// Internal plan layout shared by cqt.cu (cascade + fp32 contraction) and
// cqt_umma.cu (tcgen05 contraction).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <vector>

struct CqtOctaveDev {
  int level, hop, n_fft, n_filters, first_bin;
  float* bank;                    // device [n_fft][2*n_filters]
  std::vector<float> bank_host;   // same, host copy (tensor-path operand packing)
};

struct CqtUmmaState;    // opaque to cqt.cu
struct CqtStreamState;  // opaque to cqt.cu (cqt_umma_stream.cu)

struct saga_cqt_plan {
  int n_bins, hop, early_factor;
  int n_early_taps, n_half_taps;
  float* d_early_taps;
  float* d_early_phase = nullptr;   // polyphase image of the early filter [32][early_factor] (decimate_phase_kernel), or NULL
  float* d_half_taps;
  float early_taps2[32] = {0};   // host copies of the 32-tap (63-point symmetric) 2:1 decimators,
  float half_taps2[32] = {0};    // passed to the kernel by value
  int* d_levels;
  int* d_hops;
  int max_level;
  std::vector<CqtOctaveDev> oct;
  CqtUmmaState* umma;
  CqtStreamState* stream_tc;
};

namespace saga {

// per-level decimated signals of one exec call
struct CqtLevels {
  const float* wav;
  const int64_t* clip_offsets;
  const int64_t* clip_lens;  // NULL: every clip has max_len samples
  int64_t max_len;
  // level buffers are REFLECT-PADDED: sample s of clip c at lvl[l] + c*pitch[l] + pad[l] + s, valid for
  // s in [-pad, len_l + pad) (cqt_pad_kernel); pad[l] = n_fft/2 of the octave(s) analysed at that level
  float* const* lvl;        // [max_level+1] device buffers
  const int64_t* pitch;     // per-clip pitch of each level buffer
  const int* pad;           // per-level margin in samples (multiple of 4)
  const int32_t* clip_frames;
};

void cqt_umma_plan_init(saga_cqt_plan* p);
void cqt_umma_plan_free(saga_cqt_plan* p);
// returns SAGA_ERR_UNSUPPORTED when the plan does not fit the tensor path
// tiles with <= tail_max valid frames are skipped (the caller runs cqt_tail_kernel for them)
int cqt_umma_exec(const saga_cqt_plan* p, const CqtLevels& lv, int n_clips, int64_t max_len,
                  int64_t T_max, float* mag_out, float2* cplx_out, int64_t frame_pitch,
                  int64_t out_clip_stride, int n_split, int tail_max, cudaStream_t st);
bool cqt_umma_supported(const saga_cqt_plan* p);

// gathered rows x streamed bank (cqt_umma_stream.cu): whole transforms whose bank does not fit the resident kernel,
// and frame windows (frame_first != NULL: rows = frames [first, first + 8) of every clip, compact output)
void cqt_stream_plan_init(saga_cqt_plan* p);
void cqt_stream_plan_free(saga_cqt_plan* p);
bool cqt_stream_supported(const saga_cqt_plan* p);
int cqt_stream_exec(const saga_cqt_plan* p, const CqtLevels& lv, int n_clips, int64_t T_max,
                    const int32_t* frame_first, int frame_count, float* mag_out, float2* cplx_out,
                    int64_t frame_pitch, int64_t out_clip_stride, cudaStream_t st, int max_slices = 1,
                    float* partial = nullptr, int pstride = 0, int* slices_out = nullptr);
// peak mode of the streamed kernel (saga_cqt_peak_exec): rows packed through the device prefix sum row_start[n_clips + 1]
// of the clip frame counts, peak_out[c] = max |C| over bins and frames col_lo[c] <= t < col_hi[c] (peak_out zeroed before)
struct CqtPeakArgs {
  const int32_t* row_start;
  const int32_t* col_lo;
  const int32_t* col_hi;
  float* peak_out;
};
// several plans of equal geometry, plan i on clips [clip0[i], clip0[i] + nclips[i]) of the batch `lv` describes
int cqt_stream_exec_multi(const saga_cqt_plan* const* plans, int n_plans, const int* clip0, const int* nclips,
                          const CqtLevels& lv, int n_clips, int64_t T_max, const int32_t* frame_first, int frame_count,
                          float* mag_out, float2* cplx_out, int64_t frame_pitch, int64_t out_clip_stride,
                          cudaStream_t st, int max_slices = 1, float* partial = nullptr, int pstride = 0,
                          int* slices_out = nullptr, const CqtPeakArgs* peak = nullptr);
int cqt_stream_peak_exec(const saga_cqt_plan* p, const CqtLevels& lv, int n_clips, int64_t T_max, const CqtPeakArgs& peak,
                         cudaStream_t st);

}  // namespace saga

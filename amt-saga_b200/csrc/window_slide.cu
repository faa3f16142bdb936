// Half-window slide of the producer loop (training.py:317-328, util_audio.py:351-382) for a batch of windows:
//   audio_w.slice(h, 2h); audio_w.concat(mid_wf.section(offset + half, None, h))
// on the frame-major magnitude and phase storages, in place.  New rows [0, h) are the old rows [h, 2h) (subtractions
// and original phases included); new rows [h, 2h) are song rows [row0, row0 + h), zero past the song's end.
#include "saga_common.cuh"

namespace saga {

// One CTA per (row pair r, listed window): it reads row r + h and writes row r, then writes row r + h from the song.
// Every thread moves its own 16-byte chunks of both rows, so the read of a chunk of row r + h precedes its
// overwrite in the same thread: no other CTA touches either row, and no barrier is needed.  Chunks entirely in the
// padding columns [n_bins, pitch) are not touched; lanes of the last partial chunk past n_bins are written as 0.
__global__ void __launch_bounds__(256) window_slide_kernel(float* __restrict__ mag, float2* __restrict__ phase,
                                                           int64_t pitch, int64_t clip_stride, int half, int n_bins,
                                                           const int32_t* __restrict__ windows,
                                                           const int32_t* __restrict__ song_idx,
                                                           const int32_t* __restrict__ song_row0,
                                                           const int32_t* __restrict__ song_rows,
                                                           const float* __restrict__ song_mag,
                                                           const float2* __restrict__ song_phase,
                                                           int64_t song_clip_stride) {
  const int r = blockIdx.x, i = blockIdx.y;
  const int64_t w = windows[i];
  const bool live = r < song_rows[i];
  const int64_t lo = w * clip_stride + (int64_t)r * pitch;
  const int64_t hi = lo + (int64_t)half * pitch;
  const int64_t src = live ? (int64_t)song_idx[i] * song_clip_stride + (int64_t)(song_row0[i] + r) * pitch : 0;
  // magnitudes: 4 floats per chunk
  const int nm = (n_bins + 3) >> 2;
  for (int c = threadIdx.x; c < nm; c += blockDim.x) {
    const int k = c << 2;
    float4 v = *reinterpret_cast<const float4*>(mag + hi + k);
    float4 s = live ? __ldcs(reinterpret_cast<const float4*>(song_mag + src + k)) : make_float4(0.f, 0.f, 0.f, 0.f);
    if (k + 4 > n_bins) {
      if (k + 1 >= n_bins) v.y = s.y = 0.f;
      if (k + 2 >= n_bins) v.z = s.z = 0.f;
      v.w = s.w = 0.f;
    }
    *reinterpret_cast<float4*>(mag + lo + k) = v;
    *reinterpret_cast<float4*>(mag + hi + k) = s;
  }
  // phasors: 2 complex per chunk
  const int np_ = (n_bins + 1) >> 1;
  for (int c = threadIdx.x; c < np_; c += blockDim.x) {
    const int k = c << 1;
    float4 v = *reinterpret_cast<const float4*>(phase + hi + k);
    float4 s = live ? __ldcs(reinterpret_cast<const float4*>(song_phase + src + k)) : make_float4(0.f, 0.f, 0.f, 0.f);
    if (k + 1 >= n_bins) v.z = v.w = s.z = s.w = 0.f;
    *reinterpret_cast<float4*>(phase + lo + k) = v;
    *reinterpret_cast<float4*>(phase + hi + k) = s;
  }
}

}  // namespace saga

using namespace saga;

extern "C" int saga_window_slide_exec(float* mag, void* phase, int n_windows, int n_frames, int half, int n_bins,
                                      int64_t frame_pitch, int64_t clip_stride, const int32_t* windows,
                                      const int32_t* song_idx, const int32_t* song_row0, const int32_t* song_rows,
                                      int n_list, const float* song_mag, const void* song_phase,
                                      int64_t song_clip_stride, void* stream) {
  if (!mag || !phase || !windows || !song_idx || !song_row0 || !song_rows || !song_mag || !song_phase)
    return set_error(SAGA_ERR_INVALID, "window_slide_exec: null argument");
  if (n_windows < 0 || n_list < 0) return set_error(SAGA_ERR_INVALID, "window_slide_exec: negative count");
  if (half <= 0 || 2 * (int64_t)half > n_frames)
    return set_error(SAGA_ERR_INVALID, "window_slide_exec: need 0 < half and 2 * half <= n_frames");
  if (n_bins < 1 || n_bins > frame_pitch) return set_error(SAGA_ERR_INVALID, "window_slide_exec: need 1 <= n_bins <= frame_pitch");
  if (frame_pitch % 4) return set_error(SAGA_ERR_INVALID, "window_slide_exec: frame_pitch must be a multiple of 4");
  if (clip_stride < (int64_t)n_frames * frame_pitch || clip_stride % 4 || song_clip_stride < 0 || song_clip_stride % 4)
    return set_error(SAGA_ERR_INVALID, "window_slide_exec: bad clip stride");
  if (((reinterpret_cast<uintptr_t>(mag) | reinterpret_cast<uintptr_t>(phase) | reinterpret_cast<uintptr_t>(song_mag) |
        reinterpret_cast<uintptr_t>(song_phase)) & 15) != 0)
    return set_error(SAGA_ERR_INVALID, "window_slide_exec: storages must be 16-byte aligned");
  if (n_list > n_windows) return set_error(SAGA_ERR_INVALID, "window_slide_exec: more listed windows than windows");
  if (n_list == 0) return SAGA_OK;
  if (n_list > 65535) return set_error(SAGA_ERR_UNSUPPORTED, "window_slide_exec: at most 65535 windows per call");
  window_slide_kernel<<<dim3((unsigned)half, (unsigned)n_list), 256, 0, (cudaStream_t)stream>>>(
      mag, (float2*)phase, frame_pitch, clip_stride, half, n_bins, windows, song_idx, song_row0, song_rows, song_mag,
      (const float2*)song_phase, song_clip_stride);
  SAGA_LAUNCH_CHECK();
  return SAGA_OK;
}

/*
 * saga_b200.h -- C ABI of the B200-native AMT-SAGA feature hot path.
 *
 * The reference (RobertKajnak/AMT-SAGA) has no FFI of its own: the boundary of
 * this path is the Python class util_audio.audio_complete
 * (/root/reference/util_audio.py:32-527).  These entry points are what a ctypes
 * binding inside that class would call (INTEGRATION.md shows the stub); each
 * one names the reference lines it replaces.
 *
 * Conventions
 *   - plain C: ints, sizes, raw pointers; no torch/STL types cross the ABI.
 *   - every data pointer is a DEVICE pointer unless the name ends in _host.
 *   - the caller owns all buffers; the library only owns opaque plan handles.
 *   - `stream` is a cudaStream_t passed as void* (NULL = legacy default stream).
 *   - return value: 0 = ok, <0 = error class below; saga_last_error_string()
 *     gives the thread-local message.  Nothing throws across the boundary.
 *   - spectrogram layout is FRAME-MAJOR: element (frame t, bin k) of a clip
 *     lives at  base + t * frame_pitch + k .  Seen as [bins, frames] this is
 *     Fortran order, which is also how librosa.stft lays out its result, so the
 *     reference's `[bins, frames]` arrays are strided views of these buffers.
 *     Columns k in [n_bins, frame_pitch) are padding and are written as 0.
 */
#ifndef SAGA_B200_H
#define SAGA_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SAGA_OK 0
#define SAGA_ERR_INVALID (-1)     /* bad argument (reference: ValueError / ParameterError) */
#define SAGA_ERR_UNSUPPORTED (-2) /* valid request this build cannot run */
#define SAGA_ERR_CUDA (-3)        /* CUDA runtime error; message has the cudaError string */
#define SAGA_ERR_NOMEM (-4)

const char* saga_last_error_string(void);
/* library/ABI version, bumped on any signature change */
int saga_abi_version(void);
/* number of kernel launches this library has issued in this process (bench.py's gpu_launches) */
int64_t saga_launch_count(void);
/* Tuning / A-B switches (DESIGN.md section 5 lists them: previous-generation kernels kept as parity twins, pipeline
 * shapes).  Each is initialised once from the environment variable of the same name; saga_set_option changes it at
 * run time (value NULL = unset).  Launchers read the table, never the environment. */
int saga_set_option(const char* name, const char* value);
const char* saga_get_option(const char* name);

/* ------------------------------------------------------------------------
 * K0  PCM ingest: 16-bit PCM -> the float32 waveform audio_complete analyses.
 * The reference's waveforms are integer PCM scaled exactly once in float64:
 *   util_audio.py:894   fluidsynth `get_samples(n)[::2]` (int16, left channel of interleaved stereo)
 *   util_audio.py:776-781  `wf * (vel_max/128.0)**4 / np.abs(wf).max()`
 *   util_audio.py:964   librosa.load / soundfile: int16 / 32768
 * so the PCM itself can cross PCIe (half the bytes of float32) and
 *   wav_out[c][i] = float32( (float64(pcm[c*in_clip_stride + i*in_stride]) * mul_c) / div_c )
 * is the reference's number bit for bit.  mul_c = mul ? mul[c] : mul_all;
 * div_c = peak_div ? (double)peak_div[c] : div ? div[c] : div_all  (mul, div, peak_div: device arrays).
 * in_stride = 2 takes the left channel of an interleaved stereo stream (the reference's `[::2]`).
 * saga_pcm16_absmax_exec writes np.abs(pcm).max() per clip (int32), ready to be passed as peak_div.
 * ---------------------------------------------------------------------- */
int saga_pcm16_absmax_exec(const int16_t* pcm, int64_t in_clip_stride, int in_stride, int n_clips,
                           int64_t clip_len, int32_t* peak_out, void* stream);
int saga_pcm16_ingest_exec(const int16_t* pcm, int64_t in_clip_stride, int in_stride, float* wav_out,
                           int64_t out_clip_stride, int n_clips, int64_t clip_len, const double* mul,
                           const double* div, const int32_t* peak_div, double mul_all, double div_all,
                           void* stream);

/* ------------------------------------------------------------------------
 * K1  batched windowed real FFT -> magnitude (/ unit phasor / complex)
 * replaces librosa.stft + magphase reached from
 *   util_audio.py:127-128 (F), :147 (mag, ph), :173 (ref_mag = max(mag))
 * ---------------------------------------------------------------------- */
typedef struct saga_stft_plan saga_stft_plan;

/* n_fft in {256,...,8192} (power of two); hop >= 1; center: reflect-pad n_fft/2.
 * window_host: n_fft floats, or NULL for the periodic Hann of librosa.stft. */
int saga_stft_plan_create(saga_stft_plan** plan, int n_fft, int hop, int center,
                          const float* window_host);
int saga_stft_plan_destroy(saga_stft_plan* plan);

/* number of STFT columns librosa produces for a clip of `len` samples */
int64_t saga_stft_num_frames(const saga_stft_plan* plan, int64_t len);

/* wav:            float32 samples; clip c is wav[clip_offsets[c] .. +clip_lens[c])
 * max_len:        max over clip_lens (host knows it; sizes the grid)
 * mag_out:        [n_clips] clips, clip c at mag_out + c*out_clip_stride, frame-major
 * phase_out:      optional float2 (re,im) unit phasor exp(i*angle(F)), (1,0) where F==0;
 *                 same indexing in float2 units
 * cplx_out:       optional float2 complex STFT F
 * frame_max_out:  optional [n_clips * max_frames] per-frame max of mag
 *                 (max_frames = saga_stft_num_frames(plan, max_len))
 * clip_max_out:   optional [n_clips] max of mag per clip (== audio_complete.ref_mag)
 */
int saga_stft_exec(const saga_stft_plan* plan, const float* wav,
                   const int64_t* clip_offsets, const int64_t* clip_lens, int n_clips,
                   int64_t max_len, float* mag_out, void* phase_out, void* cplx_out,
                   int64_t frame_pitch, int64_t out_clip_stride, float* frame_max_out,
                   float* clip_max_out, void* stream);

/* The same for a FRAME RANGE per clip (the forward twin of saga_istft_rows_exec): clip c computes frames
 * t = frame0[c] + j, j in [0, n_frames), of its own centred STFT (reflect padding at the clip's true edges only) and
 * writes frame j as row dst_row0 + j of output clip dst_clip[c] (of clip c when dst_clip is NULL); output clip d is at
 * mag_out + d*out_clip_stride, out_n_frames rows of frame_pitch.  frame0 (int32) and dst_clip (int32) are device
 * arrays [n_clips]; frame0[c] >= 0.
 *   live rows (0 <= t < saga_stft_num_frames(len_c)) equal row t of saga_stft_exec on the same clip bit for bit, in
 *     magnitude and phasor (same kernels; n_fft 2048 / hop 512 uses the generic kernel, stft_exec's SAGA_STFT_RING=0);
 *   rows at or past the clip's end are zero rows: magnitude 0, phasor (0, 0);
 *   padding columns [n_bins, frame_pitch) are 0.
 * clip_max_out (optional, [n_clips], indexed by source clip) takes the atomic max over the live rows and is NOT
 * zeroed here -- unlike saga_stft_exec, which zeroes its own -- so calls over successive frame ranges accumulate a
 * clip's ref_mag.  phase_out is optional.  No per-frame maxima, no complex output. */
int saga_stft_rows_exec(const saga_stft_plan* plan, const float* wav, const int64_t* clip_offsets,
                        const int64_t* clip_lens, int n_clips, const int32_t* frame0, int n_frames,
                        const int32_t* dst_clip, int dst_row0, int out_n_frames, float* mag_out, void* phase_out,
                        int64_t frame_pitch, int64_t out_clip_stride, float* clip_max_out, void* stream);

/* ------------------------------------------------------------------------
 * K4  inverse STFT (overlap-add), replaces librosa.istft reached from
 *   util_audio.py:92-104 (wf rebuilt from mag*ph after a subtraction)
 * cplx_in frame-major float2 (or mag_in * phase_in when cplx_in is NULL);
 * wav_out clip c at c*wav_clip_stride, length hop*(T-1) when centred.
 * ---------------------------------------------------------------------- */
int saga_istft_exec(const saga_stft_plan* plan, const void* cplx_in, const float* mag_in,
                    const void* phase_in, int n_clips, int n_frames, int64_t frame_pitch,
                    int64_t in_clip_stride, float* wav_out, int64_t wav_clip_stride,
                    void* stream);

/* The same for a ROW RANGE per clip: clip c inverts rows [frame0[c], frame0[c] + n_frames) of its spectrogram as if
 * they were a clip of their own (frame0: device int32 [n_clips]).  The batched per-note step uses it to re-invert only
 * the frames a subtraction touched (util_audio.py:88-106 rebuilds the whole waveform) without first gathering them. */
int saga_istft_rows_exec(const saga_stft_plan* plan, const void* cplx_in, const float* mag_in,
                         const void* phase_in, int n_clips, const int32_t* frame0, int n_frames,
                         int64_t frame_pitch, int64_t in_clip_stride, float* wav_out,
                         int64_t wav_clip_stride, void* stream);

/* ------------------------------------------------------------------------
 * K3  generative-subtractive chain + dB epilogue, replaces
 *   util_audio.py:221-259 (subtract), :170-174 (ref_mag), :176-180 (D)
 *
 * For every window w (independent) and step j = 0..n_steps-1 (sequential):
 *   ref   = (j == 0 && ref_init && ref_init[w] >= 0) ? ref_init[w] : max(win_w)
 *   scale = normalize ? fl32(ref / guess_ref[w,j]) : 1      (numpy float32 semantics)
 *   g'    = fl32(fl32(g * scale) * overkill[w,j])
 *   win_w[:, off : off+Tg'] = relu ? max(win - g', 0) : win - g'   (Tg' clipped to T-off)
 * then  D_w = amplitude_to_db(win_w, ref = max(win_w), amin, top_db)  if D_out.
 * ---------------------------------------------------------------------- */
#define SAGA_SUB_NORMALIZE 1
#define SAGA_SUB_RELU 2
/* caller guarantees every win/guess offset is a multiple of 4 elements (16-byte vector path) */
#define SAGA_SUB_OFFSETS_ALIGNED 4
/* phase flags: SKIP_DB runs only the chain (ref_out receives every window's final max, D_out is ignored);
 * ONLY_DB runs only the dB pass over the windows as they are, with the ref_out such a call filled.
 * Lets a caller order the two phases on different streams (pipeline.py overlaps the HBM-bound dB pass with
 * the tensor-core CQT contraction). */
#define SAGA_SUB_SKIP_DB 0x100
#define SAGA_SUB_ONLY_DB 0x200

int saga_subtract_db_exec(
    float* win_mag,                /* in/out: window w at win_mag + win_offsets[w] (or w*win_stride) */
    const int64_t* win_offsets,    /* optional [n_windows] element offsets */
    int64_t win_stride,
    const float* guess_mag,        /* guess (w,j) at guess_mag + guess_offsets[w*n_steps+j] (or idx*guess_stride) */
    const int64_t* guess_offsets,  /* optional */
    int64_t guess_stride,
    const int32_t* guess_frames,   /* optional [n_windows*n_steps]; default guess_frames_all */
    int guess_frames_all,
    const int32_t* offset_frames,  /* [n_windows*n_steps] column offset of each guess (>= 0) */
    const float* overkill,         /* optional [n_windows*n_steps]; default 1 */
    const float* guess_ref,        /* optional [n_windows*n_steps] max of each guess; computed if NULL */
    const float* ref_init,         /* optional [n_windows]; <0 or NULL => max of the window */
    const float* frame_max_in,     /* optional per-frame maxima of the incoming windows (K1's
                                      frame_max_out): window w, frame t at [w*frame_max_stride + t];
                                      saves the initial full-window pass */
    int64_t frame_max_stride,
    int flags,
    float* D_out,                  /* optional, same indexing as win_mag */
    float* ref_out,                /* optional [n_windows]: max of the final window */
    int n_windows, int n_steps, int n_bins, int n_frames, int64_t frame_pitch,
    float amin, float top_db, void* stream);

/* stand-alone amplitude_to_db (util_audio.py:179) with an explicit per-clip ref
 * (ref[c] < 0 or ref == NULL => ref = max of the clip) */
int saga_amplitude_to_db_exec(const float* mag, float* D_out, const float* ref, int n_clips,
                              int n_bins, int n_frames, int64_t frame_pitch,
                              int64_t clip_stride, float amin, float top_db, void* stream);

/* ------------------------------------------------------------------------
 * K2  constant-Q transform, replaces librosa.cqt reached from
 *   util_audio.py:424-429 (slice_C)
 *
 * librosa's per-octave "rectangular STFT x sparsified FFT-domain basis" is
 * linear in the (decimated) signal, so it is folded on the host into a dense
 * real kernel bank G_o[n_fft, 2*n_filters] per octave (same numbers as
 * librosa, see DESIGN.md) and evaluated as a strided-frame GEMM
 *   C_o[t, :] = sum_n  y_o[reflect(t*hop_o + n - n_fft/2)] * G_o[n, :]
 * after the kaiser_fast decimation cascade.  The host-side plan builder
 * (amt-saga_b200/cqt_plan.py) produces this descriptor.
 * ---------------------------------------------------------------------- */
typedef struct saga_cqt_plan saga_cqt_plan;
#define SAGA_CQT_SKIP_CONTRACT 0x100
#define SAGA_CQT_SKIP_CASCADE 0x200

typedef struct saga_cqt_octave {
  int level;            /* number of 2:1 decimations after the early downsample */
  int hop;              /* hop at this level */
  int n_fft;            /* kernel length (power of two) */
  int n_filters;        /* filters in this octave */
  int first_bin;        /* output row of filter 0 (may be < 0: rows < 0 are dropped) */
  const float* bank_host; /* [n_fft][2*n_filters] (re,im interleaved per filter), all scales folded */
} saga_cqt_octave;

typedef struct saga_cqt_desc {
  int n_bins;
  int hop;                 /* hop at the input rate */
  int early_factor;        /* 1,2,4,...: single-stage decimation before the octaves */
  int n_early_taps;        /* taps[0..n) centre first, symmetric FIR, gain folded */
  const float* early_taps_host;
  int n_half_taps;         /* 2:1 decimator between levels, centre first */
  const float* half_taps_host;
  int n_octaves;
  const saga_cqt_octave* octaves;
} saga_cqt_desc;

int saga_cqt_plan_create(saga_cqt_plan** plan, const saga_cqt_desc* desc);
int saga_cqt_plan_destroy(saga_cqt_plan* plan);
/* frames librosa.cqt returns for a clip of `len` samples (min over octaves) */
int64_t saga_cqt_num_frames(const saga_cqt_plan* plan, int64_t len);
/* bytes of device scratch saga_cqt_exec needs for this batch shape */
int64_t saga_cqt_workspace_bytes(const saga_cqt_plan* plan, int n_clips, int64_t max_len);

/* clip_lens may be NULL: every clip then has exactly max_len samples (equal-length batches skip
 * the per-item length look-ups).
 * C_mag_out: |C| frame-major: (clip c, frame t, bin k) at c*out_clip_stride + t*frame_pitch + k
 * C_cplx_out: optional float2 complex CQT, same indexing in float2 units
 * impl: 0 = default: tcgen05 tensor cores with a 3xTF32 split (fp32-grade accuracy) -- the resident-bank kernel
 *       when the octave banks fit shared memory (12 bins per octave), else the streamed-bank kernel (24 / 48 / 192
 *       bins per octave: 1e-5 of peak, 2e-5 for 8192-sample kernels), else the fp32 CUDA-core path;
 *       1 = force the fp32 CUDA-core path (validation; option SAGA_CQT_STREAM=0 does the same for the streamed
 *       kernel only), 2 = force a tensor path (SAGA_ERR_UNSUPPORTED if neither fits),
 *       3 = tensor path with a single TF32 pass (measured 1.1e-4 of peak: NOT parity-grade)
 *       | SAGA_CQT_SKIP_CONTRACT: run only the decimation cascade (fills the workspace)
 *       | SAGA_CQT_SKIP_CASCADE:  run only the contraction on a workspace filled by an earlier call
 *       (the two flags let a caller time / overlap the phases separately; both calls must pass the same
 *       impl, because the cascade phase of the tensor path also writes the reflect margins of the
 *       per-level buffers in the workspace)
 * The tensor path launches one short kernel on a plan-owned side stream, forked from and joined back
 * into `stream` with per-call events: from the caller's point of view all work is ordered on `stream`. */
int saga_cqt_exec(const saga_cqt_plan* plan, const float* wav, const int64_t* clip_offsets,
                  const int64_t* clip_lens, int n_clips, int64_t max_len, float* C_mag_out,
                  void* C_cplx_out, int64_t frame_pitch, int64_t out_clip_stride,
                  void* workspace, int64_t workspace_bytes, int impl, void* stream);

/* Frame-window form of K2 for the producer loop's per-note calls (training.py:340-388): slice_C takes `C[:, s:t]`
 * of a full-window transform and `_resize`s it to 8 columns (util_audio.py:431-434, :384-409), so only columns
 * [s, s+8) are ever used.  Same cascade and reflect margins as saga_cqt_exec, but only the `frame_count` (1..8)
 * columns starting at frame_first[c] (device int32, may point past the clip: those columns are written as 0) are
 * contracted (streamed-bank tcgen05 kernel with rows = those columns; fp32 CUDA-core kernel when the plan does
 * not fit it or SAGA_CQT_STREAM=0).  Output is COMPACT: column j of clip c at C_mag_out + c*out_clip_stride +
 * j*frame_pitch. */
int saga_cqt_frames_exec(const saga_cqt_plan* plan, const float* wav, const int64_t* clip_offsets,
                         const int64_t* clip_lens, int n_clips, int64_t max_len,
                         const int32_t* frame_first, int frame_count, float* C_mag_out,
                         int64_t frame_pitch, int64_t out_clip_stride, void* workspace,
                         int64_t workspace_bytes, void* stream);

/* The same in two phases, for several plans that share ONE decimation cascade: the two note-relative transforms of a
 * per-note iteration (training.py:366-388) have a kernel bank per pitch, but pitches of equal geometry (early
 * factor, levels, kernel length) decimate the audio identically.
 *   phase 1: cascade + reflect margins for a batch of `ws_clips` clips (any plan of that geometry); frame_first /
 *            C_mag_out unused.
 *   phase 2: contraction of `frame_count` columns for clips [clip_first, clip_first + n_clips) of that batch with
 *            THIS plan's bank; frame_first / C_mag_out point at the first of those clips.
 * The caller keeps the workspace untouched between the phases and passes the same wav / clip_offsets / clip_lens /
 * max_len / workspace to both.  Plans of different geometry in one batch are the caller's error (not detectable). */
int saga_cqt_frames_shared_exec(const saga_cqt_plan* plan, const float* wav, const int64_t* clip_offsets,
                                const int64_t* clip_lens, int ws_clips, int64_t max_len, int phase,
                                int clip_first, int n_clips, const int32_t* frame_first, int frame_count,
                                float* C_mag_out, int64_t frame_pitch, int64_t out_clip_stride,
                                void* workspace, int64_t workspace_bytes, void* stream);

/* Phase 2 for SEVERAL plans of that geometry at once: plan i contracts clips [clip_first[i], clip_first[i] + clip_count[i])
 * (host arrays) of the phase-1 batch; frame_first / C_mag_out are those of the WHOLE batch (clip 0).  One tensor-core
 * launch per ~10 plans and one finish launch instead of two launches per plan.  The plans must cover every clip of the
 * batch exactly once (the finish pass of a K-split launch writes all of them). */
int saga_cqt_frames_shared_multi_exec(const saga_cqt_plan* const* plans, int n_plans, const int32_t* clip_first,
                                      const int32_t* clip_count, const float* wav, const int64_t* clip_offsets,
                                      const int64_t* clip_lens, int ws_clips, int64_t max_len,
                                      const int32_t* frame_first, int frame_count, float* C_mag_out,
                                      int64_t frame_pitch, int64_t out_clip_stride, void* workspace,
                                      int64_t workspace_bytes, void* stream);

/* Peak of a column range per clip, the whole-song normalisers of the producer loop (training.py:271-282: np.max of
 * `C[:, 0:t]`): max |C[bin, t]| over all bins and frames col_lo[c] <= t < min(col_hi[c], T_c) of clip c, written to
 * peak_out[c] (0 for an empty range).  col_lo / col_hi: device int32 [n_clips]; peak_out: device float [n_clips].
 * Same cascade, margins and contraction arithmetic as saga_cqt_exec; no image is written for the plans the streamed
 * tensor-core kernel runs (its rows are then the clips' frames packed back to back, not n_clips x T_max); the other
 * plans contract into an image inside the workspace, which saga_cqt_peak_workspace_bytes covers. */
int64_t saga_cqt_peak_workspace_bytes(const saga_cqt_plan* plan, int n_clips, int64_t max_len);
int saga_cqt_peak_exec(const saga_cqt_plan* plan, const float* wav, const int64_t* clip_offsets,
                       const int64_t* clip_lens, int n_clips, int64_t max_len,
                       const int32_t* col_lo, const int32_t* col_hi, float* peak_out,
                       void* workspace, int64_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------------
 * K5  feature gather for the classifiers (training.py:333-388)
 * ---------------------------------------------------------------------- */
/* util_audio.py:436-466 compress_bands: out[t][b] = mean(mag[t][e[b] : e[b+1]]) * inv_scale[clip]
 * (inv_scale optional, e.g. 1/song ref_mag of training.py:335-336); band_edges_host has n_bands+1 ints. */
int saga_compress_bands_exec(const float* mag, float* out, const int32_t* band_edges_host, int n_bands,
                             int n_clips, int n_frames, int64_t frame_pitch, int64_t clip_stride,
                             int64_t out_pitch, int64_t out_clip_stride, const float* inv_scale,
                             void* stream);

/* util_audio.py:469-507 resize + :334-349 section_power + training.py:347-363 normalisations in one
 * launch.  Output column j (of n_cols) copies window frame src_frames[j] (device int32; -1 = zeros), rows
 * are bins [band_min, band_min+n_rows) zero-padded past n_bins; outputs are frame-major [n_cols][out_pitch]:
 *   out_lin = mag * inv_ref,  out_log = log10(1000 mag + 1) / max(.),  out_phase = (angle(ph)+3.15)/6.3
 * (each optional; phase = float2 unit phasors, may be NULL when out_phase is NULL). */
int saga_short_window_exec(const float* mag, const void* phase, const int32_t* src_frames, int n_cols,
                           int band_min, int n_rows, int n_bins, int64_t frame_pitch, float inv_ref,
                           float* out_lin, float* out_log, float* out_phase, int64_t out_pitch, void* stream);

/* The same for a BATCH of windows (one per note of a batched step of the producer loop, training.py:337-363):
 * window w reads mag + w*clip_stride (phase likewise, float2 units), its own n_cols source frames
 * src_frames[w*n_cols ..] (device), rows [band_min[w], band_min[w]+n_rows) (band_min device array, or NULL =>
 * band_min_all for every window: the fixed C4 band of training.py:289-290), scale inv_ref[w] (or inv_ref_all),
 * and writes out_* + w*out_clip_stride.  The log10 variant is normalised by each window's own maximum. */
int saga_short_window_batch_exec(const float* mag, const void* phase, int64_t clip_stride, int64_t frame_pitch,
                                 const int32_t* src_frames, int n_cols, const int32_t* band_min, int band_min_all,
                                 int n_rows, int n_bins, const float* inv_ref, float inv_ref_all,
                                 float* out_lin, float* out_log, float* out_phase, int64_t out_pitch,
                                 int64_t out_clip_stride, int n_windows, void* stream);

/* util_audio.py:431-434 `C[:, s:t]` -> :384-409 `_resize` -> training.py:340-388 `/ ref_C` for a batch:
 *   out[w][j][k] = in[w][src_frames[w*n_cols + j]][k] * scale[w]   (k < n_bins; src -1 => zeros; scale NULL => 1)
 * in / out frame-major; columns k in [n_bins, out_pitch) are written as 0. */
int saga_gather_frames_exec(const float* in, const int32_t* src_frames, const float* scale, float* out,
                            int n_windows, int n_cols, int n_bins, int64_t frame_pitch, int64_t clip_stride,
                            int64_t out_pitch, int64_t out_clip_stride, void* stream);

/* Half-window slide of the producer loop (training.py:317-328: util_audio.py:351-365 `slice(h, 2h)` then :368-382
 * `concat(section(offset + half, None, h))`) for the n_list windows windows[i] (device int32) of a batch of
 * n_windows frame-major windows [n_windows][n_frames][frame_pitch] (mag float32, phase complex64 = float2), in place:
 *   rows [0, half)       <- rows [half, 2 half)
 *   rows [half, 2 half)  <- rows [song_row0[i], song_row0[i] + half) of song song_idx[i] of song_mag / song_phase
 *                           (stride song_clip_stride, same frame_pitch); rows j >= song_rows[i] are written as 0
 * Rows [2 half, n_frames) and windows not listed are not touched.  Padding columns: 16-byte chunks past n_bins are
 * not touched, lanes of the last partial chunk are written as 0.  All storages 16-byte aligned, frame_pitch a
 * multiple of 4.  One launch whatever n_list is. */
int saga_window_slide_exec(float* mag, void* phase, int n_windows, int n_frames, int half, int n_bins,
                           int64_t frame_pitch, int64_t clip_stride, const int32_t* windows, const int32_t* song_idx,
                           const int32_t* song_row0, const int32_t* song_rows, int n_list, const float* song_mag,
                           const void* song_phase, int64_t song_clip_stride, void* stream);

/* util_audio.py:330-332 librosa.feature.spectral_flatness(power=2): flatness_out[clip*n_frames + t] */
int saga_spectral_flatness_exec(const float* mag, float* flatness_out, int n_clips, int n_bins, int n_frames,
                                int64_t frame_pitch, int64_t clip_stride, float amin, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* SAGA_B200_H */

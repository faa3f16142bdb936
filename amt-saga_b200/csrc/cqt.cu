// K2: constant-Q transform.  Replaces librosa.cqt as reached from
// /root/reference/util_audio.py:424-429 (slice_C).
//
// librosa's recursive-downsampling CQT computes, per octave o,
//     C_o = fft_basis_o . rfft(rect-windowed frames of y_o)       (y_o: decimated signal)
// which is linear in y_o, so the host plan builder folds "rect-window FFT then
// sparse FFT-domain basis" into ONE dense real kernel bank G_o[n_fft, 2*n_filt]
// (identical numbers; DESIGN.md section "K2") and the device evaluates
//     C_o[t, :] = sum_n y_o[reflect(t*hop_o + n - n_fft/2)] * G_o[n, :]
// i.e. a GEMM whose A operand is the strided-frame (Hankel) view of the signal.
//
// This file: the kaiser_fast decimation cascade (resampy's integer-ratio case
// is a fixed symmetric FIR) and the fp32 CUDA-core contraction (impl=1, also the
// validation path for the tcgen05 kernel in cqt_umma.cu).
#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <vector>

#include "cqt_plan.cuh"
#include "saga_common.cuh"

namespace saga {

// ---------------------------------------------------------------------------
// decimation by `factor` with a symmetric FIR (taps[0] = centre), zeros outside
// the signal, output zero-padded from floor(len/factor) to ceil(len/factor)
// (librosa.resample fix=True), gain folded into the taps.
// ---------------------------------------------------------------------------
constexpr int DEC_THREADS = 256;
constexpr int DEC_PER_THREAD = 4;

__global__ void __launch_bounds__(DEC_THREADS)
decimate_kernel(const float* __restrict__ in, const int64_t* __restrict__ in_offsets,
                int64_t in_stride, const int64_t* __restrict__ clip_lens, int64_t max_len, int in_shift,
                int in_factor_total, float* __restrict__ out, int64_t out_stride,
                const float* __restrict__ taps, int n_taps, int factor, int per_thread = DEC_PER_THREAD) {
  extern __shared__ float sm[];
  const int S = n_taps - 1;
  float* tp = sm;                 // n_taps
  float* xs = sm + ((n_taps + 3) & ~3);  // tile of input
  const int clip = blockIdx.y;
  // length of this clip at the INPUT level of this stage
  int64_t len = clip_lens ? clip_lens[clip] : max_len;   // NULL = equal-length batch
  if (in_factor_total > 1) len = (len + in_factor_total - 1) / in_factor_total;  // early stage
  for (int s = 0; s < in_shift; ++s) len = (len + 1) >> 1;                        // halvings
  const int64_t n_full = len / factor;
  const int64_t n_out = (len + factor - 1) / factor;
  const int tile_out = DEC_THREADS * per_thread;
  const int64_t o0 = (int64_t)blockIdx.x * tile_out;
  if (o0 >= n_out) return;
  const float* x = in + (in_offsets ? in_offsets[clip] : (int64_t)clip * in_stride);
  for (int i = threadIdx.x; i < n_taps; i += DEC_THREADS) tp[i] = taps[i];
  const int64_t i0 = o0 * factor - S;
  const int tile_in = tile_out * factor + 2 * S;
  // the tile is stored skewed, sample i at i + i/32: consecutive outputs read samples `factor` apart, and a
  // power-of-two stride (the early stage of a 24-bins-per-octave CQT from D3 decimates by 16) would otherwise put a
  // warp's 32 reads on 32/factor banks (16-way conflicts: 9.1 ms for 600 windows; skewed: conflict-free)
  for (int i = threadIdx.x; i < tile_in; i += DEC_THREADS) {
    const int64_t s = i0 + i;
    xs[i + (i >> 5)] = (s >= 0 && s < len) ? __ldg(x + s) : 0.f;
  }
  __syncthreads();
  float* y = out + (int64_t)clip * out_stride;
  for (int u = 0; u < per_thread; ++u) {
    const int lo = threadIdx.x + u * DEC_THREADS;
    const int64_t o = o0 + lo;
    if (o >= n_out) break;
    float acc = 0.f;
    if (o < n_full) {
      const int c = lo * factor + S;          // centre sample
      acc = tp[0] * xs[c + (c >> 5)];
      for (int m = 1; m <= S; ++m) {
        const int a = c - m, b = c + m;
        acc = fmaf(tp[m], xs[a + (a >> 5)] + xs[b + (b >> 5)], acc);
      }
    }
    y[o] = acc;
  }
}

// Large early factors (a CQT that starts at a low note decimates by up to 64 first: C_velocity, training.py:382):
// the filter has 32 * factor taps, and the kernel above spends three shared-memory loads per multiply-add on it
// (112 us per pitch group of the per-note step).  Polyphase form: with j = q * factor + r,
//     y[o] = sum_r sum_{q=-16}^{15} g[q][r] * x[(o + q) * factor + r],     g[q][r] = h[|q * factor + r|]
// i.e. `factor` independent 32-tap convolutions of the stride-1 sequences x_r.  A lane owns one phase r (adjacent lanes
// = adjacent samples: every load is a coalesced 128-byte row, straight from global memory) and a run of R outputs,
// holds the 32 taps of its phase in registers and slides over R + 31 samples: 0.28 loads per multiply-add.  The
// phases are then summed across the lanes by shuffles.  factor < 32: 32 / factor runs per warp.
constexpr int DECP_Q = 16;      // taps per side and phase (kaiser_fast: 16 zero crossings)
constexpr int DECP_R = 8;       // outputs per lane
constexpr int DECP_WARPS = 8;
__global__ void __launch_bounds__(32 * DECP_WARPS, 3)
decimate_phase_kernel(const float* __restrict__ in, const int64_t* __restrict__ in_offsets, int64_t in_stride,
                      const int64_t* __restrict__ clip_lens, int64_t max_len, float* __restrict__ out,
                      int64_t out_stride, const float* __restrict__ g, int factor) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int clip = blockIdx.y;
  const int64_t len = clip_lens ? clip_lens[clip] : max_len;
  const int64_t n_full = len / factor, n_out = (len + factor - 1) / factor;
  const int fl = min(factor, 32);                    // lanes that share a run of outputs
  const int runs = 32 / fl;                          // runs per warp
  const int r0 = lane % fl, u = lane / fl;
  const int64_t o_warp = ((int64_t)blockIdx.x * DECP_WARPS + warp) * runs * DECP_R;
  if (o_warp >= n_out) return;
  const int64_t o0 = o_warp + (int64_t)u * DECP_R;
  const float* x = in + (in_offsets ? in_offsets[clip] : (int64_t)clip * in_stride);
  float acc[DECP_R];
#pragma unroll
  for (int i = 0; i < DECP_R; ++i) acc[i] = 0.f;
  for (int r = r0; r < factor; r += 32) {
    float xw[DECP_R + 2 * DECP_Q - 1];
    const int s0 = ((int)o0 - DECP_Q) * factor + r, n = (int)len;     // clips are far shorter than 2^31 samples
#pragma unroll
    for (int w = 0; w < DECP_R + 2 * DECP_Q - 1; ++w) {
      const int s = s0 + w * factor;
      xw[w] = ((unsigned)s < (unsigned)n) ? __ldg(x + s) : 0.f;
    }
    // tap by tap (each is one L1-resident load used 8 times): keeps the 32 taps out of the live register set
#pragma unroll
    for (int t = 0; t < 2 * DECP_Q; ++t) {
      const float tap = __ldg(g + t * factor + r);
#pragma unroll
      for (int i = 0; i < DECP_R; ++i) acc[i] = fmaf(tap, xw[i + t], acc[i]);
    }
  }
#pragma unroll
  for (int i = 0; i < DECP_R; ++i)
    for (int d = fl >> 1; d > 0; d >>= 1) acc[i] += __shfl_xor_sync(0xffffffffu, acc[i], d);
  // after the butterfly every lane of the run holds every sum: lane r0 stores outputs r0, r0 + fl, ...
#pragma unroll
  for (int i = 0; i < DECP_R; ++i) {
    const int64_t o = o0 + i;
    if ((i & (fl - 1)) == r0 && o < n_out) out[(int64_t)clip * out_stride + o] = o < n_full ? acc[i] : 0.f;
  }
}

static size_t decimate_smem_bytes(int n_taps, int factor, int per_thread = DEC_PER_THREAD) {
  const size_t tile_in = (size_t)DEC_THREADS * per_thread * factor + 2 * (size_t)(n_taps - 1);
  return sizeof(float) * (((n_taps + 3) & ~3) + tile_in + tile_in / 32 + 1);
}

// Factor-2 specialisation (the kaiser_fast 2:1 stage: 63 taps, S = 31), written for the packed fp32
// pipe of sm_100a.  View the input as pairs P_k = (x[2k], x[2k+1]); output o is
//     y[o] = sum_{k=-16}^{15}  te_k * x[2(o+k)] + to_k * x[2(o+k)+1],   te_k = h[|2k|] (0 for k = -16),
//                                                                        to_k = h[|2k+1|]
// i.e. 32 FFMA2 on natural (lo, hi) register pairs plus one final add of the two halves -- 33 issue
// slots per output instead of 63 scalar ones (31 symmetric pre-adds + 32 FFMA).  A thread produces
// DEC2_GROUPS x 4 consecutive outputs, each group from one 35-pair register window; the (te, to) pairs
// arrive by value (constant bank).  With fewer instructions per byte the kernel is bound by the bytes it
// keeps in flight (one-shot CTAs: load, barrier, filter), so a CTA stages DEC2_GROUPS tiles at once.
constexpr int DEC2_THREADS = 256;
constexpr int DEC2_OUT = 4;                         // consecutive outputs per register window
constexpr int DEC2_GROUPS = 2;                      // windows per thread (4: 0.63 ms, 2: 0.585 ms, 1: 0.70 ms per cascade)
constexpr int DEC2_S = 31;
constexpr int DEC2_SUB = DEC2_THREADS * DEC2_OUT;   // outputs per group
constexpr int DEC2_TILE = DEC2_SUB * DEC2_GROUPS;   // outputs per CTA
constexpr int DEC2_NIN = 2 * DEC2_TILE + 64;        // staged samples: [2*o0 - 32, 2*o0 + 2*TILE + 32)
struct Dec2Taps { float t[DEC2_S + 1]; };           // h[0..31], centre first
struct Dec2Pairs { float2 p[32]; };                 // (te_k, to_k), k = -16..15

static Dec2Pairs dec2_pairs(const float* h) {
  Dec2Pairs r;
  for (int kk = 0; kk < 32; ++kk) {
    const int k = kk - 16;
    const int me = std::abs(2 * k), mo = std::abs(2 * k + 1);
    r.p[kk] = make_float2(me <= DEC2_S ? h[me] : 0.f, h[mo]);
  }
  return r;
}

__device__ __forceinline__ unsigned long long ffma2(unsigned long long a, unsigned long long b, unsigned long long c) {
  unsigned long long d;
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c));
  return d;
}

__global__ void __launch_bounds__(DEC2_THREADS)
decimate2_kernel(const float* __restrict__ in, const int64_t* __restrict__ in_offsets, int64_t in_stride,
                 const int64_t* __restrict__ clip_lens, int64_t max_len, int in_shift, int in_factor_total,
                 float* __restrict__ out, int64_t out_stride, const Dec2Pairs taps) {
  // staged tile split by pair parity: xa = pairs 0, 2, 4, ..., xb = pairs 1, 3, 5, ...  A thread's 35-pair
  // window then is two unit-stride runs at a 16-byte lane stride: conflict-free 128-bit loads (the plain
  // contiguous layout has a 32-byte lane stride = 2-way conflicts, which made the shared-memory pipe the
  // bound: ncu r1 v7, 98.6 M wavefronts per 79 M outputs)
  __shared__ __align__(16) float2 xa[DEC2_NIN / 4];
  __shared__ __align__(16) float2 xb[DEC2_NIN / 4];
  const int clip = blockIdx.y;
  int64_t len = clip_lens ? clip_lens[clip] : max_len;   // NULL = equal-length batch
  if (in_factor_total > 1) len = (len + in_factor_total - 1) / in_factor_total;
  for (int s = 0; s < in_shift; ++s) len = (len + 1) >> 1;
  const int64_t n_full = len >> 1, n_out = (len + 1) >> 1;
  const int64_t o0 = (int64_t)blockIdx.x * DEC2_TILE;
  if (o0 >= n_out) return;
  const float* x = in + (in_offsets ? in_offsets[clip] : (int64_t)clip * in_stride);
  const int64_t i0 = 2 * o0 - 32;
  if (i0 >= 0 && i0 + DEC2_NIN <= len && ((reinterpret_cast<uintptr_t>(x + i0) & 15) == 0)) {
    const float4* src = reinterpret_cast<const float4*>(x + i0);
#pragma unroll
    for (int i = threadIdx.x; i < DEC2_NIN / 4; i += DEC2_THREADS) {
      const float4 v = __ldg(src + i);
      xa[i] = make_float2(v.x, v.y);
      xb[i] = make_float2(v.z, v.w);
    }
  } else {
    for (int i = threadIdx.x; i < DEC2_NIN; i += DEC2_THREADS) {
      const int64_t s = i0 + i;
      const float v = (s >= 0 && s < len) ? __ldg(x + s) : 0.f;      // zeros outside the signal (resampy)
      float* dst = reinterpret_cast<float*>((i & 2) ? xb : xa);
      dst[2 * (i >> 2) + (i & 1)] = v;
    }
  }
  __syncthreads();
  float* y = out + (int64_t)clip * out_stride;
#pragma unroll
  for (int grp = 0; grp < DEC2_GROUPS; ++grp) {
    // output lo = grp*SUB + 4*tid + u reads pairs lo + kk, kk = 0..31, of the staged tile
    const int p0 = grp * DEC2_SUB + 4 * threadIdx.x;          // first pair of the window (multiple of 4)
    unsigned long long w[36];
    const ulonglong2* wa = reinterpret_cast<const ulonglong2*>(xa + (p0 >> 1));
    const ulonglong2* wb = reinterpret_cast<const ulonglong2*>(xb + (p0 >> 1));
#pragma unroll
    for (int j = 0; j < 9; ++j) {
      const ulonglong2 a = wa[j], b = wb[j];
      w[4 * j] = a.x;          // pair p0 + 4j
      w[4 * j + 1] = b.x;      //         + 4j + 1
      w[4 * j + 2] = a.y;
      w[4 * j + 3] = b.y;
    }
    float acc[DEC2_OUT];
#pragma unroll
    for (int u = 0; u < DEC2_OUT; ++u) {
      unsigned long long r = 0ull;       // (+0.f, +0.f)
#pragma unroll
      for (int kk = 0; kk < 32; ++kk)
        r = ffma2(w[u + kk], *reinterpret_cast<const unsigned long long*>(&taps.p[kk]), r);
      acc[u] = __uint_as_float((unsigned)(r & 0xffffffffull)) + __uint_as_float((unsigned)(r >> 32));
    }
    const int64_t ob = o0 + p0;
    if (ob + 3 < n_full && ((reinterpret_cast<uintptr_t>(y + ob) & 15) == 0)) {
      *reinterpret_cast<float4*>(y + ob) = make_float4(acc[0], acc[1], acc[2], acc[3]);
    } else {
#pragma unroll
      for (int u = 0; u < DEC2_OUT; ++u)
        if (ob + u < n_out) y[ob + u] = (ob + u < n_full) ? acc[u] : 0.f;
    }
  }
}

// Two cascade levels in one pass: level l -> l+1 -> l+2.  The level-(l+1) tile a CTA has just produced stays in
// shared memory (same pair-parity layout) and feeds the second filter, so level l+1 is written once and never
// read back from HBM (the cascade is bound by the bytes its one-shot CTAs keep in flight, DESIGN.md section 4).
// A CTA owns DEC2X2_OUT2 = 992 outputs of level l+2; they need level-(l+1) samples [2*o2 - 32, 2*o2 + 2016) --
// exactly one 2048-output tile of the single-level kernel, computed by the same instruction sequence -- of which
// the middle 1984 are this CTA's to store (the 32-sample halos belong to the neighbours: 3 % recompute).
// Every output is produced by the same FFMA2 chain as in decimate2_kernel: results are bit-identical.
constexpr int DEC2X2_OUT2 = DEC2_TILE / 2 - 32;       // 992
static_assert(DEC2_GROUPS == 2 && DEC2X2_OUT2 % 4 == 0 && DEC2X2_OUT2 / 4 <= DEC2_THREADS, "fused tile shape");

__device__ __forceinline__ void dec2_window(const float2* xa, const float2* xb, int p0, const Dec2Pairs& taps,
                                            float (&acc)[DEC2_OUT]) {
  unsigned long long w[36];
  const ulonglong2* wa = reinterpret_cast<const ulonglong2*>(xa + (p0 >> 1));
  const ulonglong2* wb = reinterpret_cast<const ulonglong2*>(xb + (p0 >> 1));
#pragma unroll
  for (int j = 0; j < 9; ++j) {
    const ulonglong2 a = wa[j], b = wb[j];
    w[4 * j] = a.x;
    w[4 * j + 1] = b.x;
    w[4 * j + 2] = a.y;
    w[4 * j + 3] = b.y;
  }
#pragma unroll
  for (int u = 0; u < DEC2_OUT; ++u) {
    unsigned long long r = 0ull;
#pragma unroll
    for (int kk = 0; kk < 32; ++kk)
      r = ffma2(w[u + kk], *reinterpret_cast<const unsigned long long*>(&taps.p[kk]), r);
    acc[u] = __uint_as_float((unsigned)(r & 0xffffffffull)) + __uint_as_float((unsigned)(r >> 32));
  }
}

__global__ void __launch_bounds__(DEC2_THREADS)
decimate2x2_kernel(const float* __restrict__ in, const int64_t* __restrict__ in_offsets, int64_t in_stride,
                   const int64_t* __restrict__ clip_lens, int64_t max_len, int in_shift, int in_factor_total,
                   float* __restrict__ out1, int64_t out1_stride, float* __restrict__ out2, int64_t out2_stride,
                   const Dec2Pairs taps1, const Dec2Pairs taps2) {
  __shared__ __align__(16) float2 xa[DEC2_NIN / 4];
  __shared__ __align__(16) float2 xb[DEC2_NIN / 4];
  __shared__ __align__(16) float2 ya[DEC2_TILE / 4];     // level l+1 tile, even pairs
  __shared__ __align__(16) float2 yb[DEC2_TILE / 4];     //                 odd pairs
  const int clip = blockIdx.y;
  int64_t len = clip_lens ? clip_lens[clip] : max_len;
  if (in_factor_total > 1) len = (len + in_factor_total - 1) / in_factor_total;
  for (int s = 0; s < in_shift; ++s) len = (len + 1) >> 1;
  const int64_t n_full1 = len >> 1, n_out1 = (len + 1) >> 1;
  const int64_t n_full2 = n_out1 >> 1, n_out2 = (n_out1 + 1) >> 1;
  const int64_t o2_0 = (int64_t)blockIdx.x * DEC2X2_OUT2;
  if (o2_0 >= n_out2 && 2 * o2_0 >= n_out1) return;
  const int64_t o0 = 2 * o2_0 - 32;                      // first level-(l+1) sample of the tile (may be < 0)
  const float* x = in + (in_offsets ? in_offsets[clip] : (int64_t)clip * in_stride);
  const int64_t i0 = 2 * o0 - 32;
  if (i0 >= 0 && i0 + DEC2_NIN <= len && ((reinterpret_cast<uintptr_t>(x + i0) & 15) == 0)) {
    const float4* src = reinterpret_cast<const float4*>(x + i0);
#pragma unroll
    for (int i = threadIdx.x; i < DEC2_NIN / 4; i += DEC2_THREADS) {
      const float4 v = __ldg(src + i);
      xa[i] = make_float2(v.x, v.y);
      xb[i] = make_float2(v.z, v.w);
    }
  } else {
    for (int i = threadIdx.x; i < DEC2_NIN; i += DEC2_THREADS) {
      const int64_t s = i0 + i;
      const float v = (s >= 0 && s < len) ? __ldg(x + s) : 0.f;
      float* dst = reinterpret_cast<float*>((i & 2) ? xb : xa);
      dst[2 * (i >> 2) + (i & 1)] = v;
    }
  }
  __syncthreads();
  float* y1 = out1 + (int64_t)clip * out1_stride;
#pragma unroll
  for (int grp = 0; grp < DEC2_GROUPS; ++grp) {
    const int p0 = grp * DEC2_SUB + 4 * threadIdx.x;
    float acc[DEC2_OUT];
    dec2_window(xa, xb, p0, taps1, acc);
    const int64_t ob = o0 + p0;                          // multiple of 4 (possibly negative)
    // the level as the next stage sees it: zero outside [0, n_full1) (resampy zero extension; the sample
    // past floor(len/2) that librosa's fix-length appends is zero as well)
#pragma unroll
    for (int u = 0; u < DEC2_OUT; ++u)
      if (ob + u < 0 || ob + u >= n_full1) acc[u] = 0.f;
    ya[p0 >> 2] = make_float2(acc[0], acc[1]);
    yb[p0 >> 2] = make_float2(acc[2], acc[3]);
    const bool own = p0 >= 32 && p0 < DEC2_TILE - 32;     // the halo groups belong to the neighbouring CTAs
    if (own && ob < n_out1) {
      if (ob + 3 < n_out1 && ((reinterpret_cast<uintptr_t>(y1 + ob) & 15) == 0)) {
        *reinterpret_cast<float4*>(y1 + ob) = make_float4(acc[0], acc[1], acc[2], acc[3]);
      } else {
#pragma unroll
        for (int u = 0; u < DEC2_OUT; ++u)
          if (ob + u < n_out1) y1[ob + u] = acc[u];
      }
    }
  }
  __syncthreads();
  if (threadIdx.x < DEC2X2_OUT2 / 4) {
    const int p0 = 4 * threadIdx.x;
    const int64_t ob = o2_0 + p0;
    if (ob < n_out2) {
      float acc[DEC2_OUT];
      dec2_window(ya, yb, p0, taps2, acc);
      float* y2 = out2 + (int64_t)clip * out2_stride;
      if (ob + 3 < n_full2 && ((reinterpret_cast<uintptr_t>(y2 + ob) & 15) == 0)) {
        *reinterpret_cast<float4*>(y2 + ob) = make_float4(acc[0], acc[1], acc[2], acc[3]);
      } else {
#pragma unroll
        for (int u = 0; u < DEC2_OUT; ++u)
          if (ob + u < n_out2) y2[ob + u] = (ob + u < n_full2) ? acc[u] : 0.f;
      }
    }
  }
}

// ---------------------------------------------------------------------------
// fp32 contraction: CTA = 128 frames x FC output columns of one (clip, octave)
// ---------------------------------------------------------------------------
constexpr int CT_FRAMES = 128;
constexpr int CT_KC = 32;   // samples of the kernel per staged chunk
constexpr int CT_FC = 32;   // output columns (re/im interleaved) per CTA

struct ContractArgs {
  const float* sig;             // level signal base
  const int64_t* sig_offsets;   // optional per-clip offsets (level 0 without early stage = raw wav)
  int64_t sig_stride;
  const int64_t* clip_lens;     // input-rate lengths (NULL: every clip has max_len samples)
  int64_t max_len;
  int early_factor, level;
  const float* bank;            // [n_fft][ncol]
  int n_fft, ncol, hop, first_bin, n_bins;
  int zero_pad;                 // this launch also zeroes the padding columns [n_bins, frame_pitch)
  int padded;                   // sig points into a reflect-padded level buffer: samples [-n_fft/2, len + n_fft/2) are there
  float* mag_out;
  float2* cplx_out;
  int64_t frame_pitch, out_clip_stride;
  const int32_t* clip_frames;   // [n_clips] output frame count (min over octaves)
};

__global__ void __launch_bounds__(CT_FRAMES)
cqt_contract_kernel(const ContractArgs a) {
  __shared__ float ys[CT_KC][CT_FRAMES + 1];
  __shared__ __align__(16) float gs[CT_KC][CT_FC];
  const int clip = blockIdx.z;
  const int t0 = blockIdx.x * CT_FRAMES;
  const int c0 = blockIdx.y * CT_FC;
  const int T = a.clip_frames[clip];
  if (t0 >= T) return;
  int64_t len = a.clip_lens ? a.clip_lens[clip] : a.max_len;
  if (a.early_factor > 1) len = (len + a.early_factor - 1) / a.early_factor;
  for (int s = 0; s < a.level; ++s) len = (len + 1) >> 1;
  const float* y = a.sig + (a.sig_offsets ? a.sig_offsets[clip] : (int64_t)clip * a.sig_stride);
  const int tid = threadIdx.x;
  float acc[CT_FC];
#pragma unroll
  for (int f = 0; f < CT_FC; ++f) acc[f] = 0.f;
  const int half = a.n_fft >> 1;
  for (int n0 = 0; n0 < a.n_fft; n0 += CT_KC) {
    __syncthreads();
    // stage the Hankel tile ys[kk][t] = y[reflect((t0+t)*hop + n0 + kk - n_fft/2)]
    for (int i = tid; i < CT_KC * CT_FRAMES; i += CT_FRAMES) {
      const int kk = i % CT_KC, t = i / CT_KC;
      int64_t s = (int64_t)(t0 + t) * a.hop + n0 + kk - half;
      float v = 0.f;
      if (t0 + t < T) {
        if (s < 0 || s >= len) s = reflect_index(s, len);
        v = __ldg(y + s);
      }
      ys[kk][t] = v;
    }
    for (int i = tid; i < CT_KC * CT_FC; i += CT_FRAMES) {
      const int kk = i / CT_FC, f = i % CT_FC;
      gs[kk][f] = (c0 + f < a.ncol) ? __ldg(a.bank + (int64_t)(n0 + kk) * a.ncol + c0 + f) : 0.f;
    }
    __syncthreads();
#pragma unroll 4
    for (int kk = 0; kk < CT_KC; ++kk) {
      const float v = ys[kk][tid];
      const float4* g4 = reinterpret_cast<const float4*>(gs[kk]);
#pragma unroll
      for (int q = 0; q < CT_FC / 4; ++q) {
        const float4 g = g4[q];
        acc[4 * q + 0] = fmaf(v, g.x, acc[4 * q + 0]);
        acc[4 * q + 1] = fmaf(v, g.y, acc[4 * q + 1]);
        acc[4 * q + 2] = fmaf(v, g.z, acc[4 * q + 2]);
        acc[4 * q + 3] = fmaf(v, g.w, acc[4 * q + 3]);
      }
    }
  }
  const int t = t0 + tid;
  if (t >= T) return;
  const int64_t row = (int64_t)clip * a.out_clip_stride + (int64_t)t * a.frame_pitch;
#pragma unroll
  for (int f = 0; f < CT_FC; f += 2) {
    const int filt = (c0 + f) >> 1;
    const int bin = a.first_bin + filt;
    if (c0 + f < a.ncol && bin >= 0 && bin < a.n_bins) {
      const float re = acc[f], im = acc[f + 1];
      a.mag_out[row + bin] = sqrtf(re * re + im * im);
      if (a.cplx_out) a.cplx_out[row + bin] = make_float2(re, im);
    }
  }
  if (a.zero_pad && blockIdx.y == 0)
    for (int64_t k = a.n_bins; k < a.frame_pitch; ++k) {
      a.mag_out[row + k] = 0.f;
      if (a.cplx_out) a.cplx_out[row + k] = make_float2(0.f, 0.f);
    }
}

// Register-tiled form of the fp32 contraction, for the banks the resident-bank tensor path cannot hold (24 / 48 / 192
// bins per octave: the reference's per-note CQTs, training.py:340-388).  CTA = 128 frames x up to 128 output columns:
// warp w owns columns [16w, 16w + 16) -- every lane reads the same bank vector, a broadcast -- and lane l owns frames
// l, l+32, l+64, l+96: per kernel sample 4 conflict-free LDS + 4 broadcast LDS.128 feed 64 FFMA (the first version
// issued 9 LDS per 32 FFMA and staged the Hankel tile once per 32 columns instead of once per 128).
constexpr int CT2_KC = 32;
constexpr int CT2_MAXW = 8;            // warps per CTA = ceil(columns / 16), at most 8

__device__ __forceinline__ void cp_async4(float* smem_dst, const float* gsrc, bool valid) {
  const unsigned d = (unsigned)__cvta_generic_to_shared(smem_dst);
  const int sz = valid ? 4 : 0;                       // src-size 0: the 4 bytes are zero-filled, nothing is read
  asm volatile("cp.async.ca.shared.global [%0], [%1], 4, %2;" ::"r"(d), "l"(gsrc), "r"(sz) : "memory");
}

template <int FPL>                      // frames per lane: CTA tile = 32 * FPL frames
__global__ void __launch_bounds__(CT2_MAXW * 32)
cqt_contract2_kernel(const ContractArgs a, int n_warps) {
  constexpr int TF = 32 * FPL;
  constexpr int YS = CT2_KC * (TF + 1);                    // floats of the Hankel tile per stage
  const int gstride = n_warps * 16;                        // bank row pitch in shared memory = columns of this CTA
  const int STAGE = YS + CT2_KC * gstride;                 // floats per stage (sized per launch: small banks, more CTAs per SM)
  extern __shared__ __align__(16) float ct2_smem[];   // two stages: [ys | gs] [ys | gs], filled by cp.async
  const int clip = blockIdx.z;
  const int t0 = blockIdx.x * TF;
  const int c0 = blockIdx.y * (n_warps * 16);
  const int T = a.clip_frames[clip];
  if (t0 >= T) return;
  int64_t len = a.clip_lens ? a.clip_lens[clip] : a.max_len;
  if (a.early_factor > 1) len = (len + a.early_factor - 1) / a.early_factor;
  for (int s = 0; s < a.level; ++s) len = (len + 1) >> 1;
  const float* y = a.sig + (a.sig_offsets ? a.sig_offsets[clip] : (int64_t)clip * a.sig_stride);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, nthr = n_warps * 32;
  const int ncols_cta = n_warps * 16;
  float acc[FPL][16];
#pragma unroll
  for (int j = 0; j < FPL; ++j)
#pragma unroll
    for (int f = 0; f < 16; ++f) acc[j][f] = 0.f;
  const int half = a.n_fft >> 1;
  const int nT = min(TF, T - t0);        // valid frames of this tile
  const int n_chunks = a.n_fft / CT2_KC;
  const bool vec_bank = (a.ncol & 3) == 0 && ((reinterpret_cast<uintptr_t>(a.bank) & 15) == 0);

  // Hankel tile ys[kk][t] = y[(t0+t)*hop + n0 + kk - n_fft/2] and bank rows gs[kk][c] of one K-chunk, copied
  // asynchronously (the level buffers carry their reflect margins: cqt_pad_kernel); the next chunk's copies are
  // in flight while this chunk is contracted
  auto issue = [&](int chunk, int stage) {
    float* ys = ct2_smem + stage * STAGE;
    float* gs = ys + YS;
    const int n0 = chunk * CT2_KC;
    if (a.padded) {
      // thread = (kk = lane, t = warp, warp + n_warps, ...): one pointer pair advanced by a constant step
      const float* src = y + (int64_t)t0 * a.hop + n0 - half + (int64_t)warp * a.hop + lane;
      float* dst = ys + lane * (TF + 1) + warp;
      const int64_t sstep = (int64_t)n_warps * a.hop;
      for (int t = warp; t < TF; t += n_warps, src += sstep, dst += n_warps) cp_async4(dst, src, t < nT);
    } else {
      for (int i = tid; i < CT2_KC * TF; i += nthr) {
        const int kk = i % CT2_KC, t = i / CT2_KC;
        int64_t s = (int64_t)(t0 + t) * a.hop + n0 + kk - half;
        if (t < nT && (s < 0 || s >= len)) s = reflect_index(s, len);
        cp_async4(ys + kk * (TF + 1) + t, y + (t < nT ? s : 0), t < nT);
      }
    }
    if (vec_bank) {
      // bank rows are 16-byte aligned (ncol and c0 multiples of 4): 4 columns per copy
      const int q_per_row = ncols_cta >> 2;
      for (int i = tid; i < CT2_KC * q_per_row; i += nthr) {
        const int kk = i / q_per_row, f = (i % q_per_row) << 2;
        const bool ok = c0 + f < a.ncol;          // ncol % 4 == 0: a vector is entirely inside or outside
        const unsigned d = (unsigned)__cvta_generic_to_shared(gs + kk * gstride + f);
        const float* g = a.bank + (int64_t)(n0 + kk) * a.ncol + (ok ? c0 + f : 0);
        const int sz = ok ? 16 : 0;
        asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(d), "l"(g), "r"(sz) : "memory");
      }
    } else {
      for (int i = tid; i < CT2_KC * ncols_cta; i += nthr) {
        const int kk = i / ncols_cta, f = i % ncols_cta;
        const bool ok = c0 + f < a.ncol;
        cp_async4(gs + kk * gstride + f, a.bank + (int64_t)(n0 + kk) * a.ncol + (ok ? c0 + f : 0), ok);
      }
    }
    asm volatile("cp.async.commit_group;" ::: "memory");
  };

  issue(0, 0);
  for (int c = 0; c < n_chunks; ++c) {
    if (c + 1 < n_chunks) {
      issue(c + 1, (c + 1) & 1);
      asm volatile("cp.async.wait_group 1;" ::: "memory");
    } else {
      asm volatile("cp.async.wait_group 0;" ::: "memory");
    }
    __syncthreads();
    const float* ys = ct2_smem + (c & 1) * STAGE;
    const float* gs = ys + YS;
#pragma unroll 4
    for (int kk = 0; kk < CT2_KC; ++kk) {
      float v[FPL];
#pragma unroll
      for (int j = 0; j < FPL; ++j) v[j] = ys[kk * (TF + 1) + lane + 32 * j];
      const float4* g4 = reinterpret_cast<const float4*>(gs + kk * gstride + warp * 16);
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const float4 g = g4[q];
#pragma unroll
        for (int j = 0; j < FPL; ++j) {
          acc[j][4 * q + 0] = fmaf(v[j], g.x, acc[j][4 * q + 0]);
          acc[j][4 * q + 1] = fmaf(v[j], g.y, acc[j][4 * q + 1]);
          acc[j][4 * q + 2] = fmaf(v[j], g.z, acc[j][4 * q + 2]);
          acc[j][4 * q + 3] = fmaf(v[j], g.w, acc[j][4 * q + 3]);
        }
      }
    }
    __syncthreads();       // everyone is done with this stage before chunk c + 2 is copied over it
  }
#pragma unroll
  for (int j = 0; j < FPL; ++j) {
    const int t = t0 + lane + 32 * j;
    if (t >= T) continue;
    const int64_t row = (int64_t)clip * a.out_clip_stride + (int64_t)t * a.frame_pitch;
#pragma unroll
    for (int f = 0; f < 16; f += 2) {
      const int col = c0 + warp * 16 + f;
      const int bin = a.first_bin + (col >> 1);
      if (col < a.ncol && bin >= 0 && bin < a.n_bins) {
        const float re = acc[j][f], im = acc[j][f + 1];
        a.mag_out[row + bin] = sqrtf(re * re + im * im);
        if (a.cplx_out) a.cplx_out[row + bin] = make_float2(re, im);
      }
    }
    if (a.zero_pad && blockIdx.y == 0 && warp == 0)
      for (int64_t k = a.n_bins; k < a.frame_pitch; ++k) {
        a.mag_out[row + k] = 0.f;
        if (a.cplx_out) a.cplx_out[row + k] = make_float2(0.f, 0.f);
      }
  }
}

template <int FPL>
static size_t ct2_smem_bytes(int n_warps) { return sizeof(float) * 2 * (size_t)(CT2_KC * (32 * FPL + 1) + CT2_KC * n_warps * 16); }

// per-clip output frame count = min over octaves of 1 + len_o // hop_o (librosa __trim_stack)
__global__ void cqt_frames_kernel(const int64_t* clip_lens, int64_t max_len, int n_clips, int early_factor,
                                  const int* levels, const int* hops, int n_oct, int32_t* out) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= n_clips) return;
  int64_t len0 = clip_lens ? clip_lens[c] : max_len;
  if (len0 <= 0) { out[c] = 0; return; }
  if (early_factor > 1) len0 = (len0 + early_factor - 1) / early_factor;
  int64_t best = INT32_MAX;
  for (int o = 0; o < n_oct; ++o) {
    int64_t len = len0;
    for (int s = 0; s < levels[o]; ++s) len = (len + 1) >> 1;
    best = min(best, 1 + len / hops[o]);
  }
  out[c] = (int32_t)best;
}

static int64_t level_len(int64_t len, int early_factor, int level) {
  if (len <= 0) return 0;
  if (early_factor > 1) len = (len + early_factor - 1) / early_factor;
  for (int s = 0; s < level; ++s) len = (len + 1) >> 1;
  return len;
}

// reflect margin kept on both sides of every clip of a level buffer: n_fft/2 of the octave analysed there
int cqt_level_pad(const saga_cqt_plan* p, int level) {
  int pad = 0;
  for (auto& o : p->oct)
    if (o.level == level) pad = std::max(pad, ((o.n_fft / 2) + 3) & ~3);
  return pad;
}

int64_t cqt_level_pitch(const saga_cqt_plan* p, int level, int64_t max_len) {
  return (level_len(max_len, p->early_factor, level) + 2 * cqt_level_pad(p, level) + 3 + 4) & ~int64_t(3);
}

// ---------------------------------------------------------------------------
// reflect margins of the level buffers (np.pad(mode='reflect') of librosa's centred framing), written
// once per level so that the contraction kernels read plain strided tiles.  Level 0 without an early
// stage is the caller's wav: that level is copied into its padded buffer as well.
// ---------------------------------------------------------------------------
constexpr int PAD_MAX_LEVELS = 16;
struct PadArgs {
  float* lvl[PAD_MAX_LEVELS];
  int64_t pitch[PAD_MAX_LEVELS];
  int pad[PAD_MAX_LEVELS];
  const float* wav;              // raw level 0 source (early_factor == 1), else NULL
  const int64_t* clip_offsets;
  const int64_t* clip_lens;
  int64_t max_len;
  int early_factor;
};

__global__ void __launch_bounds__(256) cqt_pad_kernel(const PadArgs a) {
  const int l = blockIdx.x, clip = blockIdx.y;
  const int pad = a.pad[l];
  if (pad == 0 || !a.lvl[l]) return;
  int64_t len = a.clip_lens ? a.clip_lens[clip] : a.max_len;
  if (len <= 0) return;
  if (a.early_factor > 1) len = (len + a.early_factor - 1) / a.early_factor;
  for (int s = 0; s < l; ++s) len = (len + 1) >> 1;
  float* dst = a.lvl[l] + (int64_t)clip * a.pitch[l] + pad;
  const bool raw = (l == 0 && a.wav != nullptr);
  const float* src = raw ? a.wav + a.clip_offsets[clip] : dst;
  const int tid = blockIdx.z * blockDim.x + threadIdx.x, nth = gridDim.z * blockDim.x;
  if (raw)
    for (int64_t i = tid; i < len; i += nth) dst[i] = __ldg(src + i);
  for (int i = tid; i < 2 * pad; i += nth) {
    const int64_t s = i < pad ? (int64_t)i - pad : len + (i - pad);
    dst[s] = src[reflect_index(s, len)];
  }
}


// ---------------------------------------------------------------------------
// Frame-window contraction: only `frame_count` (<= 8) consecutive CQT columns per clip, starting at
// frame_first[clip].  The producer loop takes `C[:, s:t]` of a full-window transform and `_resize`s it to 8
// columns (util_audio.py:431-434, :384-409; training.py:340-388): whatever t - s is, every column it keeps lies
// in [s, s + 8), so 250 of the 258 columns of each of its five per-note CQTs are never looked at.  Here a warp
// owns 32 filters (lane = filter, its (re, im) bank columns are one 8-byte load) and keeps the 8 frames in
// registers: per 4 kernel samples 4 coalesced bank loads + 8 broadcast 16-byte signal loads feed 64 FFMA.  The
// decimation cascade and the reflect margins are the ones of the full transform, so interior and edge columns
// are the same numbers (fp32 summation order aside).  Output is COMPACT: [clip][frame_count][frame_pitch].
// ---------------------------------------------------------------------------
constexpr int FW_MAXF = 8;
constexpr int FW_MAX_OCT = 12;
constexpr int FW_MAX_KS = 32;          // K slices at most
constexpr int FW_TARGET_CTAS = 600;    // ~4 CTAs per SM
struct FrameWinArgs {
  const float* sig[FW_MAX_OCT];        // level buffer of the octave + its margin: sample 0 of clip 0
  int64_t sig_stride[FW_MAX_OCT];
  const float* bank[FW_MAX_OCT];
  int n_fft[FW_MAX_OCT], n_filt[FW_MAX_OCT], hop[FW_MAX_OCT], first_bin[FW_MAX_OCT];
  int n_bins, frame_count;
  const int32_t* frame_first;
  const int32_t* clip_frames;
  float* mag_out;
  int64_t frame_pitch, out_clip_stride;
  // split-K for small batches (a pitch group of the note-relative transforms is a few dozen clips): the kernel
  // length is cut into `ks` slices (blockIdx.x = column block * ks + slice), the slices' sums go to `partial`
  // [slice][clip][octave][pstride filters][8 frames][re, im] and cqt_frame_window_finish_kernel adds them in slice
  // order (deterministic) and takes the magnitudes
  int ks, n_clips, n_oct, pstride;
  float* partial;
};

template <bool VEC>
__global__ void __launch_bounds__(256) cqt_frame_window_kernel(const FrameWinArgs a) {
  const int oct = blockIdx.y, clip = blockIdx.z;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int nf = a.n_filt[oct];
  const int slice = blockIdx.x % a.ks, cblock = blockIdx.x / a.ks;
  const int filt0 = (cblock * (blockDim.x >> 5) + warp) * 32;
  if (filt0 >= nf) return;
  const int filt = min(filt0 + lane, nf - 1);
  const int T = a.clip_frames[clip], f0 = a.frame_first[clip];
  const int n_fft = a.n_fft[oct], hop = a.hop[oct];
  const float* sig = a.sig[oct] + (int64_t)clip * a.sig_stride[oct] - (n_fft >> 1);
  const float* y[FW_MAXF];
#pragma unroll
  for (int f = 0; f < FW_MAXF; ++f) {
    const int t = max(min(f0 + f, T - 1), 0);       // frames past the clip re-read the last one; zeroed on output
    y[f] = sig + (int64_t)t * hop;
  }
  float acc[FW_MAXF][2];
#pragma unroll
  for (int f = 0; f < FW_MAXF; ++f) acc[f][0] = acc[f][1] = 0.f;
  if (T > 0) {
    const float2* bk = reinterpret_cast<const float2*>(a.bank[oct]) + filt;
    float4 x[FW_MAXF], xn[FW_MAXF];
    float2 b[4], bn[4];
    auto load = [&](int k0, float4 (&xx)[FW_MAXF], float2 (&bb)[4]) {
#pragma unroll
      for (int f = 0; f < FW_MAXF; ++f) {
        if (VEC) {
          xx[f] = __ldg(reinterpret_cast<const float4*>(y[f] + k0));
        } else {
          xx[f] = make_float4(__ldg(y[f] + k0), __ldg(y[f] + k0 + 1), __ldg(y[f] + k0 + 2), __ldg(y[f] + k0 + 3));
        }
      }
#pragma unroll
      for (int i = 0; i < 4; ++i) bb[i] = __ldg(bk + (int64_t)(k0 + i) * nf);
    };
    const int k_lo = slice * (n_fft / a.ks), k_hi = k_lo + n_fft / a.ks;
    load(k_lo, x, b);
    for (int k0 = k_lo; k0 < k_hi; k0 += 4) {
      if (k0 + 4 < k_hi) load(k0 + 4, xn, bn);
#pragma unroll
      for (int f = 0; f < FW_MAXF; ++f) {
        acc[f][0] = fmaf(x[f].x, b[0].x, acc[f][0]); acc[f][1] = fmaf(x[f].x, b[0].y, acc[f][1]);
        acc[f][0] = fmaf(x[f].y, b[1].x, acc[f][0]); acc[f][1] = fmaf(x[f].y, b[1].y, acc[f][1]);
        acc[f][0] = fmaf(x[f].z, b[2].x, acc[f][0]); acc[f][1] = fmaf(x[f].z, b[2].y, acc[f][1]);
        acc[f][0] = fmaf(x[f].w, b[3].x, acc[f][0]); acc[f][1] = fmaf(x[f].w, b[3].y, acc[f][1]);
      }
#pragma unroll
      for (int f = 0; f < FW_MAXF; ++f) x[f] = xn[f];
#pragma unroll
      for (int i = 0; i < 4; ++i) b[i] = bn[i];
    }
  }
  if (a.ks > 1) {
    if (filt0 + lane < nf) {
      float4* dst = reinterpret_cast<float4*>(
          a.partial + ((((int64_t)slice * a.n_clips + clip) * a.n_oct + oct) * a.pstride + filt0 + lane) * (2 * FW_MAXF));
#pragma unroll
      for (int f = 0; f < FW_MAXF; f += 2) dst[f >> 1] = make_float4(acc[f][0], acc[f][1], acc[f + 1][0], acc[f + 1][1]);
    }
    return;
  }
  const int bin = a.first_bin[oct] + filt0 + lane;
  const bool ok = filt0 + lane < nf && bin >= 0 && bin < a.n_bins;
#pragma unroll
  for (int f = 0; f < FW_MAXF; ++f) {
    if (f >= a.frame_count) break;
    const int64_t row = (int64_t)clip * a.out_clip_stride + (int64_t)f * a.frame_pitch;
    const bool live = f0 + f >= 0 && f0 + f < T;
    if (ok) a.mag_out[row + bin] = live ? sqrtf(acc[f][0] * acc[f][0] + acc[f][1] * acc[f][1]) : 0.f;
    if (oct == 0 && blockIdx.x == 0 && warp == 0)
      for (int64_t k = a.n_bins + lane; k < a.frame_pitch; k += 32) a.mag_out[row + k] = 0.f;
  }
}

__global__ void __launch_bounds__(256) cqt_frame_window_finish_kernel(const FrameWinArgs a) {
  const int oct = blockIdx.y, clip = blockIdx.z;
  const int filt = blockIdx.x * 256 + threadIdx.x;
  const int T = a.clip_frames[clip], f0 = a.frame_first[clip];
  if (oct == 0 && blockIdx.x == 0)
    for (int f = 0; f < a.frame_count; ++f)
      for (int64_t k = a.n_bins + threadIdx.x; k < a.frame_pitch; k += 256)
        a.mag_out[(int64_t)clip * a.out_clip_stride + (int64_t)f * a.frame_pitch + k] = 0.f;
  if (filt >= a.n_filt[oct]) return;
  const int bin = a.first_bin[oct] + filt;
  if (bin < 0 || bin >= a.n_bins) return;
  float acc[2 * FW_MAXF];
#pragma unroll
  for (int i = 0; i < 2 * FW_MAXF; ++i) acc[i] = 0.f;
  for (int sl = 0; sl < a.ks; ++sl) {
    const float4* src = reinterpret_cast<const float4*>(
        a.partial + ((((int64_t)sl * a.n_clips + clip) * a.n_oct + oct) * a.pstride + filt) * (2 * FW_MAXF));
#pragma unroll
    for (int q = 0; q < FW_MAXF / 2; ++q) {
      const float4 v = src[q];
      acc[4 * q] += v.x; acc[4 * q + 1] += v.y; acc[4 * q + 2] += v.z; acc[4 * q + 3] += v.w;
    }
  }
  for (int f = 0; f < a.frame_count; ++f) {
    const bool live = f0 + f >= 0 && f0 + f < T;
    a.mag_out[(int64_t)clip * a.out_clip_stride + (int64_t)f * a.frame_pitch + bin] =
        live ? sqrtf(acc[2 * f] * acc[2 * f] + acc[2 * f + 1] * acc[2 * f + 1]) : 0.f;
  }
}

constexpr int TAIL_MAX = 16;   // partial tiles up to this many frames go to cqt_tail_kernel (cqt_umma.cu), not to the MMAs

}  // namespace saga

using namespace saga;

extern "C" int saga_cqt_plan_create(saga_cqt_plan** out, const saga_cqt_desc* d) {
  if (!out || !d) return set_error(SAGA_ERR_INVALID, "cqt_plan_create: null argument");
  *out = nullptr;
  if (d->n_octaves < 1 || !d->octaves || d->n_bins < 1 || d->hop < 1 || d->early_factor < 1)
    return set_error(SAGA_ERR_INVALID, "cqt_plan_create: bad descriptor");
  if (d->early_factor > 1 && (!d->early_taps_host || d->n_early_taps < 1))
    return set_error(SAGA_ERR_INVALID, "cqt_plan_create: early taps missing");
  saga_cqt_plan* p = new saga_cqt_plan();
  p->n_bins = d->n_bins;
  p->hop = d->hop;
  p->early_factor = d->early_factor;
  p->n_early_taps = d->n_early_taps;
  p->n_half_taps = d->n_half_taps;
  p->d_early_taps = p->d_half_taps = nullptr;
  p->d_levels = p->d_hops = nullptr;
  p->max_level = 0;
  p->umma = nullptr;
  p->stream_tc = nullptr;
  auto fail = [&](int rc) { saga_cqt_plan_destroy(p); return rc; };
  if (d->early_factor > 1) {
    if (cudaMalloc(&p->d_early_taps, sizeof(float) * d->n_early_taps) != cudaSuccess)
      return fail(set_error(SAGA_ERR_NOMEM, "cqt_plan_create: cudaMalloc"));
    cudaMemcpy(p->d_early_taps, d->early_taps_host, sizeof(float) * d->n_early_taps, cudaMemcpyHostToDevice);
    for (int i = 0; i < 32 && i < d->n_early_taps; ++i) p->early_taps2[i] = d->early_taps_host[i];
    const int F = d->early_factor;
    if (F >= 4 && (F & (F - 1)) == 0 && d->n_early_taps == DECP_Q * F) {
      std::vector<float> g((size_t)2 * DECP_Q * F, 0.f);
      for (int q = -DECP_Q; q < DECP_Q; ++q)
        for (int r = 0; r < F; ++r) {
          const int j = std::abs(q * F + r);
          if (j < d->n_early_taps) g[(size_t)(q + DECP_Q) * F + r] = d->early_taps_host[j];
        }
      if (cudaMalloc(&p->d_early_phase, sizeof(float) * g.size()) != cudaSuccess)
        return fail(set_error(SAGA_ERR_NOMEM, "cqt_plan_create: cudaMalloc"));
      cudaMemcpy(p->d_early_phase, g.data(), sizeof(float) * g.size(), cudaMemcpyHostToDevice);
    }
  }
  std::vector<int> levels, hops;
  for (int o = 0; o < d->n_octaves; ++o) {
    const saga_cqt_octave& s = d->octaves[o];
    if (s.level < 0 || s.hop < 1 || s.n_fft < 2 || (s.n_fft & (s.n_fft - 1)) || s.n_filters < 1 || !s.bank_host)
      return fail(set_error(SAGA_ERR_INVALID, "cqt_plan_create: bad octave %d", o));
    CqtOctaveDev od;
    od.level = s.level; od.hop = s.hop; od.n_fft = s.n_fft; od.n_filters = s.n_filters;
    od.first_bin = s.first_bin; od.bank = nullptr;
    const size_t n = (size_t)s.n_fft * 2 * s.n_filters;
    if (cudaMalloc(&od.bank, sizeof(float) * n) != cudaSuccess)
      return fail(set_error(SAGA_ERR_NOMEM, "cqt_plan_create: cudaMalloc"));
    cudaMemcpy(od.bank, s.bank_host, sizeof(float) * n, cudaMemcpyHostToDevice);
    od.bank_host.assign(s.bank_host, s.bank_host + n);
    p->oct.push_back(od);
    p->max_level = std::max(p->max_level, s.level);
    levels.push_back(s.level);
    hops.push_back(s.hop);
  }
  if (p->max_level > 0) {
    if (!d->half_taps_host || d->n_half_taps < 1)
      return fail(set_error(SAGA_ERR_INVALID, "cqt_plan_create: half-band taps missing"));
    if (cudaMalloc(&p->d_half_taps, sizeof(float) * d->n_half_taps) != cudaSuccess)
      return fail(set_error(SAGA_ERR_NOMEM, "cqt_plan_create: cudaMalloc"));
    cudaMemcpy(p->d_half_taps, d->half_taps_host, sizeof(float) * d->n_half_taps, cudaMemcpyHostToDevice);
    for (int i = 0; i < 32 && i < d->n_half_taps; ++i) p->half_taps2[i] = d->half_taps_host[i];
  }
  cudaMalloc(&p->d_levels, sizeof(int) * levels.size());
  cudaMalloc(&p->d_hops, sizeof(int) * hops.size());
  cudaMemcpy(p->d_levels, levels.data(), sizeof(int) * levels.size(), cudaMemcpyHostToDevice);
  cudaMemcpy(p->d_hops, hops.data(), sizeof(int) * hops.size(), cudaMemcpyHostToDevice);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return fail(set_error(SAGA_ERR_CUDA, "cqt_plan_create: %s", cudaGetErrorString(e)));
  cqt_umma_plan_init(p);  // tensor-core side tables (no-op when the plan does not fit that path)
  cqt_stream_plan_init(p);  // streamed-bank tensor path: packed banks per (octave, column group)
  *out = p;
  return SAGA_OK;
}

extern "C" int saga_cqt_plan_destroy(saga_cqt_plan* p) {
  if (!p) return SAGA_OK;
  cqt_umma_plan_free(p);
  cqt_stream_plan_free(p);
  cudaFree(p->d_early_taps);
  cudaFree(p->d_early_phase);
  cudaFree(p->d_half_taps);
  cudaFree(p->d_levels);
  cudaFree(p->d_hops);
  for (auto& o : p->oct) cudaFree(o.bank);
  delete p;
  return SAGA_OK;
}

extern "C" int64_t saga_cqt_num_frames(const saga_cqt_plan* p, int64_t len) {
  if (!p || len <= 0) return 0;
  int64_t best = INT64_MAX;
  for (auto& o : p->oct) best = std::min(best, 1 + level_len(len, p->early_factor, o.level) / o.hop);
  return best;
}

// workspace layout: [int32 clip_frames[n_clips] padded to 256 B][level 0 (only if early_factor>1)]
// [level 1] ... [level max_level], each n_clips * pitch(level) floats
static int64_t ws_header_bytes(int n_clips) { return (((int64_t)n_clips * 4) + 255) & ~int64_t(255); }

extern "C" int64_t saga_cqt_workspace_bytes(const saga_cqt_plan* p, int n_clips, int64_t max_len) {
  if (!p || n_clips <= 0 || max_len <= 0) return 256;
  int64_t b = ws_header_bytes(n_clips);
  for (int l = 0; l <= p->max_level; ++l)
    b += (int64_t)n_clips * cqt_level_pitch(p, l, max_len) * 4;
  // split-K scratch of saga_cqt_frames_exec: slices * clips * octaves <= 2 * FW_TARGET_CTAS whenever it splits
  int max_filt = 0;
  for (auto& o : p->oct) max_filt = std::max(max_filt, o.n_filters);
  b += (int64_t)2 * FW_TARGET_CTAS * ((max_filt + 31) & ~31) * 2 * FW_MAXF * 4 + 256;
  return b + 256;
}

static int cqt_exec_impl(const saga_cqt_plan* p, const float* wav, const int64_t* clip_offsets,
                         const int64_t* clip_lens, int n_clips, int64_t max_len, float* C_mag_out,
                         void* C_cplx_out, int64_t frame_pitch, int64_t out_clip_stride,
                         void* workspace, int64_t workspace_bytes, int impl, void* stream,
                         const int32_t* frame_first, int frame_count, int ws_clips = 0, int clip_first = 0) {
  if (!p || !wav || !clip_offsets || !C_mag_out || !workspace)
    return set_error(SAGA_ERR_INVALID, "cqt_exec: null argument");
  if (frame_pitch < p->n_bins) return set_error(SAGA_ERR_INVALID, "cqt_exec: frame_pitch < n_bins");
  if (n_clips <= 0 || max_len <= 0) return SAGA_OK;
  // ws_clips > 0: the workspace was laid out (and its cascade run) for a batch of ws_clips clips, of which this call
  // contracts clips [clip_first, clip_first + n_clips) -- saga_cqt_frames_shared_exec
  const int nc_ws = ws_clips > 0 ? ws_clips : n_clips;
  if (clip_first < 0 || clip_first + n_clips > nc_ws) return set_error(SAGA_ERR_INVALID, "cqt_exec: clip range outside the workspace batch");
  if (workspace_bytes < saga_cqt_workspace_bytes(p, nc_ws, max_len))
    return set_error(SAGA_ERR_INVALID, "cqt_exec: workspace too small");
  if ((reinterpret_cast<uintptr_t>(workspace) & 255) != 0)
    return set_error(SAGA_ERR_INVALID, "cqt_exec: workspace must be 256-byte aligned");
  cudaStream_t st = (cudaStream_t)stream;
  const int64_t T_max = saga_cqt_num_frames(p, max_len);
  const bool do_cascade = !(impl & SAGA_CQT_SKIP_CASCADE), do_contract = !(impl & SAGA_CQT_SKIP_CONTRACT);
  impl &= 0xFF;

  // ---- carve the workspace -------------------------------------------------------
  char* ws = (char*)workspace;
  int32_t* clip_frames = (int32_t*)ws;
  ws += ws_header_bytes(nc_ws);
  if (p->max_level + 1 > PAD_MAX_LEVELS) return set_error(SAGA_ERR_UNSUPPORTED, "cqt_exec: too many levels");
  std::vector<float*> lvl(p->max_level + 1, nullptr);   // padded buffers; sample 0 of a clip at + pad[l]
  std::vector<int64_t> pitch(p->max_level + 1, 0);
  std::vector<int> pad(p->max_level + 1, 0);
  for (int l = 0; l <= p->max_level; ++l) {
    pitch[l] = cqt_level_pitch(p, l, max_len);
    pad[l] = cqt_level_pad(p, l);
    lvl[l] = (float*)ws + (int64_t)clip_first * pitch[l];
    ws += (int64_t)nc_ws * pitch[l] * 4;
  }
  if (clip_first > 0 || ws_clips > 0) {
    if (do_cascade && (clip_first != 0 || n_clips != nc_ws))
      return set_error(SAGA_ERR_INVALID, "cqt_exec: the cascade runs on the whole workspace batch");
    clip_frames += clip_first;
  }
  const bool raw0 = (p->early_factor == 1);   // level 0 = the caller's wav (copied into lvl[0] by the pad pass)

  if (do_cascade) {      // (a contraction-only call finds the frame counts of the cascade call in the workspace header)
    cqt_frames_kernel<<<(n_clips + 127) / 128, 128, 0, st>>>(clip_lens, max_len, n_clips, p->early_factor,
                                                             p->d_levels, p->d_hops, (int)p->oct.size(),
                                                             clip_frames);
    SAGA_LAUNCH_CHECK();
  }

  // ---- decimation cascade ----------------------------------------------------------
  const int tile_out = DEC_THREADS * DEC_PER_THREAD;
  // levels 1..max_level: 2:1 stages, fused two at a time (decimate2x2_kernel) when both are the 63-tap filter
  const bool fuse = p->n_half_taps == DEC2_S + 1 && SAGA_OPT("SAGA_DEC_NO_FUSE") == nullptr;
  // Which pairs: bit i set = the pair whose FIRST output is level i is fused.  Default: every pair (one stream, kernel
  // after kernel: cascade 0.582 -> 0.516 ms, step 3.038 -> 2.971 ms; when the CQT chain ran beside the STFT chain on a
  // second stream only the two large pairs paid -- profiles/microbench/cascade_fuse_b200.txt).  SAGA_DEC_FUSE_MASK
  // overrides (tuning aid).
  unsigned fuse_mask = ~0u;
  if (const char* e = SAGA_OPT("SAGA_DEC_FUSE_MASK")) fuse_mask = (unsigned)strtoul(e, nullptr, 0);
  int l = 1;
  // the early stage itself can be the first half of a fused pair (early factor 2 with the same kind of filter)
  const bool early_is_dec2 = do_cascade && p->early_factor == 2 && p->n_early_taps == DEC2_S + 1;
  bool early_done = !(do_cascade && p->early_factor > 1);
  if (early_is_dec2 && fuse && (fuse_mask & 1u) && p->max_level >= 1) {
    const int64_t n_out2 = level_len(max_len, p->early_factor, 1);
    dim3 g((unsigned)((n_out2 + DEC2X2_OUT2 - 1) / DEC2X2_OUT2), n_clips);
    decimate2x2_kernel<<<g, DEC2_THREADS, 0, st>>>(wav, clip_offsets, 0, clip_lens, max_len, 0, 1, lvl[0] + pad[0],
                                                   pitch[0], lvl[1] + pad[1], pitch[1], dec2_pairs(p->early_taps2),
                                                   dec2_pairs(p->half_taps2));
    SAGA_LAUNCH_CHECK();
    early_done = true;
    l = 2;
  }
  if (!early_done) {
    const int64_t n_out = level_len(max_len, p->early_factor, 0);
    // outputs per thread shrink with the factor so that the staged input tile (tile_out * factor + 2 * taps) fits:
    // a 1.5-octave CQT from a low note (C_velocity, training.py:382) decimates by up to 64 first
    int per_thread = DEC_PER_THREAD;
    while (per_thread > 1 && decimate_smem_bytes(p->n_early_taps, p->early_factor, per_thread) > 160 * 1024) per_thread >>= 1;
    const int tile_e = DEC_THREADS * per_thread;
    dim3 grid((unsigned)((n_out + tile_e - 1) / tile_e), n_clips);
    const size_t smem = decimate_smem_bytes(p->n_early_taps, p->early_factor, per_thread);
    if (smem > 200 * 1024) return set_error(SAGA_ERR_UNSUPPORTED, "cqt_exec: early factor too large");
    if (smem > 48 * 1024)
      SAGA_CUDA_OK(cudaFuncSetAttribute(decimate_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    if (p->d_early_phase && !SAGA_OPT("SAGA_DEC_NO_PHASE")) {
      const int per_cta = DECP_WARPS * DECP_R * (32 / std::min(p->early_factor, 32));
      dim3 gp((unsigned)((n_out + per_cta - 1) / per_cta), n_clips);
      decimate_phase_kernel<<<gp, 32 * DECP_WARPS, 0, st>>>(wav, clip_offsets, 0, clip_lens, max_len, lvl[0] + pad[0],
                                                            pitch[0], p->d_early_phase, p->early_factor);
    } else if (early_is_dec2) {
      dim3 g2((unsigned)((n_out + DEC2_TILE - 1) / DEC2_TILE), n_clips);
      decimate2_kernel<<<g2, DEC2_THREADS, 0, st>>>(wav, clip_offsets, 0, clip_lens, max_len, 0, 1, lvl[0] + pad[0],
                                                    pitch[0], dec2_pairs(p->early_taps2));
    } else {
      decimate_kernel<<<grid, DEC_THREADS, smem, st>>>(wav, clip_offsets, 0, clip_lens, max_len, 0, 1, lvl[0] + pad[0],
                                                       pitch[0], p->d_early_taps, p->n_early_taps, p->early_factor, per_thread);
    }
    SAGA_LAUNCH_CHECK();
  }
  for (; do_cascade && l <= p->max_level; ++l) {
    const int64_t n_out = level_len(max_len, p->early_factor, l);
    dim3 grid((unsigned)((n_out + tile_out - 1) / tile_out), n_clips);
    const size_t smem = decimate_smem_bytes(p->n_half_taps, 2);
    const bool from_wav = (l == 1 && p->early_factor == 1);
    const float* src = from_wav ? wav : lvl[l - 1] + pad[l - 1];
    const int64_t* src_offs = from_wav ? clip_offsets : nullptr;
    const int64_t src_stride = from_wav ? 0 : pitch[l - 1];
    if (fuse && ((fuse_mask >> l) & 1u) && l + 1 <= p->max_level) {
      const int64_t n_out2 = level_len(max_len, p->early_factor, l + 1);
      dim3 g((unsigned)((n_out2 + DEC2X2_OUT2 - 1) / DEC2X2_OUT2), n_clips);
      decimate2x2_kernel<<<g, DEC2_THREADS, 0, st>>>(src, src_offs, src_stride, clip_lens, max_len, l - 1, p->early_factor,
                                                     lvl[l] + pad[l], pitch[l], lvl[l + 1] + pad[l + 1], pitch[l + 1],
                                                     dec2_pairs(p->half_taps2), dec2_pairs(p->half_taps2));
      ++l;
    } else if (p->n_half_taps == DEC2_S + 1) {
      dim3 g2((unsigned)((n_out + DEC2_TILE - 1) / DEC2_TILE), n_clips);
      decimate2_kernel<<<g2, DEC2_THREADS, 0, st>>>(src, src_offs, src_stride, clip_lens, max_len, l - 1, p->early_factor,
                                                    lvl[l] + pad[l], pitch[l], dec2_pairs(p->half_taps2));
    } else {
      decimate_kernel<<<grid, DEC_THREADS, smem, st>>>(src, src_offs, src_stride, clip_lens, max_len, l - 1,
                                                       p->early_factor, lvl[l] + pad[l], pitch[l], p->d_half_taps,
                                                       p->n_half_taps, 2);
    }
    SAGA_LAUNCH_CHECK();
  }

  const bool tensor_path = (impl != 1) && cqt_umma_supported(p);
  if (do_cascade) {
    // reflect margins (and the padded copy of a raw level 0): part of the cascade phase, for both contraction paths
    PadArgs pa;
    for (int l = 0; l < PAD_MAX_LEVELS; ++l) {
      const bool on = l <= p->max_level;
      pa.lvl[l] = on ? lvl[l] : nullptr;
      pa.pitch[l] = on ? pitch[l] : 0;
      pa.pad[l] = on ? pad[l] : 0;
    }
    pa.wav = raw0 ? wav : nullptr;
    pa.clip_offsets = clip_offsets;
    pa.clip_lens = clip_lens;
    pa.max_len = max_len;
    pa.early_factor = p->early_factor;
    dim3 grid(p->max_level + 1, n_clips, raw0 ? 16 : 1);
    cqt_pad_kernel<<<grid, 256, 0, st>>>(pa);
    SAGA_LAUNCH_CHECK();
  }

  if (!do_contract) return SAGA_OK;
  // ---- frame-window contraction (saga_cqt_frames_exec): a few columns per clip, compact output -------
  // SAGA_CQT_STREAM=0 keeps the fp32 CUDA-core kernels (A/B twin of the streamed tensor-core contraction)
  const bool stream_on = cqt_stream_supported(p) && !(SAGA_OPT("SAGA_CQT_STREAM") && atoi(SAGA_OPT("SAGA_CQT_STREAM")) == 0);
  if (frame_first) {
    if ((int)p->oct.size() > FW_MAX_OCT) return set_error(SAGA_ERR_UNSUPPORTED, "cqt_frames_exec: too many octaves");
    FrameWinArgs fa;
    bool vec = true;
    int max_filt = 0;
    for (size_t i = 0; i < p->oct.size(); ++i) {
      const auto& o = p->oct[i];
      fa.sig[i] = lvl[o.level] + pad[o.level];
      fa.sig_stride[i] = pitch[o.level];
      fa.bank[i] = o.bank;
      fa.n_fft[i] = o.n_fft; fa.n_filt[i] = o.n_filters; fa.hop[i] = o.hop; fa.first_bin[i] = o.first_bin;
      if ((o.hop & 3) || (o.n_fft & 7)) vec = false;
      if (o.n_fft & 3) return set_error(SAGA_ERR_UNSUPPORTED, "cqt_frames_exec: kernel length must be a multiple of 4");
      max_filt = std::max(max_filt, o.n_filters);
    }
    fa.n_bins = p->n_bins; fa.frame_count = frame_count;
    fa.frame_first = frame_first; fa.clip_frames = clip_frames;
    fa.mag_out = C_mag_out; fa.frame_pitch = frame_pitch; fa.out_clip_stride = out_clip_stride;
    fa.n_clips = n_clips; fa.n_oct = (int)p->oct.size();
    fa.pstride = (max_filt + 31) & ~31;
    fa.partial = (float*)ws;           // tail of the workspace (saga_cqt_workspace_bytes reserves it)
    if (stream_on) {
      // tensor cores (cqt_umma_stream.cu); small batches are split along K into the same scratch layout and finished
      // by the same kernel as the fp32 form
      CqtLevels lv;
      lv.wav = wav; lv.clip_offsets = clip_offsets; lv.clip_lens = clip_lens; lv.max_len = max_len;
      lv.lvl = lvl.data(); lv.pitch = pitch.data(); lv.pad = pad.data(); lv.clip_frames = clip_frames;
      int max_slices = 1;
      while (2 * max_slices <= FW_MAX_KS && (int64_t)2 * max_slices * n_clips * fa.n_oct <= 2 * FW_TARGET_CTAS) max_slices *= 2;
      int ks = 1;
      const int rc = cqt_stream_exec(p, lv, n_clips, T_max, frame_first, frame_count, C_mag_out, nullptr, frame_pitch,
                                     out_clip_stride, st, max_slices, fa.partial, fa.pstride, &ks);
      if (rc != SAGA_OK || ks == 1) return rc;
      fa.ks = ks;
      dim3 g2((unsigned)((max_filt + 255) / 256), (unsigned)p->oct.size(), n_clips);
      cqt_frame_window_finish_kernel<<<g2, 256, 0, st>>>(fa);
      SAGA_LAUNCH_CHECK();
      return SAGA_OK;
    }
    const int warps = std::min(8, (max_filt + 31) / 32);
    const int cblocks = (max_filt + warps * 32 - 1) / (warps * 32);
    // split-K until the launch has a few CTAs per SM (each CTA walks its K range serially, one L2 round trip per step)
    int min_nfft = 1 << 30;
    for (auto& o : p->oct) min_nfft = std::min(min_nfft, o.n_fft);
    int ks = 1;
    const int64_t ctas = (int64_t)cblocks * (int64_t)p->oct.size() * n_clips;
    while (ks < FW_MAX_KS && ctas * ks < FW_TARGET_CTAS && min_nfft / (2 * ks) >= 64) ks *= 2;
    fa.ks = ks;
    dim3 grid((unsigned)(cblocks * ks), (unsigned)p->oct.size(), n_clips);
    if (vec) cqt_frame_window_kernel<true><<<grid, warps * 32, 0, st>>>(fa);
    else cqt_frame_window_kernel<false><<<grid, warps * 32, 0, st>>>(fa);
    SAGA_LAUNCH_CHECK();
    if (ks > 1) {
      dim3 g2((unsigned)((max_filt + 255) / 256), (unsigned)p->oct.size(), n_clips);
      cqt_frame_window_finish_kernel<<<g2, 256, 0, st>>>(fa);
      SAGA_LAUNCH_CHECK();
    }
    return SAGA_OK;
  }
  // ---- contraction -------------------------------------------------------------------
  CqtLevels lv;
  lv.wav = wav; lv.clip_offsets = clip_offsets; lv.clip_lens = clip_lens; lv.max_len = max_len;
  lv.lvl = lvl.data(); lv.pitch = pitch.data(); lv.pad = pad.data(); lv.clip_frames = clip_frames;
  if (impl != 1) {
    int rc = cqt_umma_exec(p, lv, n_clips, max_len, T_max, C_mag_out, (float2*)C_cplx_out, frame_pitch,
                           out_clip_stride, impl == 3 ? 1 : 3, TAIL_MAX, st);
    if (rc == SAGA_OK) return SAGA_OK;
    if (rc != SAGA_ERR_UNSUPPORTED) return rc;
    // the bank does not fit the resident kernel (24 / 48 / 192 bins per octave): stream it
    if (impl != 3 && stream_on)
      return cqt_stream_exec(p, lv, n_clips, T_max, nullptr, 0, C_mag_out, (float2*)C_cplx_out, frame_pitch,
                             out_clip_stride, st);
    if (impl >= 2) return rc;
  }
  bool first = true;
  for (auto& o : p->oct) {
    ContractArgs a;
    const bool raw = (o.level == 0 && p->early_factor == 1);
    // the level buffers (a raw level 0 included: cqt_pad_kernel copies it) carry reflect margins of n_fft/2 samples;
    // a contraction-only call after a cascade-only call finds them in the workspace
    a.sig = lvl[o.level] + pad[o.level];
    a.sig_offsets = nullptr;
    a.sig_stride = pitch[o.level];
    a.padded = SAGA_OPT("SAGA_CQT_CONTRACT_V1") ? 0 : 1;
    (void)raw;
    a.clip_lens = clip_lens;
    a.max_len = max_len;
    a.early_factor = p->early_factor;
    a.level = o.level;
    a.bank = o.bank;
    a.n_fft = o.n_fft;
    a.ncol = 2 * o.n_filters;
    a.hop = o.hop;
    a.first_bin = o.first_bin;
    a.n_bins = p->n_bins;
    a.zero_pad = (first && frame_pitch > p->n_bins) ? 1 : 0;
    first = false;
    a.mag_out = C_mag_out;
    a.cplx_out = (float2*)C_cplx_out;
    a.frame_pitch = frame_pitch;
    a.out_clip_stride = out_clip_stride;
    a.clip_frames = clip_frames;
    if (SAGA_OPT("SAGA_CQT_CONTRACT_V1")) {          // first-generation kernel (A/B)
      dim3 grid((unsigned)((T_max + CT_FRAMES - 1) / CT_FRAMES), (a.ncol + CT_FC - 1) / CT_FC, n_clips);
      cqt_contract_kernel<<<grid, CT_FRAMES, 0, st>>>(a);
    } else {
      const int ny0 = (a.ncol + CT2_MAXW * 16 - 1) / (CT2_MAXW * 16);              // column blocks at full width
      const int n_warps = std::max(1, ((a.ncol + ny0 - 1) / ny0 + 15) / 16);       // even split over them (<= 8 warps)
      const int ny = (a.ncol + n_warps * 16 - 1) / (n_warps * 16);
      // frames per lane 3 or 4 (tiles of 96 / 128 frames): whichever pads the clip's frame count less
      const int64_t waste4 = (T_max + 127) / 128 * 128, waste3 = (T_max + 95) / 96 * 96;
      if (a.n_fft % CT2_KC) return set_error(SAGA_ERR_UNSUPPORTED, "cqt_exec: kernel length must be a multiple of %d", CT2_KC);
      if (waste3 < waste4) {
        SAGA_CUDA_OK(cudaFuncSetAttribute(cqt_contract2_kernel<3>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ct2_smem_bytes<3>(CT2_MAXW)));
        dim3 grid((unsigned)((T_max + 95) / 96), ny, n_clips);
        cqt_contract2_kernel<3><<<grid, n_warps * 32, ct2_smem_bytes<3>(n_warps), st>>>(a, n_warps);
      } else {
        SAGA_CUDA_OK(cudaFuncSetAttribute(cqt_contract2_kernel<4>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ct2_smem_bytes<4>(CT2_MAXW)));
        dim3 grid((unsigned)((T_max + 127) / 128), ny, n_clips);
        cqt_contract2_kernel<4><<<grid, n_warps * 32, ct2_smem_bytes<4>(n_warps), st>>>(a, n_warps);
      }
    }
    SAGA_LAUNCH_CHECK();
  }
  return SAGA_OK;
}

extern "C" int saga_cqt_exec(const saga_cqt_plan* p, const float* wav, const int64_t* clip_offsets,
                             const int64_t* clip_lens, int n_clips, int64_t max_len, float* C_mag_out,
                             void* C_cplx_out, int64_t frame_pitch, int64_t out_clip_stride,
                             void* workspace, int64_t workspace_bytes, int impl, void* stream) {
  return cqt_exec_impl(p, wav, clip_offsets, clip_lens, n_clips, max_len, C_mag_out, C_cplx_out, frame_pitch,
                       out_clip_stride, workspace, workspace_bytes, impl, stream, nullptr, 0);
}

extern "C" int saga_cqt_frames_shared_exec(const saga_cqt_plan* p, const float* wav, const int64_t* clip_offsets,
                                           const int64_t* clip_lens, int ws_clips, int64_t max_len, int phase,
                                           int clip_first, int n_clips, const int32_t* frame_first, int frame_count,
                                           float* C_mag_out, int64_t frame_pitch, int64_t out_clip_stride,
                                           void* workspace, int64_t workspace_bytes, void* stream) {
  if (phase == 1) {           // cascade + reflect margins of the whole batch
    static float dummy;       // (no output in this phase)
    return cqt_exec_impl(p, wav, clip_offsets, clip_lens, ws_clips, max_len, C_mag_out ? C_mag_out : &dummy, nullptr,
                         p ? p->n_bins : 0, 0, workspace, workspace_bytes, 1 | SAGA_CQT_SKIP_CONTRACT, stream, nullptr, 0,
                         ws_clips, 0);
  }
  if (phase != 2) return set_error(SAGA_ERR_INVALID, "cqt_frames_shared_exec: phase must be 1 (cascade) or 2 (contraction)");
  if (!frame_first) return set_error(SAGA_ERR_INVALID, "cqt_frames_shared_exec: null frame_first");
  if (frame_count < 1 || frame_count > FW_MAXF)
    return set_error(SAGA_ERR_INVALID, "cqt_frames_shared_exec: frame_count must be in 1..%d", FW_MAXF);
  return cqt_exec_impl(p, wav, clip_offsets, clip_lens, n_clips, max_len, C_mag_out, nullptr, frame_pitch,
                       out_clip_stride, workspace, workspace_bytes, 1 | SAGA_CQT_SKIP_CASCADE, stream, frame_first,
                       frame_count, ws_clips, clip_first);
}

extern "C" int saga_cqt_frames_shared_multi_exec(const saga_cqt_plan* const* plans, int n_plans, const int32_t* clip_first,
                                                 const int32_t* clip_count, const float* wav, const int64_t* clip_offsets,
                                                 const int64_t* clip_lens, int ws_clips, int64_t max_len,
                                                 const int32_t* frame_first, int frame_count, float* C_mag_out,
                                                 int64_t frame_pitch, int64_t out_clip_stride, void* workspace,
                                                 int64_t workspace_bytes, void* stream) {
  if (!plans || n_plans < 1 || !clip_first || !clip_count || !frame_first || !C_mag_out || !workspace)
    return set_error(SAGA_ERR_INVALID, "cqt_frames_shared_multi_exec: null argument");
  if (frame_count < 1 || frame_count > FW_MAXF)
    return set_error(SAGA_ERR_INVALID, "cqt_frames_shared_multi_exec: frame_count must be in 1..%d", FW_MAXF);
  const saga_cqt_plan* p = plans[0];
  const bool stream_on = cqt_stream_supported(p) && !(SAGA_OPT("SAGA_CQT_STREAM") && atoi(SAGA_OPT("SAGA_CQT_STREAM")) == 0);
  // every plan must have the geometry the cascade was run for (levels, hops, kernel lengths, filter counts, early stage)
  for (int i = 0; i < n_plans; ++i) {
    const saga_cqt_plan* q = plans[i];
    if (!q || q->oct.size() != p->oct.size() || q->early_factor != p->early_factor || q->max_level != p->max_level ||
        q->n_bins != p->n_bins || q->hop != p->hop)
      return set_error(SAGA_ERR_INVALID, "cqt_frames_shared_multi_exec: plan %d has another geometry", i);
    for (size_t o = 0; o < p->oct.size(); ++o)
      if (q->oct[o].level != p->oct[o].level || q->oct[o].hop != p->oct[o].hop || q->oct[o].n_fft != p->oct[o].n_fft ||
          q->oct[o].n_filters != p->oct[o].n_filters || q->oct[o].first_bin != p->oct[o].first_bin)
        return set_error(SAGA_ERR_INVALID, "cqt_frames_shared_multi_exec: plan %d has another geometry", i);
    if (clip_first[i] < 0 || clip_count[i] < 0 || clip_first[i] + clip_count[i] > ws_clips)
      return set_error(SAGA_ERR_INVALID, "cqt_frames_shared_multi_exec: clip range of plan %d outside the batch", i);
  }
  bool same = stream_on;
  for (int i = 0; i < n_plans && same; ++i) same = cqt_stream_supported(plans[i]);
  if (!same) {     // plan by plan (fp32 kernels, or a plan outside the tensor path's constraints)
    for (int i = 0; i < n_plans; ++i) {
      const int rc = saga_cqt_frames_shared_exec(plans[i], wav, clip_offsets, clip_lens, ws_clips, max_len, 2, clip_first[i],
                                                 clip_count[i], frame_first + clip_first[i], frame_count,
                                                 C_mag_out + (int64_t)clip_first[i] * out_clip_stride, frame_pitch,
                                                 out_clip_stride, workspace, workspace_bytes, stream);
      if (rc != SAGA_OK) return rc;
    }
    return SAGA_OK;
  }
  if (frame_pitch < p->n_bins) return set_error(SAGA_ERR_INVALID, "cqt_exec: frame_pitch < n_bins");
  if (ws_clips <= 0 || max_len <= 0) return SAGA_OK;
  if (workspace_bytes < saga_cqt_workspace_bytes(p, ws_clips, max_len))
    return set_error(SAGA_ERR_INVALID, "cqt_exec: workspace too small");
  if ((int)p->oct.size() > FW_MAX_OCT || p->max_level + 1 > PAD_MAX_LEVELS)
    return set_error(SAGA_ERR_UNSUPPORTED, "cqt_frames_shared_multi_exec: too many octaves / levels");
  cudaStream_t st = (cudaStream_t)stream;
  // the workspace layout of cqt_exec_impl for a batch of ws_clips clips
  char* ws = (char*)workspace;
  int32_t* clip_frames = (int32_t*)ws;
  ws += ws_header_bytes(ws_clips);
  std::vector<float*> lvl(p->max_level + 1, nullptr);
  std::vector<int64_t> pitch(p->max_level + 1, 0);
  std::vector<int> pad(p->max_level + 1, 0);
  for (int l = 0; l <= p->max_level; ++l) {
    pitch[l] = cqt_level_pitch(p, l, max_len);
    pad[l] = cqt_level_pad(p, l);
    lvl[l] = (float*)ws;
    ws += (int64_t)ws_clips * pitch[l] * 4;
  }
  CqtLevels lv;
  lv.wav = wav; lv.clip_offsets = clip_offsets; lv.clip_lens = clip_lens; lv.max_len = max_len;
  lv.lvl = lvl.data(); lv.pitch = pitch.data(); lv.pad = pad.data(); lv.clip_frames = clip_frames;
  int max_filt = 0;
  FrameWinArgs fa;
  for (size_t i = 0; i < p->oct.size(); ++i) {
    const auto& o = p->oct[i];
    fa.sig[i] = nullptr; fa.sig_stride[i] = 0; fa.bank[i] = nullptr;
    fa.n_fft[i] = o.n_fft; fa.n_filt[i] = o.n_filters; fa.hop[i] = o.hop; fa.first_bin[i] = o.first_bin;
    max_filt = std::max(max_filt, o.n_filters);
  }
  fa.n_bins = p->n_bins; fa.frame_count = frame_count;
  fa.frame_first = frame_first; fa.clip_frames = clip_frames;
  fa.mag_out = C_mag_out; fa.frame_pitch = frame_pitch; fa.out_clip_stride = out_clip_stride;
  fa.n_clips = ws_clips; fa.n_oct = (int)p->oct.size();
  fa.pstride = (max_filt + 31) & ~31;
  fa.partial = (float*)ws;
  int max_slices = 1;
  while (2 * max_slices <= FW_MAX_KS && (int64_t)2 * max_slices * ws_clips * fa.n_oct <= 2 * FW_TARGET_CTAS) max_slices *= 2;
  int ks = 1;
  std::vector<int> c0(clip_first, clip_first + n_plans), cn(clip_count, clip_count + n_plans);
  const int rc = cqt_stream_exec_multi(plans, n_plans, c0.data(), cn.data(), lv, ws_clips, saga_cqt_num_frames(p, max_len),
                                       frame_first, frame_count, C_mag_out, nullptr, frame_pitch, out_clip_stride, st,
                                       max_slices, fa.partial, fa.pstride, &ks);
  if (rc != SAGA_OK || ks == 1) return rc;
  fa.ks = ks;
  dim3 g2((unsigned)((max_filt + 255) / 256), (unsigned)p->oct.size(), ws_clips);
  cqt_frame_window_finish_kernel<<<g2, 256, 0, st>>>(fa);
  SAGA_LAUNCH_CHECK();
  return SAGA_OK;
}

extern "C" int saga_cqt_frames_exec(const saga_cqt_plan* p, const float* wav, const int64_t* clip_offsets,
                                    const int64_t* clip_lens, int n_clips, int64_t max_len,
                                    const int32_t* frame_first, int frame_count, float* C_mag_out,
                                    int64_t frame_pitch, int64_t out_clip_stride, void* workspace,
                                    int64_t workspace_bytes, void* stream) {
  if (!frame_first) return set_error(SAGA_ERR_INVALID, "cqt_frames_exec: null frame_first");
  if (frame_count < 1 || frame_count > FW_MAXF)
    return set_error(SAGA_ERR_INVALID, "cqt_frames_exec: frame_count must be in 1..%d", FW_MAXF);
  return cqt_exec_impl(p, wav, clip_offsets, clip_lens, n_clips, max_len, C_mag_out, nullptr, frame_pitch,
                       out_clip_stride, workspace, workspace_bytes, 1, stream, frame_first, frame_count);
}

// ---------------------------------------------------------------------------
// Peak of a column range per clip (saga_cqt_peak_exec): the whole-song normalisers of the producer loop
// (training.py:271-282) are np.max of `C[:, 0:t]` of a full transform.  Plans the streamed tensor-core kernel runs
// contract in its peak mode (packed rows, no image); every other plan contracts into an image in the workspace that
// cqt_column_peak_kernel reduces.
// ---------------------------------------------------------------------------
namespace saga {

// row_start[c] = sum of the frame counts of clips < c, row_start[n_clips] = all rows (one thread: a batch is songs)
__global__ void cqt_row_start_kernel(const int32_t* clip_frames, int n_clips, int32_t* row_start) {
  if (blockIdx.x != 0 || threadIdx.x != 0) return;
  int32_t s = 0;
  for (int c = 0; c < n_clips; ++c) {
    row_start[c] = s;
    s += clip_frames[c];
  }
  row_start[n_clips] = s;
}

// max over bins [0, n_bins) and frames [max(col_lo, 0), min(col_hi, T_c)) of clip blockIdx.y of a frame-major image
__global__ void __launch_bounds__(256) cqt_column_peak_kernel(const float* img, int64_t frame_pitch, int64_t clip_stride,
                                                             int n_bins, const int32_t* clip_frames, const int32_t* col_lo,
                                                             const int32_t* col_hi, unsigned int* peak_out) {
  const int c = blockIdx.y;
  const int lo = max(col_lo[c], 0), hi = min(col_hi[c], clip_frames[c]);
  float m = 0.f;
  for (int t = lo + blockIdx.x * blockDim.y + threadIdx.y; t < hi; t += gridDim.x * blockDim.y)
    for (int k = threadIdx.x; k < n_bins; k += blockDim.x) m = fmaxf(m, img[c * clip_stride + t * frame_pitch + k]);
  m = warp_max(m);
  if (threadIdx.x == 0 && m > 0.f) atomicMax(peak_out + c, __float_as_uint(m));      // magnitudes >= 0: bit order
}

static int64_t round256(int64_t b) { return (b + 255) & ~int64_t(255); }

// the plans saga_cqt_exec contracts with the streamed kernel (the resident kernel declines them and the option allows it)
static bool peak_streamed(const saga_cqt_plan* p) {
  const char* opt = SAGA_OPT("SAGA_CQT_STREAM");
  return cqt_stream_supported(p) && !cqt_umma_supported(p) && !(opt && atoi(opt) == 0);
}

}  // namespace saga

extern "C" int64_t saga_cqt_peak_workspace_bytes(const saga_cqt_plan* p, int n_clips, int64_t max_len) {
  if (!p || n_clips <= 0 || max_len <= 0) return 256;
  int64_t b = round256(saga_cqt_workspace_bytes(p, n_clips, max_len)) + round256(((int64_t)n_clips + 1) * 4);
  if (!peak_streamed(p)) b += (int64_t)n_clips * saga_cqt_num_frames(p, max_len) * ((p->n_bins + 3) & ~3) * 4;
  return b;
}

extern "C" int saga_cqt_peak_exec(const saga_cqt_plan* p, const float* wav, const int64_t* clip_offsets,
                                  const int64_t* clip_lens, int n_clips, int64_t max_len, const int32_t* col_lo,
                                  const int32_t* col_hi, float* peak_out, void* workspace, int64_t workspace_bytes,
                                  void* stream) {
  if (!p || !wav || !clip_offsets || !col_lo || !col_hi || !peak_out || !workspace)
    return set_error(SAGA_ERR_INVALID, "cqt_peak_exec: null argument");
  if (n_clips < 0) return set_error(SAGA_ERR_INVALID, "cqt_peak_exec: n_clips < 0");
  if (n_clips == 0) return SAGA_OK;
  if (workspace_bytes < saga_cqt_peak_workspace_bytes(p, n_clips, max_len))
    return set_error(SAGA_ERR_INVALID, "cqt_peak_exec: workspace too small");
  if ((reinterpret_cast<uintptr_t>(workspace) & 255) != 0)
    return set_error(SAGA_ERR_INVALID, "cqt_peak_exec: workspace must be 256-byte aligned");
  cudaStream_t st = (cudaStream_t)stream;
  SAGA_CUDA_OK(cudaMemsetAsync(peak_out, 0, sizeof(float) * n_clips, st));
  if (max_len <= 0) return SAGA_OK;
  const int64_t T_max = saga_cqt_num_frames(p, max_len);
  char* ws = (char*)workspace;
  const int64_t cqt_bytes = round256(saga_cqt_workspace_bytes(p, n_clips, max_len));
  int32_t* row_start = (int32_t*)(ws + cqt_bytes);
  const int32_t* clip_frames = (const int32_t*)ws;          // header of the cascade's workspace (cqt_exec_impl)
  unsigned int* peak_bits = reinterpret_cast<unsigned int*>(peak_out);
  if (!peak_streamed(p)) {
    float* img = (float*)(ws + cqt_bytes + round256(((int64_t)n_clips + 1) * 4));
    const int64_t P = (p->n_bins + 3) & ~3;
    const int rc = cqt_exec_impl(p, wav, clip_offsets, clip_lens, n_clips, max_len, img, nullptr, P, T_max * P, workspace,
                                 cqt_bytes, 0, stream, nullptr, 0);
    if (rc != SAGA_OK) return rc;
    dim3 grid((unsigned)std::min<int64_t>((T_max + 7) / 8, 64), n_clips), block(32, 8);
    cqt_column_peak_kernel<<<grid, block, 0, st>>>(img, P, T_max * P, p->n_bins, clip_frames, col_lo, col_hi, peak_bits);
    SAGA_LAUNCH_CHECK();
    return SAGA_OK;
  }
  // cascade + reflect margins exactly as saga_cqt_exec runs them, then the contraction in peak mode
  static float dummy;
  int rc = cqt_exec_impl(p, wav, clip_offsets, clip_lens, n_clips, max_len, &dummy, nullptr, p->n_bins, 0, workspace,
                         cqt_bytes, SAGA_CQT_SKIP_CONTRACT, stream, nullptr, 0);
  if (rc != SAGA_OK) return rc;
  if (p->max_level + 1 > PAD_MAX_LEVELS) return set_error(SAGA_ERR_UNSUPPORTED, "cqt_peak_exec: too many levels");
  // the workspace layout of cqt_exec_impl
  std::vector<float*> lvl(p->max_level + 1, nullptr);
  std::vector<int64_t> pitch(p->max_level + 1, 0);
  std::vector<int> pad(p->max_level + 1, 0);
  char* w = ws + ws_header_bytes(n_clips);
  for (int l = 0; l <= p->max_level; ++l) {
    pitch[l] = cqt_level_pitch(p, l, max_len);
    pad[l] = cqt_level_pad(p, l);
    lvl[l] = (float*)w;
    w += (int64_t)n_clips * pitch[l] * 4;
  }
  CqtLevels lv;
  lv.wav = wav; lv.clip_offsets = clip_offsets; lv.clip_lens = clip_lens; lv.max_len = max_len;
  lv.lvl = lvl.data(); lv.pitch = pitch.data(); lv.pad = pad.data(); lv.clip_frames = clip_frames;
  cqt_row_start_kernel<<<1, 32, 0, st>>>(clip_frames, n_clips, row_start);
  SAGA_LAUNCH_CHECK();
  CqtPeakArgs pk;
  pk.row_start = row_start; pk.col_lo = col_lo; pk.col_hi = col_hi; pk.peak_out = peak_out;
  return cqt_stream_peak_exec(p, lv, n_clips, T_max, pk, st);
}

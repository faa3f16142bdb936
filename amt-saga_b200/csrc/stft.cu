// K1: batched windowed real FFT -> magnitude / unit phasor / complex STFT.
// Replaces librosa.stft + magphase as reached from
// /root/reference/util_audio.py:127-128, :147, :173.
//
// Design (sm_100a, HBM-bound target):
//  * a CTA owns a run of F consecutive frames of one clip and stages the
//    contiguous sample span (F-1)*hop + n_fft ONCE in shared memory with
//    float4 loads (reflect padding = index mirroring at the clip edges), so the
//    n_fft/hop-fold frame overlap is served from SMEM, not L2/HBM;
//  * one warp per frame: the real frame is viewed as M = n_fft/2 complex
//    points, transformed by an in-place decimation-in-frequency FFT whose
//    passes are register-resident radix-16/32 butterflies with immediate
//    twiddles (fft_radix.cuh); data crosses lanes through a padded
//    (conflict-free) per-warp SMEM buffer, inter-pass twiddles come from
//    float64-generated fp32 tables laid out in access order;
//  * real-FFT split + |z| (+ phasor / complex) fused in the epilogue, stores
//    are 128-byte coalesced rows of the frame-major output, per-frame and
//    per-clip maxima (ref_mag) are a by-product.
#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <vector>

#include "fft_radix.cuh"
#include "saga_common.cuh"
#include "stft_plan.cuh"

namespace saga {

__device__ __forceinline__ int pidx(int i) { return i + (i >> 5); }


// table element: read-only global path, or a plain (shared-memory) load when the CTA keeps the tables in SMEM
template <bool GT>
__device__ __forceinline__ float2 tab(const float2* p) {
  if (GT) return __ldg(p);
  return *p;
}

// LANES threads work on one frame: a warp, or -- for the long transforms, whose 17 / 34 KB exchange buffers allow
// only a handful of frames per SM -- 2 or 4 warps that meet at a named barrier (id = 1 + frame slot of the CTA).
template <int LANES>
__device__ __forceinline__ void group_sync(int group) {
  if constexpr (LANES == 32) {
    __syncwarp();
  } else {
    asm volatile("bar.sync %0, %1;" ::"r"(group + 1), "n"(LANES) : "memory");
  }
}

// One DIF pass over blocks of length L with radix R, in place in `buf`.
// FIRST reads the windowed real samples instead of buf.
template <int M, int L, int R, bool FIRST, bool LAST, bool GT = true, int LANES = 32>
__device__ __forceinline__ void dif_pass(float2* buf, const float* xs, const float2* __restrict__ win2,
                                         const float2* __restrict__ tw, int lane, int group = 0) {
  constexpr int LS = L / R;       // sub-block length after this pass
  constexpr int ITEMS = M / R;    // small FFTs in this pass
  constexpr int ITERS = (ITEMS + LANES - 1) / LANES;
#pragma unroll 1
  for (int it = 0; it < ITERS; ++it) {
    const int q = lane + LANES * it;
    if ((ITEMS % LANES) != 0 && q >= ITEMS) break;
    const int b = q / LS, j = q % LS;
    const int base = b * L + j;
    float2 v[R];
    if (FIRST) {
      const bool al = ((reinterpret_cast<uintptr_t>(xs) & 7) == 0);
#pragma unroll
      for (int r = 0; r < R; ++r) {
        const int n = base + r * LS;
        float2 x;
        if (al) {
          x = *reinterpret_cast<const float2*>(xs + 2 * n);
        } else {
          x.x = xs[2 * n];
          x.y = xs[2 * n + 1];
        }
        v[r] = pmul(x, tab<GT>(win2 + n));
      }
    } else {
#pragma unroll
      for (int r = 0; r < R; ++r) v[r] = buf[pidx(base + r * LS)];
    }
    fft_reg<R>(v);
#pragma unroll
    for (int i = 0; i < R; ++i) {
      const int rp = bitrev(i, R);
      float2 o = v[i];
      if (!LAST && rp > 0) o = cmul(o, tab<GT>(tw + rp * LS + j));
      buf[pidx(base + rp * LS)] = o;
    }
  }
  group_sync<LANES>(group);
}

// position of Z[k] in buf after the digit-reversing in-place passes
template <int M, int R0, int R1, int R2>
__device__ __forceinline__ int zpos(int k) {
  constexpr int L1 = M / R0, L2 = L1 / R1;
  if (R2 == 1) return (k % R0) * L1 + (k / R0);
  return (k % R0) * L1 + ((k / R0) % R1) * L2 + (k / (R0 * R1));
}

__device__ __forceinline__ float fast_sqrt(float x) {   // sqrt.approx: ~1 ulp, exact 0 -> 0
  float r;
  asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
  return r;
}

// One pair of bins (k, M-k) of the real-FFT split.  The window table carries the factor 1/2 of
//   X[k] = 1/2 [ (Z[k] + conj Z[M-k]) - i W^k (Z[k] - conj Z[M-k]) ]
// so with s = Zk + Zm (componentwise), d = Zk - Zm:  T = W^k * (s.y, -d.x),
//   X[k] = (s.x + T.x, d.y + T.y),   X[M-k] = conj(s.x - T.x, d.y - T.y).
__device__ __forceinline__ void split_pair(float2 zk, float2 zm, float2 w, float2& Xk, float2& Xm) {
  const float2 s = cadd(zk, zm), d = csub(zk, zm);
  const float sx = s.x, dx = d.x, sy = s.y, dy = d.y;
  const float tx = fmaf(w.x, sy, w.y * dx);      // Re(w * (sy - i dx))
  const float ty = fmaf(w.y, sy, -(w.x * dx));   // Im
  Xk = make_float2(sx + tx, dy + ty);
  Xm = make_float2(sx - tx, ty - dy);
}

// Real-FFT split of one transformed frame (Z in `buf`, digit-reversed order) -> |X| (+ phasor / complex),
// coalesced rows of the frame-major output, per-frame and per-clip maxima.
template <int M, int R0, int R1, int R2, bool EXTRA, bool GT, int LANES = 32>
__device__ __forceinline__ void stft_frame_out(const float2* buf, const float2* twN, const StftArgs& a, int clip,
                                               int64_t t, int dst, int64_t drow, int lane, int group = 0,
                                               float* gmax = nullptr) {
  static_assert(LANES == 32 || R2 > 1, "multi-warp frames use the generic position map");
  // smem positions of Z[lane + 32 i] and of its partner Z[M - lane - 32 i] (digit-reversed order):
  //   zpos is affine in i for a fixed lane, so both are base + i * step
  const int zk0 = pidx(zpos<M, R0, R1, R2>(lane));
  const int zk1 = pidx(zpos<M, R0, R1, R2>(lane + 32));
  const int zm0 = pidx(zpos<M, R0, R1, R2>((M - lane) & (M - 1)));
  const int zm1 = pidx(zpos<M, R0, R1, R2>(M - lane - 32));
  const int zm2 = pidx(zpos<M, R0, R1, R2>(M - lane - 64));
  const int zk_step = zk1 - zk0, zm_step = zm2 - zm1;
  // ---- real-FFT split, |X|, outputs -----------------------------------
    const int64_t row = (int64_t)dst * a.out_clip_stride + drow * a.frame_pitch;
  float* mag_up = a.mag_out + row + lane;           // bins lane + LANES i
  float* mag_dn = a.mag_out + row + (M - lane);     // bins M - lane - LANES i
  const float2* twp = twN + lane;
  float vmax = 0.f;
  constexpr int ITERS = M / (2 * LANES);            // k = lane + LANES i < M/2
#pragma unroll 8
  for (int i = 0; i < ITERS; ++i) {
    float2 zk, zm;
    if constexpr (R2 == 1) {      // two-pass shapes: both positions are affine in i
      zk = buf[zk0 + i * zk_step];
      zm = buf[i == 0 ? zm0 : zm1 + (i - 1) * zm_step];
    } else {
      const int k = lane + LANES * i;
      zk = buf[pidx(zpos<M, R0, R1, R2>(k))];
      zm = buf[pidx(zpos<M, R0, R1, R2>((M - k) & (M - 1)))];
    }
    float2 Xk, Xm;
    split_pair(zk, zm, tab<GT>(twp + LANES * i), Xk, Xm);
    const float mk = fast_sqrt(fmaf(Xk.x, Xk.x, Xk.y * Xk.y));
    const float mm = fast_sqrt(fmaf(Xm.x, Xm.x, Xm.y * Xm.y));
    vmax = fmaxf(vmax, fmaxf(mk, mm));
    mag_up[LANES * i] = mk;
    mag_dn[-LANES * i] = mm;
    if (EXTRA) {
      const int k = lane + LANES * i;
      if (a.cplx_out) {
        float2* c = a.cplx_out + row;
        c[k] = Xk;
        c[M - k] = Xm;
      }
      if (a.phase_out) {
        float2* p = a.phase_out + row;
        p[k] = mk > 0.f ? make_float2(Xk.x / mk, Xk.y / mk) : make_float2(1.f, 0.f);
        p[M - k] = mm > 0.f ? make_float2(Xm.x / mm, Xm.y / mm) : make_float2(1.f, 0.f);
      }
    }
  }
  if (lane == 0) {
    // k = M/2 pairs with itself
    const float2 z = buf[pidx(zpos<M, R0, R1, R2>(M / 2))];
    float2 Xk, Xm;
    split_pair(z, z, tab<GT>(twN + M / 2), Xk, Xm);
    const float mk = fast_sqrt(fmaf(Xk.x, Xk.x, Xk.y * Xk.y));
    vmax = fmaxf(vmax, mk);
    a.mag_out[row + M / 2] = mk;
    if (EXTRA) {
      if (a.cplx_out) a.cplx_out[row + M / 2] = Xk;
      if (a.phase_out)
        a.phase_out[row + M / 2] = mk > 0.f ? make_float2(Xk.x / mk, Xk.y / mk) : make_float2(1.f, 0.f);
    }
  }
  // padding columns [M+1, frame_pitch) are defined as zero
  for (int64_t k = M + 1 + lane; k < a.frame_pitch; k += LANES) {
    a.mag_out[row + k] = 0.f;
    if (EXTRA) {
      if (a.cplx_out) a.cplx_out[row + k] = make_float2(0.f, 0.f);
      if (a.phase_out) a.phase_out[row + k] = make_float2(0.f, 0.f);
    }
  }
  vmax = warp_max(vmax);
  if constexpr (LANES > 32) {      // the frame's warps combine their maxima through shared memory
    if ((lane & 31) == 0) gmax[threadIdx.x >> 5] = vmax;
    group_sync<LANES>(group);
    if (lane == 0) {
#pragma unroll
      for (int i = 1; i < LANES / 32; ++i) vmax = fmaxf(vmax, gmax[(threadIdx.x >> 5) + i]);
    }
  }
  if (lane == 0) {
    if (a.frame_max_out) a.frame_max_out[(int64_t)clip * a.max_frames + t] = vmax;
    if (a.clip_max_out) atomic_max_nonneg(a.clip_max_out + clip, vmax);
  }
}

// ---- register-resident tail for the shapes whose first radix is 32 (n_fft 2048 / 1024) -----------------
// After the last pass lane l holds, in registers, exactly the bins the output stage gives it:
// position l*R + rp of the digit-reversed buffer is Z[l + 32 rp], so v[bitrev(rp)] = Z[l + 32 rp].
// The real-FFT split pairs bin k = l + 32 i with M - k = (32 - l) + 32 (R - 1 - i), which lives in lane
// (32 - l) & 31 under the SAME register index bitrev(R - 1 - i): one warp shuffle per component replaces
// the store + load round trip through shared memory (16 KB of the 60 KB a frame moves through that pipe).
// Lane 0 pairs with itself (M - 32 i = 32 (R - i)) and handles k = 0 / M/2 as before.
template <int M, int L, int R>
__device__ __forceinline__ void dif_pass_last_regs(const float2* buf, float2 (&v)[R], int lane) {
  static_assert(M / R == 32 && L == R, "one small FFT per lane, contiguous block");
  const int base = lane * L;
#pragma unroll
  for (int r = 0; r < R; ++r) v[r] = buf[pidx(base + r)];
  fft_reg<R>(v);
}

template <int M, int R, bool EXTRA, bool GT>
__device__ __forceinline__ void stft_frame_out_regs(const float2 (&v)[R], const float2* twN, const StftArgs& a,
                                                    int clip, int64_t t, int dst, int64_t drow, int lane) {
  const int64_t row = (int64_t)dst * a.out_clip_stride + drow * a.frame_pitch;
  float* mag_up = a.mag_out + row + lane;           // bins lane + 32 i
  float* mag_dn = a.mag_out + row + (M - lane);     // bins M - lane - 32 i
  const float2* twp = twN + lane;
  const int partner = (32 - lane) & 31;
  float vmax = 0.f;
  constexpr int ITERS = R / 2;                      // k = lane + 32 i < M/2
#pragma unroll
  for (int i = 0; i < ITERS; ++i) {
    const float2 zk = v[bitrev(i, R)];
    const float2 give = v[bitrev(R - 1 - i, R)];
    float2 zm;
    zm.x = __shfl_sync(0xffffffffu, give.x, partner);
    zm.y = __shfl_sync(0xffffffffu, give.y, partner);
    if (lane == 0) zm = (i == 0) ? v[0] : v[bitrev(R - i, R)];
    float2 Xk, Xm;
    split_pair(zk, zm, tab<GT>(twp + 32 * i), Xk, Xm);
    const float mk = fast_sqrt(fmaf(Xk.x, Xk.x, Xk.y * Xk.y));
    const float mm = fast_sqrt(fmaf(Xm.x, Xm.x, Xm.y * Xm.y));
    vmax = fmaxf(vmax, fmaxf(mk, mm));
    mag_up[32 * i] = mk;
    mag_dn[-32 * i] = mm;
    if (EXTRA) {
      const int k = lane + 32 * i;
      if (a.cplx_out) {
        float2* c = a.cplx_out + row;
        c[k] = Xk;
        c[M - k] = Xm;
      }
      if (a.phase_out) {
        float2* p = a.phase_out + row;
        p[k] = mk > 0.f ? make_float2(Xk.x / mk, Xk.y / mk) : make_float2(1.f, 0.f);
        p[M - k] = mm > 0.f ? make_float2(Xm.x / mm, Xm.y / mm) : make_float2(1.f, 0.f);
      }
    }
  }
  if (lane == 0) {
    // k = M/2 = 32 * (R/2) pairs with itself
    const float2 z = v[bitrev(R / 2, R)];
    float2 Xk, Xm;
    split_pair(z, z, tab<GT>(twN + M / 2), Xk, Xm);
    const float mk = fast_sqrt(fmaf(Xk.x, Xk.x, Xk.y * Xk.y));
    vmax = fmaxf(vmax, mk);
    a.mag_out[row + M / 2] = mk;
    if (EXTRA) {
      if (a.cplx_out) a.cplx_out[row + M / 2] = Xk;
      if (a.phase_out)
        a.phase_out[row + M / 2] = mk > 0.f ? make_float2(Xk.x / mk, Xk.y / mk) : make_float2(1.f, 0.f);
    }
  }
  // padding columns [M+1, frame_pitch) are defined as zero
  for (int64_t k = M + 1 + lane; k < a.frame_pitch; k += 32) {
    a.mag_out[row + k] = 0.f;
    if (EXTRA) {
      if (a.cplx_out) a.cplx_out[row + k] = make_float2(0.f, 0.f);
      if (a.phase_out) a.phase_out[row + k] = make_float2(0.f, 0.f);
    }
  }
  vmax = warp_max(vmax);
  if (lane == 0) {
    if (a.frame_max_out) a.frame_max_out[(int64_t)clip * a.max_frames + t] = vmax;
    if (a.clip_max_out) atomic_max_nonneg(a.clip_max_out + clip, vmax);
  }
}

// threads that share one frame of the forward transform
__host__ __device__ constexpr int stft_lanes(int M) { return M <= 1024 ? 32 : (M == 2048 ? 64 : 128); }

// Frame range of saga_stft_rows_exec, a kernel argument of its own: StftArgs is embedded in the ring kernel's
// arguments, whose layout stays as it is.
struct StftRows {
  const int32_t* frame0;     // clip c computes frames frame0[c] + j, j in [0, n_frames)
  const int32_t* dst_clip;   // output clip of clip c (NULL: c)
  int n_frames, dst_row0;    // frame j is written as row dst_row0 + j
};

// The frames a CTA transforms: nF consecutive frames t0 .. of the clip, frame t0 + f written as row orow0 + f of
// output clip dst.  Returns false when there are none.
//   stft_exec (ROWS false): tile `tile` of the clip's T frames, rows = frames of clip `clip`.
//   rows entry (ROWS true): frames frame0[clip] + j for the tile's j range, rows dst_row0 + j of output clip
//   dst_clip[clip]; the tile's frames outside [0, T) are written here as zero rows (magnitude 0, phasor (0, 0),
//   padding columns included) -- what a song's storage holds past its end.
template <bool ROWS, int THREADS>
__device__ __forceinline__ bool stft_tile(const StftArgs& a, const StftRows& r, int clip, int tile, int64_t T,
                                          int64_t& t0, int& nF, int& dst, int64_t& orow0) {
  if constexpr (!ROWS) {
    t0 = (int64_t)tile * a.frames_per_cta;
    if (t0 >= T) return false;
    nF = (int)min((int64_t)a.frames_per_cta, T - t0);
    dst = clip;
    orow0 = t0;
    return true;
  } else {
    const int j0 = tile * a.frames_per_cta;
    const int nJ = min(a.frames_per_cta, r.n_frames - j0);
    const int64_t ts = (int64_t)r.frame0[clip] + j0;
    const int lo = (int)min(max(-ts, (int64_t)0), (int64_t)nJ);     // frames before the clip's start
    const int hi = (int)max(min(T - ts, (int64_t)nJ), (int64_t)lo);  // first frame at or past its end
    dst = r.dst_clip ? r.dst_clip[clip] : clip;
    orow0 = (int64_t)r.dst_row0 + j0;
    float* mag = a.mag_out + (int64_t)dst * a.out_clip_stride + orow0 * a.frame_pitch;
    float2* ph = a.phase_out ? a.phase_out + (int64_t)dst * a.out_clip_stride + orow0 * a.frame_pitch : nullptr;
    const int64_t z0 = (int64_t)lo * a.frame_pitch, z1 = (int64_t)hi * a.frame_pitch, zn = (int64_t)nJ * a.frame_pitch;
    for (int64_t i = threadIdx.x; i < z0 + (zn - z1); i += THREADS) {
      const int64_t k = i < z0 ? i : z1 + (i - z0);
      mag[k] = 0.f;
      if (ph) ph[k] = make_float2(0.f, 0.f);
    }
    t0 = ts + lo;
    nF = hi - lo;
    orow0 += lo;
    return nF > 0;
  }
}

template <int M, int R0, int R1, int R2, int WARPS, bool EXTRA, bool ROWS = false>
__global__ void __launch_bounds__(WARPS * 32, 2) stft_kernel(const StftArgs a, const StftRows rows) {
  constexpr int N = 2 * M;
  constexpr int BUF = M + M / 32;
  extern __shared__ __align__(16) float smem[];
  float* span = smem;
  float2* bufs = reinterpret_cast<float2*>(smem + a.span_alloc);

  const int clip = blockIdx.x / a.tiles_per_clip;
  const int tile = blockIdx.x % a.tiles_per_clip;
  const int64_t len = a.clip_lens[clip];
  int64_t T;
  if (len <= 0) T = 0;
  else if (a.center) T = 1 + len / a.hop;
  else T = len >= N ? 1 + (len - N) / a.hop : 0;
  int64_t t0, orow0;
  int nF, dst;
  if (!stft_tile<ROWS, WARPS * 32>(a, rows, clip, tile, T, t0, nF, dst, orow0)) return;
  const float* x = a.wav + a.clip_offsets[clip];

  // ---- stage the sample span once per CTA ---------------------------------
  const int64_t s0 = t0 * a.hop - (a.center ? N / 2 : 0);
  const int span_len = (nF - 1) * a.hop + N;
  const bool interior = (s0 >= 0) && (s0 + span_len <= len);
  if (interior && ((reinterpret_cast<uintptr_t>(x + s0) & 15) == 0)) {
    const float4* src = reinterpret_cast<const float4*>(x + s0);
    float4* dst = reinterpret_cast<float4*>(span);
    const int n4 = span_len >> 2;
    for (int i = threadIdx.x; i < n4; i += WARPS * 32) dst[i] = __ldg(src + i);
    for (int i = (n4 << 2) + threadIdx.x; i < span_len; i += WARPS * 32) span[i] = __ldg(x + s0 + i);
  } else {
    for (int i = threadIdx.x; i < span_len; i += WARPS * 32) {
      int64_t s = s0 + i;
      if (s < 0 || s >= len) s = reflect_index(s, len);
      span[i] = __ldg(x + s);
    }
  }
  __syncthreads();

  // LANES threads per frame (see group_sync): one warp up to n_fft 2048, two warps for 4096, four for 8192
  constexpr int LANES = stft_lanes(M);
  constexpr int GROUPS = WARPS * 32 / LANES;
  __shared__ float gmax[WARPS];
  const int group = threadIdx.x / LANES, lane = threadIdx.x % LANES;
  float2* buf = bufs + group * BUF;
  const float2* win2 = reinterpret_cast<const float2*>(a.window);
  for (int f = group; f < nF; f += GROUPS) {
    const float* xs = span + f * a.hop;
    constexpr int L1 = M / R0, L2 = L1 / R1;
    dif_pass<M, M, R0, true, false, true, LANES>(buf, xs, win2, a.tw0, lane, group);
    if constexpr (R0 == 32 && R2 == 1) {
      // last pass stays in registers; bins k / M-k are paired by warp shuffles
      float2 v[R1];
      dif_pass_last_regs<M, L1, R1>(buf, v, lane);
      stft_frame_out_regs<M, R1, EXTRA, true>(v, a.twN, a, clip, t0 + f, dst, orow0 + f, lane);
    } else {
      dif_pass<M, L1, R1, false, (R2 == 1), true, LANES>(buf, nullptr, nullptr, a.tw1, lane, group);
      if constexpr (R2 > 1) dif_pass<M, L2, R2, false, true, true, LANES>(buf, nullptr, nullptr, nullptr, lane, group);
      stft_frame_out<M, R0, R1, R2, EXTRA, true, LANES>(buf, a.twN, a, clip, t0 + f, dst, orow0 + f, lane, group, gmax);
    }
    group_sync<LANES>(group);
  }
}

// ---- n_fft = 4096 (the reference's default N): even / odd split on the tuned 1024-point path ------------------
// The frame's 2048 complex points z[n] = (x[2n], x[2n+1]) * window are split by parity; the two warps that share
// the frame each run the two-pass radix-32 x radix-32 transform of n_fft 2048 on one half (last pass in registers),
// leave E[k] / O[k] in natural order in their exchange buffers, and the 64 lanes then finish together:
//     Z[k] = E[k] + W2048^k O[k],   Z[k + 1024] = E[k] - W2048^k O[k],
// real-FFT split of the pairs (k, 2048 - k) and (1024 - k, 1024 + k) -- four output bins from E, O at k and 1024 - k --
// magnitudes (+ phasor / complex), maxima.  2.9 k warp instructions per frame instead of 5.7 k for the three-pass
// radix-16/16/8 form.  W2048^k = twN[2k], W4096^k = twN[k]; W2048^(1024-k) = -conj(W2048^k).
template <bool EXTRA>
__device__ __forceinline__ void eo_store(const StftArgs& a, int64_t row, int k, float2 X, float& vmax) {
  const float m = fast_sqrt(fmaf(X.x, X.x, X.y * X.y));
  vmax = fmaxf(vmax, m);
  a.mag_out[row + k] = m;
  if (EXTRA) {
    if (a.cplx_out) a.cplx_out[row + k] = X;
    if (a.phase_out) a.phase_out[row + k] = m > 0.f ? make_float2(X.x / m, X.y / m) : make_float2(1.f, 0.f);
  }
}

template <int WARPS, bool EXTRA, bool ROWS = false>
__global__ void __launch_bounds__(WARPS * 32, 2) stft_eo4096_kernel(const StftArgs a, const StftRows rows) {
  constexpr int M = 2048, N = 4096, MH = 1024, BUFH = MH + MH / 32, GROUPS = WARPS / 2;
  extern __shared__ __align__(16) float smem[];
  __shared__ float gmax[WARPS];
  float* span = smem;
  float2* bufs = reinterpret_cast<float2*>(smem + a.span_alloc);

  const int clip = blockIdx.x / a.tiles_per_clip;
  const int tile = blockIdx.x % a.tiles_per_clip;
  const int64_t len = a.clip_lens[clip];
  int64_t T;
  if (len <= 0) T = 0;
  else if (a.center) T = 1 + len / a.hop;
  else T = len >= N ? 1 + (len - N) / a.hop : 0;
  int64_t t0, orow0;
  int nF, dst;
  if (!stft_tile<ROWS, WARPS * 32>(a, rows, clip, tile, T, t0, nF, dst, orow0)) return;
  const float* x = a.wav + a.clip_offsets[clip];

  const int64_t s0 = t0 * a.hop - (a.center ? N / 2 : 0);
  const int span_len = (nF - 1) * a.hop + N;
  const bool interior = (s0 >= 0) && (s0 + span_len <= len);
  if (interior && ((reinterpret_cast<uintptr_t>(x + s0) & 15) == 0)) {
    const float4* src = reinterpret_cast<const float4*>(x + s0);
    float4* dst = reinterpret_cast<float4*>(span);
    const int n4 = span_len >> 2;
    for (int i = threadIdx.x; i < n4; i += WARPS * 32) dst[i] = __ldg(src + i);
    for (int i = (n4 << 2) + threadIdx.x; i < span_len; i += WARPS * 32) span[i] = __ldg(x + s0 + i);
  } else {
    for (int i = threadIdx.x; i < span_len; i += WARPS * 32) {
      int64_t s = s0 + i;
      if (s < 0 || s >= len) s = reflect_index(s, len);
      span[i] = __ldg(x + s);
    }
  }
  __syncthreads();

  const int group = threadIdx.x >> 6, lane64 = threadIdx.x & 63, par = lane64 >> 5, lane = threadIdx.x & 31;
  float2* bufE = bufs + group * (2 * BUFH);
  float2* bufO = bufE + BUFH;
  float2* mybuf = par ? bufO : bufE;
  const float2* win2 = reinterpret_cast<const float2*>(a.window);
  for (int f = group; f < nF; f += GROUPS) {
    const float* xs = span + f * a.hop;
    {
      // first pass of this warp's half: points m = lane + 32 r are the frame's pairs 2m + par
      float2 v[32];
      const bool al = ((reinterpret_cast<uintptr_t>(xs) & 7) == 0);
#pragma unroll
      for (int r = 0; r < 32; ++r) {
        const int n = 2 * (lane + 32 * r) + par;
        float2 xv;
        if (al) {
          xv = *reinterpret_cast<const float2*>(xs + 2 * n);
        } else {
          xv.x = xs[2 * n];
          xv.y = xs[2 * n + 1];
        }
        v[r] = pmul(xv, __ldg(win2 + n));
      }
      fft_reg<32>(v);
#pragma unroll
      for (int i = 0; i < 32; ++i) {
        const int rp = bitrev(i, 32);
        float2 o = v[i];
        if (rp > 0) o = cmul(o, __ldg(a.tw_eo + rp * 32 + lane));
        mybuf[pidx(lane + rp * 32)] = o;
      }
      __syncwarp();
      // second pass in registers: v[bitrev(rp)] = half-transform bin lane + 32 rp; back to the buffer in natural order
      dif_pass_last_regs<MH, 32, 32>(mybuf, v, lane);
      __syncwarp();
#pragma unroll
      for (int rp = 0; rp < 32; ++rp) mybuf[pidx(lane + 32 * rp)] = v[bitrev(rp, 32)];
    }
    group_sync<64>(group);

    // ---- combine the halves + real-FFT split, 64 lanes: k = lane64 + 64 i in [0, 512) --------------------
    const int64_t t = t0 + f;
    const int64_t row = (int64_t)dst * a.out_clip_stride + (orow0 + f) * a.frame_pitch;
    float vmax = 0.f;
#pragma unroll 2
    for (int i = 0; i < 8; ++i) {
      const int k = lane64 + 64 * i;
      const int km = (MH - k) & (MH - 1);              // 1024 - k (0 for k = 0)
      const float2 Ek = bufE[pidx(k)], Ok = bufO[pidx(k)];
      const float2 Em = bufE[pidx(km)], Om = bufO[pidx(km)];
      const float2 wk = __ldg(a.twN + 2 * k);          // W2048^k
      const float2 T1 = cmul(wk, Ok);
      const float2 T2 = cmul(make_float2(-wk.x, wk.y), Om);   // W2048^(1024-k) = -conj(W2048^k)
      const float2 Zk = cadd(Ek, T1), Zk1 = csub(Ek, T1);      // bins k, k + 1024
      const float2 Zm = cadd(Em, T2), Zm1 = csub(Em, T2);      // bins 1024 - k, 2048 - k
      float2 Xa, Xb, Xc, Xd;
      if (k != 0) {
        split_pair(Zk, Zm1, __ldg(a.twN + k), Xa, Xb);         // X[k], X[2048 - k]
        split_pair(Zm, Zk1, __ldg(a.twN + MH - k), Xc, Xd);    // X[1024 - k], X[1024 + k]
        eo_store<EXTRA>(a, row, k, Xa, vmax);
        eo_store<EXTRA>(a, row, M - k, Xb, vmax);
        eo_store<EXTRA>(a, row, MH - k, Xc, vmax);
        eo_store<EXTRA>(a, row, MH + k, Xd, vmax);
      } else {
        // k = 0: Z[0] = E0 + O0 pairs with itself (bins 0 and 2048), Z[1024] = E0 - O0 with itself (bin 1024)
        split_pair(Zk, Zk, __ldg(a.twN), Xa, Xb);
        split_pair(Zk1, Zk1, __ldg(a.twN + MH), Xc, Xd);
        eo_store<EXTRA>(a, row, 0, Xa, vmax);
        eo_store<EXTRA>(a, row, M, Xb, vmax);
        eo_store<EXTRA>(a, row, MH, Xc, vmax);
      }
    }
    if (lane64 == 0) {
      // k = 512: 1024 - k = k, one pair (512, 1536)
      const float2 Ek = bufE[pidx(512)], Ok = bufO[pidx(512)];
      const float2 T1 = cmul(__ldg(a.twN + 1024), Ok);
      float2 Xa, Xb;
      split_pair(cadd(Ek, T1), csub(Ek, T1), __ldg(a.twN + 512), Xa, Xb);
      eo_store<EXTRA>(a, row, 512, Xa, vmax);
      eo_store<EXTRA>(a, row, 1536, Xb, vmax);
    }
    for (int64_t k = M + 1 + lane64; k < a.frame_pitch; k += 64) {
      a.mag_out[row + k] = 0.f;
      if (EXTRA) {
        if (a.cplx_out) a.cplx_out[row + k] = make_float2(0.f, 0.f);
        if (a.phase_out) a.phase_out[row + k] = make_float2(0.f, 0.f);
      }
    }
    vmax = warp_max(vmax);
    if (lane == 0) gmax[threadIdx.x >> 5] = vmax;
    group_sync<64>(group);
    if (lane64 == 0) {
      vmax = fmaxf(vmax, gmax[(threadIdx.x >> 5) + 1]);
      if (a.frame_max_out) a.frame_max_out[(int64_t)clip * a.max_frames + t] = vmax;
      if (a.clip_max_out) atomic_max_nonneg(a.clip_max_out + clip, vmax);
    }
    group_sync<64>(group);
  }
}

template <int WARPS, bool ROWS = false>
static int launch_stft_eo4096(const saga_stft_plan* p, const StftArgs& a, int n_clips, cudaStream_t st,
                              const StftRows& rows = StftRows{}) {
  const bool extra = a.phase_out || a.cplx_out;
  auto kern = extra ? stft_eo4096_kernel<WARPS, true, ROWS> : stft_eo4096_kernel<WARPS, false, ROWS>;
  SAGA_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
  const int64_t blocks = (int64_t)n_clips * a.tiles_per_clip;
  if (blocks <= 0) return SAGA_OK;
  if (blocks > 0x7fffffffLL) return set_error(SAGA_ERR_INVALID, "stft: grid too large");
  if (a.frames_per_cta > WARPS / 2) return set_error(SAGA_ERR_INVALID, "stft: more frames per CTA than frame slots");
  kern<<<(unsigned)blocks, WARPS * 32, p->smem_bytes, st>>>(a, rows);
  SAGA_LAUNCH_CHECK();
  return SAGA_OK;
}

template <int M, int R0, int R1, int R2, int WARPS, bool ROWS = false>
static int launch_stft(const saga_stft_plan* p, const StftArgs& a, int n_clips, cudaStream_t st,
                       const StftRows& rows = StftRows{}) {
  const bool extra = a.phase_out || a.cplx_out;
  auto kern = extra ? stft_kernel<M, R0, R1, R2, WARPS, true, ROWS> : stft_kernel<M, R0, R1, R2, WARPS, false, ROWS>;
  SAGA_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
  const int64_t blocks = (int64_t)n_clips * a.tiles_per_clip;
  if (blocks <= 0) return SAGA_OK;
  if (blocks > 0x7fffffffLL) return set_error(SAGA_ERR_INVALID, "stft: grid too large");
  kern<<<(unsigned)blocks, WARPS * 32, p->smem_bytes, st>>>(a, rows);
  SAGA_LAUNCH_CHECK();
  return SAGA_OK;
}


// ---------------------------------------------------------------------------
// K4: inverse STFT (librosa.istft, util_audio.py:92-104).
// A CTA owns FO*hop consecutive output samples (padded coordinates) and runs the
// inverse FFT of every frame that overlaps them (FO + halo frames, one warp per
// frame, buffers kept in SMEM); each output sample then gathers its <= n_fft/hop
// contributions in ascending frame order (the reference's accumulation order),
// divides by the window sum-of-squares (accumulated the same way) and is stored
// once -- no atomics, no scratch in HBM, deterministic.
// ---------------------------------------------------------------------------
struct IstftArgs {
  const float2* cplx_in;
  const float* mag_in;
  const float2* phase_in;
  float* wav_out;
  const float* window;
  const float2* tw0;
  const float2* tw1;
  const float2* twN;
  int64_t frame_pitch, in_clip_stride, wav_clip_stride;
  int hop, center, n_frames, FO, nbuf, tiles_per_clip;
  const int32_t* frame0;    // optional: clip c inverts rows [frame0[c], frame0[c] + n_frames) of its spectrogram
};

// threads sharing one frame of the inverse transform: 64 for n_fft 4096 when the CTA has the 16 warps for it
__host__ __device__ constexpr int istft_lanes(int M, int warps) { return (M == 2048 && warps == 16) ? 64 : 32; }

template <int M, int R0, int R1, int R2, int WARPS>
__global__ void __launch_bounds__(WARPS * 32, (M <= 1024 ? 2 : 1)) istft_kernel(const IstftArgs a) {
  constexpr int N = 2 * M;
  constexpr int BUF = M + M / 32;
  extern __shared__ __align__(16) float smem[];
  float2* bufs = reinterpret_cast<float2*>(smem);
  const int clip = blockIdx.x / a.tiles_per_clip;
  const int tile = blockIdx.x % a.tiles_per_clip;
  const int T = a.n_frames;
  const int64_t total = (int64_t)N + (int64_t)a.hop * (T - 1);   // padded signal length
  const int64_t trim = a.center ? N / 2 : 0;
  const int64_t out_len = total - 2 * trim;
  // this CTA's output range in padded coordinates
  const int64_t p0 = trim + (int64_t)tile * a.FO * a.hop;
  const int64_t p1 = min(p0 + (int64_t)a.FO * a.hop, trim + out_len);
  if (p0 >= p1) return;
  // frames overlapping [p0, p1):  t*hop <= p < t*hop + N
  int64_t t_lo = (p0 - N + 1 + a.hop - 1) / a.hop;   // ceil((p0 - N + 1)/hop) for positive numerators
  if (p0 - N + 1 <= 0) t_lo = 0;
  int64_t t_hi = (p1 - 1) / a.hop;
  if (t_hi > T - 1) t_hi = T - 1;
  const int nfr = (int)(t_hi - t_lo + 1);             // <= nbuf by construction

  // n_fft 4096: two warps per frame (named barrier per frame slot), so that the 8 frames whose buffers fit the SM
  // bring 16 warps and run in one round
  constexpr int LANES = istft_lanes(M, WARPS);
  constexpr int GROUPS = WARPS * 32 / LANES;
  const int group = threadIdx.x / LANES, lane = threadIdx.x % LANES;
  for (int f = group; f < nfr; f += GROUPS) {
    float2* buf = bufs + f * BUF;
    const int64_t row = (int64_t)clip * a.in_clip_stride + (t_lo + f + (a.frame0 ? a.frame0[clip] : 0)) * a.frame_pitch;
    // rebuild conj(Z[k]),  Z = E + iO  from the half spectrum X[0..M]; four bins per lane in flight (the loads
    // of a bin pair are six independent global reads: one pair at a time left the warp waiting on DRAM latency)
    constexpr int U = 4;
#pragma unroll 1
    for (int k0 = lane; k0 <= M / 2; k0 += LANES * U) {
      float2 xk[U], xm[U];
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const int k = k0 + LANES * u;
        if (k > M / 2) continue;
        if (a.cplx_in) {
          xk[u] = a.cplx_in[row + k];
          xm[u] = a.cplx_in[row + M - k];
        } else {
          const float mk = a.mag_in[row + k], mm = a.mag_in[row + M - k];
          const float2 pk = a.phase_in[row + k], pm = a.phase_in[row + M - k];
          xk[u] = make_float2(mk * pk.x, mk * pk.y);
          xm[u] = make_float2(mm * pm.x, mm * pm.y);
        }
      }
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const int k = k0 + LANES * u;
        if (k > M / 2) continue;
        float2 a_k = xk[u], a_m = xm[u];
        if (k == 0) { a_k.y = 0.f; a_m.y = 0.f; }          // irfft ignores Im of DC and Nyquist
        const float2 E = make_float2(0.5f * (a_k.x + a_m.x), 0.5f * (a_k.y - a_m.y));
        const float2 D = make_float2(0.5f * (a_k.x - a_m.x), 0.5f * (a_k.y + a_m.y));   // W^k O
        const float2 w = __ldg(a.twN + k);
        const float2 O = make_float2(D.x * w.x + D.y * w.y, D.y * w.x - D.x * w.y); // D * conj(w)
        // Z[k] = E + iO ; Z[M-k] = conj(E) + i conj(O);  store conjugates
        buf[pidx(k)] = make_float2(E.x - O.y, -(E.y + O.x));
        if (k != 0 && k != M / 2) buf[pidx(M - k)] = make_float2(E.x + O.y, -(O.x - E.y));
      }
    }
    group_sync<LANES>(group);
    constexpr int L1 = M / R0, L2 = L1 / R1;
    dif_pass<M, M, R0, false, false, true, LANES>(buf, nullptr, nullptr, a.tw0, lane, group);
    dif_pass<M, L1, R1, false, (R2 == 1), true, LANES>(buf, nullptr, nullptr, a.tw1, lane, group);
    if constexpr (R2 > 1) dif_pass<M, L2, R2, false, true, true, LANES>(buf, nullptr, nullptr, nullptr, lane, group);
  }
  __syncthreads();

  // ---- gather / overlap-add in frame order, normalise, store -------------------
  const float inv_m = 1.0f / (float)M;
  float* y = a.wav_out + (int64_t)clip * a.wav_clip_stride;
  // positions relative to the first buffered frame: everything below fits 32-bit integers
  const int q0 = (int)(p0 - t_lo * a.hop), q1 = (int)(p1 - t_lo * a.hop);
  if (N == 4 * a.hop && (a.hop & 1) == 0) {
    // hop = n_fft / 4 (the reference's default and the bench shape): a thread owns the sample residues r = q mod hop,
    // keeps the four window values and buffer positions of that residue in registers and walks the tile's hop slots --
    // 4 shared-memory loads and 8 FMAs per sample instead of re-deriving frame ranges, window addresses and
    // digit-reversed positions per sample (2.4 k of the kernel's 6.3 k warp instructions per output frame).
    // Contributions are still added in ascending frame order (j = 3 .. 0).
    constexpr int J = 4;
    const int s0 = q0 / a.hop, s1 = q1 / a.hop;          // q0, q1 are multiples of hop here (trim = 2 hop)
    for (int r = threadIdx.x; r < a.hop; r += WARPS * 32) {
      float wn[J];
      int zp[J];
#pragma unroll
      for (int j = 0; j < J; ++j) {
        const int n = r + j * a.hop;
        wn[j] = __ldg(a.window + n);
        zp[j] = pidx(zpos<M, R0, R1, R2>(n >> 1));
      }
      const bool odd = r & 1;
      for (int sl = s0; sl < s1; ++sl) {
        float acc = 0.f, wss = 0.f;
#pragma unroll
        for (int jj = 0; jj < J; ++jj) {
          const int j = J - 1 - jj, f = sl - j;
          if (f >= 0 && f < nfr) {
            const float2 z = bufs[f * BUF + zp[j]];
            const float xv = (odd ? -z.y : z.x) * inv_m;
            acc += wn[j] * xv;
            wss += wn[j] * wn[j];
          }
        }
        if (wss > 1.17549435e-38f) acc /= wss;
        y[t_lo * a.hop + (int64_t)sl * a.hop + r - trim] = acc;
      }
    }
    return;
  }
  for (int q = q0 + threadIdx.x; q < q1; q += WARPS * 32) {
    const int fa = (q - N + 1 <= 0) ? 0 : (q - N + a.hop) / a.hop;     // ceil((q - N + 1)/hop)
    const int fb = min(q / a.hop, nfr - 1);
    const int64_t p = q + t_lo * a.hop;
    float acc = 0.f, wss = 0.f;
    for (int f = fa; f <= fb; ++f) {
      const int n = q - f * a.hop;
      const float wn = __ldg(a.window + n);
      const float2 z = bufs[f * BUF + pidx(zpos<M, R0, R1, R2>(n >> 1))];
      const float xv = ((n & 1) ? -z.y : z.x) * inv_m;
      acc += wn * xv;
      wss += wn * wn;
    }
    if (wss > 1.17549435e-38f) acc /= wss;
    y[p - trim] = acc;
  }
}

template <int M, int R0, int R1, int R2, int WARPS>
static int launch_istft(const saga_stft_plan* p, IstftArgs& a, int n_clips, cudaStream_t st) {
  auto kern = istft_kernel<M, R0, R1, R2, WARPS>;
  constexpr int BUF = M + M / 32;
  const int halo = (2 * M + p->hop - 1) / p->hop;  // frames that can overlap a chunk beyond its own FO
  int nbuf = (int)((200 * 1024) / (BUF * sizeof(float2)));
  if (M <= 1024) nbuf = std::min(nbuf, (int)((104 * 1024) / (BUF * sizeof(float2))));
  constexpr int GROUPS = WARPS * 32 / istft_lanes(M, WARPS);
  // multi-warp frames: every buffered frame gets its own group, one round (8 frames = 4 output hops + 4 halo frames
  // at hop = n_fft/4 beats 11 frames run as 8 + 3)
  if (istft_lanes(M, WARPS) > 32 && nbuf > GROUPS && GROUPS > halo) nbuf = GROUPS;
  int FO = nbuf - halo;
  if (FO < 1) return set_error(SAGA_ERR_UNSUPPORTED, "istft: hop=%d too small for n_fft=%d", p->hop, 2 * M);
  if (FO > 2 * GROUPS) FO = 2 * GROUPS;
  a.FO = FO;
  a.nbuf = FO + halo;
  const int64_t total = (int64_t)2 * M + (int64_t)p->hop * (a.n_frames - 1);
  const int64_t out_len = total - (p->center ? 2 * M : 0);
  if (out_len <= 0) return SAGA_OK;
  a.tiles_per_clip = (int)((out_len + (int64_t)FO * p->hop - 1) / ((int64_t)FO * p->hop));
  const size_t smem = (size_t)a.nbuf * BUF * sizeof(float2);
  SAGA_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
  const int64_t blocks = (int64_t)n_clips * a.tiles_per_clip;
  if (blocks > 0x7fffffffLL) return set_error(SAGA_ERR_INVALID, "istft: grid too large");
  kern<<<(unsigned)blocks, WARPS * 32, smem, st>>>(a);
  SAGA_LAUNCH_CHECK();
  return SAGA_OK;
}

}  // namespace saga

using namespace saga;

static void stft_shape(int n_fft, int* radix, int* n_pass, int* warps) {
  const int M = n_fft / 2;
  radix[2] = 1;
  *n_pass = 2;
  *warps = 8;
  switch (M) {
    case 128: radix[0] = 16; radix[1] = 8; break;
    case 256: radix[0] = 16; radix[1] = 16; break;
    case 512: radix[0] = 32; radix[1] = 16; break;
    case 1024: radix[0] = 32; radix[1] = 32; *warps = 10; break;
    // long transforms: 2 / 4 warps per frame (stft_lanes), so that the few frames whose exchange buffers fit an SM
    // still bring 16 warps with them
    case 2048: radix[0] = 16; radix[1] = 16; radix[2] = 8; *n_pass = 3; *warps = 8; break;
    case 4096: radix[0] = 16; radix[1] = 16; radix[2] = 16; *n_pass = 3; *warps = 8; break;
    default: radix[0] = 0;
  }
}

extern "C" int saga_stft_plan_create(saga_stft_plan** out, int n_fft, int hop, int center,
                                     const float* window_host) {
  if (!out) return set_error(SAGA_ERR_INVALID, "stft_plan_create: null output");
  *out = nullptr;
  if (hop < 1) return set_error(SAGA_ERR_INVALID, "stft_plan_create: hop_length must be >= 1");
  int radix[3], n_pass, warps;
  stft_shape(n_fft, radix, &n_pass, &warps);
  if (n_fft < 256 || n_fft > 8192 || (n_fft & (n_fft - 1)) || radix[0] == 0)
    return set_error(SAGA_ERR_UNSUPPORTED, "stft_plan_create: n_fft=%d not a power of two in [256, 8192]", n_fft);
  saga_stft_plan* p = new saga_stft_plan();
  p->n_fft = n_fft;
  p->hop = hop;
  p->center = center ? 1 : 0;
  p->M = n_fft / 2;
  p->n_pass = n_pass;
  for (int i = 0; i < 3; ++i) { p->radix[i] = radix[i]; p->d_tw[i] = nullptr; }
  p->d_tw_eo = nullptr;
  p->warps = warps;
  const int M = p->M;
  const double PI = 3.14159265358979323846;

  p->default_window = window_host ? 0 : 1;
  p->d_ring_tables = nullptr;
  p->d_iring_tables = nullptr;
  p->d_wsq = nullptr;
  std::vector<float> win(n_fft);
  for (int n = 0; n < n_fft; ++n)
    win[n] = window_host ? window_host[n] : (float)(0.5 - 0.5 * std::cos(2.0 * PI * n / n_fft));
  SAGA_CUDA_OK(cudaMalloc(&p->d_window, sizeof(float) * n_fft));
  SAGA_CUDA_OK(cudaMemcpy(p->d_window, win.data(), sizeof(float) * n_fft, cudaMemcpyHostToDevice));
  // forward transform: the 1/2 of the real-FFT split is folded into the analysis window (exact: power of two)
  std::vector<float> half_win(n_fft);
  for (int n = 0; n < n_fft; ++n) half_win[n] = 0.5f * win[n];
  SAGA_CUDA_OK(cudaMalloc(&p->d_window_half, sizeof(float) * n_fft));
  SAGA_CUDA_OK(cudaMemcpy(p->d_window_half, half_win.data(), sizeof(float) * n_fft, cudaMemcpyHostToDevice));

  // inter-pass twiddles: pass with block length L and radix R multiplies output r' of
  // the small FFT at in-block offset j by exp(-2*pi*i*j*r'/L); table layout [r'][j].
  int L = M;
  for (int ps = 0; ps + 1 < n_pass; ++ps) {
    const int R = radix[ps], LS = L / R;
    std::vector<float2> tw((size_t)L);
    for (int rp = 0; rp < R; ++rp)
      for (int j = 0; j < LS; ++j) {
        const double ang = -2.0 * PI * (double)(((int64_t)j * rp) % L) / (double)L;
        tw[(size_t)rp * LS + j] = make_float2((float)std::cos(ang), (float)std::sin(ang));
      }
    SAGA_CUDA_OK(cudaMalloc(&p->d_tw[ps], sizeof(float2) * L));
    SAGA_CUDA_OK(cudaMemcpy(p->d_tw[ps], tw.data(), sizeof(float2) * L, cudaMemcpyHostToDevice));
    L = LS;
  }
  if (M == 2048) {      // first-pass twiddles of the 1024-point halves (stft_eo4096_kernel)
    std::vector<float2> tw(1024);
    for (int rp = 0; rp < 32; ++rp)
      for (int j = 0; j < 32; ++j) {
        const double ang = -2.0 * PI * (double)((j * rp) % 1024) / 1024.0;
        tw[(size_t)rp * 32 + j] = make_float2((float)std::cos(ang), (float)std::sin(ang));
      }
    SAGA_CUDA_OK(cudaMalloc(&p->d_tw_eo, sizeof(float2) * 1024));
    SAGA_CUDA_OK(cudaMemcpy(p->d_tw_eo, tw.data(), sizeof(float2) * 1024, cudaMemcpyHostToDevice));
  }
  std::vector<float2> twN(M / 2 + 1);
  for (int k = 0; k <= M / 2; ++k) {
    const double ang = -2.0 * PI * k / (double)n_fft;
    twN[k] = make_float2((float)std::cos(ang), (float)std::sin(ang));
  }
  SAGA_CUDA_OK(cudaMalloc(&p->d_twN, sizeof(float2) * twN.size()));
  SAGA_CUDA_OK(cudaMemcpy(p->d_twN, twN.data(), sizeof(float2) * twN.size(), cudaMemcpyHostToDevice));

  // frames per CTA: as many as fit a ~100 KB CTA (two CTAs per SM), at most 1 per warp
  const int groups = warps * 32 / saga::stft_lanes(M);      // frames in flight per CTA (one exchange buffer each)
  const size_t buf_bytes = (size_t)groups * (M + M / 32) * sizeof(float2);
  const size_t budget = 112 * 1024;      // two CTAs per SM for every shape
  int F = 1;
  if (budget > buf_bytes + (size_t)n_fft * 4) {
    const size_t span_floats = (budget - buf_bytes) / 4;
    F = (int)((span_floats - n_fft) / hop) + 1;
  }
  if (F > groups) F = groups;   // one frame per warp (group): measured equal to two per warp on long clips (1.04 ms) and
                                // better on short ones (128-frame guesses: 0.30 vs 0.32 ms) -- finer tiles, same overlap reuse
  if (const char* e = SAGA_OPT("SAGA_STFT_FRAMES")) F = std::max(1, std::min(F, atoi(e)));   // tuning aid
  if (F < 1) F = 1;
  p->frames_per_cta = F;
  p->span_alloc = (((F - 1) * hop + n_fft) + 3) & ~3;
  p->smem_bytes = (size_t)p->span_alloc * 4 + buf_bytes;
  if (p->smem_bytes > 200 * 1024) {
    saga_stft_plan_destroy(p);
    return set_error(SAGA_ERR_UNSUPPORTED, "stft_plan_create: hop=%d too large for n_fft=%d staging", hop, n_fft);
  }
  if (int rc = saga::stft_ring_build_tables(p)) {
    saga_stft_plan_destroy(p);
    return rc;
  }
  if (int rc = saga::istft_ring_build_tables(p)) {
    saga_stft_plan_destroy(p);
    return rc;
  }
  *out = p;
  return SAGA_OK;
}

extern "C" int saga_stft_plan_destroy(saga_stft_plan* p) {
  if (!p) return SAGA_OK;
  cudaFree(p->d_window);
  cudaFree(p->d_window_half);
  for (int i = 0; i < 3; ++i) cudaFree(p->d_tw[i]);
  cudaFree(p->d_tw_eo);
  cudaFree(p->d_twN);
  cudaFree(p->d_ring_tables);
  cudaFree(p->d_iring_tables);
  cudaFree(p->d_wsq);
  delete p;
  return SAGA_OK;
}

extern "C" int64_t saga_stft_num_frames(const saga_stft_plan* p, int64_t len) {
  if (!p || len <= 0) return 0;
  if (p->center) return 1 + len / p->hop;
  return len >= p->n_fft ? 1 + (len - p->n_fft) / p->hop : 0;
}

extern "C" int saga_stft_exec(const saga_stft_plan* p, const float* wav, const int64_t* clip_offsets,
                              const int64_t* clip_lens, int n_clips, int64_t max_len, float* mag_out,
                              void* phase_out, void* cplx_out, int64_t frame_pitch,
                              int64_t out_clip_stride, float* frame_max_out, float* clip_max_out,
                              void* stream) {
  if (!p || !wav || !clip_offsets || !clip_lens || !mag_out)
    return set_error(SAGA_ERR_INVALID, "stft_exec: null argument");
  if (n_clips < 0) return set_error(SAGA_ERR_INVALID, "stft_exec: n_clips < 0");
  if (frame_pitch < p->M + 1)
    return set_error(SAGA_ERR_INVALID, "stft_exec: frame_pitch %lld < n_bins %d", (long long)frame_pitch, p->M + 1);
  cudaStream_t st = (cudaStream_t)stream;
  const int64_t T = saga_stft_num_frames(p, max_len);
  if (n_clips == 0 || T == 0) return SAGA_OK;
  if (clip_max_out) SAGA_CUDA_OK(cudaMemsetAsync(clip_max_out, 0, sizeof(float) * n_clips, st));

  StftArgs a;
  a.wav = wav;
  a.clip_offsets = clip_offsets;
  a.clip_lens = clip_lens;
  a.mag_out = mag_out;
  a.phase_out = (float2*)phase_out;
  a.cplx_out = (float2*)cplx_out;
  a.frame_max_out = frame_max_out;
  a.clip_max_out = clip_max_out;
  a.window = p->d_window_half;
  a.tw0 = p->d_tw[0];
  a.tw1 = p->d_tw[1];
  a.twN = p->d_twN;
  a.tw_eo = p->d_tw_eo;
  a.frame_pitch = frame_pitch;
  a.out_clip_stride = out_clip_stride;
  a.hop = p->hop;
  a.center = p->center;
  a.frames_per_cta = p->frames_per_cta;
  a.span_alloc = p->span_alloc;
  a.tiles_per_clip = (int)((T + p->frames_per_cta - 1) / p->frames_per_cta);
  a.max_frames = (int)T;
  switch (p->M) {
    case 128: return launch_stft<128, 16, 8, 1, 8>(p, a, n_clips, st);
    case 256: return launch_stft<256, 16, 16, 1, 8>(p, a, n_clips, st);
    case 512: return launch_stft<512, 32, 16, 1, 8>(p, a, n_clips, st);
    case 1024: {
      // ring kernel (stft_ring.cu) for the n_fft 2048 / hop 512 / Hann shape, whatever the batch size (the choice must
      // not depend on how a caller chunks its batch: the two kernels round differently); SAGA_STFT_RING=0 keeps the
      // first-generation kernel, the A/B twin of the parity tests
      const char* ring_opt = SAGA_OPT("SAGA_STFT_RING");
      const int ring_mode = ring_opt ? atoi(ring_opt) : 1;
      if (ring_mode > 0 && saga::stft_ring_supported(p)) return saga::launch_stft_ring(p, a, n_clips, T, st);
      return launch_stft<1024, 32, 32, 1, 10>(p, a, n_clips, st);
    }
    case 2048:
      if (SAGA_OPT("SAGA_STFT_NO_EO")) return launch_stft<2048, 16, 16, 8, 8>(p, a, n_clips, st);   // three-pass form (A/B)
      return launch_stft_eo4096<8>(p, a, n_clips, st);
    case 4096: return launch_stft<4096, 16, 16, 16, 8>(p, a, n_clips, st);
  }
  return set_error(SAGA_ERR_UNSUPPORTED, "stft_exec: unsupported n_fft");
}

extern "C" int saga_stft_rows_exec(const saga_stft_plan* p, const float* wav, const int64_t* clip_offsets,
                                   const int64_t* clip_lens, int n_clips, const int32_t* frame0, int n_frames,
                                   const int32_t* dst_clip, int dst_row0, int out_n_frames, float* mag_out,
                                   void* phase_out, int64_t frame_pitch, int64_t out_clip_stride, float* clip_max_out,
                                   void* stream) {
  if (!p || !wav || !clip_offsets || !clip_lens || !frame0 || !mag_out)
    return set_error(SAGA_ERR_INVALID, "stft_rows_exec: null argument");
  if (n_clips < 0) return set_error(SAGA_ERR_INVALID, "stft_rows_exec: n_clips < 0");
  if (n_frames <= 0) return set_error(SAGA_ERR_INVALID, "stft_rows_exec: n_frames %d <= 0", n_frames);
  if (frame_pitch < p->M + 1)
    return set_error(SAGA_ERR_INVALID, "stft_rows_exec: frame_pitch %lld < n_bins %d", (long long)frame_pitch, p->M + 1);
  if (dst_row0 < 0 || (int64_t)dst_row0 + n_frames > out_n_frames)
    return set_error(SAGA_ERR_INVALID, "stft_rows_exec: dst_row0 %d + n_frames %d outside the %d output rows", dst_row0,
                     n_frames, out_n_frames);
  if (out_clip_stride < (int64_t)out_n_frames * frame_pitch)
    return set_error(SAGA_ERR_INVALID, "stft_rows_exec: out_clip_stride %lld < out_n_frames * frame_pitch",
                     (long long)out_clip_stride);
  if (n_clips == 0) return SAGA_OK;
  cudaStream_t st = (cudaStream_t)stream;

  StftArgs a;
  a.wav = wav;
  a.clip_offsets = clip_offsets;
  a.clip_lens = clip_lens;
  a.mag_out = mag_out;
  a.phase_out = (float2*)phase_out;
  a.cplx_out = nullptr;
  a.frame_max_out = nullptr;
  a.clip_max_out = clip_max_out;
  a.window = p->d_window_half;
  a.tw0 = p->d_tw[0];
  a.tw1 = p->d_tw[1];
  a.twN = p->d_twN;
  a.tw_eo = p->d_tw_eo;
  a.frame_pitch = frame_pitch;
  a.out_clip_stride = out_clip_stride;
  a.hop = p->hop;
  a.center = p->center;
  a.frames_per_cta = p->frames_per_cta;
  a.span_alloc = p->span_alloc;
  a.tiles_per_clip = (n_frames + p->frames_per_cta - 1) / p->frames_per_cta;
  a.max_frames = 0;
  const StftRows r{frame0, dst_clip, n_frames, dst_row0};
  // saga_stft_exec's kernel choice, so that a row equals that entry's row bit for bit -- except n_fft 2048 / hop 512,
  // whose ring kernel stft_exec takes by default: the generic kernel here (stft_exec's SAGA_STFT_RING=0 twin)
  switch (p->M) {
    case 128: return launch_stft<128, 16, 8, 1, 8, true>(p, a, n_clips, st, r);
    case 256: return launch_stft<256, 16, 16, 1, 8, true>(p, a, n_clips, st, r);
    case 512: return launch_stft<512, 32, 16, 1, 8, true>(p, a, n_clips, st, r);
    case 1024: return launch_stft<1024, 32, 32, 1, 10, true>(p, a, n_clips, st, r);
    case 2048:
      if (SAGA_OPT("SAGA_STFT_NO_EO")) return launch_stft<2048, 16, 16, 8, 8, true>(p, a, n_clips, st, r);
      return launch_stft_eo4096<8, true>(p, a, n_clips, st, r);
    case 4096: return launch_stft<4096, 16, 16, 16, 8, true>(p, a, n_clips, st, r);
  }
  return set_error(SAGA_ERR_UNSUPPORTED, "stft_rows_exec: unsupported n_fft");
}

static int istft_exec_impl(const saga_stft_plan* p, const void* cplx_in, const float* mag_in,
                           const void* phase_in, int n_clips, int n_frames, int64_t frame_pitch,
                           int64_t in_clip_stride, float* wav_out, int64_t wav_clip_stride,
                           const int32_t* frame0, void* stream) {
  if (!p || !wav_out || (!cplx_in && !(mag_in && phase_in)))
    return set_error(SAGA_ERR_INVALID, "istft_exec: null argument");
  if (frame_pitch < p->M + 1) return set_error(SAGA_ERR_INVALID, "istft_exec: frame_pitch < n_bins");
  if (n_clips <= 0 || n_frames <= 0) return SAGA_OK;
  IstftArgs a;
  a.cplx_in = (const float2*)cplx_in;
  a.mag_in = mag_in;
  a.phase_in = (const float2*)phase_in;
  a.wav_out = wav_out;
  a.window = p->d_window;
  a.tw0 = p->d_tw[0];
  a.tw1 = p->d_tw[1];
  a.twN = p->d_twN;
  a.frame_pitch = frame_pitch;
  a.in_clip_stride = in_clip_stride;
  a.wav_clip_stride = wav_clip_stride;
  a.hop = p->hop;
  a.center = p->center;
  a.n_frames = n_frames;
  a.frame0 = frame0;
  cudaStream_t st = (cudaStream_t)stream;
  switch (p->M) {
    case 128: return launch_istft<128, 16, 8, 1, 8>(p, a, n_clips, st);
    case 256: return launch_istft<256, 16, 16, 1, 8>(p, a, n_clips, st);
    case 512: return launch_istft<512, 32, 16, 1, 8>(p, a, n_clips, st);
    case 1024: {
      // inverse ring kernel (istft_ring.cu): every frame transformed once, in-order overlap-add; SAGA_ISTFT_RING=0 keeps
      // the first-generation kernel (A/B twin of the parity tests)
      const char* ring_opt = SAGA_OPT("SAGA_ISTFT_RING");
      const int ring_mode = ring_opt ? atoi(ring_opt) : 1;
      // the ring kernel stages whole spectrogram rows with 16-byte bulk copies and stores sample pairs
      const uintptr_t in_bits = reinterpret_cast<uintptr_t>(cplx_in) | reinterpret_cast<uintptr_t>(mag_in) |
                                reinterpret_cast<uintptr_t>(phase_in);
      const bool aligned = (wav_clip_stride & 1) == 0 && (reinterpret_cast<uintptr_t>(wav_out) & 7) == 0 &&
                           (in_bits & 15) == 0 && (frame_pitch & 3) == 0 && frame_pitch >= p->M + 4 &&
                           (in_clip_stride & 3) == 0;
      if (ring_mode > 0 && aligned && !frame0 && saga::istft_ring_supported(p))
        return saga::launch_istft_ring(p, cplx_in, mag_in, phase_in, n_clips, n_frames, frame_pitch, in_clip_stride,
                                       wav_out, wav_clip_stride, st);
      return launch_istft<1024, 32, 32, 1, 8>(p, a, n_clips, st);
    }
    case 2048:
      if (SAGA_OPT("SAGA_ISTFT_ONE_WARP")) return launch_istft<2048, 16, 16, 8, 8>(p, a, n_clips, st);   // A/B
      return launch_istft<2048, 16, 16, 8, 16>(p, a, n_clips, st);
    case 4096: return launch_istft<4096, 16, 16, 16, 4>(p, a, n_clips, st);
  }
  return set_error(SAGA_ERR_UNSUPPORTED, "istft_exec: unsupported n_fft");
}

extern "C" int saga_istft_exec(const saga_stft_plan* p, const void* cplx_in, const float* mag_in,
                               const void* phase_in, int n_clips, int n_frames, int64_t frame_pitch,
                               int64_t in_clip_stride, float* wav_out, int64_t wav_clip_stride,
                               void* stream) {
  return istft_exec_impl(p, cplx_in, mag_in, phase_in, n_clips, n_frames, frame_pitch, in_clip_stride, wav_out,
                         wav_clip_stride, nullptr, stream);
}

extern "C" int saga_istft_rows_exec(const saga_stft_plan* p, const void* cplx_in, const float* mag_in,
                                    const void* phase_in, int n_clips, const int32_t* frame0, int n_frames,
                                    int64_t frame_pitch, int64_t in_clip_stride, float* wav_out,
                                    int64_t wav_clip_stride, void* stream) {
  if (!frame0) return set_error(SAGA_ERR_INVALID, "istft_rows_exec: null frame0");
  return istft_exec_impl(p, cplx_in, mag_in, phase_in, n_clips, n_frames, frame_pitch, in_clip_stride, wav_out,
                         wav_clip_stride, frame0, stream);
}

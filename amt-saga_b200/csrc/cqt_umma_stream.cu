// K2 contraction on the tensor cores, second form: GATHERED ROWS x STREAMED BANK (tcgen05 kind::tf32, sm_100a).
//
//   C[(clip, t), :] = sum_n y_o[clip][t*hop - n_fft/2 + n] * G_o[n, :]
//
// cqt_umma.cu keeps an octave's whole bank resident in shared memory, which only the 12-bins-per-octave
// transform fits (n_fft * 4 * ncol * 4 B <= ~150 KB).  The producer loop's own shapes -- 24, 48 and 192 bins per
// octave, kernels of 1024 / 2048 / 8192 samples, 48 / 96 / 384 real columns per octave (training.py:340-388) --
// have banks of 0.4 / 1.5 / 25 MB.  Here the bank is streamed: the K loop runs in stages of 32 samples and a
// stage is
//     A_hi, A_lo : 128 rows x 32 samples, row r = 32 contiguous samples of ONE frame, gathered from the padded
//                  level signal -- in SHARED MEMORY (16 B pieces into the K-major SWIZZLE_NONE core-matrix layout:
//                  plane g = samples 4g..4g+3 of every row, 16 B per row), or in TENSOR MEMORY (lane = row, one
//                  column per sample, written with tcgen05.st) where the accumulators leave room for a ring at
//                  least as deep: then only the bank crosses the shared-memory port
//     B          : the bank's 32 rows x n_main columns for this stage, ONE bulk copy from the pre-packed
//                  [n_fft/4][n_main][4] image (TF32 hi | lo side by side along N)
// and costs 4 K-slices x (main MMA N = n_main, correction MMA N = n_lo) issued by one thread: 3xTF32 split as in
// cqt_umma.cu (hi*hi + hi*lo + lo*hi in fp32 TMEM).  TMEM holds 1, 2 or 4 partial accumulators per buffer (long
// kernels: see cqt_stream_plan_init) and two buffers when the 512 columns allow it.
// A "row" is any frame of any clip, so the same kernel serves
//   * whole transforms  : rows = every frame of every clip, 128 consecutive (clip, frame) pairs per tile --
//                         clips of 258 frames pack densely, there are no partial tiles and no tail kernel;
//   * frame windows     : rows = frames [first[clip], first[clip] + 8) of every clip (saga_cqt_frames_exec: the
//                         producer loop keeps 8 columns of each per-note transform), 16 clips per tile;
//   * column-range peaks: rows = the frames of every clip PACKED back to back (a device prefix sum of the clip frame
//                         counts, so ragged clips cost their own frames, not T_max each), nothing stored: the
//                         epilogue keeps max |C| per clip (saga_cqt_peak_exec, the kernel's PEAK instantiation).
// Column groups of <= 128 real columns (64 filters) are separate work items, ordered (octave, group)-major so
// that all CTAs stream the same bank slab out of L2 at the same time.  A work item's group also names its clip
// range and bank, so one launch can contract several plans of equal geometry (one bank per pitch:
// cqt_stream_exec_multi); frame windows of small batches are split along K (finish kernel in cqt.cu).
//
// Warp roles of the persistent CTA (one per SM): 0-3 epilogue (TMEM lanes 32w..32w+31), 4 MMA issuer (stages in
// pairs on rings of >= 4 stages, the next stage's barrier probed inside the issue block), 5 bank loader (bulk
// copies), 6-21 row loaders in groups that take the stages in turn: global -> registers (the group's next stage,
// loaded while the other groups' stages run, so the L2 round trip is not on the ring's critical path) -> hi and lo
// planes, ONE mbarrier arrive per warp; 22 an optional second issuer (measured slower, off).  (The first version
// copied rows with cp.async and split them in separate converter warps: 256 per-thread barrier arrivals and an extra
// hand-over per stage cost more than the copies.)  Waiters off the critical path are polled by lane 0 with back-off.
// DESIGN.md section 4 / K2 (5) has the measurements behind each of these choices.
#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <vector>

#include "cqt_plan.cuh"
#include "saga_common.cuh"
#include "umma_ptx.cuh"

namespace saga {

constexpr int US_TILE_M = 128;
constexpr int US_KC = 32;                                  // samples per stage
constexpr int US_PLANES = US_KC / 4;
constexpr int US_W_MMA = 4, US_W_BANK = 5, US_W_LOAD0 = 6;
constexpr int US_LOAD_WARPS = 16;
constexpr int US_W_MMA2 = US_W_LOAD0 + US_LOAD_WARPS;       // second MMA issuer (plans with >= 2 partial accumulators)
constexpr int US_THREADS = 32 * (US_W_MMA2 + 1);
constexpr int US_MAX_LOAD_GROUPS = 4;                      // stage q is filled by loader group q % groups
constexpr int US_MAX_RPT = US_PLANES * US_TILE_M / (32 * US_LOAD_WARPS / US_MAX_LOAD_GROUPS);   // 8 pieces per thread
constexpr int US_MAX_STAGES = 6;
constexpr int US_MAX_GROUPS = 64;                          // (octave, column group) pairs per launch
constexpr int US_GROUP_COLS = 128;                         // real columns per group (64 filters)
// plane pitch = 128 rows + one 16-byte pad: the row loaders write 8 planes x 4 rows per warp instruction, and a
// pitch that is a multiple of 128 B would put the 8 planes of a row on the same banks
constexpr uint32_t US_PLANE_BYTES = US_TILE_M * 16 + 16;
constexpr uint32_t US_A_BYTES = (US_PLANES * US_PLANE_BYTES + 127u) & ~127u;   // one of hi / lo per stage
constexpr uint32_t US_SMEM_LIMIT = 232448 - 1024;

struct UsGroup {
  const float* sig;       // padded level signal of the octave, element 0 = sample -n_fft/2 of clip 0
  int64_t sig_stride;     // floats per clip
  const float* b_pack;    // [n_fft/4][n_main][4]: rows [0,ncol) TF32 hi, [ncol,2ncol) lo, rest 0
  int hop, n_fft, ncol, first_bin;   // first_bin of THIS column group
  int n_main, n_lo;
  int oct, filt0;         // octave index and first filter of the group within it (split-K partial sums)
  // rows of this group: a launch may carry the groups of SEVERAL plans of equal geometry (one kernel bank per pitch),
  // each contracting its own clips [clip0, clip0 + rows / rows_per_clip) of the batch
  int clip0;
  uint32_t n_rows, tiles, item0;   // rows, 128-row tiles, and first work item of the group (items: ks * tiles)
};

struct UsArgs {
  UsGroup grp[US_MAX_GROUPS];
  int n_groups, n_clips, n_bins;
  int rows_per_clip;            // whole transform: T_max; frame window: 8
  int frame_count;              // frame window: rows j < frame_count are stored
  const int32_t* frame_first;   // NULL = whole transform
  const int32_t* clip_frames;
  uint32_t total_items;
  float* mag_out;
  float2* cplx_out;
  int64_t frame_pitch, out_clip_stride;
  uint32_t b_stage_bytes;       // bank region per stage (largest group)
  uint32_t tmem_cols, acc_stride, part_stride;
  int stages;
  int load_groups;              // 4, or 2 when the ring has fewer than 4 stages (see the row loaders)
  int unroll2;                  // the issuer handles stages in pairs (ring of >= 4 stages)
  int issuers;                  // 1 or 2 MMA issuer warps; two take the stages in turn, each owning the partial
                                // accumulator(s) of its stages (parts % issuers == 0: deterministic)
  int a_tmem;                   // 1: the A operand (rows, hi and lo) lives in TMEM, not in shared memory (see below)
  uint32_t a_tmem_col;          // first TMEM column of the A ring: 64 columns per stage (32 hi | 32 lo)
  int parts, bufs;              // partial accumulators per buffer (stage st adds into partial st % parts), buffers
  // split-K (frame windows of small batches: a pitch group of the note-relative transforms is a few dozen clips, a
  // handful of tiles, and one CTA walking an 8192-sample kernel alone takes 220 us): the kernel length is cut into `ks`
  // slices, item = (group * ks + slice) * m_tiles + tile, and the slices' complex sums go to `partial`
  // [slice][clip][octave][pstride filters][8 frames][re, im] for cqt_frame_window_finish_kernel (cqt.cu)
  int ks, n_oct, pstride;
  float* partial;
  // peak mode (saga_cqt_peak_exec): PACKED rows -- row R is frame R - row_start[c] of the clip c with
  // row_start[c] <= R < row_start[c + 1] (device prefix sum of the clip frame counts, row_start[n_clips] = all rows), so
  // every group has ceil(row_start[n_clips] / 128) tiles, read by every role at kernel start.  Nothing is stored: the
  // epilogue folds max |C| over the bins of each row with col_lo[c] <= t < col_hi[c] into peak_out[c] (atomicMax on the
  // bits of a float >= 0; peak_out zeroed by the caller)
  const int32_t* row_start;     // NULL = not peak mode
  const int32_t* col_lo;
  const int32_t* col_hi;
  unsigned int* peak_out;
  int debug;                    // SAGA_UMMA_DEBUG (timing bisection only): 1 no MMAs, 2 no row copies, 8 no bank copies, 32 no lo conversion
  int* error_flag;
  long long* prof;              // debug & 16: per-CTA cycle counters [grid][8]
};

// (clip, frame) of row R; `store` = the row has an output slot, `live` = its frame exists
struct UsRow {
  int clip, j, t;
  bool store, live;
};
// work item -> (group, K slice, tile): groups are laid out one after the other, ks * tiles items each
struct UsItem {
  uint32_t g, slice, tile;
};
// peak mode: `ptiles` = packed tiles per group (every group covers all rows once, ks = 1)
template <bool PEAK>
__device__ __forceinline__ UsItem us_item(const UsArgs& a, uint32_t item, uint32_t ptiles) {
  UsItem it;
  if (PEAK) {
    it.g = item / ptiles;
    it.slice = 0;
    it.tile = item - it.g * ptiles;
    return it;
  }
  uint32_t g = 0;
  while (g + 1 < (uint32_t)a.n_groups && item >= a.grp[g + 1].item0) ++g;
  const uint32_t local = item - a.grp[g].item0, tiles = a.grp[g].tiles;
  it.g = g;
  it.slice = local / tiles;
  it.tile = local - it.slice * tiles;
  return it;
}
template <bool PEAK>
__device__ __forceinline__ UsRow us_row(const UsArgs& a, const UsGroup& gr, uint32_t R) {
  UsRow r;
  if (PEAK) {
    // packed rows: the last clip whose first row is <= R (clips without frames share their successor's row_start)
    const uint32_t n_rows = (uint32_t)a.row_start[a.n_clips];
    if (R >= n_rows) {
      r.clip = 0; r.j = 0; r.t = 0; r.store = false; r.live = false;
      return r;
    }
    int lo = 0, hi = a.n_clips - 1;
    while (lo < hi) {
      const int mid = (lo + hi + 1) >> 1;
      if ((uint32_t)a.row_start[mid] <= R) lo = mid; else hi = mid - 1;
    }
    r.clip = lo;
    r.j = r.t = (int)(R - (uint32_t)a.row_start[lo]);
    r.store = r.live = true;
    return r;
  }
  if (R >= gr.n_rows) {
    r.clip = gr.clip0; r.j = 0; r.t = 0; r.store = false; r.live = false;
    return r;
  }
  const int c = (int)(R / (uint32_t)a.rows_per_clip);
  r.clip = gr.clip0 + c;
  r.j = (int)(R - (uint32_t)c * (uint32_t)a.rows_per_clip);
  const int T = a.clip_frames[r.clip];
  if (a.frame_first) {
    r.t = a.frame_first[r.clip] + r.j;
    r.store = r.j < a.frame_count;
    r.live = r.t >= 0 && r.t < T;
  } else {
    r.t = r.j;
    r.live = r.store = r.t < T;
  }
  return r;
}

// One stage = 4 K-slices: per slice the main MMA (A_hi x [B_hi | B_lo], N = n_main, into columns [0, n_main) of
// the partial accumulator) and the correction MMA (A_lo x B_hi, N = n_lo).  The correction goes to the hi*lo
// columns [ncol, ncol + n_lo) -- NOT on top of the main columns as in cqt_umma.cu: every MMA is one truncating add
// per accumulator element, and the large main sums should see as few of them as possible.
// Both stage helpers also PROBE the next stage's `full` barrier: the probe is issued before the MMAs and its result is
// read after them, so its round trip hides behind the issue instead of preceding it.
__device__ __forceinline__ uint32_t us_mma_stage(uint32_t d_main, uint32_t d_lo, uint64_t a_hi, uint64_t a_lo, uint64_t b,
                                                 uint32_t idesc_main, uint32_t idesc_lo, uint32_t accumulate, uint32_t da,
                                                 uint32_t db, uint32_t next_bar, uint32_t next_parity) {
  uint32_t ready;
  asm volatile(
      "{\n\t"
      ".reg .pred e, p, t, nx;\n\t"
      ".reg .b64 ah, al, bb, dda, ddb;\n\t"
      "mbarrier.test_wait.parity.shared::cta.b64 nx, [%11], %12;\n\t"
      "elect.sync _|e, 0xFFFFFFFF;\n\t"
      "setp.ne.b32 p, %8, 0;\n\t"
      "setp.eq.b32 t, 0, 0;\n\t"
      "mov.b64 ah, %3;\n\t"
      "mov.b64 al, %4;\n\t"
      "mov.b64 bb, %5;\n\t"
      "cvt.u64.u32 dda, %9;\n\t"
      "cvt.u64.u32 ddb, %10;\n\t"
      "@e tcgen05.mma.cta_group::1.kind::tf32 [%1], ah, bb, %6, p;\n\t"
      "@e tcgen05.mma.cta_group::1.kind::tf32 [%2], al, bb, %7, t;\n\t"
      "add.u64 ah, ah, dda;\n\t add.u64 al, al, dda;\n\t add.u64 bb, bb, ddb;\n\t"
      "@e tcgen05.mma.cta_group::1.kind::tf32 [%1], ah, bb, %6, t;\n\t"
      "@e tcgen05.mma.cta_group::1.kind::tf32 [%2], al, bb, %7, t;\n\t"
      "add.u64 ah, ah, dda;\n\t add.u64 al, al, dda;\n\t add.u64 bb, bb, ddb;\n\t"
      "@e tcgen05.mma.cta_group::1.kind::tf32 [%1], ah, bb, %6, t;\n\t"
      "@e tcgen05.mma.cta_group::1.kind::tf32 [%2], al, bb, %7, t;\n\t"
      "add.u64 ah, ah, dda;\n\t add.u64 al, al, dda;\n\t add.u64 bb, bb, ddb;\n\t"
      "@e tcgen05.mma.cta_group::1.kind::tf32 [%1], ah, bb, %6, t;\n\t"
      "@e tcgen05.mma.cta_group::1.kind::tf32 [%2], al, bb, %7, t;\n\t"
      "selp.u32 %0, 1, 0, nx;\n\t"
      "}\n"
      : "=r"(ready)
      : "r"(d_main), "r"(d_lo), "l"(a_hi), "l"(a_lo), "l"(b), "r"(idesc_main), "r"(idesc_lo), "r"(accumulate), "r"(da), "r"(db),
        "r"(next_bar), "r"(next_parity)
      : "memory");
  return ready;
}

// The same stage with the A operand in TENSOR MEMORY (lane = row, one 32-bit column per sample: a K-slice is 8
// columns).  An SS-mode MMA is paced by the shared-memory bytes it reads (A 4 KB + B 32 N bytes per K-slice at
// 128 B/clk, on top of the loaders' stores and the bank copies through the same port); with A in TMEM only the bank
// crosses shared memory and the row loaders write straight from registers with tcgen05.st -- no shared-memory
// stores, no generic -> async proxy fence.
__device__ __forceinline__ uint32_t us_mma_stage_ts(uint32_t d_main, uint32_t d_lo, uint32_t a_hi, uint32_t a_lo, uint64_t b,
                                                    uint32_t idesc_main, uint32_t idesc_lo, uint32_t accumulate, uint32_t db,
                                                    uint32_t next_bar, uint32_t next_parity) {
  uint32_t ready;
  asm volatile(
      "{\n\t"
      ".reg .pred e, p, t, nx;\n\t"
      ".reg .b64 bb, ddb;\n\t"
      ".reg .b32 ah, al;\n\t"
      "mbarrier.test_wait.parity.shared::cta.b64 nx, [%10], %11;\n\t"
      "elect.sync _|e, 0xFFFFFFFF;\n\t"
      "setp.ne.b32 p, %8, 0;\n\t"
      "setp.eq.b32 t, 0, 0;\n\t"
      "mov.b32 ah, %3;\n\t"
      "mov.b32 al, %4;\n\t"
      "mov.b64 bb, %5;\n\t"
      "cvt.u64.u32 ddb, %9;\n\t"
      "@e tcgen05.mma.cta_group::1.kind::tf32 [%1], [ah], bb, %6, p;\n\t"
      "@e tcgen05.mma.cta_group::1.kind::tf32 [%2], [al], bb, %7, t;\n\t"
      "add.u32 ah, ah, 8;\n\t add.u32 al, al, 8;\n\t add.u64 bb, bb, ddb;\n\t"
      "@e tcgen05.mma.cta_group::1.kind::tf32 [%1], [ah], bb, %6, t;\n\t"
      "@e tcgen05.mma.cta_group::1.kind::tf32 [%2], [al], bb, %7, t;\n\t"
      "add.u32 ah, ah, 8;\n\t add.u32 al, al, 8;\n\t add.u64 bb, bb, ddb;\n\t"
      "@e tcgen05.mma.cta_group::1.kind::tf32 [%1], [ah], bb, %6, t;\n\t"
      "@e tcgen05.mma.cta_group::1.kind::tf32 [%2], [al], bb, %7, t;\n\t"
      "add.u32 ah, ah, 8;\n\t add.u32 al, al, 8;\n\t add.u64 bb, bb, ddb;\n\t"
      "@e tcgen05.mma.cta_group::1.kind::tf32 [%1], [ah], bb, %6, t;\n\t"
      "@e tcgen05.mma.cta_group::1.kind::tf32 [%2], [al], bb, %7, t;\n\t"
      "selp.u32 %0, 1, 0, nx;\n\t"
      "}\n"
      : "=r"(ready)
      : "r"(d_main), "r"(d_lo), "r"(a_hi), "r"(a_lo), "l"(b), "r"(idesc_main), "r"(idesc_lo), "r"(accumulate), "r"(db),
        "r"(next_bar), "r"(next_parity)
      : "memory");
  return ready;
}
// 8 consecutive TMEM columns of this thread's lane <- 8 registers
__device__ __forceinline__ void tmem_st8(uint32_t taddr, const float (&v)[8]) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"r"(taddr),
               "r"(__float_as_uint(v[0])), "r"(__float_as_uint(v[1])), "r"(__float_as_uint(v[2])), "r"(__float_as_uint(v[3])),
               "r"(__float_as_uint(v[4])), "r"(__float_as_uint(v[5])), "r"(__float_as_uint(v[6])), "r"(__float_as_uint(v[7]))
               : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// Row loads for the TMEM form.  tcgen05.st wants thread = row, but a thread that reads its own row touches 32
// different cache lines per warp instruction: 1024 tag look-ups per stage, which made the row loaders the bottleneck
// (every loader warp needed ~4500 cycles per stage of its own).  So the loads are issued coalesced -- P lanes share a
// row (P consecutive 16-byte pieces), instruction i of lane (g, l) reads piece l of row P*g + i: 32 / P lines per
// instruction -- and a P x P transpose inside each group of P lanes (log2 P butterfly steps of shuffles) hands
// thread P*g + l all P pieces of row P*g + l.
template <int P>
__device__ __forceinline__ void us_transpose(float4 (&x)[8], int lane) {
#pragma unroll
  for (int b = 1; b < P; b <<= 1) {
    const bool up = (lane & b) != 0;
#pragma unroll
    for (int i = 0; i < P; ++i) {
      if (i & b) continue;
      const int j = i | b;
      float4 t = up ? x[i] : x[j];          // what the partner lane needs from here
      t.x = __shfl_xor_sync(0xffffffffu, t.x, b);
      t.y = __shfl_xor_sync(0xffffffffu, t.y, b);
      t.z = __shfl_xor_sync(0xffffffffu, t.z, b);
      t.w = __shfl_xor_sync(0xffffffffu, t.w, b);
      if (up) x[i] = t; else x[j] = t;
    }
  }
}

// lane 0 polls, the others wait at the warp barrier and then observe the completed phase themselves (one try_wait
// that succeeds: acquire for every lane) -- 700 threads polling shared memory slow the barriers down for everybody
__device__ __forceinline__ bool us_test_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
// test_wait (non-blocking) in a spin loop, NOT try_wait: a thread that try_wait suspends is woken late
// (measured here: ~1900 cycles per hand-over with try_wait, two hand-overs per stage)
// `sleep_ns`: waiters that are not on the critical path (row loaders, epilogue) back off between probes -- a warp
// that spins flat out takes issue slots from the MMA issuer on the same scheduler
__device__ __forceinline__ void us_wait(uint64_t* bar, uint32_t parity, int lane, int* error_flag, unsigned sleep_ns = 0) {
  if (lane == 0) {
    uint32_t spins = 0;
    while (!us_test_wait(bar, parity)) {
      if (sleep_ns) __nanosleep(sleep_ns);
      if (++spins > UM_SPIN_LIMIT) {
        if (error_flag) atomicExch(error_flag, 1);
        __trap();
      }
    }
  }
  __syncwarp();
  while (!us_test_wait(bar, parity)) {}
}

template <bool PEAK>
__global__ void __launch_bounds__(US_THREADS, 1) cqt_umma_stream_kernel(const __grid_constant__ UsArgs a) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  const uint32_t S = (uint32_t)a.stages;
  const uint32_t a_smem = a.a_tmem ? 0u : 2u * US_A_BYTES;
  const uint32_t stage_bytes = a_smem + a.b_stage_bytes;                // [A_hi | A_lo | B], or [B] with A in TMEM
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem_raw + S * stage_bytes);
  uint64_t* full = bars + US_MAX_STAGES;           // [S] hi / lo planes written and the bank slab landed
  uint64_t* empty = bars + 2 * US_MAX_STAGES;      // [S] the stage's MMAs retired
  uint64_t* tfull = bars + 3 * US_MAX_STAGES;      // [2]
  uint64_t* tempty = bars + 3 * US_MAX_STAGES + 2; // [2]
  uint32_t* tmem_ptr_s = reinterpret_cast<uint32_t*>(bars + 3 * US_MAX_STAGES + 4);

  const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0);
  const int lane = threadIdx.x & 31;

  if (threadIdx.x == 0) {
    for (uint32_t s = 0; s < S; ++s) {
      mbar_init(&full[s], US_LOAD_WARPS / a.load_groups + 1);      // the stage's row-loader warps + the bank loader's expect_tx arrive
      mbar_init(&empty[s], 1);
    }
    for (int s = 0; s < 2; ++s) {
      mbar_init(&tfull[s], a.issuers);
      mbar_init(&tempty[s], 4);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncwarp();
  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_ptr_s)),
                 "r"(a.tmem_cols));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::);
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = __shfl_sync(0xffffffffu, *tmem_ptr_s, 0);
  const uint32_t G = gridDim.x;
  // peak mode: the packed row count is known on the device only (every role reads the same value)
  const uint32_t ptiles = PEAK ? ((uint32_t)a.row_start[a.n_clips] + US_TILE_M - 1) / US_TILE_M : 0u;
#define US_TOTAL_ITEMS (PEAK ? (uint32_t)a.n_groups * ptiles : a.total_items)

  if (warp < 4) {
    // =========================== epilogue ===========================
    const int ew = warp;
    uint32_t it_acc = 0;
    for (uint32_t item = blockIdx.x; item < US_TOTAL_ITEMS; item += G, ++it_acc) {
      const UsItem wi = us_item<PEAK>(a, item, ptiles);
      const uint32_t g = wi.g, slice = wi.slice, tile = wi.tile;
      const UsGroup& gr = a.grp[g];
      const uint32_t acc = a.bufs == 2 ? (it_acc & 1) : 0, acc_ph = a.bufs == 2 ? ((it_acc >> 1) & 1) : (it_acc & 1);
      const UsRow r = us_row<PEAK>(a, gr, tile * US_TILE_M + (uint32_t)(ew * 32 + lane));
      us_wait(&tfull[acc], acc_ph, lane, a.error_flag, 500);
      tc_fence_after();
      const int64_t row = (int64_t)r.clip * a.out_clip_stride + (int64_t)(a.frame_first ? r.j : r.t) * a.frame_pitch;
      const uint32_t tbase = tmem_base + acc * a.acc_stride + ((uint32_t)(ew * 32) << 16);
      const bool vec_ok = ((a.frame_pitch | a.out_clip_stride | (int64_t)gr.first_bin) & 3) == 0 && !a.cplx_out &&
                          (reinterpret_cast<uintptr_t>(a.mag_out) & 15) == 0;
      // peak mode: the row counts when its frame lies in the clip's column range
      const bool in_range = PEAK && r.live && r.t >= a.col_lo[r.clip] && r.t < a.col_hi[r.clip];
      float peak = 0.f;
      for (int c0 = 0; c0 < gr.ncol; c0 += 8) {
        float hi[8], lo[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) hi[i] = lo[i] = 0.f;
        for (int pt = 0; pt < a.parts; ++pt) {
          uint32_t v[8], u[8];
          tmem_ld8(tbase + (uint32_t)pt * a.part_stride + (uint32_t)c0, v);
          tmem_ld8(tbase + (uint32_t)pt * a.part_stride + (uint32_t)(gr.ncol + c0), u);
          tmem_ld_wait();
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            hi[i] += __uint_as_float(v[i]);
            lo[i] += __uint_as_float(u[i]);
          }
        }
        if (PEAK) {
          // the storing path's arithmetic below, folded into a maximum instead of stored
          if (in_range) {
            float sum[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) sum[i] = hi[i] + lo[i];
            const int bin0 = gr.first_bin + (c0 >> 1);
#pragma unroll
            for (int i = 0; i < 4; ++i) {
              const int bin = bin0 + i;
              if (bin >= 0 && bin < a.n_bins) peak = fmaxf(peak, sqrtf(sum[2 * i] * sum[2 * i] + sum[2 * i + 1] * sum[2 * i + 1]));
            }
          }
        } else if (a.ks > 1) {
          if (r.store) {
            float2* dst = reinterpret_cast<float2*>(
                a.partial + ((((int64_t)slice * a.n_clips + r.clip) * a.n_oct + gr.oct) * a.pstride + gr.filt0 + (c0 >> 1)) * 16) + r.j;
#pragma unroll
            for (int i = 0; i < 4; ++i) dst[8 * i] = make_float2(hi[2 * i] + lo[2 * i], hi[2 * i + 1] + lo[2 * i + 1]);
          }
        } else if (r.store) {
          float sum[8], m[4];
#pragma unroll
          for (int i = 0; i < 8; ++i) sum[i] = hi[i] + lo[i];      // the correction columns are ~2^-11 of the main ones
#pragma unroll
          for (int i = 0; i < 4; ++i)
            m[i] = r.live ? sqrtf(sum[2 * i] * sum[2 * i] + sum[2 * i + 1] * sum[2 * i + 1]) : 0.f;
          const int bin0 = gr.first_bin + (c0 >> 1);
          if (vec_ok && bin0 >= 0 && bin0 + 4 <= a.n_bins) {
            *reinterpret_cast<float4*>(a.mag_out + row + bin0) = make_float4(m[0], m[1], m[2], m[3]);
          } else {
#pragma unroll
            for (int i = 0; i < 4; ++i) {
              const int bin = bin0 + i;
              if (bin >= 0 && bin < a.n_bins) {
                a.mag_out[row + bin] = m[i];
                if (a.cplx_out) a.cplx_out[row + bin] = r.live ? make_float2(sum[2 * i], sum[2 * i + 1]) : make_float2(0.f, 0.f);
              }
            }
          }
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&tempty[acc]);
      if (PEAK) {
        // the lanes of one clip (a warp's 32 consecutive rows span one or a few clips) reduce first: one atomic per
        // clip and warp.  Magnitudes are >= 0, so the order of their bit patterns as integers is the float order.
        const unsigned same = __match_any_sync(0xffffffffu, in_range ? r.clip : -1);
        const unsigned bits = __reduce_max_sync(same, in_range ? __float_as_uint(peak) : 0u);
        if (in_range && lane == __ffs(same) - 1 && bits != 0u) atomicMax(a.peak_out + r.clip, bits);
      }
    }
  } else if (warp == US_W_MMA || warp == US_W_MMA2) {
    // =========================== MMA issuer(s) ===========================
    // One thread issues a stage's 8 MMAs in ~500 cycles (the tensor pipe's pace) and then spends ~450 on commit, ring
    // bookkeeping and the fence while the pipe drains.  With two issuer warps that take the stages in turn, one
    // warp's bookkeeping runs under the other's MMAs.  Issuer w adds stage st (st % 2 == w) into partial accumulator
    // st % parts, so with parts % 2 == 0 no accumulator is shared between the warps and the sums stay deterministic.
    const uint32_t iw = warp == US_W_MMA ? 0u : 1u, NI = (uint32_t)a.issuers;
    if (iw < NI) {
    uint32_t k = iw, it_acc = 0, ring_s = iw % S, ring_ph = (iw / S) & 1u;
    bool next_ready = false;
    const bool prof_on = (a.debug & 16) != 0 && iw == 0;
    long long pr_wait = 0, pr_issue = 0, pr_commit = 0, pr_acc = 0, pt = prof_on ? clock64() : 0;
    const long long pt_start = pt;
#define US_PROF(var) do { if (prof_on) { const long long n_ = clock64(); var += n_ - pt; pt = n_; } } while (0)
#define US_TL(kk, slot) do { if ((a.debug & 128) && blockIdx.x == 0 && lane == 0 && (kk) < 96u) a.prof[2048 + (kk) * 8 + (slot)] = clock64(); } while (0)
    for (uint32_t item = blockIdx.x; item < US_TOTAL_ITEMS; item += G, ++it_acc) {
      const uint32_t g = us_item<PEAK>(a, item, ptiles).g;
      const UsGroup& gr = a.grp[g];
      // (k runs over THIS issuer's stages: iw, iw + NI, ... across items; every item has a multiple of 4 stages)
      // instruction descriptors: D = f32, A = B = tf32, K-major both, M = 128
      const uint32_t idesc_base = (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(US_TILE_M >> 4) << 24);
      const uint32_t idesc_main = idesc_base | ((uint32_t)(gr.n_main >> 3) << 17);
      const uint32_t idesc_lo = idesc_base | ((uint32_t)(gr.n_lo >> 3) << 17);
      const uint32_t acc = a.bufs == 2 ? (it_acc & 1) : 0, acc_ph = a.bufs == 2 ? ((it_acc >> 1) & 1) : (it_acc & 1);
      US_PROF(pr_issue);
      us_wait(&tempty[acc], acc_ph ^ 1, lane, a.error_flag);
      tc_fence_after();
      US_PROF(pr_acc);
      const uint32_t d_tmem0 = tmem_base + acc * a.acc_stride;
      const uint32_t bchunk16 = (uint32_t)gr.n_main;           // K-chunk pitch of the slab in 16-byte units
      const int n_st = gr.n_fft / US_KC / a.ks;
      // The tensor core adds into the fp32 accumulator with truncation: the error grows with the number of
      // accumulation steps (measured ~6.6e-9 of peak per kernel sample).  Long kernels therefore alternate between
      // `parts` partial accumulators, which the epilogue adds in fp32.
      // Stages are issued in PAIRS when the ring is deep enough (unroll 2): both stages' MMAs go out back to back
      // and the two commits follow, so the commit / bookkeeping gap in which the tensor pipe drains is paid once per
      // 16 MMAs instead of once per 8.
      const int U = (a.unroll2 && NI == 1) ? 2 : 1;
      for (int st0 = (int)iw; st0 < n_st; st0 += (int)NI * U) {
        uint32_t slot[2];
#pragma unroll
        for (int u = 0; u < 2; ++u) {
          if (u >= U) break;
          const int st = st0 + u * (int)NI;
          // ring slot / phase kept incrementally (no divisions), and the NEXT stage's barrier is probed before this
          // stage's MMAs are issued: an mbarrier probe is a ~150-cycle round trip, and with wait -> issue -> commit ->
          // wait in series the tensor pipe idled ~800 cycles per stage although the data had been there for thousands
          const uint32_t s = ring_s, ph = ring_ph;
          slot[u] = s;
          const uint32_t d_tmem = d_tmem0 + (uint32_t)(st & (a.parts - 1)) * a.part_stride;
          const uint32_t accum = st >= a.parts ? 1u : 0u;
          if (!next_ready) {
            uint32_t spins = 0;
            while (!us_test_wait(&full[s], ph)) {
              if (++spins > UM_SPIN_LIMIT) {
                if (a.error_flag) atomicExch(a.error_flag, 1);
                __trap();
              }
            }
          }
          ring_s = s + NI;                       // this issuer's next stage
          ring_ph = ph;
          if (ring_s >= S) { ring_s -= S; ring_ph ^= 1u; }
          if (ring_s >= S) { ring_s -= S; ring_ph ^= 1u; }      // (NI = 2 on a ring of 2 or 3 stages can wrap twice: S >= 2)
          const uint32_t nbar = smem_u32(&full[ring_s]);
          // A written by tcgen05.st of other threads needs the tcgen05 fence; operands that came through shared memory
          // (generic stores + proxy fence, bulk copies) are ordered by the mbarrier alone
          if (a.a_tmem) tc_fence_after();
          if (u == 0) { US_PROF(pr_wait); US_TL(k, 0); }
          const uint32_t base = smem_u32(smem_raw + s * stage_bytes);
          const uint64_t db = smem_desc(base + a_smem, bchunk16 * 16u, 128);
          // 4 K-slices of 8 samples: planes (0,1), (2,3), (4,5), (6,7) against bank chunks (0,1), ...
          if (a.debug & 1) {
            next_ready = false;
          } else if (a.a_tmem) {
            const uint32_t ta = tmem_base + a.a_tmem_col + s * 64u;
            next_ready = us_mma_stage_ts(d_tmem, d_tmem + (uint32_t)gr.ncol, ta, ta + 32u, db, idesc_main, idesc_lo, accum,
                                         2u * bchunk16, nbar, ring_ph) != 0;
          } else {
            const uint64_t dah = smem_desc(base, US_PLANE_BYTES, 128);
            const uint64_t dal = smem_desc(base + US_A_BYTES, US_PLANE_BYTES, 128);
            next_ready = us_mma_stage(d_tmem, d_tmem + (uint32_t)gr.ncol, dah, dal, db, idesc_main, idesc_lo, accum,
                                      2u * (US_PLANE_BYTES >> 4), 2u * bchunk16, nbar, ring_ph) != 0;
          }
        }
        US_PROF(pr_issue);
        US_TL(k, 1);
#pragma unroll
        for (int u = 0; u < 2; ++u) {
          if (u >= U) break;
          if (a.debug & 64) {        // timing experiment only (no MMAs in flight): plain arrive instead of tcgen05.commit
            if (lane == 0) mbar_arrive(&empty[slot[u]]);
          } else {
            tc_commit(&empty[slot[u]]);
          }
        }
        if (st0 + (int)NI * U >= n_st) tc_commit(&tfull[acc]);      // this issuer's last stage(s) of the item
        __syncwarp();
        US_PROF(pr_commit);
        US_TL(k, 2);
        k += NI * (uint32_t)U;
      }
    }
    if (prof_on && lane == 0) {
      long long* o = a.prof + (size_t)blockIdx.x * 8;
      o[0] = pr_wait; o[1] = pr_issue; o[2] = pr_commit; o[3] = pr_acc; o[4] = clock64() - pt_start; o[5] = k;
    }
    }   // iw < NI
  } else if (warp == US_W_BANK) {
    // =========================== bank loader ===========================
    if (lane == 0) {
      uint32_t k = 0;
      for (uint32_t item = blockIdx.x; item < US_TOTAL_ITEMS; item += G) {
        const UsItem wi = us_item<PEAK>(a, item, ptiles);
        const uint32_t g = wi.g, slice = wi.slice;
        const UsGroup& gr = a.grp[g];
        const uint32_t bytes = (uint32_t)gr.n_main * (US_PLANES * 16u);
        const int n_st = gr.n_fft / US_KC / a.ks;
        const uint8_t* src = reinterpret_cast<const uint8_t*>(gr.b_pack) + (size_t)slice * n_st * bytes;
        for (int st = 0; st < n_st; ++st, ++k) {
          const uint32_t s = k % S;
          while (!us_test_wait(&empty[s], ((k / S) & 1) ^ 1)) __nanosleep(100);
          US_TL(k, 3);
          if (a.debug & 8) { mbar_arrive(&full[s]); continue; }
          mbar_arrive_expect_tx(&full[s], bytes);
          bulk_g2s(smem_u32(smem_raw + s * stage_bytes + a_smem), src + (size_t)st * bytes, bytes, &full[s]);
        }
      }
    }
  } else {
    // =========================== row loaders ===========================
    // `load_groups` groups of warps; group q fills stages q, q + groups, ... of every item (the stage count is a
    // multiple of 4): the generic -> async proxy fence that has to follow the shared-memory stores costs ~1000 cycles,
    // and a warp that fenced every stage capped the pipeline at one stage per fence (measured: 1100 cycles per stage
    // with every copy and MMA switched off).  groups <= ring stages, or a group could wait for a slot two uses ahead
    // and be fooled by the barrier's phase parity.  lane = plane + 8 * row: a warp instruction reads 4 rows x 128
    // contiguous bytes (4 cache lines) and writes 4 shared-memory wavefronts (padded plane pitch); a thread owns plane
    // (t & 7) of `rpt` rows and keeps its NEXT stage in registers, loaded while the other groups' stages run.
    if (a.a_tmem) {
      // ---- A in TMEM: thread = row (TMEM lane 32 * (warp % 4) + lane, the quarter a warp may touch); a group of
      // `wpg` warps has wpg / 4 warps per quarter, which share the stage's 32 samples of each row
      const int NGt = a.load_groups, wpgt = US_LOAD_WARPS / NGt, per_q = wpgt / 4;     // per_q = 1 or 2
      const int lwt = warp - US_W_LOAD0;
      const int grpt = lwt / wpgt, sub = (lwt - grpt * wpgt) / 4;                       // sub: which part of K
      const int quarter = warp & 3;
      const int row = quarter * 32 + lane;
      const int nk = US_KC / per_q;                                                     // samples per thread and stage
      const int k_off = sub * nk;
      const uint32_t lane_addr = (uint32_t)(quarter * 32) << 16;
      uint32_t k0t = 0;
      for (uint32_t item = blockIdx.x; item < US_TOTAL_ITEMS; item += G) {
        const UsItem wi = us_item<PEAK>(a, item, ptiles);
        const uint32_t g = wi.g, slice = wi.slice, tile = wi.tile;
        const UsGroup& gr = a.grp[g];
        const int n_st = gr.n_fft / US_KC / a.ks;
        const UsRow r = us_row<PEAK>(a, gr, tile * US_TILE_M + (uint32_t)row);
        const int T = a.clip_frames[r.clip];
        const int tc = max(min(r.t, T - 1), 0);      // frames outside the clip re-read an existing one (never stored)
        const float* own = gr.sig + (int64_t)r.clip * gr.sig_stride + (int64_t)tc * gr.hop + (int)slice * n_st * US_KC + k_off;
        // P = pieces per thread and stage (8, or 4 when two warps share a quarter); lane (g, l) = (lane / P, lane % P)
        // reads piece l of rows P*g + i: fetch those rows' pointers from the lanes that own them
        const int P = US_KC / 4 / per_q, lg = lane / P, ll = lane % P;
        const float4* src[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const unsigned long long pv = __shfl_sync(0xffffffffu, (unsigned long long)own, (P * lg + (i < P ? i : 0)) & 31);
          src[i] = reinterpret_cast<const float4*>(pv) + ll;
        }
        const bool copy = !(a.debug & 2);
        float4 x[8];
#pragma unroll
        for (int i = 0; i < 8; ++i)
          x[i] = (copy && i < P) ? __ldcg(src[i] + grpt * (US_KC / 4)) : make_float4(0.f, 0.f, 0.f, 0.f);
        for (int st = grpt; st < n_st; st += NGt) {
          const uint32_t k = k0t + (uint32_t)st;
          const uint32_t s = k % S;
          if (P == 8) us_transpose<8>(x, lane); else us_transpose<4>(x, lane);   // now x[0 .. P) = this thread's row
          us_wait(&empty[s], ((k / S) & 1) ^ 1, lane, a.error_flag, 100);
          tc_fence_after();
          const uint32_t ta = tmem_base + lane_addr + a.a_tmem_col + s * 64u + (uint32_t)k_off;
#pragma unroll
          for (int i = 0; i < US_KC / 8; ++i) {
            if (8 * i >= nk) break;
            const float4 v0 = x[2 * i], v1 = x[2 * i + 1];
            const float h[8] = {v0.x, v0.y, v0.z, v0.w, v1.x, v1.y, v1.z, v1.w};
            float l[8];
#pragma unroll
            for (int j = 0; j < 8; ++j)       // kind::tf32 reads the top 19 bits: raw samples ARE hi, lo = x - trunc13(x)
              l[j] = (a.debug & 32) ? h[j] : h[j] - __uint_as_float(__float_as_uint(h[j]) & 0xFFFFE000u);
            tmem_st8(ta + 8u * (uint32_t)i, h);
            tmem_st8(ta + 32u + 8u * (uint32_t)i, l);
          }
          tmem_st_wait();
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive(&full[s]);
          US_TL(k, 4 + ((lwt - grpt * wpgt) & 3));
          if (st + NGt < n_st && copy) {
#pragma unroll
            for (int i = 0; i < 8; ++i)
              if (i < P) x[i] = __ldcg(src[i] + (st + NGt) * (US_KC / 4));
          }
        }
        k0t += (uint32_t)n_st;
      }
    } else {
    const int NG = a.load_groups, wpg = US_LOAD_WARPS / NG, rpt = 2 * NG, rstep = 64 / NG;
    const int lw = warp - US_W_LOAD0;
    const int grp = lw / wpg, t = (lw - grp * wpg) * 32 + lane;
    const int plane = t & 7, row0 = t >> 3;
    const uint32_t dst_off = (uint32_t)plane * US_PLANE_BYTES + (uint32_t)row0 * 16u;
    uint32_t k0 = 0;                                   // ring index of the item's first stage
    for (uint32_t item = blockIdx.x; item < US_TOTAL_ITEMS; item += G) {
      const UsItem wi = us_item<PEAK>(a, item, ptiles);
      const uint32_t g = wi.g, slice = wi.slice, tile = wi.tile;
      const UsGroup& gr = a.grp[g];
      const int n_st = gr.n_fft / US_KC / a.ks;
      const float4* src[US_MAX_RPT];
#pragma unroll
      for (int i = 0; i < US_MAX_RPT; ++i) {
        const UsRow r = us_row<PEAK>(a, gr, tile * US_TILE_M + (uint32_t)(row0 + rstep * (i < rpt ? i : 0)));
        const int T = a.clip_frames[r.clip];
        const int tc = max(min(r.t, T - 1), 0);      // frames outside the clip re-read an existing one (never stored)
        src[i] = reinterpret_cast<const float4*>(gr.sig + (int64_t)r.clip * gr.sig_stride + (int64_t)tc * gr.hop + 4 * plane +
                                                 (int)slice * n_st * US_KC);
      }
      float4 x[US_MAX_RPT];
      const bool copy = !(a.debug & 2);
#pragma unroll
      for (int i = 0; i < US_MAX_RPT; ++i)
        x[i] = (copy && i < rpt) ? __ldcg(src[i] + grp * (US_KC / 4)) : make_float4(0.f, 0.f, 0.f, 0.f);
      for (int st = grp; st < n_st; st += NG) {
        const uint32_t k = k0 + (uint32_t)st;
        const uint32_t s = k % S;
        long long lt0 = (a.debug & 16) ? clock64() : 0;
        us_wait(&empty[s], ((k / S) & 1) ^ 1, lane, a.error_flag, 100);
        if ((a.debug & 16) && lw == 0 && lane == 0) a.prof[(size_t)blockIdx.x * 8 + 6] += clock64() - lt0;
        lt0 = (a.debug & 16) ? clock64() : 0;
        float4* dh = reinterpret_cast<float4*>(smem_raw + s * stage_bytes + dst_off);
        float4* dl = reinterpret_cast<float4*>(smem_raw + s * stage_bytes + US_A_BYTES + dst_off);
#pragma unroll
        for (int i = 0; i < US_MAX_RPT; ++i) {
          if (i >= rpt) break;
          // kind::tf32 reads the top 19 bits of an operand: the raw fp32 samples ARE the hi operand, and
          // lo = x - trunc13(x) is exact in fp32 (cqt_umma.cu)
          const float4 v = x[i];
          float4 l;
          l.x = v.x - __uint_as_float(__float_as_uint(v.x) & 0xFFFFE000u);
          l.y = v.y - __uint_as_float(__float_as_uint(v.y) & 0xFFFFE000u);
          l.z = v.z - __uint_as_float(__float_as_uint(v.z) & 0xFFFFE000u);
          l.w = v.w - __uint_as_float(__float_as_uint(v.w) & 0xFFFFE000u);
          dh[i * rstep] = v;                      // rows row0 + rstep * i
          dl[i * rstep] = (a.debug & 32) ? v : l;
        }
        fence_proxy_async_smem();     // generic-proxy writes -> visible to the tensor core (async proxy)
        __syncwarp();
        if (lane == 0) mbar_arrive(&full[s]);
        if ((a.debug & 16) && lw == 0 && lane == 0) a.prof[(size_t)blockIdx.x * 8 + 7] += clock64() - lt0;
        // this group's next stage: in flight while the other groups' stages are consumed
        if (st + NG < n_st && copy) {
#pragma unroll
          for (int i = 0; i < US_MAX_RPT; ++i)
            if (i < rpt) x[i] = __ldcg(src[i] + (st + NG) * (US_KC / 4));
        }
      }
      k0 += (uint32_t)n_st;
    }
    }   // shared-memory A
  }

#undef US_TOTAL_ITEMS
  tc_fence_before();
  __syncthreads();
  if (warp == 0) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(a.tmem_cols));
  }
}

// columns [n_bins, pitch) of every output row are defined as zero
__global__ void cqt_stream_zero_cols_kernel(float* mag, float2* cplx, const int32_t* clip_frames, int fixed_rows,
                                            int n_bins, int64_t pitch, int64_t clip_stride) {
  const int clip = blockIdx.y;
  const int rows = fixed_rows > 0 ? fixed_rows : clip_frames[clip];
  for (int t = blockIdx.x * blockDim.y + threadIdx.y; t < rows; t += gridDim.x * blockDim.y)
    for (int64_t k = n_bins + threadIdx.x; k < pitch; k += blockDim.x) {
      mag[clip * clip_stride + t * pitch + k] = 0.f;
      if (cplx) cplx[clip * clip_stride + t * pitch + k] = make_float2(0.f, 0.f);
    }
}

struct StreamPack {
  float* d_pack = nullptr;
  int oct = 0, col0 = 0, ncol = 0, n_main = 0, n_lo = 0;
};

}  // namespace saga

struct CqtStreamState {
  std::vector<saga::StreamPack> packs;   // (octave, column group), octave-major
  bool supported = false;
  uint32_t b_stage_bytes = 0, tmem_cols = 0, acc_stride = 0, part_stride = 0;
  size_t smem_bytes = 0;
  int stages = 0, num_sms = 0, parts = 1, bufs = 2, issuers = 1;
  // second configuration: A operand in TMEM (ts_stages = 0: the accumulators leave no room for it)
  int ts_stages = 0;
  uint32_t ts_col = 0;
  size_t ts_smem_bytes = 0;
  int* d_error = nullptr;
  long long* d_prof = nullptr;
};

namespace saga {

static float us_tf32_rna_host(float x) {
  uint32_t u;
  std::memcpy(&u, &x, 4);
  if ((u & 0x7F800000u) == 0x7F800000u) return x;
  u += 0x1000u;
  u &= ~0x1FFFu;
  float r;
  std::memcpy(&r, &u, 4);
  return r;
}

void cqt_stream_plan_init(saga_cqt_plan* p) {
  CqtStreamState* st = new CqtStreamState();
  p->stream_tc = st;
  int n_main_max = 0, n_fft_max = 0;
  size_t n_groups = 0;
  for (auto& o : p->oct) n_fft_max = std::max(n_fft_max, o.n_fft);
  // The tensor core adds into its fp32 accumulator with truncation: measured ~4.5e-9 of peak per kernel sample and
  // accumulator.  Long kernels alternate between `parts` partial accumulators (added in fp32 by the epilogue) to stay
  // below ~7e-6 where the 512 TMEM columns allow it.  A 128-column group needs 256 columns per partial ([hi*hi | hi*lo]),
  // so 8192-sample kernels (192 bins per octave) get two partials: 1.7e-5 of peak against the fp32 kernel.  Groups
  // of 64 columns with four partials measured 9.5e-6 but 23.3 instead of 13.9 ms per 600 windows (every row is
  // gathered twice as often), so the wide groups stay.
  int parts = 1;
  while (parts < 4 && 4.5e-9 * n_fft_max / parts > 7e-6) parts *= 2;
  const int group_cols = US_GROUP_COLS;
  for (auto& o : p->oct) {
    const int ncol = 2 * o.n_filters;
    if (ncol % 8) return;                                   // the epilogue reads 8 columns (4 filters) at a time
    if (o.hop < 4 || (o.hop % 4) != 0 || (o.n_fft % US_KC) != 0 || o.n_fft / US_KC < 4) return;
    n_groups += (size_t)(ncol + group_cols - 1) / group_cols;
  }
  if (n_groups == 0 || n_groups > (size_t)US_MAX_GROUPS) return;
  for (size_t oi = 0; oi < p->oct.size(); ++oi) {
    const CqtOctaveDev& o = p->oct[oi];
    const int ncol_o = 2 * o.n_filters;
    for (int c0 = 0; c0 < ncol_o; c0 += group_cols) {
      StreamPack pk;
      pk.oct = (int)oi;
      pk.col0 = c0;
      pk.ncol = std::min(group_cols, ncol_o - c0);
      pk.n_main = (2 * pk.ncol + 15) & ~15;                 // [B_hi | B_lo]; M = 128 needs N % 16 == 0
      pk.n_lo = (pk.ncol + 15) & ~15;
      n_main_max = std::max(n_main_max, pk.n_main);
      const size_t n = (size_t)o.n_fft * pk.n_main;
      std::vector<float> pack(n, 0.f);
      for (int k = 0; k < o.n_fft; ++k) {
        const size_t chunk = (size_t)(k / 4) * pk.n_main;
        for (int c = 0; c < pk.ncol; ++c) {
          const float b = o.bank_host[(size_t)k * ncol_o + c0 + c];
          const float h = us_tf32_rna_host(b);
          pack[(chunk + c) * 4 + (k % 4)] = h;
          pack[(chunk + pk.ncol + c) * 4 + (k % 4)] = us_tf32_rna_host(b - h);
        }
      }
      if (cudaMalloc(&pk.d_pack, n * 4) != cudaSuccess) { cudaGetLastError(); return; }
      cudaMemcpy(pk.d_pack, pack.data(), n * 4, cudaMemcpyHostToDevice);
      st->packs.push_back(pk);
    }
  }
  st->b_stage_bytes = (uint32_t)n_main_max * (US_PLANES * 16u);
  const uint32_t stage = 2u * US_A_BYTES + st->b_stage_bytes;
  int fit = (int)((US_SMEM_LIMIT - 512u) / stage);
  fit = std::min(fit, US_MAX_STAGES);
  if (fit < 2) return;
  st->stages = fit;
  st->smem_bytes = (size_t)fit * stage + 512;
  // accumulator layout: `parts` partial accumulators per buffer, two buffers when 512 TMEM columns allow it
  const uint32_t w = ((uint32_t)n_main_max + 31u) & ~31u;
  while (parts > 1 && (uint32_t)parts * w > 512) parts /= 2;
  if (w > 512) return;
  st->issuers = parts >= 2 ? 2 : 1;        // what SAGA_CQT_STREAM_TWO_ISSUERS may use
  st->parts = parts;
  st->bufs = (2u * parts * w <= 512) ? 2 : 1;
  uint32_t cols = 32;
  while (cols < (uint32_t)(st->bufs * parts) * w) cols <<= 1;
  st->tmem_cols = cols;
  st->part_stride = w;
  st->acc_stride = parts * w;
  // A in TMEM: 64 columns per stage behind the accumulators (the allocation becomes all 512 columns)
  {
    const uint32_t acc_cols = (uint32_t)(st->bufs * parts) * w;
    int ts = acc_cols < 512 ? (int)((512 - acc_cols) / 64) : 0;
    ts = std::min(ts, std::min(US_MAX_STAGES, (int)((US_SMEM_LIMIT - 512u) / st->b_stage_bytes)));
    if (ts >= 2) {
      st->ts_stages = ts;
      st->ts_col = acc_cols;
      st->ts_smem_bytes = (size_t)ts * st->b_stage_bytes + 512;
    }
  }
  if (cudaMalloc(&st->d_error, sizeof(int)) != cudaSuccess) { cudaGetLastError(); return; }
  cudaMemset(st->d_error, 0, sizeof(int));
  if (cudaMalloc(&st->d_prof, sizeof(long long) * (2048 + 96 * 8)) != cudaSuccess) { cudaGetLastError(); return; }
  cudaMemset(st->d_prof, 0, sizeof(long long) * (2048 + 96 * 8));
  int dev = 0;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&st->num_sms, cudaDevAttrMultiProcessorCount, dev);
  // the attribute is per function, plans differ in their needs: ask for the maximum once
  if (cudaFuncSetAttribute(cqt_umma_stream_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)US_SMEM_LIMIT) != cudaSuccess ||
      cudaFuncSetAttribute(cqt_umma_stream_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)US_SMEM_LIMIT) != cudaSuccess) {
    cudaGetLastError();
    return;
  }
  st->supported = true;
}

void cqt_stream_plan_free(saga_cqt_plan* p) {
  if (!p->stream_tc) return;
  for (auto& pk : p->stream_tc->packs) cudaFree(pk.d_pack);
  cudaFree(p->stream_tc->d_error);
  cudaFree(p->stream_tc->d_prof);
  delete p->stream_tc;
  p->stream_tc = nullptr;
}

bool cqt_stream_supported(const saga_cqt_plan* p) { return p->stream_tc && p->stream_tc->supported; }

int cqt_stream_exec(const saga_cqt_plan* p, const CqtLevels& lv, int n_clips, int64_t T_max,
                    const int32_t* frame_first, int frame_count, float* mag_out, float2* cplx_out,
                    int64_t frame_pitch, int64_t out_clip_stride, cudaStream_t stream, int max_slices,
                    float* partial, int pstride, int* slices_out) {
  const int zero = 0;
  return cqt_stream_exec_multi(&p, 1, &zero, &n_clips, lv, n_clips, T_max, frame_first, frame_count, mag_out, cplx_out,
                               frame_pitch, out_clip_stride, stream, max_slices, partial, pstride, slices_out);
}

int cqt_stream_peak_exec(const saga_cqt_plan* p, const CqtLevels& lv, int n_clips, int64_t T_max, const CqtPeakArgs& peak,
                         cudaStream_t stream) {
  const int zero = 0;
  return cqt_stream_exec_multi(&p, 1, &zero, &n_clips, lv, n_clips, T_max, nullptr, 0, nullptr, nullptr, p->n_bins, 0,
                               stream, 1, nullptr, 0, nullptr, &peak);
}

// Several plans of EQUAL geometry (one kernel bank per pitch: the note-relative transforms of a per-note iteration) in
// as few launches as the 64-group argument block allows: plan i contracts clips [clip0[i], clip0[i] + nclips[i]) of the
// batch whose cascade `lv` describes.  All launches use the same K split (the caller's finish kernel runs once).
int cqt_stream_exec_multi(const saga_cqt_plan* const* plans, int n_plans, const int* clip0, const int* nclips,
                          const CqtLevels& lv, int n_clips, int64_t T_max, const int32_t* frame_first, int frame_count,
                          float* mag_out, float2* cplx_out, int64_t frame_pitch, int64_t out_clip_stride,
                          cudaStream_t stream, int max_slices, float* partial, int pstride, int* slices_out,
                          const CqtPeakArgs* peak) {
  if (n_plans < 1) return SAGA_OK;
  const saga_cqt_plan* p = plans[0];
  const CqtStreamState* st = p->stream_tc;
  if (!st || !st->supported) return set_error(SAGA_ERR_UNSUPPORTED, "cqt: plan does not fit the streamed tcgen05 path");
  for (int i = 1; i < n_plans; ++i) {
    const CqtStreamState* si = plans[i]->stream_tc;
    if (!si || !si->supported || si->packs.size() != st->packs.size() || si->b_stage_bytes != st->b_stage_bytes ||
        si->parts != st->parts || si->bufs != st->bufs || plans[i]->oct.size() != p->oct.size())
      return set_error(SAGA_ERR_INVALID, "cqt: plans of one shared-cascade launch must have the same geometry");
  }
  const int gpp = (int)st->packs.size();                       // groups per plan
  if (gpp > US_MAX_GROUPS) return set_error(SAGA_ERR_UNSUPPORTED, "cqt: too many column groups");
  const int plans_per_launch = US_MAX_GROUPS / gpp;
  const int rows_per_clip = frame_first ? 8 : (int)T_max;
  if ((int64_t)n_clips * rows_per_clip >= ((int64_t)1 << 31)) return set_error(SAGA_ERR_UNSUPPORTED, "cqt: batch too large for one launch");
  int min_st = 1 << 30;
  for (auto& o : p->oct) min_st = std::min(min_st, o.n_fft / US_KC);
  const int n_sm = st->num_sms > 0 ? st->num_sms : 148;
  // work items of the first launch decide the K split (split-K: frame windows only, the caller provides the scratch
  // and runs the finish kernel): until the launch covers most of the SMs, with >= 8 stages per slice
  int ks = 1;
  {
    int64_t items = 0;
    for (int i = 0; i < std::min(n_plans, plans_per_launch); ++i)
      items += (((int64_t)nclips[i] * rows_per_clip + US_TILE_M - 1) / US_TILE_M) * gpp;
    if (frame_first && partial)
      while (2 * ks <= max_slices && items * ks < n_sm && min_st / (2 * ks) >= 8 && min_st % (2 * ks) == 0) ks *= 2;
  }
  if (slices_out) *slices_out = ks;
  if (frame_pitch > p->n_bins && ks == 1 && !peak) {      // (the split-K finish kernel writes the padding itself)
    dim3 grid(frame_first ? 1 : 8, n_clips), block(32, 8);
    cqt_stream_zero_cols_kernel<<<grid, block, 0, stream>>>(mag_out, cplx_out, lv.clip_frames, frame_first ? frame_count : 0,
                                                            p->n_bins, frame_pitch, out_clip_stride);
    SAGA_LAUNCH_CHECK();
  }
  for (int p0 = 0; p0 < n_plans; p0 += plans_per_launch) {
  const int p1 = std::min(n_plans, p0 + plans_per_launch);
  UsArgs a;
  std::memset(&a, 0, sizeof(a));
  a.n_clips = n_clips;
  a.n_bins = p->n_bins;
  a.rows_per_clip = rows_per_clip;
  a.frame_count = frame_count;
  a.frame_first = frame_first;
  a.clip_frames = lv.clip_frames;
  a.ks = ks;
  a.n_oct = (int)p->oct.size();
  a.pstride = pstride;
  a.partial = partial;
  if (peak) {        // rows are packed on the device: the launch is sized for n_clips * T_max, the kernel runs what exists
    a.row_start = peak->row_start;
    a.col_lo = peak->col_lo;
    a.col_hi = peak->col_hi;
    a.peak_out = reinterpret_cast<unsigned int*>(peak->peak_out);
  }
  uint32_t item0 = 0;
  int ng = 0;
  for (int pi = p0; pi < p1; ++pi) {
    const saga_cqt_plan* pp = plans[pi];
    const CqtStreamState* sp = pp->stream_tc;
    const int64_t rows = (int64_t)nclips[pi] * rows_per_clip;
    if (rows <= 0) continue;
    if (clip0[pi] < 0 || clip0[pi] + nclips[pi] > n_clips) return set_error(SAGA_ERR_INVALID, "cqt: clip range outside the batch");
    const uint32_t tiles = (uint32_t)((rows + US_TILE_M - 1) / US_TILE_M);
    for (int i = 0; i < gpp; ++i) {
      const StreamPack& pk = sp->packs[i];
      const CqtOctaveDev& o = pp->oct[pk.oct];
      UsGroup& g = a.grp[ng++];
      g.sig = lv.lvl[o.level] + (lv.pad[o.level] - o.n_fft / 2);
      g.sig_stride = lv.pitch[o.level];
      g.b_pack = pk.d_pack;
      g.hop = o.hop;
      g.n_fft = o.n_fft;
      g.ncol = pk.ncol;
      g.first_bin = o.first_bin + pk.col0 / 2;
      g.n_main = pk.n_main;
      g.n_lo = pk.n_lo;
      g.oct = pk.oct;
      g.filt0 = pk.col0 / 2;
      g.clip0 = clip0[pi];
      g.n_rows = (uint32_t)rows;
      g.tiles = tiles;
      g.item0 = item0;
      item0 += tiles * (uint32_t)ks;
    }
  }
  if (ng == 0) continue;
  a.n_groups = ng;
  a.total_items = item0;
  a.mag_out = mag_out;
  a.cplx_out = cplx_out;
  a.frame_pitch = frame_pitch;
  a.out_clip_stride = out_clip_stride;
  a.b_stage_bytes = st->b_stage_bytes;
  a.tmem_cols = st->tmem_cols;
  a.acc_stride = st->acc_stride;
  a.part_stride = st->part_stride;
  a.parts = st->parts;
  a.bufs = st->bufs;
  a.stages = st->stages;
  size_t smem_bytes = st->smem_bytes;
  // default: rows in TMEM when the accumulators leave room (SAGA_CQT_STREAM_SS=1 keeps them in shared memory: A/B)
  // (a deeper shared-memory ring beats a 2-stage TMEM ring: 348/48 3.14 against 3.35 ms; at 174/24 both have 5 stages
  // and tie, and the TMEM form leaves 160 KB of shared memory unused)
  if (st->ts_stages >= 2 && (st->ts_stages >= 4 || st->ts_stages >= st->stages) && !SAGA_OPT("SAGA_CQT_STREAM_SS")) {
    a.a_tmem = 1;
    a.a_tmem_col = st->ts_col;
    a.tmem_cols = 512;
    a.stages = st->ts_stages;
    smem_bytes = st->ts_smem_bytes;
  }
  if (const char* cfg = SAGA_OPT("SAGA_UMMA_CFG")) {      // tuning aid: "stages,x" caps the ring depth
    const int cap = atoi(cfg);
    if (cap >= 2 && cap < a.stages) a.stages = cap;
  }
  // Default: ONE issuer.  Two (SAGA_CQT_STREAM_TWO_ISSUERS=1, plans with two partial accumulators) measured slower:
  // 348/48 3.78 -> 3.95 ms, 348/192 10.2 -> 15.0 ms per 600 windows (the ring must then be an even number of stages)
  a.issuers = SAGA_OPT("SAGA_CQT_STREAM_TWO_ISSUERS") ? st->issuers : 1;
  // Two issuers retire stages out of order with respect to each other.  A row-loader group only knows that the stage
  // it filled one ring lap ago has retired; for the mbarrier phase parity to stay unambiguous every earlier use of the
  // slot it waits for must have retired too, which holds when all of them belong to the SAME issuer: ring depth and
  // loader groups are kept multiples of the issuer count (and groups <= depth).
  if (a.issuers == 2) a.stages &= ~1;
  a.unroll2 = (a.stages >= 4 && !SAGA_OPT("SAGA_CQT_STREAM_NO_UNROLL")) ? 1 : 0;
  a.load_groups = a.stages >= 4 ? 4 : 2;
  a.error_flag = st->d_error;
  a.prof = st->d_prof;
  {
    const char* dbg = SAGA_OPT("SAGA_UMMA_DEBUG");
    a.debug = dbg ? atoi(dbg) : 0;
  }
  const int grid = (int)std::min<int64_t>(a.total_items, n_sm);
  if (a.debug & (16 | 128)) cudaMemsetAsync(st->d_prof, 0, sizeof(long long) * (2048 + 96 * 8), stream);
  if (peak) cqt_umma_stream_kernel<true><<<grid, US_THREADS, smem_bytes, stream>>>(a);
  else cqt_umma_stream_kernel<false><<<grid, US_THREADS, smem_bytes, stream>>>(a);
  SAGA_LAUNCH_CHECK();
  if (a.debug & 128) {
    // profiling aid only: timeline of CTA 0's first 96 stages (cycles relative to the first event)
    std::vector<long long> h(96 * 8);
    cudaStreamSynchronize(stream);
    cudaMemcpy(h.data(), st->d_prof + 2048, h.size() * sizeof(long long), cudaMemcpyDeviceToHost);
    long long t0 = 0;
    for (long long v : h) if (v && (!t0 || v < t0)) t0 = v;
    fprintf(stderr, "us_tl stage  mma.full_seen mma.issued mma.committed | bank.empty_seen | arrival of the 4 row-loader warps of the stage\n");
    for (int kk = 0; kk < 96; ++kk) {
      fprintf(stderr, "us_tl %3d ", kk);
      for (int j = 0; j < 8; ++j) fprintf(stderr, " %8lld", h[kk * 8 + j] ? h[kk * 8 + j] - t0 : -1);
      fprintf(stderr, "\n");
    }
  }
  if (a.debug & 16) {
    // profiling aid only: synchronous read-back of the MMA issuer's cycle split, mean over CTAs
    std::vector<long long> h((size_t)grid * 8);
    cudaStreamSynchronize(stream);
    cudaMemcpy(h.data(), st->d_prof, h.size() * sizeof(long long), cudaMemcpyDeviceToHost);
    static const char* names[8] = {"mma.wait_full", "mma.issue", "mma.commit", "mma.wait_tempty", "mma.total", "stages",
                                   "load0.wait_empty", "load0.store_fence_arrive"};
    fprintf(stderr, "us_prof stages/ring=%d groups=%d parts=%d bufs=%d a_tmem=%d items=%u\n", a.stages, a.load_groups, a.parts, a.bufs, a.a_tmem, a.total_items);
    for (int sidx = 0; sidx < 8; ++sidx) {
      double sum = 0;
      for (int c = 0; c < grid; ++c) sum += (double)h[(size_t)c * 8 + sidx];
      fprintf(stderr, "us_prof %-26s %12.0f per CTA\n", names[sidx], sum / grid);
    }
  }
  }   // launches
  return SAGA_OK;
}

}  // namespace saga

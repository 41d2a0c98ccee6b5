// Composite-likelihood fit for large state spaces (S > 32; the 400 x 400 co-evolution model).
//
// One epoch evaluates, for all K time buckets at once,
//     P_k = expm(t_k Q),   loss = -sum_k <C_k, log P_k>,   dloss/dQ
// with a schedule built around two facts: every bucket exponentiates the SAME matrix, and Q is
// a rate matrix, so B = Q + mu I (mu = max |Q_ii|) is entrywise non-negative.
//
//   expm(t Q) = [ e^{-tau mu} T_m(tau B) ]^(2^s),   tau = t / 2^s,   ||tau B||_inf = tau mu <= theta
//
//   1. powers B^2..B^m are formed ONCE per epoch (log-depth schedule of batched GEMMs), so the
//      degree-m Taylor polynomial of every bucket is a weighted sum of shared matrices (one
//      elementwise pass for all buckets, no GEMM per bucket); all terms are non-negative, so
//      small transition probabilities keep full relative accuracy before the log;
//   2. only buckets with tau mu > theta need squarings: s_k batched 400^3 GEMMs per bucket,
//      run level by level over the buckets that are still active;
//   3. the backward pass is the exact adjoint of 1-2: per squaring two GEMMs fused into one
//      launch (concatenated K), the bucket adjoints are folded into m weighted sums, and the
//      adjoint of the power schedule yields dloss/dB = dloss/dQ.
// Every GEMM is a hand-written FP64 tensor-core kernel (DMMA m8n8k4, cp.async pipeline,
// 80x80 CTA tiles, split-K for the small-batch power levels).  All matrices are stored padded
// to a multiple of 80 with zero padding, so the GEMM has no edge handling.
//
// Replaces torch.matrix_exp + log + sum + autograd.backward + Adam of the reference's
// train_quantization (estimation/_ratelearn/trainer.py:156-187) for S = 400.
#include <algorithm>
#include <cstdlib>
#include <mutex>
#include <unordered_map>
#include <vector>

#include "dmma.cuh"
#include "fit_common.cuh"
#include "fit_internal.cuh"

namespace {

constexpr int kDeg = 24;          // Taylor degree of the shared-power polynomial (28 with theta = 3.0 halves the squarings
                                  // of the bench workload, 13 -> 7, but lengthens the two chains and the Taylor pass:
                                  // 0.875 ms per epoch graph-replayed against 0.80, gpurun_out/r02_fit_timeline_v17_deg28.txt)
constexpr double kTheta = 2.2;    // tau*mu bound: 2.2^25/25! ~ 2e-17 (all terms non-negative)
constexpr int kSStore = 8;        // squarings kept per bucket: covers t*mu up to 2.2 * 2^8 = 563
constexpr int BT = 80, BK = 16, NSTAGE = 2;  // two stages (51 KB per CTA): THREE CTAs share an SM; three stages with two CTAs
                                              // measured 0.851 ms per epoch against 0.820 (gpurun_out/r02_fit_stage2_sweep.txt)
constexpr int GEMM_THREADS = 128;  // 4 warps, one 40x40 quadrant of the tile each
constexpr int kCtasPerSm = 3;      // persistent grids of the tile kernels: 2-stage pipeline, 51 KB and ~20 K registers per CTA
// split-K cap of the squaring kernels (graph-replayed epochs, general form, 25 tiles per product: 1 -> 1.04 ms,
// 2 -> 0.94, 5 -> 0.96; symmetric form, 15 tiles: 2 -> 0.764, 3 -> 0.741, 4 -> 0.744, 6 -> 0.749)
constexpr int kSqKsplitGeneral = 2, kSqKsplitSym = 3;
constexpr int LD_ROW = 20;        // tile stored [80][16]: k contiguous
constexpr int LD_COL = 84;        // tile stored [16][80]: m (or n) contiguous
constexpr int TILE_ELEMS = BT * LD_ROW;  // 1600 >= 16 * 84
constexpr int EW_THREADS = 256;
constexpr int kTaylorStagesS = 16;     // count loads in flight per thread of its shared-memory variant (two CTAs per SM)
constexpr int kTaylorThreads = 256;    // threads per CTA of the shared-memory variant of the fused Taylor pass (288 would make
                                       // 160 000 elements two passes of 296 CTAs instead of 2.11, but needs <= 113 registers: 96 with
                                       // 300 bytes of spills measured 213 us against 180)
constexpr int kTaylorTailUnits = 512;   // (chunk, share) CTAs of the tail split: at most 2 CTAs per SM (296 on a B200)
constexpr int kTaylorInterleave = 2;  // buckets whose dependent chains a thread of the fused Taylor pass interleaves
constexpr int kTaylorStages = 16;  // count loads in flight per thread of the fused Taylor pass
static_assert(kDeg % 4 == 0, "the elementwise kernels skip Taylor terms in blocks of four");
// The tightest shared-memory budget that depends on K: taylor_fused_kernel (the large-K Taylor pass) stages the
// weight table, three int lists and the count-load ring in the 200 KB it is allowed (see fit_large_impl).  The
// other per-K tables (poly_eval_kernel 200 K bytes, accumulate_M_kernel 204 K) fit whenever this one does.
static_assert(CHERRY_LARGE_FIT_MAX_K ==
                  (200 * 1024 - 8 - (int)sizeof(double) * kTaylorStages * EW_THREADS) / ((int)sizeof(double) * (kDeg + 1) + 3 * (int)sizeof(int)),
              "CHERRY_LARGE_FIT_MAX_K must be the K budget of taylor_fused_kernel's shared memory");

struct GemmTerm {
  const double* A;
  const double* B;
  int ta, tb;
};
struct GemmTask {
  double* C;
  int term_begin, n_terms, accumulate;
};

__device__ __forceinline__ void cp_async16(double* smem_dst, const double* gmem_src) {
  const unsigned s = (unsigned)__cvta_generic_to_shared(smem_dst);
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(s), "l"(gmem_src));
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N)); }

// tile with the k index contiguous in global memory: 80 rows x 16 doubles -> [80][LD_ROW]
__device__ __forceinline__ void load_row_tile(double* s, const double* g, int ldg, int row0, int col0) {
  for (int c = threadIdx.x; c < BT * 8; c += GEMM_THREADS) {
    const int row = c >> 3, seg = c & 7;
    cp_async16(s + row * LD_ROW + seg * 2, g + (size_t)(row0 + row) * ldg + col0 + seg * 2);
  }
}
// tile with the m/n index contiguous in global memory: 16 rows x 80 doubles -> [16][LD_COL]
__device__ __forceinline__ void load_col_tile(double* s, const double* g, int ldg, int row0, int col0) {
  for (int c = threadIdx.x; c < BK * 40; c += GEMM_THREADS) {
    const int row = c / 40, seg = c - row * 40;
    cp_async16(s + row * LD_COL + seg * 2, g + (size_t)(row0 + row) * ldg + col0 + seg * 2);
  }
}

template <bool TA, bool TB>
__device__ __forceinline__ void compute_chunk(const double* As, const double* Bs, double (&acc)[5][5][2],
                                              int rbase, int cbase, int g, int tg) {
#pragma unroll
  for (int kk = 0; kk < BK; kk += 4) {
    double a[5], b[5];
#pragma unroll
    for (int i = 0; i < 5; ++i) {
      const int row = rbase + 8 * i + g;
      a[i] = TA ? As[(kk + tg) * LD_COL + row] : As[row * LD_ROW + kk + tg];
    }
#pragma unroll
    for (int j = 0; j < 5; ++j) {
      const int col = cbase + 8 * j + g;
      b[j] = TB ? Bs[col * LD_ROW + kk + tg] : Bs[(kk + tg) * LD_COL + col];
    }
#pragma unroll
    for (int i = 0; i < 5; ++i)
#pragma unroll
      for (int j = 0; j < 5; ++j) dmma884(acc[i][j][0], acc[i][j][1], a[i], b[j]);
  }
}

// Core of every GEMM here: one 80x80 output tile, accumulated over k chunks [c_begin, c_end) of
// the concatenated terms, 3-stage cp.async pipeline, result (+ old value) stored to `out`.
// `out` is addressed as out[(m0 + r) * ld_out + n0 + c]; callers that want a compact 80x80 partial
// tile pass ld_out = BT and a pointer shifted by -(m0 * BT + n0) (compact_tile_base below).
template <typename TermFn>
__device__ __forceinline__ void gemm_tile(TermFn get_term, int Sp, int m0, int n0, int c_begin, int c_end,
                                          double* smem, double* out, bool add_old, int ld_out = 0,
                                          double* mirror = nullptr) {
  // mirror != nullptr (symmetric results): the tile is also stored transposed, mirror[(n0 + c) * Sp + m0 + r];
  // the eight lanes that share a column hold eight consecutive rows, so the transposed stores fill 64-byte
  // segments just like the direct ones
  if (ld_out == 0) ld_out = Sp;
  const int cpt = Sp / BK;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, g = lane >> 2, tg = lane & 3;
  const int rbase = (warp >> 1) * 40, cbase = (warp & 1) * 40;  // 4 warps: 2x2 quadrants of 40x40
  double acc[5][5][2];
#pragma unroll
  for (int i = 0; i < 5; ++i)
#pragma unroll
    for (int j = 0; j < 5; ++j) acc[i][j][0] = acc[i][j][1] = 0.0;
  auto issue = [&](int c, int stage) {
    const GemmTerm t = get_term(c / cpt);
    const int k0 = (c % cpt) * BK;
    double* As = smem + (size_t)stage * 2 * TILE_ELEMS;
    double* Bs = As + TILE_ELEMS;
    if (t.ta) load_col_tile(As, t.A, Sp, k0, m0); else load_row_tile(As, t.A, Sp, m0, k0);
    if (t.tb) load_row_tile(Bs, t.B, Sp, n0, k0); else load_col_tile(Bs, t.B, Sp, k0, n0);
  };
  const int n_chunks = c_end - c_begin;
#pragma unroll
  for (int s = 0; s < NSTAGE - 1; ++s) {
    if (s < n_chunks) issue(c_begin + s, s);
    cp_async_commit();
  }
  for (int i = 0; i < n_chunks; ++i) {
    cp_async_wait<NSTAGE - 2>();
    __syncthreads();
    const int nxt = i + NSTAGE - 1;
    if (nxt < n_chunks) issue(c_begin + nxt, nxt % NSTAGE);
    cp_async_commit();
    const GemmTerm t = get_term((c_begin + i) / cpt);
    const double* As = smem + (size_t)(i % NSTAGE) * 2 * TILE_ELEMS;
    const double* Bs = As + TILE_ELEMS;
    if (t.ta) {
      if (t.tb) compute_chunk<true, true>(As, Bs, acc, rbase, cbase, g, tg);
      else compute_chunk<true, false>(As, Bs, acc, rbase, cbase, g, tg);
    } else {
      if (t.tb) compute_chunk<false, true>(As, Bs, acc, rbase, cbase, g, tg);
      else compute_chunk<false, false>(As, Bs, acc, rbase, cbase, g, tg);
    }
  }
  cp_async_wait<0>();
#pragma unroll
  for (int i = 0; i < 5; ++i)
#pragma unroll
    for (int j = 0; j < 5; ++j) {
      double2* p = reinterpret_cast<double2*>(out + (ptrdiff_t)(m0 + rbase + 8 * i + g) * ld_out + n0 + cbase + 8 * j + 2 * tg);
      double2 v = make_double2(acc[i][j][0], acc[i][j][1]);
      if (add_old) {
        const double2 o = *p;
        v.x += o.x;
        v.y += o.y;
      }
      *p = v;
      if (mirror != nullptr) {
        double* q = mirror + (ptrdiff_t)(n0 + cbase + 8 * j + 2 * tg) * Sp + m0 + rbase + 8 * i + g;
        q[0] = v.x;
        q[Sp] = v.y;
      }
    }
}

// C_task = sum over the task's terms of op(A) op(B)  (+ C_task if accumulate).  Square Sp x Sp
// matrices, Sp a multiple of 80.  grid = (tiles, n_tasks, ksplit); with ksplit > 1 the CTA
// writes its partial product to `partial[(task*ksplit + z)]` and splitk_reduce_kernel finishes.
__global__ void __launch_bounds__(GEMM_THREADS)
gemm_tasks_kernel(const GemmTask* __restrict__ tasks, const GemmTerm* __restrict__ terms, int Sp,
                  int ksplit, double* __restrict__ partial) {
  extern __shared__ double smem[];
  const GemmTask task = tasks[blockIdx.y];
  const int tiles_n = Sp / BT;
  const int m0 = (blockIdx.x / tiles_n) * BT, n0 = (blockIdx.x % tiles_n) * BT;
  const int total = task.n_terms * (Sp / BK);
  const int z = blockIdx.z;
  const int c_begin = (int)((long long)total * z / ksplit), c_end = (int)((long long)total * (z + 1) / ksplit);
  double* out = (ksplit == 1) ? task.C : partial + ((size_t)blockIdx.y * ksplit + z) * (size_t)Sp * Sp;
  gemm_tile([&](int idx) { return terms[task.term_begin + idx]; }, Sp, m0, n0, c_begin, c_end, smem, out,
            (ksplit == 1) && task.accumulate);
}

// ----------------------------------------------------------- dataflow squaring chains
// All squaring levels of all buckets in ONE persistent launch.  coef_kernel publishes, per
// level, the list of buckets that are still active; CTAs pull (level, bucket, tile) items from
// an atomic queue in level-major order and, instead of a grid-wide barrier per level, wait only
// for the 25 tiles of the SAME bucket at the previous level (per-bucket completion counters).
// Items are dequeued in dependency order and every dequeued item is being executed by a
// resident CTA, so the waits cannot deadlock.
struct SqSchedule {
  int queue[2];                        // work counters: forward, backward
  int n_levels;                        // max_k s_k
  int level_off[kSStore + 1];          // prefix sums of active buckets per level
  int ks[kSStore];                     // split-K factor of the tiles of a level (few active buckets: more CTAs per tile)
  int item_off[kSStore + 1];           // prefix sums of the work items (active buckets x tiles x ks) per level
  int ksmax;                           // stride of a bucket's partial matrices
  int pad[2];                          // pad[0]: dynamic chunk counter of the fused Taylor pass
  // followed in memory by: int active[kSStore][K]; int done_fwd[K][kSStore]; int done_bwd[K][kSStore + 1];
  // int rank[K] (position of bucket k in level 0's list); int tile_arrive[K][tiles]
};
__device__ __forceinline__ int* sq_active(SqSchedule* s) { return reinterpret_cast<int*>(s + 1); }
__device__ __forceinline__ int* sq_done_fwd(SqSchedule* s, int K) { return sq_active(s) + kSStore * K; }
__device__ __forceinline__ int* sq_done_bwd(SqSchedule* s, int K) { return sq_done_fwd(s, K) + kSStore * K; }
__device__ __forceinline__ int* sq_rank(SqSchedule* s, int K) { return sq_done_bwd(s, K) + (kSStore + 1) * K; }
__device__ __forceinline__ int* sq_tile_arrive(SqSchedule* s, int K) { return sq_rank(s, K) + K; }
constexpr int kSqPartialSlots = 96;  // matrices of the split-K partial buffer (Plan::off_partial) the squarings may use

// Bounded spin (about a second): a scheduling bug must surface as an error flag, not as a hung GPU.
__device__ __forceinline__ void wait_counter(const int* ctr, int target, int* status_flag) {
  if (threadIdx.x == 0) {
    unsigned spins = 0;
    while (*reinterpret_cast<const volatile int*>(ctr) < target) {
      __nanosleep(64);
      if (++spins > (1u << 24)) {
        atomicExch(status_flag, 3);
        break;
      }
    }
    __threadfence();
  }
  __syncthreads();
}

template <bool BWD>
__global__ void __launch_bounds__(GEMM_THREADS)
squaring_dataflow_kernel(SqSchedule* __restrict__ sched, const int* __restrict__ s_arr, int K, int Sp,
                         double* __restrict__ X0, double* __restrict__ chain, int slots_per_bucket,
                         double* __restrict__ partial, int* __restrict__ status_flag, int sym) {
  // sym != 0: every matrix here is symmetric (reversible Q in the basis diag(sqrt(pi)), symmetric counts): only the
  // tiles on and above the diagonal are work items, each stores its transpose as well.  coef_kernel built the
  // schedule with the same tile count.
  extern __shared__ double smem[];
  __shared__ int s_item, s_last;
  const int tiles_n = Sp / BT, tiles = sym ? tiles_n * (tiles_n + 1) / 2 : tiles_n * tiles_n;
  const size_t n_p = (size_t)Sp * Sp;
  const int n_levels = sched->n_levels;
  const int ksmax = sched->ksmax;
  const int total_items = sched->item_off[n_levels];
  const int* active = sq_active(sched);
  int* done_fwd = sq_done_fwd(sched, K);
  int* done_bwd = sq_done_bwd(sched, K);
  const int* rank = sq_rank(sched, K);
  int* tile_arrive = sq_tile_arrive(sched, K);
  // With few active buckets a tile is split over `ksplit` CTAs (a lone CTA runs one 80x80x400
  // tile at a third of the SM's DMMA rate).  Every CTA writes its partial tile; the one that
  // arrives last adds them in z order (so the result does not depend on who is last), writes
  // the tile and moves the bucket's completion counter.
  auto finish_tile = [&](int k, int tile, int m0, int n0, double* out, int ksplit, bool mirror) -> bool {
    if (ksplit == 1) return true;
    __threadfence();
    __syncthreads();
    int* ctr = tile_arrive + rank[k] * tiles + tile;
    if (threadIdx.x == 0) {
      const int old = atomicAdd(ctr, 1);
      s_last = (old == ksplit - 1);
      if (s_last) *ctr = 0;  // ready for the next level / launch
    }
    __syncthreads();
    if (!s_last) return false;
    __threadfence();
    const double* pb = partial + (size_t)rank[k] * ksmax * n_p;
    constexpr int NQ = BT * BT / 2 / GEMM_THREADS;
    double2 v[NQ];
#pragma unroll
    for (int q = 0; q < NQ; ++q) v[q] = make_double2(0.0, 0.0);
    for (int zz = 0; zz < ksplit; ++zz) {
      double2 t[NQ];
#pragma unroll
      for (int q = 0; q < NQ; ++q) {
        const int e = threadIdx.x + q * GEMM_THREADS;
        const int r = e / (BT / 2), c2 = (e - r * (BT / 2)) * 2;
        t[q] = __ldcg(reinterpret_cast<const double2*>(pb + (size_t)zz * n_p + (size_t)(m0 + r) * Sp + n0 + c2));
      }
#pragma unroll
      for (int q = 0; q < NQ; ++q) {
        v[q].x += t[q].x;
        v[q].y += t[q].y;
      }
    }
#pragma unroll
    for (int q = 0; q < NQ; ++q) {
      const int e = threadIdx.x + q * GEMM_THREADS;
      const int r = e / (BT / 2), c2 = (e - r * (BT / 2)) * 2;
      *reinterpret_cast<double2*>(out + (size_t)(m0 + r) * Sp + n0 + c2) = v[q];
      if (mirror) {
        double* m = out + (size_t)(n0 + c2) * Sp + m0 + r;
        m[0] = v[q].x;
        m[Sp] = v[q].y;
      }
    }
    return true;
  };
  for (;;) {
    __syncthreads();
    if (threadIdx.x == 0) s_item = atomicAdd(&sched->queue[BWD ? 1 : 0], 1);
    __syncthreads();
    const int item = s_item;
    if (item >= total_items) return;
    // forward walks the levels upwards, backward downwards (the same decoding on the mirrored index)
    const int pos = BWD ? (total_items - 1 - item) : item;
    int level = 0;
    while (level + 1 < n_levels && sched->item_off[level + 1] <= pos) ++level;
    const int ksplit = sched->ks[level];
    const int local = pos - sched->item_off[level];
    const int z = local % ksplit, item_t = local / ksplit;
    const int bidx = item_t / tiles, tile = item_t - bidx * tiles;
    const int k = active[level * K + bidx];
    int ti = tile / tiles_n, tj = tile % tiles_n;
    if (sym) {  // tile = index into the upper triangle, row by row
      ti = 0;
      int rest = tile;
      while (rest >= tiles_n - ti) {
        rest -= tiles_n - ti;
        ++ti;
      }
      tj = ti + rest;
    }
    const int m0 = ti * BT, n0 = tj * BT;
    const bool mirror = sym && ti != tj;
    double* Xi = (level == 0) ? X0 + (size_t)k * n_p : chain + ((size_t)k * slots_per_bucket + (level - 1)) * n_p;
    double* out = chain + ((size_t)k * slots_per_bucket + level) * n_p;  // slot level+1
    if (!BWD) {
      if (level > 0) wait_counter(done_fwd + k * kSStore + (level - 1), tiles, status_flag);
      const GemmTerm t0{Xi, Xi, 0, 0};
      const int total = Sp / BK;
      double* dst = ksplit == 1 ? out : partial + ((size_t)rank[k] * ksmax + z) * n_p;
      gemm_tile([&](int) { return t0; }, Sp, m0, n0, total * z / ksplit, total * (z + 1) / ksplit, smem, dst, false, 0,
                (mirror && ksplit == 1) ? out : nullptr);
      if (!finish_tile(k, tile, m0, n0, out, ksplit, mirror)) continue;
      __threadfence();  // every thread publishes its part of the tile before the counter moves
      __syncthreads();
      if (threadIdx.x == 0) atomicAdd(done_fwd + k * kSStore + level, 1);
    } else {
      // Xbar_{level+1} lives in slot level+2; it is either G (written by loss_grad_kernel before
      // this launch) or the output of this kernel at level+1 of the same bucket.
      double* Xb = chain + ((size_t)k * slots_per_bucket + (level + 1)) * n_p;
      // done_bwd[k][l] counts finished tiles of backward level l of bucket k
      if (level + 1 < s_arr[k]) wait_counter(done_bwd + k * (kSStore + 1) + (level + 1), tiles, status_flag);
      const GemmTerm t0{Xb, Xi, 0, 1}, t1{Xi, Xb, 1, 0};
      const int total = 2 * (Sp / BK);
      double* dst = ksplit == 1 ? out : partial + ((size_t)rank[k] * ksmax + z) * n_p;
      gemm_tile([&](int idx) { return idx == 0 ? t0 : t1; }, Sp, m0, n0, total * z / ksplit,
                total * (z + 1) / ksplit, smem, dst, false, 0, (mirror && ksplit == 1) ? out : nullptr);
      if (!finish_tile(k, tile, m0, n0, out, ksplit, mirror)) continue;
      __threadfence();
      __syncthreads();
      if (threadIdx.x == 0) atomicAdd(done_bwd + k * (kSStore + 1) + level, 1);
    }
  }
}

// ----------------------------------------------------------- dataflow power chains
// The forward power schedule (B^2..B^m) and its adjoint are dependent chains of 400^3 products with
// 25..200 output tiles per level: launched level by level (round 1) every level paid a launch, a
// pipeline fill on 2-chunk K slices and a separate split-K reduce launch (measured: 10 us fixed +
// 58 % of the DMMA rate).  Here ONE persistent launch runs a whole chain: the host lists, in
// dependency order, work items = (output tile, K slice of 80) and groups = output-tile updates;
// CTAs pull items from an atomic queue, wait only for the operand TILES the slice reads (per-tile
// version counters, so a level starts while the previous one drains), write a compact partial tile,
// and the CTA that arrives last at a group adds the partial tiles in slice order (deterministic),
// applies the update to C and publishes the tile's new version.  Items are dequeued in dependency
// order and every dequeued item is held by a running CTA, so the waits cannot deadlock.
struct DfGroup {
  double* C;
  int m0, n0;
  int n_slices, accumulate;
  int c_mat, need_ver;  // the update applies to version need_ver of the C tile and publishes need_ver + 1
  int partial_off, n_slabs;
  int mirror, pad;      // mirror: C is symmetric and only this (upper) tile is computed -- the reduction also writes
                        // the transposed tile and publishes ITS versions (word s = column strip s of the mirrored tile)
};
struct alignas(16) DfItem {  // everything a CTA needs comes with ONE dependent load after the queue ticket
  const double* A;
  const double* B;
  int ta, tb;
  int k0, n_chunks;   // K range [k0, k0 + BK * n_chunks)
  int group, slice;   // kind 0: K slice of the group's product; kind 1: row slab of the group's reduction
  int a_mat, a_ver;   // wait until every tile of A this slice reads has version >= a_ver (a_mat < 0: no wait)
  int b_mat, b_ver;
  int kind, pad;
  DfGroup g;          // copy of the item's group
};
static_assert(sizeof(DfItem) % 16 == 0, "DfItem layout");
struct DfList {  // host-side description of one chain launch
  std::vector<DfItem> items;
  std::vector<DfGroup> groups;
  std::vector<int> pending;  // groups whose reduction items have not been emitted yet
  int n_mats = 0;
  size_t off_items = 0, off_state = 0;  // workspace offsets (every item carries a copy of its group)
  int partial_tiles = 0;
};
constexpr int kDfSlabs = 5;      // row slabs of a tile's reduction (16 rows each), one work item per slab
// device state of a list: int queue; int pad[3]; int ver[n_mats * tiles * kDfSlabs]; int arrive[n_groups]
// (a version per ROW SLAB of a tile: a slab's reduction publishes with a plain store, no ticket counter)
__host__ __device__ inline size_t df_state_ints(int n_mats, int tiles, int n_groups) {
  return 4 + (size_t)n_mats * tiles * kDfSlabs + (size_t)n_groups;
}
constexpr int kDfReduceLag = 1 << 20;  // groups between a product and its reduction items in the queue: effectively "all
                                        // of a level's products first, then its reductions" -- sweeps of 10..1000 groups
                                        // (profiles/timelines/r02_fit_reduce_lag_sweep.txt, r02_fit_chain_sweep2/3.txt): a
                                        // reduction taken before its products are done idles a CTA that could have run a product
constexpr int kDfChainTarget = 500;  // work items per level of a power chain (sweeps 300..4000:
                                     // profiles/timelines/r02_fit_chain_target_sweep.txt, r02_fit_chain_sweep3.txt)

__device__ __forceinline__ void df_wait_tile(const int* v, int target, int* status_flag) {
  unsigned spins = 0;
  while (*reinterpret_cast<const volatile int*>(v) < target) {
    __nanosleep(32);
    if (++spins > (1u << 23)) {  // a fraction of a second: a scheduling bug must not hang the GPU
      atomicExch(status_flag, 3);
      break;
    }
  }
}

__global__ void __launch_bounds__(GEMM_THREADS)
chain_dataflow_kernel(const DfItem* __restrict__ items, int n_items, int n_groups,
                      int* __restrict__ state, int n_mats, int Sp, double* __restrict__ partial,
                      int* __restrict__ status_flag, long long* __restrict__ prof) {
  extern __shared__ double smem[];
  __shared__ int s_item;
  const int tiles_n = Sp / BT, tiles = tiles_n * tiles_n;
  int* queue = state;
  int* ver = state + 4;
  int* arrive = ver + n_mats * tiles * kDfSlabs;
  // optional phase profile (CHERRY_FIT_TIMELINE): ns per CTA in {dequeue, operand wait, product,
  // arrive, reduce wait, reduce, publish}, items taken
  long long t_prev = 0;
  auto tick = [&](int phase) {
    if (prof != nullptr && threadIdx.x == 0) {
      long long now;
      asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(now));
      if (phase >= 0) prof[blockIdx.x * 8 + phase] += now - t_prev;
      t_prev = now;
    }
  };
  tick(-1);
  int next = -1;  // thread 0: ticket taken early (its latency hides behind the fence that ends an item)
  for (;;) {
    __syncthreads();
    if (threadIdx.x == 0) {
      s_item = next >= 0 ? next : atomicAdd(queue, 1);
      next = -1;
    }
    __syncthreads();
    const int idx = s_item;
    if (idx >= n_items) return;
    const DfItem it = items[idx];
    const DfGroup& g = it.g;
    const int ti = g.m0 / BT, tj = g.n0 / BT;
    if (prof != nullptr && threadIdx.x == 0) prof[blockIdx.x * 8 + 7] += 1;
    tick(0);
    if (it.kind == 0) {
      // ---- one K slice of the group's product
      if (threadIdx.x < 2 * kDfSlabs) {  // threads 0-4 wait for the slabs of A's tiles, 5-9 for B's
        const bool isA = threadIdx.x < kDfSlabs;
        const int slab = threadIdx.x - (isA ? 0 : kDfSlabs);
        const int mat = isA ? it.a_mat : it.b_mat;
        if (mat >= 0) {
          const int target = isA ? it.a_ver : it.b_ver;
          const int kz0 = it.k0 / BT, kz1 = (it.k0 + it.n_chunks * BK - 1) / BT;
          for (int kz = kz0; kz <= kz1; ++kz) {
            int tile;
            if (isA) tile = it.ta ? kz * tiles_n + ti : ti * tiles_n + kz;
            else tile = it.tb ? tj * tiles_n + kz : kz * tiles_n + tj;
            df_wait_tile(ver + (mat * tiles + tile) * kDfSlabs + slab, target, status_flag);
          }
          __threadfence();
        }
      }
      __syncthreads();
      tick(1);
      const GemmTerm t0{it.A, it.B, it.ta, it.tb};
      const bool direct = (g.n_slices == 1) && !g.accumulate;
      const int c0 = it.k0 / BK;
      if (direct) {
        gemm_tile([&](int) { return t0; }, Sp, g.m0, g.n0, c0, c0 + it.n_chunks, smem, g.C, false, 0,
                  g.mirror ? g.C : nullptr);
        tick(2);
        if (threadIdx.x == 0) next = atomicAdd(queue, 1);
        if (g.c_mat >= 0) {
          __threadfence();  // every thread publishes its part of the tile before the version moves
          __syncthreads();
          if (threadIdx.x < kDfSlabs)
            *reinterpret_cast<volatile int*>(ver + (g.c_mat * tiles + ti * tiles_n + tj) * kDfSlabs + threadIdx.x) = g.need_ver + 1;
          else if (g.mirror && threadIdx.x >= 32 && threadIdx.x < 32 + kDfSlabs)
            *reinterpret_cast<volatile int*>(ver + (g.c_mat * tiles + tj * tiles_n + ti) * kDfSlabs + (threadIdx.x - 32)) = g.need_ver + 1;
          tick(6);
        }
      } else {
        double* ptile = partial + (size_t)(g.partial_off + it.slice) * (BT * BT);
        gemm_tile([&](int) { return t0; }, Sp, g.m0, g.n0, c0, c0 + it.n_chunks, smem,
                  ptile - ((ptrdiff_t)g.m0 * BT + g.n0), false, BT);
        tick(2);
        if (threadIdx.x == 0) next = atomicAdd(queue, 1);
        __threadfence();
        __syncthreads();
        if (threadIdx.x == 0) atomicAdd(arrive + it.group, 1);  // no return value needed: a reduction
        tick(3);
      }
      continue;
    }
    // ---- one row slab of the group's reduction: C = (accumulate ? C : 0) + sum of the partial tiles, slices
    // in order (deterministic).  The items of a reduction sit in the queue behind the group's products, so
    // the wait below cannot deadlock; every slab publishes its own version of the tile.
    int* my_ver = ver + (g.c_mat * tiles + ti * tiles_n + tj) * kDfSlabs + it.slice;
    if (threadIdx.x == 0) {
      df_wait_tile(arrive + it.group, g.n_slices, status_flag);
      if (g.accumulate && g.need_ver > 0) df_wait_tile(my_ver, g.need_ver, status_flag);
      __threadfence();
    }
    __syncthreads();
    tick(4);
    {
      const int r_begin = BT * it.slice / g.n_slabs, r_end = BT * (it.slice + 1) / g.n_slabs;
      const int n_el = (r_end - r_begin) * (BT / 2);  // double2 elements of the slab
      const double* pb = partial + (size_t)g.partial_off * (BT * BT);
      constexpr int NQ = 5;  // 16 rows x 40 double2 over 128 threads
      for (int e0 = threadIdx.x; e0 < n_el; e0 += NQ * GEMM_THREADS) {
        double2 v[NQ];
        int off[NQ];
        bool on[NQ];
#pragma unroll
        for (int q = 0; q < NQ; ++q) {
          const int e = e0 + q * GEMM_THREADS;
          on[q] = e < n_el;
          const int r = r_begin + (on[q] ? e / (BT / 2) : 0), c2 = (on[q] ? e % (BT / 2) : 0) * 2;
          off[q] = r * BT + c2;
          v[q] = (g.accumulate && on[q])
                     ? __ldcg(reinterpret_cast<const double2*>(g.C + (size_t)(g.m0 + r) * Sp + g.n0 + c2))
                     : make_double2(0.0, 0.0);
        }
        for (int z = 0; z < g.n_slices; ++z) {
          const double* pz = pb + (size_t)z * (BT * BT);
          double2 t[NQ];
#pragma unroll
          for (int q = 0; q < NQ; ++q)
            t[q] = on[q] ? __ldcg(reinterpret_cast<const double2*>(pz + off[q])) : make_double2(0.0, 0.0);
#pragma unroll
          for (int q = 0; q < NQ; ++q) {
            v[q].x += t[q].x;
            v[q].y += t[q].y;
          }
        }
#pragma unroll
        for (int q = 0; q < NQ; ++q)
          if (on[q]) {
            const int r = off[q] / BT, c2 = off[q] - r * BT;
            *reinterpret_cast<double2*>(g.C + (size_t)(g.m0 + r) * Sp + g.n0 + c2) = v[q];
            if (g.mirror) {  // 16 rows x 80 columns -> 80 rows x 16 columns of the transposed tile
              double* m = g.C + (size_t)(g.n0 + c2) * Sp + g.m0 + r;
              m[0] = v[q].x;
              m[Sp] = v[q].y;
            }
          }
      }
    }
    tick(5);
    if (threadIdx.x == 0) next = atomicAdd(queue, 1);
    __threadfence();  // every thread publishes its part of the slab before the version moves
    __syncthreads();
    if (threadIdx.x == 0 && g.c_mat >= 0) {
      *reinterpret_cast<volatile int*>(my_ver) = g.need_ver + 1;
      if (g.mirror)
        *reinterpret_cast<volatile int*>(ver + (g.c_mat * tiles + tj * tiles_n + ti) * kDfSlabs + it.slice) = g.need_ver + 1;
    }
    tick(6);
  }
}

// grid = (blocks over elements, n_tasks), ksplit > 1: C = (accumulate ? C : 0) + sum_z partial[task][z], z ascending
__global__ void splitk_reduce_kernel(const GemmTask* __restrict__ tasks, int ksplit, size_t n_p,
                                     const double* __restrict__ partial) {
  const GemmTask task = tasks[blockIdx.y];
  const double* base = partial + (size_t)blockIdx.y * ksplit * n_p;
  for (size_t e = blockIdx.x * (size_t)blockDim.x + threadIdx.x; e < n_p; e += (size_t)gridDim.x * blockDim.x) {
    double v = task.accumulate ? task.C[e] : 0.0;
    for (int z = 0; z < ksplit; ++z) v += base[(size_t)z * n_p + e];
    task.C[e] = v;
  }
}

// ---------------------------------------------------------------- per-epoch small kernels
struct LargeScalars {   // lives in the workspace
  unsigned long long norm_bits;  // max row abs sum of B (bit pattern of a non-negative double)
  double mu;
  double pad[6];
};

// grid = Sp rows / 4; B = pad(Q) + mu I, row abs sums -> atomicMax (order independent)
__global__ void build_B_kernel(const double* __restrict__ Q, int S, int Sp, double* __restrict__ B,
                               LargeScalars* __restrict__ sc) {
  __shared__ double red[EW_THREADS / 32];
  double mx = 0.0;
  for (int i = threadIdx.x; i < S; i += blockDim.x) mx = fmax(mx, fabs(Q[(size_t)i * S + i]));
  for (int o = 16; o > 0; o >>= 1) mx = fmax(mx, __shfl_xor_sync(0xffffffffu, mx, o));
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = mx;
  __syncthreads();
  double mu = red[0];
  for (int w = 1; w < EW_THREADS / 32; ++w) mu = fmax(mu, red[w]);
  if (blockIdx.x == 0 && threadIdx.x == 0) sc->mu = mu;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int row = blockIdx.x * (EW_THREADS / 32) + warp; row < Sp; row += gridDim.x * (EW_THREADS / 32)) {
    double rs = 0.0;
    for (int j = lane; j < Sp; j += 32) {
      double v = 0.0;
      if (row < S && j < S) v = Q[(size_t)row * S + j] + (row == j ? mu : 0.0);
      B[(size_t)row * Sp + j] = v;
      rs += fabs(v);
    }
    for (int o = 16; o > 0; o >>= 1) rs += __shfl_xor_sync(0xffffffffu, rs, o);
    if (lane == 0) atomicMax(&sc->norm_bits, (unsigned long long)__double_as_longlong(rs));
  }
}

// one CTA: per bucket s_k, tau_k and the weights w[k][j] = e^{-tau mu} tau^j / j!, j = 0..m
// Per-bucket Taylor degree d_k <= m: the smallest degree whose truncation tail x^(d+1)/(d+1)!
// (x = tau mu <= theta, all terms non-negative) stays below 2e-17 of the SECOND-order term x^2/2,
// so that entries first reached by two substitutions keep full relative accuracy before the
// log.  Squared buckets keep the full degree.  Weights beyond d_k are zero; the elementwise
// kernels skip them in blocks of four.
__global__ void coef_kernel(const double* __restrict__ t, int K, LargeScalars* __restrict__ sc,
                            int* __restrict__ s_arr, int* __restrict__ deg_arr, double* __restrict__ w,
                            double* __restrict__ tau_arr,
                            int* __restrict__ status_flag, SqSchedule* __restrict__ sched, int tiles,
                            int n_ctas, int* __restrict__ df_state_fwd, int n_fwd_ints,
                            int* __restrict__ df_state_bwd, int n_bwd_ints, int sq_ksplit_max) {
  // the power chains' queues, tile versions and arrival counters start every epoch at zero
  for (int i = threadIdx.x; i < n_fwd_ints; i += blockDim.x) df_state_fwd[i] = 0;
  for (int i = threadIdx.x; i < n_bwd_ints; i += blockDim.x) df_state_bwd[i] = 0;
  const double norm = __longlong_as_double((long long)sc->norm_bits);
  const double mu = sc->mu;
  for (int k = threadIdx.x; k < K; k += blockDim.x) {
    const double a = fabs(t[k]) * norm;
    int s = 0;
    if (a > kTheta && a < 1e300) s = (int)ceil(log2(a / kTheta));
    if (s > kSStore) {
      atomicExch(status_flag, 2);
      s = kSStore;
    }
    const double tau = ldexp(t[k], -s);
    s_arr[k] = s;
    tau_arr[k] = tau;
    int d = kDeg;
    if (s == 0) {
      const double x = fabs(tau) * norm;
      double term = 2.0 / 6.0;  // d = 2: x^(d-1) * 2 / (d+1)!
      term *= x;
      for (d = 2; d < kDeg; ++d) {
        if (term <= 2e-17) break;
        term *= x / (double)(d + 2);
      }
    }
    deg_arr[k] = d;
    const double e = exp(-tau * mu);
    double c = e;
    for (int j = 0; j <= kDeg; ++j) {
      w[(size_t)k * (kDeg + 1) + j] = j <= d ? c : 0.0;
      c *= tau / (double)(j + 1);
    }
  }
  __syncthreads();
  if (threadIdx.x == 0) sc->norm_bits = 0ull;  // ready for the next epoch's atomicMax
  // ---- schedule of the dataflow squaring kernels: active buckets per level, counters reset
  int* active = sq_active(sched);
  int* done_fwd = sq_done_fwd(sched, K);
  int* done_bwd = sq_done_bwd(sched, K);
  for (int i = threadIdx.x; i < K * kSStore; i += blockDim.x) done_fwd[i] = 0;
  for (int i = threadIdx.x; i < K * (kSStore + 1); i += blockDim.x) done_bwd[i] = 0;
  int* rank = sq_rank(sched, K);
  int* tile_arrive = sq_tile_arrive(sched, K);
  for (int i = threadIdx.x; i < K * tiles; i += blockDim.x) tile_arrive[i] = 0;
  // s_arr was written by this CTA before the barrier above, so it is read back from global memory: K is not
  // bounded by a shared-memory array here
  __shared__ int level_n[kSStore];
  if (threadIdx.x == kSStore) {  // bucket lists of the fused Taylor pass: without / with squarings, ascending
    int* zl = deg_arr + K;
    int* ql = zl + K;
    int nz = 0, nq = 0;
    for (int k = 0; k < K; ++k) {
      if (s_arr[k] == 0) zl[nz++] = k; else ql[nq++] = k;
    }
    ql[K] = nz;
    ql[K + 1] = nq;
  }
  if (threadIdx.x < kSStore) {  // one thread per level builds that level's list
    const int lvl = threadIdx.x;
    int n = 0;
    for (int k = 0; k < K; ++k)
      if (s_arr[k] > lvl) {
        if (lvl == 0) rank[k] = n;
        active[lvl * K + n++] = k;
      }
    level_n[lvl] = n;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    int off = 0, n_levels = 0;
    for (int lvl = 0; lvl < kSStore; ++lvl) {
      sched->level_off[lvl] = off;
      if (level_n[lvl] > 0) n_levels = lvl + 1;
      off += level_n[lvl];
    }
    sched->level_off[kSStore] = off;
    // level_off beyond n_levels all equal `off`; the kernels read level_off[n_levels]
    sched->n_levels = n_levels;
    sched->queue[0] = 0;
    sched->queue[1] = 0;
    sched->pad[0] = 0;  // chunk counter of the fused Taylor pass
    // split K level by level: about 2.5 waves of work items per level (one K=400 tile is 60-100 us on a
    // CTA: with 1.1 waves of them the second wave runs nearly empty), at most sq_ksplit_max ways and within
    // the partial buffer (one slot per (bucket of level 0, z))
    int cap = sq_ksplit_max;
    if (level_n[0] > 0 && cap * level_n[0] > kSqPartialSlots) cap = kSqPartialSlots / level_n[0];
    if (cap < 1) cap = 1;
    int items = 0, ksmax = 1;
    for (int lvl = 0; lvl < kSStore; ++lvl) {
      int ks = 1;
      if (level_n[lvl] > 0) {
        ks = (5 * n_ctas / 2 + level_n[lvl] * tiles - 1) / (level_n[lvl] * tiles);
        if (ks > cap) ks = cap;
        if (ks < 1) ks = 1;
      }
      sched->ks[lvl] = ks;
      sched->item_off[lvl] = items;
      items += level_n[lvl] * tiles * ks;
      if (level_n[lvl] > 0 && ks > ksmax) ksmax = ks;
    }
    sched->item_off[kSStore] = items;
    sched->ksmax = ksmax;
  }
}

// X0_k = sum_j w[k][j] B^j for every bucket; one thread per matrix element keeps the m power
// values in registers and streams over the buckets.  powers[j-1] = B^j, j = 1..m.
__global__ void __launch_bounds__(EW_THREADS)
poly_eval_kernel(const double* __restrict__ powers, size_t n_p, int S, int Sp, int K,
                 const double* __restrict__ w, double* __restrict__ X0) {
  extern __shared__ double sw[];  // [K][m+1]
  for (int i = threadIdx.x; i < K * (kDeg + 1); i += blockDim.x) sw[i] = w[i];
  __syncthreads();
  const size_t e = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
  if (e >= n_p) return;
  const int row = (int)(e / Sp), col = (int)(e - (size_t)row * Sp);
  double pw[kDeg];
#pragma unroll
  for (int j = 0; j < kDeg; ++j) pw[j] = powers[(size_t)j * n_p + e];
  const double diag = (row == col && row < S) ? 1.0 : 0.0;
  for (int k = 0; k < K; ++k) {
    const double* wk = sw + k * (kDeg + 1);
    double v = wk[0] * diag;
#pragma unroll
    for (int j = 0; j < kDeg; ++j) v = fma(wk[j + 1], pw[j], v);
    X0[(size_t)k * n_p + e] = v;
  }
}

// Several buckets at once: the polynomial, the logarithm and the quotient of one (element, bucket) are
// ONE dependent chain of ~60 FP64 operations, and the pass runs 8 warps per SM (178 registers), so a bucket at a
// time leaves the FP64 pipe idle for most of every operation's latency (issue slots 25 % busy, r02_taylor_fused_v1).
// kTaylorInterleave independent chains interleave (four of them spill: 255 registers).  The weights beyond a bucket's degree are zero, so the four share the
// largest degree of the group (buckets are visited in ascending time = ascending degree).
template <int D, int U>
__device__ __forceinline__ void taylor_term_n(const double* const (&w)[U], const double (&pw)[kDeg], double (&acc)[kDeg],
                                              const double (&c)[U], double diag, double& part) {
  double v[U], g[U];
#pragma unroll
  for (int u = 0; u < U; ++u) v[u] = w[u][0] * diag;
#pragma unroll
  for (int j = 0; j < D; ++j)
#pragma unroll
    for (int u = 0; u < U; ++u) v[u] = fma(w[u][j + 1], pw[j], v[u]);
#pragma unroll
  for (int u = 0; u < U; ++u) {
    // c == 0: nothing is added (and padding elements, where v == 0, must not inject 0 * inf)
    const double l = log(v[u]), q = -c[u] / v[u];
    g[u] = c[u] != 0.0 ? q : 0.0;
    part -= c[u] != 0.0 ? c[u] * l : 0.0;
  }
#pragma unroll
  for (int j = 0; j < D; ++j) {
    double x = acc[j];
#pragma unroll
    for (int u = 0; u < U; ++u) x = fma(w[u][j + 1], g[u], x);
    acc[j] = x;
  }
}

// The same with the element's power values read from shared memory (spw[j * EW_THREADS], this thread's column):
// frees 48 registers, so that two CTAs share an SM (the pass is latency bound at one).
template <int D, int U, int NT>
__device__ __forceinline__ void taylor_term_n_s(const double* const (&w)[U], const double* __restrict__ spw,
                                                double (&acc)[kDeg], const double (&c)[U], double diag, double& part) {
  double v[U], g[U];
#pragma unroll
  for (int u = 0; u < U; ++u) v[u] = w[u][0] * diag;
#pragma unroll
  for (int j = 0; j < D; ++j) {
    const double pj = spw[j * NT];
#pragma unroll
    for (int u = 0; u < U; ++u) v[u] = fma(w[u][j + 1], pj, v[u]);
  }
#pragma unroll
  for (int u = 0; u < U; ++u) {
    const double l = log(v[u]), q = -c[u] / v[u];
    g[u] = c[u] != 0.0 ? q : 0.0;
    part -= c[u] != 0.0 ? c[u] * l : 0.0;
  }
#pragma unroll
  for (int j = 0; j < D; ++j) {
    double x = acc[j];
#pragma unroll
    for (int u = 0; u < U; ++u) x = fma(w[u][j + 1], g[u], x);
    acc[j] = x;
  }
}

// Fused Taylor pass (training), one thread per matrix element with its m power values in registers (48 doubles
// of state = 186 registers = one 256-thread block per SM: the pass was latency bound at 12 % of the warp slots,
// profiles/r02_taylor_fused_v1.txt).  taylor_fused_smem_kernel is the same pass with the powers in shared memory;
// this variant runs where two CTAs' weight tables do not fit an SM (large K).
//   buckets WITHOUT squarings (most of them): P_k(e) is the polynomial itself, so the loss term
//     and the bucket's whole contribution to the power adjoints, Pbar_j(e) += w[k][j] * (-C/P),
//     are formed on the spot -- nothing is stored per bucket, and an element with C_k(e) == 0
//     costs only the load of C;
//   buckets WITH squarings: X0_k(e) is stored for the squaring chain.
// Outputs: Pbar_j (j = 1..m) initialised with the no-squaring buckets' contributions, X0 of
// the squared buckets, one loss partial per block.
__global__ void __launch_bounds__(EW_THREADS)
taylor_fused_kernel(const double* __restrict__ powers, size_t n_p, int S, int Sp, int K,
                    const double* __restrict__ w, const int* __restrict__ s_arr,
                    const int* __restrict__ deg_arr, const double* __restrict__ C, double* __restrict__ X0,
                    double* __restrict__ Pbar, double* __restrict__ loss_partial_fused) {
  constexpr int U = kTaylorInterleave;
  extern __shared__ double sw[];  // [K][m+1] weights, then int lists
  __shared__ double red[EW_THREADS / 32];
  __shared__ int n_zero, n_sq;
  int* zlist = reinterpret_cast<int*>(sw + (size_t)K * (kDeg + 1));  // buckets with s == 0
  int* qlist = zlist + K;                                              // buckets with s > 0
  int* sdeg = qlist + K;                                               // Taylor degree per bucket
  for (int i = threadIdx.x; i < K * (kDeg + 1); i += blockDim.x) sw[i] = w[i];
  for (int i = threadIdx.x; i < K; i += blockDim.x) {  // lists built once per epoch by coef_kernel
    sdeg[i] = deg_arr[i];
    zlist[i] = deg_arr[K + i];
    qlist[i] = deg_arr[2 * K + i];
  }
  if (threadIdx.x == 0) {
    n_zero = deg_arr[3 * K];
    n_sq = deg_arr[3 * K + 1];
  }
  __syncthreads();
  // persistent: the weight table and the lists are staged once per CTA, the CTA walks over chunks of elements
  const size_t n_chunks = (n_p + blockDim.x - 1) / blockDim.x;
  double part = 0.0;
  for (size_t chunk = blockIdx.x; chunk < n_chunks; chunk += gridDim.x) {
    const size_t e = chunk * (size_t)blockDim.x + threadIdx.x;
    const bool in_range = e < n_p;
    const size_t ee = in_range ? e : 0;
    const int row = (int)(ee / Sp), col = (int)(ee - (size_t)row * Sp);
    const bool real = in_range && row < S && col < S;
    const double diag = (row == col && row < S) ? 1.0 : 0.0;
    double pw[kDeg], acc[kDeg];
#pragma unroll
    for (int i = 0; i < kDeg; ++i) {
      pw[i] = in_range ? powers[(size_t)i * n_p + ee] : 0.0;
      acc[i] = 0.0;
    }
    const size_t cidx = (size_t)row * S + col;
    const size_t SS = (size_t)S * S;
    // ---- buckets without squarings.  The pass is bound by the latency of the count loads (one 8-byte load per
    // bucket and thread, 87 buckets): they go through a ring of kTaylorStages cp.async stages in shared memory, so
    // that every thread keeps kTaylorStages loads in flight without holding them in registers.
    double* ring = reinterpret_cast<double*>(sdeg + K + (K & 1));  // [kTaylorStages][EW_THREADS], 8-byte aligned
    auto issue = [&](int i) {
      if (real && i < n_zero) {
        const unsigned dst = (unsigned)__cvta_generic_to_shared(ring + (i % kTaylorStages) * EW_THREADS + threadIdx.x);
        asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(dst), "l"(C + (size_t)zlist[i] * SS + cidx));
      }
      cp_async_commit();
    };
#pragma unroll
    for (int i = 0; i < kTaylorStages; ++i) issue(i);
    for (int i = 0; i < n_zero; i += U) {
      cp_async_wait<kTaylorStages - U>();
      double c[U];
#pragma unroll
      for (int u = 0; u < U; ++u)
        c[u] = (real && i + u < n_zero) ? ring[((i + u) % kTaylorStages) * EW_THREADS + threadIdx.x] : 0.0;
#pragma unroll
      for (int u = 0; u < U; ++u) issue(i + u + kTaylorStages);  // the slots just read are this thread's own
      bool nz = false;
#pragma unroll
      for (int u = 0; u < U; ++u) nz |= c[u] != 0.0;
      if (!__any_sync(0xffffffffu, nz)) continue;
      const double* wu[U];
      int d = 0;
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const int k = zlist[min(i + u, n_zero - 1)];
        wu[u] = sw + k * (kDeg + 1);
        d = max(d, sdeg[k]);
      }
      if (d <= 8) taylor_term_n<8, U>(wu, pw, acc, c, diag, part);
      else if (d <= 12) taylor_term_n<12, U>(wu, pw, acc, c, diag, part);
      else if (d <= 16) taylor_term_n<16, U>(wu, pw, acc, c, diag, part);
      else if (d <= 20) taylor_term_n<20, U>(wu, pw, acc, c, diag, part);
      else taylor_term_n<24, U>(wu, pw, acc, c, diag, part);
    }
    cp_async_wait<0>();
    // ---- buckets with squarings: store X0
    for (int i = 0; i < n_sq; ++i) {
      const int k = qlist[i];
      const double* wk = sw + k * (kDeg + 1);
      double v = wk[0] * diag;
#pragma unroll
      for (int j = 0; j < kDeg; ++j) v = fma(wk[j + 1], pw[j], v);
      if (in_range) X0[(size_t)k * n_p + e] = v;
    }
    if (in_range) {
#pragma unroll
      for (int i = 0; i < kDeg; ++i) Pbar[(size_t)i * n_p + e] = acc[i];
    }
  }
  for (int o = 16; o > 0; o >>= 1) part += __shfl_xor_sync(0xffffffffu, part, o);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = part;
  __syncthreads();
  if (threadIdx.x == 0) {
    double tot = 0.0;
    for (int wdx = 0; wdx < EW_THREADS / 32; ++wdx) tot += red[wdx];
    loss_partial_fused[blockIdx.x] = tot;
  }
}

// Element visited by thread-slot v_idx of the fused Taylor pass.  General form: the padded matrix row by row.
// Symmetric form: the elements with row <= col only -- the upper triangle folded into Sp/2 rows of Sp+1 elements
// (row f followed by row Sp-1-f), consecutive slots on consecutive columns.
template <bool SYM>
__device__ __forceinline__ void taylor_visit(size_t v_idx, int Sp, int& row, int& col) {
  if (SYM) {
    const int f = (int)(v_idx / (Sp + 1)), q = (int)(v_idx - (size_t)f * (Sp + 1));
    if (q < Sp - f) {
      row = f;
      col = f + q;
    } else {
      row = Sp - 1 - f;
      col = row + (q - (Sp - f));
    }
  } else {
    row = (int)(v_idx / Sp);
    col = (int)(v_idx - (size_t)row * Sp);
  }
}

// SYM (symmetric form, build_B_sym_kernel): every matrix is symmetric, so the pass visits the elements with
// row <= col only, stores every result at (row, col) and (col, row), and counts an off-diagonal element's loss
// term twice.
// PARTS == 1: persistent walk over the chunks [chunk_begin, chunk_end) of NT elements.
// PARTS > 1 (the tail of the pass): a chunk is one dependent chain of ~100 FP64 operations per bucket and thread,
// 60-70 us for ~100 buckets whatever else runs on the SM, so the chunks beyond a multiple of the resident CTAs
// would cost a whole extra round (314 chunks on 296 CTAs: 150 us instead of 75).  They are run as
// chunks x PARTS CTAs instead: CTA (chunk, unit) takes the unsquared buckets unit, unit + PARTS, ... and the
// squared buckets likewise, and leaves its share of the power adjoints in tailbuf[unit][j][tail element];
// taylor_tail_reduce_kernel adds the shares in unit order.
template <int UI, int NT, bool SYM, int PARTS>
__global__ void __launch_bounds__(NT, 2)
taylor_fused_smem_kernel(const double* __restrict__ powers, size_t n_p, int S, int Sp, int K,
                    const double* __restrict__ w, const int* __restrict__ s_arr,
                    const int* __restrict__ deg_arr, const double* __restrict__ C, double* __restrict__ X0,
                    double* __restrict__ Pbar, double* __restrict__ loss_partial_fused, int* __restrict__ chunk_counter,
                    int chunk_begin, int chunk_end, double* __restrict__ tailbuf) {
  constexpr bool sym = SYM;
  constexpr int NP = kDeg;
  extern __shared__ double sw[];  // [K][m+1] weights, then int lists
  __shared__ double red[NT / 32];
  __shared__ int n_zero, n_sq;
  int* zlist = reinterpret_cast<int*>(sw + (size_t)K * (kDeg + 1));  // buckets with s == 0
  int* qlist = zlist + K;                                              // buckets with s > 0
  int* sdeg = qlist + K;                                               // Taylor degree per bucket
  for (int i = threadIdx.x; i < K * (kDeg + 1); i += blockDim.x) sw[i] = w[i];
  for (int i = threadIdx.x; i < K; i += blockDim.x) {  // lists built once per epoch by coef_kernel
    sdeg[i] = deg_arr[i];
    zlist[i] = deg_arr[K + i];
    qlist[i] = deg_arr[2 * K + i];
  }
  if (threadIdx.x == 0) {
    n_zero = deg_arr[3 * K];
    n_sq = deg_arr[3 * K + 1];
  }
  __syncthreads();
  // persistent: the weight table and the lists are staged once per CTA, the CTA walks over chunks of elements
  const size_t n_visit = sym ? (size_t)(Sp / 2) * (Sp + 1) : n_p;
  double part_total = 0.0;
  __shared__ int s_chunk;
  const int unit = PARTS == 1 ? 0 : (int)(blockIdx.x % PARTS);
  const int nz_unit = PARTS == 1 ? n_zero : (n_zero - unit + PARTS - 1) / PARTS;  // this CTA's unsquared buckets
  // PARTS == 1: the first chunk of a CTA is its block index, the others come from a counter (coef_kernel zeroes it
  // every epoch): the CTAs that finish first take what is left
  for (int chunk = chunk_begin + (PARTS == 1 ? (int)blockIdx.x : (int)(blockIdx.x / PARTS)); chunk < chunk_end;) {
    const size_t v_idx = (size_t)chunk * blockDim.x + threadIdx.x;
    const bool in_range = v_idx < n_visit;
    int row, col;
    taylor_visit<SYM>(in_range ? v_idx : 0, Sp, row, col);
    const size_t e = (size_t)row * Sp + col, ee = e;
    const bool mirror = sym && in_range && row != col;
    const size_t et = (size_t)col * Sp + row;
    double part = 0.0;  // this element's loss terms
    const bool real = in_range && row < S && col < S;
    const double diag = (row == col && row < S) ? 1.0 : 0.0;
    double* ring = reinterpret_cast<double*>(sdeg + K + (K & 1));  // [kTaylorStagesS][NT], 8-byte aligned
    double* spw_all = ring + kTaylorStagesS * NT;               // [kDeg][NT]
    double acc[NP];
    double* spw = spw_all + threadIdx.x;  // this thread's column of the staged power values [kDeg][NT]
#pragma unroll
    for (int i = 0; i < NP; ++i) {
      spw[i * NT] = in_range ? powers[(size_t)i * n_p + ee] : 0.0;  // own column: no barrier needed
      acc[i] = 0.0;
    }
    const size_t cidx = (size_t)row * S + col;
    const size_t SS = (size_t)S * S;
    // ---- buckets without squarings.  The pass is bound by the latency of the count loads (one 8-byte load per
    // bucket and thread, 87 buckets): they go through a ring of kTaylorStagesS cp.async stages in shared memory, so
    // that every thread keeps kTaylorStagesS loads in flight without holding them in registers.
    auto zbucket = [&](int i) { return zlist[PARTS == 1 ? i : unit + PARTS * i]; };
    auto issue = [&](int i) {
      if (real && i < nz_unit) {
        const unsigned dst = (unsigned)__cvta_generic_to_shared(ring + (i % kTaylorStagesS) * NT + threadIdx.x);
        asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(dst), "l"(C + (size_t)zbucket(i) * SS + cidx));
      }
      cp_async_commit();
    };
#pragma unroll
    for (int i = 0; i < kTaylorStagesS; ++i) issue(i);
    {
      constexpr int U = UI;
      for (int i = 0; i < nz_unit; i += U) {
        cp_async_wait<kTaylorStagesS - U>();
        double c[U];
#pragma unroll
        for (int u = 0; u < U; ++u)
          c[u] = (real && i + u < nz_unit) ? ring[((i + u) % kTaylorStagesS) * NT + threadIdx.x] : 0.0;
#pragma unroll
        for (int u = 0; u < U; ++u) issue(i + u + kTaylorStagesS);  // the slots just read are this thread's own
        bool nz = false;
#pragma unroll
        for (int u = 0; u < U; ++u) nz |= c[u] != 0.0;
        if (!__any_sync(0xffffffffu, nz)) continue;
        const double* wu[U];
        int d = 0;
#pragma unroll
        for (int u = 0; u < U; ++u) {
          const int k = zbucket(min(i + u, nz_unit - 1));
          wu[u] = sw + k * (kDeg + 1);
          d = max(d, sdeg[k]);
        }
        if (d <= 8) taylor_term_n_s<8, U, NT>(wu, spw, acc, c, diag, part);
        else if (d <= 12) taylor_term_n_s<12, U, NT>(wu, spw, acc, c, diag, part);
        else if (d <= 16) taylor_term_n_s<16, U, NT>(wu, spw, acc, c, diag, part);
        else if (d <= 20) taylor_term_n_s<20, U, NT>(wu, spw, acc, c, diag, part);
        else taylor_term_n_s<24, U, NT>(wu, spw, acc, c, diag, part);
      }
    }
    cp_async_wait<0>();
    // ---- buckets with squarings: store X0
    for (int i = unit; i < n_sq; i += PARTS) {
      const int k = qlist[i];
      const double* wk = sw + k * (kDeg + 1);
      double v = wk[0] * diag;
#pragma unroll
      for (int j = 0; j < NP; ++j) v = fma(wk[j + 1], spw[j * NT], v);
      if (in_range) {
        X0[(size_t)k * n_p + e] = v;
        if (mirror) X0[(size_t)k * n_p + et] = v;
      }
    }
    if (PARTS == 1) {
      if (in_range) {
#pragma unroll
        for (int i = 0; i < NP; ++i) Pbar[(size_t)i * n_p + e] = acc[i];
        if (mirror) {
#pragma unroll
          for (int i = 0; i < NP; ++i) Pbar[(size_t)i * n_p + et] = acc[i];
        }
      }
    } else if (in_range) {
      const size_t tail_elems = (size_t)(chunk_end - chunk_begin) * NT;
      const size_t te = (size_t)(chunk - chunk_begin) * NT + threadIdx.x;
#pragma unroll
      for (int i = 0; i < NP; ++i) tailbuf[((size_t)unit * NP + i) * tail_elems + te] = acc[i];
    }
    part_total += mirror ? 2.0 * part : part;
    if (PARTS > 1) break;
    __syncthreads();
    if (threadIdx.x == 0) s_chunk = chunk_begin + (int)gridDim.x + atomicAdd(chunk_counter, 1);
    __syncthreads();
    chunk = s_chunk;
  }
  double part = part_total;
  for (int o = 16; o > 0; o >>= 1) part += __shfl_xor_sync(0xffffffffu, part, o);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = part;
  __syncthreads();
  if (threadIdx.x == 0) {
    double tot = 0.0;
    for (int wdx = 0; wdx < NT / 32; ++wdx) tot += red[wdx];
    loss_partial_fused[blockIdx.x] = tot;
  }
}

// Pbar_j(e) = sum over the units (in order) of the tail CTAs' shares, for the elements of the tail chunks.
// One thread per (power j, tail element), all of its loads in flight at once (a first version walked j and the
// units in one thread: 384 dependent L2 latencies, 90 us for 18 chunks).
template <bool SYM>
__global__ void taylor_tail_reduce_kernel(const double* __restrict__ tailbuf, int parts, size_t tail_elems,
                                          size_t v_begin, size_t n_visit, size_t n_p, int Sp,
                                          double* __restrict__ Pbar) {
  const size_t idx = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
  if (idx >= tail_elems * kDeg) return;
  const int j = (int)(idx / tail_elems);
  const size_t te = idx - (size_t)j * tail_elems;
  if (v_begin + te >= n_visit) return;
  double x[16];
#pragma unroll
  for (int u = 0; u < 16; ++u) x[u] = u < parts ? tailbuf[((size_t)u * kDeg + j) * tail_elems + te] : 0.0;
  double v = 0.0;
#pragma unroll
  for (int u = 0; u < 16; ++u) v += x[u];  // unit order; the absent units add +0.0
  int row, col;
  taylor_visit<SYM>(v_begin + te, Sp, row, col);
  Pbar[(size_t)j * n_p + (size_t)row * Sp + col] = v;
  if (SYM && row != col) Pbar[(size_t)j * n_p + (size_t)col * Sp + row] = v;
}

// Loss and G_k = -C_k / P_k (into chain slot s_k + 1) for the squared buckets of the list coef_kernel built (the
// fused Taylor pass did the others); P_k = X0_k if s_k == 0 else chain slot s_k.  1-D grid: block = (chunk of
// 4 * EW_THREADS elements, list position mod kLossLanes); one loss partial per block (only the SUM over the buckets
// is used downstream: loss_reduce_kernel puts it into loss_part[0]).  A grid of (blocks, K) launched 7 900 CTAs of
// which 87 % returned at once: 36 us for 13 buckets of work.
constexpr int kLossLanes = 16;  // list positions processed side by side
__global__ void __launch_bounds__(EW_THREADS)
loss_grad_kernel(const double* __restrict__ C, int S, int Sp, size_t n_p, int K, const int* __restrict__ s_arr,
                 const int* __restrict__ deg_arr, const double* __restrict__ X0, double* __restrict__ chain,
                 int slots_per_bucket, double* __restrict__ loss_partial) {
  __shared__ double red[EW_THREADS / 32];
  const int n_list = deg_arr[3 * K + 1];
  const int n_chunks = (int)((n_p + 4 * EW_THREADS - 1) / (4 * EW_THREADS));
  const int chunk = blockIdx.x % n_chunks, lane0 = blockIdx.x / n_chunks;
  double part = 0.0;
  for (int i = lane0; i < n_list; i += kLossLanes) {
    const int k = deg_arr[2 * K + i];
    const int s = s_arr[k];
    const double* P = (s == 0) ? X0 + (size_t)k * n_p
                               : chain + ((size_t)k * slots_per_bucket + (s - 1)) * n_p;
    double* G = chain + ((size_t)k * slots_per_bucket + s) * n_p;  // slot s+1 (slots are 1-based)
    const double* Ck = C + (size_t)k * S * S;
    double c[4], pv[4];
    size_t e[4];
    bool in[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      e[u] = ((size_t)chunk * 4 + u) * EW_THREADS + threadIdx.x;
      in[u] = e[u] < n_p;
      const int row = in[u] ? (int)(e[u] / Sp) : 0, col = in[u] ? (int)(e[u] - (size_t)row * Sp) : 0;
      const bool real = in[u] && row < S && col < S;
      c[u] = real ? Ck[(size_t)row * S + col] : 0.0;
      pv[u] = in[u] ? P[e[u]] : 1.0;
    }
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      double gval = 0.0;
      if (c[u] != 0.0) {
        part -= c[u] * log(pv[u]);
        gval = -c[u] / pv[u];
      }
      if (in[u]) G[e[u]] = gval;
    }
  }
  for (int o = 16; o > 0; o >>= 1) part += __shfl_xor_sync(0xffffffffu, part, o);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = part;
  __syncthreads();
  if (threadIdx.x == 0) {
    double tot = 0.0;
    for (int wdx = 0; wdx < EW_THREADS / 32; ++wdx) tot += red[wdx];
    loss_partial[blockIdx.x] = tot;
  }
}

// One CTA.  loss_part[0] = sum of the loss partials of loss_grad_kernel (block order) + of the fused Taylor pass
// (block order), loss_part[1..K) = 0: only the sum over the buckets is defined for S > 32.  Fixed orders.
__global__ void loss_reduce_kernel(const double* __restrict__ loss_partial, int K, int nblocks,
                                   double* __restrict__ loss_part, const double* __restrict__ fused_partial,
                                   int n_fused) {
  __shared__ double sh[256];
  for (int k = threadIdx.x; k < K; k += blockDim.x) loss_part[k] = 0.0;
  double v = 0.0;
  for (int b = threadIdx.x; b < nblocks; b += blockDim.x) v += loss_partial[b];
  for (int b = threadIdx.x; b < n_fused; b += blockDim.x) v += fused_partial[b];
  sh[threadIdx.x] = v;
  __syncthreads();
  if (threadIdx.x == 0) {
    double tot = 0.0;
    for (int i = 0; i < (int)blockDim.x; ++i) tot += sh[i];
    loss_part[0] = tot;
  }
}

// Pbar_j += sum_k w[k][j] * X0bar_k (chain slot 1 of bucket k), j = 1..m, over the squared buckets in order (the
// list coef_kernel built; the fused Taylor pass wrote the others' share).  Persistent: a CTA stages the weights of
// those buckets once and walks over chunks of elements.
__global__ void __launch_bounds__(EW_THREADS)
accumulate_M_kernel(const double* __restrict__ chain, int slots_per_bucket, size_t n_p, int K,
                    const double* __restrict__ w, double* __restrict__ Pbar,
                    const int* __restrict__ deg_arr) {
  extern __shared__ double sw[];  // [n_list][m+1] weights, then the bucket list
  __shared__ int n_list_s;
  if (threadIdx.x == 0) n_list_s = deg_arr[3 * K + 1];
  __syncthreads();
  const int n_list = n_list_s;
  int* list = reinterpret_cast<int*>(sw + (size_t)K * (kDeg + 1));
  for (int i = threadIdx.x; i < n_list; i += blockDim.x) list[i] = deg_arr[2 * K + i];
  __syncthreads();
  for (int i = threadIdx.x; i < n_list * (kDeg + 1); i += blockDim.x)
    sw[i] = w[(size_t)list[i / (kDeg + 1)] * (kDeg + 1) + i % (kDeg + 1)];
  __syncthreads();
  const size_t n_chunks = (n_p + blockDim.x - 1) / blockDim.x;
  for (size_t chunk = blockIdx.x; chunk < n_chunks; chunk += gridDim.x) {
    const size_t e = chunk * blockDim.x + threadIdx.x;
    if (e >= n_p) continue;
    double acc[kDeg];
#pragma unroll
    for (int j = 0; j < kDeg; ++j) acc[j] = Pbar[(size_t)j * n_p + e];
    for (int i0 = 0; i0 < n_list; i0 += 4) {
      double x[4];
#pragma unroll
      for (int u = 0; u < 4; ++u)
        x[u] = i0 + u < n_list ? chain[((size_t)list[i0 + u] * slots_per_bucket) * n_p + e] : 0.0;
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        if (i0 + u >= n_list) break;
        const double* wk = sw + (i0 + u) * (kDeg + 1);
#pragma unroll
        for (int j = 0; j < kDeg; ++j) acc[j] = fma(wk[j + 1], x[u], acc[j]);
      }
    }
#pragma unroll
    for (int j = 0; j < kDeg; ++j) Pbar[(size_t)j * n_p + e] = acc[j];
  }
}

// grid = (blocks, K): P_out[k] (S x S, unpadded) = X0_k if s_k == 0 else chain slot s_k
__global__ void extract_P_kernel(const int* __restrict__ s_arr, const double* __restrict__ X0,
                                 const double* __restrict__ chain, int slots_per_bucket, size_t n_p, int S,
                                 int Sp, double* __restrict__ P_out) {
  const int k = blockIdx.y, s = s_arr[k];
  const double* P = (s == 0) ? X0 + (size_t)k * n_p : chain + ((size_t)k * slots_per_bucket + (s - 1)) * n_p;
  for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < S * S; e += gridDim.x * blockDim.x) {
    const int i = e / S, j = e - i * S;
    P_out[(size_t)k * S * S + e] = P[(size_t)i * Sp + j];
  }
}

__global__ void unpad_kernel(const double* __restrict__ src, int S, int Sp, double* __restrict__ dst) {
  for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < S * S; e += gridDim.x * blockDim.x) {
    const int i = e / S, j = e - i * S;
    dst[e] = src[(size_t)i * Sp + j];
  }
}

// ------------------------------------------------------------------ parameter update (large S)
struct LargeUpdateArgs {
  int S, K;
  const double* mask;
  double* theta;
  double* adam_m;
  double* adam_v;
  double* Q;
  double* Q_best;
  double* Q_last;
  double* best_loss;
  double* loss_trace;
  int loss_trace_epochs;
  double* snapshots;
  int n_snapshots;
  const double* G;          // dL/dQ unnormalised [S][S]
  const double* loss_part;  // [K]
  const double* sumC;
  int* epoch_counter;
  double* grad_theta;  // [S + S(S-1)/2]
  double* dpi;         // [S]
  double* pibuf;       // [S] softmax(pi logits) of the CURRENT theta, written by the rows kernel
  double* shat;        // [S][S] mask_ij softplus(u_ij): the symmetric form of Q (off-diagonal), written with Q
  double* sr;          // [S] sqrt(pi) of the Q just built
  double lr_pi, lr_upper, beta1, beta2, eps;
  int do_adam, loss_normalization, best_mode;
};

__device__ __forceinline__ double block_sum_256(double v, double* red) {
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  __syncthreads();
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
  __syncthreads();
  double t = 0.0;
  for (int w = 0; w < EW_THREADS / 32; ++w) t += red[w];
  return t;
}
__device__ __forceinline__ double block_max_256(double v, double* red) {
  for (int o = 16; o > 0; o >>= 1) v = fmax(v, __shfl_xor_sync(0xffffffffu, v, o));
  __syncthreads();
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
  __syncthreads();
  double t = red[0];
  for (int w = 1; w < EW_THREADS / 32; ++w) t = fmax(t, red[w]);
  return t;
}
// sqrt(softmax(theta[0..S))) into sr[] (shared)
__device__ __forceinline__ void softmax_sqrt(const double* theta, int S, double* sr, double* red) {
  double mx = -INFINITY;
  for (int i = threadIdx.x; i < S; i += blockDim.x) mx = fmax(mx, theta[i]);
  mx = block_max_256(mx, red);
  double se = 0.0;
  for (int i = threadIdx.x; i < S; i += blockDim.x) se += exp(theta[i] - mx);
  se = block_sum_256(se, red);
  for (int i = threadIdx.x; i < S; i += blockDim.x) sr[i] = sqrt(exp(theta[i] - mx) / se);
  __syncthreads();
}
__device__ __forceinline__ double upper_param(const double* theta, int S, int i, int j) {
  const int lo = i < j ? i : j, hi = i < j ? j : i;
  return theta[S + cherry::triu_index(lo, hi, S)];
}

// ---- the symmetric form of a reversible model (training path only; fit_large_impl says when) ----
// Q_ij = mask_ij softplus(u_ij) sqrt(pi_j / pi_i) is similar to the SYMMETRIC matrix
//   Sh = R Q R^-1,  R = diag(sqrt(pi)):  Sh_ij = mask_ij softplus(u_ij),  Sh_ii = Q_ii,
// so expm(t Q) = R^-1 expm(t Sh) R, every power of Bh = Sh + mu I is symmetric, and for SYMMETRIC counts
// sum_ij C_ij log P_ij = sum_ij C_ij log E_ij with E = expm(t Sh) (the factors sqrt(pi_j / pi_i) cancel in
// pairs).  The whole evaluation then runs on symmetric matrices -- the forward chain and the squarings compute
// the upper tiles only -- and the result A = dL/dSh (symmetric) maps back as dL/dQ_ij = A_ij sqrt(pi_i / pi_j),
// which is the exact derivative with respect to an arbitrary perturbation of Q (R is a constant of the
// identity above).  Entry by entry (Bh^k)_ij = (B^k)_ij sqrt(pi_i / pi_j): the truncation analysis of the
// Taylor series (relative, entrywise, non-negative terms) carries over unchanged, so the scaling decisions
// keep using the row sums of B = Q + mu I.
// large_build_Q_kernel leaves Sh (off-diagonal) and sqrt(pi) next to every Q it builds, so this is build_B_kernel
// with one more operand.  grid = Sp rows / 8.
__global__ void build_B_sym_kernel(const double* __restrict__ Q, const double* __restrict__ shat, int S, int Sp,
                                   double* __restrict__ B, LargeScalars* __restrict__ sc) {
  __shared__ double red[EW_THREADS / 32];
  double mx = 0.0;
  for (int i = threadIdx.x; i < S; i += blockDim.x) mx = fmax(mx, fabs(Q[(size_t)i * S + i]));
  const double mu = block_max_256(mx, red);
  if (blockIdx.x == 0 && threadIdx.x == 0) sc->mu = mu;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int row = blockIdx.x * (EW_THREADS / 32) + warp; row < Sp; row += gridDim.x * (EW_THREADS / 32)) {
    double rs = 0.0;
    for (int j = lane; j < Sp; j += 32) {
      double v = 0.0;
      if (row < S && j < S) {
        const double q = Q[(size_t)row * S + j];
        rs += fabs(q + (row == j ? mu : 0.0));  // row sums of B = Q + mu I, as in build_B_kernel
        v = (row == j) ? q + mu : shat[(size_t)row * S + j];
      }
      B[(size_t)row * Sp + j] = v;
    }
    for (int o = 16; o > 0; o >>= 1) rs += __shfl_xor_sync(0xffffffffu, rs, o);
    if (lane == 0) atomicMax(&sc->norm_bits, (unsigned long long)__double_as_longlong(rs));
  }
}

// dL/dQ_ij = A_ij sqrt(pi_i / pi_j), A = the (symmetric up to rounding) adjoint of Bh, padded [Sp][Sp]
__global__ void unpad_sym_kernel(const double* __restrict__ src, const double* __restrict__ sr, int S, int Sp,
                                 double* __restrict__ dst) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= S * S) return;
  const int i = e / S, j = e - i * S;
  dst[e] = 0.5 * (src[(size_t)i * Sp + j] + src[(size_t)j * Sp + i]) * (sr[i] / sr[j]);
}

// flag[0] |= 1 unless mask and every count matrix are exactly symmetric
__global__ void symmetric_inputs_kernel(const double* __restrict__ mask, const double* __restrict__ C, int S, int K,
                                        int* __restrict__ flag) {
  const size_t n = (size_t)S * S;
  bool bad = false;
  for (size_t e = blockIdx.x * (size_t)blockDim.x + threadIdx.x; e < n; e += (size_t)gridDim.x * blockDim.x) {
    const int i = (int)(e / S), j = (int)(e - (size_t)i * S);
    if (j <= i) continue;
    const size_t et = (size_t)j * S + i;
    if (mask[e] != mask[et]) bad = true;
    for (int k = 0; k < K; ++k)
      if (C[(size_t)k * n + e] != C[(size_t)k * n + et]) bad = true;
  }
  if (bad) atomicOr(flag, 1);
}

// grid = S (one CTA per state i): bookkeeping copies of row i of the current Q, dL/dr_i, and the
// gradients of the upper-diagonal parameters of row i.  Nothing that other CTAs read is written.
__global__ void __launch_bounds__(EW_THREADS) large_update_rows_kernel(LargeUpdateArgs a) {
  extern __shared__ double sr[];  // [S] sqrt(pi)
  __shared__ double red[EW_THREADS / 32];
  const int S = a.S, i = blockIdx.x;
  const int epoch = a.epoch_counter[0];
  const double scale = a.loss_normalization ? 1.0 / a.sumC[0] : 1.0;
  // loss of this epoch (every CTA recomputes it in the same order -> same value)
  double lp = 0.0;
  for (int k = 0; k < a.K; ++k) lp += a.loss_part[k];
  lp *= scale;
  const bool improved = (epoch == 0 && a.best_mode == 0) ? true : (lp < a.best_loss[0]);
  const bool snap = a.snapshots && ((epoch & (epoch + 1)) == 0);
  int snap_idx = 0;
  if (snap) {
    int e1 = epoch + 1;
    while (e1 > 1) { e1 >>= 1; ++snap_idx; }
  }
  for (int j = threadIdx.x; j < S; j += blockDim.x) {
    const double q = a.Q[(size_t)i * S + j];
    a.Q_last[(size_t)i * S + j] = q;
    if (improved) a.Q_best[(size_t)i * S + j] = q;
    if (snap && snap_idx < a.n_snapshots) a.snapshots[((size_t)snap_idx * S + i) * S + j] = q;
  }
  softmax_sqrt(a.theta, S, sr, red);
  const double ri = sr[i];
  const double gii = a.G[(size_t)i * S + i];
  double col = 0.0, row = 0.0;
  for (int j = threadIdx.x; j < S; j += blockDim.x) {
    if (j == i) continue;
    const double u = upper_param(a.theta, S, i, j);
    const double sp = cherry::softplus_d(u), sg = cherry::softplus_grad_d(u);
    const double m_ij = a.mask[(size_t)i * S + j], m_ji = a.mask[(size_t)j * S + i];
    const double dM_ij = (a.G[(size_t)i * S + j] - gii) * scale;
    const double dM_ji = (a.G[(size_t)j * S + i] - a.G[(size_t)j * S + j]) * scale;
    const double rj = sr[j];
    col += dM_ji * (m_ji * sp) / rj;
    row += dM_ij * (m_ij * sp) * rj;
    if (j > i) {
      const double ds_ij = dM_ij * rj / ri, ds_ji = dM_ji * ri / rj;
      a.grad_theta[S + cherry::triu_index(i, j, S)] = sg * (m_ij * ds_ij + m_ji * ds_ji);
    }
  }
  col = block_sum_256(col, red);
  row = block_sum_256(row, red);
  if (threadIdx.x == 0) {
    a.dpi[i] = (col - row / (ri * ri)) / (2.0 * ri);
    a.pibuf[i] = ri * ri;
  }
}

// grid-stride over all parameters: softmax backward for the logits, then the optimiser step.
__global__ void __launch_bounds__(EW_THREADS) large_update_step_kernel(LargeUpdateArgs a) {
  extern __shared__ double sr[];
  __shared__ double red[EW_THREADS / 32];
  const int S = a.S, n_theta = S + S * (S - 1) / 2;
  const int epoch = a.epoch_counter[0];
  // pi comes from pibuf (written by the rows kernel), NOT from theta: other CTAs of this very
  // kernel are updating the logits while we read.
  for (int i = threadIdx.x; i < S; i += blockDim.x) sr[i] = a.pibuf[i];
  __syncthreads();
  double dot = 0.0;
  for (int i = threadIdx.x; i < S; i += blockDim.x) dot += sr[i] * a.dpi[i];
  dot = block_sum_256(dot, red);
  const int step = epoch + 1;
  const double bc1 = 1.0 - pow(a.beta1, (double)step), bc2s = sqrt(1.0 - pow(a.beta2, (double)step));
  for (int idx = blockIdx.x * blockDim.x + threadIdx.x; idx < n_theta; idx += gridDim.x * blockDim.x) {
    double g, lr;
    if (idx < S) {
      g = sr[idx] * (a.dpi[idx] - dot);
      lr = a.lr_pi;
    } else {
      g = a.grad_theta[idx];
      lr = a.lr_upper;
    }
    cherry::optimizer_step(a.theta[idx], a.adam_m[idx], a.adam_v[idx], g, lr, a.do_adam, a.beta1, a.beta2,
                           a.eps, bc1, bc2s);
  }
}

// grid = S: row i of Q(theta) (mode 1: after the step).  CTA 0 also closes the epoch's bookkeeping.
__global__ void __launch_bounds__(EW_THREADS) large_build_Q_kernel(LargeUpdateArgs a, int mode) {
  extern __shared__ double sr[];
  __shared__ double red[EW_THREADS / 32];
  const int S = a.S, i = blockIdx.x;
  softmax_sqrt(a.theta, S, sr, red);
  const double ri = sr[i];
  double rs = 0.0;
  for (int j = threadIdx.x; j < S; j += blockDim.x) {
    if (j == i) continue;
    const double u = upper_param(a.theta, S, i, j);
    const double sh = a.mask[(size_t)i * S + j] * cherry::softplus_d(u);
    const double v = sh * sr[j] / ri;
    a.Q[(size_t)i * S + j] = v;
    a.shat[(size_t)i * S + j] = sh;
    rs += v;
  }
  rs = block_sum_256(rs, red);
  if (threadIdx.x == 0) {
    a.Q[(size_t)i * S + i] = -rs;
    a.sr[i] = ri;
  }
  if (mode == 1 && i == 0 && threadIdx.x == 0) {
    const int epoch = a.epoch_counter[0];
    const double scale = a.loss_normalization ? 1.0 / a.sumC[0] : 1.0;
    double lp = 0.0;
    for (int k = 0; k < a.K; ++k) lp += a.loss_part[k];
    lp *= scale;
    if (epoch < a.loss_trace_epochs) a.loss_trace[epoch] = lp;
    const bool improved = (epoch == 0 && a.best_mode == 0) ? true : (lp < a.best_loss[0]);
    if (improved) a.best_loss[0] = lp;
    a.epoch_counter[0] = epoch + 1;
  }
}

// ------------------------------------------------------------------------------ the plan
struct Plan {
  int S, Sp, K, tiles;
  size_t n_p;
  // workspace offsets in bytes
  size_t off_sym_flag, off_sched, off_scalars, off_s, off_deg, off_tau, off_w, off_loss_partial, off_grad_theta, off_dpi, off_pibuf;
  size_t off_P, off_Pbar, off_X0, off_chain, off_partial, off_prof, total_bytes;
  size_t max_items, max_groups;  // capacity of each DfList's item array and state words in the workspace
  int slots_per_bucket;   // chain slots 1..kSStore+1
  int loss_blocks;
  DfList df_fwd, df_bwd;  // the two power chains as dataflow item lists
  DfList df_fwd_sym;      // forward chain of a symmetric B: upper tiles only, mirrored (shares df_fwd's state words)
  size_t off_sr = 0;      // [S] sqrt(pi) of the current parameters (symmetric mode)
  size_t off_shat = 0;    // [S][S] mask_ij softplus(u_ij) of the current parameters
  size_t off_tailbuf = 0; // shares of the power adjoints written by the tail CTAs of the fused Taylor pass
  bool lists_fit = true;  // every DfList's items and groups fit the workspace carved for them
};

size_t align256(size_t x) { return (x + 255) / 256 * 256; }

// Builds the layout and the item lists of the power chains (absolute device pointers if base != nullptr).
void make_plan(Plan& p, int S, int K, char* base) {
  p.S = S;
  p.K = K;
  p.Sp = (S + BT - 1) / BT * BT;
  p.tiles = (p.Sp / BT) * (p.Sp / BT);
  p.n_p = (size_t)p.Sp * p.Sp;
  p.slots_per_bucket = kSStore + 1;
  p.loss_blocks = (int)((p.n_p + 4 * EW_THREADS - 1) / (4 * EW_THREADS)) * kLossLanes;  // blocks of loss_grad_kernel
  const size_t mat = p.n_p * sizeof(double);
  const int n_theta = S + S * (S - 1) / 2;
  size_t off = 0;
  auto carve = [&](size_t bytes) { size_t o = off; off = align256(off + bytes); return o; };
  p.off_scalars = carve(sizeof(LargeScalars));
  p.off_sym_flag = carve(sizeof(int));  // result word of symmetric_inputs_kernel
  p.off_sched = carve(sizeof(SqSchedule) + sizeof(int) * ((size_t)kSStore * K * 2 + (size_t)K * (kSStore + 1) +
                                                            (size_t)K + (size_t)K * p.tiles));
  p.off_s = carve(sizeof(int) * K);
  p.off_deg = carve(sizeof(int) * (3 * (size_t)K + 2));  // degrees, then the unsquared / squared bucket lists and their lengths
  p.off_tau = carve(sizeof(double) * K);
  p.off_w = carve(sizeof(double) * K * (kDeg + 1));
  p.off_loss_partial = carve(sizeof(double) * ((size_t)p.loss_blocks + 4 * ((p.n_p + EW_THREADS - 1) / EW_THREADS) + kTaylorTailUnits + 1024));
  p.off_grad_theta = carve(sizeof(double) * n_theta);
  p.off_dpi = carve(sizeof(double) * S);
  p.off_pibuf = carve(sizeof(double) * S);
  // dataflow lists: upper bounds (fine slices everywhere): items <= 3 * (m-1) * tiles * slices
  {
    const size_t max_groups = 3 * (size_t)kDeg * p.tiles + 64;
    const size_t max_items = 3 * (size_t)kDeg * p.tiles * (p.Sp / BT) + max_groups * kDfSlabs + 64;
    p.max_items = max_items;
    p.max_groups = max_groups;
    p.df_fwd.off_items = carve(sizeof(DfItem) * max_items);
    p.df_fwd.off_state = carve(sizeof(int) * df_state_ints(kDeg, p.tiles, (int)max_groups));
    p.df_bwd.off_items = carve(sizeof(DfItem) * max_items);
    p.df_bwd.off_state = carve(sizeof(int) * df_state_ints(kDeg, p.tiles, (int)max_groups));
    p.df_fwd_sym.off_items = carve(sizeof(DfItem) * max_items);
    p.df_fwd_sym.off_state = p.df_fwd.off_state;  // one of the two forward lists runs per evaluation
    p.off_sr = carve(sizeof(double) * S);
    p.off_shat = carve(sizeof(double) * S * S);
    p.off_tailbuf = carve(sizeof(double) * kTaylorTailUnits * kDeg * kTaylorThreads);
  }
  p.off_prof = carve(sizeof(long long) * 8 * 2 * 1024);  // phase profile of the two chain launches (<= 1024 CTAs)
  p.off_P = carve(mat * kDeg);
  p.off_Pbar = carve(mat * kDeg);
  p.off_X0 = carve(mat * K);
  p.off_chain = carve(mat * K * p.slots_per_bucket);
  // ---- the two power chains as dataflow lists (pointers are only meaningful when base != nullptr)
  {
    char* b0 = base ? base : reinterpret_cast<char*>(0);
    auto Pj = [&](int j) { return reinterpret_cast<double*>(b0 + p.off_P) + (size_t)(j - 1) * p.n_p; };
    auto Pbar = [&](int j) { return reinterpret_cast<double*>(b0 + p.off_Pbar) + (size_t)(j - 1) * p.n_p; };
    const int tn = p.Sp / BT, cpt = p.Sp / BK;  // tiles per side, chunks per term
    struct TermSpec { const double* A; const double* B; int ta, tb, a_mat, a_ver, b_mat, b_ver; };
    // reduction items (one per row slab) of the `count` oldest pending groups (all of them if count < 0): the
    // queue holds them a lag behind the group's products, and always before anything that reads the result
    auto emit_reduce = [&](DfList& L, int count) {
      while (!L.pending.empty() && count != 0) {
        const int gi = L.pending.front();
        L.pending.erase(L.pending.begin());
        for (int sl = 0; sl < kDfSlabs; ++sl) {
          DfItem it{};
          it.A = nullptr; it.B = nullptr; it.group = gi; it.slice = sl; it.a_mat = it.b_mat = -1; it.kind = 1;
          it.g = L.groups[gi];
          L.items.push_back(it);
        }
        if (count > 0) --count;
      }
    };
    // one output matrix update C (+)= sum of terms, for every tile; slices of 80 (fine) or whole K per term (coarse)
    auto add_update = [&](DfList& L, double* C, int c_mat, int need_ver, int accumulate,
                          const std::vector<TermSpec>& terms, int per_term, bool upper_only = false) {
      for (int ti = 0; ti < tn; ++ti)
        for (int tj = upper_only ? ti : 0; tj < tn; ++tj) {
          DfGroup g;
          g.C = C; g.m0 = ti * BT; g.n0 = tj * BT; g.accumulate = accumulate; g.c_mat = c_mat; g.need_ver = need_ver;
          g.partial_off = L.partial_tiles; g.n_slabs = kDfSlabs;
          g.mirror = (upper_only && ti != tj) ? 1 : 0; g.pad = 0;
          g.n_slices = (int)terms.size() * per_term;
          const int gi = (int)L.groups.size();
          int slice = 0;
          for (const TermSpec& t : terms)
            for (int z = 0; z < per_term; ++z) {
              DfItem it;
              it.A = t.A; it.B = t.B; it.ta = t.ta; it.tb = t.tb;
              const int c_begin = cpt * z / per_term, c_end = cpt * (z + 1) / per_term;  // chunks of this slice
              it.k0 = c_begin * BK; it.n_chunks = c_end - c_begin;
              it.group = gi; it.slice = slice++;
              it.a_mat = t.a_ver > 0 ? t.a_mat : -1; it.a_ver = t.a_ver;
              it.b_mat = t.b_ver > 0 ? t.b_mat : -1; it.b_ver = t.b_ver;
              it.kind = 0; it.pad = 0;
              it.g = g;  // n_slices is already final (set above)
              L.items.push_back(it);
            }
          L.partial_tiles += g.n_slices;
          L.groups.push_back(g);
          const bool direct = (g.n_slices == 1) && !g.accumulate;
          if (!direct) L.pending.push_back(gi);
          if ((int)L.pending.size() > kDfReduceLag) emit_reduce(L, 1);
        }
    };
    // K slices per term of a level with `term_tiles` (term, output tile) products: as few as keep about
    // kDfChainTarget work items in the level (every item pays ~3 us of queue / fence / reduction latency, a
    // 80-deep slice is only 10 us of arithmetic), at most 5 (80-deep)
    auto slices_for = [&](int term_tiles) {
      for (int n : {1, 2, 3, 4})
        if (term_tiles * n >= kDfChainTarget) return n;
      return 5;
    };
    // forward: P_{b+r} = P_b P_r, r = 1..min(b, m-b); matrix id of P_j is j-1, version 1 once written (P_1: given).
    // Second list for a SYMMETRIC B (reversible Q in the basis diag(sqrt(pi)), see build_B_sym_kernel): every
    // power is symmetric, so only the tiles on and above the diagonal are computed and the reductions mirror them.
    for (int sym = 0; sym < 2; ++sym) {
      DfList& L = sym ? p.df_fwd_sym : p.df_fwd;
      L.items.clear(); L.groups.clear(); L.pending.clear(); L.partial_tiles = 0; L.n_mats = kDeg;
      const int tile_groups = sym ? tn * (tn + 1) / 2 : p.tiles;
      std::vector<int> ver(kDeg + 1, 0);
      for (int b = 1; b < kDeg; b *= 2) {
        // the squaring P_2b first: it is the critical path of the next level
        std::vector<int> rs;
        if (b + b <= kDeg) rs.push_back(b);
        for (int r = 1; r <= b && b + r <= kDeg; ++r)
          if (r != b) rs.push_back(r);
        const int per_term = slices_for((int)rs.size() * tile_groups);
        for (int r : rs)
          add_update(L, Pj(b + r), b + r - 1, 0, 0, {TermSpec{Pj(b), Pj(r), 0, 0, b - 1, ver[b], r - 1, ver[r]}}, per_term,
                     sym != 0);
        emit_reduce(L, -1);  // the next level reads this level's results
        for (int r : rs) ver[b + r] = 1;
      }
    }
    // backward, levels in reverse.  For P_{b+r} = P_b P_r:
    //   Pbar_r += P_b^T Pbar_{b+r} (r != b),   Pbar_b += sum_r Pbar_{b+r} P_r^T (+ P_b^T Pbar_{2b})
    // matrix id of Pbar_j is j-1; version 0 = the value accumulate_M left; P_j are inputs (no waits).
    {
      DfList& L = p.df_bwd;
      L.items.clear(); L.groups.clear(); L.pending.clear(); L.partial_tiles = 0; L.n_mats = kDeg;
      std::vector<int> ver(kDeg + 1, 0);
      std::vector<int> bases;
      for (int b = 1; b < kDeg; b *= 2) bases.push_back(b);
      for (int li = (int)bases.size() - 1; li >= 0; --li) {
        const int b = bases[li];
        const int rmax = (b + b <= kDeg) ? b : kDeg - b;
        std::vector<TermSpec> big;
        for (int r = 1; r <= rmax; ++r) big.push_back(TermSpec{Pbar(b + r), Pj(r), 0, 1, b + r - 1, ver[b + r], -1, 0});
        if (rmax == b) big.push_back(TermSpec{Pj(b), Pbar(2 * b), 1, 0, -1, 0, 2 * b - 1, ver[2 * b]});
        int n_small = 0;
        for (int r = 1; r <= rmax; ++r)
          if (r != b) ++n_small;
        const int per_term = slices_for(((int)big.size() + n_small) * p.tiles);
        // the long concatenated update first (it is the level's critical path)
        add_update(L, Pbar(b), b - 1, ver[b], 1, big, per_term);
        for (int r = 1; r <= rmax; ++r)
          if (r != b)
            add_update(L, Pbar(r), r - 1, ver[r], 1, {TermSpec{Pj(b), Pbar(b + r), 1, 0, -1, 0, b + r - 1, ver[b + r]}}, per_term);
        emit_reduce(L, -1);  // the next level reads this level's results
        ver[b]++;
        for (int r = 1; r <= rmax; ++r)
          if (r != b) ver[r]++;
      }
    }
  }
  // split-K partial buffers: the squaring dataflow kernels need kSqPartialSlots matrices, the chain
  // lists one compact 80x80 tile per (group, slice); the launches are stream ordered and share it
  {
    const size_t tile_doubles = (size_t)BT * BT;
    const size_t need = (size_t)std::max(std::max(p.df_fwd.partial_tiles, p.df_fwd_sym.partial_tiles), p.df_bwd.partial_tiles) * tile_doubles;
    size_t doubles = p.n_p * kSqPartialSlots;
    if (need > doubles) doubles = need;
    p.off_partial = carve(doubles * sizeof(double));
  }
  p.total_bytes = off;
  // fit_large_prepare uploads the item lists into the arrays carved above, and coef_kernel clears the state words
  // of groups.size() groups: the bounds are estimates, so they are checked
  for (const DfList* L : {&p.df_fwd, &p.df_bwd, &p.df_fwd_sym})
    if (L->items.size() > p.max_items || L->groups.size() > p.max_groups) p.lists_fit = false;
}

// make_plan builds ~6000 work items; the evaluation entry points run once per epoch (and per
// rank in the sharded path), so the plan of the last (S, K, workspace) is kept per host thread.
const Plan& get_plan(int S, int K, char* base) {
  static thread_local Plan cache[2];
  static thread_local int cS[2] = {0, 0}, cK[2] = {0, 0};
  static thread_local char* cbase[2] = {nullptr, nullptr};
  const int slot = base ? 1 : 0;
  if (cS[slot] != S || cK[slot] != K || cbase[slot] != base) {
    cache[slot] = Plan();
    make_plan(cache[slot], S, K, base);
    cS[slot] = S; cK[slot] = K; cbase[slot] = base;
  }
  return cache[slot];
}

int ensure_gemm_attr() {
  static bool attr_set[64] = {false};
  int dev = 0;
  CHERRY_CUDA(cudaGetDevice(&dev));
  if (dev < 64 && !attr_set[dev]) {
    CHERRY_CUDA(cudaFuncSetAttribute(gemm_tasks_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                     NSTAGE * 2 * TILE_ELEMS * (int)sizeof(double)));
    CHERRY_CUDA(cudaFuncSetAttribute(squaring_dataflow_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                     NSTAGE * 2 * TILE_ELEMS * (int)sizeof(double)));
    CHERRY_CUDA(cudaFuncSetAttribute(squaring_dataflow_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                     NSTAGE * 2 * TILE_ELEMS * (int)sizeof(double)));
    CHERRY_CUDA(cudaFuncSetAttribute(chain_dataflow_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                     NSTAGE * 2 * TILE_ELEMS * (int)sizeof(double)));
    attr_set[dev] = true;
  }
  return 0;
}

void fill_update_args(LargeUpdateArgs& u, const cherry_fit_args& a, const Plan& p, char* base) {
  u.S = a.S; u.K = a.K; u.mask = a.mask; u.theta = a.theta; u.adam_m = a.adam_m; u.adam_v = a.adam_v;
  u.Q = a.Q; u.Q_best = a.Q_best; u.Q_last = a.Q_last; u.best_loss = a.best_loss;
  u.loss_trace = a.loss_trace; u.loss_trace_epochs = a.loss_trace_epochs; u.snapshots = a.snapshots;
  u.n_snapshots = a.n_snapshots; u.G = a.dQ_part; u.loss_part = a.loss_part; u.sumC = a.sumC;
  u.epoch_counter = a.epoch_counter;
  u.grad_theta = reinterpret_cast<double*>(base + p.off_grad_theta);
  u.dpi = reinterpret_cast<double*>(base + p.off_dpi);
  u.pibuf = reinterpret_cast<double*>(base + p.off_pibuf);
  u.shat = reinterpret_cast<double*>(base + p.off_shat);
  u.sr = reinterpret_cast<double*>(base + p.off_sr);
  u.lr_pi = a.lr_pi; u.lr_upper = a.lr_upper; u.beta1 = a.beta1; u.beta2 = a.beta2; u.eps = a.eps;
  u.do_adam = a.do_adam; u.loss_normalization = a.loss_normalization; u.best_mode = a.best_mode;
}

// Sizes the large path supports; the plan of (S, K) in *plan.
int check_sizes(int S, int K, int n_problems, const Plan** plan) {
  if (n_problems != 1)
    return cherry::fail(CHERRY_ELIMIT, "fit: batched problems are supported for S <= %d only", cherry::kSmallFitMaxS);
  if (K > CHERRY_LARGE_FIT_MAX_K)
    return cherry::fail(CHERRY_ELIMIT, "fit: K=%d time buckets (or exponents) exceed the limit of %d for S > %d", K,
                        CHERRY_LARGE_FIT_MAX_K, cherry::kSmallFitMaxS);
  const Plan& p = get_plan(S, K, nullptr);
  if (!p.lists_fit)
    return cherry::fail(CHERRY_ELIMIT, "fit: the power-chain work lists of S=%d exceed their workspace", S);
  *plan = &p;
  return 0;
}

int check_large(const cherry_fit_args& a) {
  const Plan* pp = nullptr;
  int rc = check_sizes(a.S, a.K, a.n_problems, &pp);
  if (rc) return rc;
  const Plan& p = *pp;
  if (!a.workspace || a.workspace_bytes < p.total_bytes)
    return cherry::fail(CHERRY_EINVAL, "fit: workspace of %zu bytes required, got %zu", p.total_bytes,
                        a.workspace_bytes);
  return 0;
}

}  // namespace

namespace cherry {

int fit_large_workspace_bytes(int S, int K, int n_problems, size_t* bytes) {
  const Plan* p = nullptr;
  int rc = check_sizes(S, K, n_problems, &p);
  if (rc) return rc;
  *bytes = p->total_bytes;
  return 0;
}

// Which workspaces were prepared for a model whose evaluation may run in the symmetric form (mask and counts
// exactly symmetric, parameters given): decided once per fit by fit_large_prepare, read by the training entry
// points.  CHERRY_FIT_SYMMETRIC=0 is the A/B switch.
static std::mutex g_sym_mutex;
static std::unordered_map<const void*, int> g_sym_mode;
static int symmetric_mode_of(const cherry_fit_args& a) {
  if (!a.theta || !a.mask) return 0;
  std::lock_guard<std::mutex> lock(g_sym_mutex);
  auto it = g_sym_mode.find(a.workspace);
  return it == g_sym_mode.end() ? 0 : it->second;
}

int fit_large_symmetric_form(const cherry_fit_args& a) { return symmetric_mode_of(a) == 1 ? 1 : 0; }

// Uploads the item lists of the power chains (absolute pointers into this workspace) and decides the symmetric
// form.  Synchronous.
int fit_large_prepare(const cherry_fit_args& a, cudaStream_t stream) {
  int rc = check_large(a);
  if (rc) return rc;
  char* base = reinterpret_cast<char*>(a.workspace);
  const Plan& p = get_plan(a.S, a.K, base);
  CHERRY_CUDA(cudaStreamSynchronize(stream));
  for (const DfList* L : {&p.df_fwd, &p.df_bwd, &p.df_fwd_sym}) {
    CHERRY_CUDA(cudaMemcpy(base + L->off_items, L->items.data(), L->items.size() * sizeof(DfItem), cudaMemcpyHostToDevice));
  }
  CHERRY_CUDA(cudaMemset(base + p.off_scalars, 0, sizeof(LargeScalars)));
  {
    const bool sym_allowed = !(getenv("CHERRY_FIT_SYMMETRIC") && atoi(getenv("CHERRY_FIT_SYMMETRIC")) == 0);  // read per fit: tests toggle it
    int mode = 0;
    if (sym_allowed && a.theta && a.mask && a.C) {
      int* flag = reinterpret_cast<int*>(base + p.off_sym_flag);
      CHERRY_CUDA(cudaMemset(flag, 0, sizeof(int)));
      symmetric_inputs_kernel<<<256, 256>>>(a.mask, a.C, a.S, a.K, flag);
      CHERRY_LAUNCH_CHECK("symmetric_inputs_kernel");
      int bad = 1;
      CHERRY_CUDA(cudaMemcpy(&bad, flag, sizeof(int), cudaMemcpyDeviceToHost));
      mode = bad ? 0 : 1;
    }
    std::lock_guard<std::mutex> lock(g_sym_mutex);
    g_sym_mode[a.workspace] = mode;
  }
  // chain slots are read as "Xbar" for inactive levels never; but slot 1 of every bucket is
  // always written by loss_grad (s = 0) or the backward chain, so no clearing is needed.
  return 0;
}

static int fit_large_impl(const cherry_fit_args& a, cudaStream_t stream, double* P_out, bool allow_sym = false);

// Optional phase timeline (debug / profiling): when g_timeline is non-null, fit_large_impl records
// an event after every phase of one evaluation.
struct Timeline {
  static constexpr int kMax = 16;
  cudaEvent_t ev[kMax];
  const char* name[kMax];
  int n = 0;
};
static Timeline* g_timeline = nullptr;
static void mark(const char* name, cudaStream_t stream) {
  if (!g_timeline || g_timeline->n >= Timeline::kMax) return;
  cudaEventRecord(g_timeline->ev[g_timeline->n], stream);
  g_timeline->name[g_timeline->n++] = name;
}

int fit_large_expm(const cherry_fit_args& a, cudaStream_t stream, bool training) {
  return fit_large_impl(a, stream, nullptr, training);
}

// expm(t_k Q) for every bucket into P_out [K][S][S]; prepares the workspace itself (synchronous).
int fit_large_forward_only(const cherry_fit_args& a, double* P_out, cudaStream_t stream) {
  if (!P_out) return fail(CHERRY_EINVAL, "expm: null output pointer");
  int rc = fit_large_prepare(a, stream);
  if (rc) return rc;
  return fit_large_impl(a, stream, P_out);
}

static int fit_large_impl(const cherry_fit_args& a, cudaStream_t stream, double* P_out, bool allow_sym) {
  int rc = check_large(a);
  if (rc) return rc;
  if ((rc = ensure_gemm_attr())) return rc;
  char* base = reinterpret_cast<char*>(a.workspace);
  const Plan& p = get_plan(a.S, a.K, base);  // host-side tables; the device copies were uploaded by prepare
  // symmetric form (see build_B_sym_kernel): only where Q is known to be the reversible model of a.theta -- the
  // training entry points -- and fit_large_prepare found mask and counts symmetric
  const bool sym = allow_sym && P_out == nullptr && symmetric_mode_of(a) == 1;
  const int tn = p.Sp / BT, sq_tiles = sym ? tn * (tn + 1) / 2 : p.tiles;
  double* sr = reinterpret_cast<double*>(base + p.off_sr);
  LargeScalars* sc = reinterpret_cast<LargeScalars*>(base + p.off_scalars);
  int* s_arr = reinterpret_cast<int*>(base + p.off_s);
  double* tau = reinterpret_cast<double*>(base + p.off_tau);
  double* w = reinterpret_cast<double*>(base + p.off_w);
  double* loss_partial = reinterpret_cast<double*>(base + p.off_loss_partial);
  double* P = reinterpret_cast<double*>(base + p.off_P);
  double* Pbar = reinterpret_cast<double*>(base + p.off_Pbar);
  double* X0 = reinterpret_cast<double*>(base + p.off_X0);
  double* chain = reinterpret_cast<double*>(base + p.off_chain);
  const int eb = (int)((p.n_p + EW_THREADS - 1) / EW_THREADS);
  const size_t wsmem = sizeof(double) * a.K * (kDeg + 1);  // K <= CHERRY_LARGE_FIT_MAX_K (check_large)

  mark("start", stream);
  if (sym)
    build_B_sym_kernel<<<(p.Sp + 7) / 8, EW_THREADS, 0, stream>>>(a.Q, reinterpret_cast<const double*>(base + p.off_shat), a.S,
                                                                 p.Sp, P, sc);
  else
    build_B_kernel<<<(p.Sp + 7) / 8, EW_THREADS, 0, stream>>>(a.Q, a.S, p.Sp, P, sc);
  CHERRY_LAUNCH_CHECK("build_B_kernel");
  SqSchedule* sched = reinterpret_cast<SqSchedule*>(base + p.off_sched);
  int* df_state_fwd = reinterpret_cast<int*>(base + p.df_fwd.off_state);
  int* df_state_bwd = reinterpret_cast<int*>(base + p.df_bwd.off_state);
  int* deg_arr = reinterpret_cast<int*>(base + p.off_deg);
  const int persistent_grid = kCtasPerSm * sm_count();
  coef_kernel<<<1, 256, 0, stream>>>(a.t, a.K, sc, s_arr, deg_arr, w, tau, a.status_flag, sched, sq_tiles,
                                     persistent_grid, df_state_fwd,
                                     (int)df_state_ints(p.df_fwd.n_mats, p.tiles, (int)p.df_fwd.groups.size()),
                                     df_state_bwd,
                                     (int)df_state_ints(p.df_bwd.n_mats, p.tiles, (int)p.df_bwd.groups.size()),
                                     sym ? kSqKsplitSym : kSqKsplitGeneral);
  CHERRY_LAUNCH_CHECK("coef_kernel");
  mark("build_B+coef", stream);
  const size_t gemm_smem = (size_t)NSTAGE * 2 * TILE_ELEMS * sizeof(double);
  auto launch_chain = [&](const DfList& L, int* state, const char* name) -> int {
    long long* prof = nullptr;
    if (g_timeline && persistent_grid <= 1024)
      prof = reinterpret_cast<long long*>(base + p.off_prof) + (&L == &p.df_bwd ? 8 * 1024 : 0);
    chain_dataflow_kernel<<<persistent_grid, GEMM_THREADS, gemm_smem, stream>>>(
        reinterpret_cast<const DfItem*>(base + L.off_items), (int)L.items.size(), (int)L.groups.size(), state,
        L.n_mats, p.Sp,
        reinterpret_cast<double*>(base + p.off_partial), a.status_flag, prof);
    CHERRY_LAUNCH_CHECK(name);
    return 0;
  };
  if ((rc = launch_chain(sym ? p.df_fwd_sym : p.df_fwd, df_state_fwd, "chain_dataflow_kernel<fwd>"))) return rc;
  mark("powers_fwd", stream);
  static bool ew_attr[64] = {false};
  {
    int dev = 0;
    CHERRY_CUDA(cudaGetDevice(&dev));
    if (dev < 64 && !ew_attr[dev]) {
      CHERRY_CUDA(cudaFuncSetAttribute(poly_eval_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
      CHERRY_CUDA(cudaFuncSetAttribute(accumulate_M_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
      CHERRY_CUDA(cudaFuncSetAttribute(taylor_fused_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
#define CHERRY_TAYLOR_ATTR(SYM_, PARTS_)                                                               \
  CHERRY_CUDA(cudaFuncSetAttribute(taylor_fused_smem_kernel<1, kTaylorThreads, SYM_, PARTS_>,          \
                                   cudaFuncAttributeMaxDynamicSharedMemorySize, 113 * 1024))
      CHERRY_TAYLOR_ATTR(false, 1); CHERRY_TAYLOR_ATTR(false, 2); CHERRY_TAYLOR_ATTR(false, 4);
      CHERRY_TAYLOR_ATTR(false, 8); CHERRY_TAYLOR_ATTR(false, 16);
      CHERRY_TAYLOR_ATTR(true, 1); CHERRY_TAYLOR_ATTR(true, 2); CHERRY_TAYLOR_ATTR(true, 4);
      CHERRY_TAYLOR_ATTR(true, 8); CHERRY_TAYLOR_ATTR(true, 16);
#undef CHERRY_TAYLOR_ATTR
      ew_attr[dev] = true;
    }
  }
  double* fused_partial = loss_partial + (size_t)p.loss_blocks;
  int fused_blocks = 0;
  if (P_out != nullptr) {
    poly_eval_kernel<<<eb, EW_THREADS, wsmem, stream>>>(P, p.n_p, a.S, p.Sp, a.K, w, X0);
    CHERRY_LAUNCH_CHECK("poly_eval_kernel");
  } else {
    const bool two_ctas_fit = 2 * (wsmem + 3 * sizeof(int) * a.K + 8 + sizeof(double) * (kTaylorStagesS + kDeg) * kTaylorThreads + 1024) <=
                              (size_t)227 * 1024;  // else (K >= 157): the register variant, one CTA per SM
    if (two_ctas_fit) {
      // kTaylorThreads per CTA, two CTAs per SM (128 registers: the powers live in shared memory)
      constexpr int NT = kTaylorThreads;
      const size_t ssmem = wsmem + 3 * sizeof(int) * a.K + 8 + sizeof(double) * (kTaylorStagesS + kDeg) * NT;
      const size_t n_visit = sym ? (size_t)(p.Sp / 2) * (p.Sp + 1) : p.n_p;  // symmetric form: the upper triangle
      const int n_chunks = (int)((n_visit + NT - 1) / NT), slots = 2 * sm_count();
      // the chunks beyond a multiple of the resident CTAs, when they would fill less than half a round, run as
      // (chunk, share of the buckets) CTAs of their own -- see the kernel
      int tail = 0, parts = 1;
      if (n_chunks > slots && n_chunks % slots != 0 && n_chunks % slots <= slots / 2) {
        tail = n_chunks % slots;
        for (int cand : {16, 8, 4, 2})
          if (cand * tail <= slots && cand * tail <= kTaylorTailUnits) {
            parts = cand;
            break;
          }
        if (parts == 1) tail = 0;
      }
      const int n_main = n_chunks - tail;
      const int grid2 = std::min(n_main, slots), grid_tail = tail * parts;
      fused_blocks = grid2 + grid_tail;
      double* tailbuf = reinterpret_cast<double*>(base + p.off_tailbuf);
      int* counter = &sched->pad[0];
#define CHERRY_TAYLOR_S(SYM_, PARTS_, GRID_, C0_, C1_, PARTIAL_)                                                              \
  taylor_fused_smem_kernel<1, NT, SYM_, PARTS_><<<GRID_, NT, ssmem, stream>>>(P, p.n_p, a.S, p.Sp, a.K, w, s_arr, deg_arr, a.C, \
                                                                               X0, Pbar, PARTIAL_, counter, C0_, C1_, tailbuf)
      if (n_main > 0) {
        if (sym) CHERRY_TAYLOR_S(true, 1, grid2, 0, n_main, fused_partial);
        else CHERRY_TAYLOR_S(false, 1, grid2, 0, n_main, fused_partial);
      }
      if (tail > 0) {
        if (n_main > 0) CHERRY_LAUNCH_CHECK("taylor_fused_smem_kernel");
        double* tp = fused_partial + grid2;
        if (sym) {
          if (parts == 16) CHERRY_TAYLOR_S(true, 16, grid_tail, n_main, n_chunks, tp);
          else if (parts == 8) CHERRY_TAYLOR_S(true, 8, grid_tail, n_main, n_chunks, tp);
          else if (parts == 4) CHERRY_TAYLOR_S(true, 4, grid_tail, n_main, n_chunks, tp);
          else CHERRY_TAYLOR_S(true, 2, grid_tail, n_main, n_chunks, tp);
        } else {
          if (parts == 16) CHERRY_TAYLOR_S(false, 16, grid_tail, n_main, n_chunks, tp);
          else if (parts == 8) CHERRY_TAYLOR_S(false, 8, grid_tail, n_main, n_chunks, tp);
          else if (parts == 4) CHERRY_TAYLOR_S(false, 4, grid_tail, n_main, n_chunks, tp);
          else CHERRY_TAYLOR_S(false, 2, grid_tail, n_main, n_chunks, tp);
        }
        CHERRY_LAUNCH_CHECK("taylor_fused_smem_kernel<tail>");
        const size_t tail_elems = (size_t)tail * NT;
        if (sym)
          taylor_tail_reduce_kernel<true><<<tail * kDeg, NT, 0, stream>>>(tailbuf, parts, tail_elems, (size_t)n_main * NT, n_visit,
                                                                          p.n_p, p.Sp, Pbar);
        else
          taylor_tail_reduce_kernel<false><<<tail * kDeg, NT, 0, stream>>>(tailbuf, parts, tail_elems, (size_t)n_main * NT, n_visit,
                                                                           p.n_p, p.Sp, Pbar);
      }
#undef CHERRY_TAYLOR_S
    } else {
      const size_t fsmem = wsmem + 3 * sizeof(int) * a.K + 8 + sizeof(double) * kTaylorStages * EW_THREADS;
      fused_blocks = std::min(eb, sm_count());
      taylor_fused_kernel<<<fused_blocks, EW_THREADS, fsmem, stream>>>(P, p.n_p, a.S, p.Sp, a.K, w, s_arr, deg_arr, a.C,
                                                                        X0, Pbar, fused_partial);
    }
    CHERRY_LAUNCH_CHECK("taylor_fused_kernel");
  }
  mark("taylor_fused", stream);
  squaring_dataflow_kernel<false><<<persistent_grid, GEMM_THREADS, gemm_smem, stream>>>(
      sched, s_arr, a.K, p.Sp, X0, chain, p.slots_per_bucket, reinterpret_cast<double*>(base + p.off_partial),
      a.status_flag, sym ? 1 : 0);
  CHERRY_LAUNCH_CHECK("squaring_dataflow_kernel<fwd>");
  mark("squarings_fwd", stream);
  if (P_out != nullptr) {
    extract_P_kernel<<<dim3((a.S * a.S + 255) / 256, a.K), 256, 0, stream>>>(s_arr, X0, chain, p.slots_per_bucket,
                                                                             p.n_p, a.S, p.Sp, P_out);
    CHERRY_LAUNCH_CHECK("extract_P_kernel");
    return 0;
  }
  const int loss_grid = (int)((p.n_p + 4 * EW_THREADS - 1) / (4 * EW_THREADS)) * kLossLanes;
  loss_grad_kernel<<<loss_grid, EW_THREADS, 0, stream>>>(a.C, a.S, p.Sp, p.n_p, a.K, s_arr, deg_arr, X0, chain,
                                                         p.slots_per_bucket, loss_partial);
  CHERRY_LAUNCH_CHECK("loss_grad_kernel");
  loss_reduce_kernel<<<1, 256, 0, stream>>>(loss_partial, a.K, loss_grid, a.loss_part, fused_partial, fused_blocks);
  CHERRY_LAUNCH_CHECK("loss_reduce_kernel");
  mark("loss_grad", stream);
  squaring_dataflow_kernel<true><<<persistent_grid, GEMM_THREADS, gemm_smem, stream>>>(
      sched, s_arr, a.K, p.Sp, X0, chain, p.slots_per_bucket, reinterpret_cast<double*>(base + p.off_partial),
      a.status_flag, sym ? 1 : 0);
  CHERRY_LAUNCH_CHECK("squaring_dataflow_kernel<bwd>");
  mark("squarings_bwd", stream);
  accumulate_M_kernel<<<std::min(eb, 4 * sm_count()), EW_THREADS, wsmem + sizeof(int) * a.K, stream>>>(
      chain, p.slots_per_bucket, p.n_p, a.K, w, Pbar, deg_arr);
  CHERRY_LAUNCH_CHECK("accumulate_M_kernel");
  mark("accumulate_M", stream);
  if ((rc = launch_chain(p.df_bwd, df_state_bwd, "chain_dataflow_kernel<bwd>"))) return rc;
  mark("powers_bwd", stream);
  if (sym)
    unpad_sym_kernel<<<(a.S * a.S + 255) / 256, 256, 0, stream>>>(Pbar, sr, a.S, p.Sp, a.dQ_part);
  else
    unpad_kernel<<<(a.S * a.S + 255) / 256, 256, 0, stream>>>(Pbar, a.S, p.Sp, a.dQ_part);
  CHERRY_LAUNCH_CHECK("unpad_kernel");
  mark("unpad", stream);
  return 0;
}

// One evaluation with an event after every phase; prints the phase durations to stderr.
int fit_large_timeline(const cherry_fit_args& a, cudaStream_t stream) {
  Timeline tl;
  for (int i = 0; i < Timeline::kMax; ++i) CHERRY_CUDA(cudaEventCreate(&tl.ev[i]));
  // the timeline is of the training configuration: symmetric form where the fit would use it
  int rc = fit_large_impl(a, stream, nullptr, true);  // warm
  if (rc) return rc;
  const Plan& pl = get_plan(a.S, a.K, nullptr);
  char* wbase = reinterpret_cast<char*>(a.workspace);
  CHERRY_CUDA(cudaMemsetAsync(wbase + pl.off_prof, 0, sizeof(long long) * 8 * 2 * 1024, stream));
  g_timeline = &tl;
  rc = fit_large_impl(a, stream, nullptr, true);
  g_timeline = nullptr;
  if (rc) return rc;
  CHERRY_CUDA(cudaStreamSynchronize(stream));
  {
    std::vector<long long> prof(8 * 2 * 1024);
    CHERRY_CUDA(cudaMemcpy(prof.data(), wbase + pl.off_prof, prof.size() * sizeof(long long), cudaMemcpyDeviceToHost));
    const char* names[7] = {"dequeue", "operand-wait", "product", "arrive", "reduce-wait", "reduce", "publish"};
    for (int which = 0; which < 2; ++which) {
      long long sum[8] = {0}, mx_items = 0;
      int ctas = 0;
      for (int b = 0; b < 1024; ++b) {
        const long long* r = prof.data() + (size_t)which * 8 * 1024 + b * 8;
        if (r[7] == 0) continue;
        ++ctas;
        for (int k = 0; k < 8; ++k) sum[k] += r[k];
        if (r[7] > mx_items) mx_items = r[7];
      }
      if (!ctas) continue;
      fprintf(stderr, "[chain %s] %d CTAs, %lld items (max %lld per CTA); mean us per CTA:", which ? "bwd" : "fwd", ctas,
              sum[7], mx_items);
      for (int k = 0; k < 7; ++k) fprintf(stderr, " %s %.1f", names[k], sum[k] * 1e-3 / ctas);
      fprintf(stderr, "\n");
    }
  }
  float total = 0.f;
  for (int i = 1; i < tl.n; ++i) {
    float ms = 0.f;
    cudaEventElapsedTime(&ms, tl.ev[i - 1], tl.ev[i]);
    fprintf(stderr, "[timeline] %-14s %8.1f us\n", tl.name[i], ms * 1e3f);
    total += ms;
  }
  fprintf(stderr, "[timeline] %-14s %8.1f us\n", "total", total * 1e3f);
  for (int i = 0; i < Timeline::kMax; ++i) cudaEventDestroy(tl.ev[i]);
  return 0;
}

// Stand-alone batched GEMM through the same kernel (unit tests and the DMMA micro-benchmark):
// C[b] = op(A[b]) op(B[b]) (+ C[b]) for `batch` square n x n matrices (n a multiple of 80),
// consecutive in memory.  `desc` is a device scratch of cherry_gemm_desc_bytes(batch) bytes;
// `partial` is needed only when ksplit > 1 (batch * ksplit * n * n doubles).  The descriptor
// upload is synchronous; the launch itself is asynchronous on `stream`.
int gemm_f64_batched(const double* A, const double* B, double* C, int n, int batch, int ta, int tb,
                     int accumulate, int ksplit, void* desc, double* partial, cudaStream_t stream) {
  if (!A || !B || !C || !desc) return fail(CHERRY_EINVAL, "gemm: null pointer argument");
  if (n <= 0 || n % BT != 0 || batch <= 0 || ksplit < 1) return fail(CHERRY_EINVAL, "gemm: n must be a positive multiple of %d", BT);
  if (ksplit > 1 && !partial) return fail(CHERRY_EINVAL, "gemm: split-K needs a partial buffer");
  int rc = ensure_gemm_attr();
  if (rc) return rc;
  std::vector<GemmTask> tasks(batch);
  std::vector<GemmTerm> terms(batch);
  const size_t nn = (size_t)n * n;
  for (int b = 0; b < batch; ++b) {
    terms[b] = GemmTerm{A + b * nn, B + b * nn, ta, tb};
    tasks[b].C = C + b * nn; tasks[b].term_begin = b; tasks[b].n_terms = 1; tasks[b].accumulate = accumulate;
  }
  char* d = reinterpret_cast<char*>(desc);
  const size_t task_bytes = align256(sizeof(GemmTask) * batch);
  CHERRY_CUDA(cudaStreamSynchronize(stream));
  CHERRY_CUDA(cudaMemcpy(d, tasks.data(), sizeof(GemmTask) * batch, cudaMemcpyHostToDevice));
  CHERRY_CUDA(cudaMemcpy(d + task_bytes, terms.data(), sizeof(GemmTerm) * batch, cudaMemcpyHostToDevice));
  const GemmTask* dt = reinterpret_cast<const GemmTask*>(d);
  const GemmTerm* dm = reinterpret_cast<const GemmTerm*>(d + task_bytes);
  const size_t smem = (size_t)NSTAGE * 2 * TILE_ELEMS * sizeof(double);
  dim3 grid((n / BT) * (n / BT), batch, ksplit);
  gemm_tasks_kernel<<<grid, GEMM_THREADS, smem, stream>>>(dt, dm, n, ksplit, partial);
  CHERRY_LAUNCH_CHECK("gemm_tasks_kernel");
  if (ksplit > 1) {
    int bx = (int)((nn + EW_THREADS * 4 - 1) / (EW_THREADS * 4));
    splitk_reduce_kernel<<<dim3(bx, batch), EW_THREADS, 0, stream>>>(dt, ksplit, nn, partial);
    CHERRY_LAUNCH_CHECK("splitk_reduce_kernel");
  }
  return 0;
}

size_t gemm_desc_bytes(int batch) {
  return align256(sizeof(GemmTask) * (size_t)batch) + align256(sizeof(GemmTerm) * (size_t)batch);
}

// Host copy of the per-bucket squaring counts of the most recent evaluation (synchronises).
int fit_large_read_schedule(const cherry_fit_args& a, int* s_out, double* mu_out) {
  int rc = check_large(a);
  if (rc) return rc;
  const Plan& p = get_plan(a.S, a.K, nullptr);
  char* base = reinterpret_cast<char*>(a.workspace);
  CHERRY_CUDA(cudaDeviceSynchronize());
  CHERRY_CUDA(cudaMemcpy(s_out, base + p.off_s, sizeof(int) * a.K, cudaMemcpyDeviceToHost));
  if (mu_out) {
    LargeScalars sc;
    CHERRY_CUDA(cudaMemcpy(&sc, base + p.off_scalars, sizeof(sc), cudaMemcpyDeviceToHost));
    *mu_out = sc.mu;
  }
  return 0;
}

int fit_large_update(const cherry_fit_args& a, int mode, cudaStream_t stream, const double* reduced) {
  int rc = check_large(a);
  if (rc) return rc;
  const Plan& p = get_plan(a.S, a.K, nullptr);
  char* base = reinterpret_cast<char*>(a.workspace);
  if (mode == 0 && (rc = fit_large_prepare(a, stream))) return rc;
  LargeUpdateArgs u;
  fill_update_args(u, a, p, base);
  if (reduced) {  // gradient and loss already summed over the buckets of all ranks
    u.K = 1;
    u.G = reduced;
    u.loss_part = reduced + (size_t)a.S * a.S;
  }
  const size_t smem = sizeof(double) * a.S;
  if (mode == 1) {
    large_update_rows_kernel<<<a.S, EW_THREADS, smem, stream>>>(u);
    CHERRY_LAUNCH_CHECK("large_update_rows_kernel");
    const int n_theta = a.S + a.S * (a.S - 1) / 2;
    large_update_step_kernel<<<(n_theta + EW_THREADS - 1) / EW_THREADS, EW_THREADS, smem, stream>>>(u);
    CHERRY_LAUNCH_CHECK("large_update_step_kernel");
  }
  large_build_Q_kernel<<<a.S, EW_THREADS, smem, stream>>>(u, mode);
  CHERRY_LAUNCH_CHECK("large_build_Q_kernel");
  return 0;
}

}  // namespace cherry

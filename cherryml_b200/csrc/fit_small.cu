// Composite-likelihood fit for small state spaces (S <= 32: the 20x20 LG model, 21-state
// gap-augmented alphabets, per-site SiteRM batches, toy 3x3 cases).
//
// Two kernels per epoch:
//   expm_loss_grad_small   one CTA per (problem, time bucket): P = expm(t Q) by Taylor +
//                          scaling-and-squaring held in shared memory, loss_k = -<C_k, log P>,
//                          and the exact adjoint of the same algorithm back to t * dP/dQ.
//                          All S x S products run on the FP64 tensor pipe (DMMA m8n8k4).
//   fit_update_small       one CTA per problem: fixed-order reduction over buckets, loss
//                          trace, best-iterate / power-of-two snapshots, adjoint of Q(theta),
//                          Adam or SGD step, and Q(theta) for the next epoch.
//
// Replaces, in the reference (songlab-cal/CherryML v0.2.0): torch.matrix_exp + torch.log +
// sum + autograd backward + optimizer.step of train_quantization
// (estimation/_ratelearn/trainer.py:156-187), RateMatrix.forward (rate.py:167-188), and the
// batched per-site variant (_siterm/_cherryml_vectorized.py:264-293, 351-383).
#include "common.cuh"

#include "dmma.cuh"
#include "fit_common.cuh"

namespace {

using cherry::kMaxDegree;
using cherry::kMaxSquarings;

constexpr int kSmallThreads = 512;  // 16 warps: one 8x8 output tile per warp up to S = 32
constexpr int kMaxSmallS = 32;

// D = op(A) * op(B)  (+ D if ACC), all spad x spad with leading dimension ld, operands may
// live in shared or global memory (generic pointers).  Fragment layouts of m8n8k4:
//   A: lane -> (row = lane/4, k = lane%4);  B: (k = lane%4, col = lane/4);
//   C: (row = lane/4, cols = 2*(lane%4), +1).
// ld = spad + 4 makes all four access patterns bank-conflict free.
// Latency matters more than throughput here (a bucket is a dependent chain of ~50 tiny
// products): every warp owns one output tile, all operand fragments of the tile are loaded up
// front (independent loads), and the k-steps alternate between two accumulators to halve the
// DMMA dependency chain.
template <bool TA, bool TB, bool ACC, int NT, int NTL>
__device__ __forceinline__ void mm(double* D, const double* A, const double* B) {
  // NTL = tiles per side at compile time (spad = 8 NTL, ld = spad + 4): every offset below is an immediate
  // (round 2: with runtime nt / ld a product cost ~150 instructions per warp, two thirds of them address
  // arithmetic, and an LG epoch is a chain of ~45 such products per bucket)
  constexpr int nt = NTL, ld = 8 * NTL + 4, nsteps = 2 * NTL;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int g = lane >> 2, tg = lane & 3;
  for (int tile = warp; tile < nt * nt; tile += NT / 32) {
    const int r0 = (tile / nt) * 8, c0 = (tile % nt) * 8;
    double a[nsteps], b[nsteps];
    const double* Ap = TA ? A + tg * ld + r0 + g : A + (r0 + g) * ld + tg;
    const double* Bp = TB ? B + (c0 + g) * ld + tg : B + tg * ld + c0 + g;
#pragma unroll
    for (int st = 0; st < nsteps; ++st) {
      a[st] = TA ? Ap[st * 4 * ld] : Ap[st * 4];
      b[st] = TB ? Bp[st * 4] : Bp[st * 4 * ld];
    }
    double* out = D + (r0 + g) * ld + c0 + 2 * tg;
    double d0 = 0.0, d1 = 0.0, e0 = 0.0, e1 = 0.0;
    if (ACC) {
      d0 = out[0];
      d1 = out[1];
    }
#pragma unroll
    for (int st = 0; st < nsteps; st += 2) {
      dmma884(d0, d1, a[st], b[st]);
      dmma884(e0, e1, a[st + 1], b[st + 1]);
    }
    out[0] = d0 + e0;
    out[1] = d1 + e1;
  }
}

struct Slots {
  double* smem;
  double* spill;
  int n_smem;
  int slot_elems;
  __device__ __forceinline__ double* operator()(int i) const {
    return i < n_smem ? smem + (size_t)i * slot_elems : spill + (size_t)(i - n_smem) * slot_elems;
  }
};

template <int NT>
__device__ __forceinline__ double block_reduce_sum(double v, double* red) {
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  __syncthreads();
  if (lane == 0) red[warp] = v;
  __syncthreads();
  double t = 0.0;
  for (int w = 0; w < NT / 32; ++w) t += red[w];  // fixed order: deterministic
  return t;
}

template <int NT>
__device__ __forceinline__ double block_reduce_max(double v, double* red) {
  for (int o = 16; o > 0; o >>= 1) v = fmax(v, __shfl_xor_sync(0xffffffffu, v, o));
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  __syncthreads();
  if (lane == 0) red[warp] = v;
  __syncthreads();
  double t = red[0];
  for (int w = 1; w < NT / 32; ++w) t = fmax(t, red[w]);
  return t;
}

struct UpdateArgs {
  int S, K, n_problems, num_epochs_total;
  const double* mask;   // [S][S]
  double* theta;        // [P][S + S(S-1)/2]
  double* adam_m;
  double* adam_v;
  double* Q;            // [P][S][S]
  double* Q_best;       // [P][S][S]
  double* Q_last;       // [P][S][S]
  double* best_loss;    // [P]
  double* loss_trace;   // [num_epochs_total][P]
  double* snapshots;    // [n_snap][S][S] for problem 0 or null
  int n_snapshots;
  const double* dQ_part;    // [P*K][S][S]
  const double* loss_part;  // [P*K]
  const double* sumC;       // [P]
  int* epoch_counter;       // [P] device ints: epochs completed so far, per problem
  double lr_pi, lr_upper, beta1, beta2, eps;
  int do_adam, loss_normalization;
  int best_mode;  // 0: first epoch always becomes the best (trainer.py:179); 1: best starts at +inf
  int mode;       // 0: only theta -> Q; 1: full update
};

// The parameter update of one problem by one CTA of NT threads; `sm` = 4 S*S + 4 S doubles of shared memory,
// `red` = NT / 32 doubles, `sh_improved_p` = one shared int.  Called by fit_update_small (one CTA per problem)
// and, in training, by the CTA of expm_loss_grad_small that finishes a problem's last bucket.
template <int NT>
__device__ __forceinline__ void update_small_body(const UpdateArgs& a, int p, double* sm, double* red,
                                                  int* sh_improved_p) {
  int& sh_improved = *sh_improved_p;
  (void)red;  // the block reductions of this body became warp shuffles (S <= 32)
  const int tid = threadIdx.x, S = a.S, SS = S * S;
  const int n_upper = S * (S - 1) / 2, n_theta = S + n_upper;
  double* G = sm;             // dL/dQ
  double* sv = sm + SS;       // masked symmetric softplus
  double* sg = sm + 2 * SS;   // sigmoid(u) per (i<j), stored at [i][j]
  double* dM = sm + 3 * SS;
  double* pi = sm + 4 * SS;   // softmax(pi logits)
  double* rr = pi + S;        // sqrt(pi)
  double* dr = rr + S;
  double* dpi = dr + S;
  double* theta = a.theta + (size_t)p * n_theta;
  double* Q = a.Q + (size_t)p * SS;
  const int epoch = a.epoch_counter[p];

  if (a.mode == 1) {
    // ---- reduce the per-bucket pieces in bucket order
    const double scale = a.loss_normalization ? 1.0 / a.sumC[p] : 1.0;
    for (int e = tid; e < SS; e += NT) {
      // loads of 20 buckets in flight (the reduction is L2-latency bound: K / 20 round trips), added in bucket
      // order (same result as a plain loop)
      double acc = 0.0;
      const double* src = a.dQ_part + (size_t)p * a.K * SS + e;
      for (int k0 = 0; k0 < a.K; k0 += 20) {
        double v[20];
#pragma unroll
        for (int j = 0; j < 20; ++j) v[j] = (k0 + j < a.K) ? __ldcg(src + (size_t)(k0 + j) * SS) : 0.0;
#pragma unroll
        for (int j = 0; j < 20; ++j) acc += v[j];
      }
      G[e] = acc * scale;
    }
    // stage the per-bucket losses in shared memory (parallel loads), then add them in order
    for (int k = tid; k < a.K && k < SS; k += NT) sv[k] = __ldcg(a.loss_part + (size_t)p * a.K + k);
    __syncthreads();
    double lp = 0.0;
    if (tid == 0) {
      for (int k = 0; k < a.K; ++k) lp += (k < SS) ? sv[k] : __ldcg(a.loss_part + (size_t)p * a.K + k);
      lp *= scale;
      if (epoch < a.num_epochs_total) a.loss_trace[(size_t)epoch * a.n_problems + p] = lp;
      const double best = a.best_loss[p];
      // trainer.py:179 (`best_loss is None or loss < best_loss`) vs the per-site variant that
      // starts from best = +inf (_cherryml_vectorized.py:341, 366)
      const int improved = (epoch == 0 && a.best_mode == 0) ? 1 : (lp < best);
      if (improved) a.best_loss[p] = lp;
      sh_improved = improved;
    }
    __syncthreads();
    // ---- best iterate and power-of-two snapshots of the Q this loss belongs to
    const bool snap = (p == 0) && a.snapshots && ((epoch & (epoch + 1)) == 0);
    int snap_idx = 0;
    if (snap) {
      int e1 = epoch + 1;
      while (e1 > 1) { e1 >>= 1; ++snap_idx; }
    }
    for (int e = tid; e < SS; e += NT) {
      const double q = Q[e];
      if (sh_improved) a.Q_best[(size_t)p * SS + e] = q;
      a.Q_last[(size_t)p * SS + e] = q;
      if (snap && snap_idx < a.n_snapshots) a.snapshots[(size_t)snap_idx * SS + e] = q;
    }
  }
  // ---- softmax(pi logits), sqrt: S <= 32, so warp 0 does it with shuffles (one block barrier instead of five)
  auto softmax_to_shared = [&]() {
    if (tid < 32) {
      const double th = tid < S ? theta[tid] : -INFINITY;
      double mx = th;
      for (int o = 16; o > 0; o >>= 1) mx = fmax(mx, __shfl_xor_sync(0xffffffffu, mx, o));
      const double ex = tid < S ? exp(th - mx) : 0.0;
      double se = ex;
      for (int o = 16; o > 0; o >>= 1) se += __shfl_xor_sync(0xffffffffu, se, o);
      if (tid < S) {
        pi[tid] = ex / se;
        rr[tid] = sqrt(ex / se);
      }
    }
    __syncthreads();
  };
  softmax_to_shared();
  if (a.mode == 1) {
    // ---- adjoint of Q = M - diag(rowsum M), M_ij = s_ij r_j / r_i
    for (int e = tid; e < SS; e += NT) {
      const int i = e / S, j = e - i * S;
      double sval = 0.0, sig = 0.0;
      if (i != j) {
        const int lo = i < j ? i : j, hi = i < j ? j : i;
        const double u = theta[S + cherry::triu_index(lo, hi, S)];
        sval = a.mask[e] * cherry::softplus_d(u);
        sig = cherry::softplus_grad_d(u);
      }
      sv[e] = sval;
      sg[e] = sig;
      dM[e] = (i != j) ? (G[e] - G[i * S + i]) : 0.0;
    }
    __syncthreads();
    // dL/dr_i = sum_j dM_ji s_ji / r_j  -  sum_j dM_ij s_ij r_j / r_i^2
    for (int i = tid; i < S; i += NT) {
      double col = 0.0, row = 0.0;
      for (int j = 0; j < S; ++j) {
        col += dM[j * S + i] * sv[j * S + i] / rr[j];
        row += dM[i * S + j] * sv[i * S + j] * rr[j];
      }
      dr[i] = col - row / (rr[i] * rr[i]);
      dpi[i] = dr[i] / (2.0 * rr[i]);
    }
    __syncthreads();
    // every warp forms the dot product itself (S <= 32 terms, same order in every warp): no block barrier
    double dot = (tid & 31) < S ? pi[tid & 31] * dpi[tid & 31] : 0.0;
    for (int o = 16; o > 0; o >>= 1) dot += __shfl_xor_sync(0xffffffffu, dot, o);
    const int step = epoch + 1;
    const double bc1 = 1.0 - pow(a.beta1, (double)step);
    const double bc2s = sqrt(1.0 - pow(a.beta2, (double)step));
    double* am = a.adam_m + (size_t)p * n_theta;
    double* av = a.adam_v + (size_t)p * n_theta;
    // upper-diagonal parameters (before the pi logits change: their gradient uses the old r)
    for (int e = tid; e < SS; e += NT) {
      const int i = e / S, j = e - i * S;
      if (i < j) {
        const double ds_ij = dM[e] * rr[j] / rr[i], ds_ji = dM[j * S + i] * rr[i] / rr[j];
        const double g = sg[e] * (a.mask[e] * ds_ij + a.mask[j * S + i] * ds_ji);
        const int idx = S + cherry::triu_index(i, j, S);
        cherry::optimizer_step(theta[idx], am[idx], av[idx], g, a.lr_upper, a.do_adam, a.beta1,
                               a.beta2, a.eps, bc1, bc2s);
      }
    }
    for (int i = tid; i < S; i += NT) {
      const double g = pi[i] * (dpi[i] - dot);
      cherry::optimizer_step(theta[i], am[i], av[i], g, a.lr_pi, a.do_adam, a.beta1, a.beta2, a.eps,
                             bc1, bc2s);
    }
    __syncthreads();
    // ---- new softmax for the next epoch's Q
    softmax_to_shared();
  }
  // ---- Q(theta): off-diagonal M, then the diagonal from the row sums (fixed order)
  for (int e = tid; e < SS; e += NT) {
    const int i = e / S, j = e - i * S;
    double val = 0.0;
    if (i != j) {
      const int lo = i < j ? i : j, hi = i < j ? j : i;
      const double u = theta[S + cherry::triu_index(lo, hi, S)];
      val = a.mask[e] * cherry::softplus_d(u) * rr[j] / rr[i];
    }
    G[e] = val;  // reuse as M
  }
  __syncthreads();
  for (int e = tid; e < SS; e += NT) {
    const int i = e / S, j = e - i * S;
    if (i == j) {
      double rs = 0.0;
      for (int k = 0; k < S; ++k) rs += G[i * S + k];
      Q[e] = -rs;
    } else {
      Q[e] = G[e];
    }
  }
  if (a.mode == 1 && tid == 0) a.epoch_counter[p] = epoch + 1;
}


// grid.x = n_problems * K.  Problem p = blockIdx.x / K owns Q[p], buckets (p, 0..K-1).
template <int NT, int MINB, int NTL>
__global__ void __launch_bounds__(NT, MINB)
expm_loss_grad_small(const double* __restrict__ Qall, const double* __restrict__ tall,
                     const double* __restrict__ Call, int S, int K, int n_smem_slots,
                     double* __restrict__ spill_all, int spill_slots, double* __restrict__ dQ_part,
                     double* __restrict__ loss_part, int* __restrict__ overflow_flag,
                     double* __restrict__ P_out, UpdateArgs ua, int* __restrict__ arrive) {
  // arrive != nullptr (training): the CTA that finishes a problem's LAST bucket runs the parameter update of
  // that problem right here (update_small_body) instead of a second launch -- one kernel per epoch
  extern __shared__ double smem[];
  __shared__ double red[NT / 32];
  __shared__ int sh_m, sh_s, sh_last, sh_improved;
  const int tid = threadIdx.x;
  const int b = blockIdx.x, prob = b / K;
  constexpr int nt = NTL, spad = nt * 8, ld = spad + 4, slot_elems = spad * ld;  // host: NTL == (S + 7) / 8
  const double* __restrict__ Q = Qall + (size_t)prob * S * S;
  const double* __restrict__ C = Call + (size_t)b * S * S;
  const double t = tall[b];
  Slots slot{smem, spill_all + (size_t)b * spill_slots * slot_elems, n_smem_slots, slot_elems};

  // ---- ||tQ||_1 (max column abs sum), degree and scaling
  double colsum = 0.0;
  if (tid < S)
    for (int i = 0; i < S; ++i) colsum += fabs(Q[i * S + tid]);
  const double norm = fabs(t) * block_reduce_max<NT>(colsum, red);
  if (tid == 0) {
    int m, s;
    // beyond 30 squarings: report it (status 2, as the large path does) and go on with s = 30
    if (!cherry::choose_degree(norm, m, s)) atomicExch(overflow_flag, 2);
    sh_m = m;
    sh_s = s;
  }
  __syncthreads();
  const int m = sh_m, s = sh_s;
  const double tau = ldexp(t, -s);
  // slot plan: 0 = B, 1..m-1 = H_1..H_{m-1}, m..m+s = X_0..X_s, then G0, G1, Bbar
  const int sB = 0, sH = 0 /* H_j at slot j, j>=1 */, sX = m, sG0 = m + s + 1, sG1 = m + s + 2,
            sBbar = m + s + 3;
  (void)sH;
  if (sBbar >= n_smem_slots + spill_slots) {  // cannot happen with the host-side sizing; be loud
    if (tid == 0) {
      atomicExch(overflow_flag, 1);
      loss_part[b] = nan("");
    }
    for (int e = tid; e < S * S; e += NT) dQ_part[(size_t)b * S * S + e] = nan("");
    return;
  }
  double* Bm = slot(sB);
  for (int e = tid; e < slot_elems; e += NT) {
    const int i = e / ld, j = e - i * ld;
    Bm[e] = (i < S && j < S) ? tau * Q[i * S + j] : 0.0;
  }
  __syncthreads();

  // ---- Horner: H_m = c_m I, H_j = c_j I + B H_{j+1}; X_0 = H_0
  // H_{m-1} = c_{m-1} I + c_m B needs no product.
  {
    double* H = (m - 1 >= 1) ? slot(m - 1) : slot(sX);  // m == 1: H_0 = X_0 = I + B
    const double cm = cherry::inv_factorial(m), cm1 = cherry::inv_factorial(m - 1);
    for (int e = tid; e < slot_elems; e += NT) {
      const int i = e / ld, j = e - i * ld;
      H[e] = cm * Bm[e] + ((i == j && i < S) ? cm1 : 0.0);
    }
    __syncthreads();
    for (int j = m - 2; j >= 0; --j) {
      double* Hj = (j >= 1) ? slot(j) : slot(sX);
      mm<false, false, false, NT, NTL>(Hj, Bm, slot(j + 1));
      __syncthreads();
      const double cj = cherry::inv_factorial(j);
      if (tid < S) Hj[tid * ld + tid] += cj;
      __syncthreads();
    }
  }
  // ---- squarings
  for (int i = 0; i < s; ++i) {
    mm<false, false, false, NT, NTL>(slot(sX + i + 1), slot(sX + i), slot(sX + i));
    __syncthreads();
  }
  double* P = slot(sX + s);
  if (P_out != nullptr) {  // forward only: hand back expm(t Q)
    for (int e = tid; e < S * S; e += NT) {
      const int i = e / S, j = e - i * S;
      P_out[(size_t)b * S * S + e] = P[i * ld + j];
    }
    return;
  }
  // ---- loss and dL/dP (unnormalised): loss_k = -sum C log P, G = -C / P, skipping C == 0
  double* G = slot(sG0);
  double part = 0.0;
  for (int e = tid; e < slot_elems; e += NT) {
    const int i = e / ld, j = e - i * ld;
    double gval = 0.0;
    if (i < S && j < S) {
      const double c = C[i * S + j];
      if (c != 0.0) {
        const double p = P[e];
        part -= c * log(p);
        gval = -c / p;
      }
    }
    G[e] = gval;
  }
  const double loss_k = block_reduce_sum<NT>(part, red);
  if (tid == 0) loss_part[b] = loss_k;
  __syncthreads();
  // ---- adjoint of the squarings: Xbar_i = Xbar_{i+1} X_i^T + X_i^T Xbar_{i+1}
  int gcur = sG0, gnext = sG1;
  for (int i = s - 1; i >= 0; --i) {
    mm<false, true, false, NT, NTL>(slot(gnext), slot(gcur), slot(sX + i));
    __syncthreads();
    mm<true, false, true, NT, NTL>(slot(gnext), slot(sX + i), slot(gcur));
    __syncthreads();
    const int tmp = gcur;
    gcur = gnext;
    gnext = tmp;
  }
  // ---- adjoint of Horner: Bbar += Hbar_j H_{j+1}^T, Hbar_{j+1} = B^T Hbar_j; last term c_m Hbar_{m-1}
  double* Bbar = slot(sBbar);
  for (int e = tid; e < slot_elems; e += NT) Bbar[e] = 0.0;
  __syncthreads();
  for (int j = 0; j <= m - 2; ++j) {
    mm<false, true, true, NT, NTL>(Bbar, slot(gcur), slot(j + 1));
    mm<true, false, false, NT, NTL>(slot(gnext), Bm, slot(gcur));
    __syncthreads();
    const int tmp = gcur;
    gcur = gnext;
    gnext = tmp;
  }
  {
    const double cm = cherry::inv_factorial(m);
    const double* Hbar = slot(gcur);
    double* out = dQ_part + (size_t)b * S * S;
    for (int e = tid; e < S * S; e += NT) {
      const int i = e / S, j = e - i * S;
      out[e] = tau * (Bbar[i * ld + j] + cm * Hbar[i * ld + j]);
    }
  }
  if (arrive == nullptr) return;
  // ---- fused update: last arriver of the problem (every CTA of the problem gets here: the early exits above
  // are the forward-only call and an error that is reported through overflow_flag)
  __threadfence();  // this bucket's gradient and loss are visible before the ticket
  __syncthreads();
  if (tid == 0) {
    const int old = atomicAdd(arrive + prob, 1);
    sh_last = (old == K - 1);
    if (sh_last) arrive[prob] = 0;  // ready for the next epoch
  }
  __syncthreads();
  if (!sh_last) return;
  __threadfence();
  update_small_body<NT>(ua, prob, smem, red, &sh_improved);
}


// grid.x = n_problems; one CTA handles one problem.  Dynamic smem: 4 S*S + 4 S doubles.
__global__ void __launch_bounds__(kSmallThreads) fit_update_small(UpdateArgs a) {
  extern __shared__ double sm[];
  __shared__ double red[kSmallThreads / 32];
  __shared__ int sh_improved;
  update_small_body<kSmallThreads>(a, blockIdx.x, sm, red, &sh_improved);
}

}  // namespace

namespace cherry {

// Two launch shapes.  Latency shape (grid <= SMs, or S > 24): 512 threads, up to 40 resident matrix slots,
// one CTA per SM -- a bucket is a dependent chain of ~50 tiny products and the whole grid is one wave.
// Throughput shape (grid > SMs and S <= 24, e.g. the batched per-site fits: 331 sites x 4 buckets): 288
// threads (one warp per 8x8 output tile of a 24x24 matrix), <= 113 registers and 20 resident slots, so that
// TWO CTAs share an SM; slots beyond the resident ones live in the global workspace (sized for the worst
// case in both shapes, so the caller's workspace does not depend on the shape).
constexpr int kThroughputThreads = 288, kThroughputSlots = 20;
static bool throughput_shape(int S, int grid) { return S <= 24 && grid > sm_count(); }

int fit_small_workspace(int S, int* n_smem_slots, int* spill_slots, size_t* slot_bytes,
                        size_t* smem_bytes, int grid) {
  if (S <= 0 || S > kMaxSmallS) return fail(CHERRY_ELIMIT, "fit_small: S=%d outside 1..%d", S, kMaxSmallS);
  const int nt = (S + 7) / 8, spad = nt * 8, ld = spad + 4;
  const size_t sb = (size_t)spad * ld * sizeof(double);
  const size_t budget = 220 * 1024;
  const int total_needed = kMaxDegree + kMaxSquarings + 4;  // m + s_max + 4 slots
  int ns = (int)(budget / sb);
  if (ns > total_needed) ns = total_needed;
  // the workspace is sized for the shape with the fewest resident slots that this S can take
  int ns_min = ns;
  if (S <= 24 && ns_min > kThroughputSlots) ns_min = kThroughputSlots;
  if (grid >= 0 && throughput_shape(S, grid) && ns > kThroughputSlots) ns = kThroughputSlots;
  if (n_smem_slots) *n_smem_slots = ns;
  if (spill_slots) *spill_slots = total_needed - ns_min;
  if (slot_bytes) *slot_bytes = sb;
  if (smem_bytes) *smem_bytes = (size_t)ns * sb;
  return 0;
}

static UpdateArgs make_update_args(const cherry_fit_args& f, int mode, const double* reduced) {
  UpdateArgs a;
  a.S = f.S; a.K = f.K; a.n_problems = f.n_problems; a.num_epochs_total = f.loss_trace_epochs;
  a.mask = f.mask; a.theta = f.theta; a.adam_m = f.adam_m; a.adam_v = f.adam_v; a.Q = f.Q;
  a.Q_best = f.Q_best; a.Q_last = f.Q_last; a.best_loss = f.best_loss; a.loss_trace = f.loss_trace;
  a.snapshots = f.snapshots; a.n_snapshots = f.n_snapshots; a.dQ_part = f.dQ_part;
  a.loss_part = f.loss_part; a.sumC = f.sumC; a.epoch_counter = f.epoch_counter;
  a.lr_pi = f.lr_pi; a.lr_upper = f.lr_upper; a.beta1 = f.beta1; a.beta2 = f.beta2; a.eps = f.eps;
  a.do_adam = f.do_adam; a.loss_normalization = f.loss_normalization; a.best_mode = f.best_mode;
  a.mode = mode;
  if (reduced) {  // one pre-reduced piece per problem
    a.K = 1;
    a.dQ_part = reduced;
    a.loss_part = reduced + (size_t)f.n_problems * f.S * f.S;
  }
  return a;
}

// bytes of the spill area; the per-problem arrival counters of the fused update follow it (256-byte aligned)
static size_t small_spill_bytes(int sp, size_t sb, int n_problems, int K) {
  return ((size_t)sp * sb * n_problems * K + 255) / 256 * 256;
}

size_t fit_small_workspace_bytes(int S, int K, int n_problems) {
  int ns = 0, sp = 0;
  size_t sb = 0, smem = 0;
  if (fit_small_workspace(S, &ns, &sp, &sb, &smem, -1)) return 0;
  return small_spill_bytes(sp, sb, n_problems, K) + sizeof(int) * (size_t)n_problems + 256;
}

// fuse_update: training epoch -- the last CTA of every problem runs the parameter update (no second launch)
int fit_small_expm(const cherry_fit_args& a, cudaStream_t stream, double* P_out, bool fuse_update) {
  int ns = 0, sp = 0;
  size_t sb = 0, smem = 0;
  const int grid = a.n_problems * a.K;
  int rc = fit_small_workspace(a.S, &ns, &sp, &sb, &smem, grid);
  if (rc) return rc;
  const size_t need = fit_small_workspace_bytes(a.S, a.K, a.n_problems);
  if (!a.workspace || a.workspace_bytes < need)
    return fail(CHERRY_EINVAL, "fit: workspace of %zu bytes required, got %zu", need, a.workspace_bytes);
  const UpdateArgs ua = make_update_args(a, 1, nullptr);
  int* arrive = fuse_update ? reinterpret_cast<int*>(reinterpret_cast<char*>(a.workspace) +
                                                     small_spill_bytes(sp, sb, a.n_problems, a.K))
                            : nullptr;
  // the update body needs 4 S*S + 4 S doubles of the dynamic shared memory
  const size_t upd_smem = (size_t)(4 * a.S * a.S + 4 * a.S) * sizeof(double);
  if (smem < upd_smem) smem = upd_smem;
  const bool tp = throughput_shape(a.S, grid);
  const int ntl = (a.S + 7) / 8;  // tiles per side: a template parameter of the kernel
  // one instantiation per (shape, tiles per side); the attribute is set on first use per device
  static bool attr_set[64][2][5] = {};
  int dev = 0;
  CHERRY_CUDA(cudaGetDevice(&dev));
#define CHERRY_SMALL_LAUNCH(NTH, MINB, NTL_)                                                                     \
  do {                                                                                                           \
    if (dev < 64 && !attr_set[dev][MINB - 1][NTL_]) {                                                            \
      CHERRY_CUDA(cudaFuncSetAttribute(expm_loss_grad_small<NTH, MINB, NTL_>,                                    \
                                       cudaFuncAttributeMaxDynamicSharedMemorySize,                              \
                                       MINB == 1 ? 226 * 1024 : 112 * 1024));                                    \
      attr_set[dev][MINB - 1][NTL_] = true;                                                                      \
    }                                                                                                            \
    expm_loss_grad_small<NTH, MINB, NTL_><<<grid, NTH, smem, stream>>>(                                          \
        a.Q, a.t, a.C, a.S, a.K, ns, reinterpret_cast<double*>(a.workspace), sp, a.dQ_part, a.loss_part,        \
        a.status_flag, P_out, ua, arrive);                                                                       \
  } while (0)
  if (tp) {  // S <= 24
    if (ntl == 1) CHERRY_SMALL_LAUNCH(kThroughputThreads, 2, 1);
    else if (ntl == 2) CHERRY_SMALL_LAUNCH(kThroughputThreads, 2, 2);
    else CHERRY_SMALL_LAUNCH(kThroughputThreads, 2, 3);
  } else {
    if (ntl == 1) CHERRY_SMALL_LAUNCH(kSmallThreads, 1, 1);
    else if (ntl == 2) CHERRY_SMALL_LAUNCH(kSmallThreads, 1, 2);
    else if (ntl == 3) CHERRY_SMALL_LAUNCH(kSmallThreads, 1, 3);
    else CHERRY_SMALL_LAUNCH(kSmallThreads, 1, 4);
  }
#undef CHERRY_SMALL_LAUNCH
  CHERRY_LAUNCH_CHECK("expm_loss_grad_small");
  return 0;
}

int fit_small_update(const cherry_fit_args& f, int mode, cudaStream_t stream, const double* reduced) {
  const UpdateArgs a = make_update_args(f, mode, reduced);
  if (mode == 0 && f.workspace) {  // initialisation: the fused update's arrival counters start at zero
    int ns = 0, sp = 0;
    size_t sb = 0, smem_unused = 0;
    int rc = fit_small_workspace(f.S, &ns, &sp, &sb, &smem_unused, -1);
    if (rc) return rc;
    if (f.workspace_bytes >= fit_small_workspace_bytes(f.S, f.K, f.n_problems))
      CHERRY_CUDA(cudaMemsetAsync(reinterpret_cast<char*>(f.workspace) + small_spill_bytes(sp, sb, f.n_problems, f.K), 0,
                                  sizeof(int) * (size_t)f.n_problems, stream));
  }
  const size_t smem = (size_t)(4 * f.S * f.S + 4 * f.S) * sizeof(double);
  fit_update_small<<<f.n_problems, kSmallThreads, smem, stream>>>(a);
  CHERRY_LAUNCH_CHECK("fit_update_small");
  return 0;
}

}  // namespace cherry

// Tree log-likelihood by Felsenstein pruning in log space, one launch per (tree, model).
//
// Replaces the dynamic programme of dp_likelihood_computation, reference
// cherryml/evaluation/_likelihood.py:239-326.  A "unit" is an independently evolving site
// (c = 1, Su = S states) or a pair of contacting sites (c = 2, Su = S*S states, state index
// S*i + j).  Thread (g, s) of a CTA owns state s of the CTA's g-th unit and walks the tree in
// post-order; the running sum of child messages of the open node at depth d lives in
// acc[d][g][s], which only that thread touches, so the children of a node are accumulated in
// the reference's order (tree.children order) without synchronisation.  The message of child v:
//     log(max(0, sum_s' P_v[s][s'] * exp(dp_v[s'] - max dp_v) * obs_v[s'])) + max dp_v
// with P_v = expm(branch length * site rate * Q), computed beforehand by cherry_expm_batched and
// handed over TRANSPOSED (Pt[k][s] = P[s][k], cherry_tree_ll_transpose): thread s walks column s
// of Pt, so a warp reads 32 consecutive doubles per step of the dot product instead of 32
// different rows; the sum over k keeps its order.
#include <cstdint>
#include <vector>

#include "common.cuh"

namespace {

struct LlArgs {
  const cherry_ll_node* nodes;
  const int32_t* p_index;  // [n_nodes][n_cats]
  const double* P;         // [n_matrices][Su][Su], transposed: P[m][k][s] = expm(...)[s][k]
  const uint8_t* obs;      // [n_leaves][n_units][c]
  const int32_t* unit_cat; // [n_units]
  const double* pi;        // [Su]
  double* acc;             // [gridDim.x][max_depth + 1][G][Su]
  double* ll_out;          // [n_units]
  int n_nodes, n_cats, S, c, Su, n_units, G, max_depth, staged;
};

constexpr int kLlBatch = 16;

// one commit group: entries k0 .. k0+15 of this thread's column -> its slots of staging buffer `buf`
__device__ __forceinline__ void ll_stage_batch(uint32_t stage_u32, uint32_t slot_stride, const double* col, int Su,
                                               int k0, int buf) {
#pragma unroll
  for (int j = 0; j < kLlBatch; ++j)
    if (k0 + j < Su)
      asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(stage_u32 + (uint32_t)(buf * kLlBatch + j) * slot_stride),
                   "l"(col + (size_t)(k0 + j) * Su)
                   : "memory");
  asm volatile("cp.async.commit_group;" ::: "memory");
}

__device__ __forceinline__ void tree_ll_body(const LlArgs& a) {
  extern __shared__ double w[];  // [G][Su], then [G][32] partial maxima, then (Su > 64) the staging slots
  double* red = w + (size_t)a.G * a.Su;
  double* stage = red + (size_t)a.G * 32 + threadIdx.x;  // [2][kLlBatch][blockDim.x], this thread's column
  const uint32_t stage_u32 = (uint32_t)__cvta_generic_to_shared(stage);
  const uint32_t slot_stride = blockDim.x * (uint32_t)sizeof(double);
  const int Su = a.Su, S = a.S;
  const int g = threadIdx.x / Su, s = threadIdx.x - g * Su;
  const int u = blockIdx.x * a.G + g;
  const bool live = g < a.G && u < a.n_units;
  const int cat = live ? a.unit_cat[u] : 0;
  double* acc = a.acc + ((size_t)blockIdx.x * (a.max_depth + 1) * a.G + (live ? g : 0)) * Su + s;
  const size_t acc_stride = (size_t)a.G * Su;
  double* wg = w + (live ? g : 0) * Su;
  for (int i = 0; i < a.n_nodes; ++i) {
    const cherry_ll_node node = a.nodes[i];
    const bool is_leaf = node.flags & 1;
    const bool is_root = i == a.n_nodes - 1;
    // column s of the edge's matrix; the index does not depend on the running sums, so its load
    // overlaps the reduction below
    const double* col = a.P + (is_root || !live ? 0 : (size_t)a.p_index[(size_t)i * a.n_cats + cat] * Su * Su) + s;
    double m = 0.0;
    if (a.staged && live && !is_leaf && !is_root) {
      ll_stage_batch(stage_u32, slot_stride, col, Su, 0, 0);
      ll_stage_batch(stage_u32, slot_stride, col, Su, kLlBatch, 1);
    }
    if (!is_leaf) {
      // dp of this node is complete: w = exp(dp - max dp) (observation vector of an internal node = ones)
      const double v = live ? acc[(size_t)node.depth * acc_stride] : 0.0;
      if (live) wg[s] = v;
      __syncthreads();
      double mx = -INFINITY;
      if (Su > 64) {
        // two-stage maximum: 32 strided partial maxima per unit, then everyone reads those
        if (live && s < 32) {
          double r = wg[s];
          for (int k = s + 32; k < Su; k += 32) r = fmax(r, wg[k]);
          red[g * 32 + s] = r;
        }
        __syncthreads();
        if (live)
          for (int k = 0; k < 32; ++k) mx = fmax(mx, red[g * 32 + k]);
      } else {
        if (live)
          for (int k = 0; k < Su; ++k) mx = fmax(mx, wg[k]);
        __syncthreads();
      }
      if (live) wg[s] = exp(v - mx);
      __syncthreads();
      if (live) {
        double sum = 0.0;
        if (is_root) {
          if (s == 0) {
            for (int k = 0; k < Su; ++k) sum += a.pi[k] * wg[k];
            a.ll_out[u] = log(fmax(sum, 0.0)) + mx;
          }
        } else {
          if (a.staged) {
            // Two batches of 16 column entries in flight per thread through cp.async (a warp's
            // 256-byte segments come from L2 every time: the matrices of one tree do not fit in
            // L1, so the loop is bound by how many bytes are outstanding); every thread stages
            // and consumes its own slots, and the sum keeps its order in k.
            // (the first two batches were issued at the top of the node, before the reduction)
            const int nb = (Su + kLlBatch - 1) / kLlBatch;
            for (int b = 0; b < nb; ++b) {
              if (b + 1 < nb) {
                asm volatile("cp.async.wait_group 1;" ::: "memory");
              } else {
                asm volatile("cp.async.wait_group 0;" ::: "memory");
              }
              const int k0 = b * kLlBatch;
              const double* mine = stage + (size_t)(b & 1) * kLlBatch * blockDim.x;
#pragma unroll
              for (int j = 0; j < kLlBatch; ++j)
                if (k0 + j < Su) sum += mine[(size_t)j * blockDim.x] * wg[k0 + j];
              if (b + 2 < nb) ll_stage_batch(stage_u32, slot_stride, col, Su, k0 + 2 * kLlBatch, b & 1);
            }
          } else {
            for (int k = 0; k < Su; ++k) sum += col[(size_t)k * Su] * wg[k];
          }
          m = log(fmax(sum, 0.0)) + mx;
        }
      }
      __syncthreads();
    } else if (live) {
      // leaf: dp = 0, observation = one-hot, or every state compatible with the known residues
      const uint8_t* ob = a.obs + ((size_t)node.obs_row * a.n_units + u) * a.c;
      double sum = 0.0;
      if (is_root) {  // a single-node tree
        if (s == 0) {
          if (a.c == 1) {
            const int x = ob[0];
            for (int k = 0; k < Su; ++k) sum += (x == S || x == k) ? a.pi[k] : 0.0;
          } else {
            const int x = ob[0], y = ob[1];
            for (int k = 0; k < Su; ++k) sum += ((x == S || x == k / S) && (y == S || y == k % S)) ? a.pi[k] : 0.0;
          }
          a.ll_out[u] = log(fmax(sum, 0.0));
        }
      } else {
        if (a.c == 1) {
          const int x = ob[0];
          if (x != S) {
            sum = col[(size_t)x * Su];
          } else {
            for (int k = 0; k < Su; ++k) sum += col[(size_t)k * Su];
          }
        } else {
          const int x = ob[0], y = ob[1];
          if (x != S && y != S) {
            sum = col[(size_t)(x * S + y) * Su];
          } else if (x != S) {
            for (int k = 0; k < S; ++k) sum += col[(size_t)(x * S + k) * Su];
          } else if (y != S) {
            for (int k = 0; k < S; ++k) sum += col[(size_t)(k * S + y) * Su];
          } else {
            for (int k = 0; k < Su; ++k) sum += col[(size_t)k * Su];
          }
        }
        m = log(fmax(sum, 0.0));
      }
    }
    if (live && !is_root) {
      double* dst = acc + (size_t)(node.depth - 1) * acc_stride;
      *dst = (node.flags & 2) ? m : *dst + m;
    }
  }
}

__global__ void tree_ll_kernel(LlArgs a) { tree_ll_body(a); }

// The same pass for CTAs beyond tree_ll_kernel's register budget: it takes 96 registers a thread, so 64 K
// registers hold 672 threads, fewer than the G * Su of a pair model with S >= 26 (Su >= 676).  Held to 64
// registers, it launches up to 1024 threads.
__global__ void __launch_bounds__(1024) tree_ll_wide_kernel(LlArgs a) { tree_ll_body(a); }

// out[m][k][s] = in[m][s][k], 32 x 32 tiles through shared memory (both sides coalesced)
__global__ void transpose_matrices_kernel(const double* __restrict__ in, double* __restrict__ out, int Su) {
  __shared__ double tile[32][33];
  const size_t base = (size_t)blockIdx.z * Su * Su;
  const int c0 = blockIdx.x * 32, r0 = blockIdx.y * 32;
  for (int j = threadIdx.y; j < 32; j += blockDim.y) {
    const int r = r0 + j, c = c0 + threadIdx.x;
    if (r < Su && c < Su) tile[j][threadIdx.x] = in[base + (size_t)r * Su + c];
  }
  __syncthreads();
  for (int j = threadIdx.y; j < 32; j += blockDim.y) {
    const int r = c0 + j, c = r0 + threadIdx.x;
    if (r < Su && c < Su) out[base + (size_t)r * Su + c] = tile[threadIdx.x][j];
  }
}

// ---------------------------------------------------------------- edge posteriors (c = 1, S <= 32)
//
// Inside/outside pruning for the exact gradient of the log-likelihood.  The CTAs of one launch
// each hold G units of ONE rate category (units sorted by category, the last CTA of a category
// padded with dead slots), so every edge has one matrix per CTA.  Three kernels:
//   post_fwd:    the forward pass of tree_ll_kernel (same thread mapping, same arithmetic in the
//                same order, so ll_out is bitwise the same), which also stores per node and unit
//                the inside vector dp_i, the message M_i to the parent, and the sum of the
//                messages of i's EARLIER siblings (the prefix; 0 for a first child);
//   post_bwd:    reverse post-order (a parent before its children, the children last to first);
//                the outside vector of child i of p is O_i = A_p + prefix_i + suffix_i, suffix_i
//                being the running sum of the messages of i's LATER siblings (a depth stack, like
//                acc of the forward), A_root = log pi, A_i(b) = log sum_a exp(O_i(a)) P_i[a][b].
//                No "total minus M_i": a -inf message (zero-length branch, P = I) would give
//                -inf - -inf.  Pr(parent = a, i = b | data_u) = exp(O_i(a)) P_i[a][b]
//                exp(dp_i(b)) obs_i(b) / L_u; the CTA sums its units in unit order and writes one
//                S x S partial per (CTA, edge), and the root posterior per CTA;
//   post_reduce: W[m] = sum over the (edge, category) pairs of matrix m in (edge, category)
//                order, and over the category's CTAs in CTA order.  No atomics: two runs give
//                bitwise-identical W and root posteriors.
// Edge derivatives (post_bwd<true> + dtau_reduce): with G_u[a][b] = d log L_u / d P[a][b] =
// exp(O_i(a)) exp(dp_i(b)) obs_i(b) / L_u and dP/dtau = QP for P = expm(tau Q),
//     d log L_u / d tau_i = sum_ab G_u[a][b] (QP)[a][b] = sc_u sum_s (Q^T eo_u)(s) (P ei_u)(s),
// two S-vector mat-vecs per unit and edge and no division by P (P = I is harmless).  The CTA sums
// its units in unit order into one scalar per (CTA, edge); dtau[i][k] sums the CTAs of category k
// in CTA order.
struct PostArgs {
  const cherry_ll_node* nodes;
  const int32_t* p_index;  // [n_nodes][n_cats]
  const double* P;         // [n_matrices][S][S], transposed as for tree_ll_kernel
  const uint8_t* obs;      // [n_leaves][n_units]
  const double* pi;        // [S]
  const int32_t* unit_of;  // [n_ctas][G]: unit of the slot, -1 for padding
  const int32_t* cta_cat;  // [n_ctas]
  const int32_t* cat_cta;  // [n_cats + 1]: CTAs of category k are cat_cta[k] .. cat_cta[k+1]-1
  const int32_t* m_off;    // [n_matrices + 1]
  const int32_t* m_ent;    // [(n_nodes - 1) * n_cats]: node * n_cats + category, grouped by matrix
  double* dp;              // [n_ctas][n_nodes][G][S]
  double* msg;             // [n_ctas][n_nodes][G][S]
  double* pre;             // [n_ctas][n_nodes][G][S]
  double* stk;             // [n_ctas][2][max_depth + 1][G][S]: forward acc / backward A, backward suffix
  double* part;            // [n_ctas][n_nodes][S][S]
  double* root_part;       // [n_ctas][S]
  double* ll_out;          // [n_units]
  double* W_out;           // [n_matrices][S][S]
  double* root_out;        // [S]
  const double* Q;         // [S][S], not transposed (edge derivatives only)
  double* dpart;           // [n_ctas][n_nodes] (edge derivatives only)
  double* dtau_out;        // [n_nodes][n_cats] (edge derivatives only)
  int n_nodes, n_cats, S, n_units, G, max_depth, n_matrices, n_ctas;
};

__global__ void tree_ll_post_fwd_kernel(PostArgs a) {
  extern __shared__ double w[];  // [G][S]
  const int S = a.S;
  const int g = threadIdx.x / S, s = threadIdx.x - g * S;
  const int u = g < a.G ? a.unit_of[blockIdx.x * a.G + g] : -1;
  const bool live = u >= 0;
  const int cat = a.cta_cat[blockIdx.x];
  const size_t gs = (size_t)a.G * S;
  const size_t mine = (live ? g : 0) * S + s;
  double* acc = a.stk + (size_t)blockIdx.x * 2 * (a.max_depth + 1) * gs + mine;
  double* dp = a.dp + (size_t)blockIdx.x * a.n_nodes * gs + mine;
  double* msg = a.msg + (size_t)blockIdx.x * a.n_nodes * gs + mine;
  double* pre = a.pre + (size_t)blockIdx.x * a.n_nodes * gs + mine;
  double* wg = w + (live ? g : 0) * S;
  for (int i = 0; i < a.n_nodes; ++i) {
    const cherry_ll_node node = a.nodes[i];
    const bool is_leaf = node.flags & 1;
    const bool is_root = i == a.n_nodes - 1;
    const double* col = a.P + (is_root || !live ? 0 : (size_t)a.p_index[(size_t)i * a.n_cats + cat] * S * S) + s;
    double m = 0.0;
    if (!is_leaf) {
      const double v = live ? acc[(size_t)node.depth * gs] : 0.0;
      if (live) {
        wg[s] = v;
        dp[(size_t)i * gs] = v;
      }
      __syncthreads();
      double mx = -INFINITY;
      if (live)
        for (int k = 0; k < S; ++k) mx = fmax(mx, wg[k]);
      __syncthreads();
      if (live) wg[s] = exp(v - mx);
      __syncthreads();
      if (live) {
        double sum = 0.0;
        if (is_root) {
          if (s == 0) {
            for (int k = 0; k < S; ++k) sum += a.pi[k] * wg[k];
            a.ll_out[u] = log(fmax(sum, 0.0)) + mx;
          }
        } else {
          for (int k = 0; k < S; ++k) sum += col[(size_t)k * S] * wg[k];
          m = log(fmax(sum, 0.0)) + mx;
        }
      }
      __syncthreads();
    } else if (live) {
      const int x = a.obs[(size_t)node.obs_row * a.n_units + u];
      double sum = 0.0;
      if (is_root) {
        if (s == 0) {
          for (int k = 0; k < S; ++k) sum += (x == S || x == k) ? a.pi[k] : 0.0;
          a.ll_out[u] = log(fmax(sum, 0.0));
        }
      } else {
        if (x != S) {
          sum = col[(size_t)x * S];
        } else {
          for (int k = 0; k < S; ++k) sum += col[(size_t)k * S];
        }
        m = log(fmax(sum, 0.0));
      }
    }
    if (live && !is_root) {
      double* dst = acc + (size_t)(node.depth - 1) * gs;
      const bool first = node.flags & 2;
      pre[(size_t)i * gs] = first ? 0.0 : *dst;
      msg[(size_t)i * gs] = m;
      *dst = first ? m : *dst + m;
    }
  }
}

template <bool kDtau>
__global__ void tree_ll_post_bwd_kernel(PostArgs a) {
  extern __shared__ double w[];
  const int S = a.S, G = a.G, SS = S * S;
  double* Pt = w;             // [S][S] the edge's matrix, transposed: Pt[b * S + a] = P[a][b]
  double* eo = Pt + SS;       // [G][S] O_i, then exp(O_i - max O_i)
  double* ei = eo + G * S;    // [G][S] dp_i, then exp(dp_i - max dp_i) * obs_i
  double* sc = ei + G * S;    // [G] exp(max O_i + max dp_i - log L_u)
  double* Qs = sc + G;        // kDtau: [S][S] Q, not transposed
  double* prod = Qs + SS;     // kDtau: [G][S] (Q^T eo)(s) * (P ei)(s)
  double* usum = prod + G * S;  // kDtau: [G] d log L_u / d tau of the edge
  if constexpr (kDtau)
    for (int e = threadIdx.x; e < SS; e += blockDim.x) Qs[e] = a.Q[e];  // read after the root's barriers
  const int g = threadIdx.x / S, s = threadIdx.x - g * S;
  const int u = g < G ? a.unit_of[blockIdx.x * G + g] : -1;
  const bool live = u >= 0;
  const int cat = a.cta_cat[blockIdx.x];
  const size_t gs = (size_t)G * S;
  const size_t mine = (live ? g : 0) * S + s;
  double* alpha = a.stk + (size_t)blockIdx.x * 2 * (a.max_depth + 1) * gs + mine;
  double* sfx = alpha + (size_t)(a.max_depth + 1) * gs;
  const double* dp = a.dp + (size_t)blockIdx.x * a.n_nodes * gs + mine;
  const double* msg = a.msg + (size_t)blockIdx.x * a.n_nodes * gs + mine;
  const double* pre = a.pre + (size_t)blockIdx.x * a.n_nodes * gs + mine;
  const double ll = live ? a.ll_out[u] : 0.0;
  for (int i = a.n_nodes - 1; i >= 0; --i) {
    const cherry_ll_node node = a.nodes[i];
    const bool is_leaf = node.flags & 1;
    const int x = is_leaf && live ? a.obs[(size_t)node.obs_row * a.n_units + u] : S;
    if (i == a.n_nodes - 1) {
      // root: A = log pi; posterior pi_a exp(dp(a)) obs(a) / L
      double r = 0.0;
      if (live) {
        if (is_leaf) {
          r = (x == S || x == s) ? a.pi[s] * exp(-ll) : 0.0;
        } else {
          r = a.pi[s] * exp(dp[(size_t)i * gs] - ll);
          alpha[0] = log(a.pi[s]);
          sfx[0] = 0.0;
        }
      }
      if (threadIdx.x < G * S) eo[threadIdx.x] = r;
      __syncthreads();
      if ((int)threadIdx.x < S) {
        double t = 0.0;
        for (int h = 0; h < G; ++h) t += eo[h * S + threadIdx.x];
        a.root_part[(size_t)blockIdx.x * S + threadIdx.x] = t;
      }
      __syncthreads();
      continue;
    }
    const double* Pm = a.P + (size_t)a.p_index[(size_t)i * a.n_cats + cat] * SS;
    for (int e = threadIdx.x; e < SS; e += blockDim.x) Pt[e] = Pm[e];
    const int d = node.depth;
    double o = 0.0, v = 0.0;
    if (live) {
      o = alpha[(size_t)(d - 1) * gs] + pre[(size_t)i * gs] + sfx[(size_t)(d - 1) * gs];
      sfx[(size_t)(d - 1) * gs] = sfx[(size_t)(d - 1) * gs] + msg[(size_t)i * gs];
      if (!is_leaf) v = dp[(size_t)i * gs];
      eo[g * S + s] = o;
      ei[g * S + s] = v;
    }
    __syncthreads();
    double mo = -INFINITY, mi = 0.0;
    if (live) {
      for (int k = 0; k < S; ++k) mo = fmax(mo, eo[g * S + k]);
      if (!is_leaf) {
        mi = -INFINITY;
        for (int k = 0; k < S; ++k) mi = fmax(mi, ei[g * S + k]);
      }
      if (mo == -INFINITY) mo = 0.0;  // L_u = 0: every posterior is 0
      if (mi == -INFINITY) mi = 0.0;
    }
    __syncthreads();
    if (threadIdx.x < G * S) {
      eo[threadIdx.x] = live ? exp(o - mo) : 0.0;
      ei[threadIdx.x] = !live ? 0.0 : is_leaf ? ((x == S || x == s) ? 1.0 : 0.0) : exp(v - mi);
      if (s == 0) sc[g] = live ? exp(mo + mi - ll) : 0.0;
    }
    __syncthreads();
    if (live && !is_leaf) {
      // A_i(s) = log sum_a exp(O_i(a)) P_i[a][s]; this node's children start with an empty suffix
      double sum = 0.0;
      for (int k = 0; k < S; ++k) sum += eo[g * S + k] * Pt[s * S + k];
      alpha[(size_t)d * gs] = log(fmax(sum, 0.0)) + mo;
      sfx[(size_t)d * gs] = 0.0;
    }
    if constexpr (kDtau) {
      if (threadIdx.x < G * S) {  // dead slots: eo = ei = 0
        double qo = 0.0, pe = 0.0;
        for (int k = 0; k < S; ++k) {
          qo += Qs[k * S + s] * eo[g * S + k];
          pe += Pt[k * S + s] * ei[g * S + k];
        }
        prod[threadIdx.x] = qo * pe;
      }
    }
    double* part = a.part + ((size_t)blockIdx.x * a.n_nodes + i) * SS;
    for (int e = threadIdx.x; e < SS; e += blockDim.x) {
      const int ra = e / S, cb = e - ra * S;
      double t = 0.0;
      for (int h = 0; h < G; ++h) t += eo[h * S + ra] * ei[h * S + cb] * sc[h];
      part[e] = t * Pt[cb * S + ra];
    }
    __syncthreads();
    if constexpr (kDtau) {
      if (threadIdx.x < G * S && s == 0) {
        double t = 0.0;
        for (int k = 0; k < S; ++k) t += prod[g * S + k];
        usum[g] = t * sc[g];
      }
      __syncthreads();
      if (threadIdx.x == 0) {
        double t = 0.0;
        for (int h = 0; h < G; ++h) t += usum[h];
        a.dpart[(size_t)blockIdx.x * a.n_nodes + i] = t;
      }
    }
  }
}

// block m < n_matrices: W[m]; block n_matrices: the root posterior
__global__ void tree_ll_post_reduce_kernel(PostArgs a) {
  const int SS = a.S * a.S, e = threadIdx.x, m = blockIdx.x;
  if (m == a.n_matrices) {
    if (e < a.S) {
      double t = 0.0;
      for (int c = 0; c < a.n_ctas; ++c) t += a.root_part[(size_t)c * a.S + e];
      a.root_out[e] = t;
    }
    return;
  }
  if (e >= SS) return;
  double t = 0.0;
  for (int j = a.m_off[m]; j < a.m_off[m + 1]; ++j) {
    const int ent = a.m_ent[j];
    const int i = ent / a.n_cats, k = ent - i * a.n_cats;
    for (int c = a.cat_cta[k]; c < a.cat_cta[k + 1]; ++c) t += a.part[((size_t)c * a.n_nodes + i) * SS + e];
  }
  a.W_out[(size_t)m * SS + e] = t;
}

// dtau[i][k] = sum over the CTAs of category k, in CTA order, of the (CTA, edge i) derivatives;
// the root's row is 0
__global__ void tree_ll_dtau_reduce_kernel(PostArgs a) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= a.n_nodes * a.n_cats) return;
  const int i = e / a.n_cats, k = e - i * a.n_cats;
  double t = 0.0;
  if (i + 1 < a.n_nodes)
    for (int c = a.cat_cta[k]; c < a.cat_cta[k + 1]; ++c) t += a.dpart[(size_t)c * a.n_nodes + i];
  a.dtau_out[e] = t;
}

// Launch layout of the posterior pass, from the host copies of unit_cat and p_index.
struct PostLayout {
  int G = 0, n_ctas = 0;
  size_t doubles = 0, ints = 0;  // scratch: the doubles first, then the int32 tables
};

// dtau: the edge-derivative pass, which also keeps one double per (CTA, node)
bool post_layout(int S, int n_nodes, int max_depth, int n_cats, int n_matrices, int n_units,
                 const int32_t* unit_cat, bool dtau, PostLayout* L) {
  if (S < 1 || S > 32 || n_nodes < 1 || max_depth < 0 || n_cats < 1 || n_matrices < 1 || n_units < 0) return false;
  if (n_units > 0 && !unit_cat) return false;
  L->G = cherry_tree_ll_units_per_block(S, 1);
  std::vector<int64_t> count(n_cats, 0);
  for (int u = 0; u < n_units; ++u) {
    if (unit_cat[u] < 0 || unit_cat[u] >= n_cats) return false;
    ++count[unit_cat[u]];
  }
  int64_t ctas = 0;
  for (int k = 0; k < n_cats; ++k) ctas += (count[k] + L->G - 1) / L->G;
  L->n_ctas = (int)ctas;
  const size_t gs = (size_t)L->G * S;
  L->doubles = (size_t)ctas * (3 * (size_t)n_nodes * gs + 2 * (size_t)(max_depth + 1) * gs +
                               (size_t)n_nodes * S * S + S + (dtau ? (size_t)n_nodes : 0));
  L->ints = (size_t)ctas * L->G + ctas + (n_cats + 1) + (n_matrices + 1) + (size_t)(n_nodes - 1) * n_cats +
            (size_t)n_nodes * n_cats;
  return true;
}

// The host part of both posterior entry points (checks after the null checks, layout, index tables,
// upload, launches).  Q == nullptr: the edge posteriors alone; otherwise also dtau_out.
int tree_ll_post_launch(const cherry_ll_node* nodes, int n_nodes, int max_depth, const int32_t* p_index, int n_cats,
                        const double* P, int n_matrices, const uint8_t* obs, const int32_t* unit_cat, const double* pi,
                        const double* Q, int S, int n_units, void* scratch, size_t scratch_bytes, double* ll_out,
                        double* W_out, double* root_out, double* dtau_out, cudaStream_t stream) {
  if (S > 32) return cherry::fail(CHERRY_ELIMIT, "the posterior pass supports S <= 32 states (%d)", S);
  if (n_nodes < 1 || n_cats < 1 || S < 1 || max_depth < 0 || max_depth >= n_nodes || n_matrices < 1 || n_units < 0)
    return cherry::fail(CHERRY_EINVAL, "bad sizes");
  for (int i = 0; i + 1 < n_nodes; ++i)  // the root's entries are never read
    for (int k = 0; k < n_cats; ++k)
      if (p_index[(size_t)i * n_cats + k] < 0 || p_index[(size_t)i * n_cats + k] >= n_matrices)
        return cherry::fail(CHERRY_EINVAL, "p_index[%d] out of range", i * n_cats + k);
  PostLayout L;
  if (!post_layout(S, n_nodes, max_depth, n_cats, n_matrices, n_units, unit_cat, Q != nullptr, &L))
    return cherry::fail(CHERRY_EINVAL, "unit category out of range");
  if (scratch_bytes < L.doubles * sizeof(double) + L.ints * sizeof(int32_t))
    return cherry::fail(CHERRY_EINVAL, "scratch too small");
  const int G = L.G, n_ctas = L.n_ctas;
  const size_t gs = (size_t)G * S;

  // host tables: slots of each category's units in unit order, categories in order; matrix -> its
  // (node, category) pairs in (node, category) order (a counting sort)
  std::vector<int32_t> tab(L.ints);
  int32_t* unit_of = tab.data();
  int32_t* cta_cat = unit_of + (size_t)n_ctas * G;
  int32_t* cat_cta = cta_cat + n_ctas;
  int32_t* m_off = cat_cta + n_cats + 1;
  int32_t* m_ent = m_off + n_matrices + 1;
  int32_t* pidx = m_ent + (size_t)(n_nodes - 1) * n_cats;
  std::vector<int32_t> count(n_cats, 0);
  for (int u = 0; u < n_units; ++u) ++count[unit_cat[u]];
  cat_cta[0] = 0;
  for (int k = 0; k < n_cats; ++k) cat_cta[k + 1] = cat_cta[k] + (count[k] + G - 1) / G;
  std::fill(unit_of, unit_of + (size_t)n_ctas * G, -1);
  for (int k = 0; k < n_cats; ++k)
    for (int c = cat_cta[k]; c < cat_cta[k + 1]; ++c) cta_cat[c] = k;
  std::vector<int32_t> fill(n_cats, 0);
  for (int u = 0; u < n_units; ++u) {
    const int k = unit_cat[u];
    unit_of[(size_t)cat_cta[k] * G + fill[k]++] = u;
  }
  std::fill(m_off, m_off + n_matrices + 1, 0);
  for (int i = 0; i + 1 < n_nodes; ++i)
    for (int k = 0; k < n_cats; ++k) ++m_off[p_index[(size_t)i * n_cats + k] + 1];
  for (int m = 0; m < n_matrices; ++m) m_off[m + 1] += m_off[m];
  std::vector<int32_t> next(m_off, m_off + n_matrices);
  for (int i = 0; i + 1 < n_nodes; ++i)
    for (int k = 0; k < n_cats; ++k) m_ent[next[p_index[(size_t)i * n_cats + k]]++] = i * n_cats + k;
  std::copy(p_index, p_index + (size_t)n_nodes * n_cats, pidx);

  double* base = reinterpret_cast<double*>(scratch);
  int32_t* dtab = reinterpret_cast<int32_t*>(base + L.doubles);
  // pageable source: the copy is staged before cudaMemcpyAsync returns, so `tab` may go out of scope
  CHERRY_CUDA(cudaMemcpyAsync(dtab, tab.data(), L.ints * sizeof(int32_t), cudaMemcpyHostToDevice, stream));

  PostArgs a;
  a.nodes = nodes;
  a.p_index = dtab + (pidx - tab.data());
  a.P = P;
  a.obs = obs;
  a.pi = pi;
  a.unit_of = dtab;
  a.cta_cat = dtab + (cta_cat - tab.data());
  a.cat_cta = dtab + (cat_cta - tab.data());
  a.m_off = dtab + (m_off - tab.data());
  a.m_ent = dtab + (m_ent - tab.data());
  a.dp = base;
  a.msg = a.dp + (size_t)n_ctas * n_nodes * gs;
  a.pre = a.msg + (size_t)n_ctas * n_nodes * gs;
  a.stk = a.pre + (size_t)n_ctas * n_nodes * gs;
  a.part = a.stk + (size_t)n_ctas * 2 * (max_depth + 1) * gs;
  a.root_part = a.part + (size_t)n_ctas * n_nodes * S * S;
  a.dpart = a.root_part + (size_t)n_ctas * S;
  a.ll_out = ll_out;
  a.W_out = W_out;
  a.root_out = root_out;
  a.Q = Q;
  a.dtau_out = dtau_out;
  a.n_nodes = n_nodes;
  a.n_cats = n_cats;
  a.S = S;
  a.n_units = n_units;
  a.G = G;
  a.max_depth = max_depth;
  a.n_matrices = n_matrices;
  a.n_ctas = n_ctas;
  const int threads = (int)((gs + 31) / 32 * 32);
  if (n_ctas > 0) {
    tree_ll_post_fwd_kernel<<<n_ctas, threads, gs * sizeof(double), stream>>>(a);
    CHERRY_LAUNCH_CHECK("tree_ll_post_fwd_kernel");
    const size_t smem = ((size_t)S * S + 2 * gs + G) * sizeof(double);
    if (Q) {
      tree_ll_post_bwd_kernel<true><<<n_ctas, threads, smem + ((size_t)S * S + gs + G) * sizeof(double), stream>>>(a);
    } else {
      tree_ll_post_bwd_kernel<false><<<n_ctas, threads, smem, stream>>>(a);
    }
    CHERRY_LAUNCH_CHECK("tree_ll_post_bwd_kernel");
  }
  tree_ll_post_reduce_kernel<<<n_matrices + 1, (S * S + 31) / 32 * 32, 0, stream>>>(a);
  CHERRY_LAUNCH_CHECK("tree_ll_post_reduce_kernel");
  if (Q) {
    const int n = n_nodes * n_cats;
    tree_ll_dtau_reduce_kernel<<<(n + 255) / 256, 256, 0, stream>>>(a);
    CHERRY_LAUNCH_CHECK("tree_ll_dtau_reduce_kernel");
  }
  return CHERRY_OK;
}


}  // namespace

extern "C" {

int cherry_tree_ll_transpose(const double* P, int n_matrices, int Su, double* Pt, void* stream) {
  if (n_matrices == 0) return CHERRY_OK;
  if (!P || !Pt || P == Pt) return cherry::fail(CHERRY_EINVAL, "null or aliased pointer");
  if (n_matrices < 0 || Su < 1) return cherry::fail(CHERRY_EINVAL, "bad sizes");
  const int tiles = (Su + 31) / 32;
  for (int m0 = 0; m0 < n_matrices; m0 += 65535) {
    const int nm = n_matrices - m0 < 65535 ? n_matrices - m0 : 65535;
    transpose_matrices_kernel<<<dim3(tiles, tiles, nm), dim3(32, 8), 0, (cudaStream_t)stream>>>(
        P + (size_t)m0 * Su * Su, Pt + (size_t)m0 * Su * Su, Su);
  }
  CHERRY_LAUNCH_CHECK("transpose_matrices_kernel");
  return CHERRY_OK;
}

int cherry_tree_ll_units_per_block(int S, int c) {
  const int Su = c == 2 ? S * S : S;
  const int G = 256 / Su;
  return G < 1 ? 1 : G;
}

size_t cherry_tree_ll_scratch_bytes(int S, int c, int n_units, int max_depth) {
  const int Su = c == 2 ? S * S : S;
  const int G = cherry_tree_ll_units_per_block(S, c);
  const size_t blocks = (size_t)(n_units + G - 1) / G;
  return blocks * (size_t)(max_depth + 1) * G * Su * sizeof(double);
}

int cherry_tree_log_likelihood(const cherry_ll_node* nodes, int n_nodes, const int32_t* p_index, int n_cats,
                               const double* P, const uint8_t* obs, const int32_t* unit_cat, const double* pi,
                               int S, int c, int n_units, int max_depth, void* scratch, size_t scratch_bytes,
                               double* ll_out, void* stream) {
  if (n_units == 0) return CHERRY_OK;
  if (!nodes || !p_index || !P || !obs || !unit_cat || !pi || !scratch || !ll_out)
    return cherry::fail(CHERRY_EINVAL, "null pointer");
  if (n_nodes < 1 || n_cats < 1 || (c != 1 && c != 2) || S < 1 || max_depth < 0)
    return cherry::fail(CHERRY_EINVAL, "bad sizes");
  const int Su = c == 2 ? S * S : S;
  if (Su > 1024) return cherry::fail(CHERRY_ELIMIT, "more than 1024 unit states (%d)", Su);
  if (scratch_bytes < cherry_tree_ll_scratch_bytes(S, c, n_units, max_depth))
    return cherry::fail(CHERRY_EINVAL, "scratch too small");
  LlArgs a;
  a.nodes = nodes;
  a.p_index = p_index;
  a.P = P;
  a.obs = obs;
  a.unit_cat = unit_cat;
  a.pi = pi;
  a.acc = reinterpret_cast<double*>(scratch);
  a.ll_out = ll_out;
  a.n_nodes = n_nodes;
  a.n_cats = n_cats;
  a.S = S;
  a.c = c;
  a.Su = Su;
  a.n_units = n_units;
  a.G = cherry_tree_ll_units_per_block(S, c);
  a.max_depth = max_depth;
  const int threads = (a.G * Su + 31) / 32 * 32;
  const int blocks = (n_units + a.G - 1) / a.G;
  size_t smem = (size_t)a.G * (Su + 32) * sizeof(double);
  const size_t staging = (size_t)2 * kLlBatch * threads * sizeof(double);
  a.staged = Su > 64 && smem + staging <= 227 * 1024;
  // tree_ll_kernel's largest launchable CTA, which its register count decides (0 if unknown: always wide)
  static const int narrow_max_threads = [] {
    cudaFuncAttributes attr;
    return cudaFuncGetAttributes(&attr, tree_ll_kernel) == cudaSuccess ? attr.maxThreadsPerBlock : 0;
  }();
  const bool wide = threads > narrow_max_threads;
  if (a.staged) {
    smem += staging;
    const int rc = cherry::check_cuda(cudaFuncSetAttribute(wide ? tree_ll_wide_kernel : tree_ll_kernel,
                                                           cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024),
                                      "cudaFuncSetAttribute(tree_ll_kernel)");
    if (rc != 0) return rc;
  }
  if (wide) {
    tree_ll_wide_kernel<<<blocks, threads, smem, (cudaStream_t)stream>>>(a);
  } else {
    tree_ll_kernel<<<blocks, threads, smem, (cudaStream_t)stream>>>(a);
  }
  CHERRY_LAUNCH_CHECK("tree_ll_kernel");
  return CHERRY_OK;
}

size_t cherry_tree_ll_posterior_scratch_bytes(int S, int n_nodes, int max_depth, int n_cats, int n_matrices,
                                              int n_units, const int32_t* unit_cat) {
  PostLayout L;
  if (!post_layout(S, n_nodes, max_depth, n_cats, n_matrices, n_units, unit_cat, false, &L)) return 0;
  return L.doubles * sizeof(double) + L.ints * sizeof(int32_t);
}

int cherry_tree_ll_posterior(const cherry_ll_node* nodes, int n_nodes, int max_depth, const int32_t* p_index,
                             int n_cats, const double* P, int n_matrices, const uint8_t* obs, const int32_t* unit_cat,
                             const double* pi, int S, int n_units, void* scratch, size_t scratch_bytes,
                             double* ll_out, double* W_out, double* root_out, void* stream) {
  if (!nodes || !p_index || !P || !obs || !unit_cat || !pi || !scratch || !ll_out || !W_out || !root_out)
    return cherry::fail(CHERRY_EINVAL, "null pointer");
  return tree_ll_post_launch(nodes, n_nodes, max_depth, p_index, n_cats, P, n_matrices, obs, unit_cat, pi, nullptr, S,
                             n_units, scratch, scratch_bytes, ll_out, W_out, root_out, nullptr, (cudaStream_t)stream);
}

size_t cherry_tree_ll_edge_derivatives_scratch_bytes(int S, int n_nodes, int max_depth, int n_cats, int n_matrices,
                                                     int n_units, const int32_t* unit_cat) {
  PostLayout L;
  if (!post_layout(S, n_nodes, max_depth, n_cats, n_matrices, n_units, unit_cat, true, &L)) return 0;
  return L.doubles * sizeof(double) + L.ints * sizeof(int32_t);
}

int cherry_tree_ll_edge_derivatives(const cherry_ll_node* nodes, int n_nodes, int max_depth, const int32_t* p_index,
                                    int n_cats, const double* P, int n_matrices, const uint8_t* obs,
                                    const int32_t* unit_cat, const double* pi, const double* Q, int S, int n_units,
                                    void* scratch, size_t scratch_bytes, double* ll_out, double* W_out,
                                    double* root_out, double* dtau_out, void* stream) {
  if (!nodes || !p_index || !P || !obs || !unit_cat || !pi || !Q || !scratch || !ll_out || !W_out || !root_out ||
      !dtau_out)
    return cherry::fail(CHERRY_EINVAL, "null pointer");
  return tree_ll_post_launch(nodes, n_nodes, max_depth, p_index, n_cats, P, n_matrices, obs, unit_cat, pi, Q, S,
                             n_units, scratch, scratch_bytes, ll_out, W_out, root_out, dtau_out, (cudaStream_t)stream);
}

}  // extern "C"

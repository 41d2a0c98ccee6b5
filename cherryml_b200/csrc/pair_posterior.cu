// Edge posteriors of the contacting-pair model (c = 2, Su = S*S states, S <= 32) for the exact gradient of
// its log-likelihood: the inside/outside pass of tree_ll_post_*_kernel (likelihood.cu) with the pairs of a
// family as the COLUMNS of one matrix, so that an edge costs three [Su x Su] x [Su x n_pairs] FP64
// tensor-core products and its matrix is streamed once per pass for every 16 pairs, instead of once per pair.
//
// Every per-node vector is stored pair-major, [n_pairs padded to Np][Su padded to Sp], and every column
// (pair) carries its own scale: its maximum, as the per-unit maximum of the forward.
//   inside, nodes by height:  H_v = sum of the children's messages in tree order (leaf: log obs);
//                             M_v = log(P_v exp(H_v - max H_v)) + max H_v   (leaf: a gather of P_v columns);
//   outside, nodes by depth:  O_i = A_p + prefix_i + suffix_i over the siblings of i (never "total minus
//                             own": a zero-length branch gives -inf messages), A_root = log pi;
//                             A_i = log(P_i^T exp(O_i - max O_i)) + max O_i;
//   edge posteriors:          W_m = P_m o sum over the edges i of m, in node order, of U_i V_i^T with
//                             U_i = exp(O_i - max O_i), V_i = exp(H_i - max H_i) obs_i exp(max O_i + max H_i - ll).
// No atomics: each output element is summed by one thread in a fixed order.
#include <algorithm>
#include <cstdint>
#include <vector>

#include "common.cuh"
#include "dmma.cuh"

namespace {

constexpr int kPairSpAlign = 64;  // Sp: multiple of the edge kernel's 64 x 64 tile
constexpr int kPairNpAlign = 16;  // Np: multiple of the node kernel's 16-pair tile and the edge kernel's K chunk
constexpr int kPairMaxNp = 65535; // pairs ride on gridDim.y
constexpr int kPrepThreads = 128;
constexpr int kPrepPerThread = 1024 / kPrepThreads;  // Sp <= 1024
constexpr int kGemmThreads = 128;
constexpr int kNodeTM = 16, kNodeTN = 128, kBK = 16, kLdRow = 20;  // [row][k] tiles, k contiguous (bank-conflict free)
constexpr int kEdgeT = 64, kLdCol = 68;                             // [k][64] tiles

struct PairArgs {
  const double* P;         // [n_matrices][Su][Su], NOT transposed
  const uint8_t* obs;      // [n_leaves][N][2]
  const double* pi;        // [Su]
  const int32_t* pidx;     // [n_nodes]
  const int32_t* ch_off;   // [n_nodes + 1] children of node v: ch[ch_off[v] .. ch_off[v+1]) in tree order
  const int32_t* ch;       // [n_nodes]
  const int32_t* m_off;    // [n_matrices + 1]
  const int32_t* m_ent;    // [n_nodes]: non-root nodes grouped by matrix, in node order
  const int32_t* obs_row;  // [n_nodes]: leaf row of obs, -1 for an internal node
  double* hv;              // [n_nodes][Np][Sp]: H (inside), then V for non-root nodes
  double* ma;              // [n_nodes][Np][Sp]: M (message to the parent), then A (outside)
  double* uu;              // [n_nodes][Np][Sp]: exp(H - max H) as the inside product's input, then U
  double* mh;              // [n_nodes][Np]: max H
  double* mo;              // [n_nodes][Np]: max O
  double* ll_out;          // [N]
  double* W_out;           // [n_matrices][Su][Su]
  double* root_out;        // [Su]
  int S, Su, Sp, N, Np, n_nodes, root;
};

__device__ __forceinline__ size_t vec_off(const PairArgs& a, int v, int u) { return ((size_t)v * a.Np + u) * a.Sp; }

__device__ __forceinline__ bool compatible(int x, int y, int S, int k) {
  return (x == S || x == k / S) && (y == S || y == k % S);
}

// fixed-order block reductions over kPrepThreads threads (red: 4 doubles); every thread gets the result
__device__ __forceinline__ double block_max(double v, double* red) {
  for (int o = 16; o > 0; o >>= 1) v = fmax(v, __shfl_xor_sync(0xffffffffu, v, o));
  __syncthreads();
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
  __syncthreads();
  return fmax(fmax(red[0], red[1]), fmax(red[2], red[3]));
}
__device__ __forceinline__ double block_sum(double v, double* red) {
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  __syncthreads();
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
  __syncthreads();
  return (red[0] + red[1]) + (red[2] + red[3]);
}

// Leaf messages: M(a) = log sum over the states b compatible with the pair's residues of P[a][b].
// grid (leaves, Np)
__global__ void __launch_bounds__(kPrepThreads) pair_leaf_kernel(PairArgs a, const int32_t* leaves) {
  const int v = leaves[blockIdx.x], u = blockIdx.y;
  const int S = a.S, Su = a.Su;
  double* out = a.ma + vec_off(a, v, u);
  if (u >= a.N) {
    for (int k = threadIdx.x; k < a.Sp; k += kPrepThreads) out[k] = 0.0;
    return;
  }
  const uint8_t* ob = a.obs + ((size_t)a.obs_row[v] * a.N + u) * 2;
  const int x = ob[0], y = ob[1];
  const double* P = a.P + (size_t)a.pidx[v] * Su * Su;
  for (int k = threadIdx.x; k < a.Sp; k += kPrepThreads) {
    double m = 0.0;
    if (k < Su) {
      const double* row = P + (size_t)k * Su;
      double sum = 0.0;
      if (x != S && y != S) {
        sum = row[x * S + y];
      } else if (x != S) {
        for (int j = 0; j < S; ++j) sum += row[x * S + j];
      } else if (y != S) {
        for (int i = 0; i < S; ++i) sum += row[i * S + y];
      } else {
        for (int j = 0; j < Su; ++j) sum += row[j];
      }
      m = log(fmax(sum, 0.0));
    }
    out[k] = m;
  }
}

// Internal node v = list[blockIdx.x], pair u = blockIdx.y: H = sum of the children's messages in tree order,
// max H, and exp(H - max H) as the input of the inside product.  At the root: ll_out[u].
__global__ void __launch_bounds__(kPrepThreads) pair_inside_prep_kernel(PairArgs a, const int32_t* list) {
  __shared__ double red[kPrepThreads / 32];
  const int v = list[blockIdx.x], u = blockIdx.y;
  const bool live = u < a.N;
  const int c0 = a.ch_off[v], c1 = a.ch_off[v + 1];
  double* hv = a.hv + vec_off(a, v, u);
  double mx = -INFINITY;
  if (live)
    for (int k = threadIdx.x; k < a.Su; k += kPrepThreads) {
      double s = a.ma[vec_off(a, a.ch[c0], u) + k];
      for (int c = c0 + 1; c < c1; ++c) s += a.ma[vec_off(a, a.ch[c], u) + k];
      hv[k] = s;
      mx = fmax(mx, s);
    }
  mx = block_max(mx, red);
  if (mx == -INFINITY) mx = 0.0;  // L_u = 0 (or a padding column)
  double psum = 0.0;
  for (int k = threadIdx.x; k < a.Sp; k += kPrepThreads) {  // the same k as above: hv[k] is this thread's
    const double x = live && k < a.Su ? exp(hv[k] - mx) : 0.0;
    a.uu[vec_off(a, v, u) + k] = x;
    if (k < a.Su) psum += a.pi[k] * x;
  }
  if (threadIdx.x == 0) a.mh[(size_t)v * a.Np + u] = mx;
  if (v == a.root) {
    psum = block_sum(psum, red);
    if (live && threadIdx.x == 0) a.ll_out[u] = log(fmax(psum, 0.0)) + mx;
  }
}

// One level of the inside (OUTSIDE = false) or outside (OUTSIDE = true) product, for the nodes list[0 .. n):
//   inside:  ma[v][u][n] = log(sum_k uu[v][u][k] P_v[n][k]) + mh[v][u]
//   outside: ma[v][u][n] = log(sum_k uu[v][u][k] P_v[k][n]) + mo[v][u]
// A CTA computes 16 pairs x 128 states, its four warps 16 x 32 each (2 x 4 DMMA tiles).  The CTAs of one
// (node, state tile) are consecutive, so all pair tiles of an edge matrix tile read it from L2 together.
template <bool OUTSIDE>
__global__ void __launch_bounds__(kGemmThreads) pair_node_gemm_kernel(PairArgs a, const int32_t* list, int n_stile,
                                                                      int n_ptile) {
  __shared__ double As[2][kNodeTM * kLdRow];
  __shared__ double Bs[2][kNodeTN * kLdRow];
  const int b = blockIdx.x;
  const int pt = b % n_ptile, st = (b / n_ptile) % n_stile, v = list[b / n_ptile / n_stile];
  const int p0 = pt * kNodeTM, n0 = st * kNodeTN, Su = a.Su;
  const double* X = a.uu + vec_off(a, v, p0);
  const double* P = a.P + (size_t)a.pidx[v] * Su * Su;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, g = lane >> 2, tg = lane & 3;
  const int n_chunks = (Su + kBK - 1) / kBK;
  double ra[2], rb[16];
  auto load = [&](int c) {
    const int k0 = c * kBK;
#pragma unroll
    for (int r = 0; r < 2; ++r) {
      const int idx = threadIdx.x + r * kGemmThreads;
      ra[r] = X[(size_t)(idx / kBK) * a.Sp + k0 + idx % kBK];  // padding columns hold zeros
    }
#pragma unroll
    for (int r = 0; r < 16; ++r) {
      const int idx = threadIdx.x + r * kGemmThreads;
      int n, k;
      if (OUTSIDE) {
        k = idx / kNodeTN;
        n = idx % kNodeTN;
      } else {
        n = idx / kBK;
        k = idx % kBK;
      }
      const int gn = n0 + n, gk = k0 + k;
      rb[r] = gn < Su && gk < Su ? (OUTSIDE ? P[(size_t)gk * Su + gn] : P[(size_t)gn * Su + gk]) : 0.0;
    }
  };
  auto store = [&](int s) {
#pragma unroll
    for (int r = 0; r < 2; ++r) {
      const int idx = threadIdx.x + r * kGemmThreads;
      As[s][(idx / kBK) * kLdRow + idx % kBK] = ra[r];
    }
#pragma unroll
    for (int r = 0; r < 16; ++r) {
      const int idx = threadIdx.x + r * kGemmThreads;
      const int n = OUTSIDE ? idx % kNodeTN : idx / kBK, k = OUTSIDE ? idx / kNodeTN : idx % kBK;
      Bs[s][n * kLdRow + k] = rb[r];
    }
  };
  double acc[2][4][2];
#pragma unroll
  for (int i = 0; i < 2; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j][0] = acc[i][j][1] = 0.0;
  load(0);
  store(0);
  __syncthreads();
  for (int c = 0; c < n_chunks; ++c) {
    const int s = c & 1;
    if (c + 1 < n_chunks) load(c + 1);
#pragma unroll
    for (int kk = 0; kk < kBK; kk += 4) {
      double fa[2], fb[4];
#pragma unroll
      for (int i = 0; i < 2; ++i) fa[i] = As[s][(8 * i + g) * kLdRow + kk + tg];
#pragma unroll
      for (int j = 0; j < 4; ++j) fb[j] = Bs[s][(32 * warp + 8 * j + g) * kLdRow + kk + tg];
#pragma unroll
      for (int i = 0; i < 2; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) dmma884(acc[i][j][0], acc[i][j][1], fa[i], fb[j]);
    }
    if (c + 1 < n_chunks) store(s ^ 1);
    __syncthreads();
  }
  const double* scale = (OUTSIDE ? a.mo : a.mh) + (size_t)v * a.Np + p0;
#pragma unroll
  for (int i = 0; i < 2; ++i) {
    const int u = 8 * i + g;
    const double sc = scale[u];
    double* out = a.ma + vec_off(a, v, p0 + u);
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int n = n0 + 32 * warp + 8 * j + 2 * tg;
      if (n < a.Sp) {
        out[n] = log(fmax(acc[i][j][0], 0.0)) + sc;
        out[n + 1] = log(fmax(acc[i][j][1], 0.0)) + sc;
      }
    }
  }
}

// Parent p = list[blockIdx.x], pair u = blockIdx.y: O_i = A_p + prefix_i + suffix_i for every child i, then
// max O_i and U_i = exp(O_i - max O_i), the input of the outside product and of the edge posteriors.
__global__ void __launch_bounds__(kPrepThreads) pair_outside_prep_kernel(PairArgs a, const int32_t* list) {
  __shared__ double red[kPrepThreads / 32];
  const int p = list[blockIdx.x], u = blockIdx.y;
  const bool live = u < a.N;
  const int c0 = a.ch_off[p], c1 = a.ch_off[p + 1];
  if (live) {
    for (int k = threadIdx.x; k < a.Su; k += kPrepThreads) {
      double pre = 0.0;
      for (int c = c0; c < c1; ++c) {
        const int i = a.ch[c];
        a.uu[vec_off(a, i, u) + k] = pre;
        pre = pre + a.ma[vec_off(a, i, u) + k];
      }
      const double A = p == a.root ? log(a.pi[k]) : a.ma[vec_off(a, p, u) + k];
      double suf = 0.0;
      for (int c = c1 - 1; c >= c0; --c) {
        const int i = a.ch[c];
        double* o = a.uu + vec_off(a, i, u) + k;
        *o = A + *o + suf;
        suf = suf + a.ma[vec_off(a, i, u) + k];
      }
    }
  }
  for (int c = c0; c < c1; ++c) {
    const int i = a.ch[c];
    double* o = a.uu + vec_off(a, i, u);
    double o_reg[kPrepPerThread];
    double mx = -INFINITY;
#pragma unroll
    for (int r = 0; r < kPrepPerThread; ++r) {
      const int k = threadIdx.x + r * kPrepThreads;
      o_reg[r] = live && k < a.Su ? o[k] : -INFINITY;
      mx = fmax(mx, o_reg[r]);
    }
    mx = block_max(mx, red);
    if (mx == -INFINITY) mx = 0.0;
#pragma unroll
    for (int r = 0; r < kPrepPerThread; ++r) {
      const int k = threadIdx.x + r * kPrepThreads;
      if (k < a.Sp) o[k] = live && k < a.Su ? exp(o_reg[r] - mx) : 0.0;
    }
    if (threadIdx.x == 0) a.mo[(size_t)i * a.Np + u] = mx;
  }
}

// V_i = exp(H_i - max H_i) obs_i exp(max O_i + max H_i - ll_u) for every non-root node i, in place of H_i
// (a leaf: H = log obs, max H = 0).  A pair with L_u = 0 gets V = 0.  grid (n_nodes - 1, Np)
__global__ void __launch_bounds__(kPrepThreads) pair_v_kernel(PairArgs a) {
  const int i = blockIdx.x, u = blockIdx.y;
  double* out = a.hv + vec_off(a, i, u);
  const int row = a.obs_row[i];
  double sc = 0.0, mhv = 0.0;
  int x = a.S, y = a.S;
  if (u < a.N) {
    const double ll = a.ll_out[u];
    if (row < 0) mhv = a.mh[(size_t)i * a.Np + u];
    if (ll > -INFINITY) sc = exp(a.mo[(size_t)i * a.Np + u] + mhv - ll);
    if (row >= 0) {
      x = a.obs[((size_t)row * a.N + u) * 2];
      y = a.obs[((size_t)row * a.N + u) * 2 + 1];
    }
  }
  for (int k = threadIdx.x; k < a.Sp; k += kPrepThreads) {
    double v = 0.0;
    if (k < a.Su && sc != 0.0) v = row >= 0 ? (compatible(x, y, a.S, k) ? sc : 0.0) : exp(out[k] - mhv) * sc;
    out[k] = v;
  }
}

// W_m tile (64 x 64 of (parent state a, child state b)) = P_m o sum over the edges i of m (node order) and the
// pairs (16 at a time) of U_i[u][a] V_i[u][b].  grid: tiles of the matrix fastest, then m.  Four warps of
// 32 x 32 (4 x 4 DMMA tiles).
__global__ void __launch_bounds__(kGemmThreads) pair_edge_kernel(PairArgs a, int n_tile) {
  __shared__ double As[2][kBK * kLdCol];
  __shared__ double Bs[2][kBK * kLdCol];
  const int tiles = n_tile * n_tile;
  const int m = blockIdx.x / tiles, t = blockIdx.x % tiles;
  const int a0 = (t / n_tile) * kEdgeT, b0 = (t % n_tile) * kEdgeT;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, g = lane >> 2, tg = lane & 3;
  const int wm = (warp >> 1) * 32, wn = (warp & 1) * 32;
  const int e0 = a.m_off[m], n_e = a.m_off[m + 1] - e0;
  const int cpe = a.Np / kBK;
  const int n_chunks = n_e * cpe;
  double ra[8], rb[8];
  auto load = [&](int c) {
    const int node = a.m_ent[e0 + c / cpe], u0 = (c % cpe) * kBK;
    const double* U = a.uu + vec_off(a, node, u0);
    const double* V = a.hv + vec_off(a, node, u0);
#pragma unroll
    for (int r = 0; r < 8; ++r) {
      const int idx = threadIdx.x + r * kGemmThreads;
      const size_t off = (size_t)(idx / kEdgeT) * a.Sp + idx % kEdgeT;
      ra[r] = U[off + a0];
      rb[r] = V[off + b0];
    }
  };
  auto store = [&](int s) {
#pragma unroll
    for (int r = 0; r < 8; ++r) {
      const int idx = threadIdx.x + r * kGemmThreads;
      const int o = (idx / kEdgeT) * kLdCol + idx % kEdgeT;
      As[s][o] = ra[r];
      Bs[s][o] = rb[r];
    }
  };
  double acc[4][4][2];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j][0] = acc[i][j][1] = 0.0;
  if (n_chunks > 0) {
    load(0);
    store(0);
  }
  __syncthreads();
  for (int c = 0; c < n_chunks; ++c) {
    const int s = c & 1;
    if (c + 1 < n_chunks) load(c + 1);
#pragma unroll
    for (int kk = 0; kk < kBK; kk += 4) {
      double fa[4], fb[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) fa[i] = As[s][(kk + tg) * kLdCol + wm + 8 * i + g];
#pragma unroll
      for (int j = 0; j < 4; ++j) fb[j] = Bs[s][(kk + tg) * kLdCol + wn + 8 * j + g];
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) dmma884(acc[i][j][0], acc[i][j][1], fa[i], fb[j]);
    }
    if (c + 1 < n_chunks) store(s ^ 1);
    __syncthreads();
  }
  const int Su = a.Su;
  const double* P = a.P + (size_t)m * Su * Su;
  double* W = a.W_out + (size_t)m * Su * Su;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int r = a0 + wm + 8 * i + g;
    if (r >= Su) continue;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int col = b0 + wn + 8 * j + 2 * tg;
      if (col < Su) W[(size_t)r * Su + col] = P[(size_t)r * Su + col] * acc[i][j][0];
      if (col + 1 < Su) W[(size_t)r * Su + col + 1] = P[(size_t)r * Su + col + 1] * acc[i][j][1];
    }
  }
}

// Root posterior summed over pairs (pair order).  A single-leaf tree also gets its ll_out here.  One CTA.
__global__ void __launch_bounds__(256) pair_root_kernel(PairArgs a) {
  const int S = a.S, Su = a.Su, root = a.root;
  const int row = a.obs_row[root];
  if (row >= 0) {
    for (int u = threadIdx.x; u < a.N; u += blockDim.x) {
      const uint8_t* ob = a.obs + ((size_t)row * a.N + u) * 2;
      double sum = 0.0;
      for (int k = 0; k < Su; ++k) sum += compatible(ob[0], ob[1], S, k) ? a.pi[k] : 0.0;
      a.ll_out[u] = log(fmax(sum, 0.0));
    }
    __syncthreads();
  }
  for (int k = threadIdx.x; k < Su; k += blockDim.x) {
    double t = 0.0;
    for (int u = 0; u < a.N; ++u) {
      const double ll = a.ll_out[u];
      if (!(ll > -INFINITY)) continue;
      if (row >= 0) {
        const uint8_t* ob = a.obs + ((size_t)row * a.N + u) * 2;
        t += compatible(ob[0], ob[1], S, k) ? a.pi[k] * exp(-ll) : 0.0;
      } else {
        t += a.pi[k] * exp(a.hv[vec_off(a, root, u) + k] - ll);
      }
    }
    a.root_out[k] = t;
  }
}

int round_up(int x, int m) { return (x + m - 1) / m * m; }

bool pair_sizes(int S, int n_nodes, int max_depth, int n_pairs, int n_matrices, int* Sp, int* Np) {
  if (S < 1 || S > 32 || n_nodes < 1 || max_depth < 0 || n_pairs < 0 || n_matrices < 1) return false;
  *Sp = round_up(S * S, kPairSpAlign);
  *Np = round_up(std::max(n_pairs, 1), kPairNpAlign);
  return *Np <= kPairMaxNp;
}

size_t pair_scratch_bytes(int n_nodes, int n_matrices, int Sp, int Np) {
  const size_t doubles = 3 * (size_t)n_nodes * Np * Sp + 2 * (size_t)n_nodes * Np;
  const size_t ints = 8 * (size_t)n_nodes + n_matrices + 2;
  return doubles * sizeof(double) + ints * sizeof(int32_t);
}

}  // namespace

extern "C" {

size_t cherry_tree_ll_pair_posterior_scratch_bytes(int S, int n_nodes, int max_depth, int n_pairs, int n_matrices) {
  int Sp, Np;
  if (!pair_sizes(S, n_nodes, max_depth, n_pairs, n_matrices, &Sp, &Np)) return 0;
  return pair_scratch_bytes(n_nodes, n_matrices, Sp, Np);
}

int cherry_tree_ll_pair_posterior(const cherry_ll_node* nodes, int n_nodes, int max_depth, const int32_t* p_index,
                                  const double* P, int n_matrices, const uint8_t* obs, const double* pi, int S,
                                  int n_pairs, void* scratch, size_t scratch_bytes, double* ll_out, double* W_out,
                                  double* root_out, void* stream_) {
  if (!nodes || !p_index || !P || !obs || !pi || !scratch || !ll_out || !W_out || !root_out)
    return cherry::fail(CHERRY_EINVAL, "null pointer");
  if (S > 32) return cherry::fail(CHERRY_ELIMIT, "the pair posterior pass supports S <= 32 states (%d)", S);
  int Sp, Np;
  if (!pair_sizes(S, n_nodes, max_depth, n_pairs, n_matrices, &Sp, &Np)) {
    if (S >= 1 && n_pairs > 0 && round_up(n_pairs, kPairNpAlign) > kPairMaxNp)
      return cherry::fail(CHERRY_ELIMIT, "more than %d pairs (%d)", kPairMaxNp, n_pairs);
    return cherry::fail(CHERRY_EINVAL, "bad sizes");
  }
  for (int i = 0; i + 1 < n_nodes; ++i)  // the root's entry is never read
    if (p_index[i] < 0 || p_index[i] >= n_matrices) return cherry::fail(CHERRY_EINVAL, "p_index[%d] out of range", i);
  if (scratch_bytes < pair_scratch_bytes(n_nodes, n_matrices, Sp, Np))
    return cherry::fail(CHERRY_EINVAL, "scratch too small");

  // Host tables from the post-order node list: children (tree order), heights, leaves, internal nodes by
  // height and by depth, non-root nodes grouped by matrix.
  std::vector<int32_t> tab(8 * (size_t)n_nodes + n_matrices + 2, 0);
  int32_t* ch_off = tab.data();
  int32_t* ch = ch_off + n_nodes + 1;
  int32_t* by_h = ch + n_nodes;
  int32_t* by_d = by_h + n_nodes;
  int32_t* leaves = by_d + n_nodes;
  int32_t* m_off = leaves + n_nodes;
  int32_t* m_ent = m_off + n_matrices + 1;
  int32_t* pidx = m_ent + n_nodes;
  int32_t* obs_row = pidx + n_nodes;
  const int root = n_nodes - 1;
  if (nodes[root].depth != 0) return cherry::fail(CHERRY_EINVAL, "the last node is not the root");
  std::vector<std::vector<int32_t>> pending(max_depth + 2);
  std::vector<int> height(n_nodes, 0);
  int n_ch = 0, n_leaves = 0;
  for (int v = 0; v < n_nodes; ++v) {
    const int d = nodes[v].depth;
    const bool leaf = nodes[v].flags & 1;
    if (d < 0 || d > max_depth || (v < root && d == 0)) return cherry::fail(CHERRY_EINVAL, "bad node depth");
    ch_off[v] = n_ch;
    if (!leaf) {
      if (pending[d + 1].empty()) return cherry::fail(CHERRY_EINVAL, "internal node %d without children", v);
      for (int c : pending[d + 1]) {
        ch[n_ch++] = c;
        height[v] = std::max(height[v], height[c] + 1);
      }
      pending[d + 1].clear();
      obs_row[v] = -1;
    } else {
      if (nodes[v].obs_row < 0) return cherry::fail(CHERRY_EINVAL, "leaf %d without an obs row", v);
      obs_row[v] = nodes[v].obs_row;
      if (v < root) leaves[n_leaves++] = v;
    }
    pending[d].push_back(v);
  }
  ch_off[n_nodes] = n_ch;
  if (pending[0].size() != 1) return cherry::fail(CHERRY_EINVAL, "nodes are not a post-order of one tree");
  for (int d = 1; d <= max_depth + 1; ++d)
    if (!pending[d].empty()) return cherry::fail(CHERRY_EINVAL, "nodes are not a post-order of one tree");
  std::vector<int> internal;
  for (int v = 0; v < n_nodes; ++v)
    if (!(nodes[v].flags & 1)) internal.push_back(v);
  const int n_int = (int)internal.size();
  std::vector<int> h_off, d_off;  // level offsets into by_h / by_d
  std::copy(internal.begin(), internal.end(), by_h);
  std::stable_sort(by_h, by_h + n_int, [&](int x, int y) { return height[x] < height[y]; });
  std::copy(internal.begin(), internal.end(), by_d);
  std::stable_sort(by_d, by_d + n_int, [&](int x, int y) { return nodes[x].depth < nodes[y].depth; });
  for (int j = 0; j < n_int; ++j)
    if (j == 0 || height[by_h[j]] != height[by_h[j - 1]]) h_off.push_back(j);
  h_off.push_back(n_int);
  for (int j = 0; j < n_int; ++j)
    if (j == 0 || nodes[by_d[j]].depth != nodes[by_d[j - 1]].depth) d_off.push_back(j);
  d_off.push_back(n_int);
  for (int i = 0; i < root; ++i) ++m_off[p_index[i] + 1];
  for (int m = 0; m < n_matrices; ++m) m_off[m + 1] += m_off[m];
  {
    std::vector<int32_t> next(m_off, m_off + n_matrices);
    for (int i = 0; i < root; ++i) m_ent[next[p_index[i]]++] = i;
  }
  std::copy(p_index, p_index + root, pidx);
  pidx[root] = 0;

  cudaStream_t stream = (cudaStream_t)stream_;
  const int Su = S * S;
  if (n_pairs == 0) {
    CHERRY_CUDA(cudaMemsetAsync(W_out, 0, (size_t)n_matrices * Su * Su * sizeof(double), stream));
    CHERRY_CUDA(cudaMemsetAsync(root_out, 0, (size_t)Su * sizeof(double), stream));
    return CHERRY_OK;
  }
  const size_t vec = (size_t)n_nodes * Np * Sp;
  double* base = reinterpret_cast<double*>(scratch);
  int32_t* dtab = reinterpret_cast<int32_t*>(base + 3 * vec + 2 * (size_t)n_nodes * Np);
  // pageable source: the copy is staged before cudaMemcpyAsync returns, so `tab` may go out of scope
  CHERRY_CUDA(cudaMemcpyAsync(dtab, tab.data(), tab.size() * sizeof(int32_t), cudaMemcpyHostToDevice, stream));
  auto dev = [&](const int32_t* h) { return dtab + (h - tab.data()); };
  PairArgs a;
  a.P = P;
  a.obs = obs;
  a.pi = pi;
  a.pidx = dev(pidx);
  a.ch_off = dev(ch_off);
  a.ch = dev(ch);
  a.m_off = dev(m_off);
  a.m_ent = dev(m_ent);
  a.obs_row = dev(obs_row);
  a.hv = base;
  a.ma = base + vec;
  a.uu = base + 2 * vec;
  a.mh = base + 3 * vec;
  a.mo = a.mh + (size_t)n_nodes * Np;
  a.ll_out = ll_out;
  a.W_out = W_out;
  a.root_out = root_out;
  a.S = S;
  a.Su = Su;
  a.Sp = Sp;
  a.N = n_pairs;
  a.Np = Np;
  a.n_nodes = n_nodes;
  a.root = root;
  const int n_stile = (Sp + kNodeTN - 1) / kNodeTN, n_ptile = Np / kNodeTM;

  if (n_leaves > 0) {
    pair_leaf_kernel<<<dim3(n_leaves, Np), kPrepThreads, 0, stream>>>(a, dev(leaves));
    CHERRY_LAUNCH_CHECK("pair_leaf_kernel");
  }
  // inside: one height at a time; the root is alone at the greatest height and has no product
  for (size_t l = 0; l + 1 < h_off.size(); ++l) {
    const int n = h_off[l + 1] - h_off[l];
    pair_inside_prep_kernel<<<dim3(n, Np), kPrepThreads, 0, stream>>>(a, dev(by_h) + h_off[l]);
    CHERRY_LAUNCH_CHECK("pair_inside_prep_kernel");
    if (l + 2 < h_off.size()) {
      pair_node_gemm_kernel<false><<<n * n_stile * n_ptile, kGemmThreads, 0, stream>>>(a, dev(by_h) + h_off[l],
                                                                                       n_stile, n_ptile);
      CHERRY_LAUNCH_CHECK("pair_node_gemm_kernel<inside>");
    }
  }
  // outside: the parents at depth d give their children O and U; the internal children (the next depth's
  // parents) then get A by the outside product
  for (size_t l = 0; l + 1 < d_off.size(); ++l) {
    const int n = d_off[l + 1] - d_off[l];
    pair_outside_prep_kernel<<<dim3(n, Np), kPrepThreads, 0, stream>>>(a, dev(by_d) + d_off[l]);
    CHERRY_LAUNCH_CHECK("pair_outside_prep_kernel");
    if (l + 2 < d_off.size()) {
      const int nn = d_off[l + 2] - d_off[l + 1];
      pair_node_gemm_kernel<true><<<nn * n_stile * n_ptile, kGemmThreads, 0, stream>>>(a, dev(by_d) + d_off[l + 1],
                                                                                       n_stile, n_ptile);
      CHERRY_LAUNCH_CHECK("pair_node_gemm_kernel<outside>");
    }
  }
  if (root > 0) {
    pair_v_kernel<<<dim3(root, Np), kPrepThreads, 0, stream>>>(a);
    CHERRY_LAUNCH_CHECK("pair_v_kernel");
  }
  const int n_tile = Sp / kEdgeT;
  pair_edge_kernel<<<n_matrices * n_tile * n_tile, kGemmThreads, 0, stream>>>(a, n_tile);
  CHERRY_LAUNCH_CHECK("pair_edge_kernel");
  pair_root_kernel<<<1, 256, 0, stream>>>(a);
  CHERRY_LAUNCH_CHECK("pair_root_kernel");
  return CHERRY_OK;
}

}  // extern "C"

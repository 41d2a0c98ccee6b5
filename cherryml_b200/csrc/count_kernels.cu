// Transition counting for sm_100a: bucket table, LG (single-site) histogram, per-site
// histogram and the symmetrisation epilogues (co-transition counting: count_co.cu).
//
// Reference semantics (songlab-cal/CherryML v0.2.0):
//   quantisation  cherryml/utils.py:35-56  ==  counting/_count_transitions.cpp:295-307
//   LG loop       counting/_count_transitions.cpp:368-381 (cherry++), :444-506 (edge/cherry)
//   co loop       counting/_count_co_transitions.cpp:358-383, :469-531
// The reference adds 0.5 (or 0.25) to two (or four) cells per site; here each site adds ONE
// to a raw directed integer histogram and the halves/quarters are applied once at the end
// (cherry_symmetrize_*), which is exact because every addend is a multiple of 0.25.
//
// Layout in HBM (see DESIGN.md): residues are uint8 alphabet indices (255 = skip) in one
// flat buffer; a family's rows are 16-byte aligned with a row stride that is a multiple of
// 16; LG columns are sorted by site-rate category and each category is padded to a
// multiple of 4 sites, so that every aligned 32-bit word of a row has ONE category and the
// bucket of (pair, word) is a single byte lookup tab[pair][category].
#include "common.cuh"

namespace {

constexpr int kCountThreads = 1024;  // one CTA per SM, 32 warps to cover HBM latency
constexpr int kMaxSmemBytes = 227 * 1024;
// Padding cells per bucket of the LG shared-memory histogram (address-stream simulation: 2.92 -> 2.80
// wavefronts per reduction; sweep in profiles/ab/r02_count_lg_ab_v3.txt).
constexpr int kLgBucketPad = 5;

__device__ __forceinline__ uint4 ld_stream16(const uint8_t* p) {
  uint4 r;
  asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];"
               : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w)
               : "l"(p));
  return r;
}

// fp64 nearest-grid-point in relative error; -1 outside the grid.  Same expression, same
// rounding as the host definition (IEEE div.rn.f64, no contraction is possible here).
__device__ __forceinline__ int quantize_bucket(double t, const double* __restrict__ q, int K) {
  if (t < q[0] || t > q[K - 1]) return -1;
  int lo = 0, hi = K;
  while (lo < hi) {
    int mid = (lo + hi) >> 1;
    if (q[mid] < t) lo = mid + 1; else hi = mid;
  }
  if (lo == 0) return 0;
  double left = q[lo - 1], right = q[lo];
  // The reference compares t/left - 1 < right/t - 1.  In exact arithmetic that is
  // t*t < left*right; both quotients are ~1.0x, so their rounding can only flip the outcome
  // when the two sides agree to ~1e-15.  Decide by the products when the margin is clear
  // (>= 1e-12 relative) and only otherwise evaluate the reference expression itself.
  const double tt = __dmul_rn(t, t), lr = __dmul_rn(left, right);
  if (fabs(tt - lr) > 1e-12 * lr) return (tt < lr) ? lo - 1 : lo;
  double el = __dsub_rn(__ddiv_rn(t, left), 1.0);
  double er = __dsub_rn(__ddiv_rn(right, t), 1.0);
  return (el < er) ? lo - 1 : lo;
}

// Decision boundaries of the quantisation: for every pair of neighbouring grid points (left, right) the
// reference's predicate  t/left - 1 < right/t - 1  (IEEE division and subtraction, utils.py:35-56 ==
// _count_transitions.cpp:295-307) is monotone in t -- the rounded quotients are monotone -- so there is ONE
// smallest double bnd in (left, right] for which it is false, and  bucket(t) = #{i : bnd[i] <= t}.  The
// boundary is found by bisection on the bit patterns of the doubles with the predicate itself, so the
// result is the reference's by construction; quantising a value is then a float guess and two or three
// double compares instead of ~110 instructions.  Grids with repeated or non-positive points take the
// binary search of quantize_bucket instead (flag).
__device__ __forceinline__ bool quantization_predicate(double t, double left, double right) {
  return __dsub_rn(__ddiv_rn(t, left), 1.0) < __dsub_rn(__ddiv_rn(right, t), 1.0);
}
__device__ __forceinline__ double quantization_boundary(double left, double right) {
  long long lo = __double_as_longlong(left), hi = __double_as_longlong(right);  // predicate true at lo, false at hi
  // the switch point is within a few ulps of the geometric mean: bracket it there first (8 steps instead of ~50)
  const long long mid0 = __double_as_longlong(sqrt(left * right));
  if (mid0 - 128 > lo && mid0 + 128 < hi && quantization_predicate(__longlong_as_double(mid0 - 128), left, right) &&
      !quantization_predicate(__longlong_as_double(mid0 + 128), left, right)) {
    lo = mid0 - 128;
    hi = mid0 + 128;
  }
  while (hi - lo > 1) {
    const long long mid = lo + ((hi - lo) >> 1);
    const double t = __longlong_as_double(mid);
    const double el = __dsub_rn(__ddiv_rn(t, left), 1.0), er = __dsub_rn(__ddiv_rn(right, t), 1.0);
    if (el < er) lo = mid; else hi = mid;
  }
  return __longlong_as_double(hi);
}
// log2_t: float approximation of log2(t) (any value is correct, a good one saves steps of the two loops)
__device__ __forceinline__ int quantize_by_boundaries(double t, float log2_t, const double* __restrict__ q,
                                                      const double* __restrict__ bnd, int K, float log2_q0,
                                                      float inv_log2_step) {
  if (t < q[0] || t > q[K - 1]) return -1;
  const float g = (log2_t - log2_q0) * inv_log2_step;
  int b = g == g ? (int)fminf(fmaxf(g + 0.5f, 0.f), (float)(K - 1)) : 0;  // nearest grid index: the loops rarely move
  while (b > 0 && !(bnd[b - 1] <= t)) --b;
  while (b < K - 1 && bnd[b] <= t) ++b;
  return b;
}

// The bucket table, one WARP per tile: a tile's pairs belong to ONE family, so the family's rate values are
// read once per warp and a thread's only dependent load is its pair's branch length (coalesced); values are
// quantised against the precomputed decision boundaries.  Only the rows of pairs in `tiles` are written.
__global__ void __launch_bounds__(256)
bucket_table_tiles_kernel(const double* __restrict__ pair_t, const cherry_tile* __restrict__ tiles,
                          const cherry_fam_desc* __restrict__ fams, const double* __restrict__ rate_vals,
                          const double* __restrict__ grid, int K, int n_tiles, int r_pad,
                          uint8_t* __restrict__ tab) {
  extern __shared__ double sgrid[];  // [K] grid, [K] boundaries, [warps][r_pad] rate values, [warps][r_pad] floats log2(rate)
  __shared__ int general;
  double* sbnd = sgrid + K;
  double* srate = sbnd + K;
  float* slog = reinterpret_cast<float*>(srate + (size_t)(blockDim.x >> 5) * r_pad);  // [warps][r_pad] each
  if (threadIdx.x == 0) general = 0;
  for (int i = threadIdx.x; i < K; i += blockDim.x) sgrid[i] = grid[i];
  __syncthreads();
  for (int i = threadIdx.x; i < K - 1; i += blockDim.x) {
    const double left = sgrid[i], right = sgrid[i + 1];
    if (!(left > 0.0) || !(right > left) || !(right < 1e300)) {
      general = 1;
      sbnd[i] = right;
    } else {
      sbnd[i] = quantization_boundary(left, right);
    }
  }
  __syncthreads();
  const bool use_general = general != 0;
  const float log2_q0 = sgrid[0] > 0.0 ? log2f((float)sgrid[0]) : 0.0f;
  const float span = K > 1 && sgrid[0] > 0.0 ? log2f((float)(sgrid[K - 1] / sgrid[0])) : 0.0f;
  const float inv_log2_step = span > 0.0f ? (float)(K - 1) / span : 0.0f;
  // One WARP per tile from here on (no CTA barrier, so the descriptor -> family -> rates loads of the 64
  // warps of an SM overlap).  r_pad == 4: the four rate values live in registers; otherwise a warp-private
  // slice of shared memory holds them.
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, warps = blockDim.x >> 5;
  double* wrate = srate + (size_t)warp * r_pad;
  float* wlog = slog + (size_t)warp * r_pad;
  for (int tile = blockIdx.x * warps + warp; tile < n_tiles; tile += gridDim.x * warps) {
    const cherry_tile tl = tiles[tile];
    const cherry_fam_desc* fd = fams + tl.fam;
    const int n_rates = min(fd->n_rates, r_pad);
    const int rate_off = fd->rate_off;
    __syncwarp();
    for (int i = lane; i < r_pad; i += 32) {
      const double rv = i < n_rates ? __ldg(rate_vals + rate_off + i) : 0.0;
      wrate[i] = rv;
      wlog[i] = rv > 0.0 ? __log2f((float)rv) : 0.0f;
    }
    __syncwarp();
    for (int p0 = lane; p0 < tl.n_pairs; p0 += 4 * 32) {
      double t[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const int pl = p0 + u * 32;
        t[u] = pl < tl.n_pairs ? __ldg(pair_t + tl.pair_begin + pl) : 0.0;
      }
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const int pl = p0 + u * 32;
        if (pl >= tl.n_pairs) break;
        uint32_t* __restrict__ row = reinterpret_cast<uint32_t*>(tab + (int64_t)(tl.pair_begin + pl) * r_pad);
        const float lt = t[u] > 0.0 ? __log2f((float)t[u]) : 0.0f;  // one logarithm per pair: log2(t r) = log2 t + log2 r
        for (int r0 = 0; r0 < r_pad; r0 += 4) {
          uint32_t word = 0;
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            uint32_t out = CHERRY_NO_BUCKET;
            if (r0 + k < n_rates) {
              const double x = __dmul_rn(t[u], wrate[r0 + k]);
              const int b = use_general ? quantize_bucket(x, sgrid, K)
                                        : quantize_by_boundaries(x, lt + wlog[r0 + k], sgrid, sbnd, K, log2_q0, inv_log2_step);
              if (b >= 0) out = (uint32_t)b;
            }
            word |= out << (8 * k);
          }
          row[r0 >> 2] = word;
        }
      }
    }
  }
}

// ---- global-atomics fallback (histogram larger than shared memory) ----
__device__ __forceinline__ void count_word_global(unsigned long long* h64, uint32_t wa, uint32_t wb,
                                                  uint32_t bucket, int S, int SS, uint32_t S4) {
  if (bucket == CHERRY_NO_BUCKET) return;
  uint32_t m = __vcmpltu4(wa, S4) & __vcmpltu4(wb, S4);
  if (m == 0) return;
  const int base = (int)bucket * SS;
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    if (m & (0x80u << (8 * k))) {
      int x = (wa >> (8 * k)) & 0xff;
      int y = (wb >> (8 * k)) & 0xff;
      atomicAdd(h64 + base + x * S + y, 1ull);
    }
  }
}

// ---- shared-memory path: branch-free, predicated per site ----
// One aligned 32-bit word = 4 sites of one rate category (one bucket).  Validity of the 8
// residue bytes is ONE byte-parallel test: bytes are <= S (the skip code), so
// (byte + 0x80 - S) has bit 7 set iff the byte is the skip code; a word whose bucket is
// outside the grid gets all four bits set.  Per site: two IDP.4A (address = row base +
// 4*S*x + 4*y straight from the packed words, coefficient bytes select the site), one
// select, one shared-memory reduction (ATOMS.POPC.INC).  Skipped sites (a quarter of the
// lanes on Pfam-like data) all hit one junk word after the histogram, where they merge into
// a single access: fewer bank conflicts per instruction than v2's (S+1)-state junk rows and
// columns (3.4 -> ~2.9 wavefronts), which is the kernel's limiter.
// `sbase` = 32-bit shared address of the histogram [K][S][S]; bucket4 = 4*S*S;
// junk = sbase + 4*K*S*S.
// DP4A needs 4*S <= 255; otherwise the address is built with PRMT + IMAD.
struct LgCoef {
  uint32_t a[4], b[4];  // a[k] = (4*S) << 8k, b[k] = 4 << 8k
};

template <bool DP4A>
__device__ __forceinline__ void count_word_smem(uint32_t sbase, uint32_t wa, uint32_t wb,
                                                uint32_t bucket, uint32_t row4, uint32_t bucket4,
                                                uint32_t vm, uint32_t junk, const LgCoef& cf) {
  uint32_t v = ((wa + vm) | (wb + vm)) & 0x80808080u;
  if (bucket == CHERRY_NO_BUCKET) v = 0x80808080u;
  const uint32_t rowbase = sbase + bucket * bucket4;
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    uint32_t addr;
    if (DP4A) {
      addr = __dp4a(wb, cf.b[k], __dp4a(wa, cf.a[k], rowbase));
    } else {
      const uint32_t x = __byte_perm(wa, 0, 0x4440 | k);
      const uint32_t y = __byte_perm(wb, 0, 0x4440 | k);
      addr = rowbase + x * row4 + y * 4u;
    }
    // ATOMS.POPC.INC cannot be predicated (ptxas branches around it), so skipped sites are
    // redirected to ONE junk word instead: equal addresses merge into a single access.
    if (v & (0x80u << (8 * k))) addr = junk;
    asm volatile("red.shared.add.u32 [%0], 1;" ::"r"(addr) : "memory");
  }
}

// R4: the bucket-table row is exactly 4 bytes (<= 4 rate categories): one 32-bit load and a
// byte select per word instead of four byte loads.
template <bool SMEM, bool R4, bool DP4A>
__device__ __forceinline__ void count_item(uint32_t sbase, unsigned long long* h64, const uint4& va,
                                           const uint4& vb, const uint2& g,
                                           const uint8_t* __restrict__ trow, int S, int SS,
                                           uint32_t row4, uint32_t bucket4, uint32_t S4, uint32_t vm,
                                           uint32_t junk, const LgCoef& cf) {
  uint32_t b0, b1, b2, b3;
  if (R4) {
    const uint32_t t = __ldg(reinterpret_cast<const uint32_t*>(trow));
    b0 = __byte_perm(t, 0, 0x4440u | (g.x & 0xffffu));
    b1 = __byte_perm(t, 0, 0x4440u | (g.x >> 16));
    b2 = __byte_perm(t, 0, 0x4440u | (g.y & 0xffffu));
    b3 = __byte_perm(t, 0, 0x4440u | (g.y >> 16));
  } else {
    b0 = __ldg(trow + (g.x & 0xffffu));
    b1 = __ldg(trow + (g.x >> 16));
    b2 = __ldg(trow + (g.y & 0xffffu));
    b3 = __ldg(trow + (g.y >> 16));
  }
  if (SMEM) {
    count_word_smem<DP4A>(sbase, va.x, vb.x, b0, row4, bucket4, vm, junk, cf);
    count_word_smem<DP4A>(sbase, va.y, vb.y, b1, row4, bucket4, vm, junk, cf);
    count_word_smem<DP4A>(sbase, va.z, vb.z, b2, row4, bucket4, vm, junk, cf);
    count_word_smem<DP4A>(sbase, va.w, vb.w, b3, row4, bucket4, vm, junk, cf);
  } else {
    count_word_global(h64, va.x, vb.x, b0, S, SS, S4);
    count_word_global(h64, va.y, vb.y, b1, S, SS, S4);
    count_word_global(h64, va.z, vb.z, b2, S, SS, S4);
    count_word_global(h64, va.w, vb.w, b3, S, SS, S4);
  }
}

// Persistent: gridDim.x CTAs stride over tiles.  A work item is one 16-byte chunk (16
// sites) of one pair; consecutive threads take consecutive chunks, so a warp reads runs of
// contiguous bytes from the two rows.  Each thread keeps (pair, chunk) of its two in-flight
// items and advances them incrementally (no division in the loop).  SMEM=true: the whole
// [K][S][S] histogram lives in shared memory as uint32 and is flushed once; SMEM=false
// (histogram too large): global uint64 atomics.
template <bool SMEM, bool R4, bool DP4A>
__global__ void __launch_bounds__(kCountThreads, 1)
count_lg_kernel(const uint8_t* __restrict__ msa, const cherry_fam_desc* __restrict__ fams,
                const int32_t* __restrict__ pair_a, const int32_t* __restrict__ pair_b,
                const uint8_t* __restrict__ tab, int r_pad,
                const uint16_t* __restrict__ group_cat, const cherry_tile* __restrict__ tiles,
                int n_tiles, int K, int S, int bstride, unsigned long long* __restrict__ counts) {
  // bstride = cells per bucket in shared memory (>= S*S): a padded stride keeps the diagonals of different
  // buckets out of the same banks (address-stream simulation: 2.92 -> 2.80 wavefronts per reduction)
  extern __shared__ uint32_t hist[];
  const int SS = S * S;
  const int nbins = SMEM ? K * bstride : K * SS;
  const int tid = threadIdx.x;
  const uint32_t S4 = (uint32_t)S * 0x01010101u;
  const uint32_t row4 = 4u * S, bucket4 = 4u * (SMEM ? (uint32_t)bstride : (uint32_t)SS);
  const uint32_t vm = (0x80u - (uint32_t)S) * 0x01010101u;  // S <= 127 on this path
  LgCoef cf;
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    cf.a[k] = (row4 & 0xffu) << (8 * k);
    cf.b[k] = 4u << (8 * k);
  }
  uint32_t sbase = (uint32_t)__cvta_generic_to_shared(hist);
  asm volatile("" : "+r"(sbase));  // keep it in a register (ptxas re-derives it per use otherwise)
  const uint32_t junk = sbase + 4u * (uint32_t)nbins;
  if (SMEM) {
    for (int i = tid; i <= nbins; i += kCountThreads) hist[i] = 0;
    __syncthreads();
  }
  for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
    const cherry_tile tl = tiles[tile];
    const cherry_fam_desc fd = fams[tl.fam];
    const uint8_t* __restrict__ base = msa + fd.msa_off;
    const uint16_t* __restrict__ gc = group_cat + fd.aux_off;
    const uint32_t nch = (uint32_t)fd.n_chunks;
    const uint32_t n_items = (uint32_t)tl.n_pairs * nch;
    const int64_t stride = fd.row_stride;
    // per-thread (pair, chunk) cursors for items tid and tid + T, each advancing by 2T
    const uint32_t dq = (2 * kCountThreads) / nch, dr = (2 * kCountThreads) - dq * nch;
    uint32_t pl0 = (uint32_t)tid / nch, ch0 = (uint32_t)tid - pl0 * nch;
    uint32_t pl1 = (uint32_t)(tid + kCountThreads) / nch, ch1 = (uint32_t)(tid + kCountThreads) - pl1 * nch;
    for (uint32_t i = tid; i < n_items; i += 2 * kCountThreads) {
      const bool has1 = i + kCountThreads < n_items;
      const uint32_t q1 = has1 ? pl1 : pl0, c1 = has1 ? ch1 : ch0;
      const int p0 = tl.pair_begin + (int)pl0, p1 = tl.pair_begin + (int)q1;
      const int a0 = __ldg(pair_a + p0), b0 = __ldg(pair_b + p0);
      const int a1 = __ldg(pair_a + p1), b1 = __ldg(pair_b + p1);
      uint4 va0 = ld_stream16(base + a0 * stride + ch0 * 16);
      uint4 vb0 = ld_stream16(base + b0 * stride + ch0 * 16);
      uint4 va1 = ld_stream16(base + a1 * stride + c1 * 16);
      uint4 vb1 = ld_stream16(base + b1 * stride + c1 * 16);
      uint2 g0 = __ldg(reinterpret_cast<const uint2*>(gc + ch0 * 4));
      uint2 g1 = __ldg(reinterpret_cast<const uint2*>(gc + c1 * 4));
      count_item<SMEM, R4, DP4A>(sbase, counts, va0, vb0, g0, tab + (int64_t)p0 * r_pad, S, SS, row4, bucket4,
                                 S4, vm, junk, cf);
      if (has1)
        count_item<SMEM, R4, DP4A>(sbase, counts, va1, vb1, g1, tab + (int64_t)p1 * r_pad, S, SS, row4,
                                   bucket4, S4, vm, junk, cf);
      pl0 += dq; ch0 += dr;
      if (ch0 >= nch) { ch0 -= nch; ++pl0; }
      pl1 += dq; ch1 += dr;
      if (ch1 >= nch) { ch1 -= nch; ++pl1; }
    }
  }
  if (SMEM) {
    __syncthreads();
    for (int i = tid; i < K * SS; i += kCountThreads) {
      const int b = i / SS;
      const uint32_t v = hist[b * bstride + (i - b * SS)];
      if (v) atomicAdd(counts + i, (unsigned long long)v);
    }
  }
}

// Per-site counting (SiteRM): one CTA per cherry; the cherry's bucket is quantised once (fp64,
// same expression as everywhere else), then every site l adds one to counts[l][b][x][y].
__global__ void __launch_bounds__(256)
count_per_site_kernel(const uint8_t* __restrict__ xa, const uint8_t* __restrict__ xb,
                      const double* __restrict__ t, const double* __restrict__ grid, int B, int L,
                      int64_t row_stride, int S, unsigned long long* __restrict__ counts) {
  __shared__ int sb;
  const int64_t c = blockIdx.x;
  if (threadIdx.x == 0) sb = quantize_bucket(t[c], grid, B);
  __syncthreads();
  const int b = sb;
  if (b < 0) return;
  const uint8_t* ra = xa + c * row_stride;
  const uint8_t* rb = xb + c * row_stride;
  for (int l = threadIdx.x; l < L; l += blockDim.x) {
    const unsigned x = ra[l], y = rb[l];
    if (x < (unsigned)S && y < (unsigned)S)
      atomicAdd(counts + (((size_t)l * B + b) * S + x) * S + y, 1ull);
  }
}

// flag[0] |= 1 if any residue byte exceeds S (contract violation).
__global__ void validate_residues_kernel(const uint4* __restrict__ msa, int64_t n_vec, uint32_t S4,
                                         int* __restrict__ flag) {
  bool bad = false;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n_vec;
       i += (int64_t)gridDim.x * blockDim.x) {
    const uint4 v = msa[i];
    bad |= (__vcmpgtu4(v.x, S4) | __vcmpgtu4(v.y, S4) | __vcmpgtu4(v.z, S4) | __vcmpgtu4(v.w, S4)) != 0;
  }
  if (__any_sync(0xffffffffu, bad) && (threadIdx.x & 31) == 0) atomicOr(flag, 1);
}

__global__ void symmetrize_lg_kernel(const unsigned long long* __restrict__ raw, int K, int S,
                                     int directed, double* __restrict__ out) {
  const int SS = S * S;
  const int total = K * SS;
  for (int idx = blockIdx.x * blockDim.x + threadIdx.x; idx < total;
       idx += gridDim.x * blockDim.x) {
    int k = idx / SS, r = idx - k * SS;
    int x = r / S, y = r - x * S;
    unsigned long long a = raw[idx];
    if (directed) {
      out[idx] = (double)a;
    } else {
      unsigned long long b = raw[k * SS + y * S + x];
      out[idx] = 0.5 * (double)(a + b);
    }
  }
}

__global__ void symmetrize_co_kernel(const uint32_t* __restrict__ raw, int K, int S, int directed,
                                     double* __restrict__ out) {
  const size_t n = (size_t)S * S;
  const size_t total = (size_t)K * n * n;
  for (size_t idx = blockIdx.x * (size_t)blockDim.x + threadIdx.x; idx < total;
       idx += (size_t)gridDim.x * blockDim.x) {
    size_t k = idx / (n * n), r = idx - k * n * n;
    size_t s = r / n, e = r - s * n;
    size_t st = (s % S) * S + s / S, et = (e % S) * S + e / S;  // the two sites swapped
    const uint32_t* R = raw + k * n * n;
    unsigned long long v = (unsigned long long)R[s * n + e] + R[st * n + et];
    if (directed) {
      out[idx] = 0.5 * (double)v;
    } else {
      v += (unsigned long long)R[e * n + s] + R[et * n + st];
      out[idx] = 0.25 * (double)v;
    }
  }
}

int check_count_args(const void* msa, const void* fams, const void* pa, const void* pb,
                     const void* tab, const void* tiles, const void* counts, int n_tiles, int K,
                     int S, int r_pad) {
  if (!msa || !fams || !pa || !pb || !tab || !tiles || !counts)
    return cherry::fail(CHERRY_EINVAL, "count: null pointer argument");
  if (n_tiles < 0 || r_pad <= 0) return cherry::fail(CHERRY_EINVAL, "count: bad n_tiles/r_pad");
  if (K <= 0 || K > CHERRY_MAX_BUCKETS)
    return cherry::fail(CHERRY_ELIMIT, "count: K=%d outside 1..%d", K, CHERRY_MAX_BUCKETS);
  if (S <= 0 || S > 254) return cherry::fail(CHERRY_ELIMIT, "count: S=%d outside 1..254", S);
  return 0;
}

}  // namespace

extern "C" {

int cherry_count_lg(const uint8_t* msa, const cherry_fam_desc* fams, const int32_t* pair_a,
                    const int32_t* pair_b, const uint8_t* tab, int r_pad,
                    const uint16_t* group_cat, const cherry_tile* tiles, int n_tiles, int K,
                    int S, unsigned long long* counts, void* stream) {
  int rc = check_count_args(msa, fams, pair_a, pair_b, tab, tiles, counts, n_tiles, K, S, r_pad);
  if (rc) return rc;
  if (!group_cat) return cherry::fail(CHERRY_EINVAL, "count_lg: null group_cat");
  if (n_tiles == 0) return 0;
  cudaStream_t st = (cudaStream_t)stream;
  int bstride = S * S + kLgBucketPad;
  if (((size_t)K * bstride + 4) * sizeof(uint32_t) > (size_t)kMaxSmemBytes) bstride = S * S;
  const size_t hist_bytes = ((size_t)K * bstride + 4) * sizeof(uint32_t);  // + the junk word
  int grid = cherry::sm_count();
  if (grid > n_tiles) grid = n_tiles;
  const bool r4 = (r_pad == 4);
#define CHERRY_LG_LAUNCH(SM, R, D, SH)                                                          \
  count_lg_kernel<SM, R, D><<<grid, kCountThreads, SH, st>>>(msa, fams, pair_a, pair_b, tab,    \
                                                              r_pad, group_cat, tiles, n_tiles, K, S, bstride, counts)
  if (hist_bytes <= (size_t)kMaxSmemBytes && S <= 127) {
    static bool attr_set[64] = {false};
    int dev = 0;
    CHERRY_CUDA(cudaGetDevice(&dev));
    if (dev < 64 && !attr_set[dev]) {
      CHERRY_CUDA(cudaFuncSetAttribute(count_lg_kernel<true, true, true>,
                                       cudaFuncAttributeMaxDynamicSharedMemorySize, kMaxSmemBytes));
      CHERRY_CUDA(cudaFuncSetAttribute(count_lg_kernel<true, false, true>,
                                       cudaFuncAttributeMaxDynamicSharedMemorySize, kMaxSmemBytes));
      CHERRY_CUDA(cudaFuncSetAttribute(count_lg_kernel<true, false, false>,
                                       cudaFuncAttributeMaxDynamicSharedMemorySize, kMaxSmemBytes));
      attr_set[dev] = true;
    }
    if (4 * S > 255)
      CHERRY_LG_LAUNCH(true, false, false, hist_bytes);
    else if (r4)
      CHERRY_LG_LAUNCH(true, true, true, hist_bytes);
    else
      CHERRY_LG_LAUNCH(true, false, true, hist_bytes);
  } else {
    CHERRY_LG_LAUNCH(false, false, false, 0);
  }
#undef CHERRY_LG_LAUNCH
  CHERRY_LAUNCH_CHECK("count_lg_kernel");
  return 0;
}

int cherry_build_bucket_table_tiles(const double* pair_t, const cherry_tile* tiles, int n_tiles,
                                    const cherry_fam_desc* fams, const double* rate_vals, const double* grid,
                                    int K, int r_pad, uint8_t* tab, void* stream) {
  if (!pair_t || !tiles || !fams || !rate_vals || !grid || !tab)
    return cherry::fail(CHERRY_EINVAL, "bucket_table_tiles: null pointer argument");
  if (K <= 0 || K > CHERRY_MAX_BUCKETS)
    return cherry::fail(CHERRY_ELIMIT, "bucket_table_tiles: K=%d outside 1..%d", K, CHERRY_MAX_BUCKETS);
  if (n_tiles < 0 || r_pad <= 0 || r_pad % 4 != 0)
    return cherry::fail(CHERRY_EINVAL, "bucket_table_tiles: bad sizes (r_pad must be a positive multiple of 4)");
  if (n_tiles == 0) return 0;
  int blocks = (n_tiles + 7) / 8;           // 8 warps per CTA, one warp per tile
  const int cap = cherry::sm_count() * 8;  // one residency: every CTA computes the boundaries once
  if (blocks > cap) blocks = cap;
  bucket_table_tiles_kernel<<<blocks, 256, (2 * K + 8 * r_pad) * sizeof(double) + 8 * r_pad * sizeof(float), (cudaStream_t)stream>>>(
      pair_t, tiles, fams, rate_vals, grid, K, n_tiles, r_pad, tab);
  CHERRY_LAUNCH_CHECK("bucket_table_tiles_kernel");
  return 0;
}

int cherry_count_per_site(const uint8_t* xa, const uint8_t* xb, const double* t, int64_t n_cherries,
                          int L, int64_t row_stride, const double* grid, int B, int S,
                          unsigned long long* counts, void* stream) {
  if (!xa || !xb || !t || !grid || !counts) return cherry::fail(CHERRY_EINVAL, "count_per_site: null pointer");
  if (L <= 0 || B <= 0 || S <= 0 || S > 254 || row_stride < L || n_cherries < 0)
    return cherry::fail(CHERRY_EINVAL, "count_per_site: bad sizes");
  if (n_cherries == 0) return 0;
  if (n_cherries > 0x7fffffff) return cherry::fail(CHERRY_ELIMIT, "count_per_site: too many cherries");
  count_per_site_kernel<<<(unsigned)n_cherries, 256, 0, (cudaStream_t)stream>>>(xa, xb, t, grid, B, L, row_stride,
                                                                                S, counts);
  CHERRY_LAUNCH_CHECK("count_per_site_kernel");
  return 0;
}

int cherry_validate_residues(const uint8_t* msa, int64_t n_bytes, int S, int* flag, void* stream) {
  if (!msa || !flag) return cherry::fail(CHERRY_EINVAL, "validate_residues: null pointer");
  if (S <= 0 || S > 254 || n_bytes < 0 || (n_bytes % 16) != 0)
    return cherry::fail(CHERRY_EINVAL, "validate_residues: bad S or size (must be a multiple of 16)");
  if (n_bytes == 0) return 0;
  const int64_t n_vec = n_bytes / 16;
  int64_t want = (n_vec + 255) / 256;
  int cap = cherry::sm_count() * 16;
  int blocks = (int)(want < cap ? want : cap);
  validate_residues_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>(
      reinterpret_cast<const uint4*>(msa), n_vec, (uint32_t)S * 0x01010101u, flag);
  CHERRY_LAUNCH_CHECK("validate_residues_kernel");
  return 0;
}

int cherry_symmetrize_lg(const unsigned long long* raw, int K, int S, int directed, double* out,
                         void* stream) {
  if (!raw || !out) return cherry::fail(CHERRY_EINVAL, "symmetrize_lg: null pointer");
  if (K <= 0 || S <= 0) return cherry::fail(CHERRY_EINVAL, "symmetrize_lg: bad sizes");
  int total = K * S * S;
  int blocks = (total + 255) / 256;
  symmetrize_lg_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>(raw, K, S, directed, out);
  CHERRY_LAUNCH_CHECK("symmetrize_lg_kernel");
  return 0;
}

int cherry_symmetrize_co(const uint32_t* raw, int K, int S, int directed, double* out,
                         void* stream) {
  if (!raw || !out) return cherry::fail(CHERRY_EINVAL, "symmetrize_co: null pointer");
  if (K <= 0 || S <= 0) return cherry::fail(CHERRY_EINVAL, "symmetrize_co: bad sizes");
  size_t total = (size_t)K * S * S * S * S;
  size_t want = (total + 255) / 256;
  int cap = cherry::sm_count() * 16;
  int blocks = (int)(want < (size_t)cap ? want : (size_t)cap);
  symmetrize_co_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>(raw, K, S, directed, out);
  CHERRY_LAUNCH_CHECK("symmetrize_co_kernel");
  return 0;
}

}  // extern "C"

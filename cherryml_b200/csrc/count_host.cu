// Host-buffer entry point of LG counting (the end-to-end path bench.py times as `e2e`).
//
// This is what a maintainer binds in place of the `mpirun ... _count_transitions` command
// line of the reference (counting/_count_transitions.py:295-316): the caller hands over
// HOST arrays; the residue buffer is copied to the device in family segments on a copy
// stream while the compute stream counts the previous segment, the small per-pair arrays
// go first, and only the K*S*S fp64 result comes back.
#include <algorithm>
#include <vector>

#include "common.cuh"

namespace {

struct HostPathState {
  void* ws = nullptr;
  size_t ws_bytes = 0;
  cudaStream_t copy_stream = nullptr, compute_stream = nullptr;
  std::vector<cudaEvent_t> events;
  int device = -1;
};

HostPathState& state() {
  static thread_local HostPathState s;
  return s;
}

inline size_t align_up(size_t x, size_t a = 256) { return (x + a - 1) / a * a; }

int ensure_state(size_t need_bytes, int n_events) {
  HostPathState& s = state();
  int dev = 0;
  CHERRY_CUDA(cudaGetDevice(&dev));
  if (s.device != dev) {
    // first use on this device (or the thread switched device): start clean
    if (s.ws) cudaFree(s.ws);
    s.ws = nullptr;
    s.ws_bytes = 0;
    for (cudaEvent_t e : s.events) cudaEventDestroy(e);
    s.events.clear();
    if (s.copy_stream) cudaStreamDestroy(s.copy_stream);
    if (s.compute_stream) cudaStreamDestroy(s.compute_stream);
    CHERRY_CUDA(cudaStreamCreateWithFlags(&s.copy_stream, cudaStreamNonBlocking));
    CHERRY_CUDA(cudaStreamCreateWithFlags(&s.compute_stream, cudaStreamNonBlocking));
    s.device = dev;
  }
  if (s.ws_bytes < need_bytes) {
    if (s.ws) CHERRY_CUDA(cudaFree(s.ws));
    s.ws = nullptr;
    s.ws_bytes = 0;
    CHERRY_CUDA(cudaMalloc(&s.ws, need_bytes));
    s.ws_bytes = need_bytes;
  }
  while ((int)s.events.size() < n_events) {
    cudaEvent_t e;
    CHERRY_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    s.events.push_back(e);
  }
  return 0;
}

}  // namespace

extern "C" int cherry_count_lg_host(
    const uint8_t* msa, int64_t msa_bytes, const cherry_fam_desc* fams, int n_fams,
    const int32_t* pair_a, const int32_t* pair_b, const double* pair_t, int64_t n_pairs,
    const double* rate_vals, int64_t n_rate_vals, const uint16_t* group_cat, int64_t n_groups,
    const cherry_tile* tiles, int n_tiles, const double* grid, int K, int S, int r_pad, int directed,
    double* counts_out, int64_t* h2d_bytes, int64_t* d2h_bytes) {
  if (!msa || !fams || !pair_a || !pair_b || !pair_t || !rate_vals || !group_cat ||
      !tiles || !grid || !counts_out)
    return cherry::fail(CHERRY_EINVAL, "count_lg_host: null pointer argument");
  if (K <= 0 || K > CHERRY_MAX_BUCKETS)
    return cherry::fail(CHERRY_ELIMIT, "count_lg_host: K=%d outside 1..%d", K, CHERRY_MAX_BUCKETS);
  if (S <= 0 || S > 255 || r_pad <= 0 || n_fams <= 0 || n_pairs < 0 || n_tiles < 0 || msa_bytes <= 0)
    return cherry::fail(CHERRY_EINVAL, "count_lg_host: bad sizes");
  for (int t = 1; t < n_tiles; ++t)
    if (tiles[t].fam < tiles[t - 1].fam)
      return cherry::fail(CHERRY_EINVAL, "count_lg_host: tiles must be ordered by family");
  for (int f = 1; f < n_fams; ++f)
    if (fams[f].msa_off < fams[f - 1].msa_off)
      return cherry::fail(CHERRY_EINVAL, "count_lg_host: families must be ordered by msa_off");

  const size_t nb = (size_t)K * S * S;
  // carve the workspace
  size_t off = 0;
  auto carve = [&](size_t bytes) { size_t o = off; off = align_up(off + bytes); return o; };
  const size_t o_msa = carve((size_t)msa_bytes);
  const size_t o_fams = carve((size_t)n_fams * sizeof(cherry_fam_desc));
  const size_t o_pa = carve((size_t)n_pairs * 4), o_pb = carve((size_t)n_pairs * 4);
  const size_t o_pt = carve((size_t)n_pairs * 8);
  const size_t o_rv = carve((size_t)n_rate_vals * 8);
  const size_t o_gc = carve((size_t)n_groups * 2);
  const size_t o_tl = carve((size_t)n_tiles * sizeof(cherry_tile));
  const size_t o_grid = carve((size_t)K * 8);
  const size_t o_tab = carve((size_t)n_pairs * r_pad);
  const size_t o_raw = carve(nb * 8), o_out = carve(nb * 8);

  // family segments of roughly equal residue bytes
  const int max_seg = 16;
  std::vector<int> seg_fam_begin;  // family index where each segment starts
  {
    const int64_t target = std::max<int64_t>(msa_bytes / max_seg, 8 << 20);
    int64_t next = 0;
    for (int f = 0; f < n_fams; ++f) {
      if (fams[f].msa_off >= next) {
        seg_fam_begin.push_back(f);
        next = fams[f].msa_off + target;
      }
    }
  }
  const int n_seg = (int)seg_fam_begin.size();
  int rc = ensure_state(off, n_seg + 1);
  if (rc) return rc;
  HostPathState& s = state();
  char* w = (char*)s.ws;
  auto H2D = [&](size_t o, const void* src, size_t bytes) -> cudaError_t {
    if (bytes == 0) return cudaSuccess;
    return cudaMemcpyAsync(w + o, src, bytes, cudaMemcpyHostToDevice, s.copy_stream);
  };
  CHERRY_CUDA(H2D(o_fams, fams, (size_t)n_fams * sizeof(cherry_fam_desc)));
  CHERRY_CUDA(H2D(o_pa, pair_a, (size_t)n_pairs * 4));
  CHERRY_CUDA(H2D(o_pb, pair_b, (size_t)n_pairs * 4));
  CHERRY_CUDA(H2D(o_pt, pair_t, (size_t)n_pairs * 8));
  CHERRY_CUDA(H2D(o_rv, rate_vals, (size_t)n_rate_vals * 8));
  CHERRY_CUDA(H2D(o_gc, group_cat, (size_t)n_groups * 2));
  CHERRY_CUDA(H2D(o_tl, tiles, (size_t)n_tiles * sizeof(cherry_tile)));
  CHERRY_CUDA(H2D(o_grid, grid, (size_t)K * 8));
  CHERRY_CUDA(cudaEventRecord(s.events[n_seg], s.copy_stream));
  CHERRY_CUDA(cudaStreamWaitEvent(s.compute_stream, s.events[n_seg], 0));
  CHERRY_CUDA(cudaMemsetAsync(w + o_raw, 0, nb * 8, s.compute_stream));
  rc = cherry_build_bucket_table_tiles((const double*)(w + o_pt), (const cherry_tile*)(w + o_tl), n_tiles,
                                       (const cherry_fam_desc*)(w + o_fams), (const double*)(w + o_rv),
                                       (const double*)(w + o_grid), K, r_pad, (uint8_t*)(w + o_tab),
                                       s.compute_stream);
  if (rc) return rc;

  int tile_pos = 0;
  for (int sg = 0; sg < n_seg; ++sg) {
    const int f0 = seg_fam_begin[sg];
    const int f1 = (sg + 1 < n_seg) ? seg_fam_begin[sg + 1] : n_fams;
    const int64_t b0 = fams[f0].msa_off;
    const int64_t b1 = (f1 < n_fams) ? fams[f1].msa_off : msa_bytes;
    CHERRY_CUDA(H2D(o_msa + (size_t)b0, msa + b0, (size_t)(b1 - b0)));
    CHERRY_CUDA(cudaEventRecord(s.events[sg], s.copy_stream));
    CHERRY_CUDA(cudaStreamWaitEvent(s.compute_stream, s.events[sg], 0));
    int t0 = tile_pos;
    while (tile_pos < n_tiles && tiles[tile_pos].fam < f1) ++tile_pos;
    if (tile_pos > t0) {
      rc = cherry_count_lg((const uint8_t*)(w + o_msa), (const cherry_fam_desc*)(w + o_fams),
                           (const int32_t*)(w + o_pa), (const int32_t*)(w + o_pb),
                           (const uint8_t*)(w + o_tab), r_pad, (const uint16_t*)(w + o_gc),
                           (const cherry_tile*)(w + o_tl) + t0, tile_pos - t0, K, S,
                           (unsigned long long*)(w + o_raw), s.compute_stream);
      if (rc) return rc;
    }
  }
  rc = cherry_symmetrize_lg((const unsigned long long*)(w + o_raw), K, S, directed,
                            (double*)(w + o_out), s.compute_stream);
  if (rc) return rc;
  CHERRY_CUDA(cudaMemcpyAsync(counts_out, w + o_out, nb * 8, cudaMemcpyDeviceToHost,
                              s.compute_stream));
  CHERRY_CUDA(cudaStreamSynchronize(s.compute_stream));
  if (h2d_bytes)
    *h2d_bytes = msa_bytes + (int64_t)n_fams * (int64_t)sizeof(cherry_fam_desc) + n_pairs * 16 +
                 n_rate_vals * 8 + n_groups * 2 + (int64_t)n_tiles * (int64_t)sizeof(cherry_tile) +
                 (int64_t)K * 8;
  if (d2h_bytes) *d2h_bytes = (int64_t)nb * 8;
  return 0;
}

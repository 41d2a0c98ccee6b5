/* cherryml_b200 -- C ABI of the B200-native CherryML hot path.
 *
 * Every entry point takes plain pointers and sizes.  Unless a name ends in `_host`, all
 * data pointers are DEVICE pointers owned by the caller (PyTorch allocates them), no
 * entry point allocates device memory, work is enqueued on `stream` (a cudaStream_t
 * passed as void*) and the call returns without synchronising.  Return value: 0 on
 * success, a negative CHERRY_E* code otherwise; cherry_last_error() gives the message
 * of the last failure on the calling thread.
 *
 * What each entry point replaces in the reference (paths relative to the reference
 * checkout, songlab-cal/CherryML v0.2.0):
 *
 *   cherry_build_bucket_table_tiles
 *                              quantization_idx(), cherryml/utils.py:35-56 ==
 *                              counting/_count_transitions.cpp:295-307, evaluated once
 *                              per (pair, rate category) instead of once per site.
 *   cherry_count_lg            the per-site loop of _dfs()/_map_func(),
 *                              counting/_count_transitions.cpp:368-381, 444-506 and
 *                              counting/_count_transitions.py:96-126, 129-186; the CLI
 *                              it was reached through is _count_transitions.py:295-310.
 *   cherry_count_co            the per-contact loop, counting/_count_co_transitions.cpp
 *                              :358-383, 469-531 (CLI: _count_co_transitions.py:324-340).
 *   cherry_symmetrize_lg/_co   the "+= 0.5 twice" / "+= 0.25 four times" updates of the
 *                              same loops, applied once to the raw directed histogram,
 *                              and the rank-0 text-file reduction (.cpp:654-671).
 *   cherry_fit_*               RateMatrix.forward (estimation/_ratelearn/rate.py:167-188),
 *                              the epoch body of train_quantization
 *                              (estimation/_ratelearn/trainer.py:156-187: matrix_exp,
 *                              log, sum, backward, optimizer.step, best-iterate) and
 *                              torch.optim.Adam as configured at ratelearner.py:123-126.
 *   cherry_expm_batched        matrix_exponential_pytorch, markov_chain/_markov_chain.py
 *                              :22-53.
 *   cherry_fc_pair             divide_and_pair(), phylogeny_estimation/FastCherries/
 *                              pairing_algorithms.cpp:15-175 (called per family at
 *                              fast_cherries.cpp:240-244).
 *   cherry_fc_ble              ble(), FastCherries/branch_length_estimation.cpp:10-241
 *                              (fast_cherries.cpp:258-266).
 *   cherry_tree_log_likelihood the pruning loops of dp_likelihood_computation,
 *                              evaluation/_likelihood.py:239-326.
 *   cherry_fc_lengths_and_rates / cherry_fc_count_layout / cherry_fc_relayout_lg
 *                              the text hand-off between the tree estimator and the counting stage
 *                              (estimation_end_to_end/_cherry.py:279-336), done in memory with the
 *                              values the files would carry.
 *   cherry_ingest_* / cherry_fc_read_msas / cherry_fc_write_outputs / cherry_*_count_matrices /
 *   cherry_write_labelled_matrix   (host threads) the text readers and writers of cherryml/io and of
 *                              the two C++ programs, byte-identical formats.
 */
#ifndef CHERRYML_B200_H
#define CHERRYML_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CHERRY_OK 0
#define CHERRY_EINVAL (-1)  /* bad argument (null pointer, size out of range) */
#define CHERRY_ECUDA (-2)   /* CUDA runtime error; message has the cudaError string */
#define CHERRY_ELIMIT (-3)  /* size beyond what the kernels support (e.g. K > 254) */

/* Residue bytes are alphabet indices 0..S-1; the byte value S (== num_states) means "skip"
 * (gap, unknown letter, padding).  No byte may exceed S: the LG kernel indexes an
 * (S+1)-state shared-memory histogram with it without clamping. */
#define CHERRY_NO_BUCKET 255u       /* bucket-table entry for "outside the grid" */
#define CHERRY_MAX_BUCKETS 254

/* One MSA family inside the flat residue buffer.  32 bytes. */
typedef struct cherry_fam_desc {
  int64_t msa_off;    /* byte offset of the family's row 0 in the residue buffer (16-aligned) */
  int32_t row_stride; /* bytes per row, a multiple of 16; bytes past the real sites are S (skip) */
  int32_t n_chunks;   /* row_stride / 16 */
  int32_t aux_off;    /* LG: first entry of this family in group_cat[] (one per 4 sites);
                         co-transitions: first entry of this family in the host-side contact
                         list (not read by the kernels) */
  int32_t aux_cnt;    /* LG: row_stride / 4; co-transitions: number of contacting pairs
                         (row bytes 2c, 2c+1 for c < aux_cnt are residues, the rest is S) */
  int32_t rate_off;   /* first entry of this family in rate_vals[] */
  int32_t n_rates;    /* number of distinct site-rate values (co-transitions: 1) */
} cherry_fam_desc;

/* A tile is a run of consecutive pairs of one family: {family, first_pair, n_pairs, 0}. */
typedef struct cherry_tile {
  int32_t fam;
  int32_t pair_begin; /* index into pair_a / pair_b / bucket table */
  int32_t n_pairs;
  int32_t reserved;
} cherry_tile;

const char* cherry_last_error(void);
const char* cherry_version(void);
/* Number of kernels this library has launched since load (or the last reset). */
int64_t cherry_launch_count(void);
void cherry_reset_launch_count(void);

/* ---------------------------------------------------------------- counting */

/* counts[b][x][y] += #sites of all pairs with bucket b, residue x on row pair_a, residue y
 * on row pair_b (raw, directed).  group_cat[fam.aux_off + g] is the rate category of
 * sites 4g..4g+3 of the family's (category-sorted, 4-aligned) columns.
 * counts: uint64 [K][S][S], accumulated into (caller zeroes it). */
int cherry_count_lg(const uint8_t* msa, const cherry_fam_desc* fams, const int32_t* pair_a,
                    const int32_t* pair_b, const uint8_t* tab, int r_pad,
                    const uint16_t* group_cat, const cherry_tile* tiles, int n_tiles, int K,
                    int S, unsigned long long* counts, void* stream);

/* The bucket table: for every pair p of every tile in `tiles` (tile.fam = the pair's family f),
 * tab[p * r_pad + r] = bucket of (pair_t[p] * rate_vals[fams[f].rate_off + r]) for r < n_rates of f,
 * CHERRY_NO_BUCKET for n_rates <= r < r_pad; rows of pairs in no tile are not written.  grid: K ascending
 * fp64 quantization points.  fp64 throughout, bit-identical to the host definition.  Built one warp per
 * TILE (a tile's pairs share a family: its rate values are read once per warp, a pair costs one coalesced
 * load) and quantised against precomputed decision boundaries: for neighbouring grid points (left, right)
 * the reference's predicate t/left - 1 < right/t - 1 is monotone in t, so its switch point is found once
 * per launch by bisection on the doubles with the predicate itself (grids with repeated or non-positive
 * points use a binary search instead).  r_pad: a positive multiple of 4. */
int cherry_build_bucket_table_tiles(const double* pair_t, const cherry_tile* tiles, int n_tiles,
                                    const cherry_fam_desc* fams, const double* rate_vals, const double* grid,
                                    int K, int r_pad, uint8_t* tab, void* stream);

/* One sorted pair as the co-transition kernel's producer reads it.  16 bytes. */
typedef struct cherry_co_rec {
  int64_t off_a;     /* byte offset of the pair's row a in the residue buffer */
  int32_t delta_b16; /* (offset of row b - offset of row a) / 16 */
  int32_t stride;    /* bytes per row */
} cherry_co_rec;

/* Counting sort of the pairs by their bucket tab[p * r_pad] (co-transitions: one bucket per
 * pair).  Reads tab[p * r_pad] for every p < n_pairs: with a table from
 * cherry_build_bucket_table_tiles, every such pair must lie in exactly one tile.
 * order: int32 [n_pairs] (out) = pair indices grouped by bucket, ascending bucket.
 * recs: [n_pairs] (out, may be NULL) = the row addresses of order[]'s pairs, resolved here
 * through pair_fam / fams / pair_a / pair_b.
 * ws: int32 [2 * (K + 2)] (out / scratch): ws[b] = first position of bucket b in order[],
 * ws[K] = number of pairs inside the grid (the pairs outside it follow), ws[K + 1] = n_pairs.
 * The order inside a bucket is unspecified (the counts do not depend on it). */
int cherry_sort_pairs_by_bucket(const uint8_t* tab, int r_pad, int64_t n_pairs, int K,
                                const cherry_fam_desc* fams, const int32_t* pair_a,
                                const int32_t* pair_b, const int32_t* pair_fam, int32_t* order,
                                cherry_co_rec* recs, int32_t* ws, void* stream);

/* counts[b][S*xi+xj][S*yi+yj] += 1 for every (pair, contact c) with b = the pair's bucket,
 * (xi, xj) = bytes (2c, 2c+1) of row a and (yi, yj) = the same bytes of row b: rows of a
 * co-transition batch are CONTACT-PAIRED (bytes 2c, 2c+1 = residues at the two sites of
 * the family's c-th contacting pair, padded with the skip code S to row_stride).
 * recs / bucket_start: outputs of cherry_sort_pairs_by_bucket (bucket_start = ws).
 * max_row_stride: upper bound of the row strides in the batch (<= 16384).
 * counts: uint32 [K][S*S][S*S], accumulated into; the caller keeps (pairs x contacts) per
 * call below 2^32 so that no cell can wrap.
 * Replaces the per-contact loop of counting/_count_co_transitions.cpp:358-383, 469-531. */
int cherry_count_co(const uint8_t* msa, const cherry_co_rec* recs, const int32_t* bucket_start,
                    int64_t n_pairs, int max_row_stride, int K, int S, uint32_t* counts,
                    void* stream);

/* Per-site counting (SiteRM): counts[l][b][x][y] += 1 for every cherry c and site l, where
 * b = bucket of t[c] on `grid` (B ascending points), x = xa[c*row_stride + l], y = xb[...];
 * cherries outside the grid and residues >= S are skipped.  counts: uint64 [L][B][S][S],
 * accumulated into; symmetrise with cherry_symmetrize_lg(K = L*B).  Replaces
 * _get_raw_count_matrices, reference _siterm/_site_specific_rate_matrix.py:189-261. */
int cherry_count_per_site(const uint8_t* xa, const uint8_t* xb, const double* t, int64_t n_cherries,
                          int L, int64_t row_stride, const double* grid, int B, int S,
                          unsigned long long* counts, void* stream);

/* Sets flag[0] (device int, caller zeroes it) to 1 if any of the n_bytes (multiple of 16)
 * residue bytes exceeds S.  Optional guard for buffers that did not come from this
 * package's encoder. */
int cherry_validate_residues(const uint8_t* msa, int64_t n_bytes, int S, int* flag, void* stream);

/* out (fp64 [K][S][S]) = directed ? raw : (raw + raw^T) / 2. */
int cherry_symmetrize_lg(const unsigned long long* raw, int K, int S, int directed,
                         double* out, void* stream);
/* n = S*S; Pi(S*i+j) = S*j+i.  out (fp64 [K][n][n]) =
 * directed ? (R + Pi R Pi^T)/2 : (R + R^T + Pi R Pi^T + Pi R^T Pi^T)/4. */
int cherry_symmetrize_co(const uint32_t* raw, int K, int S, int directed, double* out,
                         void* stream);

/* Host-buffer entry point (end-to-end path): every pointer is a HOST pointer (pinned
 * memory makes the copies asynchronous).  Copies the batch to the device in family
 * segments overlapped with counting, and writes the symmetrised fp64 counts [K][S][S]
 * to counts_out on the host.  Synchronises before returning. */
int cherry_count_lg_host(const uint8_t* msa, int64_t msa_bytes, const cherry_fam_desc* fams,
                         int n_fams, const int32_t* pair_a, const int32_t* pair_b,
                         const double* pair_t, int64_t n_pairs,
                         const double* rate_vals, int64_t n_rate_vals,
                         const uint16_t* group_cat, int64_t n_groups,
                         const cherry_tile* tiles, int n_tiles, const double* grid, int K,
                         int S, int r_pad, int directed, double* counts_out,
                         int64_t* h2d_bytes, int64_t* d2h_bytes);

/* ------------------------------------------------------------------ ingest (host) */

/* An encoded batch built by cherry_ingest_lg / cherry_ingest_co: HOST arrays in exactly the
 * layout the counting entry points take (the library owns them; release with
 * cherry_ingest_free).  `msa` is page-locked when `pinned` is 1. */
typedef struct cherry_ingest_result {
  int32_t kind;        /* 0 = LG, 1 = co-transitions */
  int32_t pinned;
  int64_t msa_bytes;
  uint8_t* msa;
  int32_t n_fams;
  int32_t r_pad;
  cherry_fam_desc* fams;
  int64_t n_pairs;
  int32_t* pair_a;
  int32_t* pair_b;
  double* pair_t;
  int32_t* pair_fam;
  int64_t n_rate_vals;
  double* rate_vals;
  int64_t n_aux;       /* LG: entries of group_cat; co: contacting pairs */
  void* aux;           /* LG: uint16 group_cat[n_aux]; co: int32 contacts[n_aux][2] */
  int32_t n_tiles;
  int32_t max_row_stride;
  cherry_tile* tiles;
  int64_t n_items_examined; /* (pair, site) or (pair, contact) items before validity */
} cherry_ingest_result;

/* Parse `<dir>/<family>.txt` of every family with n_threads host threads and encode them
 * for cherry_count_lg: trees -> leaf pairs (edge_or_cherry = "cherry++", "cherry" or "edge"),
 * MSAs -> residue rows (alphabet = `states`, n_states one-character strings), site rates ->
 * rate categories and the category-sorted column layout.  float32_branch_lengths != 0 parses
 * branch lengths like the reference C++ program (std::stof, _count_transitions.cpp:247).
 * Replaces read_tree / read_msa / read_site_rates and _dfs of counting/_count_transitions.cpp
 * (:209-293, :316-390) with the accept/reject behaviour of the Python readers (io/_tree.py
 * :214-265, io/_msa.py:51-73, io/_site_rates.py:5-26). */
int cherry_ingest_lg(const char* tree_dir, const char* msa_dir, const char* site_rates_dir,
                     const char* const* families, int n_fams, const char* const* states,
                     int n_states, const char* edge_or_cherry, int float32_branch_lengths,
                     int n_threads, int pinned, cherry_ingest_result** out);
/* Same for cherry_count_co: contact maps -> contacting pairs (i < j, j - i >=
 * minimum_distance, map[i][j] == '1'; io/_contact_map.py:6-28, _count_co_transitions.cpp
 * :433-442) and contact-paired rows. */
int cherry_ingest_co(const char* tree_dir, const char* msa_dir, const char* contact_map_dir,
                     const char* const* families, int n_fams, const char* const* states,
                     int n_states, const char* edge_or_cherry, int minimum_distance,
                     int float32_branch_lengths, int n_threads, int pinned,
                     cherry_ingest_result** out);
void cherry_ingest_free(cherry_ingest_result* result);

/* ------------------------------------------------------------------- fit */

/* Everything the fit keeps on the device.  One "problem" is one rate matrix with its K time
 * buckets; n_problems > 1 is the batched per-site fit (independent problems, same S and K).
 * theta[p] = {S pi logits, S(S-1)/2 upper-diagonal entries in row-major order}; Q(theta) is
 * the "pande_reversible" parameterisation (reference rate.py:167-188).  All arrays fp64. */
typedef struct cherry_fit_args {
  int S, K, n_problems;
  const double* t;     /* [n_problems*K] bucket times */
  const double* C;     /* [n_problems*K][S][S] count matrices */
  const double* mask;  /* [S][S] 0/1 */
  const double* sumC;  /* [n_problems] sum of C per problem */
  double* theta;       /* [n_problems][S + S(S-1)/2] */
  double* adam_m;      /* same shape as theta, zero at start */
  double* adam_v;
  double* Q;           /* [n_problems][S][S] current rate matrix */
  double* Q_best;      /* [n_problems][S][S] */
  double* Q_last;      /* [n_problems][S][S] Q the most recent loss was evaluated at */
  double* best_loss;   /* [n_problems] (+inf at start) */
  double* loss_trace;  /* [loss_trace_epochs][n_problems] */
  int loss_trace_epochs;
  double* snapshots;   /* [n_snapshots][S][S]: Q of problem 0 at epochs 1, 2, 4, ... (or NULL) */
  int n_snapshots;
  double* dQ_part;     /* workspace [n_problems*K][S][S] */
  double* loss_part;   /* workspace [n_problems*K] */
  double* workspace;   /* see cherry_fit_workspace_bytes */
  size_t workspace_bytes;
  int* epoch_counter;  /* [n_problems] epochs completed (zero at start) */
  int* status_flag;    /* [1] zero at start; a kernel sets 1 (out of matrix slots), 2 (t * norm of Q
                          beyond the supported range, see cherry_expm_batched) or 3 (internal
                          scheduling timeout of the large path); the results are then invalid */
  double lr_pi, lr_upper, beta1, beta2, eps;
  int do_adam;             /* 1: Adam (torch semantics), 0: plain SGD */
  int loss_normalization;  /* divide loss and gradient by sumC */
  int best_mode;           /* 0: trainer.py:179 (first epoch always taken); 1: best starts at +inf */
} cherry_fit_args;

/* Largest K (time buckets, or exponents of one cherry_expm_batched call) for S > 32: the weight
 * table, bucket lists and count-load ring of the large-K Taylor pass share one CTA's 200 KB of
 * shared memory, 212 K + 32 776 bytes.  Beyond it the entry points return CHERRY_ELIMIT; callers
 * with more exponents split them into calls of at most this many. */
#define CHERRY_LARGE_FIT_MAX_K 811

/* Bytes of `workspace` the fit needs for these sizes (0 is a valid answer).  CHERRY_ELIMIT for
 * S > 32 and K > CHERRY_LARGE_FIT_MAX_K. */
int cherry_fit_workspace_bytes(int S, int K, int n_problems, size_t* bytes);
/* Q = Q(theta) for every problem (call once before the first epoch). */
int cherry_fit_init(const cherry_fit_args* args, void* stream);
/* Run `num_epochs` epochs: P_k = expm(t_k Q), loss = -sum C.log P / sumC, best-iterate and
 * snapshot bookkeeping, exact gradient, optimiser step, next Q.  No host synchronisation;
 * epochs are replayed from a CUDA graph in chunks unless `stream` is already capturing. */
int cherry_fit_run(const cherry_fit_args* args, int num_epochs, void* stream);
/* Bucket-sharded training over several GPUs (one process per GPU, each with its own subset
 * of the K buckets in `args`, replicated theta / optimiser state, args->sumC = the sum over
 * ALL ranks): one epoch is
 *     cherry_fit_epoch_local(args, packed)    loss and exact gradient of this rank's buckets,
 *                                             packed = {[n_problems][S][S] gradient totals,
 *                                             [n_problems] loss totals} (unnormalised)
 *     all-reduce(SUM) of `packed` over the ranks   (the caller: NCCL via torch.distributed)
 *     cherry_fit_epoch_update(args, packed)   bookkeeping, optimiser step and next Q from the
 *                                             reduced totals, identical on every rank.
 * This is the exchange step of l = sum_k l_k, dl/dQ = sum_k t_k G_k (reference
 * trainer.py:170-187 evaluates the same sums on one device).
 * args->Q must be the Q that cherry_fit_init / the previous cherry_fit_epoch_update built from
 * args->theta (it is, in this loop): for S > 32 the evaluation may use the symmetric form of that model
 * (cherry_fit_symmetric_form below).  For the loss and gradient of an ARBITRARY Q use cherry_fit_loss_grad. */
int cherry_fit_epoch_local(const cherry_fit_args* args, double* packed, void* stream);
int cherry_fit_epoch_update(const cherry_fit_args* args, const double* packed, void* stream);
/* One evaluation without an optimiser step (tests, evaluation): writes loss_part[p*K+k] =
 * -<C_k, log expm(t_k Q_p)> and dQ_part[p*K+k] = its gradient with respect to Q_p (S <= 32).  For S > 32
 * only the sums over k are defined: loss_part[0] holds the whole loss, dQ_part[0] the whole gradient; with
 * args->theta null (an arbitrary Q, no fit) the call prepares the workspace itself (synchronous), as
 * cherry_expm_batched does. */
int cherry_fit_loss_grad(const cherry_fit_args* args, void* stream);

/* P_out[p*K + k] = expm(t[p*K + k] * Q[p]) (fp64 [S][S] each) with the fit's forward algorithm.
 * Only S, K, n_problems, t, Q, workspace(+bytes, as for the fit) and status_flag of `args` are
 * read.  Replaces matrix_exponential_pytorch (reference markov_chain/_markov_chain.py:22-53).
 * For S > 32, K <= CHERRY_LARGE_FIT_MAX_K (else CHERRY_ELIMIT), and *status_flag is set to 2
 * when some t * max|Q_ii| exceeds 2.2 * 2^8 = 563.2 (eight squarings).  For S <= 32 the squarings
 * stop at 30, i.e. t * ||Q||_1 (max column abs sum) up to 0.0376 * 2^30 = 4.0e7; beyond it
 * *status_flag is set to 2 as well, and that exponent's result is computed with 30 squarings
 * (outside the accuracy of the path).  The same flag is set by the fit and cherry_fit_loss_grad.
 * A nan or inf t * norm sets no flag; the nan propagates to the result. */
int cherry_expm_batched(const cherry_fit_args* args, double* P_out, void* stream);

/* The FP64 tensor-core GEMM of the large-S fit, stand-alone (unit tests, micro-benchmark):
 * C[b] = op(A[b]) op(B[b]) (+ C[b] if accumulate), b < batch, square n x n row-major matrices
 * stored back to back, n a multiple of 80.  desc: device scratch of
 * cherry_gemm_desc_bytes(batch) bytes; partial: batch*ksplit*n*n doubles, needed iff ksplit > 1.
 * This is what torch.matmul does inside torch.matrix_exp in the reference
 * (estimation/_ratelearn/trainer.py:170-172). */
int cherry_gemm_f64_batched(const double* A, const double* B, double* C, int n, int batch, int trans_a,
                            int trans_b, int accumulate, int ksplit, void* desc, double* partial,
                            void* stream);
size_t cherry_gemm_desc_bytes(int batch);

/* Large-S path only (S > 32): host copy of the squarings s_k chosen for every bucket in the most
 * recent evaluation, the diagonal shift mu and the Taylor degree m.  One evaluation runs
 * (m-1) + sum_k s_k products of S x S matrices forward and twice that backward; bench.py uses
 * this to turn kernel time into executed FLOP/s.  Synchronises the device. */
int cherry_fit_schedule(const cherry_fit_args* args, int* squarings_out, double* mu_out, int* degree_out);

/* Large-S path only: 1 if the epochs of this fit (cherry_fit_run / cherry_fit_epoch_local after cherry_fit_init)
 * run in the symmetric form, 0 otherwise.  The reference's model (rate.py: pande_reversible) is
 * Q_ij = mask_ij softplus(u_ij) sqrt(pi_j / pi_i), similar to the symmetric matrix mask_ij softplus(u_ij) by
 * diag(sqrt(pi)); when mask and every count matrix are exactly symmetric (cherry counts are) the evaluation works on
 * symmetric matrices throughout and computes only the tiles on and above the diagonal of the forward products.
 * Losses and gradients are the same quantities (rounding-level differences); CHERRY_FIT_SYMMETRIC=0 turns it off. */
int cherry_fit_symmetric_form(const cherry_fit_args* args);

/* ------------------------------------------------------------------- FastCherries */

/* One MSA family for the FastCherries kernels: ALL sequences of the MSA in file order, one
 * row each, residue bytes as for counting (0..S-1, S = skip, rows padded with S).  32 bytes. */
typedef struct cherry_fc_family {
  int64_t msa_off;    /* byte offset of row 0 in the residue buffer (16-aligned) */
  int32_t n_seqs;     /* rows */
  int32_t row_stride; /* bytes per row, a multiple of 16 */
  int32_t n_sites;    /* real sites (<= row_stride) */
  int32_t cherry_off; /* first cherry of this family in pair_a/pair_b/len_idx:
                         sum of floor(n_seqs / 2) over the families before it */
  int32_t site_off;   /* first site of this family in site_cat: sum of n_sites before it */
  int32_t seq_off;    /* sum of n_seqs over the families before it */
} cherry_fc_family;

/* Device scratch both FastCherries entry points need (they may share one buffer; K, R, S as
 * passed to cherry_fc_ble). */
size_t cherry_fc_scratch_bytes(int64_t total_seqs, int64_t total_sites, int n_fams, int K, int R, int S);

/* Pairs the sequences of every family into floor(n_seqs / 2) cherries by recursive bisection
 * around two far-apart pivots under the normalised Hamming distance over sites valid in both
 * sequences.  pair_a/pair_b[fam.cherry_off + c] = row indices of the c-th cherry IN THE ORDER
 * the reference emits them; unpaired[f] = the left-over row of an odd family, else -1.
 * The random pivots are std::mt19937(seed) re-seeded per family, drawn like libstdc++'s
 * std::uniform_int_distribution<size_t> (GCC >= 11).  Exact (integer) reproduction of
 * divide_and_pair, FastCherries/pairing_algorithms.cpp:79-175. */
int cherry_fc_pair(const uint8_t* msa, const cherry_fc_family* fams, int n_fams, int64_t total_seqs, int S,
                   uint32_t seed, int32_t* pair_a, int32_t* pair_b, int32_t* unpaired, void* scratch,
                   size_t scratch_bytes, void* stream);

/* Branch-length and site-rate estimation by coordinate ascent for every family:
 * len_idx[cherry] = index into the K-point quantization grid, site_cat[site] = index into the
 * R rate categories, iters[f] = ascent iterations run (<= max_iters).
 * sym_table: fp64 [K][R][S][S], log P + (log P)^T with P = expm(q_k * rate_r * Q);
 * priors: [R] = 2 log(rate_r) - 3 rate_r; init_weights: [R] cumulative gamma-bin weights of the
 * initial site-rate assignment (fast_cherries.cpp:137-160).  S <= 32, n_seqs <= 65535.
 * Every likelihood sum is accumulated by one thread in the reference's order, so the
 * decisions equal the reference's given the same table.
 * Replaces ble(), FastCherries/branch_length_estimation.cpp:150-241. */
int cherry_fc_ble(const uint8_t* msa, const cherry_fc_family* fams, int n_fams, int64_t total_sites, int S,
                  const int32_t* pair_a, const int32_t* pair_b, const double* sym_table, int K, int R,
                  const double* priors, const double* init_weights, int max_iters, int32_t* len_idx,
                  int32_t* site_cat, int32_t* iters, void* scratch, size_t scratch_bytes, void* stream);

/* FastCherries -> LG counting without the text files.
 * cherry_fc_lengths_and_rates (HOST pointers): pair_t[cherry] and rate_table[family][category] with
 * exactly the values the counting stage would parse from the tree / site-rate files that
 * cherry_fc_write_outputs writes ('%.17f' and repr round trips, float32 when float32_lengths).
 * cherry_fc_relayout_lg (DEVICE pointers): copies the paired rows of every family into the LG
 * counting layout described by out_fams (rows 2c, 2c+1 = cherry c; column of site j = dest[j]);
 * msa_out must be pre-filled with the skip code. */
int cherry_fc_lengths_and_rates(const cherry_fc_family* fams, int n_fams, const int32_t* len_idx,
                                const int32_t* site_cat, const double* grid, int K, const double* cats, int R,
                                int float32_lengths, double* pair_t, double* rate_table, int n_threads);
/* Host metadata of that LG counting batch (HOST pointers; the ingest's layout rules: categories =
 * the site_cat values present in a family, sites in order inside a category, categories padded
 * to 4 sites, row stride a multiple of 16).  Call once with the output arrays NULL to get
 * sizes[6] = {residue bytes, group_cat entries, rate values, tiles, r_pad, (pair, site) items},
 * then with dest[total_sites], group_cat, rate_vals, out_fams[n_fams], tiles allocated.
 * chunks_per_tile: 16384 (the ingest's tile size). */
int cherry_fc_count_layout(const cherry_fc_family* fams, int n_fams, const int32_t* site_cat,
                           const double* rate_table, int R, int chunks_per_tile, int32_t* dest,
                           uint16_t* group_cat, double* rate_vals, cherry_fam_desc* out_fams, cherry_tile* tiles,
                           int64_t* sizes, int n_threads);
int cherry_fc_relayout_lg(const uint8_t* msa_in, const cherry_fc_family* fc_fams, const cherry_fam_desc* out_fams,
                          int n_fams, const int32_t* pair_a, const int32_t* pair_b, const int32_t* dest,
                          uint8_t* msa_out, void* stream);

/* Host-side text I/O of the FastCherries stage (multithreaded, one family per task). */
typedef struct cherry_fc_msas {
  int32_t n_fams;
  int32_t pinned;          /* msa is page-locked */
  int64_t msa_bytes;
  uint8_t* msa;            /* residue rows of all families, as cherry_fc_pair / cherry_fc_ble take them */
  cherry_fc_family* fams;
  int64_t total_seqs, total_sites, total_cherries;
  char* name_blob;         /* sequence names back to back */
  int64_t* name_off;       /* [total_seqs + 1] offsets into name_blob, sequences in batch order */
} cherry_fc_msas;

/* Reads and encodes `<paths[f]>` for every family like read_msa of FastCherries/io_helpers.cpp
 * :35-74 (a line starting with '>' names a sequence, the next line is the sequence; characters
 * outside `states` become the skip code).  Release with cherry_fc_free_msas. */
int cherry_fc_read_msas(const char* const* paths, int n_fams, const char* const* states, int n_states,
                        int n_threads, int pinned, cherry_fc_msas** out);
void cherry_fc_free_msas(cherry_fc_msas* msas);

/* Writes, per family, what the reference stage leaves behind (any path array except tree_paths
 * and site_rate_paths may be NULL): the star-of-cherries tree in CherryML's tree format
 * (phylogeny_estimation/_fast_cherries.py:121-141; branch length = the '%.17f' text of
 * grid[len_idx] * mean rate, read back and halved, printed like Python's repr), the newick
 * string, the site rates normalised to mean 1 in '%.17f ' format (io_helpers.cpp:91-103), the
 * constant likelihood file and the profiling file (4 numbers per family).  All pointers are
 * HOST pointers. */
int cherry_fc_write_outputs(const cherry_fc_msas* msas, const int32_t* pair_a, const int32_t* pair_b,
                            const int32_t* unpaired, const int32_t* len_idx, const int32_t* site_cat,
                            const double* grid, int K, const double* cats, int R, const char* const* tree_paths,
                            const char* const* newick_paths, const char* const* site_rate_paths,
                            const char* const* likelihood_paths, const char* const* profiling_paths,
                            const double* profiling, int n_threads);

/* Count-matrix text files (`result.txt` of the counting stages), multithreaded over the K
 * matrices; all pointers are HOST pointers.  cpp_style = 0: the layout of the reference's
 * Python writer (io/_count_matrices.py:66-81: pandas to_csv, floats as repr), 1: the layout of
 * its C++ program (counting/_count_transitions.cpp:524-548: "%g", tab after every state name).
 * The reader accepts both (io/_count_matrices.py:8-63); numbers go through strtod. */
int cherry_write_count_matrices(const char* path, const double* q, int K, const char* const* states, int S,
                                const double* counts, int cpp_style, int n_threads);
int cherry_read_count_matrices_header(const char* path, int* K, int* S);
/* states_out receives the S state names of the file's last header line, '\n'-separated. */
int cherry_read_count_matrices(const char* path, int K, int S, double* q, double* counts, char* states_out,
                               size_t states_cap, int n_threads);

/* Labelled S x S table (rate matrix file, reference io/_rate_matrix.py:37-52): fp64 numbers as
 * the shortest strings that round-trip, exponent notation like Python's repr. */
int cherry_write_labelled_matrix(const char* path, const char* const* states, int S, const double* data,
                                 int n_threads);

/* ------------------------------------------------------------------- tree log-likelihood */

/* One tree node; nodes are passed in POST-ORDER (children, in the tree's child order, before
 * their parent; the root last).  16 bytes. */
typedef struct cherry_ll_node {
  int32_t depth;    /* edges between the node and the root */
  int32_t flags;    /* bit 0: leaf; bit 1: first child of its parent */
  int32_t obs_row;  /* leaf: row of `obs`; internal node: -1 */
  int32_t reserved;
} cherry_ll_node;

int cherry_tree_ll_units_per_block(int S, int c);
size_t cherry_tree_ll_scratch_bytes(int S, int c, int n_units, int max_depth);

/* Pt[m][k][s] = P[m][s][k] for n_matrices fp64 [Su][Su] matrices (device pointers, Pt != P): the
 * layout cherry_tree_log_likelihood reads, made from cherry_expm_batched's output. */
int cherry_tree_ll_transpose(const double* P, int n_matrices, int Su, double* Pt, void* stream);

/* ll_out[u] = log-likelihood of unit u on the tree.  A unit is one site (c = 1, S states) or a
 * pair of contacting sites (c = 2, S*S states, state = S*i + j).
 * p_index[i * n_cats + k]: which matrix of P belongs to the edge above node i for rate category
 * k (ignored for the root); P: fp64 [n][Su][Su], the TRANSPOSES of the row-stochastic matrices
 * expm(branch length * rate_k * Q), i.e. P[m][k][s] = Pr(s -> k) (cherry_tree_ll_transpose); unit_cat[u]: the unit's rate category; obs: uint8 [n_leaves][n_units][c] residues
 * (S = not in the alphabet: every state is compatible); pi: [Su] root distribution.
 * Replaces the pruning loops of dp_likelihood_computation, evaluation/_likelihood.py:239-326
 * (child messages are accumulated in the same order; a pair's value is split over its two
 * sites by the caller as at :316-319). */
int cherry_tree_log_likelihood(const cherry_ll_node* nodes, int n_nodes, const int32_t* p_index, int n_cats,
                               const double* P, const uint8_t* obs, const int32_t* unit_cat, const double* pi,
                               int S, int c, int n_units, int max_depth, void* scratch, size_t scratch_bytes,
                               double* ll_out, void* stream);

/* Edge posteriors for the exact gradient of the log-likelihood of independent sites (c = 1,
 * S <= 32 states, else CHERRY_ELIMIT).  Inputs as for cherry_tree_log_likelihood, except that
 * p_index [n_nodes][n_cats] and unit_cat [n_units] are HOST arrays (the launch groups units of
 * one rate category per CTA and orders the reduction from them); P holds n_matrices matrices and
 * every p_index entry of a non-root node must be below n_matrices.  Outputs (device):
 *   ll_out[u]       bitwise what cherry_tree_log_likelihood writes for c = 1;
 *   W_out[m][a][b]  sum over units u and edges (parent(i), i) with p_index[i*n_cats + unit_cat[u]]
 *                   = m of Pr(parent(i) = a, i = b | data_u), overwritten (zero for a matrix no
 *                   edge uses);
 *   root_out[a]     sum over units of Pr(root = a | data_u), overwritten.
 * d log L / d P_m = W_m / P_m, so d log L / d Q = sum_m d/dQ <W_m, log expm(t_m Q)> with W held
 * fixed (cherry_fit_loss_grad with C = W gives minus that), and d log L / d pi_a = root_out[a] / pi_a.
 * No floating-point atomics: two calls give bitwise-identical outputs.  Synchronises the host
 * with the upload of its index tables (pageable cudaMemcpyAsync); the kernels run on `stream`. */
size_t cherry_tree_ll_posterior_scratch_bytes(int S, int n_nodes, int max_depth, int n_cats, int n_matrices,
                                              int n_units, const int32_t* unit_cat);
int cherry_tree_ll_posterior(const cherry_ll_node* nodes, int n_nodes, int max_depth, const int32_t* p_index,
                             int n_cats, const double* P, int n_matrices, const uint8_t* obs, const int32_t* unit_cat,
                             const double* pi, int S, int n_units, void* scratch, size_t scratch_bytes,
                             double* ll_out, double* W_out, double* root_out, void* stream);

/* cherry_tree_ll_posterior plus the derivative of the log-likelihood with respect to every branch
 * exponent.  Inputs and limits as for cherry_tree_ll_posterior, plus Q: device fp64 [S][S], NOT
 * transposed, the rate matrix the matrices P were made from (P = expm(tau Q)).  Outputs: ll_out,
 * W_out and root_out exactly as cherry_tree_ll_posterior writes them, and (device)
 *   dtau_out[i][k]  d log L / d tau for the edge above node i in rate category k (tau = branch length
 *                   * rate_k), summed over that category's units; the root's row is 0.
 * With dP/dtau = QP it is sum over units of (Q^T eo_u) . (P ei_u) (outside and inside vectors of
 * the edge): no division by P, so zero-length branches are fine.  d log L / d length_i =
 * sum_k rate_k dtau_out[i][k].  Null Q or dtau_out gives CHERRY_EINVAL.  No floating-point atomics:
 * two calls give bitwise-identical outputs.  The scratch size is 0 for sizes outside the limits. */
size_t cherry_tree_ll_edge_derivatives_scratch_bytes(int S, int n_nodes, int max_depth, int n_cats, int n_matrices,
                                                     int n_units, const int32_t* unit_cat);
int cherry_tree_ll_edge_derivatives(const cherry_ll_node* nodes, int n_nodes, int max_depth, const int32_t* p_index,
                                    int n_cats, const double* P, int n_matrices, const uint8_t* obs,
                                    const int32_t* unit_cat, const double* pi, const double* Q, int S, int n_units,
                                    void* scratch, size_t scratch_bytes, double* ll_out, double* W_out,
                                    double* root_out, double* dtau_out, void* stream);

/* Edge posteriors for the exact gradient of the log-likelihood of pairs of contacting sites (c = 2,
 * Su = S*S states, state S*i + j; 1 <= S <= 32, else CHERRY_ELIMIT), every pair on the same matrices
 * (no rate categories).  nodes [n_nodes] and p_index [n_nodes] are HOST arrays (the launch builds its
 * level schedule from them); every p_index entry of a non-root node must be below n_matrices.  P:
 * [n_matrices][Su][Su] as cherry_expm_batched writes it (NOT transposed); obs: uint8
 * [n_leaves][n_pairs][2] residues (S = not in the alphabet); pi: [Su].  Outputs (device):
 *   ll_out[u]       log-likelihood of pair u (what cherry_tree_log_likelihood gives for c = 2, up to
 *                   the order of the sums);
 *   W_out[m][a][b]  sum over pairs and over the edges (parent(i), i) with p_index[i] = m of
 *                   Pr(parent(i) = a, i = b | data_u), overwritten (zero for a matrix no edge uses);
 *   root_out[a]     sum over pairs of Pr(root = a | data_u), overwritten.
 * A pair with likelihood 0 contributes no posterior mass.  d log L / d P_m = W_m / P_m, so the Q
 * gradient is cherry_fit_loss_grad with C = W, as for cherry_tree_ll_posterior.  The pairs are the
 * columns of FP64 tensor-core products, so each edge matrix is read once per product for every 16
 * pairs.  No floating-point atomics: two calls give bitwise-identical outputs.  Synchronises the host
 * with the upload of its index tables (pageable cudaMemcpyAsync); the kernels run on `stream`.
 * The scratch size is 0 for sizes outside these limits. */
size_t cherry_tree_ll_pair_posterior_scratch_bytes(int S, int n_nodes, int max_depth, int n_pairs, int n_matrices);
int cherry_tree_ll_pair_posterior(const cherry_ll_node* nodes, int n_nodes, int max_depth, const int32_t* p_index,
                                  const double* P, int n_matrices, const uint8_t* obs, const double* pi, int S,
                                  int n_pairs, void* scratch, size_t scratch_bytes, double* ll_out, double* W_out,
                                  double* root_out, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* CHERRYML_B200_H */

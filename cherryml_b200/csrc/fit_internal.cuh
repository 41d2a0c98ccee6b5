// Internal entry points of the fit implementations, dispatched by fit_api.cu.
#pragma once
#include "common.cuh"

namespace cherry {

constexpr int kSmallFitMaxS = 32;

// S <= 32: everything in shared memory, one CTA per (problem, bucket).  fit_small.cu
int fit_small_workspace(int S, int* n_smem_slots, int* spill_slots, size_t* slot_bytes, size_t* smem_bytes,
                        int grid = -1);  // grid < 0: sizing only (the resident slots of the latency shape)
int fit_small_expm(const cherry_fit_args& a, cudaStream_t stream, double* P_out = nullptr, bool fuse_update = false);
size_t fit_small_workspace_bytes(int S, int K, int n_problems);
// `reduced` (optional): [P][S][S] gradient totals followed by [P] loss totals, already summed
// over the buckets (of all ranks); replaces the per-bucket pieces dQ_part / loss_part.
int fit_small_update(const cherry_fit_args& a, int mode, cudaStream_t stream, const double* reduced = nullptr);

// S > 32 (the 400 x 400 co-evolution model): batched DMMA GEMM chain.  fit_large.cu
int fit_large_workspace_bytes(int S, int K, int n_problems, size_t* bytes);
// loss_part + dQ_total in dQ_part[0].  training: a.Q is the reversible model of a.theta / a.mask (the epoch entry
// points) -- the evaluation may then run in the symmetric form, same results (fit_large.cu build_B_sym_kernel)
int fit_large_expm(const cherry_fit_args& a, cudaStream_t stream, bool training = false);
int fit_large_symmetric_form(const cherry_fit_args& a);  // 1: the training evaluations of this workspace use it
int fit_large_forward_only(const cherry_fit_args& a, double* P_out, cudaStream_t stream);
int fit_large_prepare(const cherry_fit_args& a, cudaStream_t stream);  // uploads the plan of (S, K) (synchronous)
int fit_large_update(const cherry_fit_args& a, int mode, cudaStream_t stream, const double* reduced = nullptr);
int fit_large_timeline(const cherry_fit_args& a, cudaStream_t stream);
int fit_large_read_schedule(const cherry_fit_args& a, int* s_out, double* mu_out);
int gemm_f64_batched(const double* A, const double* B, double* C, int n, int batch, int ta, int tb,
                     int accumulate, int ksplit, void* desc, double* partial, cudaStream_t stream);
size_t gemm_desc_bytes(int batch);
constexpr int kLargeDegree = 24;  // keep in sync with fit_large.cu

}  // namespace cherry

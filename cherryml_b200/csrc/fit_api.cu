// C-ABI entry points of the fit (include/cherryml_b200.h), dispatching on the state-space
// size: S <= 32 -> fit_small.cu (shared-memory resident), larger -> fit_large.cu.
#include <cstdlib>

#include "fit_internal.cuh"

namespace {

int check_args(const cherry_fit_args* a, bool training) {
  if (!a) return cherry::fail(CHERRY_EINVAL, "fit: null args");
  if (a->S <= 0 || a->K <= 0 || a->n_problems <= 0) return cherry::fail(CHERRY_EINVAL, "fit: bad sizes");
  if (!a->t || !a->C || !a->Q || !a->dQ_part || !a->loss_part || !a->status_flag)
    return cherry::fail(CHERRY_EINVAL, "fit: null pointer argument");
  if (training && (!a->mask || !a->sumC || !a->theta || !a->adam_m || !a->adam_v || !a->Q_best || !a->Q_last ||
                   !a->best_loss || !a->loss_trace || !a->epoch_counter))
    return cherry::fail(CHERRY_EINVAL, "fit: null pointer argument (training state)");
  return 0;
}

int one_epoch(const cherry_fit_args& a, cudaStream_t stream) {
  int rc;
  // S <= 32: ONE launch per epoch, the last CTA of every problem runs its parameter update (fit_small.cu)
  if (a.S <= cherry::kSmallFitMaxS) return cherry::fit_small_expm(a, stream, nullptr, true);
  if ((rc = cherry::fit_large_expm(a, stream, true))) return rc;
  return cherry::fit_large_update(a, 1, stream);
}

// packed[p][e] = sum_k dQ_part[p*K + k][e] (bucket order), packed[P*S*S + p] = sum_k loss_part.
// For the large path dQ_part[0] already is the total over this rank's buckets.
__global__ void fit_pack_partials_kernel(const double* __restrict__ dQ_part, const double* __restrict__ loss_part,
                                         int SS, int K, int P, int dq_pieces, double* __restrict__ packed) {
  const int p = blockIdx.y;
  for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < SS; e += gridDim.x * blockDim.x) {
    double acc = 0.0;
    const double* src = dQ_part + (size_t)p * dq_pieces * SS + e;
    for (int k = 0; k < dq_pieces; ++k) acc += src[(size_t)k * SS];
    packed[(size_t)p * SS + e] = acc;
  }
  if (blockIdx.x == 0 && threadIdx.x == 0) {
    double lp = 0.0;
    for (int k = 0; k < K; ++k) lp += loss_part[(size_t)p * K + k];
    packed[(size_t)P * SS + p] = lp;
  }
}

}  // namespace

extern "C" {

int cherry_fit_epoch_local(const cherry_fit_args* a, double* packed, void* stream_) {
  int rc = check_args(a, false);
  if (rc) return rc;
  if (!packed) return cherry::fail(CHERRY_EINVAL, "fit_epoch_local: null packed buffer");
  cudaStream_t stream = (cudaStream_t)stream_;
  const bool small = a->S <= cherry::kSmallFitMaxS;
  if (!small && a->n_problems != 1)
    return cherry::fail(CHERRY_EINVAL, "fit_epoch_local: the large path fits one problem");
  rc = small ? cherry::fit_small_expm(*a, stream) : cherry::fit_large_expm(*a, stream, true);
  if (rc) return rc;
  const int SS = a->S * a->S;
  dim3 grid((SS + 255) / 256 > 64 ? 64 : (SS + 255) / 256, a->n_problems);
  fit_pack_partials_kernel<<<grid, 256, 0, stream>>>(a->dQ_part, a->loss_part, SS, a->K, a->n_problems,
                                                      small ? a->K : 1, packed);
  CHERRY_LAUNCH_CHECK("fit_pack_partials_kernel");
  return 0;
}

int cherry_fit_epoch_update(const cherry_fit_args* a, const double* packed, void* stream) {
  int rc = check_args(a, true);
  if (rc) return rc;
  if (!packed) return cherry::fail(CHERRY_EINVAL, "fit_epoch_update: null packed buffer");
  if (a->S <= cherry::kSmallFitMaxS) return cherry::fit_small_update(*a, 1, (cudaStream_t)stream, packed);
  return cherry::fit_large_update(*a, 1, (cudaStream_t)stream, packed);
}

int cherry_fit_workspace_bytes(int S, int K, int n_problems, size_t* bytes) {
  if (!bytes) return cherry::fail(CHERRY_EINVAL, "fit_workspace_bytes: null pointer");
  if (S <= 0 || K <= 0 || n_problems <= 0) return cherry::fail(CHERRY_EINVAL, "fit_workspace_bytes: bad sizes");
  if (S <= cherry::kSmallFitMaxS) {
    int ns = 0, sp = 0;
    size_t sb = 0, smem = 0;
    int rc = cherry::fit_small_workspace(S, &ns, &sp, &sb, &smem);
    if (rc) return rc;
    *bytes = cherry::fit_small_workspace_bytes(S, K, n_problems);
    return 0;
  }
  return cherry::fit_large_workspace_bytes(S, K, n_problems, bytes);
}

int cherry_fit_init(const cherry_fit_args* a, void* stream) {
  if (!a || !a->mask || !a->theta || !a->Q || !a->epoch_counter)
    return cherry::fail(CHERRY_EINVAL, "fit_init: null pointer argument");
  if (a->S <= cherry::kSmallFitMaxS) return cherry::fit_small_update(*a, 0, (cudaStream_t)stream);
  return cherry::fit_large_update(*a, 0, (cudaStream_t)stream);
}

int cherry_fit_loss_grad(const cherry_fit_args* a, void* stream) {
  int rc = check_args(a, false);
  if (rc) return rc;
  if (a->S > cherry::kSmallFitMaxS && getenv("CHERRY_FIT_TIMELINE"))
    return cherry::fit_large_timeline(*a, (cudaStream_t)stream);
  if (a->S <= cherry::kSmallFitMaxS) return cherry::fit_small_expm(*a, (cudaStream_t)stream);
  // an arbitrary Q (no parameters): no cherry_fit_init has prepared this workspace for this K
  if (!a->theta && (rc = cherry::fit_large_prepare(*a, (cudaStream_t)stream))) return rc;
  return cherry::fit_large_expm(*a, (cudaStream_t)stream);
}

int cherry_expm_batched(const cherry_fit_args* a, double* P_out, void* stream) {
  if (!a || !P_out) return cherry::fail(CHERRY_EINVAL, "expm_batched: null pointer argument");
  if (a->S <= 0 || a->K <= 0 || a->n_problems <= 0 || !a->t || !a->Q || !a->status_flag)
    return cherry::fail(CHERRY_EINVAL, "expm_batched: S, K, n_problems, t, Q and status_flag are required");
  if (a->S <= cherry::kSmallFitMaxS) return cherry::fit_small_expm(*a, (cudaStream_t)stream, P_out);
  return cherry::fit_large_forward_only(*a, P_out, (cudaStream_t)stream);
}

int cherry_gemm_f64_batched(const double* A, const double* B, double* C, int n, int batch, int trans_a,
                            int trans_b, int accumulate, int ksplit, void* desc, double* partial,
                            void* stream) {
  return cherry::gemm_f64_batched(A, B, C, n, batch, trans_a, trans_b, accumulate, ksplit, desc, partial,
                                  (cudaStream_t)stream);
}

size_t cherry_gemm_desc_bytes(int batch) { return cherry::gemm_desc_bytes(batch < 1 ? 1 : batch); }

int cherry_fit_schedule(const cherry_fit_args* a, int* squarings_out, double* mu_out, int* degree_out) {
  if (!a || !squarings_out) return cherry::fail(CHERRY_EINVAL, "fit_schedule: null pointer");
  if (a->S <= cherry::kSmallFitMaxS)
    return cherry::fail(CHERRY_EINVAL, "fit_schedule: only the large-S path (S > %d) records its schedule",
                        cherry::kSmallFitMaxS);
  if (degree_out) *degree_out = cherry::kLargeDegree;
  return cherry::fit_large_read_schedule(*a, squarings_out, mu_out);
}

int cherry_fit_symmetric_form(const cherry_fit_args* a) {
  if (!a || a->S <= cherry::kSmallFitMaxS) return 0;
  return cherry::fit_large_symmetric_form(*a);
}

int cherry_fit_run(const cherry_fit_args* a, int num_epochs, void* stream_) {
  int rc = check_args(a, true);
  if (rc) return rc;
  if (num_epochs < 0) return cherry::fail(CHERRY_EINVAL, "fit_run: negative num_epochs");
  cudaStream_t stream = (cudaStream_t)stream_;
  cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
  CHERRY_CUDA(cudaStreamIsCapturing(stream, &cap));
  const int chunk = 32;
  int done = 0;
  // Epoch bodies take all their inputs from device memory (epoch counters included), so a
  // captured chunk can be replayed unchanged.  The legacy default stream cannot capture.
  if (cap == cudaStreamCaptureStatusNone && stream != nullptr && num_epochs >= 2 * chunk) {
    cudaGraph_t graph = nullptr;
    cudaGraphExec_t exec = nullptr;
    CHERRY_CUDA(cudaStreamBeginCapture(stream, cudaStreamCaptureModeThreadLocal));
    const long long before = cherry::g_launches.load();
    for (int e = 0; e < chunk && rc == 0; ++e) rc = one_epoch(*a, stream);
    const long long per_chunk = cherry::g_launches.load() - before;
    cudaError_t ce = cudaStreamEndCapture(stream, &graph);
    if (rc) {
      if (graph) cudaGraphDestroy(graph);
      return rc;
    }
    CHERRY_CUDA(ce);
    cherry::g_launches.fetch_sub(per_chunk);  // capture records, it does not launch
    ce = cudaGraphInstantiate(&exec, graph, 0);
    if (ce != cudaSuccess) {
      cudaGraphDestroy(graph);
      return cherry::check_cuda(ce, "cudaGraphInstantiate");
    }
    while (num_epochs - done >= chunk) {
      ce = cudaGraphLaunch(exec, stream);
      if (ce != cudaSuccess) break;
      cherry::count_launch((int)per_chunk);
      done += chunk;
    }
    cudaGraphExecDestroy(exec);
    cudaGraphDestroy(graph);
    CHERRY_CUDA(ce);
  }
  for (; done < num_epochs; ++done)
    if ((rc = one_epoch(*a, stream))) return rc;
  return 0;
}

}  // extern "C"

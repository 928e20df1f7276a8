// Arguments shared by the two batched kernels (batched.cu: one CTA per LFM; batched_warp.cu: one warp per LFM).
#pragma once
#include <cstring>
#include "sim_math.cuh"

struct BatchedArgs {
  int64_t B;
  int N, G;
  const double* X;
  const double* y;
  int64_t y_stride;   // 0: every LFM fits the same y (multi-start); N or more: LFM b fits y + b * y_stride (replicas / candidate TFs)
  double* u_io;       // B x P unconstrained (in/out)
  double* adam;       // B x 2P (m, v) or NULL
  double jitter, lr, b1, b2, eps;
  int first_step, steps, total_steps, fix_params, steps_per_epoch;
  double* hist; int64_t ld_hist;
  double* theta_out;  // B x P constrained result written when the last step of the fit is reached (or NULL)
  double* eval_val;   // eval-only mode: B
  double* eval_grad;  // eval-only mode: B x P
  int* info;
  int max_unique;
  long long* stamps;   // debug (lfm_debug_batched_stamps): clock64 at the phase boundaries of the first step of LFM 0
  void* struct_cache;  // NULL or lfm_batched_structure_bytes() device bytes kept by the caller between the launches of a fit
  int* queue;           // NULL or lfm_batched_queue_bytes() device bytes, initialised by lfm_batched_fit_queue: persistent workers + task queue
  int queue_chunk;      // steps per task in queue mode
  long long* step_keys; // NULL or total_steps device words: word s receives atomicMin of lfm_loss_key(loss at step s) over the batch
  long long* best_key; // NULL or one device word: atomicMin of lfm_loss_key(loss after the launch's last step) over the batch     // shared-memory matrix is sized for this many unique rows (N when unknown)
  // Heteroscedastic objective (the HET instantiations; appended so that the parameter offsets of the others stay put):
  // NULL, or the measurement variances v, Sigma = K + diag(v) + (jitter + sigma^2) I.  var_stride 0: one vector of N
  // shared by every LFM; N or more: LFM b reads var + b * var_stride (as y / y_stride).
  const double* var;
  int64_t var_stride;
};

// Order-preserving map double -> signed 64-bit integer (finite values and infinities; NaN never enters): the
// best objective of a chunk is one atomicMin per LFM and one integer MIN all-reduce across ranks.
__host__ __device__ inline long long lfm_loss_key(double v) {
  long long i;
#ifdef __CUDA_ARCH__
  i = __double_as_longlong(v);
#else
  memcpy(&i, &v, sizeof(i));
#endif
  return i >= 0 ? i : (i ^ 0x7fffffffffffffffLL);
}

// Task queue of the persistent mode (batched_warp.cu): a task is "the next queue_chunk steps of LFM b".  Layout (ints):
// [head, tail, pad, pad | done[B] | ring[B * nchunks]].  ring[t] is the LFM of ticket t (-1 = not published yet): tickets
// 0 .. B-1 are the first chunks of all LFMs; finishing chunk c of LFM b publishes b at ring[tail++].  Exactly
// B * nchunks tickets exist; a worker whose ticket is >= that exits.
struct LfmQueue {
  int* head; int* tail; int* done; int* ring; int64_t B;
  __host__ __device__ int total(int total_steps, int chunk) const { return (int)(B * ((total_steps + chunk - 1) / chunk)); }
};
__host__ __device__ inline LfmQueue lfm_queue_view(int* base, int64_t B) {
  LfmQueue q; q.head = base; q.tail = base + 1; q.done = base + 4; q.ring = base + 4 + B; q.B = B; return q;
}

// Per-row noise of the heteroscedastic objective, c_i = v_i + jitter + sigma^2, folded into one unique row u (rows i in
// u): accumulates omega = sum 1/c_i, omega2 = sum 1/c_i^2, s = sum z_i / c_i, zz = sum z_i^2 / c_i and lc = sum log c_i.
// A non-positive (or NaN) c_i makes lc NaN: the kernels report it as a failed factorisation.
__device__ __forceinline__ void lfm_het_point(double z, double v, double c, double& om, double& om2, double& s,
                                              double& zz, double& lc) {
  const double ci = v + c;
  const double inv = 1.0 / ci;
  om += inv;
  om2 += inv * inv;
  s += z * inv;
  zz += z * z * inv;
  lc += ci > 0.0 ? log(ci) : __longlong_as_double(0x7ff8000000000000LL);
}
// ... and closes the row: cbar = R / omega (the diagonal of M = diag(cbar) + R K_u), q = cbar s, the weight
// tw = R omega2 / omega^2 of M^-1_uu in tr Sigma^-1; lc -= log cbar, tr0 += omega - omega2 / omega.
__device__ __forceinline__ void lfm_het_row(double R, double om, double om2, double s, double& cbar, double& q,
                                            double& tw, double& lc, double& tr0) {
  const double cb = R / om;
  cbar = cb;
  q = cb * s;
  tw = R * om2 / (om * om);
  lc -= log(cb);
  tr0 += om - om2 / om;
}

// batched_warp.cu: launches the warp-per-LFM kernel when the problem fits its limits, else LFM_ERR_UNSUPPORTED
int lfm_batched_warp_launch(cudaStream_t st, const BatchedArgs& a, int time_grid);
size_t lfm_batched_warp_structure_bytes(int N, int G, int MU, int MT);
int lfm_batched_warp_team(int64_t B, int N, int G, int MU, int time_grid);

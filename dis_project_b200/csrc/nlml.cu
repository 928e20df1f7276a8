// NLML and its gradient for one large LFM (objectives.py:21-78 + trainer.py:86-131), plus the
// vector kernels around the dense factorisation: residual z = y - mean, triangular mat-vecs with
// W = L^-1, log-det / quadratic-form reductions (warp-shuffle), bijector chain.
#include "sim_math.cuh"

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// z_i = y_i - (B/D)[i / (N/G)] * flag_i   (model.py:143-149, positional blocks), zero padded to Npad.
// With out_mean != NULL also writes the mean itself.
__global__ void lfm_residual_kernel(int64_t N, int64_t Npad, const double* __restrict__ X,
                                    const double* __restrict__ y, int G, const double* __restrict__ theta,
                                    double* __restrict__ z, double* __restrict__ out_mean) {
  const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i >= Npad) return;
  double zi = 0.0;
  if (i < N) {
    int64_t block = N / G;
    if (block < 1) block = 1;
    int64_t m = i / block;
    if (m > G - 1) m = G - 1;
    const double flag = (double)((int)X[3 * i + 2]);
    const double mu = theta[2 * G + m] / theta[m] * flag;
    if (out_mean) out_mean[i] = mu;
    zi = (y ? y[i] : 0.0) - mu;
  }
  if (z) z[i] = zi;
}

// w_i = sum_{k <= i} W[i][k] z[k]; one warp per row.
__global__ void __launch_bounds__(256) lfm_trmv_lower_kernel(int64_t n, const double* __restrict__ W, int64_t ldw,
                                                           const double* __restrict__ z, double* __restrict__ w) {
  const int64_t row = blockIdx.x * 8 + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (row >= n) return;
  const double* r = W + row * ldw;
  double acc = 0.0;
  const int64_t kend = row + 1;
  const int64_t k2 = kend & ~(int64_t)1;
  for (int64_t k = lane * 2; k < k2; k += 64) {
    const double2 a = *reinterpret_cast<const double2*>(r + k);
    const double2 b = *reinterpret_cast<const double2*>(z + k);
    acc += a.x * b.x + a.y * b.y;
  }
  if ((kend & 1) && lane == 0) acc += r[kend - 1] * z[kend - 1];
  acc = warp_sum(acc);
  if (lane == 0) w[row] = acc;
}

// partial[chunk][j] = sum_{i in chunk, i >= j} W[i][j] w[i]; 128 columns per CTA, 512 rows per chunk.
#define TC_ROWS 128
__global__ void __launch_bounds__(128) lfm_trmv_lowerT_kernel(int64_t n, const double* __restrict__ W, int64_t ldw,
                                                            const double* __restrict__ w,
                                                            double* __restrict__ partial) {
  const int64_t j = blockIdx.x * 128 + threadIdx.x;
  const int64_t r0 = (int64_t)blockIdx.y * TC_ROWS;
  const int64_t r1 = min(n, r0 + TC_ROWS);
  double acc0 = 0.0, acc1 = 0.0, acc2 = 0.0, acc3 = 0.0;
  if (r1 > (int64_t)blockIdx.x * 128) {
    int64_t i = max(r0, (int64_t)blockIdx.x * 128);
    for (; i + 4 <= r1; i += 4) {
      const double a0 = W[i * ldw + j], a1 = W[(i + 1) * ldw + j], a2 = W[(i + 2) * ldw + j],
                   a3 = W[(i + 3) * ldw + j];
      acc0 += (i >= j) ? a0 * w[i] : 0.0;
      acc1 += (i + 1 >= j) ? a1 * w[i + 1] : 0.0;
      acc2 += (i + 2 >= j) ? a2 * w[i + 2] : 0.0;
      acc3 += (i + 3 >= j) ? a3 * w[i + 3] : 0.0;
    }
    for (; i < r1; ++i) acc0 += (i >= j) ? W[i * ldw + j] * w[i] : 0.0;
  }
  partial[(int64_t)blockIdx.y * n + j] = (acc0 + acc1) + (acc2 + acc3);
}
__global__ void lfm_sum_partials_kernel(int64_t n, int nchunk, const double* __restrict__ partial,
                                        double* __restrict__ out) {
  const int64_t j = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (j >= n) return;
  double acc = 0.0;
  for (int c = 0; c < nchunk; ++c) acc += partial[(int64_t)c * n + j];
  out[j] = acc;
}

// y[m] -= A[m x n] x[n]; one warp per row (recursive TRSV of the value-only path).
__global__ void __launch_bounds__(256) lfm_gemv_sub_kernel(int64_t m, int64_t n, const double* __restrict__ A,
                                                         int64_t lda, const double* __restrict__ x,
                                                         double* __restrict__ y) {
  const int64_t row = blockIdx.x * 8 + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (row >= m) return;
  const double* r = A + row * lda;
  double acc = 0.0;
  for (int64_t k = lane * 2; k < n; k += 64) {
    const double2 a = *reinterpret_cast<const double2*>(r + k);
    const double2 b = *reinterpret_cast<const double2*>(x + k);
    acc += a.x * b.x + a.y * b.y;
  }
  acc = warp_sum(acc);
  if (lane == 0) y[row] -= acc;
}
// z_k <- W_kk z_k for one 128-block (4 warps x 32 rows each)
__global__ void __launch_bounds__(128) lfm_leaf_trmv_kernel(const double* __restrict__ Wkk, int64_t ldw,
                                                          double* __restrict__ z) {
  __shared__ double zs[LFM_NB];
  __shared__ double os[LFM_NB];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  zs[tid] = z[tid];
  __syncthreads();
  for (int r = warp; r < LFM_NB; r += 4) {
    double acc = 0.0;
    for (int k = lane; k <= r; k += 32) acc += Wkk[(int64_t)r * ldw + k] * zs[k];
    acc = warp_sum(acc);
    if (lane == 0) os[r] = acc;
  }
  __syncthreads();
  z[tid] = os[tid];
}

static int trsv_rec(cudaStream_t st, int64_t n, const double* L, int64_t ldl, const double* Wd, int64_t ldw,
                    double* z) {
  if (n == LFM_NB) {
    lfm_leaf_trmv_kernel<<<1, 128, 0, st>>>(Wd, ldw, z);
    LFM_LAUNCHED(1);
    LFM_CUDA_OK(cudaGetLastError());
    return LFM_OK;
  }
  const int64_t n1 = (n / LFM_NB / 2) * LFM_NB, n2 = n - n1;
  LFM_TRY(trsv_rec(st, n1, L, ldl, Wd, ldw, z));
  lfm_gemv_sub_kernel<<<(unsigned)((n2 + 7) / 8), 256, 0, st>>>(n2, n1, L + n1 * ldl, ldl, z, z + n1);
  LFM_LAUNCHED(1);
  LFM_CUDA_OK(cudaGetLastError());
  return trsv_rec(st, n2, L + n1 * ldl + n1, ldl, Wd + n1 * ldw + n1, ldw, z + n1);
}

// out[0] = 1/2 [ N log 2pi + 2 sum_i log L_ii + sum_i w_i^2 ]; NaN when info != 0.
__global__ void __launch_bounds__(1024) lfm_nlml_reduce_kernel(int64_t N, int64_t Npad, const double* __restrict__ L,
                                                             int64_t ldl, const double* __restrict__ w,
                                                             const int* __restrict__ info, double* __restrict__ out) {
  __shared__ double s1[32], s2[32];
  double a = 0.0, b = 0.0;
  for (int64_t i = threadIdx.x; i < Npad; i += 1024) {
    a += log(L[i * ldl + i]);
    const double wi = w[i];
    b += wi * wi;
  }
  a = warp_sum(a); b = warp_sum(b);
  if ((threadIdx.x & 31) == 0) { s1[threadIdx.x >> 5] = a; s2[threadIdx.x >> 5] = b; }
  __syncthreads();
  if (threadIdx.x < 32) {
    a = warp_sum(s1[threadIdx.x]); b = warp_sum(s2[threadIdx.x]);
    if (threadIdx.x == 0) {
      double v = 0.5 * ((double)N * LFM_LOG_2PI + 2.0 * a + b);
      if (*info != 0) v = nan("");
      out[0] = v;
    }
  }
}

__global__ void lfm_poison_kernel(int n, const int* __restrict__ info, double* __restrict__ out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n && *info != 0) out[i] = nan("");
}

// ---- bijectors ------------------------------------------------------------------------------
__global__ void lfm_constrain_kernel(int64_t B, int G, const double* __restrict__ u, double* __restrict__ th) {
  const int P = 3 * G + 2;
  const int64_t idx = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (idx >= B * P) return;
  const int p = (int)(idx % P);
  th[idx] = (p == 3 * G) ? lfm_l_forward(u[idx]) : lfm_softplus(u[idx]);
}
__global__ void lfm_unconstrain_kernel(int64_t B, int G, const double* __restrict__ th, double* __restrict__ u) {
  const int P = 3 * G + 2;
  const int64_t idx = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (idx >= B * P) return;
  const int p = (int)(idx % P);
  u[idx] = (p == 3 * G) ? lfm_l_inverse(th[idx]) : lfm_softplus_inv(th[idx]);
}
// One launch that prepares the device state of B fits (lfm_batched_fit_init): u = unconstrain(theta0), zero Adam moments,
// NaN loss history, zero info words, INT64_MAX best-objective keys.
__global__ void lfm_fit_init_kernel(int64_t B, int G, const double* __restrict__ th0, double* __restrict__ u,
                                    double* __restrict__ adam, double* __restrict__ hist, int64_t n_hist,
                                    int* __restrict__ info, long long* __restrict__ keys, int64_t n_keys) {
  const int P = 3 * G + 2;
  const int64_t n_u = B * P;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n_u + 2 * n_u + n_hist + B + n_keys; i += stride) {
    int64_t j = i;
    if (j < n_u) { const int p = (int)(j % P); u[j] = (p == 3 * G) ? lfm_l_inverse(th0[j]) : lfm_softplus_inv(th0[j]); continue; }
    j -= n_u;
    if (j < 2 * n_u) { if (adam) adam[j] = 0.0; continue; }
    j -= 2 * n_u;
    if (j < n_hist) { if (hist) hist[j] = nan(""); continue; }
    j -= n_hist;
    if (j < B) { if (info) info[j] = 0; continue; }
    j -= B;
    if (keys) keys[j] = 0x7fffffffffffffffLL;
  }
}
extern "C" int lfm_batched_fit_init(lfm_stream_t stream, int64_t B, int G, const double* theta0, double* theta_unc,
                                    double* adam_state, double* hist, int64_t n_hist, int* info, long long* keys,
                                    int64_t n_keys) {
  if (B <= 0 || G <= 0 || !theta0 || !theta_unc || n_hist < 0 || n_keys < 0) return LFM_ERR_INVALID;
  const int64_t total = 3 * B * (3 * (int64_t)G + 2) + n_hist + B + n_keys;
  int64_t blocks = (total + 255) / 256;
  if (blocks > 148 * 8) blocks = 148 * 8;
  lfm_fit_init_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(B, G, theta0, theta_unc, adam_state, hist, n_hist,
                                                                         info, keys, n_keys);
  LFM_LAUNCHED(1);
  LFM_CUDA_OK(cudaGetLastError());
  return LFM_OK;
}
// grad_unc = grad_con * d(constrained)/d(unconstrained)
__global__ void lfm_chain_kernel(int G, const double* __restrict__ u, double* __restrict__ grad) {
  const int P = 3 * G + 2;
  const int p = blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= P) return;
  const double sg = lfm_sigmoid(u[p]);
  const double jac = (p == 3 * G) ? (LFM_L_HIGH - LFM_L_LOW) * sg * (1.0 - sg) : sg;
  grad[p] *= jac;
}

// ---- host launchers shared with posterior.cu ------------------------------------------------------
int lfm_launch_residual(cudaStream_t st, int64_t N, int64_t Npad, const double* X, const double* y, int G,
                        const double* theta, double* z, double* out_mean) {
  lfm_residual_kernel<<<(unsigned)((Npad + 255) / 256), 256, 0, st>>>(N, Npad, X, y, G, theta, z, out_mean);
  LFM_LAUNCHED(1);
  LFM_CUDA_OK(cudaGetLastError());
  return LFM_OK;
}
size_t lfm_alpha_part_doubles(int64_t Np) { return (size_t)((Np + TC_ROWS - 1) / TC_ROWS) * Np; }
// w = W z, alpha = W^T w  (W = L^-1 lower, Np x Np)
int lfm_launch_alpha(cudaStream_t st, int64_t Np, const double* W, const double* z, double* w, double* part,
                     double* alpha) {
  lfm_trmv_lower_kernel<<<(unsigned)((Np + 7) / 8), 256, 0, st>>>(Np, W, Np, z, w);
  LFM_LAUNCHED(1);
  LFM_CUDA_OK(cudaGetLastError());
  const int nchunk = (int)((Np + TC_ROWS - 1) / TC_ROWS);
  lfm_trmv_lowerT_kernel<<<dim3((unsigned)(Np / 128), (unsigned)nchunk), 128, 0, st>>>(Np, W, Np, w, part);
  LFM_LAUNCHED(1);
  LFM_CUDA_OK(cudaGetLastError());
  lfm_sum_partials_kernel<<<(unsigned)((Np + 255) / 256), 256, 0, st>>>(Np, nchunk, part, alpha);
  LFM_LAUNCHED(1);
  LFM_CUDA_OK(cudaGetLastError());
  return LFM_OK;
}

// ---- workspace layout -------------------------------------------------------------------------
struct NlmlWs {
  int64_t Np, Tu;
  double *A, *W, *z, *w, *alpha, *theta, *part, *gscratch, *grid;
  size_t total_doubles;
};
static NlmlWs nlml_ws_layout(int64_t N, int G, int64_t time_grid, void* base) {
  NlmlWs s;
  s.Np = lfm_round_up(N, LFM_NB);
  s.Tu = lfm_grid_effective(N, G, time_grid);
  double* p = reinterpret_cast<double*>(base);
  size_t off = 0;
  auto take = [&](size_t n) { double* r = p ? p + off : nullptr; off += (n + 1) & ~(size_t)1; return r; };
  s.A = take((size_t)s.Np * s.Np);
  s.W = take((size_t)s.Np * s.Np);
  s.z = take(s.Np);
  s.w = take(s.Np);
  s.alpha = take(s.Np);
  s.theta = take(3 * (size_t)G + 2);
  s.part = take(lfm_alpha_part_doubles(s.Np));
  s.gscratch = take(lfm_grad_scratch_doubles(N));
  s.grid = take(lfm_grid_ws_doubles(N, G, s.Tu));
  s.total_doubles = off;
  return s;
}

extern "C" size_t lfm_nlml_workspace_bytes_tg(int64_t N, int G, int64_t time_grid) {
  if (N <= 0 || G <= 0) return 0;
  return nlml_ws_layout(N, G, time_grid, nullptr).total_doubles * sizeof(double);
}

static int check_common(int64_t N, int G, const void* X, const void* y, const void* theta, int64_t time_grid, void* ws,
                        size_t ws_bytes, void* out, void* info) {
  if (N <= 0 || G <= 0 || !X || !y || !theta || !ws || !out || !info) return LFM_ERR_INVALID;
  if (N % G) return LFM_ERR_INVALID;  // mean_function's reshape would fail (model.py:145-149)
  if ((reinterpret_cast<uintptr_t>(ws) & 15) != 0) return LFM_ERR_INVALID;
  if (time_grid < 0) return LFM_ERR_INVALID;
  if (ws_bytes < lfm_nlml_workspace_bytes_tg(N, G, time_grid)) return LFM_ERR_WORKSPACE;
  return LFM_OK;
}

// Shared front half: z, time-grid tables, Sigma, Cholesky.  Leaves L in ws.A and the inverted diagonal
// blocks in ws.W; `grid` is the table view the gradient contraction reuses.
// `variances` (N doubles or NULL) adds diag(variances) to Sigma: the heteroscedastic objective of the GPyTorch twin
// (src/gpytorch_alfi/model_alfi.py:294-299); it touches the diagonal tiles of the Sigma build only.
static int nlml_factor(cudaStream_t st, int64_t N, int G, const double* X, const double* y, const double* variances,
                       const double* theta, double jitter, const NlmlWs& s, bool grad, LfmGrid* grid, int* info,
                       double* ldiag = nullptr, int* early_done = nullptr, cudaEvent_t chain_ready = nullptr) {
  LFM_TRY(lfm_launch_residual(st, N, s.Np, X, y, G, theta, s.z, nullptr));
  LFM_TRY(lfm_grid_build(st, N, G, X, theta, s.Tu, grad, s.grid, grid));
  // the gradient needs W = L^-1 as well: built together with the factorisation.  When that is one right-looking sweep,
  // Sigma is built in two launches -- its first two block columns (all the first leaf and the first chain step read),
  // then the rest -- and the dependent chain starts behind the first one: ~50 us of an N = 4000 evaluation in which the
  // chain partition used to wait for 8 N^2 bytes of Sigma it does not touch.
  if (grad && chain_ready && lfm_potrf_trtri_is_one_sweep(s.Np) && s.Np >= 8 * LFM_NB) {
    LFM_CUDA_OK(cudaMemsetAsync(info, 0, sizeof(int), st));
    LFM_TRY(lfm_launch_sigma_lower(st, N, s.Np, X, G, theta, variances, jitter, 1, s.A, s.Np, grid, 0, 2 * LFM_NB));
    LFM_CUDA_OK(cudaEventRecord(chain_ready, st));
    LFM_TRY(lfm_launch_sigma_lower(st, N, s.Np, X, G, theta, variances, jitter, 1, s.A, s.Np, grid, 2 * LFM_NB, s.Np));
    return lfm_potrf_trtri_diag(st, s.Np, s.A, s.Np, s.W, s.Np, info, ldiag, early_done, chain_ready);
  }
  LFM_TRY(lfm_launch_sigma_lower(st, N, s.Np, X, G, theta, variances, jitter, 1, s.A, s.Np, grid));
  return grad ? lfm_potrf_trtri_diag(st, s.Np, s.A, s.Np, s.W, s.Np, info, ldiag, early_done)
              : lfm_potrf(st, s.Np, s.A, s.Np, s.W, s.Np, info);
}

extern "C" int lfm_nlml_het_tg(lfm_stream_t stream, int64_t N, int G, const double* X, const double* y,
                               const double* variances, const double* theta, double jitter, int64_t time_grid,
                               void* ws, size_t ws_bytes, double* out, int* info) {
  LFM_TRY(check_common(N, G, X, y, theta, time_grid, ws, ws_bytes, out, info));
  cudaStream_t st = (cudaStream_t)stream;
  const NlmlWs s = nlml_ws_layout(N, G, time_grid, ws);
  LfmGrid grid;
  LFM_TRY(nlml_factor(st, N, G, X, y, variances, theta, jitter, s, false, &grid, info));
  LFM_TRY(trsv_rec(st, s.Np, s.A, s.Np, s.W, s.Np, s.z));  // z <- L^-1 z
  lfm_nlml_reduce_kernel<<<1, 1024, 0, st>>>(N, s.Np, s.A, s.Np, s.z, info, out);
  LFM_LAUNCHED(1);
  LFM_CUDA_OK(cudaGetLastError());
  return LFM_OK;
}

// Side stream of an evaluation: w = W z, alpha = W^T w and the NLML reduction only read W, z and the diagonal of L,
// so they run beside Sigma^-1 = W^T W (the longest single launch of an evaluation) instead of in front of it.
struct EvalSide {
  cudaStream_t side = nullptr;
  cudaEvent_t fork = nullptr, join = nullptr, cols = nullptr;   // cols: the first two block columns of Sigma are built
  bool ok = false;
  bool init() {
    if (ok) return true;
    if (cudaStreamCreateWithFlags(&side, cudaStreamNonBlocking) != cudaSuccess) return false;
    if (cudaEventCreateWithFlags(&cols, cudaEventDisableTiming) != cudaSuccess) return false;
    if (cudaEventCreateWithFlags(&fork, cudaEventDisableTiming) != cudaSuccess) return false;
    if (cudaEventCreateWithFlags(&join, cudaEventDisableTiming) != cudaSuccess) return false;
    ok = true;
    return true;
  }
};
static thread_local EvalSide g_eval_side[16];  // per host thread and device

static int nlml_grad_impl(cudaStream_t st, int64_t N, int G, const double* X, const double* y, const double* variances,
                          const double* theta, double jitter, const NlmlWs& s, double* out, int* info) {
  const int P = 3 * G + 2;
  LfmGrid grid;
  // the diagonal of L moves out of the way during the factorisation (the gradient scratch is idle until the contraction):
  // Sigma^-1 overwrites L -- its first half block possibly before the factorisation is over (early_done)
  double* ldiag = s.gscratch;
  int early_done = 0;
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 16) dev = -1;
  cudaEvent_t chain_ready = (dev >= 0 && g_eval_side[dev].init()) ? g_eval_side[dev].cols : nullptr;
  LFM_TRY(nlml_factor(st, N, G, X, y, variances, theta, jitter, s, true, &grid, info, ldiag, &early_done, chain_ready));
  auto lauum = [&]() { return early_done ? lfm_lauum_late(st, s.Np, s.W, s.Np, s.A, s.Np) : lfm_lauum(st, s.Np, s.W, s.Np, s.A, s.Np); };
  if (dev >= 0 && g_eval_side[dev].init()) {
    EvalSide& es = g_eval_side[dev];
    LFM_CUDA_OK(cudaEventRecord(es.fork, st));
    LFM_CUDA_OK(cudaStreamWaitEvent(es.side, es.fork, 0));
    LFM_TRY(lfm_launch_alpha(es.side, s.Np, s.W, s.z, s.w, s.part, s.alpha));
    lfm_nlml_reduce_kernel<<<1, 1024, 0, es.side>>>(N, s.Np, ldiag, 0, s.w, info, out);   // ldl = 0: L[i * 0 + i]
    LFM_LAUNCHED(1);
    LFM_CUDA_OK(cudaGetLastError());
    LFM_CUDA_OK(cudaEventRecord(es.join, es.side));
    LFM_TRY(lauum());  // Sigma^-1 (lower) overwrites L
    LFM_CUDA_OK(cudaStreamWaitEvent(st, es.join, 0));
  } else {
    LFM_TRY(lfm_launch_alpha(st, s.Np, s.W, s.z, s.w, s.part, s.alpha));
    lfm_nlml_reduce_kernel<<<1, 1024, 0, st>>>(N, s.Np, ldiag, 0, s.w, info, out);
    LFM_LAUNCHED(1);
    LFM_CUDA_OK(cudaGetLastError());
    LFM_TRY(lauum());  // Sigma^-1 (lower) overwrites L
  }
  LFM_TRY(lfm_launch_grad_contract(st, N, X, G, theta, s.A, s.Np, s.alpha, s.gscratch, out + 1, &grid));
  lfm_poison_kernel<<<(P + 255) / 256, 256, 0, st>>>(P, info, out + 1);
  LFM_LAUNCHED(1);
  LFM_CUDA_OK(cudaGetLastError());
  return LFM_OK;
}

extern "C" int lfm_nlml_grad_het_tg(lfm_stream_t stream, int64_t N, int G, const double* X, const double* y,
                                    const double* variances, const double* theta, double jitter, int64_t time_grid,
                                    void* ws, size_t ws_bytes, double* out, int* info) {
  LFM_TRY(check_common(N, G, X, y, theta, time_grid, ws, ws_bytes, out, info));
  const NlmlWs s = nlml_ws_layout(N, G, time_grid, ws);
  return nlml_grad_impl((cudaStream_t)stream, N, G, X, y, variances, theta, jitter, s, out, info);
}

extern "C" int lfm_nlml_grad_unc_het_tg(lfm_stream_t stream, int64_t N, int G, const double* X, const double* y,
                                        const double* variances, const double* theta_unc, double jitter,
                                        int64_t time_grid, void* ws, size_t ws_bytes, double* out, int* info) {
  LFM_TRY(check_common(N, G, X, y, theta_unc, time_grid, ws, ws_bytes, out, info));
  cudaStream_t st = (cudaStream_t)stream;
  const NlmlWs s = nlml_ws_layout(N, G, time_grid, ws);
  const int P = 3 * G + 2;
  lfm_constrain_kernel<<<(P + 127) / 128, 128, 0, st>>>(1, G, theta_unc, s.theta);
  LFM_LAUNCHED(1);
  LFM_CUDA_OK(cudaGetLastError());
  LFM_TRY(nlml_grad_impl(st, N, G, X, y, variances, s.theta, jitter, s, out, info));
  lfm_chain_kernel<<<(P + 127) / 128, 128, 0, st>>>(G, theta_unc, out + 1);
  LFM_LAUNCHED(1);
  LFM_CUDA_OK(cudaGetLastError());
  return LFM_OK;
}

extern "C" int lfm_constrain(lfm_stream_t stream, int64_t B, int G, const double* theta_unc, double* theta) {
  if (B <= 0 || G <= 0 || !theta_unc || !theta) return LFM_ERR_INVALID;
  const int64_t n = B * (3 * (int64_t)G + 2);
  lfm_constrain_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(B, G, theta_unc, theta);
  LFM_LAUNCHED(1);
  LFM_CUDA_OK(cudaGetLastError());
  return LFM_OK;
}
extern "C" int lfm_unconstrain(lfm_stream_t stream, int64_t B, int G, const double* theta, double* theta_unc) {
  if (B <= 0 || G <= 0 || !theta_unc || !theta) return LFM_ERR_INVALID;
  const int64_t n = B * (3 * (int64_t)G + 2);
  lfm_unconstrain_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(B, G, theta, theta_unc);
  LFM_LAUNCHED(1);
  LFM_CUDA_OK(cudaGetLastError());
  return LFM_OK;
}

extern "C" int lfm_mean_function(lfm_stream_t stream, int64_t N, const double* X, int G, const double* theta,
                                 double* out) {
  if (N <= 0 || G <= 0 || !X || !theta || !out) return LFM_ERR_INVALID;
  if (N % G) return LFM_ERR_INVALID;
  lfm_residual_kernel<<<(unsigned)((N + 255) / 256), 256, 0, (cudaStream_t)stream>>>(N, N, X, nullptr, G, theta,
                                                                                   nullptr, out);
  LFM_LAUNCHED(1);
  LFM_CUDA_OK(cudaGetLastError());
  return LFM_OK;
}

// ---- debug / roofline helpers -----------------------------------------------------------------
extern "C" int lfm_debug_dgemm_nt(lfm_stream_t stream, int64_t M, int64_t N, int64_t K, const double* A,
                                  const double* B, double* C) {
  LfmGemm g;
  g.transA = 0; g.transB = 1; g.M = M; g.N = N; g.K = K; g.A = A; g.lda = K; g.B = B; g.ldb = K;
  g.C = C; g.ldc = N; g.alpha = 1.0; g.beta = 0.0; g.lower_only = 0; g.kmode = LFM_K_FULL;
  g.batch = 1; g.strideA = g.strideB = g.strideC = 0;
  return lfm_dgemm((cudaStream_t)stream, g);
}
// C(lower tiles, m x m, ldc) -= P P^T with P m x K (ldp): the trailing update of the blocked Cholesky
extern "C" int lfm_debug_syrk(lfm_stream_t stream, int64_t m, int64_t K, const double* P, int64_t ldp, double* Cm,
                              int64_t ldc) {
  LfmGemm g;
  g.transA = 0; g.transB = 1; g.M = m; g.N = m; g.K = K; g.A = P; g.lda = ldp; g.B = P; g.ldb = ldp;
  g.C = Cm; g.ldc = ldc; g.alpha = -1.0; g.beta = 1.0; g.lower_only = 1; g.kmode = LFM_K_FULL;
  g.batch = 1; g.strideA = g.strideB = g.strideC = 0;
  return lfm_dgemm((cudaStream_t)stream, g);
}
// the same launch with 8 debug words per CTA (LfmGemm::stamps): what a tile's life is made of
extern "C" int lfm_debug_syrk_stamps(lfm_stream_t stream, int64_t m, int64_t K, const double* P, int64_t ldp, double* Cm,
                                     int64_t ldc, long long* stamps) {
  LfmGemm g;
  g.transA = 0; g.transB = 1; g.M = m; g.N = m; g.K = K; g.A = P; g.lda = ldp; g.B = P; g.ldb = ldp;
  g.C = Cm; g.ldc = ldc; g.alpha = -1.0; g.beta = 1.0; g.lower_only = 1; g.kmode = LFM_K_FULL;
  g.batch = 1; g.strideA = g.strideB = g.strideC = 0;
  g.stamps = stamps;
  return lfm_dgemm((cudaStream_t)stream, g);
}
extern "C" int lfm_debug_potrf_potri(lfm_stream_t stream, int64_t n, double* A, double* W, double* Sinv,
                                     int* info) {
  if (n <= 0 || n % LFM_NB || !A || !W || !info) return LFM_ERR_INVALID;
  cudaStream_t st = (cudaStream_t)stream;
  if (Sinv) {
    LFM_TRY(lfm_potrf_trtri(st, n, A, n, W, n, info));
    LFM_TRY(lfm_lauum(st, n, W, n, Sinv, n));
  } else {
    LFM_TRY(lfm_potrf(st, n, A, n, W, n, info));
  }
  return LFM_OK;
}
// The factorisation and Sigma^-1 exactly as nlml_grad_impl runs them on Sigma (nlml_factor with grad = true, then lauum).
extern "C" int lfm_debug_potrf_potri_eval(lfm_stream_t stream, int64_t n, double* A, double* W, double* ldiag,
                                          int chain_ready, int* early_done, int* info) {
  if (n <= 0 || n % LFM_NB || !A || !W || !ldiag || !info) return LFM_ERR_INVALID;
  cudaStream_t st = (cudaStream_t)stream;
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 16) return LFM_ERR_CUDA;
  if (!g_eval_side[dev].init()) return LFM_ERR_CUDA;
  int early = 0;
  if (chain_ready && lfm_potrf_trtri_is_one_sweep(n)) {
    LFM_CUDA_OK(cudaMemsetAsync(info, 0, sizeof(int), st));
    LFM_CUDA_OK(cudaEventRecord(g_eval_side[dev].cols, st));
    LFM_TRY(lfm_potrf_trtri_diag(st, n, A, n, W, n, info, ldiag, &early, g_eval_side[dev].cols));
  } else {
    LFM_TRY(lfm_potrf_trtri_diag(st, n, A, n, W, n, info, ldiag, &early));
  }
  LFM_TRY(early ? lfm_lauum_late(st, n, W, n, A, n) : lfm_lauum(st, n, W, n, A, n));
  if (early_done) *early_done = early;
  return LFM_OK;
}

// C-ABI glue: version / status / device check, covariance entry points and the host-buffer
// convenience layer (lfm_*_host) with its scratch-caching handle.
#include <cstdlib>
#include <cstring>
#include "lfm_common.cuh"

int lfm_launch_cross_cov(cudaStream_t st, int64_t N, int64_t M, const double* X, const double* Y, int G,
                         const double* theta, double* out, int64_t ld);

std::atomic<unsigned long long> g_lfm_launches{0};
extern "C" unsigned long long lfm_debug_launch_count(void) { return g_lfm_launches.load(std::memory_order_relaxed); }

extern "C" int lfm_abi_version(void) { return LFM_ABI_VERSION; }

extern "C" const char* lfm_status_string(int status) {
  switch (status) {
    case LFM_OK: return "ok";
    case LFM_ERR_INVALID: return "invalid argument";
    case LFM_ERR_CUDA: return "CUDA runtime error";
    case LFM_ERR_UNSUPPORTED: return "unsupported size";
    case LFM_ERR_WORKSPACE: return "workspace too small";
    case LFM_ERR_NO_DEVICE: return "no sm_100 CUDA device (there is no CPU fallback)";
    case LFM_ERR_COMM: return "NCCL is not loadable or an NCCL call failed";
    default: return "unknown status";
  }
}

extern "C" int lfm_device_check(void) {
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) { cudaGetLastError(); return LFM_ERR_NO_DEVICE; }
  cudaDeviceProp p;
  if (cudaGetDeviceProperties(&p, dev) != cudaSuccess) { cudaGetLastError(); return LFM_ERR_NO_DEVICE; }
  return p.major == 10 ? LFM_OK : LFM_ERR_NO_DEVICE;
}

extern "C" int lfm_cross_covariance(lfm_stream_t stream, int64_t N, int64_t M, const double* X, const double* Y,
                                    int G, const double* theta, double* out, int64_t ld_out) {
  if (N < 0 || M < 0 || G <= 0 || !theta) return LFM_ERR_INVALID;
  if (N == 0 || M == 0) return LFM_OK;  // empty block: nothing to write
  if (!X || !Y || !out || ld_out < M) return LFM_ERR_INVALID;
  return lfm_launch_cross_cov((cudaStream_t)stream, N, M, X, Y, G, theta, out, ld_out);
}

extern "C" int lfm_gram(lfm_stream_t stream, int64_t N, const double* X, int G, const double* theta, double* out,
                        int64_t ld_out) {
  return lfm_cross_covariance(stream, N, N, X, X, G, theta, out, ld_out);
}

// ---- evaluation plans: one NLML+grad evaluation captured as a CUDA graph ----------------------------------
// An evaluation at N = 4000 is ~140 kernel launches on three streams with ~70 cross-stream event edges; replayed
// as a graph the dependent launches of the factorisation chain start ~1 us apart instead of ~3 us.  The plan
// binds fixed device buffers (a fit loop evaluates at new theta values written into the same buffer).
struct lfm_plan {
  cudaGraph_t graph;
  cudaGraphExec_t exec;
  unsigned long long launches;  // kernels one replay launches (bench.py's gpu_launches accounting)
};

static int plan_capture(lfm_plan* p, int64_t N, int G, const double* X, const double* y, const double* variances,
                        const double* theta, double jitter, int64_t time_grid, int unconstrained, void* ws,
                        size_t ws_bytes, double* out, int* info) {
  cudaStream_t cap = nullptr;
  LFM_CUDA_OK(cudaStreamCreateWithFlags(&cap, cudaStreamNonBlocking));
  auto run = [&]() {
    return unconstrained
               ? lfm_nlml_grad_unc_het_tg(cap, N, G, X, y, variances, theta, jitter, time_grid, ws, ws_bytes, out, info)
               : lfm_nlml_grad_het_tg(cap, N, G, X, y, variances, theta, jitter, time_grid, ws, ws_bytes, out, info);
  };
  // eager warm-up: argument validation and every lazy initialisation (function attributes, library streams and
  // events) happen outside the capture
  int st = run();
  if (st == LFM_OK && cudaStreamSynchronize(cap) != cudaSuccess) st = LFM_ERR_CUDA;
  if (st != LFM_OK) { cudaStreamDestroy(cap); return st; }
  const unsigned long long l0 = g_lfm_launches.load(std::memory_order_relaxed);
  if (cudaStreamBeginCapture(cap, cudaStreamCaptureModeThreadLocal) != cudaSuccess) {
    cudaStreamDestroy(cap);
    return LFM_ERR_CUDA;
  }
  st = run();
  cudaGraph_t g = nullptr;
  const cudaError_t e = cudaStreamEndCapture(cap, &g);
  // nothing ran during the capture: take this thread's captured launches back out of the counter (other threads may
  // have launched meanwhile; a concurrent launch makes the per-replay count of THIS plan an over-estimate, never the total)
  p->launches = g_lfm_launches.load(std::memory_order_relaxed) - l0;
  g_lfm_launches.fetch_sub(p->launches, std::memory_order_relaxed);
  cudaStreamDestroy(cap);
  if (st != LFM_OK || e != cudaSuccess || !g) { if (g) cudaGraphDestroy(g); cudaGetLastError(); return st != LFM_OK ? st : LFM_ERR_CUDA; }
  p->graph = g;
  // per-node priorities (the GEMM launches carry their stream's priority as a launch attribute, dgemm.cu): without this
  // flag every node of the graph runs at the priority of the stream the graph is launched into
  if (cudaGraphInstantiate(&p->exec, g, cudaGraphInstantiateFlagUseNodePriority) != cudaSuccess) {
    cudaGetLastError();
    if (cudaGraphInstantiate(&p->exec, g, 0) != cudaSuccess) { cudaGraphDestroy(g); cudaGetLastError(); return LFM_ERR_CUDA; }
  }
  return LFM_OK;
}

extern "C" int lfm_nlml_grad_plan_create_het(lfm_plan** out_plan, int64_t N, int G, const double* X, const double* y,
                                             const double* variances, const double* theta, double jitter,
                                             int64_t time_grid, int unconstrained, void* ws, size_t ws_bytes,
                                             double* out, int* info) {
  if (!out_plan) return LFM_ERR_INVALID;
  lfm_plan* p = (lfm_plan*)calloc(1, sizeof(lfm_plan));
  if (!p) return LFM_ERR_INVALID;
  const int st = plan_capture(p, N, G, X, y, variances, theta, jitter, time_grid, unconstrained, ws, ws_bytes, out, info);
  if (st != LFM_OK) { free(p); return st; }
  *out_plan = p;
  return LFM_OK;
}
extern "C" int lfm_nlml_grad_plan_create(lfm_plan** out_plan, int64_t N, int G, const double* X, const double* y,
                                         const double* theta, double jitter, int64_t time_grid, int unconstrained,
                                         void* ws, size_t ws_bytes, double* out, int* info) {
  return lfm_nlml_grad_plan_create_het(out_plan, N, G, X, y, nullptr, theta, jitter, time_grid, unconstrained, ws,
                                       ws_bytes, out, info);
}
extern "C" int lfm_plan_launch(lfm_plan* p, lfm_stream_t stream) {
  if (!p || !p->exec) return LFM_ERR_INVALID;
  LFM_CUDA_OK(cudaGraphLaunch(p->exec, (cudaStream_t)stream));
  LFM_LAUNCHED(p->launches);
  return LFM_OK;
}
extern "C" int lfm_plan_destroy(lfm_plan* p) {
  if (!p) return LFM_OK;
  if (p->exec) cudaGraphExecDestroy(p->exec);
  if (p->graph) cudaGraphDestroy(p->graph);
  free(p);
  return LFM_OK;
}

// ---- host-buffer layer --------------------------------------------------------------------------
struct lfm_handle {
  cudaStream_t stream;
  void* ws; size_t ws_bytes;       // device scratch (grown on demand)
  double* dbuf; size_t dbuf_bytes;  // device staging for inputs / outputs
  double* hpin; size_t hpin_bytes;  // pinned host staging
  int* dinfo;
  // cached evaluation plan of lfm_nlml_grad_host (valid while the staging buffers and the shape stay the same)
  lfm_plan* plan; int64_t plan_N, plan_tg; int plan_G, plan_unc; double plan_jitter;
  void* plan_ws; double* plan_dbuf;
  // rows of the X that sits at the start of the pinned staging buffer (every *_host entry point puts X there), and the
  // distinct-time count of that X (-1: not counted yet): a fit loop that passes the same X again pays one memcmp
  int64_t x_rows, x_tg;
  bool x_ok;       // every row of that X carries flag 1
  bool plan_het;   // the cached plan binds a variances buffer
};

// Stage X at the start of the pinned buffer; returns true when it is bit-identical to the X already there.
static bool stage_X(lfm_handle* h, int64_t N, const double* X) {
  const size_t bytes = 3 * (size_t)N * 8;
  if (h->x_rows == N && memcmp(h->hpin, X, bytes) == 0) return true;
  memcpy(h->hpin, X, bytes);
  h->x_rows = N; h->x_tg = -1;
  return false;
}

static int ensure(void** p, size_t* have, size_t need, bool pinned_host) {
  if (*have >= need) return LFM_OK;
  if (*p) { if (pinned_host) cudaFreeHost(*p); else cudaFree(*p); *p = nullptr; *have = 0; }
  cudaError_t e = pinned_host ? cudaMallocHost(p, need) : cudaMalloc(p, need);
  if (e != cudaSuccess) { cudaGetLastError(); return LFM_ERR_CUDA; }
  *have = need;
  return LFM_OK;
}

extern "C" int lfm_handle_create(lfm_handle** out) {
  if (!out) return LFM_ERR_INVALID;
  LFM_TRY(lfm_device_check());
  lfm_handle* h = (lfm_handle*)calloc(1, sizeof(lfm_handle));
  if (!h) return LFM_ERR_INVALID;
  if (cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking) != cudaSuccess) { free(h); return LFM_ERR_CUDA; }
  if (cudaMalloc((void**)&h->dinfo, 4096 * sizeof(int)) != cudaSuccess) { cudaStreamDestroy(h->stream); free(h); return LFM_ERR_CUDA; }
  *out = h;
  return LFM_OK;
}

extern "C" int lfm_handle_destroy(lfm_handle* h) {
  if (!h) return LFM_OK;
  cudaStreamSynchronize(h->stream);
  if (h->plan) lfm_plan_destroy(h->plan);
  if (h->ws) cudaFree(h->ws);
  if (h->dbuf) cudaFree(h->dbuf);
  if (h->hpin) cudaFreeHost(h->hpin);
  if (h->dinfo) cudaFree(h->dinfo);
  cudaStreamDestroy(h->stream);
  free(h);
  return LFM_OK;
}

static size_t r2(size_t n) { return (n + 1) & ~(size_t)1; }

// every training row must carry flag 1 (include/lfm_b200.h, lfm_nlml): checked where a host copy is at hand
static bool training_flags_ok(int64_t N, const double* X) {
  for (int64_t i = 0; i < N; ++i)
    if (X[3 * i + 2] != 1.0) return false;
  return true;
}

extern "C" int lfm_nlml_grad_het_host(lfm_handle* h, int64_t N, int G, const double* X, const double* y,
                                      const double* variances, const double* theta, double jitter, int unconstrained,
                                      double* out, int* info) {
  if (!h || N <= 0 || G <= 0 || !X || !y || !theta || !out) return LFM_ERR_INVALID;
  const size_t P = 3 * (size_t)G + 2;
  const size_t oy = r2(3 * (size_t)N), ov = oy + r2((size_t)N), oth = ov + (variances ? r2((size_t)N) : 0);
  const size_t nin = oth + r2(P);
  const size_t nout = r2(1 + P);
  {
    void* before = h->hpin;
    LFM_TRY(ensure((void**)&h->hpin, &h->hpin_bytes, (nin + nout) * 8, true));
    if (h->hpin != before) h->x_rows = 0;   // reallocated: the staged X is gone
  }
  if (!stage_X(h, N, X)) {   // a new X: validate and count once, not per evaluation
    h->x_ok = training_flags_ok(N, X);
    h->x_tg = lfm_count_distinct_times(N, X);
  }
  if (!h->x_ok) return LFM_ERR_UNSUPPORTED;
  if (h->x_tg < 0) h->x_tg = lfm_count_distinct_times(N, X);
  const int64_t tg = h->x_tg;
  LFM_TRY(ensure(&h->ws, &h->ws_bytes, lfm_nlml_workspace_bytes_tg(N, G, tg), false));
  LFM_TRY(ensure((void**)&h->dbuf, &h->dbuf_bytes, (nin + nout) * 8, false));
  double* hp = h->hpin;
  memcpy(hp + oy, y, (size_t)N * 8);
  if (variances) memcpy(hp + ov, variances, (size_t)N * 8);
  memcpy(hp + oth, theta, P * 8);
  LFM_CUDA_OK(cudaMemcpyAsync(h->dbuf, hp, nin * 8, cudaMemcpyHostToDevice, h->stream));
  double* dX = h->dbuf;
  double* dy = dX + oy;
  double* dv = variances ? dX + ov : nullptr;
  double* dth = dX + oth;
  double* dout = h->dbuf + nin;
  // the evaluation itself is a cached CUDA graph over the staging buffers (re-captured when they or the shape change)
  const bool reuse = h->plan && h->plan_N == N && h->plan_G == G && h->plan_tg == tg && h->plan_unc == unconstrained &&
                     h->plan_jitter == jitter && h->plan_ws == h->ws && h->plan_dbuf == h->dbuf &&
                     h->plan_het == (variances != nullptr);
  int st = LFM_OK;
  if (!reuse) {
    if (h->plan) { lfm_plan_destroy(h->plan); h->plan = nullptr; }
    LFM_CUDA_OK(cudaStreamSynchronize(h->stream));  // inputs are in place before the warm-up run of the capture
    st = lfm_nlml_grad_plan_create_het(&h->plan, N, G, dX, dy, dv, dth, jitter, tg, unconstrained, h->ws, h->ws_bytes,
                                       dout, h->dinfo);
    if (st != LFM_OK) return st;
    h->plan_N = N; h->plan_G = G; h->plan_tg = tg; h->plan_unc = unconstrained; h->plan_jitter = jitter;
    h->plan_ws = h->ws; h->plan_dbuf = h->dbuf; h->plan_het = variances != nullptr;
  }
  st = lfm_plan_launch(h->plan, h->stream);
  if (st != LFM_OK) return st;
  LFM_CUDA_OK(cudaMemcpyAsync(hp + nin, dout, (1 + P) * 8, cudaMemcpyDeviceToHost, h->stream));
  int hinfo = 0;
  LFM_CUDA_OK(cudaMemcpyAsync(&hinfo, h->dinfo, sizeof(int), cudaMemcpyDeviceToHost, h->stream));
  LFM_CUDA_OK(cudaStreamSynchronize(h->stream));
  memcpy(out, hp + nin, (1 + P) * 8);
  if (info) *info = hinfo;
  return LFM_OK;
}
extern "C" int lfm_nlml_grad_host(lfm_handle* h, int64_t N, int G, const double* X, const double* y,
                                  const double* theta, double jitter, int unconstrained, double* out, int* info) {
  return lfm_nlml_grad_het_host(h, N, G, X, y, nullptr, theta, jitter, unconstrained, out, info);
}

extern "C" int lfm_latent_posterior_host(lfm_handle* h, int64_t N, int G, const double* X, const double* y,
                                         const double* variances, const double* theta, double jitter,
                                         int64_t Tstar, const double* Xstar, double* out_mean, double* out_var,
                                         int* info) {
  if (!h || N <= 0 || G <= 0 || Tstar <= 0 || !X || !y || !variances || !theta || !Xstar || !out_mean || !out_var)
    return LFM_ERR_INVALID;
  const size_t P = 3 * (size_t)G + 2;
  const size_t oX = 0, oy = oX + r2(3 * (size_t)N), ov = oy + r2((size_t)N), oth = ov + r2((size_t)N),
               oXs = oth + r2(P), nin = oXs + r2(3 * (size_t)Tstar);
  const size_t nout = 2 * r2((size_t)Tstar);
  LFM_TRY(ensure(&h->ws, &h->ws_bytes, lfm_latent_posterior_workspace_bytes(N, G, Tstar), false));
  LFM_TRY(ensure((void**)&h->dbuf, &h->dbuf_bytes, (nin + nout) * 8, false));
  {
    void* before = h->hpin;
    LFM_TRY(ensure((void**)&h->hpin, &h->hpin_bytes, (nin + nout) * 8, true));
    if (h->hpin != before) h->x_rows = 0;
  }
  double* hp = h->hpin;
  if (!stage_X(h, N, X)) h->x_ok = training_flags_ok(N, X);
  if (!h->x_ok) return LFM_ERR_UNSUPPORTED;
  memcpy(hp + oy, y, (size_t)N * 8);
  memcpy(hp + ov, variances, (size_t)N * 8);
  memcpy(hp + oth, theta, P * 8);
  memcpy(hp + oXs, Xstar, 3 * (size_t)Tstar * 8);
  LFM_CUDA_OK(cudaMemcpyAsync(h->dbuf, hp, nin * 8, cudaMemcpyHostToDevice, h->stream));
  double* d = h->dbuf;
  double* dmean = d + nin;
  double* dvar = dmean + r2((size_t)Tstar);
  LFM_TRY(lfm_latent_posterior(h->stream, N, G, d + oX, d + oy, d + ov, d + oth, jitter, Tstar, d + oXs, h->ws,
                               h->ws_bytes, dmean, dvar, h->dinfo));
  LFM_CUDA_OK(cudaMemcpyAsync(hp + nin, dmean, nout * 8, cudaMemcpyDeviceToHost, h->stream));
  int hinfo = 0;
  LFM_CUDA_OK(cudaMemcpyAsync(&hinfo, h->dinfo, sizeof(int), cudaMemcpyDeviceToHost, h->stream));
  LFM_CUDA_OK(cudaStreamSynchronize(h->stream));
  memcpy(out_mean, hp + nin, (size_t)Tstar * 8);
  memcpy(out_var, hp + nin + r2((size_t)Tstar), (size_t)Tstar * 8);
  if (info) *info = hinfo;
  return LFM_OK;
}

extern "C" int lfm_batched_fit_het_host(lfm_handle* h, int64_t B, int64_t N, int G, const double* X, const double* y,
                                        const double* variances, const double* theta0, double jitter, double lr,
                                        double b1, double b2, double eps, int steps, int fix_params,
                                        int steps_per_epoch, double* out_theta, double* out_hist, int* info) {
  if (!h || B <= 0 || N <= 0 || G <= 0 || steps < 0 || !X || !y || !theta0 || !out_theta) return LFM_ERR_INVALID;
  const size_t P = 3 * (size_t)G + 2;
  // [X | y | variances (when given) | theta0]: one host->device copy
  const size_t nv = variances ? r2((size_t)N) : 0;
  const size_t oX = 0, oy = oX + r2(3 * (size_t)N), ov = oy + r2((size_t)N), oth = ov + nv, nin = oth + r2((size_t)B * P);
  const size_t ou = nin, oadam = ou + r2((size_t)B * P), ohist = oadam + r2(2 * (size_t)B * P),
               ntot = ohist + r2((size_t)B * (size_t)(steps > 0 ? steps : 1));
  LFM_TRY(ensure((void**)&h->dbuf, &h->dbuf_bytes, ntot * 8, false));
  {
    void* before = h->hpin;
    LFM_TRY(ensure((void**)&h->hpin, &h->hpin_bytes, ntot * 8, true));
    if (h->hpin != before) h->x_rows = 0;
  }
  int* dinfo = nullptr;
  double* hp = h->hpin;
  if (!stage_X(h, N, X)) h->x_ok = training_flags_ok(N, X);
  if (!h->x_ok) return LFM_ERR_UNSUPPORTED;
  if (h->x_tg < 0) h->x_tg = lfm_count_distinct_times(N, X);
  if (B > 4096) { LFM_CUDA_OK(cudaMalloc((void**)&dinfo, (size_t)B * sizeof(int))); } else dinfo = h->dinfo;
  memcpy(hp + oy, y, (size_t)N * 8);
  if (variances) memcpy(hp + ov, variances, (size_t)N * 8);
  memcpy(hp + oth, theta0, (size_t)B * P * 8);
  double* d = h->dbuf;
  int st = cudaMemcpyAsync(h->dbuf, hp, nin * 8, cudaMemcpyHostToDevice, h->stream) == cudaSuccess ? LFM_OK : LFM_ERR_CUDA;
  if (st == LFM_OK) st = lfm_unconstrain(h->stream, B, G, d + oth, d + ou);
  if (st == LFM_OK)
    st = lfm_batched_fit_het(h->stream, B, N, G, d + oX, d + oy, 0, variances ? d + ov : nullptr, 0, d + ou, d + oadam,
                             jitter, lr, b1, b2, eps, 0, steps, steps, fix_params, steps_per_epoch,
                             lfm_count_unique_rows(N, X), (int)h->x_tg, d + ohist, steps, d + oth, dinfo, nullptr,
                             nullptr, nullptr, 0, nullptr, 0);
  // d + oth (the start points, dead after lfm_unconstrain) receives the constrained result
  if (st == LFM_OK) {
    cudaMemcpyAsync(hp + ou, d + oth, (size_t)B * P * 8, cudaMemcpyDeviceToHost, h->stream);
    if (steps > 0 && out_hist) cudaMemcpyAsync(hp + ohist, d + ohist, (size_t)B * steps * 8, cudaMemcpyDeviceToHost, h->stream);
    if (info) cudaMemcpyAsync(info, dinfo, (size_t)B * sizeof(int), cudaMemcpyDeviceToHost, h->stream);
    if (cudaStreamSynchronize(h->stream) != cudaSuccess) st = LFM_ERR_CUDA;
  }
  if (st == LFM_OK) {
    memcpy(out_theta, hp + ou, (size_t)B * P * 8);
    if (steps > 0 && out_hist) memcpy(out_hist, hp + ohist, (size_t)B * steps * 8);
  }
  if (B > 4096) cudaFree(dinfo);
  return st;
}
extern "C" int lfm_batched_fit_host(lfm_handle* h, int64_t B, int64_t N, int G, const double* X, const double* y,
                                    const double* theta0, double jitter, double lr, double b1, double b2,
                                    double eps, int steps, int fix_params, int steps_per_epoch, double* out_theta,
                                    double* out_hist, int* info) {
  return lfm_batched_fit_het_host(h, B, N, G, X, y, nullptr, theta0, jitter, lr, b1, b2, eps, steps, fix_params,
                                  steps_per_epoch, out_theta, out_hist, info);
}

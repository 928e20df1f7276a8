// Batched posteriors: latent-force and gene-expression predictions of B fitted LFMs that share the design X and the
// test inputs Xstar, one CTA per LFM (ExactLFM.latent_predict / multi_gene_predict, src/model.py:420-514).
//
// The duplicate-row compression of the batched fits (batched.cu, include/lfm_b200.h): U unique rows of uniform
// multiplicity R, incidence P (N x U), K = P K_u P^T.  With a noise c_i per point,
//   omega_u = sum_{i in u} 1/c_i,  cbar_u = R / omega_u,  q_u = cbar_u sum_{i in u} z_i / c_i,
//   M = diag(cbar) + R K_u = L L^T,  beta = M^-1 q = P^T alpha,  P^T Sigma^-1 P = R M^-1,
// so for a test row with cross-covariance k_*u against the unique rows
//   mean = mean_t + k_*u^T beta,   k_*^T Sigma^-1 k_* = R || L^-1 k_*u ||^2.
// Latent: c_i = v_i + jitter, var = k(t*,t*) + 2 jitter - R ||L^-1 k_*u||^2.
// Gene:   c_i = v_i + sigma^2, var = k(t*,t*) - R ||L^-1 k_*u||^2 + jitter;
//         cov = K_tt - R V^T V + jitter I with V = L^-1 K_ut (staged in the caller's workspace).
//
// Per LFM the CTA folds the noise per unique row, builds and factorises M in shared memory, solves for beta and then
// streams the test rows in chunks: k_*u (the flag-aware pair function of lfm_launch_cross_cov), a forward
// substitution per test row (one thread per row), mean and variance.  Every sum has a fixed order that depends on
// the LFM's own data only: LFM b's outputs do not depend on B or on b.
#include "sim_math.cuh"

#include "batched.cuh"

#define BPOST_BT 128       // threads of the per-LFM kernel; U <= 128 rows, one thread per row in the Cholesky
#define BPOST_HDR 2048     // bytes of the structure block at the start of the workspace
#define BPOST_TILE 64      // covariance tile edge
#define BPOST_KU 16        // unique rows per staged slice of V in the covariance tiles

// Structure block (ints): [U, R, status, 0 | umap[128] | urow[128]].  status -1: more unique rows than the hint.
__global__ void __launch_bounds__(128) lfm_bpost_structure_kernel(int N, const double* __restrict__ X, int MU,
                                                                   int* __restrict__ st) {
  __shared__ int rep_s[128], cnt_s[128];
  __shared__ int sU, sR;
  const int tid = threadIdx.x;
  // the rule of lfm_count_unique_rows: compress only when every distinct (time, gene, flag) row occurs R > 1 times
  if (tid < N) {
    int rep = tid;
    const double t0 = X[3 * tid], g0 = X[3 * tid + 1], f0 = X[3 * tid + 2];
    for (int j = 0; j < tid; ++j)
      if (X[3 * j] == t0 && X[3 * j + 1] == g0 && X[3 * j + 2] == f0) { rep = j; break; }
    rep_s[tid] = rep;
  }
  __syncthreads();
  if (tid < N) {
    int cnt = 0;
    for (int j = 0; j < N; ++j) cnt += rep_s[j] == rep_s[tid];
    cnt_s[tid] = cnt;
  }
  __syncthreads();
  if (tid == 0) {
    int U = 0, uniform = 1;
    const int R = cnt_s[0];
    for (int j = 0; j < N; ++j) {
      U += rep_s[j] == j;
      if (cnt_s[j] != R) uniform = 0;
    }
    if (!uniform || R == 1) { U = N; sR = 1; } else sR = R;
    sU = U;
    st[0] = U; st[1] = sR; st[2] = U > MU ? -1 : 0; st[3] = 0;
  }
  __syncthreads();
  if (tid < N) {
    int mine = tid, first = 1;
    if (sR > 1) {
      const int rep = rep_s[tid];
      mine = 0;
      for (int j = 0; j < rep; ++j) mine += rep_s[j] == j;
      first = rep == tid;
    }
    st[4 + tid] = mine;
    if (first) st[4 + 128 + mine] = tid;
  }
}

struct BPostArgs {
  int64_t B, T;
  int N, G, MU, CT;
  const double* X;
  const double* y; int64_t y_stride;
  const double* var; int64_t var_stride;
  const double* theta;
  double jitter;
  const double* Xstar;
  const int* st;
  double* V;          // NULL, or B x MU x T: L^-1 K_ut of every LFM (gene posterior with the full covariance)
  double* out_mean;   // B x T
  double* out_var;    // B x T or NULL (gene)
  int* info;          // B
};

// p -> (r, c), r >= c, p = r (r + 1) / 2 + c
__device__ __forceinline__ void bpost_pair_decode(int64_t p, int& r, int& c) {
  int64_t rr = (int64_t)((sqrt(8.0 * (double)p + 1.0) - 1.0) * 0.5);
  while ((rr + 1) * (rr + 2) / 2 <= p) ++rr;
  while (rr * (rr + 1) / 2 > p) --rr;
  r = (int)rr;
  c = (int)(p - rr * (rr + 1) / 2);
}

// Shared memory of the per-LFM kernel: doubles [S | kc | q | cbar | beta | th | mu], then LfmPoint [pts | tp], then
// ints [umap | urow].
__host__ __device__ inline size_t bpost_smem_doubles(int G, int MU, int CT) {
  return (size_t)MU * (size_t)(MU | 1) + (size_t)MU * CT + 3 * (size_t)MU + 3 * (size_t)G + 2 + (size_t)G;
}
static size_t bpost_smem_bytes(int N, int G, int MU, int CT) {
  return bpost_smem_doubles(G, MU, CT) * 8 + ((size_t)MU + CT) * sizeof(LfmPoint) + ((size_t)N + MU) * sizeof(int);
}

template <bool GENE>
__global__ void __launch_bounds__(BPOST_BT) lfm_batched_posterior_kernel(BPostArgs a) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int N = a.N, G = a.G, MU = a.MU, CT = a.CT, P = 3 * G + 2;
  const int tid = threadIdx.x;
  const int64_t b = blockIdx.x, T = a.T;
  const int U = a.st[0], R = a.st[1];
  double* S = reinterpret_cast<double*>(smem_raw);   // M -> L (lower), U x (MU | 1)
  const int ld = MU | 1;
  double* kc = S + (size_t)MU * ld;                  // k_*u chunk -> L^-1 k_*u, U x CT
  double* q = kc + (size_t)MU * CT;                  // U
  double* cbar = q + MU;                             // U
  double* beta = cbar + MU;                          // U
  double* th = beta + MU;                            // P
  double* mu = th + P;                               // G
  LfmPoint* pts = reinterpret_cast<LfmPoint*>(S + bpost_smem_doubles(G, MU, CT));   // unique points, U
  LfmPoint* tp = pts + MU;                           // the chunk's test points, CT
  int* umap = reinterpret_cast<int*>(tp + CT);       // row -> unique index, N
  int* urow = umap + N;                              // unique index -> first row, U
  __shared__ double piv;
  __shared__ int fail;

  double* om = a.out_mean + b * T;
  double* ov = a.out_var ? a.out_var + b * T : nullptr;
  if (a.st[2] != 0) {   // more unique rows than the shared memory was sized for: refuse (info = -1)
    const double nan_v = nan("");
    for (int64_t i = tid; i < T; i += BPOST_BT) {
      om[i] = nan_v;
      if (ov) ov[i] = nan_v;
    }
    if (tid == 0) a.info[b] = -1;
    return;
  }
  if (tid == 0) fail = 0;
  if (tid < P) th[tid] = a.theta[b * P + tid];
  if (tid < N) umap[tid] = a.st[4 + tid];
  if (tid < U) urow[tid] = a.st[4 + 128 + tid];
  __syncthreads();
  if (tid < G) mu[tid] = th[2 * G + tid] / th[tid];
  const double l = th[3 * G], inv_l = 1.0 / l, sigma = th[3 * G + 1];
  const double c = GENE ? sigma * sigma : a.jitter;
  const double dR = (double)R;
  const double* yb = a.y + b * a.y_stride;
  const double* vb = a.var + b * a.var_stride;
  __syncthreads();
  // ---- noise folded per unique row (lfm_het_point / lfm_het_row), the unique points --------------------------------
  if (tid < U) {
    pts[tid] = lfm_make_point(a.X + 3 * urow[tid], G, th, th + G, l, false);
    const int blk = N / G;
    double o1 = 0.0, o2 = 0.0, s = 0.0, zz = 0.0, lc = 0.0, tw, tr0 = 0.0;
    for (int i = 0; i < N; ++i) {
      if (umap[i] == tid) {
        int m = i / blk;
        if (m > G - 1) m = G - 1;
        lfm_het_point(yb[i] - mu[m] * (double)((int)a.X[3 * i + 2]), vb[i], c, o1, o2, s, zz, lc);
      }
    }
    if (!(lc == lc)) fail = 1;   // some c_i <= 0 (or NaN): Sigma is not a covariance
    lfm_het_row(dR, o1, o2, s, cbar[tid], q[tid], tw, lc, tr0);
  }
  __syncthreads();
  // ---- M = diag(cbar) + R K_u (lower) -----------------------------------------------------------------------------
  const int npairs = U * (U + 1) / 2;
  for (int p = tid; p < npairs; p += BPOST_BT) {
    int r, cc;
    bpost_pair_decode(p, r, cc);
    double k = dR * lfm_kxx(pts[r], pts[cc], l, inv_l);
    if (r == cc) k += cbar[r];
    S[r * ld + cc] = k;
  }
  __syncthreads();
  // ---- Cholesky, left-looking, one thread per row -----------------------------------------------------------------
  for (int k = 0; k < U; ++k) {
    double v = 0.0;
    if (tid >= k && tid < U) {
      const double* ri = S + tid * ld;
      const double* rk = S + k * ld;
      double s0 = 0.0, s1 = 0.0;
      int m = 0;
      for (; m + 2 <= k; m += 2) { s0 += ri[m] * rk[m]; s1 += ri[m + 1] * rk[m + 1]; }
      if (m < k) s0 += ri[m] * rk[m];
      v = ri[k] - (s0 + s1);
      if (tid == k) piv = v;
    }
    __syncthreads();
    const double pk = piv;
    if (tid == 0 && !(pk >= 0x1p-1022) && fail == 0) fail = k + 1;   // below DBL_MIN fails: the rule of every batched kernel
    if (tid >= k && tid < U) {
      const double dk = sqrt(pk);
      S[tid * ld + k] = (tid == k) ? dk : v / dk;
    }
    __syncthreads();
  }
  // ---- beta = L^-T L^-1 q, column sweeps ---------------------------------------------------------------------------
  if (tid < U) beta[tid] = q[tid];
  __syncthreads();
  for (int k = 0; k < U; ++k) {
    const double wk = beta[k] / S[k * ld + k];
    __syncthreads();
    if (tid == k) beta[k] = wk;
    else if (tid > k && tid < U) beta[tid] -= S[tid * ld + k] * wk;
    __syncthreads();
  }
  for (int k = U - 1; k >= 0; --k) {
    const double bk = beta[k] / S[k * ld + k];
    __syncthreads();
    if (tid == k) beta[k] = bk;
    else if (tid < k) beta[tid] -= S[k * ld + tid] * bk;
    __syncthreads();
  }
  const bool bad = fail != 0;
  // ---- the test rows, CT at a time ---------------------------------------------------------------------------------
  int64_t block = T / G;
  if (block < 1) block = 1;
  double* Vb = a.V ? a.V + b * (int64_t)MU * T : nullptr;
  for (int64_t t0 = 0; t0 < T; t0 += CT) {
    const int nc = (int)((T - t0 < CT) ? T - t0 : CT);
    if (tid < nc) tp[tid] = lfm_make_point(a.Xstar + 3 * (t0 + tid), G, th, th + G, l, false);
    __syncthreads();
    for (int e = tid; e < U * nc; e += BPOST_BT) {
      const int u = e / nc, j = e - u * nc;
      kc[u * CT + j] = lfm_kernel(pts[u], tp[j], l, inv_l);
    }
    __syncthreads();
    if (tid < nc) {
      const int j = tid;
      double m0 = 0.0, m1 = 0.0;
      int u = 0;
      for (; u + 2 <= U; u += 2) { m0 += kc[u * CT + j] * beta[u]; m1 += kc[(u + 1) * CT + j] * beta[u + 1]; }
      if (u < U) m0 += kc[u * CT + j] * beta[u];
      // forward substitution in place: kc[:, j] <- L^-1 kc[:, j]
      double qq = 0.0;
      for (int i = 0; i < U; ++i) {
        const double* li = S + i * ld;
        double s0 = 0.0, s1 = 0.0;
        int k = 0;
        for (; k + 2 <= i; k += 2) { s0 += li[k] * kc[k * CT + j]; s1 += li[k + 1] * kc[(k + 1) * CT + j]; }
        if (k < i) s0 += li[k] * kc[k * CT + j];
        const double v = (kc[i * CT + j] - (s0 + s1)) / li[i];
        kc[i * CT + j] = v;
        qq += v * v;
        if (Vb) Vb[(int64_t)i * T + t0 + j] = v;
      }
      const int64_t it = t0 + j;
      const LfmPoint& pt = tp[j];
      const double kdiag = lfm_kernel(pt, pt, l, inv_l);
      int64_t g = it / block;
      if (g > G - 1) g = G - 1;
      // positional mean block and flag as lfm_post_finish_kernel / lfm_gene_mean_kernel (posterior.cu)
      const double flag = GENE ? (double)((int)a.Xstar[3 * it + 2]) : (double)pt.flag;
      double mean = th[2 * G + g] / th[g] * flag + (m0 + m1);
      double var = GENE ? kdiag - dR * qq + a.jitter : kdiag + a.jitter - dR * qq + a.jitter;
      if (bad) { mean = nan(""); var = nan(""); }
      om[it] = mean;
      if (ov) ov[it] = var;
    }
    __syncthreads();
  }
  if (tid == 0) a.info[b] = fail;
}

// cov (B x T x T) = K_tt - R V^T V + jitter I: lower 64 x 64 tiles, mirrored; the diagonal also goes to var.  256
// threads: a thread owns two adjacent columns and eight rows of the tile.
__global__ void __launch_bounds__(256) lfm_bpost_cov_kernel(int64_t B, int64_t T, int G, int MU,
                                                            const double* __restrict__ theta,
                                                            const double* __restrict__ Xstar, double jitter,
                                                            const int* __restrict__ st, const double* __restrict__ V,
                                                            const int* __restrict__ info, double* __restrict__ cov,
                                                            double* __restrict__ var) {
  __shared__ LfmPoint rowp[BPOST_TILE], colp[BPOST_TILE];
  __shared__ double buf[BPOST_TILE * (BPOST_TILE + 1)];   // V slices, then the transposed tile
  double* Vr = buf;
  double* Vc = buf + BPOST_KU * BPOST_TILE;
  const int P = 3 * G + 2;
  const int tid = threadIdx.x, tx = tid & 31, ty = tid >> 5;
  int tr, tc;
  bpost_pair_decode((int64_t)blockIdx.x, tr, tc);
  const int64_t r0 = (int64_t)tr * BPOST_TILE, c0 = (int64_t)tc * BPOST_TILE;
  const int U = st[2] ? 0 : st[0];   // status -1: V was never written, the tiles are NaN (info = -1)
  const double dR = (double)st[1];
  for (int64_t b = blockIdx.y; b < B; b += gridDim.y) {
    const double* th = theta + b * P;
    const double l = th[3 * G], inv_l = 1.0 / l;
    if (tid < 2 * BPOST_TILE) {
      const int k = tid & (BPOST_TILE - 1);
      const int64_t i = (tid < BPOST_TILE ? r0 : c0) + k;
      LfmPoint p;
      if (i < T) {
        p = lfm_make_point(Xstar + 3 * i, G, th, th + G, l, false);
      } else {
        p.t = 0; p.d = 1; p.s = 0; p.gam = 0; p.eg2 = 1; p.erfg = 0; p.e = 1; p.q = 0; p.g3 = 0; p.g4 = 0;
        p.gene = 0; p.flag = 1; p.ti = 0;
      }
      (tid < BPOST_TILE ? rowp : colp)[k] = p;
    }
    double acc[8][2];
#pragma unroll
    for (int r = 0; r < 8; ++r) acc[r][0] = acc[r][1] = 0.0;
    const double* Vb = V + b * (int64_t)MU * T;
    for (int u0 = 0; u0 < U; u0 += BPOST_KU) {
      __syncthreads();
      for (int e = tid; e < BPOST_KU * BPOST_TILE; e += 256) {
        const int u = u0 + e / BPOST_TILE, k = e & (BPOST_TILE - 1);
        Vr[e] = (u < U && r0 + k < T) ? Vb[(int64_t)u * T + r0 + k] : 0.0;
        Vc[e] = (u < U && c0 + k < T) ? Vb[(int64_t)u * T + c0 + k] : 0.0;
      }
      __syncthreads();
      const int nu = (U - u0 < BPOST_KU) ? U - u0 : BPOST_KU;
      for (int uu = 0; uu < nu; ++uu) {
        const double v0 = Vc[uu * BPOST_TILE + 2 * tx], v1 = Vc[uu * BPOST_TILE + 2 * tx + 1];
#pragma unroll
        for (int r = 0; r < 8; ++r) {
          const double w = Vr[uu * BPOST_TILE + ty + 8 * r];
          acc[r][0] += w * v0;
          acc[r][1] += w * v1;
        }
      }
    }
    __syncthreads();
    const bool bad = info[b] != 0;
    double* cb = cov + b * T * T;
#pragma unroll
    for (int r = 0; r < 8; ++r) {
      const int ri = ty + 8 * r;
      const int64_t i = r0 + ri;
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        const int cj = 2 * tx + h;
        const int64_t j = c0 + cj;
        double v = 0.0;
        if (i < T && j < T) {
          v = lfm_kernel(rowp[ri], colp[cj], l, inv_l) - dR * acc[r][h] + ((i == j) ? jitter : 0.0);
          if (bad) v = nan("");
          cb[i * T + j] = v;
          if (i == j && var) var[b * T + i] = v;
        }
        buf[cj * (BPOST_TILE + 1) + ri] = v;   // transposed for the mirror
      }
    }
    __syncthreads();
    if (tr != tc) {   // upper tile (tc, tr) = transpose of this one, written along its rows
      for (int k = tid; k < BPOST_TILE * BPOST_TILE; k += 256) {
        const int cj = k / BPOST_TILE, ri = k & (BPOST_TILE - 1);
        const int64_t i = r0 + ri, j = c0 + cj;
        if (i < T && j < T) cb[j * T + i] = buf[cj * (BPOST_TILE + 1) + ri];
      }
    }
  }
}

extern "C" size_t lfm_batched_posterior_workspace_bytes(int64_t B, int64_t N, int G, int64_t Tstar,
                                                        int unique_rows_hint, int full_cov) {
  if (B <= 0 || N <= 0 || N > 128 || G <= 0 || Tstar <= 0) return 0;
  const int64_t MU = (unique_rows_hint <= 0 || unique_rows_hint > N) ? N : unique_rows_hint;
  return BPOST_HDR + (full_cov ? (size_t)B * (size_t)MU * (size_t)Tstar * sizeof(double) : 0);
}

static int bpost_run(bool gene, lfm_stream_t stream, int64_t B, int64_t N, int G, const double* X, const double* y,
                     int64_t y_stride, const double* variances, int64_t var_stride, const double* theta, double jitter,
                     int64_t Tstar, const double* Xstar, int unique_rows_hint, void* ws, size_t ws_bytes,
                     double* out_mean, double* out_cov, double* out_var, int* info) {
  if (B <= 0 || N <= 0 || G <= 0 || Tstar <= 0 || !X || !y || !variances || !theta || !Xstar || !ws || !out_mean ||
      !info || (!gene && !out_var))
    return LFM_ERR_INVALID;
  if (N % G || (gene && Tstar % G)) return LFM_ERR_INVALID;
  if ((y_stride != 0 && y_stride < N) || (var_stride != 0 && var_stride < N)) return LFM_ERR_INVALID;
  if ((reinterpret_cast<uintptr_t>(ws) & 15) != 0) return LFM_ERR_INVALID;
  if (N > 128 || B > 0x7fffffff) return LFM_ERR_UNSUPPORTED;
  const int full = gene && out_cov;
  if (ws_bytes < lfm_batched_posterior_workspace_bytes(B, N, G, Tstar, unique_rows_hint, full))
    return LFM_ERR_WORKSPACE;
  const int MU = (unique_rows_hint <= 0 || unique_rows_hint > N) ? (int)N : unique_rows_hint;
  int CT = 128;
  while (CT > 32 && bpost_smem_bytes((int)N, G, MU, CT) > 227 * 1024) CT /= 2;
  const size_t smem = bpost_smem_bytes((int)N, G, MU, CT);
  if (smem > 227 * 1024 || 3 * G + 2 > BPOST_BT) return LFM_ERR_UNSUPPORTED;
  cudaStream_t st = (cudaStream_t)stream;
  int* sb = reinterpret_cast<int*>(ws);
  lfm_bpost_structure_kernel<<<1, 128, 0, st>>>((int)N, X, MU, sb);
  LFM_LAUNCHED(1);
  LFM_CUDA_OK(cudaGetLastError());
  BPostArgs a;
  a.B = B; a.T = Tstar; a.N = (int)N; a.G = G; a.MU = MU; a.CT = CT;
  a.X = X; a.y = y; a.y_stride = y_stride; a.var = variances; a.var_stride = var_stride;
  a.theta = theta; a.jitter = jitter; a.Xstar = Xstar; a.st = sb;
  a.V = full ? reinterpret_cast<double*>(reinterpret_cast<unsigned char*>(ws) + BPOST_HDR) : nullptr;
  a.out_mean = out_mean; a.out_var = out_var; a.info = info;
  static LfmSmemConfig conf_latent, conf_gene;
  if (gene) {
    LFM_CUDA_OK(lfm_ensure_smem(lfm_batched_posterior_kernel<true>, conf_gene, smem));
    lfm_batched_posterior_kernel<true><<<(unsigned)B, BPOST_BT, smem, st>>>(a);
  } else {
    LFM_CUDA_OK(lfm_ensure_smem(lfm_batched_posterior_kernel<false>, conf_latent, smem));
    lfm_batched_posterior_kernel<false><<<(unsigned)B, BPOST_BT, smem, st>>>(a);
  }
  LFM_LAUNCHED(1);
  LFM_CUDA_OK(cudaGetLastError());
  if (full) {
    const int64_t nt = (Tstar + BPOST_TILE - 1) / BPOST_TILE;
    const int64_t tiles = nt * (nt + 1) / 2;
    if (tiles > 0x7fffffff) return LFM_ERR_UNSUPPORTED;
    dim3 grid((unsigned)tiles, (unsigned)(B < 65535 ? B : 65535));
    lfm_bpost_cov_kernel<<<grid, 256, 0, st>>>(B, Tstar, G, MU, theta, Xstar, jitter, sb, a.V, info, out_cov, out_var);
    LFM_LAUNCHED(1);
    LFM_CUDA_OK(cudaGetLastError());
  }
  return LFM_OK;
}

extern "C" int lfm_batched_latent_posterior(lfm_stream_t stream, int64_t B, int64_t N, int G, const double* X,
                                            const double* y, int64_t y_stride, const double* variances,
                                            int64_t var_stride, const double* theta, double jitter, int64_t Tstar,
                                            const double* Xstar, int unique_rows_hint, void* ws, size_t ws_bytes,
                                            double* out_mean, double* out_var, int* info) {
  return bpost_run(false, stream, B, N, G, X, y, y_stride, variances, var_stride, theta, jitter, Tstar, Xstar,
                   unique_rows_hint, ws, ws_bytes, out_mean, nullptr, out_var, info);
}

extern "C" int lfm_batched_gene_posterior(lfm_stream_t stream, int64_t B, int64_t N, int G, const double* X,
                                          const double* y, int64_t y_stride, const double* variances,
                                          int64_t var_stride, const double* theta, double jitter, int64_t Tstar,
                                          const double* Xstar, int unique_rows_hint, void* ws, size_t ws_bytes,
                                          double* out_mean, double* out_cov, double* out_var, int* info) {
  return bpost_run(true, stream, B, N, G, X, y, y_stride, variances, var_stride, theta, jitter, Tstar, Xstar,
                   unique_rows_hint, ws, ws_bytes, out_mean, out_cov, out_var, info);
}

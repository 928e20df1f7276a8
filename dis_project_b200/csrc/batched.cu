// Batched small-N path: many independent LFMs (multi-start restarts, genes x replicas x candidate TFs)
// per GPU, one CTA per LFM, the whole problem resident in shared memory for all optimiser steps.
//
// Per step (JaxTrainer.step, src/trainer.py:105-131, inside the scan of :201-216):
//   theta = constrain(u)                                   (trainer.py:103)
//   Sigma = k_xx(X,X) + (jitter + sigma^2) I                (objectives.py:70-73)
//   NLML  = 1/2 [N log 2pi + log det Sigma + z^T Sigma^-1 z] (objectives.py:76-78)
//   grad  = sum_ab K_bar_ab dK_ab/dtheta, K_bar = 1/2 (Sigma^-1 - alpha alpha^T)   (AD of trainer.py:126)
//   u <- adam(u, grad * dtheta/du); "fix p21" hook          (trainer.py:127-128, 133-160, 205-210)
//
// Duplicate-row compression (exact).  The p53 layout repeats every (time, gene) row once per replicate
// (dataset.py:380-391), so Sigma = c I + P K_u P^T with K_u the U x U Gram of the UNIQUE rows, P the
// N x U 0/1 incidence and P^T P = R I (R = replicates), c = jitter + sigma^2.  With M = c I + R K_u:
//   log det Sigma = (N - U) log c + log det M
//   P^T Sigma^-1 P = R M^-1,   beta := P^T alpha = M^-1 q,  q = P^T z,   K_u beta = (q - c beta) / R
//   z^T Sigma^-1 z = (z^T z - q^T K_u beta) / c,   alpha = (z - P K_u beta) / c
//   sum_ij K_bar_ij dSigma_ij = sum_uv 1/2 (R M^-1 - beta beta^T)_uv dK_u,uv
// so every O(N^3) / O(N^2 transcendental) term shrinks to U.  Rows without uniform duplication use
// the same code with U = N, R = 1 (then M = Sigma, beta = alpha).  The sensitivity gradient uses
// diag(P^T K_bar P K_u)_u = 1/2 (1 - c M^-1_uu - beta_u (K_u beta)_u): no second copy of K is kept.
//
// The U x U shared-memory matrix S changes role over a step: lower = M -> L -> M^-1 -> weighted
// row-gene derivative; upper = W^T (W = L^-1) -> column-gene derivative.  Every reduction has a fixed
// order: results are bit-reproducible.
#include "sim_math.cuh"


#include "batched.cuh"
#include <vector>

template <int BT>
__device__ __forceinline__ double block_sum(double v, double* red) {
  // fixed-order block reduction; all BT threads must call
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  __syncthreads();
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
  __syncthreads();
  double s = 0.0;
#pragma unroll
  for (int w = 0; w < BT / 32; ++w) s += red[w];
  return s;
}

__device__ __forceinline__ void pair_decode(int p, int& r, int& c) {
  r = (int)((sqrtf(8.0f * (float)p + 1.0f) - 1.0f) * 0.5f);
  while ((r + 1) * (r + 2) / 2 <= p) ++r;
  while (r * (r + 1) / 2 > p) --r;
  c = p - r * (r + 1) / 2;
}

// BT = 128 when the unique rows fit 64 (two threads per row in the Cholesky), else 256.
// HET: heteroscedastic objective (a.var != NULL), noise c_i = v_i + c per point; M = diag(cbar) + R K_u (header of
// include/lfm_b200.h, lfm_batched_nlml_grad_unc_het).
template <int BT, bool HET>
__global__ void __launch_bounds__(BT, (BT == 128) ? 4 : 2) lfm_batched_kernel(BatchedArgs a) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int N = a.N, G = a.G, P = 3 * G + 2;
  const int tid = threadIdx.x;
  const int64_t bidx = blockIdx.x;
  const double* yb = a.y + bidx * a.y_stride;   // this LFM's observations (y_stride = 0: shared)
  const double* vb = HET ? a.var + bidx * a.var_stride : nullptr;   // ... and their variances
  // ---- carve shared memory (matrix sized for the worst case U = N) ---------------------------------
  const int MU = a.max_unique;
  double* S = reinterpret_cast<double*>(smem_raw);
  double* q = S + (size_t)MU * (MU | 1);  // P^T z            (U)
  double* w = q + N;                    // W q                (U)
  double* beta = w + N;                 // M^-1 q             (U)
  double* kb = beta + N;                // K_u beta           (U)
  double* wdiag = kb + N;               // 1 / L_ii           (U)
  double* sdiag = wdiag + N;            // M^-1_uu            (U)
  double* dsum = sdiag + N;             // per-point decay-gradient totals (U)
  double* th = dsum + N;                // P constrained
  double* u = th + P;                   // P unconstrained
  double* gr = u + P;                   // P gradient
  double* am = gr + P;                  // P adam m
  double* av = am + P;                  // P adam v
  double* mu = av + P;                  // G positional means B/D
  double* red = mu + G;                 // 16
  double* cbar = red + 16;              // HET: R / sum_{i in u} 1/c_i     (U)
  double* tw = cbar + (HET ? N : 0);    // HET: weight of M^-1_uu in tr Sigma^-1 (U)
  LfmPoint* pts = reinterpret_cast<LfmPoint*>(red + 16 + (HET ? 2 * N : 0));
  int* umap = reinterpret_cast<int*>(pts + N);  // row -> unique index      (N)
  int* urow = umap + N;                         // unique index -> first row (N)
  __shared__ double piv;
  __shared__ int fail, sU, sR;

  if (tid < P) {
    u[tid] = a.u_io[bidx * P + tid];
    const bool have = a.adam != nullptr && a.first_step > 0;
    am[tid] = have ? a.adam[bidx * 2 * P + tid] : 0.0;
    av[tid] = have ? a.adam[bidx * 2 * P + P + tid] : 0.0;
  }
  if (tid == 0) fail = 0;
  // ---- duplicate-row detection (once): rep = first identical row; uniform multiplicity R? ----------
  if (tid < N) {
    int rep = tid;
    const double t0 = a.X[3 * tid], g0 = a.X[3 * tid + 1], f0 = a.X[3 * tid + 2];
    for (int j = 0; j < tid; ++j)
      if (a.X[3 * j] == t0 && a.X[3 * j + 1] == g0 && a.X[3 * j + 2] == f0) { rep = j; break; }
    umap[tid] = rep;  // temporarily the representative row
  }
  __syncthreads();
  if (tid < N) {
    int idx = 0, cnt = 0;
    const int rep = umap[tid];
    for (int j = 0; j < N; ++j) {
      if (j < rep && umap[j] == j) ++idx;   // unique rows before my representative
      if (umap[j] == rep) ++cnt;            // multiplicity of my class
    }
    urow[tid] = (rep == tid) ? idx : -1;    // temporarily: compact index if I am a representative
    dsum[tid] = (double)cnt;
  }
  __syncthreads();
  if (tid == 0) {
    int U = 0, R = (int)dsum[0], uniform = 1;
    for (int j = 0; j < N; ++j) {
      if (urow[j] >= 0) ++U;
      if ((int)dsum[j] != R) uniform = 0;
    }
    if (!uniform || R == 1) { U = N; R = 1; }
    if (U > MU) { U = 0; fail = -1; }  // caller's unique-row bound was wrong: refuse (info = -1)
    sU = U; sR = R;
  }
  __syncthreads();
  const int U = sU, R = sR;
  {
    int mine = 0, first = 0;
    if (tid < N) {
      if (R == 1) { mine = tid; }
      else {
        const int rep = umap[tid];
        int idx = 0;
        for (int j = 0; j < rep; ++j) if (umap[j] == j) ++idx;
        mine = idx;
      }
      first = (R == 1) ? 1 : (umap[tid] == tid);
    }
    __syncthreads();
    if (tid < N) {
      umap[tid] = mine;
      if (first) urow[mine] = tid;
    }
  }
  __syncthreads();

  const int ld = U | 1;
  const int npairs = U * (U + 1) / 2;
  const bool eval_only = a.eval_val != nullptr;
  const int nsteps = eval_only ? 1 : a.steps;
  const int blk = N / G;  // rows per positional mean block (model.py:145)
  const double dR = (double)R;

  for (int sidx = 0; sidx < nsteps; ++sidx) {
    const int step = a.first_step + sidx;
    // ---- A. constrain -----------------------------------------------------------------------
    if (tid < P) th[tid] = (tid == 3 * G) ? lfm_l_forward(u[tid]) : lfm_softplus(u[tid]);
    __syncthreads();
    const double l = th[3 * G], inv_l = 1.0 / l, sigma = th[3 * G + 1];
    const double c = a.jitter + sigma * sigma;
    // ---- B. unique points, q = P^T z, z^T z ------------------------------------------------------
    if (tid < G) mu[tid] = th[2 * G + tid] / th[tid];
    if (tid < U) pts[tid] = lfm_make_point(a.X + 3 * urow[tid], G, th, th + G, l, true);
    __syncthreads();
    double zz, lsum = 0.0, tr0 = 0.0;   // HET: zz = sum z_i^2 / c_i, lsum = sum log c_i - sum log cbar_u, tr0
    if constexpr (!HET) {
    double zz_part = 0.0;
    if (tid < N) {
      int m = tid / blk;
      if (m > G - 1) m = G - 1;
      const double zi = yb[tid] - mu[m] * (double)((int)a.X[3 * tid + 2]);
      zz_part = zi * zi;
    }
    zz = block_sum<BT>(zz_part, red);
    if (tid < U) {
      double acc = 0.0;
      for (int i = 0; i < N; ++i) {
        if (umap[i] == tid) {
          int m = i / blk;
          if (m > G - 1) m = G - 1;
          acc += yb[i] - mu[m] * (double)((int)a.X[3 * i + 2]);
        }
      }
      q[tid] = acc;
    }
    } else {
    double zp = 0.0, lp = 0.0, tp = 0.0;
    if (tid < U) {
      double om = 0.0, om2 = 0.0, s = 0.0;
      for (int i = 0; i < N; ++i) {
        if (umap[i] == tid) {
          int m = i / blk;
          if (m > G - 1) m = G - 1;
          lfm_het_point(yb[i] - mu[m] * (double)((int)a.X[3 * i + 2]), vb[i], c, om, om2, s, zp, lp);
        }
      }
      lfm_het_row(dR, om, om2, s, cbar[tid], q[tid], tw[tid], lp, tp);
    }
    zz = block_sum<BT>(zp, red);
    lsum = block_sum<BT>(lp, red);
    tr0 = block_sum<BT>(tp, red);
    if (tid == 0 && !(lsum == lsum) && fail == 0) fail = 1;   // some c_i <= 0: Sigma is not a covariance
    }
    // ---- C. M = c I + R K_u (lower + diagonal) -------------------------------------------------------
    for (int p = tid; p < npairs; p += BT) {
      int r, cc;
      pair_decode(p, r, cc);
      double k = dR * lfm_kxx(pts[r], pts[cc], l, inv_l);
      if (r == cc) k += HET ? cbar[r] : c;
      S[r * ld + cc] = k;
    }
    __syncthreads();
    // ---- D. Cholesky, left-looking, two threads per row -----------------------------------------
    {
      const int row = tid >> 1, half = tid & 1;
      for (int k = 0; k < U; ++k) {
        double v = 0.0;
        if (row >= k && row < U) {
          const double* ri = S + row * ld;
          const double* rk = S + k * ld;
          double s0 = 0.0, s1 = 0.0;
          int m = half;
          for (; m + 2 < k; m += 4) { s0 += ri[m] * rk[m]; s1 += ri[m + 2] * rk[m + 2]; }
          for (; m < k; m += 2) s0 += ri[m] * rk[m];
          v = s0 + s1;
        }
        v += __shfl_xor_sync(0xffffffffu, v, 1);
        if (row >= k && row < U) {
          v = S[row * ld + k] - v;
          if (row == k && half == 0) piv = v;
        }
        __syncthreads();
        const double p = piv;
        if (tid == 0 && !(p > 0.0) && fail == 0) fail = k + 1;
        if (row >= k && row < U && half == 0) {
          const double dk = sqrt(p);
          S[row * ld + k] = (row == k) ? dk : v / dk;
        }
        __syncthreads();
      }
    }
    // ---- E. log det M, W = L^-1 into the upper triangle (thread cc owns column cc) -----------------
    double logdet_part = 0.0;
    if (tid < U) {
      const double lii = S[tid * ld + tid];
      logdet_part = log(lii);
      wdiag[tid] = 1.0 / lii;
    }
    const double logdetM = 2.0 * block_sum<BT>(logdet_part, red);
    if (tid < U) {
      const int cc = tid;
      const double wcc = wdiag[cc];
      const int cmin = (tid >> 5) << 5;
      double* wc = S + cc * ld;  // wc[i] = W[i][cc] for i > cc (row cc of the upper triangle)
      for (int i = cmin + 1; i < U; ++i) {
        const double* li = S + i * ld;
        double s0 = 0.0, s1 = 0.0;
        int k = cmin;
        for (; k + 2 <= i; k += 2) {
          const double w0 = (k == cc) ? wcc : wc[k];
          const double w1 = (k + 1 == cc) ? wcc : wc[k + 1];
          if (k >= cc) s0 += li[k] * w0;
          if (k + 1 >= cc) s1 += li[k + 1] * w1;
        }
        for (; k < i; ++k) {
          const double w0 = (k == cc) ? wcc : wc[k];
          if (k >= cc) s0 += li[k] * w0;
        }
        if (i > cc) wc[i] = -(s0 + s1) * wdiag[i];
      }
    }
    __syncthreads();
    // ---- F. w = W q, beta = W^T w, K_u beta = (q - c beta) / R ------------------------------------------
    if (tid < U) {
      double acc = wdiag[tid] * q[tid];
      for (int k = 0; k < tid; ++k) acc += S[k * ld + tid] * q[k];
      w[tid] = acc;
    }
    __syncthreads();
    double qkb_part = 0.0, kbkb_part = 0.0;
    if (tid < U) {
      double acc = wdiag[tid] * w[tid];
      const double* uj = S + tid * ld;
      for (int i = tid + 1; i < U; ++i) acc += uj[i] * w[i];
      beta[tid] = acc;
      const double kbv = (q[tid] - (HET ? cbar[tid] : c) * acc) / dR;
      kb[tid] = kbv;
      qkb_part = (HET ? q[tid] / cbar[tid] : q[tid]) * kbv;
      kbkb_part = kbv * kbv;
    }
    const double qkb = block_sum<BT>(qkb_part, red);
    const double kbkb = block_sum<BT>(kbkb_part, red);
    const double quad = HET ? zz - qkb : (zz - qkb) / c;
    const double nlml = 0.5 * ((double)N * LFM_LOG_2PI + (HET ? lsum : (double)(N - U) * log(c)) + logdetM + quad);
    // ---- G. M^-1 = W^T W into the lower triangle (+ sdiag), every entry independent --------------------
    for (int p = tid; p < npairs; p += BT) {
      int r, cc;
      pair_decode(p, r, cc);
      // Minv[r][cc] = sum_{k >= r} W[k][r] W[k][cc];  W[k][r] = S[r][k] (k > r), W[r][r] = wdiag[r]
      const double* ur = S + r * ld;
      const double* uc = S + cc * ld;
      double s0 = wdiag[r] * ((r == cc) ? wdiag[r] : uc[r]);
      double s1 = 0.0;
      int k = r + 1;
      for (; k + 2 <= U; k += 2) { s0 += ur[k] * uc[k]; s1 += ur[k + 1] * uc[k + 1]; }
      for (; k < U; ++k) s0 += ur[k] * uc[k];
      const double v = s0 + s1;
      if (r == cc) sdiag[r] = v;
      else S[r * ld + cc] = v;  // lower; L is dead
    }
    __syncthreads();
    // ---- H. fused derivative contraction over the lower triangle of the unique pairs --------------------
    double dl_part = 0.0;
    for (int p = tid; p < npairs; p += BT) {
      int r, cc;
      pair_decode(p, r, cc);
      const double minv = (r == cc) ? sdiag[r] : S[r * ld + cc];
      const double wgt = ((r == cc) ? 0.5 : 1.0) * (dR * minv - beta[r] * beta[cc]);
      double k, dr, dc, dl;
      lfm_kxx_grad(pts[r], pts[cc], l, inv_l, k, dr, dc, dl);
      dl_part += wgt * dl;
      if (r == cc) dsum[r] = wgt * (dr + dc);
      else { S[r * ld + cc] = wgt * dr; S[cc * ld + r] = wgt * dc; }
    }
    const double gl = block_sum<BT>(dl_part, red);
    if (tid < U) {  // per-point totals: full row sums
      const double* rp = S + tid * ld;
      double s0 = dsum[tid], s1 = 0.0;
      int cc = 0;
      for (; cc + 2 <= U; cc += 2) {
        s0 += (cc == tid) ? 0.0 : rp[cc];
        s1 += (cc + 1 == tid) ? 0.0 : rp[cc + 1];
      }
      for (; cc < U; ++cc) s0 += (cc == tid) ? 0.0 : rp[cc];
      dsum[tid] = s0 + s1;
    }
    __syncthreads();
    // ---- J. fold by gene; mean-function terms; sigma ---------------------------------------------
    if (tid < G) {
      const int m = tid;
      double gd = 0.0, gs = 0.0, asum = 0.0;
      for (int i = 0; i < U; ++i) {
        if (pts[i].gene == m) {
          gd += dsum[i];
          gs += 1.0 - (HET ? cbar[i] : c) * sdiag[i] - beta[i] * kb[i];
        }
      }
      // asum_m = sum_{i in positional block m} alpha_i,  alpha_i = (z_i - (K_u beta)_{u(i)}) / c_i
      if constexpr (HET) {
        for (int i = m * blk; i < (m + 1) * blk; ++i)
          asum += (yb[i] - mu[m] * (double)((int)a.X[3 * i + 2]) - kb[umap[i]]) / (vb[i] + c);
      } else {
        for (int i = m * blk; i < (m + 1) * blk; ++i)
          asum += yb[i] - mu[m] * (double)((int)a.X[3 * i + 2]) - kb[umap[i]];
        asum /= c;
      }
      const double D = th[m], Sm = th[G + m], Bm = th[2 * G + m];
      gr[m] = gd + asum * Bm / (D * D);
      gr[G + m] = gs / Sm;
      gr[2 * G + m] = -asum / D;
    }
    if (tid == G) {
      double tr = 0.0, trSinv, aa;
      if constexpr (HET) {
        // tr Sigma^-1 = tr0 + sum_u tw_u M^-1_uu,  alpha^T alpha = sum_i alpha_i^2
        for (int i = 0; i < U; ++i) tr += tw[i] * sdiag[i];
        trSinv = tr0 + tr;
        aa = 0.0;
        for (int i = 0; i < N; ++i) {
          int m = i / blk;
          if (m > G - 1) m = G - 1;
          const double al = (yb[i] - mu[m] * (double)((int)a.X[3 * i + 2]) - kb[umap[i]]) / (vb[i] + c);
          aa += al * al;
        }
      } else {
        for (int i = 0; i < U; ++i) tr += sdiag[i];
        trSinv = ((double)(N - U) + c * tr) / c;
        aa = (zz - 2.0 * qkb + dR * kbkb) / (c * c);
      }
      gr[3 * G] = gl;
      gr[3 * G + 1] = sigma * (trSinv - aa);
    }
    __syncthreads();
    // ---- K. chain rule, Adam, hook ----------------------------------------------------------------
    const bool bad = fail != 0;
    if (tid < P) {
      const double sg = lfm_sigmoid(u[tid]);
      const double jac = (tid == 3 * G) ? (LFM_L_HIGH - LFM_L_LOW) * sg * (1.0 - sg) : sg;
      double g = gr[tid] * jac;
      if (bad) g = nan("");
      if (eval_only) {
        a.eval_grad[bidx * P + tid] = g;
      } else {
        const double m1 = a.b1 * am[tid] + (1.0 - a.b1) * g;
        const double v1 = a.b2 * av[tid] + (1.0 - a.b2) * g * g;
        am[tid] = m1; av[tid] = v1;
        const double mhat = m1 / (1.0 - pow(a.b1, (double)(step + 1)));
        const double vhat = v1 / (1.0 - pow(a.b2, (double)(step + 1)));
        double un = u[tid] - a.lr * mhat / (sqrt(vhat) + a.eps);
        if (a.fix_params && (step % a.steps_per_epoch) == 0 && G > 3) {
          if (tid == G + 3) un = 1.0;  // true_s[3]  (trainer.py:152, unconstrained space: SURVEY Q5)
          if (tid == 3) un = 0.8;      // true_d[3]  (trainer.py:153)
        }
        u[tid] = un;
      }
    }
    if (tid == 0) {
      const double v = bad ? nan("") : nlml;
      if (eval_only) a.eval_val[bidx] = v;
      else {
        if (a.hist) a.hist[bidx * a.ld_hist + step] = v;
        if (a.step_keys && v == v) atomicMin(a.step_keys + step, lfm_loss_key(v));   // best objective of EVERY step
      }
    }
    __syncthreads();
  }

  if (!eval_only && tid < P) {
    a.u_io[bidx * P + tid] = u[tid];
    if (a.adam) { a.adam[bidx * 2 * P + tid] = am[tid]; a.adam[bidx * 2 * P + P + tid] = av[tid]; }
    if (a.theta_out && a.first_step + a.steps >= a.total_steps) {
      double t = (tid == 3 * G) ? lfm_l_forward(u[tid]) : lfm_softplus(u[tid]);  // trainer.py:218
      if (a.fix_params && G > 3) {                                               // trainer.py:219-220
        if (tid == G + 3) t = 1.0;
        if (tid == 3) t = 0.8;
      }
      a.theta_out[bidx * P + tid] = t;
    }
  }
  if (tid == 0 && a.info) {
    if (a.first_step == 0 || eval_only) a.info[bidx] = fail;
    else if (fail) a.info[bidx] = fail;
  }
  if (tid == 0 && a.best_key && !eval_only && a.hist && a.steps > 0) {
    const double v = a.hist[bidx * a.ld_hist + a.first_step + a.steps - 1];
    if (v == v) atomicMin(a.best_key, lfm_loss_key(v));
  }
}

static size_t batched_smem_bytes(int N, int G, int MU, bool het) {
  const size_t P = 3 * (size_t)G + 2;
  const size_t ld = (size_t)(MU | 1);
  size_t d = (size_t)MU * ld + (het ? 9 : 7) * (size_t)N + 5 * P + (size_t)G + 16;
  return d * 8 + (size_t)N * sizeof(LfmPoint) + 2 * (size_t)N * sizeof(int);
}

static int batched_launch(cudaStream_t st, const BatchedArgs& a, int time_grid) {
  if (a.B <= 0 || a.N <= 0 || a.G <= 0 || !a.X || !a.y || !a.u_io) return LFM_ERR_INVALID;
  if (a.N % a.G) return LFM_ERR_INVALID;
  if (a.y_stride != 0 && a.y_stride < a.N) return LFM_ERR_INVALID;
  if (a.var && a.var_stride != 0 && a.var_stride < a.N) return LFM_ERR_INVALID;
  if (a.N > 128 || a.B > 0x7fffffff) return LFM_ERR_UNSUPPORTED;
  BatchedArgs b = a;
  if (b.max_unique <= 0 || b.max_unique > b.N) b.max_unique = b.N;
  if (time_grid > 0) {  // one warp per LFM with shared-memory time-grid tables, when it fits
    const int st2 = lfm_batched_warp_launch(st, b, time_grid);
    if (st2 != LFM_ERR_UNSUPPORTED) return st2;
  }
  b.queue = nullptr;   // the CTA-per-LFM kernel has no queue mode: plain launch over all the steps it was given
  const bool het = b.var != nullptr;
  const size_t smem = batched_smem_bytes(b.N, b.G, b.max_unique, het);
  if (smem > 227 * 1024) return LFM_ERR_UNSUPPORTED;
  const bool small = b.max_unique <= 64 && b.N <= 128 && 3 * b.G + 2 <= 128;
  if (!small && 3 * b.G + 2 > 256) return LFM_ERR_UNSUPPORTED;
  static LfmSmemConfig conf128, conf256, conf128h, conf256h;
  if (het) {
    if (small) {
      LFM_CUDA_OK(lfm_ensure_smem(lfm_batched_kernel<128, true>, conf128h, smem));
      lfm_batched_kernel<128, true><<<(unsigned)b.B, 128, smem, st>>>(b);
    } else {
      LFM_CUDA_OK(lfm_ensure_smem(lfm_batched_kernel<256, true>, conf256h, smem));
      lfm_batched_kernel<256, true><<<(unsigned)b.B, 256, smem, st>>>(b);
    }
  } else if (small) {
    LFM_CUDA_OK(lfm_ensure_smem(lfm_batched_kernel<128, false>, conf128, smem));
    lfm_batched_kernel<128, false><<<(unsigned)b.B, 128, smem, st>>>(b);
  } else {
    LFM_CUDA_OK(lfm_ensure_smem(lfm_batched_kernel<256, false>, conf256, smem));
    lfm_batched_kernel<256, false><<<(unsigned)b.B, 256, smem, st>>>(b);
  }
  LFM_LAUNCHED(1);
  LFM_CUDA_OK(cudaGetLastError());
  return LFM_OK;
}

extern "C" int lfm_batched_nlml_grad_unc_het(lfm_stream_t stream, int64_t B, int64_t N, int G, const double* X,
                                             const double* y, int64_t y_stride, const double* variances,
                                             int64_t var_stride, const double* theta_unc, double jitter,
                                             int unique_rows_hint, int time_grid_hint, double* out_val,
                                             double* out_grad, int* info) {
  if (!out_val || !out_grad) return LFM_ERR_INVALID;
  BatchedArgs a;
  memset(&a, 0, sizeof(a));
  a.B = B; a.N = (int)N; a.G = G; a.X = X; a.y = y; a.y_stride = y_stride;
  a.u_io = const_cast<double*>(theta_unc);  // read-only in eval mode
  a.jitter = jitter; a.steps = 1; a.total_steps = 1; a.steps_per_epoch = 1;
  a.eval_val = out_val; a.eval_grad = out_grad; a.info = info; a.max_unique = unique_rows_hint;
  a.var = variances; a.var_stride = variances ? var_stride : 0;
  if (N > 128) return LFM_ERR_UNSUPPORTED;
  return batched_launch((cudaStream_t)stream, a, time_grid_hint);
}
extern "C" int lfm_batched_nlml_grad_unc_multi(lfm_stream_t stream, int64_t B, int64_t N, int G, const double* X,
                                               const double* y, int64_t y_stride, const double* theta_unc, double jitter,
                                               int unique_rows_hint, int time_grid_hint, double* out_val,
                                               double* out_grad, int* info) {
  return lfm_batched_nlml_grad_unc_het(stream, B, N, G, X, y, y_stride, nullptr, 0, theta_unc, jitter, unique_rows_hint,
                                       time_grid_hint, out_val, out_grad, info);
}
extern "C" int lfm_batched_nlml_grad_unc_tg(lfm_stream_t stream, int64_t B, int64_t N, int G, const double* X,
                                            const double* y, const double* theta_unc, double jitter,
                                            int unique_rows_hint, int time_grid_hint, double* out_val,
                                            double* out_grad, int* info) {
  return lfm_batched_nlml_grad_unc_multi(stream, B, N, G, X, y, 0, theta_unc, jitter, unique_rows_hint, time_grid_hint,
                                         out_val, out_grad, info);
}
extern "C" int lfm_batched_nlml_grad_unc(lfm_stream_t stream, int64_t B, int64_t N, int G, const double* X,
                                         const double* y, const double* theta_unc, double jitter,
                                         int unique_rows_hint, double* out_val, double* out_grad, int* info) {
  return lfm_batched_nlml_grad_unc_tg(stream, B, N, G, X, y, theta_unc, jitter, unique_rows_hint, 0, out_val, out_grad,
                                      info);
}

extern "C" int lfm_batched_fit_tg(lfm_stream_t stream, int64_t B, int64_t N, int G, const double* X, const double* y,
                                  double* theta_unc_io, double* adam_state, double jitter, double lr, double b1,
                                  double b2, double eps, int first_step, int steps, int total_steps, int fix_params,
                                  int steps_per_epoch, int unique_rows_hint, int time_grid_hint, double* out_hist,
                                  int64_t ld_hist, double* out_theta, int* info, long long* best_key,
                                  void* structure_cache) {
  return lfm_batched_fit_multi(stream, B, N, G, X, y, 0, theta_unc_io, adam_state, jitter, lr, b1, b2, eps, first_step,
                               steps, total_steps, fix_params, steps_per_epoch, unique_rows_hint, time_grid_hint,
                               out_hist, ld_hist, out_theta, info, best_key, structure_cache);
}
extern "C" int lfm_batched_fit_multi(lfm_stream_t stream, int64_t B, int64_t N, int G, const double* X, const double* y,
                                     int64_t y_stride, double* theta_unc_io, double* adam_state, double jitter,
                                     double lr, double b1, double b2, double eps, int first_step, int steps,
                                     int total_steps, int fix_params, int steps_per_epoch, int unique_rows_hint,
                                     int time_grid_hint, double* out_hist, int64_t ld_hist, double* out_theta,
                                     int* info, long long* best_key, void* structure_cache) {
  return lfm_batched_fit_trace(stream, B, N, G, X, y, y_stride, theta_unc_io, adam_state, jitter, lr, b1, b2, eps,
                               first_step, steps, total_steps, fix_params, steps_per_epoch, unique_rows_hint,
                               time_grid_hint, out_hist, ld_hist, out_theta, info, best_key, nullptr, structure_cache);
}
// Whole fit in ONE launch with persistent workers and a device-side task queue (batched_warp.cu): see the header.
extern "C" size_t lfm_batched_queue_bytes(int64_t B, int total_steps, int chunk_steps) {
  if (B <= 0 || total_steps <= 0 || chunk_steps <= 0) return 0;
  const int64_t nchunks = (total_steps + chunk_steps - 1) / chunk_steps;
  if (B * nchunks > 0x7fffffff) return 0;
  return (size_t)(4 + B + B * nchunks) * sizeof(int);
}
// One body for the chunked (queue_ws NULL) and the persistent-queue fits, with or without variances (see the header).
extern "C" int lfm_batched_fit_het(lfm_stream_t stream, int64_t B, int64_t N, int G, const double* X, const double* y,
                                   int64_t y_stride, const double* variances, int64_t var_stride, double* theta_unc_io,
                                   double* adam_state, double jitter, double lr, double b1, double b2, double eps,
                                   int first_step, int steps, int total_steps, int fix_params, int steps_per_epoch,
                                   int unique_rows_hint, int time_grid_hint, double* out_hist, int64_t ld_hist,
                                   double* out_theta, int* info, long long* best_key, long long* step_keys,
                                   void* structure_cache, int chunk_steps, void* queue_ws, size_t queue_bytes) {
  if (steps < 0 || first_step < 0 || steps_per_epoch <= 0) return LFM_ERR_INVALID;
  if (first_step > 0 && !adam_state) return LFM_ERR_INVALID;
  if (queue_ws && (first_step != 0 || steps != total_steps)) return LFM_ERR_INVALID;   // the queue runs the whole fit
  if (N > 128) return LFM_ERR_UNSUPPORTED;
  if (queue_ws && (chunk_steps <= 0 || queue_bytes < lfm_batched_queue_bytes(B, total_steps, chunk_steps) ||
                   lfm_batched_queue_bytes(B, total_steps, chunk_steps) == 0 || !adam_state))
    return queue_bytes ? LFM_ERR_WORKSPACE : LFM_ERR_INVALID;
  BatchedArgs a;
  memset(&a, 0, sizeof(a));
  a.B = B; a.N = (int)N; a.G = G; a.X = X; a.y = y; a.y_stride = y_stride; a.u_io = theta_unc_io; a.adam = adam_state;
  a.jitter = jitter; a.lr = lr; a.b1 = b1; a.b2 = b2; a.eps = eps;
  a.first_step = first_step; a.steps = steps; a.total_steps = total_steps; a.fix_params = fix_params;
  a.steps_per_epoch = steps_per_epoch; a.hist = out_hist; a.ld_hist = ld_hist; a.theta_out = out_theta;
  a.info = info; a.max_unique = unique_rows_hint; a.best_key = best_key; a.step_keys = step_keys;
  a.struct_cache = structure_cache;
  if (queue_ws) { a.queue = (int*)queue_ws; a.queue_chunk = chunk_steps; }
  a.var = variances; a.var_stride = variances ? var_stride : 0;
  return batched_launch((cudaStream_t)stream, a, time_grid_hint);
}
extern "C" int lfm_batched_fit_queue(lfm_stream_t stream, int64_t B, int64_t N, int G, const double* X, const double* y,
                                     int64_t y_stride, double* theta_unc_io, double* adam_state, double jitter,
                                     double lr, double b1, double b2, double eps, int total_steps, int fix_params,
                                     int steps_per_epoch, int unique_rows_hint, int time_grid_hint, double* out_hist,
                                     int64_t ld_hist, double* out_theta, int* info, long long* best_key,
                                     long long* step_keys, void* structure_cache, int chunk_steps, void* queue_ws,
                                     size_t queue_bytes) {
  if (total_steps < 0) return LFM_ERR_INVALID;
  return lfm_batched_fit_het(stream, B, N, G, X, y, y_stride, nullptr, 0, theta_unc_io, adam_state, jitter, lr, b1, b2,
                             eps, 0, total_steps, total_steps, fix_params, steps_per_epoch, unique_rows_hint,
                             time_grid_hint, out_hist, ld_hist, out_theta, info, best_key, step_keys, structure_cache,
                             chunk_steps, queue_ws, queue_bytes);
}
extern "C" int lfm_batched_fit_trace(lfm_stream_t stream, int64_t B, int64_t N, int G, const double* X, const double* y,
                                     int64_t y_stride, double* theta_unc_io, double* adam_state, double jitter,
                                     double lr, double b1, double b2, double eps, int first_step, int steps,
                                     int total_steps, int fix_params, int steps_per_epoch, int unique_rows_hint,
                                     int time_grid_hint, double* out_hist, int64_t ld_hist, double* out_theta,
                                     int* info, long long* best_key, long long* step_keys, void* structure_cache) {
  return lfm_batched_fit_het(stream, B, N, G, X, y, y_stride, nullptr, 0, theta_unc_io, adam_state, jitter, lr, b1, b2,
                             eps, first_step, steps, total_steps, fix_params, steps_per_epoch, unique_rows_hint,
                             time_grid_hint, out_hist, ld_hist, out_theta, info, best_key, step_keys, structure_cache, 0,
                             nullptr, 0);
}
// Debug: one launch of `steps` >= 2 steps with clock64 stamps at the phase boundaries of the SECOND step of LFM 0
// (warp-per-LFM kernel only): A B C D E[load] E[routine] E[W^T W] E[Schur] E[store] F I J K end.
extern "C" int lfm_debug_batched_stamps(lfm_stream_t stream, int64_t B, int64_t N, int G, const double* X,
                                        const double* y, double* theta_unc_io, double* adam_state, double jitter,
                                        int steps, int unique_rows_hint, int time_grid_hint, double* out_hist,
                                        int* info, long long* stamps) {
  BatchedArgs a;
  memset(&a, 0, sizeof(a));
  a.B = B; a.N = (int)N; a.G = G; a.X = X; a.y = y; a.u_io = theta_unc_io; a.adam = adam_state;
  a.jitter = jitter; a.lr = 0.01; a.b1 = 0.9; a.b2 = 0.999; a.eps = 1e-8;
  a.first_step = 0; a.steps = steps; a.total_steps = steps; a.fix_params = 1; a.steps_per_epoch = 1000;
  a.hist = out_hist; a.ld_hist = steps; a.info = info; a.max_unique = unique_rows_hint; a.stamps = stamps;
  return batched_launch((cudaStream_t)stream, a, time_grid_hint);
}

extern "C" int lfm_batched_team_size(int64_t B, int64_t N, int G, int unique_rows_hint, int time_grid_hint) {
  if (B <= 0 || N <= 0 || N > 128 || G <= 0) return 0;
  int MU = unique_rows_hint;
  if (MU <= 0 || MU > N) MU = (int)N;
  return lfm_batched_warp_team(B, (int)N, G, MU, time_grid_hint);
}

// ---- winner of a shard: arg-min over the finite losses of one history column, packed with its theta -------------
__global__ void __launch_bounds__(256) lfm_batched_best_kernel(int64_t B, int P, const double* __restrict__ hist,
                                                               int64_t ld_hist, int64_t col,
                                                               const double* __restrict__ theta, double id0,
                                                               double* __restrict__ out) {
  __shared__ double sv[8];
  __shared__ long long si[8];
  const double inf = __longlong_as_double(0x7ff0000000000000LL);
  double best = inf;
  long long arg = -1;
  for (int64_t b = threadIdx.x; b < B; b += blockDim.x) {   // ascending b per thread: strict < keeps the smallest index
    const double v = hist[b * ld_hist + col];
    if (v - v == 0.0 && v < best) { best = v; arg = b; }
  }
  auto better = [](double v, long long i, double w, long long j) { return i >= 0 && (j < 0 || v < w || (v == w && i < j)); };
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const double v = __shfl_xor_sync(0xffffffffu, best, o);
    const long long i = __shfl_xor_sync(0xffffffffu, arg, o);
    if (better(v, i, best, arg)) { best = v; arg = i; }
  }
  if ((threadIdx.x & 31) == 0) { sv[threadIdx.x >> 5] = best; si[threadIdx.x >> 5] = arg; }
  __syncthreads();
  best = sv[0]; arg = si[0];
  for (int w = 1; w < 8; ++w)
    if (better(sv[w], si[w], best, arg)) { best = sv[w]; arg = si[w]; }
  if (threadIdx.x == 0) { out[0] = arg >= 0 ? best : inf; out[1] = arg >= 0 ? id0 + (double)arg : -1.0; }
  for (int p = threadIdx.x; p < P; p += blockDim.x) out[2 + p] = arg >= 0 ? theta[arg * P + p] : inf;
}
extern "C" int lfm_batched_best(lfm_stream_t stream, int64_t B, int P, const double* hist, int64_t ld_hist, int64_t col,
                                const double* theta, double id0, double* out_packed) {
  if (B < 0 || P <= 0 || !out_packed || col < 0 || col >= ld_hist) return LFM_ERR_INVALID;
  if (B > 0 && (!hist || !theta)) return LFM_ERR_INVALID;
  lfm_batched_best_kernel<<<1, 256, 0, (cudaStream_t)stream>>>(B, P, hist, ld_hist, col, theta, id0, out_packed);
  LFM_LAUNCHED(1);
  LFM_CUDA_OK(cudaGetLastError());
  return LFM_OK;
}

extern "C" size_t lfm_batched_structure_bytes(int64_t N, int G, int unique_rows_hint, int time_grid_hint) {
  if (N <= 0 || N > 128 || G <= 0) return 0;
  int MU = unique_rows_hint;
  if (MU <= 0 || MU > N) MU = (int)N;
  return lfm_batched_warp_structure_bytes((int)N, G, MU, time_grid_hint);
}

extern "C" int lfm_batched_fit(lfm_stream_t stream, int64_t B, int64_t N, int G, const double* X, const double* y,
                               double* theta_unc_io, double* adam_state, double jitter, double lr, double b1,
                               double b2, double eps, int first_step, int steps, int total_steps, int fix_params,
                               int steps_per_epoch, int unique_rows_hint, double* out_hist, int64_t ld_hist,
                               double* out_theta, int* info) {
  return lfm_batched_fit_tg(stream, B, N, G, X, y, theta_unc_io, adam_state, jitter, lr, b1, b2, eps, first_step, steps,
                            total_steps, fix_params, steps_per_epoch, unique_rows_hint, 0, out_hist, ld_hist, out_theta,
                            info, nullptr, nullptr);
}

// Number of rows of the duplicate-row-compressed problem for a HOST copy of X: the `unique_rows_hint` that
// lets the batched kernels size their shared memory.  Mirrors the kernels' own rule: the distinct
// (time, gene, flag) rows when every distinct row occurs the same number of times R > 1 (replicates on a
// shared design), otherwise N (no compression: e.g. one replicate with a missing measurement).
extern "C" int lfm_count_unique_rows(int64_t N, const double* X_host) {
  if (N <= 0 || !X_host) return 0;
  std::vector<int64_t> rep((size_t)N), cnt((size_t)N, 0);
  int U = 0;
  for (int64_t i = 0; i < N; ++i) {
    rep[i] = i;
    for (int64_t j = 0; j < i; ++j)
      if (X_host[3 * j] == X_host[3 * i] && X_host[3 * j + 1] == X_host[3 * i + 1] && X_host[3 * j + 2] == X_host[3 * i + 2]) {
        rep[i] = rep[j];
        break;
      }
    if (rep[i] == i) ++U;
    ++cnt[rep[i]];
  }
  const int64_t R = cnt[0];
  for (int64_t i = 0; i < N; ++i)
    if (cnt[rep[i]] != R) return (int)N;
  return R > 1 ? U : (int)N;
}

// Single-input-motif (SIM) covariance arithmetic, fp64, device side.
//
// Restates src/model.py:197-369 of the reference (k_xx :197-235, k_xf :237-282, k_ff :284-312,
// h :315-365, gamma :367-369) in a factored form: everything that depends on one point only is
// computed once per point (LfmPoint), the per-pair work is 2 exp + 4 erf for a k_xx entry.
#pragma once
#include "lfm_common.cuh"

// Per-point derived quantities for a gene-expression row (t, gene j):
struct LfmPoint {
  double t;     // time
  double d;     // D_j
  double s;     // S_j
  double gam;   // gamma_j = D_j l / 2                         (model.py:367-369)
  double eg2;   // exp(gamma_j^2)
  double erfg;  // erf(gamma_j)
  double e;     // exp(-D_j t)
  double q;     // erf(t/l - gamma_j) + erf(gamma_j)           ("second_erf_terms", model.py:355-357; lfm_erfsum)
  double g3;    // 2/sqrt(pi) exp(-(t/l - gamma_j)^2)           (gradient only)
  double g4;    // 2/sqrt(pi) exp(-gamma_j^2)                   (gradient only)
  int gene;     // resolved gene index
  int flag;     // 1 gene expression, 0 latent force
  int ti;       // index of t among the distinct times of X (time-grid tables only; else 0)
};

// jnp integer indexing semantics for the gene column (model.py:223-224): negative wraps, then clamp.
__device__ __forceinline__ int lfm_resolve_gene(double gcol, int G) {
  int g = (int)gcol;
  if (g < 0) g += G;
  g = g < 0 ? 0 : g;
  g = g >= G ? G - 1 : g;
  return g;
}

// erf(a) + erf(b) without catastrophic cancellation.  In h and k_xf the first sum R1 multiplies
// exp(-D dt) with dt < 0 (up to e^13 in the p53 regime) exactly when erf(a) ~ -1 and erf(b) ~ +1
// (SURVEY Q7): the literal sum then carries ~1e-16 * e^(D|dt|) absolute noise.  The second sum of h,
// R2 = erf(t/l - gamma) + erf(gamma), cancels for t/l < gamma and is multiplied by exp(gamma^2): the
// literal form loses ~1e-16 * exp(gamma^2) (5e-11 of the covariance scale at gamma = 4.4, 4e-2 at 7).
// For opposite-sign arguments that are both beyond 0.5 the identical quantity erfc(-n) - erfc(p) is
// used instead.  The oracle (oracle/lfm_oracle.py:erfsum) uses the same rule with the same threshold.
__device__ __forceinline__ double lfm_erfsum(double a, double b) {
  if (a * b < 0.0 && fmin(fabs(a), fabs(b)) > 0.5) {
    const double p = fmax(a, b), n = fmin(a, b);
    return erfc(-n) - erfc(p);
  }
  return erf(a) + erf(b);
}

__device__ __forceinline__ LfmPoint lfm_make_point(const double* __restrict__ row3, int G,
                                                   const double* __restrict__ d,
                                                   const double* __restrict__ s, double l, bool grad) {
  LfmPoint p;
  p.t = row3[0];
  p.gene = lfm_resolve_gene(row3[1], G);
  p.flag = ((int)row3[2]) != 0;
  p.ti = 0;
  p.d = d[p.gene];
  p.s = s[p.gene];
  p.gam = p.d * l * 0.5;
  p.eg2 = exp(p.gam * p.gam);
  p.erfg = erf(p.gam);
  p.e = exp(-p.d * p.t);
  const double x3 = p.t / l - p.gam;
  p.q = lfm_erfsum(x3, p.gam);
  if (grad) {
    p.g3 = LFM_TWO_OVER_SQRT_PI * exp(-x3 * x3);
    p.g4 = LFM_TWO_OVER_SQRT_PI * exp(-p.gam * p.gam);
  } else {
    p.g3 = 0.0;
    p.g4 = 0.0;
  }
  return p;
}

// H(a,b,u,v) = h(j=a, k=b, t1=u, t2=v) of model.py:315-365, with "b" the gene whose gamma enters.
// pa is the point (u, gene a), pb the point (v, gene b).
//   H = E0 (A1 R1 - A2 R2),  E0 = exp(gam_b^2)/(d_a+d_b), A1 = exp(-d_b (v-u)),
//   R1 = erf((v-u)/l - gam_b) + erf(u/l + gam_b), A2 = exp(-(d_b v + d_a u)) = e_a e_b, R2 = q_b.
// The transcendental factors that depend on (gene b, u, v) only -- A1, A1 R1, g1 -- and on (gene b, u) only
// -- g2 -- enter through lfm_h_core, so that they can come either from a direct evaluation (lfm_h) or
// from the distinct-time tables of a gridded data set (LfmGrid, grid.cu): G T^2 evaluations instead of N^2.
struct LfmPairTerms {
  double inv;    // 1 / (d_a + d_b)
  double A1;     // exp(-d_b (v - u))
  double A1R1;   // A1 * [erf((v-u)/l - gam_b) + erf(u/l + gam_b)]
  double g1;     // 2/sqrt(pi) exp(-((v-u)/l - gam_b)^2)    (gradient only)
  double g2;     // 2/sqrt(pi) exp(-(u/l + gam_b)^2)        (gradient only)
};
template <bool GRAD>
__device__ __forceinline__ LfmPairTerms lfm_pair_terms(double ta, double tb, double d_b, double gam_b, double inv_l) {
  LfmPairTerms r;
  const double delta = tb - ta;
  r.A1 = exp(-d_b * delta);
  const double x1 = delta * inv_l - gam_b;
  const double x2 = ta * inv_l + gam_b;
  r.A1R1 = __dmul_rn(r.A1, lfm_erfsum(x1, x2));
  if (GRAD) {
    r.g1 = __dmul_rn(LFM_TWO_OVER_SQRT_PI, exp(-x1 * x1));
    r.g2 = __dmul_rn(LFM_TWO_OVER_SQRT_PI, exp(-x2 * x2));
  } else {
    r.g1 = 0.0; r.g2 = 0.0;
  }
  r.inv = 0.0;
  return r;
}
template <bool GRAD>
__device__ __forceinline__ void lfm_h_core(const LfmPoint& pa, const LfmPoint& pb, double l, double inv_l,
                                           const LfmPairTerms& pt, double& H, double& dH_da, double& dH_db,
                                           double& dH_dl) {
  const double delta = pb.t - pa.t;
  const double inv = pt.inv;
  const double E0 = pb.eg2 * inv;
  const double A1 = pt.A1;
  const double A2 = pa.e * pb.e;
  const double A1R1 = pt.A1R1;
  const double A2R2 = __dmul_rn(A2, pb.q);
  H = E0 * (A1R1 - A2R2);
  if (GRAD) {
    const double g1 = pt.g1, g2 = pt.g2;
    const double g3 = pb.g3, g4 = pb.g4;
    const double hl = 0.5 * l;
    const double hd = 0.5 * pb.d;
    const double il2 = inv_l * inv_l;
    dH_da = -H * inv + E0 * pa.t * A2R2;
    dH_db = H * (pb.gam * l - inv) +
            E0 * (-delta * A1R1 + A1 * hl * (g2 - g1) + pb.t * A2R2 - A2 * hl * (g4 - g3));
    dH_dl = H * pb.gam * pb.d + E0 * (A1 * (g1 * (-delta * il2 - hd) + g2 * (-pa.t * il2 + hd)) -
                                      A2 * (g3 * (-pb.t * il2 - hd) + g4 * hd));
  }
}
template <bool GRAD>
__device__ __forceinline__ void lfm_h(const LfmPoint& pa, const LfmPoint& pb, double l, double inv_l,
                                      double& H, double& dH_da, double& dH_db, double& dH_dl) {
  LfmPairTerms pt = lfm_pair_terms<GRAD>(pa.t, pb.t, pb.d, pb.gam, inv_l);
  pt.inv = 1.0 / (pa.d + pb.d);
  lfm_h_core<GRAD>(pa, pb, l, inv_l, pt, H, dH_da, dH_db, dH_dl);
}

// ---- distinct-time tables ("time grid") -------------------------------------------------------------------
// When the rows of X share a small set of distinct times (the reference's layout: every gene observed on the
// same time grid, dataset.py:380-391), the pair terms above depend on (gene b, time index of a, time index
// of b) only.  grid.cu finds the distinct times on the device, tabulates the terms once per evaluation
// (G T^2 entries) and the tile kernels read them instead of evaluating exp / erf per matrix entry.
// Layouts: X[b][ia][ib] with ib fastest; the *t arrays are the (ia, ib)-transposed copies so that both
// h(col, row) and h(row, col) read consecutive addresses along a tile row.
struct LfmGrid {
  const int* tidx;     // [N] distinct-time index of every row of X
  const int* count;    // device scalar: number of distinct times found; tables are valid iff *count <= Tu
  int Tu;              // leading dimension of the tables (host-side upper bound on *count); 0: no tables
  int G;
  const double* A1R1;  const double* A1R1t;
  // gradient only: everything of dH/dd_b and dH/dl that depends on (gene b, u, v) alone, folded into ONE number each
  // when the tables are built (grid.cu), so that the contraction kernel does a dozen flops per h-term instead of ~45:
  //   Qd = (gam_b l - delta) A1R1 + A1 (l/2) (g2 - g1)
  //   Rl = gam_b d_b A1R1 + A1 (g1 (-delta / l^2 - d_b/2) + g2 (-u / l^2 + d_b/2))
  const double* Qd;    const double* Qdt;
  const double* Rl;    const double* Rlt;
  const double* inv;   // [G][G] 1 / (d_a + d_b)
};
// What a point contributes to the h-terms in which it is the "b" point (gradient only; staged beside LfmPoint):
//   phi = e q,  rho = (t - gam l) phi - e (l/2) (g4 - g3),  sig = -gam d phi - e (g3 (-t/l^2 - d/2) + g4 d/2),  ue = t e
struct LfmPointGrad { double phi, rho, sig, ue; };
__device__ __forceinline__ LfmPointGrad lfm_point_grad(const LfmPoint& p, double l, double inv_l) {
  LfmPointGrad x;
  const double hl = 0.5 * l, hd = 0.5 * p.d, il2 = inv_l * inv_l;
  x.phi = __dmul_rn(p.e, p.q);
  x.rho = (p.t - p.gam * l) * x.phi - p.e * hl * (p.g4 - p.g3);
  x.sig = -p.gam * p.d * x.phi - p.e * (p.g3 * (-p.t * il2 - hd) + p.g4 * hd);
  x.ue = p.t * p.e;
  return x;
}
// h(pa, pb) from the tables; `tr` selects the transposed copies (used for h(col, row), where the column
// index runs along ia).
__device__ __forceinline__ double lfm_h_tab(const LfmGrid& g, const LfmPoint& pa, const LfmPoint& pb, bool tr) {
  const size_t base = (size_t)pb.gene * g.Tu * g.Tu;
  const size_t off = tr ? base + (size_t)pb.ti * g.Tu + pa.ti : base + (size_t)pa.ti * g.Tu + pb.ti;
  const double A1R1 = (tr ? g.A1R1t : g.A1R1)[off];
  const double E0 = pb.eg2 * g.inv[(size_t)pa.gene * g.G + pb.gene];
  const double A2R2 = __dmul_rn(pa.e * pb.e, pb.q);
  return E0 * (A1R1 - A2R2);
}
// H and its partials from the tables, regrouped (see LfmGrid): with E0 = exp(gam_b^2) / (d_a + d_b)
//   H = E0 (A1R1 - e_a phi_b),  dH/dd_a = E0 ue_a phi_b - H inv,  dH/dd_b = E0 (Qd + e_a rho_b) - H inv,  dH/dl = E0 (Rl + e_a sig_b)
// -- the same quantities as lfm_h_core<true> (the direct path), associated differently (agreement ~1e-15 relative).
__device__ __forceinline__ void lfm_h_tab_grad(const LfmGrid& g, const LfmPoint& pa, const LfmPointGrad& xa, const LfmPoint& pb,
                                               const LfmPointGrad& xb, bool tr, double& H, double& dH_da, double& dH_db,
                                               double& dH_dl) {
  const size_t base = (size_t)pb.gene * g.Tu * g.Tu;
  const size_t off = tr ? base + (size_t)pb.ti * g.Tu + pa.ti : base + (size_t)pa.ti * g.Tu + pb.ti;
  const double T1 = (tr ? g.A1R1t : g.A1R1)[off];
  const double Q = (tr ? g.Qdt : g.Qd)[off];
  const double R = (tr ? g.Rlt : g.Rl)[off];
  const double inv = g.inv[(size_t)pa.gene * g.G + pb.gene];
  const double E0 = pb.eg2 * inv;
  H = E0 * (T1 - pa.e * xb.phi);
  const double Hinv = H * inv;
  dH_da = E0 * (xa.ue * xb.phi) - Hinv;
  dH_db = E0 * (Q + pa.e * xb.rho) - Hinv;
  dH_dl = E0 * (R + pa.e * xb.sig);
}
__device__ __forceinline__ double lfm_kxx_tab(const LfmGrid& g, const LfmPoint& pi, const LfmPoint& pj, double l,
                                              double inv_l) {
  const double H1 = lfm_h_tab(g, pj, pi, true);
  const double H2 = lfm_h_tab(g, pi, pj, false);
  return pi.s * pj.s * (LFM_SQRT_PI * 0.5 * l) * (H1 + H2);
}
__device__ __forceinline__ void lfm_kxx_grad_tab(const LfmGrid& g, const LfmPoint& pi, const LfmPointGrad& xi, const LfmPoint& pj,
                                                 const LfmPointGrad& xj, double l, double inv_l, double& k, double& dk_drow,
                                                 double& dk_dcol, double& dk_dl) {
  double H1, dH1_da, dH1_db, dH1_dl, H2, dH2_da, dH2_db, dH2_dl;
  lfm_h_tab_grad(g, pj, xj, pi, xi, true, H1, dH1_da, dH1_db, dH1_dl);
  lfm_h_tab_grad(g, pi, xi, pj, xj, false, H2, dH2_da, dH2_db, dH2_dl);
  const double mult = pi.s * pj.s * (LFM_SQRT_PI * 0.5 * l);
  k = mult * (H1 + H2);
  dk_drow = mult * (dH1_db + dH2_da);
  dk_dcol = mult * (dH1_da + dH2_db);
  dk_dl = mult * (dH1_dl + dH2_dl) + k * inv_l;
}

// k_xx between gene point pi = (t, j) and gene point pj = (t', k)  (model.py:197-235):
//   S_j S_k (sqrt(pi) l / 2) [ h(k, j, t', t) + h(j, k, t, t') ]
// H1 + H2 is rounded as written (__dadd_rn): contracted into fma(E0, ., H1) it would depend on which point is the row,
// and k_xx(X*, X*) -- the prior covariance of the gene posterior -- would not be exactly symmetric.
__device__ __forceinline__ double lfm_kxx(const LfmPoint& pi, const LfmPoint& pj, double l, double inv_l) {
  double H1, H2, u0, u1, u2;
  lfm_h<false>(pj, pi, l, inv_l, H1, u0, u1, u2);  // h(k, j, t', t): a = col gene, b = row gene
  lfm_h<false>(pi, pj, l, inv_l, H2, u0, u1, u2);  // h(j, k, t, t'): a = row gene, b = col gene
  return pi.s * pj.s * (LFM_SQRT_PI * 0.5 * l) * __dadd_rn(H1, H2);
}

// k_xx and the partials of it with respect to D of the ROW gene, D of the COLUMN gene and l.
// (dk/dS_row = k / S_row, dk/dS_col = k / S_col are formed by the caller.)
__device__ __forceinline__ void lfm_kxx_grad(const LfmPoint& pi, const LfmPoint& pj, double l, double inv_l,
                                             double& k, double& dk_drow, double& dk_dcol, double& dk_dl) {
  double H1, dH1_da, dH1_db, dH1_dl, H2, dH2_da, dH2_db, dH2_dl;
  lfm_h<true>(pj, pi, l, inv_l, H1, dH1_da, dH1_db, dH1_dl);
  lfm_h<true>(pi, pj, l, inv_l, H2, dH2_da, dH2_db, dH2_dl);
  const double mult = pi.s * pj.s * (LFM_SQRT_PI * 0.5 * l);
  k = mult * (H1 + H2);
  dk_drow = mult * (dH1_db + dH2_da);
  dk_dcol = mult * (dH1_da + dH2_db);
  dk_dl = mult * (dH1_dl + dH2_dl) + k * inv_l;
}

// k_xf between gene point pg = (t_gene, j) and a latent time (model.py:237-282).
__device__ __forceinline__ double lfm_kxf(const LfmPoint& pg, double t_latent, double l, double inv_l) {
  const double t_dist = pg.t - t_latent;
  return (0.5 * l * LFM_SQRT_PI * pg.s) * pg.eg2 * exp(-pg.d * t_dist) *
         lfm_erfsum(t_dist * inv_l - pg.gam, t_latent * inv_l + pg.gam);
}

// k_ff, latent RBF with the reference's 2*l denominator (model.py:304-312; SURVEY Q1).
__device__ __forceinline__ double lfm_kff(double t, double tp, double l) {
  const double dt = t - tp;
  return exp(-(dt * dt) / (2.0 * l));
}

// ---- host launchers shared between translation units (gram.cu / grid.cu) -------------------------------------
// Sigma (lower tiles, padded to Npad) = k_xx(X, X) + diag(diag_vec) + (diag_const [+ sigma^2]) I
int lfm_launch_sigma_lower(cudaStream_t st, int64_t N, int64_t Npad, const double* X, int G, const double* theta,
                           const double* diag_vec, double diag_const, int add_sigma2, double* out, int64_t ld,
                           const LfmGrid* tg = nullptr, int64_t col_begin = 0, int64_t col_end = -1);
size_t lfm_grad_scratch_doubles(int64_t N);
int lfm_launch_grad_contract(cudaStream_t st, int64_t N, const double* X, int G, const double* theta,
                             const double* Sinv, int64_t ld, const double* alpha, double* scratch, double* grad,
                             const LfmGrid* tg = nullptr);
int lfm_launch_cross_cov(cudaStream_t st, int64_t N, int64_t M, const double* X, const double* Y, int G,
                         const double* theta, double* out, int64_t ld);
size_t lfm_grid_ws_doubles(int64_t N, int G, int64_t Tu);
int lfm_grid_build(cudaStream_t st, int64_t N, int G, const double* X, const double* theta, int64_t Tu, bool grad,
                   void* ws, LfmGrid* grid);
// Effective table bound for a caller-supplied `time_grid`: 0 (direct evaluation) unless the tables are at
// least 8x smaller than the matrix and fit 2 GB.
static inline int64_t lfm_grid_effective(int64_t N, int G, int64_t time_grid) {
  if (time_grid <= 0 || time_grid > 46000) return 0;
  const double tab = (double)G * (double)time_grid * (double)time_grid;
  if (tab * 8.0 > (double)N * (double)N) return 0;
  if (tab * 6.0 * 8.0 > 2.0e9) return 0;
  return time_grid;
}

// ExactLFM.kernel (model.py:152-195).  Only the branch the 0/1 switches select is evaluated;
// identical to the reference's blend whenever the discarded branches are finite (SURVEY Q7).
__device__ __forceinline__ double lfm_kernel(const LfmPoint& pi, const LfmPoint& pj, double l, double inv_l) {
  if (pi.flag & pj.flag) return lfm_kxx(pi, pj, l, inv_l);
  if (pi.flag) return lfm_kxf(pi, pj.t, l, inv_l);
  if (pj.flag) return lfm_kxf(pj, pi.t, l, inv_l);
  return lfm_kff(pi.t, pj.t, l);
}

// ---- bijectors (tfp Softplus / Sigmoid(0.5, 3.5); model.py:66,79,86,93,111) -----------------
#define LFM_L_LOW 0.5
#define LFM_L_HIGH 3.5
__device__ __forceinline__ double lfm_softplus(double x) { return fmax(x, 0.0) + log1p(exp(-fabs(x))); }
__device__ __forceinline__ double lfm_softplus_inv(double y) { return y + log(-expm1(-y)); }
__device__ __forceinline__ double lfm_sigmoid(double x) { return 0.5 * (1.0 + tanh(0.5 * x)); }
__device__ __forceinline__ double lfm_l_forward(double x) {
  return LFM_L_LOW + (LFM_L_HIGH - LFM_L_LOW) * lfm_sigmoid(x);
}
__device__ __forceinline__ double lfm_l_inverse(double y) {
  const double u = (y - LFM_L_LOW) / (LFM_L_HIGH - LFM_L_LOW);
  return log(u) - log1p(-u);
}

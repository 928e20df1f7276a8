// Batched small-N path, second kernel: ONE WARP per LFM.
//
// Same mathematics as lfm_batched_kernel (batched.cu: duplicate-row compression to U unique rows with
// multiplicity R, M = c I + R K_u, everything resident in shared memory for all optimiser steps of a
// launch), restructured around three observations from the ncu profile of the CTA-per-LFM kernel
// (profiles/batched_r1_*.md): 35 % of its warp stalls were CTA barriers of phases with fewer than 128
// useful threads, 17 % were instruction-cache misses of the exp/erf code inlined at every pair
// evaluation, and the pair terms were evaluated twice per step (value pass and gradient pass).
//   * one warp owns one problem: every phase is warp-synchronous (shuffles and __syncwarp, no CTA
//     barrier), and ~10 independent problems per SM hide each other's latencies;
//   * the exp/erf factors of h (src/model.py:315-365) are tabulated once per step over
//     (gene, time index, time index) -- the time grid of sim_math.cuh/grid.cu held in shared memory:
//     G T^2 evaluations instead of 2 U^2 (p53: 245 instead of 2520), one erf/erfc call per entry;
//   * rows are mapped to lanes as {lane < U-32, (U-32) + lane}, so the triangular phases touch the
//     U - 32 "extra" rows only while they are short.
// Limits: N <= 128, U <= 36, 3G+2 <= 64, G T^2 <= 2048; anything else runs the CTA-per-LFM kernel.
#include "batched.cuh"


__device__ __forceinline__ double wsum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ void wpair_decode(int p, int& r, int& c) {
  r = (int)((sqrtf(8.0f * (float)p + 1.0f) - 1.0f) * 0.5f);
  while ((r + 1) * (r + 2) / 2 <= p) ++r;
  while (r * (r + 1) / 2 > p) --r;
  c = p - r * (r + 1) / 2;
}
// 1/sqrt(x) for x > 0 normal: MUFU.RSQ64H seed + one third-order step (branch free)
__device__ __forceinline__ double w_rsqrt(double x) {
  double y0;
  asm("rsqrt.approx.ftz.f64 %0, %1;" : "=d"(y0) : "d"(x));
  const double e = fma(-(y0 * y0), x, 1.0);
  const double t = fma(e, 0.375, 0.5);
  return fma(t, y0 * e, y0);
}

#define WEX 4             // most "extra" rows beyond 32 the warp kernel takes (U <= 36)
#define XLD (WEX + 1)
#define GJN (32 + WEX)    // padded order of the Gauss-Jordan sweep of the team kernels

// ---- team primitives: a team of NW warps (NT = 32 NW threads, one CTA) owns one LFM.  NW = 1 is the warp-synchronous
// kernel (every primitive degenerates to a shuffle / __syncwarp); NW > 1 trades CTA barriers for a shorter dependent
// chain per optimiser step and is used when the batch leaves SMs idle (few restarts per GPU).
template <int NW> __device__ __forceinline__ void tsync() {
  if (NW == 1) __syncwarp(); else __syncthreads();
}
// Team sum.  NW > 1: the warp partials go through one of two alternating slot groups of `red` (flip toggles per call),
// so ONE barrier per sum is enough: a group is rewritten only after the barrier of the next call, which every thread
// passes after it has read the group.
template <int NW> __device__ __forceinline__ double tsum(double v, double* red, int& flip) {
  v = wsum(v);
  if (NW == 1) return v;
  double* r = red + flip * 2 * NW;
  flip ^= 1;
  if ((threadIdx.x & 31) == 0) r[threadIdx.x >> 5] = v;
  __syncthreads();
  double s = r[0];
#pragma unroll
  for (int w = 1; w < NW; ++w) s += r[w];
  return s;
}
// (HET: one static red_i per kernel instantiation -- an array shared by two kernels is not demoted into either and
// would move the static shared layout of the homoscedastic ones)
template <int NW, bool HET> __device__ __forceinline__ int tsum_int(int v) {
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  if constexpr (NW == 1) {
    return v;
  } else {
    __shared__ int red_i[NW];
    if ((threadIdx.x & 31) == 0) red_i[threadIdx.x >> 5] = v;
    __syncthreads();
    int s = 0;
#pragma unroll
    for (int w = 0; w < NW; ++w) s += red_i[w];
    __syncthreads();
    return s;
  }
}
template <int NW> __device__ __forceinline__ int tany(int v) {
  if (NW == 1) return __any_sync(0xffffffffu, v);
  return __syncthreads_or(v);
}
template <int NW> __device__ __forceinline__ void tsum2(double& v0, double& v1, double* red, int& flip) {
  v0 = wsum(v0); v1 = wsum(v1);   // (two independent butterflies interleave)
  if (NW == 1) return;
  double* r = red + flip * 2 * NW;
  flip ^= 1;
  if ((threadIdx.x & 31) == 0) { r[threadIdx.x >> 5] = v0; r[NW + (threadIdx.x >> 5)] = v1; }
  __syncthreads();
  v0 = r[0]; v1 = r[NW];
#pragma unroll
  for (int w = 1; w < NW; ++w) { v0 += r[w]; v1 += r[NW + w]; }
}
// 1/x for x > 0 normal: MUFU.RCP64H seed + two Newton steps (branch free; on the pivot chain of the sweep)
__device__ __forceinline__ double w_rcp(double x) {
  double y0;
  asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(y0) : "d"(x));
  double e = fma(-x, y0, 1.0);
  y0 = fma(y0, e, y0);
  e = fma(-x, y0, 1.0);
  return fma(y0, e, y0);
}
// lfm_h_core (sim_math.cuh) with the Gaussian factors entering pre-multiplied by A1: pt.g1 = A1 g1, pt.g2 = A1 g2
template <bool GRAD>
__device__ __forceinline__ void w_h_core(const LfmPoint& pa, const LfmPoint& pb, double l, double inv_l,
                                         const LfmPairTerms& pt, double& H, double& dH_da, double& dH_db,
                                         double& dH_dl) {
  const double delta = pb.t - pa.t;
  const double inv = pt.inv;
  const double E0 = pb.eg2 * inv;
  const double A2 = pa.e * pb.e;
  const double A1R1 = pt.A1R1;
  const double A2R2 = A2 * pb.q;
  H = E0 * (A1R1 - A2R2);
  if (GRAD) {
    const double A1g1 = pt.g1, A1g2 = pt.g2;
    const double g3 = pb.g3, g4 = pb.g4;
    const double hl = 0.5 * l;
    const double hd = 0.5 * pb.d;
    const double il2 = inv_l * inv_l;
    dH_da = -H * inv + E0 * pa.t * A2R2;
    dH_db = H * (pb.gam * l - inv) + E0 * (-delta * A1R1 + hl * (A1g2 - A1g1) + pb.t * A2R2 - A2 * hl * (g4 - g3));
    dH_dl = H * pb.gam * pb.d + E0 * ((A1g1 * (-delta * il2 - hd) + A1g2 * (-pa.t * il2 + hd)) -
                                      A2 * (g3 * (-pb.t * il2 - hd) + g4 * hd));
  }
}

// The small one of erf(x) / erfc(|x|): erfc(|x|) beyond 0.5, erf(x) inside (the other is 1 - it, with x's sign).
__device__ __forceinline__ double w_erf_small(double x) {
  const double ax = fabs(x);
  return ax > 0.5 ? erfc(ax) : erf(x);
}
// x3 = t/l - gamma, formed the same way wherever its small erf value is evaluated or read back
__device__ __forceinline__ double w_x3(double t, double inv_l, double gam) { return __fma_rn(t, inv_l, -gam); }
// R2 = erf(x3) + erf(gamma) (the point's q, "second_erf_terms") from v3 = w_erf_small(x3) and vg = w_erf_small(gamma),
// gamma > 0, by lfm_erfsum's rule: erfc(-x3) - erfc(gamma) when x3 < -0.5 and gamma > 0.5, where the literal sum
// cancels (by up to 1 - erf(gamma), which exp(gamma^2) then multiplies)
__device__ __forceinline__ double w_second_erfsum(double x3, double v3, double gam, double vg) {
  const bool big3 = fabs(x3) > 0.5, bigg = gam > 0.5;
  if (x3 < 0.0 && big3 && bigg) return v3 - vg;
  return (big3 ? copysign(1.0 - v3, x3) : v3) + (bigg ? 1.0 - vg : vg);
}

// Stage-1 work items of an optimiser step (team kernels): every item is ONE transcendental of (theta, l, times).
// Flat item f -> (kind << 24) | (gene << 16) | index:
//   kind 0 / 1 / 2 : per gene: gamma and exp(gamma^2) / erf or erfc of gamma / 2/sqrt(pi) exp(-gamma^2)
//   kind 3         : per time i: exp(-t_i^2 / l^2)
//   kind 4         : per time pair p: exp(-(t_ib - t_ia)^2 / l^2)
//   kind 5 / 6 / 7 : per (gene, time i): exp(-d t) / erf and erfc of t/l + gamma / erf or erfc of t/l - gamma
//   kind 8         : per (gene, distinct time difference k): erf or erfc of dt/l - gamma
__device__ __forceinline__ int stage1_items(int G, int Tu, int nD) { return 3 * G + Tu + Tu * Tu + 3 * G * Tu + G * nD; }
__device__ __forceinline__ unsigned stage1_decode(int f, int G, int Tu, int nD) {
  if (f < 3 * G) { const int m = f / 3; return ((unsigned)(f - 3 * m) << 24) | ((unsigned)m << 16); }
  f -= 3 * G;
  if (f < Tu) return (3u << 24) | (unsigned)f;
  f -= Tu;
  if (f < Tu * Tu) return (4u << 24) | (unsigned)f;
  f -= Tu * Tu;
  if (f < 3 * G * Tu) {
    const int e = f / 3, w = f - 3 * e, b = e / Tu;
    return ((unsigned)(5 + w) << 24) | ((unsigned)b << 16) | (unsigned)(e - b * Tu);
  }
  f -= 3 * G * Tu;
  const int b = f / nD;
  return (8u << 24) | ((unsigned)b << 16) | (unsigned)(f - b * nD);
}

// The same items enumerated by cost class, so that a warp's 32 items of a round run ONE transcendental routine instead of
// diverging over two: class 0 = erf-or-erfc (kinds 1, 6, 7, 8), class 1 = exp (kinds 0, 2, 3, 4, 5).
#define STAGE1_SKIP (15u << 24)
#define STAGE1_CLASSES 2
__device__ __forceinline__ int stage1_class_count(int cls, int G, int Tu, int nD) {
  return cls == 0 ? G + 2 * G * Tu + G * nD : 2 * G + Tu + Tu * Tu + G * Tu;
}
__device__ __forceinline__ unsigned stage1_class_decode(int cls, int i, int G, int Tu, int nD) {
  if (cls == 0) {
    if (i < G) return (1u << 24) | ((unsigned)i << 16);
    i -= G;
    if (i < 2 * G * Tu) {
      const int e = i >> 1, b = e / Tu;
      return ((i & 1 ? 7u : 6u) << 24) | ((unsigned)b << 16) | (unsigned)(e - b * Tu);
    }
    i -= 2 * G * Tu;
    const int b = i / nD;
    return (8u << 24) | ((unsigned)b << 16) | (unsigned)(i - b * nD);
  }
  if (i < G) return (0u << 24) | ((unsigned)i << 16);
  i -= G;
  if (i < G) return (2u << 24) | ((unsigned)i << 16);
  i -= G;
  if (i < Tu) return (3u << 24) | (unsigned)i;
  i -= Tu;
  if (i < Tu * Tu) return (4u << 24) | (unsigned)i;
  i -= Tu * Tu;
  const int b = i / Tu;
  return (5u << 24) | ((unsigned)b << 16) | (unsigned)(i - b * Tu);
}

struct WarpLayout {
  int ld;
  size_t S, tA1R1, tA1, tG1, g2, inv, utime, e2, c2, q, beta, kb, sdiag, dsum, th, u, gr, am, av, mu, ys, ring, red, side, Msm, Xs, gterm, Em, Ep, e3, g3t, Gt, Gd, er1, dval;
  size_t vs, cbar, tw;  // heteroscedastic objective only: variances (N), cbar and the trace weights (MU)
  size_t pts;       // byte offset
  size_t ints;      // byte offset: umap[N], urow[MU], rows_of[N], mflag[N]
  size_t itab;      // byte offset (inside the integer region, so that it travels with the structure cache)
  size_t bytes;
};
#define ITAB 512          // stage-1 items of a step whose decoding is tabulated once per fit (team kernels)
__host__ __device__ inline WarpLayout warp_layout(int N, int G, int MU, int MT, bool team, bool het) {
  WarpLayout L;
  const int P = 3 * G + 2;
  L.ld = MU | 1;
  size_t o = 0;
  auto take = [&](size_t n) { size_t r = o; o += (n + 1) & ~(size_t)1; return r; };
  // S also holds W22 as Wb[32][33] (phase E) and, in phases B / C, the per-step factor tables (aliased below)
  const size_t scratch = 6 * (((size_t)G * MT + 1) & ~(size_t)1) + (((size_t)MT + 1) & ~(size_t)1) +
                         (((size_t)MT * MT + 1) & ~(size_t)1) + (((size_t)G * MT * MT + 1) & ~(size_t)1);
  size_t s_doubles = (size_t)MU * L.ld > 32 * 33 ? (size_t)MU * L.ld : 32 * 33;
  if (scratch > s_doubles) s_doubles = scratch;
  L.S = take(s_doubles);
  const size_t tab = (size_t)G * MT * MT;
  L.tA1R1 = take(tab); L.tA1 = take(tab); L.tG1 = take(tab);
  L.g2 = take((size_t)G * MT); L.inv = take((size_t)G * G); L.utime = take(MT);
  L.q = take(MU); L.beta = take(MU); L.kb = take(MU); L.sdiag = take(MU);
  L.dsum = take(MU);
  L.th = take(P); L.u = take(P); L.gr = take(P); L.am = take(P); L.av = take(P); L.mu = take(G);
  L.ys = take(N);
  L.ring = take(4 * GJN);   // NW = 1: four pivot columns in flight; NW > 1: pivot row / column, double buffered
  L.red = take(32);
  L.side = take((size_t)P + 4 + 2 * (size_t)G);   // team kernels: Jacobians of the bijectors + scalars + 1/D, 1/S prepared by the spare warp
  L.gterm = take(4 * (size_t)G);
  L.dval = take((size_t)MT * MT);
  L.vs = L.cbar = L.tw = 0;
  if (het) { L.vs = take(N); L.cbar = take(MU); L.tw = take(MU); }
  {  // aliases inside S
    size_t so = L.S;
    auto sub = [&](size_t n) { size_t r = so; so += (n + 1) & ~(size_t)1; return r; };
    L.Em = sub((size_t)G * MT); L.Ep = sub((size_t)G * MT); L.e3 = sub((size_t)G * MT); L.g3t = sub((size_t)G * MT);
    L.e2 = sub((size_t)G * MT); L.c2 = sub((size_t)G * MT);
    L.Gt = sub(MT); L.Gd = sub((size_t)MT * MT); L.er1 = sub((size_t)G * MT * MT);
  }
  L.Msm = take(WEX * 32);
  L.Xs = take(WEX * XLD);
  L.pts = o * 8;
  size_t b = L.pts + (size_t)MU * sizeof(LfmPoint);
  b = (b + 15) & ~(size_t)15;
  L.ints = b;
  b += sizeof(int) * ((size_t)3 * N + 3 * MU);
  b += sizeof(unsigned short) * ((size_t)MU * (MU + 1) / 2 + 2);  // pair table
  b += sizeof(unsigned short) * ((size_t)MT * MT + 2);             // distinct time-difference index of every time pair
  b = (b + 3) & ~(size_t)3;
  L.itab = b;
  if (team) b += sizeof(unsigned) * ITAB;                          // decoded stage-1 items (kind, gene, index)
  L.bytes = (b + 15) & ~(size_t)15;
  return L;
}

// HET: heteroscedastic objective (a.var != NULL): noise c_i = v_i + c per point, M = diag(cbar) + R K_u; the per-step
// quantities cbar, q and the trace weights come out of phase B, alpha_i = (z_i - (K_u beta)_u(i)) / c_i out of phase J.
template <int NW, bool HET>
__global__ void __launch_bounds__(32 * NW, NW == 1 ? 1 : (NW <= 4 ? 4 : 2)) lfm_batched_warp_kernel(BatchedArgs a, int MT) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  constexpr int NT = 32 * NW;
  const int N = a.N, G = a.G, P = 3 * G + 2;
  const int tid = threadIdx.x;
  const int lane = tid & 31, wid = tid >> 5;
  (void)wid;
  // queue mode (a.queue != NULL): the CTA is a WORKER that takes (LFM, chunk of steps) tasks from a device-side queue
  // until the fit is done; bidx / first_step / task_steps are then per task (see the task loop below)
  int64_t bidx = a.queue ? (int64_t)(blockIdx.x % a.B) : (int64_t)blockIdx.x;
  const int MU = a.max_unique;
  const WarpLayout L = warp_layout(N, G, MU, MT, NW > 1, HET);
  double* base = reinterpret_cast<double*>(smem_raw);
  double* S = base + L.S;
  double* tA1R1 = base + L.tA1R1; double* tA1 = base + L.tA1; double* tG1 = base + L.tG1;
  double* g2 = base + L.g2; double* inv = base + L.inv; double* utime = base + L.utime;
  double* e2 = base + L.e2; double* c2 = base + L.c2;
  double* q = base + L.q; double* beta = base + L.beta; double* kb = base + L.kb;
  double* sdiag = base + L.sdiag; double* dsum = base + L.dsum;
  double* th = base + L.th; double* u = base + L.u; double* gr = base + L.gr; double* am = base + L.am;
  double* av = base + L.av; double* mu = base + L.mu; double* ys = base + L.ys; double* ring = base + L.ring;
  double* red = base + L.red;
  double* side = base + L.side;
  (void)side;
  double* Msm = base + L.Msm; double* Xs = base + L.Xs;
  double* gterm = base + L.gterm;
  double* vs = base + L.vs; double* cbar = base + L.cbar; double* tw = base + L.tw;
  (void)vs; (void)cbar; (void)tw;
  double* Em = base + L.Em; double* Ep = base + L.Ep; double* e3 = base + L.e3;
  double* Gt = base + L.Gt; double* Gd = base + L.Gd; double* er1 = base + L.er1; double* dval = base + L.dval;
  LfmPoint* pts = reinterpret_cast<LfmPoint*>(smem_raw + L.pts);
  int* umap = reinterpret_cast<int*>(smem_raw + L.ints);  // row -> unique index       (N)
  int* urow = umap + N;                                   // unique index -> first row (MU)
  int* rows_of = urow + MU;                               // rows of class u: rows_of[u * R + r] (N)
  int* mflag = rows_of + N;                               // 2 * positional block + flag (N)
  int* pgene = mflag + N;                                 // gene of every unique row (MU)
  int* tiarr = pgene + MU;                                // distinct-time index of every unique row (MU)
  unsigned short* pairs = reinterpret_cast<unsigned short*>(tiarr + MU);  // lower-triangle pair p -> (r << 8) | c
  unsigned* itab = reinterpret_cast<unsigned*>(smem_raw + L.itab);
  (void)itab;

  int fail = 0;
  const int blk = N / G;  // rows per positional mean block (model.py:145)
  // ---- structure of X (duplicate rows, distinct times, distinct time differences, pair table): identical for every
  // LFM and every launch of a fit, so the first launch (first_step == 0) stores LFM 0's copy in a.struct_cache and
  // later launches load it instead of repeating the O(N^2) scans
  int U = 0, R = 0, Tu = 0, nD = 0, ld = 1, npairs = 0;
  int s1_rounds = 0;   // team kernels: rounds of the stage-1 schedule held in itab (0 = decode the flat list on the fly)
  (void)s1_rounds;
  unsigned short* didx = pairs + ((size_t)MU * (MU + 1) / 2 + 2);
  int* const cache_i = reinterpret_cast<int*>(a.struct_cache);
  const size_t int_bytes = L.bytes - L.ints;
  if (cache_i && a.first_step > 0 && a.eval_val == nullptr) {
    U = cache_i[0]; R = cache_i[1]; Tu = cache_i[2]; nD = cache_i[3]; fail = cache_i[4]; s1_rounds = cache_i[5];
    const int* src = cache_i + 8;
    int* dst = reinterpret_cast<int*>(smem_raw + L.ints);
    for (size_t i = tid; i < int_bytes / 4; i += NT) dst[i] = src[i];
    const double* srcd = reinterpret_cast<const double*>(reinterpret_cast<const unsigned char*>(src) + int_bytes);
    for (int i = tid; i < MT; i += NT) utime[i] = srcd[i];
    for (int i = tid; i < MT * MT; i += NT) dval[i] = srcd[MT + i];
    for (int i = tid; i < N; i += NT) ys[i] = a.y[bidx * a.y_stride + i];
    if constexpr (HET) for (int i = tid; i < N; i += NT) vs[i] = a.var[bidx * a.var_stride + i];
    ld = U | 1;
    npairs = U * (U + 1) / 2;
    tsync<NW>();
  } else {
  // ---- once per launch: duplicate rows (class representative = first identical row), multiplicity ---------
  double* Xsm = S;   // X (N x 3) staged in shared memory for the O(N^2) scans below (S is not in use yet)
  for (int i = tid; i < 3 * N; i += NT) Xsm[i] = a.X[i];
  tsync<NW>();
  for (int i = tid; i < N; i += NT) {
    int rep = i;
    const double t0 = Xsm[3 * i], g0 = Xsm[3 * i + 1], f0 = Xsm[3 * i + 2];
    for (int j = 0; j < i; ++j)
      if (Xsm[3 * j] == t0 && Xsm[3 * j + 1] == g0 && Xsm[3 * j + 2] == f0) { rep = j; break; }
    umap[i] = rep;
    ys[i] = a.y[bidx * a.y_stride + i];
    if constexpr (HET) vs[i] = a.var[bidx * a.var_stride + i];
    int m = i / blk;
    if (m > G - 1) m = G - 1;
    mflag[i] = 2 * m + (((int)f0) != 0 ? 1 : 0);
  }
  tsync<NW>();
  int uniform = 1;
  {
    int nrep = 0;
    for (int i = tid; i < N; i += NT) {
      const int rep = umap[i];
      if (rep == i) ++nrep;
      int cnt = 0;
      for (int j = 0; j < N; ++j) cnt += (umap[j] == rep);
      rows_of[i] = cnt;  // temporarily the multiplicity of row i's class
    }
    tsync<NW>();
    nrep = tsum_int<NW, HET>(nrep);
    const int cnt0 = rows_of[0];
    int bad = 0;
    for (int i = tid; i < N; i += NT) bad |= (rows_of[i] != cnt0);
    bad = tany<NW>(bad);
    U = nrep; R = cnt0; uniform = !bad;
    if (!uniform || R == 1) { U = N; R = 1; }
  }
  tsync<NW>();
  if (U > MU) { U = 0; fail = -1; }  // caller's unique-row bound was wrong: refuse (info = -1)
  if (fail == 0) {
    // compact index of every class (ordered by representative row), its rows in ascending order
    for (int i = tid; i < N; i += NT) {
      int idx = i;
      if (R > 1) {
        const int rep = umap[i];
        idx = 0;
        for (int j = 0; j < rep; ++j) idx += (umap[j] == j);
      }
      mflag[i] |= idx << 8;  // park the compact index above the 8 low bits (2 * m + flag < 256)
    }
    tsync<NW>();
    for (int i = tid; i < N; i += NT) {
      const int idx = mflag[i] >> 8;
      int ord = 0;
      if (R > 1) for (int j = 0; j < i; ++j) ord += ((mflag[j] >> 8) == idx);
      rows_of[idx * R + ord] = i;
      if (ord == 0) urow[idx] = i;
    }
    tsync<NW>();
    for (int i = tid; i < N; i += NT) { umap[i] = mflag[i] >> 8; mflag[i] &= 255; }
    tsync<NW>();
  }
  // ---- distinct times of the unique rows -> pts[].ti, utime[] ------------------------------------------------
  if (fail == 0) {
    int nfirst = 0;
    for (int r = tid; r < U; r += NT) {
      const double t = Xsm[3 * urow[r]];
      int first = 1;
      for (int j = 0; j < r; ++j) if (Xsm[3 * urow[j]] == t) { first = 0; break; }
      nfirst += first;
      pts[r].flag = first;  // temporary marker
    }
    tsync<NW>();
    Tu = tsum_int<NW, HET>(nfirst);
    if (Tu > MT) { fail = -2; }  // caller's time-grid bound was wrong: refuse (info = -2)
    else {
      for (int r = tid; r < U; r += NT) {
        const double t = Xsm[3 * urow[r]];
        int idx = 0, rep = r;
        for (int j = 0; j < r; ++j) if (Xsm[3 * urow[j]] == t) { rep = j; break; }
        for (int j = 0; j < rep; ++j) idx += pts[j].flag;
        tiarr[r] = idx;
        if (rep == r) utime[idx] = t;
      }
    }
    tsync<NW>();
  }
  if (fail != 0) { U = 0; Tu = 0; }

  ld = U | 1;
  npairs = U * (U + 1) / 2;
  for (int p = tid; p < npairs; p += NT) {
    int r, cc;
    wpair_decode(p, r, cc);
    pairs[p] = (unsigned short)((r << 8) | cc);
  }
  // distinct time differences: the erf / erfc factor of a pair term depends on (gene, t_ib - t_ia) only, and a
  // regular grid has 2 T - 1 distinct differences, not T^2 (compared bit for bit; an irregular grid keeps T^2)
  {
    const int TTp = Tu * Tu;
    for (int p = tid; p < TTp; p += NT) {
      const double dv = utime[p % Tu] - utime[p / Tu];   // pair p = ia * Tu + ib
      int first = p;
      for (int j = 0; j < p; ++j)
        if (utime[j % Tu] - utime[j / Tu] == dv) { first = j; break; }
      didx[p] = (unsigned short)first;  // temporarily the representative pair
    }
    tsync<NW>();
    for (int p = tid; p < TTp; p += NT) {
      const int rep = didx[p];
      int idx = 0;
      for (int j = 0; j < rep; ++j) idx += (didx[j] == j);
      if (rep == p) dval[idx] = utime[p % Tu] - utime[p / Tu];
      Gd[p] = (double)idx;  // park the compact index (Gd is rebuilt every step)
    }
    tsync<NW>();
    int cnt = 0;
    for (int p = tid; p < TTp; p += NT) cnt += (didx[p] == p);
    nD = tsum_int<NW, HET>(cnt);
    tsync<NW>();
    for (int p = tid; p < TTp; p += NT) didx[p] = (unsigned short)(int)Gd[p];
  }
  tsync<NW>();
  if constexpr (NW > 1) {
    // Stage-1 schedule: the items of a class are cut into chunks of 32 (one warp, one round), the chunks are handed
    // heaviest class first to the least loaded warp (erf-or-erfc 8, exp 2 cost units, measured order of
    // magnitude), and slot (round r, warp w) of itab receives its chunk: itab[(r * NW + w) * 32 + lane].  A problem
    // whose chunks do not fit ITAB keeps s1_rounds = 0 and decodes the flat item list on the fly.
    __shared__ int sched_sh[ITAB / 32 + 1];
    if (tid == 0) {
      int load[NW], used[NW];
      for (int w = 0; w < NW; ++w) { load[w] = 0; used[w] = 0; }
      for (int sl = 0; sl < ITAB / 32; ++sl) sched_sh[sl] = -1;
      int ok = 1, rounds = 0;
      for (int cls = 0; cls < STAGE1_CLASSES && ok; ++cls) {
        const int cnt = stage1_class_count(cls, G, Tu, nD), wgt = cls == 0 ? 8 : 2;
        for (int j = 0; j * 32 < cnt; ++j) {
          int best = 0;
          for (int w = 1; w < NW; ++w) if (load[w] < load[best]) best = w;
          const int sl = used[best] * NW + best;
          if (sl >= ITAB / 32 || j > 255) { ok = 0; break; }
          sched_sh[sl] = (cls << 8) | j;
          load[best] += wgt;
          if (++used[best] > rounds) rounds = used[best];
        }
      }
      sched_sh[ITAB / 32] = ok ? rounds : 0;
    }
    tsync<NW>();
    s1_rounds = sched_sh[ITAB / 32];
    for (int f = tid; f < s1_rounds * NT; f += NT) {
      const int sc = sched_sh[f >> 5];
      unsigned code = STAGE1_SKIP;
      if (sc >= 0) {
        const int cls = sc >> 8, i = (sc & 255) * 32 + (f & 31);
        if (i < stage1_class_count(cls, G, Tu, nD)) code = stage1_class_decode(cls, i, G, Tu, nD);
      }
      itab[f] = code;
    }
    tsync<NW>();
  }
  if (cache_i && a.first_step == 0 && a.eval_val == nullptr && bidx == 0) {
    if (tid == 0) { cache_i[0] = U; cache_i[1] = R; cache_i[2] = Tu; cache_i[3] = nD; cache_i[4] = fail; cache_i[5] = s1_rounds; }
    int* dst = cache_i + 8;
    const int* src = reinterpret_cast<const int*>(smem_raw + L.ints);
    for (size_t i = tid; i < int_bytes / 4; i += NT) dst[i] = src[i];
    double* dstd = reinterpret_cast<double*>(reinterpret_cast<unsigned char*>(dst) + int_bytes);
    for (int i = tid; i < MT; i += NT) dstd[i] = utime[i];
    for (int i = tid; i < MT * MT; i += NT) dstd[MT + i] = dval[i];
  }
  }
  const bool eval_only = a.eval_val != nullptr;
  // ---- task loop.  Without a queue: one pass, this CTA's LFM, the launch's steps.  With a queue: pop tasks until the
  // ticket counter passes the number of tasks of the fit.  The structure above is the same for every LFM and stays in
  // shared memory; only the iterate, the Adam moments and (with per-LFM observations) y are per task.
  const int fail_struct = fail;
  int first_step = a.first_step, task_steps = a.steps;
  __shared__ int task_sh[2];
  for (;;) {
  if (a.queue) {
    LfmQueue Q = lfm_queue_view(a.queue, a.B);
    if (tid == 0) {
      const int t = atomicAdd(Q.head, 1);
      int b = -1;
      if (t < Q.total(a.total_steps, a.queue_chunk)) {
        volatile int* slot = Q.ring + t;
        while ((b = *slot) < 0) __nanosleep(200);   // published by the worker that ran this LFM's previous chunk
        __threadfence();
      }
      task_sh[0] = b;
      task_sh[1] = b >= 0 ? *(volatile int*)(Q.done + b) : 0;
    }
    __syncthreads();
    if (task_sh[0] < 0) break;
    bidx = task_sh[0];
    first_step = task_sh[1] * a.queue_chunk;
    task_steps = min(a.queue_chunk, a.total_steps - first_step);
    if (a.y_stride != 0)
      for (int i = tid; i < N; i += NT) ys[i] = __ldcg(a.y + bidx * a.y_stride + i);
    if (HET && a.var_stride != 0)
      for (int i = tid; i < N; i += NT) vs[i] = __ldcg(a.var + bidx * a.var_stride + i);
    fail = fail_struct;
  }
  for (int p = tid; p < P; p += NT) {
    // (__ldcg: in queue mode the previous chunk of this LFM may have run on another SM; L1 is not coherent)
    u[p] = __ldcg(a.u_io + bidx * P + p);
    const bool have = a.adam != nullptr && first_step > 0;
    am[p] = have ? __ldcg(a.adam + bidx * 2 * P + p) : 0.0;
    av[p] = have ? __ldcg(a.adam + bidx * 2 * P + P + p) : 0.0;
  }
  tsync<NW>();
  const int nsteps = eval_only ? 1 : task_steps;
  const double dR = (double)R;
  const int ex = U > 32 ? U - 32 : 0;  // rows [0, ex) are the "extra" rows: lane -> rows {lane < ex, ex + lane}
  const int TT = Tu * Tu;

  int nstamp = 0;
  int flip = 0;
  int sweep_ti = 0, sweep_tj = 0;   // team kernels: tile (ti >= tj) of the symmetric sweep this thread owns
  if constexpr (NW > 1) wpair_decode(tid < (GJN / 3) * (GJN / 3 + 1) / 2 ? tid : 0, sweep_ti, sweep_tj);
  (void)flip;
  // Adam bias corrections b^(step+1), carried multiplicatively (pow once per launch, not twice per step per leaf)
  double b1t = pow(a.b1, (double)first_step), b2t = pow(a.b2, (double)first_step);
#define WSTAMP() do { if (a.stamps && bidx == 0 && sidx == 1 && tid == 0) a.stamps[nstamp++] = clock64(); } while (0)
  // finer stamps inside a phase (slots 16..31 of the same buffer; tools/team_quick.py prints them)
#define WSTAMPX(i) do { if (a.stamps && bidx == 0 && sidx == 1 && tid == 0) a.stamps[16 + (i)] = clock64(); } while (0)
  // item e of a loop of n independent items goes to thread (base + e) % NT: consecutive loops of one stage land on
  // different threads, so that a team spreads the transcendentals of a stage over all of its lanes
#define TEAM_ITEMS(e, n, base) for (int e = (tid + NT - ((base) % NT)) % NT; e < (n); e += NT)
  for (int sidx = 0; sidx < nsteps; ++sidx) {
    const int step = first_step + sidx;
    WSTAMP();
    // ---- A. constrain -----------------------------------------------------------------------
    for (int p = tid; p < P; p += NT) th[p] = (p == 3 * G) ? lfm_l_forward(u[p]) : lfm_softplus(u[p]);
    tsync<NW>();
    const double l = th[3 * G], inv_l = 1.0 / l, sigma = th[3 * G + 1];
    const double c = a.jitter + sigma * sigma;
    WSTAMP();
    // ---- B. unique points, q = P^T z, z^T z ------------------------------------------------------
    // Transcendentals, factored so that each is evaluated once per distinct argument:
    //   per gene b          : gamma_b, exp(gamma_b^2), erf or erfc of gamma_b, g4_b = 2/sqrt(pi) exp(-gamma_b^2)
    //   per time i          : Gt_i = exp(-t_i^2 / l^2)
    //   per (b, i)          : Em = exp(-d_b t_i), Ep = 1 / Em, erf / erfc of t_i/l + gamma_b, erf or erfc of t_i/l - gamma_b,
    //                         g2 = g4_b Gt_i Em, g3 = g4_b Gt_i Ep           (2 gamma_b / l = d_b)
    //   per time pair       : Gd = exp(-(t_ib - t_ia)^2 / l^2)
    //   per (b, difference) : erf or erfc of (t_ib - t_ia)/l - gamma_b
    // and per table entry (b, ia, ib) only products remain: A1 = Em[ib] Ep[ia], A1 g1 = g4_b Gd.
    // |d_b t_i| > 600 (Ep would overflow) switches the whole team to direct evaluation of A1 and g1.
    // The point's q = erf(t_i/l - gamma_b) + erf(gamma_b) is formed from the erf-or-erfc values (w_second_erfsum).
    // Stage 1: every item is ONE transcendental of (theta, l, times) alone; stage 2: the products.
    int slow = 0;
    double zz = 0.0;
    double lsum = 0.0, tr0 = 0.0;   // HET: zz = sum z_i^2 / c_i, lsum = sum log c_i - sum log cbar_u, tr0 (lfm_het_row)
    (void)lsum; (void)tr0;
    if constexpr (NW == 1) {
    double* g3t = base + L.g3t;
    for (int m = lane; m < G; m += 32) {
      mu[m] = th[2 * G + m] / th[m];
      const double gam = th[m] * l * 0.5;
      gterm[4 * m + 0] = gam;
      gterm[4 * m + 1] = exp(gam * gam);
      gterm[4 * m + 2] = w_erf_small(gam);
      gterm[4 * m + 3] = LFM_TWO_OVER_SQRT_PI * exp(-gam * gam);
    }
    for (int i = lane; i < Tu; i += 32) { const double tl = utime[i] * inv_l; Gt[i] = exp(-tl * tl); }
    for (int p = lane; p < TT; p += 32) {
      const double dl = (utime[p % Tu] - utime[p / Tu]) * inv_l;
      Gd[p] = exp(-dl * dl);
    }
    __syncwarp();
    for (int e = lane; e < G * Tu; e += 32) {
      const int b = e / Tu, i = e % Tu;
      const double t = utime[i], d_b = th[b], gam = gterm[4 * b], g4b = gterm[4 * b + 3];
      if (fabs(d_b * t) > 600.0) slow = 1;
      const double em = exp(-d_b * t), ep = 1.0 / em;
      Em[b * MT + i] = em;
      Ep[b * MT + i] = ep;
      const double x2 = t * inv_l + gam;
      e2[b * MT + i] = erf(x2);
      c2[b * MT + i] = erfc(fabs(x2));
      e3[b * MT + i] = w_erf_small(w_x3(t, inv_l, gam));
      g2[b * MT + i] = g4b * Gt[i] * em;
      g3t[b * MT + i] = g4b * Gt[i] * ep;
    }
    for (int e = lane; e < G * G; e += 32) inv[e] = 1.0 / (th[e / G] + th[e % G]);
    slow = __any_sync(0xffffffffu, slow);
    // erf-family factor per (gene, distinct difference): erfc(|x1|) beyond 0.5, erf(x1) inside
    for (int e = lane; e < G * nD; e += 32) {
      const int b = e / nD, k = e % nD;
      const double x1 = dval[k] * inv_l - gterm[4 * b];
      er1[b * MT * MT + k] = (fabs(x1) > 0.5) ? erfc(fabs(x1)) : erf(x1);
    }
    __syncwarp();
    for (int r = lane; r < U; r += 32) {
      const double* row3 = a.X + 3 * urow[r];
      LfmPoint p;
      p.t = row3[0];
      p.gene = lfm_resolve_gene(row3[1], G);
      p.flag = ((int)row3[2]) != 0;
      p.ti = tiarr[r];
      p.d = th[p.gene];
      p.s = th[G + p.gene];
      p.gam = gterm[4 * p.gene + 0];
      p.eg2 = gterm[4 * p.gene + 1];
      p.erfg = gterm[4 * p.gene + 2];   // (the small one of erf / erfc of gamma)
      p.g4 = gterm[4 * p.gene + 3];
      p.e = Em[p.gene * MT + p.ti];
      p.q = w_second_erfsum(w_x3(p.t, inv_l, p.gam), e3[p.gene * MT + p.ti], p.gam, p.erfg);
      p.g3 = slow ? LFM_TWO_OVER_SQRT_PI * exp(-(p.t * inv_l - p.gam) * (p.t * inv_l - p.gam)) : g3t[p.gene * MT + p.ti];
      pts[r] = p;
      pgene[r] = p.gene;
    }
    __syncwarp();
    if constexpr (HET) {
      for (int r = lane; r < U; r += 32) {
        double om = 0.0, om2 = 0.0, sz = 0.0;
        for (int k = 0; k < R; ++k) {
          const int i = rows_of[r * R + k];
          lfm_het_point(ys[i] - mu[mflag[i] >> 1] * (double)(mflag[i] & 1), vs[i], c, om, om2, sz, zz, lsum);
        }
        lfm_het_row(dR, om, om2, sz, cbar[r], q[r], tw[r], lsum, tr0);
      }
      zz = wsum(zz); lsum = wsum(lsum); tr0 = wsum(tr0);
      __syncwarp();
    } else {
    for (int i = lane; i < N; i += 32) {
      const double zi = ys[i] - mu[mflag[i] >> 1] * (double)(mflag[i] & 1);
      zz += zi * zi;
    }
    zz = wsum(zz);
    for (int r = lane; r < U; r += 32) {
      double acc = 0.0;
      for (int k = 0; k < R; ++k) {
        const int i = rows_of[r * R + k];
        acc += ys[i] - mu[mflag[i] >> 1] * (double)(mflag[i] & 1);
      }
      q[r] = acc;
    }
    }
    } else {
    {
      const int nloop = s1_rounds > 0 ? s1_rounds * NT : stage1_items(G, Tu, nD);
      for (int f = tid; f < nloop; f += NT) {
        const unsigned code = s1_rounds > 0 ? itab[f] : stage1_decode(f, G, Tu, nD);
        const int kind = (int)(code >> 24), b = (int)((code >> 16) & 255u), idx = (int)(code & 0xffffu);
        if (kind == 15) continue;
        const double gam = th[b] * l * 0.5;
        // ONE call site per routine (exp / erf-or-erfc): the lanes of a scheduled chunk differ in how the argument
        // is formed and where the value goes, not in the routine they run
        if (kind == 1 || kind >= 6) {
          // the small one of erf(x) / erfc(|x|) is evaluated, the other is 1 - it (kind 6 keeps both, kinds 1, 7, 8 the
          // small one)
          const double x = kind == 6 ? utime[idx] * inv_l + gam
                         : kind == 8 ? dval[idx] * inv_l - gam
                         : kind == 7 ? w_x3(utime[idx], inv_l, gam) : gam;
          const double ax = fabs(x);
          const bool big = ax > 0.5;
          const double v = big ? erfc(ax) : erf(x);
          if (kind == 6) {
            e2[b * MT + idx] = big ? copysign(1.0 - v, x) : v;
            c2[b * MT + idx] = big ? v : 1.0 - fabs(v);
          } else if (kind == 8) {
            er1[b * MT * MT + idx] = v;
          } else if (kind == 7) {
            e3[b * MT + idx] = v;
          } else {
            gterm[4 * b + 2] = v;
          }
        } else {
          double arg;
          if (kind == 0) {
            mu[b] = th[2 * G + b] / th[b];
            gterm[4 * b + 0] = gam;
            arg = gam * gam;
          } else if (kind == 2) {
            arg = -gam * gam;
          } else if (kind == 3) {
            const double tl = utime[idx] * inv_l;
            arg = -tl * tl;
          } else if (kind == 4) {
            const double dl = dval[didx[idx]] * inv_l;   // (the same difference, bit for bit)
            arg = -dl * dl;
          } else {
            const double t = utime[idx], d_b = th[b];
            if (fabs(d_b * t) > 600.0) slow = 1;
            arg = -d_b * t;
          }
          const double ev = exp(arg);
          if (kind == 0) gterm[4 * b + 1] = ev;
          else if (kind == 2) gterm[4 * b + 3] = LFM_TWO_OVER_SQRT_PI * ev;
          else if (kind == 3) Gt[idx] = ev;
          else if (kind == 4) Gd[idx] = ev;
          else Em[b * MT + idx] = ev;
        }
      }
    }
    WSTAMPX(0);
    slow = tany<NW>(slow);   // (NW > 1: also the barrier between the stages)
    tsync<NW>();
    WSTAMPX(1);
    {
      int ibase = 0;
      TEAM_ITEMS(e, G * Tu, ibase) {
        const int b = e / Tu, i = e % Tu;
        const double em = Em[b * MT + i];
        Ep[b * MT + i] = 1.0 / em;
        g2[b * MT + i] = gterm[4 * b + 3] * Gt[i] * em;
      }
      ibase += G * Tu;
      TEAM_ITEMS(r, U, ibase) {
        const double* row3 = a.X + 3 * urow[r];
        LfmPoint p;
        p.t = row3[0];
        p.gene = lfm_resolve_gene(row3[1], G);
        p.flag = ((int)row3[2]) != 0;
        p.ti = tiarr[r];
        p.d = th[p.gene];
        p.s = th[G + p.gene];
        p.gam = gterm[4 * p.gene + 0];
        p.eg2 = gterm[4 * p.gene + 1];
        p.erfg = gterm[4 * p.gene + 2];   // (the small one of erf / erfc of gamma)
        p.g4 = gterm[4 * p.gene + 3];
        p.e = Em[p.gene * MT + p.ti];
        p.q = w_second_erfsum(w_x3(p.t, inv_l, p.gam), e3[p.gene * MT + p.ti], p.gam, p.erfg);
        p.g3 = slow ? LFM_TWO_OVER_SQRT_PI * exp(-(p.t * inv_l - p.gam) * (p.t * inv_l - p.gam))
                    : p.g4 * Gt[p.ti] * (1.0 / p.e);
        pts[r] = p;
        pgene[r] = p.gene;
      }
      ibase += U;
      TEAM_ITEMS(e, G * G, ibase) inv[e] = 1.0 / (th[e / G] + th[e % G]);
      ibase += G * G;
      if constexpr (HET) {
        TEAM_ITEMS(r, U, ibase) {
          double om = 0.0, om2 = 0.0, sz = 0.0;
          for (int k = 0; k < R; ++k) {
            const int i = rows_of[r * R + k];
            lfm_het_point(ys[i] - mu[mflag[i] >> 1] * (double)(mflag[i] & 1), vs[i], c, om, om2, sz, zz, lsum);
          }
          lfm_het_row(dR, om, om2, sz, cbar[r], q[r], tw[r], lsum, tr0);
        }
      } else {
      TEAM_ITEMS(r, U, ibase) {
        double acc = 0.0;
        for (int k = 0; k < R; ++k) {
          const int i = rows_of[r * R + k];
          acc += ys[i] - mu[mflag[i] >> 1] * (double)(mflag[i] & 1);
        }
        q[r] = acc;
      }
      }
    }
    WSTAMPX(2);
    if constexpr (HET) {
      tsum2<NW>(zz, lsum, red, flip);
      tr0 = tsum<NW>(tr0, red, flip);
    } else {
    for (int i = tid; i < N; i += NT) {
      const double zi = ys[i] - mu[mflag[i] >> 1] * (double)(mflag[i] & 1);
      zz += zi * zi;
    }
    zz = tsum<NW>(zz, red, flip);
    }
    tsync<NW>();
    }
    if (HET && !(lsum == lsum) && fail == 0) fail = 1;   // some c_i <= 0: Sigma is not a covariance
    WSTAMP();
    // ---- C. time-grid tables: per (b, ia, ib) products of the factors above (tG1 holds A1 * g1) -----------------
    for (int e = tid; e < G * TT; e += NT) {
      const int b = e / TT, r2 = e % TT, ia = r2 / Tu, ib = r2 % Tu;
      const double gam = gterm[4 * b];
      const double delta = utime[ib] - utime[ia];
      const double x1 = delta * inv_l - gam;
      const double x2 = utime[ia] * inv_l + gam;
      const double ev = er1[b * MT * MT + didx[r2]];
      const bool big1 = fabs(x1) > 0.5;
      // lfm_erfsum(x1, x2): erfc(-n) - erfc(p) for opposite signs beyond 0.5, erf(x1) + erf(x2) otherwise
      double R1;
      if (x1 * x2 < 0.0 && big1 && fabs(x2) > 0.5) {
        R1 = (x1 < x2) ? (ev - c2[b * MT + ia]) : (c2[b * MT + ia] - ev);
      } else {
        const double erf1 = big1 ? copysign(1.0 - ev, x1) : ev;
        R1 = erf1 + e2[b * MT + ia];
      }
      double A1, A1g1;
      if (slow) {
        A1 = exp(-th[b] * delta);
        A1g1 = A1 * (LFM_TWO_OVER_SQRT_PI * exp(-x1 * x1));
      } else {
        A1 = Em[b * MT + ib] * Ep[b * MT + ia];
        A1g1 = gterm[4 * b + 3] * Gd[r2];
      }
      const size_t o = (size_t)b * MT * MT + (size_t)ia * MT + ib;
      tA1[o] = A1;
      tA1R1[o] = A1 * R1;
      tG1[o] = A1g1;
    }
    tsync<NW>();
    // h(pa, pb) from the shared-memory tables
    auto pair_terms = [&](const LfmPoint& pa, const LfmPoint& pb) {
      LfmPairTerms pt;
      const size_t o = (size_t)pb.gene * MT * MT + (size_t)pa.ti * MT + pb.ti;
      pt.A1 = tA1[o]; pt.A1R1 = tA1R1[o]; pt.g1 = tG1[o];              // g1 slot: A1 * g1
      pt.g2 = pt.A1 * g2[pb.gene * MT + pa.ti];                           // g2 slot: A1 * g2
      pt.inv = inv[pa.gene * G + pb.gene];
      return pt;
    };
    WSTAMP();
    // ---- D. M = c I + R K_u (lower + diagonal) -------------------------------------------------------
    // two pairs per lane and iteration: the two evaluations are independent straight-line code (loads first,
    // stores last), so their dependent chains interleave
    auto kxx_pair = [&](int p, int& r, int& cc) {
      r = pairs[p] >> 8; cc = pairs[p] & 255;
      const LfmPoint pi = pts[r], pj = pts[cc];
      double H1, H2, u0, u1, u2;
      w_h_core<false>(pj, pi, l, inv_l, pair_terms(pj, pi), H1, u0, u1, u2);
      w_h_core<false>(pi, pj, l, inv_l, pair_terms(pi, pj), H2, u0, u1, u2);
      double k = dR * (pi.s * pj.s * (LFM_SQRT_PI * 0.5 * l) * (H1 + H2));
      if (r == cc) k += HET ? cbar[r] : c;
      return k;
    };
    for (int p = tid; p < npairs; p += 2 * NT) {
      const bool two = p + NT < npairs;
      int r0, c0, r1, c1;
      if (NW == 1 || two) {   // (warp kernel: the lone pair of the last iteration is evaluated twice rather than branched on)
        const double k0 = kxx_pair(p, r0, c0);
        const double k1 = kxx_pair(two ? p + NT : p, r1, c1);
        S[r0 * ld + c0] = k0;
        if (two) S[r1 * ld + c1] = k1;
      } else {                // (team: under issue contention the duplicate would cost 16 % of the phase)
        const double k0 = kxx_pair(p, r0, c0);
        S[r0 * ld + c0] = k0;
      }
    }
    tsync<NW>();
    WSTAMP();
    // ---- E. M^-1 and log det M.  M = [[M11, M21^T], [M21, M22]] with M22 the trailing n2 = U - ex (<= 32) rows.
    // M22 is factorised AND inverted in registers (lane i owns row i of M22 / L22 and column i of W22 = L22^-1; the
    // pivot loop is fully unrolled; lanes >= n2 carry identity rows); the ex <= 4 leading rows enter through the
    // Schur complement, every per-lane quantity in registers with compile-time indices:
    //   B = M22^-1 M21,  S11 = M11 - M21^T B,  X11 = S11^-1,  Y = B X11,
    //   M^-1 = [[X11, -Y^T], [-Y, M22^-1 + Y B^T]],   log det M = log det M22 + log det S11.
    double logdetM, tr_team = 0.0;
    (void)tr_team;
    if constexpr (NW == 1) {
      const int n2 = U - ex;
      double am[32], yw[32], m21[WEX];
#pragma unroll
      for (int j = 0; j < 32; ++j) {
        am[j] = (lane < n2) ? ((j <= lane) ? S[(ex + lane) * ld + ex + j] : 0.0) : ((j == lane) ? 1.0 : 0.0);
        yw[j] = (j == lane) ? 1.0 : 0.0;
      }
#pragma unroll
      for (int j = 0; j < WEX; ++j) {
        m21[j] = (j < ex && lane < n2) ? S[(ex + lane) * ld + j] : 0.0;
        Msm[j * 32 + lane] = m21[j];                       // M21 transposed: Msm[j][c] = M21[c][j]
      }
      if (lane < ex)
        for (int b1 = 0; b1 <= lane; ++b1) Xs[lane * XLD + b1] = S[lane * ld + b1];
      __syncwarp();  // S is free from here on: it becomes Wb[32][33]
      WSTAMP();
      double my_rk = 1.0;
      double akk = __shfl_sync(0xffffffffu, am[0], 0);
#pragma unroll
      for (int k = 0; k < 32; ++k) {
        if (!(akk > 0.0) && fail == 0) fail = ex + k + 1;
        const double rk = w_rsqrt(akk);
        const double lik = (lane == k) ? akk * rk : am[k] * rk;
        double akk_next = 0.0;
        if (k + 1 < 32) akk_next = __shfl_sync(0xffffffffu, fma(-lik, lik, am[k + 1]), k + 1);
        if (lane == k) my_rk = rk;
        am[k] = lik;
        double* Tk = ring + (k & 3) * 32;
        Tk[lane] = (lane >= k) ? lik : 0.0;
        const double wk = yw[k] * rk;
        yw[k] = wk;
        __syncwarp();
        if (k + 1 < 32) {
          if ((k + 1) & 1) {
            const double l1 = Tk[k + 1];
            am[k + 1] = fma(-lik, l1, am[k + 1]);
            yw[k + 1] = fma(-l1, wk, yw[k + 1]);
          }
#pragma unroll
          for (int j = (k + 2) & ~1; j < 32; j += 2) {
            const double2 l2 = *reinterpret_cast<const double2*>(Tk + j);
            am[j] = fma(-lik, l2.x, am[j]);
            am[j + 1] = fma(-lik, l2.y, am[j + 1]);
            yw[j] = fma(-l2.x, wk, yw[j]);
            yw[j + 1] = fma(-l2.y, wk, yw[j + 1]);
          }
        }
        akk = akk_next;
      }
      WSTAMP();
      double ld22 = (lane < n2) ? -log(my_rk) : 0.0;   // log L_kk = -log(1 / L_kk)
      ld22 = 2.0 * wsum(ld22);
      // W22 -> Wb[i][c] (constant stride 33; padded lanes carry exact zeros / identity)
      double* Wb = S;
#pragma unroll
      for (int i = 0; i < 32; ++i) Wb[i * 33 + lane] = yw[i];
      __syncwarp();
      // row `lane` of M22^-1 = W22^T W22 (complete row, both sides of the diagonal)
      double mrow[32];
#pragma unroll
      for (int c = 0; c < 32; ++c) {
        double s0 = 0.0;
#pragma unroll
        for (int k = c; k < 32; ++k) s0 = fma(yw[k], Wb[k * 33 + c], s0);
        mrow[c] = s0;
      }
      WSTAMP();
      double ld11 = 0.0;
      double yrow[WEX];
#pragma unroll
      for (int j = 0; j < WEX; ++j) yrow[j] = 0.0;
      if (ex > 0) {
        double bcol[WEX];
#pragma unroll
        for (int j = 0; j < WEX; ++j) {
          double s0 = 0.0;
          if (j < ex) {
#pragma unroll
            for (int c = 0; c < 32; ++c) s0 = fma(mrow[c], Msm[j * 32 + c], s0);
          }
          bcol[j] = s0;   // B[lane][j]
        }
        // S11 = M11 - M21^T B: the ex (ex + 1) / 2 lane sums are reduced together (independent butterfly chains
        // interleave), every lane ends up with all of S11 in registers ...
        double s11[WEX][WEX];
#pragma unroll
        for (int a1 = 0; a1 < WEX; ++a1)
#pragma unroll
          for (int b1 = 0; b1 <= a1; ++b1) s11[a1][b1] = (a1 < ex) ? m21[a1] * bcol[b1] : 0.0;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1)
#pragma unroll
          for (int a1 = 0; a1 < WEX; ++a1)
#pragma unroll
            for (int b1 = 0; b1 <= a1; ++b1)
              if (a1 < ex) s11[a1][b1] += __shfl_xor_sync(0xffffffffu, s11[a1][b1], o);
#pragma unroll
        for (int a1 = 0; a1 < WEX; ++a1)
#pragma unroll
          for (int b1 = 0; b1 <= a1; ++b1) s11[a1][b1] = (a1 < ex) ? Xs[a1 * XLD + b1] - s11[a1][b1] : ((a1 == b1) ? 1.0 : 0.0);
        // ... and factorises / inverts it redundantly with compile-time indices (identity padding beyond ex):
        // L11 (in place), W11 = L11^-1, X11 = W11^T W11
        double rprod = 1.0;
        double rd[WEX];
#pragma unroll
        for (int k = 0; k < WEX; ++k) {
          const double piv = s11[k][k];
          if (k < ex && !(piv > 0.0) && fail == 0) fail = k + 1;
          const double rkk = w_rsqrt(piv);
          rd[k] = rkk;
          if (k < ex) rprod *= rkk;
          s11[k][k] = piv * rkk;
#pragma unroll
          for (int i = k + 1; i < WEX; ++i) s11[i][k] *= rkk;
#pragma unroll
          for (int i = k + 1; i < WEX; ++i)
#pragma unroll
            for (int j = k + 1; j <= i; ++j) s11[i][j] = fma(-s11[i][k], s11[j][k], s11[i][j]);
        }
        ld11 = -2.0 * log(rprod);   // log det S11 = 2 sum log L_kk = -2 log prod (1 / L_kk)
        double w11[WEX][WEX];      // lower: W11 = L11^-1
#pragma unroll
        for (int cc = 0; cc < WEX; ++cc) {
          w11[cc][cc] = rd[cc];
#pragma unroll
          for (int i = cc + 1; i < WEX; ++i) {
            double s0 = 0.0;
#pragma unroll
            for (int k = cc; k < i; ++k) s0 = fma(s11[i][k], w11[k][cc], s0);
            w11[i][cc] = -s0 * rd[i];
          }
        }
        double x11[WEX][WEX];      // full symmetric X11 = W11^T W11
#pragma unroll
        for (int a1 = 0; a1 < WEX; ++a1)
#pragma unroll
          for (int b1 = 0; b1 <= a1; ++b1) {
            double s0 = 0.0;
#pragma unroll
            for (int k = a1; k < WEX; ++k) s0 = fma(w11[k][a1], w11[k][b1], s0);
            x11[a1][b1] = s0;
            x11[b1][a1] = s0;
          }
        if (lane == 0) {
#pragma unroll
          for (int a1 = 0; a1 < WEX; ++a1)
#pragma unroll
            for (int b1 = 0; b1 <= a1; ++b1)
              if (a1 < ex) Xs[a1 * XLD + b1] = x11[a1][b1];   // for the final store of M^-1_11
        }
        // Y = B X11
#pragma unroll
        for (int a1 = 0; a1 < WEX; ++a1) {
          double s0 = 0.0;
#pragma unroll
          for (int b1 = 0; b1 < WEX; ++b1)
            if (b1 < ex) s0 = fma(bcol[b1], x11[b1][a1], s0);
          yrow[a1] = (a1 < ex) ? s0 : 0.0;   // Y[lane][a1]
        }
#pragma unroll
        for (int j = 0; j < WEX; ++j) Msm[j * 32 + lane] = bcol[j];
        __syncwarp();
#pragma unroll
        for (int c = 0; c < 32; ++c) {
          double s0 = mrow[c];
#pragma unroll
          for (int a1 = 0; a1 < WEX; ++a1)
            if (a1 < ex) s0 = fma(yrow[a1], Msm[a1 * 32 + c], s0);   // + Y[lane][a] B[c][a]
          mrow[c] = s0;
        }
      }
      WSTAMP();
      __syncwarp();  // every lane is done with Wb: S receives M^-1 (lower triangle, runtime ld) and sdiag
      if (lane < n2) {
        double* row = S + (ex + lane) * ld;
#pragma unroll
        for (int c = 0; c < 32; ++c) {
          if (c < lane) row[ex + c] = mrow[c];
          else if (c == lane) sdiag[ex + lane] = mrow[c];
        }
#pragma unroll
        for (int a1 = 0; a1 < WEX; ++a1)
          if (a1 < ex) row[a1] = -yrow[a1];               // M^-1_21 = -Y
      }
      if (lane < ex) {
        for (int b1 = 0; b1 < lane; ++b1) S[lane * ld + b1] = Xs[lane * XLD + b1];
        sdiag[lane] = Xs[lane * XLD + lane];
      }
      __syncwarp();
      logdetM = ld22 + ld11;
    } else {
      // Team version: symmetric sweep operator over the whole U x U matrix (no pivoting: M is SPD).  Sweeping pivot k,
      //   a_ij -= a_ik a_kj / d (i, j != k),   a_ik = a_ki = a_ik / d,   a_kk = -1 / d,      d = a_kk,
      // keeps the matrix symmetric, and after all U pivots it holds -M^-1; the pivots are the squares of the
      // Cholesky diagonal: log det M = sum log d_k, d_k <= 0 = not SPD.  Only the lower triangle is kept: thread
      // (ti >= tj) owns the TS x TS tile (ti, tj) in registers (diagonal tiles complete).  Per pivot the owners of row
      // k (tiles ti = k / TS) and of column k below them (tiles tj = k / TS) publish v = a_k. through shared memory --
      // double buffered, ONE barrier per pivot -- and every tile applies a_ij -= v_i v_j / d.  The pivot loop is
      // unrolled over k % TS so that every register index is a compile-time constant.
      // Warps 0-2 sweep (78 tiles of 3 x 3; their barrier is a named one for 96 threads); meanwhile warp 3 prepares
      // what depends on theta alone and would otherwise sit on the serial tail of the step: the Jacobians of the
      // bijectors, 1 / c, log c, the reciprocals of Adam's bias corrections and 1 / D, 1 / S of the fold (side[]).
      static_assert(NW >= 4, "the team kernels need a spare warp next to the three sweep warps");
      constexpr int TS = 3, SWEEP_THREADS = 96;
      constexpr int TG = GJN / TS, NTILE = TG * (TG + 1) / 2;
      static_assert(GJN % TS == 0 && NTILE <= SWEEP_THREADS, "tile grid");
      __shared__ int fail_sh;
      double mypiv = 1.0;
      if (tid < SWEEP_THREADS) {
      const bool active = tid < NTILE;
      const int ti = sweep_ti, tj = sweep_tj;
      const int r0 = ti * TS, c0 = tj * TS;
      double at[TS][TS];
#pragma unroll
      for (int ai = 0; ai < TS; ++ai)
#pragma unroll
        for (int bi = 0; bi < TS; ++bi) {
          const int i = r0 + ai, j = c0 + bi;
          double v = (i == j) ? 1.0 : 0.0;
          if (i < U && j < U) v = (i >= j) ? S[i * ld + j] : S[j * ld + i];
          at[ai][bi] = v;
        }
      // every sweep thread has read its part of S before any of them may store the result (the loop has >= 1 barrier
      // for U >= 1; with U == 0 nothing is stored)
      WSTAMP();
      // (unrolled over two tile rows = 2 TS pivots: buffer parity and register indices are compile-time constants)
      double* const dump = ring + 2 * GJN;
      double* const vr[2] = {active ? ring + r0 : dump, active ? ring + GJN + r0 : dump};
      double* const vc[2] = {active ? ring + c0 : dump, active ? ring + GJN + c0 : dump};
      for (int k0 = 0; k0 < U; k0 += 2 * TS) {
#pragma unroll
        for (int s2 = 0; s2 < 2 * TS; ++s2) {
          const int s = s2 % TS, par = s2 & 1;   // k0 is even: parity of k
          const int k = k0 + s2;
          const int kq = k0 / TS + s2 / TS;
          if (k < U) {
            const bool rowk = ti == kq, colk = tj == kq;
            {   // publish without branches: non-owners store into the dump slots behind the two buffers
              double* dst = rowk ? vc[par] : (colk ? vr[par] : dump);
#pragma unroll
              for (int x = 0; x < TS; ++x) dst[x] = rowk ? at[s][x] : at[x][s];
            }
            asm volatile("bar.sync 1, %0;" ::"n"(SWEEP_THREADS) : "memory");
            const double d = ring[par * GJN + k];
            if (!(d > 0.0) && fail == 0) fail = k + 1;
            if (tid == k) mypiv = d;
            if (active) {
              const double pinv = w_rcp(d);
              double f[TS], g[TS];
#pragma unroll
              for (int ai = 0; ai < TS; ++ai) f[ai] = vr[par][ai];
#pragma unroll
              for (int bi = 0; bi < TS; ++bi) g[bi] = vc[par][bi] * pinv;
#pragma unroll
              for (int ai = 0; ai < TS; ++ai)
#pragma unroll
                for (int bi = 0; bi < TS; ++bi) at[ai][bi] = fma(-f[ai], g[bi], at[ai][bi]);
              if (rowk) {
#pragma unroll
                for (int bi = 0; bi < TS; ++bi) at[s][bi] = g[bi];
              }
              if (colk) {
#pragma unroll
                for (int ai = 0; ai < TS; ++ai) at[ai][s] = f[ai] * pinv;
                if (rowk) at[s][s] = -pinv;
              }
            }
          }
        }
      }
      WSTAMP(); WSTAMP(); WSTAMP();
      asm volatile("bar.sync 1, %0;" ::"n"(SWEEP_THREADS) : "memory");   // every tile is in registers: S may be overwritten
      if (active) {
#pragma unroll
        for (int ai = 0; ai < TS; ++ai)
#pragma unroll
          for (int bi = 0; bi < TS; ++bi) {
            const int i = r0 + ai, j = c0 + bi;
            if (i < U && j < i) S[i * ld + j] = -at[ai][bi];
            else if (i < U && j == i) sdiag[i] = -at[ai][bi];
          }
      }
      if (tid == 0) fail_sh = fail;
      } else if (wid == 3) {
        for (int p = lane; p < P; p += 32) {
          const double sg = lfm_sigmoid(u[p]);
          side[4 + p] = (p == 3 * G) ? (LFM_L_HIGH - LFM_L_LOW) * sg * (1.0 - sg) : sg;
        }
        if (lane == 0) {
          side[0] = 1.0 / c;
          side[1] = log(c);
          side[2] = 1.0 / (1.0 - b1t * a.b1);
          side[3] = 1.0 / (1.0 - b2t * a.b2);
        }
        for (int m = lane; m < 2 * G; m += 32) side[4 + P + m] = 1.0 / th[m];   // 1 / D_m, 1 / S_m
      }
      __syncthreads();
      fail = fail_sh;
      {   // log det M and tr M^-1 in one team sum (sdiag was stored before the barrier above)
        double ldp = (tid < U) ? log(mypiv) : 0.0, trp = (tid < U) ? (HET ? tw[tid] * sdiag[tid] : sdiag[tid]) : 0.0;
        tsum2<NW>(ldp, trp, red, flip);
        logdetM = ldp;
        tr_team = trp;
      }
      tsync<NW>();
    }
    WSTAMP();
    // ---- F. beta = M^-1 q (M^-1 symmetric: lower triangle + sdiag), K_u beta = (q - c beta) / R ---------------
    double qkb = 0.0, kbkb = 0.0;
    const double inv_R = 1.0 / dR;   // (loop invariant; the team kernels multiply, the warp kernel divides as before)
    for (int r = tid; r < U; r += NT) {
      double acc = sdiag[r] * q[r];
      const double* rowr = S + r * ld;
      if (NW == 1) {
        for (int cc = 0; cc < r; ++cc) acc = fma(rowr[cc], q[cc], acc);
        for (int cc = r + 1; cc < U; ++cc) acc = fma(S[cc * ld + r], q[cc], acc);
      } else {   // the team is latency bound here: two independent chains
        double acc1 = 0.0, acc2 = 0.0, acc3 = 0.0;
        int cc = 0;
        for (; cc + 2 <= r; cc += 2) { acc = fma(rowr[cc], q[cc], acc); acc1 = fma(rowr[cc + 1], q[cc + 1], acc1); }
        if (cc < r) acc = fma(rowr[cc], q[cc], acc);
        for (cc = r + 1; cc + 2 <= U; cc += 2) {
          acc2 = fma(S[cc * ld + r], q[cc], acc2);
          acc3 = fma(S[(cc + 1) * ld + r], q[cc + 1], acc3);
        }
        if (cc < U) acc2 = fma(S[cc * ld + r], q[cc], acc2);
        acc = (acc + acc1) + (acc2 + acc3);
      }
      beta[r] = acc;
      const double cr = HET ? cbar[r] : c;
      const double kbv = (NW == 1) ? (q[r] - cr * acc) / dR : (q[r] - cr * acc) * inv_R;
      kb[r] = kbv;
      qkb += (HET ? q[r] / cr : q[r]) * kbv;
      kbkb += kbv * kbv;
    }
    WSTAMPX(5);
    tsum2<NW>(qkb, kbkb, red, flip);
    const double inv_c = (NW == 1) ? 1.0 / c : side[0];
    const double quad = HET ? zz - qkb : ((NW == 1) ? (zz - qkb) / c : (zz - qkb) * inv_c);
    const double logc = HET ? lsum : (double)(N - U) * ((NW == 1) ? log(c) : side[1]);
    const double nlml = 0.5 * ((double)N * LFM_LOG_2PI + logc + logdetM + quad);
    tsync<NW>();
    WSTAMP();
    // ---- I. fused derivative contraction over the lower triangle of the unique pairs --------------------
    double dl_part = 0.0;
    for (int r = tid; r < U; r += NT) dsum[r] = 0.0;
    tsync<NW>();
    struct GradPair { int r, cc; double wr, wc, wl; };
    auto grad_pair = [&](int p) {
      GradPair g;
      g.r = pairs[p] >> 8; g.cc = pairs[p] & 255;
      const int r = g.r, cc = g.cc;
      const double minv = (r == cc) ? sdiag[r] : S[r * ld + cc];
      const double wgt = ((r == cc) ? 0.5 : 1.0) * (dR * minv - beta[r] * beta[cc]);
      const LfmPoint pi = pts[r], pj = pts[cc];
      double H1, dH1_da, dH1_db, dH1_dl, H2, dH2_da, dH2_db, dH2_dl;
      w_h_core<true>(pj, pi, l, inv_l, pair_terms(pj, pi), H1, dH1_da, dH1_db, dH1_dl);
      w_h_core<true>(pi, pj, l, inv_l, pair_terms(pi, pj), H2, dH2_da, dH2_db, dH2_dl);
      const double mult = pi.s * pj.s * (LFM_SQRT_PI * 0.5 * l);
      const double k = mult * (H1 + H2);
      g.wr = wgt * (mult * (dH1_db + dH2_da));
      g.wc = wgt * (mult * (dH1_da + dH2_db));
      g.wl = wgt * (mult * (dH1_dl + dH2_dl) + k * inv_l);
      return g;
    };
    auto grad_store = [&](const GradPair& g) {
      if (g.r == g.cc) dsum[g.r] = g.wr + g.wc;
      else { S[g.r * ld + g.cc] = g.wr; S[g.cc * ld + g.r] = g.wc; }
    };
    // two pairs per lane and iteration (independent chains interleave); every pair reads and writes only its own
    // entries of S, so the loads of the second pair may precede the stores of the first
    for (int p = tid; p < npairs; p += 2 * NT) {
      const bool two = p + NT < npairs;
      if (NW == 1 || two) {
        const GradPair g0 = grad_pair(p);
        const GradPair g1 = grad_pair(two ? p + NT : p);
        dl_part += g0.wl;
        grad_store(g0);
        if (two) { dl_part += g1.wl; grad_store(g1); }
      } else {
        const GradPair g0 = grad_pair(p);
        dl_part += g0.wl;
        grad_store(g0);
      }
    }
    WSTAMPX(3);
    const double gl = tsum<NW>(dl_part, red, flip);
    tsync<NW>();
    WSTAMPX(4);
    for (int r = tid; r < U; r += NT) {  // per-point totals: full row sums, fixed order
      const double* rp = S + r * ld;
      double s0 = dsum[r], s1 = 0.0;
      int cc = 0;
      for (; cc + 2 <= U; cc += 2) {
        s0 += (cc == r) ? 0.0 : rp[cc];
        s1 += (cc + 1 == r) ? 0.0 : rp[cc + 1];
      }
      if (cc < U) s0 += (cc == r) ? 0.0 : rp[cc];
      dsum[r] = s0 + s1;
    }
    tsync<NW>();
    double aa_het = 0.0;   // HET: alpha^T alpha; alpha_i into S[i] (free from here to the next step)
    if constexpr (HET) {
      for (int i = tid; i < N; i += NT) {
        const double al = (ys[i] - mu[mflag[i] >> 1] * (double)(mflag[i] & 1) - kb[umap[i]]) / (vs[i] + c);
        S[i] = al;
        aa_het += al * al;
      }
      aa_het = tsum<NW>(aa_het, red, flip);
      if constexpr (NW == 1) __syncwarp();
    }
    WSTAMP();
    // ---- J. fold by gene; mean-function terms; sigma ---------------------------------------------
    if constexpr (NW == 1) {
    for (int m = lane; m < G; m += 32) {   // one lane per gene: fixed summation order, no shuffles
      double gd = 0.0, gs = 0.0, asum = 0.0;
      for (int i = 0; i < U; ++i) {
        if (pgene[i] == m) {
          gd += dsum[i];
          gs += 1.0 - (HET ? cbar[i] : c) * sdiag[i] - beta[i] * kb[i];
        }
      }
      // asum_m = sum_{i in positional block m} alpha_i,  alpha_i = (z_i - (K_u beta)_{u(i)}) / c
      if constexpr (HET) {
        for (int i = m * blk; i < (m + 1) * blk; ++i) asum += S[i];
      } else {
        for (int i = m * blk; i < (m + 1) * blk; ++i)
          asum += ys[i] - mu[m] * (double)(mflag[i] & 1) - kb[umap[i]];
        asum /= c;
      }
      const double D = th[m], Sm = th[G + m], Bm = th[2 * G + m];
      gr[m] = gd + asum * Bm / (D * D);
      gr[G + m] = gs / Sm;
      gr[2 * G + m] = -asum / D;
    }
    } else {
    {   // one half-warp per gene, lanes over the points, butterfly sums inside the half-warp (fixed order)
      const int hw = tid >> 4, hl = tid & 15;
      const unsigned hmask = 0xffffu << (16 * (hw & 1));
      for (int m = hw; m < G; m += NT / 16) {
        double gd = 0.0, gs = 0.0, asum = 0.0;
        for (int i = hl; i < U; i += 16) {
          if (pgene[i] == m) {
            gd += dsum[i];
            gs += 1.0 - (HET ? cbar[i] : c) * sdiag[i] - beta[i] * kb[i];
          }
        }
        for (int i = m * blk + hl; i < (m + 1) * blk; i += 16)
          asum += HET ? S[i] : ys[i] - mu[m] * (double)(mflag[i] & 1) - kb[umap[i]];
#pragma unroll
        for (int o = 8; o > 0; o >>= 1) {
          gd += __shfl_xor_sync(hmask, gd, o);
          gs += __shfl_xor_sync(hmask, gs, o);
          asum += __shfl_xor_sync(hmask, asum, o);
        }
        if (hl == 0) {
          if (!HET) asum *= inv_c;
          const double Bm = th[2 * G + m];
          const double rD = side[4 + P + m];
          gr[m] = gd + asum * Bm * rD * rD;
          gr[G + m] = gs * side[4 + P + G + m];
          gr[2 * G + m] = -asum * rD;
        }
      }
    }
    }
    {
      double tr = 0.0;
      if constexpr (NW == 1) {
        for (int i = tid; i < U; i += NT) tr += HET ? tw[i] * sdiag[i] : sdiag[i];
        tr = tsum<NW>(tr, red, flip);
      } else {
        tr = tr_team;
      }
      if (tid == 0) {
        // HET: tr Sigma^-1 = tr0 + sum_u tw_u M^-1_uu (tr is that weighted sum)
        const double trSinv = HET ? tr0 + tr : ((NW == 1) ? ((double)(N - U) + c * tr) / c : ((double)(N - U) + c * tr) * inv_c);
        const double aa = HET ? aa_het : ((NW == 1) ? (zz - 2.0 * qkb + dR * kbkb) / (c * c) : (zz - 2.0 * qkb + dR * kbkb) * (inv_c * inv_c));
        gr[3 * G] = gl;
        gr[3 * G + 1] = sigma * (trSinv - aa);
      }
    }
    tsync<NW>();
    WSTAMP();
    // ---- K. chain rule, Adam, hook ----------------------------------------------------------------
    const bool bad = fail != 0;
    b1t *= a.b1; b2t *= a.b2;
    for (int p = tid; p < P; p += NT) {
      double jac;
      if (NW == 1) {
        const double sg = lfm_sigmoid(u[p]);
        jac = (p == 3 * G) ? (LFM_L_HIGH - LFM_L_LOW) * sg * (1.0 - sg) : sg;
      } else {
        jac = side[4 + p];
      }
      double g = gr[p] * jac;
      if (bad) g = nan("");
      if (eval_only) {
        a.eval_grad[bidx * P + p] = g;
      } else {
        const double m1 = a.b1 * am[p] + (1.0 - a.b1) * g;
        const double v1 = a.b2 * av[p] + (1.0 - a.b2) * g * g;
        am[p] = m1; av[p] = v1;
        const double mhat = (NW == 1) ? m1 / (1.0 - b1t) : m1 * side[2];
        const double vhat = (NW == 1) ? v1 / (1.0 - b2t) : v1 * side[3];
        double un = u[p] - a.lr * mhat / (sqrt(vhat) + a.eps);
        if (a.fix_params && (step % a.steps_per_epoch) == 0 && G > 3) {
          if (p == G + 3) un = 1.0;  // true_s[3]  (trainer.py:152, unconstrained space: SURVEY Q5)
          if (p == 3) un = 0.8;      // true_d[3]  (trainer.py:153)
        }
        u[p] = un;
      }
    }
    WSTAMP();
    if (tid == 0) {
      const double v = bad ? nan("") : nlml;
      if (eval_only) a.eval_val[bidx] = v;
      else {
        if (a.hist) a.hist[bidx * a.ld_hist + step] = v;
        if (a.step_keys && v == v) atomicMin(a.step_keys + step, lfm_loss_key(v));   // best objective of EVERY step
      }
    }
    tsync<NW>();
  }

  if (!eval_only) {
    for (int p = tid; p < P; p += NT) {
      a.u_io[bidx * P + p] = u[p];
      if (a.adam) { a.adam[bidx * 2 * P + p] = am[p]; a.adam[bidx * 2 * P + P + p] = av[p]; }
      if (a.theta_out && first_step + task_steps >= a.total_steps) {
        double t = (p == 3 * G) ? lfm_l_forward(u[p]) : lfm_softplus(u[p]);  // trainer.py:218
        if (a.fix_params && G > 3) {                                         // trainer.py:219-220
          if (p == G + 3) t = 1.0;
          if (p == 3) t = 0.8;
        }
        a.theta_out[bidx * P + p] = t;
      }
    }
  }
  if (tid == 0 && a.info) {
    if (first_step == 0 || eval_only) a.info[bidx] = fail;
    else if (fail) a.info[bidx] = fail;
  }
  // (queue mode: the launch covers the whole fit, so "after the launch's last step" is the task that reaches total_steps)
  if (tid == 0 && a.best_key && !eval_only && a.hist && task_steps > 0 && (!a.queue || first_step + task_steps >= a.total_steps)) {
    const double v = a.hist[bidx * a.ld_hist + first_step + task_steps - 1];
    if (v == v) atomicMin(a.best_key, lfm_loss_key(v));
  }
  if (!a.queue) break;
  // publish the LFM's next chunk: every thread's stores of the iterate / moments precede the barrier, thread 0's fence
  // makes them visible device-wide before the ring slot is
  __syncthreads();
  if (tid == 0) {
    LfmQueue Q = lfm_queue_view(a.queue, a.B);
    const int c = task_sh[1] + 1;
    Q.done[bidx] = c;
    if (c * a.queue_chunk < a.total_steps) {
      const int slot = atomicAdd(Q.tail, 1);
      __threadfence();
      atomicExch(Q.ring + slot, (int)bidx);
    }
  }
  }   // task loop
}

size_t lfm_batched_warp_structure_bytes(int N, int G, int MU, int MT) {
  if (MU <= 0 || MT <= 0) return 0;
  const WarpLayout L = warp_layout(N, G, MU, MT, true, false);   // (the integer region does not depend on HET)
  return ((32 + (L.bytes - L.ints) + 8 * ((size_t)MT + (size_t)MT * MT)) + 15) & ~(size_t)15;
}

// Opt-in dynamic shared memory of one instantiation: only ever raised (the occupancy query and the launches of
// differently sized problems share it).
template <int NW, bool HET>
static cudaError_t team_smem(size_t bytes) {
  static LfmSmemConfig conf;
  return lfm_ensure_smem(lfm_batched_warp_kernel<NW, HET>, conf, bytes);
}
template <int NW, bool HET> static int team_slots(size_t bytes);
__global__ void lfm_queue_init_kernel(int* base, int64_t B, int total) {
  const LfmQueue q = lfm_queue_view(base, B);
  const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i == 0) { *q.head = 0; *q.tail = (int)B; base[2] = 0; base[3] = 0; }
  if (i < B) q.done[i] = 0;
  if (i < total) q.ring[i] = i < B ? (int)i : -1;
}
template <int NW, bool HET>
static int team_launch(cudaStream_t st, const BatchedArgs& a, int time_grid, size_t bytes) {
  LFM_CUDA_OK((team_smem<NW, HET>(bytes)));
  BatchedArgs b = a;
  unsigned grid = (unsigned)a.B;
  if (a.queue) {
    // Persistent workers + task queue: worth it only when a static assignment is UNBALANCED -- more LFMs than SMs, fewer
    // than resident CTA slots, and not a whole number per SM (512 LFMs on 148 SMs: 68 SMs would carry 4 teams for the
    // whole fit and 80 SMs 3; with the queue an LFM moves to a free slot after every chunk and the loads average out).
    int dev = 0, sms = 0;
    const int slots = team_slots<NW, HET>(bytes);
    if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess) sms = 0;
    const char* env = getenv("LFM_BATCHED_QUEUE");   // 0: never, 1: whenever a workspace is given (measurements)
    const int forced = env ? atoi(env) : -1;
    // Measured on B200 (profiles/batched_queue_r2.md): at 512 LFMs the loads a random hop produces are no better than the
    // static 4 / 3 split (4.11 vs 4.14 ms) and below one LFM per slot the hops cost (3.25 vs 2.74 ms at 148); the queue
    // pays when there are MORE LFMs than resident team slots (1024 LFMs, four warps each: 7.07 vs 8.03 ms), which is
    // the only case it is used in unless LFM_BATCHED_QUEUE=1 forces it.
    (void)sms;
    const bool use = forced == 1 || (forced != 0 && NW > 1 && slots > 0 && a.B > slots);
    if (use && slots > 0 && a.first_step == 0 && a.steps == a.total_steps && a.queue_chunk > 0) {
      const LfmQueue q = lfm_queue_view(a.queue, a.B);
      const int total = q.total(a.total_steps, a.queue_chunk);
      lfm_queue_init_kernel<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(a.queue, a.B, total);
      LFM_LAUNCHED(1);
      grid = (unsigned)(slots < total ? slots : total);
    } else {
      b.queue = nullptr;
    }
  }
  lfm_batched_warp_kernel<NW, HET><<<grid, 32 * NW, bytes, st>>>(b, time_grid);
  LFM_LAUNCHED(1);
  LFM_CUDA_OK(cudaGetLastError());
  return LFM_OK;
}
template <int NW, bool HET>
static int team_slots(size_t bytes) {   // LFMs of team size NW resident on the device at a time
  int dev = 0, sms = 0, per_sm = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) return 0;
  if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess) return 0;
  if (team_smem<NW, HET>(bytes) != cudaSuccess) return 0;
  if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, lfm_batched_warp_kernel<NW, HET>, 32 * NW, bytes) != cudaSuccess) return 0;
  return sms * per_sm;
}

// Team size for a batch of B LFMs.  The kernel time is the sum over waves of resident LFMs of the time of one wave;
// measured on B200 for the p53 shape (round 1; tools/team_quick.py reproduces it), in units of one warp-per-LFM fit:
//   team 1 (warp per LFM, 7 per SM):   1.00 alone, 1.11 with every slot taken -- no contention to speak of;
//   team 4 (four warps per LFM, 4 per SM): 0.42 up to one LFM per SM, 0.71 with every slot taken (issue contention).
// A full GPU keeps the warp-per-LFM kernel (most LFMs resident per wave); a shard that leaves lanes idle -- the
// multi-GPU case -- spends them on a shorter dependent chain per optimiser step.  Team 8 never wins (2 CTAs per SM)
// and is only reachable through LFM_BATCHED_TEAM = 1 | 4 | 8, which overrides the choice (debug / measurements).
template <bool HET>
static int team_choice(int64_t B, size_t bytes, size_t bytes_team) {
  const char* env = getenv("LFM_BATCHED_TEAM");
  const int forced = env ? atoi(env) : 0;
  if (forced == 1 || forced == 4 || forced == 8) return forced;
  // occupancy of the two instantiations for this layout: cached per host thread and device (a thread drives one device
  // at a time; another thread, or the same thread after cudaSetDevice, re-queries)
  thread_local size_t cached_bytes = 0, cached_team = 0;
  thread_local int cached_dev = -2, s1 = 0, s4 = 0, sms = 0;
  const int dev_now = lfm_current_device();
  if (bytes != cached_bytes || bytes_team != cached_team || dev_now != cached_dev) {
    int dev = 0;
    s1 = team_slots<1, HET>(bytes); s4 = team_slots<4, HET>(bytes_team);
    if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess) sms = 0;
    cached_bytes = bytes; cached_team = bytes_team; cached_dev = dev_now;
  }
  if (s1 <= 0 || s4 <= 0 || sms <= 0) return 1;
  auto wave1 = [&](int64_t n) { return 1.0 + 0.11 * (double)n / (double)s1; };
  auto wave4 = [&](int64_t n) { return n <= sms || s4 <= sms ? 0.42 : 0.42 + 0.29 * (double)(n - sms) / (double)(s4 - sms); };
  const double c1 = (double)(B / s1) * wave1(s1) + (B % s1 ? wave1(B % s1) : 0.0);
  const double c4 = (double)(B / s4) * wave4(s4) + (B % s4 ? wave4(B % s4) : 0.0);
  return c4 < c1 ? 4 : 1;
}

// Launch the warp- / team-per-LFM kernel if the problem fits its limits; returns LFM_ERR_UNSUPPORTED otherwise
// (the caller then runs the CTA-per-LFM kernel of batched.cu).
int lfm_batched_warp_launch(cudaStream_t st, const BatchedArgs& a, int time_grid) {
  const int P = 3 * a.G + 2;
  const int MU = a.max_unique;
  if (time_grid <= 0 || MU <= 0 || MU > 32 + WEX || a.N > 128 || P > 64) return LFM_ERR_UNSUPPORTED;
  if ((long long)a.G * time_grid * time_grid > 2048 || a.G > 127) return LFM_ERR_UNSUPPORTED;
  const bool het = a.var != nullptr;
  const WarpLayout L = warp_layout(a.N, a.G, MU, time_grid, false, het), Lt = warp_layout(a.N, a.G, MU, time_grid, true, het);
  if (Lt.bytes > 100 * 1024) return LFM_ERR_UNSUPPORTED;
  if (het) {
    switch (team_choice<true>(a.B, L.bytes, Lt.bytes)) {
      case 8: return team_launch<8, true>(st, a, time_grid, Lt.bytes);
      case 4: return team_launch<4, true>(st, a, time_grid, Lt.bytes);
      default: return team_launch<1, true>(st, a, time_grid, L.bytes);
    }
  }
  switch (team_choice<false>(a.B, L.bytes, Lt.bytes)) {
    case 8: return team_launch<8, false>(st, a, time_grid, Lt.bytes);
    case 4: return team_launch<4, false>(st, a, time_grid, Lt.bytes);
    default: return team_launch<1, false>(st, a, time_grid, L.bytes);
  }
}

// Team size lfm_batched_warp_launch would use for a batch of B LFMs of this shape on the current device (1, 4 or 8 warps
// per LFM); 0 when the shape is outside the limits of this file (the CTA-per-LFM kernel of batched.cu runs instead).
int lfm_batched_warp_team(int64_t B, int N, int G, int MU, int time_grid) {
  const int P = 3 * G + 2;
  if (time_grid <= 0 || MU <= 0 || MU > 32 + WEX || N > 128 || P > 64) return 0;
  if ((long long)G * time_grid * time_grid > 2048 || G > 127) return 0;
  const WarpLayout L = warp_layout(N, G, MU, time_grid, false, false), Lt = warp_layout(N, G, MU, time_grid, true, false);
  if (Lt.bytes > 100 * 1024) return 0;
  return team_choice<false>(B, L.bytes, Lt.bytes);
}

// Gram-block builders and the fused dK/dtheta (x) K_bar contraction.
//
//  * lfm_gram_tile_kernel      : general flag-aware N x M block of ExactLFM.cross_covariance
//                                (src/model.py:372-394 over kernel :152-195).
//  * symmetric training variant: lower-triangle tiles of Sigma = K + diag_add, padded to a
//                                multiple of LFM_NB with an identity tail (objectives.py:70-73).
//  * lfm_grad_contract_kernel  : sum_ij K_bar_ij dK_ij/dtheta for every kernel hyper-parameter in
//                                one pass, derivative blocks never leave registers
//                                (reverse-mode of model.py:392 under trainer.py:126).
//
// Tile = 64 x 64 outputs per CTA of 256 threads (32 x 8): a thread owns two adjacent columns
// (16-byte stores, 512 B contiguous per warp row) and 8 rows; the 64 row points and 64 column
// points of the tile, with all per-point exp/erf terms, are staged once in shared memory.
#include <cstring>
#include "sim_math.cuh"

#define GT 64  // tile edge
#ifndef LFM_GC_MINB
#define LFM_GC_MINB 2
#endif

__device__ __forceinline__ void lfm_stage_points(LfmPoint* sp, const double* __restrict__ X, int64_t n,
                                                 int64_t base, int G, const double* __restrict__ theta,
                                                 double l, bool grad, int lane64, const int* __restrict__ tidx = nullptr) {
  // lane64 in [0,64): one point per thread
  const int64_t i = base + lane64;
  if (i < n) {
    LfmPoint p = lfm_make_point(X + 3 * i, G, theta, theta + G, l, grad);
    if (tidx) p.ti = tidx[i];
    sp[lane64] = p;
  } else {
    LfmPoint p;
    p.t = 0; p.d = 1; p.s = 0; p.gam = 0; p.eg2 = 1; p.erfg = 0; p.e = 1; p.q = 0; p.g3 = 0; p.g4 = 0;
    p.gene = 0; p.flag = 1; p.ti = 0;
    sp[lane64] = p;
  }
}

// mode 0: general N x M block.  mode 1: symmetric training matrix, lower tiles only, padded.
template <int MODE, bool TAB>
__global__ void __launch_bounds__(256) lfm_gram_tile_kernel(int64_t N, int64_t M, const double* __restrict__ X,
                                                          const double* __restrict__ Y, int G,
                                                          const double* __restrict__ theta,
                                                          double* __restrict__ out, int64_t ld,
                                                          const double* __restrict__ diag_vec,
                                                          double diag_const, int add_sigma2, int64_t Npad,
                                                          LfmGrid grid, int tc0) {
  __shared__ LfmPoint rowp[GT];
  __shared__ LfmPoint colp[GT];
  const int64_t tr = blockIdx.y, tc = blockIdx.x + tc0;   // tc0: first column tile of this launch
  if (MODE == 1 && tc > tr) return;
  // time-grid tables (training matrix only): valid when the distinct times fit the caller's bound.  Both
  // instantiations are launched; the one that does not apply exits here.
  const bool tab = MODE == 1 && grid.Tu > 0 && *grid.count <= grid.Tu;
  if (tab != TAB) return;
  const int tid = threadIdx.y * 32 + threadIdx.x;
  const double l = theta[3 * G];
  const double inv_l = 1.0 / l;
  const int* tix = TAB ? grid.tidx : nullptr;
  if (tid < 64) lfm_stage_points(rowp, X, N, tr * GT, G, theta, l, false, tid, tix);
  else if (tid < 128) lfm_stage_points(colp, Y, M, tc * GT, G, theta, l, false, tid - 64, tix);
  __syncthreads();
  double dadd = diag_const;
  if (MODE == 1 && add_sigma2) {
    const double sg = theta[3 * G + 1];
    dadd += sg * sg;
  }
  const int c0 = threadIdx.x * 2;
  const int64_t j0 = tc * GT + c0;
  const LfmPoint pc0 = colp[c0];
  const LfmPoint pc1 = colp[c0 + 1];
  const bool vec_ok = ((ld & 1) == 0) && ((reinterpret_cast<uintptr_t>(out) & 15) == 0);
#pragma unroll 1
  for (int r = threadIdx.y; r < GT; r += 8) {
    const int64_t i = tr * GT + r;
    const LfmPoint pr = rowp[r];
    double v0, v1;
    if (MODE == 0) {
      if (i >= N) break;
      v0 = (j0 < M) ? lfm_kernel(pr, pc0, l, inv_l) : 0.0;
      v1 = (j0 + 1 < M) ? lfm_kernel(pr, pc1, l, inv_l) : 0.0;
      double* o = out + i * ld + j0;
      if (vec_ok && j0 + 1 < M) {
        *reinterpret_cast<double2*>(o) = make_double2(v0, v1);
      } else {
        if (j0 < M) o[0] = v0;
        if (j0 + 1 < M) o[1] = v1;
      }
    } else {
      // padded symmetric: inside [0,N)^2 the kernel value, identity outside
      if (i < N) {
        if (TAB) {
          v0 = (j0 < N) ? lfm_kxx_tab(grid, pr, pc0, l, inv_l) : 0.0;
          v1 = (j0 + 1 < N) ? lfm_kxx_tab(grid, pr, pc1, l, inv_l) : 0.0;
        } else {
          v0 = (j0 < N) ? lfm_kxx(pr, pc0, l, inv_l) : 0.0;
          v1 = (j0 + 1 < N) ? lfm_kxx(pr, pc1, l, inv_l) : 0.0;
        }
        const double dv = dadd + (diag_vec ? diag_vec[i] : 0.0);
        if (i == j0) v0 += dv;
        if (i == j0 + 1) v1 += dv;
      } else {
        v0 = (i == j0) ? 1.0 : 0.0;
        v1 = (i == j0 + 1) ? 1.0 : 0.0;
      }
      *reinterpret_cast<double2*>(out + i * ld + j0) = make_double2(v0, v1);
    }
  }
}

int lfm_launch_cross_cov(cudaStream_t st, int64_t N, int64_t M, const double* X, const double* Y, int G,
                         const double* theta, double* out, int64_t ld) {
  if (N <= 0 || M <= 0) return LFM_OK;
  dim3 grid((unsigned)((M + GT - 1) / GT), (unsigned)((N + GT - 1) / GT));
  if (grid.y > 65535) return LFM_ERR_UNSUPPORTED;
  LfmGrid none;
  memset(&none, 0, sizeof(none));
  lfm_gram_tile_kernel<0, false><<<grid, dim3(32, 8), 0, st>>>(N, M, X, Y, G, theta, out, ld, nullptr, 0.0, 0, 0, none, 0);
  LFM_LAUNCHED(1);
  LFM_CUDA_OK(cudaGetLastError());
  return LFM_OK;
}

// Sigma (lower tiles, padded to Npad) = k_xx(X, X) + diag(diag_vec) + (diag_const [+ sigma^2]) I
int lfm_launch_sigma_lower(cudaStream_t st, int64_t N, int64_t Npad, const double* X, int G,
                           const double* theta, const double* diag_vec, double diag_const, int add_sigma2,
                           double* out, int64_t ld, const LfmGrid* tg, int64_t col_begin, int64_t col_end) {
  // [col_begin, col_end): the block of columns this launch builds (multiples of 64; default: all of them)
  if (col_end < 0 || col_end > Npad) col_end = Npad;
  if (col_begin < 0) col_begin = 0;
  if (col_begin >= col_end) return LFM_OK;
  dim3 grid((unsigned)((col_end - col_begin) / GT), (unsigned)(Npad / GT));
  const int tc0 = (int)(col_begin / GT);
  LfmGrid tgv;
  memset(&tgv, 0, sizeof(tgv));
  if (tg) tgv = *tg;
  lfm_gram_tile_kernel<1, false><<<grid, dim3(32, 8), 0, st>>>(N, N, X, X, G, theta, out, ld, diag_vec, diag_const,
                                                              add_sigma2, Npad, tgv, tc0);
  LFM_LAUNCHED(1);
  if (tgv.Tu > 0) {
    lfm_gram_tile_kernel<1, true><<<grid, dim3(32, 8), 0, st>>>(N, N, X, X, G, theta, out, ld, diag_vec, diag_const,
                                                               add_sigma2, Npad, tgv, tc0);
    LFM_LAUNCHED(1);
  }
  LFM_CUDA_OK(cudaGetLastError());
  return LFM_OK;
}

// ---------------------------------------------------------------------------------------------
// Fused derivative contraction.  Work item = (row tile I, chunk of gc_tiles column tiles), lower
// triangle only; off-diagonal entries carry weight 2 (K_bar and dK are symmetric).
// Per entry (i,j), w = weight * K_bar_ij, K_bar_ij = 1/2 (Sinv_ij - alpha_i alpha_j):
//   rowacc[i] += w * (dk/dD_row, k)      colacc[j] += w * (dk/dD_col, k)      lacc += w * dk/dl
// Row partials go to rowpart[chunk][i][2], column partials to colpart[I][j][2]; a fixed-order
// second pass (lfm_grad_finish_kernel) folds them per gene -> deterministic results.
// ---------------------------------------------------------------------------------------------
// Column tiles per work item: few enough that the launch fills both CTA slots of every SM for more than one wave
// (N = 4000: 63 row tiles -> 1040 work items of <= 2 tiles instead of 156 of <= 16 on 296 slots; measured 3.83 -> 3.65 ms per evaluation), many for large N where
// the row partials (one N64 x 2 slab per chunk) would otherwise dominate the scratch.
static int lfm_gc_tiles(int64_t ntile) { return ntile <= 128 ? 2 : 16; }

template <bool TAB>
__global__ void __launch_bounds__(256, TAB ? LFM_GC_MINB : 1) lfm_grad_contract_kernel(int64_t N, const double* __restrict__ X, int G,
                                                              const double* __restrict__ theta,
                                                              const double* __restrict__ Sinv, int64_t ld,
                                                              const double* __restrict__ alpha,
                                                              double* __restrict__ rowpart,  // [nchunk][Npad64][2]
                                                              double* __restrict__ colpart,  // [ntile][Npad64][2]
                                                              double* __restrict__ lpart,    // [ntile][nchunk]
                                                              int64_t N64, int nchunk, int gc_tiles, LfmGrid grid) {
  __shared__ LfmPoint rowp[GT];
  __shared__ LfmPoint colp[GT];
  __shared__ double red[8][GT][2];
  __shared__ double lred[8];
  const int I = blockIdx.y;
  const int chunk = blockIdx.x;
  const int tid = threadIdx.y * 32 + threadIdx.x;
  const int lane = threadIdx.x, wy = threadIdx.y;
  const int jt0 = chunk * gc_tiles;
  if (jt0 > I) return;
  const int jt1 = min(I, jt0 + gc_tiles - 1);
  const double l = theta[3 * G];
  const double inv_l = 1.0 / l;
  const bool tab = grid.Tu > 0 && *grid.count <= grid.Tu;
  if (tab != TAB) return;   // both instantiations are launched; the one that does not apply exits here
  const int* tix = TAB ? grid.tidx : nullptr;
  __shared__ LfmPointGrad rowx[TAB ? GT : 1];   // per-point parts of the regrouped h-derivatives (table path only)
  __shared__ LfmPointGrad colx[TAB ? GT : 1];
  if (tid < 64) {
    lfm_stage_points(rowp, X, N, (int64_t)I * GT, G, theta, l, true, tid, tix);
    if (TAB) rowx[tid] = lfm_point_grad(rowp[tid], l, inv_l);
  }
  double racc_d[8], racc_k[8];
#pragma unroll
  for (int r = 0; r < 8; ++r) { racc_d[r] = 0.0; racc_k[r] = 0.0; }
  double lacc = 0.0;
  const int c0 = lane * 2;
  for (int J = jt0; J <= jt1; ++J) {
    __syncthreads();
    if (tid >= 64 && tid < 128) {
      lfm_stage_points(colp, X, N, (int64_t)J * GT, G, theta, l, true, tid - 64, tix);
      if (TAB) colx[tid - 64] = lfm_point_grad(colp[tid - 64], l, inv_l);
    }
    __syncthreads();
    const int64_t j0 = (int64_t)J * GT + c0;
    const LfmPoint pc0 = colp[c0];
    const LfmPoint pc1 = colp[c0 + 1];
    const LfmPointGrad xc0 = colx[TAB ? c0 : 0];
    const LfmPointGrad xc1 = colx[TAB ? c0 + 1 : 0];
    const double a0 = (j0 < N) ? alpha[j0] : 0.0;
    const double a1 = (j0 + 1 < N) ? alpha[j0 + 1] : 0.0;
    double cd0 = 0.0, ck0 = 0.0, cd1 = 0.0, ck1 = 0.0;
#pragma unroll 1
    for (int rr = 0; rr < 8; ++rr) {
      const int r = wy + 8 * rr;
      const int64_t i = (int64_t)I * GT + r;
      if (i >= N) continue;
      const LfmPoint pr = rowp[r];
      const LfmPointGrad xr = rowx[TAB ? r : 0];
      const double ai = alpha[i];
      const double2 sv = *reinterpret_cast<const double2*>(Sinv + i * ld + j0);
      if (j0 <= i && j0 < N) {
        const double w = (j0 == i ? 0.5 : 1.0) * (sv.x - ai * a0);
        double k, dr, dc, dl;
        if (TAB) lfm_kxx_grad_tab(grid, pr, xr, pc0, xc0, l, inv_l, k, dr, dc, dl);
        else lfm_kxx_grad(pr, pc0, l, inv_l, k, dr, dc, dl);
        racc_d[rr] += w * dr; racc_k[rr] += w * k;
        cd0 += w * dc; ck0 += w * k;
        lacc += w * dl;
      }
      if (j0 + 1 <= i && j0 + 1 < N) {
        const double w = (j0 + 1 == i ? 0.5 : 1.0) * (sv.y - ai * a1);
        double k, dr, dc, dl;
        if (TAB) lfm_kxx_grad_tab(grid, pr, xr, pc1, xc1, l, inv_l, k, dr, dc, dl);
        else lfm_kxx_grad(pr, pc1, l, inv_l, k, dr, dc, dl);
        racc_d[rr] += w * dr; racc_k[rr] += w * k;
        cd1 += w * dc; ck1 += w * k;
        lacc += w * dl;
      }
    }
    // column partials of this tile: reduce over the 8 row groups (fixed order)
    red[wy][c0][0] = cd0; red[wy][c0][1] = ck0;
    red[wy][c0 + 1][0] = cd1; red[wy][c0 + 1][1] = ck1;
    __syncthreads();
    if (tid < 128) {
      const int c = tid >> 1, q = tid & 1;
      double sacc = 0.0;
#pragma unroll
      for (int w8 = 0; w8 < 8; ++w8) sacc += red[w8][c][q];
      colpart[((int64_t)I * N64 + (int64_t)J * GT + c) * 2 + q] = sacc;
    }
  }
  // row partials: reduce across the 32 lanes of each warp (butterfly, fixed order)
#pragma unroll
  for (int rr = 0; rr < 8; ++rr) {
    double vd = racc_d[rr], vk = racc_k[rr];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      vd += __shfl_xor_sync(0xffffffffu, vd, o);
      vk += __shfl_xor_sync(0xffffffffu, vk, o);
    }
    if (lane == 0) {
      const int64_t i = (int64_t)I * GT + wy + 8 * rr;
      rowpart[((int64_t)chunk * N64 + i) * 2 + 0] = vd;
      rowpart[((int64_t)chunk * N64 + i) * 2 + 1] = vk;
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) lacc += __shfl_xor_sync(0xffffffffu, lacc, o);
  if (lane == 0) lred[wy] = lacc;
  __syncthreads();
  if (tid == 0) {
    double sacc = 0.0;
#pragma unroll
    for (int w8 = 0; w8 < 8; ++w8) sacc += lred[w8];
    lpart[(int64_t)I * nchunk + chunk] = sacc;
  }
}

// Per-point totals: pt[i] = (sum of row partials over chunks) + (sum of column partials over I >= tile(i))
__global__ void lfm_grad_point_kernel(int64_t N, int64_t N64, int ntile, int nchunk, int gc_tiles,
                                      const double* __restrict__ rowpart, const double* __restrict__ colpart,
                                      double* __restrict__ pt /* [N][2] */) {
  const int64_t idx = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (idx >= N * 2) return;
  const int64_t i = idx >> 1;
  const int q = (int)(idx & 1);
  const int ti = (int)(i / GT);
  double acc = 0.0;
  const int my_chunks = ti / gc_tiles + 1;  // chunks that exist for row tile ti
  for (int c = 0; c < my_chunks && c < nchunk; ++c) acc += rowpart[((int64_t)c * N64 + i) * 2 + q];
  for (int I = ti; I < ntile; ++I) acc += colpart[((int64_t)I * N64 + i) * 2 + q];
  pt[idx] = acc;
}

// One CTA per gene m (plus one extra CTA for l, sigma): folds per-point totals by gene in a fixed order and
// adds the mean-function terms.  grad layout: [dD(G), dS(G), dB(G), dl, dsigma].
//   dNLML/dD_m = sum_{i: g_i = m} ptD[i] + asum_m B_m / D_m^2          (positional block m, SURVEY Q3)
//   dNLML/dS_m = sum_{i: g_i = m} ptK[i] / S_m
//   dNLML/dB_m = - asum_m / D_m,   asum_m = sum_{i in positional block m} alpha_i
//   dNLML/dl   = sum lpart ;  dNLML/dsigma = 2 sigma tr(K_bar) = sigma (tr Sinv - alpha^T alpha)
// (the lower-triangle weights already carry the factor 2 of the symmetric sum.)
__global__ void __launch_bounds__(256) lfm_grad_finish_kernel(int64_t N, const double* __restrict__ X, int G,
                                                            const double* __restrict__ theta,
                                                            const double* __restrict__ pt,
                                                            const double* __restrict__ lpart, int64_t nl,
                                                            const double* __restrict__ alpha,
                                                            const double* __restrict__ Sinv, int64_t ld,
                                                            double* __restrict__ grad) {
  __shared__ double sh[3][256];
  const int m = blockIdx.x;
  const int tid = threadIdx.x;
  double a = 0.0, b = 0.0, c = 0.0;
  if (m < G) {
    for (int64_t i = tid; i < N; i += 256) {
      const int g = lfm_resolve_gene(X[3 * i + 1], G);
      if (g == m) { a += pt[2 * i]; b += pt[2 * i + 1]; }
    }
    const int64_t block = N / G;
    for (int64_t i = m * block + tid; i < (m + 1) * block; i += 256) c += alpha[i];
  } else {
    for (int64_t i = tid; i < nl; i += 256) a += lpart[i];
    for (int64_t i = tid; i < N; i += 256) { b += Sinv[i * ld + i]; c += alpha[i] * alpha[i]; }
  }
  sh[0][tid] = a; sh[1][tid] = b; sh[2][tid] = c;
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) {
    if (tid < o) { sh[0][tid] += sh[0][tid + o]; sh[1][tid] += sh[1][tid + o]; sh[2][tid] += sh[2][tid + o]; }
    __syncthreads();
  }
  if (tid == 0) {
    a = sh[0][0]; b = sh[1][0]; c = sh[2][0];
    if (m < G) {
      const double D = theta[m], S = theta[G + m], Bm = theta[2 * G + m];
      grad[m] = a + c * Bm / (D * D);
      grad[G + m] = b / S;
      grad[2 * G + m] = -c / D;
    } else {
      const double sigma = theta[3 * G + 1];
      grad[3 * G] = a;
      grad[3 * G + 1] = sigma * (b - c);
    }
  }
}

size_t lfm_grad_scratch_doubles(int64_t N) {
  const int64_t ntile = (N + GT - 1) / GT;
  const int64_t N64 = ntile * GT;
  const int64_t gct = lfm_gc_tiles(ntile);
  const int64_t nchunk = (ntile + gct - 1) / gct;
  return (size_t)(nchunk * N64 * 2 + ntile * N64 * 2 + ntile * nchunk + N * 2);
}

int lfm_launch_grad_contract(cudaStream_t st, int64_t N, const double* X, int G, const double* theta,
                             const double* Sinv, int64_t ld, const double* alpha, double* scratch,
                             double* grad, const LfmGrid* tg) {
  LfmGrid tgv;
  memset(&tgv, 0, sizeof(tgv));
  if (tg) tgv = *tg;
  const int64_t ntile = (N + GT - 1) / GT;
  const int64_t N64 = ntile * GT;
  const int gct = lfm_gc_tiles(ntile);
  const int64_t nchunk = (ntile + gct - 1) / gct;
  double* rowpart = scratch;
  double* colpart = rowpart + nchunk * N64 * 2;
  double* lpart = colpart + ntile * N64 * 2;
  double* pt = lpart + ntile * nchunk;
  // partial buffers are only sparsely written (lower triangle): clear them first
  LFM_CUDA_OK(cudaMemsetAsync(scratch, 0, sizeof(double) * (size_t)(nchunk * N64 * 2 + ntile * N64 * 2 + ntile * nchunk), st));
  dim3 grid((unsigned)nchunk, (unsigned)ntile);
  lfm_grad_contract_kernel<false><<<grid, dim3(32, 8), 0, st>>>(N, X, G, theta, Sinv, ld, alpha, rowpart, colpart,
                                                               lpart, N64, (int)nchunk, gct, tgv);
  if (tgv.Tu > 0) {
    lfm_grad_contract_kernel<true><<<grid, dim3(32, 8), 0, st>>>(N, X, G, theta, Sinv, ld, alpha, rowpart, colpart,
                                                                lpart, N64, (int)nchunk, gct, tgv);
    LFM_LAUNCHED(1);
  }
  LFM_CUDA_OK(cudaGetLastError());
  lfm_grad_point_kernel<<<(unsigned)((N * 2 + 255) / 256), 256, 0, st>>>(N, N64, (int)ntile, (int)nchunk, gct, rowpart,
                                                                        colpart, pt);
  LFM_CUDA_OK(cudaGetLastError());
  lfm_grad_finish_kernel<<<G + 1, 256, 0, st>>>(N, X, G, theta, pt, lpart, ntile * nchunk, alpha, Sinv, ld, grad);
  LFM_LAUNCHED(3);
  LFM_CUDA_OK(cudaGetLastError());
  return LFM_OK;
}

// Elementwise ExactLFM.h(j, k, t1, t2) (src/model.py:315-365) for n argument tuples.
__global__ void lfm_h_kernel(int64_t n, const double* __restrict__ j, const double* __restrict__ k,
                             const double* __restrict__ t1, const double* __restrict__ t2, int G,
                             const double* __restrict__ theta, double* __restrict__ out) {
  const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i >= n) return;
  const double l = theta[3 * G];
  double ra[3] = {t1[i], j[i], 1.0};
  double rb[3] = {t2[i], k[i], 1.0};
  const LfmPoint pa = lfm_make_point(ra, G, theta, theta + G, l, false);
  const LfmPoint pb = lfm_make_point(rb, G, theta, theta + G, l, false);
  double H, u0, u1, u2;
  lfm_h<false>(pa, pb, l, 1.0 / l, H, u0, u1, u2);
  out[i] = H;
}

extern "C" int lfm_h(lfm_stream_t stream, int64_t n, const double* j, const double* k, const double* t1,
                     const double* t2, int G, const double* theta, double* out) {
  if (n < 0 || G <= 0 || !theta) return LFM_ERR_INVALID;
  if (n == 0) return LFM_OK;
  if (!j || !k || !t1 || !t2 || !out) return LFM_ERR_INVALID;
  lfm_h_kernel<<<(unsigned)((n + 127) / 128), 128, 0, (cudaStream_t)stream>>>(n, j, k, t1, t2, G, theta, out);
  LFM_LAUNCHED(1);
  LFM_CUDA_OK(cudaGetLastError());
  return LFM_OK;
}

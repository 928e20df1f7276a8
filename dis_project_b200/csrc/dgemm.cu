// FP64 tensor-core GEMM for sm_100a: C = alpha * op(A) op(B) + beta * C (row-major).
//
// tcgen05.mma has no f64 kind, so the Blackwell FP64 tensor path is the warp-level
// mma.sync.aligned.m8n8k4.f64 (SASS DMMA.8x8x4; ptxas lowers the m16n8k{4,8,16} f64 shapes to the
// same instruction on sm_100a).  128 x 128 x 16 CTA tile, 8 warps of 64 x 32, 4-stage cp.async
// (LDGSTS) pipeline into padded shared memory so that every fragment read is bank-conflict free
// in both operand orientations.  Per-tile k-ranges (kmode) let the same kernel serve every
// triangular Level-3 shape of the blocked Cholesky / inverse (SYRK, TRMM, LAUUM, TRSM via
// inverted diagonal blocks) without multiplying structural zeros at tile granularity.
#include <cstring>
#include "lfm_common.cuh"

#define BK 16
#define STAGES 4
// k4-steps of a unit (of 8) over which the next unit's cp.async are issued.  Spreading them over all 8 steps issued the
// last eighth one k4-step (~300 cycles) before the barrier that needs it -- less than an L2 round trip, so every unit
// boundary stalled on its latest loads; over the first 4 steps every load has at least half a unit to land.  Measured on
// B200 (N = 4000 evaluation, ms per step): 8 steps 3.40, 6: 3.35, 5: 3.33, 4: 3.33, 3: 3.34, 2: 3.34, one burst behind
// the barrier 3.50; largest rank-128 update 23.7 -> 24.6 TF/s.  Over 4 steps spreading also beats one burst at large K:
// plain 8192^3 product 32.4 -> 34.8 TF/s = 0.98 of cuBLAS Dgemm, N = 32768 evaluation 1.116 -> 1.056 s.
#define SPREAD_STEPS 4
#define LDK (BK + 4)    // [row][k] layout: 20 doubles per row, == 4 (mod 16) -> conflict-free fragment reads

__device__ __forceinline__ void cp_async16(void* smem, const void* gmem) {
  const uint32_t s = (uint32_t)__cvta_generic_to_shared(smem);
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(s), "l"(gmem));
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;\n" ::"n"(N)); }

__device__ __forceinline__ void dmma884(double& c0, double& c1, double a, double b) {
  asm("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};\n"
      : "+d"(c0), "+d"(c1)
      : "d"(a), "d"(b));
}

// Load one operand tile (ROWS "rows" x 16 k) into a stage.
//  TRANS == 0: operand stored [row][k] in global (k contiguous)  -> smem [row][LDK]
//  TRANS == 1: operand stored [k][row] in global (row contiguous) -> smem [k][ROWS + 4]
template <int TRANS, int ROWS, int NT>
__device__ __forceinline__ void load_tile(double* s, const double* __restrict__ g, int64_t ld, int64_t row0,
                                          int64_t k0, int tid) {
#pragma unroll
  for (int i = 0; i < (ROWS * 8 + NT - 1) / NT; ++i) {
    const int id = tid + NT * i;
    if (ROWS * 8 % NT != 0 && id >= ROWS * 8) break;
    if (TRANS == 0) {
      const int r = id >> 3, kc = id & 7;
      cp_async16(s + r * LDK + kc * 2, g + (row0 + r) * ld + k0 + kc * 2);
    } else {
      const int kr = id / (ROWS / 2), mc = id % (ROWS / 2);
      cp_async16(s + kr * (ROWS + 4) + mc * 2, g + (k0 + kr) * ld + row0 + mc * 2);
    }
  }
}

// CTA tile (8 WM GM) x (8 WN 4): GM x 4 warps, each warp (8 WM) x (8 WN).
//   <8,4,2> 128 x 128, 8 warps     <4,4,4> 128 x 128, 16 warps (4 per scheduler: better DMMA/LDS overlap)
//   <4,4,2> 64 x 128 (in-place panel)       <4,2,2> 64 x 64 (small problems, 2 CTAs / SM)
//   <1,4,2> 16 x 128 (one 128-row panel spread over 8 CTAs: the look-ahead chain of the factorisation)
template <int TA, int TBN, int WM, int WN, int GM>  // TA: op(A)=A^T ; TBN = 1: B stored N x K ("NT"), 0: K x N
__global__ void __launch_bounds__(128 * GM, (WM * WN * GM <= 16) ? 2 : 1) lfm_dgemm_kernel(LfmGemm g, int tiles_n) {
  constexpr int BM = 8 * WM * GM, BN = 32 * WN, NT = 128 * GM;
  constexpr int A_STAGE = BM * LDK, B_STAGE = BN * LDK;  // >= 16 * (BM + 4), 16 * (BN + 4)
  extern __shared__ __align__(16) double smem[];
  double* sA = smem;
  double* sB = smem + STAGES * A_STAGE;
  const int tid = threadIdx.x;
  const int lane = tid & 31, warp = tid >> 5;
  long long* const stamp = (g.stamps && tid == 0) ? g.stamps + 8 * (int64_t)blockIdx.x : nullptr;
  if (stamp) {
    unsigned smid; long long gt;
    asm volatile("mov.u32 %0, %%smid;" : "=r"(smid));
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(gt));
    stamp[0] = smid; stamp[1] = clock64(); stamp[5] = gt;
  }
  int tm, tn;
  if (g.lower_only) {
    // blockIdx.x enumerates lower-triangle tiles, longest k-range first: row tiles descending, except
    // when the k-range starts at the row tile
    // (tiles of the first g.tri_skip rows, in units of BM, are not launched: skipped = s (s + 1) / 2)
    const int64_t srows = g.tri_skip / BM;
    const int64_t skipped = srows * (srows + 1) / 2;
    const int64_t total = (int64_t)gridDim.x;
    const bool asc = (g.kmode == LFM_K_GE_ROW || g.kmode == LFM_K_GE_ROWCOL || g.kmode == LFM_K_LAUUM_LATE);
    const int64_t t = skipped + (asc ? (int64_t)blockIdx.x : total - 1 - (int64_t)blockIdx.x);
    // row of triangular index t: single-precision estimate, exact integer correction.  (A double-precision sqrt here is
    // ~14 dependent FP64 instructions that queue behind the DMMAs of the other CTA on the SM: `tools/tile_life.py` had a
    // tile spend 2.2 k cycles -- a tenth of its life at K = 128 -- before its first memory request.)
    int64_t i = (int64_t)((sqrtf(8.0f * (float)t + 1.0f) - 1.0f) * 0.5f);
    while ((i + 1) * (i + 2) / 2 <= t) ++i;
    while (i * (i + 1) / 2 > t) --i;
    tm = (int)i;
    tn = (int)(t - i * (i + 1) / 2);
  } else {
    tm = blockIdx.x / tiles_n;
    tn = blockIdx.x % tiles_n;
  }
  const int64_t row0 = (int64_t)tm * BM, col0 = (int64_t)tn * BN;
  const double* __restrict__ gA = g.A + (int64_t)blockIdx.y * g.strideA;
  const double* __restrict__ gB = g.B + (int64_t)blockIdx.y * g.strideB;
  double* __restrict__ gC = g.C + (int64_t)blockIdx.y * g.strideC;
  int64_t kb = 0, ke = g.K;
  switch (g.kmode) {
    case LFM_K_LE_ROW: ke = min(g.K, row0 + BM); break;
    case LFM_K_GE_ROW: kb = row0; break;
    case LFM_K_GE_ROWCOL: kb = max(row0, col0); break;
    case LFM_K_LAUUM_LATE: kb = row0 < g.k_split ? g.k_split : max(row0, col0); break;
    default: break;
  }
  // (per-tile accumulate mode of LFM_K_LAUUM_LATE; every other launch: the launcher's mode word)
  const int c_mode = g.kmode == LFM_K_LAUUM_LATE ? (row0 < g.k_split ? 2 : 0) : g.c_mode;
  kb = max(kb, g.k_lo);
  ke = min(ke, g.k_hi);
  const int nk = ke > kb ? (int)((ke - kb) / BK) : 0;
  if (nk == 0 && c_mode >= 2) return;   // K-chunked accumulation: nothing of this chunk falls into the tile's k-range

  double acc[WM][WN][2];
#pragma unroll
  for (int i = 0; i < WM; ++i)
#pragma unroll
    for (int j = 0; j < WN; ++j) { acc[i][j][0] = 0.0; acc[i][j][1] = 0.0; }

  const int wm = (warp >> 2) * (8 * WM);  // warp row in the GM x 4 warp grid
  const int wn = (warp & 3) * (8 * WN);
  const int fr = lane >> 2, fc = lane & 3;

  // Two k-tiles (32 deep) per barrier: the four stages form two units; unit u is computed while unit u+1 streams
  // in, so there is one wait_group + one __syncthreads per 256 DMMAs of every warp.  The cp.async of unit u+1 are
  // issued from per-thread pointers computed once, not in one burst behind the barrier but in PIECES after each of the
  // first SPREAD_STEPS k4-steps of unit u.
  constexpr int PA = (BM * 8 + NT - 1) / NT;   // 16-byte chunks per thread and k-tile, operand A
  constexpr int PB = (BN * 8 + NT - 1) / NT;   //                                         operand B
  constexpr int PP = 2 * (PA + PB);            // chunks per thread and unit
  const double* gsrc[PA + PB];                 // global source of chunk i at k-tile 0 (advances by BK per k-tile)
  int sdst[PA + PB];                           // shared-memory offset of chunk i inside its stage (doubles)
  bool live[PA + PB];
#pragma unroll
  for (int i = 0; i < PA + PB; ++i) {
    const bool isA = i < PA;
    const int id = tid + NT * (isA ? i : i - PA);
    const int rows = isA ? BM : BN;
    const bool trans = isA ? (TA != 0) : (TBN == 0);   // operand stored [k][row]
    live[i] = id < rows * 8;
    const double* g0 = isA ? gA : gB;
    const int64_t ldg = isA ? g.lda : g.ldb;
    const int64_t r0g = isA ? row0 : col0;
    if (!trans) {
      const int r = id >> 3, kc = id & 7;
      gsrc[i] = g0 + (r0g + r) * ldg + kb + kc * 2;
      sdst[i] = r * LDK + kc * 2;
    } else {
      const int kr = id / (rows / 2), mc = id % (rows / 2);
      gsrc[i] = g0 + (kb + kr) * ldg + r0g + mc * 2;
      sdst[i] = kr * (rows + 4) + mc * 2;
    }
  }
  const int64_t kstepA = (TA != 0) ? (int64_t)BK * g.lda : BK;
  const int64_t kstepB = (TBN == 0) ? (int64_t)BK * g.ldb : BK;
  // piece q in [0, PP): k-tile t = q / (PA + PB), chunk i = q % (PA + PB)
  auto issue_piece = [&](int uslot, int kt0, int q) {
    const int t = q / (PA + PB), i = q % (PA + PB);
    if (kt0 + t < nk && live[i]) {
      const int slot = uslot * 2 + t;
      if (i < PA) cp_async16(sA + slot * A_STAGE + sdst[i], gsrc[i] + (int64_t)(kt0 + t) * kstepA);
      else cp_async16(sB + slot * B_STAGE + sdst[i], gsrc[i] + (int64_t)(kt0 + t) * kstepB);
    }
  };
  auto issue_unit = [&](int uslot, int kt0) {
#pragma unroll
    for (int q = 0; q < PP; ++q) issue_piece(uslot, kt0, q);
    cp_async_commit();
  };
  if (stamp) stamp[7] = clock64();   // address set-up done, nothing requested yet
  issue_unit(0, 0);
  // beta = 1, alpha = +-1 (the trailing updates C -= P P^T of the factorisation, K = 128: eight k-tiles, where the
  // read-modify-write of C at the end was a visible share of a tile's life): the C tile is loaded into the accumulators
  // NOW, behind the first unit's cp.async, so both latencies overlap and the epilogue only stores.  out = alpha * acc
  // with acc initialised to alpha * C gives C + alpha * A B exactly (alpha^2 = 1).
  const bool c_in_acc = c_mode >= 2 && nk > 0;
  // alpha = -1 as a flip of the sign bit (an integer instruction): the DMULs it replaces waited for the FP64 pipe too
  const int sgn = c_mode == 3 ? (int)0x80000000 : 0;
  auto flip = [&](double x) { return __hiloint2double(__double2hiint(x) ^ sgn, __double2loint(x)); };
  if (c_in_acc) {
#pragma unroll
    for (int i = 0; i < WM; ++i) {
      const int64_t r = row0 + wm + i * 8 + fr;
#pragma unroll
      for (int j = 0; j < WN; ++j) {
        const int64_t c = col0 + wn + j * 8 + fc * 2;
        const double2 old = __ldcg(reinterpret_cast<const double2*>(gC + r * g.ldc + c));
        acc[i][j][0] = flip(old.x);
        acc[i][j][1] = flip(old.y);
      }
    }
  }
  for (int u = 0; 2 * u < nk; ++u) {
    cp_async_wait<0>();
    __syncthreads();
    if (stamp && u == 0) stamp[2] = clock64();
    // the unit's (up to) 8 k4-steps with explicitly double-buffered fragments: the LDS of step s+1
    // are issued before the 32 DMMAs of step s
    const int nsteps = (2 * u + 1 < nk) ? 8 : 4;
    const bool spread = nsteps == 8;
    if (!spread) issue_unit((u + 1) & 1, 2 * (u + 1));
    const double* a_u = sA + ((u & 1) * 2) * A_STAGE;
    const double* b_u = sB + ((u & 1) * 2) * B_STAGE;
    double af[2][WM], bf[2][WN];
    auto load_frags = [&](int buf, int step) {
      const double* a_s = a_u + (step >> 2) * A_STAGE;
      const double* b_s = b_u + (step >> 2) * B_STAGE;
      const int k4 = (step & 3) * 4;
#pragma unroll
      for (int i = 0; i < WM; ++i) {
        if (TA == 0) af[buf][i] = a_s[(wm + i * 8 + fr) * LDK + k4 + fc];
        else af[buf][i] = a_s[(k4 + fc) * (BM + 4) + wm + i * 8 + fr];
      }
#pragma unroll
      for (int j = 0; j < WN; ++j) {
        if (TBN) bf[buf][j] = b_s[(wn + j * 8 + fr) * LDK + k4 + fc];
        else bf[buf][j] = b_s[(k4 + fc) * (BN + 4) + wn + j * 8 + fr];
      }
    };
    load_frags(0, 0);
#pragma unroll
    for (int step = 0; step < 8; ++step) {
      if (step < nsteps) {
        if (step + 1 < nsteps) load_frags((step + 1) & 1, step + 1);
#pragma unroll
        for (int i = 0; i < WM; ++i)
#pragma unroll
          for (int j = 0; j < WN; ++j) dmma884(acc[i][j][0], acc[i][j][1], af[step & 1][i], bf[step & 1][j]);
        if (spread) {
          // this step's share of the next unit's loads (slot (u+1)&1 was last read before this iteration's barrier)
          if (step < SPREAD_STEPS) {
#pragma unroll
            for (int q = step * PP / SPREAD_STEPS; q < (step + 1) * PP / SPREAD_STEPS; ++q) issue_piece((u + 1) & 1, 2 * (u + 1), q);
            if (step == SPREAD_STEPS - 1) cp_async_commit();
          }
        }
      }
    }
  }
  cp_async_wait<0>();
  if (stamp) stamp[3] = clock64();

  // epilogue: thread holds C[row = 8i + lane/4][col = 8j + 2*(lane%4) + {0,1}]
  const double alpha = g.alpha, beta = g.beta;
#pragma unroll
  for (int i = 0; i < WM; ++i) {
    const int64_t r = row0 + wm + i * 8 + fr;
#pragma unroll
    for (int j = 0; j < WN; ++j) {
      const int64_t c = col0 + wn + j * 8 + fc * 2;
      double2* p = reinterpret_cast<double2*>(gC + r * g.ldc + c);
      double2 o;
      if (c_in_acc) {
        o.x = flip(acc[i][j][0]);
        o.y = flip(acc[i][j][1]);
      } else {
        o.x = alpha * acc[i][j][0];
        o.y = alpha * acc[i][j][1];
      }
      if (c_mode != 0 && !c_in_acc) {
        const double2 old = *p;
        o.x += beta * old.x;
        o.y += beta * old.y;
      }
      *p = o;
    }
  }
  if (stamp) {
    long long gt;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(gt));
    stamp[4] = clock64(); stamp[6] = gt;
  }
}

// ---- optional per-launch timing (CUDA events on the launching stream) -----------------------------
#include <algorithm>
#include <cstdio>
#include <map>
#include <mutex>
#include <string>
#include <utility>
#include <vector>
// A process-wide DEBUG facility (bench.py's roofline pass, tools/): one profiling session at a time, serialised by a
// mutex so that launches from several host threads stay well-defined; it is off on every product path.
struct GemmProf {
  bool on = false;
  std::mutex mu;
  std::vector<cudaEvent_t> ev;   // pairs
  std::vector<char> is_chain;    // per pair: launched with the 16 x 128 latency tile (look-ahead chain)
  std::vector<int> variant;      // per pair: tile variant code TA TBN WM WN GM as decimal digits
  std::vector<double> pair_flops;
  std::string variants_json;     // filled by lfm_debug_profile_end
  size_t used = 0;
  double flops = 0.0;            // flops the launched tiles execute (tile-granular k-ranges), bulk launches
  double chain_flops = 0.0;
  long long launches = 0, chain_launches = 0;
  double chain_ms = 0.0, sum_ms = 0.0;
};
static GemmProf g_prof;

static double gemm_exec_flops(const LfmGemm& g, int BM, int BN) {
  const int64_t tm = g.M / BM, tn = g.N / BN;
  double f = 0.0;
  for (int64_t i = (g.lower_only ? g.tri_skip / BM : 0); i < tm; ++i) {
    const int64_t jn = g.lower_only ? (i + 1) : tn;
    for (int64_t j = 0; j < jn; ++j) {
      int64_t kb = 0, ke = g.K;
      const int64_t row0 = i * BM, col0 = j * BN;
      switch (g.kmode) {
        case LFM_K_LE_ROW: ke = g.K < row0 + BM ? g.K : row0 + BM; break;
        case LFM_K_GE_ROW: kb = row0; break;
        case LFM_K_GE_ROWCOL: kb = row0 > col0 ? row0 : col0; break;
        case LFM_K_LAUUM_LATE: kb = row0 < g.k_split ? g.k_split : (row0 > col0 ? row0 : col0); break;
        default: break;
      }
      if (kb < g.k_lo) kb = g.k_lo;
      if (ke > g.k_hi) ke = g.k_hi;
      if (ke > kb) f += 2.0 * BM * BN * (double)(ke - kb);
    }
  }
  return f;
}

extern "C" int lfm_debug_profile_begin(void) {
  std::lock_guard<std::mutex> lock(g_prof.mu);
  g_prof.variant.clear(); g_prof.pair_flops.clear(); g_prof.variants_json.clear();
  g_prof.on = true; g_prof.used = 0; g_prof.flops = 0.0; g_prof.launches = 0;
  g_prof.chain_flops = 0.0; g_prof.chain_launches = 0; g_prof.chain_ms = 0.0; g_prof.is_chain.clear();
  return LFM_OK;
}
// Synchronises the device; returns summed kernel time (ms), executed flops and launch count of the BULK
// launches of lfm_dgemm_kernel.  The 16 x 128-tile launches of the look-ahead chain (a different template
// instantiation, 8 CTAs, latency-bound by design) are accounted separately: lfm_debug_profile_chain.
extern "C" int lfm_debug_profile_end(double* total_ms, double* exec_flops, long long* launches) {
  std::lock_guard<std::mutex> lock(g_prof.mu);
  g_prof.on = false;
  LFM_CUDA_OK(cudaDeviceSynchronize());
  std::map<int, std::pair<double, std::pair<double, long long>>> per;  // variant -> (ms, (flops, launches))
  // The factorisation launches on three streams, so launches overlap: the kernel time reported is the length
  // of the UNION of the launch intervals (time during which at least one bulk GEMM launch was executing), from
  // event timestamps relative to the first event; the plain sum is kept in g_prof.sum_ms.
  std::vector<std::pair<double, double>> iv;
  double sum = 0.0, cms = 0.0;
  for (size_t i = 0; i + 1 < g_prof.used; i += 2) {
    float t0 = 0.f, t1 = 0.f;
    LFM_CUDA_OK(cudaEventElapsedTime(&t0, g_prof.ev[0], g_prof.ev[i]));
    LFM_CUDA_OK(cudaEventElapsedTime(&t1, g_prof.ev[0], g_prof.ev[i + 1]));
    if (g_prof.is_chain[i / 2]) cms += (double)t1 - (double)t0;
    else { sum += (double)t1 - (double)t0; iv.emplace_back((double)t0, (double)t1); }
    auto& b = per[g_prof.variant[i / 2]];
    b.first += (double)t1 - (double)t0; b.second.first += g_prof.pair_flops[i / 2]; b.second.second += 1;
  }
  {
    std::string js = "[";
    char buf[256];
    for (const auto& kv : per) {
      const int v = kv.first;
      snprintf(buf, sizeof buf, "%s{\"variant\": \"lfm_dgemm_kernel<%d,%d,%d,%d,%d>\", \"tile\": \"%dx%d\", \"launches\": %lld, "
               "\"ms_sum\": %.6f, \"executed_flops\": %.6e}", js.size() > 1 ? ", " : "", v / 10000 % 10, v / 1000 % 10, v / 100 % 10,
               v / 10 % 10, v % 10, 8 * (v / 100 % 10) * (v % 10), 32 * (v / 10 % 10), kv.second.second.second, kv.second.first,
               kv.second.second.first);
      js += buf;
    }
    g_prof.variants_json = js + "]";
  }
  std::sort(iv.begin(), iv.end());
  double uni = 0.0, cur_s = 0.0, cur_e = -1.0;
  for (const auto& p : iv) {
    if (cur_e < cur_s || p.first > cur_e) { if (cur_e > cur_s) uni += cur_e - cur_s; cur_s = p.first; cur_e = p.second; }
    else if (p.second > cur_e) cur_e = p.second;
  }
  if (cur_e > cur_s) uni += cur_e - cur_s;
  g_prof.chain_ms = cms;
  g_prof.sum_ms = sum;
  const double ms = uni;
  if (total_ms) *total_ms = ms;
  if (exec_flops) *exec_flops = g_prof.flops;
  if (launches) *launches = g_prof.launches;
  return LFM_OK;
}
extern "C" double lfm_debug_profile_sum_ms(void) { return g_prof.sum_ms; }
// JSON list of the last session's launches grouped by tile variant: launches, summed launch time (intervals overlap across
// streams, so the sums can exceed the union), executed flops.  Copies at most n - 1 characters; returns the full length.
extern "C" size_t lfm_debug_profile_variants(char* out, size_t n) {
  std::lock_guard<std::mutex> lock(g_prof.mu);
  if (out && n) {
    const size_t m = g_prof.variants_json.size() < n - 1 ? g_prof.variants_json.size() : n - 1;
    memcpy(out, g_prof.variants_json.data(), m);
    out[m] = 0;
  }
  return g_prof.variants_json.size();
}
extern "C" int lfm_debug_profile_chain(double* total_ms, double* exec_flops, long long* launches) {
  if (total_ms) *total_ms = g_prof.chain_ms;
  if (exec_flops) *exec_flops = g_prof.chain_flops;
  if (launches) *launches = g_prof.chain_launches;
  return LFM_OK;
}
static cudaEvent_t prof_event() {
  if (g_prof.used == g_prof.ev.size()) {
    cudaEvent_t e;
    cudaEventCreate(&e);
    g_prof.ev.push_back(e);
  }
  return g_prof.ev[g_prof.used++];
}

// `variant` (may be NULL) receives the instantiation's code TA TBN WM WN GM as decimal digits (the profiler's code)
template <int TA, int TBN, int WM, int WN, int GM>
static int launch(cudaStream_t st, const LfmGemm& g, int* variant) {
  constexpr int BM = 8 * WM * GM, BN = 32 * WN;
  constexpr int VARIANT = TA * 10000 + TBN * 1000 + WM * 100 + WN * 10 + GM;
  if (variant) *variant = VARIANT;
  constexpr int SMEM = STAGES * (BM + BN) * LDK * 8;
  auto* const kernel = &lfm_dgemm_kernel<TA, TBN, WM, WN, GM>;
  static LfmSmemConfig smem_cfg;
  {
    // Every tile variant asks for the LARGEST shared-memory carveout, whatever its own footprint: CTAs of two variants
    // can only share an SM if the SM does not have to be re-partitioned between L1 and shared memory for the newcomer
    // (that needs a drained SM).  With per-variant carveouts a 102 KB panel CTA of the highest-priority stream sat
    // behind a whole 64 x 64-tile trailing update (2 x 80 KB per SM) although slots freed every ~13 us (CUPTI
    // timeline, round 2).  The kernels read global memory through cp.async.cg / ld.cg only, so L1 size is irrelevant.
    const int dev = lfm_current_device();
    if (dev < 0 || smem_cfg.bytes[dev].load(std::memory_order_acquire) < (size_t)SMEM)
      LFM_CUDA_OK(cudaFuncSetAttribute(kernel, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
  }
  LFM_CUDA_OK(lfm_ensure_smem(kernel, smem_cfg, SMEM));
  const int64_t tm = g.M / BM, tn = g.N / BN;
  int64_t tiles = g.lower_only ? tm * (tm + 1) / 2 : tm * tn;
  if (g.lower_only && g.tri_skip > 0) {
    if (BM != BN || g.tri_skip % BM) return LFM_ERR_INVALID;
    const int64_t sr = g.tri_skip / BM;
    tiles -= sr * (sr + 1) / 2;
  }
  if (tiles <= 0) return LFM_OK;
  if (tiles > 0x7fffffff) return LFM_ERR_UNSUPPORTED;
  LfmGemm gk = g;
  gk.c_mode = g.beta == 0.0 ? 0 : ((g.beta == 1.0 && g.alpha == 1.0) ? 2 : ((g.beta == 1.0 && g.alpha == -1.0) ? 3 : 1));
  const bool prof = g_prof.on;
  std::unique_lock<std::mutex> lock(g_prof.mu, std::defer_lock);
  if (prof) {
    lock.lock();
    cudaEventRecord(prof_event(), st);
    const double f = gemm_exec_flops(g, BM, BN) * (g.batch > 1 ? g.batch : 1);
    const bool chain = BM == 16;
    g_prof.is_chain.push_back(chain ? 1 : 0);
    g_prof.variant.push_back(VARIANT);
    g_prof.pair_flops.push_back(f);
    if (chain) { g_prof.chain_flops += f; g_prof.chain_launches += 1; }
    else { g_prof.flops += f; g_prof.launches += 1; }
  }
  const dim3 grid((unsigned)tiles, (unsigned)(g.batch > 1 ? g.batch : 1));
  {
    // The launch carries its stream's priority as a launch attribute: inside a captured graph (the evaluation plans) the
    // kernel nodes otherwise run without one, and the panel stream's CTAs queued behind every pending CTA of a trailing
    // update instead of taking the next free slot (CUPTI timelines, eager vs graph, round 2).
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid; cfg.blockDim = dim3(128 * GM); cfg.dynamicSmemBytes = SMEM; cfg.stream = st;
    cudaLaunchAttribute attr[1];
    int prio = 0;
    unsigned nattr = 0;
    if (cudaStreamGetPriority(st, &prio) == cudaSuccess) {
      attr[0].id = cudaLaunchAttributePriority;
      attr[0].val.priority = prio;
      nattr = 1;
    } else {
      cudaGetLastError();
    }
    cfg.attrs = attr; cfg.numAttrs = nattr;
    LFM_CUDA_OK(cudaLaunchKernelEx(&cfg, kernel, gk, (int)tn));
  }
  if (prof) cudaEventRecord(prof_event(), st);
  LFM_LAUNCHED(1);
  LFM_CUDA_OK(cudaGetLastError());
  return LFM_OK;
}

template <int WM, int WN, int GM>
static int dispatch(cudaStream_t st, const LfmGemm& g, int* variant) {
  if (g.transA == 0 && g.transB == 1) return launch<0, 1, WM, WN, GM>(st, g, variant);
  if (g.transA == 0 && g.transB == 0) return launch<0, 0, WM, WN, GM>(st, g, variant);
  if (g.transA == 1 && g.transB == 0) return launch<1, 0, WM, WN, GM>(st, g, variant);
  return launch<1, 1, WM, WN, GM>(st, g, variant);
}

// Tile shape of a launch, WM WN GM as decimal digits, or a negative lfm_status.  Heuristic: 128 x 128 tiles once they
// fill >= 3 waves of the 148 SMs, else 64 x 64 tiles (two CTAs per SM) so that small trailing updates and panels still
// spread over the whole chip.  C aliasing A (in-place panel multiply) needs one tile across the full width N = 128; those
// tiles are not square, so they cannot serve lower_only.
static int dgemm_tile(const LfmGemm& g) {
  if ((g.transA | g.transB) & ~1) return LFM_ERR_INVALID;
  if (g.kmode != LFM_K_FULL && g.kmode != LFM_K_LE_ROW && g.kmode != LFM_K_GE_ROW && g.kmode != LFM_K_GE_ROWCOL &&
      g.kmode != LFM_K_LAUUM_LATE)
    return LFM_ERR_INVALID;
  if (g.M < 0 || g.N < 0 || g.K < 0 || g.tri_skip < 0) return LFM_ERR_INVALID;
  if (g.M % 128 || g.N % 128 || g.K % BK) return LFM_ERR_INVALID;
  if (g.k_lo % BK || g.k_hi % BK || g.k_split % BK) return LFM_ERR_INVALID;
  if (g.lower_only && g.M != g.N) return LFM_ERR_INVALID;
  const int64_t nb = g.batch > 1 ? g.batch : 1;
  if (nb > 65535) return LFM_ERR_UNSUPPORTED;
  const int64_t t128 = nb * (g.lower_only ? (g.M / 128) * (g.M / 128 + 1) / 2 : (g.M / 128) * (g.N / 128));
  const bool inplace = (const double*)g.C == g.A;
  if (g.tile == 1) {
    if (g.lower_only) return LFM_ERR_INVALID;
    return 142;
  }
  if (g.tile == 2 && !inplace) return 444;   // 128 x 128 tiles whatever the tile count
  if (g.tile == 3 && !inplace) return 422;   // 64 x 64 tiles (two CTAs per SM)
  if (inplace) {
    if (g.N != 128 || g.lower_only) return LFM_ERR_INVALID;
    if (t128 >= 148) return 842;
    return (g.M / 64 >= 148) ? 442 : 242;    // 64- or 32-row tiles: fill the SMs
  }
  if (g.tri_skip > 0) return 422;  // rank-128 trailing updates: 64 x 64 tiles measured fastest
  if (t128 >= 3 * 148) return 444;
  return 422;
}

static int dgemm_run(cudaStream_t st, const LfmGemm& g, int* variant) {
  const int t = dgemm_tile(g);
  switch (t) {
    case 142: return dispatch<1, 4, 2>(st, g, variant);
    case 242: return dispatch<2, 4, 2>(st, g, variant);
    case 422: return dispatch<4, 2, 2>(st, g, variant);
    case 442: return dispatch<4, 4, 2>(st, g, variant);
    case 444: return dispatch<4, 4, 4>(st, g, variant);
    case 842: return dispatch<8, 4, 2>(st, g, variant);
    default: return t < 0 ? t : LFM_ERR_INVALID;
  }
}

int lfm_dgemm(cudaStream_t st, const LfmGemm& g) { return dgemm_run(st, g, nullptr); }

// Debug: any launch lfm_dgemm can make, from a plain C descriptor.  What the kernel's 16-byte copies need is checked here,
// before anything is launched: aligned base pointers, even leading dimensions and batch strides.
extern "C" int lfm_debug_dgemm(lfm_stream_t stream, const lfm_gemm_desc* d, int* variant) {
  if (variant) *variant = 0;
  if (!d || !d->A || !d->B || !d->C) return LFM_ERR_INVALID;
  auto misaligned = [](const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) != 0; };
  if (misaligned(d->A) || misaligned(d->B) || misaligned(d->C)) return LFM_ERR_INVALID;
  if ((d->lda | d->ldb | d->ldc | d->strideA | d->strideB | d->strideC) & 1) return LFM_ERR_INVALID;
  LfmGemm g;
  g.transA = d->transA; g.transB = d->transB; g.M = d->M; g.N = d->N; g.K = d->K;
  g.A = d->A; g.lda = d->lda; g.B = d->B; g.ldb = d->ldb; g.C = d->C; g.ldc = d->ldc;
  g.alpha = d->alpha; g.beta = d->beta; g.lower_only = d->lower_only; g.kmode = d->kmode;
  g.batch = d->batch; g.strideA = d->strideA; g.strideB = d->strideB; g.strideC = d->strideC;
  g.tile = d->tile; g.tri_skip = d->tri_skip; g.k_split = d->k_split; g.k_lo = d->k_lo; g.k_hi = d->k_hi;
  return dgemm_run((cudaStream_t)stream, g, variant);
}

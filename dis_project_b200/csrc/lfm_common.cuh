// Shared declarations for the LFM sm_100a kernels.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <atomic>
#include "../../include/lfm_b200.h"

#define LFM_SQRT_PI 1.7724538509055160273
#define LFM_TWO_OVER_SQRT_PI 1.1283791670955125739
#define LFM_LOG_2PI 1.8378770664093454836

#define LFM_CUDA_OK(expr)                          \
  do {                                             \
    cudaError_t _e = (expr);                       \
    if (_e != cudaSuccess) return LFM_ERR_CUDA;    \
  } while (0)

#define LFM_TRY(expr)            \
  do {                           \
    int _s = (expr);             \
    if (_s != LFM_OK) return _s; \
  } while (0)

// Launch accounting (bench.py's gpu_launches): any host thread may launch.
extern std::atomic<unsigned long long> g_lfm_launches;
#define LFM_LAUNCHED(n) (g_lfm_launches.fetch_add((unsigned long long)(n), std::memory_order_relaxed))

// Function attributes (opt-in dynamic shared memory) are per DEVICE, and one process may drive several devices from
// several threads: every kernel keeps one of these (static storage, zero-initialised) and raises the attribute on
// the current device the first time a launch there needs more than it has been given.  Two threads racing on the
// same device both set the attribute, which is harmless.
#define LFM_MAX_DEVICES 16
struct LfmSmemConfig { std::atomic<size_t> bytes[LFM_MAX_DEVICES]; };
static inline int lfm_current_device() {
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= LFM_MAX_DEVICES) return -1;
  return dev;
}
template <class Kernel>
static inline cudaError_t lfm_ensure_smem(Kernel kernel, LfmSmemConfig& cfg, size_t bytes) {
  const int dev = lfm_current_device();
  if (dev >= 0 && cfg.bytes[dev].load(std::memory_order_acquire) >= bytes) return cudaSuccess;
  const cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
  if (e == cudaSuccess && dev >= 0) cfg.bytes[dev].store(bytes, std::memory_order_release);
  return e;
}

// Dense block size: every dense matrix is padded to a multiple of LFM_NB rows/cols.
#define LFM_NB 128

static inline int64_t lfm_round_up(int64_t n, int64_t m) { return (n + m - 1) / m * m; }

// theta layout (device, constrained): [d(G), s(G), b(G), l, sigma]
struct LfmTheta {
  const double* d;
  const double* s;
  const double* b;
  const double* l;      // pointer to scalar
  const double* sigma;  // pointer to scalar
};

static inline LfmTheta lfm_theta_view(const double* theta, int G) {
  LfmTheta t;
  t.d = theta;
  t.s = theta + G;
  t.b = theta + 2 * G;
  t.l = theta + 3 * G;
  t.sigma = theta + 3 * G + 1;
  return t;
}

// ---- dense primitives (dgemm.cu / chol.cu) -------------------------------------------------
// C[M x N] = alpha * op(A) op(B) + beta * C, row-major, M,N multiples of 128, K multiple of 16.
// kmode restricts the k-range per output tile (triangular operands; 2 is not a mode):
enum LfmKMode {
  LFM_K_FULL = 0,
  LFM_K_LE_ROW = 1,   // k <  row_tile_end          (A lower-triangular, op(A) = A)
  LFM_K_GE_ROW = 3,   // k >= row_tile_start        (op(A) = A^T with A lower-triangular)
  LFM_K_GE_ROWCOL = 4, // k >= max(row, col) start   (A^T A with A lower-triangular)
  LFM_K_LAUUM_LATE = 5 // as 4 for the tiles of the rows >= k_split (beta = 0); tiles of the rows < k_split ACCUMULATE (beta = 1) over
                       // k >= k_split only: the rest of S = W^T W when S11' = W11^T W11 is already in place (lfm_lauum_late), one launch
};
struct LfmGemm {
  int transA, transB;  // op(A) = A (M x K row-major) or A^T (A stored K x M row-major); same for B (op(B) is K x N;
                       // transB=1 means B stored N x K row-major, i.e. the "NT" form)
  int64_t M, N, K;
  const double* A; int64_t lda;
  const double* B; int64_t ldb;
  double* C; int64_t ldc;
  double alpha, beta;
  int lower_only;      // skip output tiles strictly above the diagonal (requires square tiling of C)
  int kmode;
  int batch;           // > 1: blockIdx.y-th problem uses A + y*strideA, B + y*strideB, C + y*strideC
  int64_t strideA, strideB, strideC;
  int tile = 0;        // 0: heuristic; 1: 16 x 128 tiles (latency-critical 128-row panels on the factorisation chain);
                       // 2: 128 x 128 tiles; 3: 64 x 64 tiles
  int tri_skip = 0;    // lower_only: skip the output tiles of the first `tri_skip` rows of C (the look-ahead chain owns them)
  int64_t k_split = 0; // LFM_K_LAUUM_LATE
  int c_mode = -1;     // set by the launcher from alpha / beta (the kernel must not compare doubles: DSETP shares the FP64 pipe
                       // with the co-resident CTA's DMMAs): 0: beta == 0; 1: general beta; 2 / 3: beta == 1 and alpha == +1 / -1 (C starts in the accumulators, signs by integer XOR)
  long long* stamps = nullptr;   // debug (lfm_debug_syrk_stamps, include/lfm_b200.h): 8 words per CTA -- SM id, clock64 at entry / first unit
                                 // landed / last DMMA issued / stores issued, globaltimer at entry and exit, clock64 when the addresses are set up
  int64_t k_lo = 0, k_hi = ((int64_t)1 << 62);   // k-window: a tile's k-range (after kmode) is clipped to [k_lo, k_hi), multiples of 16;
                       // with beta == 1 a tile whose clipped range is empty is left untouched (K-chunked accumulation)
};
int lfm_dgemm(cudaStream_t st, const LfmGemm& g);

// In-place lower Cholesky of A (n x n, ld, n multiple of 128); writes inverse diagonal blocks
// (and, through the recursion, nothing else) into W's diagonal blocks.  info (device int) receives
// 0 or the 1-based failing pivot.
int lfm_potrf(cudaStream_t st, int64_t n, double* A, int64_t lda, double* W, int64_t ldw, int* info);
// lfm_potrf followed by lfm_trtri, interleaved on three streams when the matrix is a single right-looking sweep.
int lfm_potrf_trtri(cudaStream_t st, int64_t n, double* A, int64_t lda, double* W, int64_t ldw, int* info);
// W = L^-1 (lower) given L and the inverse diagonal blocks already in W's diagonal.
int lfm_trtri(cudaStream_t st, int64_t n, const double* L, int64_t ldl, double* W, int64_t ldw);
// lfm_potrf_trtri that also returns diag(L) in `ldiag` (n doubles) and may start S = W^T W early: *early_done = 1 means the
// top-left half block of A (lower) holds W11^T W11 instead of L11 and the caller must finish with lfm_lauum_late(S = A).
// `chain_ready` (may be NULL; only when lfm_potrf_trtri_is_one_sweep(n) and lda == ldw): an event recorded on `st` when the first two
// block columns (256) of A were complete and *info zeroed, with the rest of A still being written by later work on `st`: the
// dependent chain of the factorisation starts behind the event instead of behind all of it.
bool lfm_potrf_trtri_is_one_sweep(int64_t n);
int lfm_potrf_trtri_diag(cudaStream_t st, int64_t n, double* A, int64_t lda, double* W, int64_t ldw, int* info,
                         double* ldiag, int* early_done, cudaEvent_t chain_ready = nullptr);
int lfm_lauum_late(cudaStream_t st, int64_t n, const double* W, int64_t ldw, double* S, int64_t lds);
// S(lower) = W^T W, out of place.
int lfm_lauum(cudaStream_t st, int64_t n, const double* W, int64_t ldw, double* S, int64_t lds);

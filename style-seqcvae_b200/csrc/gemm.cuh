// bf16 x bf16 -> fp32 "TN" GEMM for sm_100a:  C[M,N] = epilogue( sum_seg A_seg[M,K_seg] * B_seg[N,K_seg]^T )
// Both operands are K-major (row-major with K contiguous), i.e. activations (rows, features) and
// PyTorch-layout weights (out, in). Up to three K-segments accumulate into one TMEM accumulator, so
// a gate pre-activation like  [x_hat|h1|h_dec] W_x^T + z W_z^T  is one launch without concatenating.
#pragma once
#include "common.cuh"

namespace sscvae {

struct GemmSeg {
  const bf16* A; int lda;   // (M, K) row-major, lda in elements (multiple of 8, base 16B aligned)
  const bf16* B; int ldb;   // (N, K) row-major
  int K;
};

// Row-wise softmax statistics / cross-entropy gradient in the epilogue of the vocabulary head GEMM, so that the (rows, V)
// fp32 logits are never written (north_star kernel #3; updown_captioner.py:450, 457-466). The GEMM runs on the 128 x 128
// tile kernel; a thread owns one output row and sees the tile's 128 logits of that row.
//   mode 1: per (row, 128-column tile tn) partial  max / sum exp(x - max) / arg max (lowest index wins)  at
//           [tn * M + row]; if `target` is given, the target's logit goes to tgt_logit[row]. gemm_rowstats_tiles(N) tiles.
//   mode 2: the logit x is replaced by  gcoef[row] * (exp(x - lse[row]) - [n == target[row]])  before the normal store
//           (the bf16 d logits operand of the BPTT head GEMMs).
struct RowStatsEpi {
  int mode = 0;
  float* st_max = nullptr; float* st_sum = nullptr; int* st_arg = nullptr;
  const int* target = nullptr; float* tgt_logit = nullptr;
  const float* lse = nullptr; const float* gcoef = nullptr;
};
inline int gemm_rowstats_tiles(int N) { return (N + 127) / 128; }

struct GemmEpi {
  float alpha = 1.0f;                                  // v = alpha * acc
  const float* bias = nullptr;                         // v += bias[n]
  const float* add1 = nullptr; int ld1 = 0;            // v += add1[m, n]   (only for n < add1_cols)
  int add1_cols = 0x7fffffff;
  const float* add2 = nullptr; int ld2 = 0;            // v += add2[m, n]
  int act = 0;                                         // 1: v = tanh(v)
  const float* dtanh = nullptr; int ldd = 0;           // v *= 1 - dtanh[m,n]^2
  float* C32 = nullptr; int ldc32 = 0; int accumulate = 0;   // C32[m,n] (+)= v
  bf16* C16 = nullptr; int ldc16 = 0;                  // C16[m,n] = bf16(v)
  const char* tag = "gemm";                            // kernel class for the optional profiler (prof.cuh)
  // skinny GEMMs (M <= 256) run on the swapped-operand CTA-pair kernel with K split over a thread-block cluster;
  // 0 = the library's choice of kernel and split count, 1..4 = force the CTA-pair kernel with that K split
  // (tools/gemm_bench.py, tests)
  int splits = 0;
  const RowStatsEpi* rs = nullptr;                     // see RowStatsEpi (forces the 128 x 128 tile kernel)
};

// Launches on `stream`; returns 0 or an error code (message via get_error()).
int gemm_bf16_tn(cudaStream_t stream, int M, int N, int nseg, const GemmSeg* segs, const GemmEpi& epi);

// One problem of a grouped launch: C32[M,N] = A[M,K] * B[N,K]^T, a plain fp32 store (ldc32 in floats, any value).
struct GemmProblem {
  const bf16* A; int lda;
  const bf16* B; int ldb;
  int K, M, N;
  float* C32; int ldc32;
};
constexpr int kMaxGemmProblems = 8;

// Up to kMaxGemmProblems independent problems in ONE launch of the CTA-pair tile kernel (256 x 128 tiles), the tiles of
// the longest-K problem first; reported to the profiler under `tag`. nprob == 0 launches nothing.
int gemm_bf16_tn_grouped(cudaStream_t stream, int nprob, const GemmProblem* probs, const char* tag);

// cuTensorMapEncodeTiled resolved through the runtime (null if the driver does not export it)
void* tma_encode_fn();

// number of kernels launched by this translation unit since load (bench.py's gpu_launches)
extern unsigned long long g_launch_count;

}  // namespace sscvae

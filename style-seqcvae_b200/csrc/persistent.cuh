// Engine of the two persistent CTA-pair kernels (recurrent_fwd.cu, recurrent_bwd.cu): CTA layout, bounded waits, dataflow
// signals, the GEMM operand ring with its TMA producer and MMA issuer loops, and the host side of the launch.
// Per translation unit, like attention_dev.cuh whose ring constants it sets: the including file defines PK_NAME, the
// kernel name in the abort and error messages. Its Params type provides `flags`, `timeout_ns` and ABORT_FLAG.
#pragma once
#define ATT_TID0 64
#define ATT_STAGES_N 2
#define ATT_STAGE_BYTES_N 32768
#include "kernels.cuh"
#include "gemm.cuh"
#include "prof.cuh"
#include "ptx.cuh"
#include "tc_ptx.cuh"
#include "attention_dev.cuh"
#include <cuda.h>
#include <algorithm>
#include <vector>

namespace sscvae {

using namespace attn;

namespace {

// Warp 0: TMA producer of the GEMM operand ring (both CTAs of the pair); warp 1: MMA issuer (leader CTA); warps 2-9:
// compute (epilogues, pointwise stages, attention consumers; named barriers 1 and 2); warp 10: attention producer.
constexpr int PK_CWARPS = 8;
constexpr int PK_THREADS = 32 * (2 + PK_CWARPS + 1);
constexpr int PK_CTHREADS = 32 * PK_CWARPS;
static_assert(PK_CTHREADS == ATT_CONSUMERS, "the compute warps are the attention consumers");
constexpr int PK_X_BYTES = 128 * 64 * 2;                       // activation tile: 128 batch rows x 64 k (bf16)
constexpr int PK_W_BYTES = 64 * 64 * 2;                        // weight tile half: <= 64 rows x 64 k
constexpr int PK_STAGE_BYTES = PK_X_BYTES + PK_W_BYTES;
constexpr int PK_TMEM_COLS = 512;

// ---- bounded waits: on a timeout (or another thread's abort) raise the abort flag, print the wait that failed, trap ----
template <class P>
__device__ __noinline__ void pk_abort(const P& p, int code, int step, unsigned int have, unsigned int want) {
  if (atomicExch(&p.flags[P::ABORT_FLAG], 1u) == 0u)
    printf("[sscvae " PK_NAME "] wait timed out: cta %d thread %d code %d step %d have %u want %u\n", (int)blockIdx.x,
           (int)threadIdx.x, code, step, have, want);
  __threadfence();
  __trap();
}
template <class P>
__device__ __forceinline__ void wait_flag(const P& p, int flag, unsigned int target, int code, int step) {
  const unsigned int* f = p.flags + flag;
  unsigned long long t0 = 0;
  int n = 0;
  for (;;) {
    const unsigned int v = ld_acquire_u32(f);
    if ((int)(v - target) >= 0) return;
    if ((++n & 255) == 0) {
      const unsigned long long now = globaltimer_ns();
      if (t0 == 0) t0 = now;
      if (now - t0 > p.timeout_ns || ld_acquire_u32(p.flags + P::ABORT_FLAG)) pk_abort(p, code, step, v, target);
    }
  }
}
template <class P>
__device__ __forceinline__ void mbar_wait_bounded(const P& p, uint64_t* bar, uint32_t parity, int code, int step) {
  unsigned long long t0 = 0;
  int n = 0;
  while (!mbar_try_wait(bar, parity)) {
    if ((++n & 1023) == 0) {
      const unsigned long long now = globaltimer_ns();
      if (t0 == 0) t0 = now;
      if (now - t0 > p.timeout_ns || ld_acquire_u32(p.flags + P::ABORT_FLAG)) pk_abort(p, code, step, 0, parity);
    }
  }
}

// The compute warps signal "my part of tensor X of this step is in global memory". No per-thread membar.gl: the CTA
// barrier orders the threads' stores before thread 0's gpu-scope release (cumulativity; the pattern of cooperative-groups
// grid sync). Measured: recurrent_fwd 1.66 -> 1.57 ms, recurrent_bwd 2.26 -> 2.11 ms. `tma`: the consumers read the
// tensor through TMA (async proxy).
template <class P>
__device__ __forceinline__ void signal_done(const P& p, int flag, int ctid, bool tma = true) {
  if (tma) fence_proxy_async_global();
  ptx::bar_sync(2, PK_CTHREADS);
  if (ctid == 0) red_release_add(p.flags + flag, 1u);
}

// ---- GEMM operand ring -------------------------------------------------------------------------------------------
// Shared memory: STAGES x (X | W) tiles, the attention's region (attention_dev.cuh: carve), the ring and accumulator
// barriers, the TMEM base and this pair's jobs.
template <class Job, int STAGES, int SLOTS>
struct PkSmem {
  uint8_t* ring;           // STAGES x (X | W)
  uint8_t* att;            // attention region
  uint64_t* full;          // [STAGES]   TMA -> MMA (leader CTA's barrier collects both CTAs' bytes)
  uint64_t* empty;         // [STAGES]   MMA -> TMA (multicast commit)
  uint64_t* tfull;         // [SLOTS]    accumulator complete -> epilogue
  uint32_t* tmem_slot;
  Job* jobs;
  int* njobs;

  static size_t bytes(size_t att_bytes, int max_jobs) {
    return 1024 + (size_t)STAGES * PK_STAGE_BYTES + ((att_bytes + 127) & ~size_t(127)) + (2 * STAGES + SLOTS) * 8 + 16 +
           max_jobs * sizeof(Job) + 64;
  }
  __device__ __forceinline__ static PkSmem carve(uint8_t* smem, size_t att_bytes) {
    PkSmem sm;
    sm.ring = smem;
    sm.att = smem + STAGES * PK_STAGE_BYTES;
    sm.full = reinterpret_cast<uint64_t*>(sm.att + ((att_bytes + 127) & ~size_t(127)));
    sm.empty = sm.full + STAGES;
    sm.tfull = sm.empty + STAGES;
    sm.tmem_slot = reinterpret_cast<uint32_t*>(sm.tfull + SLOTS);
    sm.njobs = reinterpret_cast<int*>(sm.tmem_slot + 1);
    sm.jobs = reinterpret_cast<Job*>(sm.tmem_slot + 4);
    return sm;
  }
  __device__ __forceinline__ void init_barriers() const {
    for (int s = 0; s < STAGES; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], 1); }
    for (int s = 0; s < SLOTS; ++s) mbar_init(&tfull[s], 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
};

// position of the producer / the MMA issuer in the ring
template <int STAGES>
struct RingPos {
  int stage = 0;
  uint32_t phase = 0;
  __device__ __forceinline__ void advance() {
    if (++stage == STAGES) { stage = 0; phase ^= 1; }
  }
};

// TMA producer, one K segment of a job. The weight tiles do not depend on any flag: they are pulled into L2 while the
// activations they multiply are still being produced (the ring alone keeps only STAGES tiles in flight, which left the
// weight stream HBM-latency bound: ~0.4 us per k-block). `ready()` waits for the activations. Then per k-block: the
// activation tile (K column acol0 + 64 kb, this CTA's 128 batch rows, time index t_act) and the weight tile (evict_first).
template <class P, class Smem, int STAGES, class Ready>
__device__ __forceinline__ void produce_segment(const P& p, const Smem& sm, RingPos<STAGES>& pos, int step, int rank, uint32_t tx,
                                                uint64_t w_pol, const CUtensorMap* amap, int acol0, int t_act,
                                                const CUtensorMap* wmap, int wcol0, int w_row, int kblocks, Ready ready) {
  for (int kb = 0; kb < kblocks; ++kb) tma_prefetch_2d(wmap, wcol0 + kb * 64, w_row);
  ready();
  for (int kb = 0; kb < kblocks; ++kb) {
    mbar_wait_bounded(p, &sm.empty[pos.stage], pos.phase ^ 1, 1, step);
    if (rank == 0) mbar_expect_tx(&sm.full[pos.stage], tx);
    uint8_t* xs = sm.ring + (size_t)pos.stage * PK_STAGE_BYTES;
    tma_load_3d_2sm(xs, amap, &sm.full[pos.stage], acol0 + kb * 64, rank * 128, t_act);
    tma_load_2d_2sm_hint(xs + PK_X_BYTES, wmap, &sm.full[pos.stage], wcol0 + kb * 64, w_row, w_pol);
    pos.advance();
  }
}

// MMA issuer, one job: all k-blocks of its segments into the accumulator at tacc (M = 256: both CTAs' rows), then the
// "accumulator ready" commit on barrier `slot` of both CTAs.
template <class P, class Smem, int STAGES, class Job>
__device__ __forceinline__ void mma_job(const P& p, const Smem& sm, RingPos<STAGES>& pos, int step, const Job& job, uint32_t tacc,
                                        int slot) {
  const uint32_t idesc = make_idesc(256, job.N);
  bool first = true;
  for (int s = 0; s < job.nseg; ++s) {
    const int kbs = job.seg[s].kblocks;
    for (int kb = 0; kb < kbs; ++kb) {
      mbar_wait_bounded(p, &sm.full[pos.stage], pos.phase, 2, step);
      tc_fence_after();
      const uint32_t x_base = smem_u32(sm.ring + (size_t)pos.stage * PK_STAGE_BYTES);
      const uint32_t w_base = x_base + PK_X_BYTES;
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        umma_bf16_2sm(tacc, make_smem_desc(x_base + k * 32), make_smem_desc(w_base + k * 32), idesc, first ? 0u : 1u);
        first = false;
      }
      umma_commit_2sm(&sm.empty[pos.stage]);
      pos.advance();
    }
  }
  umma_commit_2sm(&sm.tfull[slot]);
}

// end of the kernel: nobody deallocates while the pair's MMAs / loads are in flight
__device__ __forceinline__ void pk_teardown(int warp, uint32_t tmem_base) {
  tc_fence_before();
  cluster_sync_all();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc_2sm<PK_TMEM_COLS>(tmem_base);
  }
}

// ---------------------------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

// activation (k, batch row, t) of a time-major bf16 tensor with row stride ld: box 64 x 128 x 1, 128B swizzle
static int encode_act3d(CUtensorMap* out, const bf16* base, int K, int B, int T, int ld) {
  EncodeTiledFn fn = reinterpret_cast<EncodeTiledFn>(tma_encode_fn());
  if (!fn) { set_error("cuTensorMapEncodeTiled not available from the driver"); return SSCVAE_ERR_DRIVER; }
  cuuint64_t dims[3] = {(cuuint64_t)K, (cuuint64_t)B, (cuuint64_t)T};
  cuuint64_t strides[2] = {(cuuint64_t)ld * 2, (cuuint64_t)B * ld * 2};
  cuuint32_t box[3] = {64, 128, 1};
  cuuint32_t estr[3] = {1, 1, 1};
  CUresult r = fn(out, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, const_cast<bf16*>(base), dims, strides, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) { set_error(PK_NAME ": activation tensor map failed (%d) K=%d B=%d T=%d ld=%d", (int)r, K, B, T, ld); return SSCVAE_ERR_DRIVER; }
  return 0;
}
// weight (k, row): box 64 x box_rows, 128B swizzle
static int encode_w2d(CUtensorMap* out, const bf16* base, int K, int rows, int ld, int box_rows) {
  EncodeTiledFn fn = reinterpret_cast<EncodeTiledFn>(tma_encode_fn());
  if (!fn) { set_error("cuTensorMapEncodeTiled not available from the driver"); return SSCVAE_ERR_DRIVER; }
  cuuint64_t dims[2] = {(cuuint64_t)K, (cuuint64_t)rows};
  cuuint64_t strides[1] = {(cuuint64_t)ld * 2};
  cuuint32_t box[2] = {64, (cuuint32_t)box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = fn(out, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<bf16*>(base), dims, strides, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) { set_error(PK_NAME ": weight tensor map failed (%d) K=%d rows=%d ld=%d box=%d", (int)r, K, rows, ld, box_rows); return SSCVAE_ERR_DRIVER; }
  return 0;
}

// CTA pairs of `kernel` that can be co-resident with `smem` bytes of dynamic shared memory (0 on failure); cached
template <class P>
static int pk_grid_pairs(void (*kernel)(P), size_t smem) {
  static int cached = -1;
  static size_t cached_smem = 0;
  if (cached >= 0 && cached_smem == smem) return cached;
  int dev = 0, n_sm = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess) return 0;
  if (cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess) {
    cudaGetLastError();
    return 0;
  }
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(2 * (n_sm / 2)); cfg.blockDim = dim3(PK_THREADS); cfg.dynamicSmemBytes = smem;
  int clusters = 0;
  if (cudaOccupancyMaxActiveClusters(&clusters, kernel, &cfg) != cudaSuccess) { cudaGetLastError(); clusters = 0; }
  cached = std::min(clusters, n_sm / 2);
  cached_smem = smem;
  return cached;
}

// every wait of both kernels gives up after SSCVAE_RF_TIMEOUT_MS (default 4 s)
static unsigned long long pk_timeout_ns() {
  static const unsigned long long ms = [] { const char* e = getenv("SSCVAE_RF_TIMEOUT_MS"); return e ? (unsigned long long)atoll(e) : 4000ull; }();
  return ms * 1000000ull;
}

// cooperative launch: all 2 * pairs CTAs are co-resident, which the dataflow counters rely on
template <class P>
static int pk_launch(void (*kernel)(P), int pairs, size_t smem, cudaStream_t s, const P& p) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(2 * pairs); cfg.blockDim = dim3(PK_THREADS); cfg.dynamicSmemBytes = smem; cfg.stream = s;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeCooperative;
  attr[0].val.cooperative = 1;
  cfg.attrs = attr; cfg.numAttrs = 1;
  CUDA_TRY(cudaLaunchKernelEx(&cfg, kernel, p));
  ++g_launch_count;
  return 0;
}

// Phase stamps (SSCVAE_RF_DBG=1 / SSCVAE_RB_DBG=1): 32 globaltimer stamps per CTA of one step, written by the kernel.
constexpr size_t PK_DBG_BYTES = 32 * 8 * 2 * 128;
// *buf = the zeroed stamp buffer, allocated on first use
static int pk_dbg_begin(cudaStream_t s, unsigned long long** buf) {
  static unsigned long long* dbg_buf = nullptr;
  if (!dbg_buf) CUDA_TRY(cudaMalloc(&dbg_buf, PK_DBG_BYTES));
  CUDA_TRY(cudaMemsetAsync(dbg_buf, 0, PK_DBG_BYTES, s));
  *buf = dbg_buf;
  return 0;
}
// after the launch: the first `nstamps` stamps of the CTAs in `show`, in us from the earliest stamp 0 of any CTA, on
// stderr as "<head> cta=<c>: i:us ..." (first 6 launches)
static int pk_dbg_print(cudaStream_t s, const unsigned long long* buf, int nctas, const char* head, const std::vector<int>& show,
                        int nstamps) {
  static int printed = 0;
  CUDA_TRY(cudaStreamSynchronize(s));
  std::vector<unsigned long long> h(32 * (size_t)nctas);
  CUDA_TRY(cudaMemcpy(h.data(), buf, h.size() * 8, cudaMemcpyDeviceToHost));
  if (printed++ >= 6) return 0;
  unsigned long long t0 = ~0ull;
  for (int c = 0; c < nctas; ++c) if (h[c * 32] && h[c * 32] < t0) t0 = h[c * 32];
  for (int c : show) {
    if (c < 0 || c >= nctas) continue;
    fprintf(stderr, "%s cta=%3d:", head, c);
    for (int i = 0; i < nstamps; ++i) fprintf(stderr, " %d:%.1f", i, h[c * 32 + i] ? (double)(h[c * 32 + i] - t0) / 1e3 : -1.0);
    fprintf(stderr, "\n");
  }
  return 0;
}

}  // namespace

}  // namespace sscvae

// tcgen05 / TMEM / TMA GEMM for sm_100a (see gemm.cuh for the contract).
//
// Three kernels: the tile kernel (one CTA per 128 x BN output tile), the CTA-pair tile kernel (a 2-CTA cluster per
// 256 x BN tile) and the swapped-operand CTA-pair kernel of the skinny GEMMs. All three share one pipeline
// (GemmSmem, gemm_setup, gemm_produce, gemm_mma, gemm_teardown), single-CTA or CTA-pair by a template parameter:
//   warp 0      : TMA producer  (cp.async.bulk.tensor.2d, 128B-swizzled K-major tiles, mbarrier ring)
//   warp 1      : TMEM allocator + single-thread tcgen05.mma issuer (kind::f16, bf16 in, fp32 accum in TMEM)
//   warps 2..5  : epilogue: tcgen05.ld (32 lanes x 32 columns per instruction) -> registers ->
//                 fused bias / addends / tanh / dtanh -> fp32 and/or bf16 global stores
// The accumulator never touches registers or shared memory until the epilogue. The two tile kernels share their
// epilogue column loop (epilogue_tile); the swapped-pair kernel reduces its K splits through distributed shared memory
// and has its own epilogue.
#include "gemm.cuh"
#include "prof.cuh"
#include "ptx.cuh"
#include "tc_ptx.cuh"
#include <cuda.h>
#include <algorithm>
#include <cstring>
#include <mutex>
#include <unordered_map>

namespace sscvae {

unsigned long long g_launch_count = 0;

static constexpr int BM = 128;
static constexpr int BK = 64;                    // 64 bf16 = 128 bytes = one swizzle-128B row
static constexpr int A_STAGE_BYTES = BM * BK * 2;
static constexpr int GEMM_THREADS = 192;
static constexpr int MAX_SEG = 3;

struct GemmParams {
  CUtensorMap ta[MAX_SEG];
  CUtensorMap tb[MAX_SEG];
  int kblocks[MAX_SEG];
  int nseg;
  int M, N;
  int vec;                                        // 1: every epilogue pointer allows 16-byte access
  int splits;                                     // pair kernel: K split = cluster z = gridDim.z
  int kb_per_split;                               // pair kernel: CTA z works on k-blocks [z*kb_per_split, ...) of the
                                                  // concatenated segments
  int tma_store;                                  // 1: plain fp32 tile (+bias): the epilogue leaves through TMA stores of `tc`
  CUtensorMap tc;                                 // fp32 output, box 32 columns x 32 rows, no swizzle
  GemmEpi epi;
  RowStatsEpi rs;                                 // vocabulary head: softmax statistics / CE gradient in the epilogue
};

// ---------------------------------------------------------------------------------------------
// epilogue math for one run of 32 consecutive columns of one row
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ float tanh_fast(float x) {
  // accurate enough for fp32 parity: tanhf via exp; the MUFU.TANH approximation is reserved for the
  // attention kernel's 27k tanh/row where the operands are bf16 anyway.
  return tanhf(x);
}

// explicit shared-memory accesses (32-bit shared addresses): pointers derived from the aligned dynamic-smem base are
// treated as generic by the compiler, and generic LD/ST that resolve to shared memory are several times slower than
// LDS/STS for a lone epilogue warp
__device__ __forceinline__ void sts_f32(uint32_t a, float v) { asm volatile("st.shared.f32 [%0], %1;" ::"r"(a), "f"(v) : "memory"); }
__device__ __forceinline__ void sts_v4(uint32_t a, const float4& v) {
  asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(a), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}
__device__ __forceinline__ float lds_f32(uint32_t a) {
  float v;
  asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(a) : "memory");
  return v;
}
__device__ __forceinline__ float4 lds_v4(uint32_t a) {
  float4 v;
  asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(a) : "memory");
  return v;
}

// Second half of the vector epilogue: the warp's 32x32 fp32 block sits in `stage` as [row][column] (pitch 36 floats);
// 8 consecutive lanes own 32 consecutive columns of ONE output row (128 contiguous bytes), 4 rows per instruction,
// for the addend loads and for the stores.
// NOTE: GemmEpi is taken BY VALUE everywhere in the epilogue. Through a reference to the __grid_constant__ kernel
// parameter the compiler must assume the output stores alias the struct and re-reads every field after each store
// (measured: ~250 cycles per store, 2-3.4k cycles per 32x32 block instead of ~300).
__device__ __forceinline__ void epilogue_block_vec(const GemmEpi e, int M, int row0, int col0, uint32_t stage,
                                                   bool add1_all) {
  constexpr int PITCH = 36;
  const int lane = threadIdx.x & 31;
  const int c4 = (lane & 7) * 4;
  const int n = col0 + c4;
  float4 bias4 = make_float4(0.f, 0.f, 0.f, 0.f);
  if (e.bias) bias4 = *reinterpret_cast<const float4*>(e.bias + n);
  // The epilogue warps run one per SM sub-partition, so the epilogue is bound by its own instruction count
  // (measured: 3.4k cycles per 32x32 block when the tanh / dtanh / accumulate forms were compiled into the one loop).
  // The common case - scaled accumulator + bias + addends -> fp32 and/or bf16 - gets its own lean loop.
  if (!e.act && !e.dtanh && !e.accumulate) {
    const float alpha = e.alpha;
    const float* a1 = add1_all ? e.add1 + n : nullptr;
    const float* a2 = e.add2 ? e.add2 + n : nullptr;
    float* c32 = e.C32 ? e.C32 + n : nullptr;
    bf16* c16 = e.C16 ? e.C16 + n : nullptr;
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      const int rr = k * 4 + (lane >> 3);
      const int r = row0 + rr;
      if (r < M) {
        float4 v = lds_v4(stage + (rr * PITCH + c4) * 4);
        v.x = fmaf(v.x, alpha, bias4.x); v.y = fmaf(v.y, alpha, bias4.y);
        v.z = fmaf(v.z, alpha, bias4.z); v.w = fmaf(v.w, alpha, bias4.w);
        if (a1) {
          const float4 b = *reinterpret_cast<const float4*>(a1 + (size_t)r * e.ld1);
          v.x += b.x; v.y += b.y; v.z += b.z; v.w += b.w;
        }
        if (a2) {
          const float4 b = *reinterpret_cast<const float4*>(a2 + (size_t)r * e.ld2);
          v.x += b.x; v.y += b.y; v.z += b.z; v.w += b.w;
        }
        if (c32) *reinterpret_cast<float4*>(c32 + (size_t)r * e.ldc32) = v;
        if (c16) {
          __nv_bfloat162 lo = __floats2bfloat162_rn(v.x, v.y), hi = __floats2bfloat162_rn(v.z, v.w);
          uint2 o;
          o.x = *reinterpret_cast<uint32_t*>(&lo);
          o.y = *reinterpret_cast<uint32_t*>(&hi);
          *reinterpret_cast<uint2*>(c16 + (size_t)r * e.ldc16) = o;
        }
      }
    }
    return;
  }
#pragma unroll
  for (int k = 0; k < 8; ++k) {
    const int rr = k * 4 + (lane >> 3);
    const int r = row0 + rr;
    if (r < M) {
      float4 v = lds_v4(stage + (rr * PITCH + c4) * 4);
      v.x = v.x * e.alpha + bias4.x; v.y = v.y * e.alpha + bias4.y;
      v.z = v.z * e.alpha + bias4.z; v.w = v.w * e.alpha + bias4.w;
      if (add1_all) {
        const float4 b = *reinterpret_cast<const float4*>(e.add1 + (size_t)r * e.ld1 + n);
        v.x += b.x; v.y += b.y; v.z += b.z; v.w += b.w;
      }
      if (e.add2) {
        const float4 b = *reinterpret_cast<const float4*>(e.add2 + (size_t)r * e.ld2 + n);
        v.x += b.x; v.y += b.y; v.z += b.z; v.w += b.w;
      }
      if (e.act == 1) { v.x = tanh_fast(v.x); v.y = tanh_fast(v.y); v.z = tanh_fast(v.z); v.w = tanh_fast(v.w); }
      if (e.dtanh) {
        const float4 t = *reinterpret_cast<const float4*>(e.dtanh + (size_t)r * e.ldd + n);
        v.x *= 1.0f - t.x * t.x; v.y *= 1.0f - t.y * t.y; v.z *= 1.0f - t.z * t.z; v.w *= 1.0f - t.w * t.w;
      }
      if (e.C32) {
        float* p = e.C32 + (size_t)r * e.ldc32 + n;
        if (e.accumulate) {
          const float4 c = *reinterpret_cast<const float4*>(p);
          v.x += c.x; v.y += c.y; v.z += c.z; v.w += c.w;
        }
        *reinterpret_cast<float4*>(p) = v;
      }
      if (e.C16) {
        __nv_bfloat162 lo = __floats2bfloat162_rn(v.x, v.y), hi = __floats2bfloat162_rn(v.z, v.w);
        uint2 o;
        o.x = *reinterpret_cast<uint32_t*>(&lo);
        o.y = *reinterpret_cast<uint32_t*>(&hi);
        *reinterpret_cast<uint2*>(e.C16 + (size_t)r * e.ldc16 + n) = o;
      }
    }
  }
}

// Plain fp32 tile (+ bias): the warp's 32x32 block goes to shared memory as 32 rows of 128 bytes in the TMA
// 128B-swizzle pattern (16-byte chunk c of row r at chunk c ^ (r & 7): 4-way instead of 32-way bank conflicts for
// lane == row) and leaves with ONE asynchronous TMA store; rows / columns beyond the matrix are clipped by the TMA
// unit. Plain STG.128 stores cost a lone epilogue warp ~220 cycles each (1.8k cycles per block, measured).
__device__ __forceinline__ void epilogue_tma_row32(const GemmEpi e, const CUtensorMap* tc, int N, int row0, int col0,
                                                   const uint32_t (&acc)[32], uint32_t stage) {
  const int lane = threadIdx.x & 31;
  if (lane == 0) tma_store_wait_read();                  // the previous store has finished reading this buffer
  __syncwarp();
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    float4 b = make_float4(0.f, 0.f, 0.f, 0.f);
    if (e.bias && col0 + 4 * j + 3 < N) b = *reinterpret_cast<const float4*>(e.bias + col0 + 4 * j);
    else if (e.bias) {
      if (col0 + 4 * j < N) b.x = e.bias[col0 + 4 * j];
      if (col0 + 4 * j + 1 < N) b.y = e.bias[col0 + 4 * j + 1];
      if (col0 + 4 * j + 2 < N) b.z = e.bias[col0 + 4 * j + 2];
    }
    const float4 v = make_float4(fmaf(__uint_as_float(acc[4 * j]), e.alpha, b.x), fmaf(__uint_as_float(acc[4 * j + 1]), e.alpha, b.y),
                                 fmaf(__uint_as_float(acc[4 * j + 2]), e.alpha, b.z), fmaf(__uint_as_float(acc[4 * j + 3]), e.alpha, b.w));
    sts_v4(stage + lane * 128 + ((j ^ (lane & 7)) << 4), v);
  }
  fence_proxy_async_smem();
  __syncwarp();
  if (lane == 0) tma_store_2d(tc, stage, col0, row0);
}

__device__ __forceinline__ void epilogue_row32(const GemmEpi e, int vec, int M, int N, int row0, int col0, int ncols,
                                               const uint32_t (&acc)[32], uint32_t stage) {
  const int lane = threadIdx.x & 31;
  const int row = row0 + lane;           // TMEM lane == output row of this thread's 32 accumulator columns
  // `ncols` < 32 only for the narrow (BN=16) tiles; add1 may cover just the first add1_cols columns
  const bool add1_all = e.add1 && (col0 + 32 <= e.add1_cols);
  const bool add1_none = !e.add1 || (col0 >= e.add1_cols);
  const bool full = (ncols == 32) && (col0 + 32 <= N) && (add1_all || add1_none);
  if (vec && full) {
    // Transpose the warp's 32x32 fp32 block through shared memory (the pipeline's stage buffers are free by
    // now) so that global traffic is coalesced: afterwards 8 consecutive lanes own 32 consecutive columns of
    // ONE row (128 contiguous bytes), 4 rows per instruction, for the addend loads and for the stores.
    constexpr int PITCH = 36;            // floats; keeps float4 alignment
#pragma unroll
    for (int j = 0; j < 8; ++j)
      sts_v4(stage + (lane * PITCH + 4 * j) * 4,
             make_float4(__uint_as_float(acc[4 * j]), __uint_as_float(acc[4 * j + 1]), __uint_as_float(acc[4 * j + 2]),
                         __uint_as_float(acc[4 * j + 3])));
    __syncwarp();
    epilogue_block_vec(e, M, row0, col0, stage, add1_all);
    __syncwarp();
    return;
  }
  if (row >= M) return;
  float v[32];
#pragma unroll
  for (int j = 0; j < 32; ++j) v[j] = __uint_as_float(acc[j]) * e.alpha;
  // scalar path (ragged right edge or unaligned pointers, e.g. gradients written straight into
  // a column block of a reference-layout weight matrix)
#pragma unroll
  for (int j = 0; j < 32; ++j) {
    const int n = col0 + j;
    if (n < N && j < ncols) {
      float x = v[j];
      if (e.bias) x += e.bias[n];
      if (e.add1 && n < e.add1_cols) x += e.add1[(size_t)row * e.ld1 + n];
      if (e.add2) x += e.add2[(size_t)row * e.ld2 + n];
      if (e.act == 1) x = tanh_fast(x);
      if (e.dtanh) { float t = e.dtanh[(size_t)row * e.ldd + n]; x *= 1.0f - t * t; }
      if (e.C32) {
        float* p = e.C32 + (size_t)row * e.ldc32 + n;
        *p = e.accumulate ? (*p + x) : x;
      }
      if (e.C16) e.C16[(size_t)row * e.ldc16 + n] = __float2bfloat16_rn(x);
    }
  }
}

// ---------------------------------------------------------------------------------------------
// the pipeline shared by the three kernels: shared-memory ring, setup, TMA producer, MMA issuer, teardown
// ---------------------------------------------------------------------------------------------
// Dynamic shared memory: STAGES slot-0 tiles, STAGES slot-1 tiles, the ring's full / empty barriers, the accumulator
// barrier and the TMEM base. bytes() is what the launcher requests (1024 bytes of alignment slack, 256 for the barriers).
template <int STAGES, int BYTES0, int BYTES1>
struct GemmSmem {
  static constexpr int kStages = STAGES, kBytes0 = BYTES0, kBytes1 = BYTES1;
  static_assert((2 * STAGES + 1) * 8 + 4 <= 256, "barriers and TMEM slot exceed their 256 bytes");
  uint8_t* s0;             // [STAGES][BYTES0]
  uint8_t* s1;             // [STAGES][BYTES1]
  uint64_t* full;          // [STAGES]   TMA -> MMA
  uint64_t* empty;         // [STAGES]   MMA -> TMA
  uint64_t* accum;         // accumulator complete -> epilogue
  uint32_t* tmem_slot;

  static constexpr int bytes() { return 1024 + STAGES * (BYTES0 + BYTES1) + 256; }
  // `smem`: the kernel's extern __shared__ __align__(1024) array; the 128B swizzle needs 1024-byte aligned tiles
  __device__ __forceinline__ static GemmSmem carve(uint8_t* smem) {
    if (threadIdx.x == 0 && (smem_u32(smem) & 1023u)) __trap();
    GemmSmem sm;
    sm.s0 = smem;
    sm.s1 = smem + STAGES * BYTES0;
    sm.full = reinterpret_cast<uint64_t*>(sm.s1 + STAGES * BYTES1);
    sm.empty = sm.full + STAGES;
    sm.accum = sm.empty + STAGES;
    sm.tmem_slot = reinterpret_cast<uint32_t*>(sm.accum + 1);
    return sm;
  }
  __device__ __forceinline__ void init_barriers() const {
    for (int s = 0; s < STAGES; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], 1); }
    mbar_init(accum, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
};

template <int BN, int STAGES> using TileSmem = GemmSmem<STAGES, A_STAGE_BYTES, BN * BK * 2>;
template <int BN, int STAGES> using PairTileSmem = GemmSmem<STAGES, A_STAGE_BYTES, BN / 2 * BK * 2>;  // half the B tile per CTA
template <int STAGES> using SwappedSmem = GemmSmem<STAGES, 128 * BK * 2, 128 * BK * 2>;              // weights | activations

__device__ __forceinline__ int total_kblocks(const GemmParams& p) {
  int total = 0;
#pragma unroll
  for (int s = 0; s < MAX_SEG; ++s) total += (s < p.nseg) ? p.kblocks[s] : 0;
  return total;
}

// PAIR: the CTA pair of a 2-cluster drives one 256-row tcgen05.mma.cta_group::2; otherwise one CTA, cta_group::1.
// Thread 0 prefetches the operand maps and initialises the barriers, warp 1 allocates the accumulator; returns its TMEM
// address once the CTA (PAIR: both CTAs, so that no remote arrival precedes the peer's barriers) has got this far.
template <bool PAIR, int TMEM_COLS, class Smem>
__device__ __forceinline__ uint32_t gemm_setup(const CUtensorMap* ta, const CUtensorMap* tb, int nseg, const Smem& sm,
                                               int warp) {
  if (threadIdx.x == 0) {
    for (int s = 0; s < nseg; ++s) { prefetch_tmap(&ta[s]); prefetch_tmap(&tb[s]); }
    sm.init_barriers();
  }
  if (warp == 1) {
    if constexpr (PAIR) tmem_alloc_2sm<TMEM_COLS>(sm.tmem_slot);
    else tmem_alloc<TMEM_COLS>(sm.tmem_slot);
  }
  tc_fence_before();
  if constexpr (PAIR) cluster_sync_all();
  else __syncthreads();
  tc_fence_after();
  return *sm.tmem_slot;
}

// TMA producer (one elected thread of warp 0) for k-blocks [kb_begin, kb_end) of the concatenated K segments: per
// k-block the slot-0 tile (map0[s], rows from row0) and the slot-1 tile (map1[s], rows from row1) of its segment s,
// which spans kblocks[s] k-blocks.
// PAIR: both CTAs load and the bytes land on the leader's `full` barrier, which alone expects them.
// EVICT_FIRST0: the slot-0 tiles are loaded with an L2 evict_first hint.
template <bool PAIR, bool EVICT_FIRST0, class Smem>
__device__ __forceinline__ void gemm_produce(const int* kblocks, const Smem& sm, const CUtensorMap* map0, int row0,
                                             const CUtensorMap* map1, int row1, int kb_begin, int kb_end, bool leader) {
  static_assert(PAIR || !EVICT_FIRST0, "the hinted load exists in the CTA-pair form only");
  constexpr uint32_t TX = (PAIR ? 2 : 1) * (Smem::kBytes0 + Smem::kBytes1);
  uint64_t pol = 0;
  if constexpr (EVICT_FIRST0) pol = ptx::l2_policy_evict_first();
  RingPos<Smem::kStages> pos;
  // segment of the current k-block, its first global index and its two maps. The maps are generic addresses fixed once
  // here (the empty asm): otherwise ptxas re-derives them from the kernel-parameter address after the `empty` wait, on
  // the critical path of every k-block (measured: +0.2 us on a 15-k-block tile GEMM).
  int s = 0, base = 0;
  const CUtensorMap* t0 = map0;
  const CUtensorMap* t1 = map1;
  asm volatile("" : "+l"(t0), "+l"(t1));
  for (int g = kb_begin; g < kb_end; ++g) {
    while (g >= base + kblocks[s]) { base += kblocks[s]; ++s; ++t0; ++t1; }
    const int kc = (g - base) * BK;
    uint64_t* bar = &sm.full[pos.stage];
    uint8_t* d0 = sm.s0 + pos.stage * Smem::kBytes0;
    uint8_t* d1 = sm.s1 + pos.stage * Smem::kBytes1;
    mbar_wait(&sm.empty[pos.stage], pos.phase ^ 1);
    if (leader) mbar_expect_tx(bar, TX);
    if constexpr (!PAIR) {
      tma_load_2d(d0, t0, bar, kc, row0);
      tma_load_2d(d1, t1, bar, kc, row1);
    } else {
      if constexpr (EVICT_FIRST0) tma_load_2d_2sm_hint(d0, t0, bar, kc, row0, pol);
      else tma_load_2d_2sm(d0, t0, bar, kc, row0);
      tma_load_2d_2sm(d1, t1, bar, kc, row1);
    }
    pos.advance();
  }
}

// MMA issuer (one elected thread of warp 1; PAIR: of the leader CTA) for k-blocks [kb_begin, kb_end): D = slot-0 tile x
// slot-1 tile^T into the accumulator at tmem_acc. A commit frees each stage once its MMAs have read it, a last one
// reports the accumulator complete. PAIR: the commits arrive on the barriers of the cluster CTAs in `mask`.
template <bool PAIR, class Smem>
__device__ __forceinline__ void gemm_mma(const Smem& sm, uint32_t tmem_acc, uint32_t idesc, int kb_begin, int kb_end,
                                         uint16_t mask = 3) {
  RingPos<Smem::kStages> pos;
  for (int kb = kb_begin; kb < kb_end; ++kb) {
    mbar_wait(&sm.full[pos.stage], pos.phase);
    tc_fence_after();
    const uint32_t a_base = smem_u32(sm.s0 + pos.stage * Smem::kBytes0);
    const uint32_t b_base = smem_u32(sm.s1 + pos.stage * Smem::kBytes1);
#pragma unroll
    for (int k = 0; k < BK / 16; ++k) {
      // advance 16 elements (32 bytes) along K inside the 128B swizzle atom
      const uint64_t ad = make_smem_desc(a_base + k * 32), bd = make_smem_desc(b_base + k * 32);
      const uint32_t accumulate = (kb > kb_begin || k > 0) ? 1u : 0u;
      if constexpr (PAIR) umma_bf16_2sm(tmem_acc, ad, bd, idesc, accumulate);
      else umma_bf16(tmem_acc, ad, bd, idesc, accumulate);
    }
    if constexpr (PAIR) umma_commit_2sm(&sm.empty[pos.stage], mask);
    else umma_commit(&sm.empty[pos.stage]);
    pos.advance();
  }
  if constexpr (PAIR) umma_commit_2sm(sm.accum, mask);
  else umma_commit(sm.accum);
}

// End of the kernel: the epilogue's TMA stores are complete, and nobody deallocates while MMAs, loads or (PAIR) the
// peer's reads of its half of the accumulator are in flight.
template <bool PAIR, int TMEM_COLS>
__device__ __forceinline__ void gemm_teardown(bool tma_store, uint32_t tmem_acc, int warp) {
  if (tma_store && warp >= 2 && (threadIdx.x & 31) == 0) tma_store_wait_all();
  tc_fence_before();
  if constexpr (PAIR) cluster_sync_all();
  else __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    if constexpr (PAIR) tmem_dealloc_2sm<TMEM_COLS>(tmem_acc);
    else tmem_dealloc<TMEM_COLS>(tmem_acc);
  }
}

// Epilogue warps 2..5 of the two tile kernels; a warp may only touch TMEM lanes [32*(warp%4), +32): the tile rows from
// m0 + 32*(warp%4). It walks the tile's columns 32 at a time; each block leaves through TMA stores or epilogue_row32.
// The output is (M, N) through `epi`; tc: the fp32 map of the TMA-store epilogue, null for the other paths (vec: see
// GemmParams). ROW_STATS: the tile kernel's vocabulary-head branch (`rs_p`). smem0: the dead stage buffers.
template <int BN, bool ROW_STATS>
__device__ __forceinline__ void epilogue_tile(const GemmEpi& epi, const RowStatsEpi& rs_p, int M, int N, int vec,
                                              const CUtensorMap* tc, uint32_t tmem_acc, uint64_t* accum, uint32_t smem0,
                                              int m0, int n0) {
  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int q = warp & 3;
  mbar_wait(accum, 0);
  tc_fence_after();
  const int row = m0 + q * 32 + lane;
  // vocabulary head (RowStatsEpi): running softmax statistics of this thread's row over the tile's columns
  const RowStatsEpi rs = ROW_STATS ? rs_p : RowStatsEpi();
  float rs_m = -INFINITY, rs_s = 0.f, rs_t = 0.f; int rs_a = 0x7fffffff;
  int rs_target = -1; float rs_lse = 0.f, rs_g = 0.f;
  if (rs.mode && row < M) {
    if (rs.target) rs_target = rs.target[row];
    if (rs.mode == 2) { rs_lse = rs.lse[row]; rs_g = rs.gcoef[row]; }
  }
#pragma unroll 1
  for (int c0 = 0; c0 < BN; c0 += 32) {
    if (n0 + c0 >= N) break;                 // warp-uniform
    uint32_t acc[32];
    tmem_ld_32x32(tmem_acc + (static_cast<uint32_t>(q * 32) << 16) + c0, acc);
    tmem_ld_wait();
    if (rs.mode) {
      // One warp per SM sub-partition runs this with nothing to hide latency behind: everything is written as
      // independent operations + tree reductions (a running  s += exp(..)  chain cost ~120 cycles per element).
      const int nb = n0 + c0;
      const bool full = nb + 32 <= N;                     // warp-uniform: only the last tile has a ragged edge
      float v[32];
#pragma unroll
      for (int j = 0; j < 32; ++j) v[j] = __uint_as_float(acc[j]) * epi.alpha;
      if (epi.bias) {
#pragma unroll
        for (int j = 0; j < 32; ++j)
          if (full || nb + j < N) v[j] += epi.bias[nb + j];
      }
      if (!full) {
#pragma unroll
        for (int j = 0; j < 32; ++j)
          if (nb + j >= N) v[j] = -INFINITY;              // exp -> 0, never the max
      }
      if (rs.mode == 1) {
        float t[16];
#pragma unroll
        for (int j = 0; j < 16; ++j) t[j] = fmaxf(v[j], v[j + 16]);
#pragma unroll
        for (int w = 8; w > 0; w >>= 1)
#pragma unroll
          for (int j = 0; j < w; ++j) t[j] = fmaxf(t[j], t[j + w]);
        const float cm = t[0];
        if (cm > rs_m) {                       // strict: an earlier column / tile keeps the arg max on ties
#pragma unroll
          for (int j = 31; j >= 0; --j)
            if (v[j] == cm) rs_a = nb + j;
          rs_s *= exp2f((rs_m - cm) * 1.4426950408889634f);
          rs_m = cm;
        }
        const float mb = rs_m * 1.4426950408889634f;
        float e[32];
#pragma unroll
        for (int j = 0; j < 32; ++j) e[j] = exp2f(fmaf(v[j], 1.4426950408889634f, -mb));
#pragma unroll
        for (int w = 16; w > 0; w >>= 1)
#pragma unroll
          for (int j = 0; j < w; ++j) e[j] += e[j + w];
        rs_s += e[0];
        if (rs_target >= nb && rs_target < nb + 32) {
#pragma unroll
          for (int j = 0; j < 32; ++j)
            if (nb + j == rs_target) rs_t = v[j];
        }
        if (!epi.C32 && !epi.C16) continue;      // statistics only: the logits are never written
      } else {
        const float lb = rs_lse * 1.4426950408889634f;
#pragma unroll
        for (int j = 0; j < 32; ++j) acc[j] = __float_as_uint(rs_g * exp2f(fmaf(v[j], 1.4426950408889634f, -lb)));
        if (rs_target >= nb && rs_target < nb + 32) {
#pragma unroll
          for (int j = 0; j < 32; ++j)
            if (nb + j == rs_target) acc[j] = __float_as_uint(__uint_as_float(acc[j]) - rs_g);
        }
        GemmEpi e2 = epi;
        e2.alpha = 1.f; e2.bias = nullptr;
        epilogue_row32(e2, vec, M, N, m0 + q * 32, n0 + c0, BN - c0 < 32 ? BN - c0 : 32, acc,
                       smem0 + (warp - 2) * 32 * 36 * 4);
        continue;
      }
    }
    if (BN >= 32 && tc) {
      epilogue_tma_row32(epi, tc, N, m0 + q * 32, n0 + c0, acc, smem0 + (warp - 2) * 4096);
    } else {
      epilogue_row32(epi, vec, M, N, m0 + q * 32, n0 + c0, BN - c0 < 32 ? BN - c0 : 32, acc,
                     smem0 + (warp - 2) * 32 * 36 * 4);
    }
  }
  if (rs.mode == 1 && row < M) {             // partial statistics of (row, this 128-column tile): lanes = consecutive rows
    const size_t o = (size_t)blockIdx.x * M + row;
    rs.st_max[o] = rs_m; rs.st_sum[o] = rs_s; rs.st_arg[o] = rs_a;
    if (rs.tgt_logit && rs_target >= n0 && rs_target < n0 + BN) rs.tgt_logit[row] = rs_t;
  }
}

// ---------------------------------------------------------------------------------------------
// the tile kernel
// ---------------------------------------------------------------------------------------------
template <int BN, int STAGES>
__global__ void __launch_bounds__(GEMM_THREADS, 2) gemm_tcgen05_kernel(const __grid_constant__ GemmParams p) {
  constexpr int TMEM_COLS = BN < 32 ? 32 : BN;          // allocation granularity: power of two >= 32
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  const auto sm = TileSmem<BN, STAGES>::carve(smem_raw);

  const int warp = threadIdx.x >> 5;
  const int m0 = blockIdx.y * BM;
  const int n0 = blockIdx.x * BN;
  const int total_kb = total_kblocks(p);
  const uint32_t tmem_acc = gemm_setup<false, TMEM_COLS>(p.ta, p.tb, p.nseg, sm, warp);

  if (warp == 0) {
    if (elect_one_sync()) gemm_produce<false, false>(p.kblocks, sm, p.ta, m0, p.tb, n0, 0, total_kb, true);
    __syncwarp();
  } else if (warp == 1) {
    if (elect_one_sync()) gemm_mma<false>(sm, tmem_acc, make_idesc(BM, BN), 0, total_kb);
    __syncwarp();
  } else {
    epilogue_tile<BN, true>(p.epi, p.rs, p.M, p.N, p.vec, p.tma_store ? &p.tc : nullptr, tmem_acc, sm.accum,
                            smem_u32(smem_raw), m0, n0);
  }
  gemm_teardown<false, TMEM_COLS>(p.tma_store, tmem_acc, warp);
}

// ---------------------------------------------------------------------------------------------
// CTA-pair kernel: a 2-CTA cluster computes one 256 x BN tile with tcgen05.mma.cta_group::2 (M = 256).
// CTA r of the pair owns rows [128r, 128r+128) of the tile: it loads its own 128 x 64 slice of A and HALF of the
// B tile (BN/2 rows), so per MMA each SM reads half the shared-memory bytes of the single-CTA kernel and the pair
// pulls B through L2 once instead of twice. Only the leader (rank 0) issues MMAs; both CTAs' TMA loads complete on
// the leader's `full` barrier; tcgen05.commit multicasts the `empty` / accumulator-ready arrivals to both CTAs.
// ---------------------------------------------------------------------------------------------
template <int BN, int STAGES>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(GEMM_THREADS, 1)
gemm_tcgen05_2cta_kernel(const __grid_constant__ GemmParams p) {
  constexpr int TMEM_COLS = BN < 32 ? 32 : BN;
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  const auto sm = PairTileSmem<BN, STAGES>::carve(smem_raw);

  const int warp = threadIdx.x >> 5;
  const uint32_t rank = cluster_ctarank();
  const int m0 = blockIdx.y * (2 * BM) + (int)rank * BM;
  const int n0 = (blockIdx.x >> 1) * BN;
  const int total_kb = total_kblocks(p);
  const uint32_t tmem_acc = gemm_setup<true, TMEM_COLS>(p.ta, p.tb, p.nseg, sm, warp);

  if (warp == 0) {
    if (elect_one_sync()) gemm_produce<true, false>(p.kblocks, sm, p.ta, m0, p.tb, n0 + (int)rank * (BN / 2), 0, total_kb, rank == 0);
    __syncwarp();
  } else if (warp == 1) {
    if (rank == 0 && elect_one_sync()) gemm_mma<true>(sm, tmem_acc, make_idesc(2 * BM, BN), 0, total_kb);
    __syncwarp();
  } else {
    epilogue_tile<BN, false>(p.epi, p.rs, p.M, p.N, p.vec, p.tma_store ? &p.tc : nullptr, tmem_acc, sm.accum,
                             smem_u32(smem_raw), m0, n0);
  }
  gemm_teardown<true, TMEM_COLS>(p.tma_store, tmem_acc, warp);
}

// ---------------------------------------------------------------------------------------------
// Grouped CTA-pair kernel (gemm_bf16_tn_grouped): the 256 x BN pair tiles of up to kMaxGemmProblems independent
// single-segment GEMMs with plain fp32 outputs in one grid. The grid is the concatenation of the problems' tile lists
// (x = 2 * tile + rank); a pair finds its problem through the prefix table tile0 and runs the pipeline of the CTA-pair
// tile kernel on that problem's maps. TMA stores are decided per problem.
// ---------------------------------------------------------------------------------------------
struct GroupedProblem {
  CUtensorMap ta, tb;                             // A (M rows, boxes of BM), B (N rows, boxes of BN / 2)
  CUtensorMap tc;                                 // fp32 output when tma_store (see choose_tma_store)
  float* C; int ldc;
  int M, N, kblocks;
  int tile0, tiles_n;                             // first pair tile of the problem in the grid, pair tiles along N
  int tma_store, vec;
};
struct GroupedParams {
  GroupedProblem prob[kMaxGemmProblems];
  int n;
};

template <int BN, int STAGES>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(GEMM_THREADS, 1)
gemm_tcgen05_2cta_grouped_kernel(const __grid_constant__ GroupedParams g) {
  constexpr int TMEM_COLS = BN;
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  const auto sm = PairTileSmem<BN, STAGES>::carve(smem_raw);

  const int warp = threadIdx.x >> 5;
  const uint32_t rank = cluster_ctarank();
  const int tile = blockIdx.x >> 1;
  int pi = 0;
  while (pi + 1 < g.n && tile >= g.prob[pi + 1].tile0) ++pi;
  const GroupedProblem& pr = g.prob[pi];
  const int local = tile - pr.tile0;
  const int m0 = (local / pr.tiles_n) * (2 * BM) + (int)rank * BM;
  const int n0 = (local % pr.tiles_n) * BN;
  const uint32_t tmem_acc = gemm_setup<true, TMEM_COLS>(&pr.ta, &pr.tb, 1, sm, warp);

  if (warp == 0) {
    if (elect_one_sync())
      gemm_produce<true, false>(&pr.kblocks, sm, &pr.ta, m0, &pr.tb, n0 + (int)rank * (BN / 2), 0, pr.kblocks, rank == 0);
    __syncwarp();
  } else if (warp == 1) {
    if (rank == 0 && elect_one_sync()) gemm_mma<true>(sm, tmem_acc, make_idesc(2 * BM, BN), 0, pr.kblocks);
    __syncwarp();
  } else {
    GemmEpi e;
    e.C32 = pr.C; e.ldc32 = pr.ldc;
    epilogue_tile<BN, false>(e, RowStatsEpi(), pr.M, pr.N, pr.vec, pr.tma_store ? &pr.tc : nullptr, tmem_acc, sm.accum,
                             smem_u32(smem_raw), m0, n0);
  }
  gemm_teardown<true, TMEM_COLS>(pr.tma_store, tmem_acc, warp);
}

// ---------------------------------------------------------------------------------------------
// Skinny-M kernel (M <= 256: the per-timestep recurrent GEMMs, M = batch): operands SWAPPED, every 256 x 256 tile
// driven by tcgen05.mma.cta_group::2 on a CTA pair, K split over a thread-block cluster, partial tiles reduced through
// distributed shared memory.
//
// Measured on B200 (tools/gemm_bench.py, profiles/README.md): an M=128 tcgen05.mma takes ~130 cycles whatever its
// N, and one SM ingests TMA operands at ~77 GB/s at most (the chip-wide L2 -> SM rate, ~6300 B/clk, B300_MICROARCH.md,
// with all SMs pulling). A skinny GEMM therefore wants (a) the <= 256 batch rows on the MMA's N side so every
// instruction is a full-width MMA, and (b) as few operand bytes per SM as possible. CTA x of a pair loads its own 128
// WEIGHT rows (16 KB) and HALF of the batch rows (16 KB) per k-block; the MMA (M = 256 weight rows, N = 256 batch rows)
// reads both halves across the pair. 32 KB per SM and k-block instead of 48 KB for one CTA that loads all 256 batch
// rows (2/3 of it the activation tile every weight-row CTA re-reads): the loads of a 128x256x64 block (~415 ns at
// 77 GB/s) hide behind its MMAs (~440 ns at the sustained tensor rate).
// Cluster = (2, 1, S): x = the pair, z = the K split (S = 1..4). Afterwards CTA (x, z) owns the batch columns
// [z*CW, z*CW+CW) of its 128 weight rows: every CTA pushes the other splits' column slices of its partial accumulator
// into their shared memory (st.shared::cluster, coalesced), a cluster barrier makes them visible, and the owner adds
// them to its own TMEM slice and runs the full epilogue.
// The accumulator is transposed (TMEM lane = output column n, TMEM column = batch row), so for a fixed batch row the
// 32 lanes of an epilogue warp hold 32 consecutive n: every global access is one coalesced 128-byte line.
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t mapa_shared(uint32_t saddr, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(saddr), "r"(rank));
  return r;
}
__device__ __forceinline__ void st_shared_cluster_f32(uint32_t addr, float v) {
  asm volatile("st.shared::cluster.f32 [%0], %1;" ::"r"(addr), "f"(v) : "memory");
}

// v[j] = value of output column n (this lane) at batch row b0 + j. The block is staged in shared memory as
// [batch row][column] (lanes write consecutive words: conflict-free, no transpose needed) and leaves through the
// same vector path as the other kernels, 16 bytes per lane. (With 4-byte stores from the 4 epilogue warps alone the
// SM sustained ~5 B/clk: 3k cycles per 32x32 block.) Ragged / unaligned blocks take a scalar loop over the staged
// block; nothing indexes the register array dynamically (that would push it to local memory).
__device__ __forceinline__ void epilogue_swapped32(const GemmEpi e, int vec, int M, int N, int n_warp0, int b0,
                                                   const float (&v)[32], uint32_t stage) {
  const int lane = threadIdx.x & 31;
#pragma unroll
  for (int j = 0; j < 32; ++j) sts_f32(stage + (j * 36 + lane) * 4, v[j]);
  __syncwarp();
  const bool add1_all = e.add1 && (n_warp0 + 32 <= e.add1_cols);
  const bool add1_none = !e.add1 || (n_warp0 >= e.add1_cols);
  if (vec && n_warp0 + 32 <= N && (add1_all || add1_none)) {
    epilogue_block_vec(e, M, b0, n_warp0, stage, add1_all);
  } else {
    const int n = n_warp0 + lane;
    if (n < N) {
      const float bias = e.bias ? e.bias[n] : 0.f;
      const bool add1 = e.add1 && n < e.add1_cols;
      const int rows = min(32, M - b0);
#pragma unroll 1
      for (int j = 0; j < rows; ++j) {
        const int b = b0 + j;
        float x = lds_f32(stage + (j * 36 + lane) * 4) * e.alpha + bias;
        if (add1) x += e.add1[(size_t)b * e.ld1 + n];
        if (e.add2) x += e.add2[(size_t)b * e.ld2 + n];
        if (e.act == 1) x = tanh_fast(x);
        if (e.dtanh) { const float t = e.dtanh[(size_t)b * e.ldd + n]; x *= 1.0f - t * t; }
        if (e.C32) {
          float* q = e.C32 + (size_t)b * e.ldc32 + n;
          *q = e.accumulate ? (*q + x) : x;
        }
        if (e.C16) e.C16[(size_t)b * e.ldc16 + n] = __float2bfloat16_rn(x);
      }
    }
  }
  __syncwarp();
}

template <int STAGES>
__global__ void __launch_bounds__(GEMM_THREADS, 1) gemm_tcgen05_swapped_pair_kernel(const __grid_constant__ GemmParams p) {
  constexpr int BW = 128, BXH = 128;                    // weight rows per CTA (half of UMMA M), batch rows LOADED per CTA
  constexpr int TCOLS = 2 * BXH;                        // accumulator: 128 lanes (this CTA's weight rows) x 256 batch rows
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  const auto sm = SwappedSmem<STAGES>::carve(smem_raw);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int xr = blockIdx.x & 1;                        // position in the pair; cluster rank = xr + 2 * z
  const int S = p.splits;
  const int rank = blockIdx.z;                          // K split of this CTA (cluster z == grid z)
  const int n0 = (blockIdx.x >> 1) * (2 * BW) + xr * BW;   // first weight row (output column) of this CTA

  const int total_kb = total_kblocks(p);
  const int kb_begin = rank * p.kb_per_split;
  const int kb_end = min(total_kb, kb_begin + p.kb_per_split);
  const uint32_t tmem_acc = gemm_setup<true, TCOLS>(p.ta, p.tb, p.nseg, sm, warp);
  const int CW = S == 1 ? 256 : S == 2 ? 128 : S == 3 ? 96 : 64;   // batch columns owned by each K split

  if (warp == 0) {
    // The weights of the skinny GEMMs (76 MB per timestep) are streamed once per launch; marking them evict_first
    // leaves L2 to the 52 MB of region features + projections the attention kernels re-read every step (measured:
    // step 8.21 -> 8.08 ms, attention_fwd 25.1 -> 23.1 us).
    if (elect_one_sync()) gemm_produce<true, true>(p.kblocks, sm, p.tb, n0, p.ta, xr * BXH, kb_begin, kb_end, xr == 0);
    __syncwarp();
  } else if (warp == 1) {
    if (xr == 0 && elect_one_sync())
      gemm_mma<true>(sm, tmem_acc, make_idesc(2 * BW, 2 * BXH), kb_begin, kb_end, static_cast<uint16_t>(3u << (2 * rank)));
    __syncwarp();
  } else {
    mbar_wait(sm.accum, 0);                             // this pair's partial tile is complete in both CTAs' TMEM
    tc_fence_after();
  }

  const int q = warp & 3;                               // epilogue warps 2..5 own TMEM lanes [32q, 32q+32)
  const int tl = q * 32 + lane;                         // TMEM lane = column n0 + tl of the output
  const uint32_t recv = smem_u32(smem_raw);             // [(S-1) sources][CW columns][128 lanes] fp32, over the dead stages
  // every CTA of the cluster has finished its main loop (stage buffers dead, also the ones the PEER's MMAs read)
  cluster_sync_all();
  if (S > 1) {
    if (warp >= 2 && kb_end > kb_begin) {
      for (int o = 0; o < S; ++o) {
        if (o == rank) continue;
        const int slot = rank < o ? rank : rank - 1;
        const uint32_t rbase = mapa_shared(recv, (uint32_t)(xr + 2 * o));
        for (int c = 0; c < CW; c += 32) {
          if (o * CW + c >= p.M || o * CW + c >= TCOLS) break;   // columns beyond the batch are never read
          uint32_t acc[32];
          tmem_ld_32x32(tmem_acc + (static_cast<uint32_t>(q * 32) << 16) + o * CW + c, acc);
          tmem_ld_wait();
#pragma unroll
          for (int j = 0; j < 32; ++j)
            st_shared_cluster_f32(rbase + (uint32_t)(((slot * CW + c + j) * 128 + tl) * 4), __uint_as_float(acc[j]));
        }
      }
    }
    cluster_sync_all();
  }
  if (warp >= 2) {
    const GemmEpi epi = p.epi;
    for (int c = 0; c < CW; c += 32) {
      const int b0 = rank * CW + c;
      if (b0 >= p.M || b0 >= TCOLS) break;
      float v[32];
      if (kb_end > kb_begin) {
        uint32_t acc[32];
        tmem_ld_32x32(tmem_acc + (static_cast<uint32_t>(q * 32) << 16) + b0, acc);
        tmem_ld_wait();
#pragma unroll
        for (int j = 0; j < 32; ++j) v[j] = __uint_as_float(acc[j]);
      } else {
#pragma unroll
        for (int j = 0; j < 32; ++j) v[j] = 0.f;
      }
      for (int o = 0; o < S; ++o) {
        if (o == rank || o * p.kb_per_split >= total_kb) continue;
        const int slot = o < rank ? o : o - 1;
#pragma unroll
        for (int j = 0; j < 32; ++j) v[j] += lds_f32(recv + (uint32_t)(((slot * CW + c + j) * 128 + tl) * 4));
      }
      if (p.tma_store) {
        const uint32_t st = smem_u32(smem_raw) + 96 * 1024 + (warp - 2) * 4096;
        const float bias = (epi.bias && n0 + tl < p.N) ? epi.bias[n0 + tl] : 0.f;
        if (lane == 0) tma_store_wait_read();
        __syncwarp();
#pragma unroll
        for (int j = 0; j < 32; ++j) sts_f32(st + (j * 32 + lane) * 4, fmaf(v[j], epi.alpha, bias));
        fence_proxy_async_smem();
        __syncwarp();
        if (lane == 0 && n0 + q * 32 < p.N) tma_store_2d(&p.tc, st, n0 + q * 32, b0);
      } else if (n0 + q * 32 < p.N) {
        epilogue_swapped32(epi, p.vec, p.M, p.N, n0 + q * 32, b0, v,
                           smem_u32(smem_raw) + 96 * 1024 + (warp - 2) * 32 * 36 * 4);
      }
    }
  }
  gemm_teardown<true, TCOLS>(p.tma_store, tmem_acc, warp);
}

// ---------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------
static EncodeTiledFn get_encode_fn() {
  static EncodeTiledFn fn = nullptr;
  static std::once_flag once;
  std::call_once(once, [] {
    void* sym = nullptr;
    cudaDriverEntryPointQueryResult qres;
    // resolved through the runtime so the library has no link-time dependency on libcuda
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &sym, cudaEnableDefault, &qres) == cudaSuccess &&
        qres == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(sym);
  });
  return fn;
}

void* tma_encode_fn() { return reinterpret_cast<void*>(get_encode_fn()); }

int encode_tmap_2d_uncached(CUtensorMap* out, const bf16* base, int rows, int K, int ld, int box_rows) {
  EncodeTiledFn fn = get_encode_fn();
  if (!fn) { set_error("cuTensorMapEncodeTiled not available from the driver"); return SSCVAE_ERR_DRIVER; }
  if ((reinterpret_cast<uintptr_t>(base) & 15) || (ld % 8) != 0) {
    set_error("gemm operand not TMA-compatible: base %p ld %d (need 16B-aligned base, ld %% 8 == 0)", (const void*)base, ld);
    return SSCVAE_ERR_BAD_ARG;
  }
  cuuint64_t dims[2] = {(cuuint64_t)K, (cuuint64_t)rows};
  cuuint64_t strides[1] = {(cuuint64_t)ld * 2};
  cuuint32_t box[2] = {(cuuint32_t)BK, (cuuint32_t)box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = fn(out, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<bf16*>(base), dims, strides, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled failed (%d) rows=%d K=%d ld=%d box_rows=%d", (int)r, rows, K, ld, box_rows);
    return SSCVAE_ERR_DRIVER;
  }
  return 0;
}

// cuTensorMapEncodeTiled costs microseconds of host time and a training step issues ~500 of them with the same
// few hundred (pointer, shape) combinations every step: memoise the encoded descriptors.
struct TmapKey {
  const void* base; int rows, K, ld, box_rows;
  bool operator==(const TmapKey& o) const { return base == o.base && rows == o.rows && K == o.K && ld == o.ld && box_rows == o.box_rows; }
};
struct TmapKeyHash {
  size_t operator()(const TmapKey& k) const {
    size_t h = reinterpret_cast<size_t>(k.base) * 0x9E3779B97F4A7C15ull;
    h ^= ((size_t)k.rows << 40) ^ ((size_t)k.K << 20) ^ ((size_t)k.ld << 4) ^ (size_t)k.box_rows;
    return h * 0xD6E8FEB86659FD93ull;
  }
};
static std::unordered_map<TmapKey, CUtensorMap, TmapKeyHash> g_tmap_cache;
static std::mutex g_tmap_mutex;

static int encode_tmap(CUtensorMap* out, const bf16* base, int rows, int K, int ld, int box_rows) {
  const TmapKey key{base, rows, K, ld, box_rows};
  std::lock_guard<std::mutex> lock(g_tmap_mutex);
  auto it = g_tmap_cache.find(key);
  if (it != g_tmap_cache.end()) { *out = it->second; return 0; }
  TRY(encode_tmap_2d_uncached(out, base, rows, K, ld, box_rows));
  if (g_tmap_cache.size() > 8192) g_tmap_cache.clear();
  g_tmap_cache.emplace(key, *out);
  return 0;
}

// operand maps of every K segment: A (M rows) with boxes of box_a rows, B (N rows) with boxes of box_b rows
static int encode_operands(GemmParams& prm, const GemmSeg* segs, int box_a, int box_b) {
  for (int s = 0; s < prm.nseg; ++s) {
    TRY(encode_tmap(&prm.ta[s], segs[s].A, prm.M, segs[s].K, segs[s].lda, box_a));
    TRY(encode_tmap(&prm.tb[s], segs[s].B, prm.N, segs[s].K, segs[s].ldb, box_b));
  }
  return 0;
}

static bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

// fp32 output tile map for TMA stores: box = 32 columns x 32 rows, dense in shared memory
static int encode_tmap_c32(CUtensorMap* out, const float* base, int rows, int cols, int ld, bool swizzle128) {
  const TmapKey key{base, rows, cols, ld, swizzle128 ? -33 : -32};
  std::lock_guard<std::mutex> lock(g_tmap_mutex);
  auto it = g_tmap_cache.find(key);
  if (it != g_tmap_cache.end()) { *out = it->second; return 0; }
  EncodeTiledFn fn = get_encode_fn();
  if (!fn) { set_error("cuTensorMapEncodeTiled not available from the driver"); return SSCVAE_ERR_DRIVER; }
  cuuint64_t dims[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
  cuuint64_t strides[1] = {(cuuint64_t)ld * 4};
  cuuint32_t box[2] = {32, 32};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = fn(out, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<float*>(base), dims, strides, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, swizzle128 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_NONE,
                  CU_TENSOR_MAP_L2_PROMOTION_NONE, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled (fp32 output) failed (%d) rows=%d cols=%d ld=%d", (int)r, rows, cols, ld);
    return SSCVAE_ERR_DRIVER;
  }
  if (g_tmap_cache.size() > 8192) g_tmap_cache.clear();
  g_tmap_cache.emplace(key, *out);
  return 0;
}

// Sets prm.tma_store, and encodes prm.tc when it is set: a plain fp32 tile (+ bias) leaves the epilogue through TMA
// stores. Never with row statistics, whose epilogue writes through epilogue_row32. bias_vec4: the epilogue reads the bias
// as float4 (the tile kernels; the swapped-pair kernel reads one bias per lane). swizzle128: the layout of the staged tile.
static bool tma_store_ok(const float* C32, int ldc32, int N) {
  // N % 4: the TMA unit clips stores at 16-byte granularity (measured: with N = 77 the columns 77..79 were written)
  return aligned16(C32) && (ldc32 % 4) == 0 && (N % 4) == 0;
}
static int choose_tma_store(GemmParams& prm, bool bias_vec4, bool swizzle128) {
  const GemmEpi& e = prm.epi;
  prm.tma_store = !prm.rs.mode && e.C32 && !e.C16 && !e.act && !e.dtanh && !e.accumulate && !e.add1 && !e.add2 &&
                  tma_store_ok(e.C32, e.ldc32, prm.N) && (!bias_vec4 || !e.bias || aligned16(e.bias));
  if (prm.tma_store) TRY(encode_tmap_c32(&prm.tc, e.C32, prm.M, prm.N, e.ldc32, swizzle128));
  return 0;
}

// GEMM_THREADS per CTA, smem bytes of dynamic shared memory; cluster_z > 0: clusters of (2, 1, cluster_z) CTAs
// (the swapped-pair kernel; the CTA-pair tile kernel declares its cluster shape itself)
static cudaLaunchConfig_t gemm_config(dim3 grid, int smem, cudaStream_t stream, int cluster_z, cudaLaunchAttribute* attr) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid;
  cfg.blockDim = dim3(GEMM_THREADS, 1, 1);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = stream;
  if (cluster_z > 0) {
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = 2; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = cluster_z;
    cfg.attrs = attr; cfg.numAttrs = 1;
  }
  return cfg;
}

// raises KERNEL's dynamic shared-memory limit to Smem::bytes(), once, before its first launch or occupancy query
template <auto KERNEL, class Smem>
static int gemm_configure() {
  static bool configured = false;
  if (!configured) {
    CUDA_TRY(cudaFuncSetAttribute(KERNEL, cudaFuncAttributeMaxDynamicSharedMemorySize, Smem::bytes()));
    configured = true;
  }
  return 0;
}

template <auto KERNEL, class Smem, class Params>
static int gemm_launch(cudaStream_t stream, dim3 grid, int cluster_z, const Params& prm) {
  TRY((gemm_configure<KERNEL, Smem>()));
  cudaLaunchAttribute attr[1];
  const cudaLaunchConfig_t cfg = gemm_config(grid, Smem::bytes(), stream, cluster_z, attr);
  CUDA_TRY(cudaLaunchKernelEx(&cfg, KERNEL, prm));
  ++g_launch_count;
  return 0;
}

template <int BN, int STAGES>
static int launch_tc(cudaStream_t stream, GemmParams& prm, const GemmSeg* segs) {
  TRY(encode_operands(prm, segs, BM, BN));
  if (BN >= 32) TRY(choose_tma_store(prm, true, true));    // a TMA store box is 32 columns wide
  return gemm_launch<gemm_tcgen05_kernel<BN, STAGES>, TileSmem<BN, STAGES>>(
      stream, dim3(ceil_div(prm.N, BN), ceil_div(prm.M, BM)), 0, prm);
}

template <int BN, int STAGES>
static int launch_tc2(cudaStream_t stream, GemmParams& prm, const GemmSeg* segs) {
  TRY(encode_operands(prm, segs, BM, BN / 2));
  TRY(choose_tma_store(prm, true, true));
  return gemm_launch<gemm_tcgen05_2cta_kernel<BN, STAGES>, PairTileSmem<BN, STAGES>>(
      stream, dim3(2 * ceil_div(prm.N, BN), ceil_div(prm.M, 2 * BM)), 0, prm);
}

// max co-resident clusters of the pair kernel for a K split of S (cluster = 2*S CTAs); 0 if the query fails
template <int STAGES>
static int pair_max_clusters(int S) {
  static int cache[5] = {-1, -1, -1, -1, -1};
  if (cache[S] >= 0) return cache[S];
  cudaLaunchAttribute attr[1];
  const cudaLaunchConfig_t cfg = gemm_config(dim3(2 * 64, 1, S), SwappedSmem<STAGES>::bytes(), 0, S, attr);
  int n = 0;
  if (cudaOccupancyMaxActiveClusters(&n, gemm_tcgen05_swapped_pair_kernel<STAGES>, &cfg) != cudaSuccess) {
    cudaGetLastError();
    n = 0;
  }
  cache[S] = n;
  return n;
}

template <int STAGES>
static int launch_swapped_pair(cudaStream_t stream, GemmParams& prm, const GemmSeg* segs, int forced_S) {
  TRY((gemm_configure<gemm_tcgen05_swapped_pair_kernel<STAGES>, SwappedSmem<STAGES>>()));
  int total_kb = 0;
  for (int s = 0; s < prm.nseg; ++s) total_kb += prm.kblocks[s];
  const int pairs = ceil_div(prm.N, 256);
  // the largest K split whose clusters are all co-resident (one wave) and that leaves every CTA >= 4 k-blocks
  int S = 1;
  if (forced_S > 0) S = forced_S;
  else
    for (int c = 4; c > 1; --c)
      if (total_kb >= 4 * c && pairs <= pair_max_clusters<STAGES>(c)) { S = c; break; }
  while (S > 1 && total_kb < S) --S;
  prm.kb_per_split = ceil_div(total_kb, S);
  S = ceil_div(total_kb, prm.kb_per_split);             // no empty trailing split
  prm.splits = S;
  TRY(encode_operands(prm, segs, 128, 128));
  TRY(choose_tma_store(prm, false, false));
  return gemm_launch<gemm_tcgen05_swapped_pair_kernel<STAGES>, SwappedSmem<STAGES>>(stream, dim3(2 * pairs, 1, S), S, prm);
}

int gemm_bf16_tn(cudaStream_t stream, int M, int N, int nseg, const GemmSeg* segs, const GemmEpi& epi) {
  REQUIRE(M > 0 && N > 0 && nseg >= 1 && nseg <= MAX_SEG, "gemm: bad shape M=%d N=%d nseg=%d", M, N, nseg);
  REQUIRE(epi.C32 || epi.C16 || (epi.rs && epi.rs->mode == 1), "gemm: no output");
  REQUIRE(epi.splits >= 0 && epi.splits <= 4, "gemm: pair split count %d (0..4)", epi.splits);
  double ksum = 0;
  for (int i = 0; i < nseg; ++i) ksum += segs[i].K;
  // instrumentation class: the skinny long-K GEMMs of the recurrence (the dominant kernel of a training step) are
  // reported on their own as "gemm.recurrent"
  int kb_all = 0;
  for (int i = 0; i < nseg; ++i) kb_all += ceil_div(segs[i].K, BK);
  const bool recurrent = M <= 256 && N >= 1024 && kb_all >= 16;
  PROF_SCOPE(stream, recurrent ? "gemm.recurrent" : epi.tag, 2.0 * M * N * ksum,
             2.0 * (M + N) * ksum + (epi.C32 ? 4.0 : 2.0) * M * N);
  GemmParams prm;
  memset(&prm, 0, sizeof(prm));
  prm.nseg = nseg; prm.M = M; prm.N = N; prm.epi = epi;
  if (epi.rs) prm.rs = *epi.rs;
  for (int s = 0; s < nseg; ++s) {
    REQUIRE(segs[s].K > 0, "gemm: empty K segment %d", s);
    prm.kblocks[s] = ceil_div(segs[s].K, BK);
  }
  bool vec = true;
  if (epi.bias) vec &= aligned16(epi.bias);
  if (epi.add1) vec &= aligned16(epi.add1) && (epi.ld1 % 4 == 0);
  if (epi.add2) vec &= aligned16(epi.add2) && (epi.ld2 % 4 == 0);
  if (epi.dtanh) vec &= aligned16(epi.dtanh) && (epi.ldd % 4 == 0);
  if (epi.C32) vec &= aligned16(epi.C32) && (epi.ldc32 % 4 == 0);
  if (epi.C16) vec &= aligned16(epi.C16) && (epi.ldc16 % 8 == 0);
  prm.vec = vec ? 1 : 0;
  int total_kb = 0;
  for (int s = 0; s < nseg; ++s) total_kb += prm.kblocks[s];
  if (epi.rs && epi.rs->mode) {                           // vocabulary head with softmax statistics / CE gradient in the epilogue
    REQUIRE(!epi.add1 && !epi.add2 && !epi.act && !epi.dtanh && !epi.accumulate,
            "gemm: row statistics take a plain (alpha, bias) epilogue");
    REQUIRE(epi.rs->mode != 1 || (epi.rs->st_max && epi.rs->st_sum && epi.rs->st_arg), "gemm: row statistics need their partial buffers");
    REQUIRE(epi.rs->mode != 2 || (epi.rs->lse && epi.rs->gcoef && epi.rs->target && epi.C16), "gemm: CE gradient needs lse, gcoef, target and a bf16 output");
    return launch_tc<128, 3>(stream, prm, segs);          // a thread sees 128 logits of its row per tile
  }
  // Skinny GEMMs with enough weight rows (the per-timestep LSTM and BPTT GEMMs, short K included: the attention-LSTM
  // recurrence, K = 2Hp) run on the swapped-operand CTA-pair kernel (see the kernel); narrow N (256x768x960) stays on
  // the plain kernel. epi.splits = 1..4 forces the pair kernel with that K split (tests, tools/gemm_bench.py).
  const bool pair_shape = N >= 1024 && total_kb >= 16;
  if (M <= 256 && (epi.splits > 0 || pair_shape)) return launch_swapped_pair<6>(stream, prm, segs, epi.splits);
  // The recurrent GEMMs have M = batch (two 128-row tiles) and stream their weights once: they are bound by
  // bytes in flight per SM, not by the tensor pipe. So: the widest N tile that still yields >= ~100 CTAs,
  // ~100 KB of TMA stages per CTA and two CTAs resident per SM (no wave-quantisation tail at 149..296 CTAs,
  // one CTA's epilogue overlaps the other's main loop).
  const long mt = ceil_div(M, BM);
  // large and long-K (the batched weight-gradient GEMMs): CTA pairs, 256x128 tiles (3600x2048x5376: 68 vs 76 us)
  if (M >= 1024 && N >= 512 && total_kb >= 32) return launch_tc2<128, 4>(stream, prm, segs);
  if (mt * ceil_div(N, 128) >= 96) return launch_tc<128, 3>(stream, prm, segs);
  // Small problems are latency-bound, not occupancy-bound: narrower tiles only add CTAs whose MMAs cost the same
  // ~130 cycles and lose the TMA-store epilogue (256x768x960: 7.9 us with 64-wide tiles, 10.4 with 16-wide).
  if (N > 32) return launch_tc<64, 4>(stream, prm, segs);
  if (N > 16) return launch_tc<32, 5>(stream, prm, segs);
  return launch_tc<16, 6>(stream, prm, segs);
}

int gemm_bf16_tn_grouped(cudaStream_t stream, int nprob, const GemmProblem* probs, const char* tag) {
  REQUIRE(nprob >= 0 && nprob <= kMaxGemmProblems, "gemm grouped: %d problems (0..%d)", nprob, kMaxGemmProblems);
  if (nprob == 0) return 0;
  constexpr int TBN = 128, STAGES = 4;
  // longest K first: the short problems' tiles fill the tail of the grid
  int order[kMaxGemmProblems];
  for (int i = 0; i < nprob; ++i) order[i] = i;
  std::stable_sort(order, order + nprob, [&](int a, int b) { return probs[a].K > probs[b].K; });
  GroupedParams g;
  memset(&g, 0, sizeof(g));
  g.n = nprob;
  double flops = 0, bytes = 0;
  int tiles = 0;
  for (int i = 0; i < nprob; ++i) {
    const GemmProblem& q = probs[order[i]];
    REQUIRE(q.M > 0 && q.N > 0 && q.K > 0 && q.C32, "gemm grouped: problem %d: M=%d N=%d K=%d C32=%p", order[i], q.M, q.N,
            q.K, (const void*)q.C32);
    GroupedProblem& pr = g.prob[i];
    TRY(encode_tmap(&pr.ta, q.A, q.M, q.K, q.lda, BM));
    TRY(encode_tmap(&pr.tb, q.B, q.N, q.K, q.ldb, TBN / 2));
    pr.C = q.C32; pr.ldc = q.ldc32; pr.M = q.M; pr.N = q.N; pr.kblocks = ceil_div(q.K, BK);
    pr.tiles_n = ceil_div(q.N, TBN);
    pr.tile0 = tiles;
    tiles += pr.tiles_n * ceil_div(q.M, 2 * BM);
    pr.vec = aligned16(q.C32) && (q.ldc32 % 4) == 0;
    pr.tma_store = tma_store_ok(q.C32, q.ldc32, q.N);
    if (pr.tma_store) TRY(encode_tmap_c32(&pr.tc, q.C32, q.M, q.N, q.ldc32, true));
    flops += 2.0 * q.M * q.N * q.K;
    bytes += 2.0 * ((double)q.M + q.N) * q.K + 4.0 * q.M * q.N;
  }
  PROF_SCOPE(stream, tag, flops, bytes);
  return gemm_launch<gemm_tcgen05_2cta_grouped_kernel<TBN, STAGES>, PairTileSmem<TBN, STAGES>>(stream, dim3(2 * tiles), 0, g);
}

}  // namespace sscvae

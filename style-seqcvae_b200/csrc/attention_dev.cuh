// Device-side building blocks of the fused region attention (attention.py:36-97, updown_cell.py:156-158), shared by the
// stand-alone kernels (attention.cu) and the persistent recurrent kernels (persistent.cuh).
#pragma once
#include "kernels.cuh"
#include "ptx.cuh"

// ATT_TID0: thread index of the first consumer thread inside the CTA (the persistent kernel runs the consumers on
// warps 2..9); the helpers below are per-translation-unit (anonymous namespace) because they depend on it.
#ifndef ATT_TID0
#define ATT_TID0 0
#endif

namespace sscvae {
namespace attn {
namespace {

__device__ __forceinline__ int attn_tid() { return (int)threadIdx.x - ATT_TID0; }

__device__ __forceinline__ float tanh_approx(float x) {
  float y;
  asm("tanh.approx.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}


constexpr int ATT_CONSUMERS = 256;                 // 8 consumer warps
constexpr int ATT_CWARPS = ATT_CONSUMERS / 32;
constexpr int ATT_THREADS = ATT_CONSUMERS + 32;    // + 1 producer warp
#ifndef ATT_STAGES_N
#define ATT_STAGES_N 4
#endif
constexpr int ATT_STAGES = ATT_STAGES_N;           // ring depth (per translation unit, like ATT_TID0)
#ifndef ATT_STAGE_BYTES_N
#define ATT_STAGE_BYTES_N 16384                    // stand-alone kernels: two CTAs per SM, their phases overlap
#endif
constexpr int ATT_STAGE_BYTES = ATT_STAGE_BYTES_N; // per translation unit: the persistent kernels use 2 x 32 KB (8 feature rows per
                                                   // chunk = one box per consumer warp: half the per-chunk handshakes)
constexpr int ATT_MAXB = 8;                        // boxes per chunk (<= consumer warps: one box per warp and chunk)
constexpr int ATT_NREG = 4;                        // boxes per lane in the softmax: N <= 128
constexpr int ATT_FV = 2;                          // 16-byte feature vectors per thread: Fp <= 4096
constexpr int ATT_PV = 2;                          // projection column pairs per thread: Ap <= 1024

struct AttnPlan {
  int nP, bP;            // chunks / boxes per chunk of the projected features
  int nF, bF;            // same for the region features
  int rows_per_cta;
};

struct AttnSmem {
  uint8_t* stage;        // ATT_STAGES x ATT_STAGE_BYTES
  uint64_t* full;        // [ATT_STAGES]
  uint64_t* empty;       // [ATT_STAGES]
  float* wa;             // Ap
  float* q0;             // 2 x Ap (double buffer, prefetched one row ahead)
  float* u;              // ATT_CWARPS x N4 partial scores (d alpha in backward): [sub-warp][box]
  float* alw;            // ATT_CWARPS x N4: every consumer warp's own copy of alpha (broadcast reads in the weighted sum)
  float* msk0;           // 2 x N4: the box mask of the row (a global-memory read per chunk put an L2 round trip, ~0.7 us,
                         // in front of every chunk of the score / d alpha loops)
  float* dx0;            // 2 x ndx x Fp (backward only; ndx = split-K slots of d xhat, summed in place before use)
  float* sv0;            // 2 x N4 (backward only: saved softmax)
  int Ap, Fp, N4, ndx, dxb;
  __device__ __forceinline__ float* q(int slot) const { return q0 + slot * Ap; }
  __device__ __forceinline__ float* msk(int slot) const { return msk0 + slot * N4; }
  __device__ __forceinline__ float* dx(int slot, int k = 0) const { return dx0 + ((dxb == 1 ? 0 : slot) * ndx + k) * Fp; }
  __device__ __forceinline__ float* sv(int slot) const { return sv0 + slot * N4; }
};

// ndx: split-K slots of d xhat; dxb: d xhat buffers (2: the next row is prefetched while this one runs, 1: the caller
// prefetches the next row's d xhat only after the d alpha phase of the current one)
__device__ __forceinline__ AttnSmem carve(uint8_t* raw, const AttnArgs& a, bool bwd, int ndx = 1, int dxb = 2) {
  AttnSmem s;
  // no integer round trip on the pointer: it would lose the shared address space and turn every access below into a
  // generic LD/ST with 64-bit address arithmetic (a third of the instructions of the first version of these kernels)
  uint8_t* p = raw;
  s.stage = p; p += ATT_STAGES * ATT_STAGE_BYTES;
  s.full = reinterpret_cast<uint64_t*>(p); p += ATT_STAGES * 8;
  s.empty = reinterpret_cast<uint64_t*>(p); p += ATT_STAGES * 8;
  float* f = reinterpret_cast<float*>(p);
  s.Ap = a.Ap; s.Fp = a.Fp; s.N4 = (a.N + 3) & ~3; s.ndx = ndx; s.dxb = dxb;
  s.wa = f; f += a.Ap;
  s.q0 = f; f += 2 * a.Ap;
  s.u = f; f += ATT_CWARPS * s.N4;
  s.alw = f; f += ATT_CWARPS * s.N4;
  s.msk0 = f; f += 2 * s.N4;
  s.dx0 = s.sv0 = nullptr;
  if (bwd) {
    s.dx0 = f; f += dxb * ndx * a.Fp;
    s.sv0 = f; f += 2 * s.N4;
  }
  return s;
}
__host__ __device__ inline size_t attn_smem_bytes(const AttnArgs& a, bool bwd, int ndx = 1, int dxb = 2) {
  size_t n = 128 + (size_t)ATT_STAGES * ATT_STAGE_BYTES + 2 * ATT_STAGES * 8;
  n += (size_t)(3 * a.Ap + (2 * ATT_CWARPS + 2) * ((a.N + 3) & ~3)) * 4;
  if (bwd) n += (size_t)(dxb * ndx * a.Fp + 2 * ((a.N + 3) & ~3)) * 4;
  return n;
}

// ring bookkeeping shared by producer and consumers (both walk the same chunk sequence)
struct Ring {
  int stage = 0;
  uint32_t phase = 0;
  __device__ __forceinline__ void advance() {
    if (++stage == ATT_STAGES) { stage = 0; phase ^= 1; }
  }
};

// Chunking of the two streams of a row: as many boxes per chunk as fit one ring stage, at most ATT_MAXB.
// rows_per_cta is left at 0 for the caller to set.
inline AttnPlan attn_chunk_plan(const AttnArgs& a) {
  auto boxes_per_chunk = [](int row_bytes) {
    int b = 1;
    while (b * 2 <= ATT_MAXB && b * 2 * row_bytes <= ATT_STAGE_BYTES) b *= 2;
    return b;
  };
  AttnPlan pl;
  pl.bP = boxes_per_chunk(a.Ap * 2); pl.nP = ceil_div(a.N, pl.bP);
  pl.bF = boxes_per_chunk(a.Fp * 2); pl.nF = ceil_div(a.N, pl.bF);
  pl.rows_per_cta = 0;
  return pl;
}

// policy: ptx::l2_policy_evict_first() in every caller. The 52 MB of features + projections are read once per timestep
// and would otherwise push the recurrent weights (76 MB, re-read every step) out of the 126 MB L2.
__device__ __forceinline__ void produce_block(const AttnSmem& sm, Ring& ring, const uint8_t* base, int N, int row_bytes,
                                              int nchunks, int bper, uint64_t policy) {
  for (int c = 0; c < nchunks; ++c) {
    const int n0 = c * bper;
    const int nb = min(bper, N - n0);
    const uint32_t bytes = (uint32_t)nb * (uint32_t)row_bytes;
    ptx::mbar_wait(&sm.empty[ring.stage], ring.phase ^ 1);
    ptx::mbar_expect_tx(&sm.full[ring.stage], bytes);
    ptx::bulk_g2s_hint(sm.stage + (size_t)ring.stage * ATT_STAGE_BYTES, base + (size_t)n0 * row_bytes, bytes, &sm.full[ring.stage],
                       policy);
    ring.advance();
  }
}

// row-vector prefetch (cp.async, 4 bytes per op: no alignment requirement on the row stride)
__device__ __forceinline__ void prefetch_vec(float* dst, const float* src, int n) {
  for (int i = attn_tid(); i < n; i += ATT_CONSUMERS) ptx::cp_async4(dst + i, src + i);
}

template <int K>
__device__ __forceinline__ float pick(const float (&v)[K], int k) {
  float r = v[0];
#pragma unroll
  for (int i = 1; i < K; ++i) r = (k == i) ? v[i] : r;
  return r;
}

// A chunk holds nb <= ATT_MAXB boxes; 8/pow2ceil(nb) warps share one box (each a slice of the vectors), so all
// consumer warps stay busy whatever the chunk size. Partial sums land in part[sub][n] and are added by the readers.
__device__ __forceinline__ int warps_per_box(int nb) { return nb > 4 ? 1 : nb > 2 ? 2 : nb > 1 ? 4 : 8; }
__device__ __forceinline__ int wpb_log2(int wpb) { return wpb == 1 ? 0 : wpb == 2 ? 1 : wpb == 4 ? 2 : 3; }
// pair: full chunks (ATT_CWARPS boxes) were reduced in "pair mode" (attn_bwd_row): two partials per box
__device__ __forceinline__ float gather_partial(const float* part, int N4, int N, int bper, int n, bool pair = false) {
  const int n0 = (n / bper) * bper;
  const int nbk = min(bper, N - n0);
  const int wpb = (pair && nbk == ATT_CWARPS) ? 2 : warps_per_box(nbk);
  float s = 0.f;
  for (int k = 0; k < wpb; ++k) s += part[k * N4 + n];
  return s;
}

// scores u_n of the boxes of one P chunk
__device__ __forceinline__ void chunk_scores(const AttnArgs& a, const bf16* buf, int n0, int nb, const float* mask_img,
                                             const float* q_s, const float* wa_s, float* part, int N4) {
  const int warp = attn_tid() >> 5, lane = threadIdx.x & 31;
  const int nvec = a.Ap >> 3;
  const int wpb = warps_per_box(nb);
  const int j = warp >> wpb_log2(wpb), sub = warp & (wpb - 1);
  if (j >= nb) return;
  const int n = n0 + j;
  float s = 0.f;
  if (mask_img[n] != 0.f) {                        // masked boxes enter the softmax as u*m = 0
    const bf16x8* p = reinterpret_cast<const bf16x8*>(buf + (size_t)j * a.Ap);
    for (int i = sub * 32 + lane; i < nvec; i += 32 * wpb) {
      const bf16x8 v = p[i];
      const float4 qa = *reinterpret_cast<const float4*>(q_s + i * 8);
      const float4 qb = *reinterpret_cast<const float4*>(q_s + i * 8 + 4);
      const float4 wa = *reinterpret_cast<const float4*>(wa_s + i * 8);
      const float4 wb = *reinterpret_cast<const float4*>(wa_s + i * 8 + 4);
      const float2 f0 = __bfloat1622float2(v.v[0]), f1 = __bfloat1622float2(v.v[1]);
      const float2 f2 = __bfloat1622float2(v.v[2]), f3 = __bfloat1622float2(v.v[3]);
      s += wa.x * tanh_approx(qa.x + f0.x) + wa.y * tanh_approx(qa.y + f0.y);
      s += wa.z * tanh_approx(qa.z + f1.x) + wa.w * tanh_approx(qa.w + f1.y);
      s += wb.x * tanh_approx(qb.x + f2.x) + wb.y * tanh_approx(qb.y + f2.y);
      s += wb.z * tanh_approx(qb.z + f3.x) + wb.w * tanh_approx(qb.w + f3.y);
    }
    s = warp_sum(s);
  }
  if (lane == 0) part[sub * N4 + n] = s;
}

// masked softmax, redundantly per warp; lane holds boxes lane, lane+32, ...
// sft[k] = softmax(u*m)[n], al[k] = alpha[n]; returns R = sum_n sft*m + 1e-13 (allennlp masked_softmax)
__device__ __forceinline__ float warp_masked_softmax(int N, const float* mask_img, const float* part, int N4, int bper,
                                                     float (&m)[ATT_NREG], float (&sft)[ATT_NREG], float (&al)[ATT_NREG]) {
  const int lane = threadIdx.x & 31;
  float x[ATT_NREG];
  float mx = -INFINITY;
#pragma unroll
  for (int k = 0; k < ATT_NREG; ++k) {
    const int n = lane + 32 * k;
    m[k] = (n < N) ? mask_img[n] : 0.f;
    x[k] = (n < N) ? gather_partial(part, N4, N, bper, n) * m[k] : -INFINITY;
    mx = fmaxf(mx, x[k]);
  }
  mx = warp_max(mx);
  float se = 0.f;
#pragma unroll
  for (int k = 0; k < ATT_NREG; ++k) {
    x[k] = (lane + 32 * k < N) ? __expf(x[k] - mx) : 0.f;
    se += x[k];
  }
  se = warp_sum(se);
  float sr = 0.f;
#pragma unroll
  for (int k = 0; k < ATT_NREG; ++k) {
    sft[k] = x[k] / se;
    sr += sft[k] * m[k];
  }
  sr = warp_sum(sr);
  const float Rn = sr + 1e-13f;
#pragma unroll
  for (int k = 0; k < ATT_NREG; ++k) al[k] = sft[k] * m[k] / Rn;
  return Rn;
}

__device__ __forceinline__ void attn_prologue(const AttnSmem& sm, const AttnArgs& a, bool bwd) {
  if (threadIdx.x == 0) {
    for (int s = 0; s < ATT_STAGES; ++s) {
      ptx::mbar_init(&sm.full[s], 1);
      ptx::mbar_init(&sm.empty[s], ATT_CWARPS);
    }
    ptx::mbar_fence_init();
  }
  for (int i = threadIdx.x; i < a.Ap; i += blockDim.x) {
    sm.wa[i] = (i < a.A) ? a.w_a[i] : 0.f;
    sm.q0[i] = 0.f;                                 // padding columns [A, Ap) stay zero: cp.async never writes them
    sm.q0[a.Ap + i] = 0.f;
  }
  if (bwd)
    for (int i = threadIdx.x; i < sm.dxb * sm.ndx * a.Fp; i += blockDim.x) sm.dx0[i] = 0.f;
  __syncthreads();
}


// One row of the forward pass, executed by the ATT_CONSUMERS consumer threads (named barrier 1). The caller has issued
// (and committed) the cp.async prefetch of this row's q into sm.q(cur); `q_next` (or null) is prefetched into the other
// buffer while this row is processed. The producer warp streams, per row, the P chunks then the feature chunks.
// `mask_g`: the row's box mask in global memory, copied to sm.msk(cur) here; null = the caller already placed it there.
__device__ __forceinline__ void attn_fwd_row(const AttnArgs& a, const AttnPlan& pl, const AttnSmem& sm, Ring& ring, int cur,
                                             const float* mask_g, const float* q_next, float* __restrict__ alpha_row,
                                             float* __restrict__ smx_row, bf16* __restrict__ xhat_row) {
  const int tid = attn_tid();
  const int warp = tid >> 5, lane = tid & 31;
  const int nfv = a.Fp >> 3;
  const float* mask_img = sm.msk(cur);
  if (mask_g && tid < a.N) sm.msk(cur)[tid] = mask_g[tid];      // buffer `cur` was last read two rows ago
  ptx::cp_async_wait_all();
  ptx::bar_sync(1, ATT_CONSUMERS);                 // q[cur] (and the mask) landed; everybody is done with the previous row
  if (q_next) {
    prefetch_vec(sm.q(cur ^ 1), q_next, a.A);
    ptx::cp_async_commit();
  }
  for (int c = 0; c < pl.nP; ++c) {
    const int n0 = c * pl.bP, nb = min(pl.bP, a.N - n0);
    ptx::mbar_wait(&sm.full[ring.stage], ring.phase);
    chunk_scores(a, reinterpret_cast<const bf16*>(sm.stage + (size_t)ring.stage * ATT_STAGE_BYTES), n0, nb, mask_img,
                 sm.q(cur), sm.wa, sm.u, sm.N4);
    __syncwarp();
    if (lane == 0) ptx::mbar_arrive(&sm.empty[ring.stage]);
    ring.advance();
  }
  ptx::bar_sync(1, ATT_CONSUMERS);                 // all N scores are in shared memory
  float m[ATT_NREG], sft[ATT_NREG], al[ATT_NREG];
  warp_masked_softmax(a.N, mask_img, sm.u, sm.N4, pl.bP, m, sft, al);
  if (warp == 0) {
#pragma unroll
    for (int k = 0; k < ATT_NREG; ++k) {
      const int n = lane + 32 * k;
      if (n < a.N) {
        alpha_row[n] = al[k];
        if (smx_row) smx_row[n] = sft[k];
      }
    }
  }
  // weighted sum: a thread owns 8 consecutive features (one 16-byte vector per box row). The inner loop is the
  // instruction hot spot of the kernel (ncu: 39 % of all issued instructions, 46 per 8 FMAs when alpha came out of
  // registers through a select chain + shuffle): alpha is read as a shared-memory broadcast from the warp's own
  // copy, bf16 -> fp32 is one shift / one mask per element, and the box loop is unrolled.
  {
    float* mine = sm.alw + warp * sm.N4;
#pragma unroll
    for (int k = 0; k < ATT_NREG; ++k)
      if (lane + 32 * k < a.N) mine[lane + 32 * k] = al[k];
    __syncwarp();
  }
  const float* alw = sm.alw + warp * sm.N4;
  const bool two = nfv > ATT_CONSUMERS;            // uniform: a second vector per thread only when Fp > 2048
  float acc[ATT_FV][8];
#pragma unroll
  for (int v = 0; v < ATT_FV; ++v)
#pragma unroll
    for (int k = 0; k < 8; ++k) acc[v][k] = 0.f;
  for (int c = 0; c < pl.nF; ++c) {
    const int n0 = c * pl.bF, nb = min(pl.bF, a.N - n0);
    ptx::mbar_wait(&sm.full[ring.stage], ring.phase);
    const uint4* buf = reinterpret_cast<const uint4*>(sm.stage + (size_t)ring.stage * ATT_STAGE_BYTES);
    if (tid < nfv) {
#pragma unroll 4
      for (int j = 0; j < nb; ++j) {
        const float w = alw[n0 + j];
        const uint4 x = buf[(size_t)j * nfv + tid];
        acc[0][0] = fmaf(w, __uint_as_float(x.x << 16), acc[0][0]);
        acc[0][1] = fmaf(w, __uint_as_float(x.x & 0xffff0000u), acc[0][1]);
        acc[0][2] = fmaf(w, __uint_as_float(x.y << 16), acc[0][2]);
        acc[0][3] = fmaf(w, __uint_as_float(x.y & 0xffff0000u), acc[0][3]);
        acc[0][4] = fmaf(w, __uint_as_float(x.z << 16), acc[0][4]);
        acc[0][5] = fmaf(w, __uint_as_float(x.z & 0xffff0000u), acc[0][5]);
        acc[0][6] = fmaf(w, __uint_as_float(x.w << 16), acc[0][6]);
        acc[0][7] = fmaf(w, __uint_as_float(x.w & 0xffff0000u), acc[0][7]);
      }
    }
    if (two && tid + ATT_CONSUMERS < nfv) {
      for (int j = 0; j < nb; ++j) {
        const float w = alw[n0 + j];
        const uint4 x = buf[(size_t)j * nfv + tid + ATT_CONSUMERS];
        acc[1][0] = fmaf(w, __uint_as_float(x.x << 16), acc[1][0]);
        acc[1][1] = fmaf(w, __uint_as_float(x.x & 0xffff0000u), acc[1][1]);
        acc[1][2] = fmaf(w, __uint_as_float(x.y << 16), acc[1][2]);
        acc[1][3] = fmaf(w, __uint_as_float(x.y & 0xffff0000u), acc[1][3]);
        acc[1][4] = fmaf(w, __uint_as_float(x.z << 16), acc[1][4]);
        acc[1][5] = fmaf(w, __uint_as_float(x.z & 0xffff0000u), acc[1][5]);
        acc[1][6] = fmaf(w, __uint_as_float(x.w << 16), acc[1][6]);
        acc[1][7] = fmaf(w, __uint_as_float(x.w & 0xffff0000u), acc[1][7]);
      }
    }
    __syncwarp();
    if (lane == 0) ptx::mbar_arrive(&sm.empty[ring.stage]);
    ring.advance();
  }
#pragma unroll
  for (int v = 0; v < ATT_FV; ++v) {
    const int vec = tid + ATT_CONSUMERS * v;
    if (vec < nfv) {
      bf16x8 o;
#pragma unroll
      for (int k = 0; k < 4; ++k) o.v[k] = __floats2bfloat162_rn(acc[v][2 * k], acc[v][2 * k + 1]);
      st_bf16x8(xhat_row + vec * 8, o);
    }
  }
}

// One row of the per-step backward (d u saved for the deferred part, d q as the bf16 operand of the query-projection
// GEMM), executed by the ATT_CONSUMERS consumer threads of the persistent BPTT kernel (recurrent_bwd.cu). Same math as
// attention.cu: attention_bwd_kernel. The caller has issued (and committed) the cp.async prefetch of this row's q,
// saved softmax and d xhat (sm.ndx split-K slots, each in the two-plane layout: quad q of the row at float offset
// (q & 1) * Fp/2 + (q >> 1) * 4) into buffer `cur`; `prefetch_next()` issues the next row's.
// The producer warp streams, per row, the feature chunks then the P chunks.
struct NoStamp { __device__ __forceinline__ void operator()(int) const {} };
// `after_dalpha()` runs once the d xhat buffer of this row is no longer needed (single-buffered d xhat: the caller issues the
// next row's d xhat prefetch there).
struct NoCall { __device__ __forceinline__ void operator()() const {} };
template <typename PrefetchNext, typename AfterDalpha = NoCall, typename Stamp = NoStamp>
__device__ __forceinline__ void attn_bwd_row(const AttnArgs& a, const AttnPlan& pl, const AttnSmem& sm, Ring& ring, int cur,
                                             const float* mask_g, PrefetchNext prefetch_next, bf16* __restrict__ dq_row,
                                             int ld_dq, float* __restrict__ du_row, AfterDalpha after_dalpha = AfterDalpha(),
                                             Stamp stamp = Stamp()) {
  const int tid = attn_tid();
  const int warp = tid >> 5, lane = tid & 31;
  const int nfv = a.Fp >> 3, npair = a.Ap >> 1;
  const float* mask_img = sm.msk(cur);               // mask_g: as for attn_fwd_row
  if (mask_g && tid < a.N) sm.msk(cur)[tid] = mask_g[tid];
  ptx::cp_async_wait_all();
  ptx::bar_sync(1, ATT_CONSUMERS);
  stamp(0);
  prefetch_next();
  float* dx_s = sm.dx(cur, 0);
  if (sm.ndx > 1) {                                  // sum the split-K slots of d xhat in place
    for (int k = 1; k < sm.ndx; ++k) {
      const float4* o = reinterpret_cast<const float4*>(sm.dx(cur, k));
      for (int i = tid; i < (a.Fp >> 2); i += ATT_CONSUMERS) {
        float4 v = reinterpret_cast<float4*>(dx_s)[i];
        const float4 w = o[i];
        v.x += w.x; v.y += w.y; v.z += w.z; v.w += w.w;
        reinterpret_cast<float4*>(dx_s)[i] = v;
      }
    }
    ptx::bar_sync(1, ATT_CONSUMERS);
  }
  stamp(1);
  // d alpha_n = d xhat . x_n. d xhat sits in shared memory as two planes (floats 0-3 / 4-7 of every group of 8: both
  // 16-byte reads of a lane are then conflict-free). A full chunk (8 boxes) runs in pair mode: a warp owns one half of
  // the vectors of TWO boxes, so that every d xhat vector it reads serves two boxes (the per-box form re-reads the
  // 8 KB of d xhat for each of the 36 boxes: 2/3 of the phase's shared-memory traffic); partials are added by the readers.
  const float4* dx_lo = reinterpret_cast<const float4*>(dx_s);
  const float4* dx_hi = reinterpret_cast<const float4*>(dx_s + (a.Fp >> 1));
  for (int c = 0; c < pl.nF; ++c) {
    const int n0 = c * pl.bF, nb = min(pl.bF, a.N - n0);
    ptx::mbar_wait(&sm.full[ring.stage], ring.phase);
    const bf16x8* buf = reinterpret_cast<const bf16x8*>(sm.stage + (size_t)ring.stage * ATT_STAGE_BYTES);
    if (nb == ATT_CWARPS) {
      const int pr = warp >> 1, half = warp & 1, hv = nfv >> 1;
      const int na = n0 + 2 * pr;
      const bool ma = mask_img[na] != 0.f, mb = mask_img[na + 1] != 0.f;
      float sa = 0.f, sb = 0.f;
      if (ma || mb) {
        const bf16x8* pa = buf + (size_t)(2 * pr) * nfv;
        const bf16x8* pb = pa + nfv;
        float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f, b0 = 0.f, b1 = 0.f, b2 = 0.f, b3 = 0.f;
#pragma unroll 2
        for (int i = half * hv + lane; i < (half + 1) * hv; i += 32) {
          const float4 da = dx_lo[i], db = dx_hi[i];
          const bf16x8 va = pa[i], vb = pb[i];
          float2 f0 = __bfloat1622float2(va.v[0]), f1 = __bfloat1622float2(va.v[1]);
          float2 f2 = __bfloat1622float2(va.v[2]), f3 = __bfloat1622float2(va.v[3]);
          a0 = fmaf(da.x, f0.x, fmaf(da.y, f0.y, a0));
          a1 = fmaf(da.z, f1.x, fmaf(da.w, f1.y, a1));
          a2 = fmaf(db.x, f2.x, fmaf(db.y, f2.y, a2));
          a3 = fmaf(db.z, f3.x, fmaf(db.w, f3.y, a3));
          f0 = __bfloat1622float2(vb.v[0]); f1 = __bfloat1622float2(vb.v[1]);
          f2 = __bfloat1622float2(vb.v[2]); f3 = __bfloat1622float2(vb.v[3]);
          b0 = fmaf(da.x, f0.x, fmaf(da.y, f0.y, b0));
          b1 = fmaf(da.z, f1.x, fmaf(da.w, f1.y, b1));
          b2 = fmaf(db.x, f2.x, fmaf(db.y, f2.y, b2));
          b3 = fmaf(db.z, f3.x, fmaf(db.w, f3.y, b3));
        }
        sa = (a0 + a1) + (a2 + a3);
        sb = (b0 + b1) + (b2 + b3);
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {             // two interleaved butterfly sums
          sa += __shfl_xor_sync(0xffffffffu, sa, o);
          sb += __shfl_xor_sync(0xffffffffu, sb, o);
        }
      }
      if (lane == 0) {
        sm.u[half * sm.N4 + na] = ma ? sa : 0.f;
        sm.u[half * sm.N4 + na + 1] = mb ? sb : 0.f;
      }
    } else {
      const int wpb = warps_per_box(nb);
      const int j = warp >> wpb_log2(wpb), sub = warp & (wpb - 1);
      if (j < nb) {
        const int n = n0 + j;
        float s = 0.f;
        if (mask_img[n] != 0.f) {
          const bf16x8* p = buf + (size_t)j * nfv;
          float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f;
#pragma unroll 2
          for (int i = sub * 32 + lane; i < nfv; i += 32 * wpb) {
            const bf16x8 v = p[i];
            const float4 da = dx_lo[i], db = dx_hi[i];
            const float2 f0 = __bfloat1622float2(v.v[0]), f1 = __bfloat1622float2(v.v[1]);
            const float2 f2 = __bfloat1622float2(v.v[2]), f3 = __bfloat1622float2(v.v[3]);
            s0 = fmaf(da.x, f0.x, fmaf(da.y, f0.y, s0));
            s1 = fmaf(da.z, f1.x, fmaf(da.w, f1.y, s1));
            s2 = fmaf(db.x, f2.x, fmaf(db.y, f2.y, s2));
            s3 = fmaf(db.z, f3.x, fmaf(db.w, f3.y, s3));
          }
          s = warp_sum((s0 + s1) + (s2 + s3));
        }
        if (lane == 0) sm.u[sub * sm.N4 + n] = s;
      }
    }
    __syncwarp();
    if (lane == 0) ptx::mbar_arrive(&sm.empty[ring.stage]);
    ring.advance();
  }
  ptx::bar_sync(1, ATT_CONSUMERS);
  after_dalpha();
  stamp(2);
  // softmax backward, redundantly per warp (see attention_bwd_kernel)
  float duv[ATT_NREG];
  {
    float m[ATT_NREG], sv[ATT_NREG], da[ATT_NREG];
    float sr = 0.f;
#pragma unroll
    for (int k = 0; k < ATT_NREG; ++k) {
      const int n = lane + 32 * k;
      const bool ok = n < a.N;
      m[k] = ok ? mask_img[n] : 0.f;
      sv[k] = ok ? sm.sv(cur)[n] : 0.f;
      da[k] = ok ? gather_partial(sm.u, sm.N4, a.N, pl.bF, n, true) : 0.f;
      sr += sv[k] * m[k];
    }
    const float Rn = warp_sum(sr) + 1e-13f;
    float dot = 0.f;
#pragma unroll
    for (int k = 0; k < ATT_NREG; ++k) dot += da[k] * (sv[k] * m[k] / Rn);
    dot = warp_sum(dot);
    float dss = 0.f;
#pragma unroll
    for (int k = 0; k < ATT_NREG; ++k) {
      da[k] = (da[k] - dot) / Rn * m[k];
      dss += da[k] * sv[k];
    }
    dss = warp_sum(dss);
#pragma unroll
    for (int k = 0; k < ATT_NREG; ++k) duv[k] = sv[k] * (da[k] - dss) * m[k];
  }
  if (warp == 0) {
#pragma unroll
    for (int k = 0; k < ATT_NREG; ++k) {
      const int n = lane + 32 * k;
      if (n < a.N) du_row[n] = duv[k];
    }
  }
  stamp(3);
  // d q_a = w_a sum_n du_n (1 - tanh^2(q_a + P_na)): a thread owns pairs of projection columns. Four boxes per iteration
  // without a branch on d u (a masked box contributes d = 0): 8 - 16 independent tanh chains per thread instead of one.
  const float* q_s = sm.q(cur);
  float g[ATT_PV][2], qv[ATT_PV][2];
#pragma unroll
  for (int v = 0; v < ATT_PV; ++v) {
    g[v][0] = g[v][1] = 0.f;
    const int cp = tid + ATT_CONSUMERS * v;
    qv[v][0] = cp < npair ? q_s[2 * cp] : 0.f;
    qv[v][1] = cp < npair ? q_s[2 * cp + 1] : 0.f;
  }
  bool any = false;                                  // padded timesteps: every d u is zero, nothing to add
#pragma unroll
  for (int k = 0; k < ATT_NREG; ++k) any = any || duv[k] != 0.f;
  any = __any_sync(0xffffffffu, any);
  for (int c = 0; c < pl.nP; ++c) {
    const int n0 = c * pl.bP, nb = min(pl.bP, a.N - n0);
    ptx::mbar_wait(&sm.full[ring.stage], ring.phase);
    const __nv_bfloat162* buf = reinterpret_cast<const __nv_bfloat162*>(sm.stage + (size_t)ring.stage * ATT_STAGE_BYTES);
    if (any) {
      for (int j0 = 0; j0 < nb; j0 += 4) {
        float d[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const int n = min(n0 + j0 + u, a.N - 1);
          const float dv = __shfl_sync(0xffffffffu, pick(duv, n >> 5), n & 31);
          d[u] = (j0 + u < nb) ? dv : 0.f;
        }
#pragma unroll
        for (int v = 0; v < ATT_PV; ++v) {
          const int cp = tid + ATT_CONSUMERS * v;
          if (cp < npair) {
#pragma unroll
            for (int u = 0; u < 4; ++u) {
              const int jj = min(j0 + u, nb - 1);    // clamped: the box exists, its weight d[u] is zero
              const float2 f = __bfloat1622float2(buf[(size_t)jj * npair + cp]);
              const float t0 = tanh_approx(qv[v][0] + f.x), t1 = tanh_approx(qv[v][1] + f.y);
              g[v][0] = fmaf(d[u], 1.f - t0 * t0, g[v][0]);
              g[v][1] = fmaf(d[u], 1.f - t1 * t1, g[v][1]);
            }
          }
        }
      }
    }
    __syncwarp();
    if (lane == 0) ptx::mbar_arrive(&sm.empty[ring.stage]);
    ring.advance();
  }
  stamp(4);
#pragma unroll
  for (int v = 0; v < ATT_PV; ++v) {
    const int cp = tid + ATT_CONSUMERS * v;
    if (cp < npair && 2 * cp < ld_dq)
      *reinterpret_cast<__nv_bfloat162*>(dq_row + 2 * cp) = __floats2bfloat162_rn(sm.wa[2 * cp] * g[v][0], sm.wa[2 * cp + 1] * g[v][1]);
  }
}

}  // namespace
}  // namespace attn
}  // namespace sscvae

// Training-step tail (SURVEY §8(f)-1): global grad-norm clipping + SGD(momentum, weight decay) fused
// over a flat fp32 parameter buffer; replaces clip_grad_norm_ / optimizer.step of
// var_updown/scripts/train.py:173-176 (~100 small launches in eager PyTorch) with three launches.
#include "../../include/sscvae.h"
#include "kernels.cuh"
#include "prof.cuh"

namespace sscvae {
extern unsigned long long g_launch_count_pw;
#define LAUNCHED() do { CUDA_TRY(cudaGetLastError()); ++g_launch_count_pw; } while (0)

static constexpr int NORM_BLOCKS = 1024;

__global__ void sqnorm_partial_kernel(const float* __restrict__ g, size_t n, float* __restrict__ partial) {
  __shared__ float red[32];
  float s = 0.f;
  const size_t n4 = n / 4;
  const float4* g4 = reinterpret_cast<const float4*>(g);
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (size_t)gridDim.x * blockDim.x) {
    const float4 v = g4[i];
    s += v.x * v.x + v.y * v.y + v.z * v.z + v.w * v.w;
  }
  if (blockIdx.x == 0)
    for (size_t i = n4 * 4 + threadIdx.x; i < n; i += blockDim.x) s += g[i] * g[i];
  s = warp_sum(s);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
  __syncthreads();
  if (threadIdx.x < 32) {
    float v = (threadIdx.x < (blockDim.x >> 5)) ? red[threadIdx.x] : 0.f;
    v = warp_sum(v);
    if (threadIdx.x == 0) partial[blockIdx.x] = v;
  }
}
__global__ void sqnorm_final_kernel(const float* __restrict__ partial, int n, float* __restrict__ out) {
  __shared__ float red[32];
  float s = 0.f;
  for (int i = threadIdx.x; i < n; i += blockDim.x) s += partial[i];
  s = warp_sum(s);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
  __syncthreads();
  if (threadIdx.x < 32) {
    float v = (threadIdx.x < (blockDim.x >> 5)) ? red[threadIdx.x] : 0.f;
    v = warp_sum(v);
    if (threadIdx.x == 0) *out = v;
  }
}

__global__ void sgd_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m, size_t n,
                           const float* __restrict__ sqnorm, float max_norm, float lr, float momentum, float wd,
                           int first) {
  // torch.nn.utils.clip_grad_norm_: coef = max_norm / (norm + 1e-6), applied only when < 1
  float coef = 1.f;
  if (sqnorm && max_norm > 0.f) coef = fminf(1.f, max_norm / (sqrtf(*sqnorm) + 1e-6f));
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
    const float w = p[i];
    float d = g[i] * coef + wd * w;
    if (momentum != 0.f) {
      const float b = first ? d : momentum * m[i] + d;
      m[i] = b;
      d = b;
    }
    p[i] = w - lr * d;
  }
}
// ---- multi-tensor form: every parameter of the model in three launches ---------------------------------
static constexpr int MT_MAX = 32;
static constexpr unsigned MT_CHUNK = 16384;            // elements per block
struct MultiTensorTable {
  float* p[MT_MAX]; const float* g[MT_MAX]; float* m[MT_MAX];
  unsigned long long n[MT_MAX];
  unsigned chunk0[MT_MAX + 1];                         // first chunk (block) of tensor i
  int first[MT_MAX];
  int count;
};

__device__ __forceinline__ int mt_find(const MultiTensorTable& t, unsigned block) {
  int i = 0;
  while (i + 1 < t.count && block >= t.chunk0[i + 1]) ++i;
  return i;
}

__global__ void __launch_bounds__(256) mt_sqnorm_kernel(const __grid_constant__ MultiTensorTable t, float gscale, float* __restrict__ partial) {
  __shared__ float red[8];
  const int ti = mt_find(t, blockIdx.x);
  const size_t lo = (size_t)(blockIdx.x - t.chunk0[ti]) * MT_CHUNK;
  const size_t hi = min((size_t)t.n[ti], lo + MT_CHUNK);
  const float* g = t.g[ti];
  float s = 0.f;
  if (g)                                               // NULL gradient = all zeros (see sscvae_sgd_step_multi)
    for (size_t i = lo + threadIdx.x; i < hi; i += 256) { const float v = g[i] * gscale; s += v * v; }
  s = warp_sum(s);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
  __syncthreads();
  if (threadIdx.x == 0) {
    float v = 0.f;
    for (int w = 0; w < 8; ++w) v += red[w];
    partial[blockIdx.x] = v;                           // fixed chunking + ordered sums: deterministic
  }
}

__global__ void __launch_bounds__(256) mt_sgd_kernel(const __grid_constant__ MultiTensorTable t, const float* __restrict__ sqnorm,
                                                     float max_norm, float lr, float momentum, float wd, float gscale) {
  const int ti = mt_find(t, blockIdx.x);
  const size_t lo = (size_t)(blockIdx.x - t.chunk0[ti]) * MT_CHUNK;
  const size_t hi = min((size_t)t.n[ti], lo + MT_CHUNK);
  float coef = 1.f;
  if (max_norm > 0.f) coef = fminf(1.f, max_norm / (sqrtf(*sqnorm) + 1e-6f));   // torch clip_grad_norm_
  coef *= gscale;                                      // gradients arrive as a SUM over ranks: the mean is taken here
  float* p = t.p[ti]; const float* g = t.g[ti]; float* m = t.m[ti];
  const bool first = t.first[ti] != 0;
  for (size_t i = lo + threadIdx.x; i < hi; i += 256) {
    const float w = p[i];
    float d = (g ? g[i] * coef : 0.f) + wd * w;
    if (momentum != 0.f) {
      const float b = first ? d : momentum * m[i] + d;
      m[i] = b;
      d = b;
    }
    p[i] = w - lr * d;
  }
}

// Fills the squared-norm partials of the table's gradients (fixed chunking, one partial per chunk) and their ordered sum
// at scratch[chunks]: the clip coefficient of every update path comes from here.
static int mt_grad_sqnorm(cudaStream_t st, const MultiTensorTable& t, float gscale, float* scratch, size_t scratch_floats) {
  const unsigned chunks = t.chunk0[t.count];
  REQUIRE(scratch_floats >= (size_t)chunks + 1, "scratch too small: need %u floats", chunks + 1);
  mt_sqnorm_kernel<<<chunks, 256, 0, st>>>(t, gscale, scratch);
  LAUNCHED();
  sqnorm_final_kernel<<<1, 1024, 0, st>>>(scratch, (int)chunks, scratch + chunks);
  LAUNCHED();
  return 0;
}
static void mt_set(MultiTensorTable& t, int i, float* p, const float* g, float* m, unsigned long long n, int first) {
  t.p[i] = p; t.g[i] = g; t.m[i] = m; t.n[i] = n; t.first[i] = first;
  t.chunk0[i + 1] = t.chunk0[i] + (unsigned)((n + MT_CHUNK - 1) / MT_CHUNK);
  t.count = i + 1;
}

// ---- clip + SGD + weight packing in one launch (kernels.cuh: SgdPackTable) ------------------------------------------
// A CTA owns a 64 x 64 tile of one source block. Update phase: each thread loads, updates (mt_sgd_kernel's expressions)
// and stores 16 elements of the tile per tensor (a warp covers 128 or 256 contiguous bytes of a row) and keeps v = w (+ w2).
// Pack phase: v goes to the fp32 images from registers, and as bf16 through a shared-memory tile of 64 rows x 128 bytes,
// 16-byte chunk c of row i stored at chunk c ^ ((i >> 3) & 7) (transpose_bf16_jobs_kernel's layout: the 16-byte row
// reads of the plain image and the 4-byte column reads of the transposed image are both free of bank conflicts), to the
// bf16 images with 16-byte stores (element stores at a ragged edge or a destination that is not 16-byte aligned).
__device__ __forceinline__ void store_bf16x8(bf16* dst, const uint4& x, int n) {
  if (n >= 8 && (reinterpret_cast<uintptr_t>(dst) & 15) == 0) { *reinterpret_cast<uint4*>(dst) = x; return; }
  const uint32_t w[4] = {x.x, x.y, x.z, x.w};
#pragma unroll
  for (int k = 0; k < 8; ++k)
    if (k < n) dst[k] = __ushort_as_bfloat16((unsigned short)(w[k >> 1] >> (16 * (k & 1))));
}

// element q of this thread: tile row / column (VW = 4: four consecutive columns per 16-byte access)
template <int VW>
__device__ __forceinline__ void tile_pos(int q, int& i, int& j) {
  const int idx = threadIdx.x + (q / VW) * 256;
  if (VW == 1) { i = idx >> 6; j = idx & 63; }
  else { i = idx >> 4; j = (idx & 15) * 4 + (q & 3); }
}

// v[q] = the (updated, when T.upd) value of element q of the tile at p + base (row stride ld, nr x nc valid)
template <int VW>
__device__ __forceinline__ void tile_update(const SgdPackTensor& T, size_t base, int ld, int nr, int nc, float coef,
                                            const SgdParams& sp, float (&v)[16]) {
  float gv[16], mv[16];
  const bool upd = T.upd != 0, has_g = upd && T.g != nullptr, first = T.first != 0, mom = sp.momentum != 0.f;
#pragma unroll
  for (int q = 0; q < 16; q += VW) {
    int i, j;
    tile_pos<VW>(q, i, j);
    if (i < nr && j < nc) {
      const size_t o = base + (size_t)i * ld + j;
      if (VW == 4) {
        const float4 a = *reinterpret_cast<const float4*>(T.p + o);
        v[q] = a.x; v[q + 1] = a.y; v[q + 2] = a.z; v[q + 3] = a.w;
        if (has_g) {
          const float4 b = *reinterpret_cast<const float4*>(T.g + o);
          gv[q] = b.x; gv[q + 1] = b.y; gv[q + 2] = b.z; gv[q + 3] = b.w;
        }
        if (upd && mom && !first) {
          const float4 c = *reinterpret_cast<const float4*>(T.m + o);
          mv[q] = c.x; mv[q + 1] = c.y; mv[q + 2] = c.z; mv[q + 3] = c.w;
        }
      } else {
        v[q] = T.p[o];
        if (has_g) gv[q] = T.g[o];
        if (upd && mom && !first) mv[q] = T.m[o];
      }
    }
  }
  if (!upd) return;
#pragma unroll
  for (int q = 0; q < 16; ++q) {
    const float w = v[q];
    float d = (has_g ? gv[q] * coef : 0.f) + sp.wd * w;
    if (mom) {
      const float b = first ? d : sp.momentum * mv[q] + d;
      mv[q] = b;
      d = b;
    }
    v[q] = w - sp.lr * d;
  }
#pragma unroll
  for (int q = 0; q < 16; q += VW) {
    int i, j;
    tile_pos<VW>(q, i, j);
    if (i < nr && j < nc) {
      const size_t o = base + (size_t)i * ld + j;
      if (VW == 4) {
        *reinterpret_cast<float4*>(T.p + o) = make_float4(v[q], v[q + 1], v[q + 2], v[q + 3]);
        if (mom) *reinterpret_cast<float4*>(T.m + o) = make_float4(mv[q], mv[q + 1], mv[q + 2], mv[q + 3]);
      } else {
        T.p[o] = v[q];
        if (mom) T.m[o] = mv[q];
      }
    }
  }
}

template <int VW>
__device__ __forceinline__ void sgd_pack_tile(const SgdPackTable& t, const SgdPackJob& j, int r0, int cb, float coef,
                                              const SgdParams& sp, uint8_t* tile) {
  const int nr = min(64, j.rows - r0), nc = min(64, j.cols - cb);
  float v[16];
  tile_update<VW>(t.t[j.w], (size_t)r0 * j.ld + j.c0 + cb, j.ld, nr, nc, coef, sp, v);
  if (j.w2 >= 0) {                                     // fold: bf16(w_ih + w_hh), pack_weights' summation order
    float v2[16];
    tile_update<VW>(t.t[j.w2], (size_t)r0 * j.ld2 + cb, j.ld2, nr, nc, coef, sp, v2);
#pragma unroll
    for (int q = 0; q < 16; ++q) v[q] += v2[q];
  }
  for (int o = 0; o < j.nout; ++o) {
    const SgdPackOut& out = j.out[o];
    if (out.kind != kPackF32) continue;
#pragma unroll
    for (int q = 0; q < 16; ++q) {
      int i, jj;
      tile_pos<VW>(q, i, jj);
      if (i < nr && jj < nc) reinterpret_cast<float*>(out.dst)[(size_t)(r0 + i) * out.ld + cb + jj] = v[q];
    }
  }
#pragma unroll
  for (int q = 0; q < 16; ++q) {
    int i, jj;
    tile_pos<VW>(q, i, jj);
    *reinterpret_cast<bf16*>(tile + i * 128 + (((jj >> 3) ^ ((i >> 3) & 7)) << 4) + (jj & 7) * 2) = __float2bfloat16_rn(v[q]);
  }
}

__global__ void __launch_bounds__(256, 3) sgd_pack_kernel(const __grid_constant__ SgdPackTable t, const SgdParams sp,
                                                       const float* __restrict__ sqnorm) {
  __shared__ __align__(16) uint8_t tile[64 * 128];
  int ji = 0;
  while (ji + 1 < t.n && (int)blockIdx.x >= t.job[ji + 1].tile0) ++ji;
  const SgdPackJob& j = t.job[ji];
  const int local = blockIdx.x - j.tile0;
  const int r0 = (local / j.tiles_x) * 64, cb = (local % j.tiles_x) * 64;
  float coef = 1.f;
  if (sp.max_norm > 0.f) coef = fminf(1.f, sp.max_norm / (sqrtf(*sqnorm) + 1e-6f));   // torch clip_grad_norm_
  coef *= sp.gscale;
  if (j.vec) sgd_pack_tile<4>(t, j, r0, cb, coef, sp, tile);
  else sgd_pack_tile<1>(t, j, r0, cb, coef, sp, tile);
  __syncthreads();
  for (int o = 0; o < j.nout; ++o) {
    const SgdPackOut& out = j.out[o];
    bf16* dst = reinterpret_cast<bf16*>(out.dst);
    if (out.kind == kPackPlain) {
#pragma unroll
      for (int it = 0; it < 2; ++it) {
        const int v = threadIdx.x + it * 256;
        const int i = v >> 3, cv = v & 7;
        const int r = r0 + i, c = cb + cv * 8;
        if (r < j.rows && c < j.cols) {
          const uint4 x = *reinterpret_cast<const uint4*>(tile + i * 128 + ((cv ^ ((i >> 3) & 7)) << 4));
          const int rd = out.gate_H ? lstm_gate_row(r / out.gate_H, r % out.gate_H) : r;
          store_bf16x8(dst + (size_t)rd * out.ld + c, x, j.cols - c);
        }
      }
    } else if (out.kind == kPackTransposed) {          // dst[c, r] = v[r, c]
      const int lane = threadIdx.x & 31, rv = lane & 7;
      const int jw = (threadIdx.x >> 5) * 4 + (lane >> 3);                  // 4-byte word = tile columns 2jw, 2jw + 1
      uint32_t w[8];
#pragma unroll
      for (int k = 0; k < 8; ++k)
        w[k] = *reinterpret_cast<const uint32_t*>(tile + (8 * rv + k) * 128 + (((jw >> 2) ^ rv) << 4) + ((jw & 3) << 2));
      uint4 lo, hi;                                                         // column 2jw / 2jw + 1, tile rows 8rv .. 8rv + 7
      lo.x = __byte_perm(w[0], w[1], 0x5410); hi.x = __byte_perm(w[0], w[1], 0x7632);
      lo.y = __byte_perm(w[2], w[3], 0x5410); hi.y = __byte_perm(w[2], w[3], 0x7632);
      lo.z = __byte_perm(w[4], w[5], 0x5410); hi.z = __byte_perm(w[4], w[5], 0x7632);
      lo.w = __byte_perm(w[6], w[7], 0x5410); hi.w = __byte_perm(w[6], w[7], 0x7632);
      const int c = cb + 2 * jw, r = r0 + 8 * rv;
      if (r < j.rows) {
        if (c < j.cols) store_bf16x8(dst + (size_t)c * out.ld + r, lo, j.rows - r);
        if (c + 1 < j.cols) store_bf16x8(dst + (size_t)(c + 1) * out.ld + r, hi, j.rows - r);
      }
    }
  }
}

static bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

static int sgd_pack_launch(cudaStream_t s, SgdPackTable& t, const SgdParams& sp, const float* sqnorm) {
  if (t.n == 0) return 0;
  double bytes = 0;
  int tiles = 0;
  bool upd = false;
  for (int i = 0; i < t.n; ++i) {
    SgdPackJob& j = t.job[i];
    REQUIRE(j.w >= 0 && j.w < kMaxSgdPackTensors && j.w2 < kMaxSgdPackTensors && j.rows > 0 && j.cols > 0 && j.nout <= 2,
            "sgd_pack: bad job %d", i);
    j.tiles_x = ceil_div(j.cols, 64);
    j.tile0 = tiles;
    tiles += j.tiles_x * ceil_div(j.rows, 64);
    const SgdPackTensor& a = t.t[j.w];
    j.vec = j.c0 % 4 == 0 && j.cols % 4 == 0 && j.ld % 4 == 0 && aligned16(a.p) && aligned16(a.g) && aligned16(a.m);
    if (j.w2 >= 0) {
      const SgdPackTensor& b = t.t[j.w2];
      j.vec = j.vec && j.ld2 % 4 == 0 && aligned16(b.p) && aligned16(b.g) && aligned16(b.m);
    }
    const double e = (double)j.rows * j.cols;
    for (int w : {j.w, j.w2}) {
      if (w < 0) continue;
      upd = upd || t.t[w].upd;
      bytes += e * (t.t[w].upd ? 8.0 + (t.t[w].g ? 4.0 : 0.0) + (sp.momentum != 0.f ? (t.t[w].first ? 4.0 : 8.0) : 0.0) : 4.0);
    }
    for (int o = 0; o < j.nout; ++o) bytes += e * (j.out[o].kind == kPackF32 ? 4.0 : 2.0);
  }
  PROF_SCOPE(s, upd ? "optim" : "pack_weights", 0, bytes);
  sgd_pack_kernel<<<tiles, 256, 0, s>>>(t, sp, sqnorm);
  LAUNCHED();
  return 0;
}

int sgd_pack(cudaStream_t s, SgdPackTable& t) {
  for (const SgdPackTensor& x : t.t) REQUIRE(!x.upd, "sgd_pack: the plain pack updates no tensor");
  return sgd_pack_launch(s, t, SgdParams{0.f, 0.f, 0.f, 0.f, 1.f}, nullptr);
}

int sgd_pack_step(cudaStream_t s, SgdPackTable& t, const int* order, int count, const SgdParams& sp, float* scratch,
                  size_t scratch_floats) {
  REQUIRE(count > 0 && count <= MT_MAX && order && scratch, "bad argument");
  MultiTensorTable mt;
  mt.chunk0[0] = 0;
  for (int i = 0; i < count; ++i) {
    const int w = order[i];
    REQUIRE(w >= 0 && w < kMaxSgdPackTensors && t.t[w].upd, "sgd_pack_step: tensor %d is not updated", w);
    mt_set(mt, i, t.t[w].p, t.t[w].g, t.t[w].m, t.t[w].n, t.t[w].first);
  }
  TRY(mt_grad_sqnorm(s, mt, sp.gscale, scratch, scratch_floats));
  return sgd_pack_launch(s, t, sp, scratch + mt.chunk0[count]);
}
}  // namespace sscvae

using namespace sscvae;
extern "C" {
int sscvae_sgd_step_multi(int count, void* const* params, const void* const* grads, void* const* momentum_bufs,
                          const uint64_t* sizes, const int32_t* first_step, float max_norm, float lr, float momentum,
                          float weight_decay, float grad_scale, float* scratch, size_t scratch_floats, void* stream) {
  REQUIRE(count > 0 && count <= MT_MAX && params && grads && sizes && first_step && scratch, "bad argument (at most %d tensors)", MT_MAX);
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  MultiTensorTable t;
  t.chunk0[0] = 0;
  for (int i = 0; i < count; ++i) {
    // grads[i] == NULL: a zero gradient (torch 1.1's zero_grad() leaves ZERO tensors behind, so a parameter frozen by
    // train.py:156-161 keeps decaying and coasting on its momentum; see FusedClipSGD(legacy_zero_grad=True))
    REQUIRE(params[i] && (momentum == 0.f || (momentum_bufs && momentum_bufs[i])), "NULL tensor %d", i);
    mt_set(t, i, reinterpret_cast<float*>(params[i]), reinterpret_cast<const float*>(grads[i]),
           momentum_bufs ? reinterpret_cast<float*>(momentum_bufs[i]) : nullptr, sizes[i], first_step[i]);
  }
  TRY(mt_grad_sqnorm(st, t, grad_scale, scratch, scratch_floats));
  const unsigned chunks = t.chunk0[count];
  mt_sgd_kernel<<<chunks, 256, 0, st>>>(t, scratch + chunks, max_norm, lr, momentum, weight_decay, grad_scale);
  LAUNCHED();
  return 0;
}

int sscvae_grad_sqnorm(const float* grads, size_t n, float* partial, float* sqnorm_out, void* stream) {
  REQUIRE(grads && partial && sqnorm_out, "NULL argument");
  REQUIRE((reinterpret_cast<uintptr_t>(grads) & 15) == 0, "grads must be 16-byte aligned");
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  sqnorm_partial_kernel<<<NORM_BLOCKS, 256, 0, st>>>(grads, n, partial);
  LAUNCHED();
  sqnorm_final_kernel<<<1, 1024, 0, st>>>(partial, NORM_BLOCKS, sqnorm_out);
  LAUNCHED();
  return 0;
}
int sscvae_sgd_step(float* params, const float* grads, float* momentum_buf, size_t n, const float* sqnorm, float max_norm,
                    float lr, float momentum, float weight_decay, int first_step, void* stream) {
  REQUIRE(params && grads && (momentum == 0.f || momentum_buf), "NULL argument");
  sgd_kernel<<<1184, 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(params, grads, momentum_buf, n, sqnorm, max_norm,
                                                                      lr, momentum, weight_decay, first_step);
  LAUNCHED();
  return 0;
}
}

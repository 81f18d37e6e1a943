// Pointwise / reduction kernels of the var_updown decoder path (everything that is not a GEMM, the
// region attention or the search). All are HBM- or latency-bound: coalesced along the feature axis,
// 16-byte vector accesses where the layout allows, warp-shuffle reductions.
#include "kernels.cuh"
#include "prof.cuh"
#include <curand_kernel.h>

namespace sscvae {

unsigned long long g_launch_count_pw = 0;
#define LAUNCHED() do { CUDA_TRY(cudaGetLastError()); ++g_launch_count_pw; } while (0)

// ---------------------------------------------------------------------------------------------
// image_prep: one CTA per image. Pass 1: bf16 copy + per-box |x| sum -> mask. Pass 2: masked mean.
// ---------------------------------------------------------------------------------------------
// TIn = float (the reference's region features) or bf16 (the bf16 feature cache of SURVEY 8(f)-3: the masked mean is taken
// over the bf16-rounded values either way, so both inputs give bit-identical featsb / avgb).
template <typename TIn>
__global__ void image_prep_kernel(const TIn* __restrict__ feats, int N, int F, bf16* __restrict__ featsb, int Fp,
                                  float* __restrict__ mask, bf16* __restrict__ avgb) {
  extern __shared__ float s_mask[];                 // N
  const int b = blockIdx.x;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nwarp = blockDim.x >> 5;
  const TIn* x = feats + (size_t)b * N * F;
  bf16* xb = featsb + (size_t)b * N * Fp;
  // 16-byte loads when the rows allow it (F % 4 == 0, 16-byte aligned base: every row then starts on a 16-byte boundary for
  // fp32 and on an 8-byte boundary for bf16 input); the scalar loop otherwise
  const bool vec = (F & 3) == 0 && (reinterpret_cast<uintptr_t>(x) & 15) == 0;
  for (int n = warp; n < N; n += nwarp) {
    float s = 0.f;
    if (vec) {
      const int nq = F >> 2;
#pragma unroll 4
      for (int q = lane; q < (Fp >> 2); q += 32) {
        float v0 = 0.f, v1 = 0.f, v2 = 0.f, v3 = 0.f;
        if (q < nq) {
          if (sizeof(TIn) == 4) {
            const float4 v = *reinterpret_cast<const float4*>(reinterpret_cast<const float*>(x) + (size_t)n * F + 4 * q);
            v0 = v.x; v1 = v.y; v2 = v.z; v3 = v.w;
          } else {
            const uint2 v = *reinterpret_cast<const uint2*>(reinterpret_cast<const bf16*>(x) + (size_t)n * F + 4 * q);
            v0 = __uint_as_float(v.x << 16); v1 = __uint_as_float(v.x & 0xffff0000u);
            v2 = __uint_as_float(v.y << 16); v3 = __uint_as_float(v.y & 0xffff0000u);
          }
        }
        s += (fabsf(v0) + fabsf(v1)) + (fabsf(v2) + fabsf(v3));
        const __nv_bfloat162 lo = __floats2bfloat162_rn(v0, v1), hi = __floats2bfloat162_rn(v2, v3);
        uint2 o;
        o.x = *reinterpret_cast<const uint32_t*>(&lo);
        o.y = *reinterpret_cast<const uint32_t*>(&hi);
        *reinterpret_cast<uint2*>(xb + (size_t)n * Fp + 4 * q) = o;
      }
    } else {
      for (int f = lane; f < Fp; f += 32) {
        float v = (f < F) ? (float)x[(size_t)n * F + f] : 0.f;
        s += fabsf(v);
        xb[(size_t)n * Fp + f] = __float2bfloat16_rn(v);
      }
    }
    s = warp_sum(s);
    if (lane == 0) { float m = s > 0.f ? 1.f : 0.f; s_mask[n] = m; mask[(size_t)b * N + n] = m; }
  }
  __syncthreads();
  float cnt = 0.f;
  for (int n = 0; n < N; ++n) cnt += s_mask[n];
  const float inv = 1.0f / fmaxf(cnt, 1e-8f);
  // masked mean over the bf16-rounded values, boxes in ascending order; a thread owns 8 consecutive features (Fp % 64 == 0)
  for (int f0 = threadIdx.x * 8; f0 < Fp; f0 += blockDim.x * 8) {
    float acc[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) acc[i] = 0.f;
    for (int n = 0; n < N; ++n)
      if (s_mask[n] != 0.f) {
        const uint4 v = *reinterpret_cast<const uint4*>(xb + (size_t)n * Fp + f0);
        acc[0] += __uint_as_float(v.x << 16); acc[1] += __uint_as_float(v.x & 0xffff0000u);
        acc[2] += __uint_as_float(v.y << 16); acc[3] += __uint_as_float(v.y & 0xffff0000u);
        acc[4] += __uint_as_float(v.z << 16); acc[5] += __uint_as_float(v.z & 0xffff0000u);
        acc[6] += __uint_as_float(v.w << 16); acc[7] += __uint_as_float(v.w & 0xffff0000u);
      }
    bf16x8 o;
#pragma unroll
    for (int i = 0; i < 4; ++i) o.v[i] = __floats2bfloat162_rn(f0 + 2 * i < F ? acc[2 * i] * inv : 0.f, f0 + 2 * i + 1 < F ? acc[2 * i + 1] * inv : 0.f);
    st_bf16x8(avgb + (size_t)b * Fp + f0, o);
  }
}

int image_prep(cudaStream_t s, const void* feats, int feats_bf16, int B, int N, int F, bf16* featsb, int Fp, float* mask, bf16* avgb) {
  PROF_SCOPE(s, "image_prep", 0, (double)B*N*(F*(feats_bf16 ? 2.0 : 4.0)+Fp*2.0));
  if (feats_bf16) image_prep_kernel<bf16><<<B, 256, N * sizeof(float), s>>>(reinterpret_cast<const bf16*>(feats), N, F, featsb, Fp, mask, avgb);
  else image_prep_kernel<float><<<B, 256, N * sizeof(float), s>>>(reinterpret_cast<const float*>(feats), N, F, featsb, Fp, mask, avgb);
  LAUNCHED();
  return 0;
}

// ---------------------------------------------------------------------------------------------
// tokens
// ---------------------------------------------------------------------------------------------
__global__ void boundary_tokens_kernel(const long long* __restrict__ cap, int B, int L, int pad, int boundary,
                                       int* __restrict__ tok, float* __restrict__ tmask, float* __restrict__ lengths) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  int len = 0;
  for (int l = 0; l < L; ++l) len += (cap[(size_t)b * L + l] != pad) ? 1 : 0;
  int* row = tok + (size_t)b * (L + 2);
  row[0] = boundary;
  for (int l = 0; l < L; ++l) row[l + 1] = (int)cap[(size_t)b * L + l];
  row[L + 1] = 0;
  row[len + 1] = boundary;
  float cnt = 0.f;
  for (int t = 0; t < L + 1; ++t) {              // targets are tok[:, 1:]
    float m = (row[t + 1] != pad) ? 1.f : 0.f;
    tmask[(size_t)t * B + b] = m;
    cnt += m;
  }
  lengths[b] = cnt;
}

int boundary_tokens(cudaStream_t s, const long long* cap, int B, int L, int pad, int boundary, int* tok, float* tmask,
                    float* lengths) {
  boundary_tokens_kernel<<<ceil_div(B, 128), 128, 0, s>>>(cap, B, L, pad, boundary, tok, tmask, lengths);
  LAUNCHED();
  return 0;
}

__global__ void embed_gather_kernel(const int* __restrict__ tok, int tok_stride_b, int tok_stride_t, int B, int rows,
                                    const bf16* __restrict__ embb, int Ep, bf16* __restrict__ out) {
  // one warp per output row, 16-byte vectors
  const int r = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (r >= rows) return;
  const int lane = threadIdx.x & 31;
  const int t = r / B, b = r % B;
  const int id = tok[(size_t)b * tok_stride_b + (size_t)t * tok_stride_t];
  const bf16x8* src = reinterpret_cast<const bf16x8*>(embb + (size_t)id * Ep);
  bf16x8* dst = reinterpret_cast<bf16x8*>(out + (size_t)r * Ep);
  for (int i = lane; i < Ep / 8; i += 32) dst[i] = src[i];
}

int embed_gather_train(cudaStream_t s, const int* tok, int B, int L, const bf16* embb, int Ep, bf16* out) {
  PROF_SCOPE(s, "embed", 0, (double)(L+1)*B*Ep*4.0);
  const int rows = (L + 1) * B;
  embed_gather_kernel<<<ceil_div(rows, 8), 256, 0, s>>>(tok, L + 2, 1, B, rows, embb, Ep, out);
  LAUNCHED();
  return 0;
}
int embed_gather_rows(cudaStream_t s, const int* tokens, int R, const bf16* embb, int Ep, bf16* out) {
  PROF_SCOPE(s, "embed", 0, (double)R*Ep*4.0);
  embed_gather_kernel<<<ceil_div(R, 8), 256, 0, s>>>(tokens, 1, 0, R, R, embb, Ep, out);
  LAUNCHED();
  return 0;
}

// ---------------------------------------------------------------------------------------------
// LSTM pointwise forward / backward: one thread per (row, hidden unit)
// ---------------------------------------------------------------------------------------------
__global__ void lstm_fwd_kernel(LstmFwdArgs a) {
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  const int r = blockIdx.y;
  if (j >= a.H) return;
  const int H = a.H;
  const int r2 = a.rowmap ? a.rowmap[r] : r;
  float g[4];
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    const int n = k * H + j;
    const int na = a.perm ? lstm_gate_row(k, j) : n;       // GEMM outputs (acc, add1, add2) share the packed row order
    float v = a.acc[(size_t)r * a.ld_acc + na];
    if (a.add1) v += a.add1[(size_t)r * a.ld1 + na];
    if (a.add2) v += a.add2[(size_t)r2 * a.ld2 + na];
    if (a.bias) v += a.bias[n];
    if (a.sent) v += a.sent[r2] * a.scol[n];
    g[k] = v;
  }
  const float i = sigmoidf_(g[0]), f = sigmoidf_(g[1]), gg = tanhf(g[2]), o = sigmoidf_(g[3]);
  const float cp = a.c_prev ? a.c_prev[(size_t)r * H + j] : 0.f;
  const float c = f * cp + i * gg;
  const float h = o * tanhf(c);
  a.c_out[(size_t)r * H + j] = c;
  if (a.gates_out) {
    float* go = a.gates_out + (size_t)r * 4 * H;
    go[j] = i; go[H + j] = f; go[2 * H + j] = gg; go[3 * H + j] = o;
  }
  const bf16 hb = __float2bfloat16_rn(h);
  if (a.h1_dst) a.h1_dst[(size_t)r * a.ld_h1 + j] = hb;
  if (a.h2_dst) a.h2_dst[(size_t)r * a.ld_h2 + j] = hb;
  if (a.h_out) a.h_out[(size_t)r * H + j] = h;
}

// 4 hidden units per thread, 16-byte accesses (H % 4 == 0 and 16-byte aligned rows: every training / decode buffer)
__device__ __forceinline__ float4 ld4(const float* p) { return *reinterpret_cast<const float4*>(p); }
__device__ __forceinline__ void fma4(float4& v, float s, const float4& w) { v.x = fmaf(s, w.x, v.x); v.y = fmaf(s, w.y, v.y); v.z = fmaf(s, w.z, v.z); v.w = fmaf(s, w.w, v.w); }
__device__ __forceinline__ void add4(float4& v, const float4& w) { v.x += w.x; v.y += w.y; v.z += w.z; v.w += w.w; }
__device__ __forceinline__ void st_bf16x4(bf16* p, float a, float b, float c, float d) {
  __nv_bfloat162 lo = __floats2bfloat162_rn(a, b), hi = __floats2bfloat162_rn(c, d);
  uint2 o;
  o.x = *reinterpret_cast<uint32_t*>(&lo);
  o.y = *reinterpret_cast<uint32_t*>(&hi);
  *reinterpret_cast<uint2*>(p) = o;
}

__global__ void __launch_bounds__(128) lstm_fwd_v4_kernel(LstmFwdArgs a) {
  const int H = a.H, H4 = H >> 2;
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= a.R * H4) return;
  const int r = idx / H4, j = (idx - r * H4) * 4;
  const int r2 = a.rowmap ? a.rowmap[r] : r;
  const float sv = a.sent ? a.sent[r2] : 0.f;
  float4 g[4];
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    const int n = k * H + j;
    const int na = a.perm ? lstm_gate_row(k, j) : n;       // GEMM outputs (acc, add1, add2) share the packed row order
    float4 v = ld4(a.acc + (size_t)r * a.ld_acc + na);
    if (a.add1) add4(v, ld4(a.add1 + (size_t)r * a.ld1 + na));
    if (a.add2) add4(v, ld4(a.add2 + (size_t)r2 * a.ld2 + na));
    if (a.bias) add4(v, ld4(a.bias + n));
    if (a.sent) fma4(v, sv, ld4(a.scol + n));
    g[k] = v;
  }
  const float4 cp = a.c_prev ? ld4(a.c_prev + (size_t)r * H + j) : make_float4(0.f, 0.f, 0.f, 0.f);
  float4 gi, gf, gg, go, c, h;
#define LSTM_LANE(X)                                                                       \
  gi.X = sigmoidf_(g[0].X); gf.X = sigmoidf_(g[1].X); gg.X = tanhf(g[2].X); go.X = sigmoidf_(g[3].X); \
  c.X = gf.X * cp.X + gi.X * gg.X; h.X = go.X * tanhf(c.X);
  LSTM_LANE(x) LSTM_LANE(y) LSTM_LANE(z) LSTM_LANE(w)
#undef LSTM_LANE
  *reinterpret_cast<float4*>(a.c_out + (size_t)r * H + j) = c;
  if (a.gates_out) {
    float* o = a.gates_out + (size_t)r * 4 * H + j;
    *reinterpret_cast<float4*>(o) = gi;
    *reinterpret_cast<float4*>(o + H) = gf;
    *reinterpret_cast<float4*>(o + 2 * H) = gg;
    *reinterpret_cast<float4*>(o + 3 * H) = go;
  }
  if (a.h1_dst) st_bf16x4(a.h1_dst + (size_t)r * a.ld_h1 + j, h.x, h.y, h.z, h.w);
  if (a.h2_dst) st_bf16x4(a.h2_dst + (size_t)r * a.ld_h2 + j, h.x, h.y, h.z, h.w);
  if (a.h_out) *reinterpret_cast<float4*>(a.h_out + (size_t)r * H + j) = h;
}

static inline bool al16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }
static inline bool al8(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 7) == 0; }

int lstm_forward(cudaStream_t s, const LstmFwdArgs& a) {
  PROF_SCOPE(s, "lstm_fwd", 0, (double)a.R*a.H*(4*4.0*2+4.0*2+2.0*2));
  const bool v4 = (a.H % 4) == 0 && al16(a.acc) && (a.ld_acc % 4) == 0 && (!a.add1 || (al16(a.add1) && (a.ld1 % 4) == 0)) &&
                  (!a.add2 || (al16(a.add2) && (a.ld2 % 4) == 0)) && (!a.bias || al16(a.bias)) && (!a.sent || al16(a.scol)) &&
                  (!a.c_prev || al16(a.c_prev)) && al16(a.c_out) && (!a.gates_out || al16(a.gates_out)) &&
                  (!a.h1_dst || (al8(a.h1_dst) && (a.ld_h1 % 4) == 0)) && (!a.h2_dst || (al8(a.h2_dst) && (a.ld_h2 % 4) == 0)) && (!a.h_out || al16(a.h_out));
  if (v4) {
    lstm_fwd_v4_kernel<<<dim3(ceil_div(a.R * (a.H / 4), 128)), dim3(128), 0, s>>>(a);
  } else {
    dim3 grid(ceil_div(a.H, 128), a.R);
    lstm_fwd_kernel<<<grid, dim3(128), 0, s>>>(a);
  }
  LAUNCHED();
  return 0;
}

__global__ void lstm_bwd_kernel(LstmBwdArgs a) {
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  const int r = blockIdx.y;
  const int H = a.H;
  if (j >= H) return;
  float dh = 0.f;
#pragma unroll
  for (int k = 0; k < 3; ++k)
    if (a.dh[k]) dh += a.dh[k][(size_t)r * a.ld_dh[k] + j];
  const float* g = a.gates + (size_t)r * 4 * H;
  const float i = g[j], f = g[H + j], gg = g[2 * H + j], o = g[3 * H + j];
  const float c = a.c[(size_t)r * H + j];
  const float cp = a.c_prev ? a.c_prev[(size_t)r * H + j] : 0.f;
  const float tc = tanhf(c);
  float dc = dh * o * (1.f - tc * tc);
  if (a.dc_in) dc += a.dc_in[(size_t)r * H + j];
  const float d_o = dh * tc;
  bf16* dg = a.dgates + (size_t)r * a.ld_dg;
  dg[j] = __float2bfloat16_rn(dc * gg * i * (1.f - i));
  dg[H + j] = __float2bfloat16_rn(dc * cp * f * (1.f - f));
  dg[2 * H + j] = __float2bfloat16_rn(dc * i * (1.f - gg * gg));
  dg[3 * H + j] = __float2bfloat16_rn(d_o * o * (1.f - o));
  a.dc_prev[(size_t)r * H + j] = dc * f;
}

__global__ void __launch_bounds__(128) lstm_bwd_v4_kernel(LstmBwdArgs a) {
  const int H = a.H, H4 = H >> 2;
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  int r, j;
  if (a.tiled) {
    // row-tiled state: a warp covers 8 rows x 4 unit-quads, so the tiled reads (8 consecutive rows = 128 contiguous
    // bytes) and the row-major accesses (4 consecutive quads = 64 contiguous bytes of a row) both use whole sectors
    const int lane = idx & 31, wg = idx >> 5;
    const int tr = (a.R + 7) >> 3, tq = (H4 + 3) >> 2;
    if (wg >= tr * tq) return;
    r = (wg % tr) * 8 + (lane & 7);
    const int jq = (wg / tr) * 4 + (lane >> 3);
    if (r >= a.R || jq >= H4) return;
    j = jq * 4;
  } else {
    if (idx >= a.R * H4) return;
    r = idx / H4; j = (idx - r * H4) * 4;
  }
  float4 dh = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
  for (int k = 0; k < 3; ++k)
    if (a.dh[k]) add4(dh, ld4(a.dh[k] + (size_t)r * a.ld_dh[k] + j));
  float4 gi, gf, gg, go, c, cp = make_float4(0.f, 0.f, 0.f, 0.f);
  if (a.tiled) {
    const float* g = a.gates + lstm_tiled_gate_offset(a.R, r, 0, j);
    const size_t gs = (size_t)a.R * 4;
    gi = ld4(g); gf = ld4(g + gs); gg = ld4(g + 2 * gs); go = ld4(g + 3 * gs);
    c = ld4(a.c + lstm_tiled_c_offset(a.R, r, j));
    if (a.c_prev) cp = ld4(a.c_prev + lstm_tiled_c_offset(a.R, r, j));
  } else {
    const float* g = a.gates + (size_t)r * 4 * H + j;
    gi = ld4(g); gf = ld4(g + H); gg = ld4(g + 2 * H); go = ld4(g + 3 * H);
    c = ld4(a.c + (size_t)r * H + j);
    if (a.c_prev) cp = ld4(a.c_prev + (size_t)r * H + j);
  }
  const float4 dci = a.dc_in ? ld4(a.dc_in + (size_t)r * H + j) : make_float4(0.f, 0.f, 0.f, 0.f);
  float4 di, df, dg, d_o, dcp;
#define LSTM_LANE(X)                                                                     \
  {                                                                                      \
    const float tc = tanhf(c.X);                                                         \
    const float dc = dh.X * go.X * (1.f - tc * tc) + dci.X;                              \
    di.X = dc * gg.X * gi.X * (1.f - gi.X);                                              \
    df.X = dc * cp.X * gf.X * (1.f - gf.X);                                              \
    dg.X = dc * gi.X * (1.f - gg.X * gg.X);                                              \
    d_o.X = dh.X * tc * go.X * (1.f - go.X);                                             \
    dcp.X = dc * gf.X;                                                                   \
  }
  LSTM_LANE(x) LSTM_LANE(y) LSTM_LANE(z) LSTM_LANE(w)
#undef LSTM_LANE
  bf16* o = a.dgates + (size_t)r * a.ld_dg + j;
  st_bf16x4(o, di.x, di.y, di.z, di.w);
  st_bf16x4(o + H, df.x, df.y, df.z, df.w);
  st_bf16x4(o + 2 * H, dg.x, dg.y, dg.z, dg.w);
  st_bf16x4(o + 3 * H, d_o.x, d_o.y, d_o.z, d_o.w);
  *reinterpret_cast<float4*>(a.dc_prev + (size_t)r * H + j) = dcp;
}

int lstm_backward(cudaStream_t s, const LstmBwdArgs& a) {
  PROF_SCOPE(s, "lstm_bwd", 0, (double)a.R*a.H*(4*4.0+4*2.0+4.0*5));
  bool v4 = (a.H % 4) == 0 && al16(a.gates) && al16(a.c) && (!a.c_prev || al16(a.c_prev)) && (!a.dc_in || al16(a.dc_in)) &&
            al16(a.dc_prev) && al8(a.dgates) && (a.ld_dg % 4) == 0;
  for (int k = 0; k < 3; ++k) v4 = v4 && (!a.dh[k] || (al16(a.dh[k]) && (a.ld_dh[k] % 4) == 0));
  REQUIRE(!a.tiled || v4, "lstm_backward: the row-tiled state layout needs H %% 4 == 0 and 16-byte aligned buffers");
  if (v4) {
    const int items = a.tiled ? ceil_div(a.R, 8) * ceil_div(a.H / 4, 4) * 32 : a.R * (a.H / 4);
    lstm_bwd_v4_kernel<<<dim3(ceil_div(items, 128)), dim3(128), 0, s>>>(a);
  } else {
    dim3 grid(ceil_div(a.H, 128), a.R);
    lstm_bwd_kernel<<<grid, dim3(128), 0, s>>>(a);
  }
  LAUNCHED();
  return 0;
}

// ---------------------------------------------------------------------------------------------
// latent
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ float philox_normal(unsigned long long seed, unsigned long long step, int r, int z, int Z) {
  curandStatePhilox4_32_10_t st;
  curand_init(seed, (unsigned long long)r * Z + z, step, &st);
  return curand_normal(&st);
}

__global__ void latent_fwd_train_kernel(LatentArgs a, const float* __restrict__ ml, int ld_ml,
                                        const float* __restrict__ bias_ml, const float* __restrict__ eps_in,
                                        const unsigned long long* __restrict__ seed_dev, unsigned long long step, float* __restrict__ mean_out,
                                        float* __restrict__ logvar_out, float* __restrict__ eps_out, bf16* __restrict__ zb,
                                        int ld_z, float* __restrict__ kl_out) {
  __shared__ float red[32];
  const int r = blockIdx.x;
  const int Z = a.Z;
  const float pm_row = a.prior_mean_row ? a.prior_mean_row[a.rowmap ? a.rowmap[r] : r] : 0.f;
  const float log_pv = logf(a.prior_var);
  float part = 0.f;
  for (int z = threadIdx.x; z < a.Zp; z += blockDim.x) {
    if (z < Z) {
      const float pm = a.prior_mean_full ? a.prior_mean_full[(size_t)r * Z + z] : pm_row;
      const float mu = ml[(size_t)r * ld_ml + z] + bias_ml[z];
      const float lv = ml[(size_t)r * ld_ml + Z + z] + bias_ml[Z + z];
      const float var = __expf(lv);
      const float e = eps_in ? eps_in[(size_t)r * Z + z] : philox_normal(seed_dev ? *seed_dev : a.seed, step, r, z, Z);
      const float zz = e * sqrtf(var) + mu;
      mean_out[(size_t)r * Z + z] = mu;
      logvar_out[(size_t)r * Z + z] = lv;
      eps_out[(size_t)r * Z + z] = e;
      zb[(size_t)r * ld_z + z] = __float2bfloat16_rn(zz);
      if (a.sentiment_vae == 0) part += 1.f + lv - mu * mu - var;
      else part += 1.f + lv - log_pv - ((mu - pm) * (mu - pm) + var) / (a.prior_var + 0.00001f);
    } else {
      zb[(size_t)r * ld_z + z] = __float2bfloat16_rn(0.f);
    }
  }
  part = warp_sum(part);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = part;
  __syncthreads();
  if (threadIdx.x < 32) {
    float v = (threadIdx.x < (blockDim.x >> 5)) ? red[threadIdx.x] : 0.f;
    v = warp_sum(v);
    if (threadIdx.x == 0) kl_out[r] = -0.5f * v;
  }
}

int latent_forward_train(cudaStream_t s, const LatentArgs& a, const float* ml, int ld_ml, const float* bias_ml,
                         const float* eps_in, const unsigned long long* seed_dev, unsigned long long step, float* mean_out,
                         float* logvar_out, float* eps_out, bf16* zb, int ld_z, float* kl_out) {
  PROF_SCOPE(s, "latent_fwd", 0, (double)a.R*a.Z*24.0);
  const int threads = min(256, round_up(a.Zp, 32));
  latent_fwd_train_kernel<<<dim3(a.R), dim3(threads), 0, s>>>(a, ml, ld_ml, bias_ml, eps_in, seed_dev, step, mean_out, logvar_out,
                                                             eps_out, zb, ld_z, kl_out);
  LAUNCHED();
  return 0;
}

__global__ void latent_fwd_eval_kernel(LatentArgs a, const float* __restrict__ eps_in, int eps_row_stride,
                                       const unsigned long long* __restrict__ seed_dev, unsigned long long step, bf16* __restrict__ zb,
                                       int ld_z) {
  const int r = blockIdx.x;
  const int img = a.rowmap ? a.rowmap[r] : r;
  const float pm_row = a.prior_mean_row ? a.prior_mean_row[img] : 0.f;
  const float sd_all = sqrtf(a.prior_var);
  for (int z = threadIdx.x; z < a.Zp; z += blockDim.x) {
    float v = 0.f;
    if (z < a.Z) {
      const float e = eps_in ? eps_in[(size_t)r * eps_row_stride * a.Z + z]
                             : philox_normal(seed_dev ? *seed_dev : a.seed, step, r, z, a.Z);
      const float pm = a.prior_mean_full ? a.prior_mean_full[(size_t)r * a.Z + z]
                     : a.prior_mean_img  ? a.prior_mean_img[(size_t)img * a.Z + z] : pm_row;
      const float sd = a.prior_var_img ? sqrtf(a.prior_var_img[(size_t)img * a.Z + z]) : sd_all;
      v = e * sd + pm;
      if (a.pm_out) a.pm_out[(size_t)r * a.Z + z] = pm;
    }
    zb[(size_t)r * ld_z + z] = __float2bfloat16_rn(v);
  }
}

int latent_forward_eval(cudaStream_t s, const LatentArgs& a, const float* eps_in, int eps_row_stride,
                        const unsigned long long* seed_dev, unsigned long long step, bf16* zb, int ld_z) {
  PROF_SCOPE(s, "latent_fwd", 0, (double)a.R*a.Z*6.0);
  const int threads = min(256, round_up(a.Zp, 32));
  latent_fwd_eval_kernel<<<dim3(a.R), dim3(threads), 0, s>>>(a, eps_in, eps_row_stride, seed_dev, step, zb, ld_z);
  LAUNCHED();
  return 0;
}

__global__ void latent_bwd_kernel(LatentArgs a, const float* __restrict__ dz, int ld_dz, const float* __restrict__ eps,
                                  const float* __restrict__ mean, const float* __restrict__ logvar,
                                  const float* __restrict__ gkld, const float* __restrict__ tmask_t,
                                  bf16* __restrict__ dml, int ld_dml) {
  const int r = blockIdx.x;
  const int Z = a.Z;
  const float pm_row = a.prior_mean_row ? a.prior_mean_row[a.rowmap ? a.rowmap[r] : r] : 0.f;
  const float w = a.upstream ? 0.f : gkld[r] * tmask_t[r];
  const float inv_pv = 1.0f / (a.prior_var + 0.00001f);
  for (int z = threadIdx.x; z < ld_dml; z += blockDim.x) {
    float out = 0.f;
    if (z < 2 * Z) {
      const int zi = (z < Z) ? z : z - Z;
      const float mu = mean[(size_t)r * Z + zi], lv = logvar[(size_t)r * Z + zi];
      const float var = __expf(lv);
      const float g = dz[(size_t)r * ld_dz + zi];
      if (z < Z) {
        const float pm = a.prior_mean_full ? a.prior_mean_full[(size_t)r * Z + zi] : pm_row;
        const float dkl = (a.sentiment_vae == 0) ? mu : (mu - pm) * inv_pv;
        if (a.upstream) out = g + (a.dmean_up ? a.dmean_up[(size_t)r * Z + zi] : 0.f);
        else out = g + w * dkl;
        if (a.dpm_out) a.dpm_out[(size_t)r * Z + zi] = -w * dkl;      // d kld / d prior_mean = -d kld / d mean
      } else {
        const float dkl = (a.sentiment_vae == 0) ? -0.5f * (1.f - var) : -0.5f * (1.f - var * inv_pv);
        const float dz_lv = g * eps[(size_t)r * Z + zi] * 0.5f * sqrtf(var);
        if (a.upstream) out = dz_lv + (a.dlogvar_up ? a.dlogvar_up[(size_t)r * Z + zi] : 0.f);
        else out = dz_lv + w * dkl;
      }
    }
    dml[(size_t)r * ld_dml + z] = __float2bfloat16_rn(out);
  }
}

int latent_backward(cudaStream_t s, const LatentArgs& a, const float* dz, int ld_dz, const float* eps, const float* mean,
                    const float* logvar, const float* gkld, const float* tmask_t, bf16* dml, int ld_dml) {
  PROF_SCOPE(s, "latent_bwd", 0, (double)a.R*a.Z*24.0);
  latent_bwd_kernel<<<dim3(a.R), dim3(min(256, round_up(ld_dml, 32))), 0, s>>>(a, dz, ld_dz, eps, mean, logvar, gkld, tmask_t, dml,
                                                                              ld_dml);
  LAUNCHED();
  return 0;
}

// ---- attribute-grounded prior (sentiment_vae == 2, updown_cell.py:160-174) ----
__global__ void prior_mean_fwd_kernel(const float* __restrict__ alpha, const float* __restrict__ obj,
                                      const int* __restrict__ rowmap, int N, int Z, float* __restrict__ pm,
                                      bf16* __restrict__ c_dst, int ld_c, int cond) {
  extern __shared__ float al_s[];
  const int r = blockIdx.x;
  const int img = rowmap ? rowmap[r] : r;
  for (int n = threadIdx.x; n < N; n += blockDim.x) al_s[n] = alpha[(size_t)r * N + n];
  __syncthreads();
  const float* o = obj + (size_t)img * N * Z;
  for (int z = threadIdx.x; z < Z; z += blockDim.x) {
    float acc = 0.f;
    for (int n = 0; n < N; ++n) acc += al_s[n] * o[(size_t)n * Z + z];
    pm[(size_t)r * Z + z] = acc;
    if (z < cond) c_dst[(size_t)r * ld_c + z] = __float2bfloat16_rn(acc);
  }
}

int prior_mean_forward(cudaStream_t s, const float* alpha, const float* obj, const int* rowmap, int R, int N, int Z,
                       float* pm, bf16* c_dst, int ld_c, int cond) {
  PROF_SCOPE(s, "prior_mean", 0, (double)R * N * Z * 4.0);
  REQUIRE(cond >= 0 && cond <= Z, "prior_mean_forward: cond=%d out of range", cond);
  prior_mean_fwd_kernel<<<dim3(R), dim3(min(256, round_up(Z, 32))), (size_t)N * sizeof(float), s>>>(alpha, obj, rowmap, N, Z, pm,
                                                                                                     c_dst, ld_c, cond);
  LAUNCHED();
  return 0;
}

__global__ void prior_mean_bwd_kernel(int N, int Z, int cond, const float* __restrict__ dpm_kl, const float* __restrict__ dc_dec,
                                      int ld_dec, const float* __restrict__ dc_enc, int ld_enc, const float* __restrict__ obj,
                                      float* __restrict__ dalpha) {
  extern __shared__ float dpm_s[];
  const int r = blockIdx.x;
  for (int z = threadIdx.x; z < Z; z += blockDim.x) {
    float v = dpm_kl[(size_t)r * Z + z];
    if (z < cond) v += dc_dec[(size_t)r * ld_dec + z] + dc_enc[(size_t)r * ld_enc + z];
    dpm_s[z] = v;
  }
  __syncthreads();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nw = blockDim.x >> 5;
  const float* o = obj + (size_t)r * N * Z;
  for (int n = warp; n < N; n += nw) {
    float acc = 0.f;
    for (int z = lane; z < Z; z += 32) acc += o[(size_t)n * Z + z] * dpm_s[z];
    acc = warp_sum(acc);
    if (lane == 0) dalpha[(size_t)r * N + n] = acc;
  }
}

int prior_mean_backward(cudaStream_t s, int R, int N, int Z, int cond, const float* dpm_kl, const float* dc_dec, int ld_dec,
                        const float* dc_enc, int ld_enc, const float* obj, float* dalpha) {
  PROF_SCOPE(s, "prior_mean", 0, (double)R * N * Z * 4.0);
  prior_mean_bwd_kernel<<<dim3(R), dim3(256), (size_t)Z * sizeof(float), s>>>(N, Z, cond, dpm_kl, dc_dec, ld_dec, dc_enc, ld_enc, obj,
                                                                               dalpha);
  LAUNCHED();
  return 0;
}

// ---------------------------------------------------------------------------------------------
// cross entropy over the vocabulary: one CTA per (t,b) row, skipped when the target is padding
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ float block_reduce(float v, float* red, bool is_max) {
  v = is_max ? warp_max(v) : warp_sum(v);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
  __syncthreads();
  float x = (threadIdx.x < (blockDim.x >> 5)) ? red[threadIdx.x] : (is_max ? -INFINITY : 0.f);
  if (threadIdx.x < 32) {
    x = is_max ? warp_max(x) : warp_sum(x);
    if (threadIdx.x == 0) red[0] = x;
  }
  __syncthreads();
  const float out = red[0];
  __syncthreads();
  return out;
}

__global__ void ce_fwd_kernel(const float* __restrict__ logits, int ld, int V, const int* __restrict__ tok, int B, int L,
                              const float* __restrict__ tmask, float* __restrict__ lse, float* __restrict__ nll) {
  __shared__ float red[32];
  const int r = blockIdx.x;
  if (tmask[r] == 0.f) { if (threadIdx.x == 0) { lse[r] = 0.f; nll[r] = 0.f; } return; }
  const int t = r / B, b = r % B;
  const float* x = logits + (size_t)r * ld;
  float m = -INFINITY;
  for (int v = threadIdx.x; v < V; v += blockDim.x) m = fmaxf(m, x[v]);
  m = block_reduce(m, red, true);
  float sum = 0.f;
  for (int v = threadIdx.x; v < V; v += blockDim.x) sum += __expf(x[v] - m);
  sum = block_reduce(sum, red, false);
  if (threadIdx.x == 0) {
    const float l = m + logf(sum);
    const int target = tok[(size_t)b * (L + 2) + t + 1];
    lse[r] = l;
    nll[r] = l - x[target];
  }
}

int ce_forward(cudaStream_t s, const float* logits, int ld, int TB, int V, const int* tok, int B, int L,
               const float* tmask, float* lse, float* nll) {
  PROF_SCOPE(s, "ce_fwd", 0, (double)TB*V*4.0*2);
  ce_fwd_kernel<<<TB, 256, 0, s>>>(logits, ld, V, tok, B, L, tmask, lse, nll);
  LAUNCHED();
  return 0;
}

__global__ void loss_reduce_kernel(const float* __restrict__ nll, const float* __restrict__ kl,
                                   const float* __restrict__ tmask, const float* __restrict__ lengths, int T, int B,
                                   float* __restrict__ loss, float* __restrict__ kld) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  float sn = 0.f, sk = 0.f;
  for (int t = 0; t < T; ++t) {
    const float m = tmask[(size_t)t * B + b];
    sn += nll[(size_t)t * B + b] * m;
    sk += kl[(size_t)t * B + b] * m;
  }
  const float len = lengths[b];
  loss[b] = len * (sn / (len + 1e-13f));
  kld[b] = sk;
}

int loss_reduce(cudaStream_t s, const float* nll, const float* kl, const float* tmask, const float* lengths, int T, int B,
                float* loss, float* kld) {
  loss_reduce_kernel<<<ceil_div(B, 128), 128, 0, s>>>(nll, kl, tmask, lengths, T, B, loss, kld);
  LAUNCHED();
  return 0;
}

__global__ void ce_bwd_kernel(const float* __restrict__ logits, int ld, int V, const int* __restrict__ tok, int B, int L,
                              const float* __restrict__ tmask, const float* __restrict__ lengths,
                              const float* __restrict__ lse, const float* __restrict__ gloss, bf16* __restrict__ dlogits,
                              int ld_d) {
  const int r = blockIdx.x;
  const int t = r / B, b = r % B;
  bf16* d = dlogits + (size_t)r * ld_d;
  if (tmask[r] == 0.f) {
    for (int v = threadIdx.x; v < ld_d; v += blockDim.x) d[v] = __float2bfloat16_rn(0.f);
    return;
  }
  const float len = lengths[b];
  const float g = gloss[b] * (len / (len + 1e-13f));
  const float l = lse[r];
  const int target = tok[(size_t)b * (L + 2) + t + 1];
  const float* x = logits + (size_t)r * ld;
  for (int v = threadIdx.x; v < ld_d; v += blockDim.x) {
    float o = 0.f;
    if (v < V) o = g * (__expf(x[v] - l) - (v == target ? 1.f : 0.f));
    d[v] = __float2bfloat16_rn(o);
  }
}

int ce_backward(cudaStream_t s, const float* logits, int ld, int TB, int V, const int* tok, int B, int L,
                const float* tmask, const float* lengths, const float* lse, const float* gloss, bf16* dlogits, int ld_d) {
  PROF_SCOPE(s, "ce_bwd", 0, (double)TB*V*6.0);
  ce_bwd_kernel<<<TB, 256, 0, s>>>(logits, ld, V, tok, B, L, tmask, lengths, lse, gloss, dlogits, ld_d);
  LAUNCHED();
  return 0;
}

// ---- vocabulary head with the softmax statistics in the GEMM epilogue (gemm.cuh: RowStatsEpi) ----------------------
// row r = t*B + b: target token and (backward) the coefficient of its CE gradient; masked rows get coefficient 0
__global__ void ce_prep_kernel(const int* __restrict__ tok, int B, int L, int TB, const float* __restrict__ tmask,
                               const float* __restrict__ lengths, const float* __restrict__ gloss, int* __restrict__ target,
                               float* __restrict__ gcoef) {
  const int r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= TB) return;
  const int t = r / B, b = r - t * B;
  target[r] = tok[(size_t)b * (L + 2) + t + 1];
  if (gcoef) {
    const float len = lengths[b];
    gcoef[r] = tmask[r] != 0.f ? gloss[b] * (len / (len + 1e-13f)) : 0.f;
  }
}
int ce_prepare(cudaStream_t s, const int* tok, int B, int L, const float* tmask, const float* lengths, const float* gloss,
               int* target, float* gcoef) {
  const int TB = (L + 1) * B;
  ce_prep_kernel<<<ceil_div(TB, 256), 256, 0, s>>>(tok, B, L, TB, tmask, lengths, gloss, target, gcoef);
  LAUNCHED();
  return 0;
}

// merges the per-tile partial (max, sum exp, arg max) of row r; partials at [tile * R + r]. One WARP per row: lanes take
// tiles lane, lane + 32, ...; (value desc, index asc) order as everywhere in the search.
__device__ __forceinline__ void merge_row_stats(const float* __restrict__ st_max, const float* __restrict__ st_sum,
                                                const int* __restrict__ st_arg, int ntiles, int R, int r, float& M, float& S,
                                                int& arg) {
  const int lane = threadIdx.x & 31;
  float m = -INFINITY; int a = 0x7fffffff;
  for (int i = lane; i < ntiles; i += 32) {
    const float v = st_max[(size_t)i * R + r];
    if (v > m) { m = v; a = st_arg[(size_t)i * R + r]; }            // strict: the lowest tile wins ties
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const float om = __shfl_xor_sync(0xffffffffu, m, o);
    const int oa = __shfl_xor_sync(0xffffffffu, a, o);
    if (om > m || (om == m && oa < a)) { m = om; a = oa; }
  }
  float s = 0.f;
  for (int i = lane; i < ntiles; i += 32) s += st_sum[(size_t)i * R + r] * __expf(st_max[(size_t)i * R + r] - m);
  S = warp_sum(s); M = m; arg = a;
}

__global__ void ce_merge_kernel(const float* __restrict__ st_max, const float* __restrict__ st_sum, const int* __restrict__ st_arg,
                                int ntiles, int TB, const float* __restrict__ tgt_logit, float* __restrict__ lse,
                                float* __restrict__ nll) {
  const int r = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (r >= TB) return;
  float M, S; int arg;
  merge_row_stats(st_max, st_sum, st_arg, ntiles, TB, r, M, S, arg);
  if ((threadIdx.x & 31) == 0) {
    const float l = M + logf(S);
    lse[r] = l;
    nll[r] = l - tgt_logit[r];
  }
}
int ce_merge(cudaStream_t s, const float* st_max, const float* st_sum, const int* st_arg, int ntiles, int TB,
             const float* tgt_logit, float* lse, float* nll) {
  PROF_SCOPE(s, "ce_fwd", 0, (double)TB * ntiles * 12.0);
  ce_merge_kernel<<<ceil_div(TB, 8), 256, 0, s>>>(st_max, st_sum, st_arg, ntiles, TB, tgt_logit, lse, nll);
  LAUNCHED();
  return 0;
}

// greedy step of the unconstrained K = 1 search (cbs.py:161-250 with S = K = P = 1): token = arg max, score = parent score
// + log-softmax of the max = -log(sum exp(x - max)); a sequence that has ended keeps emitting the boundary (cbs.py:177-181)
__global__ void greedy_merge_kernel(const float* __restrict__ st_max, const float* __restrict__ st_sum, const int* __restrict__ st_arg,
                                    int ntiles, int R, const int* __restrict__ last_tokens, const float* __restrict__ last_scores,
                                    int end_index, int* __restrict__ tok, int* __restrict__ bp, float* __restrict__ score) {
  const int r = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (r >= R) return;
  float M, S; int arg;
  merge_row_stats(st_max, st_sum, st_arg, ntiles, R, r, M, S, arg);
  if ((threadIdx.x & 31) == 0) {
    const bool forced = last_tokens != nullptr && last_tokens[r] == end_index;
    const float lp = forced ? 0.f : -logf(S);
    tok[r] = forced ? end_index : arg;
    score[r] = last_scores ? last_scores[r] + lp : lp;
    if (bp) bp[r] = 0;
  }
}
int greedy_merge(cudaStream_t s, const float* st_max, const float* st_sum, const int* st_arg, int ntiles, int R,
                 const int* last_tokens, const float* last_scores, int end_index, int* tok, int* bp, float* score) {
  PROF_SCOPE(s, "search_rows", 0, (double)R * ntiles * 12.0);
  greedy_merge_kernel<<<ceil_div(R, 8), 256, 0, s>>>(st_max, st_sum, st_arg, ntiles, R, last_tokens, last_scores, end_index, tok,
                                                    bp, score);
  LAUNCHED();
  return 0;
}

// log-softmax of the step's logits in place (updown_captioner.py:450): one warp per row merges the head GEMM's per-tile
// partials (the log-sum-exp of ce_merge) and rewrites the row with 16-byte accesses; the logits are read once, written once
__global__ void log_softmax_rows_kernel(const float* __restrict__ st_max, const float* __restrict__ st_sum,
                                        const int* __restrict__ st_arg, int ntiles, int R, int V, int vec4,
                                        float* __restrict__ x) {
  const int r = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (r >= R) return;
  const int lane = threadIdx.x & 31;
  float M, S; int arg;
  merge_row_stats(st_max, st_sum, st_arg, ntiles, R, r, M, S, arg);
  const float lse = M + logf(S);
  float* row = x + (size_t)r * V;
  if (vec4) {
    float4* row4 = reinterpret_cast<float4*>(row);
    for (int i = lane; i < (V >> 2); i += 32) {
      float4 v = row4[i];
      v.x -= lse; v.y -= lse; v.z -= lse; v.w -= lse;
      row4[i] = v;
    }
  } else {
    for (int i = lane; i < V; i += 32) row[i] -= lse;
  }
}
int log_softmax_rows(cudaStream_t s, const float* st_max, const float* st_sum, const int* st_arg, int ntiles, int R, int V,
                     float* logits) {
  PROF_SCOPE(s, "log_softmax", 0, (double)R * V * 8.0 + (double)R * ntiles * 12.0);
  const int vec4 = (V % 4) == 0 && (reinterpret_cast<uintptr_t>(logits) & 15) == 0;
  log_softmax_rows_kernel<<<ceil_div(R, 8), 256, 0, s>>>(st_max, st_sum, st_arg, ntiles, R, V, vec4, logits);
  LAUNCHED();
  return 0;
}

// one warp per row: the token and image index of the row, then (with states) its bf16 [h1 | h_dec] operand row
__global__ void step_import_kernel(const long long* __restrict__ prev, int R, int rows_per_image, const float* __restrict__ h1,
                                   const float* __restrict__ hd, int H, int Hp, int* __restrict__ tok, int* __restrict__ rowmap,
                                   bf16* __restrict__ xa, const float* __restrict__ he_in, bf16* __restrict__ he,
                                   bf16* __restrict__ xe_hd, int ld_xe) {
  const int r = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (r >= R) return;
  const int lane = threadIdx.x & 31;
  if (lane == 0) { tok[r] = (int)prev[r]; if (rowmap) rowmap[r] = r / rows_per_image; }
  if (!h1) return;
  bf16* o = xa + (size_t)r * 2 * Hp;
  for (int c = lane; c < 2 * Hp; c += 32) {
    const int j = c < Hp ? c : c - Hp;
    const float* src = c < Hp ? h1 : hd;
    o[c] = __float2bfloat16_rn(j < H ? src[(size_t)r * H + j] : 0.f);
  }
  if (he)
    for (int j = lane; j < Hp; j += 32) he[(size_t)r * Hp + j] = __float2bfloat16_rn(j < H ? he_in[(size_t)r * H + j] : 0.f);
  if (xe_hd)
    for (int j = lane; j < Hp; j += 32) xe_hd[(size_t)r * ld_xe + j] = __float2bfloat16_rn(j < H ? hd[(size_t)r * H + j] : 0.f);
}
int step_import(cudaStream_t s, const long long* prev, int R, int rows_per_image, const float* h1, const float* h_dec, int H,
                int Hp, int* tok, int* rowmap, bf16* xa, const float* h_enc, bf16* he, bf16* xe_hd, int ld_xe) {
  PROF_SCOPE(s, "step_import", 0, (double)R * (12.0 + (h1 ? 2.0 * H * 4.0 + 4.0 * Hp : 0.0)));
  REQUIRE(rows_per_image > 0 && (!h1 || (h_dec && xa)) && (!he || (h1 && h_enc)) && (!xe_hd || h1),
          "step_import: bad arguments");
  step_import_kernel<<<ceil_div(R, 8), 256, 0, s>>>(prev, R, rows_per_image, h1, h_dec, H, Hp, tok, rowmap, xa, h_enc, he,
                                                    xe_hd, ld_xe);
  LAUNCHED();
  return 0;
}

__global__ void step_export_grads_kernel(const StepGradExport a) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= a.R * a.H) return;
  const int r = idx / a.H, j = idx - r * a.H;
  const float* xa = a.dxa + (size_t)r * a.ld_xa;
  const float* xe = a.dxe + (size_t)r * a.ld_xe;
  if (a.out[0]) a.out[0][idx] = xa[j];
  if (a.out[2]) a.out[2][idx] = xe[a.off_he + j];
  if (a.out[4]) a.out[4][idx] = xe[a.off_hd + j] + xa[a.Hp + j];
  for (int k = 0; k < 3; ++k)
    if (a.out[2 * k + 1]) a.out[2 * k + 1][idx] = a.dc[k][idx];
}
int step_export_grads(cudaStream_t s, const StepGradExport& a) {
  PROF_SCOPE(s, "step_export", 0, (double)a.R * a.H * 4.0 * 10.0);
  step_export_grads_kernel<<<ceil_div(a.R * a.H, 256), 256, 0, s>>>(a);
  LAUNCHED();
  return 0;
}

// ---------------------------------------------------------------------------------------------
// layout helpers
// ---------------------------------------------------------------------------------------------
template <typename TIn>
__device__ __forceinline__ float to_f(TIn v);
template <> __device__ __forceinline__ float to_f<float>(float v) { return v; }
template <> __device__ __forceinline__ float to_f<bf16>(bf16 v) { return __bfloat162float(v); }

// out[c, r] = in[r, c]; columns of `out` in [rows, ld_out) are zero-filled so it can be a GEMM operand
__global__ void transpose_f32_kernel(const float* __restrict__ in, int rows, int cols, int ld_in, bf16* __restrict__ out,
                                     int ld_out) {
  __shared__ float tile[32][33];
  const int r0 = blockIdx.x * 32, c0 = blockIdx.y * 32;
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    const int r = r0 + i, c = c0 + threadIdx.x;
    tile[i][threadIdx.x] = (r < rows && c < cols) ? in[(size_t)r * ld_in + c] : 0.f;
  }
  __syncthreads();
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    const int c = c0 + i, r = r0 + threadIdx.x;
    if (c < cols && r < ld_out) out[(size_t)c * ld_out + r] = __float2bfloat16_rn(tile[threadIdx.x][i]);
  }
}

// ---- bf16 transposes of a whole list of operands in ONE launch; a CTA transposes one 64 x 64 tile -----------------
// The tile crosses shared memory as 64 rows of eight 16-byte chunks, chunk c of row i stored at chunk c ^ ((i >> 3) & 7):
// the 16-byte row writes and the 4-byte column reads (thread = 8 consecutive rows x 2 columns, 8 row groups per warp) are
// both free of bank conflicts. (2-byte column reads of an unswizzled tile are an 8-way bank conflict: shared memory, not
// HBM, then bounds the transpose at ~2 TB/s.)
int TransposeJobList::add(const bf16* src, int rows, int cols, int ld_in, bf16* dst, int ld_out) {
  REQUIRE(n < kMaxTransposeJobs, "transpose job list full");
  REQUIRE(rows > 0 && cols > 0 && ld_in >= cols && ld_out >= rows && ld_in % 8 == 0 && ld_out % 8 == 0 &&
              (reinterpret_cast<uintptr_t>(src) & 15) == 0 && (reinterpret_cast<uintptr_t>(dst) & 15) == 0,
          "transpose: rows %d cols %d ld_in %d ld_out %d (need ld %% 8 == 0 and 16-byte aligned bases)", rows, cols, ld_in,
          ld_out);
  TransposeJob& j = job[n++];
  j.src = src; j.dst = dst; j.rows = rows; j.cols = cols; j.ld_in = ld_in; j.ld_out = ld_out; j.tile0 = 0; j.tiles_x = 0;
  return 0;
}

struct TransposeJobTable { TransposeJob job[kMaxTransposeJobs]; int n; };

__global__ void __launch_bounds__(256) transpose_bf16_jobs_kernel(const __grid_constant__ TransposeJobTable t) {
  __shared__ __align__(16) uint8_t tile[64 * 128];
  int ji = 0;
  while (ji + 1 < t.n && (int)blockIdx.x >= t.job[ji + 1].tile0) ++ji;
  const TransposeJob& j = t.job[ji];
  const int local = blockIdx.x - j.tile0;
  const int r0 = (local % j.tiles_x) * 64, c0 = (local / j.tiles_x) * 64;   // input rows (output columns), input columns
  const int rows = j.rows, cols = j.cols;
#pragma unroll
  for (int it = 0; it < 2; ++it) {
    const int v = threadIdx.x + it * 256;
    const int i = v >> 3, cv = v & 7;
    const int r = r0 + i, c = c0 + cv * 8;
    uint4 x = make_uint4(0u, 0u, 0u, 0u);
    if (r < rows && c < cols) {
      const bf16* p = j.src + (size_t)r * j.ld_in + c;
      if (c + 8 <= cols) {
        x = *reinterpret_cast<const uint4*>(p);
      } else {                                                              // ragged right edge (cols % 8 != 0)
        bf16 e[8];
#pragma unroll
        for (int k = 0; k < 8; ++k) e[k] = c + k < cols ? p[k] : __float2bfloat16_rn(0.f);
        x = *reinterpret_cast<const uint4*>(e);
      }
    }
    *reinterpret_cast<uint4*>(tile + i * 128 + ((cv ^ ((i >> 3) & 7)) << 4)) = x;
  }
  __syncthreads();
  const int lane = threadIdx.x & 31, rv = lane & 7;
  const int jw = (threadIdx.x >> 5) * 4 + (lane >> 3);                      // 4-byte word = input columns 2jw, 2jw + 1
  uint32_t w[8];
#pragma unroll
  for (int k = 0; k < 8; ++k)
    w[k] = *reinterpret_cast<const uint32_t*>(tile + (8 * rv + k) * 128 + (((jw >> 2) ^ rv) << 4) + ((jw & 3) << 2));
  uint4 lo, hi;                                                             // column 2jw / 2jw + 1, input rows 8rv .. 8rv + 7
  lo.x = __byte_perm(w[0], w[1], 0x5410); hi.x = __byte_perm(w[0], w[1], 0x7632);
  lo.y = __byte_perm(w[2], w[3], 0x5410); hi.y = __byte_perm(w[2], w[3], 0x7632);
  lo.z = __byte_perm(w[4], w[5], 0x5410); hi.z = __byte_perm(w[4], w[5], 0x7632);
  lo.w = __byte_perm(w[6], w[7], 0x5410); hi.w = __byte_perm(w[6], w[7], 0x7632);
  const int c = c0 + 2 * jw, r = r0 + 8 * rv;
  if (r < j.ld_out) {                                                       // ld_out % 8 == 0: all 8 rows or none
    if (c < cols) *reinterpret_cast<uint4*>(j.dst + (size_t)c * j.ld_out + r) = lo;
    if (c + 1 < cols) *reinterpret_cast<uint4*>(j.dst + (size_t)(c + 1) * j.ld_out + r) = hi;
  }
}

int transpose_bf16_jobs(cudaStream_t s, TransposeJobList& jobs) {
  if (jobs.n == 0) return 0;
  TransposeJobTable t;
  double bytes = 0;
  int tiles = 0;
  for (int i = 0; i < jobs.n; ++i) {
    TransposeJob& j = jobs.job[i];
    j.tiles_x = ceil_div(j.ld_out, 64);
    j.tile0 = tiles;
    tiles += j.tiles_x * ceil_div(j.cols, 64);
    bytes += (double)j.rows * j.cols * 4.0;
    t.job[i] = j;
  }
  t.n = jobs.n;
  PROF_SCOPE(s, "transpose", 0, bytes);
  transpose_bf16_jobs_kernel<<<tiles, 256, 0, s>>>(t);
  LAUNCHED();
  jobs.n = 0;
  return 0;
}

int transpose_f32_to_bf16(cudaStream_t s, const float* in, int rows, int cols, int ld_in, bf16* out, int ld_out) {
  PROF_SCOPE(s, "transpose", 0, (double)rows*cols*6.0);
  dim3 grid(ceil_div(ld_out, 32), ceil_div(cols, 32));
  transpose_f32_kernel<<<grid, dim3(32, 8), 0, s>>>(in, rows, cols, ld_in, out, ld_out);
  LAUNCHED();
  return 0;
}

template <typename TIn>
__global__ void rowsum_kernel(const TIn* __restrict__ in, int rows, int cols, int ld, float* __restrict__ out,
                              int accumulate) {
  const int r = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (r >= rows) return;
  const int lane = threadIdx.x & 31;
  float s = 0.f;
  for (int c = lane; c < cols; c += 32) s += to_f<TIn>(in[(size_t)r * ld + c]);
  s = warp_sum(s);
  if (lane == 0) out[r] = accumulate ? out[r] + s : s;
}
int rowsum_bf16(cudaStream_t s, const bf16* in, int rows, int cols, int ld, float* out, int accumulate) {
  PROF_SCOPE(s, "reduce", 0, (double)rows*cols*2.0);
  rowsum_kernel<bf16><<<ceil_div(rows, 8), 256, 0, s>>>(in, rows, cols, ld, out, accumulate);
  LAUNCHED();
  return 0;
}
int rowsum_f32(cudaStream_t s, const float* in, int rows, int cols, int ld, float* out, int accumulate) {
  rowsum_kernel<float><<<ceil_div(rows, 8), 256, 0, s>>>(in, rows, cols, ld, out, accumulate);
  LAUNCHED();
  return 0;
}

__global__ void convert_kernel(const float* __restrict__ in, int rows, int cols, int ld_in, bf16* __restrict__ out,
                               int ld_out) {
  const int r = blockIdx.y;
  for (int c = blockIdx.x * blockDim.x + threadIdx.x; c < ld_out; c += gridDim.x * blockDim.x)
    out[(size_t)r * ld_out + c] = __float2bfloat16_rn(c < cols ? in[(size_t)r * ld_in + c] : 0.f);
}
int convert_f32_to_bf16(cudaStream_t s, const float* in, int rows, int cols, int ld_in, bf16* out, int ld_out) {
  dim3 grid(min(8, ceil_div(ld_out, 256)), rows);
  convert_kernel<<<grid, 256, 0, s>>>(in, rows, cols, ld_in, out, ld_out);
  LAUNCHED();
  return 0;
}

__global__ void timesum_kernel(const bf16* __restrict__ in, int T, int B, int n, int ld, bf16* __restrict__ out,
                               int ld_out) {
  const int b = blockIdx.y;
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= ld_out) return;
  float s = 0.f;
  if (c < n)
    for (int t = 0; t < T; ++t) s += __bfloat162float(in[((size_t)t * B + b) * ld + c]);
  out[(size_t)b * ld_out + c] = __float2bfloat16_rn(s);
}
int timesum_bf16(cudaStream_t s, const bf16* in, int T, int B, int n, int ld, bf16* out, int ld_out) {
  PROF_SCOPE(s, "reduce", 0, (double)T*B*n*2.0);
  dim3 grid(ceil_div(ld_out, 256), B);
  timesum_kernel<<<grid, 256, 0, s>>>(in, T, B, n, ld, out, ld_out);
  LAUNCHED();
  return 0;
}

__global__ void add_kernel(float* __restrict__ dst, const float* __restrict__ src, size_t n) {
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x)
    dst[i] += src[i];
}
int add_f32(cudaStream_t s, float* dst, const float* src, size_t n) {
  add_kernel<<<(int)min((size_t)1184, (n + 255) / 256), 256, 0, s>>>(dst, src, n);
  LAUNCHED();
  return 0;
}

__global__ void gather_rows_f32_kernel(const float* __restrict__ src, const int* __restrict__ idx, int n,
                                       float* __restrict__ dst) {
  const int r = blockIdx.x;
  const float* s = src + (size_t)idx[r] * n;
  for (int c = threadIdx.x; c < n; c += blockDim.x) dst[(size_t)r * n + c] = s[c];
}
int gather_rows_f32(cudaStream_t s, const float* src, const int* idx, int R, int n, float* dst) {
  gather_rows_f32_kernel<<<R, 256, 0, s>>>(src, idx, n, dst);
  LAUNCHED();
  return 0;
}
__global__ void gather_rows_bf16_kernel(const bf16* __restrict__ src, const int* __restrict__ idx, int n, int ld,
                                        bf16* __restrict__ dst) {
  const int r = blockIdx.x;
  const bf16* s = src + (size_t)idx[r] * ld;
  for (int c = threadIdx.x; c < n; c += blockDim.x) dst[(size_t)r * ld + c] = s[c];
}
int gather_rows_bf16(cudaStream_t s, const bf16* src, const int* idx, int R, int n, int ld, bf16* dst) {
  gather_rows_bf16_kernel<<<R, 256, 0, s>>>(src, idx, n, ld, dst);
  LAUNCHED();
  return 0;
}

}  // namespace sscvae

namespace sscvae {

__global__ void colsum_kernel(const float* __restrict__ in, int rows, int cols, int ld, float* __restrict__ out) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= cols) return;
  float s = 0.f;
  for (int r = 0; r < rows; ++r) s += in[(size_t)r * ld + c];
  out[c] = s;
}
int colsum_f32(cudaStream_t s, const float* in, int rows, int cols, int ld, float* out) {
  colsum_kernel<<<ceil_div(cols, 128), 128, 0, s>>>(in, rows, cols, ld, out);
  LAUNCHED();
  return 0;
}

__global__ void rowdot_kernel(const bf16* __restrict__ in, int rows, int cols, int ld, const float* __restrict__ vec,
                              int period, float* __restrict__ out, int out_stride) {
  const int r = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (r >= rows) return;
  const int lane = threadIdx.x & 31;
  float s = 0.f;
  for (int c = lane; c < cols; c += 32) s += __bfloat162float(in[(size_t)r * ld + c]) * vec[c % period];
  s = warp_sum(s);
  if (lane == 0) out[(size_t)r * out_stride] = s;
}
int rowdot_bf16(cudaStream_t s, const bf16* in, int rows, int cols, int ld, const float* vec, int period, float* out,
                int out_stride) {
  rowdot_kernel<<<ceil_div(rows, 8), 256, 0, s>>>(in, rows, cols, ld, vec, period, out, out_stride);
  LAUNCHED();
  return 0;
}

// dst[r, c] = sum_z parts[z * stride + r * ld + c]   (split-K partial tiles -> result; dst may alias parts[0])
__global__ void sum_partials_kernel(float* __restrict__ dst, int ld_dst, const float* __restrict__ parts, size_t stride,
                                    int nparts, int rows, int cols4, int ld) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  const int r = blockIdx.y;
  if (c >= cols4) return;
  float4 v = *reinterpret_cast<const float4*>(parts + (size_t)r * ld + 4 * c);
  for (int z = 1; z < nparts; ++z) {
    const float4 w = *reinterpret_cast<const float4*>(parts + z * stride + (size_t)r * ld + 4 * c);
    v.x += w.x; v.y += w.y; v.z += w.z; v.w += w.w;
  }
  *reinterpret_cast<float4*>(dst + (size_t)r * ld_dst + 4 * c) = v;
}
int sum_partials_f32(cudaStream_t s, float* dst, int ld_dst, const float* parts, size_t stride, int nparts, int rows,
                     int cols, int ld) {
  PROF_SCOPE(s, "splitk_reduce", 0, (double)rows * cols * 4.0 * (nparts + 1));
  REQUIRE(cols % 4 == 0 && ld % 4 == 0 && ld_dst % 4 == 0 && stride % 4 == 0, "sum_partials: shapes must be multiples of 4");
  dim3 grid(ceil_div(cols / 4, 128), rows);
  sum_partials_kernel<<<grid, 128, 0, s>>>(dst, ld_dst, parts, stride, nparts, rows, cols / 4, ld);
  LAUNCHED();
  return 0;
}

__global__ void scale_kernel(const float* in, float scale, float* out, int n) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = in ? in[i] * scale : 0.f;
}
int scale_rows_f32(cudaStream_t s, const float* in, float scale, float* out, int n) {
  scale_kernel<<<ceil_div(n, 256), 256, 0, s>>>(in, scale, out, n);
  LAUNCHED();
  return 0;
}

// row r = t * B + b of dx takes token tok[b * tok_stride_b + t]
__global__ void embed_scatter_kernel(const int* __restrict__ tok, int B, int tok_stride_b, int pad, const float* __restrict__ dx,
                                     int ld_dx, int E, float* __restrict__ demb) {
  const int r = blockIdx.x;
  const int t = r / B, b = r % B;
  const int id = tok[(size_t)b * tok_stride_b + t];
  if (id == pad) return;
  for (int e = threadIdx.x; e < E; e += blockDim.x) atomicAdd(&demb[(size_t)id * E + e], dx[(size_t)r * ld_dx + e]);
}
int embed_scatter_add(cudaStream_t s, const int* tok, int B, int L, int pad, const float* dx, int ld_dx, int E,
                      float* demb) {
  embed_scatter_kernel<<<(L + 1) * B, 128, 0, s>>>(tok, B, L + 2, pad, dx, ld_dx, E, demb);
  LAUNCHED();
  return 0;
}
int embed_scatter_add_rows(cudaStream_t s, const int* tok, int R, int pad, const float* dx, int ld_dx, int E, float* demb) {
  embed_scatter_kernel<<<R, 128, 0, s>>>(tok, R, 1, pad, dx, ld_dx, E, demb);
  LAUNCHED();
  return 0;
}

}  // namespace sscvae

namespace sscvae {
__global__ void fill_i32_kernel(int* dst, int value, int n, int div) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) dst[i] = div ? i / div : value;
}
int fill_i32(cudaStream_t s, int* dst, int value, int n) {
  fill_i32_kernel<<<ceil_div(n, 256), 256, 0, s>>>(dst, value, n, 0);
  LAUNCHED();
  return 0;
}
int iota_div_i32(cudaStream_t s, int* dst, int n, int div) {
  fill_i32_kernel<<<ceil_div(n, 256), 256, 0, s>>>(dst, 0, n, div);
  LAUNCHED();
  return 0;
}
}  // namespace sscvae

// Fused bottom-up/top-down region attention (north_star kernel #2), forward and backward.
//
// forward, per row r (a caption in training, an (image,state,beam) row in decode):
//   u_n   = w_a . tanh(q_r + P[img(r), n, :])             (attention.py:69-88)
//   alpha = masked_softmax(u, mask[img(r)])                (allennlp: softmax(u*m)*m / (sum + 1e-13))
//   xhat  = sum_n alpha_n * x[img(r), n, :]                (updown_cell.py:156-158)
//
// The op is a stream over the image's projected features P (N*Ap bf16) and region features x (N*Fp bf16),
// ~200 KB per row at the shipped dims, with almost no arithmetic: it is bound by bytes in flight. So the
// kernels are persistent (<= one CTA per SM, a contiguous block of rows each) and warp-specialised:
//   warp 8     : producer. One lane issues 1-D bulk async copies (cp.async.bulk -> the TMA engine) of whole
//                box-row chunks into a 4 x 32 KB shared-memory ring, completion on mbarriers. It runs ahead of
//                the consumers across chunk, phase and ROW boundaries, so the next row's data is already in
//                flight while the current row's softmax runs.
//   warps 0..7 : consumers. Scores (warp per box), masked softmax (redundantly per warp, in registers), weighted
//                sum (a thread owns 8 consecutive features). Per-row vectors (q, d xhat, saved softmax) are
//                prefetched one row ahead with cp.async into double buffers.
// Nothing intermediate goes to global memory. HBM/L2 traffic per row: N*(Ap+Fp) bf16 read once, F written.
//
// backward is split in two:
//   per step  : d alpha_n = d xhat . x_n, softmax backward -> d u (saved, (R,N) fp32), and
//               d q_a = w_a sum_n d u_n (1 - tanh^2(q_a + P_na))                        [on the BPTT critical path]
//   deferred  : d P[b,n,a] = w_a sum_t d u[t,b,n] (1 - tanh^2(q[t,b,a] + P[b,n,a])) and d w_a, ONCE after the
//               time loop, instead of a 2 x 28 MB fp32 read-modify-write of d P at every step.
#include "kernels.cuh"
#include "prof.cuh"
#include "ptx.cuh"
#include "attention_dev.cuh"

namespace sscvae {

#define LAUNCHED() do { CUDA_TRY(cudaGetLastError()); ++g_launch_count_pw; } while (0)

using namespace attn;


__global__ void __launch_bounds__(ATT_THREADS, 2)
attention_fwd_kernel(AttnArgs a, AttnPlan pl, float* __restrict__ alpha, float* __restrict__ smx, bf16* __restrict__ xhat,
                     int ld_x) {
  extern __shared__ __align__(128) uint8_t att_smem_raw[];
  const AttnSmem sm = carve(att_smem_raw, a, false);
  attn_prologue(sm, a, false);
  pdl_wait();                                        // the prologue overlaps the previous kernel's tail
  pdl_launch_dependents(2);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int r_begin = blockIdx.x * pl.rows_per_cta;
  const int r_end = min(a.R, r_begin + pl.rows_per_cta);
  Ring ring;

  if (warp == ATT_CWARPS) {                          // ---- producer
    if (lane == 0) {
      const uint64_t pol = ptx::l2_policy_evict_first();
      for (int r = r_begin; r < r_end; ++r) {
        const int img = a.rowmap ? a.rowmap[r] : r;
        produce_block(sm, ring, reinterpret_cast<const uint8_t*>(a.proj + (size_t)img * a.N * a.Ap), a.N, a.Ap * 2, pl.nP, pl.bP, pol);
        produce_block(sm, ring, reinterpret_cast<const uint8_t*>(a.feats + (size_t)img * a.N * a.Fp), a.N, a.Fp * 2, pl.nF, pl.bF, pol);
      }
    }
    return;
  }
  // ---- consumers
  if (r_begin < r_end) {
    prefetch_vec(sm.q(0), a.q + (size_t)r_begin * a.ld_q, a.A);
    ptx::cp_async_commit();
  }
  int cur = 0;
  for (int r = r_begin; r < r_end; ++r, cur ^= 1) {
    const int img = a.rowmap ? a.rowmap[r] : r;
    attn_fwd_row(a, pl, sm, ring, cur, a.mask + (size_t)img * a.N, r + 1 < r_end ? a.q + (size_t)(r + 1) * a.ld_q : nullptr,
                 alpha + (size_t)r * a.N, smx ? smx + (size_t)r * a.N : nullptr, xhat + (size_t)r * ld_x);
  }
}

// ---------------------------------------------------------------------------------------------------------------
// Decode form: the rows of an image share its features (rows r = img * rows_per_image + i are contiguous:
// (state, beam) rows of CBS, latent samples of the diverse-sampling call). attention_fwd_kernel streams the image's
// N*(Ap+Fp) bf16 (203 KB) once per ROW: at 100 rows per image that is 1.3 GB of L2 -> SM traffic per decode step
// (313 us per step of the batched sampling call, 0.6 % of the per-image HBM roofline, profiles/decode_profile_r01c.txt).
// Here a CTA owns GR = 8 rows of ONE image: the projections P are copied to shared memory once and every consumer
// warp scores its own row against all N boxes (q and w_a stay in registers; MUFU.TANH is the bound: N*A per row);
// then the features stream through a small ring ONCE for all 8 rows and a thread accumulates 8 rows x 8 feature
// columns in registers (64 FMAs per 16-byte shared-memory load).
// ---------------------------------------------------------------------------------------------------------------
namespace {
constexpr int GR = 8;                               // rows per CTA = consumer warps
constexpr int G_XSTAGES = 3;
constexpr int G_XSTAGE_BYTES = 16384;
constexpr int G_PVMAX = 4;                          // 16-byte projection vectors per lane: Ap <= 1024
}  // namespace

static size_t grouped_smem_bytes(const AttnArgs& a) {
  const int N4 = (a.N + 3) & ~3;
  return 128 + (size_t)a.N * a.Ap * 2 + (size_t)G_XSTAGES * G_XSTAGE_BYTES + (1 + 2 * G_XSTAGES) * 8 + 16 + (size_t)N4 * GR * 4 + (size_t)N4 * 4 + 64;
}

__global__ void __launch_bounds__(ATT_THREADS, 2)
attention_fwd_grouped_kernel(AttnArgs a, int rows_per_image, int chunks_per_image, int bF, int nF, float* __restrict__ alpha,
                             bf16* __restrict__ xhat, int ld_x) {
  extern __shared__ __align__(128) uint8_t att_smem_raw[];
  const int N = a.N, N4 = (N + 3) & ~3;
  uint8_t* sp = att_smem_raw;
  bf16* P_s = reinterpret_cast<bf16*>(sp); sp += (size_t)N * a.Ap * 2;
  uint8_t* x_ring = sp; sp += (size_t)G_XSTAGES * G_XSTAGE_BYTES;
  uint64_t* p_full = reinterpret_cast<uint64_t*>(sp); sp += 8;
  uint64_t* x_full = reinterpret_cast<uint64_t*>(sp); sp += G_XSTAGES * 8;
  uint64_t* x_empty = reinterpret_cast<uint64_t*>(sp); sp += G_XSTAGES * 8;
  sp += (16 - ((1 + 2 * G_XSTAGES) * 8) % 16) % 16;                          // float4 reads of al_s
  float* al_s = reinterpret_cast<float*>(sp); sp += (size_t)N4 * GR * 4;      // [box][row]
  float* mask_s = reinterpret_cast<float*>(sp);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int img = blockIdx.x / chunks_per_image, chunk = blockIdx.x - img * chunks_per_image;
  const int i0 = chunk * GR;
  const int nrows = min(GR, rows_per_image - i0);
  const int r0 = img * rows_per_image + i0;
  if (threadIdx.x == 0) {
    ptx::mbar_init(p_full, 1);
    for (int s = 0; s < G_XSTAGES; ++s) { ptx::mbar_init(&x_full[s], 1); ptx::mbar_init(&x_empty[s], ATT_CWARPS); }
    ptx::mbar_fence_init();
  }
  for (int i = threadIdx.x; i < N4 * GR; i += blockDim.x) al_s[i] = 0.f;
  __syncthreads();
  pdl_wait();
  pdl_launch_dependents(2);
  for (int i = threadIdx.x; i < N4; i += blockDim.x) mask_s[i] = i < N ? a.mask[(size_t)img * N + i] : 0.f;

  if (warp == ATT_CWARPS) {                          // ---- producer: P in one go, then the feature chunks through the ring
    if (lane == 0) {
      const uint64_t pol = ptx::l2_policy_evict_first();
      const uint8_t* pbase = reinterpret_cast<const uint8_t*>(a.proj + (size_t)img * N * a.Ap);
      const uint32_t pbytes = (uint32_t)N * a.Ap * 2;
      ptx::mbar_expect_tx(p_full, pbytes);
      for (uint32_t off = 0; off < pbytes; off += 32768) {
        const uint32_t nb = min(32768u, pbytes - off);
        ptx::bulk_g2s(reinterpret_cast<uint8_t*>(P_s) + off, pbase + off, nb, p_full);
      }
      const uint8_t* fbase = reinterpret_cast<const uint8_t*>(a.feats + (size_t)img * N * a.Fp);
      int stage = 0; uint32_t phase = 0;
      for (int c = 0; c < nF; ++c) {
        const int n0 = c * bF, nb = min(bF, N - n0);
        const uint32_t bytes = (uint32_t)nb * a.Fp * 2;
        ptx::mbar_wait(&x_empty[stage], phase ^ 1);
        ptx::mbar_expect_tx(&x_full[stage], bytes);
        ptx::bulk_g2s_hint(x_ring + (size_t)stage * G_XSTAGE_BYTES, fbase + (size_t)n0 * a.Fp * 2, bytes, &x_full[stage], pol);
        if (++stage == G_XSTAGES) { stage = 0; phase ^= 1; }
      }
    }
    return;
  }
  // ---- consumers: warp w scores row i0 + w
  ptx::bar_sync(1, ATT_CONSUMERS);                   // mask_s visible
  const int nvec = a.Ap >> 3;
  if (warp < nrows) {
    const int r = r0 + warp;
    float qv[G_PVMAX][8], wv[G_PVMAX][8];
#pragma unroll
    for (int v = 0; v < G_PVMAX; ++v) {
      const int i = lane + 32 * v;
#pragma unroll
      for (int k = 0; k < 8; ++k) {
        const int col = i * 8 + k;
        const bool ok = i < nvec && col < a.A;
        qv[v][k] = ok ? a.q[(size_t)r * a.ld_q + col] : 0.f;
        wv[v][k] = ok ? a.w_a[col] : 0.f;
      }
    }
    ptx::mbar_wait(p_full, 0);
    float u[ATT_NREG];
#pragma unroll
    for (int k = 0; k < ATT_NREG; ++k) u[k] = 0.f;
    for (int n = 0; n < N; ++n) {
      float s = 0.f;
      if (mask_s[n] != 0.f) {                        // masked boxes enter the softmax as u*m = 0
        const bf16x8* prow = reinterpret_cast<const bf16x8*>(P_s + (size_t)n * a.Ap);
#pragma unroll
        for (int v = 0; v < G_PVMAX; ++v) {
          const int i = lane + 32 * v;
          if (i < nvec) {
            const bf16x8 pv = prow[i];
            const float2 f0 = __bfloat1622float2(pv.v[0]), f1 = __bfloat1622float2(pv.v[1]);
            const float2 f2 = __bfloat1622float2(pv.v[2]), f3 = __bfloat1622float2(pv.v[3]);
            s += wv[v][0] * tanh_approx(qv[v][0] + f0.x) + wv[v][1] * tanh_approx(qv[v][1] + f0.y);
            s += wv[v][2] * tanh_approx(qv[v][2] + f1.x) + wv[v][3] * tanh_approx(qv[v][3] + f1.y);
            s += wv[v][4] * tanh_approx(qv[v][4] + f2.x) + wv[v][5] * tanh_approx(qv[v][5] + f2.y);
            s += wv[v][6] * tanh_approx(qv[v][6] + f3.x) + wv[v][7] * tanh_approx(qv[v][7] + f3.y);
          }
        }
        s = warp_sum(s);
      }
#pragma unroll
      for (int k = 0; k < ATT_NREG; ++k)
        if (n == lane + 32 * k) u[k] = s;
    }
    // masked softmax (allennlp: softmax(u*m)*m / (sum + 1e-13)); lane holds boxes lane, lane+32, ...
    float m[ATT_NREG], x[ATT_NREG];
    float mx = -INFINITY;
#pragma unroll
    for (int k = 0; k < ATT_NREG; ++k) {
      const int n = lane + 32 * k;
      m[k] = n < N ? mask_s[n] : 0.f;
      x[k] = n < N ? u[k] * m[k] : -INFINITY;
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
    for (int k = 0; k < ATT_NREG; ++k) { x[k] = x[k] / se; sr += x[k] * m[k]; }
    sr = warp_sum(sr);
    const float Rn = sr + 1e-13f;
#pragma unroll
    for (int k = 0; k < ATT_NREG; ++k) {
      const int n = lane + 32 * k;
      if (n < N) {
        const float al = x[k] * m[k] / Rn;
        alpha[(size_t)r * N + n] = al;
        al_s[n * GR + warp] = al;
      }
    }
  }
  ptx::bar_sync(1, ATT_CONSUMERS);                   // alpha of all rows of the chunk is in shared memory
  // ---- weighted sum: thread = 8 feature columns x 8 rows
  const int nfv = a.Fp >> 3;
  float acc[GR][8];
#pragma unroll
  for (int i = 0; i < GR; ++i)
#pragma unroll
    for (int k = 0; k < 8; ++k) acc[i][k] = 0.f;
  int stage = 0; uint32_t phase = 0;
  for (int c = 0; c < nF; ++c) {
    const int n0 = c * bF, nb = min(bF, N - n0);
    ptx::mbar_wait(&x_full[stage], phase);
    const uint4* buf = reinterpret_cast<const uint4*>(x_ring + (size_t)stage * G_XSTAGE_BYTES);
    if ((int)threadIdx.x < nfv) {
      for (int j = 0; j < nb; ++j) {
        const uint4 xq = buf[(size_t)j * nfv + threadIdx.x];
        float xf[8];
        xf[0] = __uint_as_float(xq.x << 16); xf[1] = __uint_as_float(xq.x & 0xffff0000u);
        xf[2] = __uint_as_float(xq.y << 16); xf[3] = __uint_as_float(xq.y & 0xffff0000u);
        xf[4] = __uint_as_float(xq.z << 16); xf[5] = __uint_as_float(xq.z & 0xffff0000u);
        xf[6] = __uint_as_float(xq.w << 16); xf[7] = __uint_as_float(xq.w & 0xffff0000u);
        const float4 w0 = *reinterpret_cast<const float4*>(al_s + (n0 + j) * GR);
        const float4 w1 = *reinterpret_cast<const float4*>(al_s + (n0 + j) * GR + 4);
        const float w[8] = {w0.x, w0.y, w0.z, w0.w, w1.x, w1.y, w1.z, w1.w};
#pragma unroll
        for (int i = 0; i < GR; ++i)
#pragma unroll
          for (int k = 0; k < 8; ++k) acc[i][k] = fmaf(w[i], xf[k], acc[i][k]);
      }
    }
    __syncwarp();
    if (lane == 0) ptx::mbar_arrive(&x_empty[stage]);
    if (++stage == G_XSTAGES) { stage = 0; phase ^= 1; }
  }
  if ((int)threadIdx.x < nfv) {
#pragma unroll
    for (int i = 0; i < GR; ++i) {
      if (i < nrows) {
        bf16x8 o;
#pragma unroll
        for (int k = 0; k < 4; ++k) o.v[k] = __floats2bfloat162_rn(acc[i][2 * k], acc[i][2 * k + 1]);
        st_bf16x8(xhat + (size_t)(r0 + i) * ld_x + threadIdx.x * 8, o);
      }
    }
  }
}

static int make_plan(const AttnArgs& a, AttnPlan& pl) {
  if (a.N > 32 * ATT_NREG || a.Fp > 8 * ATT_CONSUMERS * ATT_FV || a.Ap > 2 * ATT_CONSUMERS * ATT_PV ||
      a.Ap * 2 > ATT_STAGE_BYTES || a.Fp * 2 > ATT_STAGE_BYTES || attn_smem_bytes(a, true) > 112 * 1024) {
    set_error("attention: unsupported shape N=%d (<= %d) Fp=%d (<= %d) Ap=%d (<= %d)", a.N, 32 * ATT_NREG, a.Fp,
              8 * ATT_CONSUMERS * ATT_FV, a.Ap, 2 * ATT_CONSUMERS * ATT_PV);
    return SSCVAE_ERR_UNSUPPORTED;
  }
  REQUIRE((a.Ap % 8) == 0 && (a.Fp % 8) == 0, "attention: Ap/Fp must be multiples of 8");
  pl = attn_chunk_plan(a);
  static int n_sm = 0;
  if (n_sm == 0) {
    int dev = 0;
    CUDA_TRY(cudaGetDevice(&dev));
    CUDA_TRY(cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, dev));
  }
  pl.rows_per_cta = ceil_div(a.R, 2 * n_sm);
  return 0;
}

int attention_forward(cudaStream_t s, const AttnArgs& a, float* alpha, float* smx, bf16* xhat, int ld_x) {
  PROF_SCOPE(s, "attention_fwd", 0, (double)a.R*((double)a.N*(a.Ap+a.Fp)*2.0 + a.A*4.0 + a.Fp*2.0 + a.N*4.0));
  REQUIRE(a.R > 0 && (ld_x % 8) == 0 && (reinterpret_cast<uintptr_t>(xhat) & 15) == 0, "attention_forward: bad xhat layout");
  AttnPlan pl;
  TRY(make_plan(a, pl));
  // decode: rows of an image are contiguous and share its features -> one CTA per 8 rows of an image
  static const bool no_grouped = [] { const char* e = getenv("SSCVAE_ATT_GROUPED"); return e && e[0] == '0'; }();
  if (!no_grouped && a.rows_per_image >= 4 && smx == nullptr && a.Fp <= 8 * ATT_CONSUMERS && a.Ap <= 256 * G_PVMAX &&
      (a.R % a.rows_per_image) == 0 && grouped_smem_bytes(a) <= 113 * 1024 && pl.bF * a.Fp * 2 <= G_XSTAGE_BYTES) {
    const size_t gsmem = grouped_smem_bytes(a);
    static bool gconf = false;
    if (!gconf) {
      CUDA_TRY(cudaFuncSetAttribute(attention_fwd_grouped_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 113 * 1024));
      gconf = true;
    }
    const int cpi = ceil_div(a.rows_per_image, GR);
    const int images = a.R / a.rows_per_image;
    CUDA_TRY(launch_pdl(attention_fwd_grouped_kernel, dim3(images * cpi), dim3(ATT_THREADS), gsmem, s, a, a.rows_per_image, cpi, pl.bF,
                        pl.nF, alpha, xhat, ld_x));
    LAUNCHED();
    return 0;
  }
  const size_t smem = attn_smem_bytes(a, false);
  static bool configured = false;
  if (!configured) {
    CUDA_TRY(cudaFuncSetAttribute(attention_fwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 112 * 1024));
    configured = true;
  }
  CUDA_TRY(launch_pdl(attention_fwd_kernel, dim3(ceil_div(a.R, pl.rows_per_cta)), dim3(ATT_THREADS), smem, s, a, pl, alpha, smx, xhat, ld_x));
  LAUNCHED();
  return 0;
}

// ---- per-step backward: d u (saved) and d q ------------------------------------------------------
__global__ void __launch_bounds__(ATT_THREADS, 2)
attention_bwd_kernel(AttnArgs a, AttnPlan pl, const float* __restrict__ smx, const float* __restrict__ dxhat, int ld_dx,
                     bf16* __restrict__ dq, int ld_dq, float* __restrict__ du) {
  extern __shared__ __align__(128) uint8_t att_smem_raw[];
  const AttnSmem sm = carve(att_smem_raw, a, true);
  attn_prologue(sm, a, true);
  pdl_wait();                                        // the prologue overlaps the previous kernel's tail
  pdl_launch_dependents(2);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int r_begin = blockIdx.x * pl.rows_per_cta;
  const int r_end = min(a.R, r_begin + pl.rows_per_cta);
  Ring ring;

  if (warp == ATT_CWARPS) {                          // ---- producer: region features first, then projections
    if (lane == 0) {
      const uint64_t pol = ptx::l2_policy_evict_first();
      for (int r = r_begin; r < r_end; ++r) {
        const int img = a.rowmap ? a.rowmap[r] : r;
        produce_block(sm, ring, reinterpret_cast<const uint8_t*>(a.feats + (size_t)img * a.N * a.Fp), a.N, a.Fp * 2, pl.nF, pl.bF, pol);
        produce_block(sm, ring, reinterpret_cast<const uint8_t*>(a.proj + (size_t)img * a.N * a.Ap), a.N, a.Ap * 2, pl.nP, pl.bP, pol);
      }
    }
    return;
  }
  // ---- consumers
  auto prefetch_row = [&](int r, int slot) {
    prefetch_vec(sm.q(slot), a.q + (size_t)r * a.ld_q, a.A);
    prefetch_vec(sm.dx(slot), dxhat + (size_t)r * ld_dx, a.F);
    prefetch_vec(sm.sv(slot), smx + (size_t)r * a.N, a.N);
    ptx::cp_async_commit();
  };
  if (r_begin < r_end) prefetch_row(r_begin, 0);
  const int nfv = a.Fp >> 3, npair = a.Ap >> 1;
  int cur = 0;
  for (int r = r_begin; r < r_end; ++r, cur ^= 1) {
    const int img = a.rowmap ? a.rowmap[r] : r;
    const float* mask_img = a.mask + (size_t)img * a.N;
    ptx::cp_async_wait_all();
    ptx::bar_sync(1, ATT_CONSUMERS);
    if (r + 1 < r_end) prefetch_row(r + 1, cur ^ 1);
    const float* dx_s = sm.dx(cur);
    // d alpha_n = d xhat . x_n : warp per box
    for (int c = 0; c < pl.nF; ++c) {
      const int n0 = c * pl.bF, nb = min(pl.bF, a.N - n0);
      ptx::mbar_wait(&sm.full[ring.stage], ring.phase);
      const bf16x8* buf = reinterpret_cast<const bf16x8*>(sm.stage + (size_t)ring.stage * ATT_STAGE_BYTES);
      const int wpb = warps_per_box(nb);
      const int j = warp / wpb, sub = warp % wpb;
      if (j < nb) {
        const int n = n0 + j;
        float s = 0.f;
        if (mask_img[n] != 0.f) {
          const bf16x8* p = buf + (size_t)j * nfv;
          for (int i = sub * 32 + lane; i < nfv; i += 32 * wpb) {
            const bf16x8 v = p[i];
            const float4 da = *reinterpret_cast<const float4*>(dx_s + i * 8);
            const float4 db = *reinterpret_cast<const float4*>(dx_s + i * 8 + 4);
            const float2 f0 = __bfloat1622float2(v.v[0]), f1 = __bfloat1622float2(v.v[1]);
            const float2 f2 = __bfloat1622float2(v.v[2]), f3 = __bfloat1622float2(v.v[3]);
            s += da.x * f0.x + da.y * f0.y + da.z * f1.x + da.w * f1.y;
            s += db.x * f2.x + db.y * f2.y + db.z * f3.x + db.w * f3.y;
          }
          s = warp_sum(s);
        }
        if (lane == 0) sm.u[sub * sm.N4 + n] = s;
      }
      __syncwarp();
      if (lane == 0) ptx::mbar_arrive(&sm.empty[ring.stage]);
      ring.advance();
    }
    ptx::bar_sync(1, ATT_CONSUMERS);
    // softmax backward, redundantly per warp. alpha = r/R with r = s*m:  dr = (dalpha - sum_k dalpha_k alpha_k)/R,
    // ds = dr*m; softmax backward on x = u*m; du = dx*m
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
        da[k] = ok ? gather_partial(sm.u, sm.N4, a.N, pl.bF, n) + (a.dalpha_extra ? a.dalpha_extra[(size_t)r * a.N + n] : 0.f) : 0.f;
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
        if (n < a.N) du[(size_t)r * a.N + n] = duv[k];
      }
    }
    // d q_a = w_a sum_n du_n (1 - tanh^2(q_a + P_na)): a thread owns pairs of projection columns
    const float* q_s = sm.q(cur);
    float g[ATT_PV][2];
#pragma unroll
    for (int v = 0; v < ATT_PV; ++v) g[v][0] = g[v][1] = 0.f;
    for (int c = 0; c < pl.nP; ++c) {
      const int n0 = c * pl.bP, nb = min(pl.bP, a.N - n0);
      ptx::mbar_wait(&sm.full[ring.stage], ring.phase);
      const __nv_bfloat162* buf = reinterpret_cast<const __nv_bfloat162*>(sm.stage + (size_t)ring.stage * ATT_STAGE_BYTES);
      for (int j = 0; j < nb; ++j) {
        const int n = n0 + j;
        const float d = __shfl_sync(0xffffffffu, pick(duv, n >> 5), n & 31);
        if (d != 0.f) {                              // warp-uniform (masked boxes, padded timesteps)
#pragma unroll
          for (int v = 0; v < ATT_PV; ++v) {
            const int cp = threadIdx.x + ATT_CONSUMERS * v;
            if (cp < npair) {
              const float2 f = __bfloat1622float2(buf[(size_t)j * npair + cp]);
              const float t0 = tanh_approx(q_s[2 * cp] + f.x), t1 = tanh_approx(q_s[2 * cp + 1] + f.y);
              g[v][0] += d * (1.f - t0 * t0);
              g[v][1] += d * (1.f - t1 * t1);
            }
          }
        }
      }
      __syncwarp();
      if (lane == 0) ptx::mbar_arrive(&sm.empty[ring.stage]);
      ring.advance();
    }
#pragma unroll
    for (int v = 0; v < ATT_PV; ++v) {
      const int cp = threadIdx.x + ATT_CONSUMERS * v;
      if (cp < npair && 2 * cp < ld_dq)
        *reinterpret_cast<__nv_bfloat162*>(dq + (size_t)r * ld_dq + 2 * cp) =
            __floats2bfloat162_rn(sm.wa[2 * cp] * g[v][0], sm.wa[2 * cp + 1] * g[v][1]);
    }
  }
}

int attention_backward(cudaStream_t s, const AttnArgs& a, const float* smx, const float* dxhat, int ld_dx, bf16* dq,
                       int ld_dq, float* du) {
  PROF_SCOPE(s, "attention_bwd", 0, (double)a.R*((double)a.N*(a.Ap+a.Fp)*2.0 + a.Fp*4.0 + a.A*6.0 + a.N*8.0));
  REQUIRE(a.R > 0 && (ld_dq % 2) == 0 && (reinterpret_cast<uintptr_t>(dq) & 3) == 0, "attention_backward: bad dq layout");
  AttnPlan pl;
  TRY(make_plan(a, pl));
  const size_t smem = attn_smem_bytes(a, true);
  static bool configured = false;
  if (!configured) {
    CUDA_TRY(cudaFuncSetAttribute(attention_bwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 112 * 1024));
    configured = true;
  }
  CUDA_TRY(launch_pdl(attention_bwd_kernel, dim3(ceil_div(a.R, pl.rows_per_cta)), dim3(ATT_THREADS), smem, s, a, pl, smx, dxhat, ld_dx, dq,
                      ld_dq, du));
  LAUNCHED();
  return 0;
}

// ---- deferred backward: d P and d w_a over all timesteps at once (training layout: row = t*B + b, image b) ----
constexpr int DEF_COLS = 256;
__global__ void __launch_bounds__(DEF_COLS)
attention_bwd_deferred_kernel(int T, int B, int N, int A, int Ap, const float* __restrict__ q_all,
                              const float* __restrict__ du_all, const bf16* __restrict__ proj, const float* __restrict__ w_a,
                              float* __restrict__ dproj, float* __restrict__ dwa_rows) {
  extern __shared__ float dsm[];
  float* q_s = dsm;                         // T x DEF_COLS
  float* du_s = q_s + (size_t)T * DEF_COLS; // T x N
  int* act = reinterpret_cast<int*>(du_s + (size_t)T * N);   // T
  const int b = blockIdx.x;
  const int a0 = blockIdx.y * DEF_COLS;
  const int col = a0 + threadIdx.x;
  const bool ok = col < A;
  for (int t = threadIdx.x; t < T; t += blockDim.x) act[t] = 0;
  __syncthreads();
  for (int i = threadIdx.x; i < T * N; i += blockDim.x) {
    const int t = i / N, n = i - t * N;
    const float v = du_all[((size_t)t * B + b) * N + n];
    du_s[i] = v;
    if (v != 0.f) act[t] = 1;               // benign race: all writers store 1
  }
  for (int t = 0; t < T; ++t) q_s[t * DEF_COLS + threadIdx.x] = ok ? q_all[((size_t)t * B + b) * A + col] : 0.f;
  __syncthreads();
  const float wa = ok ? w_a[col] : 0.f;
  float dw = 0.f;
  for (int n = 0; n < N; ++n) {
    const float p = ok ? __bfloat162float(proj[((size_t)b * N + n) * Ap + col]) : 0.f;
    float acc = 0.f;
    for (int t = 0; t < T; ++t) {
      if (!act[t]) continue;                // padded timesteps carry no gradient
      const float d = du_s[t * N + n];
      const float th = tanh_approx(q_s[t * DEF_COLS + threadIdx.x] + p);
      acc += d * (1.f - th * th);
      dw += d * th;
    }
    if (ok) dproj[((size_t)b * N + n) * A + col] = wa * acc;
  }
  if (ok) dwa_rows[(size_t)b * A + col] = dw;
}

int attention_backward_deferred(cudaStream_t s, const AttnArgs& a, int T, const float* q_all, const float* du_all,
                                float* dproj, float* dwa_rows) {
  PROF_SCOPE(s, "attention_bwd_deferred", 0,
             (double)a.R * ((double)T * (a.A + a.N) * 4.0 + (double)a.N * a.Ap * 2.0 + (double)a.N * a.A * 4.0));
  REQUIRE(a.rowmap == nullptr && a.ld_q == a.A, "attention_backward_deferred: training layout only");
  const size_t smem = ((size_t)T * DEF_COLS + (size_t)T * a.N + T) * 4;
  REQUIRE(smem <= 200 * 1024, "attention_backward_deferred: T=%d too long", T);
  static bool configured = false;
  if (!configured) {
    CUDA_TRY(cudaFuncSetAttribute(attention_bwd_deferred_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
    configured = true;
  }
  dim3 grid(a.R, ceil_div(a.A, DEF_COLS));
  attention_bwd_deferred_kernel<<<grid, DEF_COLS, smem, s>>>(T, a.R, a.N, a.A, a.Ap, q_all, du_all, a.proj, a.w_a, dproj,
                                                            dwa_rows);
  LAUNCHED();
  return 0;
}

}  // namespace sscvae

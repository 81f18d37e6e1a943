// Persistent recurrent kernel of the training forward pass (north_star kernel #1): ONE cooperative launch runs all
// T teacher-forced timesteps of the UpDown cell (var_updown/var_updown/modules/updown_cell.py:123-231):
// attention LSTM -> query projection -> region attention -> posterior (encoder) LSTM -> fc_mean / fc_log_var ->
// reparameterised z + KL -> language (decoder) LSTM. Nothing is launched per step and no gate pre-activation ever
// leaves the SM: the LSTM cells, the latent sampling and the attention run where the accumulators are.
//
// Decomposition (B <= 256 rows, batch on the UMMA M side):
//   * the grid is one CTA per SM, grouped in CTA pairs (clusters of 2). A pair drives tcgen05.mma.cta_group::2 with
//     M = 256 = the whole batch (CTA r holds rows [128r, 128r+128) in its TMEM lanes) and N = a tile of weight rows, so
//     every weight byte crosses L2 -> SM exactly once per timestep;
//   * the forward LSTM weights are packed gate-interleaved (kernels.cuh: lstm_gate_row): a tile of 128 weight rows =
//     4 gates x 32 hidden units. Pair i < nt owns tile i of the attention LSTM and of the encoder LSTM, pair nt + i
//     owns tile i of the decoder LSTM; an epilogue thread (= one batch row) reads the four gates of a unit from
//     TMEM columns k*32 + u, applies the cell in registers and writes h (bf16, into every operand buffer that
//     consumes it), c and the activated gates (fp32, saved for BPTT);
//   * the remaining pairs own one Nq-column tile of the query projection and one 16-dimension tile of
//     [fc_mean ; fc_log_var] (CTA 0 of the pair loads the 16 mean rows, CTA 1 the 16 log-variance rows of the weight,
//     so the accumulator holds mean_j and log_var_j side by side) with the reparameterisation + KL in its epilogue;
//   * the region attention (attention_dev.cuh) runs on the same 8 compute warps of EVERY CTA, rows r = cta, cta + G, ...;
//     its producer warp streams the image's projections / features through its own bulk-copy ring and runs ahead
//     across timesteps.
// There is no grid-wide barrier. Producers of a tensor bump a monotonic counter in global memory (release) after their
// stores; the TMA producer thread of a consuming pair polls it (acquire) in front of the k-blocks that read the tensor.
// K segments are ordered by availability: the encoder / decoder tiles first accumulate their h_enc_{t-1}, h_dec_{t-1}
// and h1_t column blocks while the attention of step t is still streaming features, then the x_hat block, and the
// decoder tile keeps its accumulator in TMEM until z_t exists and adds the z block (K = Zp) last.
// Deadlock freedom: a pair's jobs are issued in a fixed order and no job depends on a later job of the same pair
// (q / fc tiles never share a pair with LSTM tiles); the launch is cooperative (all CTAs co-resident). Every wait
// is bounded: on a timeout the kernel raises the abort flag, prints the wait that failed and traps.
#define PK_NAME "recurrent_fwd"
#include "persistent.cuh"
#include <curand_kernel.h>

namespace sscvae {

namespace {

constexpr int RF_STAGES = 6;

// One counter per tensor family. The hidden states (FLAG_H1, FLAG_HDEC, FLAG_HENC) are bumped by both CTAs of every
// LSTM tile's pair: 2 * nt signals per timestep.
enum { FLAG_H1 = 0, FLAG_HDEC, FLAG_HENC, FLAG_XHAT, FLAG_Q, FLAG_Z, FLAG_ABORT, FLAG_COUNT };
enum { MAP_XA = 0, MAP_XE, MAP_HE, MAP_ZB, MAP_EMB, NUM_AMAPS };
enum { WMAP_ATT = 0, WMAP_Q, WMAP_ENC_X, WMAP_ENC_HH, WMAP_FC, WMAP_DEC_X, WMAP_DEC_Z, WMAP_ATT_E, NUM_WMAPS };
enum { SLOT_ATT = 0, SLOT_LSTM, SLOT_Q, SLOT_FC, NUM_SLOTS };
enum { ROLE_ENC = 0, ROLE_DEC, ROLE_SPARE };
// TMEM columns. LSTM pairs: two accumulators and the time-invariant addends of their gate pre-activations (biases,
// mean-feature block, sentiment column), written once at kernel start; the other pairs: q and [mean | log_var].
constexpr int TMEM_COL_ATT = 0, TMEM_COL_LSTM = 128, TMEM_COL_ATT_CONST = 256, TMEM_COL_LSTM_CONST = 384;
constexpr int TMEM_COL_Q = 0, TMEM_COL_FC = 128;

struct RfSeg {
  int amap, wmap;          // activation / weight tensor map
  int acol0, wcol0;        // first K column (elements) in each
  int kblocks;
  int t_off;               // the activation is read at time index t + t_off
  int flag;                // counter that must reach (t + flag_toff) * flag_mult before the segment is loaded (-1: none);
                           // FLAG_H1 / FLAG_HDEC / FLAG_HENC: (t + flag_toff) * flag_mult * nt
  int flag_mult, flag_toff;
};
struct RfJob {
  int nseg;
  RfSeg seg[4];
  int w_row[2];            // first weight row loaded by CTA 0 / CTA 1 of the pair
  int w_box_rows;          // rows per CTA (= N / 2)
  int N;                   // UMMA N
  int tmem_col;
  int slot;                // accumulator-ready barrier
};

struct RfParams {
  CUtensorMap amap[NUM_AMAPS];     // 3-D (k, batch row, t), box 64 x 128 x 1, 128B swizzle
  CUtensorMap wmap[NUM_WMAPS];     // 2-D (k, weight row), box 64 x w_box_rows
  int B, T, H, Hp, Fp, Zp, Z, A, KX, GP, Ep;
  int nt;                          // tiles per LSTM = GP / 128
  int nq, Nq;                      // query-projection tiles and their width
  int nfc;                         // latent tiles (16 dimensions each)
  int sentiment_vae;
  float prior_var;
  // LSTM cell epilogues
  const float* gavg;
  const float* b_att; const float* b_enc; const float* b_dec;
  const float* sent; const float* scol_enc; const float* scol_dec;
  float* c1; float* c_enc; float* c_dec;
  float* gates_att; float* gates_enc; float* gates_dec;
  bf16* XA; bf16* XE; bf16* HE; bf16* ZB;
  // query projection / latent epilogues
  float* q;
  const float* b_fc; const float* eps_in; const unsigned long long* seed; const float* pm_row;
  float* mean; float* logvar; float* eps_out; float* kl_part;
  // attention
  AttnArgs att; AttnPlan plan;
  float* alpha; float* smx;
  unsigned int* flags;
  static constexpr int ABORT_FLAG = FLAG_ABORT;
  unsigned long long timeout_ns;
  unsigned long long* dbg;         // SSCVAE_RF_DBG=1: globaltimer stamps of step dbg_t, 32 per CTA
  int dbg_t;
};

#define RF_STAMP(cond, i)                                                                   \
  do {                                                                                     \
    if (p.dbg && t == p.dbg_t && (cond)) p.dbg[(size_t)blockIdx.x * 32 + (i)] = globaltimer_ns(); \
  } while (0)

__device__ __forceinline__ float philox_normal_rf(unsigned long long seed, unsigned long long step, int r, int z, int Z) {
  curandStatePhilox4_32_10_t st;                       // the stream of pointwise.cu: latent_fwd_train_kernel
  curand_init(seed, (unsigned long long)r * Z + z, step, &st);
  return curand_normal(&st);
}

using RfSmem = PkSmem<RfJob, RF_STAGES, NUM_SLOTS>;

__device__ __forceinline__ float4 ld4g(const float* p) { return *reinterpret_cast<const float4*>(p); }
__device__ __forceinline__ void add4v(float* v, const float4& w) { v[0] += w.x; v[1] += w.y; v[2] += w.z; v[3] += w.w; }
__device__ __forceinline__ void fma4v(float* v, float s, const float4& w) {
  v[0] = fmaf(s, w.x, v[0]); v[1] = fmaf(s, w.y, v[1]); v[2] = fmaf(s, w.z, v[2]); v[3] = fmaf(s, w.w, v[3]);
}
__device__ __forceinline__ void st_bf16x4_rf(bf16* p, const float* h) {
  __nv_bfloat162 lo = __floats2bfloat162_rn(h[0], h[1]), hi = __floats2bfloat162_rn(h[2], h[3]);
  uint2 o;
  o.x = *reinterpret_cast<uint32_t*>(&lo);
  o.y = *reinterpret_cast<uint32_t*>(&hi);
  *reinterpret_cast<uint2*>(p) = o;
}

__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// Branch-free gate nonlinearities: the epilogue warps run two per SM sub-partition with little to hide instruction
// latency behind, and tanhf / IEEE division are ~4x the instructions. Absolute error <= 2e-7, far inside the bf16
// operand rounding of the next GEMM.
__device__ __forceinline__ float cell_sigmoid(float x) { return __fdividef(1.0f, 1.0f + __expf(-x)); }
__device__ __forceinline__ float cell_tanh(float x) { return 1.0f - __fdividef(2.0f, 1.0f + __expf(2.0f * x)); }

// Saved LSTM state in the "row-tiled" layout of the persistent kernels (kernels.cuh: lstm_tiled_*): within the block of
// one timestep, 4 consecutive hidden units of one batch row are 16 contiguous bytes and consecutive rows follow each
// other, so a warp whose lanes are 32 batch rows stores 512 contiguous bytes per instruction.

// Time-invariant part of the gate pre-activations of this thread's row, written to TMEM once: b_ih + b_hh, and for the
// attention LSTM the mean-feature block W_ih[:, avg] x_avg (hoisted GEMM `gavg`), for the encoder / decoder LSTM the
// sentiment column sent[b] * W_ih[:, cond] (updown_cell.py:143-148, 178-194, 211-229).
template <int WHICH>
__device__ __forceinline__ void init_lstm_const(const RfParams& p, int tile, uint32_t tmem_base, int cw, int lane, int rank) {
  const int qd = (cw + 2) & 3, half = cw >> 2;
  const int b = rank * 128 + qd * 32 + lane;
  const bool ok = b < p.B;
  const int H = p.H;
  const float* bias = WHICH == 0 ? p.b_att : WHICH == 1 ? p.b_enc : p.b_dec;
  const float* scol = WHICH == 1 ? p.scol_enc : WHICH == 2 ? p.scol_dec : nullptr;
  const float sv = (WHICH != 0 && p.sent && ok) ? p.sent[b] : 0.f;
  const uint32_t taddr = tmem_base + (static_cast<uint32_t>(qd * 32) << 16) + (WHICH == 0 ? TMEM_COL_ATT_CONST : TMEM_COL_LSTM_CONST);
#pragma unroll 1
  for (int k = 0; k < 4; ++k)
#pragma unroll 1
    for (int c = 0; c < 2; ++c) {
      const int u0 = half * 16 + c * 8, j0 = tile * 32 + u0;
      float v[8];
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        v[i] = 0.f;
        if (ok && j0 + i < H) {
          v[i] = bias[k * H + j0 + i];
          if (WHICH == 0) v[i] += p.gavg[(size_t)b * p.GP + tile * 128 + k * 32 + u0 + i];
          else if (p.sent) v[i] = fmaf(sv, scol[k * H + j0 + i], v[i]);
        }
      }
      tmem_st_x8(taddr + k * 32 + u0, v);
    }
  tmem_st_wait();
}

// LSTM cell epilogue (torch.nn.LSTMCell, gate order i,f,g,o; updown_cell.py:143-148, 192-194, 226-229) of one 128-column
// tile (32 hidden units x 4 gates). WHICH: 0 attention LSTM, 1 encoder, 2 decoder. A thread = one batch row x 16 units.
template <int WHICH>
__device__ __forceinline__ void epi_lstm(const RfParams& p, const RfSmem& sm, int t, int tile, uint32_t tmem_base, int cw, int lane,
                                         int rank) {
  const int qd = (cw + 2) & 3;                         // TMEM lane quadrant of this warp (warp id % 4)
  const int half = cw >> 2;                            // which 16 of the tile's 32 units
  const int b = rank * 128 + qd * 32 + lane;
  const bool ok = b < p.B;
  const int H = p.H, H4 = H >> 2, B = p.B;
  const size_t r = (size_t)t * B + b;
  float* cbuf = (WHICH == 0 ? p.c1 : WHICH == 1 ? p.c_enc : p.c_dec) + (size_t)t * B * H;           // block of step t
  float* gbuf = (WHICH == 0 ? p.gates_att : WHICH == 1 ? p.gates_enc : p.gates_dec) + (size_t)t * B * 4 * H;
  const uint32_t tlane = tmem_base + (static_cast<uint32_t>(qd * 32) << 16);
  const uint32_t tacc = tlane + (WHICH == 0 ? TMEM_COL_ATT : TMEM_COL_LSTM);
  const uint32_t tcon = tlane + (WHICH == 0 ? TMEM_COL_ATT_CONST : TMEM_COL_LSTM_CONST);
  // c_{t-1} of this thread's 16 units: independent of the accumulator, loaded before waiting for it
  float cp[2][8];
#pragma unroll
  for (int chunk = 0; chunk < 2; ++chunk) {
    const int jq0 = (tile * 32 + half * 16 + chunk * 8) >> 2;
#pragma unroll
    for (int v4 = 0; v4 < 2; ++v4) {
      float4 c4 = make_float4(0.f, 0.f, 0.f, 0.f);
      if (ok && t > 0 && jq0 + v4 < H4) c4 = ld4g(cbuf - (size_t)B * H + ((size_t)(jq0 + v4) * B + b) * 4);
      cp[chunk][v4 * 4] = c4.x; cp[chunk][v4 * 4 + 1] = c4.y; cp[chunk][v4 * 4 + 2] = c4.z; cp[chunk][v4 * 4 + 3] = c4.w;
    }
  }
  mbar_wait_bounded(p, &sm.tfull[WHICH == 0 ? SLOT_ATT : SLOT_LSTM], (uint32_t)(t & 1), 10 + WHICH, t);
  tc_fence_after();
  RF_STAMP(cw == 0 && lane == 0, WHICH == 0 ? 8 : 9);
#pragma unroll
  for (int chunk = 0; chunk < 2; ++chunk) {
    const int u0 = half * 16 + chunk * 8;              // unit inside the tile
    const int j0 = tile * 32 + u0;                     // hidden unit
    const int nv = min(8, max(0, H - j0));             // valid units of this chunk (H % 4 == 0)
    float acc[4][8], pre[4][8];
#pragma unroll
    for (int k = 0; k < 4; ++k) { tmem_ld_x8(tacc + k * 32 + u0, acc[k]); tmem_ld_x8(tcon + k * 32 + u0, pre[k]); }
    tmem_ld_wait();
    if (ok && nv > 0) {
      float gi[8], gf[8], gg[8], go[8], c[8], h[8];
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        gi[i] = cell_sigmoid(acc[0][i] + pre[0][i]);
        gf[i] = cell_sigmoid(acc[1][i] + pre[1][i]);
        gg[i] = cell_tanh(acc[2][i] + pre[2][i]);
        go[i] = cell_sigmoid(acc[3][i] + pre[3][i]);
        c[i] = gf[i] * cp[chunk][i] + gi[i] * gg[i];
        h[i] = go[i] * cell_tanh(c[i]);
      }
      bf16* h1 = nullptr; bf16* h2 = nullptr;
      if (WHICH == 0) {                                // h1_t -> XE_t[:, Fp + j] and XA_{t+1}[:, j]
        h1 = p.XE + r * p.KX + p.Fp + j0;
        h2 = p.XA + (r + B) * 2 * p.Hp + j0;
      } else if (WHICH == 1) {                         // h_enc_t -> HE_{t+1}
        h1 = p.HE + (r + B) * p.Hp + j0;
      } else {                                         // h_dec_t -> XA_{t+1}[:, Hp + j] and XE_{t+1}[:, Fp + Hp + j]
        h1 = p.XA + (r + B) * 2 * p.Hp + p.Hp + j0;
        if (t + 1 < p.T) h2 = p.XE + (r + B) * p.KX + p.Fp + p.Hp + j0;
      }
#pragma unroll
      for (int v4 = 0; v4 < 2; ++v4) {
        if (v4 * 4 < nv) {
          const int o = v4 * 4;
          const size_t jq = (size_t)((j0 >> 2) + v4);
          float* gq = gbuf + (jq * 4 * B + b) * 4;     // lstm_tiled_gate_offset(B, b, k, j) = ((jq*4 + k)*B + b)*4
          *reinterpret_cast<float4*>(gq) = make_float4(gi[o], gi[o + 1], gi[o + 2], gi[o + 3]);
          *reinterpret_cast<float4*>(gq + (size_t)B * 4) = make_float4(gf[o], gf[o + 1], gf[o + 2], gf[o + 3]);
          *reinterpret_cast<float4*>(gq + (size_t)B * 8) = make_float4(gg[o], gg[o + 1], gg[o + 2], gg[o + 3]);
          *reinterpret_cast<float4*>(gq + (size_t)B * 12) = make_float4(go[o], go[o + 1], go[o + 2], go[o + 3]);
          *reinterpret_cast<float4*>(cbuf + (jq * B + b) * 4) = make_float4(c[o], c[o + 1], c[o + 2], c[o + 3]);
          st_bf16x4_rf(h1 + o, &h[o]);
          if (h2) st_bf16x4_rf(h2 + o, &h[o]);
        }
      }
    }
  }
  tc_fence_before();
}

// q_t = W_q h1_t (attention.py:69): plain fp32 tile store
__device__ __forceinline__ void epi_q(const RfParams& p, const RfSmem& sm, int t, int tile, uint32_t tmem_base, int cw, int lane, int rank) {
  const int qd = (cw + 2) & 3, half = cw >> 2;
  const int b = rank * 128 + qd * 32 + lane;
  const bool ok = b < p.B;
  const int hw = p.Nq >> 1;                            // columns per warp half (multiple of 8)
  const uint32_t taddr = tmem_base + (static_cast<uint32_t>(qd * 32) << 16) + TMEM_COL_Q;
  mbar_wait_bounded(p, &sm.tfull[SLOT_Q], (uint32_t)(t & 1), 13, t);
  tc_fence_after();
  RF_STAMP(cw == 0 && lane == 0, 8);
  float* qrow = p.q + ((size_t)t * p.B + b) * p.A;
#pragma unroll 1
  for (int c = half * hw; c < (half + 1) * hw; c += 8) {
    float v[8];
    tmem_ld_x8(taddr + c, v);
    tmem_ld_wait();
    const int n = tile * p.Nq + c;
    if (ok) {
      if (n + 8 <= p.A && (p.A & 3) == 0) {
        *reinterpret_cast<float4*>(qrow + n) = make_float4(v[0], v[1], v[2], v[3]);
        *reinterpret_cast<float4*>(qrow + n + 4) = make_float4(v[4], v[5], v[6], v[7]);
      } else {
#pragma unroll
        for (int i = 0; i < 8; ++i)
          if (n + i < p.A) qrow[n + i] = v[i];
      }
    }
  }
  tc_fence_before();
}

// mean / log_var heads, reparameterised sample and the per-step KL terms (updown_cell.py:196-208,
// updown_captioner.py:295-303) of 16 latent dimensions: accumulator columns [0,16) = mean, [16,32) = log_var.
// eps does not depend on the accumulator: it is drawn (or loaded) before waiting for it.
__device__ __forceinline__ void epi_latent(const RfParams& p, const RfSmem& sm, int t, int tile, uint32_t tmem_base, int cw, int lane,
                                           int rank) {
  const int qd = (cw + 2) & 3, half = cw >> 2;
  const int b = rank * 128 + qd * 32 + lane;
  const bool ok = b < p.B;
  const int Z = p.Z;
  const size_t r = (size_t)t * p.B + b;
  const int z0 = tile * 16 + half * 8;
  float e[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) e[i] = 0.f;
  if (ok) {
    if (p.eps_in) {
#pragma unroll
      for (int i = 0; i < 8; i += 2)
        if (z0 + i < Z) {                              // Z even, z0 even: pairs never straddle the end
          const float2 v = *reinterpret_cast<const float2*>(p.eps_in + r * Z + z0 + i);
          e[i] = v.x; e[i + 1] = v.y;
        }
    } else {
      const unsigned long long seed = *p.seed;
#pragma unroll 1
      for (int i = 0; i < 8; ++i)
        if (z0 + i < Z) e[i] = philox_normal_rf(seed, (unsigned long long)t, b, z0 + i, Z);
    }
  }
  // pin the draws in front of the wait (the compiler would otherwise sink the register-only Philox arithmetic to its first use)
#pragma unroll
  for (int i = 0; i < 8; ++i) asm volatile("" : "+f"(e[i]));
  const uint32_t taddr = tmem_base + (static_cast<uint32_t>(qd * 32) << 16) + TMEM_COL_FC;
  mbar_wait_bounded(p, &sm.tfull[SLOT_FC], (uint32_t)(t & 1), 14, t);
  tc_fence_after();
  RF_STAMP(cw == 0 && lane == 0, 9);
  float mu[8], lv[8];
  tmem_ld_x8(taddr + half * 8, mu);
  tmem_ld_x8(taddr + 16 + half * 8, lv);
  tmem_ld_wait();
  tc_fence_before();
  if (!ok) return;
  const float pm = p.pm_row ? p.pm_row[b] : 0.f;
  const float log_pv = logf(p.prior_var);
  float part = 0.f;
  float zz[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const int z = z0 + i;
    zz[i] = 0.f;
    if (z < Z) {
      mu[i] += p.b_fc[z];
      lv[i] += p.b_fc[Z + z];
      const float var = __expf(lv[i]);
      zz[i] = e[i] * sqrtf(var) + mu[i];
      if (p.sentiment_vae == 0) part += 1.f + lv[i] - mu[i] * mu[i] - var;
      else part += 1.f + lv[i] - log_pv - ((mu[i] - pm) * (mu[i] - pm) + var) / (p.prior_var + 0.00001f);
    }
  }
#pragma unroll
  for (int i = 0; i < 8; i += 2)
    if (z0 + i < Z) {
      *reinterpret_cast<float2*>(p.mean + r * Z + z0 + i) = make_float2(mu[i], mu[i + 1]);
      *reinterpret_cast<float2*>(p.logvar + r * Z + z0 + i) = make_float2(lv[i], lv[i + 1]);
      *reinterpret_cast<float2*>(p.eps_out + r * Z + z0 + i) = make_float2(e[i], e[i + 1]);
    }
  if (z0 < p.Zp) {
    bf16x8 o;
#pragma unroll
    for (int k = 0; k < 4; ++k) o.v[k] = __floats2bfloat162_rn(zz[2 * k], zz[2 * k + 1]);
    st_bf16x8(p.ZB + r * p.Zp + z0, o);
  }
  p.kl_part[((size_t)t * 2 * p.nfc + tile * 2 + half) * p.B + b] = part;
}

__device__ __forceinline__ RfSeg make_seg(int amap, int acol0, int wmap, int wcol0, int kblocks, int t_off, int flag, int mult, int toff) {
  RfSeg s;
  s.amap = amap; s.acol0 = acol0; s.wmap = wmap; s.wcol0 = wcol0; s.kblocks = kblocks; s.t_off = t_off;
  s.flag = flag; s.flag_mult = mult; s.flag_toff = toff;
  return s;
}

// the jobs of this pair, in issue order
__device__ void build_jobs(const RfParams& p, int pair, RfJob* jobs, int* njobs) {
  const int nt = p.nt, kbH = p.Hp >> 6, kbF = p.Fp >> 6, kbZ = p.Zp >> 6;
  const int n_rows = min((int)gridDim.x, p.B);         // CTAs that signal attention rows
  int n = 0;
  if (pair < nt) {
    RfJob& a = jobs[n++];                              // attention LSTM tile: emb_t W_e^T + [h1_{t-1} | h_dec_{t-1}] W_att_rec^T
    a.nseg = 3;                                        // teacher-forced embedding block first: it needs no flag
    a.seg[0] = make_seg(MAP_EMB, 0, WMAP_ATT_E, 0, p.Ep >> 6, 0, -1, 0, 0);
    a.seg[1] = make_seg(MAP_XA, 0, WMAP_ATT, 0, kbH, 0, FLAG_H1, 2, 0);
    a.seg[2] = make_seg(MAP_XA, p.Hp, WMAP_ATT, p.Hp, kbH, 0, FLAG_HDEC, 2, 0);
    a.w_row[0] = pair * 128; a.w_row[1] = pair * 128 + 64; a.w_box_rows = 64; a.N = 128;
    a.tmem_col = TMEM_COL_ATT; a.slot = SLOT_ATT;
    RfJob& e = jobs[n++];                              // encoder LSTM tile: h_enc_{t-1}, h_dec_{t-1}, h1_t, x_hat_t
    e.nseg = 4;
    e.seg[0] = make_seg(MAP_HE, 0, WMAP_ENC_HH, 0, kbH, 0, FLAG_HENC, 2, 0);
    e.seg[1] = make_seg(MAP_XE, p.Fp + p.Hp, WMAP_ENC_X, p.Fp + p.Hp, kbH, 0, FLAG_HDEC, 2, 0);
    e.seg[2] = make_seg(MAP_XE, p.Fp, WMAP_ENC_X, p.Fp, kbH, 0, FLAG_H1, 2, 1);
    e.seg[3] = make_seg(MAP_XE, 0, WMAP_ENC_X, 0, kbF, 0, FLAG_XHAT, n_rows, 1);
    e.w_row[0] = pair * 128; e.w_row[1] = pair * 128 + 64; e.w_box_rows = 64; e.N = 128;
    e.tmem_col = TMEM_COL_LSTM; e.slot = SLOT_LSTM;
  } else if (pair < 2 * nt) {
    const int tile = pair - nt;
    RfJob& d = jobs[n++];                              // decoder LSTM tile: h_dec_{t-1}, h1_t, x_hat_t, z_t
    d.nseg = 4;
    d.seg[0] = make_seg(MAP_XE, p.Fp + p.Hp, WMAP_DEC_X, p.Fp + p.Hp, kbH, 0, FLAG_HDEC, 2, 0);
    d.seg[1] = make_seg(MAP_XE, p.Fp, WMAP_DEC_X, p.Fp, kbH, 0, FLAG_H1, 2, 1);
    d.seg[2] = make_seg(MAP_XE, 0, WMAP_DEC_X, 0, kbF, 0, FLAG_XHAT, n_rows, 1);
    d.seg[3] = make_seg(MAP_ZB, 0, WMAP_DEC_Z, 0, kbZ, 0, FLAG_Z, 2 * p.nfc, 1);
    d.w_row[0] = tile * 128; d.w_row[1] = tile * 128 + 64; d.w_box_rows = 64; d.N = 128;
    d.tmem_col = TMEM_COL_LSTM; d.slot = SLOT_LSTM;
  } else {
    const int s = pair - 2 * nt;
    if (s < p.nq) {
      RfJob& q = jobs[n++];                            // query projection tile: h1_t W_q^T
      q.nseg = 1;
      q.seg[0] = make_seg(MAP_XE, p.Fp, WMAP_Q, 0, kbH, 0, FLAG_H1, 2, 1);
      q.w_row[0] = s * p.Nq; q.w_row[1] = s * p.Nq + (p.Nq >> 1); q.w_box_rows = p.Nq >> 1; q.N = p.Nq;
      q.tmem_col = TMEM_COL_Q; q.slot = SLOT_Q;
    }
    if (s < p.nfc) {
      RfJob& f = jobs[n++];                            // latent heads tile: h_enc_t [W_mean ; W_logvar]^T
      f.nseg = 1;
      f.seg[0] = make_seg(MAP_HE, 0, WMAP_FC, 0, kbH, 1, FLAG_HENC, 2, 1);
      f.w_row[0] = s * 16; f.w_row[1] = p.Z + s * 16; f.w_box_rows = 16; f.N = 32;
      f.tmem_col = TMEM_COL_FC; f.slot = SLOT_FC;
    }
  }
  *njobs = n;
}

}  // namespace

__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(PK_THREADS, 1)
recurrent_fwd_kernel(const __grid_constant__ RfParams p) {
  extern __shared__ __align__(1024) uint8_t rf_smem_raw[];
  if (threadIdx.x == 0 && (smem_u32(rf_smem_raw) & 1023u)) __trap();
  const AttnArgs a = p.att;
  const RfSmem sm = RfSmem::carve(rf_smem_raw, attn_smem_bytes(a, false));
  const AttnSmem asm_ = carve(sm.att, a, false);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int rank = (int)cluster_ctarank();
  const int pair = blockIdx.x >> 1;
  const int cta = blockIdx.x, G = gridDim.x;
  const int role = pair < p.nt ? ROLE_ENC : pair < 2 * p.nt ? ROLE_DEC : ROLE_SPARE;

  if (threadIdx.x == 0) {
    for (int i = 0; i < NUM_AMAPS; ++i) prefetch_tmap(&p.amap[i]);
    for (int i = 0; i < NUM_WMAPS; ++i) prefetch_tmap(&p.wmap[i]);
    sm.init_barriers();
    build_jobs(p, pair, sm.jobs, sm.njobs);
  }
  if (warp == 1) tmem_alloc_2sm<PK_TMEM_COLS>(sm.tmem_slot);
  attn_prologue(asm_, a, false);                       // attention ring barriers, w_a, zeroed q buffers; __syncthreads inside
  tc_fence_before();
  cluster_sync_all();                                  // the peer's barriers exist before any remote arrival
  tc_fence_after();
  const uint32_t tmem_base = *sm.tmem_slot;
  const int njobs = *sm.njobs;
  const int T = p.T;

  if (warp == 0) {
    // ================= TMA producer of the GEMM operand ring (both CTAs of the pair) =================
    if (elect_one_sync()) {
      RingPos<RF_STAGES> pos;
      const uint64_t w_pol = ptx::l2_policy_evict_first();
      for (int t = 0; t < T; ++t) {
        for (int j = 0; j < njobs; ++j) {
          const RfJob& job = sm.jobs[j];
          const uint32_t tx = 2u * (uint32_t)(PK_X_BYTES + job.w_box_rows * 128);
          for (int s = 0; s < job.nseg; ++s) {
            const RfSeg sg = job.seg[s];
            produce_segment(p, sm, pos, t, rank, tx, w_pol, &p.amap[sg.amap], sg.acol0, t + sg.t_off, &p.wmap[sg.wmap], sg.wcol0,
                            job.w_row[rank], sg.kblocks, [&] {
              const bool hidden = sg.flag == FLAG_H1 || sg.flag == FLAG_HDEC || sg.flag == FLAG_HENC;
              const unsigned int target = sg.flag >= 0 ? (unsigned int)((t + sg.flag_toff) * sg.flag_mult * (hidden ? p.nt : 1)) : 0u;
              if (target) {
                wait_flag(p, sg.flag, target, 100 + j * 10 + s, t);
                fence_proxy_async_global();
              }
              RF_STAMP(true, 10 + j * 4 + s);
            });
          }
        }
      }
    }
    __syncwarp();
  } else if (warp == 1) {
    // ================= MMA issuer (leader CTA of the pair) =================
    if (rank == 0 && elect_one_sync()) {
      RingPos<RF_STAGES> pos;
      for (int t = 0; t < T; ++t) {
        for (int j = 0; j < njobs; ++j) {
          const RfJob& job = sm.jobs[j];
          mma_job(p, sm, pos, t, job, tmem_base + job.tmem_col, job.slot);
          RF_STAMP(true, 20 + j);
        }
      }
    }
    __syncwarp();
  } else if (warp < 2 + PK_CWARPS) {
    // ================= compute warps: epilogues + attention consumers =================
    const int cw = warp - 2;
    const int ctid = (int)threadIdx.x - 64;
    Ring ring;
    const int s_idx = pair - 2 * p.nt;
    const bool has_q = role == ROLE_SPARE && s_idx < p.nq;
    const bool has_fc = role == ROLE_SPARE && s_idx < p.nfc;
    const int tile = role == ROLE_ENC ? pair : role == ROLE_DEC ? pair - p.nt : s_idx;
    if (role == ROLE_ENC) {
      init_lstm_const<0>(p, tile, tmem_base, cw, lane, rank);
      init_lstm_const<1>(p, tile, tmem_base, cw, lane, rank);
    } else if (role == ROLE_DEC) {
      init_lstm_const<2>(p, tile, tmem_base, cw, lane, rank);
    }
    tc_fence_before();
    // the rows of this CTA are the same at every step (b = cta, cta + G): with at most two of them their box masks stay
    // in the two mask buffers of the attention for the whole kernel
    const bool mask_resident = cta + 2 * G >= p.B;
    if (mask_resident) {
      for (int k = 0; k < 2; ++k) {
        const int b = cta + k * G;
        if (b < p.B && ctid < a.N) asm_.msk(k)[ctid] = a.mask[(size_t)b * a.N + ctid];
      }
      ptx::bar_sync(1, PK_CTHREADS);
    }
    for (int t = 0; t < T; ++t) {
      RF_STAMP(ctid == 0, 0);
      if (role == ROLE_ENC) {
        epi_lstm<0>(p, sm, t, tile, tmem_base, cw, lane, rank);
        RF_STAMP(ctid == 0, 1);
        signal_done(p, FLAG_H1, ctid);
      } else if (has_q) {
        epi_q(p, sm, t, tile, tmem_base, cw, lane, rank);
        RF_STAMP(ctid == 0, 1);
        signal_done(p, FLAG_Q, ctid);
      }
      // ---- region attention of this CTA's rows (attention.py:69-93, updown_cell.py:156)
      if (cta < p.B) {
        if (ctid == 0) wait_flag(p, FLAG_Q, (unsigned int)((t + 1) * 2 * p.nq), 20, t);
        RF_STAMP(ctid == 0, 3);
        ptx::bar_sync(1, PK_CTHREADS);
        const float* q_t = p.q + (size_t)t * p.B * p.A;
        prefetch_vec(asm_.q(0), q_t + (size_t)cta * p.A, a.A);
        ptx::cp_async_commit();
        int cur = 0;
        for (int b = cta; b < p.B; b += G, cur ^= 1) {
          const size_t r = (size_t)t * p.B + b;
          attn_fwd_row(a, p.plan, asm_, ring, cur, mask_resident ? nullptr : a.mask + (size_t)b * a.N, b + G < p.B ? q_t + (size_t)(b + G) * p.A : nullptr,
                       p.alpha + r * a.N, p.smx + r * a.N, p.XE + r * p.KX);
        }
        RF_STAMP(ctid == 0, 4);
        signal_done(p, FLAG_XHAT, ctid);
      }
      RF_STAMP(ctid == 0, 5);
      if (role == ROLE_ENC) {
        epi_lstm<1>(p, sm, t, tile, tmem_base, cw, lane, rank);
        RF_STAMP(ctid == 0, 6);
        signal_done(p, FLAG_HENC, ctid);
      } else if (role == ROLE_DEC) {
        epi_lstm<2>(p, sm, t, tile, tmem_base, cw, lane, rank);
        RF_STAMP(ctid == 0, 6);
        signal_done(p, FLAG_HDEC, ctid);
      } else if (has_fc) {
        epi_latent(p, sm, t, tile, tmem_base, cw, lane, rank);
        RF_STAMP(ctid == 0, 6);
        signal_done(p, FLAG_Z, ctid);
      }
      RF_STAMP(ctid == 0, 7);
    }
  } else {
    // ================= attention producer: streams P and the region features of this CTA's rows =================
    if (lane == 0 && cta < p.B) {
      Ring ring;
      const uint64_t pol = ptx::l2_policy_evict_first();
      for (int t = 0; t < T; ++t)
        for (int b = cta; b < p.B; b += G) {
          produce_block(asm_, ring, reinterpret_cast<const uint8_t*>(a.proj + (size_t)b * a.N * a.Ap), a.N, a.Ap * 2, p.plan.nP, p.plan.bP, pol);
          produce_block(asm_, ring, reinterpret_cast<const uint8_t*>(a.feats + (size_t)b * a.N * a.Fp), a.N, a.Fp * 2, p.plan.nF, p.plan.bF, pol);
        }
    }
    __syncwarp();
  }
  pk_teardown(warp, tmem_base);
}

// kl[t*B + b] = -1/2 * sum of the per-tile partial sums (updown_captioner.py:299-303)
__global__ void kl_sum_parts_kernel(const float* __restrict__ parts, int nparts, int B, int TB, float* __restrict__ kl) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= TB) return;
  const int t = i / B, b = i - t * B;
  float s = 0.f;
  for (int k = 0; k < nparts; ++k) s += parts[((size_t)t * nparts + k) * B + b];
  kl[i] = -0.5f * s;
}

// host side
static size_t rf_smem_bytes(const AttnArgs& a) { return RfSmem::bytes(attn_smem_bytes(a, false), 2); }

size_t recurrent_forward_kl_parts(int Z) { return 2 * (size_t)((Z + 15) / 16); }

bool recurrent_forward_supported(const RecFwdArgs& r) {
  static const bool off = [] { const char* e = getenv("SSCVAE_PERSISTENT"); return e && e[0] == '0'; }();
  if (off) return false;
  if (r.B > 256 || r.B < 1 || (r.H & 3) || r.GP % 128 || (r.Hp & 63) || (r.Fp & 63) || (r.Zp & 63) || (r.Ep & 63) || (r.Z & 1)) return false;
  AttnArgs a = r.att;
  if (a.N > 32 * ATT_NREG || a.Fp > 8 * ATT_CONSUMERS * ATT_FV || a.Ap * 2 > ATT_STAGE_BYTES || a.Fp * 2 > ATT_STAGE_BYTES ||
      (a.Ap % 8) || (a.Fp % 8))
    return false;
  const size_t smem = rf_smem_bytes(a);
  if (smem > 227 * 1024) return false;
  const int NP = pk_grid_pairs(recurrent_fwd_kernel, smem);
  const int nt = r.GP / 128, spare = NP - 2 * nt;
  if (spare < 1) return false;
  const int nfc = (r.Z + 15) / 16;
  const int Nq = round_up(ceil_div(r.A, spare), 16);
  if (nfc > spare || Nq > 128 || nfc * 16 > r.Zp) return false;
  return true;
}

int recurrent_forward(cudaStream_t s, const RecFwdArgs& r) {
  RfParams p;
  memset(&p, 0, sizeof(p));
  const AttnArgs& a = r.att;
  const size_t smem = rf_smem_bytes(a);
  const int NP = pk_grid_pairs(recurrent_fwd_kernel, smem);
  REQUIRE(NP > 0, "recurrent_fwd: no co-resident CTA pairs");
  const int nt = r.GP / 128, spare = NP - 2 * nt;
  p.B = r.B; p.T = r.T; p.H = r.H; p.Hp = r.Hp; p.Fp = r.Fp; p.Zp = r.Zp; p.Z = r.Z; p.A = r.A; p.KX = r.KX; p.GP = r.GP;
  p.Ep = r.Ep;
  p.nt = nt;
  p.Nq = round_up(ceil_div(r.A, spare), 16);
  p.nq = ceil_div(r.A, p.Nq);
  p.nfc = (r.Z + 15) / 16;
  p.sentiment_vae = r.sentiment_vae; p.prior_var = r.prior_var;
  TRY(encode_act3d(&p.amap[MAP_XA], r.XA, 2 * r.Hp, r.B, r.T + 1, 2 * r.Hp));
  TRY(encode_act3d(&p.amap[MAP_XE], r.XE, r.KX, r.B, r.T, r.KX));
  TRY(encode_act3d(&p.amap[MAP_HE], r.HE, r.Hp, r.B, r.T + 1, r.Hp));
  TRY(encode_act3d(&p.amap[MAP_ZB], r.ZB, r.Zp, r.B, r.T, r.Zp));
  TRY(encode_act3d(&p.amap[MAP_EMB], r.embb_t, r.Ep, r.B, r.T, r.Ep));
  TRY(encode_w2d(&p.wmap[WMAP_ATT], r.w_att_rec, 2 * r.Hp, r.GP, 2 * r.Hp, 64));
  TRY(encode_w2d(&p.wmap[WMAP_Q], r.wq, r.Hp, r.A, r.Hp, p.Nq / 2));
  TRY(encode_w2d(&p.wmap[WMAP_ENC_X], r.w_enc_x, r.KX, r.GP, r.KX, 64));
  TRY(encode_w2d(&p.wmap[WMAP_ENC_HH], r.w_enc_hh, r.Hp, r.GP, r.Hp, 64));
  TRY(encode_w2d(&p.wmap[WMAP_FC], r.w_fc, r.Hp, 2 * r.Z, r.Hp, 16));
  TRY(encode_w2d(&p.wmap[WMAP_DEC_X], r.w_dec_x, r.KX, r.GP, r.KX, 64));
  TRY(encode_w2d(&p.wmap[WMAP_DEC_Z], r.w_dec_z, r.Zp, r.GP, r.Zp, 64));
  TRY(encode_w2d(&p.wmap[WMAP_ATT_E], r.w_att_e, r.Ep, r.GP, r.Ep, 64));
  p.gavg = r.gavg; p.b_att = r.b_att; p.b_enc = r.b_enc; p.b_dec = r.b_dec;
  p.sent = r.sent; p.scol_enc = r.scol_enc; p.scol_dec = r.scol_dec;
  p.c1 = r.c1; p.c_enc = r.c_enc; p.c_dec = r.c_dec;
  p.gates_att = r.gates_att; p.gates_enc = r.gates_enc; p.gates_dec = r.gates_dec;
  p.XA = r.XA; p.XE = r.XE; p.HE = r.HE; p.ZB = r.ZB;
  p.q = r.q; p.b_fc = r.b_fc; p.eps_in = r.eps_in; p.seed = r.seed; p.pm_row = r.pm_row;
  p.mean = r.mean; p.logvar = r.logvar; p.eps_out = r.eps_out; p.kl_part = r.kl_part;
  p.att = a; p.alpha = r.alpha; p.smx = r.smx;
  p.flags = r.flags;
  p.timeout_ns = pk_timeout_ns();
  p.plan = attn_chunk_plan(a);
  // model FLOPs of the loop (un-hoisted parts only): the three gate GEMMs, q, fc; bytes: the attention stream
  const double flops = 2.0 * r.B * r.T * ((double)r.GP * (r.Ep + 2 * r.Hp + r.KX + r.Hp + r.KX + r.Zp) + (double)r.A * r.Hp + 2.0 * r.Z * r.Hp);
  PROF_SCOPE(s, "recurrent_fwd", flops, (double)r.B * r.T * a.N * (a.Ap + a.Fp) * 2.0);
  static const bool dbg = [] { const char* e = getenv("SSCVAE_RF_DBG"); return e && e[0] == '1'; }();
  if (dbg) {
    TRY(pk_dbg_begin(s, &p.dbg));
    p.dbg_t = r.T / 2;
  }
  CUDA_TRY(cudaMemsetAsync(r.flags, 0, FLAG_COUNT * sizeof(unsigned int), s));
  TRY(pk_launch(recurrent_fwd_kernel, NP, smem, s, p));
  if (dbg) {
    char head[64];
    snprintf(head, sizeof(head), "[rfdbg] B=%d t=%d", r.B, p.dbg_t);
    TRY(pk_dbg_print(s, p.dbg, 2 * NP, head, {0, 1, 2 * nt - 2, 2 * nt, 4 * nt - 2, 4 * nt, 4 * nt + 2 * p.nfc, 2 * NP - 2}, 24));
  }
  const int TB = r.T * r.B;
  kl_sum_parts_kernel<<<ceil_div(TB, 256), 256, 0, s>>>(r.kl_part, 2 * p.nfc, r.B, TB, r.kl);
  CUDA_TRY(cudaGetLastError());
  ++g_launch_count;
  return 0;
}

}  // namespace sscvae

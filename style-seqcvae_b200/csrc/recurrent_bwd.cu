// Persistent kernel of the backward-through-time loop (north_star kernel #4): ONE cooperative launch runs all T reverse
// timesteps of the UpDown cell's backward (the autograd graph of var_updown/var_updown/modules/updown_cell.py:123-231):
//   cell_dec -> d z -> latent heads -> cell_enc -> d[x_hat | h1 | h_dec_{t-1} | h_enc_{t-1}] -> region attention backward ->
//   query projection -> cell_att -> d[h1_{t-1} | h_dec_{t-1}]
// which the per-launch path (api_train.cu) runs as ten kernels per step. Same engine as recurrent_fwd.cu (persistent.cuh):
// one CTA per SM in CTA pairs, tcgen05.mma.cta_group::2 with M = 256 = the whole batch, TMA-fed operand ring, accumulators
// in TMEM, dataflow through monotonic global counters instead of grid barriers, bounded waits.
//
// Decomposition. The data-gradient GEMMs have a long K (the 4H gate gradients, 57 k-blocks at H = 900) and few output
// columns, so they are split over K: every (tile, K part) is a job of one pair, and its epilogue stores the partial
// tile into slot `part` of the destination; the consumers add the slots. All fp32 intermediates use the row-tiled
// layout (4 consecutive columns of a row are 16 contiguous bytes, consecutive rows follow each other), so an epilogue
// warp whose lanes are 32 batch rows stores 512 contiguous bytes per instruction.
//   "big" pairs:   S6A  d[x_hat|h1|h_dec_{t-1}] = dG_dec W_dec_x + dG_enc W_enc_x   (N = 128 tiles x splitA; the decoder half is
//                       accumulated while the latent chain of the step is still running)
//                  S6B  d h_enc_{t-1} = dG_enc W_enc_hh                               (N = 64 x splitB; not needed before step t-1,
//                       runs behind the attention of step t, under the query GEMM and the attention-LSTM cell)
//                  S10  d[h1_{t-1}|h_dec_{t-1}] = dG_att W_att_rec                    (N = 128 x splitX)
//   "small" pairs: S2   d z = dG_dec W_dec_z                                          (N = 96 x splitZ)
//                  S4   d h_enc (latent heads) = d[mean|log_var] W_fc                 (N = N4 tiles, K = 2Z)
//                  S8   d h1 (query) = d q W_q                                        (N = N4 tiles, K = A)
// The pointwise stages (the three LSTM cell backwards, the latent backward) and the attention rows are spread over the
// compute warps of ALL CTAs; the attention walks the per-step list of rows that still carry gradient (rb_active_rows_kernel).
// The saved gates / cell states are read in the row-tiled layout of the persistent forward kernel or in the row-major
// layout of the per-launch forward (RbParams::tiled).
#define PK_NAME "recurrent_bwd"
#include "persistent.cuh"

namespace sscvae {

namespace {

constexpr int RB_STAGES = 5;
constexpr int RB_MAX_JOBS = 3;

enum { F_DGDEC = 0, F_DZP, F_DML, F_DHE, F_DGENC, F_DXEA, F_DQ, F_DXEB, F_DH1Q, F_DGATT, F_DXA, F_ABORT, F_COUNT };
enum { AM_DGDEC = 0, AM_DGENC, AM_DGATT, AM_DML, AM_DQ, NUM_AMAPS };
enum { WM_DECX = 0, WM_DECZ, WM_ENCX, WM_ENCH, WM_ATT, WM_FC, WM_Q, NUM_WMAPS };
enum { K_S6A = 0, K_S6B, K_S10, K_S2, K_S4, K_S8, NUM_KINDS };
// accumulator slot (TMEM column block + "accumulator ready" barrier) of a job kind: three per pair
__device__ __forceinline__ int kind_slot(int kind) { return kind % 3; }
constexpr int RB_SLOTS = 3;
constexpr int RB_TMEM_STRIDE = 128;

struct RbSeg {
  int amap, wmap;          // activation / weight tensor map
  int k0;                  // first K column (elements) of both operands
  int kblocks;
  int flag, count;         // the counter must reach (s + 1) * count before the segment is loaded
};
struct RbJob {
  int kind;
  int nseg;
  RbSeg seg[2];
  int w_row[2];            // first weight row loaded by CTA 0 / CTA 1 of the pair
  int w_box_rows;          // rows per CTA (= N / 2)
  int N;                   // UMMA N
  float* dst;              // slot base of the destination (row-tiled fp32, B rows)
  int dcol0, dlimit;       // destination column of tile column 0; columns >= dlimit are dropped
  int sig;                 // counter bumped after the epilogue
};

struct RbParams {
  CUtensorMap amap[NUM_AMAPS];     // 3-D (k, batch row, t), box 64 x 128 x 1, 128B swizzle
  CUtensorMap wmap[NUM_WMAPS];     // 2-D (k, weight row), box 64 x w_box_rows
  int B, T, H, Hp, Fp, Zp, Z, Z2p, A, Ap, KX, G, Gp, N;
  int sentiment_vae;
  float prior_var;
  int tiled;                       // saved gates / cell states: 1 row-tiled (persistent forward), 0 row-major (per-launch forward)
  // tiling
  int nbig, nsmall;
  int nA, splitA, nB, splitB, nX, splitX, nZt, splitZ, n4, N4;
  int cnt[F_COUNT];                // signals per step of every counter
  // saved forward state (row-tiled blocks per timestep)
  const float* gates_att; const float* gates_enc; const float* gates_dec;
  const float* c1; const float* c_enc; const float* c_dec;
  const float* mean; const float* logvar; const float* eps; const float* pm_row;
  const float* q; const float* smx;
  const float* dhead;              // (T*B, H) row-major: d h_dec_t from the output head
  const float* gkld; const float* tmask;
  const int* rows; const int* nrows;   // rows[t*B + i] = i-th batch row that still carries gradient at step t; nrows[t] of them
  // carried cell-state gradients (row-tiled, B x H, zero at entry)
  float* dc1; float* dc_enc; float* dc_dec;
  // outputs kept for the weight-gradient GEMMs
  bf16* dG_att; bf16* dG_enc; bf16* dG_dec; bf16* dml; bf16* dqb; float* du;
  // split-K slots and small intermediates (row-tiled)
  float* dXEA; float* dXEB; float* dXA; float* dzp; float* dhe_fc; float* dh1q;
  AttnArgs att; AttnPlan plan;
  unsigned int* flags;
  static constexpr int ABORT_FLAG = F_ABORT;
  unsigned long long timeout_ns;
  unsigned long long* dbg;         // SSCVAE_RB_DBG=1: globaltimer stamps of step dbg_s, 32 per CTA
  int dbg_s;
};

#define RB_STAMP(cond, i)                                                                   \
  do {                                                                                     \
    if (p.dbg && s == p.dbg_s && (cond)) p.dbg[(size_t)blockIdx.x * 32 + (i)] = globaltimer_ns(); \
  } while (0)

using RbSmem = PkSmem<RbJob, RB_STAGES, RB_SLOTS>;

// row-tiled fp32 matrix with B rows: element (b, col)
__device__ __forceinline__ size_t tl_off(int B, int b, int col) { return ((size_t)(col >> 2) * B + b) * 4 + (col & 3); }
__device__ __forceinline__ float4 ld4g(const float* p) { return *reinterpret_cast<const float4*>(p); }
__device__ __forceinline__ void prefetch_l2(const void* p) { asm volatile("prefetch.global.L2 [%0];" ::"l"(p)); }
__device__ __forceinline__ void add4(float4& a, const float4& b) { a.x += b.x; a.y += b.y; a.z += b.z; a.w += b.w; }
__device__ __forceinline__ void st_bf16x4_rb(bf16* p, float a, float b, float c, float d) {
  __nv_bfloat162 lo = __floats2bfloat162_rn(a, b), hi = __floats2bfloat162_rn(c, d);
  uint2 o;
  o.x = *reinterpret_cast<uint32_t*>(&lo);
  o.y = *reinterpret_cast<uint32_t*>(&hi);
  *reinterpret_cast<uint2*>(p) = o;
}

__device__ __forceinline__ void wait_all(const RbParams& p, int flag, unsigned int target, int code, int s, int ctid) {
  if (ctid == 0 && target) wait_flag(p, flag, target, code, s);
  ptx::bar_sync(1, PK_CTHREADS);
}

// ---- pointwise stages (all CTAs) ---------------------------------------------------------------------------------
// LSTM cell backward (torch.nn.LSTMCell, gate order i,f,g,o; the math of pointwise.cu: lstm_bwd_v4_kernel) of timestep t.
// WHICH: 0 attention LSTM, 1 encoder, 2 decoder. A warp covers 8 rows x 4 unit-quads.
// Inputs of one cell item (a lane = one row x 4 units) that do NOT depend on a dataflow counter: the saved gates and
// cell states, this thread's own carried d c, and (decoder) the head gradient.
struct CellPre { float4 gi, gf, gg, go, c, cp, dci, dh0; int r, j; bool ok; };

template <int WHICH>
__device__ __forceinline__ void cell_preload(const RbParams& p, int t, int wi, int lane, CellPre& in) {
  const int B = p.B, H = p.H, H4 = H >> 2;
  const int tr = (B + 7) >> 3, tq = (H4 + 3) >> 2;
  const int r = (wi % tr) * 8 + (lane & 7);
  const int jq = (wi / tr) * 4 + (lane >> 3);
  in.ok = wi < tr * tq && r < B && jq < H4;
  in.r = r; in.j = jq * 4;
  if (!in.ok) return;
  const int j = in.j;
  const float* gates = (WHICH == 0 ? p.gates_att : WHICH == 1 ? p.gates_enc : p.gates_dec) + (size_t)t * B * 4 * H;
  const float* cbuf = (WHICH == 0 ? p.c1 : WHICH == 1 ? p.c_enc : p.c_dec) + (size_t)t * B * H;
  const float* dcb = WHICH == 0 ? p.dc1 : WHICH == 1 ? p.dc_enc : p.dc_dec;
  const float* g = gates + (p.tiled ? lstm_tiled_gate_offset(B, r, 0, j) : (size_t)r * 4 * H + j);
  const size_t gs = p.tiled ? (size_t)B * 4 : (size_t)H;
  const size_t co = p.tiled ? lstm_tiled_c_offset(B, r, j) : (size_t)r * H + j;
  in.gi = ld4g(g); in.gf = ld4g(g + gs); in.gg = ld4g(g + 2 * gs); in.go = ld4g(g + 3 * gs);
  in.c = ld4g(cbuf + co);
  in.cp = make_float4(0.f, 0.f, 0.f, 0.f);
  if (t > 0) in.cp = ld4g(cbuf - (size_t)B * H + co);
  in.dci = ld4g(dcb + tl_off(B, r, j));
  in.dh0 = make_float4(0.f, 0.f, 0.f, 0.f);
  if (WHICH == 2) in.dh0 = ld4g(p.dhead + ((size_t)t * B + r) * H + j);
}

// The counter-dependent part: sum of the split-K slots that feed d h of this cell, then the LSTM cell backward
// (torch.nn.LSTMCell, gate order i,f,g,o; the math of pointwise.cu: lstm_bwd_v4_kernel).
template <int WHICH>
__device__ __forceinline__ void cell_finish(const RbParams& p, int t, bool prev, const CellPre& in) {
  if (!in.ok) return;
  const int B = p.B, H = p.H, r = in.r, j = in.j;
  // all slot loads are issued before the first add (a runtime-trip-count loop of load + add serialises the L2 round trips)
  const float4 z4 = make_float4(0.f, 0.f, 0.f, 0.f);
  float4 va[RB_MAX_SPLIT_A], vx[RB_MAX_SPLIT_X], v0 = z4;
  if (WHICH == 2) {                                    // d h_dec_t: output head + LSTM inputs of step t+1 (S6A, S10)
#pragma unroll
    for (int k = 0; k < RB_MAX_SPLIT_A; ++k) va[k] = (prev && k < p.splitA) ? ld4g(p.dXEA + (size_t)k * B * p.KX + tl_off(B, r, p.Fp + p.Hp + j)) : z4;
#pragma unroll
    for (int k = 0; k < RB_MAX_SPLIT_X; ++k) vx[k] = (prev && k < p.splitX) ? ld4g(p.dXA + (size_t)k * B * 2 * p.Hp + tl_off(B, r, p.Hp + j)) : z4;
  } else if (WHICH == 1) {                             // d h_enc_t: latent heads + recurrence (S6B of step t+1)
    v0 = ld4g(p.dhe_fc + tl_off(B, r, j));
#pragma unroll
    for (int k = 0; k < RB_MAX_SPLIT_A; ++k) va[k] = z4;
#pragma unroll
    for (int k = 0; k < RB_MAX_SPLIT_B; ++k) vx[k] = (prev && k < p.splitB) ? ld4g(p.dXEB + (size_t)k * B * p.Hp + tl_off(B, r, j)) : z4;
  } else {                                             // d h1_t: enc/dec inputs of this step + query + recurrence (S10 of t+1)
    v0 = ld4g(p.dh1q + tl_off(B, r, j));
#pragma unroll
    for (int k = 0; k < RB_MAX_SPLIT_A; ++k) va[k] = (k < p.splitA) ? ld4g(p.dXEA + (size_t)k * B * p.KX + tl_off(B, r, p.Fp + j)) : z4;
#pragma unroll
    for (int k = 0; k < RB_MAX_SPLIT_X; ++k) vx[k] = (prev && k < p.splitX) ? ld4g(p.dXA + (size_t)k * B * 2 * p.Hp + tl_off(B, r, j)) : z4;
  }
  float4 dh = in.dh0;
  add4(dh, v0);
#pragma unroll
  for (int k = 0; k < RB_MAX_SPLIT_A; ++k) add4(dh, va[k]);
#pragma unroll
  for (int k = 0; k < RB_MAX_SPLIT_X; ++k) add4(dh, vx[k]);
  const float4 gi = in.gi, gf = in.gf, gg = in.gg, go = in.go, c = in.c, cp = in.cp, dci = in.dci;
  float4 di, df, dg, d_o, dcp;
#define RB_LSTM_LANE(X)                                                                  \
  {                                                                                      \
    const float tc = tanhf(c.X);                                                         \
    const float dc = dh.X * go.X * (1.f - tc * tc) + dci.X;                              \
    di.X = dc * gg.X * gi.X * (1.f - gi.X);                                              \
    df.X = dc * cp.X * gf.X * (1.f - gf.X);                                              \
    dg.X = dc * gi.X * (1.f - gg.X * gg.X);                                              \
    d_o.X = dh.X * tc * go.X * (1.f - go.X);                                             \
    dcp.X = dc * gf.X;                                                                   \
  }
  RB_LSTM_LANE(x) RB_LSTM_LANE(y) RB_LSTM_LANE(z) RB_LSTM_LANE(w)
#undef RB_LSTM_LANE
  float* dcb = WHICH == 0 ? p.dc1 : WHICH == 1 ? p.dc_enc : p.dc_dec;
  bf16* o = (WHICH == 0 ? p.dG_att : WHICH == 1 ? p.dG_enc : p.dG_dec) + ((size_t)t * B + r) * p.Gp + j;
  st_bf16x4_rb(o, di.x, di.y, di.z, di.w);
  st_bf16x4_rb(o + H, df.x, df.y, df.z, df.w);
  st_bf16x4_rb(o + 2 * H, dg.x, dg.y, dg.z, dg.w);
  st_bf16x4_rb(o + 3 * H, d_o.x, d_o.y, d_o.z, d_o.w);
  *reinterpret_cast<float4*>(dcb + tl_off(B, r, j)) = dcp;
}

// Cell stage of timestep t (WHICH: 0 attention LSTM, 1 encoder, 2 decoder). A warp item covers 8 rows x 4 unit-quads and
// the item -> warp map is the same at every step. The stage is split around the wait for the counters its slot sums
// depend on: the saved state of the warp's first item is loaded BEFORE the wait (cell_stage_pre), so that after it only
// one L2 round trip (the slots) separates the warp from its stores (two such items per thread spill registers).
template <int WHICH>
__device__ __forceinline__ void cell_stage_pre(const RbParams& p, int t, int gw, int GW, int lane, CellPre& pre) {
  cell_preload<WHICH>(p, t, gw, lane, pre);
}
template <int WHICH>
__device__ __forceinline__ void cell_stage_post(const RbParams& p, int t, int s, int gw, int GW, int lane, const CellPre& pre) {
  const int B = p.B, H4 = p.H >> 2;
  const int total = ((B + 7) >> 3) * ((H4 + 3) >> 2);
  const bool prev = s > 0;                             // contributions of step t + 1 exist
  cell_finish<WHICH>(p, t, prev, pre);
  for (int wi = gw + GW; wi < total; wi += GW) {       // further items of this warp
    CellPre x;
    cell_preload<WHICH>(p, t, wi, lane, x);
    cell_finish<WHICH>(p, t, prev, x);
  }
}

// The saved state a cell stage reads was written milliseconds earlier (forward pass, head backward): pull the lines of
// timestep t (the NEXT step of this loop) into L2 while the current step's GEMMs run.
template <int WHICH>
__device__ __forceinline__ void cell_prefetch(const RbParams& p, int t, int gw, int GW, int lane) {
  if (t < 0) return;
  const int B = p.B, H = p.H, H4 = H >> 2;
  const int tr = (B + 7) >> 3, tq = (H4 + 3) >> 2;
  const float* gates = (WHICH == 0 ? p.gates_att : WHICH == 1 ? p.gates_enc : p.gates_dec) + (size_t)t * B * 4 * H;
  const float* cbuf = (WHICH == 0 ? p.c1 : WHICH == 1 ? p.c_enc : p.c_dec) + (size_t)t * B * H;
  for (int wi = gw; wi < tr * tq; wi += GW) {
    const int r = (wi % tr) * 8 + (lane & 7);
    const int jq = (wi / tr) * 4 + (lane >> 3);
    if (r >= B || jq >= H4) continue;
    const int j = jq * 4;
    const float* g = gates + (p.tiled ? lstm_tiled_gate_offset(B, r, 0, j) : (size_t)r * 4 * H + j);
    const size_t gs = p.tiled ? (size_t)B * 4 : (size_t)H;
    const size_t co = p.tiled ? lstm_tiled_c_offset(B, r, j) : (size_t)r * H + j;
    // tiled: 8 consecutive rows share a 128-byte line (lanes 0..7 of a quad): one prefetch per line
    if (!p.tiled || (lane & 7) == 0) {
      prefetch_l2(g); prefetch_l2(g + gs); prefetch_l2(g + 2 * gs); prefetch_l2(g + 3 * gs);
      if (t > 0) prefetch_l2(cbuf - (size_t)B * H + co);
    }
    if (WHICH == 2 && (lane >> 3) == 0) prefetch_l2(p.dhead + ((size_t)t * B + r) * H + j);   // 4 quads = 64 B of a row
  }
}

// d[mean | log_var] of timestep t from d z (sum of the S2 slots) and the KL gradient (pointwise.cu: latent_bwd_kernel;
// updown_cell.py:196-208, updown_captioner.py:295-303). A thread = one row x 4 latent dimensions.
__device__ __forceinline__ void latent_stage(const RbParams& p, int t, int gtid, int GT) {
  const int B = p.B, Z = p.Z, ZQ = (Z + 3) >> 2;
  const float inv_pv = 1.0f / (p.prior_var + 0.00001f);
  for (int idx = gtid; idx < B * ZQ; idx += GT) {
    const int r = idx % B, zq = idx / B;
    const size_t row = (size_t)t * B + r;
    // every load first (Z is even and z0 a multiple of 4: 8-byte aligned pairs)
    float4 gs[RB_MAX_SPLIT_Z];
#pragma unroll
    for (int k = 0; k < RB_MAX_SPLIT_Z; ++k)
      gs[k] = k < p.splitZ ? ld4g(p.dzp + (size_t)k * B * p.Zp + tl_off(B, r, zq * 4)) : make_float4(0.f, 0.f, 0.f, 0.f);
    const int z0 = zq * 4;
    const bool hi = z0 + 2 < Z;
    const float2 zero2 = make_float2(0.f, 0.f);
    const float2 mu0 = *reinterpret_cast<const float2*>(p.mean + row * Z + z0);
    const float2 lv0 = *reinterpret_cast<const float2*>(p.logvar + row * Z + z0);
    const float2 ep0 = *reinterpret_cast<const float2*>(p.eps + row * Z + z0);
    const float2 mu1 = hi ? *reinterpret_cast<const float2*>(p.mean + row * Z + z0 + 2) : zero2;
    const float2 lv1 = hi ? *reinterpret_cast<const float2*>(p.logvar + row * Z + z0 + 2) : zero2;
    const float2 ep1 = hi ? *reinterpret_cast<const float2*>(p.eps + row * Z + z0 + 2) : zero2;
    const float w = p.gkld[r] * p.tmask[row];
    const float pm = p.pm_row ? p.pm_row[r] : 0.f;
    float4 g4 = gs[0];
#pragma unroll
    for (int k = 1; k < RB_MAX_SPLIT_Z; ++k) add4(g4, gs[k]);
    const float gz[4] = {g4.x, g4.y, g4.z, g4.w};
    const float mu[4] = {mu0.x, mu0.y, mu1.x, mu1.y}, lv[4] = {lv0.x, lv0.y, lv1.x, lv1.y}, ep[4] = {ep0.x, ep0.y, ep1.x, ep1.y};
    bf16* out = p.dml + row * p.Z2p;
#pragma unroll
    for (int i = 0; i < 4; i += 2) {
      const int z = z0 + i;
      if (z < Z) {
        float om[2], ol[2];
#pragma unroll
        for (int u = 0; u < 2; ++u) {
          const float var = __expf(lv[i + u]);
          const float dkl_m = (p.sentiment_vae == 0) ? mu[i + u] : (mu[i + u] - pm) * inv_pv;
          const float dkl_l = (p.sentiment_vae == 0) ? -0.5f * (1.f - var) : -0.5f * (1.f - var * inv_pv);
          om[u] = gz[i + u] + w * dkl_m;
          ol[u] = gz[i + u] * ep[i + u] * 0.5f * sqrtf(var) + w * dkl_l;
        }
        *reinterpret_cast<__nv_bfloat162*>(out + z) = __floats2bfloat162_rn(om[0], om[1]);
        *reinterpret_cast<__nv_bfloat162*>(out + Z + z) = __floats2bfloat162_rn(ol[0], ol[1]);
      }
    }
  }
}
// next step's mean / log_var / eps rows into L2
__device__ __forceinline__ void latent_prefetch(const RbParams& p, int t, int gtid, int GT) {
  if (t < 0) return;
  const int B = p.B, Z = p.Z, ZQ = (Z + 3) >> 2;
  for (int idx = gtid; idx < B * ZQ; idx += GT) {
    const int r = idx % B, zq = idx / B;
    if (zq & 7) continue;                              // one prefetch per 128 bytes of a row
    const size_t o = ((size_t)t * B + r) * Z + zq * 4;
    prefetch_l2(p.mean + o); prefetch_l2(p.logvar + o); prefetch_l2(p.eps + o);
  }
}

// ---- epilogue: partial tile -> slot of the destination (row-tiled fp32) ---------------------------------------------
__device__ __forceinline__ void epi_store(const RbParams& p, const RbSmem& sm, const RbJob& job, int s, uint32_t tmem_base, int cw,
                                          int lane, int rank) {
  const int qd = (cw + 2) & 3;                         // TMEM lane quadrant of this warp (warp id % 4)
  const int half = cw >> 2;
  const int b = rank * 128 + qd * 32 + lane;
  const bool ok = b < p.B;
  const int hw = job.N >> 1;                           // columns per warp half (multiple of 8)
  const int slot = kind_slot(job.kind);
  const uint32_t taddr = tmem_base + (static_cast<uint32_t>(qd * 32) << 16) + slot * RB_TMEM_STRIDE;
  mbar_wait_bounded(p, &sm.tfull[slot], (uint32_t)(s & 1), 10 + job.kind, s);
  tc_fence_after();
  for (int c = half * hw; c < (half + 1) * hw; c += 16) {
    float v0[8], v1[8];
    const bool two = c + 8 < (half + 1) * hw;
    tmem_ld_x8(taddr + c, v0);
    if (two) tmem_ld_x8(taddr + c + 8, v1);
    tmem_ld_wait();
    if (ok) {
      const int col = job.dcol0 + c;
      float* d = job.dst + tl_off(p.B, b, col);
      const size_t qs = (size_t)p.B * 4;               // next column quad
      if (col < job.dlimit) *reinterpret_cast<float4*>(d) = make_float4(v0[0], v0[1], v0[2], v0[3]);
      if (col + 4 < job.dlimit) *reinterpret_cast<float4*>(d + qs) = make_float4(v0[4], v0[5], v0[6], v0[7]);
      if (two) {
        if (col + 8 < job.dlimit) *reinterpret_cast<float4*>(d + 2 * qs) = make_float4(v1[0], v1[1], v1[2], v1[3]);
        if (col + 12 < job.dlimit) *reinterpret_cast<float4*>(d + 3 * qs) = make_float4(v1[4], v1[5], v1[6], v1[7]);
      }
    }
  }
  tc_fence_before();
}

__device__ __forceinline__ RbSeg make_seg(int amap, int wmap, int k0_blocks, int kblocks, int flag, int count) {
  RbSeg s;
  s.amap = amap; s.wmap = wmap; s.k0 = k0_blocks * 64; s.kblocks = kblocks; s.flag = flag; s.count = count;
  return s;
}
__device__ __forceinline__ void set_tile(RbJob& j, int kind, int row0, int N, float* dst, int dcol0, int dlimit, int sig) {
  j.kind = kind; j.N = N; j.w_box_rows = N >> 1; j.w_row[0] = row0; j.w_row[1] = row0 + (N >> 1);
  j.dst = dst; j.dcol0 = dcol0; j.dlimit = dlimit; j.sig = sig;
}

// the jobs of this pair, in issue order (= the order of the dependency chain of a step)
__device__ void build_jobs(const RbParams& p, int pair, RbJob* jobs, int* njobs) {
  const int kbG = p.Gp >> 6, B = p.B;
  int n = 0;
  auto part = [&](int i, int parts, int kb, int& k0, int& k1) { k0 = (int)((long long)i * kb / parts); k1 = (int)((long long)(i + 1) * kb / parts); };
  if (pair < p.nbig) {
    const int i = pair;
    if (i < p.nA * p.splitA) {
      const int tile = i / p.splitA, pt = i % p.splitA;
      int k0, k1; part(pt, p.splitA, kbG, k0, k1);
      RbJob& j = jobs[n++];
      set_tile(j, K_S6A, tile * 128, 128, p.dXEA + (size_t)pt * B * p.KX, tile * 128, p.KX, F_DXEA);
      j.nseg = 2;
      j.seg[0] = make_seg(AM_DGDEC, WM_DECX, k0, k1 - k0, F_DGDEC, p.cnt[F_DGDEC]);
      j.seg[1] = make_seg(AM_DGENC, WM_ENCX, k0, k1 - k0, F_DGENC, p.cnt[F_DGENC]);
    }
    if (i < p.nB * p.splitB) {
      const int tile = i / p.splitB, pt = i % p.splitB;
      int k0, k1; part(pt, p.splitB, kbG, k0, k1);
      RbJob& j = jobs[n++];
      set_tile(j, K_S6B, tile * 64, 64, p.dXEB + (size_t)pt * B * p.Hp, tile * 64, p.Hp, F_DXEB);
      j.nseg = 1;
      // gated on the END of the step's attention (not on dG_enc): its operand stream would otherwise share the SM's ingest
      // with the attention's feature stream (measured: first attention row 17 us with S6B underneath, 12 us without)
      j.seg[0] = make_seg(AM_DGENC, WM_ENCH, k0, k1 - k0, F_DQ, p.cnt[F_DQ]);
    }
    if (i < p.nX * p.splitX) {
      const int tile = i / p.splitX, pt = i % p.splitX;
      int k0, k1; part(pt, p.splitX, kbG, k0, k1);
      RbJob& j = jobs[n++];
      set_tile(j, K_S10, tile * 128, 128, p.dXA + (size_t)pt * B * 2 * p.Hp, tile * 128, 2 * p.Hp, F_DXA);
      j.nseg = 1;
      j.seg[0] = make_seg(AM_DGATT, WM_ATT, k0, k1 - k0, F_DGATT, p.cnt[F_DGATT]);
    }
  } else {
    const int i = pair - p.nbig;
    if (i < p.nZt * p.splitZ) {
      const int tile = i / p.splitZ, pt = i % p.splitZ;
      int k0, k1; part(pt, p.splitZ, kbG, k0, k1);
      RbJob& j = jobs[n++];
      set_tile(j, K_S2, tile * 96, 96, p.dzp + (size_t)pt * B * p.Zp, tile * 96, p.Zp, F_DZP);
      j.nseg = 1;
      j.seg[0] = make_seg(AM_DGDEC, WM_DECZ, k0, k1 - k0, F_DGDEC, p.cnt[F_DGDEC]);
    }
    if (i < p.n4) {
      RbJob& j = jobs[n++];
      set_tile(j, K_S4, i * p.N4, p.N4, p.dhe_fc, i * p.N4, p.H, F_DHE);
      j.nseg = 1;
      j.seg[0] = make_seg(AM_DML, WM_FC, 0, p.Z2p >> 6, F_DML, p.cnt[F_DML]);
      RbJob& k = jobs[n++];
      set_tile(k, K_S8, i * p.N4, p.N4, p.dh1q, i * p.N4, p.H, F_DH1Q);
      k.nseg = 1;
      k.seg[0] = make_seg(AM_DQ, WM_Q, 0, p.Ap >> 6, F_DQ, p.cnt[F_DQ]);
    }
  }
  *njobs = n;
}

}  // namespace

__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(PK_THREADS, 1)
recurrent_bwd_kernel(const __grid_constant__ RbParams p) {
  extern __shared__ __align__(1024) uint8_t rb_smem_raw[];
  if (threadIdx.x == 0 && (smem_u32(rb_smem_raw) & 1023u)) __trap();
  const AttnArgs a = p.att;
  const int ndx = p.splitA;
  const RbSmem sm = RbSmem::carve(rb_smem_raw, attn_smem_bytes(a, true, ndx, 1));
  const AttnSmem asm_ = carve(sm.att, a, true, ndx, 1);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int rank = (int)cluster_ctarank();
  const int pair = blockIdx.x >> 1;
  const int cta = blockIdx.x, G = gridDim.x;

  if (threadIdx.x == 0) {
    for (int i = 0; i < NUM_AMAPS; ++i) prefetch_tmap(&p.amap[i]);
    for (int i = 0; i < NUM_WMAPS; ++i) prefetch_tmap(&p.wmap[i]);
    sm.init_barriers();
    build_jobs(p, pair, sm.jobs, sm.njobs);
  }
  if (warp == 1) tmem_alloc_2sm<PK_TMEM_COLS>(sm.tmem_slot);
  attn_prologue(asm_, a, true);                        // attention ring barriers, w_a, zeroed q / d xhat buffers; __syncthreads inside
  tc_fence_before();
  cluster_sync_all();                                  // the peer's barriers exist before any remote arrival
  tc_fence_after();
  const uint32_t tmem_base = *sm.tmem_slot;
  const int njobs = *sm.njobs;
  const int T = p.T;

  if (warp == 0) {
    // ================= TMA producer of the GEMM operand ring (both CTAs of the pair) =================
    if (elect_one_sync()) {
      RingPos<RB_STAGES> pos;
      const uint64_t w_pol = ptx::l2_policy_evict_first();
      for (int s = 0; s < T; ++s) {
        const int t = T - 1 - s;
        for (int j = 0; j < njobs; ++j) {
          const RbJob& job = sm.jobs[j];
          const uint32_t tx = 2u * (uint32_t)(PK_X_BYTES + job.w_box_rows * 128);
          for (int g = 0; g < job.nseg; ++g) {
            const RbSeg sg = job.seg[g];
            produce_segment(p, sm, pos, s, rank, tx, w_pol, &p.amap[sg.amap], sg.k0, t, &p.wmap[sg.wmap], sg.k0, job.w_row[rank],
                            sg.kblocks, [&] {
              wait_flag(p, sg.flag, (unsigned int)((s + 1) * sg.count), 100 + job.kind * 10 + g, s);
              fence_proxy_async_global();
              RB_STAMP(true, 20 + j * 2 + g);
            });
          }
        }
      }
    }
    __syncwarp();
  } else if (warp == 1) {
    // ================= MMA issuer (leader CTA of the pair) =================
    if (rank == 0 && elect_one_sync()) {
      RingPos<RB_STAGES> pos;
      for (int s = 0; s < T; ++s) {
        for (int j = 0; j < njobs; ++j) {
          const RbJob& job = sm.jobs[j];
          const int slot = kind_slot(job.kind);
          mma_job(p, sm, pos, s, job, tmem_base + slot * RB_TMEM_STRIDE, slot);
          RB_STAMP(true, 28 + j);
        }
      }
    }
    __syncwarp();
  } else if (warp < 2 + PK_CWARPS) {
    // ================= compute warps: pointwise stages, epilogues, attention consumers =================
    const int cw = warp - 2;
    const int ctid = (int)threadIdx.x - 64;
    const int gw = cta * PK_CWARPS + cw, GW = G * PK_CWARPS;
    // spread the (few) latent items over all CTAs: consecutive global thread ids alternate between CTAs
    const int gtid = ctid * G + cta, GT = G * PK_CTHREADS;
    Ring ring;
    const RbJob* jk[NUM_KINDS];
    for (int k = 0; k < NUM_KINDS; ++k) jk[k] = nullptr;
    for (int j = 0; j < njobs; ++j) jk[sm.jobs[j].kind] = &sm.jobs[j];
    const int B = p.B;
    auto epilogue = [&](int kind, int s) {
      if (jk[kind]) {
        epi_store(p, sm, *jk[kind], s, tmem_base, cw, lane, rank);
        signal_done(p, jk[kind]->sig, ctid, false);
      }
    };
    auto prefetch_qs = [&](int t, int b, int slot) {
      const size_t r = (size_t)t * B + b;
      prefetch_vec(asm_.q(slot), p.q + r * p.A, a.A);
      prefetch_vec(asm_.sv(slot), p.smx + r * a.N, a.N);
      prefetch_vec(asm_.msk(slot), a.mask + (size_t)b * a.N, a.N);
    };
    auto prefetch_dx = [&](int b, int slot) {
      for (int k = 0; k < ndx; ++k) {
        const float* src = p.dXEA + (size_t)k * B * p.KX;
        float* dst = asm_.dx(slot, k);
        // quad i of the row -> two-plane layout of attn_bwd_row
        for (int i = ctid; i < (a.Fp >> 2); i += PK_CTHREADS)
          ptx::cp_async16(dst + (i & 1) * (a.Fp >> 1) + (i >> 1) * 4, src + ((size_t)i * B + b) * 4);
      }
    };
    cell_prefetch<2>(p, T - 1, gw, GW, lane);
    cell_prefetch<1>(p, T - 1, gw, GW, lane);
    cell_prefetch<0>(p, T - 1, gw, GW, lane);
    latent_prefetch(p, T - 1, gtid, GT);
    for (int s = 0; s < T; ++s) {
      const int t = T - 1 - s;
      RB_STAMP(ctid == 0, 0);
      // ---- decoder cell: needs S10 (and S6A) of step t + 1
      CellPre pre;
      cell_stage_pre<2>(p, t, gw, GW, lane, pre);
      wait_all(p, F_DXA, (unsigned int)(s * p.cnt[F_DXA]), 20, s, ctid);
      RB_STAMP(ctid == 0, 1);
      cell_stage_post<2>(p, t, s, gw, GW, lane, pre);
      RB_STAMP(ctid == 0, 2);
      signal_done(p, F_DGDEC, ctid);
      cell_prefetch<2>(p, t - 1, gw, GW, lane);
      RB_STAMP(ctid == 0, 3);
      epilogue(K_S2, s);
      RB_STAMP(ctid == 0, 4);
      // ---- latent heads
      wait_all(p, F_DZP, (unsigned int)((s + 1) * p.cnt[F_DZP]), 21, s, ctid);
      RB_STAMP(ctid == 0, 5);
      latent_stage(p, t, gtid, GT);
      signal_done(p, F_DML, ctid);
      latent_prefetch(p, t - 1, gtid, GT);
      RB_STAMP(ctid == 0, 6);
      epilogue(K_S4, s);
      RB_STAMP(ctid == 0, 7);
      // ---- encoder cell: needs S4 of this step and S6B of step t + 1
      cell_stage_pre<1>(p, t, gw, GW, lane, pre);
      wait_all(p, F_DHE, (unsigned int)((s + 1) * p.cnt[F_DHE]), 22, s, ctid);
      if (s > 0) wait_all(p, F_DXEB, (unsigned int)(s * p.cnt[F_DXEB]), 23, s, ctid);
      RB_STAMP(ctid == 0, 8);
      cell_stage_post<1>(p, t, s, gw, GW, lane, pre);
      RB_STAMP(ctid == 0, 9);
      signal_done(p, F_DGENC, ctid);
      cell_prefetch<1>(p, t - 1, gw, GW, lane);
      RB_STAMP(ctid == 0, 10);
      epilogue(K_S6A, s);
      RB_STAMP(ctid == 0, 11);
      // ---- region attention backward of this CTA's share of the rows that still carry gradient (a row past the end of
      //      its caption has d x_hat = 0: its d q / d u stay at the zeros they were initialised with); q and the saved
      //      softmax of the first row do not depend on S6A
      const int nact = p.nrows[t];
      const int* act = p.rows + (size_t)t * B;
      if (cta < nact) prefetch_qs(t, act[cta], 0);
      wait_all(p, F_DXEA, (unsigned int)((s + 1) * p.cnt[F_DXEA]), 24, s, ctid);
      RB_STAMP(ctid == 0, 12);
      if (cta < nact) {
        prefetch_dx(act[cta], 0);
        ptx::cp_async_commit();
        int cur = 0;
        for (int i = cta; i < nact; i += G, cur ^= 1) {
          const int b = act[i];
          const size_t r = (size_t)t * B + b;
          const int bn = i + G < nact ? act[i + G] : -1;
          attn_bwd_row(a, p.plan, asm_, ring, cur, nullptr,
                       [&] { if (bn >= 0) { prefetch_qs(t, bn, cur ^ 1); ptx::cp_async_commit(); } },
                       p.dqb + r * p.Ap, p.Ap, p.du + r * a.N,
                       [&] { if (bn >= 0) { prefetch_dx(bn, cur ^ 1); ptx::cp_async_commit(); } },   // single d xhat buffer
                       [&](int k) { RB_STAMP(ctid == 0 && i == cta, k == 0 ? 19 : k == 1 ? 23 : k == 2 ? 25 : k == 3 ? 26 : 27); });
        }
      }
      RB_STAMP(ctid == 0, 13);
      signal_done(p, F_DQ, ctid);
      epilogue(K_S8, s);
      RB_STAMP(ctid == 0, 14);
      // ---- attention-LSTM cell: needs S8, S6A of this step, S10 of step t + 1
      cell_stage_pre<0>(p, t, gw, GW, lane, pre);
      wait_all(p, F_DH1Q, (unsigned int)((s + 1) * p.cnt[F_DH1Q]), 25, s, ctid);
      RB_STAMP(ctid == 0, 15);
      cell_stage_post<0>(p, t, s, gw, GW, lane, pre);
      RB_STAMP(ctid == 0, 16);
      signal_done(p, F_DGATT, ctid);
      cell_prefetch<0>(p, t - 1, gw, GW, lane);
      RB_STAMP(ctid == 0, 17);
      epilogue(K_S6B, s);
      epilogue(K_S10, s);
      RB_STAMP(ctid == 0, 18);
    }
  } else {
    // ================= attention producer: streams the region features and P of this CTA's rows =================
    if (lane == 0) {
      Ring ring;
      const uint64_t pol = ptx::l2_policy_evict_first();
      for (int s = 0; s < T; ++s) {
        const int t = T - 1 - s;
        const int nact = p.nrows[t];
        const int* act = p.rows + (size_t)t * p.B;
        for (int i = cta; i < nact; i += G) {
          const int b = act[i];
          produce_block(asm_, ring, reinterpret_cast<const uint8_t*>(a.feats + (size_t)b * a.N * a.Fp), a.N, a.Fp * 2, p.plan.nF, p.plan.bF, pol);
          produce_block(asm_, ring, reinterpret_cast<const uint8_t*>(a.proj + (size_t)b * a.N * a.Ap), a.N, a.Ap * 2, p.plan.nP, p.plan.bP, pol);
        }
      }
    }
    __syncwarp();
  }
  pk_teardown(warp, tmem_base);
}

// rows[t*B + i] = i-th batch row (ascending) that still carries gradient at step t, nrows[t] = how many: a row is live at t
// if any target at a step >= t is unmasked (the loss and KL of masked steps have zero weight, updown_captioner.py:295-323,
// and nothing flows into a row from later steps once all of them are masked). One block of >= B threads per timestep.
__global__ void rb_active_rows_kernel(const float* __restrict__ tmask, int T, int B, int* __restrict__ rows, int* __restrict__ nrows) {
  __shared__ int wsum[32];
  const int t = blockIdx.x;
  const int b = threadIdx.x, lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
  bool live = false;
  if (b < B)
    for (int u = t; u < T; ++u) live = live || tmask[(size_t)u * B + b] != 0.f;
  const unsigned m = __ballot_sync(0xffffffffu, live);
  if (lane == 0) wsum[warp] = __popc(m);
  __syncthreads();
  int base = 0, total = 0;
  for (int w = 0; w < nw; ++w) { if (w < warp) base += wsum[w]; total += wsum[w]; }
  if (live) rows[(size_t)t * B + base + __popc(m & ((1u << lane) - 1u))] = b;
  if (threadIdx.x == 0) nrows[t] = total;
}

// host side
static size_t rb_smem_bytes(const AttnArgs& a, int ndx) { return RbSmem::bytes(attn_smem_bytes(a, true, ndx, 1), RB_MAX_JOBS); }

// Tiling of the jobs over NP CTA pairs; false if the shape does not fit.
struct RbTiling { int nbig, nsmall, nA, splitA, nB, splitB, nX, splitX, nZt, splitZ, n4, N4; };
static bool rb_tiling(const RecBwdArgs& r, int NP, RbTiling& t) {
  if (NP < 4) return false;
  const int kbG = r.Gp / 64;
  t.nsmall = std::max(1, NP / 6);
  t.nbig = NP - t.nsmall;
  t.nA = ceil_div(r.KX, 128); t.nB = ceil_div(r.Hp, 64); t.nX = ceil_div(2 * r.Hp, 128); t.nZt = ceil_div(r.Zp, 96);
  if (t.nA > t.nbig || t.nB > t.nbig || t.nX > t.nbig || t.nZt > t.nsmall) return false;
  t.splitA = std::max(1, std::min(std::min(RB_MAX_SPLIT_A, t.nbig / t.nA), kbG));
  t.splitB = std::max(1, std::min(std::min(RB_MAX_SPLIT_B, t.nbig / t.nB), kbG));
  t.splitX = std::max(1, std::min(std::min(RB_MAX_SPLIT_X, t.nbig / t.nX), kbG));
  t.splitZ = std::max(1, std::min(std::min(RB_MAX_SPLIT_Z, t.nsmall / t.nZt), kbG));
  t.N4 = round_up(ceil_div(r.H, t.nsmall), 16);
  if (t.N4 > 128) return false;
  t.n4 = ceil_div(r.H, t.N4);
  return true;
}

static bool rb_shape_ok(const RecBwdArgs& r) {
  // Z even: the latent stage reads mean / log_var / eps as 8-byte pairs
  if (r.B > 256 || r.B < 1 || (r.H & 3) || (r.Z & 1) || (r.Hp & 63) || (r.Fp & 63) || (r.Zp & 63) || (r.Z2p & 63) || (r.Ap & 63) || (r.Gp & 63)) return false;
  const AttnArgs& a = r.att;
  if (a.N > 32 * ATT_NREG || a.Fp > 8 * ATT_CONSUMERS * ATT_FV || a.Ap * 2 > ATT_STAGE_BYTES || a.Fp * 2 > ATT_STAGE_BYTES ||
      a.Ap > 2 * ATT_CONSUMERS * ATT_PV || (a.Ap % 8) || (a.Fp % 8))
    return false;
  return true;
}

// host-only view of the job map for `pairs` co-resident CTA pairs (tests): nbig, nsmall, nA, splitA, nB, splitB, nX, splitX,
// nZt, splitZ, n4, N4; false if the shape does not fit
bool recurrent_backward_tiling(const RecBwdArgs& r, int pairs, int out[12]) {
  RbTiling t;
  if (!rb_shape_ok(r) || !rb_tiling(r, pairs, t)) return false;
  const int v[12] = {t.nbig, t.nsmall, t.nA, t.splitA, t.nB, t.splitB, t.nX, t.splitX, t.nZt, t.splitZ, t.n4, t.N4};
  for (int i = 0; i < 12; ++i) out[i] = v[i];
  return true;
}

bool recurrent_backward_supported(const RecBwdArgs& r) {
  static const bool off = [] { const char* e = getenv("SSCVAE_PERSISTENT_BWD"); return e && e[0] == '0'; }();
  if (off || !rb_shape_ok(r)) return false;
  // the split of S6A (<= RB_MAX_SPLIT_A) sizes the d xhat staging buffers: take the worst case for the occupancy query
  const size_t smem = rb_smem_bytes(r.att, RB_MAX_SPLIT_A);
  if (smem > 227 * 1024) return false;
  const int NP = pk_grid_pairs(recurrent_bwd_kernel, smem);
  RbTiling t;
  return rb_tiling(r, NP, t);
}

int recurrent_backward(cudaStream_t s, const RecBwdArgs& r) {
  RbParams p;
  memset(&p, 0, sizeof(p));
  const AttnArgs& a = r.att;
  REQUIRE(rb_shape_ok(r), "recurrent_bwd: unsupported shape");
  const size_t smem = rb_smem_bytes(a, RB_MAX_SPLIT_A);
  const int NP = pk_grid_pairs(recurrent_bwd_kernel, smem);
  RbTiling tl;
  REQUIRE(NP > 0 && rb_tiling(r, NP, tl), "recurrent_bwd: the shape does not fit the co-resident CTA pairs");
  p.B = r.B; p.T = r.T; p.H = r.H; p.Hp = r.Hp; p.Fp = r.Fp; p.Zp = r.Zp; p.Z = r.Z; p.Z2p = r.Z2p; p.A = r.A; p.Ap = r.Ap;
  p.KX = r.KX; p.G = 4 * r.H; p.Gp = r.Gp; p.N = a.N;
  p.sentiment_vae = r.sentiment_vae; p.prior_var = r.prior_var; p.tiled = r.tiled;
  p.nbig = tl.nbig; p.nsmall = tl.nsmall; p.nA = tl.nA; p.splitA = tl.splitA; p.nB = tl.nB; p.splitB = tl.splitB;
  p.nX = tl.nX; p.splitX = tl.splitX; p.nZt = tl.nZt; p.splitZ = tl.splitZ; p.n4 = tl.n4; p.N4 = tl.N4;
  const int Gr = 2 * NP;
  p.cnt[F_DGDEC] = Gr; p.cnt[F_DML] = Gr; p.cnt[F_DGENC] = Gr; p.cnt[F_DQ] = Gr; p.cnt[F_DGATT] = Gr;
  p.cnt[F_DZP] = 2 * tl.nZt * tl.splitZ; p.cnt[F_DHE] = 2 * tl.n4; p.cnt[F_DH1Q] = 2 * tl.n4;
  p.cnt[F_DXEA] = 2 * tl.nA * tl.splitA; p.cnt[F_DXEB] = 2 * tl.nB * tl.splitB; p.cnt[F_DXA] = 2 * tl.nX * tl.splitX;
  TRY(encode_act3d(&p.amap[AM_DGDEC], r.dG_dec, r.Gp, r.B, r.T, r.Gp));
  TRY(encode_act3d(&p.amap[AM_DGENC], r.dG_enc, r.Gp, r.B, r.T, r.Gp));
  TRY(encode_act3d(&p.amap[AM_DGATT], r.dG_att, r.Gp, r.B, r.T, r.Gp));
  TRY(encode_act3d(&p.amap[AM_DML], r.dml, r.Z2p, r.B, r.T, r.Z2p));
  TRY(encode_act3d(&p.amap[AM_DQ], r.dqb, r.Ap, r.B, r.T, r.Ap));
  TRY(encode_w2d(&p.wmap[WM_DECX], r.w_dec_xzT, r.Gp, r.KX, r.Gp, 64));
  TRY(encode_w2d(&p.wmap[WM_DECZ], r.w_dec_xzT + (size_t)r.KX * r.Gp, r.Gp, r.Zp, r.Gp, 48));
  TRY(encode_w2d(&p.wmap[WM_ENCX], r.w_enc_xhT, r.Gp, r.KX, r.Gp, 64));
  TRY(encode_w2d(&p.wmap[WM_ENCH], r.w_enc_xhT + (size_t)r.KX * r.Gp, r.Gp, r.Hp, r.Gp, 32));
  TRY(encode_w2d(&p.wmap[WM_ATT], r.w_att_recT, r.Gp, 2 * r.Hp, r.Gp, 64));
  TRY(encode_w2d(&p.wmap[WM_FC], r.w_fcT, r.Z2p, r.Hp, r.Z2p, tl.N4 / 2));
  TRY(encode_w2d(&p.wmap[WM_Q], r.wqT, r.Ap, r.Hp, r.Ap, tl.N4 / 2));
  p.gates_att = r.gates_att; p.gates_enc = r.gates_enc; p.gates_dec = r.gates_dec;
  p.c1 = r.c1; p.c_enc = r.c_enc; p.c_dec = r.c_dec;
  p.mean = r.mean; p.logvar = r.logvar; p.eps = r.eps; p.pm_row = r.pm_row;
  p.q = r.q; p.smx = r.smx; p.dhead = r.dhead; p.gkld = r.gkld; p.tmask = r.tmask;
  p.rows = r.rows; p.nrows = r.rows + (size_t)r.T * r.B;
  p.dc1 = r.dc1; p.dc_enc = r.dc_enc; p.dc_dec = r.dc_dec;
  p.dG_att = r.dG_att; p.dG_enc = r.dG_enc; p.dG_dec = r.dG_dec; p.dml = r.dml; p.dqb = r.dqb; p.du = r.du;
  p.dXEA = r.dXEA; p.dXEB = r.dXEB; p.dXA = r.dXA; p.dzp = r.dzp; p.dhe_fc = r.dhe_fc; p.dh1q = r.dh1q;
  p.att = a;
  p.flags = r.flags;
  p.timeout_ns = pk_timeout_ns();
  p.plan = attn_chunk_plan(a);
  // model FLOPs of the loop: the three data-gradient GEMMs, d z, latent heads, query; bytes: the attention stream
  const double G4 = 4.0 * r.H;
  const double flops = 2.0 * r.B * r.T * (G4 * (r.KX + r.Zp) + G4 * (r.KX + r.Hp) + G4 * 2.0 * r.Hp + 2.0 * r.Z * r.H + (double)r.A * r.H);
  PROF_SCOPE(s, "recurrent_bwd", flops, (double)r.B * r.T * a.N * (a.Ap + a.Fp) * 2.0);
  static const bool dbg = [] { const char* e = getenv("SSCVAE_RB_DBG"); return e && e[0] == '1'; }();
  if (dbg) {
    TRY(pk_dbg_begin(s, &p.dbg));
    p.dbg_s = r.T / 2;
  }
  CUDA_TRY(cudaMemsetAsync(r.flags, 0, 64 * sizeof(unsigned int), s));
  rb_active_rows_kernel<<<r.T, round_up(r.B, 32), 0, s>>>(r.tmask, r.T, r.B, r.rows, r.rows + (size_t)r.T * r.B);
  CUDA_TRY(cudaGetLastError());
  ++g_launch_count;
  TRY(pk_launch(recurrent_bwd_kernel, NP, smem, s, p));
  if (dbg) {
    char head[64];
    snprintf(head, sizeof(head), "[rbdbg] B=%d s=%d", r.B, p.dbg_s);
    TRY(pk_dbg_print(s, p.dbg, 2 * NP, head, {0, 1, 2 * tl.nbig - 2, 2 * tl.nbig, 2 * NP - 2}, 32));
  }
  return 0;
}

}  // namespace sscvae

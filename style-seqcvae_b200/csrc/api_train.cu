// C ABI: handle, weight packing, training forward and backward-through-time (include/sscvae.h).
//
// Data layout in HBM (all time-stacked buffers are time-major, row r = t*B + b):
//   XA  ((T+1)B, 2Hp) bf16  [h1_{t-1} | h_dec_{t-1}]            operand of the attention-LSTM recurrence
//   XE  (TB, Fp+2Hp)  bf16  [xhat_t | h1_t | h_dec_{t-1}]       operand of the encoder / decoder LSTMs
//   HE  ((T+1)B, Hp)  bf16  h_enc_{t-1}                         encoder hidden operand / fc input
//   ZB  (TB, Zp)      bf16  z_t
// Hidden states exist only as bf16 GEMM operands (written once by the LSTM pointwise kernel into
// every buffer that consumes them); cell states, gate activations, softmax/KL/CE stay fp32.
// "p" suffixes are sizes rounded up to 64 elements: every bf16 row stride and column block is a multiple of 128 bytes
// (one TMA box row = one cache line, see init_dims).
#include "api_internal.cuh"

namespace sscvae {

// ---- error string ------------------------------------------------------------------------------
static thread_local char g_err[1024] = "";
void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}
const char* get_error() { return g_err; }

// ---- dims --------------------------------------------------------------------------------------
int init_dims(const SscvaeDims* in, Dims& d) {
  REQUIRE(in != nullptr, "dims is NULL");
  d.F = in->image_feature_size; d.E = in->embedding_size; d.H = in->hidden_size;
  d.A = in->attention_projection_size; d.Z = in->z_space; d.V = in->vocab_size; d.L = in->max_caption_length;
  d.sv = in->sentiment_vae; d.simple = in->simple_vae; d.tied = in->tied_embedding;
  d.pad = in->pad_index; d.boundary = in->boundary_index; d.prior_std = in->prior_std; d.mult = in->senti_prior_multip;
  REQUIRE(d.F > 0 && d.E > 0 && d.H > 0 && d.A > 0 && d.Z > 0 && d.V > 1 && d.L > 0, "non-positive dimension");
  if (d.sv < 0 || d.sv > 2) {
    set_error("sentiment_vae=%d unsupported (0, 1 or 2)", d.sv);
    return SSCVAE_ERR_UNSUPPORTED;
  }
  d.le = in->latent_embedding;
  REQUIRE(d.sv != 2 || d.le == 0 || d.le == 1, "latent_embedding must be 0 (glove) or 1 (senti_word_net)");
  REQUIRE(d.pad >= 0 && d.pad < d.V && d.boundary >= 0 && d.boundary < d.V, "pad/boundary index out of range");
  REQUIRE(d.prior_std > 0.f, "prior_std must be positive");
  d.T = d.L + 1;
  // width of the conditioning column block of the encoder / decoder LSTM inputs (updown_cell.py:47-81); simple_vae drops it
  d.cvar = (d.sv == 2 && !d.simple) ? 1 : 0;
  d.cond = (d.simple || d.sv == 0) ? 0 : d.sv == 1 ? 1 : (d.le == 1 ? 1 : d.Z);
  // Every bf16 operand row stride and column-block offset is a multiple of 64 elements = 128 bytes, so that each
  // 128-byte row segment of a TMA box is exactly ONE cache line. With 16-byte granularity (the TMA minimum) a
  // segment straddles two lines and the TMA unit pulls both whole lines into the SM: ncu showed 2.0x the operand
  // bytes crossing the crossbar (profiles/README.md), and the per-step GEMMs are bound by exactly that ingest.
  d.Fp = round_up(d.F, kPad); d.Ep = round_up(d.E, kPad); d.Hp = round_up(d.H, kPad); d.Ap = round_up(d.A, kPad);
  d.Zp = round_up(d.Z, kPad); d.Vp = round_up(d.V, kPad);
  d.G = 4 * d.H; d.Gp = round_up(d.G, kPad); d.Z2 = 2 * d.Z; d.Z2p = round_up(d.Z2, kPad);
  d.KX = d.Fp + 2 * d.Hp;
  d.Cp = d.cvar ? round_up(d.cond, kPad) : 0;
  d.ZC = d.Zp + d.Cp;
  d.GP = lstm_gate_rows(d.H);
  { const char* e = getenv("SSCVAE_DEBUG_LOGITS"); d.debug_logits = (e && e[0] == '1') ? 1 : 0; }
  return 0;
}

// ---- region planner ----------------------------------------------------------------------------
void Plan::add(const char* name, size_t bytes) {
  Region r; r.name = name; r.off = total; r.bytes = bytes;
  regs.push_back(r);
  total += round_up_sz(bytes, 1024);
}
const Region* Plan::find(const char* name) const {
  for (const Region& r : regs)
    if (strcmp(r.name, name) == 0) return &r;
  return nullptr;
}

static void plan_packed(const Dims& d, Plan& p) {
  const size_t b = sizeof(bf16);
  const int NO = d.tied ? d.E : d.V, NOp = d.tied ? d.Ep : d.Vp;
  // --- weights streamed at every forward timestep, contiguous so one L2 access-policy window covers them.
  // Forward LSTM blocks hold GP = lstm_gate_rows(H) gate-interleaved rows (kernels.cuh: lstm_gate_row), so that one
  // 128-row GEMM tile owns all four gates of 32 hidden units and the cell can run in the GEMM epilogue.
  p.add("w_att_rec", (size_t)d.GP * 2 * d.Hp * b);
  p.add("wq", (size_t)d.A * d.Hp * b);
  p.add("w_enc_x", (size_t)d.GP * d.KX * b);
  p.add("w_enc_hh", (size_t)d.GP * d.Hp * b);
  if (d.cvar) p.add("w_enc_c", (size_t)d.GP * d.Cp * b);
  p.add("w_fc", (size_t)d.Z2 * d.Hp * b);
  p.add("w_dec_x", (size_t)d.GP * d.KX * b);
  p.add("w_dec_z", (size_t)d.GP * d.ZC * b);               // [W_z | W_c] against the [z | c] rows of ZB
  p.add("fwd_end", 0);
  // --- transposed twins streamed at every backward timestep
  p.add("w_dec_xzT", (size_t)(d.KX + d.ZC) * d.Gp * b);   // rows [0,KX): W_dec_x^T ; [KX,KX+Zp): W_dec_z^T ; then Cp rows W_dec_c^T
  p.add("w_fcT", (size_t)d.Hp * d.Z2p * b);
  p.add("w_enc_xhT", (size_t)(d.KX + d.Hp + d.Cp) * d.Gp * b);   // rows [0,KX): W_enc_x^T ; [KX,KX+Hp): W_enc_hh^T ; then Cp rows W_enc_c^T
  p.add("wqT", (size_t)d.Hp * d.Ap * b);
  p.add("w_att_recT", (size_t)2 * d.Hp * d.Gp * b);
  p.add("bwd_end", 0);
  // --- used once per sequence
  p.add("embb", (size_t)d.V * d.Ep * b);
  if (d.tied) p.add("embT", (size_t)d.E * d.Vp * b);
  p.add("w_att_e", (size_t)d.GP * d.Ep * b);
  p.add("w_att_eT", (size_t)d.Ep * d.Gp * b);
  p.add("w_att_f", (size_t)d.GP * d.Fp * b);
  p.add("wv", (size_t)d.A * d.Fp * b);
  p.add("w_out", (size_t)NO * d.Hp * b);
  p.add("w_outT", (size_t)d.Hp * NOp * b);
  p.add("b_att", (size_t)d.G * 4);
  p.add("b_enc", (size_t)d.G * 4);
  p.add("b_dec", (size_t)d.G * 4);
  p.add("scol_enc", (size_t)d.G * 4);
  p.add("scol_dec", (size_t)d.G * 4);
  p.add("b_fc", (size_t)d.Z2 * 4);
}

static void plan_train(const Dims& d, int B, int N, Plan& p) {
  const size_t b = sizeof(bf16), f = 4;
  const size_t T = d.T, TB = T * B, TBp = round_up((int)TB, kPad), BN = (size_t)B * N, BNp = round_up((int)BN, kPad);
  const size_t Bp = round_up(B, kPad);
  // ---- forward, kept for backward
  p.add("seed", 16);                                   // Philox seed of this call (device memory: graph replay)
  p.add("tok", (size_t)B * (d.L + 2) * 4);
  p.add("tmask", TB * f);
  p.add("lengths", B * f);
  p.add("pm_row", B * f);
  p.add("sent", B * f);
  p.add("featsb", BN * d.Fp * b);
  p.add("mask", BN * f);
  p.add("avgb", (size_t)B * d.Fp * b);
  p.add("projb", BN * d.Ap * b);
  p.add("embb_t", TB * d.Ep * b);
  p.add("gx_att", TB * d.GP * f);
  p.add("gavg", (size_t)B * d.GP * f);
  p.add("XA", (T + 1) * B * 2 * d.Hp * b);
  p.add("XE", TB * d.KX * b);
  p.add("HE", (T + 1) * B * d.Hp * b);
  p.add("ZB", TB * d.ZC * b);
  if (d.cvar) {
    p.add("objm", BN * d.Z * f);                        // per-box attribute means (kept for the backward)
    p.add("pm", TB * d.Z * f);                          // per-step prior mean sum_n alpha_n objm_n
    p.add("dpm", (size_t)B * d.Z * f);
    p.add("dalpha_x", (size_t)B * N * f);
  }
  p.add("acc", (size_t)B * d.GP * f);
  p.add("gates_att", TB * d.G * f);
  p.add("gates_enc", TB * d.G * f);
  p.add("gates_dec", TB * d.G * f);
  p.add("c1", TB * d.H * f);
  p.add("c_enc", TB * d.H * f);
  p.add("c_dec", TB * d.H * f);
  p.add("q", TB * d.A * f);
  p.add("alpha", TB * N * f);
  p.add("smx", TB * N * f);
  p.add("du", TB * N * f);
  p.add("ml", (size_t)B * d.Z2 * f);
  p.add("mean", TB * d.Z * f);
  p.add("logvar", TB * d.Z * f);
  p.add("eps", TB * d.Z * f);
  p.add("kl", TB * f);
  p.add("kl_part", TB * recurrent_forward_kl_parts(d.Z) * f);   // persistent recurrent kernel: per-tile KL partial sums
  p.add("rf_flags", 1024);                                      // ... and its dataflow counters
  if (d.tied) {
    p.add("ob", TB * d.Ep * b);
    p.add("o32", TB * d.E * f);
  }
  // The fp32 logits (T*B, V) are NOT materialised: the head GEMM's epilogue keeps per-tile softmax statistics
  // (gemm.cuh: RowStatsEpi) and the backward recomputes the tile to emit the bf16 CE gradient. SSCVAE_DEBUG_LOGITS=1
  // (read at sscvae_create) additionally stores them for the parity tests.
  if (d.debug_logits) p.add("logits", TB * d.V * f);
  const size_t nst = gemm_rowstats_tiles(d.V);
  p.add("rs_max", TB * nst * f);
  p.add("rs_sum", TB * nst * f);
  p.add("rs_arg", TB * nst * 4);
  p.add("rs_tgt", TB * f);
  p.add("tgt_row", TB * 4);
  p.add("gcoef", TB * f);
  p.add("lse", TB * f);
  p.add("nll", TB * f);
  // ---- backward
  p.add("dlogits", TB * d.Vp * b);
  if (d.tied) p.add("dpreo", TB * d.Ep * b);
  p.add("dhead", TB * d.H * f);
  p.add("dG_att", TB * d.Gp * b);
  p.add("dG_enc", TB * d.Gp * b);
  p.add("dG_dec", TB * d.Gp * b);
  p.add("dml", TB * d.Z2p * b);
  p.add("dqb", TB * d.Ap * b);
  p.add("dXEZ", (size_t)B * (d.KX + d.ZC) * f);          // decoder part of d[xhat|h1|h_dec], d z (and d c)
  p.add("dXEH0", (size_t)B * (d.KX + d.Hp + d.Cp) * f);  // total d[xhat|h1|h_dec], d h_enc_{t-1} (and the encoder's d c) (ping-pong)
  p.add("dXEH1", (size_t)B * (d.KX + d.Hp + d.Cp) * f);
  p.add("dXA0", (size_t)B * 2 * d.Hp * f);
  p.add("dXA1", (size_t)B * 2 * d.Hp * f);
  p.add("dhenc_fc", (size_t)B * d.H * f);
  p.add("dh1_q", (size_t)B * d.H * f);
  p.add("dc1", (size_t)B * d.H * f);
  p.add("dc_enc", (size_t)B * d.H * f);
  p.add("dc_dec", (size_t)B * d.H * f);
  // persistent BPTT kernel (recurrent_bwd.cu): dataflow counters and the split-K slots of its data-gradient GEMMs
  p.add("rb_flags", 1024);
  p.add("rb_rows", (TB + T) * 4);
  p.add("rb_dXEA", (size_t)RB_MAX_SPLIT_A * B * d.KX * f);
  p.add("rb_dXEB", (size_t)RB_MAX_SPLIT_B * B * d.Hp * f);
  p.add("rb_dXA", (size_t)RB_MAX_SPLIT_X * B * 2 * d.Hp * f);
  p.add("rb_dzp", (size_t)RB_MAX_SPLIT_Z * B * d.Zp * f);
  p.add("dproj_acc", BN * d.A * f);
  p.add("dwa_acc", (size_t)B * d.A * f);
  // ---- transposed operands of the batched-over-time weight-gradient GEMMs
  p.add("dGT", (size_t)d.G * TBp * b);
  p.add("XAT", (size_t)2 * d.Hp * TBp * b);
  p.add("XET", (size_t)d.KX * TBp * b);
  p.add("HETp", (size_t)d.Hp * TBp * b);
  p.add("HETc", (size_t)d.Hp * TBp * b);
  p.add("hdecTc", (size_t)d.Hp * TBp * b);
  p.add("ZBT", (size_t)d.ZC * TBp * b);
  p.add("embT_t", (size_t)d.Ep * TBp * b);
  p.add("dmlT", (size_t)d.Z2p * TBp * b);
  p.add("dqT", (size_t)d.Ap * TBp * b);
  if (d.tied) p.add("dpreoT", (size_t)d.Ep * TBp * b);
  else {
    p.add("dlogitsT", (size_t)d.V * TBp * b);
    p.add("dxemb", TB * d.E * f);
  }
  p.add("dGsum", (size_t)B * d.Gp * b);
  p.add("dGsumT", (size_t)d.G * Bp * b);
  p.add("avgT", (size_t)d.Fp * Bp * b);
  p.add("dPT", (size_t)d.A * BNp * b);
  p.add("featsT", (size_t)d.Fp * BNp * b);
  p.add("biasg", (size_t)std::max(d.G, std::max(d.V, d.E)) * f);
}

const Plan& Handle::train_plan(int B, int N) {
  if (tp_B != B || tp_N != N) {
    tp = Plan();
    plan_train(d, B, N, tp);
    tp_B = B; tp_N = N;
  }
  return tp;
}

// ---- weight packing ----------------------------------------------------------------------------
// The packed blob as ONE list of source blocks (kernels.cuh: SgdPackJob): every column block of every weight with the
// images it has in the blob. The plain pack (sscvae_pack_weights) and the fused clip + SGD + pack of the optimizer
// (sscvae_sgd_step_packed) both run jobs built from this list, and the source blocks of each weight split its columns
// with no overlap, so every element is updated by exactly one job.
struct SrcOut { int kind; const char* region; size_t at; int ld, gate_H; };   // `at`: element offset in the region
struct SrcBlock { int w, w2, c0, cols; int nout; SrcOut out[2]; };

// rows, columns of each weight in reference layout (include/sscvae.h); a bias is one row
static void weight_shapes(const Dims& d, int rows[SSCVAE_W_COUNT], int cols[SSCVAE_W_COUNT]) {
  const int G = d.G, H = d.H, c = d.cond, NO = d.tied ? d.E : d.V;
  auto set = [&](int w, int r, int k) { rows[w] = r; cols[w] = k; };
  set(SSCVAE_W_EMBEDDING, d.V, d.E);
  set(SSCVAE_W_ATT_IH, G, d.E + d.F + 2 * H); set(SSCVAE_W_ATT_HH, G, H);
  set(SSCVAE_W_ATT_BIH, 1, G); set(SSCVAE_W_ATT_BHH, 1, G);
  set(SSCVAE_W_QUERY_PROJ, d.A, H); set(SSCVAE_W_IMAGE_PROJ, d.A, d.F); set(SSCVAE_W_ATT_VEC, 1, d.A);
  set(SSCVAE_W_ENC_IH, G, d.F + 2 * H + c); set(SSCVAE_W_ENC_HH, G, H);
  set(SSCVAE_W_ENC_BIH, 1, G); set(SSCVAE_W_ENC_BHH, 1, G);
  set(SSCVAE_W_DEC_IH, G, d.F + 2 * H + c + d.Z); set(SSCVAE_W_DEC_HH, G, H);
  set(SSCVAE_W_DEC_BIH, 1, G); set(SSCVAE_W_DEC_BHH, 1, G);
  set(SSCVAE_W_FC_MEAN_W, d.Z, H); set(SSCVAE_W_FC_MEAN_B, 1, d.Z);
  set(SSCVAE_W_FC_LOGVAR_W, d.Z, H); set(SSCVAE_W_FC_LOGVAR_B, 1, d.Z);
  set(SSCVAE_W_OUT_PROJ_W, NO, H); set(SSCVAE_W_OUT_PROJ_B, 1, NO);
}

static int source_blocks(const Dims& d, std::vector<SrcBlock>& bl) {
  const int E = d.E, F = d.F, H = d.H, Z = d.Z, c = d.cond, NOp = d.tied ? d.Ep : d.Vp;
  bl.clear();
  auto add = [&](int w, int c0, int cols, int w2, std::initializer_list<SrcOut> outs) {
    if (cols <= 0) return;
    SrcBlock b = {w, w2, c0, cols, (int)outs.size(), {}};
    int k = 0;
    for (const SrcOut& o : outs) b.out[k++] = o;
    bl.push_back(b);
  };
  auto plain = [](const char* r, size_t at, int ld, int gate_H = 0) { return SrcOut{kPackPlain, r, at, ld, gate_H}; };
  auto trans = [](const char* r, size_t at, int ld) { return SrcOut{kPackTransposed, r, at, ld, 0}; };
  auto f32 = [](const char* r, size_t at, int ld) { return SrcOut{kPackF32, r, at, ld, 0}; };
  const size_t Gp = d.Gp;
  // embedding (gather source and, tied, the vocabulary GEMM operand)
  if (d.tied) add(SSCVAE_W_EMBEDDING, 0, E, -1, {plain("embb", 0, d.Ep), trans("embT", 0, d.Vp)});
  else add(SSCVAE_W_EMBEDDING, 0, E, -1, {plain("embb", 0, d.Ep)});
  // attention LSTM: W_ih columns [emb E | avg F | h1 H | h_dec H] (updown_cell.py:143-145); W_hh folded onto h1
  add(SSCVAE_W_ATT_IH, 0, E, -1, {plain("w_att_e", 0, d.Ep, H), trans("w_att_eT", 0, d.Gp)});
  add(SSCVAE_W_ATT_IH, E, F, -1, {plain("w_att_f", 0, d.Fp, H)});
  add(SSCVAE_W_ATT_IH, E + F, H, SSCVAE_W_ATT_HH, {plain("w_att_rec", 0, 2 * d.Hp, H), trans("w_att_recT", 0, d.Gp)});
  add(SSCVAE_W_ATT_IH, E + F + H, H, -1, {plain("w_att_rec", d.Hp, 2 * d.Hp, H), trans("w_att_recT", d.Hp * Gp, d.Gp)});
  add(SSCVAE_W_ATT_BIH, 0, d.G, SSCVAE_W_ATT_BHH, {f32("b_att", 0, d.G)});
  // attention
  add(SSCVAE_W_QUERY_PROJ, 0, H, -1, {plain("wq", 0, d.Hp), trans("wqT", 0, d.Ap)});
  add(SSCVAE_W_IMAGE_PROJ, 0, F, -1, {plain("wv", 0, d.Fp)});
  add(SSCVAE_W_ATT_VEC, 0, d.A, -1, {});                              // read by the kernels in fp32
  // encoder / decoder LSTMs: W_ih columns [xhat F | h1 H | h_dec H | cond c (| z Z)] (updown_cell.py:178-190, 211-224);
  // the decoder's W_hh is folded onto h_dec; sentiment_vae 1: the conditioning column stays fp32
  const int offs_src[3] = {0, F, F + H};
  const size_t offs_dst[3] = {0, (size_t)d.Fp, (size_t)d.Fp + d.Hp};
  const int widths[3] = {F, H, H};
  for (int k = 0; k < 3; ++k)
    add(SSCVAE_W_ENC_IH, offs_src[k], widths[k], -1, {plain("w_enc_x", offs_dst[k], d.KX, H), trans("w_enc_xhT", offs_dst[k] * Gp, d.Gp)});
  if (d.cvar) add(SSCVAE_W_ENC_IH, F + 2 * H, c, -1, {plain("w_enc_c", 0, d.Cp, H), trans("w_enc_xhT", (size_t)(d.KX + d.Hp) * Gp, d.Gp)});
  else add(SSCVAE_W_ENC_IH, F + 2 * H, c, -1, {f32("scol_enc", 0, 1)});
  add(SSCVAE_W_ENC_HH, 0, H, -1, {plain("w_enc_hh", 0, d.Hp, H), trans("w_enc_xhT", (size_t)d.KX * Gp, d.Gp)});
  add(SSCVAE_W_ENC_BIH, 0, d.G, SSCVAE_W_ENC_BHH, {f32("b_enc", 0, d.G)});
  for (int k = 0; k < 3; ++k)
    add(SSCVAE_W_DEC_IH, offs_src[k], widths[k], k == 2 ? SSCVAE_W_DEC_HH : -1,
        {plain("w_dec_x", offs_dst[k], d.KX, H), trans("w_dec_xzT", offs_dst[k] * Gp, d.Gp)});
  if (d.cvar) add(SSCVAE_W_DEC_IH, F + 2 * H, c, -1, {plain("w_dec_z", d.Zp, d.ZC, H), trans("w_dec_xzT", (size_t)(d.KX + d.Zp) * Gp, d.Gp)});
  else add(SSCVAE_W_DEC_IH, F + 2 * H, c, -1, {f32("scol_dec", 0, 1)});
  add(SSCVAE_W_DEC_IH, F + 2 * H + c, Z, -1, {plain("w_dec_z", 0, d.ZC, H), trans("w_dec_xzT", (size_t)d.KX * Gp, d.Gp)});
  add(SSCVAE_W_DEC_BIH, 0, d.G, SSCVAE_W_DEC_BHH, {f32("b_dec", 0, d.G)});
  // latent heads stacked [fc_mean ; fc_log_var]
  add(SSCVAE_W_FC_MEAN_W, 0, H, -1, {plain("w_fc", 0, d.Hp), trans("w_fcT", 0, d.Z2p)});
  add(SSCVAE_W_FC_LOGVAR_W, 0, H, -1, {plain("w_fc", (size_t)Z * d.Hp, d.Hp), trans("w_fcT", Z, d.Z2p)});
  add(SSCVAE_W_FC_MEAN_B, 0, Z, -1, {f32("b_fc", 0, Z)});
  add(SSCVAE_W_FC_LOGVAR_B, 0, Z, -1, {f32("b_fc", Z, Z)});
  // output head
  add(SSCVAE_W_OUT_PROJ_W, 0, H, -1, {plain("w_out", 0, d.Hp), trans("w_outT", 0, NOp)});
  add(SSCVAE_W_OUT_PROJ_B, 0, d.tied ? E : d.V, -1, {});             // read by the kernels in fp32
  // the blocks of each weight (its own column blocks, and the whole weight as a fold partner) split its columns
  int rows[SSCVAE_W_COUNT], cols[SSCVAE_W_COUNT];
  weight_shapes(d, rows, cols);
  REQUIRE((int)bl.size() <= kMaxSgdPackJobs, "%d source blocks > %d", (int)bl.size(), kMaxSgdPackJobs);
  for (int w = 0; w < SSCVAE_W_COUNT; ++w) {
    int next = 0;                                      // blocks are listed in column order per weight
    for (const SrcBlock& b : bl) {
      if (b.w == w) { REQUIRE(b.c0 == next, "weight %d: source block at column %d, expected %d", w, b.c0, next); next += b.cols; }
      if (b.w2 == w) {
        REQUIRE(next == 0 && rows[w] == rows[b.w] && cols[w] == b.cols, "weight %d: fold partner does not match its block", w);
        next = cols[w];
      }
    }
    REQUIRE(next == cols[w], "weight %d: source blocks cover %d of %d columns", w, next, cols[w]);
  }
  return 0;
}

static size_t out_offset(const Plan& pp, const SrcOut& o) { return pp.find(o.region)->off + o.at * (o.kind == kPackF32 ? 4 : 2); }

static void fill_job(const Dims& d, const Plan& pp, const SrcBlock& b, char* pk, SgdPackJob& j) {
  int rows[SSCVAE_W_COUNT], cols[SSCVAE_W_COUNT];
  weight_shapes(d, rows, cols);
  j = SgdPackJob();
  j.w = b.w; j.w2 = b.w2; j.c0 = b.c0; j.cols = b.cols; j.rows = rows[b.w]; j.ld = cols[b.w];
  j.ld2 = b.w2 >= 0 ? cols[b.w2] : 0;
  j.nout = b.nout;
  for (int k = 0; k < b.nout; ++k) {
    const SrcOut& o = b.out[k];
    j.out[k].dst = pk + out_offset(pp, o);
    j.out[k].kind = o.kind; j.out[k].ld = o.ld; j.out[k].gate_H = o.gate_H;
  }
}

static void fill_tensors(const Dims& d, const void* const* wv, SgdPackTable& t) {
  static_assert(kMaxSgdPackTensors == SSCVAE_W_COUNT, "one tensor slot per weight");
  int rows[SSCVAE_W_COUNT], cols[SSCVAE_W_COUNT];
  weight_shapes(d, rows, cols);
  for (int i = 0; i < SSCVAE_W_COUNT; ++i) {
    t.t[i] = SgdPackTensor();
    t.t[i].p = const_cast<float*>(reinterpret_cast<const float*>(wv[i]));
    t.t[i].n = (unsigned long long)rows[i] * cols[i];
  }
}

static int pack_weights_impl(Handle* h, const void* const* wv, char* pk, const uint8_t* dirty, cudaStream_t s) {
  const Dims& d = h->d;
  // dirty == NULL: first pack of this buffer (zero the K/N padding, pack everything); otherwise only the blocks
  // whose fp32 source changed are re-packed (the padding stays zero, frozen weights are skipped)
  for (int i = 0; i < SSCVAE_W_COUNT; ++i) REQUIRE(wv[i] != nullptr, "weight pointer %d is NULL", i);
  std::vector<SrcBlock> bl;
  TRY(source_blocks(d, bl));
  if (!dirty) CUDA_TRY(cudaMemsetAsync(pk, 0, h->pp.total, s));
  SgdPackTable t;                                      // every block below is converted by ONE kernel launch
  fill_tensors(d, wv, t);
  for (const SrcBlock& b : bl)
    if (b.nout > 0 && (!dirty || dirty[b.w] || (b.w2 >= 0 && dirty[b.w2]))) fill_job(d, h->pp, b, pk, t.job[t.n++]);
  return sgd_pack(s, t);
}


// ---- small helpers -----------------------------------------------------------------------------
static inline GemmSeg seg(const bf16* A, int lda, const bf16* B, int ldb, int K) {
  GemmSeg s; s.A = A; s.lda = lda; s.B = B; s.ldb = ldb; s.K = K; return s;
}

// Does the training forward of this shape run as the persistent recurrent kernel (recurrent_fwd.cu)? The backward asks
// the same question: the persistent kernel saves the LSTM state in the row-tiled layout.
static bool persistent_forward(const Dims& d, int B, int N) {
  if (d.cvar) return false;                            // the time-varying conditioning operand runs on the per-launch path
  RecFwdArgs rf = {};
  rf.B = B; rf.T = d.T; rf.H = d.H; rf.Hp = d.Hp; rf.Fp = d.Fp; rf.Zp = d.Zp; rf.Z = d.Z; rf.A = d.A; rf.KX = d.KX; rf.GP = d.GP;
  rf.Ep = d.Ep;
  rf.att.R = B; rf.att.N = N; rf.att.A = d.A; rf.att.Ap = d.Ap; rf.att.F = d.F; rf.att.Fp = d.Fp;
  return recurrent_forward_supported(rf);
}

// The BPTT loop runs as the persistent kernel of recurrent_bwd.cu (it reads either the
// row-tiled or row-major saved state) and the shape fits.
static void fill_rec_bwd_args(const Dims& d, int B, int N, RecBwdArgs& rb) {
  rb = RecBwdArgs();
  rb.B = B; rb.T = d.T; rb.H = d.H; rb.Hp = d.Hp; rb.Fp = d.Fp; rb.Zp = d.Zp; rb.Z = d.Z; rb.Z2p = d.Z2p; rb.A = d.A; rb.Ap = d.Ap;
  rb.KX = d.KX; rb.Gp = d.Gp;
  rb.att.R = B; rb.att.N = N; rb.att.A = d.A; rb.att.Ap = d.Ap; rb.att.F = d.F; rb.att.Fp = d.Fp;
}
static bool persistent_backward(const Dims& d, int B, int N) {
  if (d.cvar) return false;                            // the attribute-grounded prior's d alpha path runs on the per-launch path
  RecBwdArgs rb;
  fill_rec_bwd_args(d, B, N, rb);
  return recurrent_backward_supported(rb);
}

// ---- training forward --------------------------------------------------------------------------
static int train_forward_impl(Handle* h, int B, int N, const char* pk, const void* const* wv, const float* feats,
                              const long long* cap, const float* sent, const float* obj, const float* eps,
                              unsigned long long seed, char* ws, size_t ws_bytes, float* loss, float* kld, cudaStream_t s) {
  const Dims& d = h->d;
  REQUIRE(B > 0 && N > 0, "batch/num_boxes must be positive");
  const bool csent = d.cond && !d.cvar;                // sentiment_vae == 1: the time-invariant sentiment column
  REQUIRE(!csent || sent != nullptr, "sentiment is required when sentiment_vae == 1");
  REQUIRE(!d.cvar || obj != nullptr, "obj_means is required when sentiment_vae == 2");
  const Plan& tp = h->train_plan(B, N);
  if (ws_bytes < tp.total) { set_error("workspace too small: %zu < %zu", ws_bytes, tp.total); return SSCVAE_ERR_WORKSPACE; }
  REQUIRE((reinterpret_cast<uintptr_t>(ws) & 255) == 0 && (reinterpret_cast<uintptr_t>(pk) & 255) == 0,
          "workspace and packed weights must be 256-byte aligned");
  const Plan& pp = h->pp;
  auto W = [&](int i) { return reinterpret_cast<const float*>(wv[i]); };
  auto Pb = [&](const char* n) { return reinterpret_cast<const bf16*>(pk + pp.find(n)->off); };
  auto Pf = [&](const char* n) { return reinterpret_cast<const float*>(pk + pp.find(n)->off); };
  auto Wb = [&](const char* n) { return reinterpret_cast<bf16*>(ws + tp.find(n)->off); };
  auto Wf = [&](const char* n) { return reinterpret_cast<float*>(ws + tp.find(n)->off); };
  auto Wi = [&](const char* n) { return reinterpret_cast<int*>(ws + tp.find(n)->off); };
  auto zero = [&](const char* n) { return cudaMemsetAsync(ws + tp.find(n)->off, 0, tp.find(n)->bytes, s); };
  const int T = d.T, TB = T * B, GP = d.GP, H = d.H, Hp = d.Hp, KX = d.KX, Fp = d.Fp;
  const unsigned long long* seed_dev = reinterpret_cast<const unsigned long long*>(ws + tp.find("seed")->off);
  (void)seed;                                          // copied to `seed_dev` by the caller, in front of the graph

  // operand buffers carry zero padding columns and the zero initial states (updown_cell.py:131-140)
  CUDA_TRY(zero("XA")); CUDA_TRY(zero("XE")); CUDA_TRY(zero("HE")); CUDA_TRY(zero("projb")); CUDA_TRY(zero("ZB"));
  if (d.tied) CUDA_TRY(zero("ob"));

  int* tok = Wi("tok");
  float* tmask = Wf("tmask");
  TRY(boundary_tokens(s, cap, B, d.L, d.pad, d.boundary, tok, tmask, Wf("lengths")));
  TRY(image_prep(s, feats, h->opt_features_bf16, B, N, d.F, Wb("featsb"), Fp, Wf("mask"), Wb("avgb")));
  TRY(scale_rows_f32(s, csent ? sent : nullptr, d.mult, Wf("pm_row"), B));    // prior mean (updown_captioner.py:253)
  TRY(scale_rows_f32(s, csent ? sent : nullptr, 1.0f, Wf("sent"), B));
  if (d.cvar) CUDA_TRY(cudaMemcpyAsync(Wf("objm"), obj, (size_t)B * N * d.Z * sizeof(float), cudaMemcpyDeviceToDevice, s));
  {  // P = W_v x  (attention.py:125), once per image, kept in bf16
    GemmSeg sg = seg(Wb("featsb"), Fp, Pb("wv"), Fp, d.F);
    GemmEpi e; e.tag = "gemm.pre"; e.C16 = Wb("projb"); e.ldc16 = d.Ap;
    TRY(gemm_bf16_tn(s, B * N, d.A, 1, &sg, e));
  }
  TRY(embed_gather_train(s, tok, B, d.L, Pb("embb"), d.Ep, Wb("embb_t")));
  const bool persistent = persistent_forward(d, B, N);
  if (!persistent) {  // teacher-forced embedding block of the attention-LSTM gates for all T at once
    GemmSeg sg = seg(Wb("embb_t"), d.Ep, Pb("w_att_e"), d.Ep, d.E);
    GemmEpi e; e.tag = "gemm.pre"; e.C32 = Wf("gx_att"); e.ldc32 = GP;
    TRY(gemm_bf16_tn(s, TB, GP, 1, &sg, e));
  }
  {  // time-invariant mean-feature block (the biases, kept in reference order, are added by the cell)
    GemmSeg sg = seg(Wb("avgb"), Fp, Pb("w_att_f"), Fp, d.F);
    GemmEpi e; e.tag = "gemm.pre"; e.C32 = Wf("gavg"); e.ldc32 = GP;
    TRY(gemm_bf16_tn(s, B, GP, 1, &sg, e));
  }
  LatentArgs la = {}; la.R = B; la.Z = d.Z; la.Zp = d.Zp; la.sentiment_vae = d.sv; la.prior_var = d.prior_std * d.prior_std;
  la.prior_mean_row = Wf("pm_row"); la.rowmap = nullptr;
  AttnArgs aa = {}; aa.R = B; aa.N = N; aa.A = d.A; aa.Ap = d.Ap; aa.F = d.F; aa.Fp = Fp; aa.rowmap = nullptr;
  aa.proj = Wb("projb"); aa.feats = Wb("featsb"); aa.mask = Wf("mask"); aa.w_a = W(SSCVAE_W_ATT_VEC); aa.ld_q = d.A;
  // ---- the T-step recurrence: one persistent cooperative kernel (recurrent_fwd.cu) when the shape allows it,
  //      otherwise ~10 launches per timestep
  RecFwdArgs rf = {};
  rf.B = B; rf.T = T; rf.H = H; rf.Hp = Hp; rf.Fp = Fp; rf.Zp = d.Zp; rf.Z = d.Z; rf.A = d.A; rf.KX = KX; rf.GP = GP; rf.Ep = d.Ep;
  rf.embb_t = Wb("embb_t"); rf.w_att_e = Pb("w_att_e");
  rf.sentiment_vae = d.sv; rf.prior_var = d.prior_std * d.prior_std;
  rf.w_att_rec = Pb("w_att_rec"); rf.wq = Pb("wq"); rf.w_enc_x = Pb("w_enc_x"); rf.w_enc_hh = Pb("w_enc_hh");
  rf.w_fc = Pb("w_fc"); rf.w_dec_x = Pb("w_dec_x"); rf.w_dec_z = Pb("w_dec_z");
  rf.gavg = Wf("gavg"); rf.b_att = Pf("b_att"); rf.b_enc = Pf("b_enc"); rf.b_dec = Pf("b_dec");
  rf.sent = csent ? sent : nullptr; rf.scol_enc = Pf("scol_enc"); rf.scol_dec = Pf("scol_dec");
  rf.c1 = Wf("c1"); rf.c_enc = Wf("c_enc"); rf.c_dec = Wf("c_dec");
  rf.gates_att = Wf("gates_att"); rf.gates_enc = Wf("gates_enc"); rf.gates_dec = Wf("gates_dec");
  rf.XA = Wb("XA"); rf.XE = Wb("XE"); rf.HE = Wb("HE"); rf.ZB = Wb("ZB");
  rf.q = Wf("q"); rf.b_fc = Pf("b_fc"); rf.eps_in = eps; rf.seed = seed_dev; rf.pm_row = Wf("pm_row");
  rf.mean = Wf("mean"); rf.logvar = Wf("logvar"); rf.eps_out = Wf("eps"); rf.kl_part = Wf("kl_part"); rf.kl = Wf("kl");
  rf.att = aa; rf.alpha = Wf("alpha"); rf.smx = Wf("smx");
  rf.flags = reinterpret_cast<unsigned int*>(ws + tp.find("rf_flags")->off);
  if (persistent) {
    TRY(recurrent_forward(s, rf));
  } else {
    float* acc = Wf("acc");
    for (int t = 0; t < T; ++t) {
      bf16* XA_t = Wb("XA") + (size_t)t * B * 2 * Hp;
      bf16* XA_n = XA_t + (size_t)B * 2 * Hp;
      bf16* XE_t = Wb("XE") + (size_t)t * B * KX;
      bf16* XE_n = (t + 1 < T) ? XE_t + (size_t)B * KX : nullptr;
      bf16* HE_t = Wb("HE") + (size_t)t * B * Hp;
      bf16* HE_n = HE_t + (size_t)B * Hp;
      bf16* ZB_t = Wb("ZB") + (size_t)t * B * d.ZC;
      const size_t rG = (size_t)t * B * d.G, rH = (size_t)t * B * H, rZ = (size_t)t * B * d.Z;
      {  // attention LSTM (updown_cell.py:143-148): gate GEMM, then the cell
        LstmFwdArgs l = {};
        l.R = B; l.H = H; l.add1 = Wf("gx_att") + (size_t)t * B * GP; l.ld1 = GP; l.add2 = Wf("gavg"); l.ld2 = GP;
        l.bias = Pf("b_att");
        l.c_prev = t ? Wf("c1") + rH - (size_t)B * H : nullptr; l.c_out = Wf("c1") + rH; l.gates_out = Wf("gates_att") + rG;
        l.h1_dst = XE_t + Fp; l.ld_h1 = KX; l.h2_dst = XA_n; l.ld_h2 = 2 * Hp;
        l.acc = acc; l.ld_acc = GP; l.perm = 1;
        GemmSeg sg = seg(XA_t, 2 * Hp, Pb("w_att_rec"), 2 * Hp, 2 * Hp);
        GemmEpi e; e.tag = "gemm.step"; e.C32 = acc; e.ldc32 = GP;
        TRY(gemm_bf16_tn(s, B, GP, 1, &sg, e));
        TRY(lstm_forward(s, l));
      }
      {  // query projection + fused region attention (attention.py:69-93, updown_cell.py:156)
        GemmSeg sg = seg(XE_t + Fp, KX, Pb("wq"), Hp, Hp);
        GemmEpi e; e.tag = "gemm.step"; e.C32 = Wf("q") + (size_t)t * B * d.A; e.ldc32 = d.A;
        TRY(gemm_bf16_tn(s, B, d.A, 1, &sg, e));
        aa.q = Wf("q") + (size_t)t * B * d.A;
        TRY(attention_forward(s, aa, Wf("alpha") + (size_t)t * B * N, Wf("smx") + (size_t)t * B * N, XE_t, KX));
        // attribute-grounded prior (updown_cell.py:160-174): prior mean of this step from the attention weights; it is
        // also the conditioning block c of the two LSTM inputs below, stored next to z
        if (d.cvar) {
          TRY(prior_mean_forward(s, Wf("alpha") + (size_t)t * B * N, Wf("objm"), nullptr, B, N, d.Z, Wf("pm") + rZ,
                                 ZB_t + d.Zp, d.ZC, d.cond));
          la.prior_mean_full = Wf("pm") + rZ;
        }
      }
      {  // posterior (encoder) LSTM + latent heads + reparameterised sample (updown_cell.py:176-208)
        LstmFwdArgs l = {};
        l.R = B; l.H = H; l.bias = Pf("b_enc");
        if (csent) { l.sent = sent; l.scol = Pf("scol_enc"); }
        l.c_prev = t ? Wf("c_enc") + rH - (size_t)B * H : nullptr; l.c_out = Wf("c_enc") + rH;
        l.gates_out = Wf("gates_enc") + rG; l.h1_dst = HE_n; l.ld_h1 = Hp;
        l.acc = acc; l.ld_acc = GP; l.perm = 1;
        GemmSeg sg[3] = {seg(XE_t, KX, Pb("w_enc_x"), KX, KX), seg(HE_t, Hp, Pb("w_enc_hh"), Hp, Hp), GemmSeg()};
        if (d.cvar) sg[2] = seg(ZB_t + d.Zp, d.ZC, Pb("w_enc_c"), d.Cp, d.Cp);
        GemmEpi e; e.tag = "gemm.step"; e.C32 = acc; e.ldc32 = GP;
        TRY(gemm_bf16_tn(s, B, GP, d.cvar ? 3 : 2, sg, e));
        TRY(lstm_forward(s, l));
        GemmSeg sf = seg(HE_n, Hp, Pb("w_fc"), Hp, Hp);
        GemmEpi ef; ef.tag = "gemm.step"; ef.C32 = Wf("ml"); ef.ldc32 = d.Z2;
        TRY(gemm_bf16_tn(s, B, d.Z2, 1, &sf, ef));
        TRY(latent_forward_train(s, la, Wf("ml"), d.Z2, Pf("b_fc"), eps ? eps + rZ : nullptr, seed_dev, (unsigned long long)t,
                                 Wf("mean") + rZ, Wf("logvar") + rZ, Wf("eps") + rZ, ZB_t, d.ZC, Wf("kl") + (size_t)t * B));
      }
      {  // language (decoder) LSTM (updown_cell.py:211-229)
        LstmFwdArgs l = {};
        l.R = B; l.H = H; l.bias = Pf("b_dec");
        if (csent) { l.sent = sent; l.scol = Pf("scol_dec"); }
        l.c_prev = t ? Wf("c_dec") + rH - (size_t)B * H : nullptr; l.c_out = Wf("c_dec") + rH;
        l.gates_out = Wf("gates_dec") + rG; l.h1_dst = XA_n + Hp; l.ld_h1 = 2 * Hp;
        if (XE_n) { l.h2_dst = XE_n + Fp + Hp; l.ld_h2 = KX; }
        l.acc = acc; l.ld_acc = GP; l.perm = 1;
        GemmSeg sg[2] = {seg(XE_t, KX, Pb("w_dec_x"), KX, KX), seg(ZB_t, d.ZC, Pb("w_dec_z"), d.ZC, d.ZC)};
        GemmEpi e; e.tag = "gemm.step"; e.C32 = acc; e.ldc32 = GP;
        TRY(gemm_bf16_tn(s, B, GP, 2, sg, e));
        TRY(lstm_forward(s, l));
      }
    }
  }
  // output head over all T*B rows at once (updown_captioner.py:444-445) with the masked cross entropy
  // (updown_captioner.py:457-466) fused: per-row max / sum-exp / target logit come out of the vocabulary GEMM's epilogue
  const bf16* hdec_all = Wb("XA") + (size_t)B * 2 * Hp + Hp;
  TRY(ce_prepare(s, tok, B, d.L, tmask, Wf("lengths"), nullptr, Wi("tgt_row"), nullptr));
  RowStatsEpi rs;
  rs.mode = 1; rs.st_max = Wf("rs_max"); rs.st_sum = Wf("rs_sum"); rs.st_arg = Wi("rs_arg");
  rs.target = Wi("tgt_row"); rs.tgt_logit = Wf("rs_tgt");
  if (d.tied) {
    GemmSeg sg = seg(hdec_all, 2 * Hp, Pb("w_out"), Hp, Hp);
    GemmEpi e; e.tag = "gemm.head"; e.bias = W(SSCVAE_W_OUT_PROJ_B); e.act = 1; e.C32 = Wf("o32"); e.ldc32 = d.E; e.C16 = Wb("ob"); e.ldc16 = d.Ep;
    TRY(gemm_bf16_tn(s, TB, d.E, 1, &sg, e));
    GemmSeg sv = seg(Wb("ob"), d.Ep, Pb("embb"), d.Ep, d.E);
    GemmEpi ev; ev.tag = "gemm.head"; ev.rs = &rs;
    if (d.debug_logits) { ev.C32 = Wf("logits"); ev.ldc32 = d.V; }
    TRY(gemm_bf16_tn(s, TB, d.V, 1, &sv, ev));
  } else {
    GemmSeg sg = seg(hdec_all, 2 * Hp, Pb("w_out"), Hp, Hp);
    GemmEpi e; e.tag = "gemm.head"; e.bias = W(SSCVAE_W_OUT_PROJ_B); e.rs = &rs;
    if (d.debug_logits) { e.C32 = Wf("logits"); e.ldc32 = d.V; }
    TRY(gemm_bf16_tn(s, TB, d.V, 1, &sg, e));
  }
  TRY(ce_merge(s, rs.st_max, rs.st_sum, rs.st_arg, gemm_rowstats_tiles(d.V), TB, Wf("rs_tgt"), Wf("lse"), Wf("nll")));
  TRY(loss_reduce(s, Wf("nll"), Wf("kl"), tmask, Wf("lengths"), T, B, loss, kld));
  return 0;
}

// ---- training backward (BPTT) ------------------------------------------------------------------
static int train_backward_impl(Handle* h, int B, int N, const char* pk, const void* const* wv, char* ws, size_t ws_bytes,
                               const float* gloss, const float* gkld, void* const* gv, void* const* events,
                               cudaStream_t s) {
  const Dims& d = h->d;
  const Plan& tp = h->train_plan(B, N);
  if (ws_bytes < tp.total) { set_error("workspace too small: %zu < %zu", ws_bytes, tp.total); return SSCVAE_ERR_WORKSPACE; }
  const Plan& pp = h->pp;
  auto W = [&](int i) { return reinterpret_cast<const float*>(wv[i]); };
  auto Gr = [&](int i) { return reinterpret_cast<float*>(gv[i]); };
  auto Pb = [&](const char* n) { return reinterpret_cast<const bf16*>(pk + pp.find(n)->off); };
  auto Wb = [&](const char* n) { return reinterpret_cast<bf16*>(ws + tp.find(n)->off); };
  auto Wf = [&](const char* n) { return reinterpret_cast<float*>(ws + tp.find(n)->off); };
  auto Wi = [&](const char* n) { return reinterpret_cast<int*>(ws + tp.find(n)->off); };
  auto zero = [&](const char* n) { return cudaMemsetAsync(ws + tp.find(n)->off, 0, tp.find(n)->bytes, s); };
  // While the call is being captured into a graph the record becomes an EXTERNAL event-record node: every replay
  // re-records the event and streams outside the graph (the all-reduce side stream) can wait on it.
  cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
  CUDA_TRY(cudaStreamIsCapturing(s, &cap));
  auto event = [&](int g) -> int {
    if (events && events[g])
      CUDA_TRY(cudaEventRecordWithFlags(reinterpret_cast<cudaEvent_t>(events[g]), s,
                                        cap == cudaStreamCaptureStatusActive ? cudaEventRecordExternal : cudaEventRecordDefault));
    return 0;
  };
  const int T = d.T, TB = T * B, TBp = round_up(TB, kPad), G = d.G, Gp = d.Gp, H = d.H, Hp = d.Hp, KX = d.KX, Fp = d.Fp;
  const int E = d.E, F = d.F, A = d.A, Z = d.Z, V = d.V, c = d.cond, Bp = round_up(B, kPad), BN = B * N, BNp = round_up(BN, kPad);
  const int* tok = Wi("tok");
  const float* tmask = Wf("tmask");

  const int tiled = persistent_forward(d, B, N) ? 1 : 0;
  const bool pbwd = h->opt_persistent_bwd && persistent_backward(d, B, N);
  if (pbwd) {
    const char* zl[] = {"dc1", "dc_enc", "dc_dec", "dG_att", "dG_enc", "dG_dec", "dqb", "dml", "du"};
    for (const char* n : zl) CUDA_TRY(zero(n));
  } else {
    const char* zl[] = {"dc1", "dc_enc", "dc_dec", "dXEH0", "dXEH1", "dXA0", "dXA1",
                        "dG_att", "dG_enc", "dG_dec", "dqb"};
    for (const char* n : zl) CUDA_TRY(zero(n));
  }
  if (d.tied) CUDA_TRY(zero("dpreo"));

  // ---- head: d logits, d h_dec from the vocabulary projection
  // d logits = g_b (softmax - onehot) (allennlp sequence_cross_entropy_with_logits, average=None, x len_b): the vocabulary
  // GEMM is recomputed and its epilogue writes the bf16 gradient operand directly (the forward kept only lse per row)
  const bf16* hdec_all = Wb("XA") + (size_t)B * 2 * Hp + Hp;     // h_dec_t, t = 0..T-1, ld 2Hp
  TRY(ce_prepare(s, tok, B, d.L, tmask, Wf("lengths"), gloss, Wi("tgt_row"), Wf("gcoef")));
  if (d.Vp > V) CUDA_TRY(cudaMemset2DAsync(Wb("dlogits") + V, (size_t)d.Vp * 2, 0, (size_t)(d.Vp - V) * 2, (size_t)TB, s));
  {
    RowStatsEpi rs;
    rs.mode = 2; rs.target = Wi("tgt_row"); rs.lse = Wf("lse"); rs.gcoef = Wf("gcoef");
    GemmEpi e; e.tag = "gemm.head_bwd"; e.rs = &rs; e.C16 = Wb("dlogits"); e.ldc16 = d.Vp;
    if (d.tied) {
      GemmSeg sv = seg(Wb("ob"), d.Ep, Pb("embb"), d.Ep, E);
      TRY(gemm_bf16_tn(s, TB, V, 1, &sv, e));
    } else {
      GemmSeg sg = seg(hdec_all, 2 * Hp, Pb("w_out"), Hp, Hp);
      e.bias = W(SSCVAE_W_OUT_PROJ_B);
      TRY(gemm_bf16_tn(s, TB, V, 1, &sg, e));
    }
  }
  if (d.tied) {
    GemmSeg sg = seg(Wb("dlogits"), d.Vp, Pb("embT"), d.Vp, V);
    GemmEpi e; e.tag = "gemm.head_bwd"; e.dtanh = Wf("o32"); e.ldd = E; e.C16 = Wb("dpreo"); e.ldc16 = d.Ep;
    TRY(gemm_bf16_tn(s, TB, E, 1, &sg, e));
    GemmSeg s2 = seg(Wb("dpreo"), d.Ep, Pb("w_outT"), d.Ep, E);
    GemmEpi e2; e2.tag = "gemm.head_bwd"; e2.C32 = Wf("dhead"); e2.ldc32 = H;
    TRY(gemm_bf16_tn(s, TB, H, 1, &s2, e2));
  } else {
    GemmSeg sg = seg(Wb("dlogits"), d.Vp, Pb("w_outT"), d.Vp, V);
    GemmEpi e; e.tag = "gemm.head_bwd"; e.C32 = Wf("dhead"); e.ldc32 = H;
    TRY(gemm_bf16_tn(s, TB, H, 1, &sg, e));
  }
  // head weight gradients are final before the time loop starts
  TransposeJobList tj;
  TRY(tj.add(hdec_all, TB, H, 2 * Hp, Wb("hdecTc"), TBp));
  if (Gr(SSCVAE_W_OUT_PROJ_W) || Gr(SSCVAE_W_OUT_PROJ_B)) {
    if (d.tied) TRY(tj.add(Wb("dpreo"), TB, E, d.Ep, Wb("dpreoT"), TBp));
    else TRY(tj.add(Wb("dlogits"), TB, V, d.Vp, Wb("dlogitsT"), TBp));
  }
  TRY(transpose_bf16_jobs(s, tj));
  if (d.tied) {
    if (Gr(SSCVAE_W_OUT_PROJ_W)) {
      GemmSeg sg = seg(Wb("dpreoT"), TBp, Wb("hdecTc"), TBp, TB);
      GemmEpi e; e.tag = "gemm.head_bwd"; e.C32 = Gr(SSCVAE_W_OUT_PROJ_W); e.ldc32 = H;
      TRY(gemm_bf16_tn(s, E, H, 1, &sg, e));
    }
    if (Gr(SSCVAE_W_OUT_PROJ_B)) TRY(rowsum_bf16(s, Wb("dpreoT"), E, TB, TBp, Gr(SSCVAE_W_OUT_PROJ_B), 0));
  } else {
    if (Gr(SSCVAE_W_OUT_PROJ_W)) {
      GemmSeg sg = seg(Wb("dlogitsT"), TBp, Wb("hdecTc"), TBp, TB);
      GemmEpi e; e.tag = "gemm.head_bwd"; e.C32 = Gr(SSCVAE_W_OUT_PROJ_W); e.ldc32 = H;
      TRY(gemm_bf16_tn(s, V, H, 1, &sg, e));
    }
    if (Gr(SSCVAE_W_OUT_PROJ_B)) TRY(rowsum_bf16(s, Wb("dlogitsT"), V, TB, TBp, Gr(SSCVAE_W_OUT_PROJ_B), 0));
  }
  // With the persistent BPTT kernel the head group's event is recorded BEHIND the loop: the all-reduce it releases must not
  // share the GPU with a cooperative kernel whose resident CTAs spin on flags that its not-yet-resident CTAs have to set.
  // NCCL's CTAs also need to be co-resident with each other, and two such kernels placed at the same time can each hold
  // the SMs the other still needs (seen at 8 GPUs: every rank stuck behind the first warm-up steps; at 2 GPUs NCCL uses
  // too few CTAs to interleave with the placement of the 148). The all-reduce of the head bucket then overlaps the
  // weight-gradient GEMMs like the other buckets.
  const bool event0_late = pbwd;
  if (!event0_late) TRY(event(0));

  // ---- reverse time loop
  LatentArgs la = {}; la.R = B; la.Z = Z; la.Zp = d.Zp; la.sentiment_vae = d.sv; la.prior_var = d.prior_std * d.prior_std;
  la.prior_mean_row = Wf("pm_row"); la.rowmap = nullptr;
  AttnArgs aa = {}; aa.R = B; aa.N = N; aa.A = A; aa.Ap = d.Ap; aa.F = F; aa.Fp = Fp; aa.rowmap = nullptr;
  aa.proj = Wb("projb"); aa.feats = Wb("featsb"); aa.mask = Wf("mask"); aa.w_a = W(SSCVAE_W_ATT_VEC); aa.ld_q = A;
  float* dXE[2] = {Wf("dXEH0"), Wf("dXEH1")};             // [d xhat | d h1 | d h_dec_{t-1} | d h_enc_{t-1}]
  const int KXH = KX + Hp + d.Cp, KXZ = KX + d.ZC;      // [.. | d h_enc_{t-1} | d c (encoder)] and [.. | d z | d c (decoder)]
  float* dXA[2] = {Wf("dXA0"), Wf("dXA1")};
  if (pbwd) {  // the whole reverse time loop in one persistent cooperative kernel (recurrent_bwd.cu)
    RecBwdArgs rb;
    fill_rec_bwd_args(d, B, N, rb);
    rb.sentiment_vae = d.sv; rb.prior_var = d.prior_std * d.prior_std; rb.tiled = tiled;
    rb.w_dec_xzT = Pb("w_dec_xzT"); rb.w_enc_xhT = Pb("w_enc_xhT"); rb.w_att_recT = Pb("w_att_recT"); rb.w_fcT = Pb("w_fcT"); rb.wqT = Pb("wqT");
    rb.gates_att = Wf("gates_att"); rb.gates_enc = Wf("gates_enc"); rb.gates_dec = Wf("gates_dec");
    rb.c1 = Wf("c1"); rb.c_enc = Wf("c_enc"); rb.c_dec = Wf("c_dec");
    rb.mean = Wf("mean"); rb.logvar = Wf("logvar"); rb.eps = Wf("eps"); rb.pm_row = Wf("pm_row");
    rb.q = Wf("q"); rb.smx = Wf("smx"); rb.dhead = Wf("dhead"); rb.gkld = gkld; rb.tmask = tmask;
    rb.dc1 = Wf("dc1"); rb.dc_enc = Wf("dc_enc"); rb.dc_dec = Wf("dc_dec");
    rb.dG_att = Wb("dG_att"); rb.dG_enc = Wb("dG_enc"); rb.dG_dec = Wb("dG_dec"); rb.dml = Wb("dml"); rb.dqb = Wb("dqb"); rb.du = Wf("du");
    rb.dXEA = Wf("rb_dXEA"); rb.dXEB = Wf("rb_dXEB"); rb.dXA = Wf("rb_dXA"); rb.dzp = Wf("rb_dzp");
    rb.dhe_fc = Wf("dhenc_fc"); rb.dh1q = Wf("dh1_q");
    rb.att = aa;
    rb.flags = reinterpret_cast<unsigned int*>(ws + tp.find("rb_flags")->off);
    rb.rows = Wi("rb_rows");
    TRY(recurrent_backward(s, rb));
    TRY(event(0));
  }
  for (int t = T - 1; t >= 0 && !pbwd; --t) {
    const int cur = t & 1, nxt = cur ^ 1;
    const size_t rG = (size_t)t * B * G, rH = (size_t)t * B * H, rGp = (size_t)t * B * Gp, rZ = (size_t)t * B * Z;
    bf16* dGd = Wb("dG_dec") + rGp; bf16* dGe = Wb("dG_enc") + rGp; bf16* dGa = Wb("dG_att") + rGp;
    {  // decoder LSTM: d h_dec_t = head + enc/dec inputs of step t+1 + attention-LSTM input of step t+1
      LstmBwdArgs l = {};
      l.R = B; l.H = H;
      l.dh[0] = Wf("dhead") + rH; l.ld_dh[0] = H;
      l.dh[1] = dXE[nxt] + Fp + Hp; l.ld_dh[1] = KXH;
      l.dh[2] = dXA[nxt] + Hp; l.ld_dh[2] = 2 * Hp;
      l.dc_in = Wf("dc_dec"); l.dc_prev = Wf("dc_dec");
      l.gates = Wf("gates_dec") + rG; l.c = Wf("c_dec") + rH; l.c_prev = t ? Wf("c_dec") + rH - (size_t)B * H : nullptr;
      l.dgates = dGd; l.ld_dg = Gp; l.tiled = tiled;
      TRY(lstm_backward(s, l));
    }
    {  // decoder part of d[xhat|h1|h_dec_{t-1}] and d z in ONE GEMM (N = KX+Zp), then d mean / d log_var
       // (+ KL gradient) -> d h_enc
      GemmSeg sg = seg(dGd, Gp, Pb("w_dec_xzT"), Gp, G);
      GemmEpi e; e.tag = "gemm.step_bwd"; e.C32 = Wf("dXEZ"); e.ldc32 = KXZ;
      TRY(gemm_bf16_tn(s, B, KXZ, 1, &sg, e));
      bf16* dml_t = Wb("dml") + (size_t)t * B * d.Z2p;
      if (d.cvar) { la.prior_mean_full = Wf("pm") + rZ; la.dpm_out = Wf("dpm"); }
      TRY(latent_backward(s, la, Wf("dXEZ") + KX, KXZ, Wf("eps") + rZ, Wf("mean") + rZ, Wf("logvar") + rZ, gkld,
                          tmask + (size_t)t * B, dml_t, d.Z2p));
      GemmSeg s2 = seg(dml_t, d.Z2p, Pb("w_fcT"), d.Z2p, d.Z2);
      GemmEpi e2; e2.tag = "gemm.step_bwd"; e2.C32 = Wf("dhenc_fc"); e2.ldc32 = H;
      TRY(gemm_bf16_tn(s, B, H, 1, &s2, e2));
    }
    {  // encoder LSTM
      LstmBwdArgs l = {};
      l.R = B; l.H = H;
      l.dh[0] = Wf("dhenc_fc"); l.ld_dh[0] = H;
      l.dh[1] = dXE[nxt] + KX; l.ld_dh[1] = KXH;
      l.dc_in = Wf("dc_enc"); l.dc_prev = Wf("dc_enc");
      l.gates = Wf("gates_enc") + rG; l.c = Wf("c_enc") + rH; l.c_prev = t ? Wf("c_enc") + rH - (size_t)B * H : nullptr;
      l.dgates = dGe; l.ld_dg = Gp; l.tiled = tiled;
      TRY(lstm_backward(s, l));
    }
    {  // encoder part of d[xhat|h1|h_dec_{t-1}] (added onto the decoder part) and d h_enc_{t-1}: one GEMM, N = KX+Hp
      GemmSeg sg = seg(dGe, Gp, Pb("w_enc_xhT"), Gp, G);
      GemmEpi e; e.tag = "gemm.step_bwd"; e.C32 = dXE[cur]; e.ldc32 = KXH;
      e.add1 = Wf("dXEZ"); e.ld1 = KXZ; e.add1_cols = KX;
      TRY(gemm_bf16_tn(s, B, KXH, 1, &sg, e));
    }
    {  // fused attention backward, then d h1 through the query projection
      aa.q = Wf("q") + (size_t)t * B * A;
      bf16* dq_t = Wb("dqb") + (size_t)t * B * d.Ap;
      if (d.cvar) {  // d prior_mean = KL term + the two LSTMs' d c  ->  extra d alpha_n = objm_n . d prior_mean
        TRY(prior_mean_backward(s, B, N, Z, c, Wf("dpm"), Wf("dXEZ") + KX + d.Zp, KXZ, dXE[cur] + KX + Hp, KXH, Wf("objm"),
                                Wf("dalpha_x")));
        aa.dalpha_extra = Wf("dalpha_x");
      }
      TRY(attention_backward(s, aa, Wf("smx") + (size_t)t * B * N, dXE[cur], KXH, dq_t, d.Ap, Wf("du") + (size_t)t * B * N));
      GemmSeg sg = seg(dq_t, d.Ap, Pb("wqT"), d.Ap, A);
      GemmEpi e; e.tag = "gemm.step_bwd"; e.C32 = Wf("dh1_q"); e.ldc32 = H;
      TRY(gemm_bf16_tn(s, B, H, 1, &sg, e));
    }
    {  // attention LSTM
      LstmBwdArgs l = {};
      l.R = B; l.H = H;
      l.dh[0] = dXE[cur] + Fp; l.ld_dh[0] = KXH;
      l.dh[1] = Wf("dh1_q"); l.ld_dh[1] = H;
      l.dh[2] = dXA[nxt]; l.ld_dh[2] = 2 * Hp;
      l.dc_in = Wf("dc1"); l.dc_prev = Wf("dc1");
      l.gates = Wf("gates_att") + rG; l.c = Wf("c1") + rH; l.c_prev = t ? Wf("c1") + rH - (size_t)B * H : nullptr;
      l.dgates = dGa; l.ld_dg = Gp; l.tiled = tiled;
      TRY(lstm_backward(s, l));
      GemmSeg sg = seg(dGa, Gp, Pb("w_att_recT"), Gp, G);
      GemmEpi e; e.tag = "gemm.step_bwd"; e.C32 = dXA[cur]; e.ldc32 = 2 * Hp;
      TRY(gemm_bf16_tn(s, B, 2 * Hp, 1, &sg, e));
    }
  }

  // ---- weight gradients: one GEMM problem per weight block over all T*B rows (K = T*B). Per gradient group: one
  //      launch transposes the group's operands, one grouped GEMM launch computes all its weight blocks (the blocks of
  //      one LSTM share the transposed gate-gradient operand dGT), then the bias sums and the W_hh copy.
  bf16* dGT = Wb("dGT");
  GemmProblem pb[kMaxGemmProblems];
  int np = 0;
  auto wgrad_add = [&](const bf16* AT, int M, const bf16* BT, int Ncols, int K, int ldk, float* C, int ldc) -> int {
    if (!C) return 0;
    REQUIRE(np < kMaxGemmProblems, "weight-gradient group exceeds %d GEMM problems", kMaxGemmProblems);
    pb[np++] = GemmProblem{AT, ldk, BT, ldk, K, M, Ncols, C, ldc};
    return 0;
  };
  auto wgrad_launch = [&]() -> int {
    const int n = np;
    np = 0;
    return gemm_bf16_tn_grouped(s, n, pb, "gemm.wgrad");
  };
  // b_ih and b_hh get the same gradient (both are added to the gates): one row sum, copied
  auto bias_pair = [&](const bf16* dGT_, int ib, int ih) -> int {
    float* g1 = Gr(ib); float* g2 = Gr(ih);
    if (!g1 && !g2) return 0;
    TRY(rowsum_bf16(s, dGT_, G, TB, TBp, g1 ? g1 : g2, 0));
    if (g1 && g2) CUDA_TRY(cudaMemcpyAsync(g2, g1, (size_t)G * sizeof(float), cudaMemcpyDeviceToDevice, s));
    return 0;
  };
  // The forward folds W_hh onto the W_ih column block that multiplies the same operand (packed weights), so the two
  // gradients are one product: computed into W_ih's block when both are wanted and copied to W_hh afterwards (hh_copy:
  // column `col` of W_ih, row pitch ld_ih), otherwise straight into the one that is wanted.
  auto hh_pair = [&](const bf16* BT, int ih, int hh) -> int {
    if (Gr(ih)) return 0;                               // W_ih's block is a problem of the group already
    return wgrad_add(dGT, G, BT, H, TB, TBp, Gr(hh), H);
  };
  auto hh_copy = [&](int ih, int col, int ld_ih, int hh) -> int {
    if (Gr(ih) && Gr(hh))
      CUDA_TRY(cudaMemcpy2DAsync(Gr(hh), (size_t)H * sizeof(float), Gr(ih) + col, (size_t)ld_ih * sizeof(float),
                                 (size_t)H * sizeof(float), G, cudaMemcpyDeviceToDevice, s));
    return 0;
  };
  auto any = [&](std::initializer_list<int> ids) { for (int i : ids) if (gv[i]) return true; return false; };
  const bf16* xhatT = Wb("XET");                                                  // xhat_t, h1_t, h_dec_{t-1}
  const bf16* h1T = Wb("XET") + (size_t)Fp * TBp;
  const bf16* hdecpT = Wb("XET") + (size_t)(Fp + Hp) * TBp;
  const bf16* condT = Wb("ZBT") + (size_t)d.Zp * TBp;   // z_t (and, sentiment_vae == 2, the conditioning block c_t behind it)
  const float* sentv = Wf("sent");
  const int ldE = F + 2 * H + c, ldD = F + 2 * H + c + Z, ldA = E + F + 2 * H;

  // group 1: decoder LSTM. W_ih column blocks [xhat | h1 | h_dec | cond | z]; W_hh shares the h_dec operand.
  TRY(tj.add(Wb("XE"), TB, KX, KX, Wb("XET"), TBp));
  if (Gr(SSCVAE_W_DEC_IH) || (d.cvar && Gr(SSCVAE_W_ENC_IH))) TRY(tj.add(Wb("ZB"), TB, d.ZC, d.ZC, Wb("ZBT"), TBp));
  const bool dec = any({SSCVAE_W_DEC_IH, SSCVAE_W_DEC_HH, SSCVAE_W_DEC_BIH, SSCVAE_W_DEC_BHH});
  if (dec) TRY(tj.add(Wb("dG_dec"), TB, G, Gp, dGT, TBp));
  TRY(transpose_bf16_jobs(s, tj));
  if (dec) {
    float* g = Gr(SSCVAE_W_DEC_IH);
    if (g) {
      TRY(wgrad_add(dGT, G, xhatT, F, TB, TBp, g, ldD));
      TRY(wgrad_add(dGT, G, h1T, H, TB, TBp, g + F, ldD));
      TRY(wgrad_add(dGT, G, hdecpT, H, TB, TBp, g + F + H, ldD));
      TRY(wgrad_add(dGT, G, Wb("ZBT"), Z, TB, TBp, g + F + 2 * H + c, ldD));
      if (d.cvar) TRY(wgrad_add(dGT, G, condT, c, TB, TBp, g + F + 2 * H, ldD));
    }
    TRY(hh_pair(hdecpT, SSCVAE_W_DEC_IH, SSCVAE_W_DEC_HH));
    TRY(wgrad_launch());
    if (g && c && !d.cvar) TRY(rowdot_bf16(s, dGT, G, TB, TBp, sentv, B, g + F + 2 * H, ldD));
    TRY(bias_pair(dGT, SSCVAE_W_DEC_BIH, SSCVAE_W_DEC_BHH));
    TRY(hh_copy(SSCVAE_W_DEC_IH, F + H, ldD, SSCVAE_W_DEC_HH));
  }
  TRY(event(1));

  // group 2: encoder LSTM + latent heads
  const bool enc = any({SSCVAE_W_ENC_IH, SSCVAE_W_ENC_HH, SSCVAE_W_ENC_BIH, SSCVAE_W_ENC_BHH});
  const bool fc = any({SSCVAE_W_FC_MEAN_W, SSCVAE_W_FC_MEAN_B, SSCVAE_W_FC_LOGVAR_W, SSCVAE_W_FC_LOGVAR_B});
  if (enc) {
    TRY(tj.add(Wb("dG_enc"), TB, G, Gp, dGT, TBp));
    if (Gr(SSCVAE_W_ENC_HH)) TRY(tj.add(Wb("HE"), TB, Hp, Hp, Wb("HETp"), TBp));             // h_enc_{t-1}
  }
  if (fc) {
    TRY(tj.add(Wb("dml"), TB, d.Z2p, d.Z2p, Wb("dmlT"), TBp));
    TRY(tj.add(Wb("HE") + (size_t)B * Hp, TB, Hp, Hp, Wb("HETc"), TBp));                     // h_enc_t
  }
  TRY(transpose_bf16_jobs(s, tj));
  const bf16* dmT = Wb("dmlT");
  const bf16* dlT = Wb("dmlT") + (size_t)Z * TBp;
  float* ge = enc ? Gr(SSCVAE_W_ENC_IH) : nullptr;
  if (ge) {
    TRY(wgrad_add(dGT, G, xhatT, F, TB, TBp, ge, ldE));
    TRY(wgrad_add(dGT, G, h1T, H, TB, TBp, ge + F, ldE));
    TRY(wgrad_add(dGT, G, hdecpT, H, TB, TBp, ge + F + H, ldE));
    if (d.cvar) TRY(wgrad_add(dGT, G, condT, c, TB, TBp, ge + F + 2 * H, ldE));
  }
  if (enc) TRY(wgrad_add(dGT, G, Wb("HETp"), H, TB, TBp, Gr(SSCVAE_W_ENC_HH), H));
  if (fc) {
    TRY(wgrad_add(dmT, Z, Wb("HETc"), H, TB, TBp, Gr(SSCVAE_W_FC_MEAN_W), H));
    TRY(wgrad_add(dlT, Z, Wb("HETc"), H, TB, TBp, Gr(SSCVAE_W_FC_LOGVAR_W), H));
  }
  TRY(wgrad_launch());
  if (ge && c && !d.cvar) TRY(rowdot_bf16(s, dGT, G, TB, TBp, sentv, B, ge + F + 2 * H, ldE));
  if (enc) TRY(bias_pair(dGT, SSCVAE_W_ENC_BIH, SSCVAE_W_ENC_BHH));
  if (fc && Gr(SSCVAE_W_FC_MEAN_B)) TRY(rowsum_bf16(s, dmT, Z, TB, TBp, Gr(SSCVAE_W_FC_MEAN_B), 0));
  if (fc && Gr(SSCVAE_W_FC_LOGVAR_B)) TRY(rowsum_bf16(s, dlT, Z, TB, TBp, Gr(SSCVAE_W_FC_LOGVAR_B), 0));
  TRY(event(2));

  // group 3: attention LSTM. W_ih column blocks [emb | avg | h1 | h_dec]; W_hh shares the h1 operand.
  const bool need_demb = !d.tied && Gr(SSCVAE_W_EMBEDDING);
  if (need_demb || any({SSCVAE_W_ATT_IH, SSCVAE_W_ATT_HH, SSCVAE_W_ATT_BIH, SSCVAE_W_ATT_BHH})) {
    const bf16* h1pT = Wb("XAT");                                                 // h1_{t-1}, h_dec_{t-1}
    const bf16* hdecp2T = Wb("XAT") + (size_t)Hp * TBp;
    float* g = Gr(SSCVAE_W_ATT_IH);
    // mean-feature block: the operand is constant over time, so sum the gate gradients over t first
    if (g) TRY(timesum_bf16(s, Wb("dG_att"), T, B, G, Gp, Wb("dGsum"), Gp));
    TRY(tj.add(Wb("dG_att"), TB, G, Gp, dGT, TBp));
    TRY(tj.add(Wb("XA"), TB, 2 * Hp, 2 * Hp, Wb("XAT"), TBp));
    if (g) {
      TRY(tj.add(Wb("embb_t"), TB, d.Ep, d.Ep, Wb("embT_t"), TBp));
      TRY(tj.add(Wb("dGsum"), B, G, Gp, Wb("dGsumT"), Bp));
      TRY(tj.add(Wb("avgb"), B, Fp, Fp, Wb("avgT"), Bp));
    }
    TRY(transpose_bf16_jobs(s, tj));
    if (g) {
      TRY(wgrad_add(dGT, G, Wb("embT_t"), E, TB, TBp, g, ldA));
      TRY(wgrad_add(Wb("dGsumT"), G, Wb("avgT"), F, B, Bp, g + E, ldA));
      TRY(wgrad_add(dGT, G, h1pT, H, TB, TBp, g + E + F, ldA));
      TRY(wgrad_add(dGT, G, hdecp2T, H, TB, TBp, g + E + F + H, ldA));
    }
    TRY(hh_pair(h1pT, SSCVAE_W_ATT_IH, SSCVAE_W_ATT_HH));
    TRY(wgrad_launch());
    TRY(bias_pair(dGT, SSCVAE_W_ATT_BIH, SSCVAE_W_ATT_BHH));
    TRY(hh_copy(SSCVAE_W_ATT_IH, E + F, ldA, SSCVAE_W_ATT_HH));
    if (need_demb) {  // learned embedding (untied): d emb rows = dG_att W_att_ih[:, :E], scattered by token id
      GemmSeg sg = seg(Wb("dG_att"), Gp, Pb("w_att_eT"), Gp, G);
      GemmEpi e; e.tag = "gemm.wgrad"; e.C32 = Wf("dxemb"); e.ldc32 = E;
      TRY(gemm_bf16_tn(s, TB, E, 1, &sg, e));
      CUDA_TRY(cudaMemsetAsync(Gr(SSCVAE_W_EMBEDDING), 0, (size_t)V * E * sizeof(float), s));
      TRY(embed_scatter_add(s, tok, B, d.L, d.pad, Wf("dxemb"), E, E, Gr(SSCVAE_W_EMBEDDING)));
    }
  }
  TRY(event(3));

  // group 4: attention module
  if (Gr(SSCVAE_W_IMAGE_PROJ) || Gr(SSCVAE_W_ATT_VEC)) {
    // d P and d w_a for all timesteps at once (the per-step kernel only kept the score gradients d u)
    aa.q = Wf("q");
    TRY(attention_backward_deferred(s, aa, T, Wf("q"), Wf("du"), Wf("dproj_acc"), Wf("dwa_acc")));
  }
  if (Gr(SSCVAE_W_QUERY_PROJ)) TRY(tj.add(Wb("dqb"), TB, d.Ap, d.Ap, Wb("dqT"), TBp));
  if (Gr(SSCVAE_W_IMAGE_PROJ)) {
    TRY(tj.add(Wb("featsb"), BN, Fp, Fp, Wb("featsT"), BNp));
    TRY(transpose_f32_to_bf16(s, Wf("dproj_acc"), BN, A, A, Wb("dPT"), BNp));
  }
  TRY(transpose_bf16_jobs(s, tj));
  TRY(wgrad_add(Wb("dqT"), A, h1T, H, TB, TBp, Gr(SSCVAE_W_QUERY_PROJ), H));
  TRY(wgrad_add(Wb("dPT"), A, Wb("featsT"), F, BN, BNp, Gr(SSCVAE_W_IMAGE_PROJ), F));
  TRY(wgrad_launch());
  if (Gr(SSCVAE_W_ATT_VEC)) TRY(colsum_f32(s, Wf("dwa_acc"), B, A, A, Gr(SSCVAE_W_ATT_VEC)));
  TRY(event(4));
  return 0;
}

// ---- exported C ABI ----------------------------------------------------------------------------
}  // namespace sscvae

using namespace sscvae;

extern "C" {

int sscvae_abi_version(void) { return SSCVAE_ABI_VERSION; }
const char* sscvae_last_error(void) { return get_error(); }
uint64_t sscvae_launch_count(void) { return g_launch_count + g_launch_count_pw; }

int sscvae_set_option(SscvaeHandle* hh, const char* name, int value) {
  Handle* h = reinterpret_cast<Handle*>(hh);
  REQUIRE(h && name, "NULL argument");
  if (strcmp(name, "features_bf16") == 0) { h->opt_features_bf16 = value ? 1 : 0; return 0; }
  if (strcmp(name, "reuse_image_state") == 0) { h->opt_reuse_image_state = value ? 1 : 0; return 0; }
  if (strcmp(name, "fsm_packed") == 0) { h->opt_fsm_packed = value ? 1 : 0; return 0; }
  if (strcmp(name, "persistent_bwd") == 0) { h->opt_persistent_bwd = value ? 1 : 0; return 0; }
  set_error("unknown option '%s'", name);
  return SSCVAE_ERR_BAD_ARG;
}

int sscvae_train_backward_is_persistent(const SscvaeHandle* hh, int batch, int num_boxes) {
  const Handle* h = reinterpret_cast<const Handle*>(hh);
  REQUIRE(h && batch > 0 && num_boxes > 0, "bad argument");
  return h->opt_persistent_bwd && persistent_backward(h->d, batch, num_boxes) ? 1 : 0;
}

int sscvae_debug_bptt_tiling(const SscvaeHandle* hh, int batch, int num_boxes, int pairs, int32_t* out12) {
  const Handle* h = reinterpret_cast<const Handle*>(hh);
  REQUIRE(h && out12 && batch > 0 && num_boxes > 0 && pairs > 0, "bad argument");
  if (h->d.cvar) return 0;
  RecBwdArgs rb;
  fill_rec_bwd_args(h->d, batch, num_boxes, rb);
  int v[12];
  if (!recurrent_backward_tiling(rb, pairs, v)) return 0;
  for (int i = 0; i < 12; ++i) out12[i] = v[i];
  return 1;
}

int sscvae_create(const SscvaeDims* dims, SscvaeHandle** out) {
  REQUIRE(out != nullptr, "out is NULL");
  Handle* h = new Handle();
  int r = init_dims(dims, h->d);
  if (r) { delete h; return r; }
  plan_packed(h->d, h->pp);
  *out = reinterpret_cast<SscvaeHandle*>(h);
  return 0;
}
void sscvae_destroy(SscvaeHandle* h) { delete reinterpret_cast<Handle*>(h); }

size_t sscvae_packed_bytes(const SscvaeHandle* h) { return reinterpret_cast<const Handle*>(h)->pp.total; }

int sscvae_pack_weights(SscvaeHandle* hh, const void* const* weights, void* packed, size_t packed_bytes,
                        const uint8_t* dirty, void* stream) {
  Handle* h = reinterpret_cast<Handle*>(hh);
  REQUIRE(h && weights && packed, "NULL argument");
  if (packed_bytes < h->pp.total) { set_error("packed buffer too small: %zu < %zu", packed_bytes, h->pp.total); return SSCVAE_ERR_WORKSPACE; }
  REQUIRE((reinterpret_cast<uintptr_t>(packed) & 255) == 0, "packed buffer must be 256-byte aligned");
  return pack_weights_impl(h, weights, reinterpret_cast<char*>(packed), dirty, reinterpret_cast<cudaStream_t>(stream));
}

int sscvae_sgd_step_packed(SscvaeHandle* hh, const void* const* weights, const void* const* grads,
                           void* const* momentum_bufs, const int32_t* first_step, int count, const int32_t* order,
                           float max_norm, float lr, float momentum, float weight_decay, float grad_scale, void* packed,
                           size_t packed_bytes, float* scratch, size_t scratch_floats, void* stream) {
  Handle* h = reinterpret_cast<Handle*>(hh);
  REQUIRE(h && weights && grads && first_step && order && packed && scratch, "NULL argument");
  REQUIRE(count > 0 && count <= SSCVAE_W_COUNT, "count %d not in 1..%d", count, SSCVAE_W_COUNT);
  if (packed_bytes < h->pp.total) { set_error("packed buffer too small: %zu < %zu", packed_bytes, h->pp.total); return SSCVAE_ERR_WORKSPACE; }
  REQUIRE((reinterpret_cast<uintptr_t>(packed) & 255) == 0, "packed buffer must be 256-byte aligned");
  for (int i = 0; i < SSCVAE_W_COUNT; ++i) REQUIRE(weights[i] != nullptr, "weight pointer %d is NULL", i);
  const Dims& d = h->d;
  std::vector<SrcBlock> bl;
  TRY(source_blocks(d, bl));
  SgdPackTable t;
  fill_tensors(d, weights, t);
  for (int i = 0; i < count; ++i) {
    const int w = order[i];
    REQUIRE(w >= 0 && w < SSCVAE_W_COUNT && !t.t[w].upd, "order[%d] = %d: not a weight id, or repeated", i, w);
    REQUIRE(momentum == 0.f || (momentum_bufs && momentum_bufs[w]), "NULL momentum buffer of weight %d", w);
    SgdPackTensor& x = t.t[w];
    x.upd = 1; x.first = first_step[w] != 0;
    x.g = reinterpret_cast<const float*>(grads[w]);   // NULL: a zero gradient, as in sscvae_sgd_step_multi
    x.m = momentum_bufs ? reinterpret_cast<float*>(momentum_bufs[w]) : nullptr;
  }
  char* pk = reinterpret_cast<char*>(packed);
  for (const SrcBlock& b : bl)
    if (t.t[b.w].upd || (b.w2 >= 0 && t.t[b.w2].upd)) fill_job(d, h->pp, b, pk, t.job[t.n++]);
  return sgd_pack_step(reinterpret_cast<cudaStream_t>(stream), t, order, count,
                       SgdParams{max_norm, lr, momentum, weight_decay, grad_scale}, scratch, scratch_floats);
}

int sscvae_debug_sgd_pack_jobs(const SscvaeHandle* hh, int64_t* out, int max_jobs) {
  const Handle* h = reinterpret_cast<const Handle*>(hh);
  REQUIRE(h && out && max_jobs > 0, "bad argument");
  std::vector<SrcBlock> bl;
  TRY(source_blocks(h->d, bl));
  REQUIRE((int)bl.size() <= max_jobs, "%d jobs > max_jobs %d", (int)bl.size(), max_jobs);
  int rows[SSCVAE_W_COUNT], cols[SSCVAE_W_COUNT];
  weight_shapes(h->d, rows, cols);
  for (size_t i = 0; i < bl.size(); ++i) {
    const SrcBlock& b = bl[i];
    int64_t* o = out + 16 * i;
    const int64_t v[8] = {b.w, b.w2, b.c0, rows[b.w], b.cols, cols[b.w], b.w2 >= 0 ? cols[b.w2] : 0, b.nout};
    for (int k = 0; k < 8; ++k) o[k] = v[k];
    for (int k = 0; k < 2; ++k) {
      const bool on = k < b.nout;
      o[8 + 4 * k] = on ? b.out[k].kind : -1;
      o[9 + 4 * k] = on ? (int64_t)out_offset(h->pp, b.out[k]) : -1;
      o[10 + 4 * k] = on ? b.out[k].ld : 0;
      o[11 + 4 * k] = on ? b.out[k].gate_H : 0;
    }
  }
  return (int)bl.size();
}

size_t sscvae_train_workspace_bytes(const SscvaeHandle* hh, int batch, int num_boxes) {
  Handle* h = const_cast<Handle*>(reinterpret_cast<const Handle*>(hh));
  if (!h || batch <= 0 || num_boxes <= 0) return 0;
  return h->train_plan(batch, num_boxes).total;
}

int sscvae_train_region(const SscvaeHandle* hh, int batch, int num_boxes, const char* name, size_t* offset, size_t* bytes) {
  Handle* h = const_cast<Handle*>(reinterpret_cast<const Handle*>(hh));
  REQUIRE(h && name && offset && bytes, "NULL argument");
  const Region* r = h->train_plan(batch, num_boxes).find(name);
  REQUIRE(r != nullptr, "unknown workspace region '%s'", name);
  *offset = r->off; *bytes = r->bytes;
  return 0;
}

int sscvae_train_forward(SscvaeHandle* hh, int batch, int num_boxes, const void* packed, const void* const* weights,
                         const float* image_features, const int64_t* caption_tokens, const float* sentiment,
                         const float* obj_means, const float* eps, uint64_t seed, void* workspace, size_t workspace_bytes,
                         float* loss, float* kld, void* stream) {
  Handle* h = reinterpret_cast<Handle*>(hh);
  REQUIRE(h && packed && weights && image_features && caption_tokens && workspace && loss && kld, "NULL argument");
  REQUIRE(batch > 0 && num_boxes > 0, "batch/num_boxes must be positive");
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  const Plan& tp = h->train_plan(batch, num_boxes);
  if (workspace_bytes < tp.total) { set_error("workspace too small: %zu < %zu", workspace_bytes, tp.total); return SSCVAE_ERR_WORKSPACE; }
  const unsigned long long seed_host = seed;
  CUDA_TRY(cudaMemcpyAsync(reinterpret_cast<char*>(workspace) + tp.find("seed")->off, &seed_host, sizeof(seed_host),
                           cudaMemcpyHostToDevice, st));
  std::vector<uint64_t> key;
  key_add(key, (uint64_t)batch); key_add(key, (uint64_t)num_boxes); key_add(key, packed); key_add(key, image_features);
  key_add(key, (uint64_t)h->opt_features_bf16);
  key_add(key, caption_tokens); key_add(key, sentiment); key_add(key, obj_means); key_add(key, eps); key_add(key, workspace);
  key_add(key, (uint64_t)workspace_bytes); key_add(key, loss); key_add(key, kld);
  for (int i = 0; i < SSCVAE_W_COUNT; ++i) key_add(key, weights[i]);
  return run_with_graph(h->fwd_graphs, key, st, true, [&](cudaStream_t s) {
    return train_forward_impl(h, batch, num_boxes, reinterpret_cast<const char*>(packed), weights, image_features,
                              reinterpret_cast<const long long*>(caption_tokens), sentiment, obj_means, eps, seed,
                              reinterpret_cast<char*>(workspace), workspace_bytes, loss, kld, s);
  });
}

int sscvae_train_backward(SscvaeHandle* hh, int batch, int num_boxes, const void* packed, const void* const* weights,
                          void* workspace, size_t workspace_bytes, const float* grad_loss, const float* grad_kld,
                          void* const* grads, void* const* group_events, void* stream) {
  Handle* h = reinterpret_cast<Handle*>(hh);
  REQUIRE(h && packed && weights && workspace && grad_loss && grad_kld && grads, "NULL argument");
  if (group_events)                                   // a NULL entry would be silently skipped and baked into the replayed graph
    for (int g = 0; g < SSCVAE_GRAD_GROUPS; ++g) REQUIRE(group_events[g] != nullptr, "group_events[%d] is NULL (pass NULL for the whole array to disable)", g);
  std::vector<uint64_t> key;
  key_add(key, (uint64_t)batch); key_add(key, (uint64_t)num_boxes); key_add(key, packed); key_add(key, workspace);
  key_add(key, (uint64_t)workspace_bytes); key_add(key, grad_loss); key_add(key, grad_kld);
  key_add(key, (uint64_t)h->opt_persistent_bwd);
  for (int i = 0; i < SSCVAE_W_COUNT; ++i) { key_add(key, weights[i]); key_add(key, grads[i]); }
  for (int g = 0; g < SSCVAE_GRAD_GROUPS; ++g) key_add(key, group_events ? group_events[g] : nullptr);
  return run_with_graph(h->bwd_graphs, key, reinterpret_cast<cudaStream_t>(stream), true, [&](cudaStream_t s) {
    return train_backward_impl(h, batch, num_boxes, reinterpret_cast<const char*>(packed), weights,
                               reinterpret_cast<char*>(workspace), workspace_bytes, grad_loss, grad_kld, grads,
                               group_events, s);
  });
}

int sscvae_test_gemm(const void* A, int lda, const void* B, int ldb, int M, int N, int K, float* C32, int ldc,
                     const float* bias, int act_tanh, int accumulate, void* stream) {
  GemmSeg sg; sg.A = reinterpret_cast<const bf16*>(A); sg.lda = lda; sg.B = reinterpret_cast<const bf16*>(B); sg.ldb = ldb; sg.K = K;
  GemmEpi e; e.C32 = C32; e.ldc32 = ldc; e.bias = bias; e.act = act_tanh; e.accumulate = accumulate;
  int repeat = 1;                                   // tools/gemm_bench.py: back-to-back launches without Python in between
  if (const char* r = getenv("SSCVAE_TEST_GEMM_REPEAT")) repeat = std::max(1, atoi(r));
  for (int i = 0; i < repeat; ++i) TRY(gemm_bf16_tn(reinterpret_cast<cudaStream_t>(stream), M, N, 1, &sg, e));
  return 0;
}

int sscvae_test_gemm_splitk(const void* A, int lda, const void* B, int ldb, int M, int N, int K, float* C32, int ldc,
                            int splits, const float* bias, void* stream) {
  GemmSeg sg; sg.A = reinterpret_cast<const bf16*>(A); sg.lda = lda; sg.B = reinterpret_cast<const bf16*>(B); sg.ldb = ldb; sg.K = K;
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  GemmEpi e; e.C32 = C32; e.ldc32 = ldc; e.bias = bias; e.splits = splits;
  int repeat = 1;
  if (const char* r = getenv("SSCVAE_TEST_GEMM_REPEAT")) repeat = std::max(1, atoi(r));
  for (int i = 0; i < repeat; ++i) TRY(gemm_bf16_tn(st, M, N, 1, &sg, e));
  return 0;
}

int sscvae_test_gemm_grouped(int nprob, const void* const* A, const int* lda, const void* const* B, const int* ldb,
                             const int* M, const int* N, const int* K, float* const* C32, const int* ldc, void* stream) {
  REQUIRE(nprob >= 1 && nprob <= kMaxGemmProblems && A && lda && B && ldb && M && N && K && C32 && ldc, "bad argument");
  GemmProblem pb[kMaxGemmProblems];
  for (int i = 0; i < nprob; ++i)
    pb[i] = GemmProblem{reinterpret_cast<const bf16*>(A[i]), lda[i], reinterpret_cast<const bf16*>(B[i]), ldb[i], K[i], M[i],
                        N[i], C32[i], ldc[i]};
  int repeat = 1;
  if (const char* r = getenv("SSCVAE_TEST_GEMM_REPEAT")) repeat = std::max(1, atoi(r));
  for (int i = 0; i < repeat; ++i) TRY(gemm_bf16_tn_grouped(reinterpret_cast<cudaStream_t>(stream), nprob, pb, "gemm.wgrad"));
  return 0;
}

int sscvae_test_transpose_bf16(int njobs, const void* const* in, const int* rows, const int* cols, const int* ld_in,
                               void* const* out, const int* ld_out, void* stream) {
  REQUIRE(njobs >= 1 && njobs <= kMaxTransposeJobs && in && rows && cols && ld_in && out && ld_out, "bad argument");
  int repeat = 1;
  if (const char* r = getenv("SSCVAE_TEST_GEMM_REPEAT")) repeat = std::max(1, atoi(r));
  for (int k = 0; k < repeat; ++k) {
    TransposeJobList tj;
    for (int i = 0; i < njobs; ++i)
      TRY(tj.add(reinterpret_cast<const bf16*>(in[i]), rows[i], cols[i], ld_in[i], reinterpret_cast<bf16*>(out[i]), ld_out[i]));
    TRY(transpose_bf16_jobs(reinterpret_cast<cudaStream_t>(stream), tj));
  }
  return 0;
}

}  // extern "C"

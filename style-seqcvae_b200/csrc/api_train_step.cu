// C ABI: one differentiable training step of the cell, the reference's `_decode_step` in training mode
// (updown_captioner.py:371-455 with the encoder branch of updown_cell.py:176-198), forward and backward (include/sscvae.h).
//
// Three caller-owned buffers, so that any number of steps over any number of batches can be alive at once:
//   image state  the per-image operands of one (features, obj_means, weights): bf16 features and their transpose, mask, mean
//                feature, W_v projection, mean-feature gate block, per-box attribute means. Built once, read by every step.
//   tape         everything one step's backward reads: the bf16 operand rows its GEMMs consumed, the states it started
//                from, gates, cell states, attention softmax, mean / log_var / eps. One per step.
//   workspace    scratch of a single call (GEMM accumulators, gradient operands, transposes); any call may reuse it.
// Rows are images (R = B); the operand layouts are those of api_train.cu with T = 1.
#include "api_internal.cuh"

namespace sscvae {

static void plan_step_image(const Dims& d, int B, int N, Plan& p) {
  const size_t b = sizeof(bf16), f = 4, BN = (size_t)B * N;
  p.add("featsb", BN * d.Fp * b);
  p.add("projb", BN * d.Ap * b);
  p.add("avgb", (size_t)B * d.Fp * b);
  p.add("featsT", (size_t)d.Fp * round_up((int)BN, kPad) * b);
  p.add("avgT", (size_t)d.Fp * round_up(B, kPad) * b);
  p.add("mask", BN * f);
  p.add("gavg", (size_t)B * d.GP * f);
  if (d.cvar) p.add("objm", BN * d.Z * f);
}

// The bf16 operand rows come first: one memset zeroes their K-padding (no kernel writes the padding columns).
static void plan_step_tape(const Dims& d, int B, int N, Plan& p) {
  const size_t b = sizeof(bf16), f = 4;
  p.add("XAi", (size_t)B * 2 * d.Hp * b);              // [h1_{t-1} | h_dec_{t-1}]
  p.add("XAo", (size_t)B * 2 * d.Hp * b);              // [h1_t | h_dec_t]
  p.add("XE", (size_t)B * d.KX * b);                   // [xhat_t | h1_t | h_dec_{t-1}]
  p.add("HEi", (size_t)B * d.Hp * b);                  // h_enc_{t-1}
  p.add("HEo", (size_t)B * d.Hp * b);                  // h_enc_t
  p.add("ZB", (size_t)B * d.ZC * b);                   // [z_t | c_t]
  p.add("embb_r", (size_t)B * d.Ep * b);
  if (d.tied) p.add("ob", (size_t)B * d.Ep * b);
  p.add("tok", (size_t)B * 4);
  p.add("sent", (size_t)B * f);
  for (const char* n : {"c1p", "cep", "cdp", "c1", "ce", "cd"}) p.add(n, (size_t)B * d.H * f);
  for (const char* n : {"gates_att", "gates_enc", "gates_dec"}) p.add(n, (size_t)B * d.G * f);
  p.add("q", (size_t)B * d.A * f);
  p.add("smx", (size_t)B * N * f);
  for (const char* n : {"mean", "logvar", "eps"}) p.add(n, (size_t)B * d.Z * f);
  if (d.tied) p.add("o32", (size_t)B * d.E * f);
}

// The bf16 gradient operands come first: one memset per backward zeroes their padding columns (the data-gradient GEMMs read
// them with the zero-padded transposed weights, and uninitialised padding could hold NaN).
static void plan_step_ws(const Dims& d, int B, int N, Plan& p) {
  const size_t b = sizeof(bf16), f = 4, BN = (size_t)B * N;
  const size_t Bp = round_up(B, kPad), BNp = round_up((int)BN, kPad);
  p.add("dlog16", (size_t)B * d.Vp * b);
  if (d.tied) p.add("dpreo", (size_t)B * d.Ep * b);
  for (const char* n : {"dGa", "dGe", "dGd"}) p.add(n, (size_t)B * d.Gp * b);
  p.add("dml", (size_t)B * d.Z2p * b);
  p.add("dqb", (size_t)B * d.Ap * b);
  // forward scratch
  p.add("acc", (size_t)B * d.GP * f);
  p.add("ml", (size_t)B * d.Z2 * f);
  p.add("kl", (size_t)B * f);
  // backward scratch
  p.add("dhead", (size_t)B * d.H * f);
  p.add("dXEZ", (size_t)B * (d.KX + d.ZC) * f);
  p.add("dXE", (size_t)B * (d.KX + d.Hp + d.Cp) * f);
  p.add("dXA", (size_t)B * 2 * d.Hp * f);
  for (const char* n : {"dhenc_fc", "dh1_q", "dc1", "dce", "dcd"}) p.add(n, (size_t)B * d.H * f);
  if (d.cvar) {
    p.add("dpm0", (size_t)B * d.Z * f);
    p.add("dalpha_x", BN * f);
  }
  p.add("du", BN * f);
  p.add("dproj", BN * d.A * f);
  p.add("dwa", (size_t)B * d.A * f);
  if (!d.tied) p.add("dxemb", (size_t)B * d.E * f);
  // transposed operands of the weight-gradient GEMMs (K = B rows)
  for (const char* n : {"dGaT", "dGeT", "dGdT"}) p.add(n, (size_t)d.G * Bp * b);
  p.add("XET", (size_t)d.KX * Bp * b);
  p.add("ZBT", (size_t)d.ZC * Bp * b);
  p.add("XAT", (size_t)2 * d.Hp * Bp * b);
  p.add("HETp", (size_t)d.Hp * Bp * b);
  p.add("HETc", (size_t)d.Hp * Bp * b);
  p.add("hdT", (size_t)d.Hp * Bp * b);
  p.add("dmlT", (size_t)d.Z2p * Bp * b);
  p.add("embT", (size_t)d.Ep * Bp * b);
  p.add("dqT", (size_t)d.Ap * Bp * b);
  p.add("dheadT", (size_t)(d.tied ? d.E : d.V) * Bp * b);
  p.add("dPT", (size_t)d.A * BNp * b);
}

static inline GemmSeg seg(const bf16* A, int lda, const bf16* B, int ldb, int K) {
  GemmSeg s; s.A = A; s.lda = lda; s.B = B; s.ldb = ldb; s.K = K; return s;
}

// Named regions of the three buffers and of the packed weights.
struct StepViews {
  const char* pk; const Plan& pp; const void* const* wv;
  char* is; Plan ip; char* tp; Plan tpl; char* ws; Plan wpl;
  const float* W(int i) const { return reinterpret_cast<const float*>(wv[i]); }
  const bf16* Pb(const char* n) const { return reinterpret_cast<const bf16*>(pk + pp.find(n)->off); }
  const float* Pf(const char* n) const { return reinterpret_cast<const float*>(pk + pp.find(n)->off); }
  bf16* Ib(const char* n) const { return reinterpret_cast<bf16*>(is + ip.find(n)->off); }
  float* If(const char* n) const { return reinterpret_cast<float*>(is + ip.find(n)->off); }
  bf16* Tb(const char* n) const { return reinterpret_cast<bf16*>(tp + tpl.find(n)->off); }
  float* Tf(const char* n) const { return reinterpret_cast<float*>(tp + tpl.find(n)->off); }
  int* Ti(const char* n) const { return reinterpret_cast<int*>(tp + tpl.find(n)->off); }
  bf16* Wb(const char* n) const { return reinterpret_cast<bf16*>(ws + wpl.find(n)->off); }
  float* Wf(const char* n) const { return reinterpret_cast<float*>(ws + wpl.find(n)->off); }
};

static bool aligned256(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 255) == 0; }

static int check_buffer(const char* what, const void* p, size_t have, size_t need) {
  REQUIRE(p != nullptr, "NULL argument: %s", what);
  if (have < need) { set_error("%s too small: %zu < %zu", what, have, need); return SSCVAE_ERR_WORKSPACE; }
  REQUIRE(aligned256(p), "%s must be 256-byte aligned", what);
  return 0;
}

// ---- forward ----------------------------------------------------------------------------------------------------------
static int step_forward_impl(const Dims& d, const StepViews& v, int B, int N, const float* sent, const long long* prev,
                             const float* const* states_in, const float* eps, unsigned long long seed, float* logits,
                             float* const* states_out, float* mean, float* log_var, float* pm_out, float* alpha, cudaStream_t s) {
  const int GP = d.GP, H = d.H, Hp = d.Hp, Fp = d.Fp, KX = d.KX;
  const bool csent = d.cond && !d.cvar;
  const size_t BH = (size_t)B * H * sizeof(float);
  {
    const Region* first = v.tpl.find("XAi");
    const Region* last = v.tpl.find(d.tied ? "ob" : "embb_r");
    CUDA_TRY(cudaMemsetAsync(v.tp + first->off, 0, last->off + last->bytes - first->off, s));
  }
  // states in: bf16 operand rows [h1 | h_dec], h_dec_{t-1} block of XE, h_enc_{t-1}; fp32 cell states copied onto the tape
  TRY(step_import(s, prev, B, 1, states_in ? states_in[0] : nullptr, states_in ? states_in[4] : nullptr, H, Hp, v.Ti("tok"),
                  nullptr, v.Tb("XAi"), states_in ? states_in[2] : nullptr, states_in ? v.Tb("HEi") : nullptr,
                  states_in ? v.Tb("XE") + Fp + Hp : nullptr, KX));
  const char* cp[3] = {"c1p", "cep", "cdp"};
  for (int k = 0; k < 3; ++k) {
    if (states_in) CUDA_TRY(cudaMemcpyAsync(v.Tf(cp[k]), states_in[2 * k + 1], BH, cudaMemcpyDeviceToDevice, s));
    else CUDA_TRY(cudaMemsetAsync(v.Tf(cp[k]), 0, BH, s));
  }
  if (csent) CUDA_TRY(cudaMemcpyAsync(v.Tf("sent"), sent, (size_t)B * sizeof(float), cudaMemcpyDeviceToDevice, s));
  TRY(embed_gather_rows(s, v.Ti("tok"), B, v.Pb("embb"), d.Ep, v.Tb("embb_r")));
  {  // attention LSTM (updown_cell.py:143-148)
    LstmFwdArgs l = {};
    l.R = B; l.H = H; l.add2 = v.If("gavg"); l.ld2 = GP; l.bias = v.Pf("b_att");
    l.c_prev = v.Tf("c1p"); l.c_out = v.Tf("c1"); l.gates_out = v.Tf("gates_att");
    l.h1_dst = v.Tb("XE") + Fp; l.ld_h1 = KX; l.h2_dst = v.Tb("XAo"); l.ld_h2 = 2 * Hp; l.h_out = states_out[0];
    l.acc = v.Wf("acc"); l.ld_acc = GP; l.perm = 1;
    GemmSeg sg[2] = {seg(v.Tb("embb_r"), d.Ep, v.Pb("w_att_e"), d.Ep, d.E), seg(v.Tb("XAi"), 2 * Hp, v.Pb("w_att_rec"), 2 * Hp, 2 * Hp)};
    GemmEpi e; e.tag = "gemm.step"; e.C32 = v.Wf("acc"); e.ldc32 = GP;
    TRY(gemm_bf16_tn(s, B, GP, 2, sg, e));
    TRY(lstm_forward(s, l));
  }
  AttnArgs aa = {}; aa.R = B; aa.N = N; aa.A = d.A; aa.Ap = d.Ap; aa.F = d.F; aa.Fp = Fp;
  aa.proj = v.Ib("projb"); aa.feats = v.Ib("featsb"); aa.mask = v.If("mask"); aa.w_a = v.W(SSCVAE_W_ATT_VEC);
  aa.q = v.Tf("q"); aa.ld_q = d.A;
  {  // query projection + region attention (attention.py:69-93, updown_cell.py:156)
    GemmSeg sg = seg(v.Tb("XE") + Fp, KX, v.Pb("wq"), Hp, Hp);
    GemmEpi e; e.tag = "gemm.step"; e.C32 = v.Tf("q"); e.ldc32 = d.A;
    TRY(gemm_bf16_tn(s, B, d.A, 1, &sg, e));
    TRY(attention_forward(s, aa, alpha, v.Tf("smx"), v.Tb("XE"), KX));
    if (d.cvar)  // attribute-grounded prior mean of this step (updown_cell.py:160-174), also the conditioning block c
      TRY(prior_mean_forward(s, alpha, v.If("objm"), nullptr, B, N, d.Z, pm_out, v.Tb("ZB") + d.Zp, d.ZC, d.cond));
  }
  {  // posterior (encoder) LSTM + latent heads + reparameterised sample (updown_cell.py:176-208)
    LstmFwdArgs l = {};
    l.R = B; l.H = H; l.bias = v.Pf("b_enc");
    if (csent) { l.sent = v.Tf("sent"); l.scol = v.Pf("scol_enc"); }
    l.c_prev = v.Tf("cep"); l.c_out = v.Tf("ce"); l.gates_out = v.Tf("gates_enc");
    l.h1_dst = v.Tb("HEo"); l.ld_h1 = Hp; l.h_out = states_out[2];
    l.acc = v.Wf("acc"); l.ld_acc = GP; l.perm = 1;
    GemmSeg sg[3] = {seg(v.Tb("XE"), KX, v.Pb("w_enc_x"), KX, KX), seg(v.Tb("HEi"), Hp, v.Pb("w_enc_hh"), Hp, Hp), GemmSeg()};
    if (d.cvar) sg[2] = seg(v.Tb("ZB") + d.Zp, d.ZC, v.Pb("w_enc_c"), d.Cp, d.Cp);
    GemmEpi e; e.tag = "gemm.step"; e.C32 = v.Wf("acc"); e.ldc32 = GP;
    TRY(gemm_bf16_tn(s, B, GP, d.cvar ? 3 : 2, sg, e));
    TRY(lstm_forward(s, l));
    GemmSeg sf = seg(v.Tb("HEo"), Hp, v.Pb("w_fc"), Hp, Hp);
    GemmEpi ef; ef.tag = "gemm.step"; ef.C32 = v.Wf("ml"); ef.ldc32 = d.Z2;
    TRY(gemm_bf16_tn(s, B, d.Z2, 1, &sf, ef));
    // the KL it also computes goes to scratch: the caller forms the KL from mean / log_var and the prior
    LatentArgs la = {}; la.R = B; la.Z = d.Z; la.Zp = d.Zp; la.sentiment_vae = d.sv; la.prior_var = d.prior_std * d.prior_std;
    la.seed = seed;
    TRY(latent_forward_train(s, la, v.Wf("ml"), d.Z2, v.Pf("b_fc"), eps, nullptr, 0, v.Tf("mean"), v.Tf("logvar"),
                             v.Tf("eps"), v.Tb("ZB"), d.ZC, v.Wf("kl")));
  }
  {  // language (decoder) LSTM (updown_cell.py:211-229)
    LstmFwdArgs l = {};
    l.R = B; l.H = H; l.bias = v.Pf("b_dec");
    if (csent) { l.sent = v.Tf("sent"); l.scol = v.Pf("scol_dec"); }
    l.c_prev = v.Tf("cdp"); l.c_out = v.Tf("cd"); l.gates_out = v.Tf("gates_dec");
    l.h1_dst = v.Tb("XAo") + Hp; l.ld_h1 = 2 * Hp; l.h_out = states_out[4];
    l.acc = v.Wf("acc"); l.ld_acc = GP; l.perm = 1;
    GemmSeg sg[2] = {seg(v.Tb("XE"), KX, v.Pb("w_dec_x"), KX, KX), seg(v.Tb("ZB"), d.ZC, v.Pb("w_dec_z"), d.ZC, d.ZC)};
    GemmEpi e; e.tag = "gemm.step"; e.C32 = v.Wf("acc"); e.ldc32 = GP;
    TRY(gemm_bf16_tn(s, B, GP, 2, sg, e));
    TRY(lstm_forward(s, l));
  }
  // output head, raw fp32 logits (updown_captioner.py:444-445)
  const bf16* hdec = v.Tb("XAo") + Hp;
  if (d.tied) {
    GemmSeg sg = seg(hdec, 2 * Hp, v.Pb("w_out"), Hp, Hp);
    GemmEpi e; e.tag = "gemm.step"; e.bias = v.W(SSCVAE_W_OUT_PROJ_B); e.act = 1; e.C32 = v.Tf("o32"); e.ldc32 = d.E;
    e.C16 = v.Tb("ob"); e.ldc16 = d.Ep;
    TRY(gemm_bf16_tn(s, B, d.E, 1, &sg, e));
    GemmSeg sv = seg(v.Tb("ob"), d.Ep, v.Pb("embb"), d.Ep, d.E);
    GemmEpi ev; ev.tag = "gemm.step"; ev.C32 = logits; ev.ldc32 = d.V;
    TRY(gemm_bf16_tn(s, B, d.V, 1, &sv, ev));
  } else {
    GemmSeg sg = seg(hdec, 2 * Hp, v.Pb("w_out"), Hp, Hp);
    GemmEpi e; e.tag = "gemm.step"; e.bias = v.W(SSCVAE_W_OUT_PROJ_B); e.C32 = logits; e.ldc32 = d.V;
    TRY(gemm_bf16_tn(s, B, d.V, 1, &sg, e));
  }
  // outputs the caller may edit in place are copies: the backward reads the tape's own
  const char* co[3] = {"c1", "ce", "cd"};
  for (int k = 0; k < 3; ++k) CUDA_TRY(cudaMemcpyAsync(states_out[2 * k + 1], v.Tf(co[k]), BH, cudaMemcpyDeviceToDevice, s));
  const size_t BZ = (size_t)B * d.Z * sizeof(float);
  CUDA_TRY(cudaMemcpyAsync(mean, v.Tf("mean"), BZ, cudaMemcpyDeviceToDevice, s));
  CUDA_TRY(cudaMemcpyAsync(log_var, v.Tf("logvar"), BZ, cudaMemcpyDeviceToDevice, s));
  return 0;
}

// ---- backward ---------------------------------------------------------------------------------------------------------
static int step_backward_impl(const Dims& d, const StepViews& v, int B, int N, const float* d_logits,
                              const float* const* d_states_out, const float* d_mean, const float* d_log_var,
                              const float* d_prior_mean, const float* d_alpha, float* const* d_states_in, void* const* gv,
                              cudaStream_t s) {
  const int G = d.G, Gp = d.Gp, H = d.H, Hp = d.Hp, KX = d.KX, Fp = d.Fp, E = d.E, F = d.F, A = d.A, Z = d.Z, V = d.V;
  const int c = d.cond, Bp = round_up(B, kPad), BN = B * N, BNp = round_up(BN, kPad);
  const int KXH = KX + Hp + d.Cp, KXZ = KX + d.ZC;
  auto Gr = [&](int i) { return reinterpret_cast<float*>(gv[i]); };
  auto dso = [&](int k) -> const float* { return d_states_out ? d_states_out[k] : nullptr; };
  {
    const Region* first = v.wpl.find("dlog16");
    const Region* last = v.wpl.find("dqb");
    CUDA_TRY(cudaMemsetAsync(v.ws + first->off, 0, last->off + last->bytes - first->off, s));
  }
  // ---- head: d h_dec from the caller's d logits
  TRY(convert_f32_to_bf16(s, d_logits, B, V, V, v.Wb("dlog16"), d.Vp));
  if (d.tied) {
    GemmSeg sg = seg(v.Wb("dlog16"), d.Vp, v.Pb("embT"), d.Vp, V);
    GemmEpi e; e.tag = "gemm.step_bwd"; e.dtanh = v.Tf("o32"); e.ldd = E; e.C16 = v.Wb("dpreo"); e.ldc16 = d.Ep;
    TRY(gemm_bf16_tn(s, B, E, 1, &sg, e));
    GemmSeg s2 = seg(v.Wb("dpreo"), d.Ep, v.Pb("w_outT"), d.Ep, E);
    GemmEpi e2; e2.tag = "gemm.step_bwd"; e2.C32 = v.Wf("dhead"); e2.ldc32 = H;
    TRY(gemm_bf16_tn(s, B, H, 1, &s2, e2));
  } else {
    GemmSeg sg = seg(v.Wb("dlog16"), d.Vp, v.Pb("w_outT"), d.Vp, V);
    GemmEpi e; e.tag = "gemm.step_bwd"; e.C32 = v.Wf("dhead"); e.ldc32 = H;
    TRY(gemm_bf16_tn(s, B, H, 1, &sg, e));
  }
  // ---- the per-launch BPTT body for one step (api_train.cu), the next step's contributions replaced by d states_out
  {  // decoder LSTM: d h_dec_t = head + the caller's d h_decoder
    LstmBwdArgs l = {};
    l.R = B; l.H = H; l.dh[0] = v.Wf("dhead"); l.ld_dh[0] = H; l.dh[1] = dso(4); l.ld_dh[1] = H;
    l.dc_in = dso(5); l.dc_prev = v.Wf("dcd");
    l.gates = v.Tf("gates_dec"); l.c = v.Tf("cd"); l.c_prev = v.Tf("cdp");
    l.dgates = v.Wb("dGd"); l.ld_dg = Gp;
    TRY(lstm_backward(s, l));
  }
  {  // decoder part of d[xhat|h1|h_dec_{t-1}] and d z (and d c), then d mean / d log_var with the caller's upstream terms
    GemmSeg sg = seg(v.Wb("dGd"), Gp, v.Pb("w_dec_xzT"), Gp, G);
    GemmEpi e; e.tag = "gemm.step_bwd"; e.C32 = v.Wf("dXEZ"); e.ldc32 = KXZ;
    TRY(gemm_bf16_tn(s, B, KXZ, 1, &sg, e));
    LatentArgs la = {}; la.R = B; la.Z = Z; la.Zp = d.Zp; la.sentiment_vae = d.sv; la.prior_var = d.prior_std * d.prior_std;
    la.upstream = 1; la.dmean_up = d_mean; la.dlogvar_up = d_log_var;
    TRY(latent_backward(s, la, v.Wf("dXEZ") + KX, KXZ, v.Tf("eps"), v.Tf("mean"), v.Tf("logvar"), nullptr, nullptr,
                        v.Wb("dml"), d.Z2p));
    GemmSeg s2 = seg(v.Wb("dml"), d.Z2p, v.Pb("w_fcT"), d.Z2p, d.Z2);
    GemmEpi e2; e2.tag = "gemm.step_bwd"; e2.C32 = v.Wf("dhenc_fc"); e2.ldc32 = H;
    TRY(gemm_bf16_tn(s, B, H, 1, &s2, e2));
  }
  {  // encoder LSTM
    LstmBwdArgs l = {};
    l.R = B; l.H = H; l.dh[0] = v.Wf("dhenc_fc"); l.ld_dh[0] = H; l.dh[1] = dso(2); l.ld_dh[1] = H;
    l.dc_in = dso(3); l.dc_prev = v.Wf("dce");
    l.gates = v.Tf("gates_enc"); l.c = v.Tf("ce"); l.c_prev = v.Tf("cep");
    l.dgates = v.Wb("dGe"); l.ld_dg = Gp;
    TRY(lstm_backward(s, l));
    GemmSeg sg = seg(v.Wb("dGe"), Gp, v.Pb("w_enc_xhT"), Gp, G);
    GemmEpi e; e.tag = "gemm.step_bwd"; e.C32 = v.Wf("dXE"); e.ldc32 = KXH;
    e.add1 = v.Wf("dXEZ"); e.ld1 = KXZ; e.add1_cols = KX;
    TRY(gemm_bf16_tn(s, B, KXH, 1, &sg, e));
  }
  AttnArgs aa = {}; aa.R = B; aa.N = N; aa.A = A; aa.Ap = d.Ap; aa.F = F; aa.Fp = Fp;
  aa.proj = v.Ib("projb"); aa.feats = v.Ib("featsb"); aa.mask = v.If("mask"); aa.w_a = v.W(SSCVAE_W_ATT_VEC);
  aa.q = v.Tf("q"); aa.ld_q = A;
  {  // attention backward (d alpha: the caller's, plus the attribute-grounded prior's path), then d h1 through the query
    aa.dalpha_extra = d_alpha;
    if (d.cvar) {  // d prior_mean = the caller's + the two LSTMs' d c  ->  d alpha_n += objm_n . d prior_mean
      const float* dpm = d_prior_mean;
      if (!dpm) {
        CUDA_TRY(cudaMemsetAsync(v.Wf("dpm0"), 0, (size_t)B * Z * sizeof(float), s));
        dpm = v.Wf("dpm0");
      }
      TRY(prior_mean_backward(s, B, N, Z, c, dpm, v.Wf("dXEZ") + KX + d.Zp, KXZ, v.Wf("dXE") + KX + Hp, KXH, v.If("objm"),
                              v.Wf("dalpha_x")));
      if (d_alpha) TRY(add_f32(s, v.Wf("dalpha_x"), d_alpha, (size_t)BN));
      aa.dalpha_extra = v.Wf("dalpha_x");
    }
    TRY(attention_backward(s, aa, v.Tf("smx"), v.Wf("dXE"), KXH, v.Wb("dqb"), d.Ap, v.Wf("du")));
    GemmSeg sg = seg(v.Wb("dqb"), d.Ap, v.Pb("wqT"), d.Ap, A);
    GemmEpi e; e.tag = "gemm.step_bwd"; e.C32 = v.Wf("dh1_q"); e.ldc32 = H;
    TRY(gemm_bf16_tn(s, B, H, 1, &sg, e));
  }
  {  // attention LSTM
    LstmBwdArgs l = {};
    l.R = B; l.H = H;
    l.dh[0] = v.Wf("dXE") + Fp; l.ld_dh[0] = KXH; l.dh[1] = v.Wf("dh1_q"); l.ld_dh[1] = H; l.dh[2] = dso(0); l.ld_dh[2] = H;
    l.dc_in = dso(1); l.dc_prev = v.Wf("dc1");
    l.gates = v.Tf("gates_att"); l.c = v.Tf("c1"); l.c_prev = v.Tf("c1p");
    l.dgates = v.Wb("dGa"); l.ld_dg = Gp;
    TRY(lstm_backward(s, l));
    GemmSeg sg = seg(v.Wb("dGa"), Gp, v.Pb("w_att_recT"), Gp, G);
    GemmEpi e; e.tag = "gemm.step_bwd"; e.C32 = v.Wf("dXA"); e.ldc32 = 2 * Hp;
    TRY(gemm_bf16_tn(s, B, 2 * Hp, 1, &sg, e));
  }
  if (d_states_in) {
    StepGradExport x = {};
    x.R = B; x.H = H; x.Hp = Hp; x.dxa = v.Wf("dXA"); x.ld_xa = 2 * Hp; x.dxe = v.Wf("dXE"); x.ld_xe = KXH;
    x.off_hd = Fp + Hp; x.off_he = KX;
    x.dc[0] = v.Wf("dc1"); x.dc[1] = v.Wf("dce"); x.dc[2] = v.Wf("dcd");
    for (int k = 0; k < 6; ++k) x.out[k] = d_states_in[k];
    TRY(step_export_grads(s, x));
  }

  // ---- weight gradients over the B rows of this step (K = B), overwritten; NULL entries are skipped
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
  auto bias_pair = [&](const bf16* dGT, int ib, int ih) -> int {   // b_ih and b_hh get the same gradient
    float* g1 = Gr(ib); float* g2 = Gr(ih);
    if (!g1 && !g2) return 0;
    TRY(rowsum_bf16(s, dGT, G, B, Bp, g1 ? g1 : g2, 0));
    if (g1 && g2) CUDA_TRY(cudaMemcpyAsync(g2, g1, (size_t)G * sizeof(float), cudaMemcpyDeviceToDevice, s));
    return 0;
  };
  // W_hh is folded onto the W_ih block of the same operand (api_train.cu): one product, copied when both are wanted
  auto hh_pair = [&](const bf16* dGT, const bf16* BT, int ih, int hh) -> int {
    if (Gr(ih)) return 0;
    return wgrad_add(dGT, G, BT, H, B, Bp, Gr(hh), H);
  };
  auto hh_copy = [&](int ih, int col, int ld_ih, int hh) -> int {
    if (Gr(ih) && Gr(hh))
      CUDA_TRY(cudaMemcpy2DAsync(Gr(hh), (size_t)H * sizeof(float), Gr(ih) + col, (size_t)ld_ih * sizeof(float),
                                 (size_t)H * sizeof(float), G, cudaMemcpyDeviceToDevice, s));
    return 0;
  };
  const int ldE = F + 2 * H + c, ldD = F + 2 * H + c + Z, ldA = E + F + 2 * H;
  const bool csent = c && !d.cvar;
  const bf16* xhatT = v.Wb("XET");
  const bf16* h1T = v.Wb("XET") + (size_t)Fp * Bp;
  const bf16* hdecpT = v.Wb("XET") + (size_t)(Fp + Hp) * Bp;
  const bf16* condT = v.Wb("ZBT") + (size_t)d.Zp * Bp;
  const bf16* dmT = v.Wb("dmlT");
  const bf16* dlT = v.Wb("dmlT") + (size_t)Z * Bp;
  const bf16* h1pT = v.Wb("XAT");
  const bf16* hdecp2T = v.Wb("XAT") + (size_t)Hp * Bp;
  const bf16* headop = d.tied ? v.Wb("dpreo") : v.Wb("dlog16");
  const int NO = d.tied ? E : V, NOp = d.tied ? d.Ep : d.Vp;
  {  // every transposed operand in two launches (at most kMaxTransposeJobs each)
    TransposeJobList t1, t2;
    TRY(t1.add(v.Wb("dGd"), B, G, Gp, v.Wb("dGdT"), Bp));
    TRY(t1.add(v.Tb("XE"), B, KX, KX, v.Wb("XET"), Bp));
    TRY(t1.add(v.Tb("ZB"), B, d.ZC, d.ZC, v.Wb("ZBT"), Bp));
    TRY(t1.add(v.Wb("dGe"), B, G, Gp, v.Wb("dGeT"), Bp));
    TRY(t1.add(v.Tb("HEi"), B, Hp, Hp, v.Wb("HETp"), Bp));
    TRY(t1.add(v.Wb("dml"), B, d.Z2p, d.Z2p, v.Wb("dmlT"), Bp));
    TRY(t1.add(v.Tb("HEo"), B, Hp, Hp, v.Wb("HETc"), Bp));
    TRY(t2.add(v.Wb("dGa"), B, G, Gp, v.Wb("dGaT"), Bp));
    TRY(t2.add(v.Tb("XAi"), B, 2 * Hp, 2 * Hp, v.Wb("XAT"), Bp));
    TRY(t2.add(v.Tb("embb_r"), B, d.Ep, d.Ep, v.Wb("embT"), Bp));
    TRY(t2.add(v.Wb("dqb"), B, d.Ap, d.Ap, v.Wb("dqT"), Bp));
    TRY(t2.add(v.Tb("XAo") + Hp, B, H, 2 * Hp, v.Wb("hdT"), Bp));
    TRY(t2.add(headop, B, NO, NOp, v.Wb("dheadT"), Bp));
    TRY(transpose_bf16_jobs(s, t1));
    TRY(transpose_bf16_jobs(s, t2));
  }
  // decoder LSTM: W_ih column blocks [xhat | h1 | h_dec | cond | z]; W_hh shares the h_dec operand
  const bf16* dGdT = v.Wb("dGdT");
  if (float* g = Gr(SSCVAE_W_DEC_IH)) {
    TRY(wgrad_add(dGdT, G, xhatT, F, B, Bp, g, ldD));
    TRY(wgrad_add(dGdT, G, h1T, H, B, Bp, g + F, ldD));
    TRY(wgrad_add(dGdT, G, hdecpT, H, B, Bp, g + F + H, ldD));
    TRY(wgrad_add(dGdT, G, v.Wb("ZBT"), Z, B, Bp, g + F + 2 * H + c, ldD));
    if (d.cvar) TRY(wgrad_add(dGdT, G, condT, c, B, Bp, g + F + 2 * H, ldD));
  }
  TRY(hh_pair(dGdT, hdecpT, SSCVAE_W_DEC_IH, SSCVAE_W_DEC_HH));
  TRY(wgrad_launch());
  // encoder LSTM + latent heads
  const bf16* dGeT = v.Wb("dGeT");
  if (float* g = Gr(SSCVAE_W_ENC_IH)) {
    TRY(wgrad_add(dGeT, G, xhatT, F, B, Bp, g, ldE));
    TRY(wgrad_add(dGeT, G, h1T, H, B, Bp, g + F, ldE));
    TRY(wgrad_add(dGeT, G, hdecpT, H, B, Bp, g + F + H, ldE));
    if (d.cvar) TRY(wgrad_add(dGeT, G, condT, c, B, Bp, g + F + 2 * H, ldE));
  }
  TRY(wgrad_add(dGeT, G, v.Wb("HETp"), H, B, Bp, Gr(SSCVAE_W_ENC_HH), H));
  TRY(wgrad_add(dmT, Z, v.Wb("HETc"), H, B, Bp, Gr(SSCVAE_W_FC_MEAN_W), H));
  TRY(wgrad_add(dlT, Z, v.Wb("HETc"), H, B, Bp, Gr(SSCVAE_W_FC_LOGVAR_W), H));
  TRY(wgrad_launch());
  // attention LSTM (W_ih column blocks [emb | avg | h1 | h_dec]; W_hh shares the h1 operand), query / image projections, head
  const bf16* dGaT = v.Wb("dGaT");
  if (float* g = Gr(SSCVAE_W_ATT_IH)) {
    TRY(wgrad_add(dGaT, G, v.Wb("embT"), E, B, Bp, g, ldA));
    TRY(wgrad_add(dGaT, G, v.Ib("avgT"), F, B, Bp, g + E, ldA));
    TRY(wgrad_add(dGaT, G, h1pT, H, B, Bp, g + E + F, ldA));
    TRY(wgrad_add(dGaT, G, hdecp2T, H, B, Bp, g + E + F + H, ldA));
  }
  TRY(hh_pair(dGaT, h1pT, SSCVAE_W_ATT_IH, SSCVAE_W_ATT_HH));
  TRY(wgrad_add(v.Wb("dqT"), A, h1T, H, B, Bp, Gr(SSCVAE_W_QUERY_PROJ), H));
  TRY(wgrad_add(v.Wb("dheadT"), NO, v.Wb("hdT"), H, B, Bp, Gr(SSCVAE_W_OUT_PROJ_W), H));
  if (Gr(SSCVAE_W_IMAGE_PROJ) || Gr(SSCVAE_W_ATT_VEC))   // d P and d w_a from the score gradients d u (T = 1)
    TRY(attention_backward_deferred(s, aa, 1, v.Tf("q"), v.Wf("du"), v.Wf("dproj"), v.Wf("dwa")));
  if (Gr(SSCVAE_W_IMAGE_PROJ)) {
    TRY(transpose_f32_to_bf16(s, v.Wf("dproj"), BN, A, A, v.Wb("dPT"), BNp));
    TRY(wgrad_add(v.Wb("dPT"), A, v.Ib("featsT"), F, BN, BNp, Gr(SSCVAE_W_IMAGE_PROJ), F));
  }
  TRY(wgrad_launch());
  // bias sums, the sentiment column, W_hh copies, w_a, embedding rows
  if (csent) {
    if (Gr(SSCVAE_W_DEC_IH)) TRY(rowdot_bf16(s, dGdT, G, B, Bp, v.Tf("sent"), B, Gr(SSCVAE_W_DEC_IH) + F + 2 * H, ldD));
    if (Gr(SSCVAE_W_ENC_IH)) TRY(rowdot_bf16(s, dGeT, G, B, Bp, v.Tf("sent"), B, Gr(SSCVAE_W_ENC_IH) + F + 2 * H, ldE));
  }
  TRY(bias_pair(dGdT, SSCVAE_W_DEC_BIH, SSCVAE_W_DEC_BHH));
  TRY(bias_pair(dGeT, SSCVAE_W_ENC_BIH, SSCVAE_W_ENC_BHH));
  TRY(bias_pair(dGaT, SSCVAE_W_ATT_BIH, SSCVAE_W_ATT_BHH));
  TRY(hh_copy(SSCVAE_W_DEC_IH, F + H, ldD, SSCVAE_W_DEC_HH));
  TRY(hh_copy(SSCVAE_W_ATT_IH, E + F, ldA, SSCVAE_W_ATT_HH));
  if (Gr(SSCVAE_W_FC_MEAN_B)) TRY(rowsum_bf16(s, dmT, Z, B, Bp, Gr(SSCVAE_W_FC_MEAN_B), 0));
  if (Gr(SSCVAE_W_FC_LOGVAR_B)) TRY(rowsum_bf16(s, dlT, Z, B, Bp, Gr(SSCVAE_W_FC_LOGVAR_B), 0));
  if (Gr(SSCVAE_W_OUT_PROJ_B)) TRY(rowsum_bf16(s, v.Wb("dheadT"), NO, B, Bp, Gr(SSCVAE_W_OUT_PROJ_B), 0));
  if (Gr(SSCVAE_W_ATT_VEC)) TRY(colsum_f32(s, v.Wf("dwa"), B, A, A, Gr(SSCVAE_W_ATT_VEC)));
  if (!d.tied && Gr(SSCVAE_W_EMBEDDING)) {  // learned embedding: d emb rows = dG_att W_att_ih[:, :E], scattered by token id
    GemmSeg sg = seg(v.Wb("dGa"), Gp, v.Pb("w_att_eT"), Gp, G);
    GemmEpi e; e.tag = "gemm.wgrad"; e.C32 = v.Wf("dxemb"); e.ldc32 = E;
    TRY(gemm_bf16_tn(s, B, E, 1, &sg, e));
    CUDA_TRY(cudaMemsetAsync(Gr(SSCVAE_W_EMBEDDING), 0, (size_t)V * E * sizeof(float), s));
    TRY(embed_scatter_add_rows(s, v.Ti("tok"), B, d.pad, v.Wf("dxemb"), E, E, Gr(SSCVAE_W_EMBEDDING)));
  }
  return 0;
}

}  // namespace sscvae

using namespace sscvae;

extern "C" {

size_t sscvae_train_step_image_state_bytes(const SscvaeHandle* hh, int batch, int num_boxes) {
  const Handle* h = reinterpret_cast<const Handle*>(hh);
  if (!h || batch <= 0 || num_boxes <= 0) return 0;
  Plan p;
  plan_step_image(h->d, batch, num_boxes, p);
  return p.total;
}

size_t sscvae_train_step_tape_bytes(const SscvaeHandle* hh, int batch, int num_boxes) {
  const Handle* h = reinterpret_cast<const Handle*>(hh);
  if (!h || batch <= 0 || num_boxes <= 0) return 0;
  Plan p;
  plan_step_tape(h->d, batch, num_boxes, p);
  return p.total;
}

size_t sscvae_train_step_workspace_bytes(const SscvaeHandle* hh, int batch, int num_boxes) {
  const Handle* h = reinterpret_cast<const Handle*>(hh);
  if (!h || batch <= 0 || num_boxes <= 0) return 0;
  Plan p;
  plan_step_ws(h->d, batch, num_boxes, p);
  return p.total;
}

int sscvae_train_step_image_state(SscvaeHandle* hh, int batch, int num_boxes, const void* packed, const void* const* weights,
                                  const void* image_features, const float* obj_means, void* state, size_t state_bytes,
                                  void* stream) {
  Handle* h = reinterpret_cast<Handle*>(hh);
  REQUIRE(h && packed && weights && image_features, "NULL argument");
  REQUIRE(batch > 0 && num_boxes > 0, "batch/num_boxes must be positive");
  const Dims& d = h->d;
  REQUIRE(!d.cvar || obj_means != nullptr, "obj_means is required when sentiment_vae == 2");
  REQUIRE(aligned256(packed), "packed weights must be 256-byte aligned");
  Plan ip;
  plan_step_image(d, batch, num_boxes, ip);
  TRY(check_buffer("image state", state, state_bytes, ip.total));
  cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
  const int B = batch, N = num_boxes, BN = B * N;
  const char* pk = reinterpret_cast<const char*>(packed);
  char* is = reinterpret_cast<char*>(state);
  auto Ib = [&](const char* n) { return reinterpret_cast<bf16*>(is + ip.find(n)->off); };
  auto If = [&](const char* n) { return reinterpret_cast<float*>(is + ip.find(n)->off); };
  auto Pb = [&](const char* n) { return reinterpret_cast<const bf16*>(pk + h->pp.find(n)->off); };
  CUDA_TRY(cudaMemsetAsync(state, 0, ip.total, s));
  TRY(image_prep(s, image_features, h->opt_features_bf16, B, N, d.F, Ib("featsb"), d.Fp, If("mask"), Ib("avgb")));
  {  // P = W_v x (attention.py:125)
    GemmSeg sg = seg(Ib("featsb"), d.Fp, Pb("wv"), d.Fp, d.F);
    GemmEpi e; e.tag = "gemm.pre"; e.C16 = Ib("projb"); e.ldc16 = d.Ap;
    TRY(gemm_bf16_tn(s, BN, d.A, 1, &sg, e));
  }
  {  // time-invariant mean-feature block of the attention-LSTM gates
    GemmSeg sg = seg(Ib("avgb"), d.Fp, Pb("w_att_f"), d.Fp, d.F);
    GemmEpi e; e.tag = "gemm.pre"; e.C32 = If("gavg"); e.ldc32 = d.GP;
    TRY(gemm_bf16_tn(s, B, d.GP, 1, &sg, e));
  }
  TransposeJobList tj;   // operands of the W_v and mean-feature weight gradients
  TRY(tj.add(Ib("featsb"), BN, d.Fp, d.Fp, Ib("featsT"), round_up(BN, kPad)));
  TRY(tj.add(Ib("avgb"), B, d.Fp, d.Fp, Ib("avgT"), round_up(B, kPad)));
  TRY(transpose_bf16_jobs(s, tj));
  if (d.cvar) CUDA_TRY(cudaMemcpyAsync(If("objm"), obj_means, (size_t)BN * d.Z * sizeof(float), cudaMemcpyDeviceToDevice, s));
  return 0;
}

int sscvae_train_step_forward(SscvaeHandle* hh, int batch, int num_boxes, const void* packed, const void* const* weights,
                              const void* state, size_t state_bytes, const float* sentiment, const int64_t* prev_tokens,
                              const float* const* states_in, const float* eps, uint64_t seed, void* tape, size_t tape_bytes,
                              void* workspace, size_t workspace_bytes, float* logits, float* const* states_out, float* mean,
                              float* log_var, float* prior_mean_out, float* alpha, void* stream) {
  Handle* h = reinterpret_cast<Handle*>(hh);
  REQUIRE(h && packed && weights && prev_tokens && logits && states_out && mean && log_var && alpha, "NULL argument");
  for (int k = 0; k < 6; ++k) REQUIRE(states_out[k] != nullptr, "NULL argument: states_out needs all six states");
  REQUIRE(!states_in || (states_in[0] && states_in[1] && states_in[2] && states_in[3] && states_in[4] && states_in[5]),
          "NULL argument: states_in needs all six states (or is NULL for zero states)");
  REQUIRE(batch > 0 && num_boxes > 0, "batch/num_boxes must be positive");
  const Dims& d = h->d;
  const bool csent = d.cond && !d.cvar;
  REQUIRE(!csent || sentiment != nullptr, "sentiment is required when sentiment_vae == 1");
  REQUIRE(!d.cvar || prior_mean_out != nullptr, "prior_mean_out is required when sentiment_vae == 2");
  REQUIRE(aligned256(packed), "packed weights must be 256-byte aligned");
  StepViews v{reinterpret_cast<const char*>(packed), h->pp, weights, reinterpret_cast<char*>(const_cast<void*>(state)), Plan(),
              reinterpret_cast<char*>(tape), Plan(), reinterpret_cast<char*>(workspace), Plan()};
  plan_step_image(d, batch, num_boxes, v.ip);
  plan_step_tape(d, batch, num_boxes, v.tpl);
  plan_step_ws(d, batch, num_boxes, v.wpl);
  TRY(check_buffer("image state", state, state_bytes, v.ip.total));
  TRY(check_buffer("tape", tape, tape_bytes, v.tpl.total));
  TRY(check_buffer("workspace", workspace, workspace_bytes, v.wpl.total));
  return step_forward_impl(d, v, batch, num_boxes, sentiment, reinterpret_cast<const long long*>(prev_tokens), states_in, eps,
                           seed, logits, states_out, mean, log_var, prior_mean_out, alpha, reinterpret_cast<cudaStream_t>(stream));
}

int sscvae_train_step_backward(SscvaeHandle* hh, int batch, int num_boxes, const void* packed, const void* const* weights,
                               const void* state, size_t state_bytes, const void* tape, size_t tape_bytes, void* workspace,
                               size_t workspace_bytes, const float* d_logits, const float* const* d_states_out,
                               const float* d_mean, const float* d_log_var, const float* d_prior_mean, const float* d_alpha,
                               float* const* d_states_in, void* const* grads, void* stream) {
  Handle* h = reinterpret_cast<Handle*>(hh);
  REQUIRE(h && packed && weights && d_logits && grads, "NULL argument");
  REQUIRE(batch > 0 && num_boxes > 0, "batch/num_boxes must be positive");
  REQUIRE(aligned256(packed), "packed weights must be 256-byte aligned");
  const Dims& d = h->d;
  StepViews v{reinterpret_cast<const char*>(packed), h->pp, weights, reinterpret_cast<char*>(const_cast<void*>(state)), Plan(),
              reinterpret_cast<char*>(const_cast<void*>(tape)), Plan(), reinterpret_cast<char*>(workspace), Plan()};
  plan_step_image(d, batch, num_boxes, v.ip);
  plan_step_tape(d, batch, num_boxes, v.tpl);
  plan_step_ws(d, batch, num_boxes, v.wpl);
  TRY(check_buffer("image state", state, state_bytes, v.ip.total));
  TRY(check_buffer("tape", tape, tape_bytes, v.tpl.total));
  TRY(check_buffer("workspace", workspace, workspace_bytes, v.wpl.total));
  return step_backward_impl(d, v, batch, num_boxes, d_logits, d_states_out, d_mean, d_log_var, d_prior_mean, d_alpha,
                            d_states_in, grads, reinterpret_cast<cudaStream_t>(stream));
}

}  // extern "C"

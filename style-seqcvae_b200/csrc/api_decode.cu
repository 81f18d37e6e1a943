// C ABI: eval-mode decode (greedy / beam / constrained beam search) entirely on the device, plus the
// stand-alone search entry points used by the replay parity tests (include/sscvae.h).
//
// Rows r = (b*S + s)*K + k share image b's region features, projected features and mean-feature gate
// block through a row->image map; nothing image-sized is replicated per beam (the reference
// re-materialises (B*S*K, N, F) and re-projects it every step, updown_captioner.py:405-416).
#include "api_internal.cuh"
#include "search.cuh"

namespace sscvae {

// J > 1: "diverse sampling" (var_updown/scripts/inference.py:138-167 calls the model N_Z_SAMPLES times per image): every
// image is decoded J times with independent latent draws in ONE call. The search sees Bv = B*J independent sequences
// (virtual images); everything image-sized (features, projections, mean-feature gate block) stays at B and is shared
// through the row -> image map, so the per-step GEMMs run with M = B*J rows instead of J launches with M = B.
// With S > 1 or K > 1 every virtual image is one constrained beam search of S*K rows; its FSM table is the image's (the J
// samples share it) or its own (one machine per sample): `fsm_tables` = B or B*J (S,V) tables are packed.
static void plan_decode(const Dims& d, int B, int N, int S, int K, int J, int fsm_tables, Plan& p) {
  const size_t b = sizeof(bf16), f = 4;
  const size_t Bv = (size_t)B * J, R = Bv * S * K, BN = (size_t)B * N;
  const int Pmax = K;
  p.add("seed", 16);
  p.add("featsb", BN * d.Fp * b);
  p.add("mask", BN * f);
  p.add("avgb", (size_t)B * d.Fp * b);
  p.add("projb", BN * d.Ap * b);
  p.add("gavg", (size_t)B * d.GP * f);
  p.add("pm_row", B * f);
  p.add("sent", B * f);
  p.add("rowmap", R * 4);                   // row -> image
  p.add("rowmap_exp", R * 4);               // row -> its sequence's step-0 row
  p.add("rowmap0", Bv * 4);                 // step-0 row -> image
  p.add("start_tok", Bv * 4);
  p.add("XA0", R * 2 * d.Hp * b);
  p.add("XA1", R * 2 * d.Hp * b);
  p.add("c1a", R * d.H * f);
  p.add("c1b", R * d.H * f);
  p.add("cda", R * d.H * f);
  p.add("cdb", R * d.H * f);
  p.add("XE", R * (d.Fp + d.Hp) * b);
  p.add("embb_r", R * d.Ep * b);
  p.add("ZB", R * d.ZC * b);                 // [z | c]: c = the conditioning block of sentiment_vae == 2
  if (d.cvar) p.add("pm", R * d.Z * f);      // per-row prior mean of the current step (updown_cell.py:160-163)
  p.add("acc", R * d.GP * f);
  p.add("q", R * d.A * f);
  p.add("alpha_hist", (size_t)d.L * R * N * f);          // attention weights of every row of every step (step 0: Bv rows)
  if (d.tied) p.add("ob", R * d.Ep * b);
  p.add("logits", R * d.V * f);
  const size_t nst = gemm_rowstats_tiles(d.V);            // greedy: softmax statistics of the head GEMM instead of logits
  p.add("rs_max", R * nst * f);
  p.add("rs_sum", R * nst * f);
  p.add("rs_arg", R * nst * 4);
  p.add("fsm_bits", (size_t)fsm_tables * S * d.V * 4);
  p.add("cand_val", R * S * Pmax * f);
  p.add("cand_tok", R * S * Pmax * 4);
  p.add("tok_hist", (size_t)d.L * R * 4);
  p.add("bp_hist", (size_t)d.L * R * 4);
  p.add("score_hist", (size_t)d.L * R * f);
  p.add("best_samples", Bv * d.L * 8);                 // sscvae_decode_samples: the "best beam" copy of its predictions
  p.add("best_state", Bv * 4);                         // per search: the state whose beam 0 search_finish returned
  p.add("search_steps", Bv * 4);                       // per search: its step count (n_steps of its exit)
}

// The decode entry points record their shape, so sscvae_decode_attention finds the regions of the last call.
static void note_decode(Handle* h, int B, int N, int S, int K, int J, int fsm_tables) {
  h->last_B = B; h->last_N = N; h->last_S = S; h->last_K = K; h->last_J = J; h->last_T = fsm_tables;
}

const Plan& Handle::decode_plan(int B, int N, int S, int K, int J, int fsm_tables) {
  if (dp_B != B || dp_N != N || dp_S != S || dp_K != K || dp_J != J || dp_T != fsm_tables) {
    dp = Plan();
    plan_decode(d, B, N, S, K, J, fsm_tables, dp);
    dp_B = B; dp_N = N; dp_S = S; dp_K = K; dp_J = J; dp_T = fsm_tables;
  }
  return dp;
}

static inline GemmSeg seg(const bf16* A, int lda, const bf16* B, int ldb, int K) {
  GemmSeg s; s.A = A; s.lda = lda; s.B = B; s.ldb = ldb; s.K = K; return s;
}

// Named workspace regions and packed operands, shared by the fused decode and the single step.
struct Views {
  const char* pk; const Plan& pp; const void* const* wv; char* ws; const Plan& wp;
  const float* W(int i) const { return reinterpret_cast<const float*>(wv[i]); }
  const bf16* Pb(const char* n) const { return reinterpret_cast<const bf16*>(pk + pp.find(n)->off); }
  const float* Pf(const char* n) const { return reinterpret_cast<const float*>(pk + pp.find(n)->off); }
  bf16* Wb(const char* n) const { return reinterpret_cast<bf16*>(ws + wp.find(n)->off); }
  float* Wf(const char* n) const { return reinterpret_cast<float*>(ws + wp.find(n)->off); }
  int* Wi(const char* n) const { return reinterpret_cast<int*>(ws + wp.find(n)->off); }
};

// The per-image state (bf16 features, mask, mean, W_v projection, mean-feature gate block) depends on the images only:
// a caller that decodes the SAME batch again (the reference's loop over latent samples, inference.py:138-167; its
// lru_cache on the projected features, attention.py:99) sets the option "reuse_image_state" and this is skipped.
static int image_state(cudaStream_t s, const Handle* h, const Views& v, const void* feats, int B, int N) {
  const Dims& d = h->d;
  CUDA_TRY(cudaMemsetAsync(v.Wb("projb"), 0, v.wp.find("projb")->bytes, s));
  TRY(image_prep(s, feats, h->opt_features_bf16, B, N, d.F, v.Wb("featsb"), d.Fp, v.Wf("mask"), v.Wb("avgb")));
  GemmSeg sg = seg(v.Wb("featsb"), d.Fp, v.Pb("wv"), d.Fp, d.F);
  GemmEpi e; e.tag = "gemm.decode"; e.C16 = v.Wb("projb"); e.ldc16 = d.Ap;
  TRY(gemm_bf16_tn(s, B * N, d.A, 1, &sg, e));
  GemmSeg sa = seg(v.Wb("avgb"), d.Fp, v.Pb("w_att_f"), d.Fp, d.F);
  GemmEpi ea; ea.tag = "gemm.decode"; ea.C32 = v.Wf("gavg"); ea.ldc32 = d.GP;
  return gemm_bf16_tn(s, B, d.GP, 1, &sa, ea);
}

// Per-call buffers of one step of the cell; the other operands (embb_r, XE, ZB, acc, q, ob, pm and the per-image state) are
// named regions of the workspace.
struct CellIO {
  int rows, N, rows_per_image;                 // rows_per_image: consecutive rows of one image (the attention's grouping)
  const int* tokens; const int* rowmap;        // (rows) previous token; row -> image
  bool first;                                  // zero states: no recurrent GEMM segment, no previous cell state
  const float* eps; int eps_stride;            // normals of row r at eps[r * eps_stride * Z], or null -> Philox
  const unsigned long long* seed_dev; unsigned long long seed, step;   // Philox seed (device, else by value) and counter
  const bf16* xa_in; bf16* xa_out;             // [h1 | h_dec] bf16 operand rows (2 Hp) of the previous step / of this step
  const float* c1_in; float* c1_out; const float* cd_in; float* cd_out;
  float* h1_out; float* hd_out;                // optional fp32 h of this step
  float* alpha;                                // (rows, N)
  const float* sent; const float* pm_row;      // per image: sentiment column (sentiment_vae == 1), prior mean value
  const float* prior_mean; const float* prior_var; float* pm_out;   // optional (images,Z) prior; (rows,Z) mean used
  float* logits; const RowStatsEpi* rs;        // vocabulary head: fp32 logits and / or softmax statistics
};

// One eval step of the UpDown cell and the output head (updown_captioner.py:430-450, updown_cell.py:143-231).
static int decode_cell(cudaStream_t s, const Dims& d, const Views& v, const float* obj, const CellIO& c) {
  const int rows = c.rows, GP = d.GP, H = d.H, Hp = d.Hp, Fp = d.Fp, KXe = d.Fp + d.Hp, KX = d.KX;
  TRY(embed_gather_rows(s, c.tokens, rows, v.Pb("embb"), d.Ep, v.Wb("embb_r")));
  {
    LstmFwdArgs l = {};
    l.R = rows; l.H = H; l.add2 = v.Wf("gavg"); l.ld2 = GP; l.rowmap = c.rowmap; l.bias = v.Pf("b_att");
    l.c_prev = c.first ? nullptr : c.c1_in; l.c_out = c.c1_out;
    l.h1_dst = v.Wb("XE") + Fp; l.ld_h1 = KXe; l.h2_dst = c.xa_out; l.ld_h2 = 2 * Hp; l.h_out = c.h1_out;
    l.acc = v.Wf("acc"); l.ld_acc = GP; l.perm = 1;
    GemmSeg sg[2] = {seg(v.Wb("embb_r"), d.Ep, v.Pb("w_att_e"), d.Ep, d.E), seg(c.xa_in, 2 * Hp, v.Pb("w_att_rec"), 2 * Hp, 2 * Hp)};
    GemmEpi e; e.tag = "gemm.decode"; e.C32 = v.Wf("acc"); e.ldc32 = GP;
    TRY(gemm_bf16_tn(s, rows, GP, c.first ? 1 : 2, sg, e));
    TRY(lstm_forward(s, l));
  }
  {
    GemmSeg sg = seg(v.Wb("XE") + Fp, KXe, v.Pb("wq"), Hp, Hp);
    GemmEpi e; e.tag = "gemm.decode"; e.C32 = v.Wf("q"); e.ldc32 = d.A;
    TRY(gemm_bf16_tn(s, rows, d.A, 1, &sg, e));
    AttnArgs aa = {}; aa.R = rows; aa.N = c.N; aa.A = d.A; aa.Ap = d.Ap; aa.F = d.F; aa.Fp = Fp; aa.rowmap = c.rowmap;
    aa.q = v.Wf("q"); aa.ld_q = d.A; aa.proj = v.Wb("projb"); aa.feats = v.Wb("featsb"); aa.mask = v.Wf("mask");
    aa.w_a = v.W(SSCVAE_W_ATT_VEC);
    aa.rows_per_image = c.rows_per_image;
    TRY(attention_forward(s, aa, c.alpha, nullptr, v.Wb("XE"), KXe));
  }
  {  // eval: z ~ N(prior_mean, prior_var) (updown_cell.py:200-208); no encoder LSTM
    LatentArgs la = {}; la.R = rows; la.Z = d.Z; la.Zp = d.Zp; la.sentiment_vae = d.sv; la.prior_var = d.prior_std * d.prior_std;
    la.prior_mean_row = c.pm_row; la.rowmap = c.rowmap;
    la.prior_mean_img = c.prior_mean; la.prior_var_img = c.prior_var; la.pm_out = c.pm_out; la.seed = c.seed;
    if (d.cvar) {  // attribute-grounded prior: mean of this step from the row's attention weights; also the block c
      TRY(prior_mean_forward(s, c.alpha, obj, c.rowmap, rows, c.N, d.Z, v.Wf("pm"), v.Wb("ZB") + d.Zp, d.ZC, d.cond));
      la.prior_mean_full = v.Wf("pm");
    }
    TRY(latent_forward_eval(s, la, c.eps, c.eps_stride, c.seed_dev, c.step, v.Wb("ZB"), d.ZC));
  }
  {
    GemmSeg sg[3] = {seg(v.Wb("XE"), KXe, v.Pb("w_dec_x"), KX, KXe),
                     seg(v.Wb("ZB"), d.ZC, v.Pb("w_dec_z"), d.ZC, d.ZC),
                     seg(c.xa_in + Hp, 2 * Hp, v.Pb("w_dec_x") + KXe, KX, Hp)};
    LstmFwdArgs l = {};
    l.R = rows; l.H = H; l.bias = v.Pf("b_dec"); l.rowmap = c.rowmap;
    if (c.sent) { l.sent = c.sent; l.scol = v.Pf("scol_dec"); }
    l.c_prev = c.first ? nullptr : c.cd_in; l.c_out = c.cd_out;
    l.h1_dst = c.xa_out + Hp; l.ld_h1 = 2 * Hp; l.h_out = c.hd_out;
    l.acc = v.Wf("acc"); l.ld_acc = GP; l.perm = 1;
    GemmEpi e; e.tag = "gemm.decode"; e.C32 = v.Wf("acc"); e.ldc32 = GP;
    TRY(gemm_bf16_tn(s, rows, GP, c.first ? 2 : 3, sg, e));
    TRY(lstm_forward(s, l));
  }
  GemmEpi ev; ev.tag = "gemm.decode"; ev.rs = c.rs;
  if (c.logits) { ev.C32 = c.logits; ev.ldc32 = d.V; }
  if (d.tied) {
    GemmSeg sg = seg(c.xa_out + Hp, 2 * Hp, v.Pb("w_out"), Hp, Hp);
    GemmEpi e; e.tag = "gemm.decode"; e.bias = v.W(SSCVAE_W_OUT_PROJ_B); e.act = 1; e.C16 = v.Wb("ob"); e.ldc16 = d.Ep;
    TRY(gemm_bf16_tn(s, rows, d.E, 1, &sg, e));
    GemmSeg sv = seg(v.Wb("ob"), d.Ep, v.Pb("embb"), d.Ep, d.E);
    return gemm_bf16_tn(s, rows, d.V, 1, &sv, ev);
  }
  GemmSeg sg = seg(c.xa_out + Hp, 2 * Hp, v.Pb("w_out"), Hp, Hp);
  ev.bias = v.W(SSCVAE_W_OUT_PROJ_B);
  return gemm_bf16_tn(s, rows, d.V, 1, &sg, ev);
}

// gpf: search groups (virtual images) per FSM table and per num_constraints entry (1, or J when the samples of an image share
// its machine). exit_per_search: every group stops on its own (n_steps has B*J entries) instead of the batch together.
static int decode_impl(Handle* h, int B, int J, int N, int S, int K, int P, int gpf, bool exit_per_search,
                       const char* pk, const void* const* wv,
                       const void* feats, const float* sent, const float* obj, const uint8_t* fsm, const long long* num_constraints,
                       int min_sat, const float* eps, unsigned long long seed, char* ws, size_t ws_bytes,
                       long long* predictions, float* log_probs, long long* best, int32_t* n_steps, cudaStream_t s) {
  const Dims& d = h->d;
  REQUIRE(B > 0 && N > 0 && S >= 1 && S <= 32 && K >= 1 && K <= 8 && P >= 1 && P <= K, "bad decode shape B=%d N=%d S=%d K=%d P=%d", B, N, S, K, P);
  const bool csent = d.cond && !d.cvar;
  REQUIRE(!csent || sent != nullptr, "sentiment is required when sentiment_vae == 1");
  REQUIRE(!d.cvar || obj != nullptr, "obj_means is required when sentiment_vae == 2");
  REQUIRE(S == 1 || fsm != nullptr, "an FSM is required for more than one state");
  REQUIRE(J >= 1 && (gpf == 1 || gpf == J), "bad sample grouping J=%d groups per FSM=%d", J, gpf);
  const int Bv = B * J;
  const Plan& dp = h->decode_plan(B, N, S, K, J, Bv / gpf);
  if (ws_bytes < dp.total) { set_error("workspace too small: %zu < %zu", ws_bytes, dp.total); return SSCVAE_ERR_WORKSPACE; }
  REQUIRE((reinterpret_cast<uintptr_t>(ws) & 255) == 0 && (reinterpret_cast<uintptr_t>(pk) & 255) == 0,
          "workspace and packed weights must be 256-byte aligned");
  const Views v{pk, h->pp, wv, ws, dp};
  auto Wb = [&](const char* n) { return v.Wb(n); };
  auto Wf = [&](const char* n) { return v.Wf(n); };
  auto Wi = [&](const char* n) { return v.Wi(n); };
  auto zero = [&](const char* n) { return cudaMemsetAsync(ws + dp.find(n)->off, 0, dp.find(n)->bytes, s); };
  const int SK = S * K, R = Bv * SK, H = d.H, Hp = d.Hp, L = d.L;
  const unsigned long long* seed_dev = reinterpret_cast<const unsigned long long*>(ws + dp.find("seed")->off);
  (void)seed;

  CUDA_TRY(zero("XA0")); CUDA_TRY(zero("XA1")); CUDA_TRY(zero("XE")); CUDA_TRY(zero("bp_hist"));
  if (d.cvar) CUDA_TRY(zero("ZB"));                    // the padding columns behind c
  if (d.tied) CUDA_TRY(zero("ob"));
  if (!h->opt_reuse_image_state) TRY(image_state(s, h, v, feats, B, N));
  TRY(scale_rows_f32(s, csent ? sent : nullptr, d.mult, Wf("pm_row"), B));
  TRY(scale_rows_f32(s, csent ? sent : nullptr, 1.0f, Wf("sent"), B));
  TRY(iota_div_i32(s, Wi("rowmap"), R, SK * J));
  TRY(iota_div_i32(s, Wi("rowmap_exp"), R, SK));
  TRY(iota_div_i32(s, Wi("rowmap0"), Bv, J));
  TRY(fill_i32(s, Wi("start_tok"), d.boundary, Bv));                       // updown_captioner.py:326
  const uint32_t* fsm_bits = nullptr;
  if (fsm && h->opt_fsm_packed) {                      // already the (tables,S,V) uint32 bit table (sscvae_fsm_build / sscvae_fsm_pack)
    fsm_bits = reinterpret_cast<const uint32_t*>(fsm);
  } else if (fsm) {
    TRY(fsm_pack(s, fsm, Bv / gpf, S, d.V, reinterpret_cast<uint32_t*>(Wi("fsm_bits"))));
    fsm_bits = reinterpret_cast<uint32_t*>(Wi("fsm_bits"));
  }
  int* tok_hist = Wi("tok_hist"); int* bp_hist = Wi("bp_hist"); float* score_hist = Wf("score_hist");
  bf16* XA[2] = {Wb("XA0"), Wb("XA1")};
  float* c1[2] = {Wf("c1a"), Wf("c1b")};
  float* cd[2] = {Wf("cda"), Wf("cdb")};

  // Unconstrained K = 1 search (greedy decode, diverse sampling): arg max and log-sum-exp come out of the head GEMM's
  // epilogue (RowStatsEpi) and the (rows, V) fp32 logits are never written: -2 x rows x V x 4 bytes per step.
  const bool greedy = S == 1 && K == 1 && fsm == nullptr;
  RowStatsEpi rs;
  rs.mode = 1; rs.st_max = Wf("rs_max"); rs.st_sum = Wf("rs_sum"); rs.st_arg = Wi("rs_arg");
  const int nst = gemm_rowstats_tiles(d.V);
  auto cell = [&](int rows, const int* tokens, const int* rowmap, bool first, const float* eps_t, int eps_stride,
                  int step) -> int {
    CellIO c = {};
    c.rows = rows; c.N = N; c.rows_per_image = first ? J : SK * J;        // rowmap0: r / J ; rowmap: r / (SK * J)
    c.tokens = tokens; c.rowmap = rowmap; c.first = first;
    c.eps = eps_t; c.eps_stride = eps_stride; c.seed_dev = seed_dev; c.step = (unsigned long long)step;
    c.xa_in = XA[0]; c.xa_out = XA[1]; c.c1_in = c1[0]; c.c1_out = c1[1]; c.cd_in = cd[0]; c.cd_out = cd[1];
    c.alpha = Wf("alpha_hist") + (size_t)step * R * N;                   // kept for sscvae_decode_attention
    c.sent = csent ? Wf("sent") : nullptr; c.pm_row = Wf("pm_row");
    if (greedy) c.rs = &rs; else c.logits = Wf("logits");
    return decode_cell(s, d, v, obj, c);
  };

  // ---- step 0: one row per image, zero states (cbs.py:127-155)
  TRY(cell(Bv, Wi("start_tok"), Wi("rowmap0"), true, eps, SK, 0));
  if (greedy) {
    TRY(greedy_merge(s, rs.st_max, rs.st_sum, rs.st_arg, nst, Bv, nullptr, nullptr, d.boundary, tok_hist, nullptr, score_hist));
  } else {
    SearchRowsArgs a = {};
    a.logp = Wf("logits"); a.ld = d.V; a.V = d.V; a.normalized = 0; a.fsm_bits = fsm_bits; a.R = Bv; a.S = S; a.K = K;
    a.rows_per_image = 1; a.groups_per_fsm = gpf; a.P = K; a.end_index = d.boundary; a.neg_value = -INFINITY;
    a.cand_val = score_hist; a.cand_tok = tok_hist;
    TRY(search_rows(s, a));
  }
  TRY(gather_rows_bf16(s, XA[1], Wi("rowmap_exp"), R, 2 * Hp, 2 * Hp, XA[0]));
  TRY(gather_rows_f32(s, c1[1], Wi("rowmap_exp"), R, H, c1[0]));
  TRY(gather_rows_f32(s, cd[1], Wi("rowmap_exp"), R, H, cd[0]));
  // ---- steps 1..L-1 on all R rows (cbs.py:161-250); the early exit is resolved at the end
  for (int t = 1; t < L; ++t) {
    TRY(cell(R, tok_hist + (size_t)(t - 1) * R, Wi("rowmap"), false, eps ? eps + (size_t)t * R * d.Z : nullptr, 1, t));
    if (greedy) {
      TRY(greedy_merge(s, rs.st_max, rs.st_sum, rs.st_arg, nst, R, tok_hist + (size_t)(t - 1) * R, score_hist + (size_t)(t - 1) * R,
                       d.boundary, tok_hist + (size_t)t * R, bp_hist + (size_t)t * R, score_hist + (size_t)t * R));
      TRY(state_gather(s, bp_hist + (size_t)t * R, R, SK, XA[1], XA[0], 2 * Hp, c1[1], c1[0], cd[1], cd[0], H));
      continue;
    }
    SearchRowsArgs a = {};
    a.logp = Wf("logits"); a.ld = d.V; a.V = d.V; a.normalized = 0; a.fsm_bits = fsm_bits; a.R = R; a.S = S; a.K = K;
    a.rows_per_image = SK; a.groups_per_fsm = gpf; a.P = P; a.end_index = d.boundary; a.neg_value = -1e20f;
    a.last_tokens = tok_hist + (size_t)(t - 1) * R; a.last_scores = score_hist + (size_t)(t - 1) * R;
    a.cand_val = Wf("cand_val"); a.cand_tok = Wi("cand_tok");
    TRY(search_rows(s, a));
    TRY(search_merge(s, Wf("cand_val"), Wi("cand_tok"), Bv, S, K, P, tok_hist + (size_t)t * R, bp_hist + (size_t)t * R,
                     score_hist + (size_t)t * R));
    TRY(state_gather(s, bp_hist + (size_t)t * R, R, SK, XA[1], XA[0], 2 * Hp, c1[1], c1[0], cd[1], cd[0], H));
  }
  TRY(search_finish(s, tok_hist, bp_hist, score_hist, L, Bv, S, K, d.boundary, num_constraints, min_sat, gpf,
                    exit_per_search ? 1 : 0, predictions, log_probs, best, n_steps, Wi("best_state"), Wi("search_steps")));
  return 0;
}

// Single step (sscvae_decode_step). The per-image state comes first: its offsets depend on (B, N) only, so a call with
// another row count over the same workspace finds it in place. XA1, XE, ZB and ob are adjacent: one memset zeroes the
// K-padding of those operands (no kernel writes the padding columns, so it stays zero while the layout does not change).
static void plan_step(const Dims& d, int B, int R, int N, Plan& p) {
  const size_t b = sizeof(bf16), f = 4, BN = (size_t)B * N;
  p.add("featsb", BN * d.Fp * b);
  p.add("mask", BN * f);
  p.add("avgb", (size_t)B * d.Fp * b);
  p.add("projb", BN * d.Ap * b);
  p.add("gavg", (size_t)B * d.GP * f);
  p.add("pm_row", B * f);
  p.add("tok", R * 4);
  p.add("rowmap", R * 4);
  p.add("XA0", (size_t)R * 2 * d.Hp * b);
  p.add("XA1", (size_t)R * 2 * d.Hp * b);
  p.add("XE", (size_t)R * (d.Fp + d.Hp) * b);
  p.add("ZB", (size_t)R * d.ZC * b);
  if (d.tied) p.add("ob", (size_t)R * d.Ep * b);
  p.add("embb_r", (size_t)R * d.Ep * b);
  if (d.cvar) p.add("pm", (size_t)R * d.Z * f);
  p.add("acc", (size_t)R * d.GP * f);
  p.add("q", (size_t)R * d.A * f);
  const size_t nst = gemm_rowstats_tiles(d.V);
  p.add("rs_max", R * nst * f);
  p.add("rs_sum", R * nst * f);
  p.add("rs_arg", R * nst * 4);
}

const Plan& Handle::step_plan(int B, int R, int N) {
  if (sp_B != B || sp_R != R || sp_N != N) {
    sp = Plan();
    plan_step(d, B, R, N, sp);
    sp_B = B; sp_R = R; sp_N = N;
  }
  return sp;
}

}  // namespace sscvae

using namespace sscvae;

extern "C" {

int sscvae_fsm_pack(const uint8_t* fsm, int batch, int states, int vocab, uint32_t* fsm_bits, void* stream) {
  REQUIRE(fsm && fsm_bits && batch > 0 && vocab > 0, "bad argument");
  return fsm_pack(reinterpret_cast<cudaStream_t>(stream), fsm, batch, states, vocab, fsm_bits);
}

int sscvae_fsm_build(const int32_t* connections, const int32_t* connection_offsets, const int32_t* wordform_ids,
                     const int32_t* state_counts, int batch, int states, int vocab, uint32_t* fsm_bits, void* stream) {
  REQUIRE(connections && connection_offsets && wordform_ids && state_counts && fsm_bits && batch > 0 && vocab > 0, "bad argument");
  return fsm_build(reinterpret_cast<cudaStream_t>(stream), connections, connection_offsets, wordform_ids, state_counts, batch,
                   states, vocab, fsm_bits);
}

int sscvae_select_best_beam(const int64_t* predictions, const float* log_probs, const uint8_t* valid_states, int batch,
                            int states, int beam, int steps, int64_t* best, void* stream) {
  REQUIRE(predictions && log_probs && valid_states && best && batch > 0 && states > 0 && beam > 0 && steps > 0, "bad argument");
  return select_best_masked(reinterpret_cast<cudaStream_t>(stream), reinterpret_cast<const long long*>(predictions), log_probs,
                            valid_states, batch, states, beam, steps, reinterpret_cast<long long*>(best));
}

int sscvae_search_first_step(const float* logp, int batch, int states, int beam, int vocab, const uint32_t* fsm_bits,
                             int normalized, int32_t* tokens, float* scores, void* stream) {
  REQUIRE(logp && tokens && scores, "NULL argument");
  SearchRowsArgs a = {};
  a.logp = logp; a.ld = vocab; a.V = vocab; a.normalized = normalized; a.fsm_bits = fsm_bits; a.R = batch; a.S = states;
  a.K = beam; a.rows_per_image = 1; a.P = beam; a.end_index = -1; a.neg_value = -INFINITY;
  a.cand_val = scores; a.cand_tok = tokens;
  return search_rows(reinterpret_cast<cudaStream_t>(stream), a);
}

size_t sscvae_search_scratch_bytes(int batch, int states, int beam, int per_node) {
  return (size_t)batch * states * beam * states * per_node * 8 + 1024;
}

int sscvae_search_step(const float* logp, int batch, int states, int beam, int per_node, int vocab,
                       const uint32_t* fsm_bits, int normalized, int end_index, const int32_t* last_tokens,
                       const float* last_scores, void* scratch, size_t scratch_bytes, int32_t* tokens, int32_t* backptr,
                       float* scores, void* stream) {
  REQUIRE(logp && last_tokens && last_scores && scratch && tokens && backptr && scores, "NULL argument");
  const int R = batch * states * beam;
  const size_t n = (size_t)R * states * per_node;
  if (scratch_bytes < n * 8) { set_error("search scratch too small"); return SSCVAE_ERR_WORKSPACE; }
  float* cand_val = reinterpret_cast<float*>(scratch);
  int32_t* cand_tok = reinterpret_cast<int32_t*>(cand_val + n);
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  SearchRowsArgs a = {};
  a.logp = logp; a.ld = vocab; a.V = vocab; a.normalized = normalized; a.fsm_bits = fsm_bits; a.R = R; a.S = states;
  a.K = beam; a.rows_per_image = states * beam; a.P = per_node; a.end_index = end_index; a.neg_value = -1e20f;
  a.last_tokens = last_tokens; a.last_scores = last_scores; a.cand_val = cand_val; a.cand_tok = cand_tok;
  TRY(search_rows(st, a));
  return search_merge(st, cand_val, cand_tok, batch, states, beam, per_node, tokens, backptr, scores);
}

int sscvae_search_finish(const int32_t* tokens_hist, const int32_t* backptr_hist, const float* scores_hist, int steps_run,
                         int batch, int states, int beam, int end_index, const int64_t* num_constraints,
                         int min_constraints_to_satisfy, int64_t* predictions, float* final_scores, int64_t* best,
                         int32_t* n_steps, void* stream) {
  REQUIRE(tokens_hist && backptr_hist && scores_hist && predictions && final_scores && best && n_steps, "NULL argument");
  return search_finish(reinterpret_cast<cudaStream_t>(stream), tokens_hist, backptr_hist, scores_hist, steps_run, batch,
                       states, beam, end_index, reinterpret_cast<const long long*>(num_constraints),
                       min_constraints_to_satisfy, 1, 0, reinterpret_cast<long long*>(predictions), final_scores,
                       reinterpret_cast<long long*>(best), n_steps, nullptr, nullptr);
}

size_t sscvae_decode_workspace_bytes(const SscvaeHandle* hh, int batch, int num_boxes, int states, int beam) {
  Handle* h = const_cast<Handle*>(reinterpret_cast<const Handle*>(hh));
  if (!h || batch <= 0 || num_boxes <= 0 || states <= 0 || beam <= 0) return 0;
  return h->decode_plan(batch, num_boxes, states, beam, 1, batch).total;
}

size_t sscvae_decode_samples_workspace_bytes(const SscvaeHandle* hh, int batch, int samples, int num_boxes) {
  Handle* h = const_cast<Handle*>(reinterpret_cast<const Handle*>(hh));
  if (!h || batch <= 0 || num_boxes <= 0 || samples <= 0) return 0;
  return h->decode_plan(batch, num_boxes, 1, 1, samples, batch * samples).total;
}

int sscvae_decode_region(const SscvaeHandle* hh, int batch, int num_boxes, int states, int beam, const char* name,
                         size_t* offset, size_t* bytes) {
  Handle* h = const_cast<Handle*>(reinterpret_cast<const Handle*>(hh));
  REQUIRE(h && name && offset && bytes, "NULL argument");
  const Region* r = h->decode_plan(batch, num_boxes, states, beam, 1, batch).find(name);
  REQUIRE(r != nullptr, "unknown workspace region '%s'", name);
  *offset = r->off; *bytes = r->bytes;
  return 0;
}

int sscvae_decode(SscvaeHandle* hh, int batch, int num_boxes, int states, int beam, int per_node, const void* packed,
                  const void* const* weights, const float* image_features, const float* sentiment, const float* obj_means,
                  const uint8_t* fsm, const int64_t* num_constraints, int min_constraints_to_satisfy, const float* eps, uint64_t seed,
                  void* workspace, size_t workspace_bytes, int64_t* predictions, float* log_probs, int64_t* best,
                  int32_t* n_steps, void* stream) {
  Handle* h = reinterpret_cast<Handle*>(hh);
  REQUIRE(h && packed && weights && image_features && workspace && predictions && log_probs && best && n_steps, "NULL argument");
  REQUIRE(batch > 0 && num_boxes > 0 && states >= 1 && beam >= 1, "bad decode shape");
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  const Plan& dp = h->decode_plan(batch, num_boxes, states, beam, 1, batch);
  if (workspace_bytes < dp.total) { set_error("workspace too small: %zu < %zu", workspace_bytes, dp.total); return SSCVAE_ERR_WORKSPACE; }
  const unsigned long long seed_host = seed;
  CUDA_TRY(cudaMemcpyAsync(reinterpret_cast<char*>(workspace) + dp.find("seed")->off, &seed_host, sizeof(seed_host),
                           cudaMemcpyHostToDevice, st));
  std::vector<uint64_t> key;
  for (uint64_t v : {(uint64_t)batch, (uint64_t)num_boxes, (uint64_t)states, (uint64_t)beam, (uint64_t)per_node,
                     (uint64_t)min_constraints_to_satisfy, (uint64_t)workspace_bytes,
                     (uint64_t)(h->opt_fsm_packed * 4 + h->opt_features_bf16 * 2 + h->opt_reuse_image_state)})
    key_add(key, v);
  for (const void* q : {packed, (const void*)image_features, (const void*)sentiment, (const void*)obj_means, (const void*)fsm,
                        (const void*)num_constraints, (const void*)eps, (const void*)workspace, (const void*)predictions,
                        (const void*)log_probs, (const void*)best, (const void*)n_steps})
    key_add(key, q);
  for (int i = 0; i < SSCVAE_W_COUNT; ++i) key_add(key, weights[i]);
  note_decode(h, batch, num_boxes, states, beam, 1, batch);
  return run_with_graph(h->dec_graphs, key, st, true, [&](cudaStream_t s) {
    return decode_impl(h, batch, 1, num_boxes, states, beam, per_node, 1, false, reinterpret_cast<const char*>(packed), weights,
                       image_features, sentiment, obj_means, fsm, reinterpret_cast<const long long*>(num_constraints),
                       min_constraints_to_satisfy, eps, seed, reinterpret_cast<char*>(workspace), workspace_bytes,
                       reinterpret_cast<long long*>(predictions), log_probs, reinterpret_cast<long long*>(best), n_steps, s);
  });
}

int sscvae_decode_samples(SscvaeHandle* hh, int batch, int samples, int num_boxes, const void* packed,
                          const void* const* weights, const float* image_features, const float* sentiment,
                          const float* obj_means, const float* eps, uint64_t seed, void* workspace, size_t workspace_bytes, int64_t* predictions, float* log_probs,
                          int32_t* n_steps, void* stream) {
  Handle* h = reinterpret_cast<Handle*>(hh);
  REQUIRE(h && packed && weights && image_features && workspace && predictions && log_probs && n_steps, "NULL argument");
  REQUIRE(batch > 0 && num_boxes > 0 && samples >= 1, "bad decode shape");
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  const Plan& dp = h->decode_plan(batch, num_boxes, 1, 1, samples, batch * samples);
  if (workspace_bytes < dp.total) { set_error("workspace too small: %zu < %zu", workspace_bytes, dp.total); return SSCVAE_ERR_WORKSPACE; }
  const unsigned long long seed_host = seed;
  CUDA_TRY(cudaMemcpyAsync(reinterpret_cast<char*>(workspace) + dp.find("seed")->off, &seed_host, sizeof(seed_host),
                           cudaMemcpyHostToDevice, st));
  std::vector<uint64_t> key;
  for (uint64_t v : {(uint64_t)batch, (uint64_t)num_boxes, (uint64_t)samples, (uint64_t)0x5a5a, (uint64_t)workspace_bytes,
                     (uint64_t)(h->opt_features_bf16 * 2 + h->opt_reuse_image_state)})
    key_add(key, v);
  for (const void* q : {packed, (const void*)image_features, (const void*)sentiment, (const void*)obj_means, (const void*)eps,
                        (const void*)workspace, (const void*)predictions, (const void*)log_probs, (const void*)n_steps})
    key_add(key, q);
  for (int i = 0; i < SSCVAE_W_COUNT; ++i) key_add(key, weights[i]);
  char* wsb = reinterpret_cast<char*>(workspace);
  long long* best = reinterpret_cast<long long*>(wsb + dp.find("best_samples")->off);
  note_decode(h, batch, num_boxes, 1, 1, samples, batch * samples);
  return run_with_graph(h->dec_graphs, key, st, true, [&](cudaStream_t s) {
    return decode_impl(h, batch, samples, num_boxes, 1, 1, 1, 1, false, reinterpret_cast<const char*>(packed), weights, image_features,
                       sentiment, obj_means, nullptr, nullptr, 0, eps, seed, wsb, workspace_bytes, reinterpret_cast<long long*>(predictions),
                       log_probs, best, n_steps, s);
  });
}

// Constrained beam search per latent sample (the reference's loop over N_Z_SAMPLES, inference.py:138-167, with USE_CBS): every
// (image, sample) pair is one search of S*K rows, group g = b*J + j. Each search stops on its own, as the reference's batch-1
// call does (cbs.py:167 over that call's rows only).
static bool samples_search_shape_ok(int batch, int samples, int num_boxes, int states, int beam, int per_node, int fsm_per_sample) {
  return batch > 0 && samples >= 1 && num_boxes > 0 && states >= 1 && states <= 32 && per_node >= 1 && per_node <= beam &&
         beam <= 8 && (fsm_per_sample == 0 || fsm_per_sample == 1);
}

size_t sscvae_decode_samples_search_workspace_bytes(const SscvaeHandle* hh, int batch, int samples, int num_boxes, int states,
                                                    int beam, int fsm_per_sample) {
  Handle* h = const_cast<Handle*>(reinterpret_cast<const Handle*>(hh));
  if (!h || !samples_search_shape_ok(batch, samples, num_boxes, states, beam, 1, fsm_per_sample)) return 0;
  return h->decode_plan(batch, num_boxes, states, beam, samples, fsm_per_sample ? batch * samples : batch).total;
}

int sscvae_decode_samples_search_region(const SscvaeHandle* hh, int batch, int samples, int num_boxes, int states, int beam,
                                        int fsm_per_sample, const char* name, size_t* offset, size_t* bytes) {
  Handle* h = const_cast<Handle*>(reinterpret_cast<const Handle*>(hh));
  REQUIRE(h && name && offset && bytes, "NULL argument");
  REQUIRE(samples_search_shape_ok(batch, samples, num_boxes, states, beam, 1, fsm_per_sample),
          "bad decode shape B=%d J=%d N=%d S=%d K=%d", batch, samples, num_boxes, states, beam);
  const Region* r = h->decode_plan(batch, num_boxes, states, beam, samples, fsm_per_sample ? batch * samples : batch).find(name);
  REQUIRE(r != nullptr, "unknown workspace region '%s'", name);
  *offset = r->off; *bytes = r->bytes;
  return 0;
}

int sscvae_decode_samples_search(SscvaeHandle* hh, int batch, int samples, int num_boxes, int states, int beam, int per_node,
                                 const void* packed, const void* const* weights, const float* image_features,
                                 const float* sentiment, const float* obj_means, const uint8_t* fsm, int fsm_per_sample,
                                 const int64_t* num_constraints, int min_constraints_to_satisfy, const float* eps,
                                 uint64_t seed, void* workspace, size_t workspace_bytes, int64_t* predictions,
                                 float* log_probs, int64_t* best, int32_t* n_steps, void* stream) {
  Handle* h = reinterpret_cast<Handle*>(hh);
  REQUIRE(h && packed && weights && image_features && workspace && predictions && log_probs && best && n_steps, "NULL argument");
  REQUIRE(samples_search_shape_ok(batch, samples, num_boxes, states, beam, per_node, fsm_per_sample),
          "bad decode shape B=%d J=%d N=%d S=%d K=%d P=%d fsm_per_sample=%d (1 <= S <= 32, 1 <= P <= K <= 8)", batch, samples,
          num_boxes, states, beam, per_node, fsm_per_sample);
  REQUIRE(states == 1 || fsm != nullptr, "an FSM is required for more than one state");
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  const Plan& dp = h->decode_plan(batch, num_boxes, states, beam, samples, fsm_per_sample ? batch * samples : batch);
  if (workspace_bytes < dp.total) { set_error("workspace too small: %zu < %zu", workspace_bytes, dp.total); return SSCVAE_ERR_WORKSPACE; }
  const unsigned long long seed_host = seed;
  CUDA_TRY(cudaMemcpyAsync(reinterpret_cast<char*>(workspace) + dp.find("seed")->off, &seed_host, sizeof(seed_host),
                           cudaMemcpyHostToDevice, st));
  std::vector<uint64_t> key;
  for (uint64_t v : {(uint64_t)batch, (uint64_t)num_boxes, (uint64_t)samples, (uint64_t)states, (uint64_t)beam,
                     (uint64_t)per_node, (uint64_t)fsm_per_sample, (uint64_t)min_constraints_to_satisfy, (uint64_t)0x5c5c,
                     (uint64_t)workspace_bytes,
                     (uint64_t)(h->opt_fsm_packed * 4 + h->opt_features_bf16 * 2 + h->opt_reuse_image_state)})
    key_add(key, v);
  for (const void* q : {packed, (const void*)image_features, (const void*)sentiment, (const void*)obj_means, (const void*)fsm,
                        (const void*)num_constraints, (const void*)eps, (const void*)workspace, (const void*)predictions,
                        (const void*)log_probs, (const void*)best, (const void*)n_steps})
    key_add(key, q);
  for (int i = 0; i < SSCVAE_W_COUNT; ++i) key_add(key, weights[i]);
  note_decode(h, batch, num_boxes, states, beam, samples, fsm_per_sample ? batch * samples : batch);
  return run_with_graph(h->dec_graphs, key, st, true, [&](cudaStream_t s) {
    return decode_impl(h, batch, samples, num_boxes, states, beam, per_node, fsm_per_sample ? 1 : samples, true,
                       reinterpret_cast<const char*>(packed), weights, image_features, sentiment, obj_means, fsm,
                       reinterpret_cast<const long long*>(num_constraints), min_constraints_to_satisfy, eps, seed,
                       reinterpret_cast<char*>(workspace), workspace_bytes, reinterpret_cast<long long*>(predictions),
                       log_probs, reinterpret_cast<long long*>(best), n_steps, s);
  });
}

int sscvae_decode_attention(SscvaeHandle* hh, const void* workspace, size_t workspace_bytes, const uint8_t* valid_states,
                            float* attention_all, float* attention_best, void* stream) {
  Handle* h = reinterpret_cast<Handle*>(hh);
  REQUIRE(h && workspace && attention_best, "NULL argument");
  REQUIRE(h->last_B > 0, "no decode call on this handle yet");
  const Plan& dp = h->decode_plan(h->last_B, h->last_N, h->last_S, h->last_K, h->last_J, h->last_T);
  REQUIRE(workspace_bytes >= dp.total, "workspace too small for the last decode call: %zu < %zu", workspace_bytes, dp.total);
  const char* ws = reinterpret_cast<const char*>(workspace);
  auto Wi = [&](const char* n) { return reinterpret_cast<const int32_t*>(ws + dp.find(n)->off); };
  return search_attention(reinterpret_cast<cudaStream_t>(stream), Wi("tok_hist"), Wi("bp_hist"),
                          reinterpret_cast<const float*>(ws + dp.find("score_hist")->off),
                          reinterpret_cast<const float*>(ws + dp.find("alpha_hist")->off), h->d.L, h->last_B * h->last_J,
                          h->last_S, h->last_K, h->last_N, h->d.boundary, Wi("search_steps"), Wi("best_state"), valid_states,
                          attention_all, attention_best);
}


size_t sscvae_decode_step_workspace_bytes(const SscvaeHandle* hh, int batch, int rows, int num_boxes) {
  Handle* h = const_cast<Handle*>(reinterpret_cast<const Handle*>(hh));
  if (!h || batch <= 0 || rows <= 0 || num_boxes <= 0 || rows % batch != 0) return 0;
  return h->step_plan(batch, rows, num_boxes).total;
}

int sscvae_decode_step(SscvaeHandle* hh, int batch, int rows, int num_boxes, const void* packed, const void* const* weights,
                       const float* image_features, const float* sentiment, const float* obj_means, const float* prior_mean,
                       const float* prior_var, const int64_t* prev_tokens, const float* const* states_in, const float* eps,
                       uint64_t seed, void* workspace, size_t workspace_bytes, float* log_probs, float* const* states_out,
                       float* alpha, float* prior_mean_out, void* stream) {
  Handle* h = reinterpret_cast<Handle*>(hh);
  REQUIRE(h && packed && weights && image_features && prev_tokens && workspace && log_probs && states_out && alpha &&
          prior_mean_out, "NULL argument");
  REQUIRE(states_out[0] && states_out[1] && states_out[2] && states_out[3], "NULL argument: states_out needs h1, c1, h_decoder, c_decoder");
  REQUIRE(!states_in || (states_in[0] && states_in[1] && states_in[4] && states_in[5]),
          "NULL argument: states_in needs h1, c1, h_decoder and c_decoder (or is NULL for zero states)");
  REQUIRE(batch > 0 && rows > 0 && num_boxes > 0 && rows % batch == 0,
          "bad step shape B=%d R=%d N=%d (R must be a multiple of B: row r belongs to image r / (R/B))", batch, rows, num_boxes);
  const Dims& d = h->d;
  const bool csent = d.cond && !d.cvar;
  REQUIRE(!csent || sentiment != nullptr, "sentiment is required when sentiment_vae == 1");
  REQUIRE(!d.cvar || obj_means != nullptr, "obj_means is required when sentiment_vae == 2");
  const Plan& sp = h->step_plan(batch, rows, num_boxes);
  if (workspace_bytes < sp.total) { set_error("workspace too small: %zu < %zu", workspace_bytes, sp.total); return SSCVAE_ERR_WORKSPACE; }
  REQUIRE((reinterpret_cast<uintptr_t>(workspace) & 255) == 0 && (reinterpret_cast<uintptr_t>(packed) & 255) == 0,
          "workspace and packed weights must be 256-byte aligned");
  cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
  char* ws = reinterpret_cast<char*>(workspace);
  const Views v{reinterpret_cast<const char*>(packed), h->pp, weights, ws, sp};
  const int R = rows, rpi = rows / batch;
  // Launched directly, not through the graph cache: the cache keys a graph on every pointer of the call, and a search
  // hands the step new output buffers on every step, so each call would capture (and keep) a graph of its own.
  const bool reuse = h->opt_reuse_image_state != 0;
  if (!reuse || h->step_ws != workspace || h->step_R != R) {
    const Region* first = sp.find("XA1");
    const Region* last = sp.find(d.tied ? "ob" : "ZB");
    CUDA_TRY(cudaMemsetAsync(ws + first->off, 0, last->off + last->bytes - first->off, s));
  }
  if (!reuse) TRY(image_state(s, h, v, image_features, batch, num_boxes));
  h->step_ws = workspace; h->step_R = R;
  TRY(step_import(s, reinterpret_cast<const long long*>(prev_tokens), R, rpi, states_in ? states_in[0] : nullptr,
                  states_in ? states_in[4] : nullptr, d.H, d.Hp, v.Wi("tok"), v.Wi("rowmap"), v.Wb("XA0")));
  CellIO c = {};
  c.rows = R; c.N = num_boxes; c.rows_per_image = rpi; c.tokens = v.Wi("tok"); c.rowmap = v.Wi("rowmap");
  c.first = states_in == nullptr;
  c.eps = eps; c.eps_stride = 1; c.seed = seed;
  c.xa_in = v.Wb("XA0"); c.xa_out = v.Wb("XA1");
  c.c1_in = states_in ? states_in[1] : nullptr; c.cd_in = states_in ? states_in[5] : nullptr;
  c.h1_out = states_out[0]; c.c1_out = states_out[1]; c.hd_out = states_out[2]; c.cd_out = states_out[3];
  c.alpha = alpha;
  c.sent = csent ? sentiment : nullptr;
  if (!d.simple) {                                     // simple_vae: the prior mean is zero whatever is given (updown_cell.py:165-166)
    c.prior_mean = prior_mean;
    if (!prior_mean && csent) {                        // the prior forward() builds (updown_captioner.py:250-261)
      TRY(scale_rows_f32(s, sentiment, d.mult, v.Wf("pm_row"), batch));
      c.pm_row = v.Wf("pm_row");
    }
  }
  c.prior_var = prior_var; c.pm_out = prior_mean_out;
  RowStatsEpi rs;
  rs.mode = 1; rs.st_max = v.Wf("rs_max"); rs.st_sum = v.Wf("rs_sum"); rs.st_arg = v.Wi("rs_arg");
  c.logits = log_probs; c.rs = &rs;
  TRY(decode_cell(s, d, v, obj_means, c));
  return log_softmax_rows(s, rs.st_max, rs.st_sum, rs.st_arg, gemm_rowstats_tiles(d.V), R, d.V, log_probs);
}

}  // extern "C"

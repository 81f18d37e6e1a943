// Launch wrappers of the non-GEMM kernels of the var_updown decoder path. All pointers are device
// pointers; every function enqueues on `stream` and returns 0 / error code. Row index of every
// time-stacked buffer is r = t * B + b (time-major).
#pragma once
#include "common.cuh"

namespace sscvae {

// ---- pre-loop -----------------------------------------------------------------------------------
// a6 (updown_cell.py:233-270): mask = sum_f |x| > 0 ; avg = masked mean ; bf16 copy of the features.
// feats: fp32 (B,N,F), or bf16 when feats_bf16 != 0 (the bf16 feature cache, SURVEY 8(f)-3)
int image_prep(cudaStream_t s, const void* feats, int feats_bf16, int B, int N, int F, bf16* featsb, int Fp, float* mask,
               bf16* avgb);
// a16 (allennlp add_sentence_boundary_token_ids) + mask/lengths of the targets (updown_captioner.py:265-278)
int boundary_tokens(cudaStream_t s, const long long* caption_tokens, int B, int L, int pad, int boundary,
                    int* tok /*(B,L+2)*/, float* tmask /*(T,B)*/, float* lengths /*(B)*/);
// a4: embb[t*B+b, :] = Embb[tok[b, t], :]  (bf16 rows of Ep elements)
int embed_gather_train(cudaStream_t s, const int* tok, int B, int L, const bf16* embb, int Ep, bf16* out);
int embed_gather_rows(cudaStream_t s, const int* tokens, int R, const bf16* embb, int Ep, bf16* out);

// ---- LSTM pointwise (torch.nn.LSTMCell semantics, gate order i,f,g,o) ----------------------------
struct LstmFwdArgs {
  int R, H;
  const float* acc; int ld_acc;        // (R,4H) GEMM result
  const float* add1; int ld1;          // optional (R,4H)
  const float* add2; int ld2;          // optional (rows2,4H) indexed by rowmap (or row)
  const int* rowmap;                   // optional row -> add2/sent row
  const float* bias;                   // optional (4H)  (b_ih + b_hh)
  const float* sent; const float* scol;  // optional rank-1 term sent[row] * scol[4H]
  const float* c_prev;                 // (R,H) or null (zeros)
  float* c_out;                        // (R,H)
  float* gates_out;                    // optional (R,4H) activated gates, saved for BPTT
  bf16* h1_dst; int ld_h1;             // bf16 h -> up to two operand buffers
  bf16* h2_dst; int ld_h2;
  // 1: the columns of the GEMM outputs `acc`, `add1`, `add2` are in the gate-interleaved order of the packed forward LSTM weights (lstm_gate_row): tile of
  // 128 columns = 32 hidden units x 4 gates, so that one GEMM CTA owns all four gates of its units
  int perm;
};
// packed row / GEMM output column of gate k (0..3 = i,f,g,o) of hidden unit j
__host__ __device__ __forceinline__ int lstm_gate_row(int k, int j) { return (j >> 5) * 128 + k * 32 + (j & 31); }
static inline int lstm_gate_rows(int H) { return ((H + 31) / 32) * 128; }
int lstm_forward(cudaStream_t s, const LstmFwdArgs& a);

struct LstmBwdArgs {
  int R, H;
  const float* dh[3]; int ld_dh[3];    // up to three fp32 sources summed (null = skip)
  const float* dc_in;                  // (R,H) or null
  const float* gates;                  // (R,4H) saved activations
  const float* c_prev;                 // (R,H) or null (zeros)
  const float* c;                      // (R,H)
  bf16* dgates; int ld_dg;             // (R,4H) bf16 pre-activation grads (GEMM operand)
  float* dc_prev;                      // (R,H)
  int tiled;                           // 1: gates / c / c_prev are blocks in the row-tiled layout (lstm_tiled_*_offset, B = R)
};
int lstm_backward(cudaStream_t s, const LstmBwdArgs& a);

// ---- latent: reparameterised z, per-step KL (updown_cell.py:196-208, updown_captioner.py:295-303) ----
struct LatentArgs {
  int R, Z, Zp;
  int sentiment_vae;                   // 0: KL against N(0,1) ignoring the prior; else prior form
  float prior_var;                     // prior_std^2
  const float* prior_mean_row;         // (R) per-row prior mean value (broadcast over Z) or null (0)
  const int* rowmap;                   // optional row -> prior_mean_row index
  const float* prior_mean_full;        // sentiment_vae == 2: (R,Z) per-row, per-component prior mean of this step (replaces prior_mean_row)
  float* dpm_out;                      // backward, with prior_mean_full: (R,Z) gradient of the KL term w.r.t. the prior mean
};
// sentiment_vae == 2 (updown_cell.py:160-174): pm[r,:] = sum_n alpha[r,n] * obj[img(r),n,:]; the first `cond` components
// are also written as the bf16 conditioning block c of the encoder / decoder LSTM inputs (cond = Z: "glove", 1: "senti_word_net")
int prior_mean_forward(cudaStream_t s, const float* alpha, const float* obj, const int* rowmap, int R, int N, int Z,
                       float* pm /*(R,Z)*/, bf16* c_dst, int ld_c, int cond);
// d pm = dpm_kl + [d c of the decoder LSTM + d c of the encoder LSTM on the first `cond` components];
// dalpha[r,n] = obj[r,n,:] . d pm[r,:]   (training layout: image r)
int prior_mean_backward(cudaStream_t s, int R, int N, int Z, int cond, const float* dpm_kl, const float* dc_dec, int ld_dec,
                        const float* dc_enc, int ld_enc, const float* obj, float* dalpha /*(R,N)*/);
// training: ml (R,2Z) = [mean|log_var] pre-bias GEMM output
int latent_forward_train(cudaStream_t s, const LatentArgs& a, const float* ml, int ld_ml, const float* bias_ml,
                         const float* eps_in /*(R,Z) or null*/, const unsigned long long* seed_dev, unsigned long long step,
                         float* mean_out, float* logvar_out, float* eps_out, bf16* zb, int ld_z, float* kl_out);
// (the Philox seed is read from DEVICE memory so that a captured CUDA graph can be replayed with a new seed)
// eval: z = eps * prior_std + prior_mean
// eps row r is read at eps_in[r * eps_row_stride, :]
int latent_forward_eval(cudaStream_t s, const LatentArgs& a, const float* eps_in, int eps_row_stride,
                        const unsigned long long* seed_dev, unsigned long long step, bf16* zb, int ld_z);
int fill_i32(cudaStream_t s, int* dst, int value, int n);
int iota_div_i32(cudaStream_t s, int* dst, int n, int div);   // dst[i] = i / div
int latent_backward(cudaStream_t s, const LatentArgs& a, const float* dz, int ld_dz, const float* eps,
                    const float* mean, const float* logvar, const float* gkld /*(B)*/, const float* tmask_t /*(B)*/,
                    bf16* dml /*(R, ld) [dmean | dlogvar]*/, int ld_dml);

// ---- vocabulary cross-entropy (updown_captioner.py:457-466 + allennlp sequence_cross_entropy_with_logits) ----
int ce_forward(cudaStream_t s, const float* logits, int ld, int TB, int V, const int* tok, int B, int L,
               const float* tmask, float* lse, float* nll);
int loss_reduce(cudaStream_t s, const float* nll, const float* kl, const float* tmask, const float* lengths, int T,
                int B, float* loss, float* kld);
int ce_backward(cudaStream_t s, const float* logits, int ld, int TB, int V, const int* tok, int B, int L,
                const float* tmask, const float* lengths, const float* lse, const float* gloss, bf16* dlogits,
                int ld_d);

// vocabulary head with the softmax statistics in the GEMM epilogue (gemm.cuh: RowStatsEpi): the logits are never written
int ce_prepare(cudaStream_t s, const int* tok, int B, int L, const float* tmask, const float* lengths, const float* gloss /*or null*/,
               int* target /*(T*B)*/, float* gcoef /*(T*B) or null*/);
int ce_merge(cudaStream_t s, const float* st_max, const float* st_sum, const int* st_arg, int ntiles, int TB,
             const float* tgt_logit, float* lse, float* nll);
int greedy_merge(cudaStream_t s, const float* st_max, const float* st_sum, const int* st_arg, int ntiles, int R,
                 const int* last_tokens, const float* last_scores, int end_index, int* tok, int* bp, float* score);

// ---- layout helpers -------------------------------------------------------------------------------
int transpose_bf16(cudaStream_t s, const bf16* in, int rows, int cols, int ld_in, bf16* out, int ld_out);
int transpose_f32_to_bf16(cudaStream_t s, const float* in, int rows, int cols, int ld_in, bf16* out, int ld_out);
// out[r] = sum_c in[r, c]  (bf16 in, fp32 accumulate; one warp per row; deterministic)
int rowsum_bf16(cudaStream_t s, const bf16* in, int rows, int cols, int ld, float* out, int accumulate);
int rowsum_f32(cudaStream_t s, const float* in, int rows, int cols, int ld, float* out, int accumulate);
// out (rows, cols) bf16 with ld  <- fp32 in (rows, cols) with ld_in ; pad columns [cols, ld) zeroed
int convert_f32_to_bf16(cudaStream_t s, const float* in, int rows, int cols, int ld_in, bf16* out, int ld_out);
// sum over T of time-stacked (T, B, n) bf16 -> (B, n) bf16
int timesum_bf16(cudaStream_t s, const bf16* in, int T, int B, int n, int ld, bf16* out, int ld_out);
int add_f32(cudaStream_t s, float* dst, const float* src, size_t n);
// out[c] = sum_r in[r, c]   (thread per column, deterministic)
int colsum_f32(cudaStream_t s, const float* in, int rows, int cols, int ld, float* out);
// out[r * out_stride] = sum_c in[r, c] * vec[c % period]   (bf16 matrix row . periodic fp32 vector)
int rowdot_bf16(cudaStream_t s, const bf16* in, int rows, int cols, int ld, const float* vec, int period, float* out,
                int out_stride);
// strided fp32 block copy: dst[r*ld_dst + c] = src[r*ld_src + c]
int copy_block_f32(cudaStream_t s, const float* src, int ld_src, float* dst, int ld_dst, int rows, int cols);
// weight packing: dst (bf16) <- src (+ src2) fp32, optionally transposed
int pack_block(cudaStream_t s, bf16* dst, int ld_dst, int transposed, const float* src, int ld_src, int rows, int cols,
               const float* src2, int ld_src2);
// the same for a whole list of blocks in ONE launch (the per-step weight re-pack is ~30 blocks)
struct PackJob {
  const float* src; const float* src2; bf16* dst;
  int ld_src, ld_src2, ld_dst, rows, cols, transposed;
  int gate_H;                          // > 0: rows are (gate k, unit j) = r / gate_H, r % gate_H and go to row lstm_gate_row(k, j)
  int tile0, tiles_x;                  // filled by pack_blocks: first tile index, tiles along the columns
};
constexpr int kMaxPackJobs = 40;
struct PackJobList {
  PackJob job[kMaxPackJobs];
  int n = 0;
  int add(bf16* dst, int ld_dst, int transposed, const float* src, int ld_src, int rows, int cols, const float* src2,
          int ld_src2, int gate_H = 0);
};
int pack_blocks(cudaStream_t s, PackJobList& jobs);
int vec_add_f32(cudaStream_t s, const float* a, const float* b, float* out, int n);
// dst (rows, cols; ld_dst) = sum of `nparts` split-K partial tiles parts + z*stride (rows, cols; ld); dst may be parts
int sum_partials_f32(cudaStream_t s, float* dst, int ld_dst, const float* parts, size_t stride, int nparts, int rows,
                     int cols, int ld);
int scale_rows_f32(cudaStream_t s, const float* in, float scale, float* out, int n);
// dEmb[tok[b,t], :] += dx[(t*B+b), :] skipping the padding index (nn.Embedding padding_idx)
int embed_scatter_add(cudaStream_t s, const int* tok, int B, int L, int pad, const float* dx, int ld_dx, int E, float* demb);
int gather_rows_f32(cudaStream_t s, const float* src, const int* idx, int R, int n, float* dst);
int gather_rows_bf16(cudaStream_t s, const bf16* src, const int* idx, int R, int n, int ld, bf16* dst);

// ---- region attention (attention.py:36-97, updown_cell.py:156-158) -----------------------------
struct AttnArgs {
  int R, N, A, Ap, F, Fp;
  const int* rowmap;                   // row -> image (null = identity)
  const float* q; int ld_q;            // (R,A) projected query
  const bf16* proj;                    // (images, N, Ap) projected region features
  const bf16* feats;                   // (images, N, Fp)
  const float* mask;                   // (images, N)
  const float* w_a;                    // (A)
  int rows_per_image;                  // > 0: rows img*rows_per_image + i, i < rows_per_image, belong to image img (decode: the rows of
                                       // an image share its features; 0 = use rowmap / one image per row)
  const float* dalpha_extra;           // backward only: optional (R,N) added to d alpha (the attribute-grounded prior's path)
};
// smx (R,N): softmax(u*m) before the mask renormalisation, saved for the backward (null in decode)
int attention_forward(cudaStream_t s, const AttnArgs& a, float* alpha /*(R,N)*/, float* smx /*(R,N) or null*/, bf16* xhat,
                      int ld_x);
// per-step part of the backward: d q (bf16 GEMM operand) and d u (R,N), the score gradients kept for the deferred part
int attention_backward(cudaStream_t s, const AttnArgs& a, const float* smx, const float* dxhat, int ld_dx,
                       bf16* dq /*(R,Ap)*/, int ld_dq, float* du /*(R,N)*/);
// once after the time loop (training layout, a.R = B images, rows t*B+b): d P (B,N,A) and per-image d w_a rows (B,A),
// both overwritten
int attention_backward_deferred(cudaStream_t s, const AttnArgs& a, int T, const float* q_all /*(T,B,A)*/,
                                const float* du_all /*(T,B,N)*/, float* dproj, float* dwa_rows);

// ---- persistent recurrent kernel of the training forward pass (recurrent_fwd.cu) -----------------
// One cooperative launch runs all T timesteps of the UpDown cell for B <= 256 rows (training layout: row t*B + b,
// image b). Buffers and packed weights exactly as api_train.cu lays them out; the per-step outputs saved for BPTT
// (q, alpha, softmax, mean / log_var / eps, kl) are the ones the per-launch path writes; the activated gates and cell
// states are saved in the ROW-TILED layout below (lstm_backward: LstmBwdArgs::tiled).
struct RecFwdArgs {
  int B, T, H, Hp, Fp, Zp, Z, A, KX, GP, Ep;
  int sentiment_vae; float prior_var;
  const bf16* embb_t; const bf16* w_att_e;   // teacher-forced embeddings (T*B, Ep) and their attention-LSTM weight block
  const bf16* w_att_rec; const bf16* wq; const bf16* w_enc_x; const bf16* w_enc_hh; const bf16* w_fc; const bf16* w_dec_x;
  const bf16* w_dec_z;
  const float* gavg; const float* b_att; const float* b_enc; const float* b_dec;
  const float* sent; const float* scol_enc; const float* scol_dec;   // sent == null: no conditioning column
  float* c1; float* c_enc; float* c_dec; float* gates_att; float* gates_enc; float* gates_dec;
  bf16* XA; bf16* XE; bf16* HE; bf16* ZB;
  float* q;
  const float* b_fc; const float* eps_in; const unsigned long long* seed; const float* pm_row;
  float* mean; float* logvar; float* eps_out; float* kl_part; float* kl;
  AttnArgs att;                        // R = B, rowmap = null; q / ld_q unused
  float* alpha; float* smx;
  unsigned int* flags;                 // >= 1 KB of scratch for the dataflow counters
};
// Row-tiled layout of the saved LSTM state of ONE timestep (B rows, H % 4 == 0 units): 4 consecutive units of a row are
// 16 contiguous bytes and consecutive rows follow each other, so warps whose lanes are batch rows (the TMEM epilogues)
// access 512 contiguous bytes per instruction. Offsets in floats from the block of the timestep.
__host__ __device__ __forceinline__ size_t lstm_tiled_c_offset(int B, int b, int j) { return ((size_t)(j >> 2) * B + b) * 4 + (j & 3); }
__host__ __device__ __forceinline__ size_t lstm_tiled_gate_offset(int B, int b, int k, int j) {
  return (((size_t)(j >> 2) * 4 + k) * B + b) * 4 + (j & 3);
}
bool recurrent_forward_supported(const RecFwdArgs& r);
size_t recurrent_forward_kl_parts(int Z);   // number of per-row KL partial sums per timestep
int recurrent_forward(cudaStream_t s, const RecFwdArgs& r);

// ---- persistent kernel of the backward-through-time loop (recurrent_bwd.cu) -----------------------
// One cooperative launch runs the T reverse timesteps that api_train.cu otherwise issues as ten kernels per step. It
// reads the state the persistent forward kernel saved (row-tiled gates / cell states) and writes what the
// weight-gradient GEMMs behind the loop consume: dG_att / dG_enc / dG_dec (T*B, Gp), dml (T*B, Z2p), dqb (T*B, Ap) in
// bf16 (padding columns must be zero at entry) and du (T*B, N) (zero at entry: rows past the end of their caption are
// not visited). dc1 / dc_enc / dc_dec (B, H) must be zero at entry.
constexpr int RB_MAX_SPLIT_A = 2, RB_MAX_SPLIT_B = 4, RB_MAX_SPLIT_X = 4, RB_MAX_SPLIT_Z = 16;   // K splits (slots) per GEMM
struct RecBwdArgs {
  int B, T, H, Hp, Fp, Zp, Z, Z2p, A, Ap, KX, Gp;
  int sentiment_vae; float prior_var;
  int tiled;                           // layout of the saved gates / cell states: 1 row-tiled (lstm_tiled_*_offset), 0 row-major
  const bf16* w_dec_xzT; const bf16* w_enc_xhT; const bf16* w_att_recT; const bf16* w_fcT; const bf16* wqT;
  const float* gates_att; const float* gates_enc; const float* gates_dec;
  const float* c1; const float* c_enc; const float* c_dec;
  const float* mean; const float* logvar; const float* eps; const float* pm_row;
  const float* q; const float* smx;
  const float* dhead;                  // (T*B, H) fp32 row-major
  const float* gkld; const float* tmask;
  int* rows;                           // (T*B + T) ints of scratch: per-step list of the rows that still carry gradient
  float* dc1; float* dc_enc; float* dc_dec;
  bf16* dG_att; bf16* dG_enc; bf16* dG_dec; bf16* dml; bf16* dqb; float* du;
  float* dXEA;                         // RB_MAX_SPLIT_A x B x KX fp32 scratch
  float* dXEB;                         // RB_MAX_SPLIT_B x B x Hp
  float* dXA;                          // RB_MAX_SPLIT_X x B x 2Hp
  float* dzp;                          // RB_MAX_SPLIT_Z x B x Zp
  float* dhe_fc; float* dh1q;          // B x H each
  AttnArgs att;                        // R = B, rowmap = null; q / ld_q unused
  unsigned int* flags;                 // >= 256 B of scratch for the dataflow counters
};
bool recurrent_backward_supported(const RecBwdArgs& r);
bool recurrent_backward_tiling(const RecBwdArgs& r, int pairs, int out[12]);   // host only, no device needed
int recurrent_backward(cudaStream_t s, const RecBwdArgs& r);

extern unsigned long long g_launch_count_pw;   // launches from the non-GEMM kernels
}  // namespace sscvae

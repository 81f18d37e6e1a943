/* sscvae.h — C ABI of libsscvae_b200.so: the B200-native (sm_100a) implementation of the
 * Style-SeqCVAE `var_updown` sequential-decoder hot path.
 *
 * This is the drop-in boundary (SURVEY.md §8b). The reference has no FFI of its own — its hot path
 * is PyTorch eager code — so each entry point replaces a *Python* interface of the reference; the
 * reference-side binding (a ctypes stub inside the reference's UpDownCaptioner) is shown in
 * INTEGRATION.md. Paths below are relative to the reference root.
 *
 * Conventions
 *   - plain pointers and sizes only; every pointer is a DEVICE pointer unless it says "host".
 *   - the caller (PyTorch) owns all memory: inputs, outputs, packed weights and workspace. The
 *     library never allocates or frees caller-visible device memory and keeps no pointer after
 *     a call returns. The opaque handle holds host-side shape bookkeeping only.
 *   - every call enqueues work on `stream` (a cudaStream_t passed as void*) and returns
 *     immediately; 0 = success, <0 = SSCVAE_ERR_*, >0 = cudaError_t. No exception crosses the ABI;
 *     sscvae_last_error() returns the message of the last failure on the calling thread.
 *   - float tensors are fp32 row-major contiguous; token ids are int64 as in the reference.
 *   - not re-entrant on one handle; one handle per device.
 */
#ifndef SSCVAE_H_
#define SSCVAE_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SSCVAE_ABI_VERSION 6

#define SSCVAE_ERR_BAD_ARG (-1)
#define SSCVAE_ERR_WORKSPACE (-2)
#define SSCVAE_ERR_UNSUPPORTED (-3)
#define SSCVAE_ERR_DRIVER (-4)

/* Model dimensions and switches = the ctor arguments of the reference captioner
 * (var_updown/var_updown/models/updown_captioner.py:21-41) that shape the hot path. */
typedef struct SscvaeDims {
  int32_t image_feature_size;        /* F */
  int32_t embedding_size;            /* E */
  int32_t hidden_size;               /* H */
  int32_t attention_projection_size; /* A */
  int32_t z_space;                   /* Z */
  int32_t vocab_size;                /* V */
  int32_t max_caption_length;        /* L; teacher-forced steps T = L + 1 */
  int32_t sentiment_vae;             /* 0 | 1 | 2 (2 = attribute-grounded prior, updown_cell.py:160-174: per-step prior mean
                                        sum_n alpha_n * obj_means_n, also fed to the encoder / decoder LSTMs) */
  int32_t simple_vae;                /* 0 | 1 */
  int32_t tied_embedding;            /* 1: frozen embedding tied to the output layer + tanh projection (E in {300,600}) */
  int32_t pad_index;                 /* "@@UNKNOWN@@"  */
  int32_t boundary_index;            /* "@@BOUNDARY@@" */
  float prior_std;
  float senti_prior_multip;
  int32_t latent_embedding;          /* sentiment_vae == 2 only: 0 = "glove": the LSTM conditioning block is the whole prior mean
                                        (Z columns; the reference hard-codes 150 = its Z, updown_cell.py:63-70); 1 = "senti_word_net":
                                        its first column only (updown_cell.py:55-61, 168-171) */
} SscvaeDims;

/* Order of the weight / gradient pointer arrays = the reference state_dict (SURVEY §8b). */
enum SscvaeWeight {
  SSCVAE_W_EMBEDDING = 0,        /* _embedding_layer.weight                     (V,E)            */
  SSCVAE_W_ATT_IH,               /* _updown_cell._attention_lstm_cell.weight_ih (4H,E+F+2H)      */
  SSCVAE_W_ATT_HH,               /*                                  .weight_hh (4H,H)           */
  SSCVAE_W_ATT_BIH,              /*                                  .bias_ih   (4H)             */
  SSCVAE_W_ATT_BHH,              /*                                  .bias_hh   (4H)             */
  SSCVAE_W_QUERY_PROJ,           /* _butd_attention._query_vector_projection_layer.weight   (A,H) */
  SSCVAE_W_IMAGE_PROJ,           /* _butd_attention._image_features_projection_layer.weight (A,F) */
  SSCVAE_W_ATT_VEC,              /* _butd_attention._attention_layer.weight     (1,A)            */
  SSCVAE_W_ENC_IH,               /* _language_lstm_cell_encoder.weight_ih       (4H,F+2H+s)      */
  SSCVAE_W_ENC_HH,
  SSCVAE_W_ENC_BIH,
  SSCVAE_W_ENC_BHH,
  SSCVAE_W_DEC_IH,               /* _language_lstm_cell_decoder.weight_ih       (4H,F+2H+s+Z)    */
  SSCVAE_W_DEC_HH,
  SSCVAE_W_DEC_BIH,
  SSCVAE_W_DEC_BHH,
  SSCVAE_W_FC_MEAN_W,            /* fc_mean.weight (Z,H) */
  SSCVAE_W_FC_MEAN_B,
  SSCVAE_W_FC_LOGVAR_W,
  SSCVAE_W_FC_LOGVAR_B,
  SSCVAE_W_OUT_PROJ_W,           /* tied: _output_projection.0.weight (E,H)   | untied: _output_layer.weight (V,H) */
  SSCVAE_W_OUT_PROJ_B,           /* tied: _output_projection.0.bias   (E)     | untied: _output_layer.bias   (V)   */
  SSCVAE_W_COUNT
};

typedef struct SscvaeHandle SscvaeHandle;

int sscvae_abi_version(void);
const char* sscvae_last_error(void);
/* number of CUDA kernels this library has launched since it was loaded (bench.py `gpu_launches`) */
uint64_t sscvae_launch_count(void);

/* Replaces UpDownCaptioner.__init__ shape bookkeeping (updown_captioner.py:21-139). */
int sscvae_create(const SscvaeDims* dims, SscvaeHandle** out);
void sscvae_destroy(SscvaeHandle* h);

/* Packed bf16 operand copies of the weights (K-padded, recurrent blocks folded, transposed twins for
 * backward). Re-run after every optimizer step. `weights_f32` = host array of SSCVAE_W_COUNT device
 * pointers in reference layout. `dirty` = NULL for the first pack of a buffer (zero-fills the padding and
 * packs everything), else a host array of SSCVAE_W_COUNT flags: only blocks whose source weight is flagged
 * are re-packed (frozen weights — the tied embedding, the decoder LSTM under the freeze schedule of
 * var_updown/scripts/train.py:156-161 — cost nothing). */
size_t sscvae_packed_bytes(const SscvaeHandle* h);
int sscvae_pack_weights(SscvaeHandle* h, const void* const* weights_f32, void* packed, size_t packed_bytes,
                        const uint8_t* dirty, void* stream);

/* ---- training: replaces UpDownCaptioner.forward, training branch (updown_captioner.py:263-323),
 * i.e. _decode_step x T (:371-455), UpDownCell.forward (var_updown/var_updown/modules/updown_cell.py:86-231),
 * BottomUpTopDownAttention.forward (updown-baseline/updown/modules/attention.py:36-97), the KL terms
 * (:295-303) and _get_loss (:457-466). */
size_t sscvae_train_workspace_bytes(const SscvaeHandle* h, int batch, int num_boxes);
int sscvae_train_forward(SscvaeHandle* h, int batch, int num_boxes,
                         const void* packed,
                         const void* const* weights_f32,  /* host array; biases / w_a are read in fp32 */
                         const float* image_features,     /* (B,N,F) zero rows = padding boxes */
                         const int64_t* caption_tokens,   /* (B,L) pad = pad_index */
                         const float* sentiment,          /* (B,1) or NULL when sentiment_vae != 1 */
                         const float* obj_means,          /* (B,N,Z) per-box attribute means = the result of the reference's
                                                             translate_obj_atts2obj_means (updown_captioner.py:509-532);
                                                             required when sentiment_vae == 2, else NULL */
                         const float* eps,                /* (T,B,Z) N(0,1) draws, or NULL -> Philox(seed) */
                         uint64_t seed,
                         void* workspace, size_t workspace_bytes,
                         float* loss,                     /* out (B) */
                         float* kld,                      /* out (B) */
                         void* stream);
/* ---- replaces the autograd BPTT of `loss.backward()` (var_updown/scripts/train.py:172).
 * Must follow sscvae_train_forward on the same workspace. `grads_f32` = host array of
 * SSCVAE_W_COUNT device pointers in reference layout; NULL entries are skipped (frozen parameters:
 * the tied embedding always, the decoder LSTM under the freeze schedule of train.py:156-161).
 * Gradients are OVERWRITTEN, not accumulated. `group_events` = optional host array of
 * SSCVAE_GRAD_GROUPS cudaEvent_t recorded on `stream` as soon as a group's gradients are final,
 * so a data-parallel wrapper can start all-reducing that bucket while the rest still computes. */
#define SSCVAE_GRAD_GROUPS 5   /* 0 head, 1 decoder LSTM, 2 encoder LSTM + fc, 3 attention LSTM, 4 attention */
int sscvae_train_backward(SscvaeHandle* h, int batch, int num_boxes,
                          const void* packed, const void* const* weights_f32,
                          void* workspace, size_t workspace_bytes,
                          const float* grad_loss,         /* (B) dObjective/dloss_b */
                          const float* grad_kld,          /* (B) dObjective/dkld_b  */
                          void* const* grads_f32,
                          void* const* group_events,
                          void* stream);
/* Named view into the training workspace for tests ("logits", "alpha", "mean", "logvar", "kl", ...).
 * Returns 0 and fills offset/bytes, or SSCVAE_ERR_BAD_ARG for an unknown name. */
int sscvae_train_region(const SscvaeHandle* h, int batch, int num_boxes, const char* name, size_t* offset,
                        size_t* bytes);

/* ---- search: replaces ConstrainedBeamSearch.search (updown-baseline/updown/modules/cbs.py:59-277),
 * allennlp BeamSearch.search (in-tree text: var_updown/var_updown/modules/beam_search.py:592-766;
 * = the S=1, fsm==NULL case) and select_best_beam[_with_constraints]
 * (updown-baseline/updown/utils/decoding.py:10-138, cbs_simple). Declared in the search section below. */

/* One search step on given log-probabilities (replay / unit-test entry point, and the kernel the
 * full decode uses). Row r = (b*S + s)*K + k.
 *   first step : logp (B,V)      -> tokens/scores (B,S,K); backptr untouched
 *   later steps: logp (B*S*K,V)  -> tokens, backptr (index into the image's S*K rows), scores
 * fsm_bits: (B,S,V) uint32, bit i of fsm_bits[b,s,w] = reference fsm[b,s,i,w]; NULL = all allowed (plain beam).
 * normalized = 1: `logp` already holds log-softmax values; 0: raw logits, log-softmax is fused. */
int sscvae_fsm_pack(const uint8_t* fsm /*(B,S,S,V)*/, int batch, int states, int vocab, uint32_t* fsm_bits, void* stream);
/* The same bit table built ON THE DEVICE from the constraint word ids, replacing the dense tensors of
 * FiniteStateMachineBuilder.build (updown-baseline/updown/utils/constraints.py:329-478; 0.64 MB per image at S = 8,
 * V = 10 000) by a few dozen ints per image. The host lists the builder's _connect calls (:427-478) in call order:
 *   connections        (n,5) int32 rows {from_state, to_state, reset_state, first word-form, number of word-forms}
 *   connection_offsets (B+1) int32: image b owns rows [off[b], off[b+1])
 *   wordform_ids       int32 token ids the rows index into
 *   state_counts       (B,2) int32: {2**max_given_constraints = the states that start with a self loop on every word,
 *                      the number of states the image uses = the builder's next free sub-state}. The reference trims its
 *                      24-state tensor to that count (updown-baseline/updown/data/datasets.py:611-613): connections from or
 *                      to a state beyond it (a repeated constraint produces them) are dropped the same way.
 * `states` = the largest state count of the batch (states an image does not use stay without transitions, as in a
 * zero-padded batch). */
int sscvae_fsm_build(const int32_t* connections, const int32_t* connection_offsets, const int32_t* wordform_ids,
                     const int32_t* state_counts, int batch, int states, int vocab, uint32_t* fsm_bits, void* stream);
/* Best beam among an explicit set of valid states per image: the non-`cbs_simple` rule of select_best_beam_with_constraints
 * (updown-baseline/updown/utils/decoding.py:87-135), whose object / attribute state sets are host-side bookkeeping.
 * predictions (B,S,K,steps) int64, log_probs (B,S,K), valid_states (B,S) uint8 -> best (B,steps) = beam 0 of the valid
 * state with the highest beam-0 log-probability (first one on ties). */
int sscvae_select_best_beam(const int64_t* predictions, const float* log_probs, const uint8_t* valid_states, int batch,
                            int states, int beam, int steps, int64_t* best, void* stream);
int sscvae_search_first_step(const float* logp, int batch, int states, int beam, int vocab, const uint32_t* fsm_bits,
                             int normalized, int32_t* tokens, float* scores, void* stream);
int sscvae_search_step(const float* logp, int batch, int states, int beam, int per_node, int vocab,
                       const uint32_t* fsm_bits, int normalized, int end_index, const int32_t* last_tokens,
                       const float* last_scores, void* scratch, size_t scratch_bytes, int32_t* tokens,
                       int32_t* backptr, float* scores, void* stream);
size_t sscvae_search_scratch_bytes(int batch, int states, int beam, int per_node);
/* Back-trace (cbs.py:252-277) + early-exit step count (cbs.py:167) + best-beam selection.
 * tokens_hist / backptr_hist / scores_hist: (steps_run, B, S*K) as produced step by step [backptr entry 0 unused].
 * predictions (B,S,K,steps_run) int64 (entries >= n_steps are filled with end_index); final_scores (B,S,K) = the
 * scores at the reference's exit step; best (B,steps_run) int64; n_steps: device int32 = the number of steps the
 * reference would have produced (its early exit); num_constraints NULL -> plain beam rule (state 0, beam 0). */
int sscvae_search_finish(const int32_t* tokens_hist, const int32_t* backptr_hist, const float* scores_hist, int steps_run,
                         int batch, int states, int beam, int end_index, const int64_t* num_constraints,
                         int min_constraints_to_satisfy, int64_t* predictions, float* final_scores, int64_t* best,
                         int32_t* n_steps, void* stream);

/* ---- decode: replaces UpDownCaptioner.forward, eval branch (updown_captioner.py:324-366): runs the
 * whole search on the device. R = B*S*K rows, rows of one image share its region features.
 * eps: (max_steps, R, Z) external normals (parity) or NULL -> Philox(seed). Step 0 uses eps[0, b*S*K]
 * for image b (the reference draws a (B,Z) tensor there). */
size_t sscvae_decode_workspace_bytes(const SscvaeHandle* h, int batch, int num_boxes, int states, int beam);
int sscvae_decode(SscvaeHandle* h, int batch, int num_boxes, int states, int beam, int per_node,
                  const void* packed, const void* const* weights_f32,
                  const float* image_features, const float* sentiment,
                  const float* obj_means,             /* (B,N,Z) when sentiment_vae == 2 (rows of an image share them), else NULL */
                  const uint8_t* fsm,                 /* (B,S,S,V) uint8 as the reference passes it, or NULL */
                  const int64_t* num_constraints,     /* (B) or NULL */
                  int min_constraints_to_satisfy,
                  const float* eps, uint64_t seed,
                  void* workspace, size_t workspace_bytes,
                  int64_t* predictions,               /* out (B,S,K,L) */
                  float* log_probs,                   /* out (B,S,K) */
                  int64_t* best,                      /* out (B,L) */
                  int32_t* n_steps,                   /* out device int32: valid leading steps */
                  void* stream);

/* ---- diverse sampling: replaces the reference's loop `for k in range(N_Z_SAMPLES): model(image_features, ...)`
 * (var_updown/scripts/inference.py:138-167) over the eval branch with beam_size 1: every image is decoded `samples`
 * times with independent latent draws in ONE call. Row r = b*samples + j; rows of one image share its region
 * features, so the per-step GEMMs run with batch*samples rows. eps: (max_steps, batch*samples, Z) or NULL -> Philox. */
size_t sscvae_decode_samples_workspace_bytes(const SscvaeHandle* h, int batch, int samples, int num_boxes);
int sscvae_decode_samples(SscvaeHandle* h, int batch, int samples, int num_boxes,
                          const void* packed, const void* const* weights_f32,
                          const float* image_features, const float* sentiment, const float* obj_means,
                          const float* eps, uint64_t seed,
                          void* workspace, size_t workspace_bytes,
                          int64_t* predictions,               /* out (B,samples,L) */
                          float* log_probs,                   /* out (B,samples) */
                          int32_t* n_steps,                   /* out device int32: valid leading steps */
                          void* stream);

/* ---- diverse sampling under constrained beam search: the reference's inference loop
 * `for k in range(N_Z_SAMPLES): model(image_features, ..., fsm=..., num_constraints=...)` (var_updown/scripts/inference.py:138-167)
 * with USE_CBS, one constrained beam search per (image, sample), in ONE call. Search group g = b*samples + j owns the S*K rows
 * r = ((b*samples + j)*S + s)*K + k; all rows of an image share its region features, projections and mean-feature block.
 * Every search stops on its own, exactly as the reference's batch-1 call stops when all of ITS rows have emitted the boundary
 * token (updown-baseline/updown/modules/cbs.py:167): n_steps[b,j] is that call's step count, predictions / best of the search
 * hold the boundary token after it.
 *   fsm_per_sample 0: `fsm` is (B,S,S,V) uint8 (or, with option "fsm_packed", the (B,S,V) bit table) and num_constraints (B):
 *                     the samples of an image share its machine.
 *                  1: (B*samples,S,S,V) / (B*samples,S,V) and (B*samples): row b*samples + j is sample j's own machine.
 *   eps: (max_steps, B*samples*S*K, Z) or NULL -> Philox(seed); step 0 reads row (b*samples + j)*S*K.
 * Shapes: 1 <= S <= 32, 1 <= per_node <= beam <= 8, samples >= 1, an FSM whenever S > 1; otherwise SSCVAE_ERR_BAD_ARG
 * before any device work. The (B*samples*S*K, V) fp32 logits are part of the workspace. Options "fsm_packed",
 * "features_bf16" and "reuse_image_state" apply. */
size_t sscvae_decode_samples_search_workspace_bytes(const SscvaeHandle* h, int batch, int samples, int num_boxes,
                                                    int states, int beam, int fsm_per_sample);
int sscvae_decode_samples_search(SscvaeHandle* h, int batch, int samples, int num_boxes, int states, int beam, int per_node,
                                 const void* packed, const void* const* weights_f32,
                                 const float* image_features, const float* sentiment, const float* obj_means,
                                 const uint8_t* fsm, int fsm_per_sample,
                                 const int64_t* num_constraints, int min_constraints_to_satisfy,
                                 const float* eps, uint64_t seed,
                                 void* workspace, size_t workspace_bytes,
                                 int64_t* predictions,               /* out (B,samples,S,K,L) */
                                 float* log_probs,                   /* out (B,samples,S,K) */
                                 int64_t* best,                      /* out (B,samples,L) */
                                 int32_t* n_steps,                   /* out device int32 (B,samples) */
                                 void* stream);
/* Named view into the workspace of sscvae_decode_samples_search ("tok_hist", "bp_hist", "score_hist" (L,B*samples*S*K), ...). */
int sscvae_decode_samples_search_region(const SscvaeHandle* h, int batch, int samples, int num_boxes, int states, int beam,
                                        int fsm_per_sample, const char* name, size_t* offset, size_t* bytes);

/* ---- grounding: the attention weights over the boxes that stood behind every word (updown_captioner.py:371-455 returns
 * them as the last element of its eval step; attention.py:68-97). Every decode call keeps the (B*samples*S*K, N) weights
 * of each step in `workspace`; this call walks the back-pointers of each search from its exit step, as the back-trace of
 * the predictions does, and gathers, per word, the weights of the row whose log-probabilities chose it (word 0: the
 * search's single step-0 row). Words after a caption's first boundary token and steps at or after the search's own
 * n_steps are 0; the boundary word keeps its weights. Masked (all-zero) boxes are 0. One kernel launch.
 *
 * Attention over the boxes behind every word of the searches of the LAST decode call on this handle
 * (sscvae_decode / sscvae_decode_samples / sscvae_decode_samples_search) that filled `workspace`.
 * valid_states: (B*samples, S) uint8 when the caller applied the object/attribute rule (sscvae_select_best_beam),
 * else NULL (the rule search_finish applied). attention_all may be NULL.
 * samples = 1 for sscvae_decode; S = K = 1 for sscvae_decode_samples. Returns SSCVAE_ERR_BAD_ARG before any decode call on
 * the handle, for a NULL workspace or attention_best, and for a workspace smaller than the last call's. */
int sscvae_decode_attention(SscvaeHandle* h, const void* workspace, size_t workspace_bytes, const uint8_t* valid_states,
                            float* attention_all /* (B*samples,S,K,L,N) */, float* attention_best /* (B*samples,L,N) */,
                            void* stream);

/* Named view into the decode workspace for tests ("tok_hist", "bp_hist", "score_hist" (L,B*S*K), "alpha_hist" (L,B*S*K,N),
 * "logits", ...). */
int sscvae_decode_region(const SscvaeHandle* h, int batch, int num_boxes, int states, int beam, const char* name,
                         size_t* offset, size_t* bytes);

/* ---- one decode step: the reference's `_decode_step` in eval mode (updown_captioner.py:371-455), the step function its
 * forward hands to the search (updown_captioner.py:325-343), for callers that run their own search, rerank, or want the
 * per-step log-probabilities and states. R = rows rows; row r belongs to image r / (R/B), the aligned layout of every decode
 * call (the reference replicates image features with repeat_interleave but tiles sentiment / prior rows with `repeat`, which
 * agrees with this only at B = 1 or uniform sentiment: SURVEY §7 Q1).
 *   prior_mean, prior_var: (B,Z) per image, or NULL -> the prior forward() builds (sentiment * senti_prior_multip or 0;
 *     prior_std^2). With sentiment_vae == 2 the attention-weighted attribute mean replaces the mean (updown_cell.py:160-163);
 *     with simple_vae it is zero (updown_cell.py:165-166).
 *   prev_tokens: (R) int64 device ids in [0, V) (not checked here: the kernels index the embedding unchecked).
 *   states_in: host array of 6 device pointers (R,H) fp32 in the reference's order h1, c1, h_encoder, c_encoder, h_decoder,
 *     c_decoder (the encoder pair is not read in eval and may be NULL), or NULL = zero states (the search's first step).
 *   eps: (R,Z) normals, or NULL -> Philox(seed); a caller passes a new seed per call.
 *   Outputs (device, fp32): log_probs (R,V) = log-softmax of the step's logits; states_out = host array of 4 device
 *     pointers (R,H): h1, c1, h_decoder, c_decoder; alpha (R,N) attention weights; prior_mean_out (R,Z) the prior mean of
 *     the step (the prior log-variance the reference also returns is log(prior_var) of the row's image).
 * Options "features_bf16" and "reuse_image_state" (the workspace holds this batch's per-image state from an earlier step
 * call; it stays valid across calls with another row count) apply. R % B != 0, a NULL required pointer, or a missing
 * sentiment / obj_means return SSCVAE_ERR_BAD_ARG before any device work. Not captured as a CUDA graph. */
size_t sscvae_decode_step_workspace_bytes(const SscvaeHandle* h, int batch, int rows, int num_boxes);
int sscvae_decode_step(SscvaeHandle* h, int batch, int rows, int num_boxes, const void* packed, const void* const* weights_f32,
                       const float* image_features, const float* sentiment, const float* obj_means,
                       const float* prior_mean, const float* prior_var, const int64_t* prev_tokens,
                       const float* const* states_in, const float* eps, uint64_t seed, void* workspace,
                       size_t workspace_bytes, float* log_probs, float* const* states_out, float* alpha,
                       float* prior_mean_out, void* stream);

/* ---- one training step: the reference's `_decode_step` in training mode (updown_captioner.py:371-455 with the encoder branch
 * of updown_cell.py:176-198), the body of its training loop (updown_captioner.py:282-310), with a backward, so a caller can
 * build its own per-step objective (per-step KL weights, free bits, losses on the attention, scheduled sampling) and
 * back-propagate it through autograd. One row per image (R = B). Three caller-owned device buffers, 256-byte aligned:
 *   image state: the per-image operands of one batch, built by sscvae_train_step_image_state from the features, the per-box
 *     attribute means (sentiment_vae == 2) and the current weights. Every step over that batch reads it; build a new one for
 *     other features or after a weight update (replaces the reference's per-step re-projection, attention.py:99-125).
 *   tape: what one step's backward reads, written by its forward; one per step, kept until its backward has run.
 *   workspace: scratch of one call; any forward or backward of this handle may reuse it (calls on one stream).
 * The step neither reads nor returns the prior except with sentiment_vae == 2, where the prior mean is computed from the
 * attention (updown_cell.py:160-163): the caller forms the KL term (updown_captioner.py:295-303) from mean / log_var and
 * its prior. Not captured as a CUDA graph; no host synchronisation. */
size_t sscvae_train_step_image_state_bytes(const SscvaeHandle* h, int batch, int num_boxes);   /* 0 for bad arguments */
size_t sscvae_train_step_tape_bytes(const SscvaeHandle* h, int batch, int num_boxes);
size_t sscvae_train_step_workspace_bytes(const SscvaeHandle* h, int batch, int num_boxes);
/* image_features (B,N,F) fp32, or bf16 with the option "features_bf16"; obj_means (B,N,Z), required with sentiment_vae == 2
 * (NULL otherwise). */
int sscvae_train_step_image_state(SscvaeHandle* h, int batch, int num_boxes, const void* packed, const void* const* weights_f32,
                                  const void* image_features, const float* obj_means, void* state, size_t state_bytes,
                                  void* stream);
/* Forward of one step.
 *   sentiment: (B,1), required with sentiment_vae == 1 (the conditioning column, updown_cell.py:176-190), else NULL.
 *   prev_tokens: (B) int64 device ids in [0, V) (not checked here: the kernels index the embedding unchecked).
 *   states_in: host array of 6 device pointers (B,H) fp32, order h1, c1, h_encoder, c_encoder, h_decoder, c_decoder, or
 *     NULL = zero states (the first step, updown_cell.py:131-140).
 *   eps: (B,Z) normals, or NULL -> Philox(seed); a caller passes a new seed per call.
 *   Outputs (device, fp32, written in full): logits (B,V) raw (not log-softmax); states_out: host array of 6 device
 *     pointers (B,H); mean, log_var (B,Z) the posterior (updown_cell.py:196-198); prior_mean_out (B,Z) the step's prior mean,
 *     sentiment_vae == 2 only (else ignored, may be NULL); alpha (B,N) the attention weights.
 * A NULL required pointer, an incomplete state array, a missing sentiment / prior_mean_out return SSCVAE_ERR_BAD_ARG, a
 * buffer that is too small SSCVAE_ERR_WORKSPACE, all before any device work. */
int sscvae_train_step_forward(SscvaeHandle* h, int batch, int num_boxes, const void* packed, const void* const* weights_f32,
                              const void* state, size_t state_bytes, const float* sentiment, const int64_t* prev_tokens,
                              const float* const* states_in, const float* eps, uint64_t seed, void* tape, size_t tape_bytes,
                              void* workspace, size_t workspace_bytes, float* logits, float* const* states_out, float* mean,
                              float* log_var, float* prior_mean_out, float* alpha, void* stream);
/* Backward of one step (the per-launch BPTT body of sscvae_train_backward for one timestep), reading the tape and image
 * state of its forward with the same packed weights.
 *   d_logits (B,V) required. d_states_out: host array of 6 (B,H) upstream gradients of states_out, a NULL entry (or a NULL
 *     array) meaning zero. d_mean, d_log_var (B,Z), d_alpha (B,N): NULL = zero. d_prior_mean (B,Z): sentiment_vae == 2 only
 *     (the prior mean is a function of alpha there), NULL = zero.
 *   d_states_in: host array of 6 (B,H) outputs for the input states' gradients, a NULL entry (or array) = not wanted.
 *   grads: SSCVAE_W_COUNT device pointers in reference layout, OVERWRITTEN with this step's gradients (not accumulated);
 *     NULL entries (frozen parameters) are skipped with their GEMMs. The tied embedding gets no gradient (frozen GloVe,
 *     updown_captioner.py:197-216). The untied embedding's padding row stays zero (padding_idx).
 * Refusals as for the forward, before any device work. */
int sscvae_train_step_backward(SscvaeHandle* h, int batch, int num_boxes, const void* packed, const void* const* weights_f32,
                               const void* state, size_t state_bytes, const void* tape, size_t tape_bytes, void* workspace,
                               size_t workspace_bytes, const float* d_logits, const float* const* d_states_out,
                               const float* d_mean, const float* d_log_var, const float* d_prior_mean, const float* d_alpha,
                               float* const* d_states_in, void* const* grads, void* stream);

/* ---- training-step tail (SURVEY §8(f)-1): clip_grad_norm_ + SGD(momentum, weight decay) fused over
 * a flat parameter buffer; replaces var_updown/scripts/train.py:173-176. */
int sscvae_grad_sqnorm(const float* grads, size_t n, float* partial /*>= 1024 floats*/, float* sqnorm_out, void* stream);
int sscvae_sgd_step(float* params, const float* grads, float* momentum_buf, size_t n, const float* sqnorm,
                    float max_norm, float lr, float momentum, float weight_decay, int first_step, void* stream);

/* The same for ALL parameter tensors in three launches (squared-norm partials, final sum, update). Host arrays of
 * `count` (<= 32) device pointers / sizes; scratch: device floats, at least sum(ceil(size_i / 16384)) + 1. The global
 * norm is reduced with a fixed chunking and ordered sums (bit-reproducible). grads[i] == NULL = a zero gradient (torch 1.1's
 * zero_grad() semantics for a frozen parameter). `grad_scale` multiplies every gradient before the norm and the update:
 * data-parallel ranks pass 1 / world_size and all-reduce SUMS (no separate averaging pass over the buckets). */
int sscvae_sgd_step_multi(int count, void* const* params, const void* const* grads, void* const* momentum_bufs,
                          const uint64_t* sizes, const int32_t* first_step, float max_norm, float lr, float momentum,
                          float weight_decay, float grad_scale, float* scratch, size_t scratch_floats, void* stream);

/* The same update for `count` weights of this handle's model, fused with the re-pack of their images in `packed` (a
 * buffer sscvae_pack_weights has filled from the current `weights`): afterwards `packed` equals a pack of the updated
 * weights, and no re-pack is needed before the next forward. Three launches: the two norm launches of
 * sscvae_sgd_step_multi and one update + pack launch. `weights` = SSCVAE_W_COUNT device pointers as for
 * sscvae_pack_weights; grads / momentum_bufs / first_step are indexed by weight id like them and read only for the
 * weights listed in order[0..count) (a NULL gradient = a zero gradient). `order` also fixes the summation order of the
 * norm: given the same tensors in the same order, results are bit-identical to sscvae_sgd_step_multi followed by
 * sscvae_pack_weights. Weights not listed are read (fold partners, bias sums), never written. */
int sscvae_sgd_step_packed(SscvaeHandle* h, const void* const* weights, const void* const* grads,
                           void* const* momentum_bufs, const int32_t* first_step, int count, const int32_t* order,
                           float max_norm, float lr, float momentum, float weight_decay, float grad_scale, void* packed,
                           size_t packed_bytes, float* scratch, size_t scratch_floats, void* stream);

/* Per-handle options consumed by the following calls (0 = default):
 *   "features_bf16"     1: every `image_features` pointer is bf16 (B,N,F) instead of fp32 - the bf16 feature cache of SURVEY
 *                       8(f)-3 (updown-baseline/updown/data/readers.py:21-139 reads fp32 from HDF5). Results are bit-identical
 *                       to the fp32 input rounded to bf16: the kernels round the features to bf16 first either way.
 *   "fsm_packed"        1: the `fsm` pointer of sscvae_decode is the (B,S,V) uint32 bit table (sscvae_fsm_build / sscvae_fsm_pack)
 *                       instead of the reference's (B,S,S,V) uint8 tensor.
 *   "reuse_image_state" 1: the decode workspace already holds the per-image state of THIS batch (bf16 features, mask, mean
 *                       features, W_v projection): sscvae_decode / sscvae_decode_samples / sscvae_decode_step skip recomputing it. The analogue
 *                       of the reference's lru_cache on the projected features (updown-baseline/updown/modules/attention.py:99). */
int sscvae_set_option(SscvaeHandle* h, const char* name, int value);

/* 1 if sscvae_train_backward runs the BPTT loop of this shape as the persistent kernel (csrc/recurrent_bwd.cu), 0 if it
 * runs the per-launch path, < 0 on error. Option "persistent_bwd" (default 1) = 0 forces the per-launch path (tests compare
 * the two). Replaces nothing in the reference: autograd owns its backward (var_updown/scripts/train.py:172). */
int sscvae_train_backward_is_persistent(const SscvaeHandle* h, int batch, int num_boxes);

/* Host-only (no device needed): the job map of the persistent BPTT kernel for `pairs` co-resident CTA pairs (74 on a B200),
 * out12 = {big pairs, small pairs, S6A tiles, S6A K parts, S6B tiles, parts, S10 tiles, parts, d z tiles, parts, S4 / S8 tiles,
 * their width}; returns 1, or 0 if the shape does not fit (the per-launch path is used). For the CPU tests of the tiling. */
int sscvae_debug_bptt_tiling(const SscvaeHandle* h, int batch, int num_boxes, int pairs, int32_t* out12);

/* Host-only (no device needed): the source blocks that sscvae_pack_weights and sscvae_sgd_step_packed build their jobs
 * from, 16 values per block: {weight id, fold partner id or -1, first column, rows, columns, row length of the weight, row
 * length of the partner, outputs, then per output (two slots): kind (0 plain bf16, 1 transposed bf16, 2 fp32; -1 unused),
 * byte offset in the packed buffer, leading dimension, gate_H (> 0: plain rows gate-interleaved)}. Returns the number of
 * blocks (<= max_jobs) or an error. For the CPU tests of the packed layout. */
int sscvae_debug_sgd_pack_jobs(const SscvaeHandle* h, int64_t* out, int max_jobs);

/* Optional instrumentation (off by default): CUDA events around every kernel launch of the library,
 * aggregated per kernel class. report() synchronises the device and writes a JSON object
 * {"class": {"count", "ms", "flops", "bytes"}} (algorithmic FLOPs / bytes as declared at the call site). */
int sscvae_profile_enable(int on);
int sscvae_profile_report(char* buf, size_t n);

/* generic bf16 TN GEMM exposed for unit tests of the tcgen05 kernel:
 * C32[M,N] = A[M,K] (bf16, lda) * B[N,K]^T (bf16, ldb) */
int sscvae_test_gemm(const void* A, int lda, const void* B, int ldb, int M, int N, int K, float* C32, int ldc,
                     const float* bias, int act_tanh, int accumulate, void* stream);

/* the skinny-M (M <= 256) swapped-operand CTA-pair kernel with a forced cluster split of K (1..4; 0 = the library's
 * choice of kernel and split; other values return SSCVAE_ERR_BAD_ARG), for unit tests and tools/gemm_bench.py */
int sscvae_test_gemm_splitk(const void* A, int lda, const void* B, int ldb, int M, int N, int K, float* C32, int ldc,
                            int splits, const float* bias, void* stream);

/* the grouped weight-gradient GEMM: nprob (1..8) problems C32_i[M_i, N_i] = A_i[M_i, K_i] * B_i[N_i, K_i]^T (bf16, plain
 * fp32 store with row pitch ldc_i) in one launch of the CTA-pair kernel, for unit tests and tools/wgrad_bench.py */
int sscvae_test_gemm_grouped(int nprob, const void* const* A, const int* lda, const void* const* B, const int* ldb,
                             const int* M, const int* N, const int* K, float* const* C32, const int* ldc, void* stream);

/* the job-table bf16 transpose of the weight-gradient phase: for each of njobs (1..8) jobs, out[c, r] = in[r, c] for
 * c < cols, r < ld_out, zero for r >= rows; one launch. ld_in, ld_out multiples of 8, bases 16-byte aligned. */
int sscvae_test_transpose_bf16(int njobs, const void* const* in, const int* rows, const int* cols, const int* ld_in,
                               void* const* out, const int* ld_out, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* SSCVAE_H_ */

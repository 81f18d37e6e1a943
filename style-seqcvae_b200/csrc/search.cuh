// Beam / constrained-beam (CBS) selection kernels (north_star kernel #5). See search.cu.
#pragma once
#include "common.cuh"

namespace sscvae {

// bits[b,s,w] bit i = fsm[b,s,i,w] != 0   (fsm is the reference's (B,S,S,V) uint8 adjacency tensor)
int fsm_pack(cudaStream_t st, const uint8_t* fsm, int B, int S, int V, uint32_t* bits);
// the same table built on the device from the builder's connection list (include/sscvae.h: sscvae_fsm_build)
int fsm_build(cudaStream_t st, const int32_t* rec, const int32_t* rec_off, const int32_t* wf, const int32_t* counts, int B,
              int S, int V, uint32_t* bits);
// best[b,:] = predictions[b, argmax_{s: valid[b,s]} scores[b,s,0], 0, :]
int select_best_masked(cudaStream_t st, const long long* predictions, const float* scores, const uint8_t* valid, int B, int S,
                       int K, int steps, long long* best);

// Per row r and to-state i: the P best words by (value desc, word index asc), where
//   value(w) = allowed(from_state(r), i, w) ? logp[r,w] : neg_value        (+ last_scores[r] afterwards)
// and rows whose previous token is `end_index` are forced to the one-hot row (0 at end, -inf elsewhere).
// rows_per_image = S*K (1 at the first step: every row is state 0): row r belongs to search group r / rows_per_image, whose
// FSM table is group / groups_per_fsm (0 or 1: one table per group; J: the J samples of an image share one). Output (R,S,P).
struct SearchRowsArgs {
  const float* logp; int ld; int V;
  int normalized;                 // 0: raw logits, log-softmax fused
  const uint32_t* fsm_bits;       // (tables,S,V) or null (everything allowed)
  int R, S, K, rows_per_image, P;
  int groups_per_fsm;             // search groups per FSM table; 0 = 1
  int end_index;
  const int32_t* last_tokens;     // (R) or null
  const float* last_scores;       // (R) or null
  float neg_value;                // -inf at the first step (cbs.py:135), -1e20 later (cbs.py:205)
  float* cand_val; int32_t* cand_tok;   // (R,S,P)
};
int search_rows(cudaStream_t st, const SearchRowsArgs& a);

// Per image b and to-state i: K best of the S*K*P candidates by (value desc, flat index asc);
// token = candidate word, backptr = flat index / P (cbs.py:220-231).
int search_merge(cudaStream_t st, const float* cand_val, const int32_t* cand_tok, int B, int S, int K, int P,
                 int32_t* tokens, int32_t* backptr, float* scores);

// Back-trace, early exit and best beam of B search groups of S*K rows. Group b reads num_constraints[b / groups_per_table].
// groups_per_exit = 0: one exit for the whole batch (n_steps[0], the reference's batched loop, cbs.py:167); g > 0: one exit
// per set of g consecutive groups (n_steps[b / g]); 1 = every search stops on its own, as a batch-1 call would.
// best_state / group_steps (B) int32, both or neither: the state whose beam 0 group b returned and the group's step count,
// kept for search_attention.
int search_finish(cudaStream_t st, const int32_t* tokens_hist, const int32_t* backptr_hist, const float* scores_hist,
                  int steps_run, int B, int S, int K, int end_index, const long long* num_constraints, int min_sat,
                  int groups_per_table, int groups_per_exit, long long* predictions, float* final_scores, long long* best,
                  int32_t* n_steps, int32_t* best_state, int32_t* group_steps);

// Attention over the boxes behind every word of the B finished searches (one launch): alpha_hist (L, B*S*K, N) holds the
// attention weights of every row of every step (step 0: rows 0..B-1, one per group). att_all (B,S,K,L,N) or null: every
// beam; att_best (B,L,N): beam 0 of the returned state, which is best_state[b], or, with valid (B,S) uint8, the state
// select_best_masked picks. Words after a beam's first end_index token and steps >= group_steps[b] are zero.
int search_attention(cudaStream_t st, const int32_t* tokens_hist, const int32_t* backptr_hist, const float* scores_hist,
                     const float* alpha_hist, int L, int B, int S, int K, int N, int end_index, const int32_t* group_steps,
                     const int32_t* best_state, const uint8_t* valid, float* att_all, float* att_best);

// new_state[r] = old_state[img(r)*SK + bp[r]] for the four recurrent tensors of the eval cell
int state_gather(cudaStream_t st, const int32_t* bp, int R, int SK, const bf16* xa_src, bf16* xa_dst, int ld_xa,
                 const float* c1_src, float* c1_dst, const float* cd_src, float* cd_dst, int H);

}  // namespace sscvae

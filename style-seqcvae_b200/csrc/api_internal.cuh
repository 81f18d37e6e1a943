// Internal declarations shared by the C-ABI translation units.
#pragma once
#include <algorithm>
#include <cstring>
#include <initializer_list>
#include <vector>
#include "../../include/sscvae.h"
#include "common.cuh"
#include "gemm.cuh"
#include "kernels.cuh"
#include "graph_cache.cuh"

namespace sscvae {

constexpr int kPad = 64;   // elements: operand row strides / column blocks are multiples of 128 bytes (see init_dims)


struct Dims {
  int F, E, H, A, Z, V, L, T;
  int sv, simple, tied, pad, boundary, cond;
  // sentiment_vae == 2 (updown_cell.py:160-190): the conditioning block of the encoder / decoder LSTM inputs is the per-step
  // prior mean (cond = Z columns, or 1 with latent_embedding "senti_word_net"), a time-varying bf16 operand kept next to z:
  // rows of ZB are [z (Zp) | c (Cp)], ZC = Zp + Cp. cvar = 0: Cp = 0 and ZC = Zp.
  int le, cvar, Cp, ZC;
  float prior_std, mult;
  int Fp, Ep, Hp, Ap, Zp, Vp, G, Gp, Z2, Z2p, KX;
  int debug_logits;                    // SSCVAE_DEBUG_LOGITS=1 at create: the training forward also stores the fp32 logits (tests)
  int GP;                              // rows of a packed forward LSTM weight block: gate-interleaved, lstm_gate_rows(H)
};
int init_dims(const SscvaeDims* in, Dims& d);

struct Region { const char* name; size_t off, bytes; };
struct Plan {
  std::vector<Region> regs;
  size_t total = 0;
  void add(const char* name, size_t bytes);
  const Region* find(const char* name) const;
};

struct Handle {
  Dims d;
  Plan pp;                 // packed weights
  Plan tp; int tp_B = -1, tp_N = -1;   // training workspace for the last (B,N)
  Plan dp; int dp_B = -1, dp_N = -1, dp_S = -1, dp_K = -1, dp_J = -1, dp_T = -1;   // decode workspace
  // shape of the last decode call (the plan above also follows workspace-size and region queries): sscvae_decode_attention
  int last_B = -1, last_N = -1, last_S = -1, last_K = -1, last_J = -1, last_T = -1;
  Plan sp; int sp_B = -1, sp_R = -1, sp_N = -1;   // single-step workspace (sscvae_decode_step)
  const void* step_ws = nullptr; int step_R = -1;  // workspace and row count of the last step call: its zeroed operand padding
  const Plan& step_plan(int B, int R, int N);
  GraphCache fwd_graphs, bwd_graphs, dec_graphs;
  // per-handle options (sscvae_set_option), consumed by the following calls
  int opt_features_bf16 = 0;           // image_features pointers are bf16 (B,N,F) instead of fp32
  int opt_reuse_image_state = 0;       // decode / step: the workspace already holds this batch's featsb / projb / mask / avg state
  int opt_persistent_bwd = 1;          // training: run the BPTT loop as the persistent kernel (recurrent_bwd.cu) when the shape fits
  int opt_fsm_packed = 0;              // decode: `fsm` is the (B,S,V) uint32 bit table, not the (B,S,S,V) uint8 tensor
  const Plan& train_plan(int B, int N);
  const Plan& decode_plan(int B, int N, int S, int K, int J, int fsm_tables);   // fsm_tables: (S,V) bit tables packed per call
};

}  // namespace sscvae

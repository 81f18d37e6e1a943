// Beam / constrained beam search selection (north_star kernel #5).
//
// The reference (updown-baseline/updown/modules/cbs.py:200-226) sweeps the (B,S,K,V) log-prob
// tensor S times per step (masked_fill + topk per to-state). Here every row's V log-probs are read
// ONCE per step: a warp walks the row, looks up a bit-packed FSM word (bit i = "this word moves
// from-state -> state i") and keeps, per to-state, a P-entry sorted list in registers; lists are
// merged across the warp with shuffles. A second small kernel picks the K best of the S*K*P
// candidates per (image, to-state). Ordering is (value desc, index asc) everywhere, which is the
// oracle's stable-sort tie-break, so tokens / back-pointers / scores are bit-exact given identical
// log-probs. Algorithmic bytes per row-step: V*4 (log-probs) + V*4 (FSM word), streamed coalesced.
#include "search.cuh"
#include "prof.cuh"
#include <algorithm>
#include <climits>

namespace sscvae {

extern unsigned long long g_launch_count_pw;
#define LAUNCHED() do { CUDA_TRY(cudaGetLastError()); ++g_launch_count_pw; } while (0)

__device__ __forceinline__ bool better(float a, int ia, float b, int ib) { return a > b || (a == b && ia < ib); }

__global__ void fsm_pack_kernel(const uint8_t* __restrict__ fsm, int S, int V, uint32_t* __restrict__ bits, size_t total) {
  const size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;     // (b*S + s)*V + w
  if (idx >= total) return;
  const size_t w = idx % V, bs = idx / V;
  uint32_t m = 0;
  for (int i = 0; i < S; ++i) m |= (fsm[(bs * S + i) * V + w] != 0 ? 1u : 0u) << i;
  bits[idx] = m;
}
int fsm_pack(cudaStream_t st, const uint8_t* fsm, int B, int S, int V, uint32_t* bits) {
  REQUIRE(S >= 1 && S <= 32, "CBS supports 1..32 FSM states (got %d)", S);
  const size_t total = (size_t)B * S * V;
  fsm_pack_kernel<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(fsm, S, V, bits, total);
  LAUNCHED();
  return 0;
}

// ---- FSM construction on the device (constraints.py:329-478) ----
// The host turns the constraints of an image into a short list of CONNECTIONS (from, to, reset, word-form ids), in the
// order the reference's builder makes them; a thread owns one (image, from-state, word) entry of the bit table and replays
// the connections of its from-state: its word-forms move to `to`, every other word goes (back) to `reset`
// (constraints.py:427-478: reset_state is always given, so the second half of _connect always runs). The reference builds in
// a 24-state tensor and trims it to the states in use afterwards (datasets.py:611-613): a repeated constraint makes it connect
// states beyond that count, so connections from / to a state >= the image's count are dropped here the same way.
__global__ void fsm_build_kernel(const int32_t* __restrict__ rec, const int32_t* __restrict__ rec_off,
                                 const int32_t* __restrict__ wf, const int32_t* __restrict__ counts, int S, int V,
                                 uint32_t* __restrict__ bits) {
  const int w = blockIdx.x * blockDim.x + threadIdx.x, s = blockIdx.y, b = blockIdx.z;
  if (w >= V) return;
  const int n_main = counts[2 * b], n_used = counts[2 * b + 1];
  auto bit = [&](int x) { return (x >= 0 && x < n_used) ? 1u << x : 0u; };
  uint32_t m = s < n_main ? bit(s) : 0u;              // self loops for all words on the main states
  for (int i = rec_off[b]; i < rec_off[b + 1] && s < n_used; ++i) {
    const int32_t* r = rec + (size_t)i * 5;            // from, to, reset, first word-form, number of word-forms
    if (r[0] != s) continue;
    bool is_wf = false;
    for (int k = 0; k < r[4]; ++k) is_wf = is_wf || wf[r[3] + k] == w;
    if (is_wf) m |= bit(r[1]);
    m &= ~bit(s);
    if (is_wf) m &= ~bit(r[2]); else m |= bit(r[2]);
  }
  bits[((size_t)b * S + s) * V + w] = m;
}
int fsm_build(cudaStream_t st, const int32_t* rec, const int32_t* rec_off, const int32_t* wf, const int32_t* counts, int B,
              int S, int V, uint32_t* bits) {
  REQUIRE(S >= 1 && S <= 32, "CBS supports 1..32 FSM states (got %d)", S);
  fsm_build_kernel<<<dim3((V + 255) / 256, S, B), 256, 0, st>>>(rec, rec_off, wf, counts, S, V, bits);
  LAUNCHED();
  return 0;
}

// ---- the state whose beam 0 a finished search returns (decoding.py:82-135); score0[s * stride] = beam 0 of state s ----
//   valid != null: the caller's valid states (decoding.py:87-135, object / attribute rule);
//   nc >= 0:       cbs_simple, states s < 2^nc that satisfy min(nc, min_sat) constraints (decoding.py:82-86,128-134);
//   otherwise:     state 0 (plain beam search).
// The first maximum wins, like torch.argmax over the listed states; state 0 when no state qualifies.
__device__ __forceinline__ int select_state(const float* __restrict__ score0, int stride, int S, const uint8_t* __restrict__ valid, int nc,
                            int min_sat) {
  if (valid == nullptr && nc < 0) return 0;
  const int need = nc < min_sat ? nc : min_sat;
  int arg = 0; float v = 0.f; bool have = false;
  for (int s = 0; s < S; ++s) {
    if (valid ? !valid[s] : (s >= (1 << nc) || __popc(s) < need)) continue;
    const float x = score0[(size_t)s * stride];
    if (!have || x > v) { arg = s; v = x; have = true; }
  }
  return arg;
}

// ---- best beam among an explicit set of valid states (decoding.py:125-135 with the caller's valid_states) ----
__global__ void select_best_masked_kernel(const long long* __restrict__ predictions, const float* __restrict__ scores,
                                          const uint8_t* __restrict__ valid, int S, int K, int steps,
                                          long long* __restrict__ best) {
  const int b = blockIdx.x;
  __shared__ int s_best;
  if (threadIdx.x == 0) s_best = select_state(scores + (size_t)b * S * K, K, S, valid + (size_t)b * S, -1, 0);
  __syncthreads();
  const long long* src = predictions + (((size_t)b * S + s_best) * K) * steps;
  for (int t = threadIdx.x; t < steps; t += blockDim.x) best[(size_t)b * steps + t] = src[t];
}
int select_best_masked(cudaStream_t st, const long long* predictions, const float* scores, const uint8_t* valid, int B, int S,
                       int K, int steps, long long* best) {
  select_best_masked_kernel<<<B, 32, 0, st>>>(predictions, scores, valid, S, K, steps, best);
  LAUNCHED();
  return 0;
}

template <int P>
__device__ __forceinline__ void list_insert(float (&val)[P], int (&idx)[P], float v, int w) {
  if (!better(v, w, val[P - 1], idx[P - 1])) return;
  val[P - 1] = v; idx[P - 1] = w;
#pragma unroll
  for (int p = P - 1; p > 0; --p) {
    if (better(val[p], idx[p], val[p - 1], idx[p - 1])) {
      const float tv = val[p]; val[p] = val[p - 1]; val[p - 1] = tv;
      const int ti = idx[p]; idx[p] = idx[p - 1]; idx[p - 1] = ti;
    }
  }
}

// VEC = 4: 16-byte loads of the log-probs and of the FSM words (V % 4 == 0, 16-byte aligned rows). A warp walks its
// row with 313 dependent 4-byte loads per pass otherwise, which is latency-bound (341 us per step for 2560 rows of
// 10 000 log-probs; the 205 MB involved take 34 us at HBM speed).
template <int P, int SC, int VEC>
__global__ void __launch_bounds__(128) search_rows_kernel(SearchRowsArgs a) {
  const int r = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (r >= a.R) return;
  const int lane = threadIdx.x & 31;
  const int tab = r / (a.rows_per_image * (a.groups_per_fsm > 1 ? a.groups_per_fsm : 1));   // FSM table of the row's group
  const int s_from = (a.rows_per_image == 1) ? 0 : (r % a.rows_per_image) / a.K;
  const float* __restrict__ x = a.logp + (size_t)r * a.ld;
  const bool forced = a.last_tokens != nullptr && a.last_tokens[r] == a.end_index;   // cbs.py:177-181
  const int nv = a.V / VEC;
  float mx = 0.f, lsum = 0.f;
  if (!a.normalized && !forced) {
    float m = -INFINITY;
    if (VEC == 4) {
      const float4* x4 = reinterpret_cast<const float4*>(x);
#pragma unroll 4
      for (int i = lane; i < nv; i += 32) { const float4 v = x4[i]; m = fmaxf(m, fmaxf(fmaxf(v.x, v.y), fmaxf(v.z, v.w))); }
    } else {
      for (int w = lane; w < a.V; w += 32) m = fmaxf(m, x[w]);
    }
    m = warp_max(m);
    float s = 0.f;
    if (VEC == 4) {
      const float4* x4 = reinterpret_cast<const float4*>(x);
#pragma unroll 4
      for (int i = lane; i < nv; i += 32) {
        const float4 v = x4[i];
        s += (__expf(v.x - m) + __expf(v.y - m)) + (__expf(v.z - m) + __expf(v.w - m));
      }
    } else {
      for (int w = lane; w < a.V; w += 32) s += __expf(x[w] - m);
    }
    s = warp_sum(s);
    mx = m; lsum = logf(s);
  }
  const uint32_t* __restrict__ bits = a.fsm_bits ? a.fsm_bits + ((size_t)tab * a.S + s_from) * a.V : nullptr;
  for (int c0 = 0; c0 < a.S; c0 += SC) {
    float val[SC][P]; int idx[SC][P];
#pragma unroll
    for (int i = 0; i < SC; ++i)
#pragma unroll
      for (int p = 0; p < P; ++p) { val[i][p] = -INFINITY; idx[i][p] = INT_MAX; }
    auto visit = [&](float xv, uint32_t bw, int w) {
      float v;
      if (forced) v = (w == a.end_index) ? 0.f : -INFINITY;
      else v = a.normalized ? xv : (xv - mx) - lsum;
      const uint32_t b = bw >> c0;
#pragma unroll
      for (int i = 0; i < SC; ++i)
        if (c0 + i < a.S) list_insert<P>(val[i], idx[i], ((b >> i) & 1u) ? v : a.neg_value, w);
    };
    if (VEC == 4) {
      const float4* x4 = reinterpret_cast<const float4*>(x);
      const uint4* b4 = reinterpret_cast<const uint4*>(bits);
#pragma unroll 2
      for (int i = lane; i < nv; i += 32) {
        const float4 v = x4[i];
        const uint4 bw = bits ? b4[i] : make_uint4(0xffffffffu, 0xffffffffu, 0xffffffffu, 0xffffffffu);
        visit(v.x, bw.x, 4 * i); visit(v.y, bw.y, 4 * i + 1); visit(v.z, bw.z, 4 * i + 2); visit(v.w, bw.w, 4 * i + 3);
      }
    } else {
      for (int w = lane; w < a.V; w += 32) visit(x[w], bits ? bits[w] : 0xffffffffu, w);
    }
    const float add = a.last_scores ? a.last_scores[r] : 0.f;
#pragma unroll
    for (int i = 0; i < SC; ++i) {
      if (c0 + i >= a.S) break;
      for (int p = 0; p < P; ++p) {
        float bv = val[i][0]; int bi = idx[i][0];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
          const float ov = __shfl_xor_sync(0xffffffffu, bv, o);
          const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
          if (better(ov, oi, bv, bi)) { bv = ov; bi = oi; }
        }
        if (idx[i][0] == bi) {                         // winner pops its head
#pragma unroll
          for (int k = 0; k + 1 < P; ++k) { val[i][k] = val[i][k + 1]; idx[i][k] = idx[i][k + 1]; }
          val[i][P - 1] = -INFINITY; idx[i][P - 1] = INT_MAX;
        }
        if (lane == 0) {
          const size_t o = ((size_t)r * a.S + c0 + i) * P + p;
          a.cand_val[o] = a.last_scores ? bv + add : bv;     // cbs.py:210-212
          a.cand_tok[o] = bi;
        }
      }
    }
  }
}

// One CTA (8 warps) per row: the row is loaded ONCE into shared memory with every 16-byte load of the CTA in flight at
// the same time (the warp-per-row form issues ~80 dependent loads per pass and is latency-bound); max, sum-exp and the
// per-to-state selection then run from shared memory. Each warp keeps its own sorted lists over an interleaved
// slice of the row; the 8 x P warp winners of a state are merged by one warp with the same (value desc, index asc)
// order, so the result is identical to the warp-per-row kernel's.
template <int P, int SC>
__global__ void __launch_bounds__(256) search_rows_block_kernel(SearchRowsArgs a) {
  extern __shared__ __align__(16) float srow[];
  __shared__ float red[8];
  __shared__ float cv[8][SC][P];
  __shared__ int ci[8][SC][P];
  const int r = blockIdx.x;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int tab = r / (a.rows_per_image * (a.groups_per_fsm > 1 ? a.groups_per_fsm : 1));   // FSM table of the row's group
  const int s_from = (a.rows_per_image == 1) ? 0 : (r % a.rows_per_image) / a.K;
  const float4* __restrict__ x4 = reinterpret_cast<const float4*>(a.logp + (size_t)r * a.ld);
  float4* s4 = reinterpret_cast<float4*>(srow);
  const bool forced = a.last_tokens != nullptr && a.last_tokens[r] == a.end_index;   // cbs.py:177-181
  const int nv = a.V >> 2;
  float m = -INFINITY;
  for (int i = threadIdx.x; i < nv; i += 256) {
    const float4 v = x4[i];
    s4[i] = v;
    m = fmaxf(m, fmaxf(fmaxf(v.x, v.y), fmaxf(v.z, v.w)));
  }
  float mx = 0.f, lsum = 0.f;
  if (!a.normalized && !forced) {
    m = warp_max(m);
    if (lane == 0) red[warp] = m;
    __syncthreads();
    m = red[0];
#pragma unroll
    for (int w = 1; w < 8; ++w) m = fmaxf(m, red[w]);
    __syncthreads();
    float sum = 0.f;
    for (int i = threadIdx.x; i < nv; i += 256) {                       // own elements: no barrier needed yet
      const float4 v = s4[i];
      sum += (__expf(v.x - m) + __expf(v.y - m)) + (__expf(v.z - m) + __expf(v.w - m));
    }
    sum = warp_sum(sum);
    if (lane == 0) red[warp] = sum;
    __syncthreads();
    sum = 0.f;
#pragma unroll
    for (int w = 0; w < 8; ++w) sum += red[w];
    mx = m; lsum = logf(sum);
  }
  __syncthreads();
  const uint4* __restrict__ b4 = a.fsm_bits
      ? reinterpret_cast<const uint4*>(a.fsm_bits + ((size_t)tab * a.S + s_from) * a.V) : nullptr;
  const float add = a.last_scores ? a.last_scores[r] : 0.f;
  for (int c0 = 0; c0 < a.S; c0 += SC) {
    float val[SC][P]; int idx[SC][P];
#pragma unroll
    for (int i = 0; i < SC; ++i)
#pragma unroll
      for (int p = 0; p < P; ++p) { val[i][p] = -INFINITY; idx[i][p] = INT_MAX; }
    // A disallowed word enters a list with the constant neg_value. Once a thread has visited P words, every one of its
    // lists holds P entries that are >= neg_value with lower indices, PROVIDED no allowed word it has seen was below
    // neg_value (-inf log-probs, forced rows): from then on a disallowed word can never be inserted and only the set
    // bits of the FSM word (usually one) need the list test. `masked_matter` keeps the general path otherwise.
    bool masked_matter = true;
    bool seen_low = forced;
    int visited = 0;
    auto visit = [&](float xv, uint32_t bw, int w) {
      float v;
      if (forced) v = (w == a.end_index) ? 0.f : -INFINITY;
      else v = a.normalized ? xv : (xv - mx) - lsum;
      const uint32_t b = bw >> c0;
      if (masked_matter) {
#pragma unroll
        for (int i = 0; i < SC; ++i)
          if (c0 + i < a.S) list_insert<P>(val[i], idx[i], ((b >> i) & 1u) ? v : a.neg_value, w);
        seen_low |= !(v >= a.neg_value);
        masked_matter = (++visited < P) || seen_low;
      } else {
        if (!(v >= a.neg_value)) { masked_matter = true; seen_low = true; }
#pragma unroll
        for (int i = 0; i < SC; ++i)
          if (c0 + i < a.S && ((b >> i) & 1u)) list_insert<P>(val[i], idx[i], v, w);
      }
    };
    for (int i = threadIdx.x; i < nv; i += 256) {
      const float4 v = s4[i];
      const uint4 bw = b4 ? b4[i] : make_uint4(0xffffffffu, 0xffffffffu, 0xffffffffu, 0xffffffffu);
      visit(v.x, bw.x, 4 * i); visit(v.y, bw.y, 4 * i + 1); visit(v.z, bw.z, 4 * i + 2); visit(v.w, bw.w, 4 * i + 3);
    }
    // the warp's P best per state
#pragma unroll
    for (int i = 0; i < SC; ++i) {
      if (c0 + i >= a.S) break;
      for (int p = 0; p < P; ++p) {
        float bv = val[i][0]; int bi = idx[i][0];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
          const float ov = __shfl_xor_sync(0xffffffffu, bv, o);
          const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
          if (better(ov, oi, bv, bi)) { bv = ov; bi = oi; }
        }
        if (idx[i][0] == bi) {
#pragma unroll
          for (int k = 0; k + 1 < P; ++k) { val[i][k] = val[i][k + 1]; idx[i][k] = idx[i][k + 1]; }
          val[i][P - 1] = -INFINITY; idx[i][P - 1] = INT_MAX;
        }
        if (lane == 0) { cv[warp][i][p] = bv; ci[warp][i][p] = bi; }
      }
    }
    __syncthreads();
    // merge: warp i handles state c0 + i; a lane holds up to two of the 8*P warp winners
    for (int i = warp; i < SC && c0 + i < a.S; i += 8) {
      float v0 = -INFINITY, v1 = -INFINITY; int i0 = INT_MAX, i1 = INT_MAX;
      if (lane < 8 * P) { v0 = cv[lane / P][i][lane % P]; i0 = ci[lane / P][i][lane % P]; }
      if (lane + 32 < 8 * P) { v1 = cv[(lane + 32) / P][i][(lane + 32) % P]; i1 = ci[(lane + 32) / P][i][(lane + 32) % P]; }
      if (better(v1, i1, v0, i0)) { const float tv = v0; v0 = v1; v1 = tv; const int ti = i0; i0 = i1; i1 = ti; }
      for (int p = 0; p < P; ++p) {
        float bv = v0; int bi = i0;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
          const float ov = __shfl_xor_sync(0xffffffffu, bv, o);
          const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
          if (better(ov, oi, bv, bi)) { bv = ov; bi = oi; }
        }
        if (i0 == bi && v0 == bv) { v0 = v1; i0 = i1; v1 = -INFINITY; i1 = INT_MAX; }
        if (lane == 0) {
          const size_t o = ((size_t)r * a.S + c0 + i) * P + p;
          a.cand_val[o] = a.last_scores ? bv + add : bv;     // cbs.py:210-212
          a.cand_tok[o] = bi;
        }
      }
    }
    __syncthreads();
  }
}

template <int P>
static int launch_rows(cudaStream_t st, const SearchRowsArgs& a) {
  constexpr int SC = P <= 2 ? 8 : (P <= 4 ? 4 : 2);
  const bool vec = (a.V % 4) == 0 && (a.ld % 4) == 0 && (reinterpret_cast<uintptr_t>(a.logp) & 15) == 0 &&
                   (reinterpret_cast<uintptr_t>(a.fsm_bits) & 15) == 0;
  const size_t row_bytes = (size_t)a.V * 4;
  if (vec && row_bytes <= 200 * 1024) {
    static size_t configured = 0;
    if (row_bytes > 48 * 1024 && row_bytes > configured) {
      CUDA_TRY(cudaFuncSetAttribute(search_rows_block_kernel<P, SC>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)row_bytes));
      configured = row_bytes;
    }
    search_rows_block_kernel<P, SC><<<a.R, 256, row_bytes, st>>>(a);
  } else if (vec) {
    search_rows_kernel<P, SC, 4><<<ceil_div(a.R, 4), 128, 0, st>>>(a);
  } else {
    search_rows_kernel<P, SC, 1><<<ceil_div(a.R, 4), 128, 0, st>>>(a);
  }
  LAUNCHED();
  return 0;
}

int search_rows(cudaStream_t st, const SearchRowsArgs& a) {
  PROF_SCOPE(st, "search_rows", 0, (double)a.R*a.V*(a.normalized ? 4.0 : 8.0) + (a.fsm_bits ? (double)a.R*a.V*4.0*((a.S+7)/8) : 0.0));
  REQUIRE(a.V >= a.P, "vocabulary (%d) smaller than per-node beam (%d)", a.V, a.P);
  switch (a.P) {
    case 1: return launch_rows<1>(st, a);
    case 2: return launch_rows<2>(st, a);
    case 3: return launch_rows<3>(st, a);
    case 4: return launch_rows<4>(st, a);
    case 5: return launch_rows<5>(st, a);
    case 6: return launch_rows<6>(st, a);
    case 7: return launch_rows<7>(st, a);
    case 8: return launch_rows<8>(st, a);
    default:
      set_error("per-node beam size %d unsupported (1..8)", a.P);
      return SSCVAE_ERR_UNSUPPORTED;
  }
}

// one warp per (image, to-state): emit the K best candidates in sorted order
__global__ void search_merge_kernel(const float* __restrict__ cand_val, const int32_t* __restrict__ cand_tok, int B, int S,
                                    int K, int P, int32_t* __restrict__ tokens, int32_t* __restrict__ backptr,
                                    float* __restrict__ scores) {
  const int wi = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (wi >= B * S) return;
  const int lane = threadIdx.x & 31;
  const int b = wi / S, i = wi % S;
  const int n = S * K * P;
  float lastv = INFINITY; int lastj = -1;
  for (int k = 0; k < K; ++k) {
    float bv = -INFINITY; int bj = INT_MAX;
    for (int j = lane; j < n; j += 32) {
      const float v = cand_val[(((size_t)b * S * K + j / P) * S + i) * P + j % P];
      const bool after_last = (v < lastv) || (v == lastv && j > lastj);
      if (after_last && better(v, j, bv, bj)) { bv = v; bj = j; }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const float ov = __shfl_xor_sync(0xffffffffu, bv, o);
      const int oj = __shfl_xor_sync(0xffffffffu, bj, o);
      if (better(ov, oj, bv, bj)) { bv = ov; bj = oj; }
    }
    if (lane == 0) {
      const size_t o = ((size_t)b * S + i) * K + k;
      scores[o] = bv;
      tokens[o] = cand_tok[(((size_t)b * S * K + bj / P) * S + i) * P + bj % P];
      backptr[o] = bj / P;
    }
    lastv = bv; lastj = bj;
  }
}

int search_merge(cudaStream_t st, const float* cand_val, const int32_t* cand_tok, int B, int S, int K, int P,
                 int32_t* tokens, int32_t* backptr, float* scores) {
  PROF_SCOPE(st, "search_merge", 0, (double)B*S*K*S*P*8.0);
  REQUIRE(S * K * P >= K, "not enough candidates");
  search_merge_kernel<<<ceil_div(B * S, 4), 128, 0, st>>>(cand_val, cand_tok, B, S, K, P, tokens, backptr, scores);
  LAUNCHED();
  return 0;
}

// n_steps = the number of steps the reference's loop would have produced (cbs.py:161-168): it stops
// before step t when every token of step t-1 is the boundary token. Block x decides for rows [x*rows, (x+1)*rows): one
// block over all rows is the batch-wide exit, one block per search group the exit of each search on its own.
__global__ void search_nsteps_kernel(const int32_t* __restrict__ tokens_hist, int steps_run, int R, int rows,
                                     int end_index, int32_t* __restrict__ n_steps) {
  __shared__ int not_end;
  const int r0 = blockIdx.x * rows;
  int n = steps_run;
  for (int t = 1; t < steps_run; ++t) {
    if (threadIdx.x == 0) not_end = 0;
    __syncthreads();
    int local = 0;
    for (int r = threadIdx.x; r < rows; r += blockDim.x) local |= (tokens_hist[(size_t)(t - 1) * R + r0 + r] != end_index);
    if (local) atomicOr(&not_end, 1);
    __syncthreads();
    const int ne = not_end;
    __syncthreads();
    if (!ne) { n = t; break; }
  }
  if (threadIdx.x == 0) n_steps[blockIdx.x] = n;
}

__global__ void search_finish_kernel(const int32_t* __restrict__ tokens_hist, const int32_t* __restrict__ backptr_hist,
                                     const float* __restrict__ scores_hist, int steps_run, int B, int S, int K,
                                     int end_index, const long long* __restrict__ num_constraints, int min_sat,
                                     int groups_per_table, int groups_per_exit, long long* __restrict__ predictions,
                                     float* __restrict__ final_scores, long long* __restrict__ best,
                                     const int32_t* __restrict__ n_steps, int32_t* __restrict__ best_state_out,
                                     int32_t* __restrict__ steps_out) {
  extern __shared__ float s_score[];                        // S*K
  const int b = blockIdx.x;
  const int SK = S * K, R = B * SK;
  const int n = n_steps[groups_per_exit > 0 ? b / groups_per_exit : 0];
  for (int w = threadIdx.x; w < SK; w += blockDim.x) {
    long long* out = predictions + ((size_t)b * SK + w) * steps_run;
    const size_t base = (size_t)b * SK;
    out[n - 1] = tokens_hist[(size_t)(n - 1) * R + base + w];
    if (n > 1) {                                            // cbs.py:252-271
      int cur = backptr_hist[(size_t)(n - 1) * R + base + w];
      for (int t = n - 2; t >= 1; --t) {
        out[t] = tokens_hist[(size_t)t * R + base + cur];
        cur = backptr_hist[(size_t)t * R + base + cur];
      }
      out[0] = tokens_hist[base + cur];
    }
    for (int t = n; t < steps_run; ++t) out[t] = end_index;
    const float sc = scores_hist[(size_t)(n - 1) * R + base + w];
    final_scores[base + w] = sc;
    s_score[w] = sc;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    const int nc = num_constraints ? (int)num_constraints[groups_per_table > 1 ? b / groups_per_table : b] : -1;
    const int best_state = select_state(s_score, K, S, nullptr, nc, min_sat);
    const long long* src = predictions + ((size_t)b * SK + (size_t)best_state * K) * steps_run;
    for (int t = 0; t < steps_run; ++t) best[(size_t)b * steps_run + t] = src[t];
    if (best_state_out) { best_state_out[b] = best_state; steps_out[b] = n; }
  }
}

int search_finish(cudaStream_t st, const int32_t* tokens_hist, const int32_t* backptr_hist, const float* scores_hist,
                  int steps_run, int B, int S, int K, int end_index, const long long* num_constraints, int min_sat,
                  int groups_per_table, int groups_per_exit, long long* predictions, float* final_scores, long long* best,
                  int32_t* n_steps, int32_t* best_state, int32_t* group_steps) {
  REQUIRE(steps_run >= 1, "no search steps");
  REQUIRE((best_state == nullptr) == (group_steps == nullptr), "best_state and group_steps go together");
  REQUIRE(groups_per_exit >= 0 && (groups_per_exit == 0 || B % groups_per_exit == 0), "bad exit grouping %d of %d groups",
          groups_per_exit, B);
  const int R = B * S * K;
  if (groups_per_exit == 0) {
    search_nsteps_kernel<<<1, 1024, 0, st>>>(tokens_hist, steps_run, R, R, end_index, n_steps);
  } else {
    const int rows = groups_per_exit * S * K;
    search_nsteps_kernel<<<B / groups_per_exit, std::min(1024, ceil_div(rows, 32) * 32), 0, st>>>(tokens_hist, steps_run, R,
                                                                                                  rows, end_index, n_steps);
  }
  LAUNCHED();
  search_finish_kernel<<<B, 128, S * K * sizeof(float), st>>>(tokens_hist, backptr_hist, scores_hist, steps_run, B, S, K,
                                                            end_index, num_constraints, min_sat, groups_per_table,
                                                            groups_per_exit, predictions, final_scores, best, n_steps,
                                                            best_state, group_steps);
  LAUNCHED();
  return 0;
}

// Attention behind every word. Block (g, y) walks the back-pointers of search group g the way search_finish_kernel does,
// from the group's exit step n - 1, for beam w = y (y < SK, all beams) or for beam 0 of the returned state (the last y).
// Word t of the beam was chosen from the logits of one row of step t; that row's attention weights are the word's:
//   word 0: alpha[0][g] (step 0 runs one row per group);  word t >= 1: alpha[t][base + bp[t][cur_t]] = alpha[t][base + cur_(t-1)]
// with cur_(n-1) = w, cur_(t-1) = bp[t][cur_t]. Words after the first boundary token and steps >= n are zero.
__global__ void __launch_bounds__(128) search_attention_kernel(
    const int32_t* __restrict__ tokens_hist, const int32_t* __restrict__ backptr_hist, const float* __restrict__ scores_hist,
    const float* __restrict__ alpha_hist, int L, int B, int S, int K, int N, int end_index,
    const int32_t* __restrict__ group_steps, const int32_t* __restrict__ best_state, const uint8_t* __restrict__ valid,
    float* __restrict__ att_all, float* __restrict__ att_best) {
  extern __shared__ int s_mem[];
  int* s_row = s_mem;                                       // (L) alpha row of word t within step t, -1 = zero
  int* s_tok = s_mem + L;                                   // (L) word t
  const int g = blockIdx.x, SK = S * K, R = B * SK, base = g * SK;
  const bool best = att_all == nullptr || (int)blockIdx.y == SK;
  if (threadIdx.x == 0) {
    const int n = group_steps[g];
    int cur = blockIdx.y;
    if (best) {
      const int st = valid ? select_state(scores_hist + (size_t)(n - 1) * R + base, K, S, valid + (size_t)g * S, -1, 0)
                           : best_state[g];
      cur = st * K;
    }
    // both walks stay rolled: unrolled, this thread's loads spill to local memory
#pragma unroll 1
    for (int t = n - 1; t >= 1; --t) {                      // cbs.py:252-271, as search_finish_kernel
      s_tok[t] = tokens_hist[(size_t)t * R + base + cur];
      cur = backptr_hist[(size_t)t * R + base + cur];
      s_row[t] = base + cur;
    }
    s_tok[0] = tokens_hist[base + cur];
    s_row[0] = g;
    bool ended = false;
#pragma unroll 1
    for (int t = 0; t < L; ++t) {
      if (ended || t >= n) s_row[t] = -1;
      else ended = s_tok[t] == end_index;
    }
  }
  __syncthreads();
  float* out = best ? att_best + (size_t)g * L * N : att_all + ((size_t)g * SK + blockIdx.y) * L * N;
  for (int i = threadIdx.x; i < L * N; i += blockDim.x) {
    const int t = i / N, row = s_row[t];
    out[i] = row < 0 ? 0.f : alpha_hist[((size_t)t * R + row) * N + i % N];
  }
}

int search_attention(cudaStream_t st, const int32_t* tokens_hist, const int32_t* backptr_hist, const float* scores_hist,
                     const float* alpha_hist, int L, int B, int S, int K, int N, int end_index, const int32_t* group_steps,
                     const int32_t* best_state, const uint8_t* valid, float* att_all, float* att_best) {
  REQUIRE(att_best != nullptr, "attention_best is required");
  const int SK = S * K;
  const unsigned ny = att_all ? SK + 1 : 1;
  PROF_SCOPE(st, "search_attention", 0, (double)B * ny * L * N * 8.0);
  search_attention_kernel<<<dim3(B, ny), 128, 2 * L * sizeof(int), st>>>(tokens_hist, backptr_hist, scores_hist, alpha_hist, L, B,
                                                                    S, K, N, end_index, group_steps, best_state, valid,
                                                                    att_all, att_best);
  LAUNCHED();
  return 0;
}

__global__ void state_gather_kernel(const int32_t* __restrict__ bp, int SK, const bf16* __restrict__ xa_src,
                                    bf16* __restrict__ xa_dst, int ld_xa, const float* __restrict__ c1_src,
                                    float* __restrict__ c1_dst, const float* __restrict__ cd_src,
                                    float* __restrict__ cd_dst, int H) {
  const int r = blockIdx.x;
  const int src = (r / SK) * SK + bp[r];
  const bf16x8* xs = reinterpret_cast<const bf16x8*>(xa_src + (size_t)src * ld_xa);
  bf16x8* xd = reinterpret_cast<bf16x8*>(xa_dst + (size_t)r * ld_xa);
  for (int i = threadIdx.x; i < ld_xa / 8; i += blockDim.x) xd[i] = xs[i];
  for (int i = threadIdx.x; i < H; i += blockDim.x) {
    c1_dst[(size_t)r * H + i] = c1_src[(size_t)src * H + i];
    cd_dst[(size_t)r * H + i] = cd_src[(size_t)src * H + i];
  }
}
int state_gather(cudaStream_t st, const int32_t* bp, int R, int SK, const bf16* xa_src, bf16* xa_dst, int ld_xa,
                 const float* c1_src, float* c1_dst, const float* cd_src, float* cd_dst, int H) {
  state_gather_kernel<<<R, 128, 0, st>>>(bp, SK, xa_src, xa_dst, ld_xa, c1_src, c1_dst, cd_src, cd_dst, H);
  LAUNCHED();
  return 0;
}

}  // namespace sscvae

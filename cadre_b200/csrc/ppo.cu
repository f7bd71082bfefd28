// PPO minibatch update on one GPU: CadreAgent.update_policy (ppo_agent/agent.py:166-237) for W logical workers
// at once, forward and hand-written backward, plus the chief's clip + Adam (ppo_agent/chief.py:13-21).
//
// The reference runs every row through all four command experts and masks (agent.py:170-182); here rows are
// ROUTED: each row goes only through the LSTM + actor-critic of its own command (exactly the same function and
// gradient, 4x less work). Rows of a head are stably sorted by command into per-expert slots
// (expert e = head*4 + command); all eight experts run as one grid.z-batched tcgen05 GEMM per layer / step.
//
// Time-expanded buffers use 9 time slots per row ("x9" layout [E][cap][9][ld]): slot j<8 of X holds x_j, slot j of
// H / C holds h_{j-1} / c_{j-1} (j = 0 is the stored recurrent state hn/cn), slot j<8 of G / dG holds the gate
// activations / pre-activation gradients of step j and slot 8 of dG stays zero. With that layout the weight
// gradients of all eight steps are single GEMMs over K = 9*rows: dW_ih = dG^T X, dW_hh = dG^T H.
// Precision of the stored tensors: the cell state C (the recurrence's only long accumulation) and the x-part
// pre-activations stay fp32; h, the gate activations and dG are stored ONCE, as fp16 (11-bit significand like the
// TF32 operands of the other GEMMs; dG scaled by a power of two): they are tensor-core operands (recurrent GEMMs,
// weight-gradient GEMMs) or bounded activations in (-1, 1), and halving their bytes is what the L2-bound recurrence
// and weight-gradient kernels are made of.
#include "../../include/cadre_b200.h"
#include "internal.h"
#include "ptx.cuh"
#include "ppo_layout.h"
#include "lstm_seq.cuh"
#include "sampler.cuh"

#include <algorithm>
#include <cmath>
#include <vector>

namespace cadre {

using namespace ppo;

struct StorageRef {  // == cadre_storage_ref
  const float* obs;
  const long long* action;
  const float* value_preds;
  const float* returns;
  const float* action_log_probs;
  const float* adv;
  const float* hn;
  const float* cn;
  const int* command;
};

// ------------------------------------------------------------------------------------------ routing
// Stable counting sort of the R = W*mb rows of one head by command (one CTA per head).
// Minibatch indices live in a staged device table [steps][W][2][mb]; the update reads slice `*step_ctr`, which the
// update's own prep_kernel advances afterwards. A sequence of update steps therefore needs no host-to-device copy
// between steps and can be replayed from a CUDA graph (cadre_ppo_stage / cadre_ppo_update with indices_host = NULL).
// `stop` (NULL unless target-KL early stopping is on): once the phase is stopped, every expert gets zero rows, and every
// later kernel of the update sizes its work from these counts, so the remaining steps of the phase do almost nothing.
__global__ void __launch_bounds__(1024) route_kernel(const StorageRef* __restrict__ refs,
                                                     const int* __restrict__ idx_all,
                                                     const int* __restrict__ step_ctr, int W, int mb,
                                                     int* __restrict__ row_slot, int* __restrict__ row_expert,
                                                     int* __restrict__ counts, int* __restrict__ counts9,
                                                     const int* __restrict__ stop) {
  pdl_trigger();
  pdl_wait();
  if (stop && *stop) {
    if (threadIdx.x < 4) counts[blockIdx.x * 4 + threadIdx.x] = 0, counts9[blockIdx.x * 4 + threadIdx.x] = 0;
    return;
  }
  const int* idx = idx_all + static_cast<long long>(*step_ctr) * 2 * W * mb;
  __shared__ int base[4];
  __shared__ int wcnt[32][4];
  const int h = blockIdx.x, tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int R = W * mb;
  if (tid < 4) base[tid] = 0;
  __syncthreads();
  for (int tile0 = 0; tile0 < R; tile0 += 1024) {
    const int r = tile0 + tid;
    int c = -1;
    if (r < R) {
      const int w = r / mb, i = r - w * mb;
      const int t = idx[(w * 2 + h) * mb + i];
      c = refs[w * 2 + h].command[t] & 3;
    }
    int my = 0;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const unsigned bal = __ballot_sync(0xffffffffu, c == k);
      if (c == k) my = __popc(bal & ((1u << lane) - 1));
      if (lane == 0) wcnt[warp][k] = __popc(bal);
    }
    __syncthreads();
    if (r < R) {
      int off = 0;
      for (int w2 = 0; w2 < warp; ++w2) off += wcnt[w2][c];
      row_slot[h * R + r] = base[c] + off + my;
      row_expert[h * R + r] = h * 4 + c;
    }
    __syncthreads();
    if (tid < 4) {
      int tot = 0;
      for (int w2 = 0; w2 < 32; ++w2) tot += wcnt[w2][tid];
      base[tid] += tot;
    }
    __syncthreads();
  }
  if (tid < 4) {
    counts[h * 4 + tid] = base[tid];
    counts9[h * 4 + tid] = 9 * base[tid];
  }
}

// gather of one row: RolloutStorage.feed_forward_generator (storage.py:98-120) fused with the routing
struct RowScalars {
  int* action;
  int* worker;
  float* old_v;
  float* ret;
  float* old_lp;
  float* adv;
};

__global__ void __launch_bounds__(256) pack_kernel(const StorageRef* __restrict__ refs,
                                                   const int* __restrict__ idx_all,
                                                   const int* __restrict__ step_ctr, int W, int mb, int cap,
                                                   const int* __restrict__ row_slot,
                                                   const int* __restrict__ row_expert,
                                                   __half* __restrict__ X16, float* __restrict__ C9,
                                                   __half* __restrict__ H16, RowScalars sc,
                                                   const int* __restrict__ stop) {
  pdl_trigger();
  pdl_wait();
  if (stop && *stop) return;   // no routed rows (route_kernel)
  const int r = blockIdx.x, h = blockIdx.y, R = W * mb;
  const int* idx = idx_all + static_cast<long long>(*step_ctr) * 2 * R;
  const int w = r / mb, i = r - w * mb;
  const StorageRef ref = refs[w * 2 + h];
  const int t = idx[(w * 2 + h) * mb + i];
  const int e = row_expert[h * R + r], slot = row_slot[h * R + r];
  const long long row = static_cast<long long>(e) * cap + slot;
  const float* obs = ref.obs + static_cast<long long>(t) * 8 * F;
  // fp16 observations: A operand of the x-part GEMM and B operand of the W_ih weight-gradient GEMM. Eight loads
  // are in flight per thread (the kernel is latency-, not bandwidth-bound: 17 KB per block).
  __half* x16 = X16 + row * 9 * LS_LDH16;
  for (int k0 = threadIdx.x; k0 < 8 * F; k0 += 8 * 256) {
    float v[8];
#pragma unroll
    for (int u = 0; u < 8; ++u) v[u] = (k0 + u * 256 < 8 * F) ? obs[k0 + u * 256] : 0.f;
#pragma unroll
    for (int u = 0; u < 8; ++u) {
      const int k = k0 + u * 256;
      if (k < 8 * F) {
        const int j = k / F, f = k - j * F;
        x16[j * LS_LDH16 + f] = __float2half_rn(v[u]);
      }
    }
  }
  float* c0 = C9 + row * 9 * LDF;
  __half* h16 = H16 + row * 9 * LS_LDH16;    // slot 0: h_{-1}
  for (int f = threadIdx.x; f < F; f += 256) {
    h16[f] = __float2half_rn(ref.hn[static_cast<long long>(t) * F + f]);
    c0[f] = ref.cn[static_cast<long long>(t) * F + f];
  }
  if (threadIdx.x == 0) {
    sc.action[row] = static_cast<int>(ref.action[t]);
    sc.worker[row] = w;
    sc.old_v[row] = ref.value_preds[t];
    sc.ret[row] = ref.returns[t];
    sc.old_lp[row] = ref.action_log_probs[t];
    sc.adv[row] = ref.adv[t];
  }
}

// b_ih + b_hh (one bias vector for the x-part GEMM) and the compacted work list of that GEMM: (expert, 128-row tile)
// pairs covering the 9 * count[e] valid rows of each expert, so that its grid is sized by the rows that exist
// (2 * 9 * R / 128 + 8 tiles at most) instead of by the per-expert capacity (8 * 9 * cap / 128).
// It also clears the K padding of the weight-gradient GEMMs: those run over K = 9 * count rows rounded up to a whole
// 64-row k-block, i.e. they read up to 8 rows past the routed ones. The BPTT kernel writes zeros up to the next
// multiple of 32 rows only, so dG rows [count, count + 8) are zeroed here (stale rows of an earlier update with more
// rows for this expert would otherwise leak into the gradient).
constexpr int WGRAD_PAD_ROWS = 8;
__global__ void prep_kernel(const float* __restrict__ params, float* __restrict__ o, int n,
                            const int* __restrict__ counts9, int* __restrict__ tile_list, int max_tiles,
                            __half* __restrict__ dG16, int cap, int* __restrict__ step_ctr,
                            int* __restrict__ opt_step) {
  pdl_trigger();
  pdl_wait();          // the gather (previous launch) has consumed this step's index slice
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i == 0) {
    *step_ctr += 1;    // the next update step reads the next slice of the staged table
    *opt_step += 1;    // 1-based Adam step of this update (cadre_ppo_adam_step* with step = 0 reads it)
  }
  if (i < n) {
    const int e = i / G, r = i - e * G;
    const float* blk = params + OFF_LSTM + e * LSTM_BLK;
    o[i] = blk[LSTM_BIH + r] + blk[LSTM_BHH + r];
  }
  {
    constexpr int V = 9 * LS_LDG16 / 8;                       // uint4 per row (all 9 slots)
    const long long total = static_cast<long long>(E) * WGRAD_PAD_ROWS * V;
    for (long long k = i; k < total; k += static_cast<long long>(gridDim.x) * blockDim.x) {
      const int e = static_cast<int>(k / (WGRAD_PAD_ROWS * V));
      const int rr = static_cast<int>((k / V) % WGRAD_PAD_ROWS), v = static_cast<int>(k % V);
      const int row = counts9[e] / 9 + rr;
      if (row < cap)
        reinterpret_cast<uint4*>(dG16 + (static_cast<long long>(e) * cap + row) * 9 * LS_LDG16)[v] =
            make_uint4(0u, 0u, 0u, 0u);
    }
  }
  if (i == 0) {
    int nt = 0;
    for (int e = 0; e < E; ++e) {
      const int tiles = (counts9[e] + 127) >> 7;
      for (int m = 0; m < tiles && nt < max_tiles; ++m, ++nt) tile_list[1 + 2 * nt] = e, tile_list[2 + 2 * nt] = m;
    }
    tile_list[0] = nt;
  }
}

// ------------------------------------------------------------------------------------------ heads + loss
// Last actor / critic layers, Categorical log-prob + entropy (models.py:203-212, distributions.py:66-105),
// the PPO objective (agent.py:184-229) and their backward down to the ReLU of the second hidden layer.
struct HeadParams {
  const float* Y2;      // [E][cap][256] post-ReLU hidden (actor | critic)
  float* dZ2;           // [E][cap][256]
  const float* params;  // flat parameters
  float* grads;         // flat gradients (W3A / B3A / W3C / B3C written by the last CTA of each expert)
  const int* counts;
  RowScalars sc;
  float* losses;        // [W][2][3] value, action, entropy (un-scaled means), written by the last CTA of the grid
  float* partial;       // [E][cap / HEAD_ROWS][HEAD_PARTIAL] per-CTA partial sums (scratch)
  float* loss_e;        // [E][W][3] per-expert loss sums (scratch)
  float* diag;          // [W][2][4] update diagnostics (see below), written by the last CTA; NULL: not computed
  float* diag_e;        // [E][W][4] per-expert diagnostics sums (scratch)
  float* kl_sum;        // [2] per head, the sum over workers of diag[w][h][0] in worker order; NULL: not written
  unsigned* ctr;        // [E] finished CTAs per expert, [E] finished experts (zero at launch)
  int cap, W;
  float inv_mb, clip, value_coeff, clip_coeff, ent_coeff;
};

constexpr int HEAD_ROWS_PER_CTA = 32;
constexpr int HEAD_MAX_W = 64;   // workers per engine the loss reduction is sized for
// per-CTA partial: dW3A [33][128], dW3C [128], dB3A [36], dB3C [4], losses [HEAD_MAX_W][3], diagnostics [HEAD_MAX_W][4]
constexpr int HP_W3A = 0, HP_W3C = AMAX * HID, HP_B3A = HP_W3C + HID, HP_B3C = HP_B3A + B3A_LD, HP_LOSS = HP_B3C + 4;
constexpr int HP_DIAG = HP_LOSS + HEAD_MAX_W * 3;
constexpr int HEAD_PARTIAL = HP_DIAG + HEAD_MAX_W * 4;
// Update diagnostics per worker and head, means over the minibatch (d = lp - old_lp):
//   [0] approximate KL, expm1(d) - d   [1] old_lp - lp   [2] fraction of rows with |ratio - 1| > clip
//   [3] fraction of rows with |v - old_v| > clip (the value clip of agent.py:184-193)
// Per-row terms are summed unweighted through the loss terms' ordered reduction and scaled by 1 / mini_batch once at
// the end, so the clip fractions are exactly count * (1 / mini_batch).
constexpr int DIAG_TERMS = 4;

// Every sum of this kernel has a FIXED order (rows of a CTA in sequence, CTAs of an expert by block index, experts of
// a head by index), so losses and last-layer gradients are bit-reproducible from run to run: each CTA writes its
// partial sums to scratch, the last CTA of an expert to finish (device-wide counter) reduces them in block order, and
// the last expert to finish reduces the per-expert losses in expert order. No floating-point atomics.
// Launched with 256 threads. The register cap is the count the kernel had before the diagnostics terms (ptxas would
// otherwise take 73; no spills at 72, and 3 CTAs per SM either way).
__global__ void __maxnreg__(72) head_kernel(const HeadParams p) {
  pdl_trigger();
  pdl_wait();
  const int e = blockIdx.y, head = e >> 2;
  const int A = head == 0 ? 33 : 3;
  const int count = p.counts[e];
  const int rows_pad = (count + 31) & ~31;
  const int row0 = blockIdx.x * HEAD_ROWS_PER_CTA;
  if (row0 >= rows_pad) return;
  __shared__ float w3aT[HID][AMAX];      // [k][j]
  __shared__ float b3a[AMAX + 3];
  __shared__ float w3c[HID];
  __shared__ float s_y[8][2 * HID];
  __shared__ float s_dl[HEAD_ROWS_PER_CTA][AMAX + 3];  // d loss / d logits of the CTA's rows
  __shared__ float s_dv[HEAD_ROWS_PER_CTA];
  __shared__ float s_lt[HEAD_ROWS_PER_CTA][3];         // loss terms of the CTA's rows
  __shared__ float s_dg[HEAD_ROWS_PER_CTA][DIAG_TERMS]; // diagnostics terms of the CTA's rows (p.diag != NULL)
  __shared__ int s_wk[HEAD_ROWS_PER_CTA];              // worker of each row (-1: padding row)
  __shared__ int s_last;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const float* W3A = p.params + OFF_W3A + static_cast<long long>(e) * AMAX * HID;
  {   // all 17 loads of a thread in flight together (the kernel is a chain of short latency-bound phases)
    constexpr int NL = (AMAX * HID + 255) / 256;
    float wv[NL];
#pragma unroll
    for (int u = 0; u < NL; ++u) wv[u] = (tid + u * 256 < AMAX * HID) ? W3A[tid + u * 256] : 0.f;
#pragma unroll
    for (int u = 0; u < NL; ++u) {
      const int i = tid + u * 256;
      if (i < AMAX * HID) w3aT[i % HID][i / HID] = wv[u];
    }
  }
  if (tid < AMAX) b3a[tid] = p.params[OFF_B3A + e * B3A_LD + tid];
  if (tid < HID) w3c[tid] = p.params[OFF_W3C + e * HID + tid];
  for (int i = tid; i < HEAD_ROWS_PER_CTA * (AMAX + 3); i += 256) (&s_dl[0][0])[i] = 0.f;
  if (tid < HEAD_ROWS_PER_CTA) s_dv[tid] = 0.f, s_wk[tid] = -1;
  const float b3c = p.params[OFF_B3C + e * 4];
  __syncthreads();

  // ---- phase 1: one warp per row: logits, Categorical, PPO objective, backward seeds, d hidden2
  const int row_end = min(row0 + HEAD_ROWS_PER_CTA, rows_pad);
  for (int slot = row0 + warp; slot < row_end; slot += 8) {
    const long long row = static_cast<long long>(e) * p.cap + slot;
    float* dz = p.dZ2 + row * 2 * HID;
    if (slot >= count) {  // K-padding rows of the weight-gradient GEMMs must be exact zeros
#pragma unroll
      for (int q = 0; q < 8; ++q) dz[lane + 32 * q] = 0.f;
      continue;
    }
    const float* y = p.Y2 + row * 2 * HID;
    float ya[4], yc[4];
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      ya[q] = y[lane + 32 * q];
      yc[q] = y[HID + lane + 32 * q];
      s_y[warp][lane + 32 * q] = ya[q];
    }
    __syncwarp();
    float l0 = -INFINITY, l1 = -INFINITY;
    if (lane < A) {   // four independent accumulation chains (the sum order is fixed by this code, not by timing)
      float a0 = b3a[lane], a1 = 0.f, a2 = 0.f, a3 = 0.f;
#pragma unroll 8
      for (int k = 0; k < HID; k += 4) {
        a0 = fmaf(s_y[warp][k], w3aT[k][lane], a0);
        a1 = fmaf(s_y[warp][k + 1], w3aT[k + 1][lane], a1);
        a2 = fmaf(s_y[warp][k + 2], w3aT[k + 2][lane], a2);
        a3 = fmaf(s_y[warp][k + 3], w3aT[k + 3][lane], a3);
      }
      l0 = (a0 + a1) + (a2 + a3);
    }
    if (lane + 32 < A) {
      float a0 = b3a[lane + 32], a1 = 0.f, a2 = 0.f, a3 = 0.f;
#pragma unroll 8
      for (int k = 0; k < HID; k += 4) {
        a0 = fmaf(s_y[warp][k], w3aT[k][lane + 32], a0);
        a1 = fmaf(s_y[warp][k + 1], w3aT[k + 1][lane + 32], a1);
        a2 = fmaf(s_y[warp][k + 2], w3aT[k + 2][lane + 32], a2);
        a3 = fmaf(s_y[warp][k + 3], w3aT[k + 3][lane + 32], a3);
      }
      l1 = (a0 + a1) + (a2 + a3);
    }
    float v = 0.f;
#pragma unroll
    for (int q = 0; q < 4; ++q) v = fmaf(yc[q], w3c[lane + 32 * q], v);
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    v += b3c;
    // Categorical(logits): logits - logsumexp
    float mx = fmaxf(l0, l1);
    for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    float se = (lane < A ? expf(l0 - mx) : 0.f) + (lane + 32 < A ? expf(l1 - mx) : 0.f);
    for (int o = 16; o > 0; o >>= 1) se += __shfl_xor_sync(0xffffffffu, se, o);
    const float lse = mx + logf(se);
    const float lp0 = l0 - lse, lp1 = l1 - lse;
    const float p0 = lane < A ? expf(lp0) : 0.f, p1 = lane + 32 < A ? expf(lp1) : 0.f;
    float ent = -((lane < A ? p0 * lp0 : 0.f) + (lane + 32 < A ? p1 * lp1 : 0.f));
    for (int o = 16; o > 0; o >>= 1) ent += __shfl_xor_sync(0xffffffffu, ent, o);
    const int a = p.sc.action[row];
    const float lpa_src = (a < 32) ? lp0 : lp1;
    const float lp = __shfl_sync(0xffffffffu, lpa_src, a & 31);

    const float old_lp = p.sc.old_lp[row], adv = p.sc.adv[row], old_v = p.sc.old_v[row], ret = p.sc.ret[row];
    const float wgt = p.inv_mb;
    // agent.py:184-193
    const float ratio = expf(lp - old_lp);
    const float lo = 1.f - p.clip, hi = 1.f + p.clip;
    const float s1 = ratio * adv, s2 = fminf(fmaxf(ratio, lo), hi) * adv;
    const float action_term = -fminf(s1, s2);
    const float dvv = v - old_v;
    const float v_clip = old_v + fminf(fmaxf(dvv, -p.clip), p.clip);
    const float vl = (v - ret) * (v - ret), vlc = (v_clip - ret) * (v_clip - ret);
    const float value_term = 0.5f * fmaxf(vl, vlc);
    if (lane == 0) {
      s_lt[slot - row0][0] = wgt * value_term;
      s_lt[slot - row0][1] = wgt * action_term;
      s_lt[slot - row0][2] = wgt * ent;
      s_wk[slot - row0] = p.sc.worker[row];
      if (p.diag) {
        const float d = lp - old_lp;
        s_dg[slot - row0][0] = expm1f(d) - d;
        s_dg[slot - row0][1] = old_lp - lp;
        s_dg[slot - row0][2] = fabsf(ratio - 1.f) > p.clip ? 1.f : 0.f;
        s_dg[slot - row0][3] = fabsf(dvv) > p.clip ? 1.f : 0.f;
      }
    }
    // backward seeds (autograd conventions of torch.min / torch.max / clamp: ties split evenly, clamp passes
    // the gradient on the closed interval)
    const float inside_r = (ratio >= lo && ratio <= hi) ? 1.f : 0.f;
    const float g1 = s1 < s2 ? 1.f : (s1 > s2 ? 0.f : 0.5f);   // weight of surr1 in min()
    const float dmin_dlp = g1 * adv * ratio + (1.f - g1) * adv * ratio * inside_r;
    const float dlp = -p.clip_coeff * wgt * dmin_dlp;
    const float inside_v = (dvv >= -p.clip && dvv <= p.clip) ? 1.f : 0.f;
    const float gv = vl > vlc ? 1.f : (vl < vlc ? 0.f : 0.5f);
    const float dv = p.value_coeff * wgt * (gv * (v - ret) + (1.f - gv) * (v_clip - ret) * inside_v);
    const float ew = p.ent_coeff * wgt;  // total = ... - ent_coeff * mean(entropy)
    float dl0 = 0.f, dl1 = 0.f;
    if (lane < A) dl0 = dlp * ((a == lane ? 1.f : 0.f) - p0) + ew * p0 * (lp0 + ent);
    if (lane + 32 < A) dl1 = dlp * ((a == lane + 32 ? 1.f : 0.f) - p1) + ew * p1 * (lp1 + ent);
    float* dl = s_dl[slot - row0];
    if (lane < A) dl[lane] = dl0;
    if (lane + 32 < A) dl[lane + 32] = dl1;
    if (lane == 0) s_dv[slot - row0] = dv;
    __syncwarp();
    // d hidden2 = dlogits W3a (actor), dv * w3c (critic), through the ReLU
    float da[4] = {0.f, 0.f, 0.f, 0.f};
    for (int j = 0; j < A; ++j) {
      const float d = dl[j];
#pragma unroll
      for (int q = 0; q < 4; ++q) da[q] = fmaf(d, w3aT[lane + 32 * q][j], da[q]);
    }
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      dz[lane + 32 * q] = ya[q] > 0.f ? da[q] : 0.f;
      dz[HID + lane + 32 * q] = yc[q] > 0.f ? dv * w3c[lane + 32 * q] : 0.f;
    }
    __syncwarp();
  }
  __syncthreads();

  // ---- phase 2: this CTA's partial last-layer weight gradients as small register-tiled products over its rows
  // (hidden2 is re-read from L2 eight rows at a time, d logits / d value sit in shared memory) -> scratch
  const int nrows = min(count, row0 + HEAD_ROWS_PER_CTA) - row0;  // valid rows (>= 1 here; padding rows carry zeros)
  const int nblk = rows_pad / HEAD_ROWS_PER_CTA;                  // working CTAs of this expert
  float* part = p.partial + (static_cast<long long>(e) * (p.cap / HEAD_ROWS_PER_CTA) + blockIdx.x) * HEAD_PARTIAL;
  {
    const float* Ybase = p.Y2 + (static_cast<long long>(e) * p.cap + row0) * 2 * HID;
    const int k = tid & (HID - 1), jh = tid >> 7;          // column k, logits [jh*17, jh*17+17)
    const int j0 = jh * 17, j1 = min(A, j0 + 17);
    float acc[17];
#pragma unroll
    for (int i = 0; i < 17; ++i) acc[i] = 0.f;
    float accc = 0.f;
    for (int r0 = 0; r0 < nrows; r0 += 8) {
      float yv[8], ycv[8];
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const bool ok = r0 + i < nrows;
        yv[i] = ok ? Ybase[(r0 + i) * 2 * HID + k] : 0.f;
        ycv[i] = (ok && jh == 0) ? Ybase[(r0 + i) * 2 * HID + HID + k] : 0.f;
      }
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const int r = min(r0 + i, HEAD_ROWS_PER_CTA - 1);
#pragma unroll
        for (int ii = 0; ii < 17; ++ii)
          if (j0 + ii < j1) acc[ii] = fmaf(s_dl[r][j0 + ii], yv[i], acc[ii]);
        accc = fmaf(s_dv[r], ycv[i], accc);
      }
    }
#pragma unroll
    for (int i = 0; i < 17; ++i)
      if (j0 + i < j1) part[HP_W3A + (j0 + i) * HID + k] = acc[i];
    if (jh == 0) part[HP_W3C + k] = accc;
    if (tid < A) {          // bias gradients: column sums of d logits / d value
      float accb = 0.f;
      for (int r = 0; r < nrows; ++r) accb += s_dl[r][tid];
      part[HP_B3A + tid] = accb;
    } else if (tid == 64) {
      float accb = 0.f;
      for (int r = 0; r < nrows; ++r) accb += s_dv[r];
      part[HP_B3C] = accb;
    } else if (tid >= 128 && tid < 128 + p.W) {   // loss terms of worker tid - 128, rows in order
      const int w = tid - 128;
      float l0 = 0.f, l1 = 0.f, l2 = 0.f;
      for (int r = 0; r < HEAD_ROWS_PER_CTA; ++r)
        if (s_wk[r] == w) l0 += s_lt[r][0], l1 += s_lt[r][1], l2 += s_lt[r][2];
      part[HP_LOSS + w * 3 + 0] = l0, part[HP_LOSS + w * 3 + 1] = l1, part[HP_LOSS + w * 3 + 2] = l2;
    } else if (p.diag && tid >= 192 && tid < 192 + p.W) {   // diagnostics terms of worker tid - 192, rows in order
      const int w = tid - 192;
      float d0 = 0.f, d1 = 0.f, d2 = 0.f, d3 = 0.f;
      for (int r = 0; r < HEAD_ROWS_PER_CTA; ++r)
        if (s_wk[r] == w) d0 += s_dg[r][0], d1 += s_dg[r][1], d2 += s_dg[r][2], d3 += s_dg[r][3];
      float* pd = part + HP_DIAG + w * DIAG_TERMS;
      pd[0] = d0, pd[1] = d1, pd[2] = d2, pd[3] = d3;
    }
  }
  // ---- phase 3: the last CTA of the expert reduces the partials in block order
  __threadfence();
  __syncthreads();
  if (tid == 0) s_last = (atomicAdd(p.ctr + e, 1u) == static_cast<unsigned>(nblk - 1));
  __syncthreads();
  if (!s_last) return;
  __threadfence();
  const float* pe = p.partial + static_cast<long long>(e) * (p.cap / HEAD_ROWS_PER_CTA) * HEAD_PARTIAL;
  const int n_red = HP_LOSS + p.W * 3;
  for (int i0 = tid; i0 < n_red; i0 += 6 * 256) {
    float sums[6];
#pragma unroll
    for (int u = 0; u < 6; ++u) sums[u] = 0.f;
    for (int b = 0; b < nblk; ++b) {       // block order: deterministic; six independent elements per thread in flight
#pragma unroll
      for (int u = 0; u < 6; ++u)
        if (i0 + u * 256 < n_red) sums[u] += __ldcg(pe + static_cast<long long>(b) * HEAD_PARTIAL + i0 + u * 256);
    }
#pragma unroll
    for (int u = 0; u < 6; ++u) {
    const int i = i0 + u * 256;
    if (i >= n_red) continue;
    const float sum = sums[u];
    if (i < HP_W3C) {
      if (i < A * HID) p.grads[OFF_W3A + static_cast<long long>(e) * AMAX * HID + i] = sum;
    } else if (i < HP_B3A) {
      p.grads[OFF_W3C + e * HID + (i - HP_W3C)] = sum;
    } else if (i < HP_B3C) {
      if (i - HP_B3A < A) p.grads[OFF_B3A + e * B3A_LD + (i - HP_B3A)] = sum;
    } else if (i < HP_LOSS) {
      if (i == HP_B3C) p.grads[OFF_B3C + e * 4] = sum;
    } else {
      p.loss_e[e * HEAD_MAX_W * 3 + (i - HP_LOSS)] = sum;
    }
    }
  }
  if (p.diag) {
    for (int i = tid; i < p.W * DIAG_TERMS; i += 256) {
      float sum = 0.f;
      for (int b = 0; b < nblk; ++b) sum += __ldcg(pe + static_cast<long long>(b) * HEAD_PARTIAL + HP_DIAG + i);
      p.diag_e[e * HEAD_MAX_W * DIAG_TERMS + i] = sum;
    }
  }
  // ---- phase 4: the last expert to finish adds the per-expert losses in expert order
  __threadfence();
  __syncthreads();
  if (tid == 0) {
    int active = 0;
    for (int x = 0; x < E; ++x) active += p.counts[x] > 0;
    s_last = (atomicAdd(p.ctr + E, 1u) == static_cast<unsigned>(active - 1));
  }
  __syncthreads();
  if (!s_last) return;
  __threadfence();
  for (int i = tid; i < p.W * 2 * 3; i += 256) {
    const int w = i / 6, h = (i / 3) % 2, c = i % 3;
    float sum = 0.f;
    for (int x = 0; x < 4; ++x)
      if (p.counts[h * 4 + x] > 0) sum += __ldcg(p.loss_e + (h * 4 + x) * HEAD_MAX_W * 3 + w * 3 + c);
    p.losses[(w * 2 + h) * 3 + c] = sum;
  }
  if (p.diag) {
    for (int i = tid; i < p.W * 2 * DIAG_TERMS; i += 256) {
      const int w = i / (2 * DIAG_TERMS), h = (i / DIAG_TERMS) % 2, c = i % DIAG_TERMS;
      float sum = 0.f;
      for (int x = 0; x < 4; ++x)
        if (p.counts[h * 4 + x] > 0) sum += __ldcg(p.diag_e + (h * 4 + x) * HEAD_MAX_W * DIAG_TERMS + w * DIAG_TERMS + c);
      p.diag[i] = sum * p.inv_mb;
    }
    if (p.kl_sum) {     // this rank's share of the target-KL decision (kl_gate_kernel)
      __syncthreads();
      if (tid < 2) {
        float s = 0.f;
        for (int w = 0; w < p.W; ++w) s += p.diag[(w * 2 + tid) * DIAG_TERMS];
        p.kl_sum[tid] = s;
      }
    }
  }
}

// Forward-only variant for act() / get_value() / evaluate_actions (agent.py:114-164, models.py:184-212): writes,
// per routed row, [value, log-prob(action), entropy, logits[0..32]] to row_out[((worker*2+head)*mb + i)*ROW_OUT].
constexpr int ROW_OUT = 36;
__global__ void __launch_bounds__(256) head_eval_kernel(const float* __restrict__ Y2,
                                                        const float* __restrict__ params,
                                                        const int* __restrict__ row_slot,
                                                        const int* __restrict__ row_expert,
                                                        const int* __restrict__ actions_by_row, int R, int cap,
                                                        float* __restrict__ row_out) {
  pdl_trigger();
  pdl_wait();
  // one warp per (head, row r); r enumerates (worker, i) like the gather
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int g = blockIdx.x * 8 + warp;
  if (g >= 2 * R) return;
  const int head = g / R, r = g - head * R;
  const int e = row_expert[head * R + r], slot = row_slot[head * R + r];
  const int A = head == 0 ? 33 : 3;
  const long long row = static_cast<long long>(e) * cap + slot;
  const float* y = Y2 + row * 2 * HID;
  const float* W3A = params + OFF_W3A + static_cast<long long>(e) * AMAX * HID;
  float l0 = -INFINITY, l1 = -INFINITY;
  if (lane < A) {
    float acc = params[OFF_B3A + e * B3A_LD + lane];
    for (int k = 0; k < HID; ++k) acc = fmaf(y[k], W3A[lane * HID + k], acc);
    l0 = acc;
  }
  if (lane + 32 < A) {
    float acc = params[OFF_B3A + e * B3A_LD + lane + 32];
    for (int k = 0; k < HID; ++k) acc = fmaf(y[k], W3A[(lane + 32) * HID + k], acc);
    l1 = acc;
  }
  float v = 0.f;
  for (int q = 0; q < 4; ++q) v = fmaf(y[HID + lane + 32 * q], params[OFF_W3C + e * HID + lane + 32 * q], v);
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  v += params[OFF_B3C + e * 4];
  float mx = fmaxf(l0, l1);
  for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
  float se = (lane < A ? expf(l0 - mx) : 0.f) + (lane + 32 < A ? expf(l1 - mx) : 0.f);
  for (int o = 16; o > 0; o >>= 1) se += __shfl_xor_sync(0xffffffffu, se, o);
  const float lse = mx + logf(se);
  const float lp0 = l0 - lse, lp1 = l1 - lse;
  float ent = -((lane < A ? expf(lp0) * lp0 : 0.f) + (lane + 32 < A ? expf(lp1) * lp1 : 0.f));
  for (int o = 16; o > 0; o >>= 1) ent += __shfl_xor_sync(0xffffffffu, ent, o);
  const int a = actions_by_row[row];
  const float lp = __shfl_sync(0xffffffffu, (a < 32) ? lp0 : lp1, a & 31);
  float* o = row_out + static_cast<long long>(g) * ROW_OUT;
  if (lane == 0) o[0] = v, o[1] = lp, o[2] = ent;
  if (lane < A) o[3 + lane] = lp0;            // normalised logits (Categorical.logits)
  if (lane + 32 < A) o[3 + lane + 32] = lp1;
}

// Act step tail (cadre_ppo_act): block e samples both heads of environment e from head_eval_kernel's rows
// (row_out[(head * E + e) * ROW_OUT], W = 1) and writes the tick of storages 2e, 2e + 1 into the pool at `slot`
// (storage.py:45-58: everything but rewards / masks, which come from env.step afterwards).
__global__ void __launch_bounds__(256) act_write_kernel(const float* __restrict__ row_out, int E_env,
                                                        cadre_rollout_pool pool, int slot, unsigned long long seed,
                                                        unsigned long long tick, const int* __restrict__ env_ids,
                                                        const float* __restrict__ window,
                                                        const int* __restrict__ command,
                                                        const float* __restrict__ hid_h,
                                                        const float* __restrict__ hid_c,
                                                        long long* __restrict__ actions_out) {
  pdl_trigger();
  pdl_wait();
  const int e = blockIdx.x;
  const long long T1 = pool.num_steps + 1;
  if (threadIdx.x < 2) {
    const int h = threadIdx.x, A = h == 0 ? 33 : 3;
    const float* row = row_out + (static_cast<long long>(h) * E_env + e) * ROW_OUT;
    const float u = philox_uniform(philox_word(philox_words(seed, tick, env_ids[e], 0u), h));
    const int a = categorical_draw(row + 3, A, u);
    const long long at = (2LL * e + h) * T1 + slot;
    pool.action[at] = a;
    pool.action_log_probs[at] = row[3 + a];
    pool.value_preds[at] = row[0];
    pool.command[at] = command[e];
    actions_out[2 * e + h] = a;
  }
  const int win = pool.seq_length * pool.feature_dims;
  const float* src = window + static_cast<long long>(e) * win;
  float* d0 = pool.obs + (2LL * e * T1 + slot) * win;
  float* d1 = d0 + T1 * win;
  for (int k = threadIdx.x; k < win; k += blockDim.x) {
    const float v = src[k];
    d0[k] = v, d1[k] = v;
  }
  if (slot < pool.num_steps) {   // storage.py:84-87
    const int H = pool.hidden_size;
    const long long o0 = (2LL * e * T1 + slot + 1) * H, o1 = o0 + T1 * H;
    for (int k = threadIdx.x; k < H; k += blockDim.x) {
      const float vh = hid_h[k], vc = hid_c[k];
      pool.hn[o0 + k] = vh, pool.hn[o1 + k] = vh;
      pool.cn[o0 + k] = vc, pool.cn[o1 + k] = vc;
    }
  }
}

// Ensemble tail (cadre_ensemble_control, cadre_ppo_ensemble_act): one warp per environment e. Lane k (and k + 32)
// picks both heads' actions of snapshot k from row_out[k][h][e] (the sampler keyed with snapshot index k, or the first
// maximum of the log-probs in greedy mode); lane 0 then averages the snapshots' controls in float64, summed in snapshot
// order and divided by K, as numpy's mean(0) in CadreAgent.avg_action (agent.py:83-95) does.
constexpr int ENSEMBLE_MAX_K = 64;
constexpr int ENSEMBLE_WARPS = 4;
__device__ __forceinline__ int first_argmax(const float* lp, int A) {   // torch.argmax: the first maximum, NaN wins
  int best = 0;
  float bv = lp[0];
  for (int j = 1; j < A; ++j) {
    const float v = lp[j];
    if (bv == bv && (v > bv || v != v)) bv = v, best = j;
  }
  return best;
}

__global__ void __launch_bounds__(ENSEMBLE_WARPS * 32) ensemble_control_kernel(
    const float* __restrict__ row_out, int K, int E_env, unsigned long long seed, unsigned long long tick,
    const int* __restrict__ env_ids, int greedy, const double* __restrict__ steer_table,
    const double* __restrict__ throttle_table, double* __restrict__ controls_out, long long* __restrict__ actions_out) {
  pdl_trigger();
  pdl_wait();
  __shared__ unsigned char act[ENSEMBLE_WARPS][ENSEMBLE_MAX_K][2];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int e = blockIdx.x * ENSEMBLE_WARPS + warp;
  if (e >= E_env) return;
  const unsigned env_id = static_cast<unsigned>(env_ids[e]);
  for (int k = lane; k < K; k += 32) {
    const uint4 x = greedy ? make_uint4(0u, 0u, 0u, 0u) : philox_words(seed, tick, static_cast<int>(env_id), k);
    for (int h = 0; h < 2; ++h) {
      const int A = h == 0 ? 33 : 3;
      const float* lp = row_out + ((static_cast<long long>(k) * 2 + h) * E_env + e) * ROW_OUT + 3;
      const int a = greedy ? first_argmax(lp, A) : categorical_draw(lp, A, philox_uniform(philox_word(x, h)));
      act[warp][k][h] = static_cast<unsigned char>(a);
      actions_out[(static_cast<long long>(k) * E_env + e) * 2 + h] = a;
    }
  }
  __syncwarp();
  if (lane == 0) {
    double steer = 0.0, throttle = 0.0, brake = 0.0;
    for (int k = 0; k < K; ++k) {
      const int as = act[warp][k][0], at = act[warp][k][1];
      steer += steer_table[as];
      throttle += throttle_table[2 * at];
      brake += throttle_table[2 * at + 1];
    }
    const double n = static_cast<double>(K);
    steer /= n, throttle /= n, brake /= n;
    if (K > 1 && brake < 0.5) brake = 0.0;   // agent.py:92-94: several agents release a brake below one half
    controls_out[3 * e] = steer, controls_out[3 * e + 1] = throttle, controls_out[3 * e + 2] = brake;
  }
}

// Bootstrap tail (cadre_ppo_bootstrap, mini_batch = 1): next_value[w][h] = value of row (h, w), 0 for a done worker.
__global__ void bootstrap_value_kernel(const float* __restrict__ row_out, int W, unsigned long long done_mask,
                                       float* __restrict__ next_value) {
  pdl_trigger();
  pdl_wait();
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= 2 * W) return;
  const int w = i >> 1, h = i & 1;
  next_value[i] = ((done_mask >> w) & 1ull) ? 0.f : row_out[(static_cast<long long>(h) * W + w) * ROW_OUT];
}

// column sums over the valid rows of each expert (bias gradients); deterministic
__global__ void __launch_bounds__(256) colsum_kernel(const float* __restrict__ src, long long ld,
                                                     long long src_bs, const int* __restrict__ rows, int N,
                                                     float* __restrict__ dst, long long dst_bs,
                                                     float* __restrict__ dst2) {
  pdl_trigger();
  pdl_wait();
  __shared__ float sm[8][33];
  const int e = blockIdx.y;
  const int n = blockIdx.x * 32 + (threadIdx.x & 31);
  const int ry = threadIdx.x >> 5;
  const int R = rows[e];
  const float* s = src + e * src_bs;
  float acc = 0.f;
  if (n < N)
    for (int r = ry; r < R; r += 8) acc += s[r * ld + n];
  sm[ry][threadIdx.x & 31] = acc;
  __syncthreads();
  if (ry == 0 && n < N) {
    float t = 0.f;
#pragma unroll
    for (int k = 0; k < 8; ++k) t += sm[k][threadIdx.x & 31];
    dst[e * dst_bs + n] = t;
    if (dst2) dst2[e * dst_bs + n] = t;
  }
}

// ------------------------------------------------------------------------------------------ fp16 weight copies
// The LSTM weights as tensor-core operands: W_ih and W_hh rounded once per update to fp16 (the 11-bit significand of the
// TF32 operands they replace), rows padded to 544 halves, plus W_hh transposed ([unit][gate row], rows padded to 2176)
// for the BPTT kernel. Block (x, e, z): gate rows [32 x, 32 x + 32) x units [32 z, 32 z + 32) of expert e; the transpose
// goes through a padded shared-memory tile so that all global accesses are row segments. Runs on the plan's side stream while the main
// stream routes and gathers the minibatch.
__global__ void __launch_bounds__(256) wcvt_kernel(const float* __restrict__ params, __half* __restrict__ WIH16,
                                                   __half* __restrict__ WHH16, __half* __restrict__ WHHT16) {
  __shared__ float tile[32][33];
  const int e = blockIdx.y, g0 = blockIdx.x * 32, c0 = blockIdx.z * 32;   // 32 gate rows x 32 units per block
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;                 // 8 warps, 4 rows each
  const float* Wih = params + OFF_LSTM + e * LSTM_BLK + LSTM_WIH;
  const float* Whh = params + OFF_LSTM + e * LSTM_BLK + LSTM_WHH;
  __half* oih = WIH16 + static_cast<long long>(e) * G * LS_LDH16;
  __half* ohh = WHH16 + static_cast<long long>(e) * G * LS_LDH16;
  __half* oT = WHHT16 + static_cast<long long>(e) * LS_LDH16 * LS_LDG16;
  const int c = c0 + tx;
  float a[4], b[4];
#pragma unroll
  for (int k = 0; k < 4; ++k) {     // all eight loads of the thread in flight
    const int g = g0 + ty + 8 * k;
    const bool ok = g < G && c < F;
    a[k] = ok ? Wih[static_cast<long long>(g) * LDF + c] : 0.f;
    b[k] = ok ? Whh[static_cast<long long>(g) * LDF + c] : 0.f;
  }
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    const int r = ty + 8 * k, g = g0 + r;
    if (g < G) {
      oih[static_cast<long long>(g) * LS_LDH16 + c] = __float2half_rn(a[k]);
      ohh[static_cast<long long>(g) * LS_LDH16 + c] = __float2half_rn(b[k]);
    }
    tile[r][tx] = b[k];
  }
  __syncthreads();
#pragma unroll
  for (int k = 0; k < 4; ++k) {     // unit c0 + r, gate rows g0 + tx (zeros in the K padding 2120 .. 2175)
    const int r = ty + 8 * k;
    oT[static_cast<long long>(c0 + r) * LS_LDG16 + g0 + tx] = __float2half_rn(tile[tx][r]);
  }
}

__global__ void set_counters_kernel(int* ctrs, int step_ctr, int opt_step) {
  ctrs[0] = step_ctr;
  if (opt_step >= 0) ctrs[1] = opt_step;   // opt_step < 0: the Adam step continues from the device counter
}

// ------------------------------------------------------------------------------------------ target-KL early stopping
// SB3's rule (on_policy ppo.py: `if approx_kl_div > 1.5 * target_kl: continue_training = False; break`, before the
// optimizer step) applied on the device, so that a phase of staged update steps needs no host synchronisation. State
// words of the phase (cadre_ppo_kl_begin clears them):
constexpr int KS_SKIP_NORM = 0;    // the phase was stopped before the current step: no gradient norms, no Adam step
constexpr int KS_STOPPED = 1;      // the phase is stopped: no Adam step from the current step on
constexpr int KS_STEP = 2;         // update steps of the phase gated so far
constexpr int KS_RUN = 3;          // steps that ran their forward and backward: applied ones + the one that stopped
constexpr int KS_APPLIED = 4;      // steps whose Adam update was applied
constexpr int KS_STOPPED_AT = 5;   // index of the step that stopped the phase (valid while KS_STOPPED is set)
constexpr int KS_WORDS = 8;
constexpr int KL_HIST_CAP = 4096;  // steps of a phase whose KL is kept
// One thread, after the cross-rank sum of head_kernel's per-head KL sums and before the step's first norm / Adam
// launch. KL = sum over heads of (sum over the workers of all ranks) * (1 / total workers), the same operations in the
// same order on every rank, so every rank takes the same decision from the same bits. A step that is not applied gives
// back the Adam step prep_kernel took for it.
__global__ void kl_gate_kernel(const float* __restrict__ kl_sum, float inv_total, float limit, int* __restrict__ st,
                               float* __restrict__ hist, int* __restrict__ opt_step) {
  pdl_trigger();
  pdl_wait();
  const int n = st[KS_STEP];
  st[KS_STEP] = n + 1;
  st[KS_SKIP_NORM] = st[KS_STOPPED];
  if (st[KS_STOPPED]) {
    *opt_step -= 1;
    return;
  }
  const float kl = __fadd_rn(__fmul_rn(kl_sum[0], inv_total), __fmul_rn(kl_sum[1], inv_total));
  if (n < KL_HIST_CAP) hist[n] = kl;
  st[KS_RUN] += 1;
  if (kl > limit) {
    st[KS_STOPPED] = 1;
    st[KS_STOPPED_AT] = n;
    *opt_step -= 1;
  } else {
    st[KS_APPLIED] += 1;
  }
}

// ------------------------------------------------------------------------------------------ plan
constexpr int MAX_STAGED = 64;   // update steps whose minibatch indices can be staged at once (ppo_epoch x minibatches)
struct PpoPlan {
  cadre_ppo_config cfg;
  int cap = 0, R = 0;
  // device buffers
  float *XP9 = nullptr, *C9 = nullptr, *H8 = nullptr;   // H8 [E][cap][LDF]: h_8, input of the heads
  float *Y1 = nullptr, *Y2 = nullptr, *dZ1 = nullptr, *dZ2 = nullptr, *dH = nullptr, *dC = nullptr;
  float* bsum = nullptr;
  // fp16 tensors in the 9-slot layout (see the file header) + hand-off counters and prebuilt tensor maps of the
  // persistent recurrence kernels (lstm_seq.cuh)
  __half *X16 = nullptr, *H16 = nullptr, *G16 = nullptr, *dG16 = nullptr;
  __half *WIH16 = nullptr, *WHH16 = nullptr, *WHHT16 = nullptr;   // fp16 weight copies (wcvt_kernel)
  CUtensorMap tmW, tmWT;
  cudaEvent_t ev_wcvt_fork = nullptr, ev_wcvt = nullptr;
  float *head_partial = nullptr, *head_loss_e = nullptr, *head_diag_e = nullptr;   // head_kernel scratch (ordered reductions)
  float* diag_out = nullptr;       // cadre_ppo_set_diagnostics: [W][2][4] of the next update, 16 norms of the next Adam step
  float* norms_out = nullptr;
  // target-KL early stopping (cadre_ppo_set_target_kl): kl_sum = caller's rank-summed [2] (NULL: off)
  float* kl_sum = nullptr;
  float kl_limit = 0.f, kl_inv_total = 0.f;
  int* kl_state = nullptr;         // [KS_WORDS] phase state (kl_gate_kernel)
  float* kl_hist = nullptr;        // [KL_HIST_CAP] KL of each step of the phase that ran
  float* kl_diag = nullptr;        // [W][2][4] diagnostics scratch while diag_out is NULL
  unsigned* seq_sync = nullptr;          // [0, E]: forward counters + error flag, [16, 16 + E]: backward, [32, 32 + E]: head
  CUtensorMap tmH, tmDG;
  float bwd_scale = 1.f;
  RowScalars sc{};
  int *row_slot = nullptr, *row_expert = nullptr, *counts = nullptr, *counts9 = nullptr;
  int* idx_dev = nullptr;          // staged index table [MAX_STAGED][2 R]
  int* ctrs = nullptr;             // [0] step counter into idx_dev, [1] 1-based Adam step of the current update
  int32_t* idx_pinned = nullptr;   // pinned staging of the table and of the storage refs
  StorageRef* refs_pinned = nullptr;
  cudaEvent_t ev_staged = nullptr;
  int staged_steps = 0;
  int host_step = 1;               // Adam step the one-step (non-staged) path writes into ctrs[1]; see adam_step
  int* xp_tiles = nullptr;   // work list of the x-part GEMM (prep_kernel)
  int xp_max_tiles = 0;
  StorageRef* refs_dev = nullptr;
  OptTables opt;
  int launches = 0;
  // side stream for the gradient kernels that are off the critical path (dW2, dW1, bias column sums)
  cudaStream_t side = nullptr;
  cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
  // data-parallel pipeline: the LSTM weight gradients are produced per group of E / grad_groups experts, one event
  // per group; ev_mlp fires when every actor-critic gradient (side stream) is final
  int grad_groups = 1;
  cudaEvent_t ev_grp[8] = {};
  cudaEvent_t ev_mlp = nullptr;
  bool use_side = true;
};

template <typename T>
static T* dalloc(size_t n) {
  T* p = nullptr;
  CADRE_CUDA_CHECK(cudaMalloc(&p, n * sizeof(T)));
  CADRE_CUDA_CHECK(cudaMemset(p, 0, n * sizeof(T)));
  return p;
}

static PpoPlan* ppo_create(const cadre_ppo_config* cfg) {
  CADRE_REQUIRE(cfg && cfg->workers > 0 && cfg->mini_batch > 0, "ppo config");
  PpoPlan* P = new PpoPlan();
  P->cfg = *cfg;
  P->R = cfg->workers * cfg->mini_batch;
  P->cap = (P->R + 127) / 128 * 128;  // worst case: every row of a head carries the same command
  const size_t rows = static_cast<size_t>(E) * P->cap;
  P->XP9 = dalloc<float>(rows * 9 * G);
  P->H8 = dalloc<float>(rows * LDF);
  P->C9 = dalloc<float>(rows * 9 * LDF);
  P->Y1 = dalloc<float>(rows * 2 * HID);
  P->Y2 = dalloc<float>(rows * 2 * HID);
  P->dZ1 = dalloc<float>(rows * 2 * HID);
  P->dZ2 = dalloc<float>(rows * 2 * HID);
  P->dH = dalloc<float>(rows * LDF);
  P->use_side = getenv("CADRE_PPO_NO_SIDE_STREAM") == nullptr;
  CADRE_CUDA_CHECK(cudaStreamCreateWithFlags(&P->side, cudaStreamNonBlocking));
  CADRE_CUDA_CHECK(cudaEventCreateWithFlags(&P->ev_fork, cudaEventDisableTiming));
  CADRE_CUDA_CHECK(cudaEventCreateWithFlags(&P->ev_join, cudaEventDisableTiming));
  for (int i = 0; i < 8; ++i) CADRE_CUDA_CHECK(cudaEventCreateWithFlags(&P->ev_grp[i], cudaEventDisableTiming));
  CADRE_CUDA_CHECK(cudaEventCreateWithFlags(&P->ev_mlp, cudaEventDisableTiming));
  P->dC = dalloc<float>(rows * LDF);
  P->bsum = dalloc<float>(static_cast<size_t>(E) * G);
  P->X16 = dalloc<__half>(rows * 9 * LS_LDH16);
  P->H16 = dalloc<__half>(rows * 9 * LS_LDH16);
  P->G16 = dalloc<__half>(rows * 9 * G);
  P->dG16 = dalloc<__half>(rows * 9 * LS_LDG16);
  P->WIH16 = dalloc<__half>(static_cast<size_t>(E) * G * LS_LDH16);
  P->WHH16 = dalloc<__half>(static_cast<size_t>(E) * G * LS_LDH16);
  P->WHHT16 = dalloc<__half>(static_cast<size_t>(E) * LS_LDH16 * LS_LDG16);
  CADRE_CUDA_CHECK(cudaEventCreateWithFlags(&P->ev_wcvt_fork, cudaEventDisableTiming));
  CADRE_CUDA_CHECK(cudaEventCreateWithFlags(&P->ev_wcvt, cudaEventDisableTiming));
  P->seq_sync = dalloc<unsigned>(64);
  CADRE_REQUIRE(cfg->workers <= HEAD_MAX_W, "at most 64 workers per engine");
  P->head_partial = dalloc<float>(static_cast<size_t>(E) * (P->cap / HEAD_ROWS_PER_CTA) * HEAD_PARTIAL);
  P->head_loss_e = dalloc<float>(static_cast<size_t>(E) * HEAD_MAX_W * 3);
  P->head_diag_e = dalloc<float>(static_cast<size_t>(E) * HEAD_MAX_W * DIAG_TERMS);
  P->kl_state = dalloc<int>(KS_WORDS);
  P->kl_hist = dalloc<float>(KL_HIST_CAP);
  P->kl_diag = dalloc<float>(static_cast<size_t>(cfg->workers) * 2 * DIAG_TERMS);
  {
    const uint64_t dims_h[4] = {(uint64_t)F, (uint64_t)P->cap, 9, (uint64_t)E};
    const uint64_t str_h[3] = {9ull * LS_LDH16 * 2, 1ull * LS_LDH16 * 2, (uint64_t)P->cap * 9 * LS_LDH16 * 2};
    const uint32_t box[4] = {64, 128, 1, 1};
    make_tensor_map_f16(&P->tmH, 4, P->H16, dims_h, str_h, box);
    const uint64_t dims_g[4] = {(uint64_t)LS_LDG16, (uint64_t)P->cap, 9, (uint64_t)E};
    const uint64_t str_g[3] = {9ull * LS_LDG16 * 2, 1ull * LS_LDG16 * 2, (uint64_t)P->cap * 9 * LS_LDG16 * 2};
    make_tensor_map_f16(&P->tmDG, 4, P->dG16, dims_g, str_g, box);
    const uint64_t dims_w[3] = {(uint64_t)F, (uint64_t)G, (uint64_t)E};
    const uint64_t str_w[2] = {1ull * LS_LDH16 * 2, (uint64_t)G * LS_LDH16 * 2};
    const uint32_t box_w[3] = {64, 128, 1};
    make_tensor_map_f16(&P->tmW, 3, P->WHH16, dims_w, str_w, box_w);
    const uint64_t dims_t[3] = {(uint64_t)G, (uint64_t)F, (uint64_t)E};
    const uint64_t str_t[2] = {1ull * LS_LDG16 * 2, (uint64_t)LS_LDH16 * LS_LDG16 * 2};
    const uint32_t box_t[3] = {64, 32, 1};
    make_tensor_map_f16(&P->tmWT, 3, P->WHHT16, dims_t, str_t, box_t);
    // backward operands are scaled by 2^(ceil(log2(mini_batch)) + 4): the loss seeds carry a 1/mini_batch factor
    int lg = 0;
    while ((1 << lg) < cfg->mini_batch) ++lg;
    P->bwd_scale = ldexpf(1.f, std::min(lg + 4, 14));
    static size_t cfg_f[CADRE_MAX_DEVICES] = {}, cfg_b[CADRE_MAX_DEVICES] = {};
    ensure_dynamic_smem(lstm_seq_fwd_kernel, LSF_SMEM, cfg_f);
    ensure_dynamic_smem(lstm_seq_bwd_kernel, LSB_SMEM, cfg_b);
  }
  P->sc.action = dalloc<int>(rows);
  P->sc.worker = dalloc<int>(rows);
  P->sc.old_v = dalloc<float>(rows);
  P->sc.ret = dalloc<float>(rows);
  P->sc.old_lp = dalloc<float>(rows);
  P->sc.adv = dalloc<float>(rows);
  P->row_slot = dalloc<int>(2 * static_cast<size_t>(P->R));
  P->row_expert = dalloc<int>(2 * static_cast<size_t>(P->R));
  P->counts = dalloc<int>(E);
  P->counts9 = dalloc<int>(E);
  P->idx_dev = dalloc<int>(static_cast<size_t>(MAX_STAGED) * 2 * P->R);
  P->ctrs = dalloc<int>(4);
  CADRE_CUDA_CHECK(cudaHostAlloc(&P->idx_pinned, sizeof(int32_t) * MAX_STAGED * 2 * P->R, cudaHostAllocDefault));
  CADRE_CUDA_CHECK(cudaHostAlloc(&P->refs_pinned, sizeof(StorageRef) * 2 * cfg->workers, cudaHostAllocDefault));
  CADRE_CUDA_CHECK(cudaEventCreateWithFlags(&P->ev_staged, cudaEventDisableTiming));
  P->xp_max_tiles = (2 * 9 * P->R + 127) / 128 + E;   // sum_e ceil(9 count_e / 128), sum_e count_e = 2 R
  P->xp_tiles = dalloc<int>(1 + 2 * static_cast<size_t>(P->xp_max_tiles));
  P->refs_dev = dalloc<StorageRef>(2 * static_cast<size_t>(cfg->workers));

  // optimizer chunk table, grouped by module: module e = LSTM of expert e, module 8+e = actor-critic of expert e
  struct Piece {
    long long off, len;
    int mod;
  };
  std::vector<Piece> pieces;
  for (int e = 0; e < E; ++e) {
    pieces.push_back({OFF_LSTM + e * LSTM_BLK, LSTM_BLK, e});   // W_ih | W_hh | b_ih | b_hh of expert e: one module
  }
  for (int e = 0; e < E; ++e) {
    pieces.push_back({OFF_W1 + (long long)e * 2 * HID * LDF, 2LL * HID * LDF, 8 + e});
    pieces.push_back({OFF_B1 + (long long)e * 2 * HID, 2 * HID, 8 + e});
    pieces.push_back({OFF_W2 + (long long)e * 2 * HID * HID, 2LL * HID * HID, 8 + e});
    pieces.push_back({OFF_B2 + (long long)e * 2 * HID, 2 * HID, 8 + e});
    pieces.push_back({OFF_W3A + (long long)e * AMAX * HID, (long long)AMAX * HID, 8 + e});
    pieces.push_back({OFF_B3A + (long long)e * B3A_LD, B3A_LD, 8 + e});
    pieces.push_back({OFF_W3C + (long long)e * HID, HID, 8 + e});
    pieces.push_back({OFF_B3C + (long long)e * 4, 4, 8 + e});
  }
  std::stable_sort(pieces.begin(), pieces.end(), [](const Piece& a, const Piece& b) { return a.mod < b.mod; });
  std::vector<long long> coff;
  std::vector<int> clen, cmod, mfirst(17, 0);
  const int CH = 8192;
  for (const Piece& pc : pieces)
    for (long long o = 0; o < pc.len; o += CH) {
      coff.push_back(pc.off + o);
      clen.push_back(static_cast<int>(std::min<long long>(CH, pc.len - o)));
      cmod.push_back(pc.mod);
    }
  for (size_t i = 0; i < cmod.size(); ++i) mfirst[cmod[i] + 1] = static_cast<int>(i) + 1;
  for (int m = 1; m <= 16; ++m) mfirst[m] = std::max(mfirst[m], mfirst[m - 1]);
  OptTables& T = P->opt;
  T.num_chunks = static_cast<int>(coff.size());
  T.chunk_off = dalloc<long long>(coff.size());
  T.chunk_len = dalloc<int>(coff.size());
  T.chunk_mod = dalloc<int>(coff.size());
  T.mod_first = dalloc<int>(17);
  T.partial = dalloc<float>(coff.size());
  T.clip_coef = dalloc<float>(16);
  T.norms = dalloc<float>(16);
  T.scalars = dalloc<float>(2);
  CADRE_CUDA_CHECK(cudaMemcpy(T.chunk_off, coff.data(), coff.size() * 8, cudaMemcpyHostToDevice));
  CADRE_CUDA_CHECK(cudaMemcpy(T.chunk_len, clen.data(), clen.size() * 4, cudaMemcpyHostToDevice));
  CADRE_CUDA_CHECK(cudaMemcpy(T.chunk_mod, cmod.data(), cmod.size() * 4, cudaMemcpyHostToDevice));
  CADRE_CUDA_CHECK(cudaMemcpy(T.mod_first, mfirst.data(), 17 * 4, cudaMemcpyHostToDevice));
  for (int m = 0; m <= 16; ++m) T.mod_first_h[m] = mfirst[m];
  return P;
}

static void ppo_destroy(PpoPlan* P) {
  if (!P) return;
  void* ptrs[] = {P->head_partial, P->head_loss_e, P->head_diag_e, P->X16, P->H16, P->G16, P->dG16, P->WIH16, P->WHH16, P->WHHT16, P->seq_sync, P->XP9, P->H8, P->C9, P->Y1, P->Y2, P->dZ1, P->dZ2, P->dH, P->dC, P->bsum,
                  P->sc.action, P->sc.worker, P->sc.old_v, P->sc.ret, P->sc.old_lp, P->sc.adv, P->row_slot,
                  P->row_expert, P->counts, P->counts9, P->idx_dev, P->ctrs, P->xp_tiles, P->refs_dev, P->opt.chunk_off, P->opt.chunk_len,
                  P->opt.chunk_mod, P->opt.mod_first, P->opt.partial, P->opt.clip_coef, P->opt.norms, P->opt.scalars,
                  P->kl_state, P->kl_hist, P->kl_diag};
  for (void* p : ptrs) cudaFree(p);
  if (P->side) cudaStreamDestroy(P->side);
  if (P->idx_pinned) cudaFreeHost(P->idx_pinned);
  if (P->refs_pinned) cudaFreeHost(P->refs_pinned);
  if (P->ev_staged) cudaEventDestroy(P->ev_staged);
  if (P->ev_fork) cudaEventDestroy(P->ev_fork);
  if (P->ev_wcvt_fork) cudaEventDestroy(P->ev_wcvt_fork);
  if (P->ev_wcvt) cudaEventDestroy(P->ev_wcvt);
  if (P->ev_join) cudaEventDestroy(P->ev_join);
  for (cudaEvent_t ev : P->ev_grp)
    if (ev) cudaEventDestroy(ev);
  if (P->ev_mlp) cudaEventDestroy(P->ev_mlp);
  delete P;
}

static GemmArgs tf32_gemm(int a_mn, int b_mn) {
  GemmArgs g;
  g.kind = 1, g.a_mn = a_mn, g.b_mn = b_mn, g.batch = E, g.out_f32 = 1, g.block_n = 128;
  return g;
}

// Upload the storage references and the minibatch indices of `n_steps` consecutive update steps ([n_steps][W][2][mb])
// and rewind the step counter; `first_step` is the 1-based Adam step of the first of them (0: continue the device counter).
static void ppo_stage(PpoPlan* P, const cadre_storage_ref* refs_host, const int32_t* idx_host, int n_steps,
                      int first_step, cudaStream_t s) {
  CADRE_REQUIRE(n_steps >= 1 && n_steps <= MAX_STAGED, "between 1 and 64 update steps can be staged");
  const int W = P->cfg.workers, R = P->R;
  CADRE_CUDA_CHECK(cudaEventSynchronize(P->ev_staged));   // the previous upload has left the pinned buffers
  memcpy(P->idx_pinned, idx_host, sizeof(int32_t) * static_cast<size_t>(n_steps) * 2 * R);
  memcpy(P->refs_pinned, refs_host, sizeof(StorageRef) * 2 * W);
  CADRE_CUDA_CHECK(cudaMemcpyAsync(P->idx_dev, P->idx_pinned, sizeof(int32_t) * static_cast<size_t>(n_steps) * 2 * R,
                                   cudaMemcpyHostToDevice, s));
  CADRE_CUDA_CHECK(cudaMemcpyAsync(P->refs_dev, P->refs_pinned, sizeof(StorageRef) * 2 * W, cudaMemcpyHostToDevice, s));
  set_counters_kernel<<<1, 1, 0, s>>>(P->ctrs, 0, first_step - 1);
  CADRE_CUDA_CHECK(cudaGetLastError());
  CADRE_CUDA_CHECK(cudaEventRecord(P->ev_staged, s));
  P->staged_steps = n_steps;
}

// routing + gather + forward through the second hidden layer (Y2); returns the number of kernels launched.
// idx_host == nullptr: use the staged table (no host copies: capturable in a CUDA graph).
static int ppo_forward(PpoPlan* P, const cadre_storage_ref* refs_host, const int32_t* idx_host,
                       const float* params, cudaStream_t s, const int* stop = nullptr) {
  const int W = P->cfg.workers, mb = P->cfg.mini_batch, cap = P->cap, R = P->R;
  const long long rs9G = static_cast<long long>(cap) * 9 * G;
  int n = 0;
  // fp16 copies of the LSTM weights for this call (parameters may have changed since the last one: Adam step,
  // load_state_dict, update_model): on the side stream, next to the routing / gather kernels
  CADRE_CUDA_CHECK(cudaEventRecord(P->ev_wcvt_fork, s));
  CADRE_CUDA_CHECK(cudaStreamWaitEvent(P->side, P->ev_wcvt_fork, 0));
  wcvt_kernel<<<dim3(LS_LDG16 / 32, E, LS_LDH16 / 32), 256, 0, P->side>>>(params, P->WIH16, P->WHH16, P->WHHT16);
  CADRE_CUDA_CHECK(cudaGetLastError());
  ++n;
  CADRE_CUDA_CHECK(cudaEventRecord(P->ev_wcvt, P->side));
  CADRE_CUDA_CHECK(cudaMemsetAsync(P->seq_sync, 0, sizeof(unsigned) * E, s));            // forward hand-off counters
  CADRE_CUDA_CHECK(cudaMemsetAsync(P->seq_sync + 16, 0, sizeof(unsigned) * E, s));       // backward
  CADRE_CUDA_CHECK(cudaMemsetAsync(P->seq_sync + 32, 0, sizeof(unsigned) * (E + 1), s));  // head_kernel reductions
  if (idx_host != nullptr) ppo_stage(P, refs_host, idx_host, 1, P->host_step, s);   // one-step table
  launch_k(route_kernel, dim3(2), dim3(1024), 0, s, P->refs_dev, P->idx_dev, P->ctrs, W, mb, P->row_slot, P->row_expert,
           P->counts, P->counts9, stop), ++n;
  launch_k(pack_kernel, dim3(dim3(R, 2)), dim3(256), 0, s, P->refs_dev, P->idx_dev, P->ctrs, W, mb, cap, P->row_slot, P->row_expert,
                                         P->X16, P->C9, P->H16, P->sc, stop), ++n;
  launch_k(prep_kernel, dim3((E * G + 255) / 256), dim3(256), 0, s, params, P->bsum, E * G,
           P->counts9, P->xp_tiles, P->xp_max_tiles, P->dG16, cap, P->ctrs, P->ctrs + 1), ++n;
  CADRE_CUDA_CHECK(cudaGetLastError());

  // ---- forward
  CADRE_CUDA_CHECK(cudaStreamWaitEvent(s, P->ev_wcvt, 0));   // the fp16 weight copies are complete from here on
  {  // x-part of all 8 (+1 dummy) time slots: XP9 = X W_ih^T + (b_ih + b_hh), fp16 operands, fp32 accumulation
    GemmArgs g;
    g.kind = 0, g.batch = E, g.out_f32 = 1, g.block_n = 128;
    g.A = P->X16, g.lda = LS_LDH16, g.a_bs = static_cast<long long>(cap) * 9 * LS_LDH16;
    g.B = P->WIH16, g.ldb = LS_LDH16, g.b_bs = static_cast<long long>(G) * LS_LDH16;
    g.M = 9 * cap, g.N = G, g.K = F;
    g.out = P->XP9, g.ldc = G, g.out_bs = rs9G;
    g.bias = P->bsum, g.bias_bs = G;
    g.batch_rows = P->counts9;
    g.tile_list = P->xp_tiles, g.max_tiles = P->xp_max_tiles;
    launch_gemm(g, s), ++n;
  }
  {   // models.py:146-151: the 8 sequential LSTMCell steps in ONE persistent launch (lstm_seq.cuh)
    LstmFwdParams q;
    q.tmH = P->tmH, q.tmW = P->tmW, q.XP9 = P->XP9, q.G16 = P->G16, q.C9 = P->C9, q.H8 = P->H8, q.H16 = P->H16;
    q.counts = P->counts, q.sync = P->seq_sync, q.cap = cap;
    q.dbg = g_dbg_clk;
    launch_k(lstm_seq_fwd_kernel, dim3(LS_SLICES, E), dim3(LSF_THREADS), LSF_SMEM, s, q), ++n;
    CADRE_CUDA_CHECK(cudaGetLastError());
  }
  {  // first actor + critic layers share the input h_8: one N = 256 GEMM
    GemmArgs g = tf32_gemm(0, 0);
    g.A = P->H8, g.lda = LDF, g.a_bs = static_cast<long long>(cap) * LDF;
    g.B = params + OFF_W1, g.ldb = LDF, g.b_bs = 2LL * HID * LDF;
    g.M = cap, g.N = 2 * HID, g.K = F;
    g.out = P->Y1, g.ldc = 2 * HID, g.out_bs = static_cast<long long>(cap) * 2 * HID;
    g.bias = params + OFF_B1, g.bias_bs = 2 * HID, g.act = 1;
    g.batch_rows = P->counts;
    launch_gemm(g, s), ++n;
  }
  for (int br = 0; br < 2; ++br) {
    GemmArgs g = tf32_gemm(0, 0);
    g.A = P->Y1 + br * HID, g.lda = 2 * HID, g.a_bs = static_cast<long long>(cap) * 2 * HID;
    g.B = params + OFF_W2 + br * HID * HID, g.ldb = HID, g.b_bs = 2LL * HID * HID;
    g.M = cap, g.N = HID, g.K = HID;
    g.out = P->Y2 + br * HID, g.ldc = 2 * HID, g.out_bs = static_cast<long long>(cap) * 2 * HID;
    g.bias = params + OFF_B2 + br * HID, g.bias_bs = 2 * HID, g.act = 1;
    g.batch_rows = P->counts;
    launch_gemm(g, s), ++n;
  }
  return n;
}

static void ppo_update(PpoPlan* P, const cadre_storage_ref* refs_host, const int32_t* idx_host, float* params,
                       float* grads, float* losses, cudaStream_t s) {
  const int W = P->cfg.workers, mb = P->cfg.mini_batch, cap = P->cap;
  CADRE_CUDA_CHECK(cudaMemsetAsync(losses, 0, sizeof(float) * W * 2 * 3, s));
  CADRE_CUDA_CHECK(cudaMemsetAsync(grads + OFF_W3A, 0, sizeof(float) * (TOTAL - OFF_W3A), s));
  // target-KL early stopping applies to staged steps (a phase); a one-step update runs as with it off
  const bool gate = P->kl_sum != nullptr && idx_host == nullptr;
  int n = ppo_forward(P, refs_host, idx_host, params, s, gate ? P->kl_state + KS_STOPPED : nullptr);
  {
    HeadParams hp;
    hp.Y2 = P->Y2, hp.dZ2 = P->dZ2, hp.params = params, hp.grads = grads, hp.counts = P->counts, hp.sc = P->sc;
    hp.losses = losses, hp.cap = cap, hp.W = W, hp.inv_mb = 1.f / static_cast<float>(mb);
    hp.partial = P->head_partial, hp.loss_e = P->head_loss_e, hp.ctr = P->seq_sync + 32;
    hp.diag = P->diag_out, hp.diag_e = P->head_diag_e, hp.kl_sum = nullptr;
    if (gate) {
      if (hp.diag == nullptr) hp.diag = P->kl_diag;
      hp.kl_sum = P->kl_sum;
    }
    hp.clip = P->cfg.clip, hp.value_coeff = P->cfg.value_coeff, hp.clip_coeff = P->cfg.clip_coeff;
    hp.ent_coeff = P->cfg.ent_coeff;
    launch_k(head_kernel, dim3(dim3(cap / HEAD_ROWS_PER_CTA, E)), dim3(256), 0, s, hp), ++n;
    CADRE_CUDA_CHECK(cudaGetLastError());
  }

  // ---- backward. Critical path: head -> dZ1 -> dh_8 -> 8 x (LSTM cell backward, dgrad) -> LSTM weight gradients.
  // The second-layer / first-layer weight gradients and the bias column sums only consume finished tensors, so
  // they run on a side stream next to the BPTT chain (whose kernels leave most SMs idle).
  const long long bs256 = static_cast<long long>(cap) * 2 * HID;
  for (int br = 0; br < 2; ++br) {
    {  // dZ1 = (dZ2 W2) * relu'(Y1)
      GemmArgs g = tf32_gemm(0, 1);
      g.A = P->dZ2 + br * HID, g.lda = 2 * HID, g.a_bs = bs256;
      g.B = params + OFF_W2 + br * HID * HID, g.ldb = HID, g.b_bs = 2LL * HID * HID;
      g.M = cap, g.N = HID, g.K = HID;
      g.out = P->dZ1 + br * HID, g.ldc = 2 * HID, g.out_bs = bs256;
      g.mask = P->Y1 + br * HID, g.ldm = 2 * HID, g.mask_bs = bs256;
      g.batch_rows = P->counts;
      launch_gemm(g, s), ++n;
    }
  }
  cudaStream_t s2 = P->use_side ? P->side : s;
  if (P->use_side) {
    CADRE_CUDA_CHECK(cudaEventRecord(P->ev_fork, s));
    CADRE_CUDA_CHECK(cudaStreamWaitEvent(s2, P->ev_fork, 0));
  }
  for (int br = 0; br < 2; ++br) {
    {  // dW2 = dZ2^T Y1
      GemmArgs g = tf32_gemm(1, 1);
      g.A = P->dZ2 + br * HID, g.lda = 2 * HID, g.a_bs = bs256;
      g.B = P->Y1 + br * HID, g.ldb = 2 * HID, g.b_bs = bs256;
      g.M = HID, g.N = HID, g.K = cap;
      g.out = grads + OFF_W2 + br * HID * HID, g.ldc = HID, g.out_bs = 2LL * HID * HID;
      g.batch_rows = P->counts, g.rows_is_k = 1;
      launch_gemm(g, s2), ++n;
    }
  }
  launch_k(colsum_kernel, dim3(dim3(8, E)), dim3(256), 0, s2, P->dZ2, 2 * HID, bs256, P->counts, 2 * HID, grads + OFF_B2, 2 * HID,
                                           nullptr), ++n;
  launch_k(colsum_kernel, dim3(dim3(8, E)), dim3(256), 0, s2, P->dZ1, 2 * HID, bs256, P->counts, 2 * HID, grads + OFF_B1, 2 * HID,
                                           nullptr), ++n;
  {  // dW1 = dZ1^T h_8
    GemmArgs g = tf32_gemm(1, 1);
    g.A = P->dZ1, g.lda = 2 * HID, g.a_bs = bs256;
    g.B = P->H8, g.ldb = LDF, g.b_bs = static_cast<long long>(cap) * LDF;
    g.M = 2 * HID, g.N = F, g.K = cap;
    g.out = grads + OFF_W1, g.ldc = LDF, g.out_bs = 2LL * HID * LDF;
    g.batch_rows = P->counts, g.rows_is_k = 1;
    launch_gemm(g, s2), ++n;
  }
  {  // dh_8 = dZ1 W1
    GemmArgs g = tf32_gemm(0, 1);
    g.A = P->dZ1, g.lda = 2 * HID, g.a_bs = bs256;
    g.B = params + OFF_W1, g.ldb = LDF, g.b_bs = 2LL * HID * LDF;
    g.M = cap, g.N = F, g.K = 2 * HID;
    g.out = P->dH, g.ldc = LDF, g.out_bs = static_cast<long long>(cap) * LDF;
    g.batch_rows = P->counts;
    launch_gemm(g, s), ++n;
  }
  {   // BPTT: 8 x (LSTM-cell backward, dh_{t-1} = dG_t W_hh) in ONE persistent launch; it also produces the LSTM
      // bias gradients (column sums of dG)
    LstmBwdParams q;
    q.tmDG = P->tmDG, q.tmWT = P->tmWT, q.G16 = P->G16, q.C9 = P->C9, q.dG16 = P->dG16;
    q.dH8 = P->dH, q.dC = P->dC, q.counts = P->counts, q.sync = P->seq_sync + 16, q.cap = cap;
    q.scale = P->bwd_scale, q.inv_scale = 1.f / P->bwd_scale;
    q.grads = grads;
    q.dbg = g_dbg_clk ? g_dbg_clk + E * LS_SLICES * 72 : nullptr;
    launch_k(lstm_seq_bwd_kernel, dim3(LS_SLICES, E), dim3(LSB_THREADS), LSB_SMEM, s, q), ++n;
  }
  CADRE_CUDA_CHECK(cudaGetLastError());
  if (P->use_side) CADRE_CUDA_CHECK(cudaEventRecord(P->ev_join, s2));
  CADRE_CUDA_CHECK(cudaEventRecord(P->ev_mlp, s2));   // (head_kernel's last-layer gradients precede everything on s2)
  // dW_ih = dG^T X, dW_hh = dG^T H (K = 9 * rows), fp16 operands. With grad_groups > 1 (data-parallel learner) the two
  // GEMMs run per group of experts and record an event per group: the group's LSTM gradients are one contiguous range
  // of the flat buffer (ppo_layout.h), which the caller all-reduces while the next group's GEMMs run.
  const int eg = E / P->grad_groups;
  for (int grp = 0; grp < P->grad_groups; ++grp) {
    const int e0 = grp * eg;
    for (int which = 0; which < 2; ++which) {
      GemmArgs g;
      g.kind = 0, g.a_mn = 1, g.b_mn = 1, g.batch = eg, g.out_f32 = 1, g.block_n = 128;
      g.a_bs = static_cast<long long>(cap) * 9 * LS_LDG16, g.b_bs = static_cast<long long>(cap) * 9 * LS_LDH16;
      g.A = P->dG16 + e0 * g.a_bs, g.lda = LS_LDG16;
      g.B = (which ? P->H16 : P->X16) + e0 * g.b_bs, g.ldb = LS_LDH16;
      g.M = G, g.N = F, g.K = 9 * cap;
      g.alpha = 1.f / P->bwd_scale;      // dG16 holds scale * dG
      g.out = grads + OFF_LSTM + e0 * LSTM_BLK + (which ? LSTM_WHH : LSTM_WIH), g.ldc = LDF, g.out_bs = LSTM_BLK;
      g.batch_rows = P->counts9 + e0, g.rows_is_k = 1;
      launch_gemm(g, s), ++n;
    }
    CADRE_CUDA_CHECK(cudaEventRecord(P->ev_grp[grp], s));
  }
  if (P->use_side) CADRE_CUDA_CHECK(cudaStreamWaitEvent(s, P->ev_join, 0));
  CADRE_CUDA_CHECK(cudaGetLastError());
  P->launches = n;
}

}  // namespace cadre

using cadre::PpoPlan;

#define CADRE_API_BEGIN try {
#define CADRE_API_END                \
  }                                  \
  catch (const cadre::Error& e) {    \
    cadre::set_last_error(e.what()); \
    return e.code;                   \
  }                                  \
  catch (const std::exception& e) {  \
    cadre::set_last_error(e.what()); \
    return 99;                       \
  }                                  \
  return 0;

extern "C" {

int64_t cadre_ppo_param_count(void) { return cadre::ppo::TOTAL; }

int cadre_ppo_create(void** handle, const cadre_ppo_config* cfg) {
  CADRE_API_BEGIN
  CADRE_REQUIRE(handle != nullptr, "handle");
  static_assert(sizeof(cadre_storage_ref) == sizeof(cadre::StorageRef), "storage ref layout");
  *handle = cadre::ppo_create(cfg);
  CADRE_API_END
}

int cadre_ppo_destroy(void* handle) {
  CADRE_API_BEGIN
  cadre::ppo_destroy(static_cast<PpoPlan*>(handle));
  CADRE_API_END
}

int cadre_ppo_stage(void* handle, const cadre_storage_ref* storages_host, const int32_t* indices_host, int n_steps,
                    int first_adam_step, void* stream) {
  CADRE_API_BEGIN
  CADRE_REQUIRE(handle && storages_host && indices_host && first_adam_step >= 0, "ppo_stage arguments");
  cadre::ppo_stage(static_cast<PpoPlan*>(handle), storages_host, indices_host, n_steps, first_adam_step,
                   static_cast<cudaStream_t>(stream));
  CADRE_API_END
}

int cadre_ppo_update(void* handle, const cadre_storage_ref* storages_host, const int32_t* indices_host,
                     float* params, float* grads, float* losses, void* stream) {
  CADRE_API_BEGIN
  PpoPlan* P = static_cast<PpoPlan*>(handle);
  CADRE_REQUIRE(P && params && grads && losses, "ppo_update pointers");
  CADRE_REQUIRE((storages_host != nullptr) == (indices_host != nullptr), "storages and indices go together");
  CADRE_REQUIRE(indices_host != nullptr || P->staged_steps > 0, "ppo_update without indices needs cadre_ppo_stage first");
  cadre::ppo_update(P, storages_host, indices_host, params, grads, losses, static_cast<cudaStream_t>(stream));
  CADRE_API_END
}

int cadre_ppo_evaluate(void* handle, const cadre_storage_ref* storages_host, const int32_t* indices_host,
                       const float* params, float* row_out, void* stream) {
  CADRE_API_BEGIN
  PpoPlan* P = static_cast<PpoPlan*>(handle);
  CADRE_REQUIRE(P && storages_host && indices_host && params && row_out, "ppo_evaluate pointers");
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  int n = cadre::ppo_forward(P, storages_host, indices_host, params, s);
  cadre::launch_k(cadre::head_eval_kernel, dim3((2 * P->R + 7) / 8), dim3(256), 0, s, P->Y2, params, P->row_slot, P->row_expert,
                                                             P->sc.action, P->R, P->cap, row_out);
  CADRE_CUDA_CHECK(cudaGetLastError());
  P->launches = n + 1;
  CADRE_API_END
}

int cadre_ppo_act(void* handle, const cadre_storage_ref* storages_host, const int32_t* indices_host,
                  const float* params, float* row_out, const cadre_rollout_pool* pool, int slot, uint64_t seed,
                  uint64_t tick, const int32_t* env_ids, const float* hidden_hn, const float* hidden_cn,
                  int64_t* actions_out, void* stream) {
  CADRE_API_BEGIN
  cadre::check_rollout_pool(pool, slot);
  PpoPlan* P = static_cast<PpoPlan*>(handle);
  CADRE_REQUIRE(P != nullptr, "ppo_act: ppo handle is NULL");
  CADRE_REQUIRE(storages_host && indices_host && params && row_out && env_ids && hidden_hn && hidden_cn && actions_out,
                "ppo_act pointers");
  CADRE_REQUIRE(pool->obs && pool->action && pool->action_log_probs && pool->value_preds && pool->command && pool->hn &&
                    pool->cn, "ppo_act: rollout pool pointers");
  const int E_env = P->cfg.mini_batch;
  CADRE_REQUIRE(P->cfg.workers == 1, "ppo_act needs an engine with workers = 1, mini_batch = E");
  CADRE_REQUIRE(pool->storages == 2 * E_env, "ppo_act: the pool must hold 2 storages per environment");
  CADRE_REQUIRE(pool->seq_length == 8 && pool->feature_dims == cadre::ppo::F && pool->hidden_size == cadre::ppo::F,
                "ppo_act: pool windows must be [8][530] with hidden size 530");
  for (int h = 0; h < 2; ++h)
    for (int i = 0; i < E_env; ++i)
      CADRE_REQUIRE(indices_host[h * E_env + i] == i, "ppo_act: indices must be 0..E-1 for both heads");
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  int n = cadre::ppo_forward(P, storages_host, indices_host, params, s);
  cadre::launch_k(cadre::head_eval_kernel, dim3((2 * P->R + 7) / 8), dim3(256), 0, s, P->Y2, params, P->row_slot,
                  P->row_expert, P->sc.action, P->R, P->cap, row_out);
  cadre::launch_k(cadre::act_write_kernel, dim3(E_env), dim3(256), 0, s, row_out, E_env, *pool, slot,
                  static_cast<unsigned long long>(seed), static_cast<unsigned long long>(tick), env_ids,
                  storages_host[0].obs, storages_host[0].command, hidden_hn, hidden_cn,
                  reinterpret_cast<long long*>(actions_out));
  CADRE_CUDA_CHECK(cudaGetLastError());
  P->launches = n + 2;
  CADRE_API_END
}

}  // extern "C"

namespace cadre {
static void check_ensemble_args(const float* row_out, int K, int greedy, const int32_t* env_ids,
                                const double* steer_table, const double* throttle_table, const double* controls_out,
                                const int64_t* actions_out) {
  CADRE_REQUIRE(K >= 1 && K <= ENSEMBLE_MAX_K, "ensemble: K must lie in [1, 64]");
  CADRE_REQUIRE(greedy == 0 || greedy == 1, "ensemble: greedy must be 0 or 1");
  CADRE_REQUIRE(row_out && env_ids && steer_table && throttle_table && controls_out && actions_out,
                "ensemble pointers");
}

static void launch_ensemble_control(const float* row_out, int K, int E_env, uint64_t seed, uint64_t tick,
                                    const int32_t* env_ids, int greedy, const double* steer_table,
                                    const double* throttle_table, double* controls_out, int64_t* actions_out,
                                    cudaStream_t s) {
  launch_k(ensemble_control_kernel, dim3((E_env + ENSEMBLE_WARPS - 1) / ENSEMBLE_WARPS), dim3(ENSEMBLE_WARPS * 32), 0,
           s, row_out, K, E_env, static_cast<unsigned long long>(seed), static_cast<unsigned long long>(tick), env_ids,
           greedy, steer_table, throttle_table, controls_out, reinterpret_cast<long long*>(actions_out));
  CADRE_CUDA_CHECK(cudaGetLastError());
}
}  // namespace cadre

extern "C" {

int cadre_ensemble_control(const float* row_out, int K, int E, uint64_t seed, uint64_t tick, const int32_t* env_ids,
                           int greedy, const double* steer_table, const double* throttle_table, double* controls_out,
                           int64_t* actions_out, void* stream) {
  CADRE_API_BEGIN
  cadre::check_ensemble_args(row_out, K, greedy, env_ids, steer_table, throttle_table, controls_out, actions_out);
  CADRE_REQUIRE(E >= 1, "ensemble: E must be at least 1");
  cadre::launch_ensemble_control(row_out, K, E, seed, tick, env_ids, greedy, steer_table, throttle_table, controls_out,
                                 actions_out, static_cast<cudaStream_t>(stream));
  CADRE_API_END
}

int cadre_ppo_ensemble_act(void* handle, const cadre_storage_ref* storages_host, const int32_t* indices_host,
                           const float* const* params_host, int K, float* row_out, uint64_t seed, uint64_t tick,
                           const int32_t* env_ids, int greedy, const double* steer_table, const double* throttle_table,
                           double* controls_out, int64_t* actions_out, void* stream) {
  CADRE_API_BEGIN
  cadre::check_ensemble_args(row_out, K, greedy, env_ids, steer_table, throttle_table, controls_out, actions_out);
  CADRE_REQUIRE(storages_host && indices_host && params_host, "ppo_ensemble_act pointers");
  for (int k = 0; k < K; ++k) CADRE_REQUIRE(params_host[k] != nullptr, "ppo_ensemble_act: params_host[k] is NULL");
  PpoPlan* P = static_cast<PpoPlan*>(handle);
  CADRE_REQUIRE(P != nullptr, "ppo_ensemble_act: ppo handle is NULL");
  const int E_env = P->cfg.mini_batch;
  CADRE_REQUIRE(P->cfg.workers == 1, "ppo_ensemble_act needs an engine with workers = 1, mini_batch = E");
  for (int h = 0; h < 2; ++h)
    for (int i = 0; i < E_env; ++i)
      CADRE_REQUIRE(indices_host[h * E_env + i] == i, "ppo_ensemble_act: indices must be 0..E-1 for both heads");
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  // One upload of the index table for all K forwards: K identical slices, each forward's prep_kernel advances to the
  // next, so the forwards need no host copy (and no wait on the pinned staging buffer) between snapshots.
  std::vector<int32_t> tab(static_cast<size_t>(K) * 2 * E_env);
  for (int k = 0; k < K; ++k) std::copy(indices_host, indices_host + 2 * E_env, tab.begin() + static_cast<size_t>(k) * 2 * E_env);
  cadre::ppo_stage(P, storages_host, tab.data(), K, P->host_step, s);
  int n = 0;
  for (int k = 0; k < K; ++k) {
    float* rows = row_out + static_cast<size_t>(k) * 2 * E_env * cadre::ROW_OUT;
    n = cadre::ppo_forward(P, nullptr, nullptr, params_host[k], s);
    cadre::launch_k(cadre::head_eval_kernel, dim3((2 * P->R + 7) / 8), dim3(256), 0, s, P->Y2, params_host[k],
                    P->row_slot, P->row_expert, P->sc.action, P->R, P->cap, rows);
  }
  CADRE_CUDA_CHECK(cudaGetLastError());
  cadre::launch_ensemble_control(row_out, K, E_env, seed, tick, env_ids, greedy, steer_table, throttle_table,
                                 controls_out, actions_out, s);
  P->launches = K * (n + 1) + 1;
  CADRE_API_END
}

int cadre_ppo_bootstrap(void* handle, const cadre_storage_ref* storages_host, const int32_t* indices_host,
                        const float* params, float* row_out, uint64_t done_mask, float* next_value, void* stream) {
  CADRE_API_BEGIN
  PpoPlan* P = static_cast<PpoPlan*>(handle);
  CADRE_REQUIRE(P != nullptr, "ppo_bootstrap: ppo handle is NULL");
  CADRE_REQUIRE(storages_host && indices_host && params && row_out && next_value, "ppo_bootstrap pointers");
  CADRE_REQUIRE(P->cfg.mini_batch == 1, "ppo_bootstrap needs an engine with mini_batch = 1");
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  int n = cadre::ppo_forward(P, storages_host, indices_host, params, s);
  cadre::launch_k(cadre::head_eval_kernel, dim3((2 * P->R + 7) / 8), dim3(256), 0, s, P->Y2, params, P->row_slot,
                  P->row_expert, P->sc.action, P->R, P->cap, row_out);
  cadre::launch_k(cadre::bootstrap_value_kernel, dim3((2 * P->R + 127) / 128), dim3(128), 0, s, row_out, P->R,
                  static_cast<unsigned long long>(done_mask), next_value);
  CADRE_CUDA_CHECK(cudaGetLastError());
  P->launches = n + 2;
  CADRE_API_END
}

int cadre_ppo_adam_step(void* handle, float* params, const float* grads, float* exp_avg, float* exp_avg_sq,
                        float max_grad_norm, float lr, float beta1, float beta2, float eps, int step,
                        void* stream) {
  CADRE_API_BEGIN
  PpoPlan* P = static_cast<PpoPlan*>(handle);
  CADRE_REQUIRE(P && params && grads && exp_avg && exp_avg_sq && step >= 0, "adam_step arguments");
  if (step >= 1) P->host_step = step + 1;   // the one-step update path restarts the device counter from here
  cadre::launch_clip_adam(P->opt, params, grads, exp_avg, exp_avg_sq, max_grad_norm, lr, beta1, beta2, eps, step,
                          static_cast<cudaStream_t>(stream), 0, 16, P->ctrs + 1, P->norms_out,
                          P->kl_sum && step == 0 ? P->kl_state : nullptr);
  CADRE_API_END
}

int cadre_ppo_module_norms(void* handle, float* norms16_host) {
  CADRE_API_BEGIN
  PpoPlan* P = static_cast<PpoPlan*>(handle);
  CADRE_REQUIRE(P && norms16_host, "module_norms arguments");
  CADRE_CUDA_CHECK(cudaMemcpy(norms16_host, P->opt.norms, 16 * sizeof(float), cudaMemcpyDeviceToHost));
  CADRE_API_END
}

int cadre_ppo_set_grad_groups(void* handle, int groups) {
  CADRE_API_BEGIN
  PpoPlan* P = static_cast<PpoPlan*>(handle);
  CADRE_REQUIRE(P != nullptr && (groups == 1 || groups == 2 || groups == 4 || groups == 8), "grad groups: 1, 2, 4 or 8");
  P->grad_groups = groups;
  CADRE_API_END
}

int cadre_ppo_grad_range(void* handle, int group, int64_t* offset, int64_t* count, int* mod_begin, int* mod_end) {
  CADRE_API_BEGIN
  PpoPlan* P = static_cast<PpoPlan*>(handle);
  CADRE_REQUIRE(P && offset && count && mod_begin && mod_end && group >= -1 && group < P->grad_groups, "grad range");
  using namespace cadre::ppo;
  if (group < 0) {   // the actor-critic tensors of all experts
    *offset = OFF_W1, *count = TOTAL - OFF_W1, *mod_begin = 8, *mod_end = 16;
  } else {
    const int eg = E / P->grad_groups;
    *offset = OFF_LSTM + static_cast<long long>(group) * eg * LSTM_BLK, *count = eg * LSTM_BLK;
    *mod_begin = group * eg, *mod_end = (group + 1) * eg;
  }
  CADRE_API_END
}

int cadre_ppo_wait_grads(void* handle, int group, void* stream) {
  CADRE_API_BEGIN
  PpoPlan* P = static_cast<PpoPlan*>(handle);
  CADRE_REQUIRE(P != nullptr && group >= -1 && group < P->grad_groups, "grad group");
  CADRE_CUDA_CHECK(cudaStreamWaitEvent(static_cast<cudaStream_t>(stream), group < 0 ? P->ev_mlp : P->ev_grp[group], 0));
  CADRE_API_END
}

int cadre_ppo_adam_step_modules(void* handle, float* params, const float* grads, float* exp_avg, float* exp_avg_sq,
                                float max_grad_norm, float lr, float beta1, float beta2, float eps, int step,
                                int mod_begin, int mod_end, void* stream) {
  CADRE_API_BEGIN
  PpoPlan* P = static_cast<PpoPlan*>(handle);
  CADRE_REQUIRE(P && params && grads && exp_avg && exp_avg_sq && step >= 0, "adam_step arguments");
  cadre::launch_clip_adam(P->opt, params, grads, exp_avg, exp_avg_sq, max_grad_norm, lr, beta1, beta2, eps, step,
                          static_cast<cudaStream_t>(stream), mod_begin, mod_end, P->ctrs + 1, P->norms_out,
                          P->kl_sum && step == 0 ? P->kl_state : nullptr);
  CADRE_API_END
}

int cadre_ppo_set_diagnostics(void* handle, float* diag_out, float* norms_out) {
  CADRE_API_BEGIN
  PpoPlan* P = static_cast<PpoPlan*>(handle);
  CADRE_REQUIRE(P != nullptr, "set_diagnostics: ppo handle is NULL");
  P->diag_out = diag_out;
  P->norms_out = norms_out;
  CADRE_API_END
}

int cadre_ppo_set_target_kl(void* handle, float target_kl, int total_workers, float* kl_sum_dev) {
  CADRE_API_BEGIN
  CADRE_REQUIRE(std::isfinite(target_kl) && target_kl >= 0.f, "set_target_kl: target_kl must be a finite value > 0 (0: off)");
  PpoPlan* P = static_cast<PpoPlan*>(handle);
  CADRE_REQUIRE(P != nullptr, "set_target_kl: ppo handle is NULL");
  if (target_kl == 0.f) {
    P->kl_sum = nullptr;
  } else {
    CADRE_REQUIRE(kl_sum_dev != nullptr, "set_target_kl: kl_sum_dev is NULL");
    CADRE_REQUIRE(total_workers >= P->cfg.workers, "set_target_kl: total_workers is below this engine's workers");
    P->kl_limit = static_cast<float>(1.5 * static_cast<double>(target_kl));
    P->kl_inv_total = 1.f / static_cast<float>(total_workers);
    P->kl_sum = kl_sum_dev;
  }
  CADRE_API_END
}

int cadre_ppo_kl_begin(void* handle, void* stream) {
  CADRE_API_BEGIN
  PpoPlan* P = static_cast<PpoPlan*>(handle);
  CADRE_REQUIRE(P != nullptr, "kl_begin: ppo handle is NULL");
  CADRE_CUDA_CHECK(cudaMemsetAsync(P->kl_state, 0, sizeof(int) * cadre::KS_WORDS, static_cast<cudaStream_t>(stream)));
  CADRE_API_END
}

int cadre_ppo_kl_gate(void* handle, void* stream) {
  CADRE_API_BEGIN
  PpoPlan* P = static_cast<PpoPlan*>(handle);
  CADRE_REQUIRE(P != nullptr, "kl_gate: ppo handle is NULL");
  CADRE_REQUIRE(P->kl_sum != nullptr, "kl_gate: target_kl is not set (cadre_ppo_set_target_kl)");
  cadre::launch_k(cadre::kl_gate_kernel, dim3(1), dim3(1), 0, static_cast<cudaStream_t>(stream), P->kl_sum,
                  P->kl_inv_total, P->kl_limit, P->kl_state, P->kl_hist, P->ctrs + 1);
  CADRE_CUDA_CHECK(cudaGetLastError());
  CADRE_API_END
}

int cadre_ppo_early_stop(void* handle, int32_t* state_host, float* kl_host, int kl_count, void* stream) {
  CADRE_API_BEGIN
  PpoPlan* P = static_cast<PpoPlan*>(handle);
  CADRE_REQUIRE(P != nullptr && state_host != nullptr, "early_stop: NULL handle or state_host");
  CADRE_REQUIRE(kl_count >= 0 && kl_count <= cadre::KL_HIST_CAP && (kl_count == 0 || kl_host != nullptr),
                "early_stop: kl_count must be in [0, 4096] with kl_host set when positive");
  // stream-ordered reads behind the phase's gates, then a wait on that stream only
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  int st[cadre::KS_WORDS], adam = 0;
  CADRE_CUDA_CHECK(cudaMemcpyAsync(st, P->kl_state, sizeof(st), cudaMemcpyDeviceToHost, s));
  CADRE_CUDA_CHECK(cudaMemcpyAsync(&adam, P->ctrs + 1, sizeof(int), cudaMemcpyDeviceToHost, s));
  if (kl_count > 0)
    CADRE_CUDA_CHECK(cudaMemcpyAsync(kl_host, P->kl_hist, sizeof(float) * kl_count, cudaMemcpyDeviceToHost, s));
  CADRE_CUDA_CHECK(cudaStreamSynchronize(s));
  state_host[0] = st[cadre::KS_STEP];
  state_host[1] = st[cadre::KS_RUN];
  state_host[2] = st[cadre::KS_APPLIED];
  state_host[3] = st[cadre::KS_STOPPED] ? st[cadre::KS_STOPPED_AT] : -1;
  state_host[4] = adam;
  CADRE_API_END
}

int cadre_ppo_check(void* handle) {
  CADRE_API_BEGIN
  PpoPlan* P = static_cast<PpoPlan*>(handle);
  CADRE_REQUIRE(P != nullptr, "ppo handle");
  unsigned flags[32];
  CADRE_CUDA_CHECK(cudaMemcpy(flags, P->seq_sync, sizeof(flags), cudaMemcpyDeviceToHost));
  if (flags[cadre::ppo::E] != 0 || flags[16 + cadre::ppo::E] != 0)
    throw cadre::Error(4, std::string("LSTM recurrence kernel: a cross-CTA hand-off timed out (") +
                              (flags[cadre::ppo::E] ? "forward" : "backward") + "); results of that update are invalid");
  CADRE_API_END
}

int cadre_ppo_launches(void* handle) {
  PpoPlan* P = static_cast<PpoPlan*>(handle);
  return P ? P->launches : 0;
}

}  // extern "C"

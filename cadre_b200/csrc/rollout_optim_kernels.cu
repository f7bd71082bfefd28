// HBM-bound kernels around the PPO update: GAE / returns scan + advantage normalisation, segmented gradient
// norm + fused clip + Adam over the flat parameter buffer.
#include "../../include/cadre_b200.h"
#include "internal.h"
#include "ptx.cuh"
#include "sampler.cuh"

namespace cadre {

// Standalone form of the act step's sampler (sampler.cuh): one thread per row.
__global__ void __launch_bounds__(128) categorical_sample_kernel(const float* __restrict__ logp, long long ld, int rows,
                                                                 int A, unsigned long long seed, unsigned long long tick,
                                                                 const int* __restrict__ env_ids, int word,
                                                                 long long* __restrict__ action_out,
                                                                 float* __restrict__ logp_out, float* __restrict__ u_out) {
  pdl_trigger();
  pdl_wait();
  const int r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= rows) return;
  const float u = philox_uniform(philox_word(philox_words(seed, tick, env_ids[r], 0u), word));
  const float* lp = logp + r * ld;
  const int a = categorical_draw(lp, A, u);
  action_out[r] = a;
  logp_out[r] = lp[a];
  if (u_out) u_out[r] = u;
}

// ---------------------------------------------------------------------------------------------------------
// RolloutStorage.compute_returns (ppo_agent/storage.py:68-76, GAE branch) + advantage normalisation
// (ppo_agent/train.py:82-88). One warp per (env, head) sequence; the reverse-time recurrence
//   A_t = delta_t + a_t * A_{t+1},   delta_t = r_t + g V_{t+1} m_t - V_t,   a_t = g*tau*m_t
// is an affine scan: each lane composes its chunk's affine map, the 32 maps are suffix-scanned with shuffles,
// then every lane replays its chunk. Global traffic is coalesced and streamed once: 12 B read + 8 B written
// per step (V is re-read from L2 for the output pass). Only (delta, a) are staged in shared memory -- 8 B per
// step and warp -- so that ~24 warps per SM keep enough loads in flight to stream HBM.
__device__ __forceinline__ int skew(int i) { return i + (i >> 5); }

// ITERS = ceil(T / 32) when T <= 32 * ITERS is known at launch (8: T <= 256, 32: T <= 1024): every global load
// of the sequence is issued before the first use (3 * ITERS independent loads per lane, ~12 KB per warp in
// flight) and V stays in registers for the output pass. ITERS = 0 is the general loop (V re-read from L2).
__device__ __forceinline__ void cp_async_4(float* smem_dst, const float* gmem_src) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(smem_u32(smem_dst)), "l"(gmem_src) : "memory");
}
__device__ __forceinline__ void cp_async_wait_all() {
  asm volatile("cp.async.commit_group;\n\tcp.async.wait_group 0;" ::: "memory");
}

template <int ITERS>
__global__ void __launch_bounds__(256, (ITERS > 16 ? 3 : 1)) gae_kernel(const float* __restrict__ rewards, float* __restrict__ values,
                                                  const float* __restrict__ masks,
                                                  const float* __restrict__ next_value,
                                                  float* __restrict__ returns, float* __restrict__ adv, int E,
                                                  int T, float gamma, float tau, int normalize) {
  pdl_trigger();
  pdl_wait();
  extern __shared__ float gsm[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int e = blockIdx.x * (blockDim.x >> 5) + warp;
  if (e >= E) return;
  const int L = skew(T) + 1;
  float* sd = gsm + warp * 2 * L;   // delta_t, later the raw advantage
  float* sa_ = sd + L;              // a_t
  const long long base = static_cast<long long>(e) * (T + 1);
  const float nv = next_value[e];
  const float gt = gamma * tau;
  constexpr int NV = ITERS > 0 ? ITERS : 1;
  float vreg[NV];
  if constexpr (ITERS > 16) {
    // r and m travel global -> shared with cp.async (no registers held while in flight) straight into the
    // arrays that become (delta, a); V goes to registers (it is needed again for the output pass). All 3*ITERS
    // loads of the sequence are in flight at once: one memory round trip per sequence, ~60 registers.
#pragma unroll
    for (int k = 0; k < ITERS; ++k) {
      const int i = lane + 32 * k;
      if (i < T) {
        cp_async_4(&sd[skew(i)], rewards + base + i);
        cp_async_4(&sa_[skew(i)], masks + base + i);
      }
      vreg[k] = i < T ? values[base + i] : 0.f;
    }
    cp_async_wait_all();
    __syncwarp();
#pragma unroll
    for (int k = 0; k < ITERS; ++k) {
      const int i = lane + 32 * k;
      // V_{i+1}: the next lane's element, lane 31 takes lane 0's next element, the last step takes next_value
      const float dn = __shfl_down_sync(0xffffffffu, vreg[k], 1);
      const float wrap = (k + 1 < ITERS) ? __shfl_sync(0xffffffffu, vreg[k + 1 < ITERS ? k + 1 : k], 0) : nv;
      float vn = lane < 31 ? dn : wrap;
      if (i + 1 == T) vn = nv;
      if (i < T) {
        const float r = sd[skew(i)], m = sa_[skew(i)];   // this lane's own elements: in-place update is safe
        sd[skew(i)] = r + gamma * vn * m - vreg[k];
        sa_[skew(i)] = gt * m;
      }
    }
  } else if constexpr (ITERS > 0) {
    // short sequences: plain register loads (many warps per SM hide the single round trip)
    float rreg[ITERS], mreg[ITERS];
#pragma unroll
    for (int k = 0; k < ITERS; ++k) {
      const int i = lane + 32 * k;
      const bool ok = i < T;
      rreg[k] = ok ? rewards[base + i] : 0.f;
      vreg[k] = ok ? values[base + i] : 0.f;
      mreg[k] = ok ? masks[base + i] : 0.f;
    }
#pragma unroll
    for (int k = 0; k < ITERS; ++k) {
      const int i = lane + 32 * k;
      const float dn = __shfl_down_sync(0xffffffffu, vreg[k], 1);
      const float wrap = (k + 1 < ITERS) ? __shfl_sync(0xffffffffu, vreg[k + 1 < ITERS ? k + 1 : k], 0) : nv;
      float vn = lane < 31 ? dn : wrap;
      if (i + 1 == T) vn = nv;
      if (i < T) {
        sd[skew(i)] = rreg[k] + gamma * vn * mreg[k] - vreg[k];
        sa_[skew(i)] = gt * mreg[k];
      }
    }
  } else {
#pragma unroll 4
    for (int i = lane; i < T; i += 32) {
      const float r = rewards[base + i], v = values[base + i], m = masks[base + i];
      const float vn = (i + 1 == T) ? nv : values[base + i + 1];   // neighbouring lane's line: L1 hit
      sd[skew(i)] = r + gamma * vn * m - v;
      sa_[skew(i)] = gt * m;
    }
  }
  if (lane == 0) values[base + T] = nv;  // storage.py:70 value_preds[-1] = next_value
  __syncwarp();
  const int cs = (T + 31) / 32;
  const int t0 = min(T, lane * cs), t1 = min(T, t0 + cs);
  {
  // chunk map x -> a*x + b (x = gae entering the chunk from later time steps)
  // (unrolled by 8: the shared-memory loads of eight steps are issued ahead of the dependent FMA chain)
  float a = 1.f, b = 0.f;
#pragma unroll 8
  for (int t = t1 - 1; t >= t0; --t) {
    const float at = sa_[skew(t)];
    b = at * b + sd[skew(t)];   // F_t o F_chunk_so_far : later steps were composed first
    a = at * a;
  }
  // inclusive suffix composition S_l = F_l o F_{l+1} o ... o F_31
  float sa = a, sb = b;
#pragma unroll
  for (int off = 1; off < 32; off <<= 1) {
    const float oa = __shfl_down_sync(0xffffffffu, sa, off);
    const float ob = __shfl_down_sync(0xffffffffu, sb, off);
    if (lane + off < 32) {
      sb = sa * ob + sb;
      sa = sa * oa;
    }
  }
  float gae = __shfl_down_sync(0xffffffffu, sb, 1);  // S_{l+1}(0)
  if (lane == 31) gae = 0.f;
#pragma unroll 8
  for (int t = t1 - 1; t >= t0; --t) {   // replay the chunk
    gae = sd[skew(t)] + sa_[skew(t)] * gae;
    sd[skew(t)] = gae;
  }
  }
  __syncwarp();
  // returns_t = gae_t + V_t (storage.py:75); advantage_t = returns_t - V_t (train.py:82: the rounding of the
  // round trip through returns is kept); coalesced, V from L2
  float lsum = 0.f;
  if constexpr (ITERS > 0) {
#pragma unroll
    for (int k = 0; k < ITERS; ++k) {
      const int i = lane + 32 * k;
      if (i < T) {
        const float v = vreg[k];
        const float ret = sd[skew(i)] + v;
        const float ad = ret - v;
        returns[base + i] = ret;
        sd[skew(i)] = ad;
        lsum += ad;
      }
    }
  } else {
#pragma unroll 4
    for (int i = lane; i < T; i += 32) {
      const float v = values[base + i];
      const float ret = sd[skew(i)] + v;
      const float ad = ret - v;
      returns[base + i] = ret;
      sd[skew(i)] = ad;
      lsum += ad;
    }
  }
  float mean = 0.f, denom = 1.f;
  if (normalize) {
    for (int o = 16; o > 0; o >>= 1) lsum += __shfl_xor_sync(0xffffffffu, lsum, o);
    mean = lsum / static_cast<float>(T);
    float lsq = 0.f;
    for (int i = lane; i < T; i += 32) {
      const float d = sd[skew(i)] - mean;
      lsq += d * d;
    }
    for (int o = 16; o > 0; o >>= 1) lsq += __shfl_xor_sync(0xffffffffu, lsq, o);
    denom = sqrtf(lsq / static_cast<float>(T - 1)) + 1e-8f;  // torch.std is unbiased; train.py:86
  }
#pragma unroll 4
  for (int i = lane; i < T; i += 32) {
    const float ad = sd[skew(i)];
    adv[static_cast<long long>(e) * T + i] = normalize ? (ad - mean) / denom : ad;
  }
}

// ---------------------------------------------------------------------------------------------------------
// chief.py:13-21: per-module clip_grad_norm_(max_norm) on the summed gradient, then one Adam step
// (torch.optim.Adam defaults, main.py:55). The flat buffers are cut into fixed chunks; every chunk belongs to
// exactly one of the 16 modules. Pass 1 writes one partial sum of squares per chunk (deterministic), pass 2
// (one warp per module) reduces them in a fixed order, pass 3 applies clip + Adam elementwise.

__global__ void __launch_bounds__(256) sqnorm_partial_kernel(const float* __restrict__ g,
                                                             const long long* __restrict__ chunk_off,
                                                             const int* __restrict__ chunk_len,
                                                             float* __restrict__ partial,
                                                             const int* __restrict__ skip) {
  pdl_trigger();
  pdl_wait();
  if (skip && *skip) return;
  const long long off = chunk_off[blockIdx.x];
  const int len = chunk_len[blockIdx.x];
  const float4* g4 = reinterpret_cast<const float4*>(g + off);
  float s = 0.f;
  for (int i = threadIdx.x; i < (len >> 2); i += 256) {
    const float4 v = g4[i];
    s += v.x * v.x + v.y * v.y + v.z * v.z + v.w * v.w;
  }
  __shared__ float sm[8];
  for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  if ((threadIdx.x & 31) == 0) sm[threadIdx.x >> 5] = s;
  __syncthreads();
  if (threadIdx.x == 0) {
    float t = 0.f;
    for (int i = 0; i < 8; ++i) t += sm[i];
    partial[blockIdx.x] = t;
  }
}

__global__ void sqnorm_final_kernel(const float* __restrict__ partial, const int* __restrict__ mod_first,
                                    float max_norm, float* __restrict__ clip_coef, float* __restrict__ norms,
                                    int mod_begin, int step, const int* __restrict__ dev_step, float lr, float beta1,
                                    float beta2, float* __restrict__ scalars, float* __restrict__ norms_hist,
                                    const int* __restrict__ skip) {
  pdl_trigger();
  pdl_wait();
  if (skip && *skip) return;
  // one warp per module; chunks of a module are contiguous in the chunk table
  const int m = mod_begin + blockIdx.x, lane = threadIdx.x;
  if (blockIdx.x == 0 && lane == 0) {
    // torch.optim.Adam: step_size = lr / (1 - beta1^step); denom = sqrt(v) / sqrt(1 - beta2^step) + eps. The step
    // comes from the host (step >= 1) or from the device counter the update kernels advance (step = 0: CUDA graphs)
    const int st = step >= 1 ? step : *dev_step;
    const double bc1 = 1.0 - pow(static_cast<double>(beta1), static_cast<double>(st));
    const double bc2 = 1.0 - pow(static_cast<double>(beta2), static_cast<double>(st));
    scalars[0] = static_cast<float>(static_cast<double>(lr) / bc1);
    scalars[1] = static_cast<float>(sqrt(bc2));
  }
  double s = 0.0;
  for (int i = mod_first[m] + lane; i < mod_first[m + 1]; i += 32) s += static_cast<double>(partial[i]);
  for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  if (lane == 0) {
    const float total = static_cast<float>(sqrt(s));
    norms[m] = total;
    if (norms_hist) norms_hist[m] = total;   // per-step history slot (cadre_ppo_set_diagnostics)
    clip_coef[m] = fminf(max_norm / (total + 1e-6f), 1.0f);  // torch.nn.utils.clip_grad_norm_
  }
}

__global__ void __launch_bounds__(256) adam_kernel(float* __restrict__ p, const float* __restrict__ g,
                                                   float* __restrict__ m, float* __restrict__ v,
                                                   const long long* __restrict__ chunk_off,
                                                   const int* __restrict__ chunk_len,
                                                   const int* __restrict__ chunk_mod,
                                                   const float* __restrict__ clip_coef, float beta1,
                                                   float beta2, float eps, const float* __restrict__ scalars,
                                                   const int* __restrict__ skip) {
  pdl_trigger();
  pdl_wait();
  if (skip && *skip) return;
  const float step_size = scalars[0], bc2_sqrt = scalars[1];
  const long long off = chunk_off[blockIdx.x];
  const int len = chunk_len[blockIdx.x];
  const float coef = clip_coef[chunk_mod[blockIdx.x]];
  float4* p4 = reinterpret_cast<float4*>(p + off);
  const float4* g4 = reinterpret_cast<const float4*>(g + off);
  float4* m4 = reinterpret_cast<float4*>(m + off);
  float4* v4 = reinterpret_cast<float4*>(v + off);
  for (int i = threadIdx.x; i < (len >> 2); i += 256) {
    float4 pp = p4[i], gg = g4[i], mm = m4[i], vv = v4[i];
    float* pe = &pp.x;
    float* ge = &gg.x;
    float* me = &mm.x;
    float* ve = &vv.x;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const float gr = ge[k] * coef;
      me[k] = me[k] + (gr - me[k]) * (1.f - beta1);          // exp_avg.lerp_(grad, 1 - beta1)
      ve[k] = ve[k] * beta2 + (1.f - beta2) * gr * gr;       // mul_(beta2).addcmul_(grad, grad, 1 - beta2)
      const float denom = sqrtf(ve[k]) / bc2_sqrt + eps;
      pe[k] = pe[k] - step_size * (me[k] / denom);           // addcdiv_(exp_avg, denom, value=-step_size)
    }
    p4[i] = pp, m4[i] = mm, v4[i] = vv;
  }
}

void launch_clip_adam(const OptTables& t, float* params, const float* grads, float* m, float* v, float max_norm,
                      float lr, float beta1, float beta2, float eps, int step, cudaStream_t s, int mod_begin,
                      int mod_end, const int* dev_step, float* norms_hist, const int* gate) {
  CADRE_REQUIRE(mod_begin >= 0 && mod_begin < mod_end && mod_end <= 16, "module range");
  CADRE_REQUIRE(step >= 1 || dev_step != nullptr, "Adam step");
  // chunks of modules [mod_begin, mod_end) are contiguous in the chunk table (it is sorted by module)
  const int c0 = t.mod_first_h[mod_begin], nc = t.mod_first_h[mod_end] - c0;
  if (nc <= 0) return;
  // gate: the target-KL state words (ppo.cu, kl_gate_kernel): [0] the phase stopped before this step (no norms either),
  // [1] the phase is stopped (no Adam update)
  const int* skip_norm = gate;
  const int* skip_adam = gate ? gate + 1 : nullptr;
  launch_k(sqnorm_partial_kernel, dim3(nc), dim3(256), 0, s, grads, t.chunk_off + c0, t.chunk_len + c0, t.partial + c0,
           skip_norm);
  launch_k(sqnorm_final_kernel, dim3(mod_end - mod_begin), dim3(32), 0, s, t.partial, t.mod_first, max_norm, t.clip_coef,
           t.norms, mod_begin, step, dev_step, lr, beta1, beta2, t.scalars, norms_hist, skip_norm);
  launch_k(adam_kernel, dim3(nc), dim3(256), 0, s, params, grads, m, v, t.chunk_off + c0, t.chunk_len + c0, t.chunk_mod + c0,
           t.clip_coef, beta1, beta2, eps, t.scalars, skip_adam);
  CADRE_CUDA_CHECK(cudaGetLastError());
}

// ---------------------------------------------------------------------------------------------------------
// Rollout statistics after compute_returns, one warp per (env, head) sequence of T steps, in fp64 with population
// variances: out[e] = [explained variance 1 - Var(R - V) / Var(R) (NaN when Var(R) = 0, as SB3's explained_variance),
// mean and std of the raw advantage R - V, mean and std of R, mean of V]. Two passes (means, then centred sums); the
// second re-reads the sequence from L1 / L2. Lane partial sums are combined with a fixed butterfly: deterministic.
constexpr int ROLLOUT_STATS = 6;
__device__ __forceinline__ double warp_sum_f64(double s) {
  for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  return s;
}
__global__ void __launch_bounds__(256) rollout_stats_kernel(const float* __restrict__ returns,
                                                            const float* __restrict__ values, int E, int T,
                                                            float* __restrict__ out) {
  pdl_trigger();
  pdl_wait();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int e = blockIdx.x * (blockDim.x >> 5) + warp;
  if (e >= E) return;
  const float* r = returns + static_cast<long long>(e) * (T + 1);
  const float* v = values + static_cast<long long>(e) * (T + 1);
  double sr = 0.0, sv = 0.0;
  for (int i = lane; i < T; i += 32) {
    sr += static_cast<double>(r[i]);
    sv += static_cast<double>(v[i]);
  }
  const double n = static_cast<double>(T);
  const double mr = warp_sum_f64(sr) / n, mv = warp_sum_f64(sv) / n, ma = mr - mv;
  double qr = 0.0, qa = 0.0;
  for (int i = lane; i < T; i += 32) {
    const double rr = static_cast<double>(r[i]);
    const double dr = rr - mr, da = (rr - static_cast<double>(v[i])) - ma;
    qr += dr * dr;
    qa += da * da;
  }
  const double var_r = warp_sum_f64(qr) / n, var_a = warp_sum_f64(qa) / n;
  if (lane == 0) {
    float* o = out + static_cast<long long>(e) * ROLLOUT_STATS;
    o[0] = var_r == 0.0 ? __int_as_float(0x7fc00000) : static_cast<float>(1.0 - var_a / var_r);
    o[1] = static_cast<float>(ma);
    o[2] = static_cast<float>(sqrt(var_a));
    o[3] = static_cast<float>(mr);
    o[4] = static_cast<float>(sqrt(var_r));
    o[5] = static_cast<float>(mv);
  }
}

}  // namespace cadre

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

namespace cadre {
// ---------------------------------------------------------------------------------------------------------
// Sliding-window assembly of rollout observations. The env wrapper hands every tick the last `seq` frames
// (env_wrapper.py:900-914) and train.py:69-72 stores that [seq, F] feature window as obs[t] of BOTH heads'
// storages. The frozen encoder maps frames independently, so with the features U[w][k] of the T + seq - 1 UNIQUE
// frames of a worker's rollout, obs[w][head][t][j] = U[w][t + j]: a pure gather. One warp copies one feature row
// (float2, 265 per row) into its up to `seq` x 2 destinations: U is read once, obs written once.
__global__ void __launch_bounds__(256) window_scatter_kernel(const float* __restrict__ U, float* __restrict__ obs,
                                                             int W, int T, int seq, int F, long long obs_head_stride,
                                                             long long obs_step_stride) {
  pdl_trigger();
  pdl_wait();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int K = T + seq - 1;
  const long long row = static_cast<long long>(blockIdx.x) * 8 + warp;   // (worker, unique frame k)
  if (row >= static_cast<long long>(W) * K) return;
  const int w = static_cast<int>(row / K), k = static_cast<int>(row - static_cast<long long>(w) * K);
  const float2* src = reinterpret_cast<const float2*>(U + row * F);
  const int F2 = F >> 1;
  for (int c = lane; c < F2; c += 32) {
    const float2 v = src[c];
    // frame k is element j of the window of step t = k - j
    for (int j = 0; j < seq; ++j) {
      const int t = k - j;
      if (t < 0 || t >= T) continue;
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        float* dst = obs + (static_cast<long long>(w) * 2 + h) * obs_head_stride + t * obs_step_stride +
                     static_cast<long long>(j) * F;
        reinterpret_cast<float2*>(dst)[c] = v;
      }
    }
  }
}
}  // namespace cadre

extern "C" {

int cadre_gae(const float* rewards, float* values, const float* masks, const float* next_value, float* returns,
              float* adv, int E, int T, float gamma, float tau, int normalize, void* stream) {
  CADRE_API_BEGIN
  CADRE_REQUIRE(rewards && values && masks && next_value && returns && adv, "gae pointers");
  CADRE_REQUIRE(E > 0 && T > 1 && T <= 16384, "gae sizes (1 < T <= 16384)");
  const int L = T + (T >> 5) + 1;
  const size_t per_warp = 2 * static_cast<size_t>(L) * sizeof(float);
  int warps = 8;
  while (warps > 1 && warps * per_warp > 72 * 1024) warps >>= 1;
  // Warps are independent (no block-level barrier) and a block's shared memory is only released when its LAST warp is
  // done, so long sequences run in blocks of two warps: the ~26 warps an SM holds then retire and get replaced one
  // pair at a time and their load / scan / store phases stay staggered (65 536 x 1 024 sweep on B200: 4.18 TB/s with
  // 8-warp blocks, 4.56 TB/s = 71 % of the measured copy peak with 2-warp blocks).
  if (T > 256) warps = warps > 2 ? 2 : warps;
  const size_t smem = warps * per_warp;
  // (a 16-loads-per-lane instance for T <= 512 measured slower than the cp.async path: 3.07 against 4.00 TB/s)
  auto kern = T <= 256 ? cadre::gae_kernel<8> : (T <= 1024 ? cadre::gae_kernel<32> : cadre::gae_kernel<0>);
  static size_t configured[3][cadre::CADRE_MAX_DEVICES] = {};   // per kernel variant and device
  const int which = T <= 256 ? 0 : (T <= 1024 ? 1 : 2);
  if (smem > 48 * 1024) cadre::ensure_dynamic_smem(kern, smem, configured[which]);
  cadre::launch_k(kern, dim3((E + warps - 1) / warps), dim3(warps * 32), smem, static_cast<cudaStream_t>(stream),
                  rewards, values, masks, next_value, returns, adv, E, T, gamma, tau, normalize);
  CADRE_CUDA_CHECK(cudaGetLastError());
  CADRE_API_END
}

int cadre_rollout_stats(const float* returns, const float* values, int E, int T, float* out, void* stream) {
  CADRE_API_BEGIN
  CADRE_REQUIRE(returns && values && out, "rollout_stats pointers");
  CADRE_REQUIRE(E > 0 && T > 0, "rollout_stats sizes (E > 0, T > 0)");
  cadre::launch_k(cadre::rollout_stats_kernel, dim3((E + 7) / 8), dim3(256), 0, static_cast<cudaStream_t>(stream),
                  returns, values, E, T, out);
  CADRE_CUDA_CHECK(cudaGetLastError());
  CADRE_API_END
}

int cadre_window_scatter(const float* unique_feats, float* obs, int workers, int num_steps, int seq_length,
                         int feature_dims, int64_t obs_head_stride, int64_t obs_step_stride, void* stream) {
  CADRE_API_BEGIN
  CADRE_REQUIRE(unique_feats && obs && workers > 0 && num_steps > 0 && seq_length > 0, "window_scatter arguments");
  CADRE_REQUIRE(feature_dims % 2 == 0 && obs_step_stride % 2 == 0 && obs_head_stride % 2 == 0,
                "window_scatter: feature_dims and strides must be even (float2 copies)");
  const long long rows = static_cast<long long>(workers) * (num_steps + seq_length - 1);
  cadre::launch_k(cadre::window_scatter_kernel, dim3(static_cast<unsigned>((rows + 7) / 8)), dim3(256), 0,
                  static_cast<cudaStream_t>(stream), unique_feats, obs, workers, num_steps, seq_length, feature_dims,
                  static_cast<long long>(obs_head_stride), static_cast<long long>(obs_step_stride));
  CADRE_CUDA_CHECK(cudaGetLastError());
  CADRE_API_END
}

int cadre_categorical_sample(const float* logp, int ld, int rows, int A, uint64_t seed, uint64_t tick,
                             const int32_t* env_ids, int word, int64_t* action_out, float* logp_out, float* u_out,
                             void* stream) {
  CADRE_API_BEGIN
  CADRE_REQUIRE(A >= 1 && A <= 33, "categorical_sample: A must lie in [1, 33]");
  CADRE_REQUIRE(rows > 0, "categorical_sample: rows must be positive");
  CADRE_REQUIRE(ld >= A, "categorical_sample: ld must be at least A");
  CADRE_REQUIRE(word >= 0 && word <= 3, "categorical_sample: word must lie in [0, 3]");
  CADRE_REQUIRE(logp && env_ids && action_out && logp_out, "categorical_sample pointers");
  cadre::launch_k(cadre::categorical_sample_kernel, dim3((rows + 127) / 128), dim3(128), 0,
                  static_cast<cudaStream_t>(stream), logp, static_cast<long long>(ld), rows, A,
                  static_cast<unsigned long long>(seed), static_cast<unsigned long long>(tick), env_ids, word,
                  reinterpret_cast<long long*>(action_out), logp_out, u_out);
  CADRE_CUDA_CHECK(cudaGetLastError());
  CADRE_API_END
}

int cadre_rollout_env_results(const cadre_rollout_pool* pool, int slot, const float* rewards_host,
                              const float* masks_host, void* stream) {
  CADRE_API_BEGIN
  cadre::check_rollout_pool(pool, slot);
  CADRE_REQUIRE(pool->rewards && pool->masks && rewards_host && masks_host, "rollout_env_results pointers");
  // one element per storage into the column [n][slot]: destination pitch = one storage's T + 1 floats
  const size_t pitch = sizeof(float) * (static_cast<size_t>(pool->num_steps) + 1);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  CADRE_CUDA_CHECK(cudaMemcpy2DAsync(pool->rewards + slot, pitch, rewards_host, sizeof(float), sizeof(float),
                                     pool->storages, cudaMemcpyHostToDevice, s));
  CADRE_CUDA_CHECK(cudaMemcpy2DAsync(pool->masks + slot, pitch, masks_host, sizeof(float), sizeof(float),
                                     pool->storages, cudaMemcpyHostToDevice, s));
  CADRE_API_END
}

}  // extern "C"

// Counter-based categorical sampler of the device-side rollout path (cadre_categorical_sample, cadre_ppo_act).
// Replaces the host-side Categorical(probs=softmax(logits)).sample() of distributions.py:96-99 / agent.py:124-131.
//
// A draw is a pure function of (seed, env id, tick, head, log-probs); the library keeps no RNG state, so an
// environment draws the same actions whichever batch, actor or rank it is stepped in:
//   x = Philox4x32-10(counter = (tick lo, tick hi, env id, k), key = (seed lo, seed hi)), word 0 = steer, 1 = throttle;
//   k = 0 on the rollout path; an ensemble (cadre_ppo_ensemble_act) keys snapshot k's draws with its index k, so its
//   snapshot 0 draws exactly what the rollout path would draw for the same (seed, env id, tick);
//   u = (x >> 8) * 2^-24 (24 bits, exact in fp32, u in [0, 1));
//   p_j = expf(lp_j), c_j = p_0 + ... + p_j summed in index order, j < A (columns >= A are never read);
//   a = min{ j : c_j > u * c_{A-1} }, or, if rounding leaves none, max{ j : p_j > 0 } (0 if every p_j is 0).
// An action with p_j == 0 is never drawn: its c_j equals c_{j-1} exactly, so an earlier index already qualifies.
#pragma once
#include <curand_philox4x32_x.h>

namespace cadre {

__device__ __forceinline__ uint4 philox_words(unsigned long long seed, unsigned long long tick, int env_id,
                                              unsigned k) {
  const uint4 ctr = make_uint4(static_cast<unsigned>(tick), static_cast<unsigned>(tick >> 32),
                               static_cast<unsigned>(env_id), k);
  const uint2 key = make_uint2(static_cast<unsigned>(seed), static_cast<unsigned>(seed >> 32));
  return curand_Philox4x32_10(ctr, key);
}

__device__ __forceinline__ unsigned philox_word(const uint4& x, int word) {
  return word == 0 ? x.x : (word == 1 ? x.y : (word == 2 ? x.z : x.w));
}

__device__ __forceinline__ float philox_uniform(unsigned x) { return static_cast<float>(x >> 8) * 0x1p-24f; }

// lp: A log-probabilities (the normalised logits of a head_eval_kernel row); returns the drawn index
__device__ __forceinline__ int categorical_draw(const float* lp, int A, float u) {
  float total = 0.f;
  for (int j = 0; j < A; ++j) total += expf(lp[j]);
  const float t = u * total;
  float c = 0.f;
  int last = 0;
  for (int j = 0; j < A; ++j) {   // the same sums in the same order as `total`
    const float p = expf(lp[j]);
    c += p;
    if (c > t) return j;
    if (p > 0.f) last = j;
  }
  return last;
}

// host-side argument check of a cadre_rollout_pool and a cursor (include internal.h first)
inline void check_rollout_pool(const cadre_rollout_pool* p, int slot) {
  CADRE_REQUIRE(p != nullptr, "rollout pool struct is NULL");
  CADRE_REQUIRE(p->storages > 0 && p->num_steps > 0 && p->seq_length > 0 && p->feature_dims > 0 && p->hidden_size > 0,
                "rollout pool sizes");
  CADRE_REQUIRE(slot >= 0 && slot <= p->num_steps, "rollout slot must lie in [0, num_steps]");
}

}  // namespace cadre

// tcgen05 / TMEM / TMA tile kernel shared by every dense contraction on the CADRE learner path:
//   * MODE_GEMM  plain (optionally grid.z-batched) GEMM  D[M,N] = A[M,K] * B[N,K]^T  with either operand
//                K-major or MN-major in global memory (covers fwd, dgrad and wgrad without transposes);
//   * MODE_CONV  implicit-GEMM convolution over NHWC activations: one TMA box per filter tap, padding by
//                TMA out-of-bounds zero fill, stride 2 through parity sub-lattice tensor maps;
//   * MODE_STEM  the 7x7/s2 Cin=4 stem through an overlapping-stride 5-D tensor map.
// One CTA = one 128 x BLOCK_N output tile. Warp 0 lane 0 issues TMA, warp 1 lane 0 issues tcgen05.mma into a
// TMEM accumulator, warps 2..5 drain TMEM (tcgen05.ld) and run the fused epilogue.
#pragma once
#include "internal.h"
#include "ptx.cuh"

namespace cadre {

enum { MODE_GEMM = 0, MODE_CONV = 1, MODE_STEM = 2 };
enum { EPI_LINEAR = 0 };
enum { ACT_NONE = 0, ACT_RELU = 1, ACT_LEAKY = 2 };

struct ConvTap {
  short map, dw, dh, pad_;
};

struct TcGemmParams {
  CUtensorMap tmA[4];
  CUtensorMap tmB;
  int M, N, num_kb;
  // conv geometry (output map); TW == Wout
  int ntaps, cin_chunks, Hout, Wout, TH, TN, Bimg;
  ConvTap taps[12];
  // epilogue
  void* out;
  long long ldc, out_bs;
  const float* bias;
  long long bias_bs;
  const void* res;  // same dtype as out
  long long ldr, res_bs;
  int res_after_act;
  const void* mask;  // same dtype as out; output zeroed where mask <= 0 (ReLU backward)
  long long ldm, mask_bs;
  int act;
  float alpha;
  int ksplit;             // >1: blockIdx.z = batch*ksplit + ks; split ks accumulates k-blocks [ks*kb_per_split, ...)
  int kb_per_split;       //     into out + ks*split_out_stride (the consumer sums the partials)
  long long split_out_stride;
  int dbg_epi;  // experiment: 1 = skip global stores, 2 = skip phase 2, 3 = skip tmem loads
  long long* dbg_clk;  // optional [gridDim.x*y*z][8] clock64 stamps (profiling experiment)
  int dbg_a_shift, dbg_base_offset;  // experiment: A descriptor start shifted by rows (128 B each)
  const int* batch_rows;  // optional [gridDim.z]: valid rows (M) per batch, or valid K when rows_is_k
  int rows_is_k;
  // optional compacted work list (device): tile_list[0] = n, then n pairs (batch, m_tile). blockIdx.x indexes the
  // list (grid.z = 1): no CTA is launched for the unused part of a batch's row capacity
  const int* tile_list;
};

template <int KIND, int BLOCK_N, int STAGES>
struct TcGemmSmem {
  static constexpr int A_BYTES = 128 * 128;
  static constexpr int B_BYTES = BLOCK_N * 128;
  static constexpr int STAGE_BYTES = A_BYTES + B_BYTES;
  static constexpr int EPI_BYTES = 128 * (BLOCK_N + 4) * 4;  // fp32 staging tile of the coalesced epilogue
  // The staging tile ALIASES the operand stages: one tile per CTA, and the epilogue starts after tmem_full, i.e.
  // after every MMA has read its operands. That leaves room for two CTAs per SM (3 x 32 KB TF32 stages), so one
  // CTA's prologue / epilogue overlaps the other's main loop.
  static constexpr int DATA_BYTES = STAGES * STAGE_BYTES > EPI_BYTES ? STAGES * STAGE_BYTES : EPI_BYTES;
  static constexpr int TOTAL = DATA_BYTES + (2 * STAGES + 1) * 8 + 16 + 1024;
};

template <typename OutT>
__device__ __forceinline__ float load_as_float(const void* base, long long idx) {
  if constexpr (sizeof(OutT) == 2)
    return enc_to_float(reinterpret_cast<const enc_t*>(base)[idx]);
  else
    return reinterpret_cast<const float*>(base)[idx];
}

// EW = epilogue warps per TMEM lane quarter (1: 192 threads; 2: 320 threads, the two warps of a quarter split the
// columns while draining TMEM and the rows afterwards: used where the epilogue is long, i.e. the LSTM cell)
template <int KIND, int A_MN, int B_MN, int BLOCK_N, int STAGES, int MODE, int EPI, typename OutT, int EW = 1>
__global__ void __launch_bounds__(64 + 128 * EW) tc_gemm_kernel(const __grid_constant__ TcGemmParams p) {
  constexpr int ES = KIND ? 4 : 2;         // operand element bytes
  constexpr int BK = 128 / ES;             // K elements per stage (one 128-byte swizzle row)
  constexpr int CHUNK = 128 / ES;          // MN elements per 128-byte row of an MN-major operand
  constexpr int UMMA_K = 32 / ES;          // K per tcgen05.mma
  using S = TcGemmSmem<KIND, BLOCK_N, STAGES>;
  static_assert(BLOCK_N >= 32 && BLOCK_N <= 256 && (BLOCK_N & (BLOCK_N - 1)) == 0, "BLOCK_N");

  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);  // keeps the shared address space
  uint64_t* full = reinterpret_cast<uint64_t*>(smem + S::DATA_BYTES);
  uint64_t* empty = full + STAGES;
  uint64_t* tmem_full = empty + STAGES;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tmem_full + 1);

  pdl_trigger();
  pdl_wait();   // batch_rows / bias below may have been written by the previous launch (route kernel, Adam)
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  int m_tile = blockIdx.x;
  const int n_tile = blockIdx.y;
  const int ks = p.ksplit > 1 ? static_cast<int>(blockIdx.z) % p.ksplit : 0;
  int batch = p.ksplit > 1 ? static_cast<int>(blockIdx.z) / p.ksplit : static_cast<int>(blockIdx.z);
  if (p.tile_list != nullptr) {   // written by an earlier launch: read after pdl_wait (above)
    if (static_cast<int>(blockIdx.x) >= p.tile_list[0]) return;   // uniform for the whole CTA, before any barrier
    batch = p.tile_list[1 + 2 * blockIdx.x];
    m_tile = p.tile_list[2 + 2 * blockIdx.x];
  }
  const int n0 = n_tile * BLOCK_N;
  long long* clk = p.dbg_clk ? p.dbg_clk + ((static_cast<long long>(blockIdx.z) * gridDim.y + blockIdx.y) * gridDim.x + blockIdx.x) * 8 : nullptr;
  if (clk && threadIdx.x == 0) clk[0] = clock64();

  int m_valid = p.M;
  int num_kb = p.num_kb;
  const int kb0 = ks * p.kb_per_split;  // first k-block of this split (0 without split-K)
  if (p.ksplit > 1) num_kb = max(0, min(p.kb_per_split, p.num_kb - kb0));
  if (p.batch_rows != nullptr) {
    const int cnt = p.batch_rows[batch];
    if (p.rows_is_k) {
      num_kb = (cnt + BK - 1) / BK;  // operands are zero padded up to the next multiple of 128 rows
    } else {
      m_valid = min(cnt, p.M);          // a count above M must not open rows past the output
      if (m_tile * 128 >= cnt) return;  // uniform for the whole CTA, before any barrier
    }
  }

  // conv tile origin
  int img0 = 0, h0 = 0;
  if constexpr (MODE != MODE_GEMM) {
    const int tiles_h = p.Hout / p.TH;
    img0 = (m_tile / tiles_h) * p.TN;
    h0 = (m_tile % tiles_h) * p.TH;
  }

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&p.tmA[0]);
    tma_prefetch_desc(&p.tmB);
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(&full[s], 1);
      mbar_init(&empty[s], 1);
    }
    mbar_init(tmem_full, 1);
    fence_mbar_init();
  }
  if (warp == 1) {
    tmem_alloc(tmem_slot, BLOCK_N);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  if (clk && threadIdx.x == 0) clk[1] = clock64();

  if (warp == 0) {
    // ------------------------------------------------------------ TMA producer (converged warp, elected lane)
    for (int kb = 0; kb < num_kb; ++kb) {
      const int s = kb % STAGES;
      const uint32_t ph = (kb / STAGES) & 1;
      mbar_wait(&empty[s], ph ^ 1);
      if (elect_one()) {
      mbar_expect_tx(&full[s], S::STAGE_BYTES);
      uint8_t* a_s = smem + s * S::STAGE_BYTES;
      uint8_t* b_s = a_s + S::A_BYTES;
      if constexpr (MODE == MODE_GEMM) {
        if constexpr (A_MN) {
#pragma unroll
          for (int c = 0; c < 128 / CHUNK; ++c)
            tma_load_3d(a_s + c * BK * 128, &p.tmA[0], &full[s], m_tile * 128 + c * CHUNK, (kb0 + kb) * BK, batch);
        } else {
          tma_load_3d(a_s, &p.tmA[0], &full[s], (kb0 + kb) * BK, m_tile * 128, batch);
        }
      } else if constexpr (MODE == MODE_CONV) {
        const int tap = kb / p.cin_chunks, cc = kb - tap * p.cin_chunks;
        const ConvTap t = p.taps[tap];
        tma_load_4d(a_s, &p.tmA[t.map], &full[s], cc * 64, t.dw, h0 + t.dh, img0);
      } else {  // MODE_STEM: k-block kb covers filter rows 2kb, 2kb+1 (x 8 pixels x 4 channels)
        tma_load_4d(a_s, &p.tmA[0], &full[s], 0, 0, h0 + kb, img0);
      }
      if constexpr (B_MN) {
#pragma unroll
        for (int c = 0; c < BLOCK_N / CHUNK; ++c)
          tma_load_3d(b_s + c * BK * 128, &p.tmB, &full[s], n0 + c * CHUNK, (kb0 + kb) * BK, batch);
      } else {
        tma_load_3d(b_s, &p.tmB, &full[s], (kb0 + kb) * BK, n0, batch);
      }
      }
      __syncwarp();
    }
  } else if (warp == 1) {
    // ------------------------------------------------------------ MMA issuer (converged warp, elected lane)
    constexpr uint32_t idesc = umma_idesc(KIND ? 2u : (CADRE_ENC_FP16 ? 0u : 1u), A_MN, B_MN, 128, BLOCK_N);
    constexpr uint32_t A_KSTEP = A_MN ? UMMA_K * 128 : 32;
    constexpr uint32_t B_KSTEP = B_MN ? UMMA_K * 128 : 32;
    constexpr uint32_t A_LBO = A_MN ? BK * 128 : 16;
    constexpr uint32_t B_LBO = B_MN ? BK * 128 : 16;
    // MN-major TF32 uses SWIZZLE_128B_BASE32B (layout type 1): atoms of 4 K-rows x 128 B -> SBO = 512 B
    constexpr uint32_t A_SBO = (A_MN && KIND) ? 512 : 1024, B_SBO = (B_MN && KIND) ? 512 : 1024;
    constexpr uint32_t A_LAYOUT = (A_MN && KIND) ? 1 : 2, B_LAYOUT = (B_MN && KIND) ? 1 : 2;
    for (int kb = 0; kb < num_kb; ++kb) {
      const int s = kb % STAGES;
      const uint32_t ph = (kb / STAGES) & 1;
      mbar_wait(&full[s], ph);
      tc_fence_after();
      if (clk && kb == 0 && lane == 0) clk[2] = clock64();
      const uint32_t a_addr = smem_u32(smem + s * S::STAGE_BYTES);
      const uint32_t b_addr = a_addr + S::A_BYTES;
      if (elect_one()) {
#pragma unroll
      for (int k = 0; k < BK / UMMA_K; ++k) {
        uint64_t da = umma_smem_desc(a_addr + k * A_KSTEP + p.dbg_a_shift * 128, A_LBO, A_SBO, A_LAYOUT);
        da |= static_cast<uint64_t>(p.dbg_base_offset & 7) << 49;
        const uint64_t db = umma_smem_desc(b_addr + k * B_KSTEP, B_LBO, B_SBO, B_LAYOUT);
        if constexpr (KIND)
          tc_mma_tf32(tmem_base, da, db, idesc, (kb | k) != 0);
        else
          tc_mma_f16(tmem_base, da, db, idesc, (kb | k) != 0);
      }
      tc_commit(&empty[s]);  // frees the smem stage once these MMAs have read it
      if (kb == num_kb - 1) tc_commit(tmem_full);
      }
      __syncwarp();
    }
    if (clk && lane == 0) clk[3] = clock64();
  } else if (warp >= 2) {
    // ------------------------------------------------------------ epilogue
    // Phase 1 (row per thread, the TMEM access pattern): accumulator -> registers -> padded smem staging tile.
    // Phase 2 (row per warp, lane = 4 consecutive columns): every global load / store of the fused epilogue is
    // a coalesced 512-byte row segment. (Row-per-thread global stores cost ~9 cycles per 16 bytes: 37 k cycles
    // per 128x128 fp32 tile on B200, measured with clock64 stamps.)
    const int q = warp & 3;  // TMEM lane quarter this warp may access
    constexpr int LDS = BLOCK_N + 4;
    float* stg = reinterpret_cast<float*>(smem) + (q * 32) * LDS;  // this quarter's 32 rows (aliases the stages)
    const int hf = EW == 2 ? (warp - 2) >> 2 : 0;   // which of the quarter's warps
    constexpr int CPW = BLOCK_N / 32 / EW;           // 32-column TMEM loads per warp
    const int r_lo = hf * (32 / EW), r_hi = r_lo + 32 / EW;   // rows of the quarter this warp finishes
    if (num_kb > 0) {
      mbar_wait(tmem_full, 0);
      tc_fence_after();
    }
    if (clk && threadIdx.x == 64) clk[4] = clock64();
    const uint32_t taddr = tmem_base + (static_cast<uint32_t>(q * 32) << 16);
#pragma unroll 1
    for (int c = hf * CPW; c < (hf + 1) * CPW; ++c) {
      uint32_t r[32];
      if (num_kb > 0 && p.dbg_epi != 3) {
        tmem_ld_32x32(taddr + c * 32, r);
        tmem_ld_wait();
      } else {
#pragma unroll
        for (int i = 0; i < 32; ++i) r[i] = 0u;
      }
      float* dst = stg + lane * LDS + c * 32;
#pragma unroll
      for (int j = 0; j < 8; ++j)
        *reinterpret_cast<float4*>(dst + 4 * j) =
            make_float4(__uint_as_float(r[4 * j]), __uint_as_float(r[4 * j + 1]), __uint_as_float(r[4 * j + 2]),
                        __uint_as_float(r[4 * j + 3]));
    }
    if constexpr (EW == 2)
      asm volatile("bar.sync %0, 64;" ::"r"(1 + q) : "memory");   // both warps of the quarter have staged their columns
    else
      __syncwarp();
    if (clk && threadIdx.x == 64) clk[7] = clock64();

    // With one epilogue warp per scheduler nothing hides instruction latency, so phase 2 is written for few
    // instructions per row: everything that depends only on the column (bias, pointers, flags) is hoisted, rows
    // are processed four at a time (independent chains), and the rare residual / mask / tail cases branch off.
    if (p.dbg_epi != 2) {
      constexpr int C4 = (BLOCK_N / 4 + 31) / 32;  // float4 column groups per lane
      const int row_base = m_tile * 128 + q * 32;  // GEMM mode: first logical row of this warp
#pragma unroll
      for (int cc = 0; cc < C4; ++cc) {
        const int c4 = lane + 32 * cc;
        const int n = n0 + c4 * 4;
        if (c4 * 4 >= BLOCK_N || n >= p.N) continue;
        const int nv = min(4, p.N - n);
        const float* srow = stg + c4 * 4;
        if constexpr (EPI == EPI_LINEAR) {
          float4 b4 = make_float4(0.f, 0.f, 0.f, 0.f);
          if (p.bias) {
            const float* bp = p.bias + batch * p.bias_bs + n;
            b4.x = bp[0];
            if (nv > 1) b4.y = bp[1];
            if (nv > 2) b4.z = bp[2];
            if (nv > 3) b4.w = bp[3];
          }
          const float alpha = p.alpha;
          const int act = p.act;
          // the fp32 ReLU-backward mask rides the fast path; residuals, conv row mapping and 16-bit masks do not
          const bool general = (p.res != nullptr) || (MODE != MODE_GEMM) || (p.mask != nullptr && sizeof(OutT) != 4);
          OutT* obase = reinterpret_cast<OutT*>(p.out) + batch * p.out_bs + ks * p.split_out_stride + n;
          const bool vec = nv == 4 && ((reinterpret_cast<uintptr_t>(obase) | (p.ldc * sizeof(OutT))) % (4 * sizeof(OutT)) == 0);
          const bool zero_rows = (p.batch_rows != nullptr) && !p.rows_is_k;
          if (!general && vec) {
            // fast path: plain GEMM rows, coalesced 16-byte stores
#pragma unroll 1
            const float* mbase = (sizeof(OutT) == 4 && p.mask != nullptr)
                                     ? reinterpret_cast<const float*>(p.mask) + batch * p.mask_bs + n
                                     : nullptr;
            for (int rr = r_lo; rr < r_hi; rr += 4) {
              float4 a4[4], m4[4];
#pragma unroll
              for (int k = 0; k < 4; ++k) {
                a4[k] = *reinterpret_cast<const float4*>(srow + (rr + k) * LDS);
                const int m = row_base + rr + k;
                m4[k] = (mbase != nullptr && m < m_valid)
                            ? *reinterpret_cast<const float4*>(mbase + static_cast<long long>(m) * p.ldm)
                            : make_float4(1.f, 1.f, 1.f, 1.f);
              }
#pragma unroll
              for (int k = 0; k < 4; ++k) {
                const int m = row_base + rr + k;
                float v0 = fmaf(a4[k].x, alpha, b4.x), v1 = fmaf(a4[k].y, alpha, b4.y);
                float v2 = fmaf(a4[k].z, alpha, b4.z), v3 = fmaf(a4[k].w, alpha, b4.w);
                if (!(m4[k].x > 0.f)) v0 = 0.f;   // ReLU backward: zero where the forward activation was <= 0
                if (!(m4[k].y > 0.f)) v1 = 0.f;
                if (!(m4[k].z > 0.f)) v2 = 0.f;
                if (!(m4[k].w > 0.f)) v3 = 0.f;
                if (act == ACT_RELU) {
                  v0 = fmaxf(v0, 0.f), v1 = fmaxf(v1, 0.f), v2 = fmaxf(v2, 0.f), v3 = fmaxf(v3, 0.f);
                } else if (act == ACT_LEAKY) {
                  v0 = v0 > 0.f ? v0 : 0.01f * v0, v1 = v1 > 0.f ? v1 : 0.01f * v1;
                  v2 = v2 > 0.f ? v2 : 0.01f * v2, v3 = v3 > 0.f ? v3 : 0.01f * v3;
                }
                const bool ok = m < m_valid;
                if (!ok) {
                  if (!(zero_rows && m < p.M)) continue;
                  v0 = v1 = v2 = v3 = 0.f;
                }
                OutT* o = obase + static_cast<long long>(m) * p.ldc;
                if constexpr (sizeof(OutT) == 4) {
                  *reinterpret_cast<float4*>(o) = make_float4(v0, v1, v2, v3);
                } else {
                  uint2 u;
                  u.x = enc_pack2(v0, v1), u.y = enc_pack2(v2, v3);
                  *reinterpret_cast<uint2*>(o) = u;
                }
              }
            }
          } else {
            // general path: residual / ReLU-backward mask / ragged N / conv row mapping
#pragma unroll 1
            for (int rr = r_lo; rr < r_hi; ++rr) {
              const int row = q * 32 + rr;
              long long out_row;
              bool row_ok;
              if constexpr (MODE == MODE_GEMM) {
                out_row = m_tile * 128 + row;
                row_ok = out_row < m_valid;
              } else {
                const int w = row % p.Wout;
                const int hh = (row / p.Wout) % p.TH;
                const int im = row / (p.Wout * p.TH);
                const int img = img0 + im, h = h0 + hh;
                row_ok = img < p.Bimg;
                out_row = (static_cast<long long>(img) * p.Hout + h) * p.Wout + w;
              }
              const bool zf = zero_rows && !row_ok && (MODE == MODE_GEMM) && out_row < p.M;
              if (!(row_ok || zf)) continue;
              const float4 acc4 = *reinterpret_cast<const float4*>(srow + rr * LDS);
              float v[4] = {fmaf(acc4.x, alpha, b4.x), fmaf(acc4.y, alpha, b4.y), fmaf(acc4.z, alpha, b4.z),
                            fmaf(acc4.w, alpha, b4.w)};
              if (row_ok) {
                const OutT* res = p.res ? reinterpret_cast<const OutT*>(p.res) + batch * p.res_bs + out_row * p.ldr + n
                                        : nullptr;
                const OutT* mask = p.mask ? reinterpret_cast<const OutT*>(p.mask) + batch * p.mask_bs +
                                                out_row * p.ldm + n
                                          : nullptr;
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                  if (i < nv) {
                    float x = v[i];
                    if (res && !p.res_after_act) x += load_as_float<OutT>(res, i);
                    if (act == ACT_RELU) x = fmaxf(x, 0.f);
                    if (act == ACT_LEAKY) x = x > 0.f ? x : 0.01f * x;
                    if (res && p.res_after_act) x += load_as_float<OutT>(res, i);
                    if (mask && !(load_as_float<OutT>(mask, i) > 0.f)) x = 0.f;
                    v[i] = x;
                  }
                }
              } else {
                v[0] = v[1] = v[2] = v[3] = 0.f;
              }
              OutT* o = obase + out_row * p.ldc;
              if (vec) {
                if constexpr (sizeof(OutT) == 4) {
                  *reinterpret_cast<float4*>(o) = make_float4(v[0], v[1], v[2], v[3]);
                } else {
                  uint2 u;
                  u.x = enc_pack2(v[0], v[1]), u.y = enc_pack2(v[2], v[3]);
                  *reinterpret_cast<uint2*>(o) = u;
                }
              } else {
                for (int i = 0; i < nv; ++i) {
                  if constexpr (sizeof(OutT) == 4)
                    o[i] = v[i];
                  else
                    o[i] = enc_from_float(v[i]);
                }
              }
            }
          }
        }
      }
    }
  }

  if (clk && threadIdx.x == 64) clk[5] = clock64();
  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem_base, BLOCK_N);
  if (clk && threadIdx.x == 0) clk[6] = clock64();
}

}  // namespace cadre

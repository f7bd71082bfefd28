// Internal (C++) declarations shared between the translation units of libcadre_sm100.so.
#pragma once
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <string.h>

#include <stdexcept>
#include <string>

// 16-bit storage / tensor-core operand type of the encoder path. fp16 (default) keeps the 20-layer encoder at
// ~1.3e-3 relative error against the fp32 reference; bf16 sits at ~9e-3, on the edge of the 1e-2 budget
// (measured, DESIGN.md). Both run at the same tcgen05 kind::f16 rate; stores saturate instead of overflowing.
#ifndef CADRE_ENC_FP16
#define CADRE_ENC_FP16 1
#endif

namespace cadre {

#if CADRE_ENC_FP16
using enc_t = __half;
__device__ __forceinline__ enc_t enc_from_float(float f) {
  return __float2half_rn(fminf(fmaxf(f, -65504.f), 65504.f));
}
__device__ __forceinline__ float enc_to_float(enc_t h) { return __half2float(h); }
#else
using enc_t = __nv_bfloat16;
__device__ __forceinline__ enc_t enc_from_float(float f) { return __float2bfloat16_rn(f); }
__device__ __forceinline__ float enc_to_float(enc_t h) { return __bfloat162float(h); }
#endif
// two floats -> one packed 32-bit word, clamped to the finite fp16 range: ONE instruction on sm_100a
// (F2FP.SATFINITE[.RELU].F16.F32.PACK_AB) instead of clamp + clamp (+ max) + convert per value
__device__ __forceinline__ uint32_t enc_pack2(float a, float b) {
#if CADRE_ENC_FP16
  uint32_t r;
  asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(b), "f"(a));   // a -> low half
  return r;
#else
  __nv_bfloat162 h = __floats2bfloat162_rn(a, b);
  return *reinterpret_cast<uint32_t*>(&h);
#endif
}
// pack(max(a, 0), max(b, 0)): the ReLU rides in the conversion
__device__ __forceinline__ uint32_t enc_pack2_relu(float a, float b) {
#if CADRE_ENC_FP16
  uint32_t r;
  asm("cvt.rn.relu.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(b), "f"(a));
  return r;
#else
  __nv_bfloat162 h = __floats2bfloat162_rn(fmaxf(a, 0.f), fmaxf(b, 0.f));
  return *reinterpret_cast<uint32_t*>(&h);
#endif
}
// values already known to be >= 0
__device__ __forceinline__ uint32_t enc_pack2_pos(float a, float b) { return enc_pack2(a, b); }

struct Error : public std::runtime_error {
  int code;
  Error(int c, const std::string& m) : std::runtime_error(m), code(c) {}
};

void set_last_error(const std::string& msg);

#define CADRE_CUDA_CHECK(expr)                                                                       \
  do {                                                                                               \
    cudaError_t e__ = (expr);                                                                        \
    if (e__ != cudaSuccess)                                                                          \
      throw ::cadre::Error(2, std::string(#expr) + " -> " + cudaGetErrorString(e__) + " at " + __FILE__ + \
                                  ":" + std::to_string(__LINE__));                                   \
  } while (0)

#define CADRE_REQUIRE(cond, msg)                                              \
  do {                                                                        \
    if (!(cond)) throw ::cadre::Error(1, std::string("invalid argument: ") + (msg)); \
  } while (0)

// ------------------------------------------------------------------ dense tile kernel (tc_gemm.cu)
// D[M,N] = act(alpha * A*B^T + bias + res) ...; operands are either K-major ([rows=M|N][K], ld = row stride)
// or MN-major ([rows=K][M|N], ld = row stride). kind 0 = bf16 operands, 1 = fp32 operands fed as TF32.
struct GemmArgs {
  int kind = 0, a_mn = 0, b_mn = 0;
  const void* A = nullptr;
  long long lda = 0, a_bs = 0;
  const void* B = nullptr;
  long long ldb = 0, b_bs = 0;
  int M = 0, N = 0, K = 0, batch = 1;
  void* out = nullptr;
  int out_f32 = 0;
  long long ldc = 0, out_bs = 0;
  const float* bias = nullptr;
  long long bias_bs = 0;
  const void* res = nullptr;
  long long ldr = 0, res_bs = 0;
  int res_after_act = 0;
  const void* mask = nullptr;
  long long ldm = 0, mask_bs = 0;
  int act = 0;
  float alpha = 1.f;
  const int* batch_rows = nullptr;
  int rows_is_k = 0;
  const int* tile_list = nullptr;  // optional device work list {n, (batch, m_tile) x n}; grid.x = max_tiles, grid.z = 1
  int max_tiles = 0;
  int block_n = 0;  // 0 = choose
  int ksplit = 1;                  // split-K: partial sums go to out + ks * split_out_stride
  long long split_out_stride = 0;
  int dbg_a_shift = 0, dbg_base_offset = 0;
  long long* dbg_clk = nullptr;
  int dbg_epi = 0;
  // LSTM-cell epilogue (epi = 1)
  int epi = 0;
  const float* xpart = nullptr;
  long long ldx = 0, x_bs = 0;
  const float* c_prev = nullptr;
  float* c_out = nullptr;
  float* h_out = nullptr;
  float* gates_out = nullptr;
  long long ldh = 0, h_bs = 0;
};
void launch_gemm(const GemmArgs& a, cudaStream_t stream);
// cuTensorMapEncodeTiled for an fp16 tensor, 128B swizzle, zero fill out of bounds; dims / box innermost first,
// strides_bytes has rank-1 entries (dimension 0 is contiguous)
void make_tensor_map_f16(CUtensorMap* m, int rank, const void* base, const uint64_t* dims,
                         const uint64_t* strides_bytes, const uint32_t* box);

// Implicit-GEMM convolution over NHWC bf16 activations; weights [Cout][KH][KW][Cin] bf16 (BN folded).
struct ConvArgs {
  const enc_t* in = nullptr;  // [B][Hin][Win][Cin]
  int B = 0, Hin = 0, Win = 0, Cin = 0;
  const enc_t* w = nullptr;  // [Cout][KH*KW*Cin]
  int Cout = 0, KH = 1, KW = 1, stride = 1, pad = 0;
  const float* bias = nullptr;        // [Cout]
  const enc_t* res = nullptr; // [B][Hout][Wout][Cout] or null
  int res_after_act = 0;
  int act = 0;
  enc_t* out = nullptr;  // [B][Hout][Wout][Cout]
  int in_pad = 0;        // input tensor is [B][Hin+2][Win+2][Cin] with a zero border (Hin/Win stay logical)
  int out_pad = 0;       // output (and residual) tensors are [B][Hout+2][Wout+2][Cout]; the border is never written
  // Optional fused shortcut (ResNet downsample, resnet.py:152-158): out += conv1x1/stride-2 of a SECOND input,
  // executed as Cin2/64 extra k-blocks of the same implicit GEMM. `w` is then [Cout][KH*KW*Cin + Cin2] (the
  // shortcut weights appended along K) and `bias` the sum of both biases; in2 is [B][Hin2 (+2)][Win2 (+2)][Cin2]
  // with Hout = (Hin2 - 1) / 2 + 1.
  const enc_t* in2 = nullptr;
  int Cin2 = 0, in2_pad = 0, Hin2 = 0, Win2 = 0;
};
void launch_conv(const ConvArgs& a, cudaStream_t stream);

// Halo-reuse 3x3/s1/p1 64->64 convolution on zero-bordered activations [B][H+2][W+2][64] (tc_flat3x3.cuh)
struct FlatArgs {
  const enc_t* in = nullptr;
  int B = 0, H = 0, W = 0;
  const enc_t* w = nullptr;   // [64][3][3][64]
  const float* bias = nullptr;
  const enc_t* res = nullptr; // zero-bordered, same shape as out
  int act = 0;
  enc_t* out = nullptr;
};
void launch_flat3x3(const FlatArgs& a, cudaStream_t stream);
// the same for 128 -> 128 channels (ResNet layer2): [B][H+2][W+2][128], weights [128][3][3][128] (tc_halo128.cuh)
void launch_halo128(const FlatArgs& a, cudaStream_t stream);

// 7x7/s2/p3 stem over the padded 4-channel bf16 image [B][150][262][4]; weights [64][256] (K = 4 row pairs x
// 2 rows x 8 pixels x 4 ch, zero where kh==7 or kw==7); output [B][72][128][64].
struct StemArgs {
  const enc_t* in = nullptr;
  int B = 0;
  const enc_t* w = nullptr;
  const float* bias = nullptr;
  enc_t* out = nullptr;
};
void launch_stem(const StemArgs& a, cudaStream_t stream);
// fused stem + ReLU + maxpool -> zero-bordered [B][38][66][64] (tc_stem_pool.cuh); `out` of StemArgs is that buffer
void launch_stem_pool(const StemArgs& a, cudaStream_t stream);

// Segmented (per-module) gradient norm + clip + Adam over flat buffers cut into chunks (rollout_optim_kernels.cu)
struct OptTables {
  int num_chunks = 0;
  long long* chunk_off = nullptr;  // [num_chunks] element offset
  int* chunk_len = nullptr;        // [num_chunks] multiple of 4
  int* chunk_mod = nullptr;        // [num_chunks] module id 0..15, non-decreasing
  int* mod_first = nullptr;        // [17] first chunk of each module
  int mod_first_h[17] = {};        // host copy
  float* partial = nullptr;        // [num_chunks]
  float* clip_coef = nullptr;      // [16]
  float* norms = nullptr;          // [16]
  float* scalars = nullptr;        // [2] Adam step size and sqrt(1 - beta2^step) of the current step
};
// Launch with the programmatic-stream-serialization attribute (PDL, see ptx.cuh): all kernels of the library
// call pdl_wait() before touching global memory, so consecutive launches overlap prologue and launch latency
// with the predecessor's tail. CADRE_NO_PDL=1 restores plain stream order (A/B switch).
bool pdl_enabled();
extern long long* g_dbg_clk;
extern int g_dbg_persist_launch;
template <typename... KArgs, typename... Args>
inline void launch_k(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t stream, Args&&... args) {
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof(cfg));
  cfg.gridDim = grid, cfg.blockDim = block, cfg.dynamicSmemBytes = smem, cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr, cfg.numAttrs = pdl_enabled() ? 1 : 0;
  CADRE_CUDA_CHECK(cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...));
}

// cudaFuncAttributeMaxDynamicSharedMemorySize is a PER-DEVICE attribute: remember per (call site, device) which
// devices have been configured, so that a process driving several GPUs (vae_device != device_num, agent.py:21-31)
// configures each of them. `flags` is a caller-owned static array of CADRE_MAX_DEVICES entries.
constexpr int CADRE_MAX_DEVICES = 64;
inline int current_device() {
  int dev = 0;
  CADRE_CUDA_CHECK(cudaGetDevice(&dev));
  CADRE_REQUIRE(dev >= 0 && dev < CADRE_MAX_DEVICES, "device ordinal");
  return dev;
}
template <typename Kern>
inline void ensure_dynamic_smem(Kern kern, size_t smem, size_t* flags) {
  const int dev = current_device();
  if (smem > flags[dev]) {
    CADRE_CUDA_CHECK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
    flags[dev] = smem;
  }
}

// modules [mod_begin, mod_end) only (module e < 8: LSTM of expert e, 8 + e: actor-critic of expert e). `gate` (NULL:
// always step): two device words read at run time, gate[0] != 0 skips the norms and the step, gate[1] != 0 the step only.
void launch_clip_adam(const OptTables& t, float* params, const float* grads, float* m, float* v, float max_norm,
                      float lr, float beta1, float beta2, float eps, int step, cudaStream_t s, int mod_begin = 0,
                      int mod_end = 16, const int* dev_step = nullptr, float* norms_hist = nullptr,
                      const int* gate = nullptr);

}  // namespace cadre

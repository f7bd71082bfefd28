// Host side of the tcgen05 tile kernel: TMA tensor-map construction and template dispatch.
#include "internal.h"
#include "tc_gemm.cuh"
#include "tc_flat3x3.cuh"
#include "tc_halo128.cuh"
#include "tc_persist.cuh"
#include "tc_stem_pool.cuh"

#include <cstdlib>
#include <mutex>

namespace cadre {

long long* g_dbg_clk = nullptr;   // cadre_debug_clk: per-CTA cycle counters of the flat / stem / persistent kernels
int g_dbg_persist_launch = 0;     // region 3 + n for the n-th persistent launch since cadre_debug_clk()
static PersistParams with_dbg(const PersistParams& p) {
  PersistParams q = p;
  q.dbg = g_dbg_clk ? g_dbg_clk + static_cast<long long>(3 + g_dbg_persist_launch++) * 148 * 16 : nullptr;
  return q;
}


// ---------------------------------------------------------------------------------------------------------
// cuTensorMapEncodeTiled through the runtime's driver entry point (the library does not link libcuda).
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*,
                                  CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion,
                                  CUtensorMapFloatOOBfill);

static EncodeTiledFn encode_fn() {
  static EncodeTiledFn fn = nullptr;
  static std::once_flag once;
  std::call_once(once, [] {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    cudaError_t e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q);
    if (e == cudaSuccess && q == cudaDriverEntryPointSuccess) fn = reinterpret_cast<EncodeTiledFn>(p);
  });
  if (!fn) throw Error(3, "cuTensorMapEncodeTiled is not available from this driver");
  return fn;
}

// fp32 operands are loaded as CU_TENSOR_MAP_DATA_TYPE_TFLOAT32 so that TMA rounds them to TF32 (round to
// nearest) on the way to shared memory; plain FLOAT32 would leave the truncation to the tensor core, which
// biases every product towards zero (measured: 7.7e-4 -> see DESIGN.md). CADRE_TF32_TRUNCATE=1 restores that.
static const bool g_tf32_rn = getenv("CADRE_TF32_TRUNCATE") == nullptr;

// dims/box innermost first; strides_bytes has rank-1 entries (dimension 0 is contiguous).
static void make_map(CUtensorMap* m, int es, int rank, const void* base, const uint64_t* dims,
                     const uint64_t* strides_bytes, const uint32_t* box, bool atom32 = false) {
  cuuint64_t gdim[5], gstr[4];
  cuuint32_t bx[5], estr[5];
  for (int i = 0; i < rank; ++i) {
    gdim[i] = dims[i];
    bx[i] = box[i];
    estr[i] = 1;
    if (i > 0) gstr[i - 1] = strides_bytes[i - 1];
  }
  CADRE_REQUIRE(reinterpret_cast<uintptr_t>(base) % 16 == 0, "TMA base address must be 16-byte aligned");
  for (int i = 0; i + 1 < rank; ++i)
    CADRE_REQUIRE(gstr[i] % 16 == 0 && gstr[i] > 0, "TMA strides must be positive multiples of 16 bytes");
  CUresult r = encode_fn()(m, es == 4 ? (g_tf32_rn ? CU_TENSOR_MAP_DATA_TYPE_TFLOAT32 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32) : (CADRE_ENC_FP16 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16),
                           rank, const_cast<void*>(base), gdim, gstr, bx, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                           atom32 ? CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B : CU_TENSOR_MAP_SWIZZLE_128B,
                           CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                           CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) throw Error(3, "cuTensorMapEncodeTiled failed with CUresult " + std::to_string(r));
}

// fp16 tensor map with the 128B swizzle for callers outside this file (lstm_seq.cuh's exchange buffers)
void make_tensor_map_f16(CUtensorMap* m, int rank, const void* base, const uint64_t* dims,
                         const uint64_t* strides_bytes, const uint32_t* box) {
  static_assert(CADRE_ENC_FP16 == 1, "make_tensor_map_f16 relies on the fp16 build of make_map");
  make_map(m, 2, rank, base, dims, strides_bytes, box);
}

// matrix operand map: K-major -> dims {K, rows, batch}, box {BK, box_rows, 1};
//                     MN-major -> dims {rows(MN), K, batch}, box {CHUNK, BK, 1}
static void make_operand_map(CUtensorMap* m, int es, bool mn_major, const void* base, long long ld,
                             long long bs, int mn, int k, int batch, int box_rows) {
  const int bk = 128 / es;
  uint64_t dims[3], str[2];
  uint32_t box[3];
  const long long rows_stored = mn_major ? k : mn;
  str[0] = static_cast<uint64_t>(ld) * es;
  str[1] = static_cast<uint64_t>(batch > 1 ? bs : ld * rows_stored) * es;
  if (str[1] == 0 || str[1] % 16) str[1] = 16;  // batch == 1: never dereferenced beyond index 0
  if (mn_major) {
    dims[0] = mn, dims[1] = k, dims[2] = batch;
    box[0] = bk, box[1] = bk, box[2] = 1;
  } else {
    dims[0] = k, dims[1] = mn, dims[2] = batch;
    box[0] = bk, box[1] = box_rows, box[2] = 1;
  }
  // MN-major fp32 (TF32) operands only exist in the 128B swizzle with 32-byte atoms (UMMA layout type 1)
  make_map(m, es, 3, base, dims, str, box, mn_major && es == 4);
}

template <int KIND, int A_MN, int B_MN, int BN, int STAGES, int MODE, int EPI, typename OutT, int EW = 1>
static void launch_inst(const TcGemmParams& p, dim3 grid, cudaStream_t stream) {
  auto kern = tc_gemm_kernel<KIND, A_MN, B_MN, BN, STAGES, MODE, EPI, OutT, EW>;
  constexpr int smem = TcGemmSmem<KIND, BN, STAGES>::TOTAL;
  static size_t configured[CADRE_MAX_DEVICES] = {};   // per instantiation and device
  ensure_dynamic_smem(kern, smem, configured);
  launch_k(kern, dim3(grid), dim3(64 + 128 * EW), smem, stream, p);
  CADRE_CUDA_CHECK(cudaGetLastError());
}

static int num_sms() {
  static int n[CADRE_MAX_DEVICES] = {};
  const int dev = current_device();
  if (!n[dev]) CADRE_CUDA_CHECK(cudaDeviceGetAttribute(&n[dev], cudaDevAttrMultiProcessorCount, dev));
  return n[dev];
}
bool pdl_enabled() {
  static const bool on = getenv("CADRE_NO_PDL") == nullptr;
  return on;
}

// CTA-pair variant (cta_group::2): clusters of two CTAs, one 256 x BN tile per pair
template <int BN, int STAGES, int MODE>
static void launch_persist2(const PersistParams& p, cudaStream_t stream) {
  auto kern = tc_persist_kernel<BN, STAGES, MODE, true>;
  constexpr int smem = PersistSmem<BN, STAGES, true>::TOTAL;
  static size_t configured[CADRE_MAX_DEVICES] = {};   // per instantiation and device
  ensure_dynamic_smem(kern, smem, configured);
  const int pairs_needed = ((p.tiles_m + 1) / 2) * p.tiles_n;
  int pairs = num_sms() / 2;
  if (pairs_needed < pairs) pairs = pairs_needed;
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof(cfg));
  cfg.gridDim = dim3(2 * pairs), cfg.blockDim = dim3(320), cfg.dynamicSmemBytes = smem, cfg.stream = stream;
  cudaLaunchAttribute attr[2];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = 2, attr[0].val.clusterDim.y = 1, attr[0].val.clusterDim.z = 1;
  attr[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[1].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr, cfg.numAttrs = pdl_enabled() ? 2 : 1;
  CADRE_CUDA_CHECK(cudaLaunchKernelEx(&cfg, kern, with_dbg(p)));
}

template <int BN, int STAGES, int MODE>
static void launch_persist(const PersistParams& p, cudaStream_t stream) {
  auto kern = tc_persist_kernel<BN, STAGES, MODE>;
  constexpr int smem = PersistSmem<BN, STAGES>::TOTAL;
  static size_t configured[CADRE_MAX_DEVICES] = {};   // per instantiation and device
  ensure_dynamic_smem(kern, smem, configured);
  const int tiles = p.tiles_m * p.tiles_n;
  const int grid = tiles < num_sms() ? tiles : num_sms();
  launch_k(kern, dim3(grid), dim3(320), smem, stream, with_dbg(p));
  CADRE_CUDA_CHECK(cudaGetLastError());
}

static void fill_epilogue(TcGemmParams& p, const GemmArgs& a) {
  p.out = a.out, p.ldc = a.ldc, p.out_bs = a.out_bs;
  p.bias = a.bias, p.bias_bs = a.bias_bs;
  p.res = a.res, p.ldr = a.ldr, p.res_bs = a.res_bs, p.res_after_act = a.res_after_act;
  p.mask = a.mask, p.ldm = a.ldm, p.mask_bs = a.mask_bs;
  p.act = a.act, p.alpha = a.alpha;
  p.batch_rows = a.batch_rows, p.rows_is_k = a.rows_is_k;
  p.tile_list = a.tile_list;
  p.dbg_a_shift = a.dbg_a_shift, p.dbg_base_offset = a.dbg_base_offset, p.dbg_clk = a.dbg_clk, p.dbg_epi = a.dbg_epi;
}

void launch_gemm(const GemmArgs& a, cudaStream_t stream) {
  CADRE_REQUIRE(a.M > 0 && a.N > 0 && a.batch > 0, "gemm dims");
  CADRE_REQUIRE(a.K > 0, "gemm K must be positive (an empty contraction has no tensor map)");
  CADRE_REQUIRE(a.A && a.B && a.out, "gemm pointers");
  // the fp32 epilogue reads the ReLU-backward mask as float4 rows (tc_gemm.cuh fast path)
  CADRE_REQUIRE(!a.mask || !a.out_f32 ||
                    (reinterpret_cast<uintptr_t>(a.mask) % 16 == 0 && a.ldm % 4 == 0 && a.mask_bs % 4 == 0),
                "gemm fp32 mask must be 16-byte aligned with ldm and mask_bs multiples of 4");
  CADRE_REQUIRE(a.epi == EPI_LINEAR, "the LSTM-cell epilogue moved into the persistent recurrence kernels (lstm_seq.cuh)");
  const int es = a.kind ? 4 : 2;
  const int bk = 128 / es;
  int bn = a.block_n ? a.block_n : (a.N <= 64 ? 64 : 128);
  if (a.kind == 0 && !a.a_mn && !a.b_mn && a.batch == 1 && !a.out_f32 && a.epi == 0 && !a.mask &&
      !a.batch_rows && a.alpha == 1.f && a.N % 8 == 0) {
    PersistParams q;
    memset(&q, 0, sizeof(q));
    bn = a.N <= 64 ? 64 : 128;
    make_operand_map(&q.tmA[0], 2, false, a.A, a.lda, 0, a.M, a.K, 1, 128);
    make_operand_map(&q.tmB, 2, false, a.B, a.ldb, 0, a.N, a.K, 1, bn);
    {
      const uint64_t dims[3] = {(uint64_t)a.N, (uint64_t)a.M, 1};
      const uint64_t str[2] = {(uint64_t)a.ldc * 2, (uint64_t)a.ldc * 2 * a.M};
      const uint32_t box[3] = {64, 128, 1};
      make_map(&q.tmOut, 2, 3, a.out, dims, str, box);
    }
    q.num_kb = (a.K + 63) / 64;
    q.tiles_m = (a.M + 127) / 128, q.tiles_n = (a.N + bn - 1) / bn;
    q.M = a.M, q.N = a.N;
    q.bias = a.bias, q.res = static_cast<const enc_t*>(a.res), q.ldr = a.ldr;
    q.res_after_act = a.res_after_act, q.act = a.act;
    CADRE_REQUIRE(a.bias != nullptr, "persistent gemm needs a bias vector");
    if (bn == 64)
      launch_persist<64, 6, MODE_GEMM>(q, stream);
    else
      launch_persist<128, 5, MODE_GEMM>(q, stream);
    return;
  }
  TcGemmParams p;
  memset(&p, 0, sizeof(p));
  make_operand_map(&p.tmA[0], es, a.a_mn, a.A, a.lda, a.a_bs, a.M, a.K, a.batch, 128);
  make_operand_map(&p.tmB, es, a.b_mn, a.B, a.ldb, a.b_bs, a.N, a.K, a.batch, bn);
  p.M = a.M, p.N = a.N, p.num_kb = (a.K + bk - 1) / bk;
  fill_epilogue(p, a);
  {  // debug: CADRE_DBG_CLK_EPI=<epi>:<device pointer> stamps every GEMM with that epilogue kind (in-situ probe)
    static const char* spec = getenv("CADRE_DBG_CLK_EPI");
    static const char* zsel = getenv("CADRE_DBG_CLK_Z");   // optional: only launches with this grid.z
    const int gz = a.batch * (a.ksplit > 1 ? a.ksplit : 1);
    if (spec && atoi(spec) == a.epi && strchr(spec, ':') && (!zsel || atoi(zsel) == gz))
      p.dbg_clk = reinterpret_cast<long long*>(strtoull(strchr(spec, ':') + 1, nullptr, 0));
  }
  p.ksplit = a.ksplit > 1 ? a.ksplit : 1;
  p.kb_per_split = (p.num_kb + p.ksplit - 1) / p.ksplit;
  p.split_out_stride = a.split_out_stride;
  CADRE_REQUIRE(p.ksplit == 1 || (!a.bias && !a.res && !a.mask && a.act == 0 && !a.rows_is_k && a.epi == 0),
                "split-K supports plain partial sums only");
  dim3 grid((a.M + 127) / 128, (a.N + bn - 1) / bn, a.batch * p.ksplit);
  if (a.tile_list != nullptr) {
    CADRE_REQUIRE(a.max_tiles > 0 && p.ksplit == 1 && a.batch_rows != nullptr && !a.rows_is_k, "tile list arguments");
    grid = dim3(a.max_tiles, (a.N + bn - 1) / bn, 1);
  }

#define CADRE_GEMM_CASE(KIND, AMN, BMN, BN, ST, EPI, OUT_F32, OutT)                                   \
  if (a.kind == KIND && a.a_mn == AMN && a.b_mn == BMN && bn == BN && a.epi == EPI && a.out_f32 == OUT_F32) { \
    launch_inst<KIND, AMN, BMN, BN, ST, MODE_GEMM, EPI, OutT>(p, grid, stream);                       \
    return;                                                                                           \
  }
  // bf16 operands (encoder linears)
  CADRE_GEMM_CASE(0, 0, 0, 64, 4, EPI_LINEAR, 0, enc_t)
  CADRE_GEMM_CASE(0, 0, 0, 128, 4, EPI_LINEAR, 0, enc_t)
  CADRE_GEMM_CASE(0, 0, 0, 64, 4, EPI_LINEAR, 1, float)
  CADRE_GEMM_CASE(0, 0, 0, 128, 3, EPI_LINEAR, 1, float)   // PPO x-part GEMM (fp16 x W_ih^T): 2 CTAs per SM
  CADRE_GEMM_CASE(0, 0, 1, 128, 4, EPI_LINEAR, 1, float)
  CADRE_GEMM_CASE(0, 1, 1, 128, 3, EPI_LINEAR, 1, float)   // PPO LSTM weight gradients (fp16 dG^T x / h): 2 CTAs per SM
  // fp32 operands as TF32 (PPO update: forward, dgrad, wgrad, LSTM cell)
  // the PPO GEMMs are latency-bound (few CTAs, short 128-byte k-blocks): deep pipelines, one CTA per SM
  // default: 3 stages (97 KB) -> two CTAs per SM
  CADRE_GEMM_CASE(1, 0, 0, 64, 4, EPI_LINEAR, 1, float)
  CADRE_GEMM_CASE(1, 0, 0, 128, 3, EPI_LINEAR, 1, float)
  CADRE_GEMM_CASE(1, 0, 1, 128, 3, EPI_LINEAR, 1, float)
  CADRE_GEMM_CASE(1, 1, 1, 128, 3, EPI_LINEAR, 1, float)
#undef CADRE_GEMM_CASE
  throw Error(1, "launch_gemm: unsupported (kind, majors, block_n, epilogue, out dtype) combination");
}

// ---------------------------------------------------------------------------------------------------------
void launch_conv(const ConvArgs& a, cudaStream_t stream) {
  CADRE_REQUIRE(a.Cin % 64 == 0, "conv Cin must be a multiple of 64");
  CADRE_REQUIRE(a.stride == 1 || a.stride == 2, "conv stride must be 1 or 2");
  CADRE_REQUIRE(a.KH * a.KW <= 12, "conv filter too large for the tap table");
  const int Hout = (a.Hin + 2 * a.pad - a.KH) / a.stride + 1;
  const int Wout = (a.Win + 2 * a.pad - a.KW) / a.stride + 1;
  CADRE_REQUIRE(Wout <= 128 && 128 % Wout == 0, "conv output width must divide 128");
  // zero-bordered input: same taps, shifted by one pixel, on a (Hin+2) x (Win+2) tensor
  const int Hs = a.Hin + 2 * a.in_pad, Ws = a.Win + 2 * a.in_pad, pad_eff = a.pad - a.in_pad;
  const int rows_per_tile = 128 / Wout;
  int TH = 1;
  while (TH * 2 <= rows_per_tile && Hout % (TH * 2) == 0) TH *= 2;
  const int TN = rows_per_tile / TH;
  static const bool allow_bn256 = getenv("CADRE_NO_BN256") == nullptr;
  const int bn = a.Cout <= 64 ? 64 : ((a.Cout % 256 == 0 && allow_bn256) ? 256 : 128);

  TcGemmParams p;
  memset(&p, 0, sizeof(p));
  const uint64_t es = 2;
  const uint32_t box[4] = {64u, static_cast<uint32_t>(Wout), static_cast<uint32_t>(TH),
                           static_cast<uint32_t>(TN)};
  if (a.stride == 1) {
    const uint64_t dims[4] = {(uint64_t)a.Cin, (uint64_t)Ws, (uint64_t)Hs, (uint64_t)a.B};
    const uint64_t str[3] = {a.Cin * es, (uint64_t)Ws * a.Cin * es, (uint64_t)Hs * Ws * a.Cin * es};
    make_map(&p.tmA[0], 2, 4, a.in, dims, str, box);
    for (int i = 1; i < 4; ++i) p.tmA[i] = p.tmA[0];
  } else {
    for (int ph = 0; ph < 2; ++ph)
      for (int pw = 0; pw < 2; ++pw) {
        const int Hq = (Hs - ph + 1) / 2, Wq = (Ws - pw + 1) / 2;
        const uint64_t dims[4] = {(uint64_t)a.Cin, (uint64_t)Wq, (uint64_t)Hq, (uint64_t)a.B};
        const uint64_t str[3] = {2 * a.Cin * es, 2 * (uint64_t)Ws * a.Cin * es, (uint64_t)Hs * Ws * a.Cin * es};
        if (Hq > 0 && Wq > 0)
          make_map(&p.tmA[ph * 2 + pw], 2, 4, a.in + ((long long)ph * Ws + pw) * a.Cin, dims, str, box);
      }
  }
  int nt = 0;
  for (int kh = 0; kh < a.KH; ++kh)
    for (int kw = 0; kw < a.KW; ++kw) {
      ConvTap t;
      const int oh = kh - pad_eff, ow = kw - pad_eff;
      if (a.stride == 1) {
        t.map = 0, t.dh = (short)oh, t.dw = (short)ow;
      } else {
        const int ph = oh & 1, pw = ow & 1;
        t.map = (short)(ph * 2 + pw), t.dh = (short)((oh - ph) / 2), t.dw = (short)((ow - pw) / 2);
      }
      t.pad_ = 0;
      p.taps[nt++] = t;
    }
  p.ntaps = nt, p.cin_chunks = a.Cin / 64;
  p.num_kb = nt * p.cin_chunks;
  const int kb_main = p.num_kb;
  int Ktot = nt * a.Cin;
  if (a.in2 != nullptr) {
    // fused shortcut: output (h, w) reads in2 pixel (2h, 2w) -> parity sub-lattice map of the (bordered) tensor
    CADRE_REQUIRE(a.stride == 1 && a.Cin2 % 64 == 0 && a.Cin2 > 0 && nt < 12, "fused shortcut arguments");
    CADRE_REQUIRE((a.Hin2 - 1) / 2 + 1 == Hout && (a.Win2 - 1) / 2 + 1 == Wout, "fused shortcut input size");
    const int Hs2 = a.Hin2 + 2 * a.in2_pad, Ws2 = a.Win2 + 2 * a.in2_pad, par = a.in2_pad & 1;
    const int Hq = (Hs2 - par + 1) / 2, Wq = (Ws2 - par + 1) / 2;
    const uint64_t dims[4] = {(uint64_t)a.Cin2, (uint64_t)Wq, (uint64_t)Hq, (uint64_t)a.B};
    const uint64_t str[3] = {2 * a.Cin2 * es, 2 * (uint64_t)Ws2 * a.Cin2 * es, (uint64_t)Hs2 * Ws2 * a.Cin2 * es};
    make_map(&p.tmA[1], 2, 4, a.in2 + ((long long)par * Ws2 + par) * a.Cin2, dims, str, box);
    ConvTap t;
    t.map = 1, t.dh = (short)((a.in2_pad - par) / 2), t.dw = (short)((a.in2_pad - par) / 2), t.pad_ = 0;
    p.taps[nt] = t;
    p.num_kb += a.Cin2 / 64;
    Ktot += a.Cin2;
  }
  p.Hout = Hout, p.Wout = Wout, p.TH = TH, p.TN = TN, p.Bimg = a.B;
  // weights: [Cout][K] K-major
  {
    const int K = Ktot;
    make_operand_map(&p.tmB, 2, false, a.w, K, 0, a.Cout, K, 1, bn);
  }
  p.M = 0, p.N = a.Cout;
  p.out = a.out, p.ldc = a.Cout;
  p.bias = a.bias;
  p.res = a.res, p.ldr = a.Cout, p.res_after_act = a.res_after_act;
  p.act = a.act, p.alpha = 1.f;
  dim3 grid((Hout / TH) * ((a.B + TN - 1) / TN), (a.Cout + bn - 1) / bn, 1);
  {
    PersistParams q;
    memset(&q, 0, sizeof(q));
    for (int i = 0; i < 4; ++i) q.tmA[i] = p.tmA[i];
    q.tmB = p.tmB;
    {
      // out_pad: the output tensor is [B][Hout+2][Wout+2][Cout] with a zero border the stores never touch
      const int Ho2 = Hout + 2 * a.out_pad, Wo2 = Wout + 2 * a.out_pad;
      const uint64_t dims[4] = {(uint64_t)a.Cout, (uint64_t)Wo2, (uint64_t)Ho2, (uint64_t)a.B};
      const uint64_t str[3] = {(uint64_t)a.Cout * es, (uint64_t)Wo2 * a.Cout * es,
                               (uint64_t)Ho2 * Wo2 * a.Cout * es};
      make_map(&q.tmOut, 2, 4, a.out, dims, str, box);
      q.out_pad = a.out_pad;
    }
    q.num_kb = p.num_kb, q.kb_main = kb_main, q.ntaps = p.ntaps, q.cin_chunks = p.cin_chunks;
    q.Hout = Hout, q.Wout = Wout, q.TH = TH, q.TN = TN, q.Bimg = a.B;
    for (int i = 0; i < 12; ++i) q.taps[i] = p.taps[i];
    q.tiles_m = grid.x, q.tiles_n = grid.y;
    q.N = a.Cout;
    q.bias = a.bias, q.res = a.res, q.ldr = a.Cout, q.res_after_act = a.res_after_act, q.act = a.act;
    static const bool use_pairs = getenv("CADRE_NO_CTA_PAIRS") == nullptr;  // cta_group::2 pairs (A/B switch)
    if (bn == 64)
      launch_persist<64, 6, MODE_CONV>(q, stream);
    else if (bn == 128) {
      if (use_pairs) {
        make_operand_map(&q.tmB, 2, false, a.w, Ktot, 0, a.Cout, Ktot, 1, 64);  // half-tile B boxes
        launch_persist2<128, 6, MODE_CONV>(q, stream);
      } else {
        launch_persist<128, 5, MODE_CONV>(q, stream);
      }
    } else {
      if (use_pairs) {
        make_operand_map(&q.tmB, 2, false, a.w, Ktot, 0, a.Cout, Ktot, 1, 128);
        launch_persist2<256, 4, MODE_CONV>(q, stream);
      } else {
        launch_persist<256, 3, MODE_CONV>(q, stream);  // 128x256 tiles: half the A-operand smem traffic per FLOP
      }
    }
    return;
  }
}

// ---------------------------------------------------------------------------------------------------------
void launch_flat3x3(const FlatArgs& a, cudaStream_t stream) {
  CADRE_REQUIRE(a.W + 2 <= 67, "flat3x3 window is sized for W <= 65");
  FlatParams p;
  memset(&p, 0, sizeof(p));
  const int PW = a.W + 2;
  const long long P = static_cast<long long>(a.B) * (a.H + 2) * PW;
  CADRE_REQUIRE(P < (1LL << 31) - 1024, "flat3x3: too many pixels");
  const uint64_t dims[2] = {64, (uint64_t)P};
  const uint64_t str[1] = {128};
  const uint32_t box_a[2] = {64, (uint32_t)FLAT_WIN_A}, box_b[2] = {64, 128};
  make_map(&p.tmX, 2, 2, a.in, dims, str, box_a);
  make_map(&p.tmX2, 2, 2, a.in, dims, str, box_b);
  make_map(&p.tmY, 2, 2, a.out, dims, str, box_b);
  if (a.res) make_map(&p.tmR, 2, 2, a.res, dims, str, box_b);
  const uint64_t wdims[2] = {576, 64};
  const uint64_t wstr[1] = {576 * 2};
  const uint32_t wbox[2] = {64, 64};
  make_map(&p.tmW, 2, 2, a.w, wdims, wstr, wbox);
  p.P = static_cast<int>(P), p.H = a.H, p.W = a.W, p.PW = PW;
  p.num_tiles = static_cast<int>((P + 127) / 128);
  p.bias = a.bias, p.res = a.res, p.act = a.act;
  p.dbg = g_dbg_clk ? g_dbg_clk + (a.res ? 2 : 1) * 148 * 16 : nullptr;  // region 0: stem, 1: conv, 2: conv + residual
  static size_t configured[CADRE_MAX_DEVICES] = {};   // per instantiation and device
  ensure_dynamic_smem(tc_flat3x3_kernel, FLAT_SMEM, configured);
  const int grid = p.num_tiles < num_sms() ? p.num_tiles : num_sms();
  launch_k(tc_flat3x3_kernel, dim3(grid), dim3(320), FLAT_SMEM, stream, p);
  CADRE_CUDA_CHECK(cudaGetLastError());
}

// Halo-reuse 3x3/s1/p1 128 -> 128 convolution on zero-bordered activations [B][H+2][W+2][128] (tc_halo128.cuh)
void launch_halo128(const FlatArgs& a, cudaStream_t stream) {
  CADRE_REQUIRE(2 * (a.W + 2) + 2 + 256 <= HALO_WIN_ROWS, "halo128 window is sized for W <= 33");
  Halo128Params p;
  memset(&p, 0, sizeof(p));
  const int PW = a.W + 2;
  const long long P = static_cast<long long>(a.B) * (a.H + 2) * PW;
  CADRE_REQUIRE(P < (1LL << 31) - 1024, "halo128: too many pixels");
  const uint64_t dims[2] = {128, (uint64_t)P};
  const uint64_t str[1] = {256};
  const uint32_t box_a[2] = {64, (uint32_t)HALO_WIN_A}, box_b[2] = {64, 128};
  make_map(&p.tmXa, 2, 2, a.in, dims, str, box_a);
  make_map(&p.tmXb, 2, 2, a.in, dims, str, box_b);
  make_map(&p.tmY, 2, 2, a.out, dims, str, box_b);
  if (a.res) make_map(&p.tmR, 2, 2, a.res, dims, str, box_b);
  const uint64_t wdims[2] = {1152, 128};
  const uint64_t wstr[1] = {1152 * 2};
  const uint32_t wbox[2] = {64, 64};
  make_map(&p.tmW, 2, 2, a.w, wdims, wstr, wbox);
  p.P = static_cast<int>(P), p.H = a.H, p.W = a.W, p.PW = PW;
  p.num_tiles = static_cast<int>((P + 127) / 128);
  p.num_groups = (p.num_tiles + 1) / 2;
  p.num_pairs = (p.num_groups + 1) / 2;
  p.bias = a.bias, p.res = a.res, p.act = a.act;
  static size_t configured[CADRE_MAX_DEVICES] = {};   // per instantiation and device
  ensure_dynamic_smem(tc_halo128_kernel, HALO_SMEM, configured);
  int clusters = num_sms() / 2;
  if (p.num_pairs < clusters) clusters = p.num_pairs;
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof(cfg));
  cfg.gridDim = dim3(2 * clusters), cfg.blockDim = dim3(320), cfg.dynamicSmemBytes = HALO_SMEM, cfg.stream = stream;
  cudaLaunchAttribute attr[2];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = 2, attr[0].val.clusterDim.y = 1, attr[0].val.clusterDim.z = 1;
  attr[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[1].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr, cfg.numAttrs = pdl_enabled() ? 2 : 1;
  CADRE_CUDA_CHECK(cudaLaunchKernelEx(&cfg, tc_halo128_kernel, p));
  CADRE_CUDA_CHECK(cudaGetLastError());
}

// ---------------------------------------------------------------------------------------------------------
// Input layout of the stem (written by the preprocess kernel): row-pair interleaved, padded by 3 pixels on every
// side: P[n][y2 = 0..74][x = 0..261][r = 0..1][c = 0..3] (padded row 2*y2 + r), 16 bytes per (y2, x). Output pixel
// (oh, ow), filter-row pair j (kh = 2j, 2j+1) reads P[n][oh + j][2ow .. 2ow+7] = 128 contiguous bytes, so k-block j of
// the implicit GEMM is one 4-D TMA box whose ow-stride (32 B) overlaps its rows.
void launch_stem_pool(const StemArgs& a, cudaStream_t stream) {
  StemPoolParams p;
  memset(&p, 0, sizeof(p));
  const uint64_t pitch = 262 * 16;
  const uint64_t dims[4] = {64, 128, 75, (uint64_t)a.B};
  const uint64_t str[3] = {32, pitch, 75 * pitch};
  const uint32_t box[4] = {64, 128, 1, 1};
  make_map(&p.tmX, 2, 4, a.in, dims, str, box);
  const uint64_t wdims[2] = {256, 64};
  const uint64_t wstr[1] = {256 * 2};
  const uint32_t wbox[2] = {64, 64};
  make_map(&p.tmW, 2, 2, a.w, wdims, wstr, wbox);
  p.bias = a.bias, p.out = a.out, p.B = a.B;
  p.pool_rows = 12;
  p.num_units = a.B * (36 / p.pool_rows);
  p.dbg = g_dbg_clk;
  static size_t configured[CADRE_MAX_DEVICES] = {};   // per instantiation and device
  ensure_dynamic_smem(tc_stem_pool_kernel, SP_SMEM, configured);
  const int grid = p.num_units < num_sms() ? p.num_units : num_sms();
  launch_k(tc_stem_pool_kernel, dim3(grid), dim3(320), SP_SMEM, stream, p);
  CADRE_CUDA_CHECK(cudaGetLastError());
}

}  // namespace cadre

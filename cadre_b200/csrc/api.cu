// extern "C" boundary of libcadre_sm100.so (declared in include/cadre_b200.h).
#include "../../include/cadre_b200.h"

#include "internal.h"

#include <cstdlib>
#include <cstring>

namespace cadre {
static thread_local std::string g_last_error;
void set_last_error(const std::string& msg) { g_last_error = msg; }
}  // namespace cadre

#define CADRE_API_BEGIN try {
#define CADRE_API_END                                    \
  }                                                      \
  catch (const cadre::Error& e) {                        \
    cadre::set_last_error(e.what());                     \
    return e.code;                                       \
  }                                                      \
  catch (const std::exception& e) {                      \
    cadre::set_last_error(e.what());                     \
    return 99;                                           \
  }                                                      \
  return 0;

extern "C" {

const char* cadre_last_error(void) { return cadre::g_last_error.c_str(); }
const char* cadre_version(void) { return "cadre_b200 sm_100a " __DATE__; }
int cadre_enc_dtype(void) { return CADRE_ENC_FP16 ? 1 : 0; }

int cadre_memcpy_d2d(void* dst, const void* src, int64_t nbytes, void* stream) {
  CADRE_API_BEGIN
  CADRE_CUDA_CHECK(cudaMemcpyAsync(dst, src, nbytes, cudaMemcpyDeviceToDevice, static_cast<cudaStream_t>(stream)));
  CADRE_API_END
}

int cadre_gemm(const cadre_gemm_args* s, void* stream) {
  CADRE_API_BEGIN
  CADRE_REQUIRE(s != nullptr, "args");
  cadre::GemmArgs a;
  a.kind = s->kind, a.a_mn = s->a_mn, a.b_mn = s->b_mn, a.batch = s->batch;
  a.M = s->M, a.N = s->N, a.K = s->K, a.block_n = s->block_n;
  a.A = s->A, a.B = s->B, a.lda = s->lda, a.a_bs = s->a_bs, a.ldb = s->ldb, a.b_bs = s->b_bs;
  a.out = s->out, a.ldc = s->ldc, a.out_bs = s->out_bs, a.out_f32 = s->out_f32, a.act = s->act;
  a.bias = s->bias, a.bias_bs = s->bias_bs;
  a.res = s->res, a.ldr = s->ldr, a.res_bs = s->res_bs, a.res_after_act = s->res_after_act;
  a.mask = s->mask, a.ldm = s->ldm, a.mask_bs = s->mask_bs;
  a.batch_rows = s->batch_rows, a.rows_is_k = s->rows_is_k;
  a.alpha = s->alpha, a.epi = s->epi;
  if (getenv("CADRE_DBG_CLK")) a.dbg_clk = reinterpret_cast<long long*>(strtoull(getenv("CADRE_DBG_CLK"), nullptr, 0));
  if (getenv("CADRE_DBG_EPI")) a.dbg_epi = atoi(getenv("CADRE_DBG_EPI"));
  if (getenv("CADRE_DBG_A_SHIFT")) a.dbg_a_shift = atoi(getenv("CADRE_DBG_A_SHIFT"));
  if (getenv("CADRE_DBG_BASE_OFFSET")) a.dbg_base_offset = atoi(getenv("CADRE_DBG_BASE_OFFSET"));
  a.xpart = s->xpart, a.c_prev = s->c_prev, a.c_out = s->c_out, a.h_out = s->h_out;
  a.gates_out = s->gates_out, a.ldx = s->ldx, a.x_bs = s->x_bs, a.ldh = s->ldh, a.h_bs = s->h_bs;
  cadre::launch_gemm(a, static_cast<cudaStream_t>(stream));
  CADRE_API_END
}

int cadre_conv2d_nhwc(const void* in, int B, int Hin, int Win, int Cin, const void* w, int Cout, int KH,
                      int KW, int stride, int pad, const float* bias, const void* res, int res_after_act,
                      int act, void* out, int in_pad, void* stream) {
  CADRE_API_BEGIN
  cadre::ConvArgs a;
  a.in_pad = in_pad;
  a.in = static_cast<const cadre::enc_t*>(in);
  a.B = B, a.Hin = Hin, a.Win = Win, a.Cin = Cin;
  a.w = static_cast<const cadre::enc_t*>(w);
  a.Cout = Cout, a.KH = KH, a.KW = KW, a.stride = stride, a.pad = pad;
  a.bias = bias, a.res = static_cast<const cadre::enc_t*>(res), a.res_after_act = res_after_act;
  a.act = act, a.out = static_cast<cadre::enc_t*>(out);
  cadre::launch_conv(a, static_cast<cudaStream_t>(stream));
  CADRE_API_END
}

int cadre_debug_clk(long long* dev_counters) {
  cadre::g_dbg_clk = dev_counters;
  cadre::g_dbg_persist_launch = 0;
  return 0;
}

int cadre_conv3x3_flat64(const void* in, int B, int H, int W, const void* w, const float* bias, const void* res,
                         int act, void* out, void* stream) {
  CADRE_API_BEGIN
  cadre::FlatArgs a;
  a.in = static_cast<const cadre::enc_t*>(in), a.B = B, a.H = H, a.W = W;
  a.w = static_cast<const cadre::enc_t*>(w), a.bias = bias, a.res = static_cast<const cadre::enc_t*>(res);
  a.act = act, a.out = static_cast<cadre::enc_t*>(out);
  cadre::launch_flat3x3(a, static_cast<cudaStream_t>(stream));
  CADRE_API_END
}

int cadre_conv3x3_flat128(const void* in, int B, int H, int W, const void* w, const float* bias, const void* res,
                          int act, void* out, void* stream) {
  CADRE_API_BEGIN
  cadre::FlatArgs a;
  a.in = static_cast<const cadre::enc_t*>(in), a.B = B, a.H = H, a.W = W;
  a.w = static_cast<const cadre::enc_t*>(w), a.bias = bias, a.res = static_cast<const cadre::enc_t*>(res);
  a.act = act, a.out = static_cast<cadre::enc_t*>(out);
  cadre::launch_halo128(a, static_cast<cudaStream_t>(stream));
  CADRE_API_END
}

int cadre_conv2d_nhwc_bordered_out(const void* in, int B, int Hin, int Win, int Cin, const void* w, int Cout, int KH,
                                   int KW, int stride, int pad, const float* bias, int act, void* out, int in_pad,
                                   void* stream) {
  CADRE_API_BEGIN
  cadre::ConvArgs a;
  a.in_pad = in_pad, a.out_pad = 1;
  a.in = static_cast<const cadre::enc_t*>(in);
  a.B = B, a.Hin = Hin, a.Win = Win, a.Cin = Cin;
  a.w = static_cast<const cadre::enc_t*>(w);
  a.Cout = Cout, a.KH = KH, a.KW = KW, a.stride = stride, a.pad = pad;
  a.bias = bias, a.act = act, a.out = static_cast<cadre::enc_t*>(out);
  cadre::launch_conv(a, static_cast<cudaStream_t>(stream));
  CADRE_API_END
}

int cadre_conv2d_nhwc_shortcut(const void* in, int B, int Hin, int Win, int Cin, const void* w, int Cout, int KH, int KW,
                               int pad, const float* bias, int act, void* out, int in_pad, int out_pad, const void* in2,
                               int Cin2, int Hin2, int Win2, int in2_pad, void* stream) {
  CADRE_API_BEGIN
  CADRE_REQUIRE(in2 != nullptr, "conv2d_nhwc_shortcut needs the shortcut input");
  cadre::ConvArgs a;
  a.in_pad = in_pad, a.out_pad = out_pad;
  a.in = static_cast<const cadre::enc_t*>(in);
  a.B = B, a.Hin = Hin, a.Win = Win, a.Cin = Cin;
  a.w = static_cast<const cadre::enc_t*>(w);
  a.Cout = Cout, a.KH = KH, a.KW = KW, a.stride = 1, a.pad = pad;
  a.bias = bias, a.act = act, a.out = static_cast<cadre::enc_t*>(out);
  a.in2 = static_cast<const cadre::enc_t*>(in2), a.Cin2 = Cin2, a.in2_pad = in2_pad, a.Hin2 = Hin2, a.Win2 = Win2;
  cadre::launch_conv(a, static_cast<cudaStream_t>(stream));
  CADRE_API_END
}

int cadre_stem_pool(const void* in, int B, const void* w, const float* bias, void* out, void* stream) {
  CADRE_API_BEGIN
  CADRE_REQUIRE(in && w && bias && out && B > 0, "stem_pool arguments");
  cadre::StemArgs a;
  a.in = static_cast<const cadre::enc_t*>(in), a.B = B;
  a.w = static_cast<const cadre::enc_t*>(w), a.bias = bias, a.out = static_cast<cadre::enc_t*>(out);
  cadre::launch_stem_pool(a, static_cast<cudaStream_t>(stream));
  CADRE_API_END
}

}  // extern "C"

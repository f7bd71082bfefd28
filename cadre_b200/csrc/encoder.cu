// Perception encoder forward plan: DANet.get_latent_feature (carla_perception/Networks/danet.py:216-238) as a
// fixed sequence of kernel launches over NHWC bf16 activations held in library-owned HBM workspaces.
//   ingest -> stem + ReLU + maxpool (one tcgen05 kernel) -> 8 BasicBlocks (tcgen05 implicit GEMM, BN folded, residual + ReLU in
//   the epilogue) -> conv5a|conv5c as one N=256 conv -> fused PAM / fused CAM -> conv51, conv52 (+sum) ->
//   [conv8 o visual/bc 1x1 o Linear(20480,512)] folded into one [B,5120]x[5120,3072] GEMM + LeakyReLU ->
//   six Linear(512,256) as one batched GEMM -> inter-task attention (+ measurement concat).
#include "../../include/cadre_b200.h"
#include "internal.h"

#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

namespace cadre {

void launch_f32_to_enc(const float* in, enc_t* out, int n, cudaStream_t stream);
void launch_preprocess(const uint8_t* rgb, const uint8_t* route, uint8_t* route_max_ws, const enc_t* lut, enc_t* out,
                       int B, cudaStream_t stream);
void launch_pack_f32(const float* x, enc_t* out, int B, cudaStream_t stream);
static_assert(CADRE_ENC_FP16 == 1, "the fused PAM / CAM kernels are written for IEEE fp16 operands");
void launch_pam_mma(const enc_t* x, enc_t* out, const float* wqk, const float* bqk, const enc_t* wv, const float* bv,
                    float gamma, int B, int ldin, int num_sms, cudaStream_t stream);
void launch_cam(const enc_t* x, enc_t* out, float gamma, int B, int ldin, int num_sms,
                cudaStream_t stream);
void launch_intertask(const float* qkv, float* out, const double* meas, int B, int ld_out,
                      cudaStream_t stream);

struct Encoder {
  cadre_encoder_weights w;
  int max_batch = 0;
  int num_sms = 148;
  // workspaces (device)
  enc_t* padded = nullptr;   // [Bmax][75][262][8]
  enc_t* act[4] = {nullptr, nullptr, nullptr, nullptr};  // ping-pong, each [Bmax][36*64*64]
  enc_t* padact[3] = {nullptr, nullptr, nullptr};        // zero-bordered layer1 activations [Bmax][38][66][64]
  // layer2 on zero-bordered activations [Bmax][20][34][128]: its two plain 3x3 convs (layer2.1) run on the halo-reuse
  // kernel (tc_halo128.cuh), layer2.0's launches write bordered outputs for them
  bool halo2 = false;
  enc_t* pad2[3] = {nullptr, nullptr, nullptr};
  // fused shortcuts (layer2.0 / 3.0 / 4.0): conv2 weights with the 1x1 downsample appended along K, summed bias
  bool fuse_ds = true;
  enc_t* fused_w[3] = {nullptr, nullptr, nullptr};
  float* fused_b[3] = {nullptr, nullptr, nullptr};
  enc_t* head5 = nullptr;    // [Bmax][40][256]
  enc_t* sa = nullptr;       // [Bmax][40][128]
  enc_t* sc = nullptr;
  enc_t* sa_conv = nullptr;
  enc_t* feat_sum = nullptr;
  enc_t* fc1 = nullptr;      // [Bmax][3072]
  float* qkv = nullptr;              // [6][Bmax][256]
  uint8_t* route_max = nullptr;      // [Bmax]
  enc_t* lut255 = nullptr;           // k / 255 for k = 0..255, rounded like np.array(rgb / 255., dtype=float32)
  enc_t* l4 = nullptr;       // alias of the act buffer holding layer4's output after a forward
  int launches_per_forward = 0;
  // optional per-launch timing (cadre_encoder_profile)
  bool prof = false;
  cudaEvent_t ev[64];
  std::vector<std::string> names;
};

static inline void step(Encoder* e, cudaStream_t s, int& n, const char* name) {
  ++n;
  if (e->prof) {
    cudaEventRecord(e->ev[n], s);
    e->names.push_back(name);
  }
}

template <typename T>
static T* dev_alloc(size_t n, bool zero) {
  T* p = nullptr;
  CADRE_CUDA_CHECK(cudaMalloc(&p, n * sizeof(T)));
  if (zero) CADRE_CUDA_CHECK(cudaMemset(p, 0, n * sizeof(T)));
  return p;
}

static Encoder* encoder_create(const cadre_encoder_weights* w, int max_batch) {
  CADRE_REQUIRE(w != nullptr && max_batch > 0, "encoder_create arguments");
  Encoder* e = new Encoder();
  e->w = *w;
  e->max_batch = max_batch;
  int dev = 0;
  CADRE_CUDA_CHECK(cudaGetDevice(&dev));
  CADRE_CUDA_CHECK(cudaDeviceGetAttribute(&e->num_sms, cudaDevAttrMultiProcessorCount, dev));
  const size_t B = max_batch;
  e->padded = dev_alloc<enc_t>(B * 75 * 262 * 8, true);  // zero borders = conv padding
  for (int i = 0; i < 4; ++i) e->act[i] = dev_alloc<enc_t>(B * 36 * 64 * 64, false);
  for (int i = 0; i < 3; ++i) e->padact[i] = dev_alloc<enc_t>(B * 38 * 66 * 64, true);  // borders stay zero
  e->fuse_ds = getenv("CADRE_NO_SHORTCUT_FUSION") == nullptr;   // A/B switch kept for the fused-shortcut parity test
  // default on; CADRE_LAYER2_HALO=0 keeps layer2 on the implicit-GEMM kernel (A/B switch, read when the encoder is created)
  e->halo2 = e->fuse_ds && !(getenv("CADRE_LAYER2_HALO") != nullptr && atoi(getenv("CADRE_LAYER2_HALO")) == 0);
  if (e->halo2)
    for (int i = 0; i < 3; ++i) e->pad2[i] = dev_alloc<enc_t>(B * 20 * 34 * 128, true);  // borders stay zero
  if (e->fuse_ds) {
    // conv indices follow execution order: layer1 = 0..3, then per stage (conv1, conv2, downsample, conv1, conv2)
    const int planes[4] = {64, 128, 256, 512};
    for (int li = 1; li < 4; ++li) {
      const int conv2_idx = 4 + (li - 1) * 5 + 1, ds_idx = conv2_idx + 1;
      const int Cout = planes[li], Cin = planes[li - 1], K2 = 9 * Cout, Kf = K2 + Cin;
      enc_t* wf = dev_alloc<enc_t>(static_cast<size_t>(Cout) * Kf, false);
      CADRE_CUDA_CHECK(cudaMemcpy2D(wf, Kf * sizeof(enc_t), w->conv_w[conv2_idx], K2 * sizeof(enc_t),
                                    K2 * sizeof(enc_t), Cout, cudaMemcpyDeviceToDevice));
      CADRE_CUDA_CHECK(cudaMemcpy2D(wf + K2, Kf * sizeof(enc_t), w->conv_w[ds_idx], Cin * sizeof(enc_t),
                                    Cin * sizeof(enc_t), Cout, cudaMemcpyDeviceToDevice));
      std::vector<float> b2(Cout), bd(Cout);
      CADRE_CUDA_CHECK(cudaMemcpy(b2.data(), w->conv_b[conv2_idx], Cout * sizeof(float), cudaMemcpyDeviceToHost));
      CADRE_CUDA_CHECK(cudaMemcpy(bd.data(), w->conv_b[ds_idx], Cout * sizeof(float), cudaMemcpyDeviceToHost));
      for (int i = 0; i < Cout; ++i) b2[i] += bd[i];
      float* bf = dev_alloc<float>(Cout, false);
      CADRE_CUDA_CHECK(cudaMemcpy(bf, b2.data(), Cout * sizeof(float), cudaMemcpyHostToDevice));
      e->fused_w[li - 1] = wf, e->fused_b[li - 1] = bf;
    }
  }
  e->head5 = dev_alloc<enc_t>(B * 40 * 256, false);
  e->sa = dev_alloc<enc_t>(B * 40 * 128, false);
  e->sc = dev_alloc<enc_t>(B * 40 * 128, false);
  e->sa_conv = dev_alloc<enc_t>(B * 40 * 128, false);
  e->feat_sum = dev_alloc<enc_t>(B * 40 * 128, false);
  e->fc1 = dev_alloc<enc_t>(B * 3072, false);
  e->qkv = dev_alloc<float>(6 * B * 256, false);
  e->route_max = dev_alloc<uint8_t>(B, true);
  {
    // agent.py:46: float64 division, cast to float32 (then to the 16-bit operand type of the stem)
    std::vector<float> lf(256);
    for (int k = 0; k < 256; ++k) lf[k] = static_cast<float>(k / 255.0);
    float* tmp = dev_alloc<float>(256, false);
    CADRE_CUDA_CHECK(cudaMemcpy(tmp, lf.data(), 256 * sizeof(float), cudaMemcpyHostToDevice));
    e->lut255 = dev_alloc<enc_t>(256, false);
    launch_f32_to_enc(tmp, e->lut255, 256, 0);
    CADRE_CUDA_CHECK(cudaDeviceSynchronize());
    cudaFree(tmp);
  }
  return e;
}

static void encoder_destroy(Encoder* e) {
  if (!e) return;
  cudaFree(e->padded);
  for (int i = 0; i < 4; ++i) cudaFree(e->act[i]);
  for (int i = 0; i < 3; ++i) cudaFree(e->padact[i]);
  for (int i = 0; i < 3; ++i) cudaFree(e->pad2[i]);
  cudaFree(e->head5), cudaFree(e->sa), cudaFree(e->sc), cudaFree(e->sa_conv), cudaFree(e->feat_sum);
  cudaFree(e->fc1), cudaFree(e->qkv), cudaFree(e->route_max), cudaFree(e->lut255);
  for (int i = 0; i < 3; ++i) cudaFree(e->fused_w[i]), cudaFree(e->fused_b[i]);
  delete e;
}

static void conv(Encoder* e, int idx, const enc_t* in, int B, int H, int W, int Cin, int Cout, int k,
                 int stride, int pad, const enc_t* res, int act, enc_t* out,
                 cudaStream_t s, bool in_pad = false, bool out_pad = false) {
  ConvArgs a;
  a.in_pad = in_pad ? 1 : 0;
  a.out_pad = out_pad ? 1 : 0;
  a.in = in, a.B = B, a.Hin = H, a.Win = W, a.Cin = Cin;
  a.w = static_cast<const enc_t*>(e->w.conv_w[idx]);
  a.bias = e->w.conv_b[idx];
  a.Cout = Cout, a.KH = k, a.KW = k, a.stride = stride, a.pad = pad;
  a.res = res, a.act = act, a.out = out;
  launch_conv(a, s);
}

// everything after the ingest kernel; `B` frames already sit in e->padded
static void encoder_trunk(Encoder* e, int B, const double* meas, float* out, int ld_out, cudaStream_t s) {
  int n = 0;
  if (e->prof) {
    e->names.clear();
    cudaEventRecord(e->ev[0], s);
  }
  StemArgs st;
  st.in = e->padded, st.B = B, st.w = static_cast<const enc_t*>(e->w.stem_w), st.bias = e->w.stem_b;
  st.out = e->padact[0];   // the pooled map lands in layer1's zero-bordered input; the stem activation never reaches HBM
  launch_stem_pool(st, s), step(e, s, n, "stem+pool");

  // ResNet-18 BasicBlocks (resnet.py:39-55, 116-119); conv indices follow execution order
  int cur = 0, ci = 0, H = 36, W = 64, C = 64;
  const int planes[4] = {64, 128, 256, 512};
  const enc_t* padded_in = nullptr;  // layer1 output in zero-bordered layout (input of layer2.0)
  {
    // layer1 (4 convs 64->64, 3x3/s1) through the halo-reuse kernel on zero-bordered buffers
    enc_t* x = e->padact[0];
    enc_t* t = e->padact[1];
    enc_t* o = e->padact[2];
    for (int bi = 0; bi < 2; ++bi) {
      FlatArgs f;
      f.B = B, f.H = 36, f.W = 64, f.act = 1;
      f.in = x, f.w = static_cast<const enc_t*>(e->w.conv_w[ci]), f.bias = e->w.conv_b[ci], f.out = t;
      launch_flat3x3(f, s), ++ci;
      step(e, s, n, (std::string("layer1.") + std::to_string(bi) + ".conv1").c_str());
      f.in = t, f.w = static_cast<const enc_t*>(e->w.conv_w[ci]), f.bias = e->w.conv_b[ci], f.out = o, f.res = x;
      launch_flat3x3(f, s), ++ci;
      step(e, s, n, (std::string("layer1.") + std::to_string(bi) + ".conv2").c_str());
      enc_t* tmp = x;
      x = o, o = tmp;
    }
    padded_in = x;
  }
  for (int li = 1; li < 4; ++li) {
    if (li == 1 && e->halo2) {
      // layer2 on zero-bordered buffers: 2.0.conv1 (3x3/s2) and 2.0.conv2 + shortcut on the implicit-GEMM kernel with
      // bordered outputs, 2.1.conv1 / 2.1.conv2 (plain 3x3/s1, 128 -> 128) on the halo-reuse kernel
      enc_t* t0 = e->pad2[0];
      enc_t* y0 = e->pad2[1];
      enc_t* t1 = e->pad2[2];
      conv(e, ci++, padded_in, B, 36, 64, 64, 128, 3, 2, 1, nullptr, 1, t0, s, true, true);
      step(e, s, n, "layer2.0.conv1");
      {
        ++ci, ++ci;   // conv2 and the downsample conv are folded into fused_w[0]
        ConvArgs a;
        a.in = t0, a.in_pad = 1, a.B = B, a.Hin = 18, a.Win = 32, a.Cin = 128;
        a.w = e->fused_w[0], a.bias = e->fused_b[0];
        a.Cout = 128, a.KH = 3, a.KW = 3, a.stride = 1, a.pad = 1;
        a.act = 1, a.out = y0, a.out_pad = 1;
        a.in2 = padded_in, a.Cin2 = 64, a.in2_pad = 1, a.Hin2 = 36, a.Win2 = 64;
        launch_conv(a, s);
        step(e, s, n, "layer2.0.conv2+shortcut");
      }
      FlatArgs f;
      f.B = B, f.H = 18, f.W = 32, f.act = 1;
      f.in = y0, f.w = static_cast<const enc_t*>(e->w.conv_w[ci]), f.bias = e->w.conv_b[ci], f.out = t1;
      launch_halo128(f, s), ++ci;
      step(e, s, n, "layer2.1.conv1");
      f.in = t1, f.w = static_cast<const enc_t*>(e->w.conv_w[ci]), f.bias = e->w.conv_b[ci], f.out = t0, f.res = y0;
      launch_halo128(f, s), ++ci;
      step(e, s, n, "layer2.1.conv2");
      padded_in = t0;
      H = 18, W = 32, C = 128;
      continue;
    }
    for (int bi = 0; bi < 2; ++bi) {
      const int stride = (li > 0 && bi == 0) ? 2 : 1;
      const int Cout = planes[li];
      const int Ho = (H + 2 - 3) / stride + 1, Wo = (W + 2 - 3) / stride + 1;
      const bool from_pad = (padded_in != nullptr && bi == 0 && (li == 1 || (li == 2 && e->halo2)));
      const enc_t* x = from_pad ? padded_in : e->act[cur];
      enc_t* t = e->act[(cur + 1) & 3];
      enc_t* ds = e->act[(cur + 2) & 3];
      enc_t* o = e->act[(cur + 3) & 3];
      conv(e, ci++, x, B, H, W, C, Cout, 3, stride, 1, nullptr, 1, t, s, from_pad);
      step(e, s, n, (std::string("layer") + std::to_string(li + 1) + "." + std::to_string(bi) + ".conv1").c_str());
      const enc_t* idn = x;
      const int conv2_idx = ci++;
      if (stride == 2 && e->fuse_ds) {
        // BasicBlock with downsample (resnet.py:47-53): relu(bn2(conv2(t)) + bn_d(conv1x1_s2(x))) as ONE
        // implicit GEMM: the shortcut is Cin/64 extra k-blocks reading x on its stride-2 sub-lattice
        ++ci;
        ConvArgs a;
        a.in = t, a.B = B, a.Hin = Ho, a.Win = Wo, a.Cin = Cout;
        a.w = e->fused_w[li - 1], a.bias = e->fused_b[li - 1];
        a.Cout = Cout, a.KH = 3, a.KW = 3, a.stride = 1, a.pad = 1;
        a.act = 1, a.out = o;
        a.in2 = x, a.Cin2 = C, a.in2_pad = from_pad ? 1 : 0, a.Hin2 = H, a.Win2 = W;
        launch_conv(a, s);
        step(e, s, n, (std::string("layer") + std::to_string(li + 1) + ".0.conv2+shortcut").c_str());
        cur = (cur + 3) & 3;
        H = Ho, W = Wo, C = Cout;
        continue;
      }
      if (stride == 2) {
        conv(e, ci++, x, B, H, W, C, Cout, 1, 2, 0, nullptr, 0, ds, s, from_pad);
        step(e, s, n, (std::string("layer") + std::to_string(li + 1) + ".0.downsample").c_str());
        idn = ds;
      }
      conv(e, conv2_idx, t, B, Ho, Wo, Cout, Cout, 3, 1, 1, idn, 1, o, s);
      step(e, s, n, (std::string("layer") + std::to_string(li + 1) + "." + std::to_string(bi) + ".conv2").c_str());
      cur = (cur + 3) & 3;
      H = Ho, W = Wo, C = Cout;
    }
  }
  e->l4 = e->act[cur];

  // DANetHead (danet.py:43-69)
  {
    ConvArgs a;
    a.in = e->l4, a.B = B, a.Hin = 5, a.Win = 8, a.Cin = 512;
    a.w = static_cast<const enc_t*>(e->w.head5_w), a.bias = e->w.head5_b;
    a.Cout = 256, a.KH = 3, a.KW = 3, a.stride = 1, a.pad = 1, a.act = 1, a.out = e->head5;
    launch_conv(a, s), step(e, s, n, "conv5a|conv5c");
  }
  launch_pam_mma(e->head5, e->sa, e->w.pam_wqk, e->w.pam_bqk, static_cast<const enc_t*>(e->w.pam_wv), e->w.pam_bv,
                 e->w.pam_gamma, B, 256, e->num_sms, s);
  step(e, s, n, "pam (value conv fused)");
  launch_cam(e->head5 + 128, e->sc, e->w.cam_gamma, B, 256, e->num_sms, s), step(e, s, n, "cam");
  {
    ConvArgs a;
    a.in = e->sa, a.B = B, a.Hin = 5, a.Win = 8, a.Cin = 128;
    a.w = static_cast<const enc_t*>(e->w.conv51_w), a.bias = e->w.conv51_b;
    a.Cout = 128, a.KH = 3, a.KW = 3, a.stride = 1, a.pad = 1, a.act = 1, a.out = e->sa_conv;
    launch_conv(a, s), step(e, s, n, "conv51");
    a.in = e->sc;
    a.w = static_cast<const enc_t*>(e->w.conv52_w), a.bias = e->w.conv52_b;
    a.res = e->sa_conv, a.res_after_act = 1, a.out = e->feat_sum;  // feat_sum = relu(conv52) + sa_conv
    launch_conv(a, s), step(e, s, n, "conv52+sum");
  }
  // conv8 -> {visual_conv, bc_conv} -> six Linear(20480,512): all linear, folded offline into fc1 (K = 40*128)
  {
    GemmArgs g;
    g.kind = 0, g.A = e->feat_sum, g.lda = 5120, g.B = e->w.fc1_w, g.ldb = 5120;
    g.M = B, g.N = 3072, g.K = 5120;
    g.out = e->fc1, g.ldc = 3072, g.out_f32 = 0, g.bias = e->w.fc1_b, g.act = 2;
    launch_gemm(g, s), step(e, s, n, "fc1(folded)");
  }
  {
    GemmArgs g;
    g.kind = 0, g.batch = 6;
    g.A = e->fc1, g.lda = 3072, g.a_bs = 512;
    g.B = e->w.fc2_w, g.ldb = 512, g.b_bs = 256 * 512;
    g.M = B, g.N = 256, g.K = 512;
    g.out = e->qkv, g.ldc = 256, g.out_bs = static_cast<long long>(B) * 256, g.out_f32 = 1;
    g.bias = e->w.fc2_b, g.bias_bs = 256;
    launch_gemm(g, s), step(e, s, n, "fc2");
  }
  launch_intertask(e->qkv, out, meas, B, ld_out, s), step(e, s, n, "intertask");
  e->launches_per_forward = n + 2;
}

}  // namespace cadre

using cadre::Encoder;

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

int cadre_encoder_create(void** handle, const cadre_encoder_weights* w, int max_batch) {
  CADRE_API_BEGIN
  CADRE_REQUIRE(handle != nullptr, "handle");
  *handle = cadre::encoder_create(w, max_batch);
  CADRE_API_END
}

int cadre_encoder_destroy(void* handle) {
  CADRE_API_BEGIN
  cadre::encoder_destroy(static_cast<Encoder*>(handle));
  CADRE_API_END
}

int cadre_encoder_forward_u8(void* handle, const uint8_t* rgb, const uint8_t* route_fig,
                             const double* measurements, int B, float* out, int ld_out, void* stream) {
  CADRE_API_BEGIN
  Encoder* e = static_cast<Encoder*>(handle);
  CADRE_REQUIRE(e && rgb && route_fig && out, "encoder_forward_u8 pointers");
  CADRE_REQUIRE(B > 0 && B <= e->max_batch, "batch exceeds the encoder's max_batch");
  CADRE_REQUIRE(ld_out >= (measurements ? 530 : 512), "ld_out too small");
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  cadre::launch_preprocess(rgb, route_fig, e->route_max, e->lut255, e->padded, B, s);
  cadre::encoder_trunk(e, B, measurements, out, ld_out, s);
  CADRE_API_END
}

int cadre_encoder_forward_f32(void* handle, const float* x_nchw, int B, float* out, int ld_out, void* stream) {
  CADRE_API_BEGIN
  Encoder* e = static_cast<Encoder*>(handle);
  CADRE_REQUIRE(e && x_nchw && out, "encoder_forward_f32 pointers");
  CADRE_REQUIRE(B > 0 && B <= e->max_batch, "batch exceeds the encoder's max_batch");
  CADRE_REQUIRE(ld_out >= 512, "ld_out too small");
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  cadre::launch_pack_f32(x_nchw, e->padded, B, s);
  cadre::encoder_trunk(e, B, nullptr, out, ld_out, s);
  CADRE_API_END
}

int cadre_encoder_buffer(void* handle, int which, void** ptr, int64_t* elems_per_frame) {
  CADRE_API_BEGIN
  Encoder* e = static_cast<Encoder*>(handle);
  CADRE_REQUIRE(e && ptr && elems_per_frame, "encoder_buffer pointers");
  switch (which) {
    case 0: *ptr = e->l4, *elems_per_frame = 40 * 512; break;          // layer4 output, NHWC bf16
    case 1: *ptr = e->feat_sum, *elems_per_frame = 40 * 128; break;    // sa_conv + sc_conv, NHWC bf16
    case 2: *ptr = e->head5, *elems_per_frame = 40 * 256; break;       // conv5a|conv5c output
    case 3: *ptr = e->sa, *elems_per_frame = 40 * 128; break;          // PAM output
    case 4: *ptr = e->sc, *elems_per_frame = 40 * 128; break;          // CAM output
    case 5: *ptr = e->fc1, *elems_per_frame = 3072; break;             // six folded Linear(20480,512) + LeakyReLU
    case 6: *ptr = e->padded, *elems_per_frame = 75 * 262 * 8; break;  // ingested image, stem input layout
    default: throw cadre::Error(1, "encoder_buffer: unknown buffer id");
  }
  CADRE_API_END
}

int cadre_encoder_profile(void* handle, int B, float* out, int ld_out, float* ms_out, char* names_out,
                          int names_cap, int* n_out, void* stream) {
  CADRE_API_BEGIN
  Encoder* e = static_cast<Encoder*>(handle);
  CADRE_REQUIRE(e && out && ms_out && names_out && n_out, "encoder_profile pointers");
  CADRE_REQUIRE(B > 0 && B <= e->max_batch, "batch exceeds the encoder's max_batch");
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  for (int i = 0; i < 64; ++i) CADRE_CUDA_CHECK(cudaEventCreate(&e->ev[i]));
  e->prof = true;
  cadre::encoder_trunk(e, B, nullptr, out, ld_out, s);   // re-runs the trunk on the frames already ingested
  e->prof = false;
  CADRE_CUDA_CHECK(cudaStreamSynchronize(s));
  const int n = static_cast<int>(e->names.size());
  std::string joined;
  for (int i = 0; i < n; ++i) {
    CADRE_CUDA_CHECK(cudaEventElapsedTime(&ms_out[i], e->ev[i], e->ev[i + 1]));
    joined += e->names[i] + (i + 1 < n ? ";" : "");
  }
  for (int i = 0; i < 64; ++i) cudaEventDestroy(e->ev[i]);
  CADRE_REQUIRE(static_cast<int>(joined.size()) < names_cap, "names buffer too small");
  memcpy(names_out, joined.c_str(), joined.size() + 1);
  *n_out = n;
  CADRE_API_END
}

int cadre_encoder_launches(void* handle) {
  Encoder* e = static_cast<Encoder*>(handle);
  return e ? e->launches_per_forward : 0;
}

}  // extern "C"

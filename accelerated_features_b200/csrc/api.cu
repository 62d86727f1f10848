// C-ABI glue: context, error reporting and the backbone schedule (XFeatModel.forward, model.py:123-154).
#include <stdarg.h>

#include <map>
#include <mutex>
#include <utility>
#include <vector>

#include "common.cuh"

namespace xf {

static thread_local char g_err[1024] = "";
unsigned long long g_launches = 0;
int g_conv_impl = 2;  // 0 = fp32 CUDA-core convs everywhere, 1 = tcgen05 for the 64->64 stride-1 layers (default)

// (device, kernel) -> largest dynamic shared-memory size opted into so far
int ensure_dyn_smem(const void* func, size_t bytes) {
  static std::mutex mu;
  static std::map<std::pair<int, const void*>, size_t> done;
  int dev = 0;
  XF_CUDA(cudaGetDevice(&dev));
  std::lock_guard<std::mutex> lock(mu);
  size_t& cur = done[std::make_pair(dev, func)];
  if (bytes > cur) {
    XF_CUDA(cudaFuncSetAttribute(func, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes));
    cur = bytes;
  }
  return XF_OK;
}

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

// Activation buffers of one forward pass (NHWC fp32), carved from the caller's workspace.
struct NetWs {
  float *a1, *a2, *a3, *x1s, *t4a, *x2;       // stem + block2 (1/1, 1/2, 1/4 res)
  float *t8a, *t8b, *x3, *fin, *f1, *f2;      // 1/8 res, 64 ch
  float *t16a, *t16b, *x4;                    // 1/16 res, 64 ch
  float *t32a, *t32b, *x5;                    // 1/32 res, 128/128/64 ch
};

static void carve_net(Bump& bump, int B, int H, int W, NetWs& ws) {
  const size_t p1 = (size_t)B * H * W, p2 = p1 / 4, p4 = p1 / 16, p8 = p1 / 64, p16 = p1 / 256, p32 = p1 / 1024;
  ws.a1 = bump.take<float>(p1 * 4);
  ws.a2 = bump.take<float>(p2 * 8);
  ws.a3 = bump.take<float>(p2 * 8);
  ws.x1s = bump.take<float>(p4 * 32);   // 24 fp32 channels, or split fp16 [hi(32) | lo(32)] = 128 B per pixel
  ws.t4a = bump.take<float>(p4 * 32);
  ws.x2 = bump.take<float>(p4 * 32);
  ws.t8a = bump.take<float>(p8 * 64);
  ws.t8b = bump.take<float>(p8 * 64);
  ws.x3 = bump.take<float>(p8 * 64);
  ws.fin = bump.take<float>(p8 * 64);
  ws.f1 = bump.take<float>(p8 * 64);
  ws.f2 = bump.take<float>(p8 * 64);
  ws.t16a = bump.take<float>(p16 * 64);
  ws.t16b = bump.take<float>(p16 * 64);
  ws.x4 = bump.take<float>(p16 * 64);
  ws.t32a = bump.take<float>(p32 * 128);
  ws.t32b = bump.take<float>(p32 * 128);
  ws.x5 = bump.take<float>(p32 * 64);
}

}  // namespace xf

extern "C" int xfeat_abi_version(void) { return XFEAT_ABI_VERSION; }
extern "C" const char* xfeat_last_error(void) { return xf::g_err; }
extern "C" unsigned long long xfeat_launch_count(void) { return xf::g_launches; }
extern "C" size_t xfeat_packed_weight_floats(void) { return xf::make_layer_table().total; }

extern "C" int xfeat_create(xfeat_ctx** out, int device, const float* packed_host, size_t n_floats) {
  XF_REQUIRE(out && packed_host, "create: null pointer");
  const xf::LayerTable t = xf::make_layer_table();
  XF_REQUIRE(n_floats == t.total, "create: packed blob has %zu floats, expected %zu", n_floats, t.total);
  xf::DeviceGuard guard(device);   // the caller's current device is restored on every return path
  XF_REQUIRE(guard.ok, "create: cudaSetDevice(%d) failed", device);
  cudaDeviceProp prop;
  XF_CUDA(cudaGetDeviceProperties(&prop, device));
  if (prop.major != 10) {
    xf::set_error("create: device %d is sm_%d%d; this library contains sm_100a code only", device, prop.major, prop.minor);
    return XF_E_UNSUPPORTED;
  }
  xfeat_ctx* c = new xfeat_ctx();
  c->device = device;
  c->sm_count = prop.multiProcessorCount;
  c->table = t;
  c->h_weights = (float*)malloc(sizeof(float) * t.total);
  memcpy(c->h_weights, packed_host, sizeof(float) * t.total);
  c->d_weights = nullptr;
  cudaError_t e = cudaMalloc(&c->d_weights, sizeof(float) * t.total);
  if (e == cudaSuccess) e = cudaMemcpy(c->d_weights, packed_host, sizeof(float) * t.total, cudaMemcpyHostToDevice);
  if (e != cudaSuccess) {
    xf::set_error("create: weight upload failed: %s", cudaGetErrorString(e));
    if (c->d_weights) cudaFree(c->d_weights);
    free(c->h_weights);
    delete c;
    return XF_E_CUDA;
  }
  c->d_tcw = nullptr;
  c->d_mlpw = nullptr;
  int rc = xf::conv_tc_prepare(c);
  if (rc == XF_OK) rc = xf::mlp_tc_prepare(c);
  if (rc != XF_OK) {
    cudaFree(c->d_weights);
    if (c->d_tcw) cudaFree(c->d_tcw);
    if (c->d_mlpw) cudaFree(c->d_mlpw);
    free(c->h_weights);
    delete c;
    return rc;
  }
  *out = c;
  return XF_OK;
}

extern "C" void xfeat_set_conv_impl(int impl) { xf::g_conv_impl = (impl < 0 || impl > 2) ? 1 : impl; }
extern "C" int xfeat_get_conv_impl(void) { return xf::g_conv_impl; }

extern "C" void xfeat_destroy(xfeat_ctx* ctx) {
  if (!ctx) return;
  xf::DeviceGuard guard(ctx->device);
  if (ctx->d_weights) cudaFree(ctx->d_weights);
  if (ctx->d_tcw) cudaFree(ctx->d_tcw);
  if (ctx->d_mlpw) cudaFree(ctx->d_mlpw);
  free(ctx->h_weights);
  delete ctx;
}

extern "C" size_t xfeat_net_workspace_bytes(int B, int H, int W) {
  xf::Bump bump(nullptr, 0);
  xf::NetWs ws;
  xf::carve_net(bump, B, H, W, ws);
  return bump.used();
}

extern "C" int xfeat_net(xfeat_ctx* ctx, const float* d_xn, int B, int H, int W, float* d_feats, float* d_heat,
                         float* d_reliability, float* d_kpt_logits, void* d_ws, size_t ws_bytes, void* stream) {
  using namespace xf;
  XF_REQUIRE(ctx && d_xn && d_feats && d_heat && d_reliability && d_ws, "net: null pointer");
  XF_REQUIRE(B > 0 && B <= 65535 && H > 0 && W > 0 && H % 32 == 0 && W % 32 == 0, "net: bad shape B=%d H=%d W=%d", B, H, W);
  XF_CUDA(cudaSetDevice(ctx->device));
  cudaStream_t st = (cudaStream_t)stream;
  Bump bump(d_ws, ws_bytes);
  NetWs ws;
  carve_net(bump, B, H, W, ws);
  if (!bump.ok) {
    set_error("net: workspace too small (%zu < %zu)", ws_bytes, bump.used());
    return XF_E_WORKSPACE;
  }
  const int H4 = H / 4, W4 = W / 4, H8 = H / 8, W8 = W / 8, H16 = H / 16, W16 = W / 16, H32 = H / 32, W32 = W / 32;
  int rc;
#define XF_RUN(call) \
  if ((rc = (call)) != XF_OK) return rc
  if (g_conv_impl == 0) {
    // ------------------------------ all layers on the fp32 CUDA-core kernels ------------------------------
    // block1 + skip1 -> x1 + skip1(x)                                            model.py:139-140
    XF_RUN(launch_stem_chain(ctx->h_weights, ctx->table, d_xn, ws.a1, ws.a2, ws.a3, ws.x1s, nullptr, B, H, W, st));
    XF_RUN(launch_conv_layer(ctx, L_B2_0, ws.x1s, IN_NHWC, B, H4, W4, ws.t4a, st));                  // block2, model.py:140
    XF_RUN(launch_conv_layer(ctx, L_B2_1, ws.t4a, IN_NHWC, B, H4, W4, ws.x2, st));
    XF_RUN(launch_conv_layer(ctx, L_B3_0, ws.x2, IN_NHWC, B, H4, W4, ws.t8a, st));                   // block3, model.py:141
    XF_RUN(launch_conv_layer(ctx, L_B3_1, ws.t8a, IN_NHWC, B, H8, W8, ws.t8b, st));
    XF_RUN(launch_conv_layer(ctx, L_B3_2, ws.t8b, IN_NHWC, B, H8, W8, ws.x3, st));
    XF_RUN(launch_conv_layer(ctx, L_B4_0, ws.x3, IN_NHWC, B, H8, W8, ws.t16a, st));                  // block4, model.py:142
    XF_RUN(launch_conv_layer(ctx, L_B4_1, ws.t16a, IN_NHWC, B, H16, W16, ws.t16b, st));
    XF_RUN(launch_conv_layer(ctx, L_B4_2, ws.t16b, IN_NHWC, B, H16, W16, ws.x4, st));
    XF_RUN(launch_conv_layer(ctx, L_B5_0, ws.x4, IN_NHWC, B, H16, W16, ws.t32a, st));                // block5, model.py:143
  } else {
    // ---- block2 .. block5.0 on tcgen05; activations between tensor-core layers travel as split fp16 [hi | lo] ----
    __half *s4a = (__half*)ws.x1s, *s4b = (__half*)ws.t4a, *s4c = (__half*)ws.x2;
    __half *s8a = (__half*)ws.t8a, *s8b = (__half*)ws.t8b, *s16a = (__half*)ws.t16a, *s16b = (__half*)ws.t16b;
    if (g_conv_impl == 2) {
      // block1.0/1.1 on CUDA cores (K = 9 / 36), block1.2 and block1.3 + skip1 (stride 2) in one tcgen05 kernel with 32-byte
      // operand rows [hi(8)|lo(8)] (block1_tc.cu)                                  model.py:43-48,139-140
      XF_RUN(launch_stem_chain(ctx->h_weights, ctx->table, d_xn, ws.a1, ws.a2, ws.a3, nullptr, nullptr, B, H, W, st, 1));
      XF_RUN(launch_block1_tail(ctx, (const __half*)ws.a2, d_xn, B, H4, W4, (__half*)ws.a3, s4a, nullptr, st));
    } else {
      XF_RUN(launch_stem_chain(ctx->h_weights, ctx->table, d_xn, ws.a1, ws.a2, ws.a3, nullptr, s4a, B, H, W, st));
    }
    XF_RUN(launch_conv_tc(ctx, L_B2_0, s4a, B, H4, W4, s4b, nullptr, st));                           // block2, model.py:140
    XF_RUN(launch_conv_tc(ctx, L_B2_1, s4b, B, H4, W4, s4c, nullptr, st));
    XF_RUN(launch_conv_tc(ctx, L_B3_0, s4c, B, H4, W4, s8a, nullptr, st));                           // block3 (stride 2), model.py:141
    XF_RUN(launch_conv_tc(ctx, L_B3_1, s8a, B, H8, W8, s8b, nullptr, st));
    XF_RUN(launch_conv_tc(ctx, L_B3_2, s8b, B, H8, W8, s8a, nullptr, st));     // x3 stays split: block4.0 and the fusion read it
    XF_RUN(launch_conv_tc(ctx, L_B4_0, s8a, B, H8, W8, s16a, nullptr, st));                          // block4 (stride 2), model.py:142
    XF_RUN(launch_conv_tc(ctx, L_B4_1, s16a, B, H16, W16, s16b, nullptr, st));
    XF_RUN(launch_conv_tc(ctx, L_B4_2, s16b, B, H16, W16, s16a, nullptr, st)); // x4 stays split: block5.0 and the fusion read it
    // block5: 128 channels, split tensors are [hi(128) | lo(128)] = 512 B per pixel            model.py:143
    __half *s32a = (__half*)ws.t32a, *s32b = (__half*)ws.t32b;
    XF_RUN(launch_conv_tc(ctx, L_B5_0, s16a, B, H16, W16, s32a, nullptr, st));
    XF_RUN(launch_conv_tc(ctx, L_B5_1, s32a, B, H32, W32, s32b, nullptr, st));
    XF_RUN(launch_conv_tc(ctx, L_B5_2, s32b, B, H32, W32, s32a, nullptr, st));
    XF_RUN(launch_conv_tc(ctx, L_B5_3, s32a, B, H32, W32, s32b, nullptr, st));  // x5 (64 ch) split, for the fusion
  }
  if (g_conv_impl == 0) {   // rest of block5 on the fp32 CUDA-core kernel                  model.py:143
    XF_RUN(launch_conv_layer(ctx, L_B5_1, ws.t32a, IN_NHWC, B, H32, W32, ws.t32b, st));
    XF_RUN(launch_conv_layer(ctx, L_B5_2, ws.t32b, IN_NHWC, B, H32, W32, ws.t32a, st));
    XF_RUN(launch_conv_layer(ctx, L_B5_3, ws.t32a, IN_NHWC, B, H32, W32, ws.x5, st));
  }
  if (g_conv_impl == 0) {
    // pyramid fusion                                                             model.py:146-148
    XF_RUN(launch_fuse_pyramid(ws.x3, ws.x4, ws.x5, ws.fin, nullptr, B, H8, W8, st));
    XF_RUN(launch_conv_layer(ctx, L_FU_0, ws.fin, IN_NHWC, B, H8, W8, ws.f1, st));
    XF_RUN(launch_conv_layer(ctx, L_FU_1, ws.f1, IN_NHWC, B, H8, W8, ws.f2, st));
    XF_RUN(launch_conv_layer(ctx, L_FU_2, ws.f2, IN_NHWC, B, H8, W8, d_feats, st));
    // reliability head                                                           model.py:151
    XF_RUN(launch_conv_layer(ctx, L_HH_0, d_feats, IN_NHWC, B, H8, W8, ws.t8a, st));
    XF_RUN(launch_conv_layer(ctx, L_HH_1, ws.t8a, IN_NHWC, B, H8, W8, ws.t8b, st));
    XF_RUN(launch_reliability(ctx, ws.t8b, d_reliability, (int64_t)B * H8 * W8, st));
    // keypoint head on the 8x8-unfolded gray image, softmax + depth-to-space      model.py:152, xfeat.py:242-247
    XF_RUN(launch_conv_layer(ctx, L_KH_0, d_xn, IN_UNFOLD8, B, H8, W8, ws.t8a, st));
    XF_RUN(launch_conv_layer(ctx, L_KH_1, ws.t8a, IN_NHWC, B, H8, W8, ws.t8b, st));
    XF_RUN(launch_conv_layer(ctx, L_KH_2, ws.t8b, IN_NHWC, B, H8, W8, ws.t8a, st));
    XF_RUN(launch_kpt_softmax(ctx, ws.t8a, d_heat, d_kpt_logits, B, H8, W8, st));
  } else {
    __half *s8a = (__half*)ws.t8a, *s8b = (__half*)ws.t8b, *sfin = (__half*)ws.fin, *sf1 = (__half*)ws.f1, *sf2 = (__half*)ws.f2;
    XF_RUN(launch_fuse_pyramid_split(s8a, (const __half*)ws.t16a, (const __half*)ws.t32b, sfin, B, H8, W8, st));  // model.py:146-148
    XF_RUN(launch_conv_tc(ctx, L_FU_0, sfin, B, H8, W8, sf1, nullptr, st));
    XF_RUN(launch_conv_tc(ctx, L_FU_1, sf1, B, H8, W8, sf2, nullptr, st));
    XF_RUN(launch_conv_tc(ctx, L_FU_2, sf2, B, H8, W8, s8a, d_feats, st));      // fp32 feats for the samplers + split for the head
    if (g_conv_impl == 2) {
      // fused head chains: activations stay in shared memory / TMEM between the 1x1 layers (head_chain_tc.cu)
      XF_RUN(launch_head_chain(ctx, 1, s8a, B, H8, W8, d_reliability, nullptr, st));                 // model.py:151
      XF_RUN(launch_head_chain(ctx, 0, d_xn, B, H8, W8, d_heat, d_kpt_logits, st));   // unfold8 (model.py:152) inside; + xfeat.py:242-247
      return XF_OK;
    }
    XF_RUN(launch_conv_tc(ctx, L_HH_0, s8a, B, H8, W8, s8b, nullptr, st));                          // model.py:151
    XF_RUN(launch_conv_tc(ctx, L_HH_1, s8b, B, H8, W8, nullptr, ws.t8a, st));
    XF_RUN(launch_reliability(ctx, ws.t8a, d_reliability, (int64_t)B * H8 * W8, st));
    XF_RUN(launch_unfold8_split(d_xn, s8b, B, H8, W8, st));                                          // model.py:152
    XF_RUN(launch_conv_tc(ctx, L_KH_0, s8b, B, H8, W8, s8a, nullptr, st));
    XF_RUN(launch_conv_tc(ctx, L_KH_1, s8a, B, H8, W8, s8b, nullptr, st));
    XF_RUN(launch_conv_tc(ctx, L_KH_2, s8b, B, H8, W8, nullptr, ws.t8a, st));
    XF_RUN(launch_kpt_softmax(ctx, ws.t8a, d_heat, d_kpt_logits, B, H8, W8, st));
  }
#undef XF_RUN
  return XF_OK;
}

// Shared helpers for libxfeat_sm100.so (sm_100a only).
#pragma once
#include <cuda.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string>

#include "../../include/xfeat_b200.h"
#include "layers.h"

namespace xf {

void set_error(const char* fmt, ...);


#define XF_CUDA(expr)                                                                      \
  do {                                                                                     \
    cudaError_t _e = (expr);                                                               \
    if (_e != cudaSuccess) {                                                               \
      xf::set_error("%s:%d: %s -> %s", __FILE__, __LINE__, #expr, cudaGetErrorString(_e)); \
      return XF_E_CUDA;                                                                    \
    }                                                                                      \
  } while (0)

// every launch of one of OUR kernels passes through here: counted for bench.py's gpu_launches claim
extern unsigned long long g_launches;
#define XF_LAUNCH_CHECK()          \
  do {                             \
    ++xf::g_launches;              \
    XF_CUDA(cudaGetLastError());   \
  } while (0)

#define XF_REQUIRE(cond, ...)       \
  do {                              \
    if (!(cond)) {                  \
      xf::set_error(__VA_ARGS__);   \
      return XF_E_INVALID;          \
    }                               \
  } while (0)

// cudaFuncAttributeMaxDynamicSharedMemorySize is a per-DEVICE (per-context) attribute: remembered per (current device,
// kernel), so a second XFeat(device=1) in the same process sets it again there (api.cu).
int ensure_dyn_smem(const void* func, size_t bytes);
#define XF_DYN_SMEM(kernel, bytes)                                                   \
  do {                                                                               \
    int _rc = xf::ensure_dyn_smem((const void*)(kernel), (size_t)(bytes));           \
    if (_rc != XF_OK) return _rc;                                                    \
  } while (0)

// cudaSetDevice(dev) for the scope, then back to whatever the caller had current (xfeat_create / xfeat_destroy must not
// change the caller's device as a side effect).
struct DeviceGuard {
  int prev;
  bool ok;
  explicit DeviceGuard(int dev) : prev(-1), ok(false) {
    if (cudaGetDevice(&prev) != cudaSuccess) prev = -1;
    ok = (cudaSetDevice(dev) == cudaSuccess);
  }
  ~DeviceGuard() {
    if (prev >= 0) cudaSetDevice(prev);
  }
};

static inline int cdiv(int a, int b) { return (a + b - 1) / b; }
static inline size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

// Bump allocator over a caller-provided workspace.
struct Bump {
  char* base;
  size_t off, cap;
  bool ok;
  Bump(void* p, size_t bytes) : base((char*)p), off(0), cap(bytes), ok(true) {}
  template <typename T>
  T* take(size_t n) {
    off = align_up(off, 256);
    size_t b = n * sizeof(T);
    if (base != nullptr && off + b > cap) ok = false;
    T* r = base ? (T*)(base + off) : nullptr;
    off += b;
    return r;
  }
  size_t used() const { return align_up(off, 256); }
};

// float <-> order-preserving uint32 (larger float -> larger uint). -0 is canonicalised by the callers (v + 0.0f).
__host__ __device__ __forceinline__ uint32_t f2ord(float f) {
#ifdef __CUDA_ARCH__
  uint32_t u = __float_as_uint(f);
#else
  uint32_t u;
  memcpy(&u, &f, 4);
#endif
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__host__ __device__ __forceinline__ float ord2f(uint32_t o) {
  uint32_t u = (o & 0x80000000u) ? (o & 0x7fffffffu) : ~o;
#ifdef __CUDA_ARCH__
  return __uint_as_float(u);
#else
  float f;
  memcpy(&f, &u, 4);
  return f;
#endif
}
// (value, index) packed so that unsigned max == "largest value, then lowest index" (torch.max tie rule).
__device__ __forceinline__ unsigned long long pack_vi(float v, uint32_t idx) {
  return ((unsigned long long)f2ord(v + 0.0f) << 32) | (unsigned long long)(0xffffffffu - idx);
}
__device__ __forceinline__ uint32_t packed_idx(unsigned long long p) { return 0xffffffffu - (uint32_t)(p & 0xffffffffu); }
__device__ __forceinline__ float packed_val(unsigned long long p) { return ord2f((uint32_t)(p >> 32)); }

// Source coordinate of InterpolateSparse2d for integer position p (interpolator.py:17-19 + ATen
// grid_sampler_unnormalize, align_corners=False), in the same fp32 operation order as the oracle's source_coord.
__device__ __forceinline__ float sparse_src_coord(int p, int size_pos, int size_map) {
  float g = __fsub_rn(__fmul_rn(2.0f, __fdiv_rn((float)p, (float)(size_pos - 1))), 1.0f);
  return __fdiv_rn(__fsub_rn(__fmul_rn(__fadd_rn(g, 1.0f), (float)size_map), 1.0f), 2.0f);
}

// ATen upsample_bilinear2d source index (align_corners=False): src = scale*(dst+0.5)-0.5 clamped at 0.
// packed fp32 pairs (sm_100: FFMA2 / FMUL2): two independent IEEE round-to-nearest operations per instruction
__device__ __forceinline__ float2 f2_fma(float2 a, float2 b, float2 c) {
  float2 r;
  asm("fma.rn.f32x2 %0, %1, %2, %3;"
      : "=l"(*reinterpret_cast<unsigned long long*>(&r))
      : "l"(*reinterpret_cast<const unsigned long long*>(&a)), "l"(*reinterpret_cast<const unsigned long long*>(&b)),
        "l"(*reinterpret_cast<const unsigned long long*>(&c)));
  return r;
}
__device__ __forceinline__ float2 f2_mul(float2 a, float2 b) {
  float2 r;
  asm("mul.rn.f32x2 %0, %1, %2;"
      : "=l"(*reinterpret_cast<unsigned long long*>(&r))
      : "l"(*reinterpret_cast<const unsigned long long*>(&a)), "l"(*reinterpret_cast<const unsigned long long*>(&b)));
  return r;
}

struct LinTap {
  int i0, i1;
  float l0, l1;
};
__device__ __forceinline__ LinTap lin_tap(int dst, float scale, int in_size) {
  float src = __fsub_rn(__fmul_rn(scale, __fadd_rn((float)dst, 0.5f)), 0.5f);
  if (src < 0.f) src = 0.f;
  LinTap t;
  t.i0 = (int)src;
  if (t.i0 > in_size - 1) t.i0 = in_size - 1;
  t.i1 = t.i0 + ((t.i0 < in_size - 1) ? 1 : 0);
  t.l1 = __fsub_rn(src, (float)t.i0);
  t.l0 = __fsub_rn(1.0f, t.l1);
  return t;
}

}  // namespace xf

struct xfeat_ctx {
  int device;
  int sm_count;
  float* d_weights;     // packed blob on device
  float* h_weights;     // host copy (stem weights travel as kernel parameters)
  xf::LayerTable table; // offsets into d_weights
  // tensor-core path (conv_tc.cu): pre-split fp16 weights [tap][term][cout][cin], their TMA maps, 2^-k rescale
  void* d_tcw;
  size_t tc_off[xf::L_COUNT];
  float tc_inv_wscale[xf::L_COUNT];
  // fine-matcher MLP on the tensor cores (mlp_tc.cu): split fp16 weights [N][whi(K) | wlo(K)] of the five Linear layers
  void* d_mlpw;
  size_t mlp_off[5];
  float mlp_inv_scale[5];
};

// ---- stage launchers shared between translation units -------------------------------------------------
namespace xf {
enum { IN_NHWC = 0, IN_UNFOLD8 = 1 };
int launch_conv_layer(const xfeat_ctx* ctx, int layer, const float* in, int in_mode, int B, int Hi, int Wi,
                      float* out, cudaStream_t st, const int* n_live = nullptr, __half* out_split = nullptr);
extern int g_conv_impl;  // 0 = fp32 CUDA cores, 1 = tcgen05 (per-tap operand loads), 2 = tcgen05 + halo-patch reuse for 3x3/s1
bool conv_tc_eligible(int layer);
int launch_conv_tc_halo(const xfeat_ctx* ctx, int layer, const __half* in_split, int B, int H, int W, __half* out_split,
                        float* out_f32, cudaStream_t st);
int launch_topk_select_sort(const unsigned long long* keys, const int* n_keep, int n_const, int cap, int top_k, int B,
                            unsigned long long* sorted, cudaStream_t st);
int conv_tc_prepare(xfeat_ctx* ctx);
int mlp_tc_prepare(xfeat_ctx* ctx);
int launch_fine_mlp_tc(const xfeat_ctx* ctx, const __half* X_split, int rows_cap, const int* n_live, __half* act_a, __half* act_b,
                       float* logits, cudaStream_t st);
int launch_conv_tc(const xfeat_ctx* ctx, int layer, const __half* in_split, int B, int H, int W, __half* out_split,
                   float* out_f32, cudaStream_t st, const float* skip_xn = nullptr);
int launch_block1_tail(const xfeat_ctx* ctx, const __half* a2_split, const float* xn, int B, int H4, int W4, __half* a3_split,
                       __half* out_split, float* out_f32, cudaStream_t st);
int launch_head_chain(const xfeat_ctx* ctx, int mode, const void* in, int B, int Hc, int Wc, float* out, float* logits,
                      cudaStream_t st);
int launch_split_nhwc(const float* in, __half* out, int64_t npix, int C, int CP, cudaStream_t st);
int launch_unfold8_split(const float* xn, __half* out, int B, int Hc, int Wc, cudaStream_t st);
int launch_stem_chain(const float* h_weights, const LayerTable& t, const float* xn, float* a1, float* a2, float* a3,
                      float* x1s, __half* x1s_split32, int B, int H, int W, cudaStream_t st, int tc_tail = 0);
int launch_fuse_pyramid(const float* x3, const float* x4, const float* x5, float* out, __half* out_split, int B, int H3,
                        int W3, cudaStream_t st);
int launch_fuse_pyramid_split(const __half* x3, const __half* x4, const __half* x5, __half* out_split, int B, int H3, int W3,
                              cudaStream_t st);
int launch_reliability(const xfeat_ctx* ctx, const float* t, float* out, int64_t npix, cudaStream_t st);
int launch_kpt_softmax(const xfeat_ctx* ctx, const float* t, float* heat, float* logits, int B, int Hc, int Wc,
                       cudaStream_t st);
}

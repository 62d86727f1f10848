// block1.2 (3x3 stride 1, 8 -> 8) and block1.3 (3x3 stride 2, 8 -> 24) + skip1 in ONE persistent tcgen05 kernel: the
// half-resolution activation between the two layers stays in shared memory instead of a 32-byte-per-pixel HBM round trip.
//
// A tile is TQH x TQW quarter-resolution outputs.  They read the (2*TQH+1) x (2*TQW+1) half-resolution block1.2 outputs
// starting at half-res (2*qy0-1, 2*qx0-1), which in turn read the (2*TQH+3) x (2*TQW+3) patch of a2 loaded by one TMA box
// (out-of-image coordinates zero-filled = block1.2's padding).
//   * block1.2 is the halo scheme of conv_tc_halo.cu: GEMM rows m = h * PW2 + w over the patch pitch PW2 = 2*TQW+3, the
//     taps are shifted shared-memory descriptors; M2 = ceil((2*TQH+1) * PW2 / 128) M-tiles of 128 rows, 16 TMEM columns each.
//   * the block1.2 epilogue re-splits its outputs into four POLYPHASE planes (even|odd half-res row) x (even|odd column),
//     plane pitch PQW = TQW+1, in the SWIZZLE_32B K-major layout the next UMMA reads.  Half-res positions outside the image
//     are stored as zeros: block1.3's zero padding.
//   * block1.3: quarter-res output (i,j), tap (ky,kx) reads half-res (2i-1+ky, 2j-1+kx) = plane (ky&1, kx&1) at
//     (i + (ky>>1), j + (kx>>1)): with GEMM rows m = i * PQW + j every stride-2 tap is a shifted descriptor over one plane.
// Both layers issue the UMMAs of conv_tc_halo_kernel<8,8> / conv_tc_kernel<3,8,32> on bit-identical operands and their
// epilogues do the same fp32 operations, so the output equals the two-kernel path bit for bit.
//
// Warp roles: 0 TMA, 1 MMA (issue order per tile: block1.2 of tile t+1 before block1.3 of tile t, so the tensor pipe has
// work while the block1.2 epilogue of tile t fills the planes), 2-9 block1.2 epilogue (two warps per TMEM lane quarter,
// alternate M-tiles), 10-13 block1.3 + skip1 epilogue.
#include <cuda_fp16.h>

#include <stdlib.h>

#include "common.cuh"
#include "tc_common.cuh"

namespace xf {

constexpr int B1_THREADS = 448;
constexpr int B1_NP = 4;                       // a2 patch ring
constexpr int B1_W2_BYTES = 9 * 2 * 8 * 32;    // block1.2 weights: [tap][whi|whi ; wlo|0][8 rows] x 32 B
constexpr int B1_W3_BYTES = 9 * 2 * 32 * 32;   // block1.3 weights: [tap][whi|whi ; wlo|0][32 rows] x 32 B
constexpr int B1_W_PAD = 23 * 1024;            // both weight sets, padded so that the patch and plane buffers are 1024-aligned
constexpr int B1_PB_MAX = 30 * 1024;           // bytes per patch buffer
constexpr int B1_PLANE_MAX = 6 * 1024;         // bytes per polyphase plane (4 planes per buffer, 2 buffers)

struct Block1Params {
  CUtensorMap amap;    // a2 split (B,H2,W2,16) halves; box {16, PW2, 2*TQH+3, 1}, SWIZZLE_32B
  CUtensorMap w2map;   // block1.2 weights, box {16, 8}
  CUtensorMap w3map;   // block1.3 weights, box {16, 32}
  const float* bias2;
  const float* bias3;
  const float* skip_w;   // 24 weights then 24 biases
  const float* xn;       // (B, 4*H4, 4*W4) normalised gray image
  float inv_ws2, inv_ws3;
  int B, H4, W4;         // output (quarter-res) size; the half-res input is 2*H4 x 2*W4
  int TQH, TQW, PW2, PQW, M2;
  int PB, PLB;           // patch buffer / plane bytes (multiples of 1024)
  int tmem_cols;
  __half* out_split;     // (B,H4,W4,64) [hi(32) | lo(32)] or null
  float* out_f32;        // (B,H4,W4,24) or null
  FastDiv div_img, div_x;
};

__global__ void __launch_bounds__(B1_THREADS, 1) block1_tc_kernel(const __grid_constant__ Block1Params P) {
  extern __shared__ unsigned char smem_raw[];
  unsigned char* base = reinterpret_cast<unsigned char*>(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
  unsigned char* sW2 = base;
  unsigned char* sW3 = sW2 + B1_W2_BYTES;
  unsigned char* sP = base + B1_W_PAD;
  unsigned char* sQ = sP + (size_t)B1_NP * P.PB;                          // plane buffers [2][4][PLB]
  uint64_t* bars = reinterpret_cast<uint64_t*>(sQ + (size_t)8 * P.PLB);
  uint64_t* w_full = bars;
  uint64_t* p_full = bars + 1;                 // [NP]
  uint64_t* p_empty = p_full + B1_NP;          // [NP]
  uint64_t* acc2_full = p_empty + B1_NP;       // [2]
  uint64_t* acc2_empty = acc2_full + 2;        // [2]
  uint64_t* q_full = acc2_empty + 2;           // [2] planes written
  uint64_t* q_empty = q_full + 2;              // [2] planes read by the block1.3 MMAs
  uint64_t* acc3_full = q_empty + 2;           // [2]
  uint64_t* acc3_empty = acc3_full + 2;        // [2]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(acc3_empty + 2);
  float* sB2 = reinterpret_cast<float*>(tmem_slot + 2);   // [8]
  float* sB3 = sB2 + 8;                                    // [32]
  float* sSkip = sB3 + 32;                                 // [2][32]

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int tiles_x = (P.W4 + P.TQW - 1) / P.TQW, tiles_y = (P.H4 + P.TQH - 1) / P.TQH;
  const int tiles_img = tiles_x * tiles_y;
  const int n_tiles = tiles_img * P.B;
  const int H2 = 2 * P.H4, W2 = 2 * P.W4;
  const int ACC2 = P.M2 * 16;                  // TMEM columns per block1.2 accumulator buffer
  const uint32_t acc3_col = 2u * ACC2;         // block1.3 accumulators follow: 2 x 64 columns

  if (threadIdx.x < 8) sB2[threadIdx.x] = __ldg(P.bias2 + threadIdx.x);
  if (threadIdx.x < 32) sB3[threadIdx.x] = threadIdx.x < 24 ? __ldg(P.bias3 + threadIdx.x) : 0.f;
  if (threadIdx.x < 64) {
    const int c = threadIdx.x % 32, wb = threadIdx.x / 32;
    sSkip[threadIdx.x] = c < 24 ? __ldg(P.skip_w + wb * 24 + c) : 0.f;
  }
  if (warp == 0 && lane == 0) {
    tc::tma_prefetch_desc(&P.amap);
    tc::tma_prefetch_desc(&P.w2map);
    tc::tma_prefetch_desc(&P.w3map);
    tc::mbar_init(w_full, 1);
    for (int i = 0; i < B1_NP; ++i) {
      tc::mbar_init(&p_full[i], 1);
      tc::mbar_init(&p_empty[i], 1);
    }
    for (int i = 0; i < 2; ++i) {
      tc::mbar_init(&acc2_full[i], 1);
      tc::mbar_init(&acc2_empty[i], 8);
      tc::mbar_init(&q_full[i], 8);
      tc::mbar_init(&q_empty[i], 1);
      tc::mbar_init(&acc3_full[i], 1);
      tc::mbar_init(&acc3_empty[i], 4);
    }
    tc::fence_barrier_init();
  }
  if (warp == 1) {
    tc::tmem_alloc(tmem_slot, P.tmem_cols);
    tc::tmem_relinquish();
  }
  tc::tc_fence_before();
  __syncthreads();
  tc::tc_fence_after();
  const uint32_t tmem = *tmem_slot;

  if (warp == 0) {
    if (tc::elect_one()) {
      tc::mbar_expect_tx(w_full, (uint32_t)(B1_W2_BYTES + B1_W3_BYTES));
      for (int i = 0; i < 18; ++i) tc::tma_load_2d(sW2 + i * 256, &P.w2map, w_full, 0, i * 8);
      for (int i = 0; i < 18; ++i) tc::tma_load_2d(sW3 + i * 1024, &P.w3map, w_full, 0, i * 32);
      const uint32_t patch_tx = (uint32_t)(2 * P.TQH + 3) * P.PW2 * 32;
      uint32_t tcount = 0;
      for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, ++tcount) {
        const int b = (int)fdiv((unsigned)tile, P.div_img), rem = tile - b * tiles_img;
        const int ty_ = (int)fdiv((unsigned)rem, P.div_x), tx_ = rem - ty_ * tiles_x;
        const int s = tcount % B1_NP;
        tc::mbar_wait(&p_empty[s], ((tcount / B1_NP) & 1) ^ 1);
        tc::mbar_expect_tx(&p_full[s], patch_tx);
        tc::tma_load_4d(sP + (size_t)s * P.PB, &P.amap, &p_full[s], 0, 2 * tx_ * P.TQW - 2, 2 * ty_ * P.TQH - 2, b);
      }
    }
    __syncwarp();
  } else if (warp == 1) {
    if (tc::elect_one()) {
      constexpr uint32_t idesc2 = tc::make_idesc(/*F16*/ 0, 128, 16);   // block1.2: [whi|whi ; wlo|0], N = 2 x 8
      constexpr uint32_t idesc3 = tc::make_idesc(/*F16*/ 0, 128, 64);   // block1.3: [whi|whi ; wlo|0], N = 2 x 32
      tc::mbar_wait(w_full, 0);
      const uint32_t w2_base = tc::smem_u32(sW2), w3_base = tc::smem_u32(sW3);
      const uint32_t p_base = tc::smem_u32(sP), q_base = tc::smem_u32(sQ);
      const int n_mine = n_tiles > (int)blockIdx.x ? (n_tiles - 1 - (int)blockIdx.x) / (int)gridDim.x + 1 : 0;
      for (int t = 0; t <= n_mine; ++t) {
        if (t < n_mine) {   // ---- block1.2 of tile t (conv_tc_halo_kernel<8,8>'s UMMAs, per M-tile) ----
          const int s = t % B1_NP, a = t & 1;
          tc::mbar_wait(&acc2_empty[a], ((t >> 1) & 1) ^ 1);
          tc::mbar_wait(&p_full[s], (t / B1_NP) & 1);
          tc::tc_fence_after();
          const uint32_t pb = p_base + (uint32_t)s * P.PB;
          for (int mt = 0; mt < P.M2; ++mt) {
            const uint32_t d = tmem + (uint32_t)(a * ACC2 + mt * 16);
            for (int tap = 0; tap < 9; ++tap) {
              const uint32_t row = (uint32_t)(mt * 128 + (tap / 3) * P.PW2 + (tap % 3));
              tc::umma_f16(d, tc::make_desc_sw32(pb + row * 32u, 256), tc::make_desc_sw32(w2_base + tap * 512u, 256), idesc2,
                           tap ? 1u : 0u);
            }
          }
          tc::umma_commit(&p_empty[s]);
          tc::umma_commit(&acc2_full[a]);
        }
        if (t > 0) {        // ---- block1.3 of tile t-1 from the planes (conv_tc_kernel<3,8,32>'s UMMAs) ----
          const int u = t - 1, a = u & 1;
          tc::mbar_wait(&acc3_empty[a], ((u >> 1) & 1) ^ 1);
          tc::mbar_wait(&q_full[a], (u >> 1) & 1);
          tc::tc_fence_after();
          const uint32_t qb = q_base + (uint32_t)a * 4u * P.PLB;
          const uint32_t d = tmem + acc3_col + (uint32_t)a * 64u;
          for (int tap = 0; tap < 9; ++tap) {
            const int ky = tap / 3, kx = tap % 3;
            const uint32_t addr = qb + (uint32_t)((ky & 1) * 2 + (kx & 1)) * P.PLB + (uint32_t)((ky >> 1) * P.PQW + (kx >> 1)) * 32u;
            tc::umma_f16(d, tc::make_desc_sw32(addr, 256), tc::make_desc_sw32(w3_base + tap * 2048u, 256), idesc3, tap ? 1u : 0u);
          }
          tc::umma_commit(&q_empty[a]);
          tc::umma_commit(&acc3_full[a]);
        }
      }
    }
    __syncwarp();
  } else if (warp < 10) {
    // ---- block1.2 epilogue: TMEM -> bias + ReLU -> split fp16 -> polyphase planes (zeros outside the half-res image) ----
    const int q = warp & 3, eg = (warp - 2) >> 2;
    const int hmax = 2 * P.TQH + 1, wmax = 2 * P.TQW + 1;
    uint32_t tcount = 0;
    for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, ++tcount) {
      const int a = tcount & 1;
      const int b = (int)fdiv((unsigned)tile, P.div_img), rem = tile - b * tiles_img;
      const int ty_ = (int)fdiv((unsigned)rem, P.div_x), tx_ = rem - ty_ * tiles_x;
      const int y0 = 2 * ty_ * P.TQH - 1, x0 = 2 * tx_ * P.TQW - 1;   // half-res coordinates of GEMM row 0
      unsigned char* qb = sQ + (size_t)a * 4 * P.PLB;
      tc::mbar_wait(&acc2_full[a], (tcount >> 1) & 1);
      tc::mbar_wait(&q_empty[a], ((tcount >> 1) & 1) ^ 1);
      tc::tc_fence_after();
      for (int mt = eg; mt < P.M2; mt += 2) {
        uint32_t v[16];
        __syncwarp();
        tc::tmem_ld_32x16(tmem + ((uint32_t)(q * 32) << 16) + (uint32_t)(a * ACC2 + mt * 16), v);
        tc::tmem_ld_wait();
        const int m = mt * 128 + q * 32 + lane;
        const int h = m / P.PW2, w = m - h * P.PW2;
        if (h < hmax && w < wmax) {   // junk lanes of the pitch enumeration store nothing
          const int y = y0 + h, x = x0 + w;
          uint32_t hw[4] = {0u, 0u, 0u, 0u}, lw[4] = {0u, 0u, 0u, 0u};
          if (y >= 0 && y < H2 && x >= 0 && x < W2) {
            float o[8];
#pragma unroll
            for (int c = 0; c < 8; ++c) o[c] = fmaxf(fmaf(__uint_as_float(v[c]) + __uint_as_float(v[8 + c]), P.inv_ws2, sB2[c]), 0.f);
#pragma unroll
            for (int j = 0; j < 4; ++j) {   // tc::store_split_row<8>'s split
              const __half2 hh = __floats2half2_rn(o[2 * j], o[2 * j + 1]);
              const float2 hf = __half22float2(hh);
              const __half2 ll = __floats2half2_rn(o[2 * j] - hf.x, o[2 * j + 1] - hf.y);
              hw[j] = *reinterpret_cast<const uint32_t*>(&hh);
              lw[j] = *reinterpret_cast<const uint32_t*>(&ll);
            }
          }
          // plane (h&1, w&1), row (h>>1) * PQW + (w>>1); 32-byte swizzle: 16-byte chunk c of row r sits at c ^ ((r >> 2) & 1)
          const int r = (h >> 1) * P.PQW + (w >> 1);
          unsigned char* rp = qb + (size_t)((h & 1) * 2 + (w & 1)) * P.PLB + r * 32;
          const int sw = (r >> 2) & 1;
          *reinterpret_cast<uint4*>(rp + (sw << 4)) = make_uint4(hw[0], hw[1], hw[2], hw[3]);
          *reinterpret_cast<uint4*>(rp + ((sw ^ 1) << 4)) = make_uint4(lw[0], lw[1], lw[2], lw[3]);
        }
      }
      tc::fence_proxy_async();        // generic-proxy smem writes -> visible to the tensor core (async proxy)
      tc::tc_fence_before();
      __syncwarp();
      if (lane == 0) {
        tc::mbar_arrive(&acc2_empty[a]);
        tc::mbar_arrive(&q_full[a]);
      }
    }
  } else {
    // ---- block1.3 + skip1 epilogue: conv_tc_kernel<3,8,32>'s arithmetic ----
    // The skip branch's 4x4 xn window of the NEXT tile is loaded while this tile's accumulator is drained and stored: one
    // group of four warps drains every tile, so a global-load latency per tile would otherwise pace the whole kernel.
    const int q = warp & 3;
    const int m = q * 32 + lane;
    const int i = m / P.PQW, j = m - i * P.PQW;
    const bool lane_ok = (i < P.TQH) && (j < P.TQW);
    const int W0 = P.W4 * 4;
    auto fetch_xn = [&](int tile, float4 (&xv)[4]) {
      if (tile >= n_tiles) return;
      const int b = (int)fdiv((unsigned)tile, P.div_img), rem = tile - b * tiles_img;
      const int ty_ = (int)fdiv((unsigned)rem, P.div_x), tx_ = rem - ty_ * tiles_x;
      const int y = ty_ * P.TQH + i, x = tx_ * P.TQW + j;
      if (lane_ok && y < P.H4 && x < P.W4) {
        const float* xp = P.xn + ((int64_t)b * P.H4 * 4 + y * 4) * W0 + x * 4;
#pragma unroll
        for (int rr = 0; rr < 4; ++rr) xv[rr] = __ldg(reinterpret_cast<const float4*>(xp + (int64_t)rr * W0));
      }
    };
    float4 xv[4] = {};
    fetch_xn(blockIdx.x, xv);
    uint32_t tcount = 0;
    for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, ++tcount) {
      const int a = tcount & 1;
      const int b = (int)fdiv((unsigned)tile, P.div_img), rem = tile - b * tiles_img;
      const int ty_ = (int)fdiv((unsigned)rem, P.div_x), tx_ = rem - ty_ * tiles_x;
      const int y = ty_ * P.TQH + i, x = tx_ * P.TQW + j;
      float4 xnext[4] = {};
      fetch_xn(tile + (int)gridDim.x, xnext);
      tc::mbar_wait(&acc3_full[a], (tcount >> 1) & 1);
      tc::tc_fence_after();
      uint32_t v[64];
      __syncwarp();
#pragma unroll
      for (int c = 0; c < 2; ++c) {
        uint32_t t[32];
        tc::tmem_ld_32x32(tmem + ((uint32_t)(q * 32) << 16) + acc3_col + (uint32_t)a * 64u + c * 32, t);
#pragma unroll
        for (int k = 0; k < 32; ++k) v[c * 32 + k] = t[k];
      }
      tc::tmem_ld_wait();
      tc::tc_fence_before();
      __syncwarp();
      if (lane == 0) tc::mbar_arrive(&acc3_empty[a]);
      if (lane_ok && y < P.H4 && x < P.W4) {
        const int64_t pix = ((int64_t)b * P.H4 + y) * P.W4 + x;
        float o[32];
#pragma unroll
        for (int c = 0; c < 32; ++c) o[c] = fmaxf(fmaf(__uint_as_float(v[c]) + __uint_as_float(v[32 + c]), P.inv_ws3, sB3[c]), 0.f);
        // AvgPool2d(4,4) of the normalised gray image, then 1x1 conv 1 -> 24 with bias, added AFTER the ReLU (model.py:140)
        float sacc = 0.f;
#pragma unroll
        for (int rr = 0; rr < 4; ++rr) {
          sacc += xv[rr].x; sacc += xv[rr].y; sacc += xv[rr].z; sacc += xv[rr].w;
        }
        const float skipv = sacc * (1.0f / 16.0f);
#pragma unroll
        for (int c = 0; c < 32; ++c) o[c] += fmaf(skipv, sSkip[c], sSkip[32 + c]);
        if (P.out_f32) tc::store_f32_row<32>(P.out_f32 + pix * 24, o, 24);
        if (P.out_split) {
          __half* hp = P.out_split + pix * 64;
          tc::store_split_row<32>(hp, hp + 32, o);
        }
      }
#pragma unroll
      for (int rr = 0; rr < 4; ++rr) xv[rr] = xnext[rr];
    }
  }
  tc::tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc::tc_fence_after();
    tc::tmem_dealloc(tmem, P.tmem_cols);
  }
}

struct Block1Tile { int TQH, TQW, M2; };

// Tile shape: the quarter-res tile fills at most 128 block1.3 GEMM rows (TQH * (TQW+1) <= 128); the block1.2 rows of its
// halo-extended half-res region are the bulk of the tensor work.  Cost = MMA rows of both layers + a term for patch bytes.
static Block1Tile pick_block1_tile(int H4, int W4) {
  Block1Tile best = {0, 0, 0};
  double best_cost = 1e30;
  for (int tqw = 4; tqw <= 62; ++tqw) {
    const int pqw = tqw + 1, pw2 = 2 * tqw + 3;
    for (int tqh = 1; tqh * pqw <= 128; ++tqh) {
      const int m2 = cdiv((2 * tqh + 1) * pw2, 128);
      if ((m2 * 128 + 2 * pw2 + 2) * 32 > B1_PB_MAX || (128 + pqw + 1) * 32 > B1_PLANE_MAX) continue;
      const double tiles = (double)cdiv(W4, tqw) * cdiv(H4, tqh);
      const double cost = tiles * ((m2 + 1) * 128.0 + 0.15 * (2 * tqh + 3) * pw2);
      if (cost < best_cost) { best_cost = cost; best = {tqh, tqw, m2}; }
    }
  }
  return best;
}

int g_block1_fused = 1;   // XFEAT_BLOCK1_UNFUSED=1 in the environment selects the two-kernel path (A/B measurements)

static bool block1_fused() {
  static const bool unfused = getenv("XFEAT_BLOCK1_UNFUSED") != nullptr;
  return g_block1_fused && !unfused;
}

static int launch_block1_fused(const xfeat_ctx* ctx, const __half* a2_split, const float* xn, int B, int H4, int W4,
                               __half* out_split, float* out_f32, cudaStream_t st) {
  PFN_encodeTiled enc = get_encode_tiled();
  if (!enc) {
    set_error("cuTensorMapEncodeTiled entry point not available");
    return XF_E_CUDA;
  }
  const Block1Tile tl = pick_block1_tile(H4, W4);
  Block1Params P;
  P.TQH = tl.TQH; P.TQW = tl.TQW; P.M2 = tl.M2;
  P.PW2 = 2 * tl.TQW + 3;
  P.PQW = tl.TQW + 1;
  P.PB = (int)align_up((size_t)(tl.M2 * 128 + 2 * P.PW2 + 2) * 32, 1024);
  P.PLB = (int)align_up((size_t)(128 + P.PQW + 1) * 32, 1024);
  int cols = 32;
  while (cols < 2 * tl.M2 * 16 + 128) cols *= 2;
  P.tmem_cols = cols;
  const int H2 = 2 * H4, W2 = 2 * W4;
  const cuuint64_t dims[4] = {16, (cuuint64_t)W2, (cuuint64_t)H2, (cuuint64_t)B};
  const cuuint64_t strides[3] = {32, (cuuint64_t)W2 * 32, (cuuint64_t)H2 * W2 * 32};
  const cuuint32_t box[4] = {16, (cuuint32_t)P.PW2, (cuuint32_t)(2 * P.TQH + 3), 1};
  const cuuint32_t estr[4] = {1, 1, 1, 1};
  CUresult r = enc(&P.amap, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 4, (void*)a2_split, dims, strides, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_32B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled(block1 a2 patch) failed: %d", (int)r);
    return XF_E_CUDA;
  }
  const int layers[2] = {L_B1_2, L_B1_3}, nrows[2] = {8, 32};
  CUtensorMap* maps[2] = {&P.w2map, &P.w3map};
  for (int k = 0; k < 2; ++k) {
    const cuuint64_t wdims[2] = {16, (cuuint64_t)18 * nrows[k]};
    const cuuint64_t wstrides[1] = {32};
    const cuuint32_t wbox[2] = {16, (cuuint32_t)nrows[k]};
    const cuuint32_t westr[2] = {1, 1};
    r = enc(maps[k], CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, (void*)((__half*)ctx->d_tcw + ctx->tc_off[layers[k]]), wdims, wstrides,
            wbox, westr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_32B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
            CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
      set_error("cuTensorMapEncodeTiled(block1 weights, layer %d) failed: %d", layers[k], (int)r);
      return XF_E_CUDA;
    }
  }
  P.bias2 = ctx->d_weights + ctx->table.b_off[L_B1_2];
  P.bias3 = ctx->d_weights + ctx->table.b_off[L_B1_3];
  P.skip_w = ctx->d_weights + ctx->table.w_off[L_SKIP1];   // 24 weights; the 24 biases follow (layers.h packing)
  P.xn = xn;
  P.inv_ws2 = ctx->tc_inv_wscale[L_B1_2];
  P.inv_ws3 = ctx->tc_inv_wscale[L_B1_3];
  P.B = B; P.H4 = H4; P.W4 = W4;
  P.out_split = out_split;
  P.out_f32 = out_f32;
  const int tiles_img = cdiv(H4, P.TQH) * cdiv(W4, P.TQW);
  const int n_tiles = tiles_img * B;
  XF_REQUIRE(n_tiles < (1 << 22), "block1_tc: too many tiles (%d)", n_tiles);
  P.div_img = make_fastdiv((unsigned)tiles_img);
  P.div_x = make_fastdiv((unsigned)cdiv(W4, P.TQW));
  const size_t smem = 1024 + B1_W_PAD + (size_t)B1_NP * P.PB + (size_t)8 * P.PLB + 1024;
  const int grid = n_tiles < ctx->sm_count ? n_tiles : ctx->sm_count;
  XF_DYN_SMEM(block1_tc_kernel, smem);
  block1_tc_kernel<<<grid, B1_THREADS, smem, st>>>(P);
  XF_LAUNCH_CHECK();
  return XF_OK;
}

// a2_split (B,2*H4,2*W4,16) [hi(8)|lo(8)] -> block1.2 -> block1.3 + skip1(xn) -> out_split (B,H4,W4,64) and/or out_f32
// (B,H4,W4,24).  The two-kernel path (XFEAT_BLOCK1_UNFUSED / xfeat_set_block1_fused(0)) writes block1.2's output to a3_split.
int launch_block1_tail(const xfeat_ctx* ctx, const __half* a2_split, const float* xn, int B, int H4, int W4, __half* a3_split,
                       __half* out_split, float* out_f32, cudaStream_t st) {
  XF_REQUIRE(ctx->d_tcw && ctx->tc_off[L_B1_2] != (size_t)-1 && ctx->tc_off[L_B1_3] != (size_t)-1,
             "block1_tc: block1 weights not prepared for the tensor-core path");
  XF_REQUIRE(out_split || out_f32, "block1_tc: no output");
  if (block1_fused()) return launch_block1_fused(ctx, a2_split, xn, B, H4, W4, out_split, out_f32, st);
  int rc = launch_conv_tc(ctx, L_B1_2, a2_split, B, 2 * H4, 2 * W4, a3_split, nullptr, st);
  if (rc) return rc;
  return launch_conv_tc(ctx, L_B1_3, a3_split, B, 2 * H4, 2 * W4, out_split, out_f32, st, xn);
}

}  // namespace xf

extern "C" void xfeat_set_block1_fused(int on) { xf::g_block1_fused = on ? 1 : 0; }
extern "C" int xfeat_get_block1_fused(void) { return xf::block1_fused() ? 1 : 0; }

// Test hook: block1.2 -> block1.3 + skip1 on caller tensors.  a2 (B,H/2,W/2,8) fp32 NHWC, xn (B,H,W) -> x1s (B,H/4,W/4,24).
extern "C" int xfeat_debug_block1_tail(xfeat_ctx* ctx, const float* d_a2, const float* d_xn, int B, int H, int W, float* d_x1s,
                                       void* d_scratch, size_t scratch_bytes, void* stream) {
  XF_REQUIRE(ctx && d_a2 && d_xn && d_x1s && d_scratch, "debug_block1_tail: null pointer");
  XF_REQUIRE(B > 0 && B <= 65535 && H > 0 && W > 0 && H % 4 == 0 && W % 4 == 0, "debug_block1_tail: bad shape B=%d H=%d W=%d", B,
             H, W);
  const int64_t npix2 = (int64_t)B * (H / 2) * (W / 2);
  XF_REQUIRE(scratch_bytes >= (size_t)npix2 * 64, "debug_block1_tail: scratch must hold B*(H/2)*(W/2)*64 bytes");
  XF_CUDA(cudaSetDevice(ctx->device));
  cudaStream_t st = (cudaStream_t)stream;
  __half* a2s = (__half*)d_scratch;
  int rc = xf::launch_split_nhwc(d_a2, a2s, npix2, 8, 8, st);
  if (rc) return rc;
  return xf::launch_block1_tail(ctx, a2s, d_xn, B, H / 4, W / 4, a2s + npix2 * 16, nullptr, d_x1s, st);
}

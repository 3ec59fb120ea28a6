// Input gradient of the stem: d(clip) of the 1x7x7, stride (1,2,2), pad (0,3,3) spatial convolution
// (r21d_byol.py:198), from the stem unit's d(raw) (bf16 NDHWC, the tensor the BatchNorm backward of that unit writes).
//
//   dx[n][c][t][h][w] = sum over co < cout, kh, kw with oh = (h + 3 - kh) / 2 and ow = (w + 3 - kw) / 2 integral and
//                       inside the d(raw) plane of  g[n][t][oh][ow][co] * bf16(w[co][c][0][kh][kw])
//
// The weight is rounded to bf16 as the packed weights of every other dgrad are, so each product of two bf16 values is
// exact in fp32 and every fmaf is one rounded addition.  The order is fixed: channel pairs (2p, 2p + 1) ascending, then
// kh ascending, then kw ascending, then the two channels of the pair; a float32 stand-in reproduces the bits
// (tests/emulate_stem_dgrad.py).  No atomics: one thread owns each output element.
//
// Tiling: tiles of (n, t, 8 rows, 64 columns) of the clip, taken in grid strides by persistent CTAs (two per SM) that
// stage the weights once.  A warp covers one row parity and one column parity, so
// its tap counts (3 or 4 per axis) are uniform; each thread owns rows h and h + 2 of one column, which read the same
// weight with d(raw) rows oh and oh + 1.  The d(raw) tile (7 x 35 positions, channel pairs as bf16x2 words, pair-major:
// the lanes of a warp read consecutive words) and the weights (float4 {c0, c1, c2, 0} per (co, kh, kw), read as warp
// broadcasts) are staged in shared memory; the fp32 result goes back through shared memory for 16-byte stores.
#include "common.h"

#include <cuda_bf16.h>

namespace cstp {

constexpr int kSdThreads = 256;
constexpr int kSdTileH = 8;
constexpr int kSdTileW = 64;
constexpr int kSdRows = kSdTileH / 2 + 3;      // d(raw) rows one tile reads
constexpr int kSdCols = kSdTileW / 2 + 3;
constexpr int kSdPlane = kSdRows * kSdCols;
constexpr int kSdMaxCout = 128;

static size_t stem_dgrad_smem_bytes(int cout) {
  const int pairs = (cout + 1) / 2;
  const size_t wbytes = sizeof(float4) * 2 * pairs * 49;
  size_t gbytes = sizeof(uint32_t) * pairs * kSdPlane;
  const size_t obytes = sizeof(float) * 3 * kSdTileH * kSdTileW;
  if (gbytes < obytes) gbytes = obytes;
  return wbytes + gbytes;
}

__device__ __forceinline__ float bf16_lo(uint32_t v) { return __uint_as_float(v << 16); }
__device__ __forceinline__ float bf16_hi(uint32_t v) { return __uint_as_float(v & 0xffff0000u); }

template <int NKH, int NKW>
__device__ __forceinline__ void stem_dgrad_accumulate(float (&acc)[2][3], const uint32_t* __restrict__ gs,
                                                      const float4* __restrict__ ws, int pairs, int row0, int col0) {
  // row0 / col0: tile-local d(raw) row and column of the first tap (kh = kh0, kw = kw0); each further tap steps back one
#pragma unroll 1
  for (int p = 0; p < pairs; ++p) {
    const uint32_t* g = gs + p * kSdPlane;
    const float4* w0 = ws + (2 * p) * 49;
    const float4* w1 = w0 + 49;
#pragma unroll
    for (int i = 0; i < NKH; ++i) {
      const int kh = (NKH == 4 ? 0 : 1) + 2 * i;
#pragma unroll
      for (int j = 0; j < NKW; ++j) {
        const int kw = (NKW == 4 ? 0 : 1) + 2 * j;
        const int at = (row0 - i) * kSdCols + col0 - j;
        const uint32_t ga = g[at], gb = g[at + kSdCols];
        const float4 a = w0[kh * 7 + kw], b = w1[kh * 7 + kw];
        const float a0 = bf16_lo(ga), a1 = bf16_hi(ga), b0 = bf16_lo(gb), b1 = bf16_hi(gb);
        acc[0][0] = fmaf(a0, a.x, acc[0][0]);
        acc[0][1] = fmaf(a0, a.y, acc[0][1]);
        acc[0][2] = fmaf(a0, a.z, acc[0][2]);
        acc[1][0] = fmaf(b0, a.x, acc[1][0]);
        acc[1][1] = fmaf(b0, a.y, acc[1][1]);
        acc[1][2] = fmaf(b0, a.z, acc[1][2]);
        acc[0][0] = fmaf(a1, b.x, acc[0][0]);
        acc[0][1] = fmaf(a1, b.y, acc[0][1]);
        acc[0][2] = fmaf(a1, b.z, acc[0][2]);
        acc[1][0] = fmaf(b1, b.x, acc[1][0]);
        acc[1][1] = fmaf(b1, b.y, acc[1][1]);
        acc[1][2] = fmaf(b1, b.z, acc[1][2]);
      }
    }
  }
}

__global__ void __launch_bounds__(kSdThreads) stem_dgrad_kernel(const __nv_bfloat16* __restrict__ g, int Cg,
                                                                const float* __restrict__ w, int cout,
                                                                float* __restrict__ dx, int T, int H, int W,
                                                                int tiles_h, int tiles_w, long long ntiles) {
  extern __shared__ __align__(16) unsigned char sd_smem[];
  const int pairs = (cout + 1) / 2;
  float4* ws = reinterpret_cast<float4*>(sd_smem);
  uint32_t* gs = reinterpret_cast<uint32_t*>(sd_smem + sizeof(float4) * 2 * pairs * 49);
  const int tid = threadIdx.x;
  // weights: ws[co][kh*7 + kw] = {bf16(w[co][0][kh][kw]), bf16(w[co][1]..), bf16(w[co][2]..), 0}; co >= cout is zero
  for (int i = tid; i < 2 * pairs * 49; i += kSdThreads) {
    const int co = i / 49, k = i % 49;
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (co < cout) {
      const float* src = w + static_cast<long long>(co) * 3 * 49 + k;
      v.x = __bfloat162float(__float2bfloat16_rn(src[0]));
      v.y = __bfloat162float(__float2bfloat16_rn(src[49]));
      v.z = __bfloat162float(__float2bfloat16_rn(src[98]));
    }
    ws[i] = v;
  }
  const uint32_t* g32 = reinterpret_cast<const uint32_t*>(g);
  const int Ho = H / 2, Wo = W / 2;
  const int warp = tid >> 5, lane = tid & 31;
  const int hp = warp & 1, wp = (warp >> 1) & 1, rq = warp >> 2;
  const int hl = rq * 4 + hp;                   // tile-local rows hl and hl + 2
  const int wl = 2 * lane + wp;                 // tile-local column
  // first tap kh0 = 1 - hp: oh = (h + 3 - kh0) / 2, tile-local row = that - oh_lo
  const int row0 = (hl + 2 + hp) / 2 + 1;
  const int col0 = (wl + 2 + wp) / 2 + 1;
  float* os = reinterpret_cast<float*>(gs);     // [c][row][col] of the tile (after the accumulation)

  // persistent CTAs: the weights are staged once, the tiles are taken in grid strides
  for (long long tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
    const int tw = static_cast<int>(tile % tiles_w);
    const long long b = tile / tiles_w;
    const int th = static_cast<int>(b % tiles_h);
    const long long nt = b / tiles_h;             // n * T + t
    const int n = static_cast<int>(nt / T), t = static_cast<int>(nt % T);
    const int h0 = th * kSdTileH, w0 = tw * kSdTileW;
    const int oh_lo = h0 / 2 - 1, ow_lo = w0 / 2 - 1;
    __syncthreads();                              // the previous tile's output staging (os aliases gs) has been read
    // d(raw) tile: gs[p][r][c] = channels (2p, 2p + 1) of g[n][t][oh_lo + r][ow_lo + c], zero outside the plane
    const long long plane = nt * Ho;
    for (int i = tid; i < pairs * kSdPlane; i += kSdThreads) {
      const int p = i % pairs, rc = i / pairs;
      const int r = rc / kSdCols, c = rc % kSdCols;
      const int oh = oh_lo + r, ow = ow_lo + c;
      uint32_t v = 0u;
      if (oh >= 0 && oh < Ho && ow >= 0 && ow < Wo) {
        v = g32[(((plane + oh) * Wo + ow) * Cg >> 1) + p];
        if (2 * p + 1 >= cout) v &= 0xffffu;
      }
      gs[p * kSdPlane + rc] = v;
    }
    __syncthreads();

    float acc[2][3] = {{0.f, 0.f, 0.f}, {0.f, 0.f, 0.f}};
    if (hp) {
      if (wp) stem_dgrad_accumulate<4, 4>(acc, gs, ws, pairs, row0, col0);
      else stem_dgrad_accumulate<4, 3>(acc, gs, ws, pairs, row0, col0);
    } else {
      if (wp) stem_dgrad_accumulate<3, 4>(acc, gs, ws, pairs, row0, col0);
      else stem_dgrad_accumulate<3, 3>(acc, gs, ws, pairs, row0, col0);
    }
    __syncthreads();
  #pragma unroll
    for (int c = 0; c < 3; ++c) {
      os[(c * kSdTileH + hl) * kSdTileW + wl] = acc[0][c];
      os[(c * kSdTileH + hl + 2) * kSdTileW + wl] = acc[1][c];
    }
    __syncthreads();
    for (int i = tid; i < 3 * kSdTileH * kSdTileW / 4; i += kSdThreads) {
      const int c = i / (kSdTileH * kSdTileW / 4), rem = i % (kSdTileH * kSdTileW / 4);
      const int r = rem / (kSdTileW / 4), q = rem % (kSdTileW / 4);
      const int h = h0 + r, x = w0 + 4 * q;
      if (h < H && x < W) {
        const float4 v = reinterpret_cast<const float4*>(os)[(c * kSdTileH + r) * (kSdTileW / 4) + q];
        float* dst = dx + ((((static_cast<long long>(n) * 3 + c) * T + t) * H + h) * W + x);
        *reinterpret_cast<float4*>(dst) = v;
      }
    }
  }
}

}  // namespace cstp

using namespace cstp;

extern "C" int cstp_stem_dgrad(const void* g, int Cg, const float* w, int cout, float* dx, int N, int T, int H, int W,
                               void* stream) {
  CSTP_REQUIRE(g && w && dx && N > 0 && T > 0 && H > 0 && W > 0 && H % 2 == 0 && W % 4 == 0);
  CSTP_REQUIRE(cout > 0 && cout <= kSdMaxCout && Cg % 2 == 0 && Cg >= cout);
  CSTP_REQUIRE((reinterpret_cast<uintptr_t>(g) % 4) == 0 && (reinterpret_cast<uintptr_t>(dx) % 16) == 0 &&
               (reinterpret_cast<uintptr_t>(w) % 4) == 0);
  const size_t smem = stem_dgrad_smem_bytes(cout);
  static bool attr_set = false;
  if (!attr_set) {
    CSTP_CUDA(cudaFuncSetAttribute(stem_dgrad_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                   static_cast<int>(stem_dgrad_smem_bytes(kSdMaxCout))));
    attr_set = true;
  }
  const int tiles_h = (H + kSdTileH - 1) / kSdTileH, tiles_w = (W + kSdTileW - 1) / kSdTileW;
  const long long tiles = static_cast<long long>(N) * T * tiles_h * tiles_w;
  const long long grid = tiles < 2LL * num_sms() ? tiles : 2LL * num_sms();     // two 107 KB CTAs fit an SM
  stem_dgrad_kernel<<<static_cast<unsigned>(grid), kSdThreads, smem, static_cast<cudaStream_t>(stream)>>>(
      static_cast<const __nv_bfloat16*>(g), Cg, w, cout, dx, T, H, W, tiles_h, tiles_w, tiles);
  CSTP_LAUNCHED();
  return CSTP_OK;
}

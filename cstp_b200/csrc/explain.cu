// Grad-CAM of a finetuned classifier (cstp_b200.explain): the seed of the score's backward pass, the class-activation map
// of one stage and its trilinear upsampling to the clip with per-clip min-max normalisation.
//
//   cam_seed      k[b] = classes[b], or the argmax over the n_cls valid logit columns (ties to the lower class, the rule
//                 of cstp_video_finalize); dlogits[b] = one-hot(k[b]).  Rows >= n and padding columns are zero.
//   gradcam       alpha[b][c] = (sum over positions p of dA[b][p][c]) / P;  cam[b][p] = relu(sum_c alpha[b][c] * A[b][p][c])
//   cam_upsample  F.interpolate(mode="trilinear", align_corners=False) to T x H x W, then (v - min) / (max - min) per clip
//                 (all zeros where max == min)
//
// Every floating-point operation is one separately rounded _rn intrinsic in a fixed order (no contraction, no atomics),
// so a numpy float32 stand-in reproduces the bits (tests/emulate_explain.py):
//   * the position sum of alpha runs in eight interleaved lanes (lane j adds positions j, j + 8, j + 16, ... in order),
//     whose partials are then added in lane order, and is divided by P;
//   * the channel sum of the map adds the rounded products alpha_c * A_c in ascending channel order;
//   * the upsampling takes torch's source index per axis -- scale = in / out, src = max(scale * (d + 0.5) - 0.5, 0),
//     i0 = (int)src, i1 = i0 + (i0 < in - 1), l = src - i0 -- and blends along w, then h, then t as a + l * (b - a),
//     which keeps a constant map exactly constant (the l0 * a + l1 * b form can move it by an ulp, which the min-max
//     normalisation would blow up to [0, 1]).
// The activations and gradients are the bf16 NDHWC tensors of the engine (channels padded to Cp; padding is ignored).
#include "common.h"

#include <cuda_bf16.h>

namespace cstp {

constexpr int kSeedThreads = 128;
constexpr int kAlphaLanes = 8;               // interleaved position lanes of the alpha sum
constexpr int kAlphaChannels = 32;           // channels of one alpha CTA (one warp per lane)
constexpr int kCamThreads = 256;
constexpr int kCamMaxC = 512;
constexpr int kUpThreads = 1024;

// (v, i) ranks ahead of (w, j): larger value first, the lower class index on equal values
__device__ __forceinline__ bool cam_ranks_before(float v, int i, float w, int j) {
  return v > w || (v == w && i < j);
}

__global__ void __launch_bounds__(kSeedThreads) cam_seed_kernel(const float* __restrict__ logits, int ld, int n, int n_cls,
                                                                const int64_t* __restrict__ classes_in,
                                                                int64_t* __restrict__ classes_out,
                                                                float* __restrict__ dlogits) {
  __shared__ float s_val[kSeedThreads / 32];
  __shared__ int s_idx[kSeedThreads / 32];
  __shared__ int s_k;
  const int b = blockIdx.x;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  int k = -1;
  if (b < n && classes_in != nullptr) {
    k = static_cast<int>(classes_in[b]);
  } else if (b < n) {
    const float* row = logits + static_cast<long long>(b) * ld;
    float bv = -INFINITY;
    int bi = -1;
    for (int c = threadIdx.x; c < n_cls; c += blockDim.x) {
      const float v = row[c];
      if (bi < 0 || cam_ranks_before(v, c, bv, bi)) bv = v, bi = c;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const float ov = __shfl_xor_sync(0xffffffffu, bv, o);
      const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
      if (oi >= 0 && (bi < 0 || cam_ranks_before(ov, oi, bv, bi))) bv = ov, bi = oi;
    }
    if (lane == 0) s_val[warp] = bv, s_idx[warp] = bi;
    __syncthreads();
    if (threadIdx.x == 0) {
      float v = s_val[0];
      int i = s_idx[0];
      for (int w = 1; w < kSeedThreads / 32; ++w)
        if (s_idx[w] >= 0 && (i < 0 || cam_ranks_before(s_val[w], s_idx[w], v, i))) v = s_val[w], i = s_idx[w];
      s_k = i;
    }
    __syncthreads();
    k = s_k;
  }
  if (threadIdx.x == 0) classes_out[b] = b < n ? k : 0;
  float* d = dlogits + static_cast<long long>(b) * ld;
  for (int c = threadIdx.x; c < ld; c += blockDim.x) d[c] = (b < n && c == k && c < n_cls) ? 1.f : 0.f;
}

// alpha[b][c0 + x] for one clip b and 32 channels: lane j = threadIdx.x / 32 sums positions j, j + 8, ... in order
__global__ void __launch_bounds__(kAlphaLanes * kAlphaChannels) gradcam_alpha_kernel(const __nv_bfloat16* __restrict__ dA,
                                                                                   long long P, int C, int Cp,
                                                                                   float* __restrict__ alpha) {
  __shared__ float part[kAlphaLanes][kAlphaChannels];
  const int b = blockIdx.y;
  const int cl = threadIdx.x & (kAlphaChannels - 1), j = threadIdx.x / kAlphaChannels;
  const int c = blockIdx.x * kAlphaChannels + cl;
  float acc = 0.f;
  if (c < C) {
    const __nv_bfloat16* src = dA + static_cast<long long>(b) * P * Cp + c;
    long long p = j;
    for (; p + 3 * kAlphaLanes < P; p += 4 * kAlphaLanes) {
      const float v0 = __bfloat162float(src[p * Cp]);
      const float v1 = __bfloat162float(src[(p + kAlphaLanes) * Cp]);
      const float v2 = __bfloat162float(src[(p + 2 * kAlphaLanes) * Cp]);
      const float v3 = __bfloat162float(src[(p + 3 * kAlphaLanes) * Cp]);
      acc = __fadd_rn(__fadd_rn(__fadd_rn(__fadd_rn(acc, v0), v1), v2), v3);
    }
    for (; p < P; p += kAlphaLanes) acc = __fadd_rn(acc, __bfloat162float(src[p * Cp]));
  }
  part[j][cl] = acc;
  __syncthreads();
  if (j == 0 && c < C) {
    float s = part[0][cl];
#pragma unroll
    for (int q = 1; q < kAlphaLanes; ++q) s = __fadd_rn(s, part[q][cl]);
    alpha[static_cast<long long>(b) * C + c] = __fdiv_rn(s, static_cast<float>(P));
  }
}

// cam[b][p]: one thread per position, channels in ascending order (16-byte loads of eight bf16 channels)
__global__ void __launch_bounds__(kCamThreads) gradcam_map_kernel(const __nv_bfloat16* __restrict__ A, long long P, int C,
                                                                  int Cp, const float* __restrict__ alpha,
                                                                  float* __restrict__ cam) {
  __shared__ float s_alpha[kCamMaxC];
  const int b = blockIdx.y;
  for (int c = threadIdx.x; c < C; c += blockDim.x) s_alpha[c] = alpha[static_cast<long long>(b) * C + c];
  __syncthreads();
  const long long p = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (p >= P) return;
  const uint4* src = reinterpret_cast<const uint4*>(A + (static_cast<long long>(b) * P + p) * Cp);
  float acc = 0.f;
  for (int v = 0; v < C / 8; ++v) {
    const uint4 q = src[v];
    const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&q);
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const float2 f = __bfloat1622float2(h[e]);
      acc = __fadd_rn(acc, __fmul_rn(s_alpha[8 * v + 2 * e], f.x));
      acc = __fadd_rn(acc, __fmul_rn(s_alpha[8 * v + 2 * e + 1], f.y));
    }
  }
  cam[static_cast<long long>(b) * P + p] = acc > 0.f ? acc : 0.f;
}

struct UpAxis {
  int i0, i1;
  float l;
};

// torch's area_pixel_compute_source_index (align_corners=False, linear modes) and the neighbours it blends
__device__ __forceinline__ UpAxis up_axis(int d, int in, int out) {
  const float scale = __fdiv_rn(static_cast<float>(in), static_cast<float>(out));
  float src = __fsub_rn(__fmul_rn(scale, __fadd_rn(static_cast<float>(d), 0.5f)), 0.5f);
  src = src < 0.f ? 0.f : src;
  UpAxis a;
  a.i0 = static_cast<int>(src);
  a.i1 = a.i0 + (a.i0 < in - 1 ? 1 : 0);
  a.l = __fsub_rn(src, static_cast<float>(a.i0));
  return a;
}

__device__ __forceinline__ float up_mix(float a, float l, float b) {
  return __fadd_rn(a, __fmul_rn(l, __fsub_rn(b, a)));
}

// One CTA per clip: the upsampled map is written with its min / max reduced on the way, then normalised in place
__global__ void __launch_bounds__(kUpThreads) cam_upsample_kernel(const float* __restrict__ cam, int t, int h, int w,
                                                                  int T, int H, int W, float* __restrict__ out) {
  __shared__ float s_min[kUpThreads / 32], s_max[kUpThreads / 32];
  const int b = blockIdx.x;
  const float* x = cam + static_cast<long long>(b) * t * h * w;
  float* o = out + static_cast<long long>(b) * T * H * W;
  const long long total = static_cast<long long>(T) * H * W;
  float mn = INFINITY, mx = -INFINITY;
  for (long long i = threadIdx.x; i < total; i += blockDim.x) {
    const int ow = static_cast<int>(i % W), oh = static_cast<int>((i / W) % H), ot = static_cast<int>(i / (W * H));
    const UpAxis at = up_axis(ot, t, T), ah = up_axis(oh, h, H), aw = up_axis(ow, w, W);
    auto plane = [&](int ti) {
      const float* r0 = x + (static_cast<long long>(ti) * h + ah.i0) * w;
      const float* r1 = x + (static_cast<long long>(ti) * h + ah.i1) * w;
      return up_mix(up_mix(r0[aw.i0], aw.l, r0[aw.i1]), ah.l, up_mix(r1[aw.i0], aw.l, r1[aw.i1]));
    };
    const float v = up_mix(plane(at.i0), at.l, plane(at.i1));
    o[i] = v;
    mn = fminf(mn, v);
    mx = fmaxf(mx, v);
  }
#pragma unroll
  for (int k = 16; k > 0; k >>= 1) {
    mn = fminf(mn, __shfl_xor_sync(0xffffffffu, mn, k));
    mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, k));
  }
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (lane == 0) s_min[warp] = mn, s_max[warp] = mx;
  __syncthreads();
  mn = s_min[0];
  mx = s_max[0];
  for (int k = 1; k < kUpThreads / 32; ++k) mn = fminf(mn, s_min[k]), mx = fmaxf(mx, s_max[k]);
  const bool flat = !(mx > mn);
  const float range = __fsub_rn(mx, mn);
  // each thread reads back only the elements it wrote
  for (long long i = threadIdx.x; i < total; i += blockDim.x) o[i] = flat ? 0.f : __fdiv_rn(__fsub_rn(o[i], mn), range);
}

}  // namespace cstp

using namespace cstp;

extern "C" int cstp_cam_seed(const float* logits, int B, int ld, int n, int n_cls, const int64_t* classes_in,
                             int64_t* classes_out, float* dlogits, void* stream) {
  CSTP_REQUIRE(logits && classes_out && dlogits && B > 0 && n > 0 && n <= B && n_cls > 0 && n_cls <= ld);
  cam_seed_kernel<<<B, kSeedThreads, 0, static_cast<cudaStream_t>(stream)>>>(logits, ld, n, n_cls, classes_in,
                                                                              classes_out, dlogits);
  CSTP_LAUNCHED();
  return CSTP_OK;
}

extern "C" int cstp_gradcam(const void* act, const void* grad, int n, long long P, int C, int Cp, float* alpha, float* cam,
                            void* stream) {
  CSTP_REQUIRE(act && grad && alpha && cam && n > 0 && P > 0 && C > 0 && C <= kCamMaxC && C % 8 == 0 && Cp >= C &&
               Cp % 8 == 0);
  CSTP_REQUIRE((reinterpret_cast<uintptr_t>(act) % 16) == 0 && (reinterpret_cast<uintptr_t>(grad) % 2) == 0);
  const cudaStream_t st = static_cast<cudaStream_t>(stream);
  gradcam_alpha_kernel<<<dim3(ceil_div(C, kAlphaChannels), n), kAlphaLanes * kAlphaChannels, 0, st>>>(
      static_cast<const __nv_bfloat16*>(grad), P, C, Cp, alpha);
  CSTP_LAUNCHED();
  gradcam_map_kernel<<<dim3(ceil_div(P, kCamThreads), n), kCamThreads, 0, st>>>(static_cast<const __nv_bfloat16*>(act), P,
                                                                                 C, Cp, alpha, cam);
  CSTP_LAUNCHED();
  return CSTP_OK;
}

extern "C" int cstp_cam_upsample(const float* cam, int n, int t, int h, int w, int T, int H, int W, float* out,
                                 void* stream) {
  CSTP_REQUIRE(cam && out && n > 0 && t > 0 && h > 0 && w > 0 && T > 0 && H > 0 && W > 0);
  cam_upsample_kernel<<<n, kUpThreads, 0, static_cast<cudaStream_t>(stream)>>>(cam, t, h, w, T, H, W, out);
  CSTP_LAUNCHED();
  return CSTP_OK;
}

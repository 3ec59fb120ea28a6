// Video-level test scoring (test.py:76-93): the logits of a video's clips are averaged and ranked on the device.
// A video's clips may arrive in several consecutive batches, so its fp32 sum lives in a slot that keeps accumulating
// across launches.  Additions run in clip order inside one thread per class column (no float atomics): two runs give
// identical bits, and the sum equals a sequential fp32 loop over the video's clips.  Both launches read their work lists
// from device tables the host rewrites in place, so they can sit in a captured CUDA graph; entries with a count <= 0
// are skipped.  Latency-bound work on a few kilobytes: one CTA per table entry.
#include "common.h"

namespace cstp {

constexpr int kVideoThreads = 128;
constexpr int kVideoMaxK = 8;

__global__ void __launch_bounds__(kVideoThreads) video_accumulate_kernel(const float* __restrict__ logits, int rows, int ld,
                                                                         int n_cls, const int32_t* __restrict__ seg,
                                                                         float* __restrict__ sums, int n_slots) {
  const int slot = seg[3 * blockIdx.x], first = seg[3 * blockIdx.x + 1], count = seg[3 * blockIdx.x + 2];
  if (count <= 0 || slot < 0 || slot >= n_slots || first < 0 || first + count > rows) return;
  float* s = sums + static_cast<long long>(slot) * n_cls;
  for (int c = threadIdx.x; c < n_cls; c += blockDim.x) {
    float acc = s[c];
    for (int r = first; r < first + count; ++r) acc += logits[static_cast<long long>(r) * ld + c];
    s[c] = acc;
  }
}

// (v, i) ranks ahead of (w, j): larger value first, the lower class index on equal values
__device__ __forceinline__ bool ranks_before(float v, int i, float w, int j) {
  return v > w || (v == w && i < j);
}

__global__ void __launch_bounds__(kVideoThreads) video_finalize_kernel(float* __restrict__ sums, int n_slots, int n_cls,
                                                                       const int32_t* __restrict__ fin, int n_videos, int k,
                                                                       const int64_t* __restrict__ labels,
                                                                       float* __restrict__ mean_out,
                                                                       int64_t* __restrict__ topk_out,
                                                                       unsigned long long* __restrict__ hits) {
  __shared__ float s_val[kVideoThreads / 32];
  __shared__ int s_idx[kVideoThreads / 32];
  __shared__ int s_pick[kVideoMaxK];
  const int slot = fin[3 * blockIdx.x], count = fin[3 * blockIdx.x + 1], video = fin[3 * blockIdx.x + 2];
  if (count <= 0 || slot < 0 || slot >= n_slots || video < 0 || video >= n_videos) return;
  float* s = sums + static_cast<long long>(slot) * n_cls;
  const float n = static_cast<float>(count);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int kk = min(max(k, 5), n_cls);                 // top-5 hits are counted even when fewer indices are written
  float prev_v = INFINITY;
  int prev_i = -1;
  for (int j = 0; j < kk; ++j) {
    // best (mean, class) that ranks strictly behind the previous pick
    float bv = -INFINITY;
    int bi = -1;
    for (int c = threadIdx.x; c < n_cls; c += blockDim.x) {
      const float v = s[c] / n;
      if (j > 0 && !ranks_before(prev_v, prev_i, v, c)) continue;
      if (bi < 0 || ranks_before(v, c, bv, bi)) bv = v, bi = c;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const float ov = __shfl_xor_sync(0xffffffffu, bv, o);
      const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
      if (oi >= 0 && (bi < 0 || ranks_before(ov, oi, bv, bi))) bv = ov, bi = oi;
    }
    if (lane == 0) s_val[warp] = bv, s_idx[warp] = bi;
    __syncthreads();
    if (threadIdx.x == 0) {
      float v = s_val[0];
      int i = s_idx[0];
      for (int w = 1; w < kVideoThreads / 32; ++w)
        if (s_idx[w] >= 0 && (i < 0 || ranks_before(s_val[w], s_idx[w], v, i))) v = s_val[w], i = s_idx[w];
      s_pick[j] = i;
      s_val[0] = v;
      s_idx[0] = i;
    }
    __syncthreads();
    prev_v = s_val[0];
    prev_i = s_idx[0];
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    for (int j = 0; j < k; ++j) topk_out[static_cast<long long>(video) * k + j] = j < kk ? s_pick[j] : -1;
    if (hits != nullptr) {
      const int64_t y = labels[video];
      bool in5 = false;
      for (int j = 0; j < min(5, kk); ++j) in5 |= s_pick[j] == y;
      if (s_pick[0] == y) atomicAdd(hits, 1ull);
      if (in5) atomicAdd(hits + 1, 1ull);
    }
  }
  // the slot is left zero for the next video that uses it
  for (int c = threadIdx.x; c < n_cls; c += blockDim.x) {
    if (mean_out != nullptr) mean_out[static_cast<long long>(video) * n_cls + c] = s[c] / n;
    s[c] = 0.f;
  }
}

}  // namespace cstp

using namespace cstp;

extern "C" int cstp_video_accumulate(const float* logits, int rows, int ld, int n_cls, const int32_t* seg, int n_seg,
                                     float* sums, int n_slots, void* stream) {
  CSTP_REQUIRE(logits && seg && sums && rows > 0 && n_cls > 0 && n_cls <= ld && n_seg > 0 && n_slots > 0);
  video_accumulate_kernel<<<n_seg, kVideoThreads, 0, static_cast<cudaStream_t>(stream)>>>(logits, rows, ld, n_cls, seg,
                                                                                          sums, n_slots);
  CSTP_LAUNCHED();
  return CSTP_OK;
}

extern "C" int cstp_video_finalize(float* sums, int n_slots, int n_cls, const int32_t* fin, int n_fin, int n_videos, int k,
                                   const int64_t* labels, float* mean_out, int64_t* topk_out, int64_t* hits,
                                   void* stream) {
  CSTP_REQUIRE(sums && fin && topk_out && n_slots > 0 && n_cls > 0 && n_fin > 0 && n_videos > 0);
  CSTP_REQUIRE(k >= 1 && k <= kVideoMaxK && (hits == nullptr || labels != nullptr));
  video_finalize_kernel<<<n_fin, kVideoThreads, 0, static_cast<cudaStream_t>(stream)>>>(
      sums, n_slots, n_cls, fin, n_videos, k, labels, mean_out, topk_out, reinterpret_cast<unsigned long long*>(hits));
  CSTP_LAUNCHED();
  return CSTP_OK;
}

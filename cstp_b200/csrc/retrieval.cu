// Nearest-neighbour video retrieval (the VCOP / Pace protocol): cosine similarity of every query feature against every
// gallery feature and the k best gallery rows per query, without ever writing the query x gallery matrix.
//
// Arithmetic is defined to the bit so that a float32 stand-in reproduces it and results do not depend on the tiling:
//   norm(x)   = max(sqrt(sum of squares), 1e-12), the squares summed lane-strided over a warp (lane l adds columns l,
//               l + 32, ... in order), then a fixed xor butterfly; y = x / norm, correctly rounded.
//   s(q, g)   = ((0 + q[0] g[0]) + q[1] g[1]) + ... + q[d-1] g[d-1], every product and sum rounded separately (no FMA).
// Neighbours are ranked by a strict total order -- similarity descending, then the lower gallery index -- so the top-k
// of a query is unique: any split of the gallery, merged, gives the same bits.  FP32 SIMT on purpose: bf16 / TF32 tensor
// cores round the features of one class (which sit close together) enough to reorder neighbours.
#include "common.h"

namespace cstp {

constexpr int kNormThreads = 256;

// One warp per row.
__global__ void __launch_bounds__(kNormThreads) l2_normalize_rows_kernel(const float* __restrict__ x, int n, int d, int ld,
                                                                        float* __restrict__ y) {
  const int row = (blockIdx.x * kNormThreads + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (row >= n) return;
  const float* xr = x + static_cast<long long>(row) * ld;
  float ss = 0.f;
  for (int j = lane; j < d; j += 32) ss = __fadd_rn(ss, __fmul_rn(xr[j], xr[j]));
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) ss = __fadd_rn(ss, __shfl_xor_sync(0xffffffffu, ss, o));
  const float nrm = fmaxf(__fsqrt_rn(ss), 1e-12f);
  float* yr = y + static_cast<long long>(row) * d;
  for (int j = lane; j < d; j += 32) yr[j] = __fdiv_rn(xr[j], nrm);
}

// ---- partial top-k: one CTA per (tile of kKnnBQ queries, gallery split)
constexpr int kKnnThreads = 256;
constexpr int kKnnBQ = 64;                      // query rows per CTA
constexpr int kKnnBG = 128;                     // gallery rows per shared-memory tile
constexpr int kKnnDK = 32;                      // feature columns staged per step
constexpr int kKnnMaxK = 64;
constexpr int kKnnMaxSplits = 32;               // one lane of the merge warp per split
constexpr int kQPad = kKnnBQ + 4;               // staged tiles are transposed ([column][row]); +4 keeps float4 alignment
constexpr int kGPad = kKnnBG + 4;
constexpr int kSPad = kKnnBG + 1;               // similarity tile [query][gallery]: the owner threads read rows
constexpr int kStageFloats = kKnnDK * (kQPad + kGPad);
constexpr int kUnionFloats = kStageFloats > kKnnBQ * kSPad ? kStageFloats : kKnnBQ * kSPad;

// (v, i) ranks ahead of (w, j): larger similarity first, the lower gallery index on equal values
__device__ __forceinline__ bool knn_before(float v, int i, float w, int j) { return v > w || (v == w && i < j); }

static size_t knn_smem_bytes(int k) { return sizeof(float) * kUnionFloats + 2 * sizeof(float) * k * kKnnBQ; }

// One feature column j of a thread's 4x8 register tile: every chain adds its rounded product (no contraction).
__device__ __forceinline__ void knn_column_step(float (&acc)[4][8], const float* Qs, const float* Gs, int j, int tq,
                                                int tg) {
  const float4 a = *reinterpret_cast<const float4*>(Qs + j * kQPad + tq * 4);
  const float4 b0 = *reinterpret_cast<const float4*>(Gs + j * kGPad + tg * 4);
  const float4 b1 = *reinterpret_cast<const float4*>(Gs + j * kGPad + 64 + tg * 4);
  const float av[4] = {a.x, a.y, a.z, a.w};
  const float bv[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
#pragma unroll
  for (int x = 0; x < 4; ++x)
#pragma unroll
    for (int y = 0; y < 8; ++y) acc[x][y] = __fadd_rn(acc[x][y], __fmul_rn(av[x], bv[y]));
}

// Thread (tq, tg) = (t / 16, t % 16) owns queries 4 tq .. 4 tq + 3 against gallery columns 4 tg .. 4 tg + 3 and
// 64 + 4 tg .. 64 + 4 tg + 3 of the tile: 32 independent accumulation chains.  After a tile, its similarities go to
// shared memory, and thread t < kKnnBQ merges row t into query t's running top-k (kept sorted, [k][kKnnBQ]); candidates
// that do not beat the current k-th entry cost one comparison.
__global__ void __launch_bounds__(kKnnThreads, 3) knn_partial_kernel(const float* __restrict__ q, int nq,
                                                                    const float* __restrict__ g, int ng, int d, int k,
                                                                    int splits, float* __restrict__ part_val,
                                                                    int32_t* __restrict__ part_idx) {
  extern __shared__ float4 smem4[];
  float* sm = reinterpret_cast<float*>(smem4);
  float* Qs = sm;                                // [kKnnDK][kQPad]
  float* Gs = sm + kKnnDK * kQPad;               // [kKnnDK][kGPad]
  float* S = sm;                                 // [kKnnBQ][kSPad], reuses the staging area after a tile's last step
  float* lv = sm + kUnionFloats;                 // [k][kKnnBQ]
  int* li = reinterpret_cast<int*>(lv + k * kKnnBQ);
  const int q0 = blockIdx.x * kKnnBQ, split = blockIdx.y;
  const int g_begin = static_cast<int>(static_cast<long long>(ng) * split / splits);
  const int g_end = static_cast<int>(static_cast<long long>(ng) * (split + 1) / splits);
  const int t = threadIdx.x, tq = t >> 4, tg = t & 15;
  for (int i = t; i < k * kKnnBQ; i += kKnnThreads) lv[i] = -INFINITY, li[i] = -1;

  for (int g0 = g_begin; g0 < g_end; g0 += kKnnBG) {
    float acc[4][8];
#pragma unroll
    for (int a = 0; a < 4; ++a)
#pragma unroll
      for (int b = 0; b < 8; ++b) acc[a][b] = 0.f;
    for (int j0 = 0; j0 < d; j0 += kKnnDK) {
      __syncthreads();                           // the previous step (or the previous tile's top-k pass) is done
      const int dk = min(kKnnDK, d - j0);        // a multiple of 4
      for (int e = t; e < kKnnBQ * kKnnDK / 4; e += kKnnThreads) {
        const int r = e >> 3, c = (e & 7) * 4;
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (q0 + r < nq && c < dk) v = *reinterpret_cast<const float4*>(q + static_cast<long long>(q0 + r) * d + j0 + c);
        Qs[(c + 0) * kQPad + r] = v.x;
        Qs[(c + 1) * kQPad + r] = v.y;
        Qs[(c + 2) * kQPad + r] = v.z;
        Qs[(c + 3) * kQPad + r] = v.w;
      }
      for (int e = t; e < kKnnBG * kKnnDK / 4; e += kKnnThreads) {
        const int r = e >> 3, c = (e & 7) * 4;
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (g0 + r < g_end && c < dk) v = *reinterpret_cast<const float4*>(g + static_cast<long long>(g0 + r) * d + j0 + c);
        Gs[(c + 0) * kGPad + r] = v.x;
        Gs[(c + 1) * kGPad + r] = v.y;
        Gs[(c + 2) * kGPad + r] = v.z;
        Gs[(c + 3) * kGPad + r] = v.w;
      }
      __syncthreads();
      if (dk == kKnnDK) {
#pragma unroll
        for (int j = 0; j < kKnnDK; ++j) knn_column_step(acc, Qs, Gs, j, tq, tg);
      } else {
        for (int j = 0; j < dk; ++j) knn_column_step(acc, Qs, Gs, j, tq, tg);
      }
    }
    __syncthreads();                             // every thread is done reading the staged columns
#pragma unroll
    for (int x = 0; x < 4; ++x)
#pragma unroll
      for (int y = 0; y < 8; ++y) S[(tq * 4 + x) * kSPad + (y < 4 ? tg * 4 + y : 64 + tg * 4 + y - 4)] = acc[x][y];
    __syncthreads();
    if (t < kKnnBQ && q0 + t < nq) {
      const int n = min(kKnnBG, g_end - g0);
      float tv = lv[(k - 1) * kKnnBQ + t];
      int ti = li[(k - 1) * kKnnBQ + t];
      for (int c = 0; c < n; ++c) {
        const float v = S[t * kSPad + c];
        const int gi = g0 + c;
        if (ti >= 0 && !knn_before(v, gi, tv, ti)) continue;
        int p = k - 1;                           // insertion into the sorted list; empty entries (index -1) sit last
        for (; p > 0; --p) {
          const int pi = li[(p - 1) * kKnnBQ + t];
          const float pv = lv[(p - 1) * kKnnBQ + t];
          if (pi >= 0 && !knn_before(v, gi, pv, pi)) break;
          lv[p * kKnnBQ + t] = pv;
          li[p * kKnnBQ + t] = pi;
        }
        lv[p * kKnnBQ + t] = v;
        li[p * kKnnBQ + t] = gi;
        tv = lv[(k - 1) * kKnnBQ + t];
        ti = li[(k - 1) * kKnnBQ + t];
      }
    }
  }
  __syncthreads();
  for (int i = t; i < kKnnBQ * k; i += kKnnThreads) {
    const int r = i / k, j = i - r * k;
    if (q0 + r >= nq) continue;
    const long long o = (static_cast<long long>(split) * nq + q0 + r) * k + j;
    part_val[o] = lv[j * kKnnBQ + r];
    part_idx[o] = li[j * kKnnBQ + r];
  }
}

// One warp per query: lane s holds the head of split s's sorted list; k rounds of a warp-wide max under the total order.
// Every gallery index lives in exactly one split, so the winner's lane is the one whose head carries the winning index.
__global__ void __launch_bounds__(256) knn_merge_kernel(const float* __restrict__ part_val,
                                                        const int32_t* __restrict__ part_idx, int nq, int k, int splits,
                                                        int64_t* __restrict__ idx_out, float* __restrict__ sim_out,
                                                        const int64_t* __restrict__ q_labels,
                                                        const int64_t* __restrict__ g_labels,
                                                        const int32_t* __restrict__ cutoffs, int n_cut,
                                                        unsigned long long* __restrict__ hits) {
  const int qi = (blockIdx.x * 256 + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (qi >= nq) return;
  const long long base = (static_cast<long long>(lane) * nq + qi) * k;
  const int64_t y = hits != nullptr ? q_labels[qi] : 0;
  int head = 0, first_hit = k;
  for (int j = 0; j < k; ++j) {
    float v = -INFINITY;
    int i = -1;
    if (lane < splits && head < k) v = part_val[base + head], i = part_idx[base + head];
    float bv = v;
    int bi = i;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const float ov = __shfl_xor_sync(0xffffffffu, bv, o);
      const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
      if (oi >= 0 && (bi < 0 || knn_before(ov, oi, bv, bi))) bv = ov, bi = oi;
    }
    if (bi >= 0 && i == bi) ++head;
    if (lane == 0) {
      idx_out[static_cast<long long>(qi) * k + j] = bi;
      sim_out[static_cast<long long>(qi) * k + j] = bi >= 0 ? bv : -INFINITY;
      if (hits != nullptr && bi >= 0 && first_hit == k && g_labels[bi] == y) first_hit = j;
    }
  }
  if (lane == 0 && hits != nullptr)
    for (int c = 0; c < n_cut; ++c)
      if (first_hit < cutoffs[c]) atomicAdd(hits + c, 1ull);
}

}  // namespace cstp

using namespace cstp;

extern "C" int cstp_l2_normalize_rows(const float* x, int n, int d, int ld, float* y, void* stream) {
  CSTP_REQUIRE(x && y && n > 0 && d > 0 && ld >= d);
  const int rows_per_cta = kNormThreads / 32;
  l2_normalize_rows_kernel<<<(n + rows_per_cta - 1) / rows_per_cta, kNormThreads, 0, static_cast<cudaStream_t>(stream)>>>(
      x, n, d, ld, y);
  CSTP_LAUNCHED();
  return CSTP_OK;
}

extern "C" int cstp_knn_partial(const float* q, int nq, const float* g, int ng, int d, int k, int splits, float* part_val,
                                int32_t* part_idx, void* stream) {
  CSTP_REQUIRE(q && g && part_val && part_idx && nq > 0 && ng > 0 && d > 0);
  CSTP_REQUIRE(d % 4 == 0 && k >= 1 && k <= kKnnMaxK && splits >= 1 && splits <= kKnnMaxSplits);
  CSTP_REQUIRE(reinterpret_cast<uintptr_t>(q) % 16 == 0 && reinterpret_cast<uintptr_t>(g) % 16 == 0);
  const size_t smem = knn_smem_bytes(k);
  CSTP_CUDA(cudaFuncSetAttribute(knn_partial_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
  const dim3 grid((nq + kKnnBQ - 1) / kKnnBQ, splits);
  knn_partial_kernel<<<grid, kKnnThreads, smem, static_cast<cudaStream_t>(stream)>>>(q, nq, g, ng, d, k, splits, part_val,
                                                                                  part_idx);
  CSTP_LAUNCHED();
  return CSTP_OK;
}

extern "C" int cstp_knn_merge(const float* part_val, const int32_t* part_idx, int nq, int k, int splits, int64_t* idx_out,
                              float* sim_out, const int64_t* q_labels, const int64_t* g_labels, const int32_t* cutoffs,
                              int n_cut, int64_t* hits, void* stream) {
  CSTP_REQUIRE(part_val && part_idx && idx_out && sim_out && nq > 0);
  CSTP_REQUIRE(k >= 1 && k <= kKnnMaxK && splits >= 1 && splits <= kKnnMaxSplits);
  CSTP_REQUIRE(hits == nullptr || (q_labels && g_labels && cutoffs && n_cut > 0));
  knn_merge_kernel<<<(nq + 7) / 8, 256, 0, static_cast<cudaStream_t>(stream)>>>(
      part_val, part_idx, nq, k, splits, idx_out, sim_out, q_labels, g_labels, cutoffs, n_cut,
      reinterpret_cast<unsigned long long*>(hits));
  CSTP_LAUNCHED();
  return CSTP_OK;
}

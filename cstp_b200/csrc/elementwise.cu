// HBM-bound kernels of the hot path: weight packing, stem row packing, training-mode BatchNorm (statistics,
// finalize, apply + ReLU + residual, backward reduce / apply), average pooling, column sums and casts.
// All activations are bf16 [rows][Cp] (NDHWC flattened), processed as 16-byte vectors of 8 channels.
// Replaces ATen/cuDNN batch_norm, relu, add, adaptive_avg_pool3d behind models/pace/r21d_byol.py:83-97,141-148,210-223.
#include "common.h"
#include "ptx.cuh"

namespace cstp {

__device__ __forceinline__ void unpack8(const uint4& v, float (&f)[8]) {
  f[0] = bf16_lo(v.x); f[1] = bf16_hi(v.x);
  f[2] = bf16_lo(v.y); f[3] = bf16_hi(v.y);
  f[4] = bf16_lo(v.z); f[5] = bf16_hi(v.z);
  f[6] = bf16_lo(v.w); f[7] = bf16_hi(v.w);
}
__device__ __forceinline__ uint4 pack8(const float (&f)[8]) {
  uint4 v;
  v.x = pack_bf16x2(f[0], f[1]);
  v.y = pack_bf16x2(f[2], f[3]);
  v.z = pack_bf16x2(f[4], f[5]);
  v.w = pack_bf16x2(f[6], f[7]);
  return v;
}

// ------------------------------------------------------------------------------------------- weight packing
__global__ void pack_weight_kernel(const float* __restrict__ w, int cout, int cin, int taps, int transpose,
                                   __nv_bfloat16* __restrict__ packed, int Rp, int Kc) {
  const long long total = static_cast<long long>(Rp) * taps * Kc;
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int c = static_cast<int>(i % Kc);
    const int tap = static_cast<int>((i / Kc) % taps);
    const int r = static_cast<int>(i / (static_cast<long long>(Kc) * taps));
    float v = 0.f;
    if (transpose == 0) {
      if (r < cout && c < cin) v = w[(static_cast<long long>(r) * cin + c) * taps + tap];
    } else if (transpose == 1) {
      if (r < cin && c < cout) v = w[(static_cast<long long>(c) * cin + r) * taps + tap];
    } else {
      // stem layout: w is (cout, 3, 1, 7, 7); tap = row pair j, packed column c = hpar*32 + kw*3 + ci (cstp_stem_pack)
      const int k = c & 31, kh = 2 * tap + (c >> 5) - 1;
      if (r < cout && c < 64 && k < 21 && kh >= 0 && kh < 7) v = w[((static_cast<long long>(r) * 3 + k % 3) * 7 + kh) * 7 + k / 3];
    }
    packed[i] = __float2bfloat16_rn(v);
  }
}

// All weight tensors of a network in ONE launch: job j packs w_j (fp32 reference layout) into packed_j exactly as
// pack_weight_kernel does; `jobs` is a device table of 8 int64 per job {w, packed, cout, cin, taps, transpose, Rp, Kc},
// `prefix[j]` the first global element index of job j (prefix[n_jobs] = total).  97 launches per step -> 2.
__global__ void __launch_bounds__(256) pack_weights_batched_kernel(const long long* __restrict__ jobs,
                                                                   const long long* __restrict__ prefix, int n_jobs,
                                                                   long long total) {
  // Each CTA owns a contiguous span of kPackSpan elements: ONE binary search per CTA (first element of the span), then
  // every thread walks forward from there (a span rarely crosses more than one job boundary); 32-bit index arithmetic
  // inside a job.  The per-element search + 64-bit div/mod version took 0.28 ms per launch for 0.2 GB of traffic.
  constexpr int kPackSpan = 256 * 16;
  __shared__ int job0;
  for (long long base = static_cast<long long>(blockIdx.x) * kPackSpan; base < total;
       base += static_cast<long long>(gridDim.x) * kPackSpan) {
    __syncthreads();
    if (threadIdx.x == 0) {
      int lo = 0, hi = n_jobs - 1;
      while (lo < hi) {                       // last job whose prefix <= base
        const int mid = (lo + hi + 1) >> 1;
        if (prefix[mid] <= base) lo = mid; else hi = mid - 1;
      }
      job0 = lo;
    }
    __syncthreads();
    int lo = job0;
    // eight consecutive K columns per thread: one 16-byte store, eight independent loads (a job's size and every row of
    // Kc columns are multiples of 64 elements, so a group of eight never straddles a row, a tap or a job)
    for (int e = threadIdx.x * 8; e < kPackSpan; e += 256 * 8) {
      const long long g = base + e;
      if (g >= total) break;
      while (lo + 1 < n_jobs && prefix[lo + 1] <= g) ++lo;
      const long long* jb = jobs + static_cast<long long>(lo) * 8;
      const float* w = reinterpret_cast<const float*>(jb[0]);
      __nv_bfloat16* packed = reinterpret_cast<__nv_bfloat16*>(jb[1]);
      const unsigned cout = static_cast<unsigned>(jb[2]), cin = static_cast<unsigned>(jb[3]), taps = static_cast<unsigned>(jb[4]);
      const int transpose = static_cast<int>(jb[5]);
      const unsigned Kc = static_cast<unsigned>(jb[7]);
      const unsigned i = static_cast<unsigned>(g - prefix[lo]);          // a job holds < 2^32 elements
      const unsigned c0 = i % Kc;
      const unsigned q = i / Kc;
      const unsigned tap = q % taps;
      const unsigned r = q / taps;
      float v[8];
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const unsigned c = c0 + j;
        v[j] = 0.f;
        if (transpose == 0) {
          if (r < cout && c < cin) v[j] = __ldg(w + (static_cast<size_t>(r) * cin + c) * taps + tap);
        } else if (transpose == 1) {
          if (r < cin && c < cout) v[j] = __ldg(w + (static_cast<size_t>(c) * cin + r) * taps + tap);
        } else {                                           // stem layout (see pack_weight_kernel)
          const unsigned k = c & 31;
          const int kh = 2 * static_cast<int>(tap) + static_cast<int>(c >> 5) - 1;
          if (r < cout && c < 64 && k < 21 && kh >= 0 && kh < 7)
            v[j] = __ldg(w + ((static_cast<size_t>(r) * 3 + k % 3) * 7 + kh) * 7 + k / 3);
        }
      }
      *reinterpret_cast<uint4*>(packed + i) = pack8(v);
    }
  }
}

// ------------------------------------------------------------------------------------------- stem row packing
// The 1x7x7 s(1,2,2) p(0,3,3) stem (r21d_byol.py:198) as a FOUR-tap stride-1 convolution over row pairs: the seven kw taps
// and the three input channels of every output column are packed into a 32-channel vector, and the two frame rows
// 2*h2, 2*h2 + 1 share one 64-channel pixel,
//   P[n][t][h2][wo][hpar*32 + kw*3 + ci] = x[n][ci][t][2*h2 + hpar][2*wo + kw - 3]   (0 outside the frame; k >= 21 zero).
// Output row ho reads frame rows 2*ho - 3 .. 2*ho + 3 = row pairs ho - 2 .. ho + 1: a (1,4,1) stride-1 implicit GEMM over
// P with padding 2 below / 1 above (TMA zero fill = the h padding), tap j and pixel channel hpar*32 + kw*3 + ci holding
// w[co][ci][0][kh = 2*j + hpar - 1][kw] (zero for kh = -1).  P holds 64 bytes per (frame row, output column): 0.77 GB per
// batch of 60 against 1.93 GB for the materialised im2col rows (K = 147 -> 160) it replaces; K grows to 256, which the
// tensor pipe does not notice on this HBM-bound layer.  One CTA per (n, t, h2): six input rows staged in shared memory.
constexpr int kStemMaxW = 256;
constexpr int kStemRowPairs = 4;     // row pairs per CTA: 24 input rows staged with float4 loads, 28 KB written per CTA
__global__ void __launch_bounds__(256) stem_pack_kernel(const float* __restrict__ x, int T, int H, int W,
                                                        uint4* __restrict__ P) {
  __shared__ __align__(16) float rows[kStemRowPairs][2][3][kStemMaxW + 8];   // [pair][hpar][ci][4 + wi]: zero columns around
  const int Wo = W / 2, H2 = H / 2;
  const int groups = (H2 + kStemRowPairs - 1) / kStemRowPairs;
  int b = blockIdx.x;
  const int h2_0 = (b % groups) * kStemRowPairs;
  b /= groups;
  const int t = b % T;
  const int n = b / T;
  const int np = min(kStemRowPairs, H2 - h2_0);
  // (column c of a staged row holds x[wi = c - 4]: the float4 loads stay 16-byte aligned; columns 0..3 and W+4.. are zero)
  const int W4 = W / 4;
  for (int i = threadIdx.x; i < np * 6 * (W4 + 2); i += blockDim.x) {
    const int q = i % (W4 + 2), row = i / (W4 + 2);          // row = (pair*2 + hpar)*3 + ci
    const int ci = row % 3, hp = (row / 3) & 1, pr = row / 6;
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (q >= 1 && q <= W4)
      v = __ldg(reinterpret_cast<const float4*>(
                    x + (((static_cast<long long>(n) * 3 + ci) * T + t) * H + 2 * (h2_0 + pr) + hp) * W) + (q - 1));
    *reinterpret_cast<float4*>(&rows[pr][hp][ci][4 * q]) = v;
  }
  __syncthreads();
  uint4* dst = P + (((static_cast<long long>(n) * T + t) * H2 + h2_0) * Wo) * 8;
  for (int i = threadIdx.x; i < np * Wo * 8; i += blockDim.x) {
    const int v = i & 3, hp = (i >> 2) & 1;          // eight 16-byte vectors (8 channels each) per output column
    const int wo = (i >> 3) % Wo, pr = (i >> 3) / Wo;
    float f[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const int k = v * 8 + j;                       // k = kw*3 + ci
      const int kw = (k * 11) >> 5;                  // k / 3 for k < 32
      f[j] = k < 21 ? rows[pr][hp][k - 3 * kw][2 * wo + kw + 1] : 0.f;      // x[2*wo + kw - 3] sits in column 2*wo + kw + 1
    }
    dst[i] = pack8(f);
  }
}

// ------------------------------------------------------------------------------------------- BN statistics
// Per-block partial sums.  grid = (nblocks, groups, channel segments of <=1024 channels).
// partials layout: [nblocks][groups][2][Cp].
constexpr int kSegVecs = 128;

// Backward flavour: s0 = sum(dy), s1 = sum(dy * x) over RAW x; bn_bwd_finalize converts to sum(dy * xhat) =
// invstd * (s1 - mean * s0) in double, so the streaming loop carries no per-channel statistics (registers ->
// occupancy -> bytes in flight: this kernel ran at 45% of HBM peak with mean/invstd held per thread).
template <bool kBackward>
__global__ void __launch_bounds__(256, 4) bn_reduce_kernel(const uint4* __restrict__ a, const uint4* __restrict__ act,
                                                        const uint4* __restrict__ raw, long long rows_per_group, int Cp,
                                                        const float* __restrict__ mean, const float* __restrict__ invstd,
                                                        const float* __restrict__ mscale, const float* __restrict__ mshift,
                                                        float* __restrict__ partials) {
  __shared__ float red[256 * 2];
  const int nvec = Cp / 8;
  const int g = blockIdx.y;
  const int seg0 = blockIdx.z * kSegVecs;
  const int seg_vecs = min(kSegVecs, nvec - seg0);
  const int rows_per_pass = 256 / seg_vecs;
  const int cv = threadIdx.x % seg_vecs;
  const int rl = threadIdx.x / seg_vecs;
  float s0[8], s1[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) s0[j] = s1[j] = 0.f;
  if (rl < rows_per_pass) {
    float ms[8], mb[8];
    if (kBackward && mscale != nullptr) {
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        ms[j] = mscale[g * Cp + (seg0 + cv) * 8 + j];
        mb[j] = mshift[g * Cp + (seg0 + cv) * 8 + j];
      }
    }
    const long long base = static_cast<long long>(g) * rows_per_group;
    long long r = static_cast<long long>(blockIdx.x) * rows_per_pass + rl;
    const long long rstep = static_cast<long long>(gridDim.x) * rows_per_pass;
    if (!kBackward) {
      // one stream only: four independent 16-byte loads in flight per thread before the (order-preserving) accumulation
      for (; r + 3 * rstep < rows_per_group; r += 4 * rstep) {
        uint4 v[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) v[u] = a[(base + r + u * rstep) * nvec + seg0 + cv];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          float x[8];
          unpack8(v[u], x);
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            s0[j] += x[j];
            s1[j] += x[j] * x[j];
          }
        }
      }
    }
#pragma unroll 2
    for (; r < rows_per_group; r += rstep) {
      const long long idx = (base + r) * nvec + seg0 + cv;
      float x[8];
      if (!kBackward) {
        unpack8(a[idx], x);
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          s0[j] += x[j];
          s1[j] += x[j] * x[j];
        }
      } else {
        float d[8];
        unpack8(a[idx], d);
        unpack8(raw[idx], x);
        if (act != nullptr) {
          float y[8];
          unpack8(act[idx], y);
#pragma unroll
          for (int j = 0; j < 8; ++j) d[j] = y[j] > 0.f ? d[j] : 0.f;
        } else if (mscale != nullptr) {
#pragma unroll
          for (int j = 0; j < 8; ++j) d[j] = fmaf(x[j], ms[j], mb[j]) > 0.f ? d[j] : 0.f;
        }
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          s0[j] += d[j];
          s1[j] = fmaf(d[j], x[j], s1[j]);
        }
      }
    }
  }
  // Cross-row reduction through 2 KB of shared memory (a 16 KB staging buffer kept this kernel from sharing an SM with
  // a one-CTA-per-SM tensor-core kernel on the other stream): 8 rounds, each over one channel pair (j, j+1) of one
  // quantity; thread (rl, cv) writes at (rl*seg_vecs + cv)*2 + jo, the sum over rl runs in row order (deterministic).
#pragma unroll
  for (int q = 0; q < 2; ++q) {
#pragma unroll
    for (int jj = 0; jj < 4; ++jj) {
      red[threadIdx.x * 2 + 0] = q == 0 ? s0[2 * jj] : s1[2 * jj];
      red[threadIdx.x * 2 + 1] = q == 0 ? s0[2 * jj + 1] : s1[2 * jj + 1];
      __syncthreads();
      if (threadIdx.x < seg_vecs * 2) {
        const int cvv = threadIdx.x >> 1, jo = threadIdx.x & 1;
        float acc = 0.f;
        for (int r = 0; r < rows_per_pass; ++r) acc += red[(r * seg_vecs + cvv) * 2 + jo];
        partials[((static_cast<long long>(blockIdx.x) * gridDim.y + g) * 2 + q) * Cp + (seg0 + cvv) * 8 + 2 * jj + jo] = acc;
      }
      __syncthreads();
    }
  }
}

// Deterministic tree over the per-block partials: kRedWarps warps x 32 channels per CTA; warp w owns blocks w, w + kRedWarps,
// ... and adds them in that order, the warp sums are then combined in fixed order in double.  The loop is latency bound (a
// serial version of it cost 130 us per launch; 8 warps with 8 + a serial tail of loads in flight 11 us): 32 warps, kG
// statistics groups at a time, four blocks x both quantities per trip (296 blocks: 3 trips per warp).
// partials: [nblocks][groups][2][Cp].
constexpr int kRedWarps = 32;
constexpr int kRedThreads = kRedWarps * 32;
template <int kG>
__device__ __forceinline__ void reduce_partials(const float* __restrict__ partials, int nblocks, int groups, int g0, int Cp,
                                                int c, bool active, double (*red)[4][32], double (&s)[kG], double (&ss)[kG]) {
  constexpr int kU = 4;
  const int ty = threadIdx.x >> 5, tx = threadIdx.x & 31;
  double a0[kG], a1[kG];
#pragma unroll
  for (int q = 0; q < kG; ++q) a0[q] = a1[q] = 0.0;
  if (active) {
    const long long bstride = static_cast<long long>(groups) * 2 * Cp;
    const float* base = partials + static_cast<long long>(g0) * 2 * Cp + c;
    int b = ty;
    for (; b + (kU - 1) * kRedWarps < nblocks; b += kU * kRedWarps) {
      float v0[kG][kU], v1[kG][kU];
#pragma unroll
      for (int j = 0; j < kU; ++j) {
        const float* p = base + (b + kRedWarps * j) * bstride;
#pragma unroll
        for (int q = 0; q < kG; ++q) {
          v0[q][j] = __ldg(p + q * 2 * Cp);
          v1[q][j] = __ldg(p + q * 2 * Cp + Cp);
        }
      }
#pragma unroll
      for (int j = 0; j < kU; ++j) {
#pragma unroll
        for (int q = 0; q < kG; ++q) {
          a0[q] += static_cast<double>(v0[q][j]);
          a1[q] += static_cast<double>(v1[q][j]);
        }
      }
    }
    for (; b < nblocks; b += kRedWarps) {
      const float* p = base + b * bstride;
#pragma unroll
      for (int q = 0; q < kG; ++q) {
        a0[q] += static_cast<double>(__ldg(p + q * 2 * Cp));
        a1[q] += static_cast<double>(__ldg(p + q * 2 * Cp + Cp));
      }
    }
  }
  __syncthreads();
#pragma unroll
  for (int q = 0; q < kG; ++q) {
    red[ty][2 * q][tx] = a0[q];
    red[ty][2 * q + 1][tx] = a1[q];
  }
  __syncthreads();
#pragma unroll
  for (int q = 0; q < kG; ++q) {
    s[q] = 0.0;
    ss[q] = 0.0;
    if (ty == 0) {          // (only the leading warp uses the sums)
      for (int w = 0; w < kRedWarps; ++w) {
        s[q] += red[w][2 * q][tx];
        ss[q] += red[w][2 * q + 1][tx];
      }
    }
  }
}

// f(g, sum, sum2) for every statistics group in ascending order; the groups are reduced two at a time.
template <class F>
__device__ __forceinline__ void for_each_group_sum(const float* __restrict__ partials, int nblocks, int groups, int Cp, int c,
                                                   bool active, double (*red)[4][32], F f) {
  int g = 0;
  for (; g + 1 < groups; g += 2) {
    double s[2], ss[2];
    reduce_partials<2>(partials, nblocks, groups, g, Cp, c, active, red, s, ss);
    f(g, s[0], ss[0]);
    f(g + 1, s[1], ss[1]);
  }
  if (g < groups) {
    double s[1], ss[1];
    reduce_partials<1>(partials, nblocks, groups, g, Cp, c, active, red, s, ss);
    f(g, s[0], ss[0]);
  }
}

// Collapses the per-block partials to one row [groups][2][Cp] (fp32): the payload of the cross-rank statistics
// all-reduce in world-synchronised BatchNorm (SyncBN); the finalize kernels then run with nblocks = 1.
__global__ void __launch_bounds__(kRedThreads) bn_partials_reduce_kernel(const float* __restrict__ partials, int nblocks, int groups,
                                                                 int Cp, float* __restrict__ out) {
  __shared__ double red[kRedWarps][4][32];
  const int c = blockIdx.x * 32 + (threadIdx.x & 31);
  const bool lead = (threadIdx.x >> 5) == 0 && c < Cp;
  for_each_group_sum(partials, nblocks, groups, Cp, c, c < Cp, red, [&](int g, double s, double ss) {
    if (lead) {
      out[(g * 2 + 0) * Cp + c] = static_cast<float>(s);
      out[(g * 2 + 1) * Cp + c] = static_cast<float>(ss);
    }
  });
}

__global__ void __launch_bounds__(kRedThreads) bn_finalize_kernel(const float* __restrict__ partials, int nblocks, int groups,
                                                          long long rows_per_group, int C, int Cp,
                                                          const float* __restrict__ gamma, const float* __restrict__ beta,
                                                          float eps, float momentum, float* __restrict__ running_mean,
                                                          float* __restrict__ running_var, float* __restrict__ scale,
                                                          float* __restrict__ shift, float* __restrict__ mean_out,
                                                          float* __restrict__ invstd_out) {
  __shared__ double red[kRedWarps][4][32];
  const int c = blockIdx.x * 32 + (threadIdx.x & 31);
  const bool lead = (threadIdx.x >> 5) == 0 && c < Cp;
  float rm = 0.f, rv = 0.f;
  if (lead && c < C && running_mean != nullptr) {
    rm = running_mean[c];
    rv = running_var[c];
  }
  for_each_group_sum(partials, nblocks, groups, Cp, c, c < C, red, [&](int g, double s, double ss) {
    if (!lead) return;
    if (c >= C) {
      scale[g * Cp + c] = 0.f;
      shift[g * Cp + c] = 0.f;
      mean_out[g * Cp + c] = 0.f;
      invstd_out[g * Cp + c] = 0.f;
      return;
    }
    const double n = static_cast<double>(rows_per_group);
    const double mu = s / n;
    double var = ss / n - mu * mu;
    if (var < 0.0) var = 0.0;
    const float istd = static_cast<float>(1.0 / sqrt(var + static_cast<double>(eps)));
    const float sc = gamma[c] * istd;
    scale[g * Cp + c] = sc;
    shift[g * Cp + c] = beta[c] - static_cast<float>(mu) * sc;
    mean_out[g * Cp + c] = static_cast<float>(mu);
    invstd_out[g * Cp + c] = istd;
    // the views pass through the module one after the other: the running statistics advance once per group
    const double unbiased = n > 1.0 ? var * n / (n - 1.0) : var;
    rm = (1.f - momentum) * rm + momentum * static_cast<float>(mu);
    rv = (1.f - momentum) * rv + momentum * static_cast<float>(unbiased);
  });
  if (lead && c < C && running_mean != nullptr) {
    running_mean[c] = rm;
    running_var[c] = rv;
  }
}

// Shared row/channel geometry of the BatchNorm streaming kernels: grid = (row blocks, groups, channel segments of
// <= 1024 channels); every thread owns ONE 8-channel vector (its per-channel coefficients live in registers) and
// walks the rows of its group.
struct BnThread {
  int g, cvec, rl, rows_per_pass;
  bool active;
};
__device__ __forceinline__ BnThread bn_thread(int Cp) {
  BnThread t;
  const int nvec = Cp / 8;
  const int seg0 = blockIdx.z * kSegVecs;
  const int seg_vecs = min(kSegVecs, nvec - seg0);
  t.rows_per_pass = 256 / seg_vecs;
  t.cvec = seg0 + static_cast<int>(threadIdx.x) % seg_vecs;
  t.rl = static_cast<int>(threadIdx.x) / seg_vecs;
  t.g = blockIdx.y;
  t.active = t.rl < t.rows_per_pass;
  return t;
}
__device__ __forceinline__ void load8(const float* __restrict__ p, float (&f)[8]) {
  const float4 a = __ldg(reinterpret_cast<const float4*>(p)), b = __ldg(reinterpret_cast<const float4*>(p) + 1);
  f[0] = a.x; f[1] = a.y; f[2] = a.z; f[3] = a.w;
  f[4] = b.x; f[5] = b.y; f[6] = b.z; f[7] = b.w;
}

// out = act(raw*scale + shift + residual).  Two rows per trip with every load issued before the first use (one 16-byte
// load in flight per thread and four CTAs per SM keep 16 KB per SM in the air: 4.7 TB/s; the HBM pipe wants ~3x that).
// kCoef2: the residual carries its own BatchNorm coefficients (res_mode 2 / 3): 32 more registers, three CTAs per SM.
template <bool kCoef2>
__global__ void __launch_bounds__(256, kCoef2 ? 3 : 4) bn_apply_kernel(const uint4* __restrict__ raw, int Cp, long long rows_per_group,
                                                          const float* __restrict__ scale, const float* __restrict__ shift,
                                                          int relu, int res_mode, const uint4* __restrict__ res,
                                                          const float* __restrict__ scale2, const float* __restrict__ shift2,
                                                          uint4* __restrict__ out) {
  const BnThread t = bn_thread(Cp);
  if (!t.active) return;
  const int nvec = Cp / 8;
  float s[8], b[8], s2[8], b2[8];
  load8(scale + t.g * Cp + t.cvec * 8, s);
  load8(shift + t.g * Cp + t.cvec * 8, b);
  if (kCoef2) {
    load8(scale2 + t.g * Cp + t.cvec * 8, s2);
    load8(shift2 + t.g * Cp + t.cvec * 8, b2);
  }
  auto apply = [&](const uint4& a, const uint4& q) {
    float x[8];
    unpack8(a, x);
#pragma unroll
    for (int j = 0; j < 8; ++j) x[j] = fmaf(x[j], s[j], b[j]);
    if (res_mode == 1) {
      float y[8];
      unpack8(q, y);
#pragma unroll
      for (int j = 0; j < 8; ++j) x[j] += y[j];
    } else if (kCoef2 && res_mode == 2) {
      float y[8];
      unpack8(q, y);
#pragma unroll
      for (int j = 0; j < 8; ++j) x[j] += fmaf(y[j], s2[j], b2[j]);
    } else if (kCoef2 && res_mode == 3) {
      // the shortcut is an activation that was never materialised: rebuild the bf16 value its consumers see
      float y[8];
      unpack8(q, y);
#pragma unroll
      for (int j = 0; j < 8; ++j) x[j] += __bfloat162float(__float2bfloat16_rn(fmaxf(fmaf(y[j], s2[j], b2[j]), 0.f)));
    }
    if (relu) {
#pragma unroll
      for (int j = 0; j < 8; ++j) x[j] = fmaxf(x[j], 0.f);
    }
    return pack8(x);
  };
  const long long base = static_cast<long long>(t.g) * rows_per_group;
  const long long rstep = static_cast<long long>(gridDim.x) * t.rows_per_pass;
  long long r = static_cast<long long>(blockIdx.x) * t.rows_per_pass + t.rl;
  constexpr int kRows = 2;       // (four rows per trip measured neutral, profiles/r02f_bn_rows_ab.txt)
  for (; r + (kRows - 1) * rstep < rows_per_group; r += kRows * rstep) {
    long long i[kRows];
    uint4 a[kRows], q[kRows];
#pragma unroll
    for (int k = 0; k < kRows; ++k) {
      i[k] = (base + r + k * rstep) * nvec + t.cvec;
      a[k] = raw[i[k]];
    }
#pragma unroll
    for (int k = 0; k < kRows; ++k) q[k] = res_mode != 0 ? res[i[k]] : a[k];
#pragma unroll
    for (int k = 0; k < kRows; ++k) out[i[k]] = apply(a[k], q[k]);
  }
  for (; r < rows_per_group; r += rstep) {
    const long long i = (base + r) * nvec + t.cvec;
    const uint4 a = raw[i];
    uint4 q = a;
    if (res_mode != 0) q = res[i];
    out[i] = apply(a, q);
  }
}

__global__ void __launch_bounds__(kRedThreads) bn_bwd_finalize_kernel(const float* __restrict__ partials, int nblocks, int groups,
                                                              long long rows_per_group, int C, int Cp,
                                                              const float* __restrict__ gamma,
                                                              const float* __restrict__ mean,
                                                              const float* __restrict__ invstd, float* __restrict__ dgamma,
                                                              float* __restrict__ dbeta, int accumulate,
                                                              float* __restrict__ coef) {
  __shared__ double red[kRedWarps][4][32];
  const int c = blockIdx.x * 32 + (threadIdx.x & 31);
  const bool lead = (threadIdx.x >> 5) == 0 && c < Cp;
  double dg = 0.0, db = 0.0;
  for_each_group_sum(partials, nblocks, groups, Cp, c, c < C, red, [&](int g, double s, double sx) {
    if (!lead) return;
    float* cf = coef + static_cast<long long>(g) * 3 * Cp;
    if (c >= C) {
      cf[c] = 0.f;
      cf[Cp + c] = 0.f;
      cf[2 * Cp + c] = 0.f;
      return;
    }
    // partials hold sum(dy * x) over raw x: sum(dy * xhat) = invstd * (sum(dy*x) - mean * sum(dy))
    sx = static_cast<double>(invstd[g * Cp + c]) * (sx - static_cast<double>(mean[g * Cp + c]) * s);
    const double n = static_cast<double>(rows_per_group);
    cf[c] = gamma[c] * invstd[g * Cp + c];
    cf[Cp + c] = static_cast<float>(s / n);
    cf[2 * Cp + c] = static_cast<float>(sx / n);
    db += s;
    dg += sx;
  });
  if (lead && c < C && dgamma != nullptr) {
    dgamma[c] = accumulate ? dgamma[c] + static_cast<float>(dg) : static_cast<float>(dg);
    dbeta[c] = accumulate ? dbeta[c] + static_cast<float>(db) : static_cast<float>(db);
  }
}

// g = c0*(dy - c1 - xhat*c2) with dy = d masked by the ReLU of the forward pass:
//   act != NULL            mask = act > 0            (block outputs: the pre-activation includes the residual)
//   mscale != NULL         mask = raw*mscale + mshift > 0, the same fmaf the forward apply evaluated (saves the act read)
//   neither                no ReLU behind this BatchNorm
__global__ void __launch_bounds__(256, 2) bn_bwd_apply_kernel(const uint4* __restrict__ d, const uint4* __restrict__ act,
                                                           const uint4* __restrict__ raw, int Cp, long long rows_per_group,
                                                           const float* __restrict__ mean, const float* __restrict__ invstd,
                                                           const float* __restrict__ coef, const float* __restrict__ mscale,
                                                           const float* __restrict__ mshift, uint4* __restrict__ gout,
                                                           uint4* __restrict__ dz) {
  const BnThread t = bn_thread(Cp);
  if (!t.active) return;
  const int nvec = Cp / 8;
  const int co = t.g * Cp + t.cvec * 8;
  float A[8], Bc[8], Cc[8], ms[8], mb[8];
  {
    // g = c0*(dy - c1 - (x - mu)*istd*c2) = A*dy + Bc*x + Cc with Bc = -c0*c2*istd, Cc = -c0*c1 - Bc*mu
    float mu[8], is[8], c1[8], c2[8];
    load8(mean + co, mu);
    load8(invstd + co, is);
    load8(coef + static_cast<long long>(t.g) * 3 * Cp + t.cvec * 8, A);
    load8(coef + static_cast<long long>(t.g) * 3 * Cp + Cp + t.cvec * 8, c1);
    load8(coef + static_cast<long long>(t.g) * 3 * Cp + 2 * Cp + t.cvec * 8, c2);
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      Bc[j] = -A[j] * c2[j] * is[j];
      Cc[j] = -A[j] * c1[j] - Bc[j] * mu[j];
    }
  }
  if (mscale != nullptr) {
    load8(mscale + co, ms);
    load8(mshift + co, mb);
  }
  const long long base = static_cast<long long>(t.g) * rows_per_group;
  const long long rstep = static_cast<long long>(gridDim.x) * t.rows_per_pass;
  // one row: d (and act) and raw are already loaded as 16-byte vectors
  auto row = [&](long long i, const uint4& vd, const uint4& vx, const uint4& vy) {
    float dy[8], x[8];
    unpack8(vd, dy);
    unpack8(vx, x);
    if (act != nullptr) {
      float y[8];
      unpack8(vy, y);
#pragma unroll
      for (int j = 0; j < 8; ++j) dy[j] = y[j] > 0.f ? dy[j] : 0.f;
    } else if (mscale != nullptr) {
#pragma unroll
      for (int j = 0; j < 8; ++j) dy[j] = fmaf(x[j], ms[j], mb[j]) > 0.f ? dy[j] : 0.f;
    }
    if (dz != nullptr) dz[i] = pack8(dy);
    float o[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) o[j] = fmaf(A[j], dy[j], fmaf(Bc[j], x[j], Cc[j]));
    gout[i] = pack8(o);
  };
  long long r = static_cast<long long>(blockIdx.x) * t.rows_per_pass + t.rl;
  // kRows rows per trip with every load issued before the first use: 2 (3 with act) independent 16-byte loads per row.
  // Four rows (120 registers, two CTAs per SM: 64 KB in flight per SM) against two: 144-channel pass 5.5 -> 6.4 TB/s,
  // batch-60 step -0.4 ms (profiles/r02f_bn_rows_ab.txt)
  constexpr int kRows = 4;
  for (; r + (kRows - 1) * rstep < rows_per_group; r += kRows * rstep) {
    long long i[kRows];
    uint4 vd[kRows], vx[kRows], vy[kRows];
#pragma unroll
    for (int k = 0; k < kRows; ++k) {
      i[k] = (base + r + k * rstep) * nvec + t.cvec;
      vd[k] = d[i[k]];
      vx[k] = raw[i[k]];
    }
#pragma unroll
    for (int k = 0; k < kRows; ++k) vy[k] = act != nullptr ? act[i[k]] : make_uint4(0, 0, 0, 0);
#pragma unroll
    for (int k = 0; k < kRows; ++k) row(i[k], vd[k], vx[k], vy[k]);
  }
  for (; r < rows_per_group; r += rstep) {
    const long long i = (base + r) * nvec + t.cvec;
    row(i, d[i], raw[i], act != nullptr ? act[i] : make_uint4(0, 0, 0, 0));
  }
}

// ------------------------------------------------------------------------------------------- pooling
// Sample n lands in output row n % rows_out at column offset (n / rows_out) * Cp of a row of ld_out elements:
// rows_out == N gives the plain [N][Cp] layout, rows_out == N/2 the cat(feat1, feat2) layout of r21d_byol.py:374.
__global__ void avgpool_fwd_kernel(const uint4* __restrict__ x, int P, int Cp, float* __restrict__ out_f32,
                                   __nv_bfloat16* __restrict__ out_bf16, int rows_out, int ld_out) {
  const int nvec = Cp / 8;
  const int n = blockIdx.x;
  const long long obase = static_cast<long long>(n % rows_out) * ld_out + static_cast<long long>(n / rows_out) * Cp;
  for (int cv = threadIdx.x; cv < nvec; cv += blockDim.x) {
    float acc[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) acc[j] = 0.f;
    for (int p = 0; p < P; ++p) {
      float f[8];
      unpack8(x[(static_cast<long long>(n) * P + p) * nvec + cv], f);
#pragma unroll
      for (int j = 0; j < 8; ++j) acc[j] += f[j];
    }
    const float inv = 1.f / static_cast<float>(P);
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      acc[j] *= inv;
      if (out_f32) out_f32[obase + cv * 8 + j] = acc[j];
    }
    if (out_bf16) *reinterpret_cast<uint4*>(out_bf16 + obase + cv * 8) = pack8(acc);
  }
}

// dx[n][p][c] = (dfeat[n][c] + dcat[n % rows_cat][(n / rows_cat) * Cp + c]) / P   (dcat optional)
__global__ void avgpool_bwd_kernel(const float* __restrict__ dfeat, const float* __restrict__ dcat, int rows_cat,
                                   int ld_cat, int P, int Cp, uint4* __restrict__ dx, long long total) {
  const int nvec = Cp / 8;
  const float inv = 1.f / static_cast<float>(P);
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int cv = static_cast<int>(i % nvec);
    const long long n = i / nvec / P;
    float f[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      float v = dfeat[n * Cp + cv * 8 + j];
      if (dcat != nullptr) v += dcat[(n % rows_cat) * ld_cat + (n / rows_cat) * Cp + cv * 8 + j];
      f[j] = v * inv;
    }
    dx[i] = pack8(f);
  }
}

// ------------------------------------------------------------------------------------------- misc
__global__ void colsum_kernel(const __nv_bfloat16* __restrict__ x, long long rows, int Cp, int C, float* __restrict__ out,
                              int accumulate) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= C) return;
  float acc = 0.f;
  for (long long r = 0; r < rows; ++r) acc += __bfloat162float(x[r * Cp + c]);
  out[c] = accumulate ? out[c] + acc : acc;
}

__global__ void cast_pad_kernel(const float* __restrict__ x, long long rows, int cols, int ld_in,
                                __nv_bfloat16* __restrict__ out, int ld_out, const float* __restrict__ scale_dev) {
  const float s = scale_dev ? *scale_dev : 1.f;
  const long long total = rows * ld_out;
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int c = static_cast<int>(i % ld_out);
    const long long r = i / ld_out;
    out[i] = __float2bfloat16_rn(c < cols ? x[r * ld_in + c] * s : 0.f);
  }
}

// Row-block count of the BatchNorm streaming kernels (see bn_thread): enough CTAs to fill the machine a few times.
static inline dim3 bn_grid(long long rows_per_group, int Cp, int groups) {
  const int nvec = Cp / 8;
  const int segs = ceil_div(nvec, kSegVecs);
  const int seg_vecs = nvec < kSegVecs ? nvec : kSegVecs;
  const int rows_per_pass = 256 / seg_vecs;
  long long want = (static_cast<long long>(num_sms()) * kStreamCtasPerSm + groups * segs - 1) / (groups * segs);
  long long have = (rows_per_group + rows_per_pass - 1) / rows_per_pass;
  if (want > have) want = have;
  if (want < 1) want = 1;
  return dim3(static_cast<unsigned>(want), static_cast<unsigned>(groups), static_cast<unsigned>(segs));
}

static inline int grid_for(long long total, int threads) {
  long long b = (total + threads - 1) / threads;
  const long long cap = static_cast<long long>(num_sms()) * 16;
  if (b > cap) b = cap;
  if (b < 1) b = 1;
  return static_cast<int>(b);
}

}  // namespace cstp

using namespace cstp;
#define ST(s) static_cast<cudaStream_t>(s)

extern "C" int cstp_pack_weight(const float* w, int cout, int cin, int taps, int transpose, void* packed, int Rp, int Kc,
                                void* stream) {
  CSTP_REQUIRE(w && packed && cout > 0 && cin > 0 && taps > 0 && Rp > 0 && Kc > 0 && Kc % 64 == 0);
  CSTP_REQUIRE(transpose == 0 || transpose == 1 || (transpose == 2 && cin == 64 && taps == 4));
  CSTP_REQUIRE(transpose == 1 ? (Rp >= cin && Kc >= cout) : (Rp >= cout && Kc >= cin));
  const long long total = static_cast<long long>(Rp) * taps * Kc;
  pack_weight_kernel<<<grid_for(total, 256), 256, 0, ST(stream)>>>(w, cout, cin, taps, transpose,
                                                                  reinterpret_cast<__nv_bfloat16*>(packed), Rp, Kc);
  CSTP_LAUNCHED();
  return CSTP_OK;
}

extern "C" int cstp_pack_weights_batched(const int64_t* jobs_dev, const int64_t* prefix_dev, int n_jobs, int64_t total,
                                         void* stream) {
  CSTP_REQUIRE(jobs_dev && prefix_dev && n_jobs > 0 && total > 0);
  static_assert(sizeof(long long) == sizeof(int64_t), "job table is int64");
  pack_weights_batched_kernel<<<grid_for((total + 15) / 16, 256), 256, 0, ST(stream)>>>(
      reinterpret_cast<const long long*>(jobs_dev), reinterpret_cast<const long long*>(prefix_dev), n_jobs, total);
  CSTP_LAUNCHED();
  return CSTP_OK;
}

extern "C" int cstp_stem_pack(const float* x, int N, int T, int H, int W, void* P, void* stream) {
  CSTP_REQUIRE(x && P && N > 0 && T > 0 && H > 0 && W > 0 && W % 4 == 0 && H % 2 == 0 && W <= kStemMaxW);
  CSTP_REQUIRE((reinterpret_cast<uintptr_t>(P) % 16) == 0 && (reinterpret_cast<uintptr_t>(x) % 16) == 0);
  const int groups = (H / 2 + kStemRowPairs - 1) / kStemRowPairs;
  stem_pack_kernel<<<N * T * groups, 256, 0, ST(stream)>>>(x, T, H, W, reinterpret_cast<uint4*>(P));
  CSTP_LAUNCHED();
  return CSTP_OK;
}

extern "C" int cstp_bn_stats(const void* raw, int64_t rows, int Cp, int groups, float* partials, int nblocks,
                             void* stream) {
  CSTP_REQUIRE(raw && partials && rows > 0 && groups > 0 && rows % groups == 0 && Cp % 16 == 0 && nblocks > 0);
  const dim3 grid(nblocks, groups, ceil_div(Cp / 8, kSegVecs));
  bn_reduce_kernel<false><<<grid, 256, 0, ST(stream)>>>(reinterpret_cast<const uint4*>(raw), nullptr, nullptr,
                                                       rows / groups, Cp, nullptr, nullptr, nullptr, nullptr, partials);
  CSTP_LAUNCHED();
  return CSTP_OK;
}

extern "C" int cstp_bn_partials_reduce(const float* partials, int nblocks, int groups, int Cp, float* out, void* stream) {
  CSTP_REQUIRE(partials && out && nblocks > 0 && groups > 0 && Cp % 16 == 0);
  bn_partials_reduce_kernel<<<ceil_div(Cp, 32), kRedThreads, 0, ST(stream)>>>(partials, nblocks, groups, Cp, out);
  CSTP_LAUNCHED();
  return CSTP_OK;
}

extern "C" int cstp_bn_finalize(const float* partials, int nblocks, int groups, int64_t rows_per_group, int C, int Cp,
                                const float* gamma, const float* beta, float eps, float momentum, float* running_mean,
                                float* running_var, float* scale, float* shift, float* mean, float* invstd,
                                void* stream) {
  CSTP_REQUIRE(partials && gamma && beta && scale && shift && mean && invstd && C <= Cp);
  bn_finalize_kernel<<<ceil_div(Cp, 32), kRedThreads, 0, ST(stream)>>>(partials, nblocks, groups, rows_per_group, C, Cp, gamma, beta,
                                                               eps, momentum, running_mean, running_var, scale, shift,
                                                               mean, invstd);
  CSTP_LAUNCHED();
  return CSTP_OK;
}

extern "C" int cstp_bn_apply(const void* raw, int64_t rows, int Cp, int groups, const float* scale, const float* shift,
                             int relu, int res_mode, const void* res, const float* scale2, const float* shift2,
                             void* out, void* stream) {
  CSTP_REQUIRE(raw && out && scale && shift && rows > 0 && groups > 0 && rows % groups == 0 && Cp % 16 == 0);
  CSTP_REQUIRE(res_mode >= 0 && res_mode <= 3 && (res_mode == 0 || res != nullptr));
  CSTP_REQUIRE(res_mode < 2 || (scale2 && shift2));
  auto kernel = res_mode >= 2 ? bn_apply_kernel<true> : bn_apply_kernel<false>;
  kernel<<<bn_grid(rows / groups, Cp, groups), 256, 0, ST(stream)>>>(
      reinterpret_cast<const uint4*>(raw), Cp, rows / groups, scale, shift, relu, res_mode,
      reinterpret_cast<const uint4*>(res), scale2, shift2, reinterpret_cast<uint4*>(out));
  CSTP_LAUNCHED();
  return CSTP_OK;
}

extern "C" int cstp_bn_bwd_reduce(const void* d, const void* act, const void* raw, int64_t rows, int Cp, int groups,
                                  const float* mean, const float* invstd, const float* mask_scale,
                                  const float* mask_shift, float* partials, int nblocks, void* stream) {
  CSTP_REQUIRE(d && raw && mean && invstd && partials && rows > 0 && groups > 0 && rows % groups == 0 && Cp % 16 == 0);
  CSTP_REQUIRE((mask_scale == nullptr) == (mask_shift == nullptr));
  CSTP_REQUIRE(act == nullptr || mask_scale == nullptr);
  const dim3 grid(nblocks, groups, ceil_div(Cp / 8, kSegVecs));
  bn_reduce_kernel<true><<<grid, 256, 0, ST(stream)>>>(reinterpret_cast<const uint4*>(d),
                                                      reinterpret_cast<const uint4*>(act),
                                                      reinterpret_cast<const uint4*>(raw), rows / groups, Cp, mean,
                                                      invstd, mask_scale, mask_shift, partials);
  CSTP_LAUNCHED();
  return CSTP_OK;
}

extern "C" int cstp_bn_bwd_finalize(const float* partials, int nblocks, int groups, int64_t rows_per_group, int C,
                                    int Cp, const float* gamma, const float* mean, const float* invstd, float* dgamma,
                                    float* dbeta, int accumulate, float* coef, void* stream) {
  CSTP_REQUIRE(partials && gamma && mean && invstd && coef && C <= Cp);
  bn_bwd_finalize_kernel<<<ceil_div(Cp, 32), kRedThreads, 0, ST(stream)>>>(partials, nblocks, groups, rows_per_group, C, Cp, gamma,
                                                                  mean, invstd, dgamma, dbeta, accumulate, coef);
  CSTP_LAUNCHED();
  return CSTP_OK;
}

extern "C" int cstp_bn_bwd_apply(const void* d, const void* act, const void* raw, int64_t rows, int Cp, int groups,
                                 const float* mean, const float* invstd, const float* coef, const float* mask_scale,
                                 const float* mask_shift, void* g, void* dz, void* stream) {
  CSTP_REQUIRE(d && raw && mean && invstd && coef && g && rows > 0 && groups > 0 && rows % groups == 0 && Cp % 16 == 0);
  CSTP_REQUIRE((mask_scale == nullptr) == (mask_shift == nullptr));
  CSTP_REQUIRE(act == nullptr || mask_scale == nullptr);
  // (64 registers / 4 CTAs per SM was measured: it spills and is 7 % slower than 80 registers / 3 CTAs)
  bn_bwd_apply_kernel<<<bn_grid(rows / groups, Cp, groups), 256, 0, ST(stream)>>>(
      reinterpret_cast<const uint4*>(d), reinterpret_cast<const uint4*>(act), reinterpret_cast<const uint4*>(raw), Cp,
      rows / groups, mean, invstd, coef, mask_scale, mask_shift, reinterpret_cast<uint4*>(g),
      reinterpret_cast<uint4*>(dz));
  CSTP_LAUNCHED();
  return CSTP_OK;
}

extern "C" int cstp_avgpool_fwd(const void* x, int N, int P, int Cp, float* out_f32, void* out_bf16, int rows_out,
                                int ld_out, void* stream) {
  CSTP_REQUIRE(x && (out_f32 || out_bf16) && N > 0 && P > 0 && Cp % 16 == 0);
  CSTP_REQUIRE(rows_out > 0 && N % rows_out == 0 && ld_out >= (N / rows_out) * Cp && ld_out % 8 == 0);
  avgpool_fwd_kernel<<<N, 64, 0, ST(stream)>>>(reinterpret_cast<const uint4*>(x), P, Cp, out_f32,
                                              reinterpret_cast<__nv_bfloat16*>(out_bf16), rows_out, ld_out);
  CSTP_LAUNCHED();
  return CSTP_OK;
}

extern "C" int cstp_avgpool_bwd(const float* dfeat, const float* dcat, int rows_cat, int ld_cat, int N, int P, int Cp,
                                void* dx, void* stream) {
  CSTP_REQUIRE(dfeat && dx && N > 0 && P > 0 && Cp % 16 == 0);
  CSTP_REQUIRE(dcat == nullptr || (rows_cat > 0 && N % rows_cat == 0 && ld_cat >= (N / rows_cat) * Cp));
  const long long total = static_cast<long long>(N) * P * (Cp / 8);
  avgpool_bwd_kernel<<<grid_for(total, 256), 256, 0, ST(stream)>>>(dfeat, dcat, rows_cat > 0 ? rows_cat : 1, ld_cat, P, Cp,
                                                                  reinterpret_cast<uint4*>(dx), total);
  CSTP_LAUNCHED();
  return CSTP_OK;
}

extern "C" int cstp_colsum(const void* x, int64_t rows, int Cp, int C, float* out, int accumulate, void* stream) {
  CSTP_REQUIRE(x && out && rows > 0 && C > 0 && C <= Cp);
  colsum_kernel<<<ceil_div(C, 128), 128, 0, ST(stream)>>>(reinterpret_cast<const __nv_bfloat16*>(x), rows, Cp, C, out,
                                                         accumulate);
  CSTP_LAUNCHED();
  return CSTP_OK;
}

extern "C" int cstp_cast_pad(const float* x, int64_t rows, int cols, int ld_in, void* out, int ld_out,
                             const float* scale_dev, void* stream) {
  CSTP_REQUIRE(x && out && rows > 0 && cols > 0 && cols <= ld_in && cols <= ld_out);
  const long long total = rows * ld_out;
  cast_pad_kernel<<<grid_for(total, 256), 256, 0, ST(stream)>>>(x, rows, cols, ld_in,
                                                               reinterpret_cast<__nv_bfloat16*>(out), ld_out, scale_dev);
  CSTP_LAUNCHED();
  return CSTP_OK;
}

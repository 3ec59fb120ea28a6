// Loss kernels (BYOL regression, six pretext cross-entropies, NT-Xent) and the optimiser-side HBM-bound
// kernels (EMA target update, global-norm clip + SGD momentum step) of the CSTP pretraining step.
// Reductions are performed in a fixed order so that results are run-to-run bit-reproducible.
#include "common.h"
#include "ptx.cuh"

namespace cstp {

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// ------------------------------------------------------------------------------------------- BYOL loss
// models/pace/r21d_byol.py:346-355,382.  One block; warp w handles rows w, w+nwarps, ...
__global__ void __launch_bounds__(1024) byol_loss_kernel(const float* __restrict__ pred, const float* __restrict__ tproj,
                                                         int B, int D, int ld, float* __restrict__ loss_out,
                                                         const float* __restrict__ upstream, float* __restrict__ dpred) {
  __shared__ float wsum[32];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nwarps = blockDim.x >> 5;
  const float up = upstream ? *upstream : 1.f;
  float acc = 0.f;
  for (int i = warp; i < B; i += nwarps) {
#pragma unroll
    for (int pair = 0; pair < 2; ++pair) {
      const float* x = pred + static_cast<long long>(pair == 0 ? i : B + i) * ld;
      const float* y = tproj + static_cast<long long>(pair == 0 ? B + i : i) * ld;
      float xx = 0.f, yy = 0.f, xy = 0.f;
      for (int c = lane; c < D; c += 32) {
        const float a = x[c], b = y[c];
        xx += a * a;
        yy += b * b;
        xy += a * b;
      }
      xx = warp_sum(xx);
      yy = warp_sum(yy);
      xy = warp_sum(xy);
      const float nx = fmaxf(sqrtf(xx), 1e-12f), ny = fmaxf(sqrtf(yy), 1e-12f);
      const float cosv = xy / (nx * ny);
      acc += 2.f - 2.f * cosv;
      if (dpred != nullptr) {
        float* dx = dpred + static_cast<long long>(pair == 0 ? i : B + i) * ld;
        const float k = -2.f * up / (static_cast<float>(B) * nx);
        for (int c = lane; c < D; c += 32) dx[c] = k * (y[c] / ny - (x[c] / nx) * cosv);
        for (int c = D + lane; c < ld; c += 32) dx[c] = 0.f;
      }
    }
  }
  if (lane == 0) wsum[warp] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    float t = 0.f;
    for (int w = 0; w < nwarps; ++w) t += wsum[w];
    loss_out[0] = t / static_cast<float>(B);
  }
}

// ------------------------------------------------------------------------------------------- pretext CE x6
struct CeArgs {
  const float* logits[6];
  const int64_t* labels[6];
  float* dlogits[6];
};

// main_byol.py:62-73: six mean cross-entropies and their weighted sum.  One block, one thread per row.
__global__ void __launch_bounds__(1024) pretext_ce_kernel(CeArgs a, int B, int n_cls, int ld,
                                                          const float* __restrict__ weights5,
                                                          float* __restrict__ losses_out) {
  __shared__ float red[1024];
  __shared__ float head_loss[6];
  const float w[6] = {weights5[1], weights5[2], weights5[3], weights5[3], weights5[4], weights5[4]};
  for (int h = 0; h < 6; ++h) {
    float acc = 0.f;
    for (int i = threadIdx.x; i < B; i += blockDim.x) {
      const float* l = a.logits[h] + static_cast<long long>(i) * ld;
      const int y = static_cast<int>(a.labels[h][i]);
      float m = l[0];
      for (int c = 1; c < n_cls; ++c) m = fmaxf(m, l[c]);
      float s = 0.f;
      for (int c = 0; c < n_cls; ++c) s += expf(l[c] - m);
      const float lse = m + logf(s);
      acc += lse - l[y];
      if (a.dlogits[h] != nullptr) {
        float* d = a.dlogits[h] + static_cast<long long>(i) * ld;
        const float k = w[h] / static_cast<float>(B);
        for (int c = 0; c < ld; ++c) d[c] = c < n_cls ? k * (expf(l[c] - lse) - (c == y ? 1.f : 0.f)) : 0.f;
      }
    }
    red[threadIdx.x] = acc;
    __syncthreads();
    for (int s = blockDim.x >> 1; s > 0; s >>= 1) {
      if (threadIdx.x < s) red[threadIdx.x] += red[threadIdx.x + s];
      __syncthreads();
    }
    if (threadIdx.x == 0) head_loss[h] = red[0] / static_cast<float>(B);
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    float tot = 0.f;
    for (int h = 0; h < 6; ++h) {
      losses_out[h] = head_loss[h];
      tot += w[h] * head_loss[h];
    }
    losses_out[6] = tot;
  }
}

// ------------------------------------------------------------------------------------------- finetune head
// F.normalize(feat, p=2, dim=1) of the finetune / test branch (models/pace/r21d_byol.py:394-399): y = x / max(|x|, eps),
// written as bf16 rows for the BatchNorm1d / Linear kernels; the norms are kept for the backward.
__global__ void l2norm_fwd_kernel(const float* __restrict__ x, int rows, int d, int ld, float eps,
                                  __nv_bfloat16* __restrict__ y, int ld_y, float* __restrict__ norms) {
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (warp >= rows) return;
  const float* xr = x + static_cast<long long>(warp) * ld;
  float ss = 0.f;
  for (int c = lane; c < d; c += 32) ss += xr[c] * xr[c];
  ss = warp_sum(ss);
  const float n = fmaxf(sqrtf(ss), eps);
  for (int c = lane; c < ld_y; c += 32) y[static_cast<long long>(warp) * ld_y + c] = __float2bfloat16_rn(c < d ? xr[c] / n : 0.f);
  if (lane == 0) norms[warp] = n;
}

// dx = (g - y (y . g)) / norm with y = x / norm (rows whose norm was clamped to eps pass g / eps, as torch does).
__global__ void l2norm_bwd_kernel(const float* __restrict__ x, const float* __restrict__ norms,
                                  const __nv_bfloat16* __restrict__ g, int rows, int d, int ld, int ld_g,
                                  float* __restrict__ dx) {
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (warp >= rows) return;
  const float* xr = x + static_cast<long long>(warp) * ld;
  const __nv_bfloat16* gr = g + static_cast<long long>(warp) * ld_g;
  const float inv = 1.f / norms[warp];
  float dot = 0.f, ss = 0.f;
  for (int c = lane; c < d; c += 32) {
    dot += xr[c] * inv * __bfloat162float(gr[c]);
    ss += xr[c] * xr[c];
  }
  dot = warp_sum(dot);
  ss = warp_sum(ss);
  const bool clamped = sqrtf(ss) < norms[warp];        // |x| < eps: the forward divided by the constant eps
  for (int c = lane; c < ld; c += 32) {
    float v = 0.f;
    if (c < d) v = clamped ? __bfloat162float(gr[c]) * inv : (__bfloat162float(gr[c]) - xr[c] * inv * dot) * inv;
    dx[static_cast<long long>(warp) * ld + c] = v;
  }
}

// nn.CrossEntropyLoss() (mean) over [B][ld] logits with n_cls classes (main_ft_mp.py:188,203) + gradient.
// One block; warp w handles rows w, w + nwarps, ...; the row losses are summed in row order.
__global__ void __launch_bounds__(1024) ce_loss_kernel(const float* __restrict__ logits, const int64_t* __restrict__ labels,
                                                       int B, int n_cls, int ld, float* __restrict__ loss_out,
                                                       float* __restrict__ dlogits, float* __restrict__ row_loss) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nwarps = blockDim.x >> 5;
  for (int i = warp; i < B; i += nwarps) {
    const float* l = logits + static_cast<long long>(i) * ld;
    const int y = static_cast<int>(labels[i]);
    float m = -INFINITY;
    for (int c = lane; c < n_cls; c += 32) m = fmaxf(m, l[c]);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
    float s = 0.f;
    for (int c = lane; c < n_cls; c += 32) s += expf(l[c] - m);
    s = warp_sum(s);
    const float lse = m + logf(s);
    if (lane == 0) row_loss[i] = lse - l[y];
    if (dlogits != nullptr) {
      float* dr = dlogits + static_cast<long long>(i) * ld;
      const float k = 1.f / static_cast<float>(B);
      for (int c = lane; c < ld; c += 32) dr[c] = c < n_cls ? k * (expf(l[c] - lse) - (c == y ? 1.f : 0.f)) : 0.f;
    }
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    float t = 0.f;
    for (int i = 0; i < B; ++i) t += row_loss[i];
    loss_out[0] = t / static_cast<float>(B);
  }
}

// Eval-mode BatchNorm as an affine map: scale = gamma / sqrt(running_var + eps), shift = beta - running_mean * scale
// (model.eval() in main_ft_mp.py:281-289 / test.py:76-93); the forward then only needs cstp_bn_apply.
__global__ void bn_eval_coeffs_kernel(const float* __restrict__ gamma, const float* __restrict__ beta,
                                      const float* __restrict__ rm, const float* __restrict__ rv, int C, int Cp, int groups,
                                      float eps, float* __restrict__ scale, float* __restrict__ shift) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= Cp) return;
  float sc = 0.f, sh = 0.f;
  if (c < C) {
    sc = gamma[c] / sqrtf(rv[c] + eps);
    sh = beta[c] - rm[c] * sc;
  }
  for (int g = 0; g < groups; ++g) {
    scale[g * Cp + c] = sc;
    shift[g * Cp + c] = sh;
  }
}

// ------------------------------------------------------------------------------------------- NT-Xent
// loss/NTXent.py:46-62 in closed form (SURVEY.md A.3): no rows x rows matrix is ever materialised.
constexpr int kNtBM = 64, kNtBN = 64, kNtBK = 32;

__global__ void ntxent_normalize_kernel(const float* __restrict__ z, int rows, int d, int use_cosine,
                                        float* __restrict__ zn, float* __restrict__ norms) {
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (warp >= rows) return;
  const float* x = z + static_cast<long long>(warp) * d;
  float ss = 0.f;
  for (int c = lane; c < d; c += 32) ss += x[c] * x[c];
  ss = warp_sum(ss);
  const float n = use_cosine ? fmaxf(sqrtf(ss), 1e-8f) : 1.f;
  for (int c = lane; c < d; c += 32) zn[static_cast<long long>(warp) * d + c] = x[c] / n;
  if (lane == 0) norms[warp] = n;
}

// S tile (64x64) of zn_i . zn_j * inv_tau; thread (ty,tx) of a 16x16 block owns rows ty*4.., cols tx*4...
__device__ __forceinline__ void ntxent_s_tile(const float* __restrict__ zn, int rows, int d, int i0, int j0,
                                              float inv_tau, float (*As)[kNtBM + 4], float (*Bs)[kNtBN + 4],
                                              float (&s)[4][4]) {
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
#pragma unroll
  for (int a = 0; a < 4; ++a)
#pragma unroll
    for (int b = 0; b < 4; ++b) s[a][b] = 0.f;
  for (int k0 = 0; k0 < d; k0 += kNtBK) {
    __syncthreads();
    // 64 rows x 32 k for each operand: 2048 elements, 256 threads -> 8 each.
    for (int e = threadIdx.x; e < kNtBM * kNtBK; e += 256) {
      const int r = e / kNtBK, k = e % kNtBK;
      const int gi = i0 + r, gj = j0 + r, gk = k0 + k;
      As[k][r] = (gi < rows && gk < d) ? zn[static_cast<long long>(gi) * d + gk] : 0.f;
      Bs[k][r] = (gj < rows && gk < d) ? zn[static_cast<long long>(gj) * d + gk] : 0.f;
    }
    __syncthreads();
#pragma unroll 8
    for (int k = 0; k < kNtBK; ++k) {
      const float4 av = *reinterpret_cast<const float4*>(&As[k][ty * 4]);
      const float4 bv = *reinterpret_cast<const float4*>(&Bs[k][tx * 4]);
      const float a4[4] = {av.x, av.y, av.z, av.w};
      const float b4[4] = {bv.x, bv.y, bv.z, bv.w};
#pragma unroll
      for (int a = 0; a < 4; ++a)
#pragma unroll
        for (int b = 0; b < 4; ++b) s[a][b] = fmaf(a4[a], b4[b], s[a][b]);
    }
  }
#pragma unroll
  for (int a = 0; a < 4; ++a)
#pragma unroll
    for (int b = 0; b < 4; ++b) s[a][b] *= inv_tau;
}

__global__ void __launch_bounds__(256) ntxent_fwd_kernel(const float* __restrict__ zn, int rows, int d, float inv_tau,
                                                         float* __restrict__ lse, float* __restrict__ row_loss) {
  __shared__ float As[kNtBK][kNtBM + 4];
  __shared__ float Bs[kNtBK][kNtBN + 4];
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
  const int i0 = blockIdx.x * kNtBM;
  const int half = rows / 2;
  float m[4], l[4], spos[4];
#pragma unroll
  for (int a = 0; a < 4; ++a) {
    m[a] = -INFINITY;
    l[a] = 0.f;
    spos[a] = 0.f;
  }
  for (int j0 = 0; j0 < rows; j0 += kNtBN) {
    float s[4][4];
    ntxent_s_tile(zn, rows, d, i0, j0, inv_tau, As, Bs, s);
#pragma unroll
    for (int a = 0; a < 4; ++a) {
      const int gi = i0 + ty * 4 + a;
      const int pos = gi < half ? gi + half : gi - half;
      float tm = -INFINITY;
#pragma unroll
      for (int b = 0; b < 4; ++b) {
        const int gj = j0 + tx * 4 + b;
        if (gj == pos) spos[a] = s[a][b];
        if (gj >= rows || gj == gi) s[a][b] = -INFINITY;
        tm = fmaxf(tm, s[a][b]);
      }
#pragma unroll
      for (int o = 8; o > 0; o >>= 1) tm = fmaxf(tm, __shfl_xor_sync(0xffffffffu, tm, o));
      const float mn = fmaxf(m[a], tm);
      float ts = 0.f;
      if (mn > -INFINITY) {
#pragma unroll
        for (int b = 0; b < 4; ++b) ts += __expf(s[a][b] - mn);
      }
#pragma unroll
      for (int o = 8; o > 0; o >>= 1) ts += __shfl_xor_sync(0xffffffffu, ts, o);
      l[a] = (mn > -INFINITY ? l[a] * __expf(m[a] - mn) : 0.f) + ts;
      m[a] = mn;
    }
  }
#pragma unroll
  for (int a = 0; a < 4; ++a) {
    float sp = spos[a];
#pragma unroll
    for (int o = 8; o > 0; o >>= 1) sp += __shfl_xor_sync(0xffffffffu, sp, o);
    const int gi = i0 + ty * 4 + a;
    if (tx == 0 && gi < rows) {
      const float v = m[a] + logf(l[a]);
      lse[gi] = v;
      row_loss[gi] = v - sp;
    }
  }
}

__global__ void __launch_bounds__(1024) ntxent_loss_reduce_kernel(const float* __restrict__ row_loss, int rows,
                                                                  float* __restrict__ loss_out) {
  __shared__ float red[1024];
  float acc = 0.f;
  for (int i = threadIdx.x; i < rows; i += blockDim.x) acc += row_loss[i];
  red[threadIdx.x] = acc;
  __syncthreads();
  for (int s = blockDim.x >> 1; s > 0; s >>= 1) {
    if (threadIdx.x < s) red[threadIdx.x] += red[threadIdx.x + s];
    __syncthreads();
  }
  if (threadIdx.x == 0) loss_out[0] = red[0] / static_cast<float>(rows);
}

// dzn_i = (1/(tau*rows)) * sum_j (P_ij + P_ji - 2[j = pos(i)]) zn_j, then the cosine-normalisation Jacobian.
// One CTA per 64 rows and per 128-wide slice of d (blockIdx.y).
__global__ void __launch_bounds__(256) ntxent_bwd_kernel(const float* __restrict__ zn, const float* __restrict__ norms,
                                                         const float* __restrict__ lse, int rows, int d, float inv_tau,
                                                         int use_cosine, float* __restrict__ dzn) {
  extern __shared__ float sm[];
  float(*As)[kNtBM + 4] = reinterpret_cast<float(*)[kNtBM + 4]>(sm);
  float(*Bs)[kNtBN + 4] = reinterpret_cast<float(*)[kNtBN + 4]>(sm + kNtBK * (kNtBM + 4));
  float(*Ws)[kNtBN + 1] = reinterpret_cast<float(*)[kNtBN + 1]>(sm + 2 * kNtBK * (kNtBM + 4));
  float(*Zs)[128] = reinterpret_cast<float(*)[128]>(sm + 2 * kNtBK * (kNtBM + 4) + kNtBM * (kNtBN + 1));
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
  const int i0 = blockIdx.x * kNtBM;
  const int d0 = blockIdx.y * 128;
  const int half = rows / 2;
  const int r2 = threadIdx.x >> 2, dq = threadIdx.x & 3;  // second GEMM: row r2, dims dq*32..+31 of the slice
  float acc[32];
#pragma unroll
  for (int e = 0; e < 32; ++e) acc[e] = 0.f;
  float lse_i[4];
#pragma unroll
  for (int a = 0; a < 4; ++a) {
    const int gi = i0 + ty * 4 + a;
    lse_i[a] = gi < rows ? lse[gi] : 0.f;
  }
  for (int j0 = 0; j0 < rows; j0 += kNtBN) {
    float s[4][4];
    ntxent_s_tile(zn, rows, d, i0, j0, inv_tau, As, Bs, s);
#pragma unroll
    for (int a = 0; a < 4; ++a) {
      const int gi = i0 + ty * 4 + a;
      const int pos = gi < half ? gi + half : gi - half;
#pragma unroll
      for (int b = 0; b < 4; ++b) {
        const int gj = j0 + tx * 4 + b;
        float wv = 0.f;
        if (gi < rows && gj < rows && gj != gi) {
          wv = __expf(s[a][b] - lse_i[a]) + __expf(s[a][b] - lse[gj]);
          if (gj == pos) wv -= 2.f;
        }
        Ws[ty * 4 + a][tx * 4 + b] = wv;
      }
    }
    for (int e = threadIdx.x; e < kNtBN * 128; e += 256) {
      const int r = e >> 7, c = e & 127;
      const int gj = j0 + r, gc = d0 + c;
      Zs[r][c] = (gj < rows && gc < d) ? zn[static_cast<long long>(gj) * d + gc] : 0.f;
    }
    __syncthreads();
#pragma unroll 4
    for (int j = 0; j < kNtBN; ++j) {
      const float wv = Ws[r2][j];
#pragma unroll
      for (int e4 = 0; e4 < 8; ++e4) {
        const float4 zv = *reinterpret_cast<const float4*>(&Zs[j][dq * 32 + e4 * 4]);
        acc[e4 * 4 + 0] = fmaf(wv, zv.x, acc[e4 * 4 + 0]);
        acc[e4 * 4 + 1] = fmaf(wv, zv.y, acc[e4 * 4 + 1]);
        acc[e4 * 4 + 2] = fmaf(wv, zv.z, acc[e4 * 4 + 2]);
        acc[e4 * 4 + 3] = fmaf(wv, zv.w, acc[e4 * 4 + 3]);
      }
    }
  }
  const int gi = i0 + r2;
  if (gi < rows) {
    const float k = inv_tau / static_cast<float>(rows);
#pragma unroll
    for (int e = 0; e < 32; ++e) {
      const int gc = d0 + dq * 32 + e;
      if (gc < d) dzn[static_cast<long long>(gi) * d + gc] = acc[e] * k;
    }
  }
  (void)norms;
  (void)use_cosine;
}

// dz_i = (dzn_i - zn_i (zn_i . dzn_i)) / norm_i   (cosine) ;  dz_i = dzn_i (dot similarity)
__global__ void ntxent_bwd_norm_kernel(const float* __restrict__ zn, const float* __restrict__ norms,
                                       const float* dzn, int rows, int d, int use_cosine, float* dz) {
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (warp >= rows) return;
  const long long o = static_cast<long long>(warp) * d;
  if (!use_cosine) {
    for (int c = lane; c < d; c += 32) dz[o + c] = dzn[o + c];
    return;
  }
  float dot = 0.f;
  for (int c = lane; c < d; c += 32) dot += zn[o + c] * dzn[o + c];
  dot = warp_sum(dot);
  const float inv = 1.f / norms[warp];
  for (int c = lane; c < d; c += 32) dz[o + c] = (dzn[o + c] - zn[o + c] * dot) * inv;
}

// ------------------------------------------------------------------------------------------- EMA
// r21d_byol.py:331-337: param_k * m + param_q * (1 - m) with separately rounded products (no FMA contraction).
__global__ void __launch_bounds__(256) ema_kernel(float4* __restrict__ k, const float4* __restrict__ q, long long n4,
                                                  float* __restrict__ kt, const float* __restrict__ qt, int tail, float m,
                                                  float om) {
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < n4;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    float4 a = k[i];
    const float4 b = q[i];
    a.x = __fadd_rn(__fmul_rn(a.x, m), __fmul_rn(b.x, om));
    a.y = __fadd_rn(__fmul_rn(a.y, m), __fmul_rn(b.y, om));
    a.z = __fadd_rn(__fmul_rn(a.z, m), __fmul_rn(b.z, om));
    a.w = __fadd_rn(__fmul_rn(a.w, m), __fmul_rn(b.w, om));
    k[i] = a;
  }
  if (blockIdx.x == 0 && static_cast<int>(threadIdx.x) < tail)
    kt[threadIdx.x] = __fadd_rn(__fmul_rn(kt[threadIdx.x], m), __fmul_rn(qt[threadIdx.x], om));
}

// ------------------------------------------------------------------------------------------- clip + SGD
constexpr int kNormBlocks = 1024;

__global__ void __launch_bounds__(256) sumsq_partial_kernel(const float* __restrict__ g, long long n,
                                                            float* __restrict__ partials) {
  __shared__ float red[256];
  float acc = 0.f;
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < n;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const float v = g[i];
    acc = fmaf(v, v, acc);
  }
  red[threadIdx.x] = acc;
  __syncthreads();
  for (int s = 128; s > 0; s >>= 1) {
    if (threadIdx.x < s) red[threadIdx.x] += red[threadIdx.x + s];
    __syncthreads();
  }
  if (threadIdx.x == 0) partials[blockIdx.x] = red[0];
}

// main_byol.py:88-91,229-232: clip_grad_norm_(18) then SGD(momentum 0.9, wd on every parameter, dampening 0).
__global__ void __launch_bounds__(256) sgd_step_kernel(float* __restrict__ p, const float* __restrict__ g,
                                                       float* __restrict__ mom, long long n, float lr, float momentum,
                                                       float wd, float max_norm, int do_clip, int first_step,
                                                       const float* __restrict__ partials, float* __restrict__ norm_out,
                                                       const float* __restrict__ hyper) {
  if (hyper != nullptr) {      // hyper-parameters from device memory: a captured CUDA graph follows the lr schedule
    lr = hyper[0];
    momentum = hyper[1];
    wd = hyper[2];
    max_norm = hyper[3];
    do_clip = hyper[4] != 0.f;
    first_step = hyper[5] != 0.f;
  }
  __shared__ double red[256];
  double acc = 0.0;
  for (int i = threadIdx.x; i < kNormBlocks; i += blockDim.x) acc += static_cast<double>(partials[i]);
  red[threadIdx.x] = acc;
  __syncthreads();
  for (int s = 128; s > 0; s >>= 1) {
    if (threadIdx.x < s) red[threadIdx.x] += red[threadIdx.x + s];
    __syncthreads();
  }
  const float total_norm = static_cast<float>(sqrt(red[0]));
  float coef = 1.f;
  if (do_clip) {
    coef = max_norm / (total_norm + 1e-6f);
    coef = coef > 1.f ? 1.f : coef;
  }
  if (blockIdx.x == 0 && threadIdx.x == 0 && norm_out != nullptr) {
    norm_out[0] = total_norm;
    norm_out[1] = coef;
  }
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < n;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const float w = p[i];
    float gr = g[i] * coef;
    gr = fmaf(wd, w, gr);
    const float b = first_step ? gr : fmaf(momentum, mom[i], gr);
    mom[i] = b;
    p[i] = w - lr * b;
  }
}

// ------------------------------------------------------------------------------------------- clip + Adam / AdamW
// clip_grad_norm_ (main_byol.py:88-90): every block reduces the kNormBlocks partial sums of squares in the same fixed
// order (in double) and derives the clip coefficient max_norm / (norm + 1e-6), capped at 1; block 0 reports both.
// Kept operation for operation equal to the prologue of sgd_step_kernel: both optimisers clip by the same norm.
__device__ __forceinline__ float clip_coefficient(const float* __restrict__ partials, int do_clip, float max_norm,
                                                  float* __restrict__ norm_out) {
  __shared__ double red[256];
  double acc = 0.0;
  for (int i = threadIdx.x; i < kNormBlocks; i += blockDim.x) acc += static_cast<double>(partials[i]);
  red[threadIdx.x] = acc;
  __syncthreads();
  for (int s = 128; s > 0; s >>= 1) {
    if (threadIdx.x < s) red[threadIdx.x] += red[threadIdx.x + s];
    __syncthreads();
  }
  const float total_norm = static_cast<float>(sqrt(red[0]));
  float coef = 1.f;
  if (do_clip) {
    coef = max_norm / (total_norm + 1e-6f);
    coef = coef > 1.f ? 1.f : coef;
  }
  if (blockIdx.x == 0 && threadIdx.x == 0 && norm_out != nullptr) {
    norm_out[0] = total_norm;
    norm_out[1] = coef;
  }
  return coef;
}

// torch.optim.Adam / AdamW (_single_tensor_adam) per element, each operation rounded on its own so that a float32
// restatement reproduces the bits (include/cstp_b200.h has the formula).
__device__ __forceinline__ void adam_element(float& w, float gr, float& m, float& v, const cstp_adam_hyper& h,
                                             float coef) {
  gr = __fmul_rn(gr, coef);
  w = __fmul_rn(w, h.decay);
  gr = __fadd_rn(gr, __fmul_rn(h.l2, w));
  m = __fadd_rn(m, __fmul_rn(__fsub_rn(gr, m), h.one_minus_beta1));
  v = __fadd_rn(__fmul_rn(v, h.beta2), __fmul_rn(__fmul_rn(h.one_minus_beta2, gr), gr));
  const float den = __fadd_rn(__fdiv_rn(__fsqrt_rn(v), h.bc2_sqrt), h.eps);
  w = __fsub_rn(w, __fdiv_rn(__fmul_rn(h.step_size, m), den));
}

// One float4 of each buffer per thread and iteration (4 loads, 3 stores); block 0 also takes the n % 4 tail.
__global__ void __launch_bounds__(256) adam_step_kernel(float4* __restrict__ p, const float4* __restrict__ g,
                                                        float4* __restrict__ m, float4* __restrict__ v, long long n4,
                                                        int tail, cstp_adam_hyper h, const float* __restrict__ partials,
                                                        float* __restrict__ norm_out,
                                                        const cstp_adam_hyper* __restrict__ hyper) {
  if (hyper != nullptr) h = *hyper;
  const float coef = clip_coefficient(partials, h.do_clip != 0.f, h.max_norm, norm_out);
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < n4;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    float4 w = p[i], a = m[i], b = v[i];
    const float4 gr = g[i];
    adam_element(w.x, gr.x, a.x, b.x, h, coef);
    adam_element(w.y, gr.y, a.y, b.y, h, coef);
    adam_element(w.z, gr.z, a.z, b.z, h, coef);
    adam_element(w.w, gr.w, a.w, b.w, h, coef);
    p[i] = w;
    m[i] = a;
    v[i] = b;
  }
  if (blockIdx.x == 0 && static_cast<int>(threadIdx.x) < tail) {
    const long long i = n4 * 4 + threadIdx.x;
    float* pt = reinterpret_cast<float*>(p);
    float* mt = reinterpret_cast<float*>(m);
    float* vt = reinterpret_cast<float*>(v);
    adam_element(pt[i], reinterpret_cast<const float*>(g)[i], mt[i], vt[i], h, coef);
  }
}

int ntxent_tensor_path(const float* zn, int rows, int d, float temperature, bool backward, float* row_loss, float* ws,
                       float** dzn_out, cudaStream_t stream);

static inline int grid_cap(long long total, int threads) {
  long long b = (total + threads - 1) / threads;
  const long long cap = static_cast<long long>(num_sms()) * 8;
  if (b > cap) b = cap;
  if (b < 1) b = 1;
  return static_cast<int>(b);
}

}  // namespace cstp

using namespace cstp;
#define ST(s) static_cast<cudaStream_t>(s)

extern "C" int cstp_byol_loss(const float* pred, const float* tproj, int B, int D, int ld, float* loss_out,
                              const float* upstream, float* dpred, void* stream) {
  CSTP_REQUIRE(pred && tproj && loss_out && B > 0 && D > 0 && D <= ld);
  byol_loss_kernel<<<1, 1024, 0, ST(stream)>>>(pred, tproj, B, D, ld, loss_out, upstream, dpred);
  CSTP_LAUNCHED();
  return CSTP_OK;
}

extern "C" int cstp_pretext_ce(const float* const* logits, const int64_t* const* labels, float* const* dlogits, int B,
                               int n_cls, int ld, const float* weights5, float* losses_out, void* stream) {
  CSTP_REQUIRE(logits && labels && weights5 && losses_out && B > 0 && n_cls > 0 && n_cls <= ld);
  CeArgs a;
  for (int h = 0; h < 6; ++h) {
    CSTP_REQUIRE(logits[h] != nullptr && labels[h] != nullptr);
    a.logits[h] = logits[h];
    a.labels[h] = labels[h];
    a.dlogits[h] = dlogits ? dlogits[h] : nullptr;
  }
  pretext_ce_kernel<<<1, 1024, 0, ST(stream)>>>(a, B, n_cls, ld, weights5, losses_out);
  CSTP_LAUNCHED();
  return CSTP_OK;
}

extern "C" int cstp_l2norm_fwd(const float* x, int rows, int d, int ld, float eps, void* y_bf16, int ld_y, float* norms,
                               void* stream) {
  CSTP_REQUIRE(x && y_bf16 && norms && rows > 0 && d > 0 && d <= ld && d <= ld_y);
  l2norm_fwd_kernel<<<ceil_div(static_cast<long long>(rows) * 32, 256), 256, 0, ST(stream)>>>(
      x, rows, d, ld, eps, reinterpret_cast<__nv_bfloat16*>(y_bf16), ld_y, norms);
  CSTP_LAUNCHED();
  return CSTP_OK;
}

extern "C" int cstp_l2norm_bwd(const float* x, const float* norms, const void* g_bf16, int rows, int d, int ld, int ld_g,
                               float* dx, void* stream) {
  CSTP_REQUIRE(x && norms && g_bf16 && dx && rows > 0 && d > 0 && d <= ld && d <= ld_g);
  l2norm_bwd_kernel<<<ceil_div(static_cast<long long>(rows) * 32, 256), 256, 0, ST(stream)>>>(
      x, norms, reinterpret_cast<const __nv_bfloat16*>(g_bf16), rows, d, ld, ld_g, dx);
  CSTP_LAUNCHED();
  return CSTP_OK;
}

extern "C" int cstp_ce_loss(const float* logits, const int64_t* labels, int B, int n_cls, int ld, float* loss_out,
                            float* dlogits, float* workspace, void* stream) {
  CSTP_REQUIRE(logits && labels && loss_out && workspace && B > 0 && n_cls > 0 && n_cls <= ld);
  ce_loss_kernel<<<1, 1024, 0, ST(stream)>>>(logits, labels, B, n_cls, ld, loss_out, dlogits, workspace);
  CSTP_LAUNCHED();
  return CSTP_OK;
}

extern "C" int cstp_bn_eval_coeffs(const float* gamma, const float* beta, const float* running_mean,
                                   const float* running_var, int C, int Cp, int groups, float eps, float* scale,
                                   float* shift, void* stream) {
  CSTP_REQUIRE(gamma && beta && running_mean && running_var && scale && shift && C > 0 && C <= Cp && groups > 0);
  bn_eval_coeffs_kernel<<<ceil_div(Cp, 128), 128, 0, ST(stream)>>>(gamma, beta, running_mean, running_var, C, Cp, groups,
                                                                  eps, scale, shift);
  CSTP_LAUNCHED();
  return CSTP_OK;
}

extern "C" long long cstp_ntxent_workspace_floats(int rows, int d);

extern "C" int cstp_ntxent(const float* z, int rows, int d, float temperature, int use_cosine, float* loss_out,
                           float* dz, float* workspace, long long workspace_floats, void* stream) {
  CSTP_REQUIRE(z && loss_out && workspace && rows >= 2 && rows % 2 == 0 && d > 0 && temperature > 0.f);
  CSTP_REQUIRE(workspace_floats >= 3LL * rows + static_cast<long long>(rows) * d);
  float* norms = workspace;
  float* lse = workspace + rows;
  float* row_loss = workspace + 2 * static_cast<long long>(rows);
  float* zn = workspace + 3 * static_cast<long long>(rows);
  const float inv_tau = 1.f / temperature;
  ntxent_normalize_kernel<<<ceil_div(static_cast<long long>(rows) * 32, 256), 256, 0, ST(stream)>>>(z, rows, d, use_cosine,
                                                                                                  zn, norms);
  CSTP_LAUNCHED();
  // Tensor-core path (ntxent_tc.cu) when the shape allows and the caller provided its larger workspace; the SIMT
  // kernels below serve small / odd shapes (rows < 256, d not a multiple of 64).
  if (rows >= 256 && d % 64 == 0 && d <= 256 && workspace_floats >= cstp_ntxent_workspace_floats(rows, d) &&
      (reinterpret_cast<uintptr_t>(workspace) % 16) == 0) {
    float* dzn = nullptr;
    float* tc_ws = zn + static_cast<long long>(rows) * d;
    tc_ws += (8 - (reinterpret_cast<uintptr_t>(tc_ws) / 4) % 8) % 8;        // 32-byte alignment (STG.256 of the dZn partials)
    int rc = ntxent_tensor_path(zn, rows, d, temperature, dz != nullptr, row_loss, tc_ws, &dzn, ST(stream));
    if (rc != CSTP_OK) return rc;
    ntxent_loss_reduce_kernel<<<1, 1024, 0, ST(stream)>>>(row_loss, rows, loss_out);
    CSTP_LAUNCHED();
    if (dz != nullptr) {
      ntxent_bwd_norm_kernel<<<ceil_div(static_cast<long long>(rows) * 32, 256), 256, 0, ST(stream)>>>(
          zn, norms, dzn, rows, d, use_cosine, dz);
      CSTP_LAUNCHED();
    }
    return CSTP_OK;
  }
  ntxent_fwd_kernel<<<ceil_div(rows, kNtBM), 256, 0, ST(stream)>>>(zn, rows, d, inv_tau, lse, row_loss);
  CSTP_LAUNCHED();
  ntxent_loss_reduce_kernel<<<1, 1024, 0, ST(stream)>>>(row_loss, rows, loss_out);
  CSTP_LAUNCHED();
  if (dz != nullptr) {
    // dzn is staged in dz itself, then normalised in place row by row (each row is owned by one warp).
    const int smem = (2 * kNtBK * (kNtBM + 4) + kNtBM * (kNtBN + 1) + kNtBN * 128) * static_cast<int>(sizeof(float));
    static bool attr_set = false;
    if (!attr_set) {
      CSTP_CUDA(cudaFuncSetAttribute(ntxent_bwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
      attr_set = true;
    }
    const dim3 grid(ceil_div(rows, kNtBM), ceil_div(d, 128));
    ntxent_bwd_kernel<<<grid, 256, smem, ST(stream)>>>(zn, norms, lse, rows, d, inv_tau, use_cosine, dz);
    CSTP_LAUNCHED();
    ntxent_bwd_norm_kernel<<<ceil_div(static_cast<long long>(rows) * 32, 256), 256, 0, ST(stream)>>>(zn, norms, dz, rows, d,
                                                                                                   use_cosine, dz);
    CSTP_LAUNCHED();
  }
  return CSTP_OK;
}

extern "C" int cstp_ema_update(float* k, const float* q, int64_t n, float m, float one_minus_m, void* stream) {
  CSTP_REQUIRE(k && q && n > 0);
  CSTP_REQUIRE((reinterpret_cast<uintptr_t>(k) % 16) == 0 && (reinterpret_cast<uintptr_t>(q) % 16) == 0);
  const long long n4 = n / 4;
  const int tail = static_cast<int>(n % 4);
  ema_kernel<<<grid_cap(n4 > 0 ? n4 : 1, 256), 256, 0, ST(stream)>>>(reinterpret_cast<float4*>(k),
                                                                    reinterpret_cast<const float4*>(q), n4, k + n4 * 4,
                                                                    q + n4 * 4, tail, m, one_minus_m);
  CSTP_LAUNCHED();
  return CSTP_OK;
}

extern "C" int cstp_sgd_clip_step(float* p, const float* g, float* mom, int64_t n, float lr, float momentum, float wd,
                                  float max_norm, int do_clip, int first_step, float* norm_out, float* workspace,
                                  void* stream) {
  CSTP_REQUIRE(p && g && mom && workspace && n > 0);
  sumsq_partial_kernel<<<kNormBlocks, 256, 0, ST(stream)>>>(g, n, workspace);
  CSTP_LAUNCHED();
  sgd_step_kernel<<<grid_cap(n, 256), 256, 0, ST(stream)>>>(p, g, mom, n, lr, momentum, wd, max_norm, do_clip, first_step,
                                                           workspace, norm_out, nullptr);
  CSTP_LAUNCHED();
  return CSTP_OK;
}

extern "C" int cstp_sgd_clip_step_dev(float* p, const float* g, float* mom, int64_t n, const float* hyper, float* norm_out,
                                      float* workspace, void* stream) {
  CSTP_REQUIRE(p && g && mom && workspace && hyper && n > 0);
  sumsq_partial_kernel<<<kNormBlocks, 256, 0, ST(stream)>>>(g, n, workspace);
  CSTP_LAUNCHED();
  sgd_step_kernel<<<grid_cap(n, 256), 256, 0, ST(stream)>>>(p, g, mom, n, 0.f, 0.f, 0.f, 0.f, 0, 0, workspace, norm_out, hyper);
  CSTP_LAUNCHED();
  return CSTP_OK;
}

static int adam_launch(float* p, const float* g, float* m, float* v, int64_t n, const cstp_adam_hyper& h,
                       const cstp_adam_hyper* hyper_dev, float* norm_out, float* workspace, void* stream) {
  CSTP_REQUIRE(p && g && m && v && workspace && n > 0);
  for (const void* ptr : {static_cast<const void*>(p), static_cast<const void*>(g), static_cast<const void*>(m),
                          static_cast<const void*>(v)})
    CSTP_REQUIRE(reinterpret_cast<uintptr_t>(ptr) % 16 == 0);
  sumsq_partial_kernel<<<kNormBlocks, 256, 0, ST(stream)>>>(g, n, workspace);
  CSTP_LAUNCHED();
  const long long n4 = n / 4;
  adam_step_kernel<<<grid_cap(n4 > 0 ? n4 : 1, 256), 256, 0, ST(stream)>>>(
      reinterpret_cast<float4*>(p), reinterpret_cast<const float4*>(g), reinterpret_cast<float4*>(m),
      reinterpret_cast<float4*>(v), n4, static_cast<int>(n % 4), h, workspace, norm_out, hyper_dev);
  CSTP_LAUNCHED();
  return CSTP_OK;
}

extern "C" int cstp_adam_clip_step(float* p, const float* g, float* m, float* v, int64_t n, cstp_adam_hyper hyper,
                                   float* norm_out, float* workspace, void* stream) {
  return adam_launch(p, g, m, v, n, hyper, nullptr, norm_out, workspace, stream);
}

extern "C" int cstp_adam_clip_step_dev(float* p, const float* g, float* m, float* v, int64_t n,
                                       const cstp_adam_hyper* hyper, float* norm_out, float* workspace, void* stream) {
  CSTP_REQUIRE(hyper != nullptr);
  return adam_launch(p, g, m, v, n, cstp_adam_hyper{}, hyper, norm_out, workspace, stream);
}

// Pretraining clip pipeline (SURVEY.md 8 f-2): decoded uint8 frames in HBM -> the two fp32 NCDHW clips of every sample,
// one CTA per (frame, view).  Replaces the reference's per-frame Pillow / torchvision calls
// (data_process/datasets.py:888-932, data_process/preprocess_data.py:514-515, 537-562, 1112-1122).
//
// The arithmetic is Pillow's own, restated in integers so that the result equals the reference's clip bit for bit:
//   * Image.transpose(ROTATE_90/180/270) + Image.crop          -> an index map, pixels outside the frame read 0
//   * Image.resize((S, S), BICUBIC)                             -> two passes (horizontal into shared memory, then
//     vertical) with the Q22 tap tables the host precomputes exactly as Pillow does (uint8 rounding between the passes)
//   * Image.rotate(angle) (NEAREST)                             -> the 16.16 fixed-point affine walk
//   * ImageEnhance Brightness / Contrast / Color (Image.blend)  -> fp32 blend with truncation / clipping
//   * torchvision adjust_hue (convert('HSV'), uint8 wrap, back) -> Pillow's rgb2hsv / hsv2rgb float-double mix
//   * ClipRandomGray                                            -> channel replicate
//   * ImageFilter.GaussianBlur                                  -> 3 + 3 passes of the extended box blur in Q24
//   * flip, ToTensor, Normalize('tf')                           -> (v / 255) * 2 - 1 in fp32 (three rounded operations)
// No FMA contraction may happen in the float / double expressions: they use the _rn intrinsics.
#include <cooperative_groups.h>

#include "common.h"

namespace cg = cooperative_groups;

namespace cstp {

constexpr int kClipThreads = 1024;   // one CTA per SM (the staging buffers fill shared memory): all 32 warps hide the gather latency
constexpr int kPrecisionBits = 22;                       // Pillow: 32 - 8 - 2
constexpr int kCoefStride = 2 + CSTP_CLIP_KMAX;

__device__ __forceinline__ uint8_t clip8_q22(int v) {
  v >>= kPrecisionBits;
  return static_cast<uint8_t>(v < 0 ? 0 : (v > 255 ? 255 : v));
}

// Image.blend(degenerate, image, alpha) for one uint8 sample (libImaging/Blend.c)
__device__ __forceinline__ uint8_t blend_u8(int deg, int img, float alpha, bool inside) {
  const float t = __fadd_rn(static_cast<float>(deg), __fmul_rn(alpha, static_cast<float>(img - deg)));
  if (inside) return static_cast<uint8_t>(static_cast<int>(t));
  if (t <= 0.f) return 0;
  if (t >= 255.f) return 255;
  return static_cast<uint8_t>(static_cast<int>(t));
}

__device__ __forceinline__ int luma_u8(int r, int g, int b) {            // convert('L'): ITU-R 601-2, Q16
  return (r * 19595 + g * 38470 + b * 7471 + 0x8000) >> 16;
}

__device__ __forceinline__ int clip255(int v) { return v < 0 ? 0 : (v > 255 ? 255 : v); }

// libImaging/Convert.c rgb2hsv_row
__device__ __forceinline__ void rgb2hsv_u8(int r, int g, int b, int& uh, int& us, int& uv) {
  const int maxc = max(r, max(g, b)), minc = min(r, min(g, b));
  uv = maxc;
  if (minc == maxc) {
    uh = 0;
    us = 0;
    return;
  }
  const float cr = static_cast<float>(maxc - minc);
  const float s = __fdiv_rn(cr, static_cast<float>(maxc));
  const float rc = __fdiv_rn(static_cast<float>(maxc - r), cr);
  const float gc = __fdiv_rn(static_cast<float>(maxc - g), cr);
  const float bc = __fdiv_rn(static_cast<float>(maxc - b), cr);
  float h;
  if (r == maxc) {
    h = __fsub_rn(bc, gc);
  } else if (g == maxc) {
    h = static_cast<float>(__dsub_rn(__dadd_rn(2.0, static_cast<double>(rc)), static_cast<double>(bc)));
  } else {
    h = static_cast<float>(__dsub_rn(__dadd_rn(4.0, static_cast<double>(gc)), static_cast<double>(rc)));
  }
  const double hh = __dadd_rn(__ddiv_rn(static_cast<double>(h), 6.0), 1.0);
  h = static_cast<float>(hh - floor(hh));                                  // fmod(x, 1.0) for x in (0, 2): exact
  uh = clip255(static_cast<int>(__dmul_rn(static_cast<double>(h), 255.0)));
  us = clip255(static_cast<int>(__dmul_rn(static_cast<double>(s), 255.0)));
}

// libImaging/Convert.c hsv2rgb
__device__ __forceinline__ void hsv2rgb_u8(int h, int s, int v, int& r, int& g, int& b) {
  if (s == 0) {
    r = g = b = v;
    return;
  }
  const double hf = __ddiv_rn(__dmul_rn(static_cast<double>(h), 6.0), 255.0);
  const int i = static_cast<int>(floor(hf));
  const float f = static_cast<float>(__dsub_rn(hf, static_cast<double>(i)));
  const float fs = static_cast<float>(__ddiv_rn(static_cast<double>(s), 255.0));
  const double dv = static_cast<double>(v);
  const int p = clip255(static_cast<int>(round(__dmul_rn(dv, __dsub_rn(1.0, static_cast<double>(fs))))));
  const int q = clip255(static_cast<int>(round(__dmul_rn(dv, __dsub_rn(1.0, static_cast<double>(__fmul_rn(fs, f)))))));
  const int t = clip255(static_cast<int>(round(
      __dmul_rn(dv, __dsub_rn(1.0, __dmul_rn(static_cast<double>(fs), __dsub_rn(1.0, static_cast<double>(f))))))));
  switch (i % 6) {
    case 0: r = v; g = t; b = p; break;
    case 1: r = q; g = v; b = p; break;
    case 2: r = p; g = v; b = t; break;
    case 3: r = p; g = q; b = v; break;
    case 4: r = t; g = p; b = v; break;
    default: r = v; g = p; b = q; break;
  }
}

// libImaging/BoxBlur.c ImagingLineBoxBlur8 for one line of one channel of n elements; element i of the line is
// src0[i * stride].  kSplit: a column that a cluster pair splits by rows -- elements [0, half) are in src0 / dst0 (rank
// 0), element i >= half is src1[(i - half) * stride] (rank 1).
template <bool kSplit>
__device__ void box_blur_line(const uint8_t* __restrict__ src0, const uint8_t* __restrict__ src1, uint8_t* __restrict__ dst0,
                              uint8_t* __restrict__ dst1, int half, int stride, int n, int radius, int edge_a, int edge_b,
                              uint32_t ww, uint32_t fw) {
  const int lastx = n - 1;
#define LN(i) static_cast<uint32_t>(!kSplit || (i) < half ? src0[(i) * stride] : src1[((i) - half) * stride])
#define STEP(x, sub, add, left, right)                              \
  do {                                                              \
    acc += LN(add) - LN(sub);                                       \
    const uint32_t bulk = acc * ww + (LN(left) + LN(right)) * fw;   \
    const uint8_t o = static_cast<uint8_t>((bulk + (1u << 23)) >> 24); \
    if (!kSplit || (x) < half) dst0[(x) * stride] = o;              \
    else dst1[((x) - half) * stride] = o;                           \
  } while (0)
  uint32_t acc = LN(0) * static_cast<uint32_t>(radius + 1);
  for (int x = 0; x < edge_a - 1; ++x) acc += LN(x);
  acc += LN(lastx) * static_cast<uint32_t>(radius - edge_a + 1);
  if (edge_a <= edge_b) {
    for (int x = 0; x < edge_a; ++x) STEP(x, 0, x + radius, 0, x + radius + 1);
    for (int x = edge_a; x < edge_b; ++x) STEP(x, x - radius - 1, x + radius, x - radius - 1, x + radius + 1);
    for (int x = edge_b; x <= lastx; ++x) STEP(x, x - radius - 1, lastx, x - radius - 1, lastx);
  } else {
    for (int x = 0; x < edge_b; ++x) STEP(x, 0, x + radius, 0, x + radius + 1);
    for (int x = edge_b; x < edge_a; ++x) STEP(x, 0, lastx, 0, lastx);
    for (int x = edge_a; x <= lastx; ++x) STEP(x, x - radius - 1, lastx, x - radius - 1, lastx);
  }
#undef STEP
#undef LN
}

// Row y of a staged buffer (tmp: crop rows; cur / oth: image rows) at the same shared-memory offset `buf` of each CTA.
// One CTA holds every row.  A cluster pair splits the rows: rank r holds rows [r * half, (r + 1) * half), and the
// other CTA's rows are reached through distributed shared memory.
template <int CL>
struct StagedRows {
  uint8_t* base[CL];
  int half, row_bytes;
  __device__ __forceinline__ StagedRows(uint8_t* buf, int half_, int row_bytes_) : half(half_), row_bytes(row_bytes_) {
    if constexpr (CL == 1) {
      base[0] = buf;
    } else {
      cg::cluster_group cluster = cg::this_cluster();
      base[0] = cluster.map_shared_rank(buf, 0);
      base[1] = cluster.map_shared_rank(buf, 1);
    }
  }
  __device__ __forceinline__ uint8_t* operator()(int y) const {
    if constexpr (CL == 1) return base[0] + y * row_bytes;
    else return y < half ? base[0] + y * row_bytes : base[1] + (y - half) * row_bytes;
  }
};

template <int CL>
__device__ __forceinline__ void clip_sync() {
  if constexpr (CL == 1) __syncthreads();
  else cg::this_cluster().sync();
}

// CL = 1: one CTA per (frame, view) holds tmp, cur and oth.  CL = 2: a cluster pair per (frame, view) (blockIdx.x =
// 2 * frame + rank) splits every buffer by rows and oth reuses tmp's rows (tmp is dead once the vertical pass ends).
// Each thread works on the rows its own CTA holds; only the vertical resampling taps, the rotation walk and the vertical
// blur passes read (and the vertical blur writes) the other CTA's rows, and each of those steps ends in a cluster barrier.
template <int CL>
__global__ void __launch_bounds__(kClipThreads) clip_assemble_kernel(const cstp_clip_view* __restrict__ views, int T, int S,
                                                                    int tmp_bytes, int img_bytes) {
  extern __shared__ __align__(16) uint8_t clip_smem[];
  __shared__ unsigned int red_sum;
  const cstp_clip_view& v = views[blockIdx.y];
  const int t = blockIdx.x / CL;
  int rank = 0;
  if constexpr (CL == 2) rank = static_cast<int>(cg::this_cluster().block_rank());
  uint8_t* tmp = clip_smem;                       // [crop_h][S][3] after the horizontal pass
  uint8_t* cur = clip_smem + tmp_bytes;           // [S][S][3]
  uint8_t* oth = CL == 1 ? cur + img_bytes : clip_smem;
  const int W = v.W, H = v.H, rot = v.rot;
  const uint8_t* __restrict__ frame = v.video + static_cast<size_t>(v.frames[t]) * W * H * 3;
  const int bx = v.box[0], by = v.box[1];
  const int ch = v.box[3] - v.box[1];
  const int Wr = (rot & 1) ? H : W, Hr = (rot & 1) ? W : H;
  const int32_t* __restrict__ cx = v.coef;
  const int32_t* __restrict__ cy = v.coef + S * kCoefStride;
  const int npix = S * S;
  // this CTA's rows: crop rows [t_lo, t_hi) of tmp, image rows [i_lo, i_lo + nloc / S) of cur / oth
  const int t_half = (ch + CL - 1) / CL, i_half = (S + CL - 1) / CL;
  const int t_lo = rank * t_half, t_hi = CL == 1 ? ch : min(ch, t_lo + t_half);
  const int i_lo = rank * i_half;
  const int nloc = CL == 1 ? npix : (min(S, i_lo + i_half) - i_lo) * S;

  // ---- 1. horizontal resampling pass over every row of the crop (rotation and crop folded into the fetch)
  for (int i = t_lo * S + threadIdx.x; i < t_hi * S; i += blockDim.x) {
    const int y = i / S, xx = i - y * S;
    const int32_t* k = cx + xx * kCoefStride;
    const int x0 = k[0], n = k[1];
    int a0 = 1 << (kPrecisionBits - 1), a1 = a0, a2 = a0;
    const int ry = by + y;
    if (ry >= 0 && ry < Hr) {
      for (int j = 0; j < n; ++j) {
        const int rx = bx + x0 + j;
        if (rx < 0 || rx >= Wr) continue;
        int xi, yi;
        switch (rot) {                              // Image.transpose: where the rotated pixel (rx, ry) comes from
          case 0: xi = rx; yi = ry; break;
          case 1: xi = W - 1 - ry; yi = rx; break;                   // ROTATE_90 (counter-clockwise)
          case 2: xi = W - 1 - rx; yi = H - 1 - ry; break;           // ROTATE_180
          default: xi = ry; yi = H - 1 - rx; break;                  // ROTATE_270
        }
        const uint8_t* p = frame + (static_cast<size_t>(yi) * W + xi) * 3;
        const int kk = k[2 + j];
        a0 += static_cast<int>(p[0]) * kk;
        a1 += static_cast<int>(p[1]) * kk;
        a2 += static_cast<int>(p[2]) * kk;
      }
    }
    const int o = i - t_lo * S;
    tmp[o * 3 + 0] = clip8_q22(a0);
    tmp[o * 3 + 1] = clip8_q22(a1);
    tmp[o * 3 + 2] = clip8_q22(a2);
  }
  clip_sync<CL>();
  // ---- 2. vertical pass
  {
    const StagedRows<CL> trow(tmp, t_half, S * 3);
    for (int i = threadIdx.x; i < nloc; i += blockDim.x) {
      const int g = i_lo * S + i;
      const int yy = g / S, xx = g - yy * S;
      const int32_t* k = cy + yy * kCoefStride;
      const int y0 = k[0], n = k[1];
      int a0 = 1 << (kPrecisionBits - 1), a1 = a0, a2 = a0;
      for (int j = 0; j < n; ++j) {
        const uint8_t* p = trow(y0 + j) + xx * 3;
        const int kk = k[2 + j];
        a0 += static_cast<int>(p[0]) * kk;
        a1 += static_cast<int>(p[1]) * kk;
        a2 += static_cast<int>(p[2]) * kk;
      }
      cur[i * 3 + 0] = clip8_q22(a0);
      cur[i * 3 + 1] = clip8_q22(a1);
      cur[i * 3 + 2] = clip8_q22(a2);
    }
  }
  clip_sync<CL>();

  // ---- 3. base-transform chain (absent for the null chain)
  if (v.rotate) {                                   // libImaging/Geometry.c affine_fixed, nearest neighbour
    const int f0 = v.rot_fix[0], f1 = v.rot_fix[1], f2 = v.rot_fix[2], f3 = v.rot_fix[3], f4 = v.rot_fix[4], f5 = v.rot_fix[5];
    const StagedRows<CL> crow(cur, i_half, S * 3);
    for (int i = threadIdx.x; i < nloc; i += blockDim.x) {
      const int g = i_lo * S + i;
      const int y = g / S, x = g - y * S;
      const int xin = (f2 + x * f0 + y * f1) >> 16, yin = (f5 + x * f3 + y * f4) >> 16;
      const bool ok = xin >= 0 && xin < S && yin >= 0 && yin < S;
      const uint8_t* p = crow(yin) + xin * 3;
      oth[i * 3 + 0] = ok ? p[0] : 0;
      oth[i * 3 + 1] = ok ? p[1] : 0;
      oth[i * 3 + 2] = ok ? p[2] : 0;
    }
    clip_sync<CL>();
    uint8_t* s = cur;
    cur = oth;
    oth = s;
  }
  for (int j = 0; j < v.n_jitter; ++j) {
    const int op = v.jitter_op[j];
    const float alpha = v.jitter_f[j];
    const bool inside = alpha >= 0.f && alpha <= 1.f;
    if (op == 0) {                                  // ImageEnhance.Brightness: blend with black
      for (int i = threadIdx.x; i < nloc * 3; i += blockDim.x) cur[i] = blend_u8(0, cur[i], alpha, inside);
    } else if (op == 1) {                           // ImageEnhance.Contrast: blend with the rounded mean of convert('L')
      unsigned int* sum = &red_sum;                 // the pair sums into rank 0's counter
      if constexpr (CL == 2) sum = cg::this_cluster().map_shared_rank(&red_sum, 0);
      if (threadIdx.x == 0 && rank == 0) red_sum = 0;
      clip_sync<CL>();
      unsigned int part = 0;
      for (int i = threadIdx.x; i < nloc; i += blockDim.x) part += luma_u8(cur[i * 3], cur[i * 3 + 1], cur[i * 3 + 2]);
      for (int o = 16; o > 0; o >>= 1) part += __shfl_xor_sync(0xffffffffu, part, o);
      if ((threadIdx.x & 31) == 0) atomicAdd(sum, part);
      clip_sync<CL>();
      const int mean = static_cast<int>(__dadd_rn(__ddiv_rn(static_cast<double>(*sum), static_cast<double>(npix)), 0.5));
      for (int i = threadIdx.x; i < nloc * 3; i += blockDim.x) cur[i] = blend_u8(mean, cur[i], alpha, inside);
    } else if (op == 2) {                           // ImageEnhance.Color: blend with convert('L')
      for (int i = threadIdx.x; i < nloc; i += blockDim.x) {
        const int r = cur[i * 3], g = cur[i * 3 + 1], b = cur[i * 3 + 2];
        const int l = luma_u8(r, g, b);
        cur[i * 3 + 0] = blend_u8(l, r, alpha, inside);
        cur[i * 3 + 1] = blend_u8(l, g, alpha, inside);
        cur[i * 3 + 2] = blend_u8(l, b, alpha, inside);
      }
    } else {                                        // torchvision adjust_hue
      for (int i = threadIdx.x; i < nloc; i += blockDim.x) {
        int h, s, val, r, g, b;
        rgb2hsv_u8(cur[i * 3], cur[i * 3 + 1], cur[i * 3 + 2], h, s, val);
        h = (h + v.hue_shift) & 255;
        hsv2rgb_u8(h, s, val, r, g, b);
        cur[i * 3 + 0] = static_cast<uint8_t>(r);
        cur[i * 3 + 1] = static_cast<uint8_t>(g);
        cur[i * 3 + 2] = static_cast<uint8_t>(b);
      }
    }
    clip_sync<CL>();
  }
  const int gch = v.gray[t];
  if (gch >= 0) {                                   // ClipRandomGray.grayscale
    for (int i = threadIdx.x; i < nloc; i += blockDim.x) {
      const uint8_t c = cur[i * 3 + gch];
      cur[i * 3 + 0] = c;
      cur[i * 3 + 1] = c;
      cur[i * 3 + 2] = c;
    }
    clip_sync<CL>();
  }
  if (v.blur) {                                     // ImagingGaussianBlur: 3 horizontal passes, then 3 vertical ones
    for (int pass = 0; pass < 6; ++pass) {
      const bool vertical = pass >= 3;
      // horizontal lines are this CTA's rows; the pair's vertical lines (columns) are shared out over both CTAs
      const bool pair_cols = CL == 2 && vertical;
      const int jobs = vertical ? S * 3 : nloc / S * 3;
      const StagedRows<CL> crow(cur, i_half, S * 3), orow(oth, i_half, S * 3);
      for (int job = (pair_cols ? rank * blockDim.x : 0) + threadIdx.x; job < jobs; job += (pair_cols ? CL : 1) * blockDim.x) {
        const int line = job / 3, c = job - line * 3;
        if (pair_cols) {
          const int col = line * 3 + c;
          box_blur_line<true>(crow(0) + col, crow(i_half) + col, orow(0) + col, orow(i_half) + col, i_half, S * 3, S,
                              v.blur_radius, v.blur_edge_a, v.blur_edge_b, v.blur_ww, v.blur_fw);
        } else {
          const int base = (vertical ? line : line * S) * 3 + c;
          box_blur_line<false>(cur + base, nullptr, oth + base, nullptr, S, (vertical ? S : 1) * 3, S, v.blur_radius,
                               v.blur_edge_a, v.blur_edge_b, v.blur_ww, v.blur_fw);
        }
      }
      clip_sync<CL>();
      uint8_t* s = cur;
      cur = oth;
      oth = s;
    }
  }

  // ---- 4. flip, ToTensor, Normalize('tf'); (3, T, S, S) fp32, coalesced along x
  float* __restrict__ out = v.out;
  for (int i = threadIdx.x; i < nloc * 3; i += blockDim.x) {
    const int c = i / nloc, r = i - c * nloc;
    const int y = r / S, x = r - y * S;
    const int sx = v.flip ? S - 1 - x : x;
    const float val = static_cast<float>(cur[(y * S + sx) * 3 + c]);
    out[(static_cast<size_t>(c) * T + t) * npix + i_lo * S + r] = __fsub_rn(__fmul_rn(__fdiv_rn(val, 255.f), 2.f), 1.f);
  }
}

}  // namespace cstp

using namespace cstp;

namespace {

constexpr int kClipSmemLimit = 226 * 1024;      // 227 KB per CTA minus the kernel's static shared memory

struct ClipLayout {
  int cluster, tmp_bytes, img_bytes, smem;
};

// One CTA per (frame, view) when tmp [crop_h][S][3] and two [S][S][3] images fit; else a cluster pair, each CTA holding
// half the rows of tmp (aliased by oth) and of cur.  Chosen from (S, max_crop_h) alone.
int clip_layout(int S, int max_crop_h, ClipLayout* L) {
  const int row = S * 3;
  L->cluster = 1;
  L->tmp_bytes = (max_crop_h * row + 15) & ~15;
  L->img_bytes = (S * row + 15) & ~15;
  L->smem = L->tmp_bytes + 2 * L->img_bytes;
  if (L->smem <= kClipSmemLimit) return CSTP_OK;
  const int half_h = (max_crop_h + 1) / 2, half_s = (S + 1) / 2;
  L->cluster = 2;
  L->tmp_bytes = ((half_h > half_s ? half_h : half_s) * row + 15) & ~15;
  L->img_bytes = (half_s * row + 15) & ~15;
  L->smem = L->tmp_bytes + L->img_bytes;
  if (L->smem <= kClipSmemLimit) return CSTP_OK;
  set_error("invalid argument: crop height %d needs %d bytes of shared memory (limit %d)", max_crop_h, L->smem, kClipSmemLimit);
  return CSTP_EINVAL;
}

}  // namespace

extern "C" int cstp_clip_layout(int S, int max_crop_h, int* cluster, int* smem_bytes) {
  CSTP_REQUIRE(S >= 8 && S <= CSTP_CLIP_S && max_crop_h > 0);
  ClipLayout L;
  const int rc = clip_layout(S, max_crop_h, &L);
  if (rc != CSTP_OK) return rc;
  if (cluster) *cluster = L.cluster;
  if (smem_bytes) *smem_bytes = L.smem;
  return CSTP_OK;
}

extern "C" int cstp_clip_assemble(const cstp_clip_view* views, int n_views, int T, int S, int max_crop_h, void* stream) {
  CSTP_REQUIRE(views != nullptr && n_views > 0 && T > 0 && T <= CSTP_CLIP_T && S >= 8 && S <= CSTP_CLIP_S && max_crop_h > 0);
  ClipLayout L;
  const int rc = clip_layout(S, max_crop_h, &L);
  if (rc != CSTP_OK) return rc;
  static bool attr_set = false;
  if (!attr_set) {
    CSTP_CUDA(cudaFuncSetAttribute(clip_assemble_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, kClipSmemLimit));
    CSTP_CUDA(cudaFuncSetAttribute(clip_assemble_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, kClipSmemLimit));
    attr_set = true;
  }
  if (L.cluster == 1) {
    clip_assemble_kernel<1><<<dim3(T, n_views), kClipThreads, L.smem, static_cast<cudaStream_t>(stream)>>>(views, T, S, L.tmp_bytes,
                                                                                                       L.img_bytes);
  } else {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(static_cast<unsigned>(2 * T), static_cast<unsigned>(n_views), 1);
    cfg.blockDim = dim3(kClipThreads, 1, 1);
    cfg.dynamicSmemBytes = static_cast<size_t>(L.smem);
    cfg.stream = static_cast<cudaStream_t>(stream);
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = 2;
    at[0].val.clusterDim.y = 1;
    at[0].val.clusterDim.z = 1;
    cfg.attrs = at;
    cfg.numAttrs = 1;
    CSTP_CUDA(cudaLaunchKernelEx(&cfg, clip_assemble_kernel<2>, views, T, S, L.tmp_bytes, L.img_bytes));
  }
  CSTP_LAUNCHED();
  return CSTP_OK;
}

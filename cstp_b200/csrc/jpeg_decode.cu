// Baseline JPEG decoding on the GPU, byte-exact with Pillow on libjpeg-turbo (JDCT_ISLOW, fancy upsampling).
//
// One batch of streams is decoded by three launches on the caller's stream:
//   A. jpeg_entropy_kernel: one warp per image.  Lane 0 walks the marker segments and builds the tables in shared
//      memory; the warp fills the Huffman lookahead tables, zeroes the image's coefficient slice and finds the restart
//      markers; then each lane entropy-decodes whole restart intervals (lane l takes intervals l, l + 32, ...) into
//      de-zigzagged int16 coefficient blocks.
//   B. jpeg_idct_kernel: one thread per 8x8 block: dequantise + ISLOW IDCT into uint8 component planes.
//   C. jpeg_colour_kernel: one thread per output pixel: fancy upsampling of the chroma planes + YCbCr -> RGB.
//
// The arithmetic follows the code Pillow runs, not the C reference alone:
//   * IDCT: libjpeg-turbo's SIMD jpeg_idct_islow.  It forms coef * quant and the sums x0 +- x4, x7 + x3, x5 + x1 in
//     16 bits, keeps the rotations' products exact in 32 bits, saturates each pass's descaled output to int16 and the
//     final one to [-128, 127] (a clamp where jidctint.c's range-limit table would wrap).  Valid streams reach none of
//     these limits; the stand-in tests/emulate_jpeg.py pins them against Pillow with scaled-up quantisation tables.
//   * Upsampling: jdsample.c's h2v1 / h2v2 fancy upsamplers (biases +1 / +2 and +8 / +7, edge columns replicated), plain
//     replication when the chroma plane is at most 2 samples wide (jinit_upsampler), context rows clamped to the last
//     real row of the component (jdmainct.c), never the IDCT's padding rows.
//   * Colour: jdcolor.c's Q16 tables (FIX(1.40200), FIX(1.77200), -FIX(0.71414), -FIX(0.34414), ONE_HALF), clamped.
//
// Robustness by construction: every stream read is bounded by src_bytes, every coefficient / plane / interval write
// by counts derived from the expected size (which SOF must match), and the Huffman decoder consumes a bounded number
// of symbols per block.  Where libjpeg would warn and fill in zeros (bad Huffman code, data running out, extraneous
// bytes, a wrong restart marker), the image is reported as CSTP_JPEG_MALFORMED instead.
#include "common.h"

namespace cstp {

constexpr int kJpegHdrBytes = 512;
constexpr int kIdctThreads = 128;
constexpr int kIdctCtasPerImage = 8;
constexpr int kColourThreads = 256;
constexpr int kColourCtasPerImage = 16;
constexpr int kHuffSlots = 8;          // (class, id): DC 0-3, AC 0-3

__host__ __device__ inline long long align256(long long x) { return (x + 255) & ~255ll; }
__host__ __device__ inline long long cdiv(long long a, long long b) { return (a + b - 1) / b; }

// Upper bound of coefficient blocks (MCU-padded) over every supported sampling: 4:4:4 (3 per 8x8 MCU), 4:2:2 (4 per
// 16x8), 4:2:0 (6 per 16x16), grayscale (1 per 8x8).
__host__ __device__ inline long long jpeg_max_blocks(int w, int h) {
  const long long b8 = cdiv(w, 8) * cdiv(h, 8), b422 = 4 * cdiv(w, 16) * cdiv(h, 8), b420 = 6 * cdiv(w, 16) * cdiv(h, 16);
  const long long m = 3 * b8 > b422 ? 3 * b8 : b422;
  return m > b420 ? m : b420;
}

// Per-image workspace: [header][int16 coefficients][uint8 planes][restart intervals (begin, end)].
struct JpegWs {
  long long coef, plane, iv, total;
};
__host__ __device__ inline JpegWs jpeg_ws(int w, int h) {
  const long long nb = jpeg_max_blocks(w, h);
  JpegWs s;
  s.coef = kJpegHdrBytes;
  s.plane = s.coef + align256(nb * 128);
  s.iv = s.plane + align256(nb * 64);
  s.total = s.iv + align256(cdiv(w, 8) * cdiv(h, 8) * 8);
  return s;
}

struct JpegHdr {                        // written by stage A for a decoded image, read by B and C
  int32_t ncomp;
  int32_t h[3], v[3];
  uint16_t q[3][64];                    // natural order
};
static_assert(sizeof(JpegHdr) <= kJpegHdrBytes, "header slot");

struct JpegLayout {
  int ncomp, hmax, vmax, mcux, mcuy;
  int h[3], v[3], bw[3], bh[3], dw[3], dh[3];
  long long cbase[3], nblocks;          // first block of each component, total blocks
};

__device__ inline JpegLayout jpeg_layout(int ncomp, const int* h, const int* v, int w, int ht) {
  JpegLayout L;
  L.ncomp = ncomp;
  L.hmax = L.vmax = 1;
#pragma unroll
  for (int c = 0; c < 3; ++c)
    if (c < ncomp) L.hmax = max(L.hmax, h[c]), L.vmax = max(L.vmax, v[c]);
  L.mcux = static_cast<int>(cdiv(w, 8 * L.hmax));
  L.mcuy = static_cast<int>(cdiv(ht, 8 * L.vmax));
  long long base = 0;
#pragma unroll
  for (int c = 0; c < 3; ++c) {              // unused components get an empty block grid
    const int hc = c < ncomp ? h[c] : 0, vc = c < ncomp ? v[c] : 0;
    L.h[c] = hc, L.v[c] = vc;
    L.bw[c] = L.mcux * hc, L.bh[c] = L.mcuy * vc;
    L.dw[c] = static_cast<int>(cdiv(static_cast<long long>(w) * hc, L.hmax));
    L.dh[c] = static_cast<int>(cdiv(static_cast<long long>(ht) * vc, L.vmax));
    L.cbase[c] = base;
    base += static_cast<long long>(L.bw[c]) * L.bh[c];
  }
  L.nblocks = base;
  return L;
}

__constant__ uint8_t kZigzag[64] = {0,  1,  8,  16, 9,  2,  3,  10, 17, 24, 32, 25, 18, 11, 4,  5,
                                    12, 19, 26, 33, 40, 48, 41, 34, 27, 20, 13, 6,  7,  14, 21, 28,
                                    35, 42, 49, 56, 57, 50, 43, 36, 29, 22, 15, 23, 30, 37, 44, 51,
                                    58, 59, 52, 45, 38, 31, 39, 46, 53, 60, 61, 54, 47, 55, 62, 63};

// ---------------------------------------------------------------------------------------------------------------
// Stage A
struct HuffTab {
  uint16_t lut[512];                    // 9-bit lookahead: (length << 8) | symbol, 0 when the code is longer
  int32_t maxcode[18];                  // largest code of each length, -1 when there is none
  int32_t valoff[17];                   // vals index of code c of length l: valoff[l] + c
  uint8_t vals[256];
};

struct ParseState {
  int status;
  int ncomp, dri, data;                 // data: first byte of the entropy-coded segment
  int id[3], h[3], v[3], tq[3], td[3], ta[3];
  int defined_q, defined_h;             // bit masks
};

struct EntropySmem {
  HuffTab tab[kHuffSlots];
  uint16_t q[4][64];
  ParseState ps;
};

__device__ inline int rd16(const uint8_t* d, int p) { return (d[p] << 8) | d[p + 1]; }

// A DHT table: jpeg_make_d_derived_tbl's checks, then maxcode / valoff.  Returns false when libjpeg would reject it.
__device__ bool jpeg_define_huff(HuffTab& t, const uint8_t* counts, bool dc) {
  int code = 0, k = 0;
  for (int l = 1; l <= 16; ++l) {
    const int n = counts[l - 1];
    t.maxcode[l] = -1;
    if (n) {
      t.valoff[l] = k - code;
      code += n;
      k += n;
      if (code > (1 << l)) return false;
      t.maxcode[l] = code - 1;
    }
    code <<= 1;
  }
  t.maxcode[17] = 1 << 30;
  if (dc)
    for (int i = 0; i < k; ++i)
      if (t.vals[i] > 15) return false;
  return true;
}

// Lane 0's marker walk from SOI to the end of the SOS header.  Mirrors tests/emulate_jpeg.py::parse.
__device__ int jpeg_parse(const uint8_t* d, int n, int width, int height, EntropySmem& sm) {
  ParseState& ps = sm.ps;
  ps.defined_q = ps.defined_h = 0;
  ps.dri = 0;
  ps.ncomp = 0;
  bool saw_jfif = false;
  int adobe = -1;
  if (n < 4 || d[0] != 0xFF || d[1] != 0xD8) return CSTP_JPEG_MALFORMED;
  int pos = 2;
  for (;;) {
    if (pos >= n || d[pos] != 0xFF) return CSTP_JPEG_MALFORMED;
    while (pos < n && d[pos] == 0xFF) ++pos;
    if (pos + 3 > n) return CSTP_JPEG_MALFORMED;
    const int m = d[pos++];
    if ((m >= 0xC2 && m <= 0xCF && m != 0xC4) || m == 0xDE || m == 0xDF) return CSTP_JPEG_UNSUPPORTED;
    if (!(m == 0xC0 || m == 0xC1 || m == 0xC4 || m == 0xDA || m == 0xDB || m == 0xDD || m == 0xFE ||
          (m >= 0xE0 && m <= 0xEF)))
      return CSTP_JPEG_MALFORMED;
    const int seg = rd16(d, pos), end = pos + seg;
    if (seg < 2 || end > n) return CSTP_JPEG_MALFORMED;
    int p = pos + 2;
    if (m == 0xC0 || m == 0xC1) {
      if (ps.ncomp != 0 || seg < 8) return CSTP_JPEG_MALFORMED;
      if (d[p] != 8) return CSTP_JPEG_UNSUPPORTED;
      const int h = rd16(d, p + 1), w = rd16(d, p + 3), nf = d[p + 5];
      if (seg != 8 + 3 * nf || nf == 0) return CSTP_JPEG_MALFORMED;
      if ((nf != 1 && nf != 3) || h == 0) return CSTP_JPEG_UNSUPPORTED;
      for (int c = 0; c < nf; ++c) {
        const int hv = d[p + 7 + 3 * c], tq = d[p + 8 + 3 * c];
        ps.id[c] = d[p + 6 + 3 * c];
        ps.h[c] = hv >> 4, ps.v[c] = hv & 15, ps.tq[c] = tq;
        if (ps.h[c] < 1 || ps.h[c] > 4 || ps.v[c] < 1 || ps.v[c] > 4 || tq > 3) return CSTP_JPEG_MALFORMED;
      }
      if (w == 0) return CSTP_JPEG_MALFORMED;
      if (w != width || h != height) return CSTP_JPEG_SIZE;
      if (nf == 3) {
        const bool y_ok = (ps.h[0] == 1 && ps.v[0] == 1) || (ps.h[0] == 2 && (ps.v[0] == 1 || ps.v[0] == 2));
        if (!y_ok || ps.h[1] != 1 || ps.v[1] != 1 || ps.h[2] != 1 || ps.v[2] != 1) return CSTP_JPEG_UNSUPPORTED;
      }
      ps.ncomp = nf;
    } else if (m == 0xC4) {
      while (p < end) {
        const int tc = d[p] >> 4, th = d[p] & 15;
        if (tc > 1 || th > 3 || p + 17 > end) return CSTP_JPEG_MALFORMED;
        int tot = 0;
        for (int i = 0; i < 16; ++i) tot += d[p + 1 + i];
        if (tot > 256 || p + 17 + tot > end) return CSTP_JPEG_MALFORMED;
        HuffTab& t = sm.tab[tc * 4 + th];
        for (int i = 0; i < tot; ++i) t.vals[i] = d[p + 17 + i];
        if (!jpeg_define_huff(t, d + p + 1, tc == 0)) return CSTP_JPEG_MALFORMED;
        ps.defined_h |= 1 << (tc * 4 + th);
        p += 17 + tot;
      }
    } else if (m == 0xDB) {
      while (p < end) {
        const int pq = d[p] >> 4, tq = d[p] & 15;
        if (pq > 1 || tq > 3 || p + 1 + 64 * (pq + 1) > end) return CSTP_JPEG_MALFORMED;
        for (int k = 0; k < 64; ++k) sm.q[tq][kZigzag[k]] = pq ? rd16(d, p + 1 + 2 * k) : d[p + 1 + k];
        ps.defined_q |= 1 << tq;
        p += 1 + 64 * (pq + 1);
      }
    } else if (m == 0xDD) {
      if (seg != 4) return CSTP_JPEG_MALFORMED;
      ps.dri = rd16(d, p);
    } else if (m == 0xE0) {
      if (seg - 2 >= 14 && d[p] == 'J' && d[p + 1] == 'F' && d[p + 2] == 'I' && d[p + 3] == 'F' && d[p + 4] == 0)
        saw_jfif = true;
    } else if (m == 0xEE) {
      if (seg - 2 >= 12 && d[p] == 'A' && d[p + 1] == 'd' && d[p + 2] == 'o' && d[p + 3] == 'b' && d[p + 4] == 'e')
        adobe = d[p + 11];
    } else if (m == 0xDA) {
      if (ps.ncomp == 0 || seg < 3) return CSTP_JPEG_MALFORMED;
      const int ns = d[p];
      if (seg != 6 + 2 * ns) return CSTP_JPEG_MALFORMED;
      if (ns != ps.ncomp) return CSTP_JPEG_UNSUPPORTED;      // one interleaved scan only
      for (int c = 0; c < ns; ++c) {
        const int cs = d[p + 1 + 2 * c], t = d[p + 2 + 2 * c];
        if (cs != ps.id[c]) return CSTP_JPEG_UNSUPPORTED;
        if ((t >> 4) > 3 || (t & 15) > 3) return CSTP_JPEG_MALFORMED;
        ps.td[c] = t >> 4, ps.ta[c] = t & 15;
      }
      const int q = p + 1 + 2 * ns;
      if (d[q] != 0 || d[q + 1] != 63 || d[q + 2] != 0) return CSTP_JPEG_UNSUPPORTED;
      for (int c = 0; c < ns; ++c) {
        if (!((ps.defined_q >> ps.tq[c]) & 1)) return CSTP_JPEG_MALFORMED;
        // libjpeg-turbo would substitute the standard tables (Motion-JPEG); not supported here
        if (!((ps.defined_h >> ps.td[c]) & 1) || !((ps.defined_h >> (4 + ps.ta[c])) & 1)) return CSTP_JPEG_UNSUPPORTED;
      }
      if (ns == 3 && !saw_jfif && (adobe == 0 || (adobe < 0 && ps.id[0] == 82 && ps.id[1] == 71 && ps.id[2] == 66)))
        return CSTP_JPEG_UNSUPPORTED;                          // RGB, not YCbCr
      if (ns == 1) ps.h[0] = ps.v[0] = 1;                     // a one-component scan codes one block per MCU
      ps.data = end;
      return 0;
    }
    pos = end;
  }
}

struct BitReader {
  const uint8_t* d;
  int pos, end, fake;
  int nb;
  uint64_t acc;                         // left-aligned

  __device__ __forceinline__ void fill() {   // leaves nb >= 32
    if (pos + 4 <= end) {
      const uint32_t b0 = d[pos], b1 = d[pos + 1], b2 = d[pos + 2], b3 = d[pos + 3];
      if (b0 != 0xFF && b1 != 0xFF && b2 != 0xFF && b3 != 0xFF) {
        acc |= static_cast<uint64_t>((b0 << 24) | (b1 << 16) | (b2 << 8) | b3) << (32 - nb);
        nb += 32;
        pos += 4;
        return;
      }
    }
    while (nb <= 56) {
      uint32_t v = 0;
      if (pos < end) {
        v = d[pos];
        pos += v == 0xFF ? 2 : 1;       // every 0xFF inside an interval is followed by its stuffed 0x00
      } else {
        ++fake;
      }
      acc |= static_cast<uint64_t>(v) << (56 - nb);
      nb += 8;
    }
  }
  __device__ __forceinline__ uint32_t get(int k) {
    const uint32_t v = static_cast<uint32_t>(acc >> (64 - k));
    acc <<= k;
    nb -= k;
    return v;
  }
  // Huffman symbol, or -1 for a code no table entry matches
  __device__ __forceinline__ int sym(const HuffTab& t) {
    const uint32_t e = t.lut[acc >> 55];
    if (e >> 8) {
      get(e >> 8);
      return e & 0xFF;
    }
    for (int l = 10; l <= 16; ++l) {
      const int code = static_cast<int>(acc >> (64 - l));
      if (code <= t.maxcode[l]) {
        get(l);
        return t.vals[t.valoff[l] + code];
      }
    }
    return -1;
  }
};

__device__ __forceinline__ int huff_extend(uint32_t v, int s) {
  return v < (1u << (s - 1)) ? static_cast<int>(v) - (1 << s) + 1 : static_cast<int>(v);
}

__global__ void __launch_bounds__(32) jpeg_entropy_kernel(const uint8_t* __restrict__ data,
                                                          const cstp_jpeg_image* __restrict__ images,
                                                          int32_t* __restrict__ status, uint8_t* __restrict__ ws,
                                                          long long ws_bytes) {
  __shared__ EntropySmem sm;
  const int img = blockIdx.x, lane = threadIdx.x;
  const cstp_jpeg_image im = images[img];
  const int W = im.width, H = im.height;
  if (W <= 0 || H <= 0 || W > 65535 || H > 65535 || im.ws_offset < 0 || (im.ws_offset & 255) != 0 ||
      im.ws_offset + jpeg_ws(W, H).total > ws_bytes || im.src_offset < 0 || im.src_bytes < 0 ||
      im.src_bytes > 0x7fffffff) {
    if (lane == 0) status[img] = CSTP_JPEG_SIZE;
    return;
  }
  const uint8_t* d = data + im.src_offset;
  const int n = static_cast<int>(im.src_bytes);
  uint8_t* base = ws + im.ws_offset;
  const JpegWs off = jpeg_ws(W, H);
  if (lane == 0) sm.ps.status = jpeg_parse(d, n, W, H, sm);
  __syncwarp();
  int st = sm.ps.status;
  if (st != 0) {
    if (lane == 0) status[img] = st;
    return;
  }
  const ParseState& ps = sm.ps;
  // Huffman lookahead tables of every defined slot
  for (int s = 0; s < kHuffSlots; ++s) {
    if (!((ps.defined_h >> s) & 1)) continue;
    HuffTab& t = sm.tab[s];
    for (int i = lane; i < 512; i += 32) {
      uint16_t e = 0;
      for (int l = 1; l <= 9; ++l) {
        const int code = i >> (9 - l);
        if (code <= t.maxcode[l]) {
          e = static_cast<uint16_t>((l << 8) | t.vals[t.valoff[l] + code]);
          break;
        }
      }
      t.lut[i] = e;
    }
  }
  const JpegLayout L = jpeg_layout(ps.ncomp, ps.h, ps.v, W, H);
  int16_t* coef = reinterpret_cast<int16_t*>(base + off.coef);
  {
    int4* z = reinterpret_cast<int4*>(coef);
    for (long long i = lane; i < L.nblocks * 8; i += 32) z[i] = make_int4(0, 0, 0, 0);
  }
  // Restart intervals: the warp tests 32 positions per step for a marker (0xFF followed by neither 0x00 nor 0xFF)
  const long long total = static_cast<long long>(L.mcux) * L.mcuy;
  const int ri = ps.dri ? ps.dri : static_cast<int>(total);
  const int n_int = static_cast<int>(cdiv(total, ri));
  int2* iv = reinterpret_cast<int2*>(base + off.iv);
  {
    int k = 0, begin = ps.data;
    bool done = false, bad = false;
    for (int b0 = ps.data; !done; b0 += 32) {
      const int p = b0 + lane;
      const bool mk = p + 1 < n && d[p] == 0xFF && d[p + 1] != 0x00 && d[p + 1] != 0xFF;
      unsigned m = __ballot_sync(0xffffffffu, mk);
      while (m && !done) {
        const int mp = b0 + __ffs(m) - 1;
        m &= m - 1;
        const int code = d[mp + 1];
        int e = mp;
        while (e > begin && d[e - 1] == 0xFF) --e;
        if (lane == 0) iv[k] = make_int2(begin, e);
        if (code == 0xD9) {
          bad = k != n_int - 1;
          done = true;
        } else if (code != 0xD0 + (k & 7) || k >= n_int - 1) {
          bad = done = true;
        } else {
          ++k;
          begin = mp + 2;
        }
      }
      if (!done && b0 + 31 >= n - 2) bad = done = true;   // no closing marker: truncated
    }
    if (bad) {
      if (lane == 0) status[img] = CSTP_JPEG_MALFORMED;
      return;
    }
  }
  __syncwarp();
  bool err = false;
  for (int k = lane; k < n_int && !err; k += 32) {
    const int2 be = iv[k];
    BitReader br{d, be.x, be.y, 0, 0, 0ull};
    int pred[3] = {0, 0, 0};
    const long long m_end = min(total, static_cast<long long>(k + 1) * ri);
    for (long long m = static_cast<long long>(k) * ri; m < m_end && !err; ++m) {
      const int my = static_cast<int>(m / L.mcux), mx = static_cast<int>(m - static_cast<long long>(my) * L.mcux);
#pragma unroll
      for (int c = 0; c < 3; ++c) {
        if (c >= L.ncomp || err) break;
        const HuffTab& dc = sm.tab[ps.td[c]];
        const HuffTab& ac = sm.tab[4 + ps.ta[c]];
        for (int by = 0; by < L.v[c] && !err; ++by)
          for (int bx = 0; bx < L.h[c] && !err; ++bx) {
            int16_t* blk = coef + (L.cbase[c] + static_cast<long long>(my * L.v[c] + by) * L.bw[c] + mx * L.h[c] + bx) * 64;
            if (br.nb < 32) br.fill();
            int s = br.sym(dc);
            if (s < 0) {
              err = true;
              break;
            }
            if (s) {
              if (br.nb < 32) br.fill();
              pred[c] += huff_extend(br.get(s), s);
            }
            blk[0] = static_cast<int16_t>(pred[c]);
            for (int z = 1; z < 64; ++z) {
              if (br.nb < 32) br.fill();
              const int rs = br.sym(ac);
              if (rs < 0) {
                err = true;
                break;
              }
              const int r = rs >> 4;
              s = rs & 15;
              if (s) {
                z += r;
                if (z > 63) {
                  err = true;
                  break;
                }
                blk[kZigzag[z]] = static_cast<int16_t>(huff_extend(br.get(s), s));
              } else if (r == 15) {
                z += 15;
              } else {
                break;
              }
            }
          }
      }
    }
    // ran into the zeros past the interval's data, or left whole bytes of it unread
    if (br.nb < 8 * br.fake || br.pos < br.end || br.nb - 8 * br.fake >= 8) err = true;
  }
  err = __any_sync(0xffffffffu, err);
  if (err) {
    if (lane == 0) status[img] = CSTP_JPEG_MALFORMED;
    return;
  }
  JpegHdr* hdr = reinterpret_cast<JpegHdr*>(base);
  for (int i = lane; i < L.ncomp * 64; i += 32) hdr->q[i >> 6][i & 63] = sm.q[ps.tq[i >> 6]][i & 63];
  if (lane == 0) {
    hdr->ncomp = L.ncomp;
    for (int c = 0; c < 3; ++c) hdr->h[c] = c < L.ncomp ? L.h[c] : 1, hdr->v[c] = c < L.ncomp ? L.v[c] : 1;
    status[img] = 0;
  }
}

// ---------------------------------------------------------------------------------------------------------------
// Stage B: libjpeg-turbo's SIMD jpeg_idct_islow (see the file comment for its 16-bit steps).
constexpr int F0298 = 2446, F0390 = 3196, F0541 = 4433, F0765 = 6270, F0899 = 7373, F1175 = 9633, F1501 = 12299,
              F1847 = 15137, F1961 = 16069, F2053 = 16819, F2562 = 20995, F3072 = 25172;

__device__ __forceinline__ int s16(int x) { return static_cast<int16_t>(x); }

// x[0..7] in, the 8 undescaled outputs back into x
__device__ __forceinline__ void islow_1d(int (&x)[8]) {
  const int t3 = x[2] * (F0541 + F0765) + x[6] * F0541;
  const int t2 = x[2] * F0541 + x[6] * (F0541 - F1847);
  const int t0 = s16(x[0] + x[4]) * 8192;
  const int t1 = s16(x[0] - x[4]) * 8192;
  const int t10 = t0 + t3, t13 = t0 - t3, t11 = t1 + t2, t12 = t1 - t2;
  const int z3a = s16(x[7] + x[3]), z4a = s16(x[5] + x[1]);
  const int z3 = z3a * (F1175 - F1961) + z4a * F1175;
  const int z4 = z3a * F1175 + z4a * (F1175 - F0390);
  const int o0 = x[7] * (F0298 - F0899) + x[1] * -F0899 + z3;
  const int o1 = x[5] * (F2053 - F2562) + x[3] * -F2562 + z4;
  const int o2 = x[5] * -F2562 + x[3] * (F3072 - F2562) + z3;
  const int o3 = x[7] * -F0899 + x[1] * (F1501 - F0899) + z4;
  x[0] = t10 + o3, x[7] = t10 - o3;
  x[1] = t11 + o2, x[6] = t11 - o2;
  x[2] = t12 + o1, x[5] = t12 - o1;
  x[3] = t13 + o0, x[4] = t13 - o0;
}

__global__ void __launch_bounds__(kIdctThreads) jpeg_idct_kernel(const cstp_jpeg_image* __restrict__ images,
                                                                 const int32_t* __restrict__ status,
                                                                 uint8_t* __restrict__ ws) {
  __shared__ int q[3][64];
  const int img = blockIdx.y;
  if (status[img] != 0) return;
  const cstp_jpeg_image im = images[img];
  uint8_t* base = ws + im.ws_offset;
  const JpegWs off = jpeg_ws(im.width, im.height);
  const JpegHdr* hdr = reinterpret_cast<const JpegHdr*>(base);
  const int ncomp = hdr->ncomp;
  const int hh[3] = {hdr->h[0], hdr->h[1], hdr->h[2]}, vv[3] = {hdr->v[0], hdr->v[1], hdr->v[2]};
  const JpegLayout L = jpeg_layout(ncomp, hh, vv, im.width, im.height);
  for (int i = threadIdx.x; i < ncomp * 64; i += kIdctThreads) q[i >> 6][i & 63] = hdr->q[i >> 6][i & 63];
  __syncthreads();
  const int16_t* coef = reinterpret_cast<const int16_t*>(base + off.coef);
  uint8_t* planes = base + off.plane;
  for (long long j = static_cast<long long>(blockIdx.x) * kIdctThreads + threadIdx.x; j < L.nblocks;
       j += static_cast<long long>(gridDim.x) * kIdctThreads) {
    const int c = j >= L.cbase[2] ? 2 : (j >= L.cbase[1] ? 1 : 0);
    const long long cbase = c == 0 ? 0 : (c == 1 ? L.cbase[1] : L.cbase[2]);
    const int bw = c == 0 ? L.bw[0] : (c == 1 ? L.bw[1] : L.bw[2]);
    const long long local = j - cbase;
    const int by = static_cast<int>(local / bw), bx = static_cast<int>(local - static_cast<long long>(by) * bw);
    int ws_[8][8];                      // [row][col] after pass 1
    {
      const int4* src = reinterpret_cast<const int4*>(coef + j * 64);
      int cf[64];
#pragma unroll
      for (int r = 0; r < 8; ++r) {
        const int4 v = src[r];
        const int w4[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          cf[r * 8 + 2 * e] = s16(static_cast<int16_t>(w4[e] & 0xFFFF) * q[c][r * 8 + 2 * e]);
          cf[r * 8 + 2 * e + 1] = s16(static_cast<int16_t>(static_cast<uint32_t>(w4[e]) >> 16) * q[c][r * 8 + 2 * e + 1]);
        }
      }
#pragma unroll
      for (int col = 0; col < 8; ++col) {
        int x[8];
#pragma unroll
        for (int u = 0; u < 8; ++u) x[u] = cf[u * 8 + col];
        islow_1d(x);
#pragma unroll
        for (int y = 0; y < 8; ++y) ws_[y][col] = min(max((x[y] + 1024) >> 11, -32768), 32767);
      }
    }
    uint8_t* dst = planes + cbase * 64 + static_cast<long long>(by * 8) * (bw * 8) + bx * 8;
#pragma unroll
    for (int y = 0; y < 8; ++y) {
      int x[8];
#pragma unroll
      for (int v = 0; v < 8; ++v) x[v] = ws_[y][v];
      islow_1d(x);
      uint32_t lo = 0, hi = 0;
#pragma unroll
      for (int v = 0; v < 8; ++v) {
        const uint32_t px = static_cast<uint32_t>(min(max((x[v] + (1 << 17)) >> 18, -128), 127) + 128);
        if (v < 4) lo |= px << (8 * v);
        else hi |= px << (8 * (v - 4));
      }
      *reinterpret_cast<uint2*>(dst + static_cast<long long>(y) * (bw * 8)) = make_uint2(lo, hi);
    }
  }
}

// ---------------------------------------------------------------------------------------------------------------
// Stage C
__device__ __forceinline__ int jpeg_chroma(const uint8_t* p, int stride, int dw, int dh, int hs, int vs, int x, int y) {
  if (hs == 1 && vs == 1) return p[static_cast<long long>(y) * stride + x];
  if (dw <= 2) return p[static_cast<long long>(y / vs) * stride + x / hs];     // jinit_upsampler: no fancy upsampling
  const int j = x >> 1, odd = x & 1;
  const int nb = odd ? min(j + 1, dw - 1) : max(j - 1, 0);
  if (vs == 1) {
    const uint8_t* r = p + static_cast<long long>(y) * stride;
    return (3 * r[j] + r[nb] + (odd ? 2 : 1)) >> 2;
  }
  const int i = y >> 1;
  const int vn = (y & 1) ? min(i + 1, dh - 1) : max(i - 1, 0);
  const uint8_t* r0 = p + static_cast<long long>(i) * stride;
  const uint8_t* r1 = p + static_cast<long long>(vn) * stride;
  const int cs = 3 * r0[j] + r1[j], cn = 3 * r0[nb] + r1[nb];
  return (3 * cs + cn + (odd ? 7 : 8)) >> 4;
}

__global__ void __launch_bounds__(kColourThreads) jpeg_colour_kernel(const cstp_jpeg_image* __restrict__ images,
                                                                     const int32_t* __restrict__ status,
                                                                     const uint8_t* __restrict__ ws) {
  const int img = blockIdx.y;
  if (status[img] != 0) return;
  const cstp_jpeg_image im = images[img];
  const uint8_t* base = ws + im.ws_offset;
  const JpegWs off = jpeg_ws(im.width, im.height);
  const JpegHdr* hdr = reinterpret_cast<const JpegHdr*>(base);
  const int ncomp = hdr->ncomp;
  const int hh[3] = {hdr->h[0], hdr->h[1], hdr->h[2]}, vv[3] = {hdr->v[0], hdr->v[1], hdr->v[2]};
  const JpegLayout L = jpeg_layout(ncomp, hh, vv, im.width, im.height);
  const uint8_t* planes = base + off.plane;
  const int W = im.width;
  const long long npx = static_cast<long long>(W) * im.height;
  for (long long p = static_cast<long long>(blockIdx.x) * kColourThreads + threadIdx.x; p < npx;
       p += static_cast<long long>(gridDim.x) * kColourThreads) {
    const int y = static_cast<int>(p / W), x = static_cast<int>(p - static_cast<long long>(y) * W);
    const int Y = planes[static_cast<long long>(y) * (L.bw[0] * 8) + x];
    uint8_t* o = im.out + p * 3;
    if (ncomp == 1) {
      o[0] = o[1] = o[2] = static_cast<uint8_t>(Y);
      continue;
    }
    const int cb = jpeg_chroma(planes + L.cbase[1] * 64, L.bw[1] * 8, L.dw[1], L.dh[1], L.hmax / L.h[1], L.vmax / L.v[1], x,
                               y) - 128;
    const int cr = jpeg_chroma(planes + L.cbase[2] * 64, L.bw[2] * 8, L.dw[2], L.dh[2], L.hmax / L.h[2], L.vmax / L.v[2], x,
                               y) - 128;
    const int r = Y + ((91881 * cr + 32768) >> 16);
    const int g = Y + ((-22554 * cb + 32768 - 46802 * cr) >> 16);
    const int b = Y + ((116130 * cb + 32768) >> 16);
    o[0] = static_cast<uint8_t>(min(max(r, 0), 255));
    o[1] = static_cast<uint8_t>(min(max(g, 0), 255));
    o[2] = static_cast<uint8_t>(min(max(b, 0), 255));
  }
}

}  // namespace cstp

using namespace cstp;

extern "C" long long cstp_jpeg_workspace_bytes(int width, int height) {
  if (width <= 0 || height <= 0 || width > 65535 || height > 65535) {
    fail_inval("width and height in 1 .. 65535");
    return -1;
  }
  return jpeg_ws(width, height).total;
}

extern "C" int cstp_jpeg_decode(const uint8_t* data, const cstp_jpeg_image* images, int n_images, int32_t* status,
                                void* workspace, long long workspace_bytes, void* stream) {
  CSTP_REQUIRE(data && images && status && workspace && n_images > 0 && n_images <= 65535 && workspace_bytes > 0);
  CSTP_REQUIRE(reinterpret_cast<uintptr_t>(workspace) % 256 == 0);
  const cudaStream_t s = static_cast<cudaStream_t>(stream);
  uint8_t* ws = static_cast<uint8_t*>(workspace);
  jpeg_entropy_kernel<<<n_images, 32, 0, s>>>(data, images, status, ws, workspace_bytes);
  CSTP_LAUNCHED();
  jpeg_idct_kernel<<<dim3(kIdctCtasPerImage, n_images), kIdctThreads, 0, s>>>(images, status, ws);
  CSTP_LAUNCHED();
  jpeg_colour_kernel<<<dim3(kColourCtasPerImage, n_images), kColourThreads, 0, s>>>(images, status, ws);
  CSTP_LAUNCHED();
  return CSTP_OK;
}

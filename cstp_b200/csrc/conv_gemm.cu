// Implicit-GEMM convolution (forward and dgrad) and linear layers on tcgen05 tensor cores.
//
// One persistent CTA per SM, warp-specialised:
//   warp 0 (one lane)  TMA producer: per K-block one 5-D box of activations (128 positions x 64 channels, the tap
//                      shift folded into the box origin; out-of-range taps are zero-filled by TMA = conv padding)
//                      and one 2-D box of packed weights (n_tile x 64).
//   warp 1 (one lane)  tcgen05.mma issuer: D[128 x n_tile] fp32 in TMEM, double-buffered across tiles.
//   warp 2             TMEM allocator.
//   warps 4..7         epilogue: tcgen05.ld -> (+bias, +previous) -> bf16 / fp32 rows to global.
// CTA pairs (thread-block clusters of two, launched with the cluster attribute): the two CTAs take neighbouring M tiles of
// the SAME N tile in lockstep; each loads half of the weight tile and multicasts it into both shared memories, and a stage
// is released by the MMA commits of both (multicast arrive).  The kernel is bound by the L2 -> SM feed on the deep layers
// (16 KB of activations + 24-32 KB of weights per 64-channel K-block): the pair reads every weight tile from L2 once.
// Replaces cuDNN conv3d fwd/dgrad and cuBLAS addmm behind models/pace/r21d_byol.py:81-97,236-253.
#include "common.h"
#include "ptx.cuh"

namespace cstp {

constexpr int kConvThreads = 256;
constexpr int kConvXformThreads = 256;      // warps 8..15: operand prologue (BatchNorm affine + ReLU on the staged A box)
constexpr uint32_t kABytes = 128 * 64 * 2;  // one A stage: 128 positions x 64 bf16 channels
constexpr int kMaxStages = 8;
constexpr int kSmemLimit = 232448;  // 227 KB

struct ConvKParams {
  CUtensorMap amap[CSTP_MAX_AMAPS];
  CUtensorMap bmap;
  CUtensorMap bmap_half;   // boxes of n_tile / 2 rows: what one CTA of a pair loads (and multicasts)
  int tiles_w, tiles_h, tiles_t, tiles_n, n_ntiles;
  int bw, bh, bt, bn;
  int Wt, Ht, Tt, Nt;
  int n_taps, chunks_per_tap, last_ksteps;
  int n_tile, Np;
  int stages, tmem_cols;
  uint32_t b_bytes, idesc;
  int accumulate;
  int fast_store;          // bf16 output only, no bias, 32-byte aligned rows: pipelined epilogue with STG.256
  const float* pro_scale;  // operand prologue (kXform): fp32 [pro_groups][pro_cp] BatchNorm affine of the producer of A
  const float* pro_shift;
  int pro_groups, pro_cp;
  __nv_bfloat16* out;
  float* out_f32;
  const float* bias;
  long long out_off, osw, osh, ost, osn;
  int n_classes;                          // tap classes (stride-parity classes of a dgrad) run as one launch
  int cls_first_tap[8], cls_n_taps[8];
  long long cls_out_off[8];
  cstp_tap taps[CSTP_MAX_TAPS];
};

struct TileCoord {
  int w0, h0, t0, n0, ntile, cls;
};

// Class of a tile.  Class-minor order (the classes of one M tile are neighbours in the tile order and run at the same
// time on neighbouring CTAs), rotated by the M tile index: with a plain tile % n_classes a persistent CTA (stride = grid
// size, a multiple of the class count) would see ONE class for ever -- and the classes differ in taps (1, 2, 2, 4 for a
// stride-2 1x3x3 dgrad: measured 1.78x slower than balanced).
__device__ __forceinline__ int tile_class(int n_classes, int tile) {
  return (tile + tile / n_classes) % n_classes;
}

// (csize, crank): CTAs per cluster and this CTA's rank -- a "tile" of a pair is two neighbouring M tiles (the second one
// may lie beyond the tile space: its loads are zero-filled, its rows fail the validity test of the epilogue).
__device__ __forceinline__ TileCoord decode_tile(const ConvKParams& p, int tile, int csize = 1, int crank = 0) {
  TileCoord c;
  c.cls = tile_class(p.n_classes, tile);
  tile /= p.n_classes;
  c.ntile = tile % p.n_ntiles;
  int pt = (tile / p.n_ntiles) * csize + crank;
  c.w0 = (pt % p.tiles_w) * p.bw;
  pt /= p.tiles_w;
  c.h0 = (pt % p.tiles_h) * p.bh;
  pt /= p.tiles_h;
  c.t0 = (pt % p.tiles_t) * p.bt;
  pt /= p.tiles_t;
  c.n0 = pt * p.bn;
  return c;
}

template <bool kXform>
__global__ void __launch_bounds__(kXform ? kConvThreads + kConvXformThreads : kConvThreads, 1)
    conv_gemm_kernel(const __grid_constant__ ConvKParams p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  const uint32_t stage_bytes = kABytes + p.b_bytes;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + static_cast<size_t>(p.stages) * stage_bytes);
  uint64_t* full = bars;
  uint64_t* empty = bars + kMaxStages;
  uint64_t* tfull = bars + 2 * kMaxStages;
  uint64_t* tempty = bars + 2 * kMaxStages + 2;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * kMaxStages + 4);
  uint64_t* xfull = bars + 2 * kMaxStages + 5;          // [kMaxStages]: staged A box transformed (kXform)

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int csize = kXform ? 1 : static_cast<int>(cluster_nctarank());      // 1, or 2: CTA pair
  const int crank = kXform ? 0 : static_cast<int>(cluster_ctarank());
  const int m_tiles = p.tiles_w * p.tiles_h * p.tiles_t * p.tiles_n;
  const int total_tiles = ((m_tiles + csize - 1) / csize) * p.n_ntiles * p.n_classes;
  const int tile0 = static_cast<int>(blockIdx.x) / csize, tile_step = static_cast<int>(gridDim.x) / csize;

  if (warp == 0 && lane == 0) {
    for (int i = 0; i < CSTP_MAX_AMAPS; ++i) tma_prefetch_desc(&p.amap[i]);
    tma_prefetch_desc(&p.bmap);
  }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < p.stages; ++s) {
      mbar_init(&full[s], 1);
      mbar_init(&empty[s], static_cast<uint32_t>(csize));        // released by the MMA commits of every CTA of the pair
      if constexpr (kXform) mbar_init(&xfull[s], kConvXformThreads / 32);
    }
    for (int a = 0; a < 2; ++a) {
      mbar_init(&tfull[a], 1);
      mbar_init(&tempty[a], 4);
    }
    fence_mbar_init();
  }
  if (warp == 2) {
    tmem_alloc(tmem_slot, static_cast<uint32_t>(p.tmem_cols));
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  if constexpr (!kXform) cluster_sync_all();      // the peer's mbarriers exist before anything is multicast to them
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  // Roles run warp-converged with one elected issuing lane (see conv_halo.cu: a single-lane branch makes every
  // UTCHMMA pay an ELECT / R2UR round trip).
  if (warp == 0) {
    // ------------------------------------------------------------ TMA producer
    const bool leader = elect_one();
    int stage = 0;
    uint32_t phase = 0;
    for (int tile = tile0; tile < total_tiles; tile += tile_step) {
      const TileCoord tc = decode_tile(p, tile, csize, crank);
      const int tap0 = p.cls_first_tap[tc.cls], tap1 = tap0 + p.cls_n_taps[tc.cls];
      for (int t = tap0; t < tap1; ++t) {
        const cstp_tap tap = p.taps[t];
        for (int c = 0; c < p.chunks_per_tap; ++c) {
          mbar_wait(&empty[stage], phase ^ 1u);
          if (leader) {
            uint8_t* sa = smem + static_cast<size_t>(stage) * stage_bytes;
            mbar_expect_tx(&full[stage], kABytes + p.b_bytes);
            tma_load_5d(sa, &p.amap[tap.map_id], &full[stage], c * 64, tc.w0 + tap.dw, tc.h0 + tap.dh, tc.t0 + tap.dt,
                        tc.n0);
            if (csize == 1) {
              tma_load_2d(sa + kABytes, &p.bmap, &full[stage], tap.k_off + c * 64, tc.ntile * p.n_tile);
            } else {          // my half of the weight tile, into both CTAs (the peer sends the other half)
              tma_load_2d_mc(sa + kABytes + static_cast<uint32_t>(crank) * (p.b_bytes >> 1), &p.bmap_half, &full[stage],
                             tap.k_off + c * 64, tc.ntile * p.n_tile + crank * (p.n_tile >> 1), 0x3);
            }
          }
          __syncwarp();
          if (++stage == p.stages) {
            stage = 0;
            phase ^= 1u;
          }
        }
      }
    }
  } else if (warp == 1) {
    // ------------------------------------------------------------ MMA issuer
    const bool leader = elect_one();
    int stage = 0;
    uint32_t phase = 0;
    int it = 0;
    // loop-invariant parameters live in registers and the MMAs are issued without a compiler memory clobber (see
    // conv_halo.cu: otherwise every UTCHMMA waits for a fresh LDCU of the kernel parameters)
    const int chunks_per_tap = p.chunks_per_tap, last_ksteps = p.last_ksteps, stages = p.stages;
    const int n_tile = p.n_tile, n_classes = p.n_classes;
    uint32_t idesc;
    asm volatile("mov.u32 %0, %1;" : "=r"(idesc) : "r"(p.idesc));
    const uint32_t smem_addr0 = smem_u32(smem);
    const uint64_t dhi = umma_desc_hi(16, 1024);
    for (int tile = tile0; tile < total_tiles; tile += tile_step, ++it) {
      const int as = it & 1;
      const uint32_t aphase = (it >> 1) & 1;
      mbar_wait(&tempty[as], aphase ^ 1u);
      tc_fence_after();
      const uint32_t d_tmem = tmem_base + static_cast<uint32_t>(as * n_tile);
      const int n_taps = p.cls_n_taps[tile_class(n_classes, tile)];
      const int kblocks = n_taps * chunks_per_tap;
      int kb = 0;
      for (int t = 0; t < n_taps; ++t) {
        for (int c = 0; c < chunks_per_tap; ++c, ++kb) {
          mbar_wait(kXform ? &xfull[stage] : &full[stage], phase);
          tc_fence_after();
          if (leader) {
            const uint32_t a_addr = smem_addr0 + static_cast<uint32_t>(stage) * stage_bytes;
            const uint64_t da = umma_desc_at(dhi, a_addr);
            const uint64_t db = umma_desc_at(dhi, a_addr + kABytes);
            umma_bf16_nc(d_tmem, da, db, idesc, kb != 0 ? 1u : 0u);
            if (c != chunks_per_tap - 1 || last_ksteps == 4) {
              umma_bf16_acc_nc(d_tmem, da + 2, db + 2, idesc);
              umma_bf16_acc_nc(d_tmem, da + 4, db + 4, idesc);
              umma_bf16_acc_nc(d_tmem, da + 6, db + 6, idesc);
            } else {
              for (int k = 1; k < last_ksteps; ++k) umma_bf16_acc_nc(d_tmem, da + 2 * k, db + 2 * k, idesc);
            }
            if (csize == 1) umma_commit(&empty[stage]);
            else umma_commit_mc(&empty[stage], 0x3);
            if (kb == kblocks - 1) umma_commit(&tfull[as]);
          }
          __syncwarp();
          if (++stage == stages) {
            stage = 0;
            phase ^= 1u;
          }
        }
      }
    }
  } else if (kXform && warp >= 8) {
    // ------------------------------------------------------------ operand prologue: BatchNorm affine + ReLU in place
    // Thread t owns the 16-byte units t, t + 256, ... of every staged A box (one swizzle phase = one 8-channel vector of
    // the chunk; coefficients from a table built once in shared memory).  Box rows run (w, h, t, n): the rows of samples
    // below Nt / 2 take the coefficients of statistics group 0, the others those of group 1.
    const uint32_t tid = threadIdx.x - kConvThreads;
    const uint32_t smem_addr0 = smem_u32(smem);
    const int chunks_per_tap = p.chunks_per_tap, stages = p.stages;
    float* xtab = reinterpret_cast<float*>(reinterpret_cast<uint8_t*>(bars) + 256);
    xform_table_fill<kConvXformThreads>(xtab, p.pro_scale, p.pro_shift, p.pro_groups, p.pro_cp, tid);
    xform_bar_sync<kConvXformThreads>();
    const uint32_t xtab_addr = smem_u32(xtab);
    const int rows_per_n = p.bw * p.bh * p.bt;
    constexpr uint32_t kUnits = kABytes / 16;
    int stage = 0;
    uint32_t phase = 0;
    for (int tile = tile0; tile < total_tiles; tile += tile_step) {
      const TileCoord tc = decode_tile(p, tile, csize, crank);
      uint32_t split = kUnits;                     // units below `split` belong to group 0
      if (p.pro_groups == 2) {
        const int rb = (p.Nt / 2 - tc.n0) * rows_per_n;
        split = rb <= 0 ? 0u : (rb >= 128 ? kUnits : static_cast<uint32_t>(rb) * 8u);
      }
      const int n_taps = p.cls_n_taps[tc.cls];
      for (int t = 0; t < n_taps; ++t) {
        for (int c = 0; c < chunks_per_tap; ++c) {
          const uint32_t s_addr = smem_addr0 + static_cast<uint32_t>(stage) * stage_bytes;
          const int cj = xform_unit_channel(s_addr + tid * 16u, 7u);
          XformCoef k0, k1;
          if (split > 0) xform_load_smem(k0, xtab_addr, chunks_per_tap, 0, c, cj);
          if (split < kUnits) xform_load_smem(k1, xtab_addr, chunks_per_tap, 1, c, cj);
          mbar_wait(&full[stage], phase);
          if (split > 0) xform_span<kConvXformThreads>(s_addr, tid, split, k0);
          if (split < kUnits) xform_span<kConvXformThreads>(s_addr, xform_first<kConvXformThreads>(split, tid), kUnits, k1);
          fence_proxy_async();
          __syncwarp();
          if (lane == 0) mbar_arrive(&xfull[stage]);
          if (++stage == stages) {
            stage = 0;
            phase ^= 1u;
          }
        }
      }
    }
  } else if (warp >= 4 && warp < 8) {
    // ------------------------------------------------------------ epilogue (warp w owns TMEM lanes 32*(w%4)..)
    const int q = warp - 4;
    const int row = q * 32 + lane;
    const int rw = row % p.bw;
    const int rh = (row / p.bw) % p.bh;
    const int rt = (row / (p.bw * p.bh)) % p.bt;
    const int rn = row / (p.bw * p.bh * p.bt);
    int it = 0;
    for (int tile = tile0; tile < total_tiles; tile += tile_step, ++it) {
      const int as = it & 1;
      const uint32_t aphase = (it >> 1) & 1;
      const TileCoord tc = decode_tile(p, tile, csize, crank);
      const int w = tc.w0 + rw, h = tc.h0 + rh, t = tc.t0 + rt, n = tc.n0 + rn;
      const bool valid = (w < p.Wt) && (h < p.Ht) && (t < p.Tt) && (n < p.Nt);
      const int col0 = tc.ntile * p.n_tile;
      const int ncols = min(p.n_tile, p.Np - col0);
      const long long off = p.cls_out_off[tc.cls] + w * p.osw + h * p.osh + t * p.ost + n * p.osn + col0;
      mbar_wait(&tfull[as], aphase);
      tc_fence_after();
      const uint32_t taddr = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + static_cast<uint32_t>(as * p.n_tile);
      if (p.fast_store) {        // plain bf16 output: pipelined TMEM loads, one 32-byte store per 16 columns (ptx.cuh)
        if (p.accumulate) epilogue_row_bf16<true>(taddr, ncols, p.out + off, valid);
        else epilogue_row_bf16<false>(taddr, ncols, p.out + off, valid);
      } else
      for (int c0 = 0; c0 < ncols; c0 += 16) {
        uint32_t v[16];
        tmem_ld16(taddr + c0, v);
        tmem_ld_wait();
        if (valid) {
          float f[16];
#pragma unroll
          for (int i = 0; i < 16; ++i) f[i] = __uint_as_float(v[i]);
          if (p.bias != nullptr) {
#pragma unroll
            for (int i = 0; i < 16; ++i) f[i] += __ldg(p.bias + col0 + c0 + i);
          }
          if (p.out != nullptr) {
            uint4* dst = reinterpret_cast<uint4*>(p.out + off + c0);
            if (p.accumulate) {
              const uint4 o0 = dst[0], o1 = dst[1];
              const uint32_t o[8] = {o0.x, o0.y, o0.z, o0.w, o1.x, o1.y, o1.z, o1.w};
#pragma unroll
              for (int i = 0; i < 8; ++i) {
                f[2 * i] += bf16_lo(o[i]);
                f[2 * i + 1] += bf16_hi(o[i]);
              }
            }
            uint4 s0, s1;
            s0.x = pack_bf16x2(f[0], f[1]);
            s0.y = pack_bf16x2(f[2], f[3]);
            s0.z = pack_bf16x2(f[4], f[5]);
            s0.w = pack_bf16x2(f[6], f[7]);
            s1.x = pack_bf16x2(f[8], f[9]);
            s1.y = pack_bf16x2(f[10], f[11]);
            s1.z = pack_bf16x2(f[12], f[13]);
            s1.w = pack_bf16x2(f[14], f[15]);
            dst[0] = s0;
            dst[1] = s1;
          }
          if (p.out_f32 != nullptr) {
            float4* dstf = reinterpret_cast<float4*>(p.out_f32 + off + c0);
            if (p.accumulate && p.out == nullptr) {
#pragma unroll
              for (int i = 0; i < 4; ++i) {
                const float4 o = dstf[i];
                f[4 * i] += o.x;
                f[4 * i + 1] += o.y;
                f[4 * i + 2] += o.z;
                f[4 * i + 3] += o.w;
              }
            }
#pragma unroll
            for (int i = 0; i < 4; ++i) dstf[i] = make_float4(f[4 * i], f[4 * i + 1], f[4 * i + 2], f[4 * i + 3]);
          }
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&tempty[as]);
    }
  }

  tc_fence_before();
  __syncthreads();
  if constexpr (!kXform) cluster_sync_all();      // no CTA leaves while its peer may still signal its mbarriers
  if (warp == 2) {
    tc_fence_after();
    tmem_dealloc(tmem_base, static_cast<uint32_t>(p.tmem_cols));
  }
}

}  // namespace cstp

struct cstp_conv_plan {
  cstp::ConvKParams kp;
  int grid;
  int smem_bytes;
  int cluster;      // CTAs per cluster: 1, or 2 (grid is then even)
};

using namespace cstp;

static int encode_tensor5(CUtensorMap* map, const cstp_tensor5& t, const uint32_t box[5], bool oob_nan = false) {
  uint64_t dims[5], strides[4];
  for (int i = 0; i < 5; ++i) {
    if (t.dims[i] <= 0) return fail_inval("tensor5 dim <= 0");
    dims[i] = static_cast<uint64_t>(t.dims[i]);
  }
  for (int i = 0; i < 4; ++i) {
    if (t.strides[i] <= 0 || (t.strides[i] % 16) != 0) return fail_inval("tensor5 stride must be a positive multiple of 16 bytes");
    strides[i] = static_cast<uint64_t>(t.strides[i]);
  }
  if ((reinterpret_cast<uintptr_t>(t.ptr) % 16) != 0 || t.ptr == nullptr) return fail_inval("tensor5 ptr must be 16B aligned");
  return encode_tmap_bf16(map, t.ptr, 5, dims, strides, box, 128, oob_nan);
}

extern "C" int cstp_conv_plan_create(const cstp_conv_desc* d, cstp_conv_plan** out_plan) {
  CSTP_REQUIRE(d != nullptr && out_plan != nullptr);
  CSTP_REQUIRE(d->n_amaps >= 1 && d->n_amaps <= CSTP_MAX_AMAPS);
  CSTP_REQUIRE(d->n_taps >= 1 && d->n_taps <= CSTP_MAX_TAPS);
  CSTP_REQUIRE(d->a_channels >= 16 && d->a_channels % 16 == 0);
  CSTP_REQUIRE(d->Np >= 16 && d->Np % 16 == 0);
  CSTP_REQUIRE(d->n_tile >= 16 && d->n_tile % 16 == 0 && d->n_tile <= 256);
  CSTP_REQUIRE(d->Ktot >= 64 && d->Ktot % 64 == 0);
  CSTP_REQUIRE(d->bw >= 1 && d->bh >= 1 && d->bt >= 1 && d->bn >= 1);
  CSTP_REQUIRE(d->bw * d->bh * d->bt * d->bn == 128);
  CSTP_REQUIRE(d->bw <= 256 && d->bh <= 256 && d->bt <= 256 && d->bn <= 256);
  CSTP_REQUIRE(d->Wt >= 1 && d->Ht >= 1 && d->Tt >= 1 && d->Nt >= 1);
  CSTP_REQUIRE(d->w_packed != nullptr);
  CSTP_REQUIRE(d->out_bf16 != nullptr || d->out_f32 != nullptr);
  CSTP_REQUIRE(d->osw % 8 == 0 && d->osh % 8 == 0 && d->ost % 8 == 0 && d->osn % 8 == 0 && d->out_off % 8 == 0);
  const int n_classes = d->n_classes > 1 ? d->n_classes : 1;
  CSTP_REQUIRE(n_classes <= 8);
  if (n_classes > 1) {
    int covered = 0;
    for (int c = 0; c < n_classes; ++c) {
      CSTP_REQUIRE(d->cls_first_tap[c] == covered && d->cls_n_taps[c] >= 1 && d->cls_out_off[c] % 8 == 0);
      covered += d->cls_n_taps[c];
    }
    CSTP_REQUIRE(covered == d->n_taps);
  }
  const bool xform = d->pro.scale != nullptr;
  if (xform) {
    CSTP_REQUIRE(d->pro.shift != nullptr && (d->pro.groups == 1 || d->pro.groups == 2) && d->Nt % d->pro.groups == 0);
    CSTP_REQUIRE(d->pro.Cp == d->a_channels);
    CSTP_REQUIRE(reinterpret_cast<uintptr_t>(d->pro.scale) % 16 == 0 && reinterpret_cast<uintptr_t>(d->pro.shift) % 16 == 0);
  }

  cstp_conv_plan* plan = new (std::nothrow) cstp_conv_plan();
  if (!plan) {
    set_error("out of host memory");
    return CSTP_ENOMEM;
  }
  ConvKParams& k = plan->kp;
  memset(&k, 0, sizeof(k));
  const uint32_t abox[5] = {64u, (uint32_t)d->bw, (uint32_t)d->bh, (uint32_t)d->bt, (uint32_t)d->bn};
  for (int i = 0; i < CSTP_MAX_AMAPS; ++i) {
    // Unused slots alias map 0 so the descriptor prefetch in the kernel always sees a valid descriptor.
    const cstp_tensor5& t = d->amap[i < d->n_amaps ? i : 0];
    int rc = encode_tensor5(&k.amap[i], t, abox, xform);
    if (rc != CSTP_OK) {
      delete plan;
      return rc;
    }
  }
  {
    const uint64_t dims[2] = {(uint64_t)d->Ktot, (uint64_t)d->Np};
    const uint64_t strides[1] = {(uint64_t)d->Ktot * 2};
    const uint32_t box[2] = {64u, (uint32_t)d->n_tile};
    int rc = encode_tmap_bf16(&k.bmap, d->w_packed, 2, dims, strides, box);
    if (rc == CSTP_OK) {
      const uint32_t half[2] = {64u, (uint32_t)(d->n_tile / 2 >= 8 ? d->n_tile / 2 : 8)};
      rc = encode_tmap_bf16(&k.bmap_half, d->w_packed, 2, dims, strides, half);
    }
    if (rc != CSTP_OK) {
      delete plan;
      return rc;
    }
  }
  k.tiles_w = ceil_div(d->Wt, d->bw);
  k.tiles_h = ceil_div(d->Ht, d->bh);
  k.tiles_t = ceil_div(d->Tt, d->bt);
  k.tiles_n = ceil_div(d->Nt, d->bn);
  k.n_ntiles = ceil_div(d->Np, d->n_tile);
  k.bw = d->bw; k.bh = d->bh; k.bt = d->bt; k.bn = d->bn;
  k.Wt = d->Wt; k.Ht = d->Ht; k.Tt = d->Tt; k.Nt = d->Nt;
  k.n_taps = d->n_taps;
  k.chunks_per_tap = ceil_div(d->a_channels, 64);
  k.last_ksteps = ((d->a_channels - 1) % 64) / 16 + 1;
  k.n_tile = d->n_tile;
  k.Np = d->Np;
  k.b_bytes = static_cast<uint32_t>(d->n_tile) * 128u;
  k.idesc = umma_idesc_bf16(128, static_cast<uint32_t>(d->n_tile), 0, 0);
  k.accumulate = d->accumulate;
  k.out = reinterpret_cast<__nv_bfloat16*>(d->out_bf16);
  k.out_f32 = d->out_f32;
  k.bias = d->bias;
  k.out_off = d->out_off; k.osw = d->osw; k.osh = d->osh; k.ost = d->ost; k.osn = d->osn;
  k.n_classes = n_classes;
  bool offs16 = true;
  for (int c = 0; c < n_classes; ++c) {
    k.cls_first_tap[c] = n_classes > 1 ? d->cls_first_tap[c] : 0;
    k.cls_n_taps[c] = n_classes > 1 ? d->cls_n_taps[c] : d->n_taps;
    k.cls_out_off[c] = n_classes > 1 ? d->cls_out_off[c] : d->out_off;
    offs16 = offs16 && k.cls_out_off[c] % 16 == 0;
  }
  k.fast_store = d->out_bf16 != nullptr && d->out_f32 == nullptr && d->bias == nullptr &&
                 reinterpret_cast<uintptr_t>(d->out_bf16) % 32 == 0 && offs16 && d->osw % 16 == 0 &&
                 d->osh % 16 == 0 && d->ost % 16 == 0 && d->osn % 16 == 0 && d->n_tile % 16 == 0;
  k.pro_scale = d->pro.scale;
  k.pro_shift = d->pro.shift;
  k.pro_groups = d->pro.groups;
  k.pro_cp = d->pro.Cp;
  for (int t = 0; t < d->n_taps; ++t) {
    const cstp_tap& tp = d->taps[t];
    if (tp.map_id < 0 || tp.map_id >= d->n_amaps || tp.k_off < 0 || tp.k_off % 64 != 0 ||
        tp.k_off + k.chunks_per_tap * 64 > d->Ktot) {
      delete plan;
      return fail_inval("tap map_id / k_off out of range");
    }
    k.taps[t] = tp;
  }
  const uint32_t stage_bytes = kABytes + k.b_bytes;
  const int bar_bytes = 256;       // 5 + 3 * kMaxStages mbarriers + the TMEM slot
  const int xtab_bytes = xform ? static_cast<int>(xform_table_bytes(d->pro.groups, d->pro.Cp)) : 0;      // prologue coefficient table
  int stages = (kSmemBudget - 1024 - bar_bytes - xtab_bytes) / static_cast<int>(stage_bytes);
  if (stages > kMaxStages) stages = kMaxStages;
  if (stages < 2) {
    delete plan;
    return fail_inval("n_tile too large for the shared-memory pipeline");
  }
  k.stages = stages;
  int cols = 32;
  while (cols < 2 * d->n_tile) cols *= 2;
  k.tmem_cols = cols;
  plan->smem_bytes = 1024 + stages * static_cast<int>(stage_bytes) + bar_bytes + xtab_bytes;
  if (plan->smem_bytes < 120 * 1024) plan->smem_bytes = 120 * 1024;  // keep one CTA per SM (TMEM ownership)
  const long long m_tiles = 1LL * k.tiles_w * k.tiles_h * k.tiles_t * k.tiles_n;
  const long long total = m_tiles * k.n_ntiles * n_classes;
  const int sms = num_sms();
  plan->grid = static_cast<int>(total < sms ? total : sms);
  plan->cluster = 1;
  // CTA pairs when the persistent grid is full anyway (deep layers: many tiles, weight tiles of 16-32 KB per K-block)
  if (!xform && total >= 2LL * sms && m_tiles >= 2 && d->n_tile % 16 == 0 && d->n_tile >= 32) {
    static int max_pairs = -1;        // co-resident clusters of two with this kernel's footprint (one CTA per SM)
    if (max_pairs < 0) {
      max_pairs = 0;
      cudaLaunchConfig_t cfg = {};
      cfg.gridDim = dim3(static_cast<unsigned>(sms & ~1), 1, 1);
      cfg.blockDim = dim3(kConvThreads, 1, 1);
      cfg.dynamicSmemBytes = kSmemLimit;
      cudaLaunchAttribute at[1];
      at[0].id = cudaLaunchAttributeClusterDimension;
      at[0].val.clusterDim.x = 2;
      at[0].val.clusterDim.y = 1;
      at[0].val.clusterDim.z = 1;
      cfg.attrs = at;
      cfg.numAttrs = 1;
      int n = 0;
      if (cudaFuncSetAttribute(conv_gemm_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemLimit) == cudaSuccess &&
          cudaOccupancyMaxActiveClusters(&n, conv_gemm_kernel<false>, &cfg) == cudaSuccess)
        max_pairs = n;
      else
        (void)cudaGetLastError();
    }
    const long long pair_tiles = ((m_tiles + 1) / 2) * k.n_ntiles * n_classes;
    long long pairs = max_pairs < pair_tiles ? max_pairs : pair_tiles;
    if (pairs >= (sms * 9) / 20) {        // (a machine that cannot hold ~all SMs in pairs keeps single CTAs)
      plan->cluster = 2;
      plan->grid = static_cast<int>(2 * pairs);
    }
  }
  *out_plan = plan;
  return CSTP_OK;
}

extern "C" int cstp_conv_plan_cluster(const cstp_conv_plan* plan) { return plan ? plan->cluster : CSTP_EINVAL; }

extern "C" int cstp_conv_plan_run(const cstp_conv_plan* plan, void* stream) {
  CSTP_REQUIRE(plan != nullptr);
  static bool attr_set = false;
  if (!attr_set) {
    CSTP_CUDA(cudaFuncSetAttribute(conv_gemm_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemLimit));
    CSTP_CUDA(cudaFuncSetAttribute(conv_gemm_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemLimit));
    attr_set = true;
  }
  if (plan->kp.pro_scale != nullptr)
    conv_gemm_kernel<true><<<plan->grid, kConvThreads + kConvXformThreads, plan->smem_bytes, static_cast<cudaStream_t>(stream)>>>(plan->kp);
  else if (plan->cluster > 1) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(static_cast<unsigned>(plan->grid), 1, 1);
    cfg.blockDim = dim3(kConvThreads, 1, 1);
    cfg.dynamicSmemBytes = static_cast<size_t>(plan->smem_bytes);
    cfg.stream = static_cast<cudaStream_t>(stream);
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = static_cast<unsigned>(plan->cluster);
    at[0].val.clusterDim.y = 1;
    at[0].val.clusterDim.z = 1;
    cfg.attrs = at;
    cfg.numAttrs = 1;
    CSTP_CUDA(cudaLaunchKernelEx(&cfg, conv_gemm_kernel<false>, plan->kp));
  } else
    conv_gemm_kernel<false><<<plan->grid, kConvThreads, plan->smem_bytes, static_cast<cudaStream_t>(stream)>>>(plan->kp);
  CSTP_LAUNCHED();
  return CSTP_OK;
}

extern "C" void cstp_conv_plan_destroy(cstp_conv_plan* plan) { delete plan; }

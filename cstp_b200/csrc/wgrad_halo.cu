// Weight-gradient GEMM for the wide, shallow layers (stride-1 1x3x3 / 3x1x1 convs of conv1..conv3): every CTA computes
// ALL taps of dW for its slice of the position (K) axis.
//
//   P[split][chunk*64 + r][n] = sum_{pos in split} X[pos + tap(chunk), c_off(chunk) + r] * G[pos, n]
//
// wgrad.cu gives every (tap, 64-channel chunk) pair of X its own CTA column, so the same activations are fetched once
// per tap and G once per M tile: those layers (K = 6M positions, 64..144 channels) ran at 150-380 TFLOP/s, bound by the
// L2->SM feed.  Here one K-block of 64 positions is staged ONCE: X as a box with a halo along the tap axis (the taps
// of that axis are the same shared-memory rows, shifted by a multiple of 8 rows, i.e. whole 128B-swizzle atoms), G as
// plain boxes; the tcgen05 issuer then runs one 128 x n_tile MMA per pair of (tap, chunk) row blocks into its own
// TMEM accumulator (n_mtiles * n_tile <= 512 columns).  Taps along the fastest axis (kw) cannot be expressed as an
// aligned row shift and are staged as separately shifted boxes ("groups").
//
// Round 2: (a) M CLASSES.  When all M tiles at the full N width do not fit TMEM (5 x 144 columns for the 64 -> 144 1x3x3
// layers) the N axis used to be cut in two (96 + 48 columns): narrow MMAs re-read their 4 KB A slice from shared memory
// per 24-48 tensor cycles, and the kernel sat at 62 % tensor-pipe activity bound by shared-memory bandwidth.  Now the M
// tiles are dealt to CTA classes (3 + 2 tiles, every MMA 144 columns wide = 119 B/clk of shared-memory reads) and the
// split-K CTAs are shared out in proportion to the work of a class.  (b) Either operand may carry the taps: the host may
// hand G in as the "x" tensor (halo + row-shifted chunks) and X as the "g" tensor, which puts (tap, cout) on M and the wide
// cin on N for the 144 -> 64 3x1x1 layers (N = 64 MMAs want 192 B/clk); pro_on_b then moves the operand prologue to the
// N-side boxes.
// Replaces cuDNN conv3d wgrad behind main_byol.py:87 for models/pace/r21d_byol.py:81-92 layers with stride 1.
#include "common.h"
#include "ptx.cuh"

namespace cstp {

constexpr int kWhThreads = 256;
constexpr int kWhXformThreads = 256;   // warps 8..15: operand prologue (BatchNorm affine + ReLU on the staged boxes)
constexpr int kWhMaxStages = 8;
constexpr int kWhSmemLimit = 232448;
constexpr int kWhMaxMtiles = 16;
constexpr int kWhMaxBoxes = 16;      // (group, channel chunk) X boxes per stage
constexpr uint32_t kGBoxBytes = 64 * 64 * 2;
constexpr int kWhMaxClasses = 8;     // CTA classes along M (each owns mt_per_class accumulators of n_tile columns)

struct WhXBox {
  int c_off, dw, dh, dt;  // channel offset and tile-origin offset of this staged box
};
struct WhMtile {
  uint32_t a_off;  // byte offset (inside a stage) of the first 64-row block
  uint32_t lbo;    // byte distance to the second 64-row block (== 0: single block, upper 64 lanes unused)
};

struct WgradHaloKParams {
  CUtensorMap xmap;
  CUtensorMap gmap;
  int tiles_w, tiles_h, tiles_t, tiles_n;
  int bw, bh, bt, bn;
  int Wt, Ht, Tt;
  int box_w, box_h, box_t;   // extents of a staged M-side box, halo included
  int a_w, a_h, a_t;         // extents of the M-side tensor
  int n_xboxes, n_mtiles, n_chunks, Np, n_tile, n_gboxes;
  int total_kblocks;
  int n_ntiles, mt_per_class, n_mclasses, pro_on_b;
  int class_splits[kWhMaxClasses], class_kps[kWhMaxClasses];   // split-K CTAs and K-blocks per CTA of every M class
  int stages, tmem_cols;
  uint32_t xbox_bytes, stage_bytes, idesc;
  uint32_t x_tx_bytes;     // bytes the X boxes of one stage really carry (xbox_bytes is their 1024-aligned pitch)
  uint32_t a_sbo;          // bytes between consecutive 8-position atoms of a chunk inside its staged box
  uint32_t a_kstep;        // descriptor start-address advance (>> 4) per 16-position K step: two atoms
  float* partials;
  const float* pro_scale;  // operand prologue (kXform): fp32 [pro_groups][pro_cp] BatchNorm affine of the producer of X
  const float* pro_shift;
  int pro_groups, pro_cp, Nt;
  uint32_t xbox_units;     // 16-byte units one staged X box really carries
  WhXBox xboxes[kWhMaxBoxes];
  WhMtile mtiles[kWhMaxMtiles];
};

template <bool kXform>
__global__ void __launch_bounds__(kXform ? kWhThreads + kWhXformThreads : kWhThreads, 1) wgrad_halo_kernel(const __grid_constant__ WgradHaloKParams p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + static_cast<size_t>(p.stages) * p.stage_bytes);
  uint64_t* full = bars;
  uint64_t* empty = bars + kWhMaxStages;
  uint64_t* tfull = bars + 2 * kWhMaxStages;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * kWhMaxStages + 1);
  uint64_t* xfull = bars + 2 * kWhMaxStages + 2;        // [kWhMaxStages]: staged X boxes transformed (kXform)

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int ntile = blockIdx.x % p.n_ntiles, mclass = blockIdx.x / p.n_ntiles, split = blockIdx.y;
  if (split >= p.class_splits[mclass]) return;          // classes with less work own fewer split-K CTAs
  const int mt0 = mclass * p.mt_per_class;
  const int nmt = min(p.n_mtiles - mt0, p.mt_per_class);
  const int kb_begin = split * p.class_kps[mclass];
  const int kb_end = min(p.total_kblocks, kb_begin + p.class_kps[mclass]);
  const uint32_t x_bytes = static_cast<uint32_t>(p.n_xboxes) * p.xbox_bytes;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&p.xmap);
    tma_prefetch_desc(&p.gmap);
  }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < p.stages; ++s) {
      mbar_init(&full[s], 1);
      mbar_init(&empty[s], 1);
      if constexpr (kXform) mbar_init(&xfull[s], kWhXformThreads / 32);
    }
    mbar_init(tfull, 1);
    fence_mbar_init();
  }
  if (warp == 2) {
    tmem_alloc(tmem_slot, static_cast<uint32_t>(p.tmem_cols));
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (kXform && warp >= 8) {
    // ------------------------------------------------------------ operand prologue: BatchNorm affine + ReLU on X in place
    // Thread t owns the 16-byte units t, t + 256, ... of every staged X box (one swizzle phase = one 8-channel vector of
    // the box's chunk; coefficients from a table built once in shared memory); one K-block is one sample (bn == 1),
    // hence one statistics group.
    const uint32_t tid = threadIdx.x - kWhThreads;
    const uint32_t smem_addr0 = smem_u32(smem);
    const int slab = p.tiles_w * p.tiles_h * p.tiles_t, stages = p.stages;
    // the boxes to transform: the staged A-side boxes, or (pro_on_b) the 64-channel boxes of this CTA's N tile
    const bool on_b = p.pro_on_b != 0;
    const int n_boxes = on_b ? p.n_gboxes : p.n_xboxes;
    const uint32_t box0 = on_b ? x_bytes : 0u, box_pitch = on_b ? kGBoxBytes : p.xbox_bytes;
    const uint32_t box_units = on_b ? kGBoxBytes / 16u : p.xbox_units;
    const int chunk0 = on_b ? (ntile * p.n_tile) >> 6 : 0;
    const int tchunks = (p.pro_cp + 63) / 64;
    float* xtab = reinterpret_cast<float*>(reinterpret_cast<uint8_t*>(bars) + 256);
    xform_table_fill<kWhXformThreads>(xtab, p.pro_scale, p.pro_shift, p.pro_groups, p.pro_cp, tid);
    xform_bar_sync<kWhXformThreads>();
    const uint32_t xtab_addr = smem_u32(xtab);
    // stages and boxes are 1024-byte aligned: a thread's swizzle phase, hence its 8-channel vector, never changes
    const int cj = xform_unit_channel(smem_addr0 + tid * 16u, 7u);
    // Up to three boxes of at most two units per thread (the N-side boxes of the flipped form): the coefficients of the
    // thread's vector in every box stay in registers (reloaded when the statistics group changes, once per launch) and the
    // loads of a box are issued before the previous box is finished.  Measured (tools/prologue_probe.py): the
    // cost of the prologue is the arithmetic of the transform warps (ALU pipe), not the proxy fence or the second barrier
    // hop; sixteen warps instead of eight made it worse.
    const bool small = n_boxes <= 3 && box_units <= 2u * kWhXformThreads;
    const bool two = box_units > static_cast<uint32_t>(kWhXformThreads) && tid + kWhXformThreads < box_units;
    const bool one = tid < box_units;
    // N-side boxes on an exact tiling are never out of range and the MMA never reads channels beyond n_tile: the cheaper
    // ReLU-in-the-conversion form applies (its NaN stays NaN)
    const bool exact = on_b && p.tiles_w * p.bw == p.Wt && p.tiles_h * p.bh == p.Ht && p.tiles_t * p.bt == p.Tt &&
                       p.tiles_n * p.bn == p.Nt;
    XformCoef kc[3];
    int cur_grp = -1;
    int stage = 0;
    uint32_t phase = 0;
    // K-blocks of the second statistics group (bn == 1: K-block kb belongs to sample kb / slab)
    const int kb_grp1 = p.pro_groups == 2 ? ((p.Nt + 1) / 2) * slab : p.total_kblocks;
    for (int kb = kb_begin; kb < kb_end; ++kb) {
      const int grp = kb >= kb_grp1 ? 1 : 0;
      const uint32_t s_addr = smem_addr0 + static_cast<uint32_t>(stage) * p.stage_bytes + box0;
      if (small) {
        if (grp != cur_grp) {
          cur_grp = grp;
#pragma unroll
          for (int b = 0; b < 3; ++b)
            if (b < n_boxes) xform_load_smem(kc[b], xtab_addr, tchunks, grp, on_b ? chunk0 + b : p.xboxes[b].c_off >> 6, cj);
        }
        mbar_wait(&full[stage], phase);
        const uint32_t a0 = s_addr + tid * 16u;
        uint4 v0 = make_uint4(0, 0, 0, 0), v1 = v0;
        if (one) v0 = lds128(a0);
        if (two) v1 = lds128(a0 + kWhXformThreads * 16u);
#pragma unroll
        for (int b = 0; b < 3; ++b) {
          if (b < n_boxes) {
            const uint32_t a = a0 + static_cast<uint32_t>(b) * box_pitch;
            uint4 w0 = v0, w1 = v1;
            if (b + 1 < n_boxes) {             // next box's loads in flight while this one is computed
              if (one) w0 = lds128(a + box_pitch);
              if (two) w1 = lds128(a + box_pitch + kWhXformThreads * 16u);
            }
            if (exact) {
              if (one) sts128(a, xform_unit_relu(v0, kc[b]));
              if (two) sts128(a + kWhXformThreads * 16u, xform_unit_relu(v1, kc[b]));
            } else {
              if (one) sts128(a, xform_unit(v0, kc[b]));
              if (two) sts128(a + kWhXformThreads * 16u, xform_unit(v1, kc[b]));
            }
            v0 = w0;
            v1 = w1;
          }
        }
      } else {
        XformCoef k;
        xform_load_smem(k, xtab_addr, tchunks, grp, on_b ? chunk0 : p.xboxes[0].c_off >> 6, cj);
        int pt = kb;
        const int w0 = (pt % p.tiles_w) * p.bw;
        pt /= p.tiles_w;
        const int h0 = (pt % p.tiles_h) * p.bh;
        const int t0 = ((pt / p.tiles_h) % p.tiles_t) * p.bt;
        mbar_wait(&full[stage], phase);
        for (int b = 0; b < n_boxes; ++b) {
          // a box inside the tensor with a full channel chunk has no NaN fill to turn into zero: cheaper transform
          bool inside = exact;
          if (!on_b) {
            const WhXBox xb = p.xboxes[b];
            const int bw0 = w0 + xb.dw, bh0 = h0 + xb.dh, bt0 = t0 + xb.dt;
            inside = bw0 >= 0 && bw0 + p.box_w <= p.a_w && bh0 >= 0 && bh0 + p.box_h <= p.a_h && bt0 >= 0 &&
                     bt0 + p.box_t <= p.a_t && xb.c_off + 64 <= p.pro_cp;
          }
          if (inside)
            xform_span<kWhXformThreads, true>(s_addr + static_cast<uint32_t>(b) * box_pitch, tid, box_units, k);
          else
            xform_span<kWhXformThreads>(s_addr + static_cast<uint32_t>(b) * box_pitch, tid, box_units, k);
          if (b + 1 < n_boxes) xform_load_smem(k, xtab_addr, tchunks, grp, on_b ? chunk0 + b + 1 : p.xboxes[b + 1].c_off >> 6, cj);
        }
      }
      fence_proxy_async();
      __syncwarp();
      if (lane == 0) mbar_arrive(&xfull[stage]);
      if (++stage == stages) {
        stage = 0;
        phase ^= 1u;
      }
    }
  }

  // Roles run warp-converged with one elected issuing lane (see conv_halo.cu).
  if (warp == 0) {
    // ------------------------------------------------------------ TMA producer
    const bool leader = elect_one();
    int stage = 0;
    uint32_t phase = 0;
    for (int kb = kb_begin; kb < kb_end; ++kb) {
      int pt = kb;
      const int w0 = (pt % p.tiles_w) * p.bw;
      pt /= p.tiles_w;
      const int h0 = (pt % p.tiles_h) * p.bh;
      pt /= p.tiles_h;
      const int t0 = (pt % p.tiles_t) * p.bt;
      pt /= p.tiles_t;
      const int n0 = pt * p.bn;
      mbar_wait(&empty[stage], phase ^ 1u);
      if (leader) {
        uint8_t* st = smem + static_cast<size_t>(stage) * p.stage_bytes;
        mbar_expect_tx(&full[stage], p.x_tx_bytes + static_cast<uint32_t>(p.n_gboxes) * kGBoxBytes);
        for (int b = 0; b < p.n_xboxes; ++b) {
          const WhXBox xb = p.xboxes[b];
          tma_load_5d(st + static_cast<size_t>(b) * p.xbox_bytes, &p.xmap, &full[stage], xb.c_off, w0 + xb.dw, h0 + xb.dh,
                      t0 + xb.dt, n0);
        }
        for (int j = 0; j < p.n_gboxes; ++j)
          tma_load_5d(st + x_bytes + j * kGBoxBytes, &p.gmap, &full[stage], ntile * p.n_tile + j * 64, w0, h0, t0, n0);
      }
      __syncwarp();
      if (++stage == p.stages) {
        stage = 0;
        phase ^= 1u;
      }
    }
  } else if (warp == 1) {
    // ------------------------------------------------------------ MMA issuer: n_mtiles accumulators per K-block
    const bool leader = elect_one();
    const uint32_t smem_addr0 = smem_u32(smem);
    const uint64_t dhi_b = umma_desc_hi(kGBoxBytes, 1024);
    // loop invariants in registers, clobber-free MMA issue (see conv_halo.cu)
    const int stages = p.stages, n_tile = p.n_tile;
    const uint32_t stage_bytes = p.stage_bytes, a_sbo = p.a_sbo;
    const uint64_t k1 = p.a_kstep, k2 = 2ull * p.a_kstep, k3 = 3ull * p.a_kstep;
    uint32_t idesc;
    asm volatile("mov.u32 %0, %1;" : "=r"(idesc) : "r"(p.idesc));
    int stage = 0;
    uint32_t phase = 0;
    for (int kb = kb_begin; kb < kb_end; ++kb) {
      mbar_wait(kXform ? &xfull[stage] : &full[stage], phase);
      tc_fence_after();
      if (leader) {
        const uint32_t s_addr = smem_addr0 + static_cast<uint32_t>(stage) * stage_bytes;
        const uint64_t db = umma_desc_at(dhi_b, s_addr + x_bytes);
        // MN-major, 128B swizzle: 16 K-rows (positions) per step = 2048 B (+128 in the address field); LBO = next
        // 64-channel block of the M (resp. N) axis, SBO = next 8 K-rows.
        const uint32_t acc = kb > kb_begin ? 1u : 0u;
        for (int mt = 0; mt < nmt; ++mt) {
          const WhMtile m = p.mtiles[mt0 + mt];
          const uint64_t da = umma_desc_at(umma_desc_hi(m.lbo != 0 ? m.lbo : 1024u, a_sbo), s_addr + m.a_off);
          const uint32_t d_tmem = tmem_base + static_cast<uint32_t>(mt * n_tile);
          umma_bf16_nc(d_tmem, da, db, idesc, acc);
          umma_bf16_acc_nc(d_tmem, da + k1, db + 128, idesc);
          umma_bf16_acc_nc(d_tmem, da + k2, db + 256, idesc);
          umma_bf16_acc_nc(d_tmem, da + k3, db + 384, idesc);
        }
        umma_commit(&empty[stage]);
        if (kb == kb_end - 1) umma_commit(tfull);
      }
      __syncwarp();
      if (++stage == stages) {
        stage = 0;
        phase ^= 1u;
      }
    }
  } else if (warp >= 4 && warp < 8) {
    // ------------------------------------------------------------ epilogue: TMEM -> fp32 partials
    const int q = warp - 4;
    const int row = q * 32 + lane;
    const int col0 = ntile * p.n_tile;
    const int ncols = min(p.n_tile, p.Np - col0);
    const long long mtot = static_cast<long long>(p.n_chunks) * 64;
    mbar_wait_idle(tfull, 0);
    tc_fence_after();
    for (int mt = 0; mt < nmt; ++mt) {
      const bool valid = ((mt0 + mt) * 2 + (row >> 6)) < p.n_chunks;
      float* dst = p.partials + (static_cast<long long>(split) * mtot + static_cast<long long>(mt0 + mt) * 128 + row) * p.Np + col0;
      const uint32_t taddr = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + static_cast<uint32_t>(mt * p.n_tile);
      epilogue_row_f32(taddr, ncols, dst, valid);     // pipelined TMEM loads, 32-byte stores (ptx.cuh)
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 2) {
    tc_fence_after();
    tmem_dealloc(tmem_base, static_cast<uint32_t>(p.tmem_cols));
  }
}

}  // namespace cstp

struct cstp_wgrad_halo_plan {
  cstp::WgradHaloKParams kp;
  dim3 grid;
  int smem_bytes;
  int splits;                     // the largest split count of a class: rows of the partials buffer
};

using namespace cstp;

static int encode5(CUtensorMap* map, const cstp_tensor5& t, const uint32_t box[5], bool oob_nan = false) {
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

extern "C" int cstp_wgrad_halo_plan_create(const cstp_wgrad_halo_desc* d, cstp_wgrad_halo_plan** out_plan) {
  CSTP_REQUIRE(d != nullptr && out_plan != nullptr);
  CSTP_REQUIRE(d->n_chunks >= 1 && d->n_chunks <= 2 * kWhMaxMtiles);
  CSTP_REQUIRE(d->n_xboxes >= 1 && d->n_xboxes <= kWhMaxBoxes);
  CSTP_REQUIRE(d->Np >= 16 && d->Np % 16 == 0);
  CSTP_REQUIRE(d->n_tile >= 16 && d->n_tile % 16 == 0 && d->n_tile <= 256);
  CSTP_REQUIRE(d->bw >= 1 && d->bh >= 1 && d->bt >= 1 && d->bn >= 1 && d->bw * d->bh * d->bt * d->bn == 64);
  CSTP_REQUIRE(d->halo_w >= 0 && d->halo_h >= 0 && d->halo_t >= 0);
  CSTP_REQUIRE(d->Wt >= 1 && d->Ht >= 1 && d->Tt >= 1 && d->Nt >= 1);
  CSTP_REQUIRE(d->splits >= 1 && d->partials != nullptr && reinterpret_cast<uintptr_t>(d->partials) % 32 == 0);   // 32-byte stores
  const int n_mtiles = (d->n_chunks + 1) / 2;
  const int mt_per_class = d->mt_per_class > 0 && d->mt_per_class < n_mtiles ? d->mt_per_class : n_mtiles;
  const int n_mclasses = ceil_div(n_mtiles, mt_per_class);
  CSTP_REQUIRE(mt_per_class * d->n_tile <= 512 && n_mclasses <= kWhMaxClasses);
  const int xrows = (d->bw + d->halo_w) * (d->bh + d->halo_h) * (d->bt + d->halo_t) * d->bn;
  CSTP_REQUIRE(d->bw + d->halo_w <= 256 && d->bh + d->halo_h <= 256 && d->bt + d->halo_t <= 256);
  // atom pitch: 8 rows when the 64 positions of a chunk are contiguous rows of the staged box; with a halo along w (bw == 8)
  // every run of 8 positions is one atom and consecutive atoms are one box row (bw + halo_w positions) apart
  const int pitch = d->atom_pitch_rows > 0 ? d->atom_pitch_rows : 8;
  CSTP_REQUIRE(d->halo_w == 0 ? (pitch == 8 && xrows % 8 == 0) : (d->bw == 8 && pitch == d->bw + d->halo_w));
  const bool xform = d->pro.scale != nullptr;
  if (xform) {
    CSTP_REQUIRE(d->pro.shift != nullptr && (d->pro.groups == 1 || d->pro.groups == 2) && d->Nt % d->pro.groups == 0);
    CSTP_REQUIRE(d->pro.Cp == (d->pro_on_b ? d->gmap.dims[0] : d->xmap.dims[0]) && d->bn == 1);
    CSTP_REQUIRE(!d->pro_on_b || d->n_tile % 64 == 0 || d->n_tile >= d->Np);       // N-tile origins on 64-channel chunks
    CSTP_REQUIRE(reinterpret_cast<uintptr_t>(d->pro.scale) % 16 == 0 && reinterpret_cast<uintptr_t>(d->pro.shift) % 16 == 0);
  }

  cstp_wgrad_halo_plan* plan = new (std::nothrow) cstp_wgrad_halo_plan();
  if (!plan) {
    set_error("out of host memory");
    return CSTP_ENOMEM;
  }
  WgradHaloKParams& k = plan->kp;
  memset(&k, 0, sizeof(k));
  const uint32_t xbox[5] = {64u, (uint32_t)(d->bw + d->halo_w), (uint32_t)(d->bh + d->halo_h),
                            (uint32_t)(d->bt + d->halo_t), (uint32_t)d->bn};
  const uint32_t gbox[5] = {64u, (uint32_t)d->bw, (uint32_t)d->bh, (uint32_t)d->bt, (uint32_t)d->bn};
  int rc = encode5(&k.xmap, d->xmap, xbox, xform && !d->pro_on_b);
  if (rc == CSTP_OK) rc = encode5(&k.gmap, d->gmap, gbox, xform && d->pro_on_b);
  if (rc != CSTP_OK) {
    delete plan;
    return rc;
  }
  k.tiles_w = ceil_div(d->Wt, d->bw);
  k.tiles_h = ceil_div(d->Ht, d->bh);
  k.tiles_t = ceil_div(d->Tt, d->bt);
  k.tiles_n = ceil_div(d->Nt, d->bn);
  k.bw = d->bw; k.bh = d->bh; k.bt = d->bt; k.bn = d->bn;
  k.n_xboxes = d->n_xboxes;
  k.n_chunks = d->n_chunks;
  k.n_mtiles = n_mtiles;
  k.Np = d->Np;
  k.n_tile = d->n_tile;
  k.n_gboxes = ceil_div(d->n_tile, 64);
  k.xbox_bytes = (static_cast<uint32_t>(xrows) * 128u + 1023u) & ~1023u;
  k.x_tx_bytes = static_cast<uint32_t>(d->n_xboxes) * static_cast<uint32_t>(xrows) * 128u;
  k.a_sbo = static_cast<uint32_t>(pitch) * 128u;
  k.a_kstep = (2u * k.a_sbo) >> 4;
  k.stage_bytes = static_cast<uint32_t>(d->n_xboxes) * k.xbox_bytes + static_cast<uint32_t>(k.n_gboxes) * kGBoxBytes;
  k.total_kblocks = k.tiles_w * k.tiles_h * k.tiles_t * k.tiles_n;
  k.n_ntiles = ceil_div(d->Np, d->n_tile);
  k.mt_per_class = mt_per_class;
  k.n_mclasses = n_mclasses;
  k.pro_on_b = xform && d->pro_on_b;
  // d->splits split-K CTAs per N tile, dealt to the M classes in proportion to their M tiles (at least one each)
  int max_splits = 0, left = d->splits, tiles_left = n_mtiles;
  for (int c = 0; c < n_mclasses; ++c) {
    const int tiles = (c + 1 < n_mclasses) ? mt_per_class : n_mtiles - c * mt_per_class;
    int s = (c + 1 < n_mclasses) ? (d->splits * tiles + n_mtiles / 2) / n_mtiles : left;
    if (s > left - (n_mclasses - 1 - c)) s = left - (n_mclasses - 1 - c);
    if (s < 1) s = 1;
    left -= s;
    tiles_left -= tiles;
    if (s > k.total_kblocks) s = k.total_kblocks;
    k.class_kps[c] = ceil_div(k.total_kblocks, s);
    k.class_splits[c] = ceil_div(k.total_kblocks, k.class_kps[c]);
    if (k.class_splits[c] > max_splits) max_splits = k.class_splits[c];
  }
  (void)tiles_left;
  const int splits = max_splits;
  plan->splits = splits;
  k.idesc = umma_idesc_bf16(128, static_cast<uint32_t>(d->n_tile), 1, 1);
  k.partials = d->partials;
  k.pro_scale = d->pro.scale;
  k.pro_shift = d->pro.shift;
  k.pro_groups = d->pro.groups;
  k.pro_cp = d->pro.Cp;
  k.Nt = d->Nt;
  k.Wt = d->Wt; k.Ht = d->Ht; k.Tt = d->Tt;
  k.box_w = d->bw + d->halo_w; k.box_h = d->bh + d->halo_h; k.box_t = d->bt + d->halo_t;
  k.a_w = d->xmap.dims[1]; k.a_h = d->xmap.dims[2]; k.a_t = d->xmap.dims[3];
  k.xbox_units = static_cast<uint32_t>(xrows) * 8u;
  for (int i = 0; i < d->n_xboxes; ++i) {
    const cstp_xbox& b = d->xboxes[i];
    if (b.c_off < 0 || b.c_off % 8 != 0 || (xform && b.c_off % 64 != 0)) {
      delete plan;
      return fail_inval("xbox c_off");
    }
    k.xboxes[i] = WhXBox{b.c_off, b.dw, b.dh, b.dt};
  }
  // chunk i = 64 rows starting at stage byte offset chunk_off[i] (a row shift of a staged X box); consecutive chunks
  // are paired into one 128-row MMA, so offsets must ascend inside a pair and keep 1024-byte (8-row) alignment.
  const uint32_t x_bytes = static_cast<uint32_t>(d->n_xboxes) * k.xbox_bytes;
  for (int mt = 0; mt < n_mtiles; ++mt) {
    const uint32_t a = d->chunk_off[2 * mt];
    const bool two = 2 * mt + 1 < d->n_chunks;
    const uint32_t b = two ? d->chunk_off[2 * mt + 1] : a;
    const uint32_t align = pitch == 8 ? 1024u : 128u;
    if (a % align != 0 || b % align != 0 || (two && b <= a) || b + 7u * k.a_sbo + 1024u > x_bytes ||
        (b - a) / 16 >= (1u << 14)) {
      delete plan;
      return fail_inval("chunk_off must be atom- (row- with a w halo) aligned, ascending within a pair and inside the staged X boxes");
    }
    k.mtiles[mt] = WhMtile{a, two ? b - a : 0u};
  }
  const int bar_bytes = 256;
  const int xtab_bytes = xform ? static_cast<int>(xform_table_bytes(d->pro.groups, d->pro.Cp)) : 0;      // prologue coefficient table
  int stages = (kSmemBudget - 1024 - bar_bytes - xtab_bytes) / static_cast<int>(k.stage_bytes);
  if (stages > kWhMaxStages) stages = kWhMaxStages;
  if (stages < 2) {
    delete plan;
    return fail_inval("stage too large for the shared-memory pipeline");
  }
  k.stages = stages;
  int cols = 32;
  while (cols < mt_per_class * d->n_tile) cols *= 2;
  k.tmem_cols = cols;
  plan->smem_bytes = 1024 + stages * static_cast<int>(k.stage_bytes) + bar_bytes + xtab_bytes;
  if (plan->smem_bytes < 120 * 1024) plan->smem_bytes = 120 * 1024;   // one CTA per SM (TMEM ownership)
  plan->grid = dim3(static_cast<unsigned>(k.n_ntiles * n_mclasses), static_cast<unsigned>(splits), 1);
  *out_plan = plan;
  return CSTP_OK;
}

extern "C" int cstp_wgrad_halo_plan_splits(const cstp_wgrad_halo_plan* plan) { return plan ? plan->splits : CSTP_EINVAL; }

extern "C" int cstp_wgrad_halo_plan_chunk_splits(const cstp_wgrad_halo_plan* plan, int32_t* out, int n_chunks) {
  CSTP_REQUIRE(plan != nullptr && out != nullptr && n_chunks == plan->kp.n_chunks);
  for (int i = 0; i < n_chunks; ++i) out[i] = plan->kp.class_splits[(i / 2) / plan->kp.mt_per_class];
  return CSTP_OK;
}

extern "C" int cstp_wgrad_halo_plan_run(const cstp_wgrad_halo_plan* plan, void* stream) {
  CSTP_REQUIRE(plan != nullptr);
  static bool attr_set = false;
  if (!attr_set) {
    CSTP_CUDA(cudaFuncSetAttribute(wgrad_halo_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, kWhSmemLimit));
    CSTP_CUDA(cudaFuncSetAttribute(wgrad_halo_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, kWhSmemLimit));
    attr_set = true;
  }
  if (plan->kp.pro_scale != nullptr)
    wgrad_halo_kernel<true><<<plan->grid, kWhThreads + kWhXformThreads, plan->smem_bytes, static_cast<cudaStream_t>(stream)>>>(plan->kp);
  else
    wgrad_halo_kernel<false><<<plan->grid, kWhThreads, plan->smem_bytes, static_cast<cudaStream_t>(stream)>>>(plan->kp);
  CSTP_LAUNCHED();
  return CSTP_OK;
}

extern "C" void cstp_wgrad_halo_plan_destroy(cstp_wgrad_halo_plan* plan) { delete plan; }

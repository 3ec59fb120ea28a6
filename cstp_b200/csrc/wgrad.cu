// Weight-gradient GEMM on tcgen05: P[m, n] = sum_pos X[pos + tap(m), c(m)] * G[pos, n].
//
// Both operands come straight out of NDHWC activations, so both are "MN-major" for the tensor core: the
// reduction (K) axis is the position axis, channels are contiguous.  One K-block is a TMA box of 64 positions;
// the M tile (128 rows) is two 64-channel chunks of X, each with its own tap shift, so that 3x3 / 3x1x1 taps of
// narrow layers (Cin = 64) still fill the 128-row MMA.  A CTA owns up to four such M tiles (mt_per_cta, one TMEM
// accumulator each) that share ONE staged G tile per K-block: the kernel is bound by the L2 -> SM feed of its operands
// (a 128 x 256 tile re-loads 48 KB per 64 positions), and every extra M tile per CTA removes one re-load of G.
// Split-K over position tiles; fp32 partials are reduced in
// fixed order by cstp_wgrad_finalize, which also scatters into the reference (Cout, Cin, kT, kH, kW) layout.
// Replaces cuDNN conv3d wgrad / cuBLAS addmm wgrad behind main_byol.py:87.
#include "common.h"
#include "ptx.cuh"

namespace cstp {

constexpr int kWgThreads = 256;
constexpr int kWgXformThreads = 256;   // warps 8..15: operand prologue (BatchNorm affine + ReLU on the staged X boxes)
constexpr uint32_t kBoxBytes = 64 * 64 * 2;  // 64 positions x 64 channels
constexpr int kWgMaxStages = 8;
constexpr int kWgSmemLimit = 232448;
constexpr int kWgMaxMt = 4;            // M tiles per CTA: n_mt * n_tile <= 512 TMEM columns

struct WgradKParams {
  CUtensorMap amap[CSTP_MAX_AMAPS];
  CUtensorMap gmap;
  int tiles_w, tiles_h, tiles_t, tiles_n;
  int bw, bh, bt, bn;
  int n_mchunks, Np, n_tile, n_gboxes;
  int n_mt;                // M tiles (128 rows = two chunks) per CTA, 1..kWgMaxMt
  int total_kblocks, kblocks_per_split;
  int stages, tmem_cols;
  uint32_t idesc;
  float* partials;
  const float* pro_scale;  // operand prologue (kXform): fp32 [pro_groups][pro_cp] BatchNorm affine of the producer of X
  const float* pro_shift;
  int pro_groups, pro_cp, Nt;
  cstp_mchunk mchunks[CSTP_MAX_MCHUNKS];
};

template <bool kXform>
__global__ void __launch_bounds__(kXform ? kWgThreads + kWgXformThreads : kWgThreads, 1) wgrad_gemm_kernel(const __grid_constant__ WgradKParams p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  const uint32_t a_bytes = 2u * static_cast<uint32_t>(p.n_mt) * kBoxBytes;
  const uint32_t stage_bytes = a_bytes + static_cast<uint32_t>(p.n_gboxes) * kBoxBytes;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + static_cast<size_t>(p.stages) * stage_bytes);
  uint64_t* full = bars;
  uint64_t* empty = bars + kWgMaxStages;
  uint64_t* tfull = bars + 2 * kWgMaxStages;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * kWgMaxStages + 1);
  uint64_t* xfull = bars + 2 * kWgMaxStages + 2;        // [kWgMaxStages]: staged X boxes transformed (kXform)

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int mtile = blockIdx.x, ntile = blockIdx.y, split = blockIdx.z;
  const int chunk0 = mtile * 2 * p.n_mt;
  const int nchunks = min(2 * p.n_mt, p.n_mchunks - chunk0);       // (the prologue variant runs with n_mt == 1)
  const int mts = (nchunks + 1) >> 1;                              // M tiles of this CTA that hold at least one chunk
  const int kb_begin = split * p.kblocks_per_split;
  const int kb_end = min(p.total_kblocks, kb_begin + p.kblocks_per_split);

  if (warp == 0 && lane == 0) {
    for (int i = 0; i < CSTP_MAX_AMAPS; ++i) tma_prefetch_desc(&p.amap[i]);
    tma_prefetch_desc(&p.gmap);
  }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < p.stages; ++s) {
      mbar_init(&full[s], 1);
      mbar_init(&empty[s], 1);
      if constexpr (kXform) mbar_init(&xfull[s], kWgXformThreads / 32);
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
    // Thread t owns the 16-byte units t, t + 256, ... of the (up to) two staged X boxes (coefficients from a table built
    // once in shared memory); box rows run (w, h, t, n): rows of samples below Nt / 2 take the coefficients of statistics
    // group 0, the others those of group 1.
    const uint32_t tid = threadIdx.x - kWgThreads;
    const uint32_t smem_addr0 = smem_u32(smem);
    const int stages = p.stages;
    const int tchunks = (p.pro_cp + 63) / 64;
    float* xtab = reinterpret_cast<float*>(reinterpret_cast<uint8_t*>(bars) + 256);
    xform_table_fill<kWgXformThreads>(xtab, p.pro_scale, p.pro_shift, p.pro_groups, p.pro_cp, tid);
    xform_bar_sync<kWgXformThreads>();
    const uint32_t xtab_addr = smem_u32(xtab);
    const int rows_per_n = p.bw * p.bh * p.bt;
    const int kb_per_n = p.tiles_w * p.tiles_h * p.tiles_t;
    constexpr uint32_t kUnits = kBoxBytes / 16;
    const int c_off[2] = {p.mchunks[chunk0].c_off, p.mchunks[nchunks > 1 ? chunk0 + 1 : chunk0].c_off};
    int stage = 0;
    uint32_t phase = 0;
    for (int kb = kb_begin; kb < kb_end; ++kb) {
      const int n0 = (kb / kb_per_n) * p.bn;
      uint32_t split = kUnits;                     // units below `split` belong to group 0
      if (p.pro_groups == 2) {
        const int rb = (p.Nt / 2 - n0) * rows_per_n;
        split = rb <= 0 ? 0u : (rb >= 64 ? kUnits : static_cast<uint32_t>(rb) * 8u);
      }
      const uint32_t s_addr = smem_addr0 + static_cast<uint32_t>(stage) * stage_bytes;
      const int cj = xform_unit_channel(s_addr + tid * 16u, 7u);
      XformCoef k0[2], k1[2];
#pragma unroll
      for (int b = 0; b < 2; ++b) {
        if (b >= nchunks) break;
        if (split > 0) xform_load_smem(k0[b], xtab_addr, tchunks, 0, c_off[b] >> 6, cj);
        if (split < kUnits) xform_load_smem(k1[b], xtab_addr, tchunks, 1, c_off[b] >> 6, cj);
      }
      mbar_wait(&full[stage], phase);
#pragma unroll
      for (int b = 0; b < 2; ++b) {
        if (b >= nchunks) break;
        const uint32_t box = s_addr + static_cast<uint32_t>(b) * kBoxBytes;
        if (split > 0) xform_span<kWgXformThreads>(box, tid, split, k0[b]);
        if (split < kUnits) xform_span<kWgXformThreads>(box, xform_first<kWgXformThreads>(split, tid), kUnits, k1[b]);
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
        uint8_t* sa = smem + static_cast<size_t>(stage) * stage_bytes;
        mbar_expect_tx(&full[stage], static_cast<uint32_t>(nchunks + p.n_gboxes) * kBoxBytes);
        for (int b = 0; b < nchunks; ++b) {
          const cstp_mchunk mc = p.mchunks[chunk0 + b];
          tma_load_5d(sa + static_cast<uint32_t>(b) * kBoxBytes, &p.amap[mc.map_id], &full[stage], mc.c_off, w0 + mc.dw,
                      h0 + mc.dh, t0 + mc.dt, n0);
        }
        for (int j = 0; j < p.n_gboxes; ++j)
          tma_load_5d(sa + a_bytes + j * kBoxBytes, &p.gmap, &full[stage], ntile * p.n_tile + j * 64, w0, h0, t0, n0);
      }
      __syncwarp();
      if (++stage == p.stages) {
        stage = 0;
        phase ^= 1u;
      }
    }
  } else if (warp == 1) {
    const bool leader = elect_one();
    int stage = 0;
    uint32_t phase = 0;
    const uint32_t smem_addr0 = smem_u32(smem);
    const uint64_t dhi = umma_desc_hi(kBoxBytes, 1024);
    const int stages = p.stages;        // loop invariants in registers, clobber-free MMA issue (see conv_halo.cu)
    const uint32_t n_tile = static_cast<uint32_t>(p.n_tile);
    uint32_t idesc;
    asm volatile("mov.u32 %0, %1;" : "=r"(idesc) : "r"(p.idesc));
    for (int kb = kb_begin; kb < kb_end; ++kb) {
      mbar_wait(kXform ? &xfull[stage] : &full[stage], phase);
      tc_fence_after();
      if (leader) {
        const uint32_t a_addr = smem_addr0 + static_cast<uint32_t>(stage) * stage_bytes;
        // MN-major, 128B swizzle: 16 K-rows per step = 2048 B (+128 in the address field); LBO = next 64-channel
        // chunk, SBO = next 8 K-rows.  M tile mt: its two X boxes, accumulator mt (n_tile columns each), the shared G tile
        // (a tile whose second chunk does not exist multiplies stale rows that the epilogue never stores).
        const uint64_t db = umma_desc_at(dhi, a_addr + a_bytes);
        for (int mt = 0; mt < mts; ++mt) {
          const uint64_t da = umma_desc_at(dhi, a_addr + static_cast<uint32_t>(mt) * 2u * kBoxBytes);
          const uint32_t d_tmem = tmem_base + static_cast<uint32_t>(mt) * n_tile;
          umma_bf16_nc(d_tmem, da, db, idesc, kb > kb_begin ? 1u : 0u);
          umma_bf16_acc_nc(d_tmem, da + 128, db + 128, idesc);
          umma_bf16_acc_nc(d_tmem, da + 256, db + 256, idesc);
          umma_bf16_acc_nc(d_tmem, da + 384, db + 384, idesc);
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
    const int q = warp - 4;
    const int row = q * 32 + lane;
    const int col0 = ntile * p.n_tile;
    const int ncols = min(p.n_tile, p.Np - col0);
    const long long mtot = static_cast<long long>(p.n_mchunks) * 64;
    mbar_wait_idle(tfull, 0);
    tc_fence_after();
    for (int mt = 0; mt < mts; ++mt) {
      const bool valid = (2 * mt + (row >> 6)) < nchunks;
      float* dst = p.partials +
                   (static_cast<long long>(split) * mtot + (static_cast<long long>(mtile) * p.n_mt + mt) * 128 + row) * p.Np + col0;
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

// dW[(co*cin + ci)*taps + tap] = sum_s P[s][chunk*64 + r][co], ci = c_off(chunk) + r.  One thread per (row, co).
// layout 1 (stem, cstp_stem_pack): the X channel ci = hpar*32 + kw*3 + c of row pair tap j is w[co][c][0][2*j + hpar - 1][kw]
// of a (cout, 3, 1, 7, 7) weight; channels / taps without a weight element are skipped.
__global__ void wgrad_finalize_kernel(const float* __restrict__ partials, int splits, int n_mchunks, int Np,
                                      const int* __restrict__ chunk_tap, const int* __restrict__ chunk_coff, int cout,
                                      int cin, int taps, float* __restrict__ dw, int accumulate, int layout,
                                      const int* __restrict__ chunk_splits) {
  const long long mtot = static_cast<long long>(n_mchunks) * 64;
  // rows carry (tap, row channel), columns the other channel axis: (cin rows, cout columns) -- or, layout 2, the reverse
  const int ncol = layout == 2 ? cin : cout, nrow = layout == 2 ? cout : cin;
  const long long total = mtot * ncol;
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int col = static_cast<int>(i % ncol);
    const long long row = i / ncol;
    const int chunk = static_cast<int>(row >> 6);
    const int rc = chunk_coff[chunk] + static_cast<int>(row & 63);
    if (rc >= nrow) continue;
    const int ns = chunk_splits != nullptr ? chunk_splits[chunk] : splits;
    float acc = 0.f;
    for (int s = 0; s < ns; ++s) acc += partials[(static_cast<long long>(s) * mtot + row) * Np + col];
    const int co = layout == 2 ? rc : col, ci = layout == 2 ? col : rc;
    long long o;
    if (layout == 0 || layout == 2) {
      o = (static_cast<long long>(co) * cin + ci) * taps + chunk_tap[chunk];
    } else {
      const int k = ci & 31, kh = 2 * chunk_tap[chunk] + (ci >> 5) - 1;
      if (k >= 21 || kh < 0 || kh > 6) continue;
      o = ((static_cast<long long>(co) * 3 + k % 3) * 7 + kh) * 7 + k / 3;
    }
    dw[o] = accumulate ? dw[o] + acc : acc;
  }
}

}  // namespace cstp

struct cstp_wgrad_plan {
  cstp::WgradKParams kp;
  dim3 grid;
  int smem_bytes;
  int splits;
};

using namespace cstp;

static int encode_tensor5_w(CUtensorMap* map, const cstp_tensor5& t, const uint32_t box[5], bool oob_nan = false) {
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

extern "C" int cstp_wgrad_plan_create(const cstp_wgrad_desc* d, cstp_wgrad_plan** out_plan) {
  CSTP_REQUIRE(d != nullptr && out_plan != nullptr);
  CSTP_REQUIRE(d->n_amaps >= 1 && d->n_amaps <= CSTP_MAX_AMAPS);
  CSTP_REQUIRE(d->n_mchunks >= 1 && d->n_mchunks <= CSTP_MAX_MCHUNKS);
  CSTP_REQUIRE(d->Np >= 16 && d->Np % 16 == 0);
  CSTP_REQUIRE(d->n_tile >= 16 && d->n_tile % 16 == 0 && d->n_tile <= 256);
  CSTP_REQUIRE(d->Np <= d->n_tile || d->n_tile % 64 == 0);
  CSTP_REQUIRE(d->bw >= 1 && d->bh >= 1 && d->bt >= 1 && d->bn >= 1);
  CSTP_REQUIRE(d->bw * d->bh * d->bt * d->bn == 64);
  CSTP_REQUIRE(d->Wt >= 1 && d->Ht >= 1 && d->Tt >= 1 && d->Nt >= 1);
  CSTP_REQUIRE(d->splits >= 1 && d->partials != nullptr && reinterpret_cast<uintptr_t>(d->partials) % 32 == 0);   // 32-byte stores
  const bool xform = d->pro.scale != nullptr;
  const int n_mt = d->mt_per_cta > 0 ? d->mt_per_cta : 1;
  CSTP_REQUIRE(n_mt <= kWgMaxMt && n_mt * d->n_tile <= 512 && (!xform || n_mt == 1));
  if (xform) {
    CSTP_REQUIRE(d->pro.shift != nullptr && (d->pro.groups == 1 || d->pro.groups == 2) && d->Nt % d->pro.groups == 0);
    CSTP_REQUIRE(d->pro.Cp == d->amap[0].dims[0]);
    CSTP_REQUIRE(reinterpret_cast<uintptr_t>(d->pro.scale) % 16 == 0 && reinterpret_cast<uintptr_t>(d->pro.shift) % 16 == 0);
  }

  cstp_wgrad_plan* plan = new (std::nothrow) cstp_wgrad_plan();
  if (!plan) {
    set_error("out of host memory");
    return CSTP_ENOMEM;
  }
  WgradKParams& k = plan->kp;
  memset(&k, 0, sizeof(k));
  const uint32_t box[5] = {64u, (uint32_t)d->bw, (uint32_t)d->bh, (uint32_t)d->bt, (uint32_t)d->bn};
  for (int i = 0; i < CSTP_MAX_AMAPS; ++i) {
    int rc = encode_tensor5_w(&k.amap[i], d->amap[i < d->n_amaps ? i : 0], box, xform);
    if (rc != CSTP_OK) {
      delete plan;
      return rc;
    }
  }
  {
    int rc = encode_tensor5_w(&k.gmap, d->gmap, box);
    if (rc != CSTP_OK) {
      delete plan;
      return rc;
    }
  }
  k.tiles_w = ceil_div(d->Wt, d->bw);
  k.tiles_h = ceil_div(d->Ht, d->bh);
  k.tiles_t = ceil_div(d->Tt, d->bt);
  k.tiles_n = ceil_div(d->Nt, d->bn);
  k.bw = d->bw; k.bh = d->bh; k.bt = d->bt; k.bn = d->bn;
  k.n_mchunks = d->n_mchunks;
  k.Np = d->Np;
  k.n_tile = d->n_tile;
  k.n_gboxes = ceil_div(d->n_tile, 64);
  k.n_mt = n_mt;
  k.total_kblocks = k.tiles_w * k.tiles_h * k.tiles_t * k.tiles_n;
  int splits = d->splits < k.total_kblocks ? d->splits : k.total_kblocks;
  k.kblocks_per_split = ceil_div(k.total_kblocks, splits);
  splits = ceil_div(k.total_kblocks, k.kblocks_per_split);
  plan->splits = splits;
  k.idesc = umma_idesc_bf16(128, static_cast<uint32_t>(d->n_tile), 1, 1);
  k.partials = d->partials;
  k.pro_scale = d->pro.scale;
  k.pro_shift = d->pro.shift;
  k.pro_groups = d->pro.groups;
  k.pro_cp = d->pro.Cp;
  k.Nt = d->Nt;
  for (int i = 0; i < d->n_mchunks; ++i) {
    const cstp_mchunk& mc = d->mchunks[i];
    if (mc.map_id < 0 || mc.map_id >= d->n_amaps || mc.c_off < 0 || mc.c_off % 8 != 0 || (xform && mc.c_off % 64 != 0)) {
      delete plan;
      return fail_inval("mchunk map_id / c_off out of range");
    }
    k.mchunks[i] = mc;
  }
  const uint32_t stage_bytes = (2u * static_cast<uint32_t>(n_mt) + static_cast<uint32_t>(k.n_gboxes)) * kBoxBytes;
  const int bar_bytes = 256;
  const int xtab_bytes = xform ? static_cast<int>(xform_table_bytes(d->pro.groups, d->pro.Cp)) : 0;      // prologue coefficient table
  int stages = (kSmemBudget - 1024 - bar_bytes - xtab_bytes) / static_cast<int>(stage_bytes);
  if (stages > kWgMaxStages) stages = kWgMaxStages;
  if (stages < 2) {
    delete plan;
    return fail_inval("wgrad stage (mt_per_cta X boxes + the G tile) too large for a two-stage shared-memory pipeline");
  }
  k.stages = stages;
  int cols = 32;
  while (cols < n_mt * d->n_tile) cols *= 2;
  k.tmem_cols = cols;
  plan->smem_bytes = 1024 + stages * static_cast<int>(stage_bytes) + bar_bytes + xtab_bytes;
  if (plan->smem_bytes < 120 * 1024) plan->smem_bytes = 120 * 1024;
  plan->grid = dim3(static_cast<unsigned>(ceil_div(d->n_mchunks, 2 * n_mt)), static_cast<unsigned>(ceil_div(d->Np, d->n_tile)),
                    static_cast<unsigned>(splits));
  *out_plan = plan;
  return CSTP_OK;
}

extern "C" int cstp_wgrad_plan_splits(const cstp_wgrad_plan* plan) { return plan ? plan->splits : CSTP_EINVAL; }

extern "C" int cstp_wgrad_plan_run(const cstp_wgrad_plan* plan, void* stream) {
  CSTP_REQUIRE(plan != nullptr);
  static bool attr_set = false;
  if (!attr_set) {
    CSTP_CUDA(cudaFuncSetAttribute(wgrad_gemm_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, kWgSmemLimit));
    CSTP_CUDA(cudaFuncSetAttribute(wgrad_gemm_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, kWgSmemLimit));
    attr_set = true;
  }
  if (plan->kp.pro_scale != nullptr)
    wgrad_gemm_kernel<true><<<plan->grid, kWgThreads + kWgXformThreads, plan->smem_bytes, static_cast<cudaStream_t>(stream)>>>(plan->kp);
  else
    wgrad_gemm_kernel<false><<<plan->grid, kWgThreads, plan->smem_bytes, static_cast<cudaStream_t>(stream)>>>(plan->kp);
  CSTP_LAUNCHED();
  return CSTP_OK;
}

extern "C" void cstp_wgrad_plan_destroy(cstp_wgrad_plan* plan) { delete plan; }

extern "C" int cstp_wgrad_finalize(const float* partials, int splits, int n_mchunks, int Np, const int32_t* chunk_tap,
                                   const int32_t* chunk_coff, int cout, int cin, int taps, float* dw, int accumulate,
                                   int layout, const int32_t* chunk_splits, void* stream) {
  CSTP_REQUIRE(partials && chunk_tap && chunk_coff && dw);
  CSTP_REQUIRE(layout == 0 || layout == 2 || (layout == 1 && cin == 64 && taps == 4));
  CSTP_REQUIRE(splits >= 1 && n_mchunks >= 1 && n_mchunks <= CSTP_MAX_MCHUNKS && (layout == 2 ? cin : cout) <= Np);
  // chunk_tap / chunk_coff are device pointers (tiny int arrays uploaded once by the host at plan time).
  const long long total = static_cast<long long>(n_mchunks) * 64 * (layout == 2 ? cin : cout);
  int blocks = ceil_div(total, 256);
  if (blocks > 4 * num_sms()) blocks = 4 * num_sms();
  wgrad_finalize_kernel<<<blocks, 256, 0, static_cast<cudaStream_t>(stream)>>>(partials, splits, n_mchunks, Np, chunk_tap,
                                                                             chunk_coff, cout, cin, taps, dw, accumulate,
                                                                             layout, chunk_splits);
  CSTP_LAUNCHED();
  return CSTP_OK;
}

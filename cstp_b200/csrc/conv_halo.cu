// Implicit-GEMM convolution (forward and dgrad) for the stride-1 1x3x3 / 3x1x1 layers with a large spatial extent
// (conv1.temporal, conv2.*, conv3.block1.conv2.*), where conv_gemm.cu is bound by the L2->SM feed, not by the tensor
// pipe: it stages one 128-position activation box PER FILTER TAP (9x / 3x the same data) and one weight tile per tap
// for every output tile.  Here
//   * the activation box is staged once per "load group" with a HALO along the tap axis; the taps of that axis are the
//     same shared-memory rows shifted by a multiple of 8 rows (whole 128B-swizzle atoms), i.e. just another UMMA
//     descriptor start address.  Taps along the fastest axis (kw) are separate groups (a one-row shift is not
//     atom aligned);
//   * when all weight K-blocks of one N tile fit next to the activation pipeline they are loaded ONCE per CTA
//     ("resident B"); every CTA then keeps its N tile for its whole life (blockIdx.y) and walks M tiles only.
//   * "slab mode" (64-column dgrad of the 1x3x3 layers): a tcgen05.mma of 128 x 64 x 16 cannot be fed faster than one
//     per ~76 cycles (its 4 KB A slice comes out of shared memory at 64 B/clk) while the tensor pipe needs 32.  So G
//     consecutive output rows (slabs along h) share one accumulator of G x 64 columns: every INPUT slab is staged once
//     and multiplied, in ONE MMA of up to 3 x 64 columns, with the stacked weights [tap +1 | tap 0 | tap -1] of the
//     output slabs it feeds (a row offset into the resident weight block picks the sub-range at the tile's borders).
//     36 tap units of a 1x3x3 tile with G = 4 take 18 MMA series instead of 36, and every A slice is read once instead
//     of three times.
// Same math, epilogue and output layout as conv_gemm.cu.
// Replaces cuDNN conv3d fwd/dgrad behind models/pace/r21d_byol.py:81-97 (main_byol.py:87 for the dgrad).
#include "common.h"
#include "ptx.cuh"

namespace cstp {

constexpr int kHcThreads = 256;
constexpr int kHcXformThreads = 256;     // warps 8..15: operand prologue
constexpr int kHcMaxStages = 8;
constexpr int kHcSmemLimit = 232448;
constexpr int kHcMaxGroups = 4;
constexpr int kHcMaxTaps = 16;
constexpr int kHcMaxSlabs = 8;           // staged input slabs per tile in slab mode (G + taps along h - 1)

struct HcGroup {
  int dw, dh, dt;       // origin offset of the staged (halo) box from the tile origin
  int first_tap, n_taps;
};
struct HcTap {
  uint32_t a_shift;     // byte offset of this tap's first row inside the staged box (multiple of 1024)
  int k_off;            // column of its first 64-channel chunk in the packed weight matrix
};

struct ConvHaloKParams {
  CUtensorMap amap;
  CUtensorMap bmap;
  CUtensorMap amap_tail;   // channel tail (16 or 32 channels beyond a multiple of 64): boxes with 32 / 64-byte rows
  CUtensorMap bmap_tail;
  int tail;                // 0, 16 or 32 channels in the last chunk (then staged with its own narrow boxes)
  uint32_t a_bytes_tail, b_bytes_tail, tap_bytes;   // tap_bytes: resident weight bytes of one tap (all chunks)
  int tiles_w, tiles_h, tiles_t, tiles_n;
  int bw, bh, bt, bn;
  int Wt, Ht, Tt, Nt;
  int n_groups, n_taps, chunks, last_ksteps;
  int n_tile, Np;
  int stages, tmem_cols, resident;
  uint32_t a_bytes, b_bytes, stage_bytes, res_bytes, idesc;
  uint32_t a_stride;       // a_bytes rounded up to 1024: where the per-stage weight tiles start (non-resident mode)
  int group_taps;          // taps per load group (all groups hold the same number)
  int tap_nw;              // regular tap walk of a load group: tap j sits (j % tap_nw) * tap_sw + (j / tap_nw) * tap_sh
  uint32_t tap_sw, tap_sh; // bytes into the staged box (validated against taps[].a_shift when the plan is built)
  uint32_t a_sbo;          // bytes between consecutive 8-row atoms of a tap's rows inside the staged box (128-byte rows)
  int accumulate;
  float* stats;            // optional fused BatchNorm statistics: partials [gridDim.x][stats_groups][2][Np] (Np == 64)
  int stats_groups;
  int fast_store;          // bf16 output only, no bias, 32-byte aligned rows: pipelined epilogue with STG.256
  // operand prologue (kXform): A is the producer's raw output; BatchNorm affine + ReLU applied to every staged box
  const float* pro_scale;  // fp32 [pro_groups][pro_cp]
  const float* pro_shift;
  int pro_groups, pro_cp;
  uint32_t xtab_off;       // byte offset (from the mbarrier block) of the prologue's coefficient table in shared memory
  __nv_bfloat16* out;
  float* out_f32;
  const float* bias;
  long long out_off, osw, osh, ost, osn;
  int step_h;              // tile step along h (bh, or G in slab mode)
  // slab mode (slab_g > 1): G output rows of slab_cols columns each on the accumulator's N axis
  int slab_g;
  int slab_in;             // staged input slabs per tile
  int slab_nslots;         // taps along h (weights of one w tap: nslots stacked blocks of slab_cols rows)
  int slab_cols;
  uint32_t res_tap_stride, res_chunk_stride, res_tail_base, res_tail_tap_stride;     // resident weight block layout
  int slab_order[kHcMaxSlabs];    // load / issue order of the input slabs (the first MMA of an accumulator column range
  int slab_init[kHcMaxSlabs];     // must overwrite: slabs flagged `init` come first and cover disjoint column ranges)
  int slab_doff[kHcMaxSlabs];     // first accumulator column this input slab feeds
  int slab_brow[kHcMaxSlabs];     // first row of the stacked weight block it multiplies with
  uint32_t slab_idesc[kHcMaxSlabs];
  HcGroup groups[kHcMaxGroups];
  HcTap taps[kHcMaxTaps];
};

// Fused BatchNorm statistics (kStats): one 16-column chunk of a 64-column tile -- pack, store, and add the values AS
// STORED (bf16-rounded) to this thread's running sum / sum of squares of its row (acc[c], acc[64 + c]; static indices).
template <int kC0>
__device__ __forceinline__ void stats_chunk(const uint32_t (&v)[16], __nv_bfloat16* dst, bool valid, float (&acc)[128]) {
  uint32_t w[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) w[i] = pack_bf16x2(__uint_as_float(v[2 * i]), __uint_as_float(v[2 * i + 1]));
  if (valid) {
    st_global_256(dst + kC0, w);
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const float lo = bf16_lo(w[i]), hi = bf16_hi(w[i]);
      acc[kC0 + 2 * i] += lo;
      acc[kC0 + 2 * i + 1] += hi;
      acc[64 + kC0 + 2 * i] = fmaf(lo, lo, acc[64 + kC0 + 2 * i]);
      acc[64 + kC0 + 2 * i + 1] = fmaf(hi, hi, acc[64 + kC0 + 2 * i + 1]);
    }
  }
}

// Adds the 128 per-thread accumulators of the four epilogue warps (= 128 rows) into tot[e] (e = quantity * 64 + column),
// in a fixed order, and clears them.  Reduce-scatter butterfly: after the five steps lane L holds entries 4L .. 4L+3.
__device__ __forceinline__ void stats_flush(float (&acc)[128], float* wsum, float* tot, int q, int lane) {
#pragma unroll
  for (int half = 64, m = 16; half >= 4; half >>= 1, m >>= 1) {
    const bool up = (lane & m) != 0;
#pragma unroll
    for (int i = 0; i < half; ++i) {
      const float send = up ? acc[i] : acc[i + half];
      const float keep = up ? acc[i + half] : acc[i];
      acc[i] = keep + __shfl_xor_sync(0xffffffffu, send, m);
    }
  }
#pragma unroll
  for (int j = 0; j < 4; ++j) wsum[q * 128 + 4 * lane + j] = acc[j];
  asm volatile("bar.sync 1, 128;" ::: "memory");
  const int e = q * 32 + lane;
  tot[e] += ((wsum[e] + wsum[128 + e]) + wsum[256 + e]) + wsum[384 + e];
  asm volatile("bar.sync 1, 128;" ::: "memory");
#pragma unroll
  for (int i = 0; i < 128; ++i) acc[i] = 0.f;
}

// One K-block of one load group with FULL 64-channel chunks (four K steps per tap), for the tap walks this network uses:
// kTaps taps, kNw of them along w.  Every descriptor is the first tap's plus a compile-time combination of three loop
// invariants (the 14-bit start-address field never carries: shared addresses stay below 256 KB), so the issuing thread
// spends two adds per tcgen05.mma.  The generic walk below costs ~35 uniform-datapath instructions per tap, two of them
// constant-bank loads: the N = 64 layers (32 tensor cycles per MMA) ran at 76 issue cycles per MMA, 42 % tensor-pipe
// activity (ncu r02_c2s_dgrad_plain).
template <int kTaps, int kNw>
__device__ __forceinline__ void issue_group_full(uint32_t d_tmem, uint64_t da0, uint64_t db0, uint64_t sw16, uint64_t sh16,
                                                 uint64_t bstep16, uint32_t idesc, uint32_t first) {
#pragma unroll
  for (int j = 0; j < kTaps; ++j) {
    const uint64_t da = da0 + static_cast<uint64_t>(j % kNw) * sw16 + static_cast<uint64_t>(j / kNw) * sh16;
    const uint64_t db = db0 + static_cast<uint64_t>(j) * bstep16;
    if (j == 0) umma_bf16_nc(d_tmem, da, db, idesc, first ? 0u : 1u);
    else umma_bf16_acc_nc(d_tmem, da, db, idesc);
    umma_bf16_acc_nc(d_tmem, da + 2, db + 2, idesc);
    umma_bf16_acc_nc(d_tmem, da + 4, db + 4, idesc);
    umma_bf16_acc_nc(d_tmem, da + 6, db + 6, idesc);
  }
}

// kXform: eight more warps (8..15) rewrite every staged activation box in place -- BatchNorm affine + ReLU of the producing
// unit (ptx.cuh) -- between the TMA arrival (full[]) and the MMA issue (xfull[]).
template <bool kStats, bool kXform>
__global__ void __launch_bounds__(kXform ? kHcThreads + kHcXformThreads : kHcThreads, 1)
    conv_halo_kernel(const __grid_constant__ ConvHaloKParams p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* stage0 = smem + p.res_bytes;
  uint64_t* bars = reinterpret_cast<uint64_t*>(stage0 + static_cast<size_t>(p.stages) * p.stage_bytes);
  uint64_t* full = bars;
  uint64_t* empty = bars + kHcMaxStages;
  uint64_t* tfull = bars + 2 * kHcMaxStages;
  uint64_t* tempty = bars + 2 * kHcMaxStages + 2;
  uint64_t* bfull = bars + 2 * kHcMaxStages + 4;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * kHcMaxStages + 5);
  uint64_t* xfull = bars + 2 * kHcMaxStages + 6;        // [kHcMaxStages]: staged box transformed (kXform)

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int ntile = blockIdx.y;
  const int m_tiles = p.tiles_w * p.tiles_h * p.tiles_t * p.tiles_n;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&p.amap);
    tma_prefetch_desc(&p.bmap);
  }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < p.stages; ++s) {
      mbar_init(&full[s], 1);
      mbar_init(&empty[s], 1);
      if constexpr (kXform) mbar_init(&xfull[s], kHcXformThreads / 32);
    }
    for (int a = 0; a < 2; ++a) {
      mbar_init(&tfull[a], 1);
      mbar_init(&tempty[a], 4);
    }
    mbar_init(bfull, 1);
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
  // kStats && kXform: 384 threads leave 168 registers each, but the statistics epilogue keeps 128 accumulators per thread:
  // the producer / issuer warpgroup and the transform warpgroup hand registers to the epilogue warpgroup (setmaxnreg at
  // the head of each warpgroup's branch, where ptxas can see which code runs under which budget).
  constexpr bool kRealloc = kStats && kXform;
  // slab mode (plain dgrad only) is compiled into the instantiation without prologue and statistics
  constexpr bool kSlabOk = !kStats && !kXform;

  // Roles run WARP-CONVERGED: all 32 lanes walk the loops and poll the mbarriers, one elected lane issues the TMA /
  // tcgen05 instructions.  (With a single-lane branch the compiler cannot keep descriptors and addresses in uniform
  // registers and wraps every UTCHMMA in an ELECT / R2UR loop: the issuer then ran at ~25 cycles per instruction and
  // the N=64 layers sat at 19% tensor-pipe activity, ncu r01_conv_halo.)
  if (warp < 4) {
   if constexpr (kRealloc) warpgroup_reg_dec<120>();
   if (warp == 0) {
    // ------------------------------------------------------------ TMA producer
    const bool leader = elect_one();
    const int full_chunks = p.tail ? p.chunks - 1 : p.chunks;
    if (p.resident && leader) {
      mbar_expect_tx(bfull, p.res_bytes);
      for (int t = 0; t < p.n_taps; ++t) {
        uint8_t* tb = smem + static_cast<size_t>(t) * p.res_tap_stride;
        for (int c = 0; c < full_chunks; ++c)
          tma_load_2d(tb + static_cast<size_t>(c) * p.res_chunk_stride, &p.bmap, bfull, p.taps[t].k_off + c * 64,
                      ntile * p.n_tile);
        if (p.tail)
          tma_load_2d(smem + p.res_tail_base + static_cast<size_t>(t) * p.res_tail_tap_stride, &p.bmap_tail, bfull,
                      p.taps[t].k_off + full_chunks * 64, ntile * p.n_tile);
      }
    }
    int stage = 0;
    uint32_t phase = 0;
    const int pslab = kSlabOk ? p.slab_g : 0;
    const int n_loads = pslab ? p.slab_in : p.n_groups;
    for (int tile = blockIdx.x; tile < m_tiles; tile += gridDim.x) {
      int pt = tile;
      const int w0 = (pt % p.tiles_w) * p.bw;
      pt /= p.tiles_w;
      const int h0 = (pt % p.tiles_h) * p.step_h;
      pt /= p.tiles_h;
      const int t0 = (pt % p.tiles_t) * p.bt;
      pt /= p.tiles_t;
      const int n0 = pt * p.bn;
      for (int g = 0; g < n_loads; ++g) {
        HcGroup gr = p.groups[pslab ? 0 : g];
        if (pslab) gr.dh += p.slab_order[g];      // input slab s of the tile: the first slab's origin moved s rows along h
        for (int c = 0; c < p.chunks; ++c) {
          mbar_wait(&empty[stage], phase ^ 1u);
          if (leader) {
            uint8_t* st = stage0 + static_cast<size_t>(stage) * p.stage_bytes;
            const bool tl = p.tail && c == p.chunks - 1;
            const uint32_t ab = tl ? p.a_bytes_tail : p.a_bytes, bb = tl ? p.b_bytes_tail : p.b_bytes;
            mbar_expect_tx(&full[stage], ab + (p.resident ? 0u : static_cast<uint32_t>(gr.n_taps) * bb));
            tma_load_5d(st, tl ? &p.amap_tail : &p.amap, &full[stage], c * 64, w0 + gr.dw, h0 + gr.dh, t0 + gr.dt, n0);
            if (!p.resident) {
              for (int j = 0; j < gr.n_taps; ++j)
                tma_load_2d(st + p.a_stride + static_cast<size_t>(j) * p.b_bytes, tl ? &p.bmap_tail : &p.bmap, &full[stage],
                            p.taps[gr.first_tap + j].k_off + c * 64, ntile * p.n_tile);
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
    // Every loop-invariant parameter is copied out of the constant bank once, the tap walk is pure uniform arithmetic
    // (tap j of a group sits (j % nw) * sw + (j / nw) * sh bytes into the staged box; its weights follow the previous
    // tap's), and the MMAs are issued without a compiler memory clobber: with the taps[] table and the clobbering
    // wrappers the issuing warp spent ~85 cycles per UTCHMMA on LDCU round trips (ncu source page, profiles/README.md)
    // while a 128x64x16 MMA occupies the tensor pipe for 32.
    const bool leader = elect_one();
    const uint32_t stage_bytes = p.stage_bytes, a_stride = p.a_stride, b_bytes = p.b_bytes, tap_bytes = p.tap_bytes;
    uint32_t idesc;             // pinned in a register: the compiler otherwise re-loads it in front of every tap
    asm volatile("mov.u32 %0, %1;" : "=r"(idesc) : "r"(p.idesc));
    const int slab_g = kSlabOk ? p.slab_g : 0;
    const int n_groups = slab_g ? p.slab_in : p.n_groups, chunks = p.chunks, last_ksteps = p.last_ksteps, stages = p.stages,
              n_tile = p.n_tile;
    // (copied through registers once: the compiler otherwise re-loads them from the constant bank inside the tap loop)
    int nw, group_taps;
    asm volatile("mov.u32 %0, %1;" : "=r"(nw) : "r"(p.tap_nw));
    asm volatile("mov.u32 %0, %1;" : "=r"(group_taps) : "r"(p.group_taps));
    const bool resident = p.resident != 0, has_tail = p.tail != 0;
    const int tail_shift = p.tail == 16 ? 2 : 1;        // shifts are in 128-byte rows; tail rows are 32 / 64 bytes
    const uint32_t sw_full = p.tap_sw, sh_full = p.tap_sh;
    const int full_chunks = has_tail ? chunks - 1 : chunks;
    if (resident) {
      mbar_wait(bfull, 0);
      tc_fence_after();
    }
    const uint32_t res_addr = smem_u32(smem);
    const uint32_t stage_addr0 = smem_u32(stage0);
    const uint64_t dhi_b = umma_desc_hi(16, 1024);
    const uint64_t dhi_a = umma_desc_hi(16, p.a_sbo);
    const uint64_t dhi_tail_b = umma_desc_hi_kmajor(static_cast<uint32_t>(p.tail) * 2u);
    // tail rows are 32 / 64 bytes wide: the atom pitch shrinks with the row width
    const uint64_t dhi_tail_a = umma_desc_hi_kmajor_sbo(static_cast<uint32_t>(p.tail) * 2u, p.a_sbo / 128u * static_cast<uint32_t>(p.tail) * 2u);
    int stage = 0;
    uint32_t phase = 0;
    int it = 0;
    for (int tile = blockIdx.x; tile < m_tiles; tile += gridDim.x, ++it) {
      const int as = it & 1;
      const uint32_t aphase = (it >> 1) & 1;
      mbar_wait(&tempty[as], aphase ^ 1u);
      tc_fence_after();
      const uint32_t d_tmem = tmem_base + static_cast<uint32_t>(as * n_tile);
      uint32_t first = 1;
      for (int g = 0; g < n_groups; ++g) {
        const int g_first = g * group_taps, g_taps = group_taps;        // groups are equal-sized (checked at plan creation)
        for (int c = 0; c < chunks; ++c) {
          mbar_wait(kXform ? &xfull[stage] : &full[stage], phase);
          tc_fence_after();
          if (leader) {
            const uint32_t s_addr = stage_addr0 + static_cast<uint32_t>(stage) * stage_bytes;
            const bool tl = has_tail && c == chunks - 1;
            const int ks = (c == chunks - 1) ? last_ksteps : 4;
            const uint64_t hi_a = tl ? dhi_tail_a : dhi_a, hi_b = tl ? dhi_tail_b : dhi_b;
            const uint32_t sw = tl ? sw_full >> tail_shift : sw_full, sh = tl ? sh_full >> tail_shift : sh_full;
            if (slab_g) {
              // slab mode: this stage holds ONE input slab; w tap j multiplies it with the stacked weight blocks of the
              // output slabs it feeds (brow rows into the [nslots x slab_cols]-row block of tap j), ncols wide, into the
              // accumulator columns doff .. doff + ncols
              const uint32_t rowb = tl ? static_cast<uint32_t>(p.tail) * 2u : 128u;
              const uint32_t blk = static_cast<uint32_t>(p.slab_nslots) * (tl ? p.res_tail_tap_stride : p.res_tap_stride);
              const uint32_t b0 = res_addr + (tl ? p.res_tail_base : static_cast<uint32_t>(c) * p.res_chunk_stride) +
                                  static_cast<uint32_t>(p.slab_brow[g]) * rowb;
              const uint32_t sidesc = p.slab_idesc[g];
              const uint32_t dcol = d_tmem + static_cast<uint32_t>(p.slab_doff[g]);
              uint32_t acc = (p.slab_init[g] && c == 0) ? 0u : 1u;
              for (int j = 0; j < nw; ++j) {
                const uint64_t da = umma_desc_at(hi_a, s_addr + static_cast<uint32_t>(j) * sw);
                const uint64_t db = umma_desc_at(hi_b, b0 + static_cast<uint32_t>(j) * blk);
                umma_bf16_nc(dcol, da, db, sidesc, acc);
                acc = 1u;
                for (int k = 1; k < ks; ++k) umma_bf16_acc_nc(dcol, da + 2 * k, db + 2 * k, sidesc);
              }
              umma_commit(&empty[stage]);
              if (g == n_groups - 1 && c == chunks - 1) umma_commit(&tfull[as]);
            } else {
            uint32_t b_addr = resident ? res_addr + static_cast<uint32_t>(g_first) * tap_bytes +
                                             static_cast<uint32_t>(tl ? full_chunks : c) * b_bytes
                                       : s_addr + a_stride;
            const uint32_t b_step = resident ? tap_bytes : b_bytes;
            if (ks == 4 && nw == 3 && (g_taps == 9 || g_taps == 3)) {
              const uint64_t da0 = umma_desc_at(hi_a, s_addr), db0 = umma_desc_at(hi_b, b_addr);
              if (g_taps == 9) issue_group_full<9, 3>(d_tmem, da0, db0, sw >> 4, sh >> 4, b_step >> 4, idesc, first);
              else issue_group_full<3, 3>(d_tmem, da0, db0, sw >> 4, sh >> 4, b_step >> 4, idesc, first);
              first = 0;
            } else {
            uint32_t a_addr = s_addr, a_row0 = s_addr;       // a_addr walks along w, a_row0 is the start of its h row
            int jw = 0;
            for (int j = 0; j < g_taps; ++j) {
              // the swizzle XOR follows the absolute shared-memory address: a start that is a whole number of rows but
              // not 1024-aligned needs no descriptor base offset (measured: setting it breaks the result)
              const uint64_t da = umma_desc_at(hi_a, a_addr);
              const uint64_t db = umma_desc_at(hi_b, b_addr);
              umma_bf16_nc(d_tmem, da, db, idesc, first ? 0u : 1u);
              first = 0;
              if (ks == 4) {
                umma_bf16_acc_nc(d_tmem, da + 2, db + 2, idesc);
                umma_bf16_acc_nc(d_tmem, da + 4, db + 4, idesc);
                umma_bf16_acc_nc(d_tmem, da + 6, db + 6, idesc);
              } else {
                for (int k = 1; k < ks; ++k) umma_bf16_acc_nc(d_tmem, da + 2 * k, db + 2 * k, idesc);
              }
              b_addr += b_step;
              if (++jw == nw) {
                jw = 0;
                a_row0 += sh;
                a_addr = a_row0;
              } else {
                a_addr += sw;
              }
            }
            }
            umma_commit(&empty[stage]);
            if (g == n_groups - 1 && c == chunks - 1) umma_commit(&tfull[as]);
            }
          }
          first = 0;
          __syncwarp();
          if (++stage == stages) {
            stage = 0;
            phase ^= 1u;
          }
        }
      }
    }
   }
  } else if (kXform && warp >= 8) {
    if constexpr (kRealloc) warpgroup_reg_dec<88>();
    // ------------------------------------------------------------ operand prologue: BatchNorm affine + ReLU in place
    // Thread t owns the 16-byte units t, t + 256, ... of every staged box: a fixed swizzle phase, i.e. one 8-channel
    // vector of the chunk, whose coefficients come from a table the transform warps build once in shared memory.
    const uint32_t tid = threadIdx.x - kHcThreads;
    float* xtab = reinterpret_cast<float*>(reinterpret_cast<uint8_t*>(bars) + p.xtab_off);
    xform_table_fill<kHcXformThreads>(xtab, p.pro_scale, p.pro_shift, p.pro_groups, p.pro_cp, tid);
    xform_bar_sync<kHcXformThreads>();
    const uint32_t xtab_addr = smem_u32(xtab);
    const uint32_t stage_addr0 = smem_u32(stage0);
    const uint32_t stage_bytes = p.stage_bytes;
    const int n_groups = p.n_groups, chunks = p.chunks, stages = p.stages;
    const bool has_tail = p.tail != 0;
    const uint32_t units_full = p.a_bytes >> 4, units_tail = p.a_bytes_tail >> 4;
    const uint32_t mask_tail = p.tail == 16 ? 1u : 3u;
    const int slab = p.tiles_w * p.tiles_h * p.tiles_t;        // tiles per bn samples (all of one statistics group)
    int stage = 0;
    uint32_t phase = 0;
    for (int tile = blockIdx.x; tile < m_tiles; tile += gridDim.x) {
      const int n0 = (tile / slab) * p.bn;
      const int grp = (p.pro_groups == 2 && 2 * n0 >= p.Nt) ? 1 : 0;
      for (int g = 0; g < n_groups; ++g) {
        for (int c = 0; c < chunks; ++c) {
          const bool tl = has_tail && c == chunks - 1;
          const uint32_t s_addr = stage_addr0 + static_cast<uint32_t>(stage) * stage_bytes;
          XformCoef k;
          xform_load_smem(k, xtab_addr, chunks, grp, c, xform_unit_channel(s_addr + tid * 16u, tl ? mask_tail : 7u));
          mbar_wait(&full[stage], phase);
          xform_span<kHcXformThreads>(s_addr, tid, tl ? units_tail : units_full, k);
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
    if constexpr (kRealloc) warpgroup_reg_inc<216>();
    // ------------------------------------------------------------ epilogue (warp w owns TMEM lanes 32*(w%4)..)
    const int q = warp - 4;
    const int row = q * 32 + lane;
    const int rw = row % p.bw;
    const int rh = (row / p.bw) % p.bh;
    const int rt = (row / (p.bw * p.bh)) % p.bt;
    const int rn = row / (p.bw * p.bh * p.bt);
    const int col0 = ntile * p.n_tile;
    const int ncols = min(p.n_tile, p.Np - col0);
    // fused statistics: [4 warps][128] cross-warp staging + [2 groups][128] CTA totals behind the mbarriers
    float* wsum = reinterpret_cast<float*>(reinterpret_cast<uint8_t*>(bars) + 256);
    float* tot = wsum + 512;
    float acc[128];            // only touched (and only allocated) in the kStats instantiation
    int cur_group = -1;
    if constexpr (kStats) {
#pragma unroll
      for (int i = 0; i < 128; ++i) acc[i] = 0.f;
      tot[row] = 0.f;
      tot[128 + row] = 0.f;
    }
    int it = 0;
    for (int tile = blockIdx.x; tile < m_tiles; tile += gridDim.x, ++it) {
      const int as = it & 1;
      const uint32_t aphase = (it >> 1) & 1;
      int pt = tile;
      const int w = (pt % p.tiles_w) * p.bw + rw;
      pt /= p.tiles_w;
      const int h = (pt % p.tiles_h) * p.step_h + rh;
      pt /= p.tiles_h;
      const int t = (pt % p.tiles_t) * p.bt + rt;
      pt /= p.tiles_t;
      const int n_first = pt * p.bn;                          // first sample of the tile
      const int n = n_first + rn;
      const bool valid = (w < p.Wt) && (h < p.Ht) && (t < p.Tt) && (n < p.Nt);
      const long long off = p.out_off + w * p.osw + h * p.osh + t * p.ost + n * p.osn + col0;
      mbar_wait(&tfull[as], aphase);
      tc_fence_after();
      const uint32_t taddr = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + static_cast<uint32_t>(as * p.n_tile);
      if constexpr (kStats) {
        // 64-column tile, plain bf16 output, bn == 1: the whole tile belongs to ONE statistics group (the halves of the N
        // axis are the two views); the accumulators are flushed when the group changes (at most once per CTA) and at
        // the end -- no shuffle and no shared memory per tile, two FMAs per element
        const int g = (p.stats_groups == 2 && 2 * n_first >= p.Nt) ? 1 : 0;  // all bn samples of a tile share the group
        if (g != cur_group) {
          if (cur_group >= 0) stats_flush(acc, wsum, tot + cur_group * 128, q, lane);
          cur_group = g;
        }
        __nv_bfloat16* dst = p.out + off;
        uint32_t va[16], vb[16];
        tmem_ld16(taddr, va);
        tmem_ld_wait();
        tmem_ld16(taddr + 16, vb);
        stats_chunk<0>(va, dst, valid, acc);
        tmem_ld_wait();
        tmem_ld16(taddr + 32, va);
        stats_chunk<16>(vb, dst, valid, acc);
        tmem_ld_wait();
        tmem_ld16(taddr + 48, vb);
        stats_chunk<32>(va, dst, valid, acc);
        tmem_ld_wait();
        stats_chunk<48>(vb, dst, valid, acc);
      } else if (kSlabOk && p.slab_g) {
        // slab mode: column block o of the accumulator is output row h + o (plain bf16 rows)
        for (int o = 0; o < p.slab_g; ++o) {
          const bool ok = valid && h + o < p.Ht;
          const uint32_t ta = taddr + static_cast<uint32_t>(o * p.slab_cols);
          if (p.accumulate) epilogue_row_bf16<true>(ta, p.slab_cols, p.out + off + o * p.osh, ok);
          else epilogue_row_bf16<false>(ta, p.slab_cols, p.out + off + o * p.osh, ok);
        }
      } else if (p.fast_store) {
        // plain bf16 output (optionally accumulated into what is there): pipelined, one 32-byte store per 16 columns.
        // (The row-per-thread layout makes every 16-byte store a half-written sector; with nine serial
        // load -> wait -> 2 x STG.128 rounds the epilogue warps were busy 93 % of a 64->144 tile and the issuer waited
        // on the accumulator 21 % of the time: ncu source page, profiles/README.md.)
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
    if constexpr (kStats) {
      if (cur_group >= 0) stats_flush(acc, wsum, tot + cur_group * 128, q, lane);
      // every CTA publishes a row for every group (zeros for a group it never saw): cstp_bn_finalize sums all blocks
      for (int g = 0; g < p.stats_groups; ++g)
        p.stats[((static_cast<long long>(blockIdx.x) * p.stats_groups + g) * 2 + (row >> 6)) * p.Np + (row & 63)] =
            tot[g * 128 + row];
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

struct cstp_conv_halo_plan {
  cstp::ConvHaloKParams kp;
  dim3 grid;
  int smem_bytes;
};

using namespace cstp;

extern "C" int cstp_conv_halo_plan_create(const cstp_conv_halo_desc* d, cstp_conv_halo_plan** out_plan) {
  CSTP_REQUIRE(d != nullptr && out_plan != nullptr);
  CSTP_REQUIRE(d->n_groups >= 1 && d->n_groups <= kHcMaxGroups);
  CSTP_REQUIRE(d->n_taps >= 1 && d->n_taps <= kHcMaxTaps);
  CSTP_REQUIRE(d->a_channels >= 16 && d->a_channels % 16 == 0);
  CSTP_REQUIRE(d->Np >= 16 && d->Np % 16 == 0);
  CSTP_REQUIRE(d->n_tile >= 16 && d->n_tile % 16 == 0 && d->n_tile <= 256);
  CSTP_REQUIRE(d->Ktot >= 64 && d->Ktot % 64 == 0);
  CSTP_REQUIRE(d->bw >= 1 && d->bh >= 1 && d->bt >= 1 && d->bn >= 1 && d->bw * d->bh * d->bt * d->bn == 128);
  CSTP_REQUIRE(d->halo_w >= 0 && d->halo_h >= 0 && d->halo_t >= 0);
  CSTP_REQUIRE(d->Wt >= 1 && d->Ht >= 1 && d->Tt >= 1 && d->Nt >= 1);
  CSTP_REQUIRE(d->w_packed != nullptr && (d->out_bf16 != nullptr || d->out_f32 != nullptr));
  CSTP_REQUIRE(d->osw % 8 == 0 && d->osh % 8 == 0 && d->ost % 8 == 0 && d->osn % 8 == 0 && d->out_off % 8 == 0);
  const int xrows = (d->bw + d->halo_w) * (d->bh + d->halo_h) * (d->bt + d->halo_t) * d->bn;
  CSTP_REQUIRE(d->bw + d->halo_w <= 256 && d->bh + d->halo_h <= 256 && d->bt + d->halo_t <= 256);
  // atom pitch: 8 rows when a tap's 128 rows are contiguous in the staged box (halo along the slowest tile axes only);
  // a halo along w breaks the rows into runs of bw, which must then be exactly one 8-row atom each
  const int pitch = d->atom_pitch_rows > 0 ? d->atom_pitch_rows : 8;
  CSTP_REQUIRE(pitch >= 8 && pitch <= 64);
  CSTP_REQUIRE(d->halo_w == 0 ? (pitch == 8 && xrows % 8 == 0) : (d->bw == 8 && pitch == d->bw + d->halo_w));
  const bool xform = d->pro.scale != nullptr;
  const int G = d->slabs.n_slabs > 1 ? d->slabs.n_slabs : 0;
  if (G) {
    // slab mode: taps[] lists, for every w tap j, the nslots stacked weight blocks (tap offset along h DEscending);
    // groups[0] is the origin of the first input slab; one tile = 128 positions x G output rows
    const cstp_halo_slabs& sl = d->slabs;
    if (sl.axis != 1 || xform || d->stats_partials != nullptr)
      return fail_inval("slab mode runs along h (axis 1) without an operand prologue or fused statistics");
    CSTP_REQUIRE(sl.nslots >= 1 && sl.nslots <= 4 && d->n_taps % sl.nslots == 0);
    CSTP_REQUIRE(G + sl.nslots - 1 <= kHcMaxSlabs && d->n_groups == 1 && d->groups[0].n_taps == d->n_taps);
    CSTP_REQUIRE(d->Np % 16 == 0 && d->n_tile == G * d->Np && d->n_tile <= 256 && sl.nslots * d->Np <= 256);
    CSTP_REQUIRE(d->bh == 1 && d->halo_h == 0);
    CSTP_REQUIRE(d->allow_resident && d->bias == nullptr && d->out_f32 == nullptr);
  }
  if (xform) {
    // the prologue picks its coefficient row per tile: one sample per tile, the statistics groups split the N axis evenly
    CSTP_REQUIRE(d->pro.shift != nullptr && (d->pro.groups == 1 || d->pro.groups == 2) && d->Nt % d->pro.groups == 0);
    CSTP_REQUIRE(d->pro.Cp == d->a_channels && (d->Nt / d->pro.groups) % d->bn == 0);    // a tile's samples share one group
    CSTP_REQUIRE(reinterpret_cast<uintptr_t>(d->pro.scale) % 16 == 0 && reinterpret_cast<uintptr_t>(d->pro.shift) % 16 == 0);
  }

  cstp_conv_halo_plan* plan = new (std::nothrow) cstp_conv_halo_plan();
  if (!plan) {
    set_error("out of host memory");
    return CSTP_ENOMEM;
  }
  ConvHaloKParams& k = plan->kp;
  memset(&k, 0, sizeof(k));
  {
    uint64_t dims[5], strides[4];
    for (int i = 0; i < 5; ++i) dims[i] = static_cast<uint64_t>(d->amap.dims[i]);
    for (int i = 0; i < 4; ++i) strides[i] = static_cast<uint64_t>(d->amap.strides[i]);
    bool ok = d->amap.ptr != nullptr && (reinterpret_cast<uintptr_t>(d->amap.ptr) % 16) == 0;
    for (int i = 0; i < 5; ++i) ok = ok && d->amap.dims[i] > 0;
    for (int i = 0; i < 4; ++i) ok = ok && d->amap.strides[i] > 0 && d->amap.strides[i] % 16 == 0;
    if (!ok) {
      delete plan;
      return fail_inval("amap: dims > 0, strides positive multiples of 16 bytes, ptr 16B aligned");
    }
    const uint32_t abox[5] = {64u, (uint32_t)(d->bw + d->halo_w), (uint32_t)(d->bh + d->halo_h),
                              (uint32_t)(d->bt + d->halo_t), (uint32_t)d->bn};
    int rc = encode_tmap_bf16(&k.amap, d->amap.ptr, 5, dims, strides, abox, 128, xform);
    if (rc == CSTP_OK) {
      const uint64_t bdims[2] = {(uint64_t)d->Ktot, (uint64_t)d->Np};
      const uint64_t bstr[1] = {(uint64_t)d->Ktot * 2};
      const uint32_t bbox[2] = {64u, (uint32_t)(G ? d->Np : d->n_tile)};
      rc = encode_tmap_bf16(&k.bmap, d->w_packed, 2, bdims, bstr, bbox);
    }
    // channel tail: exactly 16 or 32 channels beyond a multiple of 64 get their own narrow (32 / 64-byte row) boxes
    const int tail = d->a_channels % 64;
    k.tail = (d->use_tail_boxes && (tail == 16 || tail == 32) && d->a_channels > 64) ? tail : 0;
    if (rc == CSTP_OK && k.tail) {
      const uint32_t abox_t[5] = {(uint32_t)k.tail, abox[1], abox[2], abox[3], abox[4]};
      rc = encode_tmap_bf16(&k.amap_tail, d->amap.ptr, 5, dims, strides, abox_t, k.tail * 2, xform);
      if (rc == CSTP_OK) {
        const uint64_t bdims[2] = {(uint64_t)d->Ktot, (uint64_t)d->Np};
        const uint64_t bstr[1] = {(uint64_t)d->Ktot * 2};
        const uint32_t bbox_t[2] = {(uint32_t)k.tail, (uint32_t)(G ? d->Np : d->n_tile)};
        rc = encode_tmap_bf16(&k.bmap_tail, d->w_packed, 2, bdims, bstr, bbox_t, k.tail * 2);
      }
    } else if (rc == CSTP_OK) {
      k.amap_tail = k.amap;
      k.bmap_tail = k.bmap;
    }
    if (rc != CSTP_OK) {
      delete plan;
      return rc;
    }
  }
  k.step_h = G ? G : d->bh;
  k.tiles_w = ceil_div(d->Wt, d->bw);
  k.tiles_h = ceil_div(d->Ht, k.step_h);
  k.tiles_t = ceil_div(d->Tt, d->bt);
  k.tiles_n = ceil_div(d->Nt, d->bn);
  k.bw = d->bw; k.bh = d->bh; k.bt = d->bt; k.bn = d->bn;
  k.Wt = d->Wt; k.Ht = d->Ht; k.Tt = d->Tt; k.Nt = d->Nt;
  k.n_groups = d->n_groups;
  k.n_taps = d->n_taps;
  k.chunks = ceil_div(d->a_channels, 64);
  k.last_ksteps = ((d->a_channels - 1) % 64) / 16 + 1;
  k.n_tile = d->n_tile;
  k.Np = d->Np;
  k.a_bytes = static_cast<uint32_t>(xrows) * 128u;
  k.a_stride = (k.a_bytes + 1023u) & ~1023u;
  k.a_sbo = static_cast<uint32_t>(pitch) * 128u;
  const uint32_t b_rows = static_cast<uint32_t>(G ? d->Np : d->n_tile);      // rows of one staged weight block
  k.b_bytes = b_rows * 128u;
  k.a_bytes_tail = static_cast<uint32_t>(xrows) * static_cast<uint32_t>(k.tail) * 2u;
  k.b_bytes_tail = b_rows * static_cast<uint32_t>(k.tail) * 2u;
  k.tap_bytes = k.tail ? static_cast<uint32_t>(k.chunks - 1) * k.b_bytes + k.b_bytes_tail
                       : static_cast<uint32_t>(k.chunks) * k.b_bytes;
  {
    // resident weight blocks: classic [tap][chunk], slab mode [chunk][w tap][slot] (the stacked blocks of one w tap are
    // consecutive rows of ONE K-major operand)
    const uint32_t full_chunks = static_cast<uint32_t>(k.tail ? k.chunks - 1 : k.chunks);
    if (G) {
      k.res_tap_stride = k.b_bytes;
      k.res_chunk_stride = static_cast<uint32_t>(d->n_taps) * k.b_bytes;
      k.res_tail_base = full_chunks * k.res_chunk_stride;
      k.res_tail_tap_stride = k.b_bytes_tail;
    } else {
      k.res_tap_stride = k.tap_bytes;
      k.res_chunk_stride = k.b_bytes;
      k.res_tail_base = full_chunks * k.b_bytes;
      k.res_tail_tap_stride = k.tap_bytes;
    }
  }
  if (G) {
    const cstp_halo_slabs& sl = d->slabs;
    const int span = sl.nslots - 1, n_in = G + span;
    k.slab_g = G;
    k.slab_in = n_in;
    k.slab_nslots = sl.nslots;
    k.slab_cols = d->Np;
    // input slab s feeds the output slabs o = max(0, s - span) .. min(G - 1, s) with the taps s - o (descending):
    // stacked blocks (span - s + o_lo) ..; the slabs that cover disjoint column ranges and together all G x Np columns
    // (s = span, span + nslots, ...) go first and overwrite the accumulator
    int order[kHcMaxSlabs], n_ord = 0, covered = 0;
    bool used[kHcMaxSlabs] = {false};
    while (covered < G) {
      int s = covered + span;                         // its lowest output slab is `covered`
      if (s > n_in - 1) s = n_in - 1;
      int o_lo = s - span > 0 ? s - span : 0;
      if (o_lo != covered) {                          // cannot happen: s - span == covered unless clamped to the last slab
        delete plan;
        return fail_inval("slab mode: no overwrite cover of the accumulator");
      }
      order[n_ord++] = s;
      used[s] = true;
      covered = (s < G - 1 ? s : G - 1) + 1;
    }
    const int n_init = n_ord;
    for (int s = 0; s < n_in; ++s)
      if (!used[s]) order[n_ord++] = s;
    for (int i = 0; i < n_in; ++i) {
      const int s = order[i];
      const int o_lo = s - span > 0 ? s - span : 0, o_hi = s < G - 1 ? s : G - 1;
      k.slab_order[i] = s;
      k.slab_init[i] = i < n_init ? 1 : 0;
      k.slab_doff[i] = o_lo * d->Np;
      k.slab_brow[i] = (span - s + o_lo) * d->Np;
      k.slab_idesc[i] = umma_idesc_bf16(128, static_cast<uint32_t>((o_hi - o_lo + 1) * d->Np), 0, 0);
    }
  }
  k.idesc = umma_idesc_bf16(128, static_cast<uint32_t>(d->n_tile), 0, 0);
  k.accumulate = d->accumulate;
  k.out = reinterpret_cast<__nv_bfloat16*>(d->out_bf16);
  k.out_f32 = d->out_f32;
  k.bias = d->bias;
  k.out_off = d->out_off; k.osw = d->osw; k.osh = d->osh; k.ost = d->ost; k.osn = d->osn;
  k.fast_store = d->out_bf16 != nullptr && d->out_f32 == nullptr && d->bias == nullptr &&
                 reinterpret_cast<uintptr_t>(d->out_bf16) % 32 == 0 && d->out_off % 16 == 0 && d->osw % 16 == 0 &&
                 d->osh % 16 == 0 && d->ost % 16 == 0 && d->osn % 16 == 0 && d->n_tile % 16 == 0;
  k.stats = d->stats_partials;
  k.stats_groups = d->stats_groups;
  k.pro_scale = d->pro.scale;
  k.pro_shift = d->pro.shift;
  k.pro_groups = d->pro.groups;
  k.pro_cp = d->pro.Cp;
  if (d->stats_partials != nullptr &&
      !(k.fast_store && !d->accumulate && d->Np == 64 && d->n_tile == 64 &&
        (d->stats_groups == 1 || d->stats_groups == 2) && d->Nt % d->stats_groups == 0 &&
        (d->Nt / d->stats_groups) % d->bn == 0)) {
    delete plan;
    return fail_inval("fused statistics need Np == 64 (one 64-column tile), a plain aligned bf16 output and 1 or 2 groups "
                      "dividing N into multiples of bn");
  }
  const int stats_bytes = d->stats_partials != nullptr ? 3072 : 0;
  const int xtab_bytes = xform ? static_cast<int>(xform_table_bytes(d->pro.groups, d->pro.Cp)) : 0;
  int max_group_taps = 0, seen = 0;
  for (int g = 0; g < d->n_groups; ++g) {
    const cstp_halo_group& gr = d->groups[g];
    if (gr.n_taps < 1 || gr.first_tap != seen) {
      delete plan;
      return fail_inval("groups must partition the tap list in order");
    }
    seen += gr.n_taps;
    if (gr.n_taps > max_group_taps) max_group_taps = gr.n_taps;
    k.groups[g] = HcGroup{gr.dw, gr.dh, gr.dt, gr.first_tap, gr.n_taps};
  }
  if (seen != d->n_taps) {
    delete plan;
    return fail_inval("groups must cover every tap");
  }
  for (int t = 0; t < d->n_taps; ++t) {
    const cstp_halo_tap& tp = d->taps[t];
    if (tp.a_shift % (pitch == 8 ? 1024u : 128u) != 0 || tp.a_shift + 15u * k.a_sbo + 1024u > k.a_bytes || tp.k_off < 0 ||
        tp.k_off % 64 != 0 ||
        tp.k_off + k.chunks * 64 > d->Ktot) {
      delete plan;
      return fail_inval("tap a_shift (whole atoms, or whole rows with a w halo; 128 rows inside the staged box) / k_off out of range");
    }
    k.taps[t] = HcTap{tp.a_shift, tp.k_off};
  }
  if (G) {
    // slab mode: taps[j * nslots + slot] share the w shift j * sw (whole rows of the staged box)
    const int ns = d->slabs.nslots, nwt = d->n_taps / ns;
    const uint32_t sw = nwt > 1 ? d->taps[ns].a_shift : 0u;
    bool ok = k.fast_store != 0;
    for (int t = 0; t < d->n_taps; ++t) ok = ok && d->taps[t].a_shift == static_cast<uint32_t>(t / ns) * sw;
    if (!ok) {
      delete plan;
      return fail_inval("slab mode: taps must be listed w tap by w tap (equal shifts within one w tap), plain aligned bf16 output");
    }
    k.group_taps = d->n_taps;
    k.tap_nw = nwt;
    k.tap_sw = sw;
    k.tap_sh = 0;
  } else
  // the issuer walks the taps of a group arithmetically: derive (nw, sw, sh) from the first group and hold every group to it
  {
    const cstp_halo_group& g0 = d->groups[0];
    const uint32_t base0 = d->taps[g0.first_tap].a_shift;
    uint32_t sw = g0.n_taps > 1 ? d->taps[g0.first_tap + 1].a_shift - base0 : 0u;
    int nw = g0.n_taps;
    for (int j = 1; j < g0.n_taps; ++j)
      if (d->taps[g0.first_tap + j].a_shift - base0 != static_cast<uint32_t>(j) * sw) {
        nw = j;
        break;
      }
    const uint32_t sh = nw < g0.n_taps ? d->taps[g0.first_tap + nw].a_shift - base0 : 0u;
    bool regular = base0 == 0;
    for (int g = 0; g < d->n_groups && regular; ++g)
      for (int j = 0; j < d->groups[g].n_taps; ++j)
        regular = regular && d->taps[d->groups[g].first_tap + j].a_shift ==
                                 static_cast<uint32_t>(j % nw) * sw + static_cast<uint32_t>(j / nw) * sh;
    if (!regular) {
      delete plan;
      return fail_inval("tap shifts of a load group must form a regular (w, h) walk starting at 0");
    }
    for (int g = 0; g < d->n_groups; ++g) regular = regular && d->groups[g].n_taps == d->groups[0].n_taps;
    if (!regular) {
      delete plan;
      return fail_inval("load groups must hold the same number of taps");
    }
    k.group_taps = d->groups[0].n_taps;
    k.tap_nw = nw;
    k.tap_sw = sw;
    k.tap_sh = sh;
  }
  // shared-memory plan: resident weights when every K-block of this N tile fits beside >= 3 activation stages
  const int bar_bytes = 256;
  const long long res_all = 1LL * d->n_taps * k.tap_bytes;
  const long long budget = kSmemBudget - 1024 - bar_bytes - stats_bytes - xtab_bytes;
  k.xtab_off = static_cast<uint32_t>(bar_bytes + stats_bytes);
  if (d->allow_resident && res_all + (pitch == 8 ? 3LL : 2LL) * k.a_stride <= budget) {
    k.resident = 1;
    k.res_bytes = static_cast<uint32_t>(res_all);
    k.stage_bytes = k.a_stride;
  } else {
    k.resident = 0;
    k.res_bytes = 0;
    k.stage_bytes = k.a_stride + static_cast<uint32_t>(max_group_taps) * k.b_bytes;
  }
  int stages = static_cast<int>((budget - k.res_bytes) / k.stage_bytes);
  if (stages > kHcMaxStages) stages = kHcMaxStages;
  if (stages < 2) {
    delete plan;
    return fail_inval("stage too large for the shared-memory pipeline");
  }
  if (G && !k.resident) {
    delete plan;
    return fail_inval("slab mode needs the weights resident in shared memory");
  }
  k.stages = stages;
  int cols = 32;
  while (cols < 2 * d->n_tile) cols *= 2;
  k.tmem_cols = cols;
  plan->smem_bytes = 1024 + static_cast<int>(k.res_bytes) + stages * static_cast<int>(k.stage_bytes) + bar_bytes + stats_bytes +
                     xtab_bytes;
  if (plan->smem_bytes < 120 * 1024) plan->smem_bytes = 120 * 1024;  // keep one CTA per SM (TMEM ownership)
  const int n_ntiles = ceil_div(d->Np, d->n_tile);
  const long long m_tiles = 1LL * k.tiles_w * k.tiles_h * k.tiles_t * k.tiles_n;
  long long gx = num_sms() / n_ntiles;
  if (gx < 1) gx = 1;
  if (gx > m_tiles) gx = m_tiles;
  plan->grid = dim3(static_cast<unsigned>(gx), static_cast<unsigned>(n_ntiles), 1);
  *out_plan = plan;
  return CSTP_OK;
}

extern "C" int cstp_conv_halo_plan_resident(const cstp_conv_halo_plan* plan) { return plan ? plan->kp.resident : CSTP_EINVAL; }
extern "C" int cstp_conv_halo_plan_stat_blocks(const cstp_conv_halo_plan* plan) {
  return plan ? (plan->kp.stats != nullptr ? static_cast<int>(plan->grid.x) : 0) : CSTP_EINVAL;
}


extern "C" int cstp_conv_halo_plan_run(const cstp_conv_halo_plan* plan, void* stream) {
  CSTP_REQUIRE(plan != nullptr);
  static bool attr_set = false;
  if (!attr_set) {
    CSTP_CUDA(cudaFuncSetAttribute(conv_halo_kernel<false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, kHcSmemLimit));
    CSTP_CUDA(cudaFuncSetAttribute(conv_halo_kernel<true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, kHcSmemLimit));
    CSTP_CUDA(cudaFuncSetAttribute(conv_halo_kernel<false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, kHcSmemLimit));
    CSTP_CUDA(cudaFuncSetAttribute(conv_halo_kernel<true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, kHcSmemLimit));
    attr_set = true;
  }
  const cudaStream_t st = static_cast<cudaStream_t>(stream);
  const bool stats = plan->kp.stats != nullptr, xform = plan->kp.pro_scale != nullptr;
  const int threads = xform ? kHcThreads + kHcXformThreads : kHcThreads;
  if (stats && xform) conv_halo_kernel<true, true><<<plan->grid, threads, plan->smem_bytes, st>>>(plan->kp);
  else if (stats) conv_halo_kernel<true, false><<<plan->grid, threads, plan->smem_bytes, st>>>(plan->kp);
  else if (xform) conv_halo_kernel<false, true><<<plan->grid, threads, plan->smem_bytes, st>>>(plan->kp);
  else conv_halo_kernel<false, false><<<plan->grid, threads, plan->smem_bytes, st>>>(plan->kp);
  CSTP_LAUNCHED();
  return CSTP_OK;
}

extern "C" void cstp_conv_halo_plan_destroy(cstp_conv_halo_plan* plan) { delete plan; }

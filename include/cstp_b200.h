/*
 * cstp_b200 C ABI -- the drop-in boundary of the B200-native CSTP `r21d_byol` pretraining hot path.
 *
 * The reference (KT27-A/CSTP) is pure Python/PyTorch and has no FFI of its own: every entry point below
 * replaces a PyTorch library op that the reference invokes at the cited call site (paths relative to the
 * reference repo).  Conventions:
 *   - extern "C", plain pointers and sizes only; all tensors are caller-owned DEVICE pointers.
 *   - every function returns 0 on success, <0 (CSTP_E*) on failure; cstp_last_error() gives the message
 *     (thread-local).  No function synchronises the device; every launch goes to the `stream` argument
 *     (a cudaStream_t passed as void*).
 *   - "plans" hold host-encoded TMA descriptors and launch geometry; they own no device memory.
 *   - activations are NDHWC bf16 with the channel count padded to a multiple of 16 ("Cp").
 */
#ifndef CSTP_B200_H_
#define CSTP_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CSTP_OK 0
#define CSTP_EINVAL (-1)  /* bad argument / unsupported geometry */
#define CSTP_ECUDA (-2)   /* CUDA runtime / driver error */
#define CSTP_ENOMEM (-3)

#define CSTP_MAX_AMAPS 4
#define CSTP_MAX_TAPS 32
#define CSTP_MAX_MCHUNKS 96

const char* cstp_last_error(void);
int cstp_version(void);
/* Number of kernels this library has launched since load (all entry points; for bench.py `gpu_launches`). */
long long cstp_launch_count(void);

/* A 5-D view (C, W, H, T, N) of an NDHWC bf16 tensor, possibly a stride-parity sub-lattice of it.
 * dims[0] is the channel extent; strides[i] is the BYTE stride of dims[i+1]. */
typedef struct {
  const void* ptr;
  int32_t dims[5];
  int64_t strides[4];
} cstp_tensor5;

/* One filter tap of an implicit GEMM: which A view it reads, the (w,h,t) offset added to the tile origin,
 * and the column (K) offset of its first 64-channel chunk inside the packed weight matrix. */
typedef struct {
  int32_t map_id;
  int32_t dw, dh, dt;
  int32_t k_off;
} cstp_tap;

/* Optional operand prologue of the conv-forward and weight-gradient kernels: the activation operand is the RAW output
 * of the producing convolution and the kernel applies the producer's BatchNorm affine map and ReLU,
 *   a = bf16(max(raw * scale[g][c] + shift[g][c], 0)),
 * to the TMA-staged tiles in shared memory before the tensor cores read them -- bit for bit the tensor cstp_bn_apply
 * (relu = 1, no residual) would have written, which then never exists in HBM (conv -> bn -> relu -> conv,
 * models/pace/r21d_byol.py:94-97).  scale / shift: fp32 [groups][Cp] as cstp_bn_finalize / cstp_bn_eval_coeffs write
 * them (zero for padded channels); `groups` (1 or 2) equal parts of the operand's N axis use their own rows.  The
 * convolution's zero padding stays exactly zero.  scale == NULL: the operand is used as it is. */
typedef struct {
  const float* scale;
  const float* shift;
  int32_t groups;
  int32_t Cp;
} cstp_prologue;

/* ---- implicit-GEMM convolution / linear: forward and dgrad ---------------------------------------------
 * Replaces nn.Conv3d forward (models/pace/r21d_byol.py:81-82,91-92,94-97) and its autograd dgrad
 * (main_byol.py:87), and nn.Linear forward/dgrad (r21d_byol.py:236-239,250-253,276-291).
 * D[m, n] = sum_taps sum_c A[pos(m)+tap, c] * Wp[n, tap.k_off + c]   (+ bias[n]) (+ previous out if accumulate)
 * M tiles are boxes (bw,bh,bt,bn) of 128 positions in the (Wt,Ht,Tt,Nt) tile space; out-of-range taps read 0. */
typedef struct {
  int32_t n_amaps;
  cstp_tensor5 amap[CSTP_MAX_AMAPS];
  int32_t a_channels;           /* padded channel count of A (multiple of 16) */
  int32_t n_taps;
  cstp_tap taps[CSTP_MAX_TAPS];
  const void* w_packed;         /* bf16 [Np][Ktot], K-major */
  int32_t Np;                   /* padded output channels (multiple of 16) */
  int32_t Ktot;                 /* packed K extent (multiple of 64) */
  int32_t n_tile;               /* N per tile: multiple of 16, <= 256 */
  int32_t Wt, Ht, Tt, Nt;       /* tile-space extents */
  int32_t bw, bh, bt, bn;       /* box: bw*bh*bt*bn == 128 */
  void* out_bf16;               /* may be NULL */
  float* out_f32;               /* may be NULL */
  int64_t out_off;              /* element offset of tile-space origin */
  int64_t osw, osh, ost, osn;   /* element strides of the tile-space axes in `out` */
  const float* bias;            /* fp32 [Np] or NULL */
  int32_t accumulate;           /* 1: out += D (read-modify-write) */
  cstp_prologue pro;            /* BatchNorm + ReLU applied to A on the way in (scale NULL: none) */
  /* Tap classes (0 or 1: one class holding every tap).  A strided convolution's dgrad is one implicit GEMM per
   * stride-parity class of dx, each with its own taps and output origin but the same tile space: n_classes > 1 runs them
   * as ONE launch -- class c covers taps [cls_first_tap[c], + cls_n_taps[c]) and writes at cls_out_off[c] (out_off is
   * ignored); the classes of one M tile run on neighbouring CTAs at the same time, so the activation boxes they share
   * come from L2 once. */
  int32_t n_classes;
  int32_t cls_first_tap[8];
  int32_t cls_n_taps[8];
  int64_t cls_out_off[8];
} cstp_conv_desc;

typedef struct cstp_conv_plan cstp_conv_plan;
int cstp_conv_plan_create(const cstp_conv_desc* desc, cstp_conv_plan** plan);
int cstp_conv_plan_run(const cstp_conv_plan* plan, void* stream);
/* CTAs per thread-block cluster the plan launches with: 1, or 2 (CTA pairs, each weight tile multicast into both shared
 * memories; chosen when the persistent grid is full). */
int cstp_conv_plan_cluster(const cstp_conv_plan* plan);
void cstp_conv_plan_destroy(cstp_conv_plan* plan);

/* Stride-1 1xkxk / kx1x1 convolutions with a large spatial extent: the activation box is staged once per "load group"
 * with a halo along the tap axis and every tap of the group is a row shift (`a_shift` bytes, whole 8-row swizzle
 * atoms) of that box; weights stay resident in shared memory when they fit (csrc/conv_halo.cu).  Same math and
 * output conventions as cstp_conv_desc; taps must be listed group by group. */
typedef struct {
  int32_t dw, dh, dt;          /* origin of the staged box relative to the tile origin */
  int32_t first_tap, n_taps;
} cstp_halo_group;

typedef struct {
  uint32_t a_shift;
  int32_t k_off;
} cstp_halo_tap;

/* "Slab mode" for layers with few output channels (Np <= 64): n_slabs = G > 1 consecutive output slabs along h
 * (`axis` must be 1) share one accumulator of n_tile = G * Np columns.  Every input slab of the tile (G + nslots - 1 of
 * them, the first at the origin groups[0]) is staged once and multiplied, per w tap, with the stacked weight blocks of the
 * output slabs it feeds: a 128 x 64 x 16 tcgen05.mma is bound by the shared-memory read of its A slice, an MMA of 2 - 3 x 64
 * columns is not.  taps[] then lists, w tap by w tap, the nslots taps along h in DEscending offset order; the tile covers
 * bw*bh*bt*bn == 128 positions with bh == 1.  Needs resident weights, a plain bf16 output, no prologue, no fused
 * statistics. */
typedef struct {
  int32_t n_slabs;              /* 0 / 1: off */
  int32_t axis;                 /* 1 (h) */
  int32_t nslots;
} cstp_halo_slabs;

typedef struct {
  cstp_tensor5 amap;
  int32_t a_channels;
  int32_t n_groups;
  cstp_halo_group groups[4];
  int32_t n_taps;
  cstp_halo_tap taps[16];
  const void* w_packed;
  int32_t Np, Ktot, n_tile;
  int32_t Wt, Ht, Tt, Nt;
  int32_t bw, bh, bt, bn;       /* product == 128 */
  int32_t halo_w, halo_h, halo_t;
  void* out_bf16;
  float* out_f32;
  int64_t out_off;
  int64_t osw, osh, ost, osn;
  const float* bias;
  int32_t accumulate;
  int32_t allow_resident;
  /* 1: when a_channels is 16 or 32 beyond a multiple of 64, stage that channel tail (activations and weights) as boxes
   * with 32 / 64-byte rows (TMA + UMMA 32B / 64B swizzle) instead of zero-padded 128-byte rows. */
  int32_t use_tail_boxes;
  /* Rows between consecutive 8-row atoms of one tap's 128 rows inside the staged box.  0 / 8: the rows are contiguous
   * (halo only along the slower tile axes, a_shift in whole 1024-byte atoms).  bw + halo_w with bw == 8: the box also
   * carries a halo along w (all k x k taps of a 1 x k x k filter read ONE staged box; a_shift in whole 128-byte rows). */
  int32_t atom_pitch_rows;
  /* Optional fused BatchNorm statistics of the stored (bf16-rounded) output (replaces a cstp_bn_stats pass over it):
   * stats_groups (1 or 2) equal parts of the N axis are separate statistics groups; fp32
   * [stat_blocks][stats_groups][2: sum, sum of squares][Np], the partials layout cstp_bn_finalize consumes with
   * nblocks = cstp_conv_halo_plan_stat_blocks.  Needs a single 64-column N tile (Np == n_tile == 64), bn == 1, a plain
   * bf16 output: every epilogue thread keeps the sums of its row's 64 columns in registers. */
  int32_t stats_groups;
  float* stats_partials;
  cstp_prologue pro;            /* BatchNorm + ReLU applied to A on the way in (scale NULL: none) */
  cstp_halo_slabs slabs;        /* n_slabs <= 1: classic tiles */
} cstp_conv_halo_desc;

typedef struct cstp_conv_halo_plan cstp_conv_halo_plan;
int cstp_conv_halo_plan_create(const cstp_conv_halo_desc* desc, cstp_conv_halo_plan** plan);
int cstp_conv_halo_plan_stat_blocks(const cstp_conv_halo_plan* plan);   /* 0: no fused statistics */
int cstp_conv_halo_plan_resident(const cstp_conv_halo_plan* plan);   /* 1 when the weights are kept in shared memory */
int cstp_conv_halo_plan_run(const cstp_conv_halo_plan* plan, void* stream);
void cstp_conv_halo_plan_destroy(cstp_conv_halo_plan* plan);

/* ---- weight gradient ------------------------------------------------------------------------------------
 * Replaces the autograd wgrad of nn.Conv3d / nn.Linear (main_byol.py:87).
 * The M axis is a list of 64-row chunks, each one (tap, 64 input channels) of the conv input X; the N axis
 * is the output-channel axis of G = dL/d(conv output); K runs over all output positions:
 *   P[split][chunk*64 + r][n] = sum_{pos in split} X[pos + tap(chunk), c_off(chunk) + r] * G[pos, n]
 * cstp_wgrad_finalize then reduces the splits in fixed order and scatters into the reference weight layout. */
typedef struct {
  int32_t map_id;
  int32_t dw, dh, dt;
  int32_t c_off;
} cstp_mchunk;

typedef struct {
  int32_t n_amaps;
  cstp_tensor5 amap[CSTP_MAX_AMAPS];   /* views of X */
  int32_t n_mchunks;
  cstp_mchunk mchunks[CSTP_MAX_MCHUNKS];
  cstp_tensor5 gmap;                    /* view of G */
  int32_t Np;                           /* padded G channels (multiple of 16) */
  int32_t n_tile;                       /* multiple of 16, <= 256 */
  int32_t Wt, Ht, Tt, Nt;               /* position space */
  int32_t bw, bh, bt, bn;               /* box: product == 64 */
  int32_t splits;                       /* requested split-K factor (>=1) */
  float* partials;                      /* fp32 [splits_eff][n_mchunks*64][Np] */
  cstp_prologue pro;                    /* BatchNorm + ReLU applied to X on the way in (scale NULL: none) */
  int32_t mt_per_cta;                   /* 128-row M tiles per CTA sharing one staged G tile (0 / 1 .. 4; mt_per_cta * n_tile
                                           <= 512 TMEM columns; 1 with a prologue): fewer re-loads of G through L2 */
} cstp_wgrad_desc;

typedef struct cstp_wgrad_plan cstp_wgrad_plan;
int cstp_wgrad_plan_create(const cstp_wgrad_desc* desc, cstp_wgrad_plan** plan);
int cstp_wgrad_plan_splits(const cstp_wgrad_plan* plan);      /* effective split count */
int cstp_wgrad_plan_run(const cstp_wgrad_plan* plan, void* stream);
void cstp_wgrad_plan_destroy(cstp_wgrad_plan* plan);
/* dW[(co*cin + ci)*taps + tap] (+)= sum_s partials[s][row(chunk,ci)][co]; chunk_tap/chunk_coff are DEVICE int32
 * arrays of length n_mchunks (tap index and first input channel of every 64-row chunk). */
int cstp_wgrad_finalize(const float* partials, int splits, int n_mchunks, int Np, const int32_t* chunk_tap,
                        const int32_t* chunk_coff, int cout, int cin, int taps, float* dw, int accumulate,
                        int layout, const int32_t* chunk_splits, void* stream);
/* chunk_splits (DEVICE, may be NULL = `splits` for every chunk): partials of chunk i exist for split < chunk_splits[i].
 * layout 2: the transposed product -- partial rows are (tap, cout) (chunk_coff = first OUTPUT channel of the chunk), the
 * Np columns are the input channels; dW is (cout, cin, taps) as for layout 0.
 * layout 0: dW is (cout, cin, taps) as above.  layout 1 (the stem over cstp_stem_pack row pairs: cin = 64 pixel
 * channels hpar*32 + kw*3 + c, taps = 4 row pairs j): dW is the reference's (cout, 3, 1, 7, 7) tensor, element
 * ((co*3 + c)*7 + kh)*7 + kw with kh = 2*j + hpar - 1; channels / taps outside the filter are skipped. */

/* Weight gradient of the wide, shallow stride-1 layers: every CTA computes all taps for its slice of positions.
 * One K-block (box of 64 positions) stages `n_xboxes` boxes of X, each 64 channels wide and extended by
 * (halo_w, halo_h, halo_t) positions so that the taps of one axis are row shifts of the same shared-memory box, and
 * the G boxes of one N tile.  chunk i of the M axis is the 64 rows found `chunk_off[i]` bytes into the staged X
 * region (1024-byte aligned: whole 8-row swizzle atoms); chunks are paired into 128-row MMAs.  Output partials have
 * the layout of cstp_wgrad_desc (chunk-major rows), so cstp_wgrad_finalize applies unchanged. */
typedef struct {
  int32_t c_off;        /* first channel of the box */
  int32_t dw, dh, dt;   /* offset of the box origin from the K-block origin */
} cstp_xbox;

typedef struct {
  cstp_tensor5 xmap;
  cstp_tensor5 gmap;
  int32_t n_xboxes;
  cstp_xbox xboxes[16];
  int32_t n_chunks;                     /* <= 32 */
  uint32_t chunk_off[32];
  int32_t Np, n_tile;                   /* ceil(n_chunks/2) * n_tile <= 512 TMEM columns */
  int32_t Wt, Ht, Tt, Nt;
  int32_t bw, bh, bt, bn;               /* product == 64 */
  int32_t halo_w, halo_h, halo_t;
  int32_t splits;
  float* partials;                      /* fp32 [splits_eff][n_chunks*64][Np] */
  /* 0 / 8: the 64 positions of a chunk are contiguous box rows (chunk_off in whole 1024-byte atoms).  bw + halo_w with
   * bw == 8: the box carries a halo along w as well (all k x k taps of a 1 x k x k filter read ONE staged box per channel
   * chunk; chunk_off in whole 128-byte rows). */
  int32_t atom_pitch_rows;
  cstp_prologue pro;                    /* BatchNorm + ReLU applied to X on the way in (scale NULL: none) */
  /* M classes: > 0 and < ceil(n_chunks/2): the M tiles are dealt to CTA classes of this many tiles each (the TMEM bound
   * becomes mt_per_class * n_tile <= 512) and `splits` split-K CTAs per N tile are shared out in proportion to the tiles
   * of a class; rows of class c exist for split < its split count (cstp_wgrad_halo_plan_chunk_splits). */
  int32_t mt_per_class;
  /* Operand roles are symmetric: the caller may pass dL/d(raw) as `xmap` (halo, row-shifted chunks: M = (tap, cout)) and
   * the activations as `gmap` (N = cin); pro_on_b != 0 then applies the prologue to the gmap boxes (n_tile % 64 == 0 or one
   * N tile).  The partial rows are then (tap, cout-chunk) and the columns cin: cstp_wgrad_finalize layout 2. */
  int32_t pro_on_b;
} cstp_wgrad_halo_desc;

typedef struct cstp_wgrad_halo_plan cstp_wgrad_halo_plan;
int cstp_wgrad_halo_plan_create(const cstp_wgrad_halo_desc* desc, cstp_wgrad_halo_plan** plan);
int cstp_wgrad_halo_plan_splits(const cstp_wgrad_halo_plan* plan);     /* rows of splits in the partials buffer */
/* out[i] = number of split-K partials that exist for chunk i (differs between M classes). */
int cstp_wgrad_halo_plan_chunk_splits(const cstp_wgrad_halo_plan* plan, int32_t* out, int n_chunks);
int cstp_wgrad_halo_plan_run(const cstp_wgrad_halo_plan* plan, void* stream);
void cstp_wgrad_halo_plan_destroy(cstp_wgrad_halo_plan* plan);

/* ---- packing / layout -----------------------------------------------------------------------------------
 * fp32 reference-layout weight (rows_out, cin, taps) -> bf16 K-major packed [Rp][taps*Kc].
 * transpose=0: packed[r=co][tap*Kc + ci] (forward);  transpose=1: packed[r=ci][tap*Kc + co] (dgrad);
 * transpose=2: the stem's (cout, 3, 1, 7, 7) weight for cstp_stem_pack row pairs (call with cin = 64, taps = 4):
 * packed[co][j*Kc + hpar*32 + kw*3 + c] = w[co][c][0][2*j + hpar - 1][kw], zero where no such filter element exists. */
int cstp_pack_weight(const float* w, int cout, int cin, int taps, int transpose, void* packed, int Rp, int Kc,
                     void* stream);
/* The same for a whole list of tensors in one launch.  jobs_dev: DEVICE int64 [n_jobs][8] = {w ptr, packed ptr, cout,
 * cin, taps, transpose, Rp, Kc}; prefix_dev: DEVICE int64 [n_jobs + 1], prefix[j] = sum of Rp*taps*Kc of the jobs
 * before j; total = prefix[n_jobs]. */
int cstp_pack_weights_batched(const int64_t* jobs_dev, const int64_t* prefix_dev, int n_jobs, int64_t total, void* stream);
/* Stem, packed row pairs: fp32 NCDHW clip (N,3,T,H,W), H and W even -> bf16 P (N,T,H/2,W/2,64) with
 * P[n][t][h2][wo][hpar*32 + kw*3 + c] = x[n][c][t][2*h2 + hpar][2*wo + kw - 3] (zero outside the frame, k = 21..31 of
 * each half zero): the 1x7x7 s(1,2,2) p(0,3,3) convolution (r21d_byol.py:198) becomes a four-tap (1,4,1) stride-1
 * implicit GEMM over P (row pairs ho-2 .. ho+1) whose packed weights come from cstp_pack_weight(s) with transpose = 2
 * and whose weight gradient is scattered by cstp_wgrad_finalize layout 1. */
int cstp_stem_pack(const float* x, int N, int T, int H, int W, void* P, void* stream);
/* Input gradient of the same convolution: g is the stem unit's d(raw), bf16 (N,T,H/2,W/2,Cg) with Cg even and >= cout;
 * w the fp32 (cout, 3, 1, 7, 7) weight (rounded to bf16 on load, as the packed weights of every dgrad are); dx the fp32
 * NCDHW (N,3,T,H,W) clip gradient, overwritten.  dx[n][c][t][h][w] = sum of g[n][t][oh][ow][co] * w[co][c][0][kh][kw]
 * over oh = (h + 3 - kh) / 2, ow = (w + 3 - kw) / 2 integral and in range, summed in a fixed order (channel pairs, kh,
 * kw, channel) with one fmaf per term and no atomics (csrc/stem_dgrad.cu).  H even, W a multiple of 4, cout <= 128,
 * g 4-byte and dx 16-byte aligned. */
int cstp_stem_dgrad(const void* g, int Cg, const float* w, int cout, float* dx, int N, int T, int H, int W,
                    void* stream);

/* ---- BatchNorm (training mode), fused with ReLU / residual ---------------------------------------------
 * Replaces nn.BatchNorm3d / BatchNorm1d forward+backward and the ReLU / residual adds around them
 * (r21d_byol.py:83,95,126,133,138,141-148,199,216).  `groups` splits the rows evenly into independent
 * statistics groups (the two views, which the reference pushes through the net one after the other). */
int cstp_bn_stats(const void* raw, int64_t rows, int Cp, int groups, float* partials, int nblocks, void* stream);
int cstp_bn_finalize(const float* partials, int nblocks, int groups, int64_t rows_per_group, int C, int Cp,
                     const float* gamma, const float* beta, float eps, float momentum, float* running_mean,
                     float* running_var, float* scale, float* shift, float* mean, float* invstd, void* stream);
/* Sums the per-block partials of cstp_bn_stats / cstp_bn_bwd_reduce into one row fp32 [groups][2][Cp]: the payload of
 * the cross-rank all-reduce of world-synchronised BatchNorm; finalize then runs with nblocks = 1 and the global row
 * count. */
int cstp_bn_partials_reduce(const float* partials, int nblocks, int groups, int Cp, float* out, void* stream);
/* out = act(raw*scale+shift + residual); res_mode 0 none, 1 bf16 tensor, 2 raw2*scale2+shift2 (the shortcut is a
 * BatchNorm output, r21d_byol.py:144-145), 3 bf16(relu(raw2*scale2+shift2)) (the shortcut is a BatchNorm + ReLU
 * activation that only exists as its producer's raw output, see cstp_prologue). */
int cstp_bn_apply(const void* raw, int64_t rows, int Cp, int groups, const float* scale, const float* shift,
                  int relu, int res_mode, const void* res, const float* scale2, const float* shift2, void* out,
                  void* stream);
/* dy = d masked by the forward ReLU; partials of sum(dy), sum(dy*raw) per (group, channel) (cstp_bn_bwd_finalize turns
 * the second into sum(dy*xhat)).  The mask is
 * act > 0 when `act` is given (block outputs, whose pre-activation includes the residual), else
 * raw*mask_scale + mask_shift > 0 when the forward affine coefficients are given (no read of act), else none. */
int cstp_bn_bwd_reduce(const void* d, const void* act, const void* raw, int64_t rows, int Cp, int groups,
                       const float* mean, const float* invstd, const float* mask_scale, const float* mask_shift,
                       float* partials, int nblocks, void* stream);
/* Reduces partials; writes dgamma/dbeta (summed over groups, optionally accumulated) and the apply coefficients
 * coef[g][3][Cp] = {gamma*invstd, sum(dy)/n, sum(dy*xhat)/n}. */
int cstp_bn_bwd_finalize(const float* partials, int nblocks, int groups, int64_t rows_per_group, int C, int Cp,
                         const float* gamma, const float* mean, const float* invstd, float* dgamma, float* dbeta,
                         int accumulate, float* coef, void* stream);
/* g = c0*(dy - c1 - xhat*c2) (bf16), same masking as cstp_bn_bwd_reduce; optionally also writes dz = dy. */
int cstp_bn_bwd_apply(const void* d, const void* act, const void* raw, int64_t rows, int Cp, int groups,
                      const float* mean, const float* invstd, const float* coef, const float* mask_scale,
                      const float* mask_shift, void* g, void* dz, void* stream);

/* AdaptiveAvgPool3d(1) over `P` positions (r21d_byol.py:210,222-223) and its backward broadcast.
 * Forward: sample n is written to row n % rows_out, column offset (n / rows_out)*Cp of a row of ld_out elements
 * (rows_out == N: plain [N][Cp]; rows_out == N/2: the cat(feat1, feat2) layout of r21d_byol.py:374).
 * Backward: dx[n][p][:] = (dfeat[n] + dcat[n % rows_cat][(n / rows_cat)*Cp ...]) / P, dcat optional. */
int cstp_avgpool_fwd(const void* x, int N, int P, int Cp, float* out_f32, void* out_bf16, int rows_out, int ld_out,
                     void* stream);
int cstp_avgpool_bwd(const float* dfeat, const float* dcat, int rows_cat, int ld_cat, int N, int P, int Cp, void* dx,
                     void* stream);

/* Column sums of a bf16 [rows][Cp] matrix into fp32 (bias gradients): out[c] (+)= sum_r x[r][c]. */
int cstp_colsum(const void* x, int64_t rows, int Cp, int C, float* out, int accumulate, void* stream);
/* fp32 [rows][ld_in] -> bf16 [rows][ld_out] (zero padded), optional scale read from a device scalar. */
int cstp_cast_pad(const float* x, int64_t rows, int cols, int ld_in, void* out, int ld_out, const float* scale_dev,
                  void* stream);

/* ---- losses ---------------------------------------------------------------------------------------------
 * BYOL regression loss (r21d_byol.py:346-355,382): pred/tproj are fp32 [2B][ld]; rows [0,B) view 1, [B,2B) view 2.
 * loss_out[0] = mean_i[(2-2cos(p1_i,t2_i)) + (2-2cos(p2_i,t1_i))]; dpred = upstream * dloss/dpred
 * (`upstream` is a device scalar, NULL = 1). */
int cstp_byol_loss(const float* pred, const float* tproj, int B, int D, int ld, float* loss_out,
                   const float* upstream, float* dpred, void* stream);
/* Representation (collapse) statistics of one step.  Blocks k = 0..3 are fp32 [2B][ld_k] rows (512 valid columns,
 * ld_k >= 512; NULL = not given, its entries are 0): the online pooled feature, projector, predictor and target projector
 * outputs.  Per view v (rows [vB, (v+1)B)) and block, with every operation rounded on its own, in this order:
 *   n_r = sqrt(ss_r): lane l of a warp adds x[l]^2, x[l+32]^2, ... in order, then an xor butterfly over offsets
 *         16, 8, 4, 2, 1 sums the lanes;  z_rj = x_rj / max(n_r, 1e-12)  (F.normalize);
 *   per column j: d_rj = z_rj - z_0j, m_j = (sum_r d_rj, r ascending) / B, std_j = sqrt((sum_r (d_rj - m_j)^2) / (B - 1));
 *   s = (pairwise tree sum of std_j: a[i] += a[i + h] for h = 256, 128, ..., 1) / 512.
 * out fp32 [2][5]: out[v][k] = s of block k, out[v][4] = (sum_r n_r of block 0, r ascending) / B.  s is about
 * 1/sqrt(512) = 0.0442 for well-spread rows and exactly 0 when the view's rows are equal.  2 <= B <= 8192. */
int cstp_repr_stats(const float* feat, int ld_feat, const float* proj, int ld_proj, const float* pred, int ld_pred,
                    const float* tproj, int ld_tproj, int B, float* out, void* stream);
/* Six nn.CrossEntropyLoss() (mean) over [B][ld] logits with 5 classes + the weighted sum of main_byol.py:63-73.
 * logits[h], labels[h] (int64), dlogits[h] for h in spa, tem, pb1, pb2, rot1, rot2; weights[5] = --loss_weight.
 * losses_out[0..5] = the six CE values, losses_out[6] = weighted sum of them (BYOL term excluded). */
int cstp_pretext_ce(const float* const* logits, const int64_t* const* labels, float* const* dlogits, int B,
                    int n_cls, int ld, const float* weights5, float* losses_out, void* stream);
/* NT-Xent (loss/NTXent.py:46-62), closed form: z = cat(zjs, zis) [rows=2N][d] fp32;
 * loss = mean_i[LSE_{j!=i}(cos_ij/tau) - cos_i,pos(i)/tau]; dz optional (NULL = forward only).
 * use_cosine=0 uses raw dot products.  workspace: 16-byte aligned fp32 scratch of `workspace_floats` elements, at
 * least 3*rows + rows*d; with cstp_ntxent_workspace_floats(rows, d) elements (and rows >= 256, d a multiple of 64,
 * d <= 256) the similarity matrix runs on the tensor cores (bf16 operands, fp32 accumulation and softmax). */
long long cstp_ntxent_workspace_floats(int rows, int d);
int cstp_ntxent(const float* z, int rows, int d, float temperature, int use_cosine, float* loss_out, float* dz,
                float* workspace, long long workspace_floats, void* stream);

/* ---- finetune / test branch (models/pace/r21d_byol.py:394-399, main_ft_mp.py:179-289, test.py:76-93) ----------
 * F.normalize(x, p=2, dim=1): y = x / max(|x|_2, eps) for fp32 [rows][ld] -> bf16 [rows][ld_y] (zero padded); norms kept. */
int cstp_l2norm_fwd(const float* x, int rows, int d, int ld, float eps, void* y_bf16, int ld_y, float* norms, void* stream);
/* dx = (g - y (y.g)) / norm for the bf16 gradient g w.r.t. y. */
int cstp_l2norm_bwd(const float* x, const float* norms, const void* g_bf16, int rows, int d, int ld, int ld_g, float* dx,
                    void* stream);
/* nn.CrossEntropyLoss() (mean) over fp32 [B][ld] logits with n_cls classes and int64 labels; dlogits optional;
 * workspace: fp32 [B]. */
int cstp_ce_loss(const float* logits, const int64_t* labels, int B, int n_cls, int ld, float* loss_out, float* dlogits,
                 float* workspace, void* stream);
/* Eval-mode BatchNorm as the affine map cstp_bn_apply consumes: scale = gamma/sqrt(running_var+eps),
 * shift = beta - running_mean*scale, replicated for `groups` groups. */
int cstp_bn_eval_coeffs(const float* gamma, const float* beta, const float* running_mean, const float* running_var, int C,
                        int Cp, int groups, float eps, float* scale, float* shift, void* stream);
/* Video-level scoring of test.py:76-93 (csrc/video_eval.cu).  A video's clip logits are summed into an fp32 slot
 * sums[slot][n_cls] that keeps accumulating across launches, in clip order (no float atomics: bit-reproducible, equal to a
 * sequential fp32 loop).  Work lists are DEVICE int32 tables the host may rewrite in place between graph replays; an entry
 * whose count is <= 0 (or that points outside the buffers) is skipped.
 * accumulate: seg[n_seg][3] = {slot, first row, row count}; adds rows [first, first + count) of logits (fp32 [rows][ld],
 *   first n_cls columns) to sums[slot].  Rows no entry names are never read. */
int cstp_video_accumulate(const float* logits, int rows, int ld, int n_cls, const int32_t* seg, int n_seg, float* sums,
                          int n_slots, void* stream);
/* finalize: fin[n_fin][3] = {slot, clip count, video}; mean = sums[slot] / count (fp32), optionally written to
 * mean_out[video][n_cls]; topk_out[video][k] (1 <= k <= 8) = class indices by mean, descending, ties to the lower index;
 * with hits: hits[0] += (top-1 == labels[video]), hits[1] += (labels[video] among the top 5) (int64 counters).  The slot
 * is left zero. */
int cstp_video_finalize(float* sums, int n_slots, int n_cls, const int32_t* fin, int n_fin, int n_videos, int k,
                        const int64_t* labels, float* mean_out, int64_t* topk_out, int64_t* hits, void* stream);

/* Nearest-neighbour retrieval (csrc/retrieval.cu).  Defined fp32 arithmetic, no contraction: results are bit-identical
 * for every tiling and split.
 * l2_normalize_rows: y[n][d] = x / max(||x||_2, 1e-12) (F.normalize), x fp32 [n][ld].  The sum of squares is lane-strided
 *   over a warp (lane l adds x[l]^2, x[l+32]^2, ... in order) and then reduced by an xor butterfly over offsets 16, 8, 4,
 *   2, 1; sqrt and the division are correctly rounded. */
int cstp_l2_normalize_rows(const float* x, int n, int d, int ld, float* y, void* stream);
/* knn_partial: q fp32 [nq][d], g fp32 [ng][d] (rows normalised, 16-byte aligned, d % 4 == 0).  s(q, g) is the sequential
 * chain acc = acc + q[j] * g[j], j = 0 .. d-1, each product and sum rounded.  Gallery split s = rows
 * [ng*s/splits, ng*(s+1)/splits); part_val / part_idx [splits][nq][k] receive each split's top-k (similarity descending,
 * then the lower gallery index), empty entries -inf / -1.  1 <= k <= 64, 1 <= splits <= 32; the similarity matrix is
 * never written. */
int cstp_knn_partial(const float* q, int nq, const float* g, int ng, int d, int k, int splits, float* part_val,
                     int32_t* part_idx, void* stream);
/* knn_merge: the splits' lists -> idx_out int64 [nq][k], sim_out fp32 [nq][k] in the same order (-1 / -inf past ng).
 * With hits (then q_labels int64 [nq], g_labels int64 [ng], cutoffs int32 [n_cut], all device): for every cutoff c,
 * hits[c] += (one of the first c neighbours has g_labels == q_labels[i]), int64 counters. */
int cstp_knn_merge(const float* part_val, const int32_t* part_idx, int nq, int k, int splits, int64_t* idx_out,
                   float* sim_out, const int64_t* q_labels, const int64_t* g_labels, const int32_t* cutoffs, int n_cut,
                   int64_t* hits, void* stream);

/* Grad-CAM of a finetuned classifier (csrc/explain.cu).  Every floating-point operation is one rounded _rn intrinsic in
 * a fixed order, so a float32 stand-in reproduces the bits.
 * cam_seed: for rows b < n, k = classes_in[b] (device int64, optional) or the argmax over the n_cls valid columns of
 *   logits fp32 [B][ld] (ties to the lower class); classes_out[b] = k (int64), dlogits[b] = one-hot(k) fp32 [B][ld].
 *   Rows >= n get class 0 and a zero row; padding columns are zero. */
int cstp_cam_seed(const float* logits, int B, int ld, int n, int n_cls, const int64_t* classes_in, int64_t* classes_out,
                  float* dlogits, void* stream);
/* gradcam: act / grad bf16 NDHWC [n][P positions][Cp] (C valid channels, C % 8 == 0, C <= 512, act 16-byte aligned):
 *   alpha[b][c] = (sum_p grad[b][p][c]) / P, the sum in eight interleaved position lanes (lane j: p = j, j + 8, ... in
 *   order) then lane order; cam[b][p] = relu(sum_c alpha[b][c] * act[b][p][c]), rounded products added in channel order.
 *   alpha fp32 [n][C], cam fp32 [n][P].  Two launches. */
int cstp_gradcam(const void* act, const void* grad, int n, long long P, int C, int Cp, float* alpha, float* cam,
                 void* stream);
/* cam_upsample: cam fp32 [n][t][h][w] -> out fp32 [n][T][H][W], trilinear with torch's align_corners=False source index
 *   (per axis: scale = in / out, src = max(scale * (d + 0.5) - 0.5, 0), i0 = (int)src, i1 = min(i0 + 1, in - 1),
 *   l = src - i0; blends a + l * (b - a) along w, then h, then t), then per clip (v - min) / (max - min), zeros where
 *   max == min. */
int cstp_cam_upsample(const float* cam, int n, int t, int h, int w, int T, int H, int W, float* out, void* stream);

/* ---- optimiser side -------------------------------------------------------------------------------------
 * EMA target update (r21d_byol.py:331-337): k = k*m + q*(1-m), bit-exact fp32 (two rounded products, one add). */
int cstp_ema_update(float* k, const float* q, int64_t n, float m, float one_minus_m, void* stream);
/* clip_grad_norm_(params, max_norm) + SGD(momentum, weight_decay) (main_byol.py:88-91,229-232) over flat buffers.
 * norm_out[0] = total grad norm (before clipping), norm_out[1] = clip coefficient. first_step: buf = g. */
int cstp_sgd_clip_step(float* p, const float* g, float* mom, int64_t n, float lr, float momentum, float wd,
                       float max_norm, int do_clip, int first_step, float* norm_out, float* workspace,
                       void* stream);
/* The same with the hyper-parameters read from DEVICE memory at run time, hyper = {lr, momentum, wd, max_norm, do_clip,
 * first_step} (flags: nonzero = set): the launch can sit in a captured CUDA graph while the host follows the per-epoch
 * learning-rate schedule (scheduler/cosine_anneal.py) by rewriting six floats. */
int cstp_sgd_clip_step_dev(float* p, const float* g, float* mom, int64_t n, const float* hyper, float* norm_out,
                           float* workspace, void* stream);
/* Scalars of one Adam / AdamW step, in the form torch.optim.Adam(W) (foreach=False) uses them.  step_size =
 * lr / (1 - beta1^t) and bc2_sqrt = sqrt(1 - beta2^t) are computed by the caller in double, as torch does; so are
 * 1 - beta1, 1 - beta2 and decay.  Adam: l2 = weight_decay, decay = 1.  AdamW: l2 = 0, decay = 1 - lr * weight_decay.
 * Flags: nonzero = set.  Ten floats, so a device copy is a plain float[10]. */
typedef struct {
  float step_size, bc2_sqrt, one_minus_beta1, beta2, one_minus_beta2, eps, l2, decay, max_norm, do_clip;
} cstp_adam_hyper;
/* clip_grad_norm_ (as cstp_sgd_clip_step) + one Adam / AdamW step over flat fp32 buffers p, g, m (exp_avg), v
 * (exp_avg_sq), all 16-byte aligned.  Per element, every operation rounded on its own (no FMA contraction):
 *   g *= coef; p *= decay; g += l2 * p; m += (g - m) * (1 - beta1); v = beta2 * v + ((1 - beta2) * g) * g;
 *   p -= (step_size * m) / (sqrt(v) / bc2_sqrt + eps).
 * norm_out[0] = total grad norm (before clipping), norm_out[1] = clip coefficient. */
int cstp_adam_clip_step(float* p, const float* g, float* m, float* v, int64_t n, cstp_adam_hyper hyper, float* norm_out,
                        float* workspace, void* stream);
/* The same with the scalars read from DEVICE memory at run time: the launch can sit in a captured CUDA graph while the
 * host rewrites the step-dependent scalars before every replay. */
int cstp_adam_clip_step_dev(float* p, const float* g, float* m, float* v, int64_t n, const cstp_adam_hyper* hyper,
                            float* norm_out, float* workspace, void* stream);

/* ---- pretraining clip pipeline (SURVEY.md 8 f-2) -----------------------------------------------------------
 * Replaces the pixel work of the reference's CPU data pipeline for one batch of pretraining samples:
 *   data_process/datasets.py:888-932 (Image.open + Image.transpose(ROTATE_*) per frame),
 *   data_process/preprocess_data.py:514-515,537-562 (crop + resize((112,112), BICUBIC)),
 *   data_process/preprocess_data.py:1112-1122 (RandomRotation -> ColorJitter -> ClipRandomGray -> GaussianBlur ->
 *   horizontal flip -> ToTensor -> Normalize 'tf').
 * Every random decision has been taken on the host (cstp_b200/data_process/clip_plan.py, bit-exact with the reference's
 * draw order); a view descriptor carries them as integers / fixed-point tables, and one launch turns decoded uint8
 * frames resident in HBM into the two fp32 NCDHW clips the model consumes.  The arithmetic is Pillow's, restated in
 * integers (Q22 resampling taps, 16.16 affine walk, Q24 box blur, uint8 HSV), so the output equals the reference's
 * clips bit for bit. */
#define CSTP_CLIP_T 64     /* frames per clip (opts.sample_duration) upper bound */
#define CSTP_CLIP_S 224    /* clip side (opts.sample_size) upper bound */
#define CSTP_CLIP_KMAX 24  /* resampling taps per output pixel upper bound (crop side <= 616 for a 112 output) */
typedef struct {
  const uint8_t* video;  /* device: frame 0 of this sample's decoded video, uint8 [F][H][W][3] */
  float* out;            /* device: this view's clip, fp32 (3, T, S, S) */
  const int32_t* coef;   /* device: [2][S][2 + CSTP_CLIP_KMAX]: x tables, then y tables; per output index: first source
                            index, tap count, Q22 taps (Pillow's precompute_coeffs + normalize_coeffs_8bpc) */
  int32_t W, H;          /* stored frame size */
  int32_t frames[CSTP_CLIP_T];
  int32_t rot;           /* rotation label: frame turned rot x 90 degrees counter-clockwise before cropping */
  int32_t box[4];        /* crop (x0, y0, x1, y1) in the rotated frame; outside pixels read 0 */
  int32_t flip;
  int32_t rotate;        /* 1: Image.rotate(angle), NEAREST, as the 16.16 fixed-point affine walk rot_fix[a0..a5] */
  int32_t rot_fix[6];
  int32_t n_jitter;
  int32_t jitter_op[4];  /* 0 brightness, 1 contrast, 2 saturation, 3 hue -- in application order */
  float jitter_f[4];     /* blend factor of ops 0-2 */
  int32_t hue_shift;     /* uint8 increment of the H channel (op 3) */
  int32_t gray[CSTP_CLIP_T]; /* per frame: -1, or the channel copied into R, G and B */
  int32_t blur;          /* 1: Pillow's 3-pass extended box blur with the parameters below (both axes) */
  int32_t blur_radius, blur_edge_a, blur_edge_b;
  uint32_t blur_ww, blur_fw;
} cstp_clip_view;
/* views: DEVICE array of n_views descriptors; max_crop_h: largest (box[3]-box[1]) among them (sizes the shared-memory
 * staging of the horizontal pass; CSTP_EINVAL when it does not fit).  8 <= S <= CSTP_CLIP_S, T <= CSTP_CLIP_T.
 * One CTA per (frame, view) when the crop rows and two S x S images fit its shared memory, else a thread-block cluster
 * of two CTAs per (frame, view) that splits every staged buffer by rows (see cstp_clip_layout). */
int cstp_clip_assemble(const cstp_clip_view* views, int n_views, int T, int S, int max_crop_h, void* stream);
/* The launch layout cstp_clip_assemble picks for (S, max_crop_h): *cluster = 1 (one CTA holds
 * align16(max_crop_h * S * 3) + 2 * align16(S * S * 3) bytes) or 2 (each CTA of the pair holds
 * align16(max(ceil(max_crop_h / 2), ceil(S / 2)) * S * 3) + align16(ceil(S / 2) * S * 3) bytes); *smem_bytes per CTA.
 * CSTP_EINVAL, naming the crop height, when neither fits 226 KB.  Host only: needs no GPU. */
int cstp_clip_layout(int S, int max_crop_h, int* cluster, int* smem_bytes);

/* ---- JPEG decoding (csrc/jpeg_decode.cu) -------------------------------------------------------------------
 * Baseline / extended-sequential Huffman JPEG (SOF0 / SOF1, 8-bit samples, one interleaved scan; grayscale or YCbCr
 * 4:4:4, 4:2:2 (h2v1), 4:2:0 (h2v2); restart intervals; any size) decoded to RGB uint8 [height][width][3], byte for
 * byte what Pillow on libjpeg-turbo returns for Image.open(...).convert("RGB") (ISLOW IDCT, fancy upsampling).  One call
 * decodes a batch on `stream`: stage A parses and entropy-decodes (one warp per image, one lane per restart interval),
 * stage B runs the IDCT per block, stage C upsamples and converts colour per pixel.  status[i] becomes 0 or one of the
 * codes below; a rejected image leaves its `out` unspecified and touches nothing outside its own stream, output and
 * workspace slice.  Where libjpeg would warn and fill in zeros (corrupt or truncated entropy data), this decoder
 * reports CSTP_JPEG_MALFORMED. */
#define CSTP_JPEG_UNSUPPORTED 1 /* progressive / arithmetic / lossless / hierarchical, 12-bit, CMYK or RGB, other
                                   sampling, several scans, no Huffman table (Motion-JPEG) */
#define CSTP_JPEG_MALFORMED 2   /* truncated or corrupt stream, a missing quantisation table */
#define CSTP_JPEG_SIZE 3        /* SOF size differs from (width, height), or an invalid size / workspace slice */
typedef struct {
  int64_t src_offset, src_bytes; /* this image's stream inside `data` */
  uint8_t* out;                  /* device: RGB uint8 [height][width][3] */
  int32_t width, height;         /* expected size: a stream of another size is rejected */
  int64_t ws_offset;             /* this image's slice of the workspace (a multiple of 256, workspace_bytes long) */
} cstp_jpeg_image;
/* Workspace bytes one image of this size needs, whatever its sampling; -1 outside 1 .. 65535. */
long long cstp_jpeg_workspace_bytes(int width, int height);
/* data: DEVICE, the concatenated streams; images: DEVICE array of n_images descriptors; status: DEVICE int32
 * [n_images]; workspace: DEVICE, 256-byte aligned, workspace_bytes long. */
int cstp_jpeg_decode(const uint8_t* data, const cstp_jpeg_image* images, int n_images, int32_t* status,
                     void* workspace, long long workspace_bytes, void* stream);

/* ---- SyncBN statistics exchange over NVLink peer memory ----------------------------------------------------
 * The all-reduce(SUM) of the [groups][2][Cp] row a world-synchronised BatchNorm call exchanges (the north star's SyncBN;
 * no counterpart in the reference, whose --sync_bn group holds one rank: models/model.py:95-96), as ONE kernel that
 * stores the local row into every peer's receive buffer, publishes a flag, waits for every peer's flag and sums the rows
 * in rank order (csrc/p2p_sync.cu).  peer_buffers: DEVICE array of `world` pointers to the per-rank buffers
 * (peer-mapped, e.g. torch symmetric memory), each cstp_bn_sync_buffer_bytes(world, slots, row_max) bytes, zeroed before
 * the first call; seq = 1, 2, ... per buffer set, identical on every rank -- either passed by the host (seq != 0,
 * seq_dev NULL) or kept by the kernel in a DEVICE counter (seq == 0, *seq_dev incremented per call: the launch can then
 * be replayed from a CUDA graph); out may alias row; *err_flag becomes 1 + peer when a peer's flag did not arrive within
 * the spin limit. */
long long cstp_bn_sync_buffer_bytes(int world, int slots, int row_max);
int cstp_bn_sync_exchange(const float* row, int n, const uint64_t* peer_buffers, int world, int rank, int slots,
                          int row_max, uint32_t seq, uint32_t* seq_dev, float* out, int* err_flag, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* CSTP_B200_H_ */

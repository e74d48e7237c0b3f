/*
 * pcb200.h -- C ABI of libpcb200.so: the B200 (sm_100a) replacement for the native half of the
 * MinkowskiEngine v0.4.3 operator library on PointContrast's Res16UNet34C hot path.
 *
 * What each entry point replaces (reference call sites are relative to /root/reference; the ME
 * native sources are an external, un-vendored dependency pinned at README.md:24,34):
 *
 *   pcb_coords_* / pcb_hash_* / pcb_kernel_map*   ME CoordsManager (CPU hash map): initialize, stride, getKernelMap.
 *        Reached implicitly from every `ME.SparseTensor(F, coords=C)` (pretrain/pointcontrast/lib/ddp_trainer.py:290-297,392-398)
 *        and every strided / 3x3x3 convolution (pretrain/pointcontrast/model/res16unet.py:47-190).
 *   pcb_conv_forward / pcb_conv_wgrad / pcb_weight_prep
 *        ME ConvolutionForwardGPU / ConvolutionBackwardGPU (and the Transpose variants), bound in ME's python as
 *        MinkowskiConvolutionFunction.apply(input_features, kernel, tensor_stride, stride, kernel_size, dilation,
 *        region_type, region_offset, in_coords_key, out_coords_key, coords_manager) -- signature evidenced by
 *        downstream/votenet_det_new/models/backbone/sparseconv/models/conditional_random_fields.py:135-137;
 *        constructed at pretrain/pointcontrast/model/modules/common.py:130-138,159-167.
 *   pcb_bn_*      MinkowskiBatchNorm == torch.nn.BatchNorm1d on .F (model/modules/common.py:21, model/resnet.py:95-97).
 *   pcb_nce_*     PointInfoNCE (lib/ddp_trainer.py:420-426 + lib/criterion.py:15-19).
 *   pcb_pdist_rowmin   pdist + min(1) of the hardest-contrastive loss (lib/ddp_trainer.py:182-184,215-219).
 *   pcb_sgd_step  optim.SGD(momentum, weight_decay) step (lib/ddp_trainer.py:107-111,319,435).
 *
 * Conventions
 *   - every function returns 0 on success, non-zero on failure; pcb_last_error() returns the message
 *     of the last failure on the calling thread.  Nothing throws across this boundary.
 *   - all data pointers are CALLER-OWNED DEVICE memory (16-byte aligned); the library never allocates
 *     device memory.  Workspaces are sized by the *_ws_bytes queries.
 *   - `stream` is a cudaStream_t passed as void*; every call is asynchronous on it unless stated.
 *   - feature matrices are fp32 row-major [rows, channels]; coordinates int32 [rows, 4] = (batch, x, y, z).
 *   - a kernel map is a dense neighbour table  tbl[K][n_out]  (int32): tbl[k][j] = input row feeding output
 *     row j through kernel offset k, or -1.  The ME per-offset (in,out) pair lists are exactly the
 *     non-negative entries of row k, in ascending j.
 */
#ifndef PCB200_H_
#define PCB200_H_

#include <stdint.h>
#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PCB_OK 0
#define PCB_ERR_CUDA 1
#define PCB_ERR_ARG 2
#define PCB_ERR_RANGE 3      /* coordinate outside the packable range */
#define PCB_ERR_DUPLICATE 4  /* duplicate coordinates in a SparseTensor */
#define PCB_MAX_KERNEL_VOLUME 27

const char* pcb_last_error(void);
/* "pcb200 <version> sm_100a" */
const char* pcb_version(void);
/* Number of kernels this library has launched on this process since load (bench.py's gpu_launches). */
uint64_t pcb_launch_count(void);
/* The library links its own (static) CUDA runtime: select the device the caller's pointers/streams live on. */
int pcb_set_device(int device);
/* Measurement aid (bench.py's roofline): while enabled, every convolution / weight-gradient entry point (including the ones
 * issued inside pcb_unit_*) is bracketed by CUDA events on its stream.  pcb_profile_read synchronises with them, returns the
 * elapsed ms and kind (0 = convolution forward / data gradient, 1 = weight gradient) of up to max_records records in issue
 * order, *count = records taken since the last read, and clears the list.  Not thread-safe; off by default. */
int pcb_profile_enable(int on);
int pcb_profile_read(float* ms, int32_t* kinds, int max_records, int* count);

/* ----------------------------------------------------------------------------------------------- coordinates */
/* (b,x,y,z) -> 64-bit keys whose unsigned order is lexicographic (b,x,y,z).  b in [0,65535), |x|,|y|,|z| < 32768.
 * `status` (device int32, caller-zeroed) receives PCB_ERR_RANGE bits on violation. */
int pcb_coords_pack(const int32_t* coords, int64_t n, uint64_t* keys, int32_t* status, void* stream);
int pcb_coords_unpack(const uint64_t* keys, int64_t n, int32_t* coords, void* stream);

/* Open-addressing hash table key -> row.  capacity must be a power of two >= 2n.  `status` gets
 * PCB_ERR_DUPLICATE if a key occurs twice. */
int pcb_hash_build(const uint64_t* keys, int64_t n, uint64_t* table_keys, int32_t* table_vals,
                   int64_t capacity, int32_t* status, void* stream);

/* Stride a level: coarse = floor(c / new_ts) * new_ts, unique, rows ordered by key (canonical order).
 * Writes out_keys[0..*n_out) and parent[i] = coarse row of fine row i.
 * SYNCHRONISES the stream once to return *n_out on the host. */
size_t pcb_coords_stride_ws_bytes(int64_t n);
int pcb_coords_stride(const uint64_t* keys, int64_t n, int32_t new_ts, uint64_t* out_keys, int32_t* parent,
                      int64_t* n_out, void* ws, size_t ws_bytes, void* stream);

/* tbl[k][j] = row of (out_coord[j] + offsets[k]) in the hashed level, or -1.  offsets: HOST int32 [K][3]. */
int pcb_kernel_map(const uint64_t* out_keys, int64_t n_out, const uint64_t* table_keys,
                   const int32_t* table_vals, int64_t capacity, const int32_t* offsets, int K, int32_t* tbl,
                   void* stream);
/* counts[k] = number of non-negative entries of row k (device int64 [K]). */
int pcb_kernel_map_count(const int32_t* tbl, int K, int64_t n_out, int64_t* counts, void* stream);

/* ----------------------------------------------------------------------------------------------- data preparation (SURVEY.md 8f-2) */
/* One point per occupied voxel: voxel index = floor(xyz / voxel_size) per axis (fp32, |index| < 2^20).  Writes the M occupied voxels'
 * indices (int32 [M,3], sorted by (x,y,z)) and sel[M] = the smallest index of a point in each voxel -- np.unique(return_index=True) /
 * `ME.utils.sparse_quantize(xyz / voxel_size, return_index=True)` of `pretrain/pointcontrast/lib/ddp_data_loaders.py:228-241`.
 * out_coords / sel hold up to n rows.  SYNCHRONISES the stream once to return *m_out. */
size_t pcb_voxelize_ws_bytes(int64_t n);
int pcb_voxelize(const float* xyz, int64_t n, float voxel_size, int32_t* out_coords, int32_t* sel, int64_t* m_out, void* ws,
                 size_t ws_bytes, void* stream);
/* All (i, j) with |src_i - dst_j| < radius (fp32, strict), i ascending, j ascending within i -- `get_matching_indices`
 * (`ddp_data_loaders.py:36-49`: an open3d KD-tree radius search per source point; radius = 1.5 voxels) on a hashed uniform grid of
 * cell size `radius`.  *n_pairs = total number of pairs (SYNCHRONISES once); at most `cap` of them are written ([cap,2] int32;
 * pairs == NULL: count only). */
size_t pcb_radius_pairs_ws_bytes(int64_t ns, int64_t nd);
int pcb_radius_pairs(const float* src, int64_t ns, const float* dst, int64_t nd, float radius, int32_t* pairs, int64_t cap,
                     int64_t* n_pairs, void* ws, size_t ws_bytes, void* stream);

/* ----------------------------------------------------------------------------------------------- convolution */
/* fp32 W[K][Cin][Cout] -> bf16 hi/lo split planes in the same layout (w_hi, w_lo) and per-offset transposed
 * [K][Cout][Cin] (wt_hi, wt_lo).  x ~= hi + lo with |x - hi - lo| <= 2^-17 |x|. */
int pcb_weight_prep(const float* W, int K, int Cin, int Cout, uint16_t* w_hi, uint16_t* w_lo,
                    uint16_t* wt_hi, uint16_t* wt_lo, void* stream);

/* Y[j, :] = bias + sum_k X[tbl[kmap[k]][j], :] . W[k]      (j < n_out)      -- fp32 operands (the modular ME-style surface)
 *   X  : [*, Cin] row stride ldx (floats);  Y: [n_out, Cout] row stride ldy.
 *   wk_hi/wk_lo : the weights of THIS call's roles as bf16 hi/lo planes, K-major = [K][Cout][Cin] (pcb_weight_prep: the wt_* planes for
 *               the forward roles; the w_* planes with swapped channel counts for the data gradient).  Tensor-core path (tcgen05, fp32 rows
 *               split to bf16 hi/lo in the producers' registers, fp32 accumulate in TMEM): Cin % 32 == 0, Cout % 32 == 0, K <= 27.
 *   w_f32     : fp32 weights [K][Cin][Cout] for the exact SIMT path (other widths, the 3-channel stem, PCB_CONV_FORCE_SIMT); may be NULL
 *               when the tensor-core path applies.
 *   kmap      : HOST int32 [K] table row used by weight k (NULL = identity). */
#define PCB_CONV_FORCE_SIMT 1
#define PCB_CONV_ACCUMULATE 4  /* Y += result (tensor-core paths) / dW += result (weight gradients) */
#define PCB_PLANES_A_FP16 8    /* split-operand calls: the GATHERED operand's planes are fp16 hi/lo (default: bf16 hi/lo) */
#define PCB_PLANES_B_FP16 16   /* pcb_conv_forward_split: the weight tiles are fp16 x 2^10 (pcb_weight_tile with this flag);
                                  pcb_conv_wgrad_split: the ROW-ALIGNED operand's planes are fp16.  Both operands of a call must
                                  use the same format (tcgen05.mma.kind::f16 rejects fp16 x bf16): set both flags or neither. */
/* Small levels split the (offset, channel-chunk) loop over extra CTAs and reduce through `ws` (deterministic). */
size_t pcb_conv_forward_ws_bytes(int K, int64_t n_out, int Cin, int Cout);
int pcb_conv_forward(const float* X, int ldx, const int32_t* tbl, int64_t tbl_stride, const int32_t* kmap, int K,
                     int64_t n_out, int Cin, int Cout, const uint16_t* wk_hi, const uint16_t* wk_lo, const float* w_f32,
                     const float* bias, float* Y, int ldy, void* ws, size_t ws_bytes, int flags, void* stream);

/* Y[j, :] = sum_k X[tbl[kmap[k]][j], :];  cnt[j] (optional) = number of neighbours present.  The sum / average pooling and unpooling
 * layers of the sibling models (MinkowskiSumPooling / AvgPooling / PoolingTranspose / AvgUnpooling, `model/modules/common.py:170-214`,
 * `model/resnet.py:63`) and their backward passes (the same sum over the transposed table).  C % 4 == 0. */
int pcb_gather_sum(const float* X, int ldx, const int32_t* tbl, int64_t tbl_stride, const int32_t* kmap, int K, int64_t n_out, int C,
                   float* Y, int ldy, float* cnt, void* stream);

/* dW[k] = sum_j A[tbl[k][j], :]^T . B[j, :]       A: gathered [*, Ca] (lda), B: contiguous rows [n_out, Cb] (ldb).
 *   transpose_out = 0: dW is [K][Ca][Cb];  1: dW is [K][Cb][Ca].
 * pcb_conv_wgrad: EXACT fp32 kernels on fp32 operands (the 3-channel stem layer, widths the tensor-core tiling does not cover, cross-checks);
 * the tensor-core weight gradient is pcb_conv_wgrad_split on split operands. */
size_t pcb_conv_wgrad_ws_bytes(int K, int64_t n_out, int Ca, int Cb);
int pcb_conv_wgrad(const float* A, int lda, const float* B, int ldb, const int32_t* tbl, int64_t tbl_stride, int K,
                   int64_t n_out, int Ca, int Cb, float* dW, int transpose_out, void* ws, size_t ws_bytes,
                   int flags, void* stream);

/* Split-operand variants (tcgen05 only): the gathered / row-aligned operands are bf16 hi/lo planes (see pcb_split_rows),
 * row strides lds/lda/ldb in ELEMENTS (multiples of 8).  Same semantics as pcb_conv_forward / pcb_conv_wgrad; the kernels'
 * operand staging is then a pure asynchronous copy (cp.async, zero-filled where a neighbour is missing). */
/* pcb_weight_tile: fp32 W[K][Cin][Cout] -> split weights pre-tiled as the shared-memory images of the split conv kernel (one
 * contiguous blob per (offset, 32-channel chunk, column block), fetched by ONE TMA bulk copy per pipeline stage):
 * `fwd_tiles` for the forward roles, `dgrad_tiles` for the data-gradient roles (Cin/Cout swapped).  flags & PCB_PLANES_B_FP16:
 * the FORWARD tiles hold fp16 hi/lo of W * 2^10 (|W| < 60; the kernel rescales its output), the data-gradient tiles stay bf16. */
size_t pcb_weight_tile_bytes(int K, int Cin, int Cout, int dgrad_roles);
int pcb_weight_tile(const float* W, int K, int Cin, int Cout, void* fwd_tiles, void* dgrad_tiles, int flags, void* stream);
/* The same for every convolution of a network in ONE launch: fill a HOST array of descriptors with pcb_tile_desc_fill (start = running
 * sum of K*Cin*Cout), copy it to the device, call pcb_weight_tile_batch(device array, n <= 256, total elements) after every optimiser step. */
typedef struct pcb_tile_desc {
  const float* W; void* fwd; void* dgrad;
  int32_t K, Cin, Cout, flags, bn_f, bn_d;
  int64_t start;
} pcb_tile_desc;
int pcb_tile_desc_fill(pcb_tile_desc* d, const float* W, int K, int Cin, int Cout, void* fwd_tiles, void* dgrad_tiles, int flags, int64_t start);
int pcb_weight_tile_batch(const pcb_tile_desc* descs_dev, int n, int64_t total, void* stream);
int pcb_conv_forward_split(const uint16_t* Xhi, const uint16_t* Xlo, int lds, const int32_t* tbl, int64_t tbl_stride,
                           const int32_t* kmap, int K, int64_t n_out, int Cin, int Cout, const void* w_tiles,
                           const float* bias, float* Y, int ldy, void* ws, size_t ws_bytes, int flags, void* stream);
size_t pcb_conv_wgrad_split_ws_bytes(int K, int64_t n_out, int Ca, int Cb);
int pcb_conv_wgrad_split(const uint16_t* Ahi, const uint16_t* Alo, int lda, const uint16_t* Bhi, const uint16_t* Blo, int ldb,
                         const int32_t* tbl, int64_t tbl_stride, int K, int64_t n_out, int Ca, int Cb, float* dW,
                         int transpose_out, void* ws, size_t ws_bytes, int flags, void* stream);

/* ----------------------------------------------------------------------------------------------- batch norm */
/* Training-mode statistics over n rows: mean[C], invstd[C] = 1/sqrt(var_biased + eps); if running_* non-NULL:
 * running = (1-momentum)*running + momentum*{mean, var_unbiased}.  ws: pcb_bn_ws_bytes(n, C). */
size_t pcb_bn_ws_bytes(int64_t n, int C);
int pcb_bn_stats(const float* X, int64_t n, int C, float eps, float momentum, float* mean, float* invstd,
                 float* running_mean, float* running_var, void* ws, size_t ws_bytes, void* stream);
/* Y = (X - mean) * invstd * gamma + beta  [+ residual] [relu].   Y may alias X. */
int pcb_bn_apply(const float* X, int64_t n, int C, const float* mean, const float* invstd, const float* gamma,
                 const float* beta, const float* residual, int relu, float* Y, void* stream);
/* Backward of the affine-normalise (no relu): given dY and X, writes dX, dgamma[C], dbeta[C]. */
int pcb_bn_backward(const float* dY, const float* X, int64_t n, int C, const float* mean, const float* invstd,
                    const float* gamma, float* dX, float* dgamma, float* dbeta, void* ws, size_t ws_bytes,
                    void* stream);

/* Strided / row-segmented variants used by the fused network executor (pointcontrast_b200/fused.py).  All ld* are row strides
 * in floats (>= C, multiples of 4), so inputs/outputs may be column slices of wider (concatenated) buffers.
 *   apply   : Y = [relu]( (X-mean)*invstd*gamma+beta [+ residual] ), as fp32 (Y, may be NULL) and/or split planes (Yhi/Ylo);
 *             flags: PCB_BN_RELU, PCB_PLANES_A_FP16 (Yhi/Ylo are fp16 hi/lo instead of bf16 hi/lo; Ybhi/Yblo, if non-NULL, then
 *             receive the bf16 hi/lo planes as well)
 *   backward: g = dY * (relu_out > 0) if relu_out else dY;   dgamma/dbeta (+)= sum(g*xhat) / sum(g);
 *             dX = gamma*invstd*(g - mean(g) - xhat*mean(g*xhat));   gout (=|+=) g  (gout_mode 0 none, 1 write, 2 add)
 *             -- gout is the gradient of the residual input of the forward unit; it may alias dY. */
#define PCB_BN_RELU 1
/* Row-segmented variants: rows [0, n0) and [n0, n) are two independent BatchNorm batches -- the two views of a scene pair
 * stacked in one feature matrix, each normalised with its own statistics exactly as the reference's two forward calls do
 * (`lib/ddp_trainer.py:290-297,392-398`).  mean / invstd are [2][C]; the running statistics are updated with segment 0 and
 * then with segment 1; dgamma / dbeta sum over both segments.  n0 == n degenerates to the single-batch functions above. */
int pcb_bn_stats_seg(const float* X, int ldx, int64_t n, int64_t n0, int C, float eps, float momentum, float* mean, float* invstd,
                     float* running_mean, float* running_var, void* ws, size_t ws_bytes, void* stream);
int pcb_bn_apply_seg(const float* X, int ldx, int64_t n, int64_t n0, int C, const float* mean, const float* invstd,
                     const float* gamma, const float* beta, const float* residual, int ldr, int flags, float* Y, int ldy,
                     uint16_t* Yhi, uint16_t* Ylo, int lds, uint16_t* Ybhi, uint16_t* Yblo, void* stream);
int pcb_bn_backward_seg(const float* dY, int lddy, const float* X, int ldx, const float* relu_out, int ldm, int64_t n, int64_t n0,
                        int C, const float* mean, const float* invstd, const float* gamma, float* dX, int lddx, float* dgamma,
                        float* dbeta, int accumulate_param_grads, float* gout, int ldg, int gout_mode, uint16_t* dXhi,
                        uint16_t* dXlo, int lds, void* ws, size_t ws_bytes, void* stream);
/* "Split" operand format of the tensor-core conv kernels: an fp32 matrix stored as two 16-bit planes, x ~= hi + lo: bf16 planes
 * (2^-17 relative, fp32's exponent range: gradients) or, with PCB_PLANES_A_FP16, fp16 planes (2^-22 relative, |x| < 65504: the
 * activations gathered by the FORWARD convolutions -- the forward pass sets the whole-network gradient error, profiles/r2_results.md);
 * row stride lds in ELEMENTS.  The elementwise producers above can emit it directly (Yhi/Ylo, dXhi/dXlo; NULL = off; dX may
 * then be NULL), so the conv kernels' gather becomes a pure asynchronous copy.  pcb_split_rows converts an fp32 matrix. */
int pcb_split_rows(const float* X, int ldx, int64_t n, int C, uint16_t* hi, uint16_t* lo, int lds, int flags, void* stream);

/* ----------------------------------------------------------------------------------------------- fused units */
/* One "unit" of the Res16UNet graph = convolution -> BatchNorm (training statistics) -> [+ residual] -> [ReLU]
 * (`model/res16unet.py:206-268`, `model/modules/resnet_block.py:44-60`: a BasicBlock is two units).  pcb_unit_forward issues the whole
 * unit from ONE call -- on the small levels, where the convolution runs offset-split, its reduction pass also produces the BatchNorm
 * column statistics (no separate pass over z) --
 * and pcb_unit_backward issues its reverse: ReLU mask + BatchNorm backward + residual-gradient fan-out in one elementwise
 * pass, then the weight gradient (accumulated into dW) and the data gradient (written or accumulated into gin).
 * The caller (pointcontrast_b200/fused.py; a C++ host would do the same) owns every buffer; the struct is plain data.
 *
 * Matrices: fp32 pointer `*_p` (row stride `*_ld` floats) and/or bf16 split planes `*_hi`/`*_lo` (row stride `*_lds` elements).
 *   x    : unit input  [n_in, Cin]   (split planes when Cin % 32 == 0, else fp32: the 3-channel stem)
 *   z    : convolution output [n_out, Cout], fp32 (kept for the backward pass)
 *   out  : unit output [n_out, Cout]: split planes (always) and fp32 (only if out_p != NULL: it feeds a residual add)
 *   res  : residual input, fp32 (or NULL);  rows [0, n0) / [n0, n_out) are the two views of a stacked pair (n0 == n_out: one)
 *   g    : gradient of `out` (fp32, complete when pcb_unit_backward is called)
 *   dz   : scratch for the gradient of z: split planes [n_out, Cout] (+ fp32 `dz_p` when Cout or Cin is not a multiple of 32)
 *   gin  : gradient of x (fp32) -- written (gin_mode 1) or accumulated (2); 0: not wanted (network input)
 *   gres : gradient of the residual input -- written (1) / accumulated (2) / none (0)
 * Tables (device int32 [K][stride]) and kmaps (HOST int32 [K] or NULL) as for pcb_conv_forward / pcb_conv_wgrad.
 * ws: pcb_unit_ws_bytes(K, n_in, n_out, Cin, Cout) bytes of scratch. */
typedef struct pcb_unit {
  int64_t n_in, n_out, n0;
  int32_t K, Cin, Cout, relu;
  const int32_t* fwd_tbl; int64_t fwd_stride; const int32_t* fwd_kmap;
  const int32_t* dg_tbl; int64_t dg_stride; const int32_t* dg_kmap;
  const int32_t* wg_tbl; int64_t wg_stride; int32_t wg_gather_x;
  const float* W; const void* wt_fwd; const void* wt_dg; float* dW;
  const float* gamma; const float* beta; float* running_mean; float* running_var; float* dgamma; float* dbeta;
  float eps, momentum;
  float* mean; float* invstd;                       /* [segments][Cout], written by forward, read by backward */
  const float* x_p; int32_t x_ld; const uint16_t* x_hi; const uint16_t* x_lo; int32_t x_lds;
  const uint16_t* x_bhi; const uint16_t* x_blo;     /* PCB_UNIT_FP16_FORWARD: x once more as bf16 hi/lo planes (the weight gradient pairs it
                                                       with the bf16 gradient planes: tcgen05.mma takes ONE format for both operands) */
  float* z_p; int32_t z_ld;
  float* out_p; int32_t out_ld; uint16_t* out_hi; uint16_t* out_lo; int32_t out_lds;
  uint16_t* out_bhi; uint16_t* out_blo;             /* PCB_UNIT_FP16_FORWARD: bf16 hi/lo copy of `out` (row stride out_lds) */
  const float* res_p; int32_t res_ld;
  const float* g_p; int32_t g_ld;
  float* dz_p; uint16_t* dz_hi; uint16_t* dz_lo; int32_t dz_ld;
  float* gin_p; int32_t gin_ld; int32_t gin_mode;
  float* gres_p; int32_t gres_ld; int32_t gres_mode;
  void* ws; size_t ws_bytes;
  int32_t flags;                                    /* PCB_UNIT_* */
} pcb_unit;
#define PCB_UNIT_SEPARATE_STATS 1   /* forward: BatchNorm statistics always by a separate pass over z (cross-check of the fused reduce+statistics pass) */
#define PCB_UNIT_FP16_FORWARD 2     /* activations are gathered by the forward convolutions as fp16 hi/lo planes (x_hi/x_lo, out_hi/out_lo)
                                       against fp16 weight tiles (pcb_weight_tile with PCB_PLANES_B_FP16): 2^-22 products in the
                                       forward pass.  Gradients (dz) and the data-gradient tiles stay bf16 hi/lo (fp32's exponent
                                       range); tcgen05.mma.kind::f16 rejects mixed fp16 x bf16 operands (illegal instruction,
                                       profiles/probes/mixed_fmt_probe.cu), so every activation also carries bf16 hi/lo planes
                                       (x_bhi/x_blo, out_bhi/out_blo) for the weight gradient. */
#define PCB_UNIT_EVAL 4             /* forward only, eval-mode BatchNorm: normalise with running_mean / running_var (not updated) */
size_t pcb_unit_ws_bytes(int K, int64_t n_in, int64_t n_out, int Cin, int Cout);
int pcb_unit_forward(const pcb_unit* u, void* stream);
int pcb_unit_backward(const pcb_unit* u, void* stream);

/* ----------------------------------------------------------------------------------------------- losses */
/* PointInfoNCE on gathered rows q,k [n, D]: loss = mean_i(logsumexp_j(q_i.k_j/T) - q_i.k_i/T).
 * Writes loss (device float), dq, dk (= d loss / d q, d k).  ws: pcb_nce_ws_bytes(n).
 * D = 32 or 64: fused tcgen05 kernels (nce_tc5.cu) -- q k^T tiles in Tensor Memory from fp16 hi/lo operands (|q|,|k| <= ~1: the
 * L2-normalised features), softmax statistics and both gradients straight from the tiles, the n x n logits never stored.
 * Other widths (or PCB_NCE_SIMT=1): exact fp32 SIMT kernels that materialise the logits in ws. */
size_t pcb_nce_ws_bytes(int64_t n);
int pcb_nce_forward_backward(const float* q, const float* k, int64_t n, int D, float inv_T, float* loss, float* dq,
                             float* dk, void* ws, size_t ws_bytes, void* stream);
/* nn.CrossEntropyLoss(ignore_index) on logits [n, C] with int64 targets (`downstream/semseg/lib/train.py:68,120`): writes the mean loss
 * over the non-ignored rows (device float) and dlogits = grad_scale * d loss / d logits.  ws: pcb_ce_ws_bytes(n). */
size_t pcb_ce_ws_bytes(int64_t n);
int pcb_ce_forward_backward(const float* logits, const int64_t* target, int64_t n, int C, int64_t ignore_index, float grad_scale,
                            float* loss, float* dlogits, void* ws, size_t ws_bytes, void* stream);
/* Semantic-segmentation metrics of one batch (`downstream/semseg/lib/test.py:119-149`, `lib/utils.py:117-133`) on logits [n, C]
 * (contiguous fp32) and int64 targets.  A row is valid when 0 <= target < C and target != ignore_index; the others count in no loss,
 * precision or histogram term and are negatives for every class in the average precision.
 *   pred  [n] int32: first maximal index of each row (may be NULL)
 *   hist  [C*C] int64, ACCUMULATED (+=): hist[target * C + pred] over the valid rows
 *   stats [4] fp64 = {sum of the cross-entropy over the valid rows, #valid, #(pred == target) among them, n}
 *   ap    [C] fp64: uninterpolated average precision of softmax column c against target == c, equal scores ranked as one group;
 *         NaN for a class without a positive row
 *   prob  [n, C] fp32: the softmax the average precision ranked by (may be NULL)
 * 2 <= C <= 64, n >= 1, n * C < 2^31.  ws: pcb_seg_eval_ws_bytes(n, C).  Deterministic: repeated calls give bit-identical stats / ap. */
size_t pcb_seg_eval_ws_bytes(int64_t n, int C);
int pcb_seg_eval(const float* logits, const int64_t* target, int64_t n, int C, int64_t ignore_index, int32_t* pred, int64_t* hist,
                 double* stats, double* ap, float* prob, void* ws, size_t ws_bytes, void* stream);
/* Row-wise L2 normalisation of the output features, y = x / ||x||_2 with no epsilon (`model/res16unet.py:262-266`), and its
 * backward dx = (dy - y (y.dy)) / ||x||.  inv_norm: [n] scratch written by forward, read by backward. */
int pcb_l2norm_forward(const float* X, int64_t n, int C, float* Y, float* inv_norm, void* stream);
int pcb_l2norm_backward(const float* dY, const float* Y, const float* inv_norm, int64_t n, int C, float* dX, void* stream);
/* minval[i] = min_j sqrt(sum_d (A[i,d]-B[j,d])^2 + 1e-7), argmin[i] = smallest such j.   packed: u64 scratch [P]. */
int pcb_pdist_rowmin(const float* A, int64_t P, const float* B, int64_t S, int D, float* minval, int32_t* argmin,
                     uint64_t* packed, void* stream);

/* ----------------------------------------------------------------------------------------------- optimiser */
/* torch.optim.SGD semantics on a flat buffer:  d = g*grad_scale + wd*p;  buf = first ? d : momentum*buf + (1-dampening)*d;  p -= lr*buf
 * (pretraining: dampening 0, `lib/ddp_trainer.py:107-111`; semseg finetuning: 0.1, `downstream/semseg/lib/solvers.py:50-57`) */
int pcb_sgd_step(float* p, const float* g, float* buf, int64_t n, float lr, float momentum, float weight_decay,
                 float grad_scale, int first, float dampening, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* PCB200_H_ */

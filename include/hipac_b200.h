/*
 * hipac_b200.h -- C ABI of the B200-native HiPAC hot path (libhipac_b200.so).
 *
 * The reference (anacarsi/ss25_Hierarchical_Multiscale_Image_Classification) has no FFI
 * or plugin layer: its boundary is plain Python functions (SURVEY.md section 8b).  Each entry
 * point below names the reference code it replaces; the Python mirror of the
 * reference interface (package ss25_hierarchical_multiscale_image_classification_b200)
 * binds these symbols with ctypes.  INTEGRATION.md shows the reference-side stub.
 *
 * Conventions
 *   - every pointer named d_* is DEVICE memory owned by the caller (PyTorch),
 *     h_* is host memory; the library allocates no persistent device memory
 *     except small constant tables.
 *   - every call is asynchronous on `stream` (a cudaStream_t passed as void*).
 *   - return 0 on success, negative on error; hipac_last_error() gives the text.
 *     Nothing throws across the ABI.
 */
#ifndef HIPAC_B200_H
#define HIPAC_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define HIPAC_ABI_VERSION 2

/* batch layouts written by hipac_tile_scan / consumed by hipac_resnet18_forward */
#define HIPAC_LAYOUT_NHWC3_BF16 1 /* bf16 [N,224,224,3], (u8/255-mean)/std, the reference's tensor (src/main.py:815-816) in NHWC */
#define HIPAC_LAYOUT_S2D16_BF16 2 /* bf16 [N,112,115,16]: 2x2 space-to-depth of the above, ch=(dy*2+dx)*3+c, 12..15 zero; column X of the
                                    image sits at index X+2, columns 0,1,114 are zero (conv1's W padding made explicit so that the four
                                    W-taps of a filter row are one contiguous 128-byte TMA row) */
#define HIPAC_S2D16_WIDTH 115

/* stage-1 algorithm selector */
#define HIPAC_SCAN_AUTO   0 /* fused read-once path when stride %% (P/224) == 0, else direct */
#define HIPAC_SCAN_DIRECT 1 /* one window reduction + one resample per patch (any stride) */
#define HIPAC_SCAN_FUSED  2 /* single streaming pass over the level image (error if not applicable) */
#define HIPAC_SCAN_NO_STREAM 0x200 /* OR-able flag: run the fused path with its cp.async kernels (two reads of the image) instead of the
                                      TMA streaming pass; the two are bit-identical, the flag exists for the cross-check tests */
#define HIPAC_SCAN_KEEP_ALL 0x100 /* OR-able flag: skip the tissue rejection (every candidate survives); used when the input
                                     is a stack of already-extracted patches, as in the reference's extract_features */

const char* hipac_last_error(void);
int hipac_abi_version(void);

/* ---------------------------------------------------------------------------------------
 * Stage 1: multiscale patch extraction of ONE level image resident in HBM.
 * Replaces the hot loop of extract_patches (reference src/main.py:682-727): candidate grid
 * x in range(0,W,S), y in range(0,H,S) (x outer), white padding of border patches (688-703),
 * tissue test mean>240 -> reject (718-720, integer form sum <= 240*3*P*P), lesion label
 * any(mask[y:y+P,x:x+P]>0) (705-716), and -- instead of the PNG round trip -- the
 * Resize((224,224)) + ToTensor + Normalize of src/main.py:812-818 (Pillow-exact antialiased
 * bilinear in 22-bit fixed point, two uint8 passes).
 *
 *   d_rgb        uint8 [H][pitch_bytes], 3 bytes per pixel (RGB), level-L image
 *   d_mask       uint8 [H][mask_pitch] rasterised lesion mask (>0 = lesion) or NULL (all "normal")
 *   P, S         patch size (1792>>level) and stride (reference CLI: 224)
 *   iy_begin/end candidate grid rows y/S in [iy_begin, iy_end)  (the multi-GPU shard unit)
 *   outputs      survivors in the reference's emission order (x outer, y inner):
 *     d_coords   int32 [capacity][2] (x, y) level-L pixel coordinates
 *     d_labels   uint8 [capacity]    1 = tumor, 0 = normal
 *     d_batch_u8 uint8 [capacity][224][224][3] Pillow-exact resized patch, or NULL
 *     d_batch    bf16 batch in `layout`, or NULL
 *     d_count    int32 [2]: {survivors, candidates}; survivors may exceed capacity, in which
 *                case only the first `capacity` are written (caller re-runs with a smaller row range)
 *   d_workspace  >= hipac_tile_scan_workspace_bytes(...) bytes, 256-byte aligned
 * ------------------------------------------------------------------------------------- */
size_t hipac_tile_scan_workspace_bytes(int H, int W, int P, int S, int iy_begin, int iy_end, int mode);

int hipac_tile_scan(const uint8_t* d_rgb, int H, int W, int64_t pitch_bytes,
                    const uint8_t* d_mask, int64_t mask_pitch,
                    int P, int S, int iy_begin, int iy_end,
                    int32_t* d_coords, uint8_t* d_labels,
                    uint8_t* d_batch_u8, void* d_batch, int layout,
                    int32_t* d_count, int capacity,
                    void* d_workspace, size_t workspace_bytes,
                    int mode, void* stream);

/* ---------------------------------------------------------------------------------------
 * Tissue segmentation (opt-in stage 1 background rejection; the reference has none, see SURVEY.md fact 1).  The CLAM-style
 * recipe of CAMELYON16 pipelines on a low-resolution level, bit-exact against OpenCV 4.13's 8-bit code:
 *   cv2.cvtColor(RGB2HSV) saturation -> cv2.medianBlur(S, ksize) (replicated borders) -> cv2.threshold(BINARY | OTSU),
 * or a fixed threshold.  S = (d * sdiv[v] + 2048) >> 12 with v = max(R,G,B), d = v - min(R,G,B), sdiv[i] = round(255*4096/i);
 * mask = blurred > t ? 255 : 0.
 *   d_rgb        uint8 [H][pitch_bytes] RGB (channel order does not matter), pitch_bytes >= 3*W
 *   ksize        1, 3, 5 or 7
 *   threshold    -1 = Otsu's threshold of the blurred plane's histogram (OpenCV's fp64 loop), else t in [0, 255]
 *   d_mask       uint8 [H][mask_pitch] output, 0 / 255
 *   d_threshold  int32 [1] output: the t that was used (device memory; nothing waits on the host)
 *   d_blur       uint8 [H][blur_pitch] output of the median blur, or NULL (kept in the workspace only)
 *   d_workspace  >= hipac_tissue_workspace_bytes(H, W) bytes, 256-byte aligned
 * Three kernels on `stream` (saturation + median + histogram, Otsu, binarize). */
size_t hipac_tissue_workspace_bytes(int H, int W);
int hipac_tissue_segment(const uint8_t* d_rgb, int H, int W, int64_t pitch_bytes, int ksize, int threshold,
                         uint8_t* d_mask, int64_t mask_pitch, int32_t* d_threshold,
                         uint8_t* d_blur, int64_t blur_pitch,
                         void* d_workspace, size_t workspace_bytes, void* stream);

/* hipac_tile_scan with a tissue mask instead of the mean > 240 rule.  d_tissue: uint8 [tissue_h][tissue_pitch] (> 0 = tissue)
 * at scale m = tissue_scale (1, 2, 4, 8, 16 or 32; S % m == 0 and P % m == 0): mask pixel (u, v) covers level pixels
 * [v*m, v*m+m) x [u*m, u*m+m), row 0 = row 0 of d_rgb (a shard passes the mask rows of its own origin, a multiple of m).
 * A candidate (x, y) survives iff at least min_tissue_pixels mask pixels > 0 lie inside [y/m, (y+P)/m) x [x/m, (x+P)/m);
 * pixels outside the mask's extent count as background.  Everything else -- grid, emission order, labels, compaction,
 * capacity, resample, HIPAC_SCAN_KEEP_ALL -- is as in hipac_tile_scan.
 * d_workspace >= hipac_tile_scan_tissue_workspace_bytes(...) bytes, 256-byte aligned. */
size_t hipac_tile_scan_tissue_workspace_bytes(int H, int W, int P, int S, int iy_begin, int iy_end, int mode, int tissue_scale);
int hipac_tile_scan_tissue(const uint8_t* d_rgb, int H, int W, int64_t pitch_bytes,
                           const uint8_t* d_mask, int64_t mask_pitch,
                           int P, int S, int iy_begin, int iy_end,
                           int32_t* d_coords, uint8_t* d_labels,
                           uint8_t* d_batch_u8, void* d_batch, int layout,
                           int32_t* d_count, int capacity,
                           void* d_workspace, size_t workspace_bytes, int mode,
                           const uint8_t* d_tissue, int tissue_h, int tissue_w, int64_t tissue_pitch,
                           int tissue_scale, int min_tissue_pixels, void* stream);

/* ---------------------------------------------------------------------------------------
 * Coarse-to-fine cascade: tile a finer level only where a coarser level's classifier fires.
 * Levels are exact powers of two; the coarse level Lc and the fine level Lf < Lc differ by shift = Lc - Lf >= 1.
 *
 * hipac_roi_grid  builds the ROI: uint8 d_grid [ny][nx] over the coarse CANDIDATE grid (nx, ny = the coarse level's grid
 *                 shape at `stride`), cell (i, j) = 1 iff some survivor s < min(d_count[0], capacity) with
 *                 d_scores[s] >= threshold has its cell (x / stride, y / stride) within Chebyshev distance `dilate`
 *                 (cells) of (i, j); 0 otherwise.  d_coords int32 [capacity][2], d_scores float [capacity] (e.g.
 *                 logits[:,1] - logits[:,0] with threshold = log(tau / (1 - tau))).  d_count is read on the device (the
 *                 tile scan's survivor counter): nothing waits on the host.  Two kernels (clear, scatter) on `stream`.
 *                 hipac_roi_grid_bytes(nx, ny) = nx * ny.
 * hipac_tile_scan_roi  hipac_tile_scan_tissue (tissue_scale > 0) or hipac_tile_scan (tissue_scale = 0: no tissue mask, the
 *                 mean > 240 rule; the tissue arguments are ignored), then the ROI test ANDed into the keep bit before the
 *                 compaction.  A candidate at fine pixel (x, y_origin + y) -- y_origin = fine-level row of d_rgb's row 0 --
 *                 is in the ROI iff its footprint [x, x+P) x [y, y+P) (white-padded border patches included) overlaps with
 *                 positive area the footprint [i*roi_stride << shift, (i*roi_stride + roi_patch) << shift) (same on y) of
 *                 at least one set cell of d_roi [roi_ny][roi_nx] (shift = roi_level_shift; cells outside the grid are
 *                 not set).  Grid, emission order, labels, capacity, resample and d_count[1] (= candidates of the row
 *                 range) are as in hipac_tile_scan.  HIPAC_SCAN_KEEP_ALL is refused.
 *                 d_workspace >= hipac_tile_scan_roi_workspace_bytes(...) bytes, 256-byte aligned. */
size_t hipac_roi_grid_bytes(int nx, int ny);
int hipac_roi_grid(const int32_t* d_coords, const float* d_scores, const int32_t* d_count, int capacity, float threshold,
                   int stride, int nx, int ny, int dilate, uint8_t* d_grid, void* stream);
size_t hipac_tile_scan_roi_workspace_bytes(int H, int W, int P, int S, int iy_begin, int iy_end, int mode, int tissue_scale);
int hipac_tile_scan_roi(const uint8_t* d_rgb, int H, int W, int64_t pitch_bytes,
                        const uint8_t* d_mask, int64_t mask_pitch,
                        int P, int S, int iy_begin, int iy_end,
                        int32_t* d_coords, uint8_t* d_labels,
                        uint8_t* d_batch_u8, void* d_batch, int layout,
                        int32_t* d_count, int capacity,
                        void* d_workspace, size_t workspace_bytes, int mode,
                        const uint8_t* d_tissue, int tissue_h, int tissue_w, int64_t tissue_pitch,
                        int tissue_scale, int min_tissue_pixels,
                        const uint8_t* d_roi, int roi_nx, int roi_ny, int roi_level_shift, int roi_stride, int roi_patch,
                        int64_t y_origin, void* stream);

/* ---------------------------------------------------------------------------------------
 * Macenko stain normalisation (torchstain's NumpyMacenkoNormalizer, the stain matrix estimated once per slide).
 * OD(v) = -log((v + 1) / Io) per channel, fp64.
 *
 * Stain block, fp64 [HIPAC_STAIN_BLOCK_DOUBLES]: [0..5] HE row-major [3][2] (column 0 haematoxylin, column 1 eosin),
 * [6..7] maxC, [8] valid (1 or 0), [9] n_hat (pixels whose three ODs are all >= beta), [10..15] zero.
 * Parameter block, fp64 [HIPAC_STAIN_PARAMS_DOUBLES]: [0] valid, [1] Io, [2..10] M row-major [3][3], [11..266] od[256].
 *
 * hipac_stain_estimate  (HE, maxC) of the uint8 RGB image d_rgb [H][pitch] (e.g. a slide thumbnail): ODhat = the pixels with
 *                       all three ODs >= beta; E = the eigenvectors of np.cov(ODhat) with the two largest eigenvalues;
 *                       phi = atan2 of ODhat . E; vMin / vMax = E (cos, sin) of numpy's linear percentiles alpha and
 *                       100 - alpha of phi; HE = [vMin, vMax] if vMin[0] > vMax[0] else [vMax, vMin]; C = P . OD over all
 *                       pixels with P below; maxC = the 99th percentiles of C's rows.  valid = 0 when n_hat < 2,
 *                       det(HE^T HE) <= 0, a value is not finite or maxC <= 0.  A fixed sequence of kernels on `stream`
 *                       with no host wait and no floating-point atomics: the block is the same bits on every run.
 *                       Io in 1..255, alpha in (0, 50), beta finite and >= 0; H * W < 2^31.
 *                       d_ws >= hipac_stain_workspace_bytes(H, W) bytes (16 per pixel + 48 KB), 256-byte aligned.
 * hipac_stain_normalizer  the parameter block that maps d_src's stain to d_target's (NULL: torchstain's reference,
 *                       HERef = [[0.5626, 0.2159], [0.7201, 0.8012], [0.4062, 0.5581]], maxCRef = [1.9705, 1.0308]).
 *                       In fp64, every operation rounded on its own:  g_ij = (HE[0][i] HE[0][j] + HE[1][i] HE[1][j])
 *                       + HE[2][i] HE[2][j];  det = g00 g11 - g01 g01;  P = [[g11, -g01], [-g01, g00]] / det . HE^T;
 *                       s_i = maxCRef_i / maxC_i;  M[c][j] = (HERef[c][0] s_0) P[0][j] + (HERef[c][1] s_1) P[1][j];
 *                       od[v] = -log((v + 1) / Io).  valid = both blocks valid, det > 0 and M finite.  One kernel.
 * hipac_stain_apply     d_in uint8 [n_patches][224][224][3]; per pixel and channel c
 *                       y = (M[c][0] od[r] + M[c][1] od[g]) + M[c][2] od[b] (products rounded, no FMA) and
 *                       out_c = #{v in 0..254 : y <= od[v]}, which is uint8(min(255, Io exp(-y))) = torchstain's
 *                       normalize with the source's (HE, maxC).  valid = 0: out = in.  Outputs: d_out_u8 (uint8, may be
 *                       d_in itself, otherwise disjoint) and / or d_batch in `layout` (the stage-1 ToTensor/Normalize
 *                       of out; S2D16 padding columns and channels 12..15 written as zero; layout 0 = no d_batch).
 *                       d_count: NULL = all n_patches, else only patches < clamp(d_count[0] - n_base, 0, n_patches)
 *                       are read and written.  Buffers 16-byte aligned.  One kernel.
 * ------------------------------------------------------------------------------------- */
#define HIPAC_STAIN_BLOCK_DOUBLES 16
#define HIPAC_STAIN_PARAMS_DOUBLES 267
size_t hipac_stain_workspace_bytes(int H, int W);
int hipac_stain_estimate(const uint8_t* d_rgb, int H, int W, int64_t pitch, int Io, double alpha, double beta, double* d_stain,
                         void* d_ws, size_t ws_bytes, void* stream);
int hipac_stain_normalizer(const double* d_src, const double* d_target, int Io, double* d_params, void* stream);
int hipac_stain_apply(const uint8_t* d_in, int n_patches, const int32_t* d_count, int n_base, const double* d_params,
                      uint8_t* d_out_u8, void* d_batch, int layout, void* stream);

/* Early survivor count.  If a pinned host buffer int32[2] is registered (calling thread), every hipac_tile_scan copies
 * {survivors, candidates} into it right after the compaction kernel and records an event; hipac_tile_scan_wait_count
 * blocks only until that copy has landed -- the resample / gather kernels of the same call keep running, so the caller
 * can enqueue the next stage without a pipeline bubble.  Pass NULL to unregister. */
int hipac_tile_scan_set_count_buffer(int32_t* h_count_pinned);
int hipac_tile_scan_wait_count(void);

/* Host -> device copy of `rows` rows of `row_bytes` bytes between pitched buffers (one cudaMemcpy2DAsync on `stream`).
 * The read-once streaming pass of hipac_tile_scan needs a level image whose row pitch is a multiple of 16 bytes and whose
 * base is 16-byte aligned (TMA bulk copies); 3*W generally is not, so callers allocate the device image with
 * pitch = (3*W + 15) & ~15 and land the reader's [rows][3*W] host rows in it with this call (no extra pass over HBM).
 * Replaces the `slide.read_region(...)` -> numpy hand-over of the reference's loop (src/main.py:693-697) as the point
 * where pixels enter the path. */
int hipac_upload_rows(void* d_dst, int64_t dst_pitch, const void* h_src, int64_t src_pitch, int64_t row_bytes, int64_t rows,
                      void* stream);

/* ---------------------------------------------------------------------------------------
 * Lesion-mask rasterisation on the device (SURVEY.md section 8f-3): replaces the Pillow call inside parse_xml_mask
 * (reference src/main.py:388-409: ImageDraw.polygon(coords, outline=255, fill=255) on an "L" image of the level size, one
 * call per annotation), bit-exact against Pillow 12.2.0's polygon fill.  The vertices are the reference's
 * (int(X * level_w / w0), int(Y * level_h / h0)) pairs, computed by the caller.
 *   h_xy / h_offsets  HOST arrays: int32 [total][2] vertices of all polygons back to back, int32 [num_polygons + 1] offsets
 *   d_xy              the same vertices in device memory (8-byte aligned)
 *   H, W              size of the level image the vertices refer to (Pillow clamps the scan range to it)
 *   y_begin, n_rows   the row window [y_begin, y_begin + n_rows) of that image which is rasterised (a slab of the level)
 *   d_mask            uint8 [n_rows][pitch], row 0 = level row y_begin; every covered pixel becomes 255; `clear` zeroes the
 *                     n_rows x W window first
 *   d_workspace       >= hipac_polygon_workspace_bytes() bytes; holds the overflow flag read by hipac_polygon_overflowed
 *                     (1 if some scan line crossed more than 1024 edges: the mask is then incomplete)
 * Asynchronous on `stream` (hipac_polygon_overflowed synchronises it). */
size_t hipac_polygon_workspace_bytes(int num_polygons);
int hipac_polygon_fill(const int32_t* h_xy, const int32_t* h_offsets, int num_polygons, const int32_t* d_xy, uint8_t* d_mask,
                       int H, int W, int64_t pitch, int y_begin, int n_rows, int clear, void* d_workspace, size_t workspace_bytes,
                       void* stream);
int hipac_polygon_overflowed(const void* d_workspace, void* stream);

/* Pillow coefficient tables used by the kernels (known-answer hook for the CPU tests; no GPU needed).
 * scale in {2,4,8}; writes interior[2*scale], left_edge[3*scale/2], right_edge[3*scale/2] (22-bit fixed point). */
int hipac_pillow_coeffs(int scale, int32_t* h_interior, int32_t* h_left, int32_t* h_right);

/* float32 -> bf16 bits of the ToTensor+Normalize LUT, [256][3] (known-answer hook, host only). */
int hipac_normalize_lut_bf16(uint16_t* h_lut);

/* ---------------------------------------------------------------------------------------
 * Stage 2: ResNet18 forward (reference src/models/resnet.py:22-77 = torchvision resnet18
 * trunk, eval-mode BN, global average pool [+ Linear(512,k)]) on a bf16 batch.
 * ------------------------------------------------------------------------------------- */

/* Number of fp32 tensors hipac_resnet18_pack expects and their order: see INTEGRATION.md
 * (conv weight, bn weight, bn bias, bn running_mean, bn running_var per conv, network order;
 * then fc weight [k][512] and fc bias [k], or NULL,NULL for the headless feature extractor). */
#define HIPAC_RESNET18_NUM_CONVS 20
#define HIPAC_RESNET18_NUM_TENSORS (HIPAC_RESNET18_NUM_CONVS * 5 + 2)

size_t hipac_resnet18_packed_bytes(int num_classes);

/* Fold eval-mode BatchNorm into the conv weights (fp32), convert to the bf16 K-major layouts the
 * implicit-GEMM kernels read, write the blob to HOST memory `h_packed` (caller uploads it). */
int hipac_resnet18_pack(const float* const* h_tensors, int num_tensors, int num_classes, float bn_eps,
                        void* h_packed, size_t packed_bytes);

size_t hipac_resnet18_workspace_bytes(int n_patches, int chunk);

/* d_batch: bf16 batch of n_patches in `layout` (HIPAC_LAYOUT_S2D16_BF16 is the native one).
 * d_feats: float32 [n][512]; d_logits: float32 [n][num_classes] or NULL. */
int hipac_resnet18_forward(const void* d_packed, int num_classes,
                           const void* d_batch, int layout, int n_patches,
                           float* d_feats, float* d_logits,
                           void* d_workspace, size_t workspace_bytes, int chunk, void* stream);

/* Same forward with the patch count on the DEVICE: buffers, grids and tensor maps are sized for `capacity` patches and
 * every kernel reads d_count[0] (e.g. the survivor counter written by hipac_tile_scan) when it starts, working on
 * min(d_count[0], capacity) patches.  Nothing waits on the host, so tile scan + forward of one level image are enqueued
 * back to back (and the sequence is CUDA-graph capturable); rows >= d_count[0] of d_feats / d_logits are left untouched.
 * Workspace as for hipac_resnet18_workspace_bytes(capacity, chunk). */
int hipac_resnet18_forward_dcount(const void* d_packed, int num_classes,
                                  const void* d_batch, int layout, int capacity, const int32_t* d_count,
                                  float* d_feats, float* d_logits,
                                  void* d_workspace, size_t workspace_bytes, int chunk, void* stream);

/* Rotation/flip test-time augmentation: the forward on the eight views of every patch under the dihedral group D4, with the
 * features averaged.  View v = 4*f + k (f in {0,1}, k in {0,1,2,3}) of an NHWC image x is
 * torch.rot90(torch.flip(x, dims=[W]) if f else x, k, dims=(H, W)).  d_feats = (((f_0 + f_1) + ...) + f_7) * 0.125 in fp32,
 * f_v = the features hipac_resnet18_forward gives for view v; d_logits = the head applied to d_feats.  Each chunk runs the
 * view kernel (skipped for view 0 of an S2D16 batch), the network and an accumulating pool eight times: 8x the launches of
 * hipac_resnet18_forward (+7 for an S2D16 batch).  Validation and workspace as for hipac_resnet18_forward.  d_count: NULL =
 * host count (n_patches patches), else device-count mode as in hipac_resnet18_forward_dcount (n_patches = capacity; rows
 * >= d_count[0] of d_feats / d_logits are left untouched). */
int hipac_resnet18_forward_d4(const void* d_packed, int num_classes,
                              const void* d_batch, int layout, int n_patches, const int32_t* d_count,
                              float* d_feats, float* d_logits,
                              void* d_workspace, size_t workspace_bytes, int chunk, void* stream);

/* Test hook: D4 view `view` (0..7, see hipac_resnet18_forward_d4) of a bf16 batch in `layout` -> S2D16 d_out
 * [n_patches][112][115][16] (padding columns and channels 12..15 written as zero).  View 0 of an NHWC3 batch is the repack
 * hipac_resnet18_forward runs.  d_count / n_base as for the hooks below: only patches < clamp(d_count[0] - n_base, 0,
 * n_patches) are written.  d_out must not overlap d_in. */
int hipac_batch_d4_view(const void* d_in, int layout, int n_patches, int view, void* d_out, const int32_t* d_count, int n_base,
                        void* stream);

/* The three test hooks below run one stage-2 kernel with the launch state the forward gives it:
 *   reverse  nonzero: walk the tiles from the last to the first (the forward alternates the order from launch to launch);
 *   d_count  NULL: work on all n_patches patches; else device-count mode as in hipac_resnet18_forward_dcount, the kernel
 *            reads d_count[0] when it starts and works on clamp(d_count[0] - n_base, 0, n_patches) patches, leaving the
 *            output rows of the others untouched;
 *   n_base   >= 0: index of the first patch of d_in in the count (the forward's chunk offset).
 * The output does not depend on `reverse`. */

/* Test hook: one conv layer of the network on its own (layer index 1..19 in network order, except 7), bf16 NHWC in/out,
 * optional residual.  Used by the per-layer parity tests.  Layer 0 (conv1) exists only fused with the max pool and layer 7
 * (layer2.0's projection shortcut) only fused into layer2.0.conv2: both are refused with -1, see hipac_resnet18_stem and
 * hipac_resnet18_conv_ds_fused. */
int hipac_resnet18_conv_layer(const void* d_packed, int num_classes, int layer,
                              const void* d_in, const void* d_residual, void* d_out,
                              int n_patches, int relu, void* stream, int reverse, const int32_t* d_count, int n_base);

/* Test hook: conv2 of layer{2,3,4}.0 with its 1x1/stride-2 projection shortcut fused into the same accumulator:
 * out = relu(conv3x3(d_in) + bn + conv1x1_s2(d_block_in) + bn); stage 0/1/2 = layer2/3/4. */
int hipac_resnet18_conv_ds_fused(const void* d_packed, int num_classes, int stage, const void* d_in, const void* d_block_in,
                                 void* d_out, int n_patches, void* stream, int reverse, const int32_t* d_count, int n_base);

/* Test hook: the fused stem (conv1 + folded BN + ReLU + 3x3/s2 max pool): S2D16 batch -> bf16 [n][56][56][64]. */
int hipac_resnet18_stem(const void* d_packed, int num_classes, const void* d_in, void* d_out, int n_patches, void* stream,
                        int reverse, const int32_t* d_count, int n_base);

/* ---------------------------------------------------------------------------------------
 * The exchange step (SURVEY.md section 8e): per-segment survivors -> ONE canonically ordered result.
 * A segment = the outputs of one tile-scan + forward pass over a contiguous range of candidate grid rows (a rank's
 * shard, or one row group of it): rows in emission order (x outer, y inner), count on the device.  The reference has no
 * counterpart (nn.DataParallel only, src/main.py:839-842); the contract is array equality with a single-rank run, whose
 * row order is the reference's loop order (src/main.py:682-683).
 *
 *   hipac_exchange_pack   writes segment = [1 + capacity][row_bytes] bytes: header row {count}, then per survivor
 *                         {x, y + y_offset, label, features[512], logits[num_classes]}.  Segments of equal capacity laid
 *                         side by side are the send / receive buffers of one fixed-size all-gather (the counts ride in
 *                         the headers: no separate count exchange, no host round trip).
 *   hipac_exchange_merge  num_segments segments, ordered by ascending y range (rank after rank, row group after row
 *                         group) -> final arrays in (x, y) order: a binary search per (segment, grid column), one prefix
 *                         sum, one scatter.  d_total[0] = number of rows (device memory; rows beyond out_capacity are
 *                         dropped), d_total[1] = out_capacity.  stride / nx = candidate grid stride and column count.
 * ------------------------------------------------------------------------------------- */
#define HIPAC_FEATURE_DIM 512
/* feat_dim is 512 (rows carry the features) or 0 (coords / labels / logits only, e.g. the heatmap of configs[3]).
 * cyclic_world: 0 = the segments are stored in ascending y order (contiguous row shards); W > 0 = block-cyclic sharding over W
 * ranks (stored rank-major, as an all-gather delivers them): local segment g of rank r is grid-row block g * W + r, which balances
 * spatially clumped tissue across the ranks.
 * hipac_exchange_pack: `capacity` = rows available in the INPUT tensors (<= the segment's row capacity); min(*d_count,
 * capacity) rows are packed.  hipac_exchange_merge: `capacity` = row capacity of every segment (segment stride =
 * hipac_exchange_segment_bytes(capacity, ...)). */
size_t hipac_exchange_row_bytes(int feat_dim, int num_classes);
size_t hipac_exchange_segment_bytes(int capacity, int feat_dim, int num_classes);
size_t hipac_exchange_workspace_bytes(int num_segments, int nx);
int hipac_exchange_pack(const int32_t* d_coords, const uint8_t* d_labels, const float* d_feats, const float* d_logits,
                        int feat_dim, int num_classes, const int32_t* d_count, int capacity, int y_offset, void* d_segment, void* stream);
int hipac_exchange_merge(const void* d_segments, int num_segments, int capacity, int feat_dim, int num_classes, int stride, int nx,
                         int cyclic_world, int32_t* d_coords, uint8_t* d_labels, float* d_feats, float* d_logits, int32_t* d_total,
                         int out_capacity, void* d_workspace, size_t workspace_bytes, void* stream);

/* ---------------------------------------------------------------------------------------
 * ABMIL head over a bag of patch features (SURVEY.md section 8f-4): MILAttentionPooling + MILClassifier of the reference
 * (src/models/mil_classifier.py:5-45), fp32:  a = softmax_i(u . tanh(V x_i + bV) + bu);  M = sum_i a_i x_i;
 * logits = W2 relu(W1 M + b1) + b2.  pooling: 0 attention, 1 mean (x.mean(0)), 2 max (x.max(0)).
 *   hipac_mil_pack     host repack of the module's tensors (torch layouts: V [128][512], bV [128], u = attn_U.weight [1][128],
 *                      bu [1], W1 [128][512], b1 [128], W2 [k][128], b2 [k]; V/bV/u/bu may be NULL for mean / max pooling)
 *                      into hipac_mil_packed_floats(k) floats; the caller uploads the blob.
 *   hipac_mil_forward  d_x float32 [n_instances][512] (e.g. hipac_resnet18_forward's features); d_count: optional int32 device
 *                      counter (min(*d_count, n_instances) instances are pooled, nothing waits on the host);
 *                      d_logits [k]; d_attention [n_instances] or NULL (attention weights, the module's second output);
 *                      d_pooled [512] or NULL.
 * ------------------------------------------------------------------------------------- */
size_t hipac_mil_packed_floats(int num_classes);
int hipac_mil_pack(const float* V, const float* bV, const float* u, const float* bu, const float* W1, const float* b1,
                   const float* W2, const float* b2, int num_classes, float* h_packed);
size_t hipac_mil_workspace_bytes(int n_instances);
int hipac_mil_forward(const float* d_x, int n_instances, const int32_t* d_count, const float* d_packed, int num_classes, int pooling,
                      float* d_logits, float* d_attention, float* d_pooled, void* d_workspace, size_t workspace_bytes, void* stream);

/* Number of kernel launches issued by this library on the calling thread since the last reset
 * (bench.py's "gpu_launches"). */
long long hipac_launch_count(int reset);

/* Test hook for the shifted-descriptor mechanism of the row-tile conv kernels:
 * D[m][n] = sum_k A[m + shift_rows][k] * B[n][k] (m < 128, n < 64) with A [256][K], B [64][K] bf16,
 * K = 64 (swizzle_bytes = 128) or 16 (swizzle_bytes = 32); A and B are TMA-loaded whole, the UMMA A
 * descriptor starts shift_rows rows into the tile. */
int hipac_debug_umma_shift(const void* d_A, const void* d_B, float* d_D, int shift_rows, int swizzle_bytes, void* stream);

/* Optional per-kernel profiler (calling thread): when enabled every kernel launch of the library is
 * bracketed by CUDA events on its stream.  hipac_profile_report synchronises them, writes one line per
 * kernel "<name> <launches> <total_ms> <total_work>" (work = algorithmic bytes for the stage-1 kernels,
 * flops for the conv kernels), clears the records and returns the report length. */
int hipac_profile_enable(int on);
long long hipac_profile_report(char* buf, size_t cap);

#ifdef __cplusplus
}
#endif
#endif /* HIPAC_B200_H */

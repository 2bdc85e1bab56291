/* ssp_b200 -- C ABI of the B200-native homography-warp correspondence path of Semantic-SuperPoint.
 *
 * The reference (Gabriel-SGama/Semantic-SuperPoint) has no FFI: its boundary for this path is a set of
 * Python callables in utils/utils.py, Train_model_heatmap_all.py, export.py and models/model_wrap.py.  Every entry point below
 * names the reference callable (file:line) it serves; the Python host side (semantic-superpoint_b200/*.py)
 * re-exports those callables with unchanged signatures and binds them to this library through ctypes.
 *
 * Conventions
 *   - all pointers are DEVICE pointers unless the name ends in _host; tensors are contiguous fp32 NCHW
 *   - the caller owns every buffer (inputs, outputs, workspaces); nothing is allocated or freed here
 *   - `stream` is a cudaStream_t; calls are stream-ordered and never synchronise, except ssp_nms_fast /
 *     ssp_box_nms whose reference API returns host data (they sync the stream to read counters)
 *   - return value: 0 = ok, < 0 = argument error, > 0 = cudaError_t; ssp_last_error() gives the text
 */
#ifndef SSP_B200_H
#define SSP_B200_H
#include <stddef.h>
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

int ssp_version(void);
const char* ssp_last_error(void);

/* ---- a1 / a10: warp_points (utils/utils.py:315-343), filter_points (:303-311),
 *      warp_keypoints / keep_true_keypoints (evaluations/detector_evaluation.py:139-191) ---- */
int ssp_warp_points_mask(const float* pts /*[P,2] x,y*/, int P, const float* H /*[B,3,3]*/, int B, float shape_x,
                         float shape_y, float* out /*[B,P,2]*/, uint8_t* keep /*[B,P] 0<=p<=shape-1, or NULL*/,
                         void* stream);
int ssp_warp_keypoints_f64(const double* kp /*[K,2] x,y pixels*/, int K, const double* H /*[3,3]*/, double W,
                           double Hh, double* out /*[K,2]*/, uint8_t* keep /*[K] 0<=x<W,0<=y<H*/, void* stream);

/* ---- a2: inv_warp_image_batch / inv_warp_image (utils/utils.py:347-405).
 *      xs[W], ys[H] = the normalised sampling grid (torch.linspace(-1,1,n) of the reference, :375).
 *      mode 0 = bilinear, 1 = nearest (any other value is an argument error); zeros padding, align_corners=True.
 *      One gather kernel: each thread computes the source coordinates of 4 output pixels once and reads their taps
 *      straight from global memory for every channel. ---- */
int ssp_inv_warp_image(const float* img /*[B,C,H,W]*/, int B, int C, int H, int W, const float* Hinv /*[B,3,3]*/,
                       const float* xs, const float* ys, int mode, float* out /*[B,C,H,W]*/, void* stream);

/* ---- a3: compute_valid_mask (utils/utils.py:715-742): nearest warp of ones + erosion by an explicit
 *      structuring element kern[kh,kw] (device, uint8) with anchor (ax,ay); kh == kw == 0 -> no erosion ---- */
int ssp_valid_mask(int B, int H, int W, const float* Hinv, const float* xs, const float* ys, const uint8_t* kern,
                   int kh, int kw, int ax, int ay, float* out /*[B,H,W]*/, void* stream);

/* ---- a4: labels2Dto3D (utils/utils.py:408-440), getMasks (Train_model_frontend_all.py:373-386),
 *      detector_loss (Train_model_heatmap_all.py:155-179) forward / backward.
 *      fused2d = 0: target [B,65,Hc,Wc], mask [B,Hc,Wc] (the reference call signature)
 *      fused2d = 1: target = labels_2D [B,1,H,W], mask = mask_2D [B,1,H,W] (labels2Dto3D+getMasks fused in)
 *      out3 = { loss, numerator, sum(mask)+1e-5 } ---- */
int ssp_labels2d_to_3d(const float* labels /*[B,1,H,W]*/, int B, int H, int W, int add_dustbin,
                       float* out /*[B,64|65,H/8,W/8]*/, void* stream);
int ssp_cell_mask(const float* mask2d /*[B,1,H,W]*/, int B, int H, int W, float* out /*[B,H/8,W/8]*/, void* stream);
size_t ssp_detector_loss_ws_bytes(int B, int Hc, int Wc);
/* one loss (semi1 == NULL: problem 1's pointers are ignored) or both losses of a training pair (image, warped image) in
 * one launch; semi [B,65,Hc,Wc], gout [1]; ws = one region of ws_bytes rounded up to 16 per loss;
 * cellmask1 (optional, [B,Hc,Wc]) receives getMasks() of problem 1 as a by-product */
int ssp_detector_loss_fwd_pair(const float* semi0, const float* target0, const float* mask0, const float* semi1,
                               const float* target1, const float* mask1, int B, int Hc, int Wc, int fused2d,
                               float* out3_0, float* out3_1, float* cellmask1, void* ws, size_t ws_bytes, void* stream);
int ssp_detector_loss_bwd_pair(const float* semi0, const float* target0, const float* mask0, const float* semi1,
                               const float* target1, const float* mask1, int B, int Hc, int Wc, int fused2d,
                               const float* fwd0, const float* fwd1, const float* gout0, const float* gout1,
                               float* dsemi0, float* dsemi1, void* stream);

/* ---- a6: flattenDetection (utils/utils.py:515-560) ---- */
int ssp_flatten_detection(const float* semi /*[N,65,Hc,Wc]*/, int N, int Hc, int Wc, float* heat /*[N,1,8Hc,8Wc]*/,
                          void* stream);

/* a6 fused with the valid mask of each view (the heat * mask product of export.py:53): heat where mask == 1, -1 where mask == 0;
 * *flag (device int, zeroed by the caller) is raised by any other mask value.  Input of ssp_combine_heatmap_signed. */
int ssp_flatten_detection_masked(const float* semi /*[N,65,Hc,Wc]*/, const float* mask /*[N,8Hc,8Wc] 0/1*/, int N, int Hc,
                                 int Wc, float* heat /*[N,1,8Hc,8Wc]*/, int* flag, void* stream);

/* ---- a7: combine_heatmap (export.py:49-60), batched over I source images ---- */
int ssp_combine_heatmap(const float* heat /*[I,N,H,W]*/, const float* mask /*[I,N,H,W]*/,
                        const float* Hinv /*[I,N,3,3]*/, int I, int N, int H, int W, const float* xs, const float* ys,
                        float* out /*[I,H,W]*/, void* stream);
/* the same aggregation from the signed heat of ssp_flatten_detection_masked: one gather per tap (bit-identical results for
 * 0/1 masks; a raised flag turns the output into NaN) */
int ssp_combine_heatmap_signed(const float* heat_signed /*[I,N,H,W]*/, const float* Hinv /*[I,N,3,3]*/, int I, int N, int H,
                               int W, const float* xs, const float* ys, const int* flag /*or NULL*/, float* out /*[I,H,W]*/,
                               void* stream);

/* ---- a8 / a9: getPtsFromHeatmap + nms_fast (utils/utils.py:581-609, 653-712), box_nms (:612-650).
 *      stencil: device (2R+1)^2 bytes, 1 = suppressed offset.  pts: [I,3,capacity] float64 rows x,y,conf,
 *      confidence-descending.  counts_host: HOST int[I].  0 <= R <= 48. ---- */
size_t ssp_nms_ws_bytes(int I, int H, int W, int capacity);
/* byte offset in ssp_nms_fast's workspace of its per-image keypoint counts (device unsigned int[I], valid after the call) */
size_t ssp_nms_ws_counts_offset(int I, int H, int W);
int ssp_nms_fast(const float* heat /*[I,H,W]*/, int I, int H, int W, float conf_thresh, int R, const uint8_t* stencil,
                 int border, int capacity, double* pts, int* counts_host, void* ws, size_t ws_bytes, void* stream);
int ssp_box_nms(const float* prob /*[I,H,W]*/, int I, int H, int W, float min_prob, int R, const uint8_t* stencil,
                float* out /*[I,H,W]*/, void* ws, size_t ws_bytes, void* stream);

/* ---- sub-pixel keypoints (SURVEY 8a): SuperPointFrontend_torch.soft_argmax_points (models/model_wrap.py:212-248) with
 *      extract_patch_from_points / norm_patches / do_log / soft_argmax_2d (utils/losses.py; torchgeometry 0.1.2
 *      SpatialSoftArgmax2d, normalized_coordinates=False), the step the shipped COCO export config runs between NMS and
 *      top-k (configs/magicpoint_coco_export.yaml:44-45, export.py:309-314).  pts: the [I,3,capacity] float64 layout of
 *      ssp_nms_fast, refined in place; image i refines its first min(counts[i], limit, capacity) points.  counts: device
 *      unsigned int[I], e.g. ssp_nms_fast's own (ssp_nms_ws_counts_offset), so no host round trip.  Per point,
 *      (xi, yi) = (int)(x, y), patch = heat[yi - patch/2 + r, xi - patch/2 + c] (zero outside the image), q = patch /
 *      (sum + 1e-6), q < 0 -> 1e-6, l = log q, e = exp(l - max l), s = 1 / (sum e + 1e-6), then in float64
 *      x += sum((c * e) * s) - patch/2 and y += sum((r * e) * s) - patch/2; conf is unchanged.  1 <= patch <= 15. ---- */
int ssp_soft_argmax_points(const float* heat /*[I,H,W]*/, int I, int H, int W, double* pts, int capacity,
                           const unsigned int* counts, int limit, int patch, void* stream);

/* ---- a5: descriptor_loss (utils/utils.py:779-893), forward and backward, split into stages.
 *      Nc = Hc*Wc, Nc_pad = ceil(Nc/256)*256.  wpts [B,Nc_pad,2], mv_pad [B,Nc_pad],
 *      bitsR/bitsC [B,Nc_pad/32,Nc_pad] u32 indicator bit-matrices (element j of a word at bit (j>>1)|((j&1)<<4)),
 *      partials = per-CTA (unweighted, weighted) double pairs.
 *      out8 = { loss, pos_sum, neg_sum, norm, num_loss, num_pos, num_neg, sum(mask_valid) }
 *      mvbits (optional, [B,Nc_pad/32] u32): mask_valid != 0 per cell in the same bit order, for the "fold" mode of the
 *      tensor-core engine (mask folded into the indicator words; a non-binary mask then poisons the normaliser: NaN) ---- */
int ssp_desc_geometry_nblocks(int B, int Nc); /* length of ssp_desc_pack2_geometry's mv_part */
int ssp_desc_pos_nblocks(int B, int Nc);
int ssp_desc_maxp(void); /* DESC_MAXP: list slots per row / column */
/* sparse positive pairs: exact fp32 dots, partial sums (4 doubles per block: pos_u, pos_w, negcorr_u, negcorr_w)
 * and the pair lists rowcol/rowdot/colrow/coldot [B,Nc_pad,DESC_MAXP], colcnt [B,Nc_pad] used by the backward */
int ssp_desc_pos_fwd(const float* D /*[B,Dch,Hc,Wc]*/, const float* Dw, const float* wpts, const float* mv_pad, int B,
                     int Hc, int Wc, int Dch, int cell, float dist, float lamda, float mpos, float mneg,
                     double* partials, int* rowcol, float* rowdot, int* colcnt, int* colrow, float* coldot,
                     void* stream);
/* Same contract from the packed hi/lo planes [B,Nc_pad,256] bf16 of D (A*) and Dw (B*) written by ssp_desc_pack2_geometry
 * (bf16x3 engine): a cell's descriptor is 2 x 512 contiguous bytes there instead of 256 channels 4*Nc bytes apart. */
int ssp_desc_pos_planes_nblocks(int B, int Nc);
int ssp_desc_pos_fwd_planes(const void* Ahi, const void* Alo, const void* Bhi, const void* Blo, const float* wpts,
                            const float* mv_pad, int B, int Hc, int Wc, int cell, float dist, float lamda, float mpos,
                            float mneg, double* partials, int* rowcol, float* rowdot, int* colcnt, int* colrow,
                            float* coldot, void* stream);
int ssp_desc_dense_simt_nblocks(int B, int Nc);
int ssp_desc_dense_fwd_simt(const float* D, const float* Dw, const float* mv_pad, int B, int Hc, int Wc, int Dch,
                            float mneg, double* partials, uint32_t* bitsR, uint32_t* bitsC,
                            float* dbgS /*[B,Nc,Nc] or NULL*/, void* stream);
int ssp_desc_pack(const float* src /*[B,Dch,Nc]*/, const float* scale /*[B,Nc_pad] or NULL*/, int B, int Dch, int Nc,
                  void* hi /*bf16 [B,Nc_pad,Dch]*/, void* lo /*or NULL*/, void* stream);
/* ssp_desc_pack of two tensors (unscaled) and the geometry (warped cell centres wpts, mv_pad and the per-block sums mv_part
 * of mask_valid) as ONE launch: they do not depend on each other.  hi0 == hi1 == NULL: the geometry alone (src*, lo* and
 * Dch unused).  mask2d is used when mask_valid is NULL: [B,1,8Hc,8Wc], getMasks fused in (cell must be 8). */
int ssp_desc_pack2_geometry(const float* src0, const float* src1, int B, int Dch, int Hc, int Wc, void* hi0 /*or NULL*/,
                            void* lo0 /*or NULL*/, void* hi1 /*or NULL*/, void* lo1 /*or NULL*/, const float* H /*[B,3,3]*/,
                            const float* mask_valid /*[B,Nc] or NULL*/, const float* mask2d /*or NULL*/, int cell,
                            float* wpts, float* mv_pad, double* mv_part /*[geometry_nblocks]*/, uint32_t* mvbits /*or NULL*/,
                            void* stream);
int ssp_desc_dense_tc_nblocks(int B, int Nc);
/* tcgen05 forward (CTA-pair MMAs, M=256): negative hinge over all pairs + row-orientation indicator words bitsR (their
 * transpose bitsC comes from ssp_desc_pos_coef).  The lo planes must lie above their hi planes in memory (one allocation).
 * mvbits != NULL ("fold"): the indicator words drop the columns whose mask_valid is 0, so the dD indicator GEMM can take
 * the unscaled forward planes of Dw and one scalar (valid when mask_valid is binary and g_neg = 0). */
int ssp_desc_dense_fwd_tc(const void* Ahi, const void* Alo, const void* Bhi, const void* Blo, const float* mv_pad,
                          const uint32_t* mvbits /*or NULL*/, int B, int Hc, int Wc, float mneg, double* partials,
                          uint32_t* bitsR, float* dbgS, void* stream);
/* overflow (optional) = &colcnt[B*Nc_pad], the counter of positive pairs that did not fit the sparse lists: non-zero
 * makes loss / pos_sum NaN (loud without a host sync) */
int ssp_desc_finalize(const double* pos_part, int npos, const double* neg_part, int nneg, const double* mv_part,
                      int nmv, int B, int Hc, int Wc, const int* overflow, float* out8,
                      const float* det0 /*or NULL*/, const float* det1, float lambda_loss, float* total /*or NULL: fused
                      loss step, total = det0.loss + det1.loss + lambda_loss * loss_desc*/, void* stream);
int ssp_desc_pair_mask(const float* wpts, int B, int Hc, int Wc, int cell, float dist, float* mask /*[B,Nc,Nc]*/,
                       void* stream);
int ssp_desc_alpha(const float* mv_pad, const float* g3 /*[3] dL/d(loss,pos,neg)*/, const float* out8, int B,
                   int Nc_pad, float* alpha /*[B,Nc_pad]*/, void* stream);
/* backward coefficients of the positive pairs (and removal of their negative term).  colrow_sorted receives the column
 * lists ordered by row index (deterministic summation order) with their coefficients in colcoef; the forward's lists
 * are left untouched, so a second backward over the same graph sees the same inputs.
 * g3: gmode 0 -> {dL/dloss, dL/dpos, dL/dneg}; gmode 1 -> g3[0] = dL/dloss only (fused step); both scaled by gscale.
 * alpha_out (optional, [B,Nc_pad]): what ssp_desc_alpha would write for the same scaled gradients; srow_out (optional,
 * [B,Nc_pad]): the same coefficient at mask_valid = 1, the row scale of the folded backward.
 * bitsC_out (optional, then Nc = unpadded cell count): bitsC transposed from bitsR by extra blocks of the same launch. */
int ssp_desc_pos_coef(const int* rowcol, const float* rowdot, const int* colcnt, const int* colrow, const float* coldot,
                      const uint32_t* bitsR, const float* mv_pad, const float* g3, float gscale, int gmode,
                      const float* out8, int B, int Nc_pad, float lamda, float mpos, float* rowcoef, int* colrow_sorted,
                      float* colcoef, float* alpha_out, float* srow_out, uint32_t* bitsC_out, int Nc, void* stream);
/* Backward prologue of the fused loss step (Train_model_heatmap_all.py:295-365 differentiated through the uniform total):
 * ssp_detector_loss_bwd_pair (labels / masks at pixel resolution, both images, one upstream gradient) and ssp_desc_pos_coef
 * (incl. alpha / srow / bitsC outputs) as ONE launch of heterogeneous blocks.  Same results as the two calls. */
int ssp_step_bwd_prologue(const float* semi0, const float* labels0, const float* mask0, const float* semi1,
                          const float* labels1, const float* mask1, int B, int Hc, int Wc, const float* fwd0 /*out3*/,
                          const float* fwd1, const float* gout /*[1]*/, float* dsemi0, float* dsemi1,
                          const int* rowcol, const float* rowdot, const int* colcnt, const int* colrow, const float* coldot,
                          const uint32_t* bitsR, const float* mv_pad, const float* g3, float gscale, int gmode,
                          const float* out8, float lamda, float mpos, float* rowcoef, int* colrow_sorted, float* colcoef,
                          float* alpha_out, float* srow_out, uint32_t* bitsC_out, void* stream);
/* dD[b,:,r] += sum_n rowcoef[b,r,n] Dw[b,:,rowcol[b,r,n]];  dDw[b,:,c] += sum_n colcoef[b,c,n] D[b,:,colrow[b,c,n]] */
int ssp_desc_pos_apply(const int* rowcol, const float* rowcoef, const int* colrow, const float* colcoef, const float* D,
                       const float* Dw, int B, int Dch, int Nc, float* dD, float* dDw, void* stream);
/* indicator GEMM  out[b,d,r] = rowscale[b,r] * sum_k bit(r,k) * colscale[b,k] * src[b,d,k]  (scales may be NULL) */
int ssp_desc_bits_gemm_simt(const uint32_t* bits, const float* src /*[B,Dch,Nc]*/, const float* colscale,
                            const float* rowscale, int B, int Dch, int Nc, float* out /*[B,Dch,Nc]*/, void* stream);
/* tcgen05 indicator GEMMs of the backward (job 0: dD, job 1: dDw) in ONE persistent launch (CTA-pair MMAs, A = indicator
 * bits expanded into TMEM, B = packed planes [B,Nc_pad,256] bf16, Blo above Bhi in memory or NULL), out [B,256,Nc]
 *   out[b,d,r] = rowscale[b,r] * sum_k bit(r,k) * B[b,k,d] + sum_n pcoef[b,r,n] * pos[b,plist[b,r,n],d]
 * with the positive-pair partners read from the packed planes pos_hi (+ pos_lo); plist may be NULL. */
int ssp_desc_bits_gemm_tc_pair(const uint32_t* bits0, const void* Bhi0, const void* Blo0, const float* rowscale0,
                               const int* plist0, const float* pcoef0, const void* pos_hi0, const void* pos_lo0,
                               float* out0, const uint32_t* bits1, const void* Bhi1, const void* Blo1,
                               const float* rowscale1, const int* plist1, const float* pcoef1, const void* pos_hi1,
                               const void* pos_lo1, float* out1, int B, int Nc, void* stream);

/* ---- semantic head: cross entropy with ignore_index, optionally fused with the x8 bilinear upsample ------------
 * (SURVEY 8f rank 1; not part of the five north-star pieces, same boundary.)
 * Replaces Train_model_heatmap_all.py:181-193 (sem_loss = nn.CrossEntropyLoss(ignore_index=133)) and, for the
 * _up8 entry points, also models/SuperPointNet_gauss2_ssmall.py:90 (F.interpolate(sem, x_hw, "bilinear",
 * align_corners=False)): the [B,C,H,W] logits never exist.
 * labels: int64 [B,H,W]; values outside [0,C) other than ignore_index are not counted (the reference asserts).
 * out3 = { loss = sum / count (NaN when nothing is counted), sum, count }.  ws: ssp_sem_ce_ws_bytes(), 8-byte aligned. */
size_t ssp_sem_ce_ws_bytes(int B, int C, int H, int W, int upsampled);
int ssp_sem_ce_fwd(const float* logits /*[B,C,H,W]*/, const long long* labels, int B, int C, int H, int W,
                   int ignore_index, float* lse2 /*[B,H,W] log2-domain log-sum-exp, kept for the backward*/,
                   float* out3, void* ws, size_t ws_bytes, void* stream);
int ssp_sem_ce_bwd(const float* logits, const long long* labels, const float* lse2, int B, int C, int H, int W,
                   int ignore_index, const float* out3, const float* gout /*device scalar*/,
                   float* dlogits /*[B,C,H,W]*/, void* stream);
/* logits_lr [B,C,Hc,Wc], labels [B,8Hc,8Wc], 2 <= C <= 256.  gsum (optional, [B,C,Hc,Wc]) receives the un-normalised
 * gradient sum_pixels w(pixel,cell) (softmax - onehot); ssp_sem_ce_up8_bwd scales it by gout / count. */
int ssp_sem_ce_up8(const float* logits_lr, const long long* labels, int B, int C, int Hc, int Wc, int ignore_index,
                   float* gsum, float* out3, void* ws, size_t ws_bytes, void* stream);
int ssp_sem_ce_up8_bwd(const float* gsum, const float* out3, const float* gout, int B, int C, int Hc, int Wc,
                       float* dlogits /*[B,C,Hc,Wc]*/, void* stream);

/* ---- sparse descriptors: sampling at keypoints and two-way nearest-neighbour matching (SURVEY 8f rank 3) ---------
 * ssp_sample_desc_batch replaces SuperPointFrontend_torch.sample_desc_from_points (models/model_wrap.py:295-313); with
 *   I = 1 and capacity = limit = K: coarse [D,Hc,Wc] fp32, pts = the reference's [3,K] float64 array (x row, y row,
 *   conf row; device memory), desc [D,K] fp32 = bilinear samples (grid_sample align_corners=True, zero padding),
 *   L2-normalised per point.
 * ssp_nn_match replaces the K1 x K2 part of PointTracker.nn_match_two_way (models/model_wrap.py:451-494):
 *   best1[i] = (bits(min_j dist(i,j)) << 32 | argmin_j), best2[j] likewise over i, dist = sqrt(2 - 2 clip(d1_i . d2_j, -1, 1));
 *   ties go to the lowest index (np.argmin).  The threshold / mutual test on 2K numbers stays with the caller. */
int ssp_nn_match(const float* desc1 /*[D,K1]*/, const float* desc2 /*[D,K2]*/, int D, int K1, int K2,
                 unsigned long long* best1 /*[K1]*/, unsigned long long* best2 /*[K2]*/, void* stream);
/* Batched forms for the descriptor export of a batch of image pairs.
 * ssp_sample_desc_batch: coarse [I,D,Hc,Wc], pts [I,3,capacity] float64 (ssp_nms_fast's layout), counts device unsigned[I]
 *   (e.g. ssp_nms_fast's own, ssp_nms_ws_counts_offset).  Image i samples its first min(counts[i], limit) points into
 *   desc [I,D,limit]; its later columns are zeros.  limit <= capacity.
 * ssp_nn_match_batch: P pairs on the tensor cores.  hi1/lo1 [P,R1,256], hi2/lo2 [P,R2,256] = ssp_desc_pack's bf16 planes of
 *   [P,256,limit] fp32 descriptors (R = ceil(limit/256)*256, lo above hi), multiplied as hi*hi + lo*hi + hi*lo (fp32-grade
 *   dots).  Pair p matches its first n1 = min(counts1[p], limit, R1) points against the first n2 = min(counts2[p], limit, R2):
 *   dist, ties and the mutual test of ssp_nn_match / nn_match_two_way, dist < nn_thresh compared in fp32.  matches
 *   [P,3,R1] float64 receives (index 1, index 2, dist) of pair p's nmatch[p] matches (device unsigned[P]) in increasing
 *   index-1 order.  ws: ssp_nn_match_batch_ws_bytes(P, R1, R2) bytes, 8-byte aligned. */
int ssp_sample_desc_batch(const float* coarse, const double* pts, int capacity, const unsigned int* counts, int limit,
                          int I, int D, int Hc, int Wc, int cell, float* desc, void* stream);
size_t ssp_nn_match_batch_ws_bytes(int P, int R1, int R2);
int ssp_nn_match_batch(const void* hi1, const void* lo1, int R1, const void* hi2, const void* lo2, int R2,
                       const unsigned int* counts1, const unsigned int* counts2, int limit, int P, float nn_thresh,
                       double* matches, unsigned int* nmatch, void* ws, size_t ws_bytes, void* stream);

/* ---- sparse descriptor loss (SURVEY 8f rank 2): utils/loss_functions/sparse_loss.py:65-284 with
 * pixelwise_contrastive_loss.py:140-265 (dist "cos", method "1d").  The reference samples K matches and Kn non-matches per
 * image on the host; the lists ia / ib [B, K+Kn] (int32 cell indices into `descriptors` / `descriptors_warped`, matches
 * first) are inputs.  Dt / Dwt are the descriptors in cell-major layout [B, Nc, Dch] (ssp_transpose_batched of NCHW).
 * out3 = batch means {loss, match, nonmatch}; dots [B,K+Kn] and stats [B,4] {match, nonmatch, loss, hard count} feed the
 * backward, which scatters into cell-major gradients dDt / dDwt (zeroed by the call; fp32 atomics). ---- */
int ssp_transpose_batched(const float* src /*[B,rows,cols]*/, int B, int rows, int cols, float* dst /*[B,cols,rows]*/,
                          void* stream);
int ssp_sparse_desc_loss_fwd(const float* Dt, const float* Dwt, const int* ia, const int* ib, int B, int Nc, int Dch, int K,
                             int Kn, float lamda, float mpos, float mneg, float* dots, float* stats, float* out3,
                             void* stream);
int ssp_sparse_desc_loss_bwd(const float* Dt, const float* Dwt, const int* ia, const int* ib, const float* dots,
                             const float* stats, const float* g3 /*device [3]*/, int B, int Nc, int Dch, int K, int Kn,
                             float lamda, float mpos, float mneg, float* dDt, float* dDwt, void* stream);
/* ssp_sparse_sample draws those lists on the device, with the distribution of the reference's sample_correspondences
 * (sparse_loss.py:170-255, correspondence_finder.py:191-320), not its RNG stream.  Per image b: the candidates are the cells
 * a whose warp by T^-1 mat_H[b] T (normalised -> cell coordinates), rounded half to even, lands in [0,Wc-1] x [0,Hc-1]
 * (M[b] of them); the K matches are a uniformly random K-subset of them in random order (M >= K), or all M in random order
 * followed by K - M draws with replacement (M < K); the K*nper non-matches pair matches_a[k] (repeated nper times) with
 * uniform cells.  ia / ib [B, K + K*nper] int32, matches first.  Hc * Wc <= 8192.  state [4] uint64 device: {seed, launch
 * counter, 0, images with M = 0 so far}; the launch reads the counter and advances it by one (no host involvement: graph
 * replays draw fresh lists).  An image with M = 0 gets ia = ib = -1 (it adds nothing to the loss) and counts in state[3].
 * ssp_sparse_finalize (optional M, total) turns out3 into NaN when some M[b] = 0 and writes
 * total = det0[0] + det1[0] + lambda_loss * out3[0] (det0 / det1: detector-loss triples) when total is not NULL. */
int ssp_sparse_sample(const float* mat_H /*[B,3,3]*/, int B, int Hc, int Wc, int K, int nper, unsigned long long* state,
                      int* ia, int* ib, int* M /*[B]*/, void* stream);
int ssp_sparse_finalize(const int* M /*[B] or NULL*/, int B, float* out3, const float* det0, const float* det1,
                        float lambda_loss, float* total /*or NULL*/, void* stream);

/* ---- homography sampler (SURVEY 8f rank 4): sample_homography_np (utils/homographies.py:12-141) on the device, at the
 * arguments of its call sites (datasets/Coco.py:261-277, :342-347): shape [2,2], shift -1, allow_artifacts, no translation
 * overflow.  The distribution of the reference, not its RNG stream; one thread per homography, float64 arithmetic.
 * flags: 1 perspective, 2 scaling, 4 rotation, 8 translation.  homographies [B,3,3] = the inverse of the sampled transform
 * (the callers' convention, Coco.py:345), inv_homographies [B,3,3] = the inverse of that fp32 matrix; with group > 0 every
 * index that is a multiple of group is the identity (Coco.py:271, one group per source image).  state [4] uint64 device:
 * {seed, launch counter, 0, unused}; the launch reads the counter and advances it by one, as ssp_sparse_sample does, from
 * disjoint Philox counters (one seed serves both samplers). ---- */
int ssp_sample_homography(int B, int flags, int n_scales, int n_angles, double scaling_amplitude,
                          double perspective_amplitude_x, double perspective_amplitude_y, double patch_ratio, double max_angle,
                          int group, unsigned long long* state, float* homographies, float* inv_homographies, void* stream);

/* ---- label warping of the warped training pair (SURVEY 8f rank 4): datasets/data_tools.py:37-63 warpLabels (+ :6-34
 * get_labels_bi), call sites datasets/Coco.py:330,367.  pnts [B,Pmax,2] (x, y) fp32, counts[b] valid points per image
 * (device), Hpix [B,3,3] = homography_scaling_torch(homography, H, W) (pixel coordinates, computed by the host like the
 * reference).  labels [B,1,H,W], res [B,H,W,2], labels_bi [B,1,H,W] (bilinear != 0), warped [B,Pmax,2] holding kept[b]
 * in-bounds warped points in their original order.  Duplicate targets: the last point wins, like the reference's
 * sequential index_put.  ws: ssp_warp_labels_ws_bytes(). ---- */
size_t ssp_warp_labels_ws_bytes(int B, int H, int W);
int ssp_warp_labels(const float* pnts, const int* counts, int B, int Pmax, int H, int W, const float* Hpix, int bilinear,
                    float* labels, float* res, float* labels_bi /*or NULL*/, float* warped, int* kept, void* ws,
                    size_t ws_bytes, void* stream);

/* ---- evaluation of exported image pairs (evaluation.py:86-499 of the reference lineage, with
 * evaluations/detector_evaluation.py and evaluations/descriptor_evaluation.py).  Pair p's points are pts1 / pts2
 * [P,3,cap] float64 (x, y, conf rows, as ssp_nms_fast writes them); it uses its first min(counts[p], limit) points of each
 * image.  Hs [P,2,9] float64: H (image 1 -> image 2, pixel coordinates) and its inverse as the caller computes it.  Matches
 * [P,3,Lmax] float64 (index 1, index 2, distance) with nmatch[p] valid entries: ssp_nn_match_batch's output.
 *
 * ssp_ransac_homography: n = n_sets * P problems; problem q = set * P + p takes pair p's matches, all of them (set 0) or, in
 * set 1, those with distance < subset_dist, in list order; Lmax <= 8192.  M hypotheses per problem, all evaluated: 4
 * distinct matches from Philox4x32-10 (key seed, counter (q, hypothesis, draw block, 1 << 31)), OpenCV's
 * haveCollinearPoints (every triple, both images) and checkSubset sign test, the 4-point DLT (h33 = 1) in float64; a
 * rejected sample scores nothing.  Match j is an inlier when ||pi(H p1_j) - p2_j||^2 <= thresh^2 (|w| <= FLT_EPSILON: an
 * outlier); coordinates enter as fp32 (exact for integer positions).  The hypothesis with the most inliers wins, the lowest
 * index on ties; H [n,9] is OpenCV's normalised DLT refit on its inliers (h33 = 1, no Levenberg-Marquardt step), ninl [n]
 * and mask [n,Lmax] (uint8, over the problem's list) its inliers, best [n] its index.  No estimate (fewer than 4 matches,
 * no hypothesis with 4 inliers, a degenerate refit): H all NaN, ninl 0, mask 0, best -1.  samples [n,M,4] int32 (the drawn
 * indices, -1 when the problem has fewer than 4 matches) and hyp_inliers [n,M] int32 (-1 = rejected sample) are optional
 * outputs (NULL in production).  ws: ssp_ransac_homography_ws_bytes(n, M).
 *
 * ssp_eval_repeatability: out [P,2] = (repeatability, localisation error) of compute_repeatability
 * (detector_evaluation.py:152-283): float64 warps, strict in-bounds masks, the keep_k most confident points of each side
 * (ties at the cut resolved as a stable sort), mutual nearest distances <= dist_thresh; (0, -1) when nothing matches.
 *
 * ssp_eval_match_metrics: out [P,3+T] = (mean corner distance of H_est[p] from H, matching score, NN mAP, then
 * mean_dist <= correctness_thresh[t] as 0 / 1), from the RANSAC results of ssp_ransac_homography (problems 0..P-1 on all
 * matches; with map_gt == 0 problems P..2P-1 on the matches closer than subset_dist, whose inlier masks label the mAP
 * matches; map_gt == 1 labels them by ||pi(H p1) - p2|| < 3).  correctness_thresh: HOST array of T <= 8 values.  The
 * matching score is 2 ninl / (K1 + K2'), K2' counting image 2's points whose integer-truncated back-warp by fp32(H^-1)
 * lies inside the image (warpLabels' arithmetic); AP is average_precision_score with score = -distance. ---- */
size_t ssp_ransac_homography_ws_bytes(int n, int M);
int ssp_ransac_homography(const double* pts1, int cap1, const double* pts2, int cap2, const double* matches,
                          const unsigned int* nmatch, int Lmax, int P, int n_sets, double subset_dist, int M, double thresh,
                          unsigned long long seed, double* H, int* ninl, unsigned char* mask, int* best,
                          int* samples /*or NULL*/, int* hyp_inliers /*or NULL*/, void* ws, size_t ws_bytes, void* stream);
int ssp_eval_repeatability(const double* pts1, int cap1, const unsigned int* counts1, const double* pts2, int cap2,
                           const unsigned int* counts2, int limit, int P, const double* Hs, int Himg, int Wimg, int keep_k,
                           double dist_thresh, double* out, void* stream);
int ssp_eval_match_metrics(const double* pts1, int cap1, const unsigned int* counts1, const double* pts2, int cap2,
                           const unsigned int* counts2, int limit, int P, const double* Hs, int Himg, int Wimg,
                           const double* matches, const unsigned int* nmatch, int Lmax, double subset_dist,
                           const double* H_est, const int* ninl, const unsigned char* mask, int map_gt,
                           const double* correctness_thresh, int T, double* out, void* stream);

/* ---- multi-GPU (SURVEY 8e): exchange of the global-batch normalisers of the loss step as ONE kernel over peer memory.
 * The reference is single-GPU; what has to agree with it on a batch sharded by pair is the whole-batch divisors of
 * detector_loss (Train_model_heatmap_all.py:178), descriptor_loss (utils/utils.py:886-887) and sem_loss (:181-193).
 * Every rank owns one exchange buffer (ssp_xchg_alloc: the only allocation this library makes, because cudaIpc can
 * only export a cudaMalloc'ed base pointer), exports it as a 64-byte cudaIpcMemHandle_t (HOST memory) and maps the
 * buffers of the other ranks of the node (ssp_xchg_open).  ssp_loss_exchange pushes the local sums into every rank's
 * buffer (peer stores over NVLink + release flag), waits for everybody's flags in local memory, adds in rank order
 * and rewrites det0/det1 {loss, numerator, sum(mask)+1e-5}, desc8 (out8 of ssp_desc_finalize) and sem0/sem1
 * {loss, sum, count} in place with the global-batch values (any of them may be NULL).  Stream-ordered, graph
 * capturable, no NCCL.  A peer that does not arrive within timeout_s poisons the outputs with NaN and sets the
 * sticky error that ssp_xchg_status reports (it synchronises the stream). ---- */
int ssp_xchg_max_ranks(void);
int ssp_xchg_alloc(void** buf, void* ipc_handle64_host);
int ssp_xchg_open(const void* ipc_handle64_host, void** peer_buf);
int ssp_xchg_close(void* peer_buf);
int ssp_xchg_free(void* buf);
int ssp_xchg_status(const void* local_buf, void* stream);
int ssp_loss_exchange(const void* const* bufs_host /*[world] device pointers, own buffer at [rank]*/, int rank, int world,
                      float* det0, float* det1, float* desc8, float* sem0, float* sem1, int B_local, int Hc, int Wc,
                      float lambda_loss, float* total /*or NULL: det0.loss + det1.loss + lambda_loss * desc.loss*/,
                      double timeout_s, void* stream);

/* ---- profiling aid (not on the product path): timeline trace of the two tcgen05 kernels.  Only a library built with
 * -DSSP_TRACE (SSP_TRACE=1 python -m ...build) records anything; the default build returns an error.  buf holds
 * grid * 4 roles * ssp_debug_trace_cap() int64 records (clock64 << 8 | tag), NULL switches tracing off. ---- */
int ssp_debug_trace(void* buf);
int ssp_debug_trace_cap(void);

#ifdef __cplusplus
}
#endif
#endif /* SSP_B200_H */

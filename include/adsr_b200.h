/* adsr_b200 -- C ABI of the B200-native DRCT / DRN super-resolution + anomaly-scoring hot path.
 *
 * The reference (Benedict3007/anomaly-detection-super-resolution) has NO FFI / operator layer: its
 * seams are Python symbols (SURVEY.md section 8b).  Each entry point below therefore cites the reference
 * Python call site(s) whose device work it replaces.  The Python host side
 * (anomaly-detection-super-resolution_b200/{drct,drn,metrics,evaluate}.py) binds these with ctypes;
 * INTEGRATION.md shows the stub a reference maintainer would add.
 *
 * Conventions
 *   - every pointer is a raw DEVICE pointer unless named host_*; bf16 tensors are passed as void*
 *   - nothing is allocated here: outputs and workspaces are caller-owned
 *   - `stream` is a cudaStream_t passed as void*; every call only ENQUEUES work on it, never syncs
 *   - return value: 0 = ok, otherwise one of ADSR_ERR_* (never aborts, never prints)
 *   - stateless and re-entrant (the only cached state is the per-process max-shared-memory opt-in)
 *   - activations are token-major ("NHWC") bf16: row m = (b*H + y)*W + x, `ld*` = row pitch in elements
 */
#ifndef ADSR_B200_H_
#define ADSR_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define ADSR_ABI_VERSION 21

#define ADSR_OK 0
#define ADSR_ERR_BAD_SHAPE 1   /* unsupported dimensions (e.g. window size whose N does not tile 64) */
#define ADSR_ERR_BAD_ALIGN 2   /* pointer / pitch alignment requirement violated */
#define ADSR_ERR_LAUNCH 3      /* kernel launch failed (cudaGetLastError) */
#define ADSR_ERR_CUDA 4        /* a CUDA runtime call failed */
#define ADSR_ERR_ARCH 5        /* device is not sm_100 */

#define ADSR_ACT_NONE 0
#define ADSR_ACT_LRELU 1
#define ADSR_ACT_GELU 2        /* exact erf GELU (nn.GELU default, src/drct.py:175) */
#define ADSR_ACT_RELU 3

#define ADSR_OUT_ROWS 0            /* out[m*ldo + ocol0 + n] */
#define ADSR_OUT_PIXEL_SHUFFLE2 1  /* nn.PixelShuffle(2): n = c*4+i*2+j -> out[b,2y+i,2x+j,c] */

int adsr_abi_version(void);
const char* adsr_status_string(int status);
/* 0 if the current device is compute capability 10.x, ADSR_ERR_ARCH otherwise; *num_sms receives the SM count */
int adsr_device_check(int* host_num_sms);

/* ---- tcgen05 GEMM: out = alpha * act(A[M,K] * W^T + bias) + res ------------------------------------
 * replaces nn.Linear qkv / proj / fc1 / fc2 (src/drct.py:278, 300, 185-188) and the 1x1 `adjust` convs
 * with their LeakyReLU / 0.2*x5 + x epilogues (src/drct.py:334-374, 389-396).
 * w_packed / bias_padded come from pack.pack_gemm_weight(): n_tiles tiles of BN rows, K padded to 64.
 * ln_colsum != NULL fuses the preceding nn.LayerNorm(K, eps=ln_eps) (norm1 / norm2, src/drct.py:432, 438, 481, 510):
 * A then holds the RAW rows, w_packed carries gamma (pack.pack_ln_gemm_weight), bias_padded carries beta W^T + b,
 * ln_colsum[n] = sum_k gamma_k W[n,k]; row mean / rstd come from ln_stats_in: per row `stats_in_stride` (sum, sumsq)
 * float pairs of which the first `stats_in_slots` are added up.
 * stats_out != NULL makes THIS call emit such partials for its own output rows (over the N valid columns, after
 * bias / activation / alpha / residual): slot = stats_out_slot0 + 2 * n_tile + {0,1}; needs slot0 + 2*n_tiles <= stride.
 * reverse_tiles != 0 (row-tile kernel, also adsr_swin_mlp*_bf16): the persistent CTAs walk the 128-row tiles from the LAST one down --
 * when the kernel that produced A wrote it front to back, the rows it wrote last are the ones still in the 126 MB L2. */
int adsr_tc_gemm_bf16(const void* A, int64_t lda, int M, int K,
                      const void* w_packed, const float* bias_padded, int N, int BN, int n_tiles,
                      int act, float slope, float alpha,
                      const void* res, int64_t ldres,
                      void* out, int64_t ldo, int ocol0, int n_store,
                      const float* ln_colsum, float ln_eps, const float* ln_stats_in, int stats_in_slots, int stats_in_stride,
                      float* stats_out, int stats_out_slot0, int stats_out_stride,
                      int reverse_tiles, int num_sms, void* stream);

/* ---- fused Swin MLP half: z = y + fc2(GELU(fc1(LayerNorm(y))))   (one kernel, hidden activations stay in TMEM) ----
 * replaces norm2 + Mlp.forward + the second residual of SwinTransformerBlock.forward (src/drct.py:510, 173-190).
 * w1_packed / w2_packed / bias1 / colsum1 / bias2 / plan come from pack.pack_swin_mlp(): the fc1 weights carry the
 * LayerNorm gamma, fc2 carries the 0.5 of GELU; `plan` (host memory, int32) is the static tiling
 *   [ks1, k1steps, nc, hc, n2, acc1_col0, acc1_col1, n_pieces, piece_rows0, piece_rows1, w1_slots, w1_slot_bytes,
 *    w2_slots, w2_slot_bytes, hcw[8]].
 * Row mean / rstd come from ln_stats_in exactly as in adsr_tc_gemm_bf16.  y and z must not alias. */
int adsr_swin_mlp_bf16(const void* y, int64_t ldy, int M, int C,
                       const void* w1_packed, const void* w2_packed,
                       const float* bias1, const float* colsum1, const float* bias2,
                       const int32_t* plan, int plan_len, float ln_eps,
                       const float* ln_stats_in, int stats_in_slots, int stats_in_stride,
                       void* z, int64_t ldz, int reverse_tiles, int num_sms, void* stream);

/* Same kernel with the adjust 1x1 conv of the RDG folded in (src/drct.py:389-393: x_k = LReLU_0.2(adjust_k(swin_k(...))) appended to
 * the dense feature slab): out[:, ocol0 + n] = LReLU(z W_adj^T + b_adj)[n] for the 32 new channels, where z is the MLP result above.
 * fc2 and the conv have nothing non-linear between them and nothing else reads z, so the conv is folded INTO fc2:
 *   W_adj (y + W2 g + b2) = y W_adj^T + g (W_adj W2)^T + (b_adj + W_adj b2)
 * -- w2_packed holds the 32 rows of W_adj W2 (n2 = 32), the accumulator starts as y W_adj^T (wadj_packed, resident in shared
 * memory), bias_adj is the combined bias, and there is no z and no residual pass.  All of it comes from
 * pack.pack_swin_mlp(..., adjust_w, adjust_b), whose plan is extended by (0, 1): plan[23] != 0 marks the folded layout (plan_len
 * >= 24 is required here, and adsr_swin_mlp_bf16 rejects such a pack).  stats_out receives the per-row (sum, sumsq) of the 32 new
 * columns in slot stats_out_slot0 (slot0 + 1 is zeroed), for the LayerNorm folds of the following blocks. */
int adsr_swin_mlp_adjust_bf16(const void* y, int64_t ldy, int M, int C,
                              const void* w1_packed, const void* w2_packed,
                              const float* bias1, const float* colsum1, const float* bias2,
                              const int32_t* plan, int plan_len, float ln_eps,
                              const float* ln_stats_in, int stats_in_slots, int stats_in_stride,
                              const void* wadj_packed, const float* bias_adj, float slope,
                              void* out, int64_t ldo, int ocol0,
                              float* stats_out, int stats_out_slot0, int stats_out_stride, int reverse_tiles, int num_sms, void* stream);

/* Same kernel with a WIDE 1x1 conv and its residual folded in -- adjust5 of the RDG (src/drct.py:394-396: `x5 = adjust5(swin5(...));
 * return x5 * 0.2 + x`):   out[:, :c_out] = res[:, :c_out] + alpha (W_a z + b_a),  z = the MLP result above, computed as
 *   res + y (alpha W_a)^T + g (alpha W_a W2)^T + alpha (b_a + W_a b2)
 * -- w2_packed holds, per tile, the (K slab, N piece) slabs of alpha W_a followed by the chunk slabs of alpha W_a W2; bias2 is the
 * combined bias (n2 = c_out rounded up to 16 entries); the plan ends in (0, 2).  All of it comes from
 * pack.pack_swin_mlp_conv_res().  The residual tile replaces the consumed y tile in shared memory and the result leaves by TMA, so
 * res and out need 16-byte aligned rows (ld % 8 == 0) and MAY alias (the in-place update of the dense-feature slab).  stats_out
 * (optional) receives the row's (sum, sumsq) over the c_out output columns as FOUR partial slots stats_out_slot0 .. +3 (one per
 * column group of the epilogue; a consumer's LayerNorm fold adds its slots up).  z is never written. */
int adsr_swin_mlp_conv_res_bf16(const void* y, int64_t ldy, int M, int C,
                                const void* w1_packed, const void* w2_packed,
                                const float* bias1, const float* colsum1, const float* bias2,
                                const int32_t* plan, int plan_len, float ln_eps,
                                const float* ln_stats_in, int stats_in_slots, int stats_in_stride,
                                const void* res, int64_t ldres, void* out, int64_t ldo, int c_out,
                                float* stats_out, int stats_out_slot0, int stats_out_stride, int reverse_tiles, int num_sms, void* stream);

/* ---- fused attention half of a Swin block for 8 x 8 windows ------------------------------------------------------
 *   y = x + proj( WindowAttention( LayerNorm(x) ) )
 * replaces norm1 + torch.roll + window_partition + WindowAttention.forward (qkv Linear, q k^T * scale + relative position
 * bias + shift mask, softmax, P v, proj Linear) + window_reverse + torch.roll + the first residual of
 * SwinTransformerBlock.forward (src/drct.py:478-509, 271-302, 193-220, 449-470) in ONE kernel: q | k | v and the
 * attention output stay in tensor memory / shared memory.
 * x: [B*H*W, >= C] bf16 raw token rows (row pitch ldx >= C rounded up to 16), row statistics from ln_stats_in exactly as
 * in adsr_tc_gemm_bf16.  w1_packed / w2_packed / bias_qkv / colsum_qkv / bias_proj come from pack.pack_swin_attn().
 * adsr_swin_attn_mode(C, heads, head_dim_padded, allow_proj) tells what the kernel covers for a block shape:
 *   2 = the whole half (fuse_proj = 1: out = y [M, >= C], stats_out receives the per-row (sum, sumsq) of y for the norm2
 *       fold of adsr_swin_mlp_bf16),
 *   1 = qkv + attention only (fuse_proj = 0: out = attention rows [M, heads * head_dim_padded]; the proj Linear and the
 *       residual are then one adsr_tc_gemm_bf16 call),
 *   0 = shape not covered (use adsr_tc_gemm_bf16 + adsr_window_attention).
 * Requires H % 8 == W % 8 == 0 and an even number of windows; x and out must not alias. */
int adsr_swin_attn_mode(int C, int heads, int head_dim_padded, int allow_proj);
int adsr_swin_attn_bf16(const void* x, int64_t ldx, int B, int H, int W, int C, int shift, int heads, int head_dim,
                        int head_dim_padded, const void* w1_packed, const void* w2_packed,
                        const float* bias_qkv, const float* colsum_qkv, const float* bias_proj, const float* bias_table,
                        float ln_eps, const float* ln_stats_in, int stats_in_slots, int stats_in_stride,
                        int fuse_proj, void* out, int64_t ldo,
                        float* stats_out, int stats_out_slot0, int stats_out_stride, int num_sms, void* stream);

/* ---- tcgen05 implicit-GEMM 3x3 convolution (pad 1, stride 1|2) on NHWC bf16 -------------------------
 * replaces conv_after_body / conv_before_upsample(+LeakyReLU) / Upsample convs + nn.PixelShuffle(2)
 * (src/drct.py:837, 844-845, 702-705, 893-895) and DRN's default_conv / DownBlock convs
 * (src/drn.py:29-32, 83-119).  out_mode selects plain rows or the fused PixelShuffle(2) store. */
int adsr_conv3x3_igemm_bf16(const void* in, int64_t ld_in, int B, int Hin, int Win, int Cin, int stride,
                            const void* w_packed, const float* bias_padded, int N, int BN, int n_tiles,
                            int act, float slope, float alpha,
                            const void* res, int64_t ldres,
                            void* out, int64_t ldo, int ocol0, int out_mode, int n_store,
                            int num_sms, void* stream);

/* ---- halo-tile 3x3 convolution (pad 1, stride 1) with weights resident in shared memory ----------------
 * replaces the two default_conv of every RCAB (src/drn.py:143-158; 80 -> 80 channels in DRN-L): Cin <= 128, Cout <= 128,
 * 8 <= W <= 126, plain-row output with bias and optional ReLU / LeakyReLU.  `w_compact` is the K-concatenated image of
 * pack.pack_conv3x3_weight(...).compact.  ADSR_ERR_BAD_SHAPE = shape not covered (use adsr_conv3x3_igemm_bf16).
 * chan_part (nullable): fp32 [B * parts, BN], parts = 4 * ceil(H * (W + 2) / 128): per-image partial column sums of the outputs
 * (fp32, before the bf16 rounding), the input of adsr_channel_mean_parts -- CALayer's AdaptiveAvgPool2d(1) (src/drn.py:126, 137)
 * without a second pass over the conv output. */
int adsr_conv3x3_halo_bf16(const void* in, int64_t ld_in, int B, int H, int W, int Cin,
                           const void* w_compact, const float* bias_padded, int N, int BN,
                           int act, float slope, void* out, int64_t ldo, int ocol0, int n_store,
                           float* chan_part, int num_sms, void* stream);
/* mean[b, c] = (sum over the `parts` partial rows of image b) / HW, summed in a fixed order (deterministic).  With w1 != NULL the
 * kernel continues with CALayer's conv_du (src/drn.py:128-133) and writes sigmoid(W2 relu(W1 mean + b1) + b2) into `mean` instead:
 * adsr_rcab_ca_scale then takes that buffer as its scales. */
int adsr_channel_mean_parts(const float* chan_part, int B, int parts, int ld_part, int C, int HW, float* mean,
                            const float* w1, const float* b1, const float* w2, const float* b2, int Cr, void* stream);

/* ---- LayerNorm over the first C columns of each row (eps, affine); writes round16(C) columns ---------
 * replaces nn.LayerNorm norm1 / norm2 / final norm (src/drct.py:432, 438, 833, 881). */
int adsr_layernorm_rows(const void* in, int64_t ldi, void* out, int64_t ldo,
                        const float* gamma, const float* beta, int M, int C, float eps, void* stream);

/* ---- fused (shifted-)window multi-head attention ------------------------------------------------------
 * replaces torch.roll + window_partition + WindowAttention.forward (q*scale, q@k^T, +relative position
 * bias, +shift mask (-100), softmax, @v) + window_reverse + roll back
 * (src/drct.py:482-505, 193-220, 271-299, 449-470).
 * qkv: [B*H*W, ldq] with q|k|v blocks of nH heads, each head padded to hdp (multiple of 16) columns;
 * out: [B*H*W, ldo], head h at column h*hdp, written at the ORIGINAL (un-shifted) token position.
 * bias_table: fp32 [(2ws-1)^2, nH] = relative_position_bias_table. */
int adsr_window_attention(const void* qkv, int64_t ldq, void* out, int64_t ldo, const float* bias_table,
                          int B, int H, int W, int ws, int shift, int nH, int hd, int hdp, void* stream);

/* ---- index maps (bit-exact objects): gather map of roll+partition and region ids of calculate_mask ------
 * src/drct.py:193-204, 449-463, 482-489.  src_index / region_id: int32 [ (H/ws)*(W/ws) * ws*ws ]. */
int adsr_window_index_map(int H, int W, int ws, int shift, int32_t* src_index, int32_t* region_id, void* stream);

/* ---- standalone LayerNorm + cyclic shift + window partition, and its inverse (first parity slice) -------
 * src/drct.py:481-489 and 497-505.  windows: [B*nW*N, ldw]. */
int adsr_ln_shift_partition(const void* x, int64_t ldx, void* windows, int64_t ldw,
                            const float* gamma, const float* beta, float eps,
                            int B, int H, int W, int C, int ws, int shift, void* stream);
int adsr_window_reverse_unshift(const void* windows, int64_t ldw, void* x, int64_t ldx,
                                int B, int H, int W, int C, int ws, int shift, void* stream);

/* ---- DRCT head: (x - mean)*img_range -> conv_first 3x3 -> x0 (long skip) and LayerNorm(x0) -> slab -------
 * src/drct.py:887-892, 650-654 (patch_embed.norm).  x: fp32 NCHW, weights fp32 [C, nc, 3, 3].
 * stats_out (optional): (sum, sumsq) of each slab row in slot 0 and zeros in slots 1..3 (the slots the adjust5 epilogue
 * fills from the second RDG on), for the first folded LayerNorm. */
int adsr_drct_head(const float* x_nchw, int B, int nc, int H, int W,
                   const float* weight, const float* bias, const float* mean, float img_range,
                   const float* ln_gamma, const float* ln_beta, float eps, int C,
                   void* x0, int64_t ld0, void* slab, int64_t lds,
                   float* stats_out, int stats_out_stride, void* stream);

/* ---- DRCT tail: conv_last 3x3 (Cin -> nc) + x/img_range + mean, fused uint8 truncation ------------------
 * src/drct.py:895-897 and the quantisation of src/evaluate.py:212-215
 * (u8 = trunc(clamp(sr * 255/rgb_range, 0, 255)), HWC).  Either output pointer may be NULL. */
int adsr_conv_last_quant(const void* in, int64_t ld_in, int B, int H, int W, int Cin,
                         const float* weight, const float* bias, int nc, const float* mean, float img_range,
                         float rgb_range, float* out_nchw, uint8_t* out_u8_hwc, void* stream);

/* uint8 HWC images (PNG decoder output, host-pinned then copied as bytes: a quarter of the fp32 traffic) -> fp32 NCHW in
 * [0, rgb_range]: the reference loader's np2Tensor, `tensor.mul_(rgb_range / 255)` (src/data.py:11-17), on the device. */
int adsr_u8_to_float_nchw(const uint8_t* x_u8_hwc, int B, int nc, int H, int W, float rgb_range, float* out_nchw, void* stream);

/* ---- uint8 truncation of an fp32 NCHW image batch (HR side of src/evaluate.py:215) ----------------------- */
int adsr_quantize_u8(const float* x_nchw, int B, int nc, int H, int W, float rgb_range, uint8_t* out_u8_hwc,
                     void* stream);

/* ---- DRN-only bandwidth-bound pieces --------------------------------------------------------------------------
 * adsr_bicubic_affine: nn.Upsample(scale, 'bicubic', align_corners=False) + the sub_mean MeanShift 1x1 conv
 *   (src/drn.py:174-175, 243-246); mat = [nc, nc] fp32, bias = [nc].   fp32 NCHW in and out.
 * adsr_conv3x3_small: `head` conv, Cin <= 3 (fp32 NCHW) -> C <= 64 channels NHWC bf16 (src/drn.py:187, 247), written to
 *   out1 and, optionally, to the column slice col2.. of out2 (the skip-connection half of the later torch.cat).
 * adsr_channel_mean: the pooling partials of CALayer (src/drn.py:126, 137) where the halo conv does not run: x [B, HW, ld] bf16
 *   (C % 8 == 0, 16-byte aligned rows) -> part[(b * slices + s) * ld_part + c] = column sums of pixel slice s, for
 *   adsr_channel_mean_parts(part, B, slices, ...): a fixed summation order, so the result does not depend on scheduling or the batch.
 * adsr_rcab_ca_scale: out = res * scale[b] + x   (src/drn.py:139, 155-158), scale [B, C] from adsr_channel_mean_parts with the MLP. */
int adsr_bicubic_affine(const float* x_nchw, int B, int nc, int h, int w, int scale, const float* mat,
                        const float* bias, float* out_nchw, void* stream);
int adsr_conv3x3_small(const float* x_nchw, int B, int nc, int H, int W, const float* weight, const float* bias,
                       int C, void* out1, int64_t ld1, void* out2, int64_t ld2, int col2, void* stream);
int adsr_channel_mean(const void* x, int64_t ld, int B, int HW, int C, int slices, float* part, int64_t ld_part, void* stream);
int adsr_rcab_ca_scale(const void* res, int64_t ldr, const void* x, int64_t ldx, void* out, int64_t ldo,
                       const float* scale, int B, int HW, int C, void* stream);

/* ---- per-image anomaly scores ---------------------------------------------------------------------------------
 * replaces ssim_numpy (src/metrics.py:26-67) for every window size of the sweep (src/evaluate.py:233-248),
 * MSE (src/evaluate.py:259-260) and psnr_numpy (src/metrics.py:15-23) on uint8 HWC pairs.
 * host_ws_list: int32 [n_ws <= 128] in HOST memory (odd window sizes, ws/2 < min(H,W)): the evaluator's full sweep of images up to
 * the kernels' limit of W <= 1024 columns (102 window sizes at 1024 px);
 * scores: fp64 [B, n_ws + 2] = ssim(ws_0..), mse, psnr (+inf when mse == 0).  An image's row is bit-identical whatever batch it is
 * scored in; an identical pair gives exactly 1 / 0 / +inf. */
int adsr_score_images(const uint8_t* sr_u8_hwc, const uint8_t* hr_u8_hwc, int B, int H, int W, int C,
                      const int32_t* host_ws_list, int n_ws, double* scores, void* stream);

/* Same kernel behind the reference's generic metric signatures: psnr_numpy / ssim_numpy on float arrays
 * (src/metrics.py:15-67) and psnr_torch / ssim_torch (src/metrics.py:70-108: zero-padded box filter, /rgb_range,
 * clamp, 255^2-scaled constants).  sr/hr: uint8 (is_f32=0) or fp32 (is_f32=1) with element strides
 * host_strides_* = {image, row, column, channel}; value = clamp?(raw / div); zero_pad selects F.conv2d-style
 * padding instead of np.pad reflect; c1/c2 are the SSIM constants, psnr_peak the PSNR data range. */
int adsr_score_images_strided(const void* sr, const void* hr, int is_f32, int B, int H, int W, int C,
                              const int64_t* host_strides_sr, const int64_t* host_strides_hr, float div,
                              int clamp01, int zero_pad, double c1, double c2, double psnr_peak,
                              const int32_t* host_ws_list, int n_ws, double* scores, void* stream);

/* Per-pixel anomaly maps of uint8 HWC SR / HR pairs (same pixel conventions as adsr_score_images), for defect localisation.
 * ssim_map, se_map: fp32 [B, H, W]; scratch: fp32 [B, H, W], needed only when sigma > 0 (NULL otherwise);
 * map_max: fp64 [B, 2] = per-image max of the (smoothed) ssim_map and se_map.
 *   ssim_map = 1 - SSIM(hr, sr) per pixel for ONE odd win_size (gray conversion, / 255, reflect padding and C1 / C2 of ssim_numpy;
 *              fp64 sums, stored as fp32): its mean is 1 - the adsr_score_images SSIM of that window size;
 *   se_map   = mean over channels of (sr / 255 - hr / 255)^2: its mean is the MSE column.
 * sigma > 0 smooths both maps with scipy.ndimage.gaussian_filter(map, sigma, mode="reflect", truncate=4.0) semantics: radius
 * r = int(4 sigma + 0.5) <= 64, normalised taps exp(-x^2 / 2 sigma^2), half-sample reflection at the borders; sigma == 0: no smoothing.
 * ADSR_ERR_BAD_SHAPE: C not 1 or 3, H < 2, W < 2, W > 1024, even win_size, win_size/2 >= min(H, W), r >= min(H, W), r > 64,
 * sigma < 0, or sigma > 0 with scratch == NULL.  Deterministic; image i does not depend on the rest of the batch. */
int adsr_anomaly_maps(const uint8_t* sr_u8_hwc, const uint8_t* hr_u8_hwc, int B, int H, int W, int C,
                      int win_size, float sigma, float* ssim_map, float* se_map, float* scratch,
                      double* map_max, void* stream);

/* Multi-scale gradient-magnitude-similarity (MSGMS) map of uint8 HWC SR / HR pairs (RIAD, Zavrtanik et al. 2021, after GMSD, Xue et
 * al. 2014), for defect localisation next to adsr_anomaly_maps.  On the gray plane of the 1 - SSIM map (x = HR, y = SR, in [0, 1]):
 * 4 pyramid levels (level k + 1 = avg_pool2d(level k, 2, 2), odd sizes floored); at each level Prewitt gradient magnitudes
 * g = sqrt(gx^2 + gy^2 + 1e-12) (kernels [[1/3, 0, -1/3]] x 3 and its transpose, zero padding) and
 * gms = (2 g_x g_y + c) / (g_x^2 + g_y^2 + c), c = 0.0026; the map is (1/4) sum_k up_k(1 - gms_k), up_k = bilinear resize to H x W
 * (align_corners = False), summed in level order.  sigma > 0 smooths it with the Gaussian of adsr_anomaly_maps (same radius rule and
 * limit).  fp32 arithmetic; the GMS products are rounded one by one, so an identical pair gives exact zeros.
 * gms_map: fp32 [B, H, W]; map_max: fp64 [B] = per-image max of the final map; workspace: adsr_gms_workspace_bytes(B, H, W) bytes,
 * 4-byte aligned (pyramids of both images, per-level similarity planes, Gaussian scratch).  No allocation, no synchronisation; the
 * launch count is fixed by (B, H, W, sigma): 4 kernels, 6 with smoothing.
 * ADSR_ERR_BAD_SHAPE: C not 1 or 3, H < 8, W < 8, B H W >= 2^31, sigma NaN or < 0, r > 64, r >= min(H, W), or a NULL workspace or
 * output with B > 0.  Deterministic; image i does not depend on the rest of the batch.
 * adsr_gms_workspace_bytes: -1 for negative sizes. */
int64_t adsr_gms_workspace_bytes(int B, int H, int W);
int adsr_gms_map(const uint8_t* sr_u8_hwc, const uint8_t* hr_u8_hwc, int B, int H, int W, int C, float sigma, float* gms_map,
                 double* map_max, void* workspace, void* stream);

/* Localisation metrics of ONE anomaly map over a whole test set: pixel AUROC, AU-PRO@fpr_limit, pixel AP and F1-max with its threshold,
 * exact (no threshold binning).
 * scores: fp32 [n] (all pixels of all images, higher = more anomalous); regions: int32 [n], -1 = defect-free pixel, else the index of
 * the pixel's defect region (8-connected component of a ground-truth mask) in region_sizes: int64 [n_regions] pixel counts.
 * n_ok = number of defect-free pixels.  All pixels are ranked by score, descending (-0.0 = +0.0); equal scores form one curve point.
 *   pixel AUROC = sklearn.metrics.roc_auc_score(regions >= 0, scores) (ties count one half);
 *   AU-PRO      = (1 / fpr_limit) * trapezoid area under (FPR, PRO) from FPR 0 to fpr_limit, the crossing segment cut by linear
 *                 interpolation; FPR = share of the defect-free pixels at or above the score, PRO = mean over the regions of the share
 *                 of the region's pixels at or above it.
 * With runs = maximal sets of equal scores in that order, and d_k / o_k = the defect / defect-free pixels at or above run k's score,
 * N_def = n - n_ok:
 *   pixel AP    = sum_k (d_k - d_{k-1}) / N_def * d_k / (d_k + o_k) = sklearn.metrics.average_precision_score(regions >= 0, scores);
 *   F1-max      = max_k 2 d_k / (d_k + o_k + N_def), exact (the fractions are compared as integers), a tie going to the higher score;
 *   F1 threshold = the fp32 score of that run (-0.0 reported as +0.0): `scores >= threshold` is the mask that attains F1-max.  It is
 *                 an oracle threshold: chosen with the ground truth of the very pixels it is scored on.
 * out: fp64 [8] = {pixel AUROC, AU-PRO, NaN scores, defect-free pixels seen, region indices out of range, pixel AP, F1-max,
 * F1 threshold}: indices 2-4 are checks for the caller (the metrics are only valid when they read 0, n_ok, 0).  workspace:
 * adsr_localisation_workspace_bytes(n) bytes, 16-byte aligned.  Deterministic (integer sort and counts, exact F1 max, fixed-order fp64
 * area and AP sums) and a function of the pixel sequence alone.
 * ADSR_ERR_BAD_SHAPE: n < 1, n_regions < 1, n_ok < 1, n_ok >= n, fpr_limit outside (0, 1], a NULL pointer or a short workspace. */
int64_t adsr_localisation_workspace_bytes(int64_t n);
int adsr_localisation_metrics(const float* scores, const int32_t* regions, int64_t n, const int64_t* region_sizes, int n_regions,
                              int64_t n_ok, double fpr_limit, void* workspace, int64_t workspace_bytes, double* out, void* stream);

/* Thresholds calibrated on defect-free images, and the metrics of one fixed threshold; both read the scores without sorting them,
 * take the same workspace as adsr_localisation_metrics (adsr_localisation_workspace_bytes(n) bytes, 16-byte aligned), are integer-exact
 * and deterministic, and do not synchronise with the host.
 * adsr_score_quantile: the exact k-th smallest of the n fp32 scores, 1 <= k <= n (np.quantile(scores.astype(float64), q,
 *   method="inverted_cdf") for k = max(1, ceil(q n))): an MSD radix select over the order-preserving 32-bit keys, 4 passes of 8 bits, ~16 B read per pixel.
 *   -0.0 ranks as +0.0 and is reported as +0.0; NaN scores are counted, not ranked.
 *   out: fp64 [2] = {score, NaN scores} (score = NaN when fewer than k scores are not NaN).
 * adsr_threshold_metrics: one pass over the pixels with the rule `score >= threshold` (threshold not NaN); regions / region_sizes /
 *   n_regions as in adsr_localisation_metrics, except that n_regions may be 0 (region_sizes may then be NULL).
 *   out: fp64 [7] = {TP, FP, FN, TN, PRO@threshold, NaN scores, region indices out of range}: counts of predicted / actual defect
 *   pixels (a NaN score is never predicted); PRO@threshold = mean over the regions of the share of the region's pixels predicted,
 *   from the fixed-point weights the AU-PRO curve sums (NaN when n_regions == 0).  The last two are checks for the caller.
 * ADSR_ERR_BAD_SHAPE: n < 1, k outside [1, n], n_regions < 0, a NaN threshold, a NULL pointer or a short workspace. */
int adsr_score_quantile(const float* scores, int64_t n, int64_t k, void* workspace, int64_t workspace_bytes, double* out, void* stream);
int adsr_threshold_metrics(const float* scores, const int32_t* regions, int64_t n, const int64_t* region_sizes, int n_regions,
                           float threshold, void* workspace, int64_t workspace_bytes, double* out, void* stream);

/* Defect regions of a [B, H, W] batch, image by image: the 8-connected components of the foreground (scipy.ndimage.label with
 * structure = ones((3, 3))), components of fewer than min_area >= 1 pixels dropped, the kept ones numbered 1..n in raster order of their
 * first pixel (0 = background).  Exact and deterministic: the same labels whatever the scheduling, and image i does not depend on the
 * rest of the batch.
 * adsr_label_regions: foreground = scores >= threshold (fp32 scores, threshold not NaN; a NaN score is never foreground) or mask != 0
 *   (uint8): exactly one of scores / mask is given.  labels: int32 [B, H, W]; counts: int32 [B] regions kept per image.
 *   workspace: adsr_regions_workspace_bytes(B, H, W) bytes, 16-byte aligned; its first 4 bytes (uint32) count union / find loops that
 *   hit their iteration cap (the pixel count of a tile or an image; each pass strictly lowers a root index, so 0 unless memory was
 *   corrupted): the labels are only valid when it reads 0.  Nine launches (two memsets, seven kernels).
 * adsr_region_stats: one pass over labels (as adsr_label_regions left them) with integer atomics.  row_offsets: int64 [B + 1] device,
 *   region l of image b is table row row_offsets[b] + l - 1 (row_offsets[B] = n_rows); table: int64 [n_rows, 9] =
 *   {area, y min, x min, y max, x max, sum of y, sum of x, peak key, ground-truth pixels}, the peak key = (k << 32) | ~(y W + x) as an
 *   unsigned 64-bit value with k the order-preserving key of the fp32 score (-0.0 as +0.0; sign bit set for scores >= 0, all bits
 *   flipped for negative ones): the highest score wins, a tie goes to the first raster pixel.  scores NULL: peak keys stay 0.
 *   gt_labels (nullable): int32 [B, H, W] ground-truth regions (adsr_label_regions of the mask, min_area 1) with gt_offsets int64 [B + 1]
 *   as row_offsets; field 8 counts the region's pixels with gt_labels > 0 and gt_hit: int32 [n_gt] is 1 for every ground-truth region
 *   that holds a pixel of a region, else 0.  The workspace (that of adsr_label_regions) receives the number of labels out of range in
 *   its first 4 bytes.  Two kernels.
 * ADSR_ERR_BAD_SHAPE: B, H or W < 1, H W >= 2^31, min_area < 1, a NaN threshold, neither or both of scores / mask, n_rows or n_gt < 0, a
 *   NULL output or a short workspace.  adsr_regions_workspace_bytes: -1 for unsupported sizes. */
int64_t adsr_regions_workspace_bytes(int B, int H, int W);
int adsr_label_regions(const float* scores, float threshold, const uint8_t* mask, int B, int H, int W, int min_area, int32_t* labels,
                       int32_t* counts, void* workspace, int64_t workspace_bytes, void* stream);
int adsr_region_stats(const int32_t* labels, const float* scores, const int32_t* gt_labels, int B, int H, int W,
                      const int64_t* row_offsets, int64_t n_rows, const int64_t* gt_offsets, int64_t n_gt, int64_t* table,
                      int32_t* gt_hit, void* workspace, int64_t workspace_bytes, void* stream);

/* Validation metrics of the reference's training loop, `Trainer.test` (src/trainer.py:242-304), for a batch of fp32 image
 * pairs: the SR value is first quantised with ROUNDING (`quantize`, src/trainer.py:45-47: round(clamp(x * 255 / rgb_range, 0,
 * 255)) / (255 / rgb_range) -- the evaluator truncates instead), then calc_psnr / calc_ssim = psnr_torch / ssim_torch
 * (src/metrics.py:70-108: / rgb_range, clamp [0,1] for the SSIM, zero-padded win_size box, C1/C2 scaled by 255^2).
 * sr / hr: fp32 with element strides {image, row, column, channel} (pass the 4-px shaved crop as a strided view).
 * scores: fp64 [B, 3] = ssim, mse (of the unclamped (sr_q - hr) / rgb_range), psnr per image. */
int adsr_validate_images(const void* sr, const void* hr, int B, int H, int W, int C,
                         const int64_t* host_strides_sr, const int64_t* host_strides_hr, float rgb_range, int win_size,
                         double* scores, void* stream);

/* ---- host-side weight packing and workspace sizes (SURVEY.md 8b: pack_weights_*, *_workspace_bytes) -----------------
 * Pure HOST functions (no stream, no device work): the tensor-core operand images are built once per checkpoint
 * (replacing nothing in the reference: its nn.Linear / nn.Conv2d weights, src/drct.py:245-249, 334-374, are used as stored)
 * and uploaded with one plain copy per buffer.
 * adsr_pack_slab_sw128: fp32 [rows, >= cols] (row pitch ld, cols <= 64) -> bf16 [rows x 64] slab in the K-major 128-byte-swizzle
 *   shared-memory layout (row r at byte r*128, its 16-byte chunk c at position c ^ (r % 8)); columns >= cols are zeros.
 * adsr_pack_tiles_sw128: fp32 weight [n, k] (nn.Linear layout) -> n_tiles tiles x ceil(k/64) K slabs of [bn x 64] in that
 *   layout (what adsr_tc_gemm_bf16 streams); rows >= n and columns >= k are zeros.  host_dst: n_tiles*ceil(k/64)*bn*128 bytes.
 * adsr_drct_workspace_bytes: bytes of caller-owned scratch one DRCT forward of [B, *, H, W] LR inputs needs (dense slab, per-block
 *   scratch rows with qkv_cols / att_cols head-padded columns, row-statistics slots, PixelShuffle stages); -1 on bad arguments.
 * adsr_score_workspace_bytes: 0 (the scorer keeps its planes and prefix sums in shared memory). */
int adsr_pack_slab_sw128(const float* host_src, int64_t ld, int rows, int cols, void* host_dst);
int adsr_pack_tiles_sw128(const float* host_w, int64_t ld, int n, int k, int bn, int n_tiles, void* host_dst);
int64_t adsr_drct_workspace_bytes(int B, int H, int W, int embed_dim, int gc, int upscale, int qkv_cols, int att_cols);
int64_t adsr_score_workspace_bytes(int B, int H, int W, int C, int n_ws);

/* ---- first slice of the training step (reference: Trainer.train src/trainer.py:141-227, Loss "1*L1" src/loss.py:83-84, 108-121,
 * Adam src/trainer.py:49-59).  The backward of the tcgen05 blocks is not built; these cover the loss and the last layer.
 * adsr_l1_loss_grad: nn.L1Loss (mean) of fp32 sr / hr (n elements, 16-byte aligned) and d loss / d sr = sign(sr - hr) * grad_scale / n
 *   in one pass; partial_ws: fp64 [n_partial] scratch (n_partial = number of thread blocks); loss: fp32 [1] on the device.
 * adsr_conv_last_bwd: backward of conv_last (3x3, pad 1, Cin = 64 -> nc <= 3, src/drct.py:847, 895): x bf16 NHWC rows (pitch ldx),
 *   grad_out fp32 NCHW [B, nc, H, W], weight fp32 [nc, 64, 3, 3] -> dx bf16 NHWC rows (may be NULL), dw fp32 [nc, 64, 3, 3] and db
 *   fp32 [nc] (both NULL to skip); workspace: adsr_conv_last_bwd_workspace_bytes(B, H, 64) bytes; reductions in a fixed order.
 * adsr_adam_step: torch.optim.Adam step `step` (1-based; amsgrad off) fused over many fp32 tensors: tensor_table = device array of
 *   {float* p; const float* g; float* m; float* v; int64 n}, chunk_table = device array of int32 pairs {tensor index, chunk index},
 *   one thread block per chunk of chunk_elems elements. */
int adsr_l1_loss_grad(const float* sr, const float* hr, int64_t n, float grad_scale, float* grad, double* partial_ws, int n_partial,
                      float* loss, void* stream);
int64_t adsr_conv_last_bwd_workspace_bytes(int B, int H, int Cin);
int adsr_conv_last_bwd(const void* x, int64_t ldx, const float* grad_out_nchw, const float* weight, int B, int H, int W, int Cin, int nc,
                       void* dx, int64_t ld_dx, float* dw, float* db, float* workspace, void* stream);
int adsr_adam_step(const void* tensor_table, const void* chunk_table, int n_chunks, int chunk_elems, float lr, float beta1, float beta2,
                   float eps, float weight_decay, int step, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* ADSR_B200_H_ */

/* mgw.h -- C ABI of the B200-native multi-grid warp library (libmgw_b200.so).
 *
 * This is the drop-in boundary for the hot path of cxjyxxme/deep-online-video-stabilization: the
 * transformer(U, theta[, out_size]) / interpolate(im, x, y, out_size) operators and the loss epilogue
 * fused onto them.  The reference has no FFI of its own (it is a TensorFlow-1.3 Python graph); each
 * entry point below names the reference expression it replaces (file:line under the reference repo).
 * INTEGRATION.md shows the ctypes binding the reference's scripts would add.
 *
 * Conventions
 *   - Every pointer is a DEVICE pointer to fp32 (int32 where stated), contiguous, NHWC for images.
 *   - The caller allocates every buffer; the library never frees or retains one.  Pointers documented
 *     "nullable" may be NULL to skip that output.
 *   - `stream` is a cudaStream_t (NULL = legacy default stream).  All calls are asynchronous and
 *     stream-ordered; no call synchronises the device.
 *   - Return 0 on success, a negative MGW_ERR_* otherwise; mgw_last_error() gives the thread-local text.
 *   - No CPU fallback exists: without a CUDA device every compute call returns MGW_ERR_CUDA.
 *
 * Shapes: N batch, H x W image, C channels, gh x gw mesh cells, P = N*H*W.
 */
#ifndef MGW_H_
#define MGW_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(__GNUC__)
#define MGW_API __attribute__((visibility("default")))
#else
#define MGW_API
#endif

#define MGW_OK 0
#define MGW_ERR_INVALID (-1)     /* bad argument: null pointer, non-positive size, misalignment */
#define MGW_ERR_UNSUPPORTED (-2) /* shape outside what the kernels implement */
#define MGW_ERR_CUDA (-3)        /* CUDA runtime / driver error (text in mgw_last_error) */

MGW_API int mgw_version(void);
MGW_API const char* mgw_last_error(void);

/* Number of kernels this library has launched on the calling process so far (bench.py's gpu_launches). */
MGW_API uint64_t mgw_launch_count(void);

/* Kernel family: chosen per call from shape and alignment (forward: a persistent TMA pipeline, else one TMA tile per CTA;
 * backward: one TMA tile per CTA; else the generic global-gather kernels).  Tests and tuning runs can force one through the
 * environment variable MGW_IMPL = auto | generic | tma | pipe ("tma" / "pipe" fail instead of falling back; "pipe" selects the
 * forward pipeline and, for the backward, the tile kernels like "tma"); the library keeps no such state. */

/* ---- a0: get_4_pts, s_net_bundle_nobm.py:29-71 --------------------------------------------------------
 * head [N, 2*(gh+1)*(gw+1)] -> pts2 [N,gh+1,gw+1,2] (absolute clamped vertices, (x,y) last),
 * pts1 [N,gh,gw,8] nullable (per-cell [x_tl,x_tr,x_bl,x_br,y_tl,y_tr,y_bl,y_br]).  do_crop_rate = 0.8 in v2_93. */
MGW_API int mgw_vertices_fwd(const float* head, int N, int gh, int gw, float do_crop_rate, float* pts2, float* pts1,
                     void* stream);
/* d_pts2 / d_pts1 nullable (treated as zero) -> d_head [N, 2*(gh+1)*(gw+1)] */
MGW_API int mgw_vertices_bwd(const float* head, const float* d_pts2, const float* d_pts1, int N, int gh, int gw,
                     float do_crop_rate, float* d_head, void* stream);

/* ---- a1/a2: get_Hs / get_H / pinv, spatial_transformer3.py:144-198 ------------------------------------
 * theta [N,gh+1,gw+1,2] -> Hs [N,gh,gw,9]; h = inverse(A + 1e-4 I).b per cell, H[8] = 1. */
MGW_API int mgw_solve_h_fwd(const float* theta, int N, int gh, int gw, float* Hs, void* stream);
/* dHs [N,gh,gw,9] (slot 8 ignored) -> dtheta [N,gh+1,gw+1,2] */
MGW_API int mgw_solve_h_bwd(const float* theta, const float* Hs, const float* dHs, int N, int gh, int gw, float* dtheta,
                    void* stream);

/* ---- a3-a5: _transform3 given Hs, spatial_transformer3.py:218-301 -------------------------------------
 * U [N,H,W,C], Hs [N,gh,gw,9] -> out [N,H,W,C] ("output_img"), black [N,H,W] ("black_pix", 1.0/0.0),
 * img [N,H,W,2] (x_map,y_map interleaved), cell_idx [N,H,W] int32 (debug).  All four outputs nullable. */
MGW_API int mgw_warp_fwd(const float* U, const float* Hs, int N, int H, int W, int C, int gh, int gw, float* out,
                 float* black, float* img, int32_t* cell_idx, void* stream);
/* Backward of mgw_warp_fwd.  d_out [N,H,W,C]; d_img [N,H,W,2] nullable (gradient arriving on x_map/y_map);
 * dU [N,H,W,C] nullable -- OVERWRITTEN with the gradient (the library zero-fills it first);
 * dHs [N,gh,gw,9] overwritten (slot 8 = 0); nullable when a workspace is given and a tile family serves the shape: the per-tile
 * partials then stay in the workspace and the final reduction launch is skipped (bench.py times the backward kernel alone so).
 * workspace: nullable device scratch of at least mgw_warp_bwd_workspace_bytes() (deterministic dHs reduction);
 * with NULL the library reduces dHs with fp32 atomics. */
MGW_API size_t mgw_warp_bwd_workspace_bytes(int N, int H, int W, int C, int gh, int gw);
MGW_API int mgw_warp_bwd(const float* U, const float* Hs, const float* d_out, const float* d_img, int N, int H, int W,
                 int C, int gh, int gw, float* dU, float* dHs, void* workspace, void* stream);
/* The same, but dU is ACCUMULATED INTO (dU += gradient) and never zero-filled by the library: the caller owns its initial
 * contents -- gradient accumulation across micro-batches, or a zero-fill issued earlier on another stream so that it
 * overlaps the forward pass (what bench.py does).  dHs is still overwritten. */
MGW_API int mgw_warp_bwd_acc(const float* U, const float* Hs, const float* d_out, const float* d_img, int N, int H, int W,
                     int C, int gh, int gw, float* dU, float* dHs, void* workspace, void* stream);

/* ---- fused a1-a5: spatial_transformer3.transformer(U, theta), :19-365 ---------------------------------
 * theta [N,gh+1,gw+1,2] mesh vertices.  Hs is an output too (deploy_bundle.py:54 fetches it). */
MGW_API int mgw_mesh_warp_fwd(const float* U, const float* theta, int N, int H, int W, int C, int gh, int gw, float* Hs,
                      float* out, float* black, float* img, void* stream);
/* -> dU nullable (overwritten), dtheta [N,gh+1,gw+1,2] (overwritten).  workspace as for mgw_warp_bwd plus
 * N*gh*gw*9 floats; query with mgw_mesh_warp_bwd_workspace_bytes (required, not nullable). */
MGW_API size_t mgw_mesh_warp_bwd_workspace_bytes(int N, int H, int W, int C, int gh, int gw);
MGW_API int mgw_mesh_warp_bwd(const float* U, const float* theta, const float* Hs, const float* d_out, const float* d_img,
                      int N, int H, int W, int C, int gh, int gw, float* dU, float* dtheta, void* workspace,
                      void* stream);
/* dU += gradient (see mgw_warp_bwd_acc); dtheta overwritten */
MGW_API int mgw_mesh_warp_bwd_acc(const float* U, const float* theta, const float* Hs, const float* d_out, const float* d_img,
                          int N, int H, int W, int C, int gh, int gw, float* dU, float* dtheta, void* workspace,
                          void* stream);

/* ---- fused a1-a5 + a8: transformer(U, theta) with the img_loss epilogue (s_net_bundle_nobm.py:332,347-352) ----------
 * Forward: as mgw_mesh_warp_fwd (out, black required) plus sums [N,2] = per-sample (sum ((out-y)(1-black))^2,
 * sum (1-black)) accumulated inside the warp kernel -- no second pass over out / y / black.
 * upstream_dev (here and in the other loss backwards): nullable DEVICE scalar multiplied onto `upstream` inside the kernel --
 * the autograd upstream gradient without a host read, so that a whole training step can be enqueued / graph-captured.
 * Backward: the upstream gradient of out is the loss's, d_out = upstream*2/batch * (out-y)(1-black)^2/(sums[n][1]+1e-8),
 * formed in registers inside the backward kernel (no d_out tensor is written or read); d_img nullable as before; d_out_extra
 * (nullable, [N,H,W,C]) = the gradient another consumer of `out` sends back (temp_loss), added to the loss's inside the kernel.
 * loss = sum_n sums[n][0]/(sums[n][1]+1e-8)/batch is N scalars of arithmetic left to the caller. */
MGW_API int mgw_mesh_warp_img_loss_fwd(const float* U, const float* theta, const float* y, int N, int H, int W, int C, int gh,
                               int gw, float* Hs, float* out, float* black, float* img, float* sums, void* stream);
MGW_API size_t mgw_mesh_warp_img_loss_bwd_workspace_bytes(int N, int H, int W, int C, int gh, int gw);
MGW_API int mgw_mesh_warp_img_loss_bwd(const float* U, const float* theta, const float* Hs, const float* out, const float* y,
                               const float* black, const float* sums, float upstream, const float* upstream_dev, float batch,
                               const float* d_img, const float* d_out_extra, int N, int H, int W, int C, int gh, int gw, float* dU,
                               float* dtheta, void* workspace, void* stream);

/* feature_loss backward taken straight to the homographies: dH_part [N*gh*gw, 8] = the dH terms (as mgw_warp_bwd forms them from a
 * dense d_img) of d(loss)/d(flow map), which is non-zero at the <= M match pixels of a sample only -- no dense [N,H,W,2] gradient
 * is written or read.  img = the forward's flow map, Hs its homographies, facc [N,2] = per-sample (sum of masked residuals, sum of
 * mask) (only the count is read); upstream as mgw_feature_loss_bwd.  Feed dH_part to the solve backward as one more partial. */
MGW_API int mgw_feature_loss_dh(const float* matches, const float* mask, const float* img, const float* Hs, const float* facc,
                        float upstream, const float* upstream_dev, int N, int M, int H, int W, int gh, int gw, float* dH_part,
                        void* stream);

/* the O(N) scalar epilogue of img_loss / temp_loss (clamp = 0: out[0] = scale * sum_n sums[n][0] / (sums[n][1] + 1e-8)) and of
 * feature_loss given per-sample (sum, count) pairs (clamp = 1: ... / max(sums[n][1], 1)) as one launch.  sums [N,2], out [1]. */
MGW_API int mgw_loss_ratio_sum(const float* sums, int N, int clamp, float scale, float* out, void* stream);

/* ---- one training pass: s_net_bundle_nobm.py:266-381 after the network head, as a handful of launches -------------------
 * head [N, 2(gh+1)(gw+1)] (the network's output) -> get_4_pts (:29-71) -> transformer + img_loss (:332,:347-352) ->
 * feature_loss / warp_pts (:215-230,:335-343) -> id / black_pos / distortion / consistency terms (:139-210,:246) -> total (:354-359).
 * coef: HOST array of 11 floats = the multipliers of the vertex sums [4] (id, black_pos, distortion, consistency: configured
 * multipliers, use_black_loss and element counts folded in), the multipliers of IMG = sum_n e2_n/(nb_n+1e-8)/batch, FEAT =
 * sum_n acc_n/max(cnt_n,1)/batch and of the weight regulariser REGU (*regu_dev, nullable device scalar), the shares of the id term
 * reported as theta_loss / grid_theta_loss, 1/batch (the GLOBAL batch under data parallelism), gate = 1 - use_theta_only:
 * total = id + gate * (everything else), the parts are reported without the gate (:354-375).
 * Forward outputs: pts1 [N,gh,gw,8], pts2 [N,gh+1,gw+1,2], Hs, out, black, img as mgw_mesh_warp_fwd (all required), acc [4N+4]
 * (img sums [N,2], feature sums [N,2], vertex sums [4]), warpped [N,M,2] (nullable), result [9] = total, then the weighted parts
 * theta, grid_theta, black, distortion, consistency, feature, img, regu (the reference's ret[...]).
 * Backward: d_head [N, 2(gh+1)(gw+1)] = d(total * *g_total_dev)/d(head) (g_total_dev nullable = 1); d_out_extra (nullable) is a
 * gradient reaching `out` from another consumer (temp_loss, train_bundle_nobm.py:115-125), added inside the warp backward; dU
 * nullable.  The gradient of feature_loss goes straight to one dH partial per cell: no dense d(flow map) is written or read.
 * The flow map `img` therefore must have no other differentiable consumer in this form. */
MGW_API int mgw_train_pass_fwd(const float* head, const float* U, const float* y, const float* matches, const float* mask,
                       const float* regu_dev, const float* coef, int N, int H, int W, int C, int gh, int gw, int M, float do_crop_rate,
                       float* pts1, float* pts2, float* Hs, float* out, float* black, float* img, float* acc, float* warpped,
                       float* result, void* stream);
MGW_API size_t mgw_train_pass_bwd_workspace_bytes(int N, int H, int W, int C, int gh, int gw);
MGW_API int mgw_train_pass_bwd(const float* head, const float* pts1, const float* pts2, const float* U, const float* y,
                       const float* matches, const float* mask, const float* Hs, const float* out, const float* black,
                       const float* img, const float* acc, const float* g_total_dev, const float* d_out_extra, const float* coef,
                       int N, int H, int W, int C, int gh, int gw, int M, float do_crop_rate, float* dU, float* d_head,
                       void* workspace, void* stream);

/* ---- f1 (deploy side): warpRevBundle2(img, x_map, y_map), deploy_bundle.py:136-146 ---------------------------------
 * img [N,H,W,C] uint8 (the unstable frame at network size), xy [N,H,W,2] = the operator's x_map,y_map (the `img` output of
 * mgw_warp_fwd / mgw_mesh_warp_fwd) -> dst [N,H,W,C] uint8: maps smoothed by cv2.resize /4 then x4, converted to pixel
 * coordinates, cv2.remap(INTER_LINEAR, constant border 0).  Bit-exact with OpenCV's plain C++ path.  C in {1,3,4}.
 * workspace: device scratch of mgw_remap_bundle_u8_workspace_bytes() (the /4 maps). */
MGW_API size_t mgw_remap_bundle_u8_workspace_bytes(int N, int H, int W);
MGW_API int mgw_remap_bundle_u8(const uint8_t* img, const float* xy, int N, int H, int W, int C, uint8_t* dst, void* workspace,
                        void* stream);

/* cv2.resize(frame, (width, height)) of the uint8 colour frame, deploy_bundle.py:301 (INTER_LINEAR, OpenCV's 8-bit fixed-point
 * path, byte-exact; an exact 2x2 decimation takes OpenCV's INTER_AREA shortcut and needs no tables).  img [H,W,C] -> dst
 * [out_h,out_w,C]; xtab [out_w][4], ytab [out_h][4] = {i0, i1, a0, a1}: the two source indices and their 11-bit weights
 * (device int32, 16-byte aligned; computed by the host binding as resize.cpp does). */
MGW_API int mgw_resize_linear_u8(const uint8_t* img, int H, int W, int C, const int32_t* xtab, const int32_t* ytab, int out_h,
                         int out_w, uint8_t* dst, void* stream);

/* cvt_img2train(img, crop_rate), config.py:6-21 (the producer of every frame the network and the warp see): bgr [H,W,3] uint8 ->
 * cv2 BGR2GRAY -> Pillow resize(BILINEAR) [-> centre crop] -> v*(1/255) - 0.5 -> out [out_h,out_w] fp32, exact.
 * kx [out_w,ksx] / ky [out_h,ksy]: Pillow's 22-bit fixed-point weights of each output column / row, x0 / y0 the first source
 * column / row of its window, xn / yn the window length (device int32 tables; the host binding computes them in double as
 * Resample.c does and slices them for the crop).  tmp: device scratch of H*out_w bytes (the horizontally resampled image). */
MGW_API int mgw_cvt_img2train_u8(const uint8_t* bgr, int H, int W, const int32_t* kx, const int32_t* x0, const int32_t* xn, int ksx,
                         const int32_t* ky, const int32_t* y0, const int32_t* yn, int ksy, int out_h, int out_w, uint8_t* tmp,
                         float* out, void* stream);

/* warpRevBundle(img, Hs), deploy_bundle.py:148-173 (the per-cell cv2.warpPerspective variant; its call at :300 is commented
 * out in the reference): Hs_cvt [N,gh,gw,9] DOUBLE on the device = cvt_theta_mat_bundle(Hs) (:121-134: scale_mat . H .
 * inv(scale_mat), computed by the host binding with the reference's own numpy expressions); dst cell (i, j) = that region of
 * cv2.warpPerspective(img, Hs_cvt[i][j], dsize=(W,H), WARP_INVERSE_MAP | INTER_LINEAR), byte-exact with OpenCV 4.x. */
MGW_API int mgw_warp_rev_bundle_u8(const uint8_t* img, const double* Hs_cvt, int N, int H, int W, int C, int gh, int gw,
                           uint8_t* dst, void* stream);

/* ---- f2 (deploy side): the streaming state of deploy_bundle.py:204-232,259-295,319-327 -----------------------------
 * frames, masks: device rings [depth][H][W] (the reference's before_frames / before_masks lists, depth = before_ch = 32);
 * `head` = slot of the newest entry, so that list[-i] is slot (head - (i-1)) mod depth.
 * mgw_stream_assemble: in_x [H,W,nch] = [masks[-i] for i in taps (if use_masks)] + [frames[-i] for i in taps] + [cur]
 *   (taps: HOST array of ntaps <= 32 ints, the reference's indices[1:] = 1,2,4,8,16,32; cur [H,W] = the current frame).
 * mgw_stream_push: frame = img + black*(-1) -> frames[slot], black -> masks[slot] (either ring nullable), and optionally
 *   frame -> frame_out[p * out_stride] (the refine re-feed tmp_in_x[..., -1] = frame: pass in_x + nch-1 and nch). */
MGW_API int mgw_stream_assemble(const float* frames, const float* masks, int depth, int head, const int* taps, int ntaps,
                        int use_masks, const float* cur, int H, int W, float* in_x, void* stream);
MGW_API int mgw_stream_push(float* frames, float* masks, int depth, int slot, const float* img, const float* black, int H, int W,
                    float* frame_out, int out_stride, void* stream);

/* ---- f4 (training side): the vertex regularisers of s_net_bundle_nobm.py ------------------------------------------------
 * theta [N, 2*(gh+1)*(gw+1)] (the head output), pts1 [N,gh,gw,8], pts2 [N,gh+1,gw+1,2] (mgw_vertices_fwd's outputs); each
 * nullable, its terms are then skipped.  sums[4] (device, overwritten):
 *   [0] sum |theta|                       id loss :246-247        = sums[0] / (N*2*(gh+1)*(gw+1)) * id_mul
 *   [1] sum black_err^2 over pts1         black_pos :139-148,313-317   mean = sums[1] / (N*gh*gw*8)  (times use_black_loss)
 *   [2] sum of the 8 squared rotated-edge residuals per cell   distortion :150-184   loss = sums[2] / (N*gh*gw*2) / 8
 *   [3] sum of squared lattice second differences over pts2    consistency :186-210  loss = sums[3] / (N*2*K),
 *       K = 2*((gh-1)*(gw+1) + (gh+1)*(gw-1)) listed terms (0 terms -> loss 0)
 * black_err [N,gh,gw,8] nullable = get_black_pos(pts1) before the reshape.
 * mgw_vertex_losses_bwd: f[4] (device) = d(total)/d(sums[k]); d_theta (id term only), d_pts1, d_pts2 nullable, overwritten. */
MGW_API int mgw_vertex_losses_fwd(const float* theta, const float* pts1, const float* pts2, int N, int gh, int gw,
                          float do_crop_rate, float* sums, float* black_err, void* stream);
MGW_API int mgw_vertex_losses_bwd(const float* theta, const float* pts1, const float* pts2, int N, int gh, int gw,
                          float do_crop_rate, const float* f, float* d_theta, float* d_pts1,
                          float* d_pts2, void* stream);

/* ---- frame transport -------------------------------------------------------------------------------------------------
 * Frames cross PCIe as uint8 (the reference's frames ARE uint8: config.py:6-21, deploy_bundle.py:301) and are widened on the device.
 * mgw_u8_to_train_f32: dst[i] = float32(src[i] * (1./255) - 0.5), the double-precision expression of config.py:19 and the
 *   float32 cast of the network's placeholder; exact.
 * mgw_train_f32_to_u8: cvt_train2img, deploy_bundle.py:75 = ((x + 0.5) * 255).astype(np.uint8) on float32 (truncation; values
 *   outside [0,256) wrap like numpy on x86).
 * mgw_fill_zero: zero-fill of `bytes` (multiple of 16, 16-byte aligned) device bytes; keep_in_l2 != 0 writes the lines with an
 *   L2 evict_last policy -- for the dU buffer that mgw_*_bwd_acc accumulates into next (its reductions then hit L2). */
MGW_API int mgw_u8_to_train_f32(const uint8_t* src, float* dst, size_t n, void* stream);
MGW_API int mgw_train_f32_to_u8(const float* src, uint8_t* dst, size_t n, void* stream);
MGW_API int mgw_fill_zero(void* p, size_t bytes, int keep_in_l2, void* stream);

/* ---- f4 (deploy side): the crop of deploy_bundle.py:240,291,344-365 -------------------------------------------------
 * mgw_black_accumulate: all_black[p] += round(black[p])  (all_black = all_black + np.round(black).astype(np.int64), :291;
 *   int32 counts: one increment per network evaluation).
 * mgw_crop_rect: rect[4] (device) = the reference's `ans` = [top, left, bottom, right] (inclusive) of the largest rectangle
 *   free of ever-black pixels whose top-left corner (i, j) has i in range(0, H/2, step), j in range(0, W/2, step)
 *   (step = 10 in the reference), ties resolved like the reference's loops (first found); rect = -1,-1,-1,-1 when every
 *   corner is black (the reference raises IndexError there).  workspace: mgw_crop_rect_workspace_bytes() device bytes. */
MGW_API int mgw_black_accumulate(const float* black, int32_t* all_black, int n, void* stream);
MGW_API size_t mgw_crop_rect_workspace_bytes(int H, int W);
MGW_API int mgw_crop_rect(const int32_t* all_black, int H, int W, int step, void* workspace, int32_t* rect, void* stream);

/* The same with the ring head on the DEVICE (head_dev: one int32, the slot of the newest entry): no launch parameter changes
 * from frame to frame, so the whole per-frame loop can be captured once in a CUDA graph and replayed.  mgw_stream_push_dev
 * writes the slot after the head and then advances the head (two launches). */
MGW_API int mgw_stream_assemble_dev(const float* frames, const float* masks, int depth, const int32_t* head_dev, const int* taps,
                            int ntaps, int use_masks, const float* cur, int H, int W, float* in_x, void* stream);
MGW_API int mgw_stream_push_dev(float* frames, float* masks, int depth, int32_t* head_dev, const float* img, const float* black,
                        int H, int W, void* stream);

/* ---- f1/f2 batched: S independent videos of one source size advanced by one set of launches ----------------------------
 * Every per-stream result is bit-identical to the single-stream call on that stream's slice.  0 <= S <= 65535; S = 0 returns
 * MGW_OK and launches nothing.
 * mgw_cvt_img2train_u8_batch: bgr [S,H,W,3] -> out [S,out_h,out_w]; the tables as for mgw_cvt_img2train_u8 (shared by all S
 *   frames), tmp: S*H*out_w bytes.
 * mgw_resize_linear_u8_batch: img [S,H,W,C] -> dst [S,out_h,out_w,C]; the tables as for mgw_resize_linear_u8.
 * mgw_streams_assemble: frames, masks [S,depth,H,W] (stream s's rings are byte for byte those of mgw_stream_assemble_dev),
 *   heads_dev [S] int32 (device), cur [S,H,W] -> in_x [S,H,W,nch].
 * mgw_streams_push: img, black [S,H,W]: writes slot heads_dev[s]+1 of every stream, then advances all S heads (two launches).
 * The refine re-feed and mgw_black_accumulate are element-wise: call mgw_stream_push (frame_out, H = S*H) and
 * mgw_black_accumulate (n = S*H*W) on the [S,H,W] buffers as they are. */
MGW_API int mgw_cvt_img2train_u8_batch(const uint8_t* bgr, int S, int H, int W, const int32_t* kx, const int32_t* x0, const int32_t* xn,
                               int ksx, const int32_t* ky, const int32_t* y0, const int32_t* yn, int ksy, int out_h, int out_w,
                               uint8_t* tmp, float* out, void* stream);
MGW_API int mgw_resize_linear_u8_batch(const uint8_t* img, int S, int H, int W, int C, const int32_t* xtab, const int32_t* ytab,
                               int out_h, int out_w, uint8_t* dst, void* stream);
MGW_API int mgw_streams_assemble(const float* frames, const float* masks, int S, int depth, const int32_t* heads_dev, const int* taps,
                         int ntaps, int use_masks, const float* cur, int H, int W, float* in_x, void* stream);
MGW_API int mgw_streams_push(float* frames, float* masks, int S, int depth, int32_t* heads_dev, const float* img, const float* black,
                     int H, int W, void* stream);

/* ---- f1/f2 from YUV 4:2:0 frames, as video decoders emit them ----------------------------------------------------------
 * yuv [S,3H/2,W] uint8 in OpenCV's 4:2:0 layout, H and W even: the Y plane (H rows of W), then
 *   MGW_YUV420_NV12: H/2 rows of W bytes of interleaved U,V;
 *   MGW_YUV420_I420: the U plane, then the V plane (H/2 x W/2 bytes each, contiguous: byte offsets H*W and H*W + H*W/4).
 * Each call gives byte for byte what its BGR batch call gives on cv2.cvtColor(yuv, COLOR_YUV2BGR_NV12 / _I420) of every frame:
 * OpenCV's BT.601 limited-range 20-bit fixed point, one chroma sample per 2x2 block, converted inside the kernels that read the
 * source.  The frame the network sees is BGR2GRAY of that BGR frame, not the Y plane.  (cv2.VideoCapture converts with FFmpeg's
 * swscale, which is not byte-identical to cvtColor.)  Pitched decoder surfaces: the plane-table calls (mgw_*_planes) below.
 * mgw_cvt_img2train_yuv420_batch: -> out [S,out_h,out_w]; tables and tmp (S*H*out_w bytes) as for mgw_cvt_img2train_u8_batch.
 * mgw_resize_linear_yuv420_batch: -> dst [S,out_h,out_w,3] BGR; tables as for mgw_resize_linear_u8_batch.
 * Checked in the order of the BGR batch calls: sizes and format (S <= 65535, H, W even and positive, S*(3H/2)*W < 2^31), then
 * S = 0 returns MGW_OK and launches nothing, then the pointers and the 16-byte table alignment. */
#define MGW_YUV420_NV12 1
#define MGW_YUV420_I420 2
MGW_API int mgw_cvt_img2train_yuv420_batch(const uint8_t* yuv, int format, int S, int H, int W, const int32_t* kx, const int32_t* x0,
                               const int32_t* xn, int ksx, const int32_t* ky, const int32_t* y0, const int32_t* yn, int ksy, int out_h,
                               int out_w, uint8_t* tmp, float* out, void* stream);
MGW_API int mgw_resize_linear_yuv420_batch(const uint8_t* yuv, int format, int S, int H, int W, const int32_t* xtab, const int32_t* ytab,
                               int out_h, int out_w, uint8_t* dst, void* stream);

/* ---- f1/f2 for a batch of videos of different source sizes: per-slot source geometry ----------------------------------
 * The batch has a capacity (max_h, max_w); slot s owns the region src + s * frame_bytes(max_h, max_w) of the pool (frame_bytes =
 * 3*H*W for MGW_BGR24, 3H/2*W for YUV 4:2:0), and its frame lies contiguous at the start of that region in the slot's own size
 * sizes[s] = (H_s, W_s): BGR [H_s,W_s,3] or YUV [3H_s/2,W_s] in the layouts above.  sizes: device int32 [S,2], 8-byte aligned.
 * Per-slot tables, each slot's rows those of the uniform call at the slot's size:
 *   mgw_cvt_img2train_mixed: kx [S,out_w,ksx], x0 / xn [S,out_w], ky [S,out_h,ksy], y0 / yn [S,out_h]; ksx / ksy are the window
 *     lengths of the capacity (Pillow's 2*ceil(max(in/out,1))+1 does not decrease as the input grows), a slot's shorter rows
 *     zero-padded; tmp [S,max_h,out_w] bytes; -> out [S,out_h,out_w].
 *   mgw_resize_linear_mixed: xtab [S,out_w,4], ytab [S,out_h,4] (16-byte aligned, required even where a slot takes the 2x2
 *     shortcut, which is chosen per slot: H_s == 2*out_h and W_s == 2*out_w); -> dst [S,out_h,out_w,3] BGR.
 * Every active slot's result is bit-identical to the uniform batch call (mgw_*_u8_batch / mgw_*_yuv420_batch) at that slot's size.
 * A slot whose size is 0, larger than the capacity, or odd for a YUV format is idle: its blocks write nothing (out / tmp / dst rows
 * keep what they held).  The tables' contents are trusted, as in the uniform calls.
 * Checked in the order of the batch calls: sizes and format (0 <= S <= 65535, capacity positive and even for YUV, the uniform
 * calls' 32-bit limits over the capacity: S*max_h*max_w < 2^29 for BGR, S*(3max_h/2)*max_w < 2^31 for YUV; ksx, ksy > 0), then
 * S = 0 returns MGW_OK and launches nothing, then the pointers and their alignment. */
#define MGW_BGR24 0
MGW_API int mgw_cvt_img2train_mixed(const uint8_t* src, int format, int S, int max_h, int max_w, const int32_t* sizes,
                               const int32_t* kx, const int32_t* x0, const int32_t* xn, int ksx, const int32_t* ky, const int32_t* y0,
                               const int32_t* yn, int ksy, int out_h, int out_w, uint8_t* tmp, float* out, void* stream);
MGW_API int mgw_resize_linear_mixed(const uint8_t* src, int format, int S, int max_h, int max_w, const int32_t* sizes,
                               const int32_t* xtab, const int32_t* ytab, int out_h, int out_w, uint8_t* dst, void* stream);

/* ---- f1 at any output size: warpRevBundle2 of the frame at its own size ---------------------------------------------
 * src [S,H,W,3] (MGW_BGR24) or [S,3H/2,W] (MGW_YUV420_NV12 / _I420), xy [S,h,w,2] (the operator's x_map,y_map at the network
 * size) -> dst [S,H,W,3] BGR = cv2.remap of the frame with the /4 maps resized to (W, H) and scaled by (W, H), constant border 0
 * (a YUV frame is read as the BGR frame cv2.cvtColor makes of it).  (H, W) == (h, w) with MGW_BGR24 is mgw_remap_bundle_u8, bit
 * for bit.  workspace: device scratch of mgw_remap_bundle_frame_workspace_bytes() (the /4 maps), 8-byte aligned like xy.
 * Checked in the order of the batch calls: sizes and format (0 <= S <= 65535, h, w >= 8, 1 <= H, W <= 32767, H and W even for
 * YUV, S*H*W*3 < 2^31, S*h*w < 2^31), then S = 0 returns MGW_OK and launches nothing, then the pointers and their alignment. */
MGW_API size_t mgw_remap_bundle_frame_workspace_bytes(int S, int h, int w, int H, int W);
MGW_API int mgw_remap_bundle_frame(const uint8_t* src, int format, const float* xy, int S, int h, int w, int H, int W,
                               uint8_t* dst, void* workspace, void* stream);

/* ---- f1 for the encoder: the stabilised frames as YUV 4:2:0 ------------------------------------------------------------
 * mgw_remap_bundle_frame with the result written as dst [S,3H/2,W] uint8 in dst_format, MGW_YUV420_NV12 (what NVENC takes) or
 * MGW_YUV420_I420 (yuv420p, what libx264 / libavcodec take), in the layouts above: byte for byte cv2.cvtColor(F,
 * COLOR_BGR2YUV_I420) of the BGR frame F that mgw_remap_bundle_frame gives, its U and V planes interleaved for NV12.  That is
 * BT.601 limited range in 20-bit fixed point, Y of every pixel and U, V of the top-left pixel of each 2x2 block (no chroma
 * averaging); the conversion runs inside the warp and the BGR frame is never written.  Half the bytes of the BGR result.  The
 * rows are packed (pitch W); mgw_remap_bundle_frame_planes below writes pitched encoder surfaces.  Same workspace as
 * mgw_remap_bundle_frame.
 * Checked in the order of the batch calls: mgw_remap_bundle_frame's sizes and source format with H and W even for every source,
 * and dst_format NV12 or I420 (MGW_BGR24 is rejected: that result is mgw_remap_bundle_frame's), then S = 0 returns MGW_OK and
 * launches nothing, then the pointers and their alignment. */
MGW_API int mgw_remap_bundle_frame_yuv420(const uint8_t* src, int format, const float* xy, int S, int h, int w, int H, int W,
                               int dst_format, uint8_t* dst, void* workspace, void* stream);

/* ---- f1 for a batch of videos of different source sizes, each stabilised at its own size -------------------------------
 * src is a pool of the per-slot calls above (format, capacity (max_h, max_w), sizes [S,2] device int32, 8-byte aligned), xy
 * [S,h,w,2] as for mgw_remap_bundle_frame.  dst holds S regions of dst_frame_bytes(max_h, max_w) (3*max_h*max_w for MGW_BGR24,
 * 3*max_h*max_w/2 for YUV 4:2:0); slot s's result lies contiguous at the start of its region in the slot's own size: BGR
 * [H_s,W_s,3] or, for dst_format MGW_YUV420_NV12 / _I420, [3H_s/2,W_s].  Every active slot's bytes are those of
 * mgw_remap_bundle_frame (MGW_BGR24) or mgw_remap_bundle_frame_yuv420 on that slot's frame alone at (H_s, W_s) with xy[s].  Bytes
 * past a slot's result inside its region are not written, nor is any byte of an idle slot's region: size 0, above the capacity,
 * or odd when either format is YUV.  workspace: mgw_remap_bundle_frame_workspace_bytes(S, h, w, ., .).
 * Checked in the order of the batch calls: both formats and the sizes (0 <= S <= 65535, h, w >= 8, 1 <= max_h, max_w <= 32767,
 * the capacity even when either format is YUV, S*max_h*max_w*3 < 2^31, S*h*w < 2^31), then S = 0 returns MGW_OK and launches
 * nothing, then the pointers and the 8-byte alignment of xy, workspace and sizes. */
MGW_API int mgw_remap_bundle_frame_mixed(const uint8_t* src, int format, int S, int max_h, int max_w, const int32_t* sizes,
                               const float* xy, int h, int w, int dst_format, uint8_t* dst, void* workspace, void* stream);

/* ---- moving a pool of per-slot frames across PCIe: exactly each slot's bytes --------------------------------------------
 * src and dst are pools of the per-slot calls above (format, capacity (max_h, max_w), sizes [S,2] device int32, 8-byte
 * aligned).  For every active slot s the first frame_bytes(format, sizes[s]) bytes of src + s * frame_bytes(max_h, max_w) are
 * copied to the same offset of dst; bytes past them, and every byte of an idle slot's region (size 0, above the capacity, odd
 * for YUV), are neither read nor written.  One kernel, which reads the sizes when it runs, so a captured graph keeps working
 * when a slot changes size.  Unlike every other call here, src and dst may each be pinned host memory (cudaHostAlloc /
 * cudaHostRegister, read or written through its mapped device address across PCIe) as well as device or managed memory: the
 * upload of a pinned host pool into the device pool, the download of an output pool, or a device copy.  Pageable host memory
 * is refused (MGW_ERR_INVALID, "pageable" in mgw_last_error()) before anything is launched.
 * Checked in the order of the batch calls: the format, the sizes (0 <= S <= 65535, 1 <= max_h, max_w <= 32767, even for YUV,
 * S * frame_bytes(max_h, max_w) < 2^31), then S = 0 returns MGW_OK and launches nothing, then null pointers, src and dst 16-byte
 * aligned, sizes 8-byte aligned, then the first and the last byte of src and of dst must be device, managed or pinned host
 * memory (cudaPointerGetAttributes; legal inside a stream capture). */
MGW_API int mgw_copy_slots_mixed(const uint8_t* src, uint8_t* dst, int format, int S, int max_h, int max_w, const int32_t* sizes,
                               void* stream);

/* ---- f1/f2 straight from decoder surfaces into encoder surfaces: per-slot plane pointers and pitches ---------------------
 * A batch of S frames of one size H x W whose frames lie wherever a decoder (or an encoder's input pool) put them: each slot is
 * described by one mgw_planes entry of a table in device memory, [S] entries, 16-byte aligned (48 bytes each: every entry is).
 * plane[k] is a device address and pitch[k] its row pitch in bytes (any value, aligned or not; planes need not be adjacent):
 *   MGW_BGR24:       plane[0] holds H rows of 3W used bytes.
 *   MGW_YUV420_NV12: plane[0] is Y (H rows of W bytes), plane[1] interleaved U,V (H/2 rows of W bytes); NVDEC's layout of a
 *                    1080p surface is plane[1] = plane[0] + pitch * 1088.
 *   MGW_YUV420_I420: plane[0] is Y, plane[1] / plane[2] are U / V (H/2 rows of W/2 bytes each), e.g. an AVFrame's data[0..2]
 *                    with linesize[0..2].
 * Unused planes, pitches and `reserved` are ignored.  A slot is idle when a plane its format needs is 0 or a needed pitch is below
 * that plane's row bytes: its blocks return before writing anything (no tmp, out or dst rows, no byte of a destination surface),
 * so clearing an entry stops a slot and a bad entry can only stop it, never move an access.  The tables are read when the
 * kernels run, so a captured graph follows whatever surfaces the entries hold at each replay.  The tables travel as const void*.
 * mgw_cvt_img2train_planes: src table in `format` -> out [S,out_h,out_w]; tables and tmp (S*H*out_w bytes) as for the uniform
 *   batch call; byte for byte mgw_cvt_img2train_u8_batch / _yuv420_batch on the packed frames.
 * mgw_resize_linear_planes: -> dst [S,out_h,out_w,3] BGR, contiguous; tables as for the uniform batch call (2x2 INTER_AREA shortcut
 *   included); byte for byte mgw_resize_linear_u8_batch / _yuv420_batch on the packed frames.
 * mgw_remap_bundle_frame_planes: xy [S,h,w,2]; src table in `format`, dst table in dst_format (MGW_BGR24, MGW_YUV420_NV12 or
 *   _I420), both of frames H x W.  Each active slot's used bytes are mgw_remap_bundle_frame's (MGW_BGR24) or
 *   mgw_remap_bundle_frame_yuv420's on the packed frame; pitch padding and anything between planes is never written.  A
 *   contiguous buffer is the table whose pitches are the row bytes.  workspace: mgw_remap_bundle_frame_workspace_bytes().
 * Checked in the order of the batch calls: formats and sizes as for the uniform calls (H and W even when a format is YUV), then
 * S = 0 returns MGW_OK and launches nothing, then null pointers and alignment: the tables 16 bytes, xy and workspace 8 bytes, the
 * coefficient tables as in the uniform calls. */
/* 48 bytes: three 8-byte addresses and three 4-byte pitches take 36, and padding to 48 keeps every entry of a table 16-byte
 * aligned, so a block reads BGR / NV12 entries in two 16-byte loads (I420's V pitch in a third). */
typedef struct { uint64_t plane[3]; int32_t pitch[3]; int32_t reserved[3]; } mgw_planes;
MGW_API int mgw_cvt_img2train_planes(const void* src, int format, int S, int H, int W, const int32_t* kx, const int32_t* x0,
                               const int32_t* xn, int ksx, const int32_t* ky, const int32_t* y0, const int32_t* yn, int ksy, int out_h,
                               int out_w, uint8_t* tmp, float* out, void* stream);
MGW_API int mgw_resize_linear_planes(const void* src, int format, int S, int H, int W, const int32_t* xtab, const int32_t* ytab,
                               int out_h, int out_w, uint8_t* dst, void* stream);
MGW_API int mgw_remap_bundle_frame_planes(const void* src, int format, const float* xy, int S, int h, int w, int H, int W,
                               const void* dst, int dst_format, void* workspace, void* stream);

/* ---- f1/f2 for a batch of videos of different source sizes, straight from decoder surfaces into encoder surfaces -----------
 * The _mixed calls above with the pool replaced by a table of mgw_planes (the layouts of the plane-table calls): slot s's frame
 * has the size sizes[s] (device int32 [S,2], 8-byte aligned) and lies in the planes of entry s.  That entry also names the size
 * of the frame it describes: reserved[0] = its height, reserved[1] = its width (the plane-table calls above ignore `reserved`).
 * The capacity (max_h, max_w) and the per-slot tables, tmp [S,max_h,out_w] and out rows are those of the _mixed calls.
 * mgw_cvt_img2train_mixed_planes: -> out [S,out_h,out_w], as mgw_cvt_img2train_mixed.
 * mgw_resize_linear_mixed_planes: -> dst [S,out_h,out_w,3] BGR, packed, as mgw_resize_linear_mixed.
 * mgw_remap_bundle_frame_mixed_planes: xy [S,h,w,2]; each slot's result goes into entry s of the dst table (dst_format) at the
 *   slot's own size sizes[s], which that entry must carry too; pitch padding and anything between planes is never written.
 * Every active slot's bytes are bit-identical to the _mixed call on the packed pool of the same frames.  A slot is idle when
 * sizes[s] is idle under the _mixed rule (0, above the capacity, odd when a format is YUV), when a plane its format needs is 0 or
 * a needed pitch is below the plane's row bytes at the slot's width, or when an entry's size (reserved[0], reserved[1]) is not
 * sizes[s]: an idle slot writes no tmp / out / dst row and no byte of a destination surface.  So a slot that joins again at
 * another size stops until its entries name surfaces of the new size: a stale entry cannot move an access past its surface.
 * Checked in the order of the _mixed calls, with their checks except the limits on the pool's offsets: the capacity's 32-bit
 * limits hold for one frame (max_h*max_w < 2^29 for BGR, (3max_h/2)*max_w < 2^31 for YUV; 1 <= max_h, max_w <= 32767 for the
 * warp), the limits on tmp (S*max_h*out_w < 2^31), out (S*out_h*out_w < 2^29) and xy (S*h*w < 2^31) for all S; then S = 0
 * returns MGW_OK and launches nothing, then the pointers and their alignment, the tables last (16 bytes). */
MGW_API int mgw_cvt_img2train_mixed_planes(const void* src, int format, int S, int max_h, int max_w, const int32_t* sizes,
                               const int32_t* kx, const int32_t* x0, const int32_t* xn, int ksx, const int32_t* ky, const int32_t* y0,
                               const int32_t* yn, int ksy, int out_h, int out_w, uint8_t* tmp, float* out, void* stream);
MGW_API int mgw_resize_linear_mixed_planes(const void* src, int format, int S, int max_h, int max_w, const int32_t* sizes,
                               const int32_t* xtab, const int32_t* ytab, int out_h, int out_w, uint8_t* dst, void* stream);
MGW_API int mgw_remap_bundle_frame_mixed_planes(const void* src, int format, int S, int max_h, int max_w, const int32_t* sizes,
                               const float* xy, int h, int w, const void* dst, int dst_format, void* workspace, void* stream);

/* ---- a6: interpolate(im, x, y, out_size), spatial_transformer.py:200-281 ------------------------------
 * im [N,IH,IW,C]; x,y [N,OH,OW] normalised coords -> out [N,OH,OW,C]. */
MGW_API int mgw_interp_fwd(const float* im, const float* x, const float* y, int N, int IH, int IW, int C, int OH, int OW,
                   float* out, void* stream);
/* d_im [N,IH,IW,C] nullable (overwritten), dx, dy [N,OH,OW] nullable */
MGW_API int mgw_interp_bwd(const float* im, const float* x, const float* y, const float* d_out, int N, int IH, int IW,
                   int C, int OH, int OW, float* d_im, float* dx, float* dy, void* stream);

/* ---- a7: spatial_transformer.transformer(U, theta[N,9], out_size), spatial_transformer.py:143-193 -----
 * theta is divided by theta[8] (:151-153); black is [N,OH,OW].  The reference reshapes black with the input
 * dims (:184) and therefore only works for out_size == (H,W); this entry point accepts any out_size. */
MGW_API int mgw_homography_warp_fwd(const float* U, const float* theta, int N, int H, int W, int C, int OH, int OW,
                            float* out, float* black, float* img, void* stream);
MGW_API int mgw_homography_warp_bwd(const float* U, const float* theta, const float* d_out, int N, int H, int W, int C,
                            int OH, int OW, float* dU, float* dtheta, void* stream);

/* ---- a8: img_loss, s_net_bundle_nobm.py:347-352 --------------------------------------------------------
 * sums [N,2] = per-sample (sum e^2, sum (1-black)), e = (out - y)*(1-black); loss = sum_b s0/(s1+1e-8)/N is
 * finished by the caller (N scalars).  bwd: d_out = upstream * 2 e (1-black) / (s1+1e-8) / N. */
MGW_API int mgw_img_loss_fwd(const float* out, const float* y, const float* black, int N, int H, int W, int C,
                     float* sums, void* stream);
MGW_API int mgw_img_loss_bwd(const float* out, const float* y, const float* black, const float* sums, float upstream,
                     const float* upstream_dev, int N, int H, int W, int C, float* d_out, void* stream);

/* ---- a9: feature_loss / warp_pts, s_net_bundle_nobm.py:215-230,335-343 ---------------------------------
 * matches [N,M,4] (sx,sy,ux,uy), mask [N,M], img [N,H,W,2] -> warpped [N,M,2] nullable, per_sample [N]
 * (= sum_m mask*(|gx-ux|+|gy-uy|)/max(sum mask,1)); loss = mean_b per_sample.
 * bwd: d_img [N,H,W,2] must be zeroed by the caller or carry a gradient to accumulate into (sparse +=). */
MGW_API int mgw_feature_loss_fwd(const float* matches, const float* mask, const float* img, int N, int M, int H, int W,
                         float* warpped, float* per_sample, void* stream);
MGW_API int mgw_feature_loss_bwd(const float* matches, const float* mask, const float* img, float upstream,
                         const float* upstream_dev, int N, int M, int H, int W, float* d_img, void* stream);

/* ---- a10: temp_loss, train_bundle_nobm.py:115-125 -------------------------------------------------------
 * out1,out2 [N,H,W,C], black1,black2 [N,H,W], flow [N,H,W,2] -> sums [N,2] = (sum e^2, sum m),
 * m = (1-black1)*interp(1-black2, flow), e = (out1 - interp(out2, flow))*m.
 * bwd: d_out1 (overwritten), d_out2 (overwritten, scatter), upstream includes use_temp_loss. */
MGW_API int mgw_temp_loss_fwd(const float* out1, const float* black1, const float* out2, const float* black2,
                      const float* flow, int N, int H, int W, int C, float* sums, void* stream);
MGW_API int mgw_temp_loss_bwd(const float* out1, const float* black1, const float* out2, const float* black2,
                      const float* flow, const float* sums, float upstream, const float* upstream_dev, int N, int H, int W,
                      int C, float* d_out1, float* d_out2, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* MGW_H_ */

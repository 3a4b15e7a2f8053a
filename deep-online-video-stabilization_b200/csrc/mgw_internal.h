// Internal declarations shared by the .cu files of libmgw_b200.so (not part of the ABI).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stddef.h>

#include "../../include/mgw.h"
#include "mgw_device.cuh"

namespace mgw {

int set_error(int code, const char* fmt, ...);
int check_launch(const char* what);          // counts the launch, maps cudaGetLastError() to MGW_ERR_CUDA
void count_launches(int n);
int impl_mode();                             // MGW_IMPL environment override: 0 auto, 1 generic, 2 tma tiles, 3 forward pipeline (backward: tma tiles)

// Launch with (pdl = true) the programmatic-stream-serialization attribute: the kernel may be scheduled while the previous
// kernel of the stream is still running and synchronises with it through griddep_wait() (mgw_device.cuh).
template <typename... KArgs, typename... Args>
static inline cudaError_t launch_ex(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, bool pdl, Args&&... args)
{
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = st;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = at; cfg.numAttrs = pdl ? 1 : 0;
    return cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}
bool pdl_enabled();                          // MGW_PDL=0 switches programmatic dependent launch off (tuning / debugging aid)

struct WarpShape {
    int N, H, W, C;          // source image (and output, for the mesh op)
    int OH, OW;              // output size
    int gh, gw;              // mesh cells (1x1 for the single-homography op)
};

// mgw_solve.cu
int launch_vertices_fwd(const float* head, int N, int gh, int gw, float do_crop_rate, float* pts2, float* pts1, cudaStream_t st);
// id_coef / id_dev: optional id-loss term added to d_head: id_coef * (id_dev ? *id_dev : 1) * sign(head)  (s_net_bundle_nobm.py:246)
int launch_vertices_bwd(const float* head, const float* d_pts2, const float* d_pts1, int N, int gh, int gw,
                        float do_crop_rate, float* d_head, cudaStream_t st, float id_coef = 0.0f, const float* id_dev = nullptr);
int launch_solve_h_fwd(const float* theta, int N, int gh, int gw, float* Hs, cudaStream_t st);
int launch_solve_h_bwd(const float* theta, const float* Hs, const float* dHs_part, int nparts, int part_stride,
                       int N, int gh, int gw, float* dtheta, cudaStream_t st, bool after_own_warp_kernel = false,
                       const float* extra_part = nullptr /*[cells,8] one more partial per cell*/);

// mgw_warp_generic.cu : any shape, global gather / global atomics
// normalize: Hs holds raw [N,9] homographies to be divided by H[8] (spatial_transformer.py:151-153)
int launch_warp_fwd_generic(const float* U, const float* Hs, const WarpShape& s, bool normalize, float* out,
                            float* black, float* img, int32_t* cell_idx, cudaStream_t st);
int launch_warp_bwd_generic(const float* U, const float* Hs, const float* d_out, const float* d_img,
                            const WarpShape& s, bool normalize, float* dU, float* dHs /*[cells,9] zeroed*/,
                            cudaStream_t st);
int launch_homography_finish_bwd(const float* theta, const float* dHn, int N, float* dtheta, cudaStream_t st);

// mgw_interp.cu
int launch_interp_fwd(const float* im, const float* x, const float* y, int N, int IH, int IW, int C, int OH, int OW,
                      float* out, cudaStream_t st);
int launch_interp_bwd(const float* im, const float* x, const float* y, const float* d_out, int N, int IH, int IW,
                      int C, int OH, int OW, float* d_im, float* dx, float* dy, cudaStream_t st);

// mgw_loss.cu
int launch_img_loss_fwd(const float* out, const float* y, const float* black, int N, int H, int W, int C, float* sums, cudaStream_t st);
int launch_img_loss_bwd(const float* out, const float* y, const float* black, const float* sums, float upstream,
                        const float* up_dev, int N, int H, int W, int C, float* d_out, cudaStream_t st, const float* add = nullptr);
int launch_feature_loss_fwd(const float* matches, const float* mask, const float* img, int N, int M, int H, int W,
                            float* warpped, float* per_sample, cudaStream_t st);
int launch_feature_loss_bwd(const float* matches, const float* mask, const float* img, float upstream, const float* up_dev, int N, int M,
                            int H, int W, float* d_img, cudaStream_t st);
int launch_temp_loss_fwd(const float* out1, const float* black1, const float* out2, const float* black2,
                         const float* flow, int N, int H, int W, int C, float* sums, cudaStream_t st);
int launch_temp_loss_bwd(const float* out1, const float* black1, const float* out2, const float* black2,
                         const float* flow, const float* sums, float upstream, const float* up_dev, int N, int H, int W, int C,
                         float* d_out1, float* d_out2, cudaStream_t st);

// mgw_loss_tile.cu : temp_loss on TMA-staged tiles (locally compact flow fields; per-pixel fallback inside)
bool temp_loss_tile_supported(const float* out2, const float* black2, const float* d_out2, int N, int H, int W, int C);
int launch_temp_loss_tile_fwd(const float* out1, const float* black1, const float* out2, const float* black2, const float* flow, int N,
                              int H, int W, int C, float* sums, cudaStream_t st);
int launch_temp_loss_tile_bwd(const float* out1, const float* black1, const float* out2, const float* black2, const float* flow,
                              const float* sums, float upstream, const float* up_dev, int N, int H, int W, int C, float* d_out1,
                              float* d_out2, cudaStream_t st);

// mgw_warp_tma.cu : TMA-staged tiles (fast path)
struct FusedImgLoss {            // img_loss fused onto the warp (s_net_bundle_nobm.py:347-352)
    const float* out;            // backward: the forward's output_img
    const float* y;              // target frames [N,H,W,C]
    const float* black;          // backward: the forward's black_pix
    const float* sums;           // backward: [N,2] per-sample (sum e^2, sum (1-black)) from the fused forward
    float kscale;                // backward: upstream * 2 / batch
    const float* kscale_dev;     // backward, nullable: device scalar multiplied onto kscale (the autograd upstream, no host sync)
};
bool tma_fwd_supported(const WarpShape& s);
// y_tgt / sums nullable: when given, the img_loss partial sums are accumulated into sums[N,2] (must be zeroed)
int launch_warp_fwd_tma(const float* U, const float* Hs, const WarpShape& s, float* out, float* black, float* img,
                        const float* y_tgt, float* sums, cudaStream_t st);
bool tma_bwd_supported(const WarpShape& s);
size_t tma_bwd_workspace_bytes(const WarpShape& s);
// fl nullable: when given, d_out is ignored and the upstream gradient is the fused img_loss's
int launch_warp_bwd_tma(const float* U, const float* Hs, const float* d_out, const float* d_img, const WarpShape& s,
                        float* dU, float* dHs_part, int* nparts, const FusedImgLoss* fl, cudaStream_t st,
                        bool behind_own_fill = false);      // true: the kernel right before us in `st` is the library's zero-fill of dU

// mgw_warp_pipe.cu : forward as a persistent warp-specialised pipeline over TMA-staged tiles (serves the full call:
// out + black + img)
bool pipe_fwd_supported(const WarpShape& s);
int launch_warp_fwd_pipe(const float* U, const float* Hs, const WarpShape& s, float* out, float* black, float* img, cudaStream_t st);

// mgw_deploy.cu : deploy-side colour-frame warp (deploy_bundle.py:136-146)
size_t remap_bundle_workspace_bytes(int N, int H, int W);
int launch_remap_bundle_u8(const uint8_t* img, const float* xy, int N, int H, int W, int C, uint8_t* dst, void* workspace,
                           cudaStream_t st);
// the same warp with maps xy [N,h,w,2] of the network's size applied to frames of the output's size H x W: BGR / C-channel
// [N,H,W,C] (src_fmt 0) or YUV 4:2:0 [N,3H/2,W] (C = 3) -> dst [N,H,W,C]; the workspace is remap_bundle_workspace_bytes(N, h, w)
int launch_remap_bundle(const uint8_t* src, int src_fmt, int C, const float* xy, int N, int h, int w, int H, int W, uint8_t* dst,
                        void* workspace, cudaStream_t st);
// the same warp (C = 3, H and W even) with the result as YUV 4:2:0, dst [N,3H/2,W] in dst_fmt (MGW_YUV420_NV12 / _I420): Y, U, V as
// cv2.cvtColor(COLOR_BGR2YUV_I420) computes them from the BGR result, converted inside the warp
int launch_remap_bundle_yuv420(const uint8_t* src, int src_fmt, const float* xy, int N, int h, int w, int H, int W, int dst_fmt,
                               uint8_t* dst, void* workspace, cudaStream_t st);
// the warp per slot at the slot's own size sizes[s] (int32 [S,2], 8-byte aligned): slot s's frame at src + s * frame_bytes(max_h,
// max_w) in src_fmt, its result at dst + s * dst_frame_bytes(max_h, max_w) in dst_fmt (MGW_BGR24 or YUV 4:2:0); xy [S,h,w,2].
// Slots with a size of 0, above the capacity or odd (either format YUV) write nothing.
int launch_remap_bundle_mixed(const uint8_t* src, int src_fmt, int S, int max_h, int max_w, const int32_t* sizes, const float* xy,
                              int h, int w, int dst_fmt, uint8_t* dst, void* workspace, cudaStream_t st);
// each active slot's frame_bytes(fmt, sizes[s]) bytes from src + s * stride to dst + s * stride (stride = frame_bytes(fmt, max_h,
// max_w)); src / dst 16-byte aligned device addresses (a pinned host buffer's mapped one), sizes 8-byte aligned; idle slots as above
int launch_copy_slots_mixed(const uint8_t* src, uint8_t* dst, int fmt, int S, int max_h, int max_w, const int32_t* sizes, cudaStream_t st);

// S frames of one size ([S,H,W,C] -> [S,out_h,out_w,C]; S >= 1, the single-frame calls pass 1).  src_fmt: 0 for the BGR / C-channel
// frames, MGW_YUV420_NV12 or MGW_YUV420_I420 for YUV 4:2:0 frames [S,3H/2,W] read as the BGR frames cvtColor makes of them (C = 3)
int launch_resize_linear_u8(const uint8_t* img, int S, int H, int W, int C, const int32_t* xtab, const int32_t* ytab, int out_h, int out_w,
                            uint8_t* dst, cudaStream_t st, int src_fmt = 0);
int launch_cvt_img2train_u8(const uint8_t* bgr, int S, int H, int W, const int32_t* kx, const int32_t* x0, const int32_t* xn, int ksx,
                            const int32_t* ky, const int32_t* y0, const int32_t* yn, int ksy, int out_h, int out_w, uint8_t* tmp,
                            float* out, cudaStream_t st, int src_fmt = 0);
// per-slot source geometry: slot s's frame of size sizes[s] (int32 [S,2], 8-byte aligned) at src + s * frame_bytes(max_h, max_w),
// per-slot tables; BGR (src_fmt 0) or YUV 4:2:0, C = 3.  Slots with a size of 0, above the capacity or odd (YUV) write nothing.
int launch_cvt_img2train_mixed(const uint8_t* src, int src_fmt, int S, int max_h, int max_w, const int32_t* sizes, const int32_t* kx,
                               const int32_t* x0, const int32_t* xn, int ksx, const int32_t* ky, const int32_t* y0, const int32_t* yn,
                               int ksy, int out_h, int out_w, uint8_t* tmp, float* out, cudaStream_t st);
int launch_resize_linear_mixed(const uint8_t* src, int src_fmt, int S, int max_h, int max_w, const int32_t* sizes, const int32_t* xtab,
                               const int32_t* ytab, int out_h, int out_w, uint8_t* dst, cudaStream_t st);
// per-slot planes: slot s's source frame (and, for the warp, its result) described by entry s of a device table of mgw_planes
// (16-byte aligned); S frames of one size H x W, uniform tables; slots whose entry lacks a plane or has a short pitch write nothing
int launch_cvt_img2train_planes(const mgw_planes* src, int src_fmt, int S, int H, int W, const int32_t* kx, const int32_t* x0,
                                const int32_t* xn, int ksx, const int32_t* ky, const int32_t* y0, const int32_t* yn, int ksy, int out_h,
                                int out_w, uint8_t* tmp, float* out, cudaStream_t st);
int launch_resize_linear_planes(const mgw_planes* src, int src_fmt, int S, int H, int W, const int32_t* xtab, const int32_t* ytab,
                                int out_h, int out_w, uint8_t* dst, cudaStream_t st);
int launch_remap_bundle_planes(const mgw_planes* src, int src_fmt, const float* xy, int S, int h, int w, int H, int W,
                               const mgw_planes* dst, int dst_fmt, void* workspace, cudaStream_t st);
int launch_warp_rev_bundle_u8(const uint8_t* img, const double* Hs_cvt, int N, int H, int W, int C, int gh, int gw, uint8_t* dst,
                              cudaStream_t st);

// frame transport: uint8 <-> the network's fp32 range (config.py:19, deploy_bundle.py:75), and a zero-fill that can leave its
// lines resident in L2 (the dU buffer the backward accumulates into)
int launch_u8_to_train(const uint8_t* src, float* dst, size_t n, cudaStream_t st);
int launch_train_to_u8(const float* src, uint8_t* dst, size_t n, cudaStream_t st);
int launch_fill_zero(void* p, size_t bytes, bool keep_in_l2, cudaStream_t st);

// mgw_vertex_loss.cu : vertex regularisers (s_net_bundle_nobm.py:139-210,246-247)
int launch_vertex_losses_fwd(const float* theta, const float* pts1, const float* pts2, int N, int gh, int gw, float do_crop_rate,
                             float* sums, float* black_err, cudaStream_t st, bool sums_zeroed = false /* true: several blocks, reduce-adds */);
int launch_vertex_losses_bwd(const float* theta, const float* pts1, const float* pts2, int N, int gh, int gw, float do_crop_rate,
                             const float* f, float* d_theta, float* d_pts1, float* d_pts2,
                             cudaStream_t st);
// the same with f[k] = coef[k] * (g_dev ? *g_dev : 1) and d_pts2 += instead of = (the warp's dtheta is already in it)
int launch_vertex_losses_bwd_coef(const float* pts1, const float* pts2, int N, int gh, int gw, float do_crop_rate, const float coef[4],
                                  const float* g_dev, float* d_pts1, float* d_pts2_acc, cudaStream_t st);

// mgw_pass.cu : the pieces that turn one training pass (s_net_bundle_nobm.py:266-381) into a handful of launches
struct PassCoef {            // total = v[0] vsums[0] + gate * (sum_{k>0} v[k] vsums[k] + img IMG + feat FEAT + regu REGU)   (:354-359)
    float v[4];              // multipliers of the vertex sums (id, black_pos, distortion, consistency), element counts folded in
    float img, feat, regu;   // IMG = sum_n e2_n / (nb_n + 1e-8) / batch, FEAT = sum_n acc_n / max(cnt_n, 1) / batch
    float theta_share, grid_theta_share;   // split of the id term into ret['theta_loss'] / ret['grid_theta_loss']
    float inv_batch;
    float gate;              // 1 - use_theta_only; the parts of `ret` are reported without it, as the reference does
};
int launch_ratio_sum(const float* sums /*[N,2]*/, int N, bool clamp, float scale, float* out, cudaStream_t st);
int launch_feature_acc_fwd(const float* matches, const float* mask, const float* img, int N, int M, int H, int W, float* warpped,
                           float* facc /*[N,2] zeroed*/, cudaStream_t st);
int launch_feature_dh(const float* matches, const float* mask, const float* img, const float* Hs, const float* facc, float upstream,
                      const float* up_dev, int N, int M, int H, int W, int gh, int gw, float* extra_part /*[cells,8]*/, cudaStream_t st);
int launch_objective_fwd(const float* img_sums, const float* facc, const float* vsums, const float* regu_dev, int N, const PassCoef& c,
                         float* result /*[9]: total, then the 8 weighted parts*/, cudaStream_t st);

// mgw_crop.cu : deploy-side crop (deploy_bundle.py:240,291,344-365)
int launch_black_accumulate(const float* black, int32_t* all_black, int n, cudaStream_t st);
size_t crop_rect_workspace_bytes(int H, int W);
int launch_crop_rect(const int32_t* all_black, int H, int W, int step, void* workspace, int32_t* rect, cudaStream_t st);

// mgw_stream.cu : deploy-side streaming state (device-resident history rings, deploy_bundle.py:204-232,259-295,319-327)
// S > 1 (device heads only): S independent streams, rings [S][depth][H][W], heads head_dev[S], pixels [S][H][W]
int launch_stream_assemble(const float* frames, const float* masks, int depth, int head, const int* taps_host, int ntaps, int use_masks,
                           const float* cur, int H, int W, float* in_x, cudaStream_t st, const int* head_dev = nullptr, int S = 1);
int launch_stream_push(float* frames, float* masks, int depth, int slot, const float* img, const float* black, int H, int W,
                       float* frame_out, int out_stride, cudaStream_t st, const int* head_dev = nullptr, int S = 1);
int launch_stream_advance(int* head_dev, int depth, cudaStream_t st, int S = 1);

}  // namespace mgw

// Deploy-side streaming state (deploy_bundle.py:204-232 initialisation, :259-272 input assembly, :283-295 refine re-feed,
// :319-327 update): the reference keeps the last `before_ch` = 32 stabilised frames and their black masks in Python lists
// and rebuilds the 13-channel network input on the host every frame.  Here both histories are device-resident rings
// [depth][H][W]; one launch assembles the NHWC input from the index taps (masks[-i] for the taps, frames[-i] for the taps,
// the current frame), one launch pushes the new stabilised frame (img + black * (-1), :292) and its mask.  Pure data
// movement and one fp32 operation: exact.
#include "mgw_internal.h"

namespace mgw {

namespace {

constexpr int kMaxTaps = 32;
struct Taps32 { int slot[kMaxTaps]; };

// in_x[p][c]: c < nmask -> masks[slot[c]][p]; then frames[slot[c - nmask]][p]; last channel = cur[p]
// head_dev != nullptr: taps.slot[] holds the tap DISTANCES i (list[-i]) and the slot is resolved here from the device-resident
// head, so that the launch parameters never change from frame to frame (CUDA-graph replay of the whole frame loop)
// Several independent streams (StreamBatch): blockIdx.y = stream s, whose rings are frames / masks + s*depth*HW, its head
// head_dev[s] and its pixels cur / img / black + s*HW.  The stream goes in the grid's y dimension rather than being folded
// into the pixel index: a block offsets its base pointers once and the per-pixel arithmetic stays that of one stream, so the
// single-stream calls (gridDim.y = 1) run the same instructions as before the batch existed.
__device__ __forceinline__ int ring_slot(int head, int i, int depth) { return ((head - (i - 1)) % depth + depth) % depth; }

__global__ void __launch_bounds__(256)
stream_assemble_kernel(const float* __restrict__ frames, const float* __restrict__ masks, const __grid_constant__ Taps32 taps_in,
                       int ntaps, int use_masks, const float* __restrict__ cur, int HW, float* __restrict__ in_x,
                       const int* __restrict__ head_dev, int depth)
{
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= HW) return;
    const int s = blockIdx.y;
    const size_t ring = (size_t)s * depth * HW;
    frames += ring;
    if (use_masks) masks += ring;
    cur += (size_t)s * HW;
    Taps32 taps = taps_in;
    if (head_dev) {
        const int head = __ldg(head_dev + s);
        for (int k = 0; k < ntaps; ++k) taps.slot[k] = ring_slot(head, taps_in.slot[k], depth);
    }
    const int nch = (use_masks ? 2 : 1) * ntaps + 1;
    float* o = in_x + ((size_t)s * HW + p) * nch;
    int c = 0;
    if (use_masks)
        for (int k = 0; k < ntaps; ++k) o[c++] = __ldg(masks + (size_t)taps.slot[k] * HW + p);
    for (int k = 0; k < ntaps; ++k) o[c++] = __ldg(frames + (size_t)taps.slot[k] * HW + p);
    o[c] = __ldg(cur + p);
}

__global__ void __launch_bounds__(256)
stream_push_kernel(float* __restrict__ frame_slot, float* __restrict__ mask_slot, const float* __restrict__ img,
                   const float* __restrict__ black, int HW, float* __restrict__ frame_out, int out_stride,
                   const int* __restrict__ head_dev, int depth)
{
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= HW) return;
    const int s = blockIdx.y;
    if (head_dev) {                                   // frame_slot / mask_slot are the ring bases: write the slot after the head
        const size_t off = ((size_t)s * depth + (__ldg(head_dev + s) + 1) % depth) * HW;
        if (frame_slot) frame_slot += off;
        if (mask_slot) mask_slot += off;
    }
    img += (size_t)s * HW;
    black += (size_t)s * HW;
    const float b = __ldg(black + p);
    const float f = __fadd_rn(__ldg(img + p), __fmul_rn(b, -1.0f));         // frame = img + black * (-1)   (:292)
    if (frame_slot) frame_slot[p] = f;
    if (mask_slot) mask_slot[p] = b;
    if (frame_out) frame_out[(size_t)p * out_stride] = f;                    // refine: tmp_in_x[..., -1] = frame  (:295)
}

__global__ void stream_advance_kernel(int* head, int S, int depth)
{
    const int s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s < S) head[s] = (head[s] + 1) % depth;
}

}  // namespace

int launch_stream_assemble(const float* frames, const float* masks, int depth, int head, const int* taps_host, int ntaps, int use_masks,
                           const float* cur, int H, int W, float* in_x, cudaStream_t st, const int* head_dev, int S)
{
    if (ntaps < 0 || ntaps > kMaxTaps) return set_error(MGW_ERR_INVALID, "stream_assemble: at most %d taps (got %d)", kMaxTaps, ntaps);
    Taps32 t{};
    for (int k = 0; k < ntaps; ++k) {
        const int i = taps_host[k];
        if (i < 1 || i > depth) return set_error(MGW_ERR_INVALID, "stream_assemble: tap %d outside [1, depth = %d]", i, depth);
        t.slot[k] = head_dev ? i : ((head - (i - 1)) % depth + depth) % depth;    // list[-i] with the newest entry at `head`
    }
    const int HW = H * W;
    stream_assemble_kernel<<<dim3((HW + 255) / 256, S), 256, 0, st>>>(frames, masks, t, ntaps, use_masks, cur, HW, in_x, head_dev, depth);
    return check_launch("stream_assemble");
}

int launch_stream_push(float* frames, float* masks, int depth, int slot, const float* img, const float* black, int H, int W,
                       float* frame_out, int out_stride, cudaStream_t st, const int* head_dev, int S)
{
    const int HW = H * W;
    float* fs = frames ? frames + (head_dev ? 0 : (size_t)slot * HW) : nullptr;
    float* ms = masks ? masks + (head_dev ? 0 : (size_t)slot * HW) : nullptr;
    stream_push_kernel<<<dim3((HW + 255) / 256, S), 256, 0, st>>>(fs, ms, img, black, HW, frame_out, out_stride, head_dev, depth);
    return check_launch("stream_push");
}

int launch_stream_advance(int* head_dev, int depth, cudaStream_t st, int S)
{
    const int threads = S < 256 ? S : 256;
    stream_advance_kernel<<<(S + threads - 1) / threads, threads, 0, st>>>(head_dev, S, depth);
    return check_launch("stream_advance");
}

}  // namespace mgw

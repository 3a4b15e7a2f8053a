// Deploy-side colour-frame warp: warpRevBundle2 of deploy_bundle.py:136-146.
//   x_map, y_map (the operator's outputs, [N,H,W,2] interleaved)  --cv2.resize /4-->  small maps  --cv2.resize x4-->
//   smoothed maps  --((m+1)/2*size)-->  pixel coordinates  --cv2.remap(INTER_LINEAR, constant border 0)-->  uint8 frame
// Two launches: K5a writes the /4 maps (a 74 KB scratch at 288x512, L2 resident), K5b upsamples them per output pixel,
// converts to OpenCV's 1/32-pixel fixed point and blends the uint8 taps with OpenCV's 15-bit integer weights.  The
// arithmetic restates OpenCV's published algorithm (resize.cpp resizeGeneric_/HResizeLinear/VResizeLinear, plain C++
// path; imgwarp.cpp remapBilinear) operation by operation: deploy_ref.py (test infrastructure) is the numpy statement of the same thing
// and is pinned bit-exact against cv2 (tests/golden/deploy_remap.npz).  HBM-bound byte work: no tensor cores.
#include "mgw_internal.h"

namespace mgw {

namespace {

struct Lin { int i0, i1; float a0, a1; };

// resize.cpp: inv_scale = dsize / (double)ssize, scale = 1. / inv_scale, fx = (float)((d + 0.5) * scale - 0.5).  The scale is the
// same IEEE double on the host and the device, so a kernel may take it as a launch argument (resize_scale) instead of dividing.
__host__ __device__ __forceinline__ double resize_scale(int n_out, int n_in) { return 1.0 / ((double)n_out / (double)n_in); }

__device__ __forceinline__ float src_pos_s(int d, double scale) { return (float)(((double)d + 0.5) * scale - 0.5); }

__device__ __forceinline__ float src_pos(int d, int n_out, int n_in) { return src_pos_s(d, resize_scale(n_out, n_in)); }

// horizontal taps: a tap outside the row is folded onto the border with weight 0
__device__ __forceinline__ Lin hcoef_at(float fx, int n_in)
{
    int sx = (int)floorf(fx);
    fx = __fsub_rn(fx, (float)sx);
    if (sx < 0) { sx = 0; fx = 0.0f; }
    if (sx >= n_in - 1) { sx = n_in - 1; fx = 0.0f; }
    Lin l;
    l.i0 = sx; l.i1 = min(sx + 1, n_in - 1); l.a0 = __fsub_rn(1.0f, fx); l.a1 = fx;
    return l;
}

// vertical taps: row indices clamped, weights kept
__device__ __forceinline__ Lin vcoef_at(float fy, int n_in)
{
    const int sy = (int)floorf(fy);
    fy = __fsub_rn(fy, (float)sy);
    Lin l;
    l.i0 = min(max(sy, 0), n_in - 1); l.i1 = min(max(sy + 1, 0), n_in - 1); l.a0 = __fsub_rn(1.0f, fy); l.a1 = fy;
    return l;
}

__device__ __forceinline__ Lin hcoef(int d, int n_out, int n_in) { return hcoef_at(src_pos(d, n_out, n_in), n_in); }
__device__ __forceinline__ Lin vcoef(int d, int n_out, int n_in) { return vcoef_at(src_pos(d, n_out, n_in), n_in); }

// one bilinear resize sample of an interleaved (x,y) map: rows first horizontally, then vertically, fp32 mul / add
__device__ __forceinline__ float2 resize_sample(const float2* __restrict__ s, int sw, const Lin& h, const Lin& v)
{
    const float2 p00 = __ldg(s + (size_t)v.i0 * sw + h.i0), p01 = __ldg(s + (size_t)v.i0 * sw + h.i1);
    const float2 p10 = __ldg(s + (size_t)v.i1 * sw + h.i0), p11 = __ldg(s + (size_t)v.i1 * sw + h.i1);
    const float r0x = __fadd_rn(__fmul_rn(p00.x, h.a0), __fmul_rn(p01.x, h.a1));
    const float r1x = __fadd_rn(__fmul_rn(p10.x, h.a0), __fmul_rn(p11.x, h.a1));
    const float r0y = __fadd_rn(__fmul_rn(p00.y, h.a0), __fmul_rn(p01.y, h.a1));
    const float r1y = __fadd_rn(__fmul_rn(p10.y, h.a0), __fmul_rn(p11.y, h.a1));
    return make_float2(__fadd_rn(__fmul_rn(r0x, v.a0), __fmul_rn(r1x, v.a1)), __fadd_rn(__fmul_rn(r0y, v.a0), __fmul_rn(r1y, v.a1)));
}

__global__ void __launch_bounds__(256)
maps_down_kernel(const float2* __restrict__ xy, int N, int H, int W, int h4, int w4, float2* __restrict__ small)
{
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= N * h4 * w4) return;
    const int c = t % w4, r = (t / w4) % h4, n = t / (w4 * h4);
    const Lin h = hcoef(c, w4, W), v = vcoef(r, h4, H);
    small[t] = resize_sample(xy + (size_t)n * H * W, W, h, v);
}

constexpr int SRC_BGR = 0;

// cv2.cvtColor(COLOR_YUV2BGR_NV12 / _I420), color_yuv.simd.hpp: BT.601 limited range in 20-bit fixed point, one chroma sample per
// 2x2 block, no chroma interpolation.  The chroma terms (rounding constant included) are formed once per chroma sample.
struct Chroma { int r, g, b; };

__device__ __forceinline__ Chroma yuv_chroma(int U, int V)
{
    const int u = U - 128, v = V - 128;
    return Chroma{(1 << 19) + 1673527 * v, (1 << 19) - 852492 * v - 409993 * u, (1 << 19) + 2116026 * u};
}

// the per-pixel half: y = max(0, Y-16)*CY, channel = sat8((y + chroma term) >> 20); every sum fits int32
__device__ __forceinline__ int3 yuv_to_bgr(int Y, const Chroma& c)
{
    const int y = max(Y - 16, 0) * 1220542;
    return make_int3(min(max((y + c.b) >> 20, 0), 255), min(max((y + c.g) >> 20, 0), 255), min(max((y + c.r) >> 20, 0), 255));
}

// the chroma sample of pixel (row, x) in a frame [3H/2, W]: after the H*W bytes of the Y plane, NV12 interleaves U,V in rows of W
// bytes; I420 has the U plane (H/2 rows of W/2) and then the V plane -- contiguous planes, so byte offsets, not row offsets
template <int FMT>
__device__ __forceinline__ Chroma yuv_chroma_at(const uint8_t* __restrict__ f, int H, int W, int row, int x)
{
    const uint8_t* c = f + (size_t)H * W;
    if constexpr (FMT == MGW_YUV420_NV12) {
        const uint8_t* p = c + (size_t)(row >> 1) * W + (x & ~1);
        return yuv_chroma(__ldg(p), __ldg(p + 1));
    } else {
        const uint8_t* p = c + (size_t)(row >> 1) * (W >> 1) + (x >> 1);
        return yuv_chroma(__ldg(p), __ldg(p + (size_t)(H >> 1) * (W >> 1)));
    }
}

// bytes of one source frame: a batch's frames are contiguous
template <int FMT>
__device__ __forceinline__ size_t src_frame_bytes(int H, int W)
{
    return FMT == SRC_BGR ? (size_t)H * W * 3 : (size_t)H * W * 3 / 2;
}

// Per-slot geometry (MIXED kernels): a slot is idle -- its blocks return before they write anything -- when its size is 0, larger
// than the capacity, or odd for a YUV format (the source's, or the result's in the warp): never-joined slots, and a bad
// device-side size cannot move an access outside the slot's region.
template <int FMT>
__device__ __forceinline__ bool slot_active(int2 sz, int max_h, int max_w)
{
    return sz.x > 0 && sz.y > 0 && sz.x <= max_h && sz.y <= max_w && (FMT == SRC_BGR || ((sz.x | sz.y) & 1) == 0);
}

// Per-slot planes (PLANES kernels): slot s's frame is described by entry s of a table of mgw_planes in device memory, each plane
// at its own address with its own row pitch, row r of plane k at p[k] + (size_t)r * pitch[k].  Block (., s) loads the entry once
// -- two 16-byte loads, a third for I420's V plane -- and the slot is idle (its blocks return before they write anything) when a
// plane FMT uses is 0 or its pitch is below that plane's row bytes at the frame size H x W: a bad device-side entry cannot move an
// access past the rows it describes.
struct Planes { uint8_t* p[3]; size_t pitch[3]; };

template <int FMT>
__device__ __forceinline__ bool load_planes(const mgw_planes* __restrict__ tab, int s, int W, Planes& f)
{
    const uint4* e = reinterpret_cast<const uint4*>(tab + s);
    const uint4 a = __ldg(e), b = __ldg(e + 1);
    f.p[0] = reinterpret_cast<uint8_t*>(a.x | ((uint64_t)a.y << 32));
    f.p[1] = reinterpret_cast<uint8_t*>(a.z | ((uint64_t)a.w << 32));
    f.p[2] = reinterpret_cast<uint8_t*>(b.x | ((uint64_t)b.y << 32));
    const int q0 = (int)b.z, q1 = (int)b.w;
    f.pitch[0] = (size_t)(unsigned)q0; f.pitch[1] = (size_t)(unsigned)q1;
    if constexpr (FMT == SRC_BGR) return f.p[0] && q0 >= 3 * W;
    else if constexpr (FMT == MGW_YUV420_NV12) return f.p[0] && f.p[1] && q0 >= W && q1 >= W;
    else {
        const int q2 = (int)__ldg(e + 2).x;
        f.pitch[2] = (size_t)(unsigned)q2;
        return f.p[0] && f.p[1] && f.p[2] && q0 >= W && q1 >= (W >> 1) && q2 >= (W >> 1);
    }
}

// MIXED && PLANES: slot s's entry at the slot's size sz = sizes[s] (its width for the pitch rule), and only when the entry's own
// frame size, reserved[0] x reserved[1] (the third 16-byte word of the entry), equals sz: a slot that re-joined at another size
// while its entry still names the old surface is idle, so a stale entry cannot move an access past the surface it describes
template <int FMT>
__device__ __forceinline__ bool load_planes_at(const mgw_planes* __restrict__ tab, int s, int2 sz, Planes& f)
{
    const int4 c = __ldg(reinterpret_cast<const int4*>(tab + s) + 2);
    return c.y == sz.x && c.z == sz.y && load_planes<FMT>(tab, s, sz.y, f);
}

// yuv_chroma_at / yuv_bgr_at on pitched planes: NV12's UV rows in p[1], I420's U and V in p[1] and p[2]
template <int FMT>
__device__ __forceinline__ Chroma planes_chroma_at(const Planes& f, int row, int x)
{
    const size_t r = (size_t)(row >> 1);
    if constexpr (FMT == MGW_YUV420_NV12) {
        const uint8_t* p = f.p[1] + r * f.pitch[1] + (x & ~1);
        return yuv_chroma(__ldg(p), __ldg(p + 1));
    } else {
        const size_t c = (size_t)(x >> 1);
        return yuv_chroma(__ldg(f.p[1] + r * f.pitch[1] + c), __ldg(f.p[2] + r * f.pitch[2] + c));
    }
}

// the BGR value of pixel (row, x) of a pitched source: the bytes of a BGR row, or the pixel cvtColor makes of a YUV 4:2:0 one
template <int FMT>
__device__ __forceinline__ int3 planes_bgr_at(const Planes& f, int row, int x)
{
    if constexpr (FMT == SRC_BGR) {
        const uint8_t* p = f.p[0] + (size_t)row * f.pitch[0] + (size_t)x * 3;
        return make_int3(__ldg(p), __ldg(p + 1), __ldg(p + 2));
    } else {
        return yuv_to_bgr(__ldg(f.p[0] + (size_t)row * f.pitch[0] + x), planes_chroma_at<FMT>(f, row, x));
    }
}

// cvRound(v) as x86 does it (cvtss2si: round half to even; out of range / NaN -> INT_MIN)
__device__ __forceinline__ int cv_round(float v)
{
    return (fabsf(v) < 2147483648.0f) ? __float2int_rn(v) : (int)0x80000000;
}

// a YUV 4:2:0 source (FMT = MGW_YUV420_*, C = 3) is read as the BGR frame cvtColor makes of it: each tap is converted
template <int FMT>
__device__ __forceinline__ int3 yuv_bgr_at(const uint8_t* __restrict__ f, int H, int W, int row, int x)
{
    return yuv_to_bgr(__ldg(f + (size_t)row * W + x), yuv_chroma_at<FMT>(f, H, W, row, x));
}

// remapBilinear on 1/32-pixel fixed-point source coordinates: taps clamped to int16, 15-bit integer weights summing to 2^15,
// constant border 0 (imgwarp.cpp); shared by cv2.remap (float maps) and cv2.warpPerspective (its own fixed-point maps).
// base: one frame [H,W,C] (SRC_BGR) or [3H/2,W] (YUV 4:2:0, C = 3: every tap converted as cvtColor converts it)
template <int C, int FMT = SRC_BGR>
__device__ __forceinline__ void bilinear_fixed_u8(const uint8_t* __restrict__ base, int H, int W, int sx, int sy, uint8_t* __restrict__ o)
{
    static_assert(FMT == SRC_BGR || C == 3, "a YUV 4:2:0 source is sampled as BGR");
    const int ix = min(max(sx >> 5, -32768), 32767), iy = min(max(sy >> 5, -32768), 32767);
    const int fx = sx & 31, fy = sy & 31;
    const int w00 = (32 - fx) * (32 - fy) * 32, w01 = fx * (32 - fy) * 32, w10 = (32 - fx) * fy * 32, w11 = fx * fy * 32;
    const bool x0 = (unsigned)ix < (unsigned)W, x1 = (unsigned)(ix + 1) < (unsigned)W;
    const bool y0 = (unsigned)iy < (unsigned)H, y1 = (unsigned)(iy + 1) < (unsigned)H;
    int acc[C];
#pragma unroll
    for (int ch = 0; ch < C; ++ch) acc[ch] = 1 << 14;
    if constexpr (FMT == SRC_BGR) {
        const uint8_t* p00 = base + ((long long)iy * W + ix) * C;
        if (y0 && x0) {
#pragma unroll
            for (int ch = 0; ch < C; ++ch) acc[ch] += w00 * (int)__ldg(p00 + ch);
        }
        if (y0 && x1) {
#pragma unroll
            for (int ch = 0; ch < C; ++ch) acc[ch] += w01 * (int)__ldg(p00 + C + ch);
        }
        if (y1 && x0) {
#pragma unroll
            for (int ch = 0; ch < C; ++ch) acc[ch] += w10 * (int)__ldg(p00 + (long long)W * C + ch);
        }
        if (y1 && x1) {
#pragma unroll
            for (int ch = 0; ch < C; ++ch) acc[ch] += w11 * (int)__ldg(p00 + (long long)W * C + C + ch);
        }
    } else {
        const auto add = [&](int w, int3 p) { acc[0] += w * p.x; acc[1] += w * p.y; acc[2] += w * p.z; };
        if (y0 && x0) add(w00, yuv_bgr_at<FMT>(base, H, W, iy, ix));
        if (y0 && x1) add(w01, yuv_bgr_at<FMT>(base, H, W, iy, ix + 1));
        if (y1 && x0) add(w10, yuv_bgr_at<FMT>(base, H, W, iy + 1, ix));
        if (y1 && x1) add(w11, yuv_bgr_at<FMT>(base, H, W, iy + 1, ix + 1));
    }
#pragma unroll
    for (int ch = 0; ch < C; ++ch) o[ch] = (uint8_t)min(max(acc[ch] >> 15, 0), 255);
}

// bilinear_fixed_u8 (C = 3) on a pitched source: the same taps, weights and order; a tap's row is addressed only when it is inside
template <int FMT>
__device__ __forceinline__ void bilinear_fixed_planes(const Planes& f, int H, int W, int sx, int sy, uint8_t* __restrict__ o)
{
    const int ix = min(max(sx >> 5, -32768), 32767), iy = min(max(sy >> 5, -32768), 32767);
    const int fx = sx & 31, fy = sy & 31;
    const int w00 = (32 - fx) * (32 - fy) * 32, w01 = fx * (32 - fy) * 32, w10 = (32 - fx) * fy * 32, w11 = fx * fy * 32;
    const bool x0 = (unsigned)ix < (unsigned)W, x1 = (unsigned)(ix + 1) < (unsigned)W;
    const bool y0 = (unsigned)iy < (unsigned)H, y1 = (unsigned)(iy + 1) < (unsigned)H;
    int acc[3] = {1 << 14, 1 << 14, 1 << 14};
    const auto add = [&](int w, int3 p) { acc[0] += w * p.x; acc[1] += w * p.y; acc[2] += w * p.z; };
    if (y0 && x0) add(w00, planes_bgr_at<FMT>(f, iy, ix));
    if (y0 && x1) add(w01, planes_bgr_at<FMT>(f, iy, ix + 1));
    if (y1 && x0) add(w10, planes_bgr_at<FMT>(f, iy + 1, ix));
    if (y1 && x1) add(w11, planes_bgr_at<FMT>(f, iy + 1, ix + 1));
#pragma unroll
    for (int ch = 0; ch < 3; ++ch) o[ch] = (uint8_t)min(max(acc[ch] >> 15, 0), 255);
}

// warpRevBundle (deploy_bundle.py:148-173): output cell (i, j) = that region of cv2.warpPerspective(img, Hs_cvt[i][j],
// WARP_INVERSE_MAP | INTER_LINEAR).  OpenCV walks the destination in blocks of bw columns and evaluates, in double,
//   X0 = M0*bx + M1*y + M2 (left to right), W = W0 + M6*x1, W = W ? 32/W : 0, fX = clamp((X0 + M0*x1)*W), X = cvRound(fX)
// with bx the block's first column and x1 = x - bx; restated operation by operation (no contraction: __dmul_rn / __dadd_rn).
__device__ __forceinline__ int persp_fixed(double a, double b, double c, double bx, double y, double x1, double Wq)
{
    const double X0 = __dadd_rn(__dadd_rn(__dmul_rn(a, bx), __dmul_rn(b, y)), c);
    double f = __dmul_rn(__dadd_rn(X0, __dmul_rn(a, x1)), Wq);
    f = (f < 2147483647.0) ? f : 2147483647.0;                    // std::min((double)INT_MAX, f)
    f = (-2147483648.0 < f) ? f : -2147483648.0;                  // std::max((double)INT_MIN, f)
    return __double2int_rn(f);                                    // cvRound: round half to even
}

template <int C>
__global__ void __launch_bounds__(256)
warp_rev_bundle_kernel(const uint8_t* __restrict__ img, const double* __restrict__ Hc, int N, int H, int W, int gh, int gw, int bw,
                       uint8_t* __restrict__ dst)
{
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= N * H * W) return;
    const int x = t % W, y = (t / W) % H, n = t / (W * H);
    const int ci = min(y / (H / gh), gh - 1), cj = min(x / (W / gw), gw - 1);       // the last cell takes the remainder (:162-165)
    const double* M = Hc + ((size_t)(n * gh + ci) * gw + cj) * 9;
    const int bxi = (x / bw) * bw;
    const double bx = (double)bxi, x1 = (double)(x - bxi), yd = (double)y;
    const double W0 = __dadd_rn(__dadd_rn(__dmul_rn(__ldg(M + 6), bx), __dmul_rn(__ldg(M + 7), yd)), __ldg(M + 8));
    double Wq = __dadd_rn(W0, __dmul_rn(__ldg(M + 6), x1));
    Wq = (Wq != 0.0) ? __ddiv_rn(32.0, Wq) : 0.0;
    const int sx = persp_fixed(__ldg(M + 0), __ldg(M + 1), __ldg(M + 2), bx, yd, x1, Wq);
    const int sy = persp_fixed(__ldg(M + 3), __ldg(M + 4), __ldg(M + 5), bx, yd, x1, Wq);
    bilinear_fixed_u8<C>(img + (size_t)n * H * W * C, H, W, sx, sy, dst + (size_t)t * C);
}

// K5b: output pixel (r, c) of frame n samples the /4 maps (h4 x w4) bilinearly at the output size H x W, turns them into pixel
// coordinates of the frame and remaps the frame, which has the output's size.  Each thread takes a run of REMAP_RUN adjacent
// pixels of the frame's row-major order (a run may cross rows), so that it stores whole words: C words of 4 pixels.  The
// per-column and per-row map coefficients are the device functions of maps_down at the output size; their resize scales
// (a double division each) are launch arguments.  blockIdx.y is the frame.
// MIXED = per-slot geometry (see cvt_img2train below): H, W are the capacity, slot s's source frame of size sizes[s] lies at the
// start of its region [s * src_frame_bytes(H, W), ...) and its result at the start of [s * dst_frame_bytes(H, W), ...); block
// (., s) reads the slot's size once, computes the slot's scales (bit for bit the host's launch arguments) and then runs the
// per-pixel code of the uniform batch at the slot's size.
constexpr int REMAP_RUN = 4;

// a slot's two resize scales, computed by two threads of the block and broadcast through shared memory
__device__ __forceinline__ void slot_scales(int H, int W, int h4, int w4, double& xscale, double& yscale)
{
    __shared__ double sc[2];
    if (threadIdx.x < 2) sc[threadIdx.x] = threadIdx.x == 0 ? resize_scale(W, w4) : resize_scale(H, h4);
    __syncthreads();
    xscale = sc[0]; yscale = sc[1];
}

// pixel (c, r) of the output: its source position in 1/32 pixel from the /4 maps, as remap_up_kernel computes it
__device__ __forceinline__ int2 remap_src_fixed(const float2* __restrict__ small, int w4, const Lin& h, const Lin& v, int H, int W)
{
    const float2 m = resize_sample(small, w4, h, v);
    // (map + 1) / 2 * size in fp32 (deploy_bundle.py:142-143)
    const float xp = __fmul_rn(__fmul_rn(__fadd_rn(m.x, 1.0f), 0.5f), (float)W);
    const float yp = __fmul_rn(__fmul_rn(__fadd_rn(m.y, 1.0f), 0.5f), (float)H);
    return make_int2(cv_round(__fmul_rn(xp, 32.0f)), cv_round(__fmul_rn(yp, 32.0f)));
}

// PLANES (C = 3): the source frame and the BGR result are slot blockIdx.y's entries of the tables sp (FMT) and dp (BGR), src and dst
// unused.  A pitched row cannot be continued by the next one, so the threads are laid out over rows x ceil(W / REMAP_RUN) column
// groups, as in remap_up_yuv_kernel: each stores the 3 * REMAP_RUN bytes of its group (fewer at the row's end) as 3 words where the
// address is aligned and byte by byte otherwise.  MIXED && PLANES: H, W are the capacity; block (., s) applies the MIXED rule to
// sizes[s], loads both entries at that size (load_planes_at) and runs the PLANES code at the slot's size and scales.
template <int C, int FMT, bool MIXED = false, bool PLANES = false>
__global__ void __launch_bounds__(256)
remap_up_kernel(const uint8_t* __restrict__ src, const float2* __restrict__ small, int H, int W, int h4, int w4, double xscale,
                double yscale, uint8_t* __restrict__ dst, const int2* __restrict__ sizes, const mgw_planes* __restrict__ sp,
                const mgw_planes* __restrict__ dp)
{
    if constexpr (PLANES) {
        static_assert(C == 3, "a table's slot is a colour frame");
        Planes f, d;
        if constexpr (MIXED) {
            const int2 sz = __ldg(sizes + blockIdx.y);
            // block-uniform: before the barrier of slot_scales
            if (!slot_active<FMT>(sz, H, W) || !load_planes_at<FMT>(sp, blockIdx.y, sz, f) || !load_planes_at<SRC_BGR>(dp, blockIdx.y, sz, d))
                return;
            H = sz.x; W = sz.y;                             // launched over the capacity's rows x column groups: the rest return below
            slot_scales(H, W, h4, w4, xscale, yscale);
        } else if (!load_planes<FMT>(sp, blockIdx.y, W, f) || !load_planes<SRC_BGR>(dp, blockIdx.y, W, d)) return;
        const int gw = (W + REMAP_RUN - 1) / REMAP_RUN;
        const int t = blockIdx.x * blockDim.x + threadIdx.x;
        if (t >= H * gw) return;
        const int r = t / gw, c0 = (t - r * gw) * REMAP_RUN, ncol = min(REMAP_RUN, W - c0);
        small += (size_t)blockIdx.y * h4 * w4;
        const Lin v = vcoef_at(src_pos_s(r, yscale), h4);
        uint8_t px[REMAP_RUN * 3];
#pragma unroll
        for (int k = 0; k < REMAP_RUN; ++k) {
            // past the row's end (c0 + k >= W) the pixel is computed as any other and not stored
            const int2 q = remap_src_fixed(small, w4, hcoef_at(src_pos_s(c0 + k, xscale), w4), v, H, W);
            bilinear_fixed_planes<FMT>(f, H, W, q.x, q.y, px + k * 3);
        }
        uint8_t* o = d.p[0] + (size_t)r * d.pitch[0] + (size_t)c0 * 3;
        if (ncol == REMAP_RUN && (reinterpret_cast<uintptr_t>(o) & 3) == 0) {
#pragma unroll
            for (int q = 0; q < 3; ++q)
                reinterpret_cast<uint32_t*>(o)[q] = (uint32_t)px[4 * q] | ((uint32_t)px[4 * q + 1] << 8) | ((uint32_t)px[4 * q + 2] << 16) |
                                                    ((uint32_t)px[4 * q + 3] << 24);
        } else {
#pragma unroll
            for (int i = 0; i < REMAP_RUN * 3; ++i)
                if (i < ncol * 3) o[i] = px[i];
        }
        return;
    }
    if constexpr (MIXED) {
        static_assert(C == 3, "a slot's result is BGR");
        const int2 sz = __ldg(sizes + blockIdx.y);
        if (!slot_active<FMT>(sz, H, W)) return;            // block-uniform: before the barrier of slot_scales
        src += (size_t)blockIdx.y * src_frame_bytes<FMT>(H, W);
        small += (size_t)blockIdx.y * h4 * w4;
        dst += (size_t)blockIdx.y * H * W * 3;
        H = sz.x; W = sz.y;                                 // launched over the capacity's pixels: runs past the slot's return below
        slot_scales(H, W, h4, w4, xscale, yscale);
    }
    const int HW = H * W;
    const int p0 = (blockIdx.x * blockDim.x + threadIdx.x) * REMAP_RUN;
    if (p0 >= HW) return;
    const size_t n = MIXED ? 0 : blockIdx.y;
    const uint8_t* f = src + n * (FMT == SRC_BGR ? (size_t)HW * C : (size_t)HW * 3 / 2);
    small += n * h4 * w4;
    uint8_t* o = dst + (n * HW + p0) * C;
    int r = p0 / W, c = p0 - r * W;
    Lin v = vcoef_at(src_pos_s(r, yscale), h4);
    uint8_t px[REMAP_RUN * C];
#pragma unroll
    for (int k = 0; k < REMAP_RUN; ++k) {
        if (k > 0 && ++c == W) { c = 0; ++r; v = vcoef_at(src_pos_s(r, yscale), h4); }
        // past the frame's last pixel r = H: its map rows clamp and its taps fall outside, and nothing of it is stored
        const Lin h = hcoef_at(src_pos_s(c, xscale), w4);
        const float2 m = resize_sample(small, w4, h, v);
        // (map + 1) / 2 * size in fp32 (deploy_bundle.py:142-143)
        const float xp = __fmul_rn(__fmul_rn(__fadd_rn(m.x, 1.0f), 0.5f), (float)W);
        const float yp = __fmul_rn(__fmul_rn(__fadd_rn(m.y, 1.0f), 0.5f), (float)H);
        const int sx = cv_round(__fmul_rn(xp, 32.0f)), sy = cv_round(__fmul_rn(yp, 32.0f));
        bilinear_fixed_u8<C, FMT>(f, H, W, sx, sy, px + k * C);
    }
    if (p0 + REMAP_RUN <= HW && (reinterpret_cast<uintptr_t>(o) & 3) == 0) {
#pragma unroll
        for (int q = 0; q < C; ++q)
            reinterpret_cast<uint32_t*>(o)[q] = (uint32_t)px[4 * q] | ((uint32_t)px[4 * q + 1] << 8) | ((uint32_t)px[4 * q + 2] << 16) |
                                                ((uint32_t)px[4 * q + 3] << 24);
    } else {
        const int n_bytes = min(REMAP_RUN, HW - p0) * C;
#pragma unroll
        for (int i = 0; i < REMAP_RUN * C; ++i)
            if (i < n_bytes) o[i] = px[i];
    }
}

template <int C, int FMT>
int launch_remap_up(const uint8_t* src, const float2* small, int N, int H, int W, int h4, int w4, uint8_t* dst, cudaStream_t st)
{
    const unsigned gx = (unsigned)((((long long)H * W + REMAP_RUN - 1) / REMAP_RUN + 255) / 256);
    const double xscale = resize_scale(W, w4), yscale = resize_scale(H, h4);
    // the frame index is gridDim.y: a batch of more than 65535 frames (mgw_remap_bundle_u8 allows it) takes several launches
    for (int n0 = 0; n0 < N; n0 += 65535) {
        const int n = min(N - n0, 65535);
        remap_up_kernel<C, FMT><<<dim3(gx, n), 256, 0, st>>>(src + (size_t)n0 * (FMT == SRC_BGR ? (size_t)H * W * C : (size_t)H * W * 3 / 2),
                                                             small + (size_t)n0 * h4 * w4, H, W, h4, w4, xscale, yscale,
                                                             dst + (size_t)n0 * H * W * C, nullptr, nullptr, nullptr);
        if (int rc = check_launch("remap_up")) return rc;
    }
    return MGW_OK;
}

// cv2.cvtColor(COLOR_BGR2YUV_I420), color_yuv.simd.hpp: BT.601 limited range in 20-bit fixed point.  Y of every pixel; U and V
// of the top-left pixel of each 2x2 block only (no averaging).  Every sum lies in [16 << 20, 241 << 20): no clamp is needed.
__device__ __forceinline__ int bgr_y(const uint8_t* p)
{
    return (269484 * p[2] + 528482 * p[1] + 102760 * p[0] + (16 << 20) + (1 << 19)) >> 20;
}
__device__ __forceinline__ int bgr_u(const uint8_t* p)
{
    return (-155188 * p[2] - 305135 * p[1] + 460324 * p[0] + (128 << 20) + (1 << 19)) >> 20;
}
__device__ __forceinline__ int bgr_v(const uint8_t* p)
{
    return (460324 * p[2] - 385875 * p[1] - 74448 * p[0] + (128 << 20) + (1 << 19)) >> 20;
}

// n (2 or 4) bytes b[0..n) to o: one word (or half word) where o is aligned, single bytes otherwise
__device__ __forceinline__ void store_run(uint8_t* o, const uint8_t* b, int n)
{
    const uintptr_t a = reinterpret_cast<uintptr_t>(o);
    if (n == 4 && (a & 3) == 0)
        *reinterpret_cast<uint32_t*>(o) = (uint32_t)b[0] | ((uint32_t)b[1] << 8) | ((uint32_t)b[2] << 16) | ((uint32_t)b[3] << 24);
    else if (n == 2 && (a & 1) == 0)
        *reinterpret_cast<uint16_t*>(o) = (uint16_t)(b[0] | (b[1] << 8));
    else {
#pragma unroll
        for (int i = 0; i < 4; ++i)
            if (i < n) o[i] = b[i];
    }
}

// K5b with the result as YUV 4:2:0 (DST_FMT = MGW_YUV420_NV12 / _I420, [3H/2,W] per frame; H and W even): each thread takes a
// block of 2 rows x YUV_RUN columns of the output, the columns starting at a multiple of YUV_RUN inside one row pair (when W is
// not a multiple of 4 the last block of a row is 2 columns wide).  Every pixel's BGR value is remap_up_kernel's, by the same
// device functions; the column coefficients are shared by the two rows.  The thread writes the block's Y bytes and the U, V of
// its two (or one) 2x2 chroma blocks, so the BGR frame never reaches memory.  MIXED: as remap_up_kernel, with a YUV result region
// of 3H/2*W bytes per slot; a slot of odd size is idle.  PLANES: the source and the result are slot blockIdx.y's entries of the
// tables sp (SRC_FMT) and dp (DST_FMT), src and dst unused; the same threads and arithmetic, pitched loads and stores.  MIXED &&
// PLANES: the MIXED rule on sizes[s], both entries loaded at that size (load_planes_at), then the PLANES code at the slot's size.
constexpr int YUV_RUN = 4;

template <int SRC_FMT, int DST_FMT, bool MIXED = false, bool PLANES = false>
__global__ void __launch_bounds__(256)
remap_up_yuv_kernel(const uint8_t* __restrict__ src, const float2* __restrict__ small, int H, int W, int h4, int w4, double xscale,
                    double yscale, uint8_t* __restrict__ dst, const int2* __restrict__ sizes, const mgw_planes* __restrict__ sp,
                    const mgw_planes* __restrict__ dp)
{
    [[maybe_unused]] Planes sf, df;
    if constexpr (PLANES) {
        if constexpr (MIXED) {
            const int2 sz = __ldg(sizes + blockIdx.y);
            if (!slot_active<SRC_FMT>(sz, H, W) || !slot_active<DST_FMT>(sz, H, W) || !load_planes_at<SRC_FMT>(sp, blockIdx.y, sz, sf) ||
                !load_planes_at<DST_FMT>(dp, blockIdx.y, sz, df))
                return;                                     // block-uniform: before the barrier of slot_scales
            H = sz.x; W = sz.y;
            slot_scales(H, W, h4, w4, xscale, yscale);
        } else if (!load_planes<SRC_FMT>(sp, blockIdx.y, W, sf) || !load_planes<DST_FMT>(dp, blockIdx.y, W, df)) return;
        small += (size_t)blockIdx.y * h4 * w4;
    } else if constexpr (MIXED) {
        const int2 sz = __ldg(sizes + blockIdx.y);
        // the result is 4:2:0, so every active slot is even (DST_FMT's rule covers an odd size from a BGR source)
        if (!slot_active<SRC_FMT>(sz, H, W) || !slot_active<DST_FMT>(sz, H, W)) return;
        src += (size_t)blockIdx.y * src_frame_bytes<SRC_FMT>(H, W);
        small += (size_t)blockIdx.y * h4 * w4;
        dst += (size_t)blockIdx.y * H * W * 3 / 2;
        H = sz.x; W = sz.y;                                 // launched over the capacity's row pairs: blocks past the slot's return below
        slot_scales(H, W, h4, w4, xscale, yscale);
    }
    const int gw = (W + YUV_RUN - 1) / YUV_RUN;
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= (H >> 1) * gw) return;
    const int r = (t / gw) * 2, c0 = (t % gw) * YUV_RUN;
    const int ncol = min(YUV_RUN, W - c0);
    const size_t n = (MIXED || PLANES) ? 0 : blockIdx.y;
    const uint8_t* f = src + n * src_frame_bytes<SRC_FMT>(H, W);
    small += n * h4 * w4;
    uint8_t* y = dst + n * ((size_t)H * W * 3 / 2);
    uint8_t* uv = y + (size_t)H * W;
    const Lin v0 = vcoef_at(src_pos_s(r, yscale), h4), v1 = vcoef_at(src_pos_s(r + 1, yscale), h4);
    uint8_t ys[2][YUV_RUN], us[YUV_RUN / 2], vs[YUV_RUN / 2];
#pragma unroll
    for (int k = 0; k < YUV_RUN; ++k) {
        // past the row's end (c0 + k >= W) the taps are computed as for any column and nothing of them is stored
        const Lin hc = hcoef_at(src_pos_s(c0 + k, xscale), w4);
#pragma unroll
        for (int i = 0; i < 2; ++i) {
            const float2 m = resize_sample(small, w4, hc, i ? v1 : v0);
            // (map + 1) / 2 * size in fp32 (deploy_bundle.py:142-143)
            const float xp = __fmul_rn(__fmul_rn(__fadd_rn(m.x, 1.0f), 0.5f), (float)W);
            const float yp = __fmul_rn(__fmul_rn(__fadd_rn(m.y, 1.0f), 0.5f), (float)H);
            const int sx = cv_round(__fmul_rn(xp, 32.0f)), sy = cv_round(__fmul_rn(yp, 32.0f));
            uint8_t px[3];
            if constexpr (PLANES) bilinear_fixed_planes<SRC_FMT>(sf, H, W, sx, sy, px);
            else bilinear_fixed_u8<3, SRC_FMT>(f, H, W, sx, sy, px);
            ys[i][k] = (uint8_t)bgr_y(px);
            if (i == 0 && (k & 1) == 0) { us[k >> 1] = (uint8_t)bgr_u(px); vs[k >> 1] = (uint8_t)bgr_v(px); }
        }
    }
    if constexpr (PLANES) {
        store_run(df.p[0] + (size_t)r * df.pitch[0] + c0, ys[0], ncol);
        store_run(df.p[0] + (size_t)(r + 1) * df.pitch[0] + c0, ys[1], ncol);
        const size_t cr = (size_t)(r >> 1);
        if constexpr (DST_FMT == MGW_YUV420_NV12) {
            const uint8_t b[YUV_RUN] = {us[0], vs[0], us[1], vs[1]};
            store_run(df.p[1] + cr * df.pitch[1] + c0, b, ncol);
        } else {
            store_run(df.p[1] + cr * df.pitch[1] + (c0 >> 1), us, ncol >> 1);
            store_run(df.p[2] + cr * df.pitch[2] + (c0 >> 1), vs, ncol >> 1);
        }
        return;
    }
    store_run(y + (size_t)r * W + c0, ys[0], ncol);
    store_run(y + (size_t)(r + 1) * W + c0, ys[1], ncol);
    if constexpr (DST_FMT == MGW_YUV420_NV12) {
        const uint8_t b[YUV_RUN] = {us[0], vs[0], us[1], vs[1]};
        store_run(uv + (size_t)(r >> 1) * W + c0, b, ncol);
    } else {
        const size_t q = (size_t)(r >> 1) * (W >> 1) + (c0 >> 1);
        store_run(uv + q, us, ncol >> 1);
        store_run(uv + (size_t)(H >> 1) * (W >> 1) + q, vs, ncol >> 1);
    }
}

template <int SRC_FMT, int DST_FMT>
int launch_remap_up_yuv(const uint8_t* src, const float2* small, int N, int H, int W, int h4, int w4, uint8_t* dst, cudaStream_t st)
{
    const long long threads = (long long)(H / 2) * ((W + YUV_RUN - 1) / YUV_RUN);
    remap_up_yuv_kernel<SRC_FMT, DST_FMT><<<dim3((unsigned)((threads + 255) / 256), N), 256, 0, st>>>(
        src, small, H, W, h4, w4, resize_scale(W, w4), resize_scale(H, h4), dst, nullptr, nullptr, nullptr);
    return check_launch("remap_up_yuv");
}

// K5b over a pool of per-slot frames: the grid covers the capacity (max_h, max_w), gridDim.y is the slot
template <int SRC_FMT>
int launch_remap_up_mixed(int dst_fmt, const uint8_t* src, const float2* small, int S, int max_h, int max_w, int h4, int w4,
                          const int2* sizes, uint8_t* dst, cudaStream_t st)
{
    if (dst_fmt == SRC_BGR) {
        const unsigned gx = (unsigned)((((long long)max_h * max_w + REMAP_RUN - 1) / REMAP_RUN + 255) / 256);
        remap_up_kernel<3, SRC_FMT, true><<<dim3(gx, S), 256, 0, st>>>(src, small, max_h, max_w, h4, w4, 0.0, 0.0, dst, sizes, nullptr,
                                                                       nullptr);
        return check_launch("remap_up");
    }
    const long long threads = (long long)(max_h / 2) * ((max_w + YUV_RUN - 1) / YUV_RUN);
    const dim3 grid((unsigned)((threads + 255) / 256), S);
    switch (dst_fmt) {
    case MGW_YUV420_NV12:
        remap_up_yuv_kernel<SRC_FMT, MGW_YUV420_NV12, true><<<grid, 256, 0, st>>>(src, small, max_h, max_w, h4, w4, 0.0, 0.0, dst, sizes,
                                                                                  nullptr, nullptr);
        break;
    case MGW_YUV420_I420:
        remap_up_yuv_kernel<SRC_FMT, MGW_YUV420_I420, true><<<grid, 256, 0, st>>>(src, small, max_h, max_w, h4, w4, 0.0, 0.0, dst, sizes,
                                                                                  nullptr, nullptr);
        break;
    default: return set_error(MGW_ERR_INVALID, "remap_bundle_frame_mixed: unknown destination format %d", dst_fmt);
    }
    return check_launch("remap_up_yuv");
}

// K5b between two tables of planes (S slots of one size H x W): BGR results over rows x column groups, YUV ones over row pairs
template <int SRC_FMT>
int launch_remap_up_planes(int dst_fmt, const mgw_planes* sp, const float2* small, int S, int H, int W, int h4, int w4,
                           const mgw_planes* dp, cudaStream_t st)
{
    const double xscale = resize_scale(W, w4), yscale = resize_scale(H, h4);
    const long long groups = (W + REMAP_RUN - 1) / REMAP_RUN;
    if (dst_fmt == SRC_BGR) {
        const dim3 grid((unsigned)(((long long)H * groups + 255) / 256), S);
        remap_up_kernel<3, SRC_FMT, false, true><<<grid, 256, 0, st>>>(nullptr, small, H, W, h4, w4, xscale, yscale, nullptr, nullptr, sp, dp);
        return check_launch("remap_up");
    }
    const dim3 grid((unsigned)(((long long)(H / 2) * ((W + YUV_RUN - 1) / YUV_RUN) + 255) / 256), S);
    switch (dst_fmt) {
    case MGW_YUV420_NV12:
        remap_up_yuv_kernel<SRC_FMT, MGW_YUV420_NV12, false, true><<<grid, 256, 0, st>>>(nullptr, small, H, W, h4, w4, xscale, yscale, nullptr,
                                                                                         nullptr, sp, dp);
        break;
    case MGW_YUV420_I420:
        remap_up_yuv_kernel<SRC_FMT, MGW_YUV420_I420, false, true><<<grid, 256, 0, st>>>(nullptr, small, H, W, h4, w4, xscale, yscale, nullptr,
                                                                                         nullptr, sp, dp);
        break;
    default: return set_error(MGW_ERR_INVALID, "remap_bundle_frame_planes: unknown destination format %d", dst_fmt);
    }
    return check_launch("remap_up_yuv");
}

// K5b of a batch of per-slot sizes between two tables of planes: the grid covers the capacity, gridDim.y is the slot
template <int SRC_FMT>
int launch_remap_up_mixed_planes(int dst_fmt, const mgw_planes* sp, const float2* small, int S, int max_h, int max_w, int h4, int w4,
                                 const int2* sizes, const mgw_planes* dp, cudaStream_t st)
{
    if (dst_fmt == SRC_BGR) {
        const long long groups = (max_w + REMAP_RUN - 1) / REMAP_RUN;
        const dim3 grid((unsigned)(((long long)max_h * groups + 255) / 256), S);
        remap_up_kernel<3, SRC_FMT, true, true><<<grid, 256, 0, st>>>(nullptr, small, max_h, max_w, h4, w4, 0.0, 0.0, nullptr, sizes, sp, dp);
        return check_launch("remap_up");
    }
    const dim3 grid((unsigned)(((long long)(max_h / 2) * ((max_w + YUV_RUN - 1) / YUV_RUN) + 255) / 256), S);
    switch (dst_fmt) {
    case MGW_YUV420_NV12:
        remap_up_yuv_kernel<SRC_FMT, MGW_YUV420_NV12, true, true><<<grid, 256, 0, st>>>(nullptr, small, max_h, max_w, h4, w4, 0.0, 0.0,
                                                                                        nullptr, sizes, sp, dp);
        break;
    case MGW_YUV420_I420:
        remap_up_yuv_kernel<SRC_FMT, MGW_YUV420_I420, true, true><<<grid, 256, 0, st>>>(nullptr, small, max_h, max_w, h4, w4, 0.0, 0.0,
                                                                                        nullptr, sizes, sp, dp);
        break;
    default: return set_error(MGW_ERR_INVALID, "remap_bundle_frame_mixed_planes: unknown destination format %d", dst_fmt);
    }
    return check_launch("remap_up_yuv");
}

template <int SRC_FMT>
int launch_remap_up_yuv_to(int dst_fmt, const uint8_t* src, const float2* small, int N, int H, int W, int h4, int w4, uint8_t* dst,
                           cudaStream_t st)
{
    switch (dst_fmt) {
    case MGW_YUV420_NV12: return launch_remap_up_yuv<SRC_FMT, MGW_YUV420_NV12>(src, small, N, H, W, h4, w4, dst, st);
    case MGW_YUV420_I420: return launch_remap_up_yuv<SRC_FMT, MGW_YUV420_I420>(src, small, N, H, W, h4, w4, dst, st);
    default: return set_error(MGW_ERR_INVALID, "remap_bundle_yuv420: unknown destination format %d", dst_fmt);
    }
}

// K5a: the /4 maps of every frame (h4 = int(height / rate), w4 = int(width / rate)) into the workspace
float2* launch_maps_down(const float* xy, int N, int h, int w, void* workspace, cudaStream_t st)
{
    float2* small = reinterpret_cast<float2*>(workspace);
    const int h4 = h / 4, w4 = w / 4, t1 = N * h4 * w4;
    maps_down_kernel<<<(t1 + 255) / 256, 256, 0, st>>>(reinterpret_cast<const float2*>(xy), N, h, w, h4, w4, small);
    return small;
}

}  // namespace

size_t remap_bundle_workspace_bytes(int N, int H, int W) { return sizeof(float) * 2 * (size_t)N * (H / 4) * (W / 4); }

// K5a at the maps' size h x w, then K5b at the output size H x W; the frame src has the output's size
int launch_remap_bundle(const uint8_t* src, int src_fmt, int C, const float* xy, int N, int h, int w, int H, int W, uint8_t* dst,
                        void* workspace, cudaStream_t st)
{
    const int h4 = h / 4, w4 = w / 4;
    float2* small = launch_maps_down(xy, N, h, w, workspace, st);
    if (int rc = check_launch("maps_down")) return rc;
    if (src_fmt != SRC_BGR && C != 3) return set_error(MGW_ERR_UNSUPPORTED, "remap_bundle: a YUV 4:2:0 source gives C = 3 (got %d)", C);
    switch (src_fmt) {
    case SRC_BGR:
        switch (C) {
        case 1: return launch_remap_up<1, SRC_BGR>(src, small, N, H, W, h4, w4, dst, st);
        case 3: return launch_remap_up<3, SRC_BGR>(src, small, N, H, W, h4, w4, dst, st);
        case 4: return launch_remap_up<4, SRC_BGR>(src, small, N, H, W, h4, w4, dst, st);
        default: return set_error(MGW_ERR_UNSUPPORTED, "remap_bundle_u8: C must be 1, 3 or 4 (got %d)", C);
        }
    case MGW_YUV420_NV12: return launch_remap_up<3, MGW_YUV420_NV12>(src, small, N, H, W, h4, w4, dst, st);
    case MGW_YUV420_I420: return launch_remap_up<3, MGW_YUV420_I420>(src, small, N, H, W, h4, w4, dst, st);
    default: return set_error(MGW_ERR_INVALID, "remap_bundle: unknown source format %d", src_fmt);
    }
}

int launch_remap_bundle_u8(const uint8_t* img, const float* xy, int N, int H, int W, int C, uint8_t* dst, void* workspace,
                           cudaStream_t st)
{
    return launch_remap_bundle(img, SRC_BGR, C, xy, N, H, W, H, W, dst, workspace, st);
}

// launch_remap_bundle's warp (C = 3) with the result written as YUV 4:2:0: the same K5a, then the YUV variant of K5b
int launch_remap_bundle_yuv420(const uint8_t* src, int src_fmt, const float* xy, int N, int h, int w, int H, int W, int dst_fmt,
                               uint8_t* dst, void* workspace, cudaStream_t st)
{
    const int h4 = h / 4, w4 = w / 4;
    float2* small = launch_maps_down(xy, N, h, w, workspace, st);
    if (int rc = check_launch("maps_down")) return rc;
    switch (src_fmt) {
    case SRC_BGR: return launch_remap_up_yuv_to<SRC_BGR>(dst_fmt, src, small, N, H, W, h4, w4, dst, st);
    case MGW_YUV420_NV12: return launch_remap_up_yuv_to<MGW_YUV420_NV12>(dst_fmt, src, small, N, H, W, h4, w4, dst, st);
    case MGW_YUV420_I420: return launch_remap_up_yuv_to<MGW_YUV420_I420>(dst_fmt, src, small, N, H, W, h4, w4, dst, st);
    default: return set_error(MGW_ERR_INVALID, "remap_bundle_yuv420: unknown source format %d", src_fmt);
    }
}

// the same K5a, then K5b per slot at the slot's own size: src / dst are pools of capacity-sized regions, sizes [S,2]
int launch_remap_bundle_mixed(const uint8_t* src, int src_fmt, int S, int max_h, int max_w, const int32_t* sizes, const float* xy,
                              int h, int w, int dst_fmt, uint8_t* dst, void* workspace, cudaStream_t st)
{
    const int h4 = h / 4, w4 = w / 4;
    float2* small = launch_maps_down(xy, S, h, w, workspace, st);
    if (int rc = check_launch("maps_down")) return rc;
    const int2* sz = reinterpret_cast<const int2*>(sizes);
    switch (src_fmt) {
    case SRC_BGR: return launch_remap_up_mixed<SRC_BGR>(dst_fmt, src, small, S, max_h, max_w, h4, w4, sz, dst, st);
    case MGW_YUV420_NV12: return launch_remap_up_mixed<MGW_YUV420_NV12>(dst_fmt, src, small, S, max_h, max_w, h4, w4, sz, dst, st);
    case MGW_YUV420_I420: return launch_remap_up_mixed<MGW_YUV420_I420>(dst_fmt, src, small, S, max_h, max_w, h4, w4, sz, dst, st);
    default: return set_error(MGW_ERR_INVALID, "remap_bundle_frame_mixed: unknown source format %d", src_fmt);
    }
}

// the same K5a, then K5b from the source table's planes into the destination table's
int launch_remap_bundle_planes(const mgw_planes* src, int src_fmt, const float* xy, int S, int h, int w, int H, int W,
                               const mgw_planes* dst, int dst_fmt, void* workspace, cudaStream_t st)
{
    const int h4 = h / 4, w4 = w / 4;
    float2* small = launch_maps_down(xy, S, h, w, workspace, st);
    if (int rc = check_launch("maps_down")) return rc;
    switch (src_fmt) {
    case SRC_BGR: return launch_remap_up_planes<SRC_BGR>(dst_fmt, src, small, S, H, W, h4, w4, dst, st);
    case MGW_YUV420_NV12: return launch_remap_up_planes<MGW_YUV420_NV12>(dst_fmt, src, small, S, H, W, h4, w4, dst, st);
    case MGW_YUV420_I420: return launch_remap_up_planes<MGW_YUV420_I420>(dst_fmt, src, small, S, H, W, h4, w4, dst, st);
    default: return set_error(MGW_ERR_INVALID, "remap_bundle_frame_planes: unknown source format %d", src_fmt);
    }
}

// the same K5a, then K5b per slot at the slot's own size from the source table's planes into the destination table's
int launch_remap_bundle_mixed_planes(const mgw_planes* src, int src_fmt, int S, int max_h, int max_w, const int32_t* sizes,
                                     const float* xy, int h, int w, const mgw_planes* dst, int dst_fmt, void* workspace, cudaStream_t st)
{
    const int h4 = h / 4, w4 = w / 4;
    float2* small = launch_maps_down(xy, S, h, w, workspace, st);
    if (int rc = check_launch("maps_down")) return rc;
    const int2* sz = reinterpret_cast<const int2*>(sizes);
    switch (src_fmt) {
    case SRC_BGR: return launch_remap_up_mixed_planes<SRC_BGR>(dst_fmt, src, small, S, max_h, max_w, h4, w4, sz, dst, st);
    case MGW_YUV420_NV12: return launch_remap_up_mixed_planes<MGW_YUV420_NV12>(dst_fmt, src, small, S, max_h, max_w, h4, w4, sz, dst, st);
    case MGW_YUV420_I420: return launch_remap_up_mixed_planes<MGW_YUV420_I420>(dst_fmt, src, small, S, max_h, max_w, h4, w4, sz, dst, st);
    default: return set_error(MGW_ERR_INVALID, "remap_bundle_frame_mixed_planes: unknown source format %d", src_fmt);
    }
}

// ---------------------------------------------------------------------------------------------------------------------
// Exact-bytes transfer of a pool of per-slot frames (MIXED): slot s's frame_bytes(sizes[s]) bytes from src + s * stride to
// dst + s * stride, stride = frame_bytes(max_h, max_w); nothing past them is read or written, and an idle slot (the MIXED rule)
// moves nothing.  Either side may be pinned host memory reached through its mapped device address, so the kernel is the
// upload, the download or a device copy; a copy-engine node of a captured graph has a fixed size, this kernel reads the sizes
// at replay.  src and dst are 16-byte aligned, so both sides of a slot share the misalignment of s * stride: a head of under
// 16 bytes up to the boundary, the body in 16-byte vectors (COPY_UNROLL independent loads in flight per thread, to cover
// the round trip of a read across PCIe), a tail of under 16 bytes.  gridDim.y is the slot, gridDim.x blocks share its body.
namespace {

constexpr int COPY_THREADS = 256, COPY_UNROLL = 4;

// FMT = SRC_BGR or MGW_YUV420_NV12 (I420 has NV12's bytes per frame and idle rule)
template <int FMT>
__global__ void __launch_bounds__(COPY_THREADS)
copy_slots_kernel(const uint8_t* __restrict__ src, uint8_t* __restrict__ dst, int max_h, int max_w, const int2* __restrict__ sizes)
{
    const int2 sz = __ldg(sizes + blockIdx.y);
    if (!slot_active<FMT>(sz, max_h, max_w)) return;
    const size_t off = (size_t)blockIdx.y * src_frame_bytes<FMT>(max_h, max_w);
    src += off;
    dst += off;
    const int n = (int)src_frame_bytes<FMT>(sz.x, sz.y);                  // < 2^31: the call checks S * stride
    const int head = min((int)((16 - (off & 15)) & 15), n);
    const int n16 = (n - head) >> 4, tail = head + (n16 << 4);
    const int t = blockIdx.x * COPY_THREADS + threadIdx.x, nt = gridDim.x * COPY_THREADS;
    if (t < head) dst[t] = __ldcs(src + t);
    if (t < n - tail) dst[tail + t] = __ldcs(src + tail + t);
    const uint4* s4 = reinterpret_cast<const uint4*>(src + head);
    uint4* d4 = reinterpret_cast<uint4*>(dst + head);
    int i = t;
    for (; i + (COPY_UNROLL - 1) * nt < n16; i += COPY_UNROLL * nt) {
        uint4 v[COPY_UNROLL];
#pragma unroll
        for (int k = 0; k < COPY_UNROLL; ++k) v[k] = __ldcs(s4 + i + k * nt);
#pragma unroll
        for (int k = 0; k < COPY_UNROLL; ++k) __stcs(d4 + i + k * nt, v[k]);
    }
    for (; i < n16; i += nt) __stcs(d4 + i, __ldcs(s4 + i));
}

}  // namespace

// gridDim.x: COPY_BLOCKS_PER_SM blocks per SM spread over the slots, no more than one pass over a full slot needs
int launch_copy_slots_mixed(const uint8_t* src, uint8_t* dst, int fmt, int S, int max_h, int max_w, const int32_t* sizes, cudaStream_t st)
{
    constexpr long long COPY_BLOCKS_PER_SM = 8;
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    const long long stride = fmt == SRC_BGR ? 3LL * max_h * max_w : 3LL * max_h * max_w / 2;
    const long long pass = (long long)COPY_THREADS * COPY_UNROLL * 16;
    const long long full = (stride + pass - 1) / pass, spread = (sms * COPY_BLOCKS_PER_SM + S - 1) / S;
    const dim3 grid((unsigned)(full < spread ? full : spread), S);
    const int2* sz = reinterpret_cast<const int2*>(sizes);
    switch (fmt) {
    case SRC_BGR: copy_slots_kernel<SRC_BGR><<<grid, COPY_THREADS, 0, st>>>(src, dst, max_h, max_w, sz); break;
    case MGW_YUV420_NV12:
    case MGW_YUV420_I420: copy_slots_kernel<MGW_YUV420_NV12><<<grid, COPY_THREADS, 0, st>>>(src, dst, max_h, max_w, sz); break;
    default: return set_error(MGW_ERR_INVALID, "copy_slots_mixed: unknown format %d", fmt);
    }
    return check_launch("copy_slots");
}

// ---------------------------------------------------------------------------------------------------------------------
// cvt_img2train (config.py:6-21): BGR uint8 frame -> cv2 BGR2GRAY -> Pillow resize(BILINEAR) [-> crop] -> v*(1/255) - 0.5.
// The host binding computes Pillow's 22-bit fixed-point coefficient tables (double arithmetic, Resample.c) once per shape
// and slices them for the crop; the two passes below are Pillow's: horizontal first into a uint8 image, then vertical.
// A batch of S frames of one size shares the tables; blockIdx.y is the frame (the stream index of a StreamBatch): each block
// offsets its base pointers once, the per-pixel index arithmetic is the single-frame one, and S = 1 is the single-frame call.
// The source frame is BGR (SRC_BGR) or YUV 4:2:0 in OpenCV's layout (MGW_YUV420_NV12 / MGW_YUV420_I420): the kernels then read
// the BGR frame cv2.cvtColor would make of it, converted per pixel on the fly.
// MIXED = per-slot source geometry (a batch of videos of different sizes): H, W are the batch's capacity, slot s owns the region
// [s * frame_bytes(H, W), +frame_bytes(H, W)) of the source and its frame of size sizes[s] lies at the start of it, and the slot
// has its own tables (kx [S,out_w,ks], ...) and tmp rows [S,H,out_w].  Block (., s) reads sizes[s] once, offsets its pointers to
// the slot, and then runs the per-pixel code of the uniform batch at the slot's size with frame index 0.
// PLANES = per-slot planes (a uniform batch whose frames lie wherever a decoder put them): slot s's source is entry s of the table
// `planes` (see load_planes), bgr is unused; the tables, tmp and out are the uniform batch's, and an idle slot writes no row of either.
// MIXED && PLANES: the MIXED slot (its size, tables and tmp / out rows at the capacity) read from its entry (load_planes_at).
namespace {

template <int FMT, bool MIXED = false, bool PLANES = false>
__global__ void __launch_bounds__(256)
gray_hpass_kernel(const uint8_t* __restrict__ bgr, int H, int W, const int32_t* __restrict__ kx, const int32_t* __restrict__ x0,
                  const int32_t* __restrict__ xn, int ks, int out_w, uint8_t* __restrict__ tmp, const int2* __restrict__ sizes,
                  const mgw_planes* __restrict__ planes)
{
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if constexpr (PLANES) {
        Planes f;
        if constexpr (MIXED) {
            const int2 sz = __ldg(sizes + blockIdx.y);
            if (!slot_active<FMT>(sz, H, W) || !load_planes_at<FMT>(planes, blockIdx.y, sz, f)) return;
            tmp += (size_t)blockIdx.y * H * out_w;          // the slot's tmp rows, laid out at the capacity
            kx += (size_t)blockIdx.y * out_w * ks;
            x0 += (size_t)blockIdx.y * out_w;
            xn += (size_t)blockIdx.y * out_w;
            H = sz.x;
        } else if (!load_planes<FMT>(planes, blockIdx.y, W, f)) return;
        if (t >= H * out_w) return;
        if constexpr (!MIXED) tmp += (size_t)blockIdx.y * H * out_w;
        const int xx = t % out_w, row = t / out_w;
        const int n = __ldg(xn + xx), xs = __ldg(x0 + xx);
        int acc = 1 << 21;
        if constexpr (FMT == SRC_BGR) {
            const uint8_t* p = f.p[0] + (size_t)row * f.pitch[0] + (size_t)xs * 3;
            for (int k = 0; k < n; ++k, p += 3) {
                const int g = ((int)__ldg(p) * 3735 + (int)__ldg(p + 1) * 19235 + (int)__ldg(p + 2) * 9798 + (1 << 14)) >> 15;
                acc += g * __ldg(kx + (size_t)xx * ks + k);
            }
        } else {
            const uint8_t* py = f.p[0] + (size_t)row * f.pitch[0] + xs;
            Chroma c;
#pragma unroll 1
            for (int k = 0; k < n; ++k) {
                if (k == 0 || ((xs + k) & 1) == 0) c = planes_chroma_at<FMT>(f, row, xs + k);
                const int3 p = yuv_to_bgr(__ldg(py + k), c);
                const int g = (p.x * 3735 + p.y * 19235 + p.z * 9798 + (1 << 14)) >> 15;
                acc += g * __ldg(kx + (size_t)xx * ks + k);
            }
        }
        tmp[t] = (uint8_t)min(max(acc >> 22, 0), 255);
        return;
    }
    if constexpr (MIXED) {
        const int2 sz = __ldg(sizes + blockIdx.y);
        if (!slot_active<FMT>(sz, H, W)) return;
        bgr += (size_t)blockIdx.y * src_frame_bytes<FMT>(H, W);
        tmp += (size_t)blockIdx.y * H * out_w;
        kx += (size_t)blockIdx.y * out_w * ks;
        x0 += (size_t)blockIdx.y * out_w;
        xn += (size_t)blockIdx.y * out_w;
        H = sz.x; W = sz.y;                                 // launched over the capacity's rows: rows >= H return below
    }
    const unsigned s = MIXED ? 0u : blockIdx.y;             // the frame index of a uniform batch
    if (t >= H * out_w) return;
    tmp += (size_t)s * H * out_w;
    const int xx = t % out_w, row = t / out_w;
    const int n = __ldg(xn + xx);
    int acc = 1 << 21;
    if constexpr (FMT == SRC_BGR) {
        bgr += (size_t)s * H * W * 3;
        const uint8_t* p = bgr + ((size_t)row * W + __ldg(x0 + xx)) * 3;
        for (int k = 0; k < n; ++k, p += 3) {
            // RGB2Gray<uchar>: (B*3735 + G*19235 + R*9798 + 2^14) >> 15
            const int g = ((int)__ldg(p) * 3735 + (int)__ldg(p + 1) * 19235 + (int)__ldg(p + 2) * 9798 + (1 << 14)) >> 15;
            acc += g * __ldg(kx + (size_t)xx * ks + k);
        }
    } else {
        // the BGR pixel cvtColor makes, then the same gray; a pair of pixels (even x, x+1) shares one chroma sample
        const uint8_t* f = bgr + (size_t)s * src_frame_bytes<FMT>(H, W);
        const int xs = __ldg(x0 + xx);
        const uint8_t* py = f + (size_t)row * W + xs;
        Chroma c;
#pragma unroll 1        // unrolled, the NV12 loop spills at 40 registers; rolled, both formats take 32 and none
        for (int k = 0; k < n; ++k) {
            if (k == 0 || ((xs + k) & 1) == 0) c = yuv_chroma_at<FMT>(f, H, W, row, xs + k);
            const int3 p = yuv_to_bgr(__ldg(py + k), c);
            const int g = (p.x * 3735 + p.y * 19235 + p.z * 9798 + (1 << 14)) >> 15;
            acc += g * __ldg(kx + (size_t)xx * ks + k);
        }
    }
    tmp[t] = (uint8_t)min(max(acc >> 22, 0), 255);
}

// MIXED: H is the capacity's height (the tmp rows of a slot), max_w its width; the slot's rows of ky / y0 / yn
// PLANES: max_w is the source width; a slot that gray_hpass found idle is skipped by the same rule (MIXED && PLANES: at the slot's size)
template <int FMT = SRC_BGR, bool MIXED = false, bool PLANES = false>
__global__ void __launch_bounds__(256)
vpass_norm_kernel(const uint8_t* __restrict__ tmp, int H, int out_w, const int32_t* __restrict__ ky, const int32_t* __restrict__ y0,
                  const int32_t* __restrict__ yn, int ks, int out_h, float* __restrict__ out, const int2* __restrict__ sizes, int max_w,
                  const mgw_planes* __restrict__ planes)
{
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if constexpr (PLANES) {
        Planes f;
        if constexpr (MIXED) {
            const int2 sz = __ldg(sizes + blockIdx.y);
            if (!slot_active<FMT>(sz, H, max_w) || !load_planes_at<FMT>(planes, blockIdx.y, sz, f)) return;
        } else if (!load_planes<FMT>(planes, blockIdx.y, max_w, f)) return;
    }
    if constexpr (MIXED) {
        if (!PLANES && !slot_active<FMT>(__ldg(sizes + blockIdx.y), H, max_w)) return;
        ky += (size_t)blockIdx.y * out_h * ks;
        y0 += (size_t)blockIdx.y * out_h;
        yn += (size_t)blockIdx.y * out_h;
    }
    if (t >= out_h * out_w) return;
    tmp += (size_t)blockIdx.y * H * out_w;
    out += (size_t)blockIdx.y * out_h * out_w;
    const int xx = t % out_w, yy = t / out_w;
    const uint8_t* p = tmp + (size_t)__ldg(y0 + yy) * out_w + xx;
    const int n = __ldg(yn + yy);
    int acc = 1 << 21;
    for (int k = 0; k < n; ++k, p += out_w) acc += (int)__ldg(p) * __ldg(ky + (size_t)yy * ks + k);
    const int v = min(max(acc >> 22, 0), 255);
    // img * (1. / 255) - 0.5 in double (numpy), then the float32 cast of the network's placeholder
    out[t] = (float)__dadd_rn(__dmul_rn((double)v, 1.0 / 255), -0.5);
}

}  // namespace

int launch_cvt_img2train_u8(const uint8_t* bgr, int S, int H, int W, const int32_t* kx, const int32_t* x0, const int32_t* xn, int ksx,
                            const int32_t* ky, const int32_t* y0, const int32_t* yn, int ksy, int out_h, int out_w, uint8_t* tmp,
                            float* out, cudaStream_t st, int src_fmt)
{
    const dim3 g1((H * out_w + 255) / 256, S);
    switch (src_fmt) {
    case SRC_BGR: gray_hpass_kernel<SRC_BGR><<<g1, 256, 0, st>>>(bgr, H, W, kx, x0, xn, ksx, out_w, tmp, nullptr, nullptr); break;
    case MGW_YUV420_NV12:
        gray_hpass_kernel<MGW_YUV420_NV12><<<g1, 256, 0, st>>>(bgr, H, W, kx, x0, xn, ksx, out_w, tmp, nullptr, nullptr); break;
    case MGW_YUV420_I420:
        gray_hpass_kernel<MGW_YUV420_I420><<<g1, 256, 0, st>>>(bgr, H, W, kx, x0, xn, ksx, out_w, tmp, nullptr, nullptr); break;
    default: return set_error(MGW_ERR_INVALID, "cvt_img2train: unknown source format %d", src_fmt);
    }
    if (int rc = check_launch("gray_hpass")) return rc;
    vpass_norm_kernel<<<dim3((out_h * out_w + 255) / 256, S), 256, 0, st>>>(tmp, H, out_w, ky, y0, yn, ksy, out_h, out, nullptr, 0, nullptr);
    return check_launch("vpass_norm");
}

template <int FMT>
static int cvt_planes(const mgw_planes* src, int S, int H, int W, const int32_t* kx, const int32_t* x0, const int32_t* xn, int ksx,
                      const int32_t* ky, const int32_t* y0, const int32_t* yn, int ksy, int out_h, int out_w, uint8_t* tmp, float* out,
                      cudaStream_t st)
{
    gray_hpass_kernel<FMT, false, true><<<dim3((H * out_w + 255) / 256, S), 256, 0, st>>>(nullptr, H, W, kx, x0, xn, ksx, out_w, tmp,
                                                                                        nullptr, src);
    if (int rc = check_launch("gray_hpass")) return rc;
    vpass_norm_kernel<FMT, false, true><<<dim3((out_h * out_w + 255) / 256, S), 256, 0, st>>>(tmp, H, out_w, ky, y0, yn, ksy, out_h, out,
                                                                                            nullptr, W, src);
    return check_launch("vpass_norm");
}

int launch_cvt_img2train_planes(const mgw_planes* src, int src_fmt, int S, int H, int W, const int32_t* kx, const int32_t* x0,
                                const int32_t* xn, int ksx, const int32_t* ky, const int32_t* y0, const int32_t* yn, int ksy, int out_h,
                                int out_w, uint8_t* tmp, float* out, cudaStream_t st)
{
    switch (src_fmt) {
    case SRC_BGR: return cvt_planes<SRC_BGR>(src, S, H, W, kx, x0, xn, ksx, ky, y0, yn, ksy, out_h, out_w, tmp, out, st);
    case MGW_YUV420_NV12: return cvt_planes<MGW_YUV420_NV12>(src, S, H, W, kx, x0, xn, ksx, ky, y0, yn, ksy, out_h, out_w, tmp, out, st);
    case MGW_YUV420_I420: return cvt_planes<MGW_YUV420_I420>(src, S, H, W, kx, x0, xn, ksx, ky, y0, yn, ksy, out_h, out_w, tmp, out, st);
    default: return set_error(MGW_ERR_INVALID, "cvt_img2train_planes: unknown source format %d", src_fmt);
    }
}

template <int FMT>
static int cvt_mixed(const uint8_t* src, int S, int max_h, int max_w, const int2* sizes, const int32_t* kx, const int32_t* x0,
                     const int32_t* xn, int ksx, const int32_t* ky, const int32_t* y0, const int32_t* yn, int ksy, int out_h, int out_w,
                     uint8_t* tmp, float* out, cudaStream_t st)
{
    gray_hpass_kernel<FMT, true><<<dim3((max_h * out_w + 255) / 256, S), 256, 0, st>>>(src, max_h, max_w, kx, x0, xn, ksx, out_w, tmp, sizes,
                                                                                      nullptr);
    if (int rc = check_launch("gray_hpass")) return rc;
    vpass_norm_kernel<FMT, true><<<dim3((out_h * out_w + 255) / 256, S), 256, 0, st>>>(tmp, max_h, out_w, ky, y0, yn, ksy, out_h, out,
                                                                                      sizes, max_w, nullptr);
    return check_launch("vpass_norm");
}

int launch_cvt_img2train_mixed(const uint8_t* src, int src_fmt, int S, int max_h, int max_w, const int32_t* sizes, const int32_t* kx,
                               const int32_t* x0, const int32_t* xn, int ksx, const int32_t* ky, const int32_t* y0, const int32_t* yn,
                               int ksy, int out_h, int out_w, uint8_t* tmp, float* out, cudaStream_t st)
{
    const int2* sz = reinterpret_cast<const int2*>(sizes);
    switch (src_fmt) {
    case SRC_BGR: return cvt_mixed<SRC_BGR>(src, S, max_h, max_w, sz, kx, x0, xn, ksx, ky, y0, yn, ksy, out_h, out_w, tmp, out, st);
    case MGW_YUV420_NV12: return cvt_mixed<MGW_YUV420_NV12>(src, S, max_h, max_w, sz, kx, x0, xn, ksx, ky, y0, yn, ksy, out_h, out_w, tmp, out, st);
    case MGW_YUV420_I420: return cvt_mixed<MGW_YUV420_I420>(src, S, max_h, max_w, sz, kx, x0, xn, ksx, ky, y0, yn, ksy, out_h, out_w, tmp, out, st);
    default: return set_error(MGW_ERR_INVALID, "cvt_img2train_mixed: unknown source format %d", src_fmt);
    }
}

template <int FMT>
static int cvt_mixed_planes(const mgw_planes* src, int S, int max_h, int max_w, const int2* sizes, const int32_t* kx, const int32_t* x0,
                            const int32_t* xn, int ksx, const int32_t* ky, const int32_t* y0, const int32_t* yn, int ksy, int out_h,
                            int out_w, uint8_t* tmp, float* out, cudaStream_t st)
{
    gray_hpass_kernel<FMT, true, true><<<dim3((max_h * out_w + 255) / 256, S), 256, 0, st>>>(nullptr, max_h, max_w, kx, x0, xn, ksx, out_w,
                                                                                           tmp, sizes, src);
    if (int rc = check_launch("gray_hpass")) return rc;
    vpass_norm_kernel<FMT, true, true><<<dim3((out_h * out_w + 255) / 256, S), 256, 0, st>>>(tmp, max_h, out_w, ky, y0, yn, ksy, out_h,
                                                                                           out, sizes, max_w, src);
    return check_launch("vpass_norm");
}

int launch_cvt_img2train_mixed_planes(const mgw_planes* src, int src_fmt, int S, int max_h, int max_w, const int32_t* sizes,
                                      const int32_t* kx, const int32_t* x0, const int32_t* xn, int ksx, const int32_t* ky,
                                      const int32_t* y0, const int32_t* yn, int ksy, int out_h, int out_w, uint8_t* tmp, float* out,
                                      cudaStream_t st)
{
    const int2* sz = reinterpret_cast<const int2*>(sizes);
    switch (src_fmt) {
    case SRC_BGR:
        return cvt_mixed_planes<SRC_BGR>(src, S, max_h, max_w, sz, kx, x0, xn, ksx, ky, y0, yn, ksy, out_h, out_w, tmp, out, st);
    case MGW_YUV420_NV12:
        return cvt_mixed_planes<MGW_YUV420_NV12>(src, S, max_h, max_w, sz, kx, x0, xn, ksx, ky, y0, yn, ksy, out_h, out_w, tmp, out, st);
    case MGW_YUV420_I420:
        return cvt_mixed_planes<MGW_YUV420_I420>(src, S, max_h, max_w, sz, kx, x0, xn, ksx, ky, y0, yn, ksy, out_h, out_w, tmp, out, st);
    default: return set_error(MGW_ERR_INVALID, "cvt_img2train_mixed_planes: unknown source format %d", src_fmt);
    }
}

// ---------------------------------------------------------------------------------------------------------------------
// cv2.resize(frame, (width, height)) of the uint8 colour frame (deploy_bundle.py:301; INTER_LINEAR): OpenCV's 8-bit path --
// 11-bit fixed-point weights (tables from the host binding: x0, x1, a0, a1 per output column / row), int32 horizontal sums,
// ((b0*(S0>>4))>>16) + ((b1*(S1>>4))>>16) + 2) >> 2 vertically; an exact 2x2 decimation is OpenCV's INTER_AREA shortcut.
// blockIdx.y is the frame of a batch of S frames of one size (as for cvt_img2train above).
namespace {

__device__ __forceinline__ int ch_of(const int3& p, int ch) { return ch == 0 ? p.x : (ch == 1 ? p.y : p.z); }

// MIXED: H, W are the capacity (see cvt_img2train above); xtab [S,out_w], ytab [S,out_h]; the 2x2 shortcut is the slot's own
// PLANES: slot s's source is entry s of the table `planes` (img unused), the uniform tables and dst; an idle slot writes nothing
// MIXED && PLANES: the MIXED slot (size rule, tables, its own 2x2 shortcut) read from its entry (load_planes_at)
template <int C, int FMT = SRC_BGR, bool MIXED = false, bool PLANES = false>
__global__ void __launch_bounds__(256)
resize_u8_kernel(const uint8_t* __restrict__ img, int H, int W, const int4* __restrict__ xtab, const int4* __restrict__ ytab,
                 int out_h, int out_w, int area2, uint8_t* __restrict__ dst, const int2* __restrict__ sizes,
                 const mgw_planes* __restrict__ planes)
{
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= out_h * out_w) return;
    if constexpr (PLANES) {
        static_assert(C == 3, "a table's slot is a colour frame");
        Planes f;
        if constexpr (MIXED) {
            const int2 sz = __ldg(sizes + blockIdx.y);
            if (!slot_active<FMT>(sz, H, W) || !load_planes_at<FMT>(planes, blockIdx.y, sz, f)) return;
            xtab += (size_t)blockIdx.y * out_w;
            ytab += (size_t)blockIdx.y * out_h;
            area2 = sz.y == 2 * out_w && sz.x == 2 * out_h;
        } else if (!load_planes<FMT>(planes, blockIdx.y, W, f)) return;
        const int x = t % out_w, y = t / out_w;
        uint8_t* o = dst + ((size_t)blockIdx.y * out_h * out_w + t) * 3;
        int3 p00, p01, p10, p11;
        if (area2) {
            if constexpr (FMT == SRC_BGR) {
                p00 = planes_bgr_at<FMT>(f, 2 * y, 2 * x); p01 = planes_bgr_at<FMT>(f, 2 * y, 2 * x + 1);
                p10 = planes_bgr_at<FMT>(f, 2 * y + 1, 2 * x); p11 = planes_bgr_at<FMT>(f, 2 * y + 1, 2 * x + 1);
            } else {
                // the 2x2 block starts at even coordinates: four Y samples, one chroma sample
                const uint8_t* py = f.p[0] + (size_t)(2 * y) * f.pitch[0] + 2 * x;
                const Chroma c = planes_chroma_at<FMT>(f, 2 * y, 2 * x);
                p00 = yuv_to_bgr(__ldg(py), c); p01 = yuv_to_bgr(__ldg(py + 1), c);
                p10 = yuv_to_bgr(__ldg(py + f.pitch[0]), c); p11 = yuv_to_bgr(__ldg(py + f.pitch[0] + 1), c);
            }
            o[0] = (uint8_t)((p00.x + p01.x + p10.x + p11.x + 2) >> 2);
            o[1] = (uint8_t)((p00.y + p01.y + p10.y + p11.y + 2) >> 2);
            o[2] = (uint8_t)((p00.z + p01.z + p10.z + p11.z + 2) >> 2);
            return;
        }
        const int4 xt = __ldg(xtab + x), yt = __ldg(ytab + y);        // {i0, i1, a0, a1}
        p00 = planes_bgr_at<FMT>(f, yt.x, xt.x); p01 = planes_bgr_at<FMT>(f, yt.x, xt.y);
        p10 = planes_bgr_at<FMT>(f, yt.y, xt.x); p11 = planes_bgr_at<FMT>(f, yt.y, xt.y);
#pragma unroll
        for (int ch = 0; ch < 3; ++ch) {
            const int h0 = ch_of(p00, ch) * xt.z + ch_of(p01, ch) * xt.w;
            const int h1 = ch_of(p10, ch) * xt.z + ch_of(p11, ch) * xt.w;
            const int v = (((yt.z * (h0 >> 4)) >> 16) + ((yt.w * (h1 >> 4)) >> 16) + 2) >> 2;
            o[ch] = (uint8_t)min(max(v, 0), 255);
        }
        return;
    }
    if constexpr (MIXED) {
        static_assert(C == 3, "a slot's frame is BGR or YUV 4:2:0");
        const int2 sz = __ldg(sizes + blockIdx.y);
        if (!slot_active<FMT>(sz, H, W)) return;
        img += (size_t)blockIdx.y * src_frame_bytes<FMT>(H, W);
        xtab += (size_t)blockIdx.y * out_w;
        ytab += (size_t)blockIdx.y * out_h;
        H = sz.x; W = sz.y;
        area2 = W == 2 * out_w && H == 2 * out_h;
    }
    const unsigned s = MIXED ? 0u : blockIdx.y;             // the source frame index of a uniform batch
    if constexpr (FMT != SRC_BGR) {
        static_assert(C == 3, "a YUV 4:2:0 source resizes to BGR");
        const uint8_t* f = img + (size_t)s * src_frame_bytes<FMT>(H, W);
        dst += (size_t)blockIdx.y * out_h * out_w * 3;
        const int x = t % out_w, y = t / out_w;
        uint8_t* o = dst + (size_t)t * 3;
        if (area2) {
            // the 2x2 block starts at even coordinates: four Y samples, one chroma sample
            const uint8_t* py = f + (size_t)(2 * y) * W + 2 * x;
            const Chroma c = yuv_chroma_at<FMT>(f, H, W, 2 * y, 2 * x);
            const int3 p00 = yuv_to_bgr(__ldg(py), c), p01 = yuv_to_bgr(__ldg(py + 1), c);
            const int3 p10 = yuv_to_bgr(__ldg(py + W), c), p11 = yuv_to_bgr(__ldg(py + W + 1), c);
            o[0] = (uint8_t)((p00.x + p01.x + p10.x + p11.x + 2) >> 2);
            o[1] = (uint8_t)((p00.y + p01.y + p10.y + p11.y + 2) >> 2);
            o[2] = (uint8_t)((p00.z + p01.z + p10.z + p11.z + 2) >> 2);
            return;
        }
        const int4 xt = __ldg(xtab + x), yt = __ldg(ytab + y);        // {i0, i1, a0, a1}
        const int3 p00 = yuv_bgr_at<FMT>(f, H, W, yt.x, xt.x), p01 = yuv_bgr_at<FMT>(f, H, W, yt.x, xt.y);
        const int3 p10 = yuv_bgr_at<FMT>(f, H, W, yt.y, xt.x), p11 = yuv_bgr_at<FMT>(f, H, W, yt.y, xt.y);
#pragma unroll
        for (int ch = 0; ch < 3; ++ch) {
            const int h0 = ch_of(p00, ch) * xt.z + ch_of(p01, ch) * xt.w;
            const int h1 = ch_of(p10, ch) * xt.z + ch_of(p11, ch) * xt.w;
            const int v = (((yt.z * (h0 >> 4)) >> 16) + ((yt.w * (h1 >> 4)) >> 16) + 2) >> 2;
            o[ch] = (uint8_t)min(max(v, 0), 255);
        }
        return;
    }
    img += (size_t)s * H * W * C;
    dst += (size_t)blockIdx.y * out_h * out_w * C;
    const int x = t % out_w, y = t / out_w;
    uint8_t* o = dst + (size_t)t * C;
    if (area2) {
        const uint8_t* p = img + ((size_t)(2 * y) * W + 2 * x) * C;
#pragma unroll
        for (int ch = 0; ch < C; ++ch)
            o[ch] = (uint8_t)(((int)__ldg(p + ch) + (int)__ldg(p + C + ch) + (int)__ldg(p + (size_t)W * C + ch) +
                               (int)__ldg(p + (size_t)W * C + C + ch) + 2) >> 2);
        return;
    }
    const int4 xt = __ldg(xtab + x), yt = __ldg(ytab + y);            // {i0, i1, a0, a1}
    const uint8_t* r0 = img + (size_t)yt.x * W * C;
    const uint8_t* r1 = img + (size_t)yt.y * W * C;
#pragma unroll
    for (int ch = 0; ch < C; ++ch) {
        const int h0 = (int)__ldg(r0 + xt.x * C + ch) * xt.z + (int)__ldg(r0 + xt.y * C + ch) * xt.w;
        const int h1 = (int)__ldg(r1 + xt.x * C + ch) * xt.z + (int)__ldg(r1 + xt.y * C + ch) * xt.w;
        const int v = (((yt.z * (h0 >> 4)) >> 16) + ((yt.w * (h1 >> 4)) >> 16) + 2) >> 2;
        o[ch] = (uint8_t)min(max(v, 0), 255);
    }
}

}  // namespace

int launch_resize_linear_u8(const uint8_t* img, int S, int H, int W, int C, const int32_t* xtab, const int32_t* ytab, int out_h, int out_w,
                            uint8_t* dst, cudaStream_t st, int src_fmt)
{
    const int area2 = (W == 2 * out_w && H == 2 * out_h) ? 1 : 0;
    if (!area2 && (!xtab || !ytab)) return set_error(MGW_ERR_INVALID, "resize_linear_u8: coefficient tables are required");
    const dim3 grid((out_h * out_w + 255) / 256, S);
    const int4* xt = reinterpret_cast<const int4*>(xtab);
    const int4* yt = reinterpret_cast<const int4*>(ytab);
    if (src_fmt != SRC_BGR) {
        if (C != 3) return set_error(MGW_ERR_UNSUPPORTED, "resize_linear_u8: a YUV 4:2:0 source gives C = 3 (got %d)", C);
        switch (src_fmt) {
        case MGW_YUV420_NV12:
            resize_u8_kernel<3, MGW_YUV420_NV12><<<grid, 256, 0, st>>>(img, H, W, xt, yt, out_h, out_w, area2, dst, nullptr, nullptr); break;
        case MGW_YUV420_I420:
            resize_u8_kernel<3, MGW_YUV420_I420><<<grid, 256, 0, st>>>(img, H, W, xt, yt, out_h, out_w, area2, dst, nullptr, nullptr); break;
        default: return set_error(MGW_ERR_INVALID, "resize_linear_u8: unknown source format %d", src_fmt);
        }
        return check_launch("resize_u8");
    }
    switch (C) {
    case 1: resize_u8_kernel<1><<<grid, 256, 0, st>>>(img, H, W, xt, yt, out_h, out_w, area2, dst, nullptr, nullptr); break;
    case 3: resize_u8_kernel<3><<<grid, 256, 0, st>>>(img, H, W, xt, yt, out_h, out_w, area2, dst, nullptr, nullptr); break;
    case 4: resize_u8_kernel<4><<<grid, 256, 0, st>>>(img, H, W, xt, yt, out_h, out_w, area2, dst, nullptr, nullptr); break;
    default: return set_error(MGW_ERR_UNSUPPORTED, "resize_linear_u8: C must be 1, 3 or 4 (got %d)", C);
    }
    return check_launch("resize_u8");
}

int launch_resize_linear_planes(const mgw_planes* src, int src_fmt, int S, int H, int W, const int32_t* xtab, const int32_t* ytab,
                                int out_h, int out_w, uint8_t* dst, cudaStream_t st)
{
    const int area2 = (W == 2 * out_w && H == 2 * out_h) ? 1 : 0;
    const dim3 grid((out_h * out_w + 255) / 256, S);
    const int4* xt = reinterpret_cast<const int4*>(xtab);
    const int4* yt = reinterpret_cast<const int4*>(ytab);
    switch (src_fmt) {
    case SRC_BGR:
        resize_u8_kernel<3, SRC_BGR, false, true><<<grid, 256, 0, st>>>(nullptr, H, W, xt, yt, out_h, out_w, area2, dst, nullptr, src); break;
    case MGW_YUV420_NV12:
        resize_u8_kernel<3, MGW_YUV420_NV12, false, true><<<grid, 256, 0, st>>>(nullptr, H, W, xt, yt, out_h, out_w, area2, dst, nullptr, src);
        break;
    case MGW_YUV420_I420:
        resize_u8_kernel<3, MGW_YUV420_I420, false, true><<<grid, 256, 0, st>>>(nullptr, H, W, xt, yt, out_h, out_w, area2, dst, nullptr, src);
        break;
    default: return set_error(MGW_ERR_INVALID, "resize_linear_planes: unknown source format %d", src_fmt);
    }
    return check_launch("resize_u8");
}

int launch_resize_linear_mixed(const uint8_t* src, int src_fmt, int S, int max_h, int max_w, const int32_t* sizes, const int32_t* xtab,
                               const int32_t* ytab, int out_h, int out_w, uint8_t* dst, cudaStream_t st)
{
    const dim3 grid((out_h * out_w + 255) / 256, S);
    const int2* sz = reinterpret_cast<const int2*>(sizes);
    const int4* xt = reinterpret_cast<const int4*>(xtab);
    const int4* yt = reinterpret_cast<const int4*>(ytab);
    switch (src_fmt) {
    case SRC_BGR: resize_u8_kernel<3, SRC_BGR, true><<<grid, 256, 0, st>>>(src, max_h, max_w, xt, yt, out_h, out_w, 0, dst, sz, nullptr); break;
    case MGW_YUV420_NV12:
        resize_u8_kernel<3, MGW_YUV420_NV12, true><<<grid, 256, 0, st>>>(src, max_h, max_w, xt, yt, out_h, out_w, 0, dst, sz, nullptr); break;
    case MGW_YUV420_I420:
        resize_u8_kernel<3, MGW_YUV420_I420, true><<<grid, 256, 0, st>>>(src, max_h, max_w, xt, yt, out_h, out_w, 0, dst, sz, nullptr); break;
    default: return set_error(MGW_ERR_INVALID, "resize_linear_mixed: unknown source format %d", src_fmt);
    }
    return check_launch("resize_u8");
}

int launch_resize_linear_mixed_planes(const mgw_planes* src, int src_fmt, int S, int max_h, int max_w, const int32_t* sizes,
                                      const int32_t* xtab, const int32_t* ytab, int out_h, int out_w, uint8_t* dst, cudaStream_t st)
{
    const dim3 grid((out_h * out_w + 255) / 256, S);
    const int2* sz = reinterpret_cast<const int2*>(sizes);
    const int4* xt = reinterpret_cast<const int4*>(xtab);
    const int4* yt = reinterpret_cast<const int4*>(ytab);
    switch (src_fmt) {
    case SRC_BGR:
        resize_u8_kernel<3, SRC_BGR, true, true><<<grid, 256, 0, st>>>(nullptr, max_h, max_w, xt, yt, out_h, out_w, 0, dst, sz, src); break;
    case MGW_YUV420_NV12:
        resize_u8_kernel<3, MGW_YUV420_NV12, true, true><<<grid, 256, 0, st>>>(nullptr, max_h, max_w, xt, yt, out_h, out_w, 0, dst, sz, src);
        break;
    case MGW_YUV420_I420:
        resize_u8_kernel<3, MGW_YUV420_I420, true, true><<<grid, 256, 0, st>>>(nullptr, max_h, max_w, xt, yt, out_h, out_w, 0, dst, sz, src);
        break;
    default: return set_error(MGW_ERR_INVALID, "resize_linear_mixed_planes: unknown source format %d", src_fmt);
    }
    return check_launch("resize_u8");
}

int launch_warp_rev_bundle_u8(const uint8_t* img, const double* Hs_cvt, int N, int H, int W, int C, int gh, int gw, uint8_t* dst,
                              cudaStream_t st)
{
    // WarpPerspectiveInvoker's block width: bh0 = min(16, H); bw0 = min(1024 / bh0, W)
    const int bh0 = H < 16 ? H : 16;
    const int bw = (1024 / bh0) < W ? (1024 / bh0) : W;
    const int t = N * H * W, grid = (t + 255) / 256;
    switch (C) {
    case 1: warp_rev_bundle_kernel<1><<<grid, 256, 0, st>>>(img, Hs_cvt, N, H, W, gh, gw, bw, dst); break;
    case 3: warp_rev_bundle_kernel<3><<<grid, 256, 0, st>>>(img, Hs_cvt, N, H, W, gh, gw, bw, dst); break;
    case 4: warp_rev_bundle_kernel<4><<<grid, 256, 0, st>>>(img, Hs_cvt, N, H, W, gh, gw, bw, dst); break;
    default: return set_error(MGW_ERR_UNSUPPORTED, "warp_rev_bundle_u8: C must be 1, 3 or 4 (got %d)", C);
    }
    return check_launch("warp_rev_bundle");
}

// ---------------------------------------------------------------- frame transport
// config.py:19: img * (1. / 255) - 0.5 in double (numpy: uint8 array times a Python float), then the float32 cast of the network's
// placeholder.  Frames cross PCIe as uint8 (a quarter of the fp32 bytes) and are widened here.
__global__ void u8_to_train_kernel(const uint8_t* __restrict__ src, float* __restrict__ dst, size_t n)
{
    const size_t i4 = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) * 4;
    if (i4 >= n) return;
    if (i4 + 4 <= n && ((reinterpret_cast<uintptr_t>(src) | (reinterpret_cast<uintptr_t>(dst) >> 2)) & 3) == 0) {
        const uchar4 v = *reinterpret_cast<const uchar4*>(src + i4);
        float4 o;
        o.x = (float)__dadd_rn(__dmul_rn((double)v.x, 1.0 / 255), -0.5); o.y = (float)__dadd_rn(__dmul_rn((double)v.y, 1.0 / 255), -0.5);
        o.z = (float)__dadd_rn(__dmul_rn((double)v.z, 1.0 / 255), -0.5); o.w = (float)__dadd_rn(__dmul_rn((double)v.w, 1.0 / 255), -0.5);
        *reinterpret_cast<float4*>(dst + i4) = o;
    } else {
        for (size_t i = i4; i < n && i < i4 + 4; ++i) dst[i] = (float)__dadd_rn(__dmul_rn((double)src[i], 1.0 / 255), -0.5);
    }
}

// cvt_train2img, deploy_bundle.py:75: ((x + 0.5) * 255).astype(np.uint8) on a float32 array: two fp32 operations, truncation
// towards zero; values outside [0, 256) wrap like the x86 conversion numpy compiles to (int32 truncation, low byte; NaN -> 0).
__device__ __forceinline__ uint8_t train_to_u8(float x)
{
    const float v = __fmul_rn(__fadd_rn(x, 0.5f), 255.0f);
    const int t = (fabsf(v) < 2147483648.0f) ? __float2int_rz(v) : (int)0x80000000;
    return (uint8_t)(t & 0xff);
}

__global__ void train_to_u8_kernel(const float* __restrict__ src, uint8_t* __restrict__ dst, size_t n)
{
    const size_t i4 = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) * 4;
    if (i4 >= n) return;
    if (i4 + 4 <= n && (((reinterpret_cast<uintptr_t>(src) >> 2) | reinterpret_cast<uintptr_t>(dst)) & 3) == 0) {
        const float4 v = *reinterpret_cast<const float4*>(src + i4);
        *reinterpret_cast<uchar4*>(dst + i4) = make_uchar4(train_to_u8(v.x), train_to_u8(v.y), train_to_u8(v.z), train_to_u8(v.w));
    } else {
        for (size_t i = i4; i < n && i < i4 + 4; ++i) dst[i] = train_to_u8(src[i]);
    }
}

// 16 bytes per thread and iteration; keep = the lines are written with an L2 evict_last policy, so that a buffer which is
// accumulated into next (dU of the backward: reductions at L2) is still resident when its kernel starts
// Small blocks with a handful of registers on purpose: the fill is meant to run NEXT TO the persistent warp kernels, which
// leave only ~3 K registers and a few hundred thread slots per SM free (a 256-thread block does not fit and would wait for
// them to finish).
template <bool KEEP>
__global__ void __launch_bounds__(64) fill_zero_kernel(uint4* __restrict__ p, size_t n16)
{
    // programmatic dependent launch on both sides: the blocks may be scheduled under the tail of the previous kernel (the forward
    // warp) and the next one (the backward warp) may set itself up while the fill runs
    griddep_wait();
    griddep_launch_dependents();
    uint64_t pol = 0;
    if (KEEP) asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(pol));
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n16; i += (size_t)gridDim.x * blockDim.x) {
        if (KEEP) asm volatile("st.global.L2::cache_hint.v4.b32 [%0], {%1, %1, %1, %1}, %2;" ::"l"(p + i), "r"(0), "l"(pol) : "memory");
        else p[i] = make_uint4(0, 0, 0, 0);
    }
}

int launch_u8_to_train(const uint8_t* src, float* dst, size_t n, cudaStream_t st)
{
    const size_t blocks = ((n + 3) / 4 + 255) / 256;
    if (blocks > 0x7fffffffULL) return set_error(MGW_ERR_INVALID, "u8_to_train: too many elements");
    u8_to_train_kernel<<<(unsigned)blocks, 256, 0, st>>>(src, dst, n);
    return check_launch("u8_to_train");
}

int launch_train_to_u8(const float* src, uint8_t* dst, size_t n, cudaStream_t st)
{
    const size_t blocks = ((n + 3) / 4 + 255) / 256;
    if (blocks > 0x7fffffffULL) return set_error(MGW_ERR_INVALID, "train_to_u8: too many elements");
    train_to_u8_kernel<<<(unsigned)blocks, 256, 0, st>>>(src, dst, n);
    return check_launch("train_to_u8");
}

int launch_fill_zero(void* p, size_t bytes, bool keep_in_l2, cudaStream_t st)
{
    const size_t n16 = bytes / 16;
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    // 24 blocks of 64 threads per SM: measured next to the tile backward that now starts under the fill (step at config #2 with
    // 4 / 8 / 16 / 24 / 32 blocks per SM: 131.7 / 118.1 / 109.6 / 108.3 / 108.7 us)
    size_t per_sm = 24;
    if (const char* e = getenv("MGW_FILL_BLOCKS_PER_SM")) { const int v = atoi(e); if (v > 0) per_sm = (size_t)v; }      // tuning aid
    const size_t want = (n16 + 63) / 64, cap = (size_t)sms * per_sm;
    const unsigned grid = (unsigned)(want < cap ? want : cap);
    const cudaError_t e = keep_in_l2 ? launch_ex(fill_zero_kernel<true>, dim3(grid), dim3(64), 0, st, pdl_enabled(), reinterpret_cast<uint4*>(p), n16)
                                     : launch_ex(fill_zero_kernel<false>, dim3(grid), dim3(64), 0, st, pdl_enabled(), reinterpret_cast<uint4*>(p), n16);
    if (e != cudaSuccess) { count_launches(1); return set_error(MGW_ERR_CUDA, "fill_zero: %s", cudaGetErrorString(e)); }
    return check_launch("fill_zero");
}

}  // namespace mgw

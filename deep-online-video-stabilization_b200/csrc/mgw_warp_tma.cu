// K2/K3, TMA-staged tile variant (the fast path of the multi-grid warp on sm_100a).
//
// One CTA = one output tile of TH x TW pixels lying inside ONE mesh cell (so one homography), 256 threads; thread
// (tx, g) owns column tx and the K consecutive rows g*K..g*K+K-1 (TH = K * 256/TW), so a warp always touches 32
// consecutive pixels of a row: 12-byte lane strides in shared memory, conflict free.
//   forward : warp 0 decodes the tile, projects its 4 corners and issues ONE TMA load (cp.async.bulk.tensor.3d,
//             SASS UTMALDG) of the source bounding box while all threads compute the per-pixel projective map; the
//             bilinear gather reads shared memory; out / x_map,y_map / black_pix are staged in shared memory and
//             leave by TMA stores (UTMASTG).
//   backward: the same source box of U by TMA, requested before anything else; in the plain variant (dU wanted, no fused loss)
//             the tile's d_out / d_img arrive by TMA too, into the accumulator box before it is zeroed (as 24 strided LDGs
//             per thread they queued in the LSU for thousands of cycles).  dU is pre-accumulated in a shared-memory box in
//             FIXED POINT with native integer shared atomics (ATOMS.ADD, ~1 cycle per warp instruction measured on B200,
//             against ~4-6 cycles and a serialising ~300-cycle round trip for the CAS loop behind atomicAdd(float*)); the
//             scale is a power of two chosen per tile from max|d_out|, kBits = 30 - floor(log2(TH*TW)) <= 22 bits per term:
//             a term rounds to at most 2^kBits and TH*TW of them stay below 2^31, so the int32 sums provably cannot
//             overflow.  The box leaves as fp32 by 16-byte reductions
//             (red.global.add.v4.f32, REDG; all-zero groups skipped) straight from the fixed-point words -- no conversion
//             back into shared memory, no third barrier, no TMA read wait before the CTA exits.
//             Launched programmatically behind the library's zero-fill of dU, the kernel runs next to it up to its first
//             access to dU (griddepcontrol.wait).  The 8 dH terms are reduced warp-shuffle -> shared -> one deterministic
//             partial per tile (no global atomics).
// Every tap is checked against the staged box; taps outside it (folded cells, extreme magnification, far
// out-of-range pixels) and weights outside [-1,1] fall back to global loads / global fp32 atomics, so results never
// depend on the box heuristic.  Arithmetic is mgw_device.cuh's, bit-identical to the generic kernels and the C oracle.
#include "mgw_tile.cuh"

#ifdef MGW_PROBE
__device__ unsigned long long g_probe[16];
extern "C" __attribute__((visibility("default"))) int mgw_debug_probe(unsigned long long* out, int reset)
{
    cudaDeviceSynchronize();
    cudaMemcpyFromSymbol(out, g_probe, sizeof(g_probe));
    if (reset) { unsigned long long z[16] = {}; cudaMemcpyToSymbol(g_probe, z, sizeof(z)); }
    return 0;
}
#define PROBE(i) do { if (threadIdx.x == MGW_PROBE_TID) { const long long t_ = clock64(); atomicAdd(&g_probe[i], (unsigned long long)(t_ - tprev)); tprev = t_; } } while (0)
#else
#define PROBE(i) do {} while (0)
#endif
#ifndef MGW_PROBE_TID
#define MGW_PROBE_TID 32
#endif

namespace mgw {

constexpr int kMaxWarps = 16;

template <int C, int TW, int K, int NT>
struct Geo {
    static constexpr int kGroups = NT / TW;
    static constexpr int TH = kGroups * K;
    static constexpr int kXalign = (C % 4 == 0) ? 1 : ((C % 2 == 0) ? 2 : 4);
    // Row pitch of the staged box in floats = TMA box inner dimension (<= 256 elements).  It is a multiple of 32 so
    // that a tap's bank depends only on its column: lanes of a warp that sit on different source rows (rotation,
    // shear) then never collide (a 252-float pitch made 40-50 % of the shared wavefronts conflict replays).  The
    // box need not hold a whole number of pixels; SBW is the number of complete pixels in a row.
    static constexpr int kWantF = (((TW * 13 + 9) / 10 + 4 + (kXalign - 1)) * C + 31) / 32 * 32;
    static constexpr int kRowF = kWantF < 256 ? kWantF : 256;
    static constexpr int SBW = kRowF / C;                                            // staged source box, pixels
    static constexpr int SBH = (TH * 13 + 9) / 10 + 4;
    static constexpr int kBoxF = SBH * kRowF;                                        // floats (multiple of 32)
    static constexpr int kOutF = (TH * TW * C + 31) / 32 * 32;
    static_assert(SBW >= TW + 4, "source box too narrow for this tile width / channel count");
};

// what warp 0 works out per tile for everyone else
struct TileInfo {
    int bx0, by0;                   // first column / row of the staged source box
    int interior;                   // every tap of every pixel of the tile is unclipped AND inside the staged box
    float wmax[kMaxWarps];          // backward: per-warp max|d_out|
};

struct Tile {
    int n, r0, c0, vr0, vc0, cell, part;
};

__device__ __forceinline__ Tile this_tile(const TileCfg& cfg)
{
    Tile t;
    const int ty = blockIdx.y, tx = blockIdx.x;
    t.n = blockIdx.z;
    t.r0 = cfg.rows.start[ty]; t.vr0 = cfg.rows.vstart[ty];
    t.c0 = cfg.cols.start[tx]; t.vc0 = cfg.cols.vstart[tx];
    t.cell = (t.n * cfg.gh + cfg.rows.cell[ty]) * cfg.gw + cfg.cols.cell[tx];
    t.part = cfg.rows.part[ty] * cfg.parts_x + cfg.cols.part[tx];
    return t;
}

// Source box of the tile, by warp 0 (lanes 0-3 project one corner each): bbox of the 4 projected corners (+1 px for
// rounding, +1 for the x1/y1 taps), clipped to the image like the taps are.  A projective map with no pole inside the
// tile (z of one sign at the corners) sends the rectangle into the convex hull of its corner images, so the box holds
// every tap.  `interior` says so, and additionally that no tap is clipped: such tiles (the vast majority) run a
// per-pixel path without clipping, bounds tests or address arithmetic; all other tiles test every tap and fall back
// to global memory for the ones outside the box.
template <int C, int TW, int K, int NT>
__device__ __forceinline__ void source_box(const TileCfg& cfg, const Tile& tl, const float (&Hc)[9], float stepx, float stepy,
                                           int& bx0, int& by0, int& interior, int* complete = nullptr)
{
    using G = Geo<C, TW, K, NT>;
    const int k4 = threadIdx.x & 3;
    const int rr = tl.r0 + ((k4 & 2) ? G::TH - 1 : 0), cc = tl.c0 + ((k4 & 1) ? TW - 1 : 0);
    const Proj q = project(Hc, lin_at(cc, stepx), lin_at(rr, stepy));
    const float x = (q.xn + 1.0f) * (float)cfg.W * 0.5f, y = (q.yn + 1.0f) * (float)cfg.H * 0.5f;
    bool ok = (fabsf(x) < 1.0e8f) && (fabsf(y) < 1.0e8f);
    int sgn = (q.zs > 0.0f) ? 1 : -1;
    float xmin = x, xmax = x, ymin = y, ymax = y;
#pragma unroll
    for (int o = 1; o < 4; o <<= 1) {
        xmin = fminf(xmin, __shfl_xor_sync(0xffffffffu, xmin, o));
        xmax = fmaxf(xmax, __shfl_xor_sync(0xffffffffu, xmax, o));
        ymin = fminf(ymin, __shfl_xor_sync(0xffffffffu, ymin, o));
        ymax = fmaxf(ymax, __shfl_xor_sync(0xffffffffu, ymax, o));
        sgn += __shfl_xor_sync(0xffffffffu, sgn, o);
        ok = ok && (__shfl_xor_sync(0xffffffffu, (int)ok, o) != 0);
    }
    ok = ok && (sgn == 4 || sgn == -4);
    bx0 = 0; by0 = 0; interior = 0;
    if (complete) *complete = 0;
    if (ok) {
        const int ux0 = (int)floorf(xmin) - 1, ux1 = (int)floorf(xmax) + 2;      // unclipped tap range, 1 px of slack
        const int uy0 = (int)floorf(ymin) - 1, uy1 = (int)floorf(ymax) + 2;
        const int ix0 = clipi(ux0, 0, cfg.W - 1), ix1 = clipi(ux1, 0, cfg.W - 1);
        const int iy0 = clipi(uy0, 0, cfg.H - 1), iy1 = clipi(uy1, 0, cfg.H - 1);
        const int needw = ix1 - ix0 + 1, needh = iy1 - iy0 + 1;
        bx0 = needw <= G::SBW ? ix0 : ix0 + (needw - G::SBW) / 2;
        by0 = needh <= G::SBH ? iy0 : iy0 + (needh - G::SBH) / 2;
        // TMA needs the box to start on a 16-byte boundary of global memory (measured on B200: a start that is not
        // a multiple of 4 floats raises "illegal instruction"): round the first column down
        bx0 -= bx0 % G::kXalign;
        interior = (ux0 >= 0 && ux1 <= cfg.W - 1 && uy0 >= 0 && uy1 <= cfg.H - 1 &&
                    ux1 - bx0 < G::SBW && uy1 - by0 < G::SBH) ? 1 : 0;
        // every tap that survives clipping lies inside the box (the backward skips pixels with a clipped tap, see below)
        if (complete) *complete = (ix0 >= bx0 && ix1 - bx0 < G::SBW && iy0 >= by0 && iy1 - by0 < G::SBH) ? 1 : 0;
    }
}

// taps of an INTERIOR pixel: no clipping can occur, so x0f = floor(x), x1f = x0f + 1 (exact) and the reference's
// weights (spatial_transformer3.py:114-121) reduce to these expressions bit for bit
struct FastTaps { int x0, y0; float ax, bx, ay, by; };
__device__ __forceinline__ FastTaps make_taps_interior(float xn, float yn, int IH, int IW)
{
    const float x = __fmul_rn(__fmul_rn(__fadd_rn(xn, 1.0f), (float)IW), 0.5f);
    const float y = __fmul_rn(__fmul_rn(__fadd_rn(yn, 1.0f), (float)IH), 0.5f);
    const float fx = floorf(x), fy = floorf(y);
    FastTaps t;
    t.x0 = __float2int_rz(fx); t.y0 = __float2int_rz(fy);
    t.ax = __fsub_rn(__fadd_rn(fx, 1.0f), x); t.bx = __fsub_rn(x, fx);
    t.ay = __fsub_rn(__fadd_rn(fy, 1.0f), y); t.by = __fsub_rn(y, fy);
    return t;
}

__device__ __forceinline__ float blend4(float ax, float bx, float ay, float by, float Ia, float Ib, float Ic, float Id)
{
    const float wa = __fmul_rn(ax, ay), wb = __fmul_rn(ax, by), wc = __fmul_rn(bx, ay), wd = __fmul_rn(bx, by);
    float s = __fmul_rn(wa, Ia);
    s = __fadd_rn(s, __fmul_rn(wb, Ib));
    s = __fadd_rn(s, __fmul_rn(wc, Ic));
    s = __fadd_rn(s, __fmul_rn(wd, Id));
    return s;
}

// ------------------------------------------------------------------------------------------------ forward
#ifndef MGW_FWD_MINB
#define MGW_FWD_MINB (NT == 256 ? (LOSS ? 3 : 4) : 2)
#endif
// LOSS = true fuses the img_loss epilogue (s_net_bundle_nobm.py:347-352) onto the warped tile: per-sample
// sums[n] += (sum over owned pixels of ((out - y)*(1-black))^2, sum of (1-black)).
template <int C, int TW, int K, int NT, bool LOSS>
__global__ void __launch_bounds__(NT, MGW_FWD_MINB)
warp_fwd_tma_kernel(const __grid_constant__ CUtensorMap mapU, const __grid_constant__ CUtensorMap mapOut,
                    const float* __restrict__ U, const float* __restrict__ Hs, const __grid_constant__ TileCfg cfg,
                    float* __restrict__ out, float* __restrict__ img, float* __restrict__ black,
                    const float* __restrict__ y_tgt, float* __restrict__ sums)
{
    using G = Geo<C, TW, K, NT>;
    extern __shared__ __align__(1024) unsigned char smem_raw[];
    float* s_src = reinterpret_cast<float*>(smem_raw);
    float* s_out = s_src + G::kBoxF;
    uint64_t* bar = reinterpret_cast<uint64_t*>(s_out + G::kOutF);
    TileInfo* ti = reinterpret_cast<TileInfo*>(bar + 2);

    const int tid = threadIdx.x;
    if (tid == 0) {
        tma::mbar_init(bar, 1);
        tma::fence_barrier_init();
    }
    const Tile tl = this_tile(cfg);
    float Hc[9];
#pragma unroll
    for (int k = 0; k < 9; ++k) Hc[k] = __ldg(Hs + (size_t)tl.cell * 9 + k);
    const float stepx = cfg.stepx, stepy = cfg.stepy;
    __syncthreads();                                  // barrier initialised; nobody has waited on anything long yet
    if (tid < 32 && out) {
        int bx0, by0, interior;
        source_box<C, TW, K, NT>(cfg, tl, Hc, stepx, stepy, bx0, by0, interior);
        if (tid == 0) {
            ti->bx0 = bx0; ti->by0 = by0; ti->interior = interior;
            tma::mbar_expect_tx(bar, (uint32_t)(G::kBoxF * sizeof(float)));     // release: publishes ti
            tma::load_3d(s_src, &mapU, bar, bx0 * C, by0, tl.n);
        }
    }

    const int tx = tid % TW, g = tid / TW;
    const float xt = lin_at(tl.c0 + tx, stepx);
    const float hx0 = __fmul_rn(Hc[0], xt), hx3 = __fmul_rn(Hc[3], xt), hx6 = __fmul_rn(Hc[6], xt);   // first term of hrow()
    float xn[K], yn[K];
    float yv[LOSS ? K : 1][C], nbv[LOSS ? K : 1];          // fused loss: target pixels and (1 - black) of the owned pixels
    {
        size_t p = ((size_t)tl.n * cfg.H + tl.r0 + g * K) * cfg.W + tl.c0 + tx;
#pragma unroll
        for (int k = 0; k < K; ++k, p += cfg.W) {
            if (LOSS) {
#pragma unroll
                for (int ch = 0; ch < C; ++ch) yv[k][ch] = __ldg(y_tgt + p * C + ch);
            }
            const float yt = lin_at(tl.r0 + g * K + k, stepy);
            const float xs = __fadd_rn(__fmaf_rn(Hc[1], yt, hx0), Hc[2]);
            const float ys = __fadd_rn(__fmaf_rn(Hc[4], yt, hx3), Hc[5]);
            float zs = __fadd_rn(__fmaf_rn(Hc[7], yt, hx6), Hc[8]);
            zs = __fadd_rn(zs, (zs >= 0.0f) ? 1e-8f : -1e-8f);
            div2_rn(xs, ys, zs, xn[k], yn[k]);
            // x_map,y_map and black_pix are 8 / 4 contiguous bytes per lane: plain coalesced stores, no staging
            const float bk = black_of(xn[k], yn[k]);
            if (img) reinterpret_cast<float2*>(img)[p] = make_float2(xn[k], yn[k]);
            if (black) black[p] = bk;
            if (LOSS) nbv[k] = (tl.r0 + g * K + k >= tl.vr0 && tl.c0 + tx >= tl.vc0) ? 1.0f - bk : -1.0f;    // -1: not owned
        }
    }
    if (!out) return;
    float se = 0.0f, sm = 0.0f;
    tma::mbar_wait(bar, 0);                           // acquire: the source box has landed and ti is visible
    const int bx0 = ti->bx0, by0 = ti->by0;
    if (ti->interior) {
#pragma unroll
        for (int k = 0; k < K; ++k) {
            const FastTaps t = make_taps_interior(xn[k], yn[k], cfg.H, cfg.W);
            const float* pa = s_src + ((t.y0 - by0) * G::kRowF + (t.x0 - bx0) * C);
            float* o = s_out + ((g * K + k) * TW + tx) * C;
#pragma unroll
            for (int ch = 0; ch < C; ++ch) {
                const float v = blend4(t.ax, t.bx, t.ay, t.by, pa[ch], pa[G::kRowF + ch], pa[C + ch], pa[G::kRowF + C + ch]);
                o[ch] = v;
                if (LOSS && nbv[k] >= 0.0f) { const float e = (v - yv[k][ch]) * nbv[k]; se = fmaf(e, e, se); }
            }
            if (LOSS && nbv[k] >= 0.0f) sm += nbv[k];
        }
    } else {
        const float* Un = U + (size_t)tl.n * cfg.H * cfg.W * C;
#pragma unroll
        for (int k = 0; k < K; ++k) {
            const Taps t = make_taps(xn[k], yn[k], cfg.H, cfg.W);
            const int sx0 = t.x0 - bx0, sx1 = t.x1 - bx0, sy0 = t.y0 - by0, sy1 = t.y1 - by0;
            float* o = s_out + ((g * K + k) * TW + tx) * C;
            if (sx0 >= 0 && sx1 < G::SBW && sy0 >= 0 && sy1 < G::SBH) {
                const float* pa = s_src + sy0 * G::kRowF + sx0 * C;
                const float* pb = s_src + sy1 * G::kRowF + sx0 * C;
                const float* pc = s_src + sy0 * G::kRowF + sx1 * C;
                const float* pd = s_src + sy1 * G::kRowF + sx1 * C;
#pragma unroll
                for (int ch = 0; ch < C; ++ch) o[ch] = blend(t, pa[ch], pb[ch], pc[ch], pd[ch]);
            } else {
                const float* pa = Un + ((size_t)t.y0 * cfg.W + t.x0) * C;
                const float* pb = Un + ((size_t)t.y1 * cfg.W + t.x0) * C;
                const float* pc = Un + ((size_t)t.y0 * cfg.W + t.x1) * C;
                const float* pd = Un + ((size_t)t.y1 * cfg.W + t.x1) * C;
#pragma unroll
                for (int ch = 0; ch < C; ++ch) o[ch] = blend(t, __ldg(pa + ch), __ldg(pb + ch), __ldg(pc + ch), __ldg(pd + ch));
            }
            if (LOSS && nbv[k] >= 0.0f) {
#pragma unroll
                for (int ch = 0; ch < C; ++ch) { const float e = (o[ch] - yv[k][ch]) * nbv[k]; se = fmaf(e, e, se); }
                sm += nbv[k];
            }
        }
    }
    if (LOSS) {
        se = warp_sum(se); sm = warp_sum(sm);
        float* s_loss = reinterpret_cast<float*>(ti + 1);             // [warps][2]
        if ((tid & 31) == 0) { s_loss[(tid >> 5) * 2] = se; s_loss[(tid >> 5) * 2 + 1] = sm; }
    }
    tma::fence_proxy_async();
    __syncthreads();
    if (tid == 0) {
        tma::store_3d(&mapOut, s_out, tl.c0 * C, tl.r0, tl.n);
        tma::commit_group();
        if (LOSS) {
            const float* s_loss = reinterpret_cast<const float*>(ti + 1);
            float a = 0.0f, b = 0.0f;
#pragma unroll
            for (int w = 0; w < NT / 32; ++w) { a += s_loss[2 * w]; b += s_loss[2 * w + 1]; }
            atomicAdd(sums + 2 * tl.n, a);
            atomicAdd(sums + 2 * tl.n + 1, b);
        }
        tma::wait_group_read0();
    }
}

// ------------------------------------------------------------------------------------------------ backward
// float <-> fixed point without the conversion unit (F2I / I2F issue at a quarter rate on the XU pipe and there are 12
// per pixel): adding 1.5*2^23 leaves round-to-nearest-even(v) in the low mantissa bits for |v| <= 2^22.
constexpr float kMagic = 12582912.0f;          // 1.5 * 2^23
constexpr int kMagicBits = 0x4B400000;
__device__ __forceinline__ int fixed_of(float w, float gs) { return __float_as_int(__fmaf_rn(w, gs, kMagic)) - kMagicBits; }
__device__ __forceinline__ float float_of_fixed(int v) { return (float)v; }      // sums of coincident taps may exceed 2^22: plain I2F
constexpr int bit_width(int v) { return v > 0 ? 1 + bit_width(v >> 1) : 0; }       // floor(log2 v) + 1

// dH terms of one pixel (SURVEY.md 8a-bwd) accumulated into the thread's 8 partial sums
__device__ __forceinline__ void accumulate_dh(float (&dh)[8], float gxn, float gyn, float xn, float yn, float zs, float xt, float yt)
{
    const float rz = __frcp_rn(zs);
    const float dxs = gxn * rz, dys = gyn * rz;
    const float dzs = -(gxn * xn + gyn * yn) * rz;
    dh[0] = fmaf(dxs, xt, dh[0]); dh[1] = fmaf(dxs, yt, dh[1]); dh[2] += dxs;
    dh[3] = fmaf(dys, xt, dh[3]); dh[4] = fmaf(dys, yt, dh[4]); dh[5] += dys;
    dh[6] = fmaf(dzs, xt, dh[6]); dh[7] = fmaf(dzs, yt, dh[7]);
}

// the same with the reciprocal of zs already at hand (the shared-reciprocal division of the fast path)
__device__ __forceinline__ void accumulate_dh_r(float (&dh)[8], float gxn, float gyn, float xn, float yn, float rz, float xt, float yt)
{
    const float dxs = gxn * rz, dys = gyn * rz;
    const float dzs = -(gxn * xn + gyn * yn) * rz;
    dh[0] = fmaf(dxs, xt, dh[0]); dh[1] = fmaf(dxs, yt, dh[1]); dh[2] += dxs;
    dh[3] = fmaf(dys, xt, dh[3]); dh[4] = fmaf(dys, yt, dh[4]); dh[5] += dys;
    dh[6] = fmaf(dzs, xt, dh[6]); dh[7] = fmaf(dzs, yt, dh[7]);
}

// LOSS = true takes the upstream gradient from the fused img_loss instead of a d_out tensor:
// d_out = kscale/(sums[n][1]+1e-8) * (out - y) * (1-black)^2, computed in registers from the forward's out / black; a d_out tensor
// given on top of that (nullable) is added to it (the gradient of another consumer of `output`, e.g. temp_loss).
struct LossBwd {
    const float* out;       // forward output_img
    const float* y;         // target
    const float* black;     // forward black_pix
    const float* sums;      // [N,2] from the fused forward
    float kscale;           // upstream * 2 / batch
    const float* kscale_dev;    // nullable device factor on kscale
};

#ifndef MGW_BWD_MINB
#define MGW_BWD_MINB (NT == 256 ? (K <= 3 ? 4 : 3) : 2)
#endif
#ifndef MGW_BWD_NODU_MINB
#define MGW_BWD_NODU_MINB (NT == 256 ? 4 : 2)
#endif
// DU = false is the variant for a placeholder U (the reference's own training graph, s_net_bundle_nobm.py:281): no
// accumulator box, no scatter code, fewer registers -> one more CTA per SM.
template <int C, int TW, int K, int NT, bool LOSS, bool DU>
__global__ void __launch_bounds__(NT, DU ? MGW_BWD_MINB : MGW_BWD_NODU_MINB)
warp_bwd_tma_kernel(const __grid_constant__ CUtensorMap mapU, const __grid_constant__ CUtensorMap mapG,
                    const __grid_constant__ CUtensorMap mapGI, const float* __restrict__ U, const float* __restrict__ Hs, const float* __restrict__ d_out,
                    const float* __restrict__ d_img, const __grid_constant__ TileCfg cfg, float* __restrict__ dU,
                    float* __restrict__ parts, const LossBwd loss)
{
    using G = Geo<C, TW, K, NT>;
    extern __shared__ __align__(1024) unsigned char smem_raw[];
    float* s_src = reinterpret_cast<float*>(smem_raw);
    float* s_red = s_src + G::kBoxF;                                   // [warps][8] dH partials (<= 128 floats)
    uint64_t* bar = reinterpret_cast<uint64_t*>(s_red + 128);
    TileInfo* ti = reinterpret_cast<TileInfo*>(bar + 2);
    int* s_acc = reinterpret_cast<int*>(s_red + 256);                  // fixed-point dU box (only when dU != nullptr)

    // STAGE: the tile's d_out / d_img arrive by TMA too, into the (not yet zeroed) accumulator box, and every thread picks its
    // pixels up from shared memory (12-byte lane stride: conflict free).  As 24 LDGs per thread with a 12-byte lane stride
    // (three lines per request) they queued in the LSU for ~3500 cycles next to the other CTAs' shared-memory traffic and
    // the CTA spent more than half of its life before its first pixel.
    constexpr bool STAGE = DU && !LOSS && (G::kBoxF >= G::TH * TW * (C + 2));
    constexpr int kStageOut = G::TH * TW * C;         // floats of the staged d_out tile; the d_img tile follows it
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
#ifdef MGW_PROBE
    long long tprev = clock64();
    if (tid == MGW_PROBE_TID) atomicAdd(&g_probe[15], 1ull);
#endif
    if (tid == 0) {
        tma::mbar_init(bar, 1);
        if (STAGE) tma::mbar_init(bar + 1, 1);
        tma::fence_barrier_init();
    }
    griddep_launch_dependents();                      // K4 (launched programmatically) may run its factorisation under this kernel
    PROBE(11);     // barrier init
    const Tile tl = this_tile(cfg);
    PROBE(12);     // tile decode
    if (STAGE && tid == 0) {
        float* sg = reinterpret_cast<float*>(s_acc);
        tma::mbar_expect_tx(bar + 1, (uint32_t)((kStageOut + (d_img ? G::TH * TW * 2 : 0)) * sizeof(float)));
        tma::load_3d(sg, &mapG, bar + 1, tl.c0 * C, tl.r0, tl.n);
        if (d_img) tma::load_3d(sg + kStageOut, &mapGI, bar + 1, tl.c0 * 2, tl.r0, tl.n);
    }
    float Hc[9];
#pragma unroll
    for (int k = 0; k < 9; ++k) Hc[k] = __ldg(Hs + (size_t)tl.cell * 9 + k);
    const float stepx = cfg.stepx, stepy = cfg.stepy;
    const int tx = tid % TW, g = tid / TW;
    const int col = tl.c0 + tx;

    // warp 0 issues the TMA load of the source box FIRST, ahead of everybody's gradient loads (24 LDGs per thread that queue in
    // the LSU for ~3500 cycles next to the other CTAs' shared-memory traffic: issued behind them, the box arrived ~4000 cycles
    // after the first barrier).  Thread 0 initialised the barrier itself; everybody else meets it after the __syncthreads below.
    if (tid < 32) {
        int bx0, by0, interior, complete;
        source_box<C, TW, K, NT>(cfg, tl, Hc, stepx, stepy, bx0, by0, interior, &complete);
        if (tid == 0) {
            ti->bx0 = bx0; ti->by0 = by0; ti->interior = complete;      // backward: "interior" = complete
            tma::mbar_expect_tx(bar, (uint32_t)(G::kBoxF * sizeof(float)));
            tma::load_3d(s_src, &mapU, bar, bx0 * C, by0, tl.n);
        }
    }
    // this thread's K pixels of d_out / d_img: 12 / 8 contiguous bytes per lane, coalesced, all loads in flight at once
    PROBE(13);     // Hs loads issued, lin_step
    float gout[K][C], gimg[K][2];
    if (STAGE) {
        __syncthreads();                              // the barriers thread 0 initialised are visible to everybody
        tma::mbar_wait(bar + 1, 0);
        const float* sg = reinterpret_cast<const float*>(s_acc) + (g * K * TW + tx) * C;
        const float2* si = reinterpret_cast<const float2*>(reinterpret_cast<const float*>(s_acc) + kStageOut) + g * K * TW + tx;
#pragma unroll
        for (int k = 0; k < K; ++k) {
#pragma unroll
            for (int ch = 0; ch < C; ++ch) gout[k][ch] = sg[k * TW * C + ch];
            if (d_img) {
                const float2 di = si[k * TW];
                gimg[k][0] = di.x; gimg[k][1] = di.y;
            } else {
                gimg[k][0] = 0.0f; gimg[k][1] = 0.0f;
            }
        }
    } else {
        size_t p = ((size_t)tl.n * cfg.H + tl.r0 + g * K) * cfg.W + col;
        const float kn = LOSS ? (loss.kscale_dev ? loss.kscale * __ldg(loss.kscale_dev) : loss.kscale) / (__ldg(loss.sums + 2 * tl.n + 1) + 1e-8f) : 0.0f;
#pragma unroll
        for (int k = 0; k < K; ++k, p += cfg.W) {
            if (LOSS) {
                const float nb = 1.0f - __ldg(loss.black + p);
                const float kk = kn * nb * nb;
#pragma unroll
                for (int ch = 0; ch < C; ++ch) {
                    gout[k][ch] = kk * (__ldg(loss.out + p * C + ch) - __ldg(loss.y + p * C + ch));
                    if (d_out) gout[k][ch] += __ldg(d_out + p * C + ch);       // gradient reaching `output` from elsewhere (temp_loss)
                }
            } else {
#pragma unroll
                for (int ch = 0; ch < C; ++ch) gout[k][ch] = __ldg(d_out + p * C + ch);
            }
            if (d_img) {
                const float2 di = __ldg(reinterpret_cast<const float2*>(d_img) + p);
                gimg[k][0] = di.x; gimg[k][1] = di.y;
            } else {
                gimg[k][0] = 0.0f; gimg[k][1] = 0.0f;
            }
        }
    }
    PROBE(0);      // gradients in registers (STAGE) / their loads issued
    // ---- per-tile fixed-point scale from max|d_out| (Inf/NaN anywhere in the tile disables the fixed-point path)
    if (DU) {
        // max over |d_out| as unsigned bit patterns: Inf/NaN (>= 0x7f800000) win the max, one REDUX per warp
        unsigned m = 0u;
#pragma unroll
        for (int k = 0; k < K; ++k)
#pragma unroll
            for (int ch = 0; ch < C; ++ch) m = max(m, (unsigned)__float_as_int(gout[k][ch]) & 0x7fffffffu);
        m = __reduce_max_sync(0xffffffffu, m);
        if (lane == 0) ti->wmax[warp] = __int_as_float((int)m);
    }
    if (DU) {
        if (STAGE) __syncthreads();                   // everybody has taken its gradients out of the box
        int4* a4 = reinterpret_cast<int4*>(s_acc);
#pragma unroll
        for (int i = 0; i < (G::kBoxF / 4 + NT - 1) / NT; ++i)
            if (i * NT + tid < G::kBoxF / 4) a4[i * NT + tid] = make_int4(0, 0, 0, 0);
    }
    PROBE(1);      // source box / zero / max (includes the wait for the gradient loads)
    __syncthreads();                                  // wmax, box and the zeroed accumulator are visible
    PROBE(2);      // barrier 1
    const int bx0 = ti->bx0, by0 = ti->by0;
    int fixed = 0;
    float scale = 0.0f, inv_scale = 0.0f;
    if (DU) {
        unsigned mb = 0u;
#pragma unroll
        for (int w = 0; w < NT / 32; ++w) mb = max(mb, (unsigned)__float_as_int(ti->wmax[w]));
        const float mm = __int_as_float((int)mb);
        const int e = (int)(mb >> 23) - 127;                                // floor(log2 mm) for normal mm; 128 for Inf/NaN
        // |w*g*scale| < 2^kBits per term before rounding (tap weights are in [0,1] on this path), but fixed_of() rounds to
        // nearest, so a term can reach 2^kBits exactly.  A pixel adds at most ONE term to a word (its four taps are four
        // different pixels), so a word receives at most kTerms = TH*TW terms: with kBits = 31 - bit_width(kTerms), i.e.
        // 30 - floor(log2 kTerms), their sum stays below 2^31 whatever the map does (no magnification heuristic).  Each term
        // is exact to 2^-kBits of the tile's max|d_out| (2^-20 for the 64 x 24 tile: a millionth, against a 1e-4 tolerance)
        constexpr int kTerms = G::TH * TW;
        constexpr int kBits = 31 - bit_width(kTerms);
        // (never more than 22: fixed_of()'s magic-number rounding holds |v| <= 2^22)
        static_assert(kBits <= 22 && ((long long)kTerms << kBits) < (1LL << 31), "fixed-point headroom");
        fixed = (mm > 0.0f) && (e > -100) && (e < 100);
        scale = __int_as_float((kBits - 1 - e + 127) << 23);
        inv_scale = __int_as_float((e - (kBits - 1) + 127) << 23);
    }

    const float xt = lin_at(col, stepx);
    const float hx0 = __fmul_rn(Hc[0], xt), hx3 = __fmul_rn(Hc[3], xt), hx6 = __fmul_rn(Hc[6], xt);
    float dh[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) dh[k] = 0.0f;
    const float halfW = 0.5f * (float)cfg.W, halfH = 0.5f * (float)cfg.H;

    PROBE(3);
    tma::mbar_wait(bar, 0);
    PROBE(4);      // wait for the TMA box
    if (ti->interior && (fixed || !DU)) {
        // ---- fast path: every UNCLIPPED tap lies inside the box; shared-memory offsets are compile-time constants.
        // A pixel with a clipped tap (its sample point is outside the image) contributes nothing but its d_img term: clipping
        // collapses a tap pair onto one pixel with weights that are exact negatives (mgw_device.cuh, taps_scatter), so its
        // dU terms cancel and gx = sum_c g_c (Ic-Ia)(ay+by) = 0, gy likewise -- the reference keeps only the rounding residue
        // of those cancellations (~1e-8 relative), far below the gradient tolerance.  Border tiles therefore run this loop
        // too, with the gather / scatter of such pixels predicated off, instead of the general per-tap loop below.
#pragma unroll
        for (int k = 0; k < K; ++k) {
            const int row = tl.r0 + g * K + k;
            if (row >= tl.vr0 && col >= tl.vc0) {
                const float yt = lin_at(row, stepy);
                const float xs = __fadd_rn(__fmaf_rn(Hc[1], yt, hx0), Hc[2]);
                const float ys = __fadd_rn(__fmaf_rn(Hc[4], yt, hx3), Hc[5]);
                float zs = __fadd_rn(__fmaf_rn(Hc[7], yt, hx6), Hc[8]);
                zs = __fadd_rn(zs, (zs >= 0.0f) ? 1e-8f : -1e-8f);
                float xn, yn;
                const float rz = div2_rn(xs, ys, zs, xn, yn);
                const FastTaps t = make_taps_interior(xn, yn, cfg.H, cfg.W);
                float gx = 0.0f, gy = 0.0f;
                if ((unsigned)t.x0 < (unsigned)(cfg.W - 1) && (unsigned)t.y0 < (unsigned)(cfg.H - 1)) {      // no tap clipped
                    const int ia = ((t.y0 - by0) * G::kRowF + (t.x0 - bx0) * C);
                    const float* pa = s_src + ia;
                    int* qa = s_acc + ia;
                    const float wa = t.ax * t.ay, wb = t.ax * t.by, wc = t.bx * t.ay, wd = t.bx * t.by;
                    // gx = sum_c g_c [(Ic-Ia) ay + (Id-Ib) by], gy = sum_c g_c [(Ib-Ia) ax + (Id-Ic) bx], with the channel sums
                    // taken per tap first (4 FMAs per channel instead of 10 operations)
                    float sa = 0.0f, sb = 0.0f, sc = 0.0f, sd = 0.0f;
#pragma unroll
                    for (int ch = 0; ch < C; ++ch) {
                        const float gch = gout[k][ch];
                        sa = fmaf(gch, pa[ch], sa); sb = fmaf(gch, pa[G::kRowF + ch], sb);
                        sc = fmaf(gch, pa[C + ch], sc); sd = fmaf(gch, pa[G::kRowF + C + ch], sd);
                        if (DU) {
                            const float gs = gch * scale;
                            atomicAdd(qa + ch, fixed_of(wa, gs));
                            atomicAdd(qa + G::kRowF + ch, fixed_of(wb, gs));
                            atomicAdd(qa + C + ch, fixed_of(wc, gs));
                            atomicAdd(qa + G::kRowF + C + ch, fixed_of(wd, gs));
                        }
                    }
                    gx = fmaf(sc - sa, t.ay, (sd - sb) * t.by); gy = fmaf(sb - sa, t.ax, (sd - sc) * t.bx);
                }
                accumulate_dh_r(dh, fmaf(gx, halfW, gimg[k][0]), fmaf(gy, halfH, gimg[k][1]), xn, yn, rz, xt, yt);
            }
        }
    } else {
        if (DU) griddep_wait();                       // this path adds to dU from inside the loop: the zero-fill before us must be complete
        const float* Un = U + (size_t)tl.n * cfg.H * cfg.W * C;
        float* dUn = DU ? dU + (size_t)tl.n * cfg.H * cfg.W * C : nullptr;
#pragma unroll
        for (int k = 0; k < K; ++k) {
            const int row = tl.r0 + g * K + k;
            if (row >= tl.vr0 && col >= tl.vc0) {
                const float yt = lin_at(row, stepy);
                const float xs = __fadd_rn(__fmaf_rn(Hc[1], yt, hx0), Hc[2]);
                const float ys = __fadd_rn(__fmaf_rn(Hc[4], yt, hx3), Hc[5]);
                float zs = __fadd_rn(__fmaf_rn(Hc[7], yt, hx6), Hc[8]);
                zs = __fadd_rn(zs, (zs >= 0.0f) ? 1e-8f : -1e-8f);
                const float xn = __fdiv_rn(xs, zs), yn = __fdiv_rn(ys, zs);
                const Taps t = make_taps(xn, yn, cfg.H, cfg.W);
                const int sx0 = t.x0 - bx0, sx1 = t.x1 - bx0, sy0 = t.y0 - by0, sy1 = t.y1 - by0;
                const bool inbox = sx0 >= 0 && sx1 < G::SBW && sy0 >= 0 && sy1 < G::SBH;
                const float wa = t.ax * t.ay, wb = t.ax * t.by, wc = t.bx * t.ay, wd = t.bx * t.by;
                float gx = 0.0f, gy = 0.0f;
                const bool scatter = DU && taps_scatter(t);
                const size_t ga = ((size_t)t.y0 * cfg.W + t.x0) * C, gb = ((size_t)t.y1 * cfg.W + t.x0) * C;
                const size_t gc = ((size_t)t.y0 * cfg.W + t.x1) * C, gd = ((size_t)t.y1 * cfg.W + t.x1) * C;
                const int ia = sy0 * G::kRowF + sx0 * C, ib = sy1 * G::kRowF + sx0 * C;
                const int ic = sy0 * G::kRowF + sx1 * C, id = sy1 * G::kRowF + sx1 * C;
#pragma unroll
                for (int ch = 0; ch < C; ++ch) {
                    const float gch = gout[k][ch];
                    float Ia, Ib, Ic, Id;
                    if (inbox) { Ia = s_src[ia + ch]; Ib = s_src[ib + ch]; Ic = s_src[ic + ch]; Id = s_src[id + ch]; }
                    else { Ia = __ldg(Un + ga + ch); Ib = __ldg(Un + gb + ch); Ic = __ldg(Un + gc + ch); Id = __ldg(Un + gd + ch); }
                    gx = fmaf(gch, fmaf(Ic - Ia, t.ay, (Id - Ib) * t.by), gx);
                    gy = fmaf(gch, fmaf(Ib - Ia, t.ax, (Id - Ic) * t.bx), gy);
                    if (scatter) {
                        if (inbox && fixed) {      // unclipped taps have weights in [0,1], so |w*g| <= max|d_out|
                            const float gs = gch * scale;
                            atomicAdd(s_acc + ia + ch, fixed_of(wa, gs));
                            atomicAdd(s_acc + ib + ch, fixed_of(wb, gs));
                            atomicAdd(s_acc + ic + ch, fixed_of(wc, gs));
                            atomicAdd(s_acc + id + ch, fixed_of(wd, gs));
                        } else {
                            atomicAdd(dUn + ga + ch, wa * gch);
                            atomicAdd(dUn + gb + ch, wb * gch);
                            atomicAdd(dUn + gc + ch, wc * gch);
                            atomicAdd(dUn + gd + ch, wd * gch);
                        }
                    }
                }
                accumulate_dh(dh, fmaf(gx, halfW, gimg[k][0]), fmaf(gy, halfH, gimg[k][1]), xn, yn, zs, xt, yt);
            }
        }
    }
    PROBE(5);      // pixel loop
    // dH: halving butterfly (9 shuffles for the 8 sums instead of 40) -> shared -> one partial per tile.
    // After the three halving steps lane l holds term (l>>2)&7 summed over the lanes that share l's low two bits ... the
    // last two steps finish the sum, so lanes 0,4,..,28 hold terms 0..7.
    {
        float v4[4], v2[2], v1;
        const bool hi16 = lane & 16, hi8 = lane & 8, hi4 = lane & 4;
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const float send = hi16 ? dh[i] : dh[i + 4], keep = hi16 ? dh[i + 4] : dh[i];
            v4[i] = keep + __shfl_xor_sync(0xffffffffu, send, 16);
        }
#pragma unroll
        for (int i = 0; i < 2; ++i) {
            const float send = hi8 ? v4[i] : v4[i + 2], keep = hi8 ? v4[i + 2] : v4[i];
            v2[i] = keep + __shfl_xor_sync(0xffffffffu, send, 8);
        }
        {
            const float send = hi4 ? v2[0] : v2[1], keep = hi4 ? v2[1] : v2[0];
            v1 = keep + __shfl_xor_sync(0xffffffffu, send, 4);
        }
        v1 += __shfl_xor_sync(0xffffffffu, v1, 2);
        v1 += __shfl_xor_sync(0xffffffffu, v1, 1);
        // lane l now holds term  4*bit4(l) + 2*bit3(l) + bit2(l)
        if ((lane & 3) == 0) s_red[warp * 8 + ((lane >> 4) & 1) * 4 + ((lane >> 3) & 1) * 2 + ((lane >> 2) & 1)] = v1;
    }
    PROBE(6);      // dH shuffles
    __syncthreads();                                  // also orders every shared atomic before the drain below
    PROBE(7);      // barrier 2
    if (tid < 8) {
        float v = 0.0f;
#pragma unroll
        for (int w = 0; w < NT / 32; ++w) v += s_red[w * 8 + tid];
        parts[((size_t)tl.cell * (cfg.parts_y * cfg.parts_x) + tl.part) * 8 + tid] = v;
    }
    if (fixed) {
        // Launched programmatically behind the zero-fill of dU (mgw_capi.cu), this kernel has run up to here NEXT TO it: nothing
        // above reads or writes dU.  From here on the fill must be complete and visible (a no-op under a plain launch).
        griddep_wait();
        // fixed point -> fp32 straight from the accumulator into dU by 16-byte reductions (red.global.add.v4.f32, fire and
        // forget through the LSU): no conversion back into shared memory, no proxy fence, no third barrier, and nothing of this
        // CTA waits in the SM's TMA unit in front of the next CTA's box load
        const int4* a4 = reinterpret_cast<const int4*>(s_acc);
        constexpr int kQ = G::kRowF / 4;                                   // 16-byte groups per box row
        const int rows = min(G::SBH, cfg.H - by0);                           // the part of the box inside the image
        const int nq = min(G::kRowF, (cfg.W - bx0) * C) / 4;                 // ((W - bx0) * C is a multiple of 4 floats)
        float* base = dU + (((size_t)tl.n * cfg.H + by0) * cfg.W + bx0) * C;
        const int pitch = cfg.W * C;
#pragma unroll
        for (int i = 0; i < (G::kBoxF / 4 + NT - 1) / NT; ++i) {
            const int j = i * NT + tid;
            const int row = j / kQ, q = j % kQ;
            if (row < rows && q < nq) {
                const int4 v = a4[j];
                if ((v.x | v.y | v.z | v.w) != 0)      // most of the box outside the tile's own footprint received nothing: no traffic for +0
                    tma::red_add_v4(base + row * pitch + q * 4, float_of_fixed(v.x) * inv_scale, float_of_fixed(v.y) * inv_scale,
                                    float_of_fixed(v.z) * inv_scale, float_of_fixed(v.w) * inv_scale);
            }
        }
        PROBE(8);
    }
}

struct Plan {
    TileCfg cfg;
    int TW, K, NT, TH, nty, ntx;
};

// compiled (TW, K, threads) variants: TH = K * threads/TW
constexpr int kNumVariants = 6;
static const int kVariants[kNumVariants][3] = {{64, 6, 256}, {64, 3, 512}, {64, 3, 256}, {32, 3, 256}, {32, 2, 256}, {32, 1, 256}};

// Picks the tiling for a shape; false if the TMA path cannot serve it (the generic kernels then do).
static bool plan(const WarpShape& s, Plan* out)
{
    if (s.OH != s.H || s.OW != s.W) return false;
    if (s.C != 1 && s.C != 3 && s.C != 4) return false;
    if (s.H > 65535 || s.W > 65535 || s.gh > 255 || s.gw > 255 || s.N > 65535) return false;
    // tiles start at cell boundaries (or cell end - TW) and every TMA start address must be 16-byte aligned for
    // out (C floats/px): columns of cell boundaries must be multiples of 4
    const int cell_h = s.H / s.gh, cell_w = s.W / s.gw;
    if (s.W % 4 != 0 || cell_w % 4 != 0) return false;
    double best_eff = 0;
    int best = -1;
    for (int v = 0; v < kNumVariants; ++v) {
        const int tw = kVariants[v][0], k = kVariants[v][1], th = (kVariants[v][2] / tw) * k;
        if (tw > cell_w || th > cell_h) continue;
        if (s.C == 4 && tw == 64) continue;                      // 64 px x 4 ch leaves no room for a halo in a 256-element box
        const double ey = (double)cell_h / (((cell_h + th - 1) / th) * th), ex = (double)cell_w / (((cell_w + tw - 1) / tw) * tw);
        const double eff = ey * ex * (tw == 64 ? 1.0 : 0.93) * (th >= 12 ? 1.0 : 0.9);      // larger tiles amortise the halo
        if (eff > best_eff) { best_eff = eff; best = v; }
    }
    if (const char* force = getenv("MGW_TILE")) {                  // tuning aid: MGW_TILE=64x3 forces a compiled variant if it fits
        int tw = 0, k = 0, nt = 256;
        if (sscanf(force, "%dx%dx%d", &tw, &k, &nt) >= 2)
            for (int v = 0; v < kNumVariants; ++v)
                if (kVariants[v][0] == tw && kVariants[v][1] == k && kVariants[v][2] == nt && tw <= cell_w && (nt / tw) * k <= cell_h &&
                    !(s.C == 4 && tw == 64)) best = v;
    }
    if (best < 0) return false;
    Plan p;
    p.TW = kVariants[best][0]; p.K = kVariants[best][1]; p.NT = kVariants[best][2]; p.TH = (p.NT / p.TW) * p.K;
    TileCfg& c = p.cfg;
    c.N = s.N; c.H = s.H; c.W = s.W; c.gh = s.gh; c.gw = s.gw;
    tile_steps(&c);
    p.nty = fill_axis(&c.rows, s.gh, cell_h, s.H, p.TH, &c.parts_y);
    p.ntx = fill_axis(&c.cols, s.gw, cell_w, s.W, p.TW, &c.parts_x);
    if (p.nty < 0 || p.ntx < 0 || c.parts_y > 255 || c.parts_x > 255) return false;
    *out = p;
    return true;
}

bool tma_fwd_supported(const WarpShape& s) { Plan p; return plan(s, &p); }
bool tma_bwd_supported(const WarpShape& s) { Plan p; return plan(s, &p); }

size_t tma_bwd_workspace_bytes(const WarpShape& s)
{
    Plan p;
    if (!plan(s, &p)) return 0;
    return (size_t)s.N * s.gh * s.gw * p.cfg.parts_y * p.cfg.parts_x * 8 * sizeof(float);
}

template <int C, int TW, int K, int NT>
static int launch_fwd_v(const float* U, const float* Hs, const Plan& p, float* out, float* black, float* img, const float* y_tgt,
                        float* sums, cudaStream_t st)
{
    using G = Geo<C, TW, K, NT>;
    const TileCfg& c = p.cfg;
    CUtensorMap mU, mOut;
    TRY_RC(make_map(&mU, U, c.W * C, c.H, c.N, G::kRowF, G::SBH));
    TRY_RC(make_map(&mOut, out ? out : U, c.W * C, c.H, c.N, TW * C, G::TH));
    const size_t smem = (size_t)(G::kBoxF + G::kOutF) * 4 + 16 + sizeof(TileInfo) + 2 * kMaxWarps * 4 + 64;
    if (y_tgt) {
        static bool attr_l[64] = {};
        TRY_RC(allow_smem(warp_fwd_tma_kernel<C, TW, K, NT, true>, attr_l, "warp_fwd_tma(loss)"));
        warp_fwd_tma_kernel<C, TW, K, NT, true><<<dim3(p.ntx, p.nty, c.N), NT, smem, st>>>(mU, mOut, U, Hs, c, out, img, black, y_tgt, sums);
        return check_launch("warp_fwd_tma(loss)");
    }
    static bool attr[64] = {};
    TRY_RC(allow_smem(warp_fwd_tma_kernel<C, TW, K, NT, false>, attr, "warp_fwd_tma"));
    warp_fwd_tma_kernel<C, TW, K, NT, false><<<dim3(p.ntx, p.nty, c.N), NT, smem, st>>>(mU, mOut, U, Hs, c, out, img, black, nullptr, nullptr);
    return check_launch("warp_fwd_tma");
}

template <int C, int TW, int K, int NT>
static int launch_bwd_v(const float* U, const float* Hs, const float* d_out, const float* d_img, const Plan& p, float* dU,
                        float* parts, const LossBwd* loss, cudaStream_t st, bool behind_own_fill)
{
    using G = Geo<C, TW, K, NT>;
    const TileCfg& c = p.cfg;
    CUtensorMap mU;
    TRY_RC(make_map(&mU, U, c.W * C, c.H, c.N, G::kRowF, G::SBH));
    CUtensorMap mG = mU, mGI = mU;                  // staged d_out / d_img tiles (plain backward with dU only)
    if (dU && !loss) {
        TRY_RC(make_map(&mG, d_out, c.W * C, c.H, c.N, TW * C, G::TH));
        if (d_img) TRY_RC(make_map(&mGI, d_img, c.W * 2, c.H, c.N, TW * 2, G::TH));
    }
    size_t smem = (size_t)(G::kBoxF + 256 + (dU ? G::kBoxF : 0)) * 4 + 64;
    if (const char* e = getenv("MGW_BWD_PAD_SMEM")) smem += (size_t)atoi(e);      // tuning aid: fewer CTAs per SM (occupancy experiments)
    const dim3 grid(p.ntx, p.nty, c.N);
    if (loss && dU) {
        static bool attr[64] = {};
        TRY_RC(allow_smem(warp_bwd_tma_kernel<C, TW, K, NT, true, true>, attr, "warp_bwd_tma(loss)"));
        warp_bwd_tma_kernel<C, TW, K, NT, true, true><<<grid, NT, smem, st>>>(mU, mG, mGI, U, Hs, d_out, d_img, c, dU, parts, *loss);
    } else if (loss) {
        static bool attr[64] = {};
        TRY_RC(allow_smem(warp_bwd_tma_kernel<C, TW, K, NT, true, false>, attr, "warp_bwd_tma(loss, no dU)"));
        warp_bwd_tma_kernel<C, TW, K, NT, true, false><<<grid, NT, smem, st>>>(mU, mG, mGI, U, Hs, d_out, d_img, c, nullptr, parts, *loss);
    } else if (dU) {
        static bool attr[64] = {};
        TRY_RC(allow_smem(warp_bwd_tma_kernel<C, TW, K, NT, false, true>, attr, "warp_bwd_tma"));
        const cudaError_t e = launch_ex(warp_bwd_tma_kernel<C, TW, K, NT, false, true>, grid, dim3(NT), smem, st, behind_own_fill && pdl_enabled(),
                                        mU, mG, mGI, U, Hs, d_out, d_img, c, dU, parts, LossBwd{});
        if (e != cudaSuccess) { count_launches(1); return set_error(MGW_ERR_CUDA, "warp_bwd_tma: %s", cudaGetErrorString(e)); }
    } else {
        static bool attr[64] = {};
        TRY_RC(allow_smem(warp_bwd_tma_kernel<C, TW, K, NT, false, false>, attr, "warp_bwd_tma(no dU)"));
        warp_bwd_tma_kernel<C, TW, K, NT, false, false><<<grid, NT, smem, st>>>(mU, mG, mGI, U, Hs, d_out, d_img, c, nullptr, parts, LossBwd{});
    }
    return check_launch("warp_bwd_tma");
}

template <int C>
static int launch_fwd_c(const Plan& p, const float* U, const float* Hs, float* out, float* black, float* img, const float* y_tgt,
                        float* sums, cudaStream_t st)
{
    if (p.NT == 256 && p.TW == 32 && p.K == 3) return launch_fwd_v<C, 32, 3, 256>(U, Hs, p, out, black, img, y_tgt, sums, st);
    if (p.NT == 256 && p.TW == 32 && p.K == 2) return launch_fwd_v<C, 32, 2, 256>(U, Hs, p, out, black, img, y_tgt, sums, st);
    if (p.NT == 256 && p.TW == 32 && p.K == 1) return launch_fwd_v<C, 32, 1, 256>(U, Hs, p, out, black, img, y_tgt, sums, st);
    if constexpr (C != 4) {
        if (p.NT == 256 && p.TW == 64 && p.K == 6) return launch_fwd_v<C, 64, 6, 256>(U, Hs, p, out, black, img, y_tgt, sums, st);
        if (p.NT == 512 && p.TW == 64 && p.K == 3) return launch_fwd_v<C, 64, 3, 512>(U, Hs, p, out, black, img, y_tgt, sums, st);
        if (p.NT == 256 && p.TW == 64 && p.K == 3) return launch_fwd_v<C, 64, 3, 256>(U, Hs, p, out, black, img, y_tgt, sums, st);
    }
    return set_error(MGW_ERR_UNSUPPORTED, "warp_fwd_tma: no tile variant");
}

template <int C>
static int launch_bwd_c(const Plan& p, const float* U, const float* Hs, const float* d_out, const float* d_img, float* dU,
                        float* parts, const LossBwd* loss, cudaStream_t st, bool behind_own_fill)
{
    if (p.NT == 256 && p.TW == 32 && p.K == 3) return launch_bwd_v<C, 32, 3, 256>(U, Hs, d_out, d_img, p, dU, parts, loss, st, behind_own_fill);
    if (p.NT == 256 && p.TW == 32 && p.K == 2) return launch_bwd_v<C, 32, 2, 256>(U, Hs, d_out, d_img, p, dU, parts, loss, st, behind_own_fill);
    if (p.NT == 256 && p.TW == 32 && p.K == 1) return launch_bwd_v<C, 32, 1, 256>(U, Hs, d_out, d_img, p, dU, parts, loss, st, behind_own_fill);
    if constexpr (C != 4) {
        if (p.NT == 256 && p.TW == 64 && p.K == 6) return launch_bwd_v<C, 64, 6, 256>(U, Hs, d_out, d_img, p, dU, parts, loss, st, behind_own_fill);
        if (p.NT == 512 && p.TW == 64 && p.K == 3) return launch_bwd_v<C, 64, 3, 512>(U, Hs, d_out, d_img, p, dU, parts, loss, st, behind_own_fill);
        if (p.NT == 256 && p.TW == 64 && p.K == 3) return launch_bwd_v<C, 64, 3, 256>(U, Hs, d_out, d_img, p, dU, parts, loss, st, behind_own_fill);
    }
    return set_error(MGW_ERR_UNSUPPORTED, "warp_bwd_tma: no tile variant");
}

int launch_warp_fwd_tma(const float* U, const float* Hs, const WarpShape& s, float* out, float* black, float* img,
                        const float* y_tgt, float* sums, cudaStream_t st)
{
    Plan p;
    if (!plan(s, &p)) return set_error(MGW_ERR_UNSUPPORTED, "warp_fwd_tma: unsupported shape");
    if (s.C == 1) return launch_fwd_c<1>(p, U, Hs, out, black, img, y_tgt, sums, st);
    if (s.C == 3) return launch_fwd_c<3>(p, U, Hs, out, black, img, y_tgt, sums, st);
    return launch_fwd_c<4>(p, U, Hs, out, black, img, y_tgt, sums, st);
}

int launch_warp_bwd_tma(const float* U, const float* Hs, const float* d_out, const float* d_img, const WarpShape& s, float* dU,
                        float* parts, int* nparts, const FusedImgLoss* fl, cudaStream_t st, bool behind_own_fill)
{
    LossBwd lb{};
    const LossBwd* loss = nullptr;
    if (fl) { lb.out = fl->out; lb.y = fl->y; lb.black = fl->black; lb.sums = fl->sums; lb.kscale = fl->kscale; lb.kscale_dev = fl->kscale_dev; loss = &lb; }
    Plan p;
    if (!plan(s, &p)) return set_error(MGW_ERR_UNSUPPORTED, "warp_bwd_tma: unsupported shape");
    *nparts = p.cfg.parts_y * p.cfg.parts_x;
    // cells with fewer tiles than parts_y*parts_x leave slots untouched: zero them (a few hundred KB at most).  Every cell of
    // a uniform mesh has the same tiling, i.e. every slot is written by its tile: no zero-fill (one launch less on the
    // critical path between forward and backward).
    const int cell_h = s.H / s.gh, cell_w = s.W / s.gw;
    const bool all_slots_written = (s.H % s.gh == 0) && (s.W % s.gw == 0) && (p.nty == s.gh * ((cell_h + p.TH - 1) / p.TH)) &&
                                   (p.ntx == s.gw * ((cell_w + p.TW - 1) / p.TW));
    if (!all_slots_written && cudaMemsetAsync(parts, 0, tma_bwd_workspace_bytes(s), st) != cudaSuccess)
        return set_error(MGW_ERR_CUDA, "memset parts: %s", cudaGetErrorString(cudaGetLastError()));
    if (!all_slots_written) behind_own_fill = false;          // the memset sits between the fill and us
    if (s.C == 1) return launch_bwd_c<1>(p, U, Hs, d_out, d_img, dU, parts, loss, st, behind_own_fill);
    if (s.C == 3) return launch_bwd_c<3>(p, U, Hs, d_out, d_img, dU, parts, loss, st, behind_own_fill);
    return launch_bwd_c<4>(p, U, Hs, d_out, d_img, dU, parts, loss, st, behind_own_fill);
}

}  // namespace mgw

// extern "C" entry points of libmgw_b200.so (see include/mgw.h): argument validation, workspace carving,
// kernel selection.  No torch types, no hidden allocation, no CPU fallback.
#include <atomic>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>

#include "mgw_internal.h"

namespace mgw {

static thread_local char g_err[512] = "";
static std::atomic<uint64_t> g_launches{0};

int set_error(int code, const char* fmt, ...)
{
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
    return code;
}

void count_launches(int n) { g_launches.fetch_add((uint64_t)n, std::memory_order_relaxed); }

int check_launch(const char* what)
{
    count_launches(1);
    const cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return set_error(MGW_ERR_CUDA, "%s: %s", what, cudaGetErrorString(e));
    return MGW_OK;
}

// Kernel-family override for tests and tuning: environment variable MGW_IMPL = auto | generic | tma | pipe, read at every
// call (there is no setter in the ABI and no state in the library).
int impl_mode()
{
    const char* e = getenv("MGW_IMPL");
    if (!e) return 0;
    switch (e[0]) { case 'g': return 1; case 't': return 2; case 'p': return 3; default: return 0; }
}

bool pdl_enabled()
{
    static const bool on = [] { const char* e = getenv("MGW_PDL"); return !(e && e[0] == '0'); }();
    return on;
}

static bool aligned(const void* p, size_t a) { return (reinterpret_cast<uintptr_t>(p) % a) == 0; }

#define REQUIRE(cond, ...) do { if (!(cond)) return set_error(MGW_ERR_INVALID, __VA_ARGS__); } while (0)
#define TRY(expr) do { const int rc_ = (expr); if (rc_ != MGW_OK) return rc_; } while (0)

static int check_memset(cudaError_t e, const char* what)
{
    if (e != cudaSuccess) return set_error(MGW_ERR_CUDA, "%s: %s", what, cudaGetErrorString(e));
    return MGW_OK;
}

static int validate_mesh_shape(const char* fn, int N, int H, int W, int C, int gh, int gw)
{
    REQUIRE(N > 0 && H > 1 && W > 1 && C > 0, "%s: need N>0, H>1, W>1, C>0 (got N=%d H=%d W=%d C=%d)", fn, N, H, W, C);
    REQUIRE(gh > 0 && gw > 0 && gh <= H && gw <= W, "%s: need 1 <= gh <= H and 1 <= gw <= W (got gh=%d gw=%d)", fn, gh, gw);
    REQUIRE((long long)N * H * W < (1LL << 31), "%s: N*H*W must fit in int32", fn);
    return MGW_OK;
}

// dHs accumulators for the atomic reduction live either in the caller's dHs buffer (zeroed here)
static size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

__global__ void reduce_parts_kernel(const float* __restrict__ parts, int nparts, int ncell, float* __restrict__ dHs)
{
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= ncell * 9) return;
    const int cell = t / 9, k = t % 9;
    double s = 0;
    if (k < 8) for (int p = 0; p < nparts; ++p) s += (double)parts[((size_t)cell * nparts + p) * 8 + k];
    dHs[t] = (float)s;
}

}  // namespace mgw

using namespace mgw;

extern "C" {

int mgw_version(void) { return 102; }

const char* mgw_last_error(void) { return g_err; }

uint64_t mgw_launch_count(void) { return g_launches.load(std::memory_order_relaxed); }

int mgw_vertices_fwd(const float* head, int N, int gh, int gw, float do_crop_rate, float* pts2, float* pts1, void* stream)
{
    REQUIRE(head && pts2, "mgw_vertices_fwd: null pointer");
    REQUIRE(N > 0 && gh > 0 && gw > 0 && do_crop_rate > 0.0f, "mgw_vertices_fwd: bad sizes");
    return launch_vertices_fwd(head, N, gh, gw, do_crop_rate, pts2, pts1, (cudaStream_t)stream);
}

int mgw_vertices_bwd(const float* head, const float* d_pts2, const float* d_pts1, int N, int gh, int gw,
                     float do_crop_rate, float* d_head, void* stream)
{
    REQUIRE(head && d_head, "mgw_vertices_bwd: null pointer");
    REQUIRE(N > 0 && gh > 0 && gw > 0 && do_crop_rate > 0.0f, "mgw_vertices_bwd: bad sizes");
    return launch_vertices_bwd(head, d_pts2, d_pts1, N, gh, gw, do_crop_rate, d_head, (cudaStream_t)stream);
}

int mgw_solve_h_fwd(const float* theta, int N, int gh, int gw, float* Hs, void* stream)
{
    REQUIRE(theta && Hs, "mgw_solve_h_fwd: null pointer");
    REQUIRE(N > 0 && gh > 0 && gw > 0, "mgw_solve_h_fwd: bad sizes");
    return launch_solve_h_fwd(theta, N, gh, gw, Hs, (cudaStream_t)stream);
}

int mgw_solve_h_bwd(const float* theta, const float* Hs, const float* dHs, int N, int gh, int gw, float* dtheta, void* stream)
{
    REQUIRE(theta && Hs && dHs && dtheta, "mgw_solve_h_bwd: null pointer");
    REQUIRE(N > 0 && gh > 0 && gw > 0, "mgw_solve_h_bwd: bad sizes");
    return launch_solve_h_bwd(theta, Hs, dHs, 1, 9, N, gh, gw, dtheta, (cudaStream_t)stream);
}

static bool use_tma_fwd(const WarpShape& s, const float* U, const float* out, const float* black, const float* img, int* rc)
{
    *rc = MGW_OK;
    const int mode = impl_mode();
    if (mode == 1 || mode == 3) return false;
    const bool ok = tma_fwd_supported(s) && aligned(U, 16) && (!out || aligned(out, 16)) && (!black || aligned(black, 16)) &&
                    (!img || aligned(img, 16));
    if (!ok && mode == 2) *rc = set_error(MGW_ERR_UNSUPPORTED, "TMA path required (MGW_IMPL=tma) but shape/alignment does not allow it");
    return ok;
}

// the persistent pipeline serves the full call (warped image + maps + mask); partial calls take the one-tile-per-CTA kernels
static bool use_pipe_fwd(const WarpShape& s, const float* U, const float* out, const float* black, const float* img, int* rc)
{
    *rc = MGW_OK;
    const int mode = impl_mode();
    if (mode == 1 || mode == 2) return false;
    const bool ok = out && black && img && pipe_fwd_supported(s) && aligned(U, 16) && aligned(out, 16) && aligned(black, 16) &&
                    aligned(img, 16);
    if (!ok && mode == 3) *rc = set_error(MGW_ERR_UNSUPPORTED, "pipeline path required (MGW_IMPL=pipe) but shape/alignment does not allow it");
    return ok;
}

int mgw_warp_fwd(const float* U, const float* Hs, int N, int H, int W, int C, int gh, int gw, float* out, float* black,
                 float* img, int32_t* cell_idx, void* stream)
{
    REQUIRE(U && Hs, "mgw_warp_fwd: null pointer");
    TRY(validate_mesh_shape("mgw_warp_fwd", N, H, W, C, gh, gw));
    REQUIRE(!img || aligned(img, 8), "mgw_warp_fwd: img must be 8-byte aligned");
    const WarpShape s{N, H, W, C, H, W, gh, gw};
    cudaStream_t st = (cudaStream_t)stream;
    int rc = MGW_OK;
    if (!cell_idx && use_pipe_fwd(s, U, out, black, img, &rc)) return launch_warp_fwd_pipe(U, Hs, s, out, black, img, st);
    if (rc != MGW_OK) return rc;
    if (!cell_idx && use_tma_fwd(s, U, out, black, img, &rc)) return launch_warp_fwd_tma(U, Hs, s, out, black, img, nullptr, nullptr, st);
    if (rc != MGW_OK) return rc;
    return launch_warp_fwd_generic(U, Hs, s, false, out, black, img, cell_idx, st);
}

size_t mgw_warp_bwd_workspace_bytes(int N, int H, int W, int C, int gh, int gw)
{
    return tma_bwd_workspace_bytes(WarpShape{N, H, W, C, H, W, gh, gw});      // 0 when the tile kernels cannot serve the shape
}

// shared by mgw_warp_bwd and mgw_mesh_warp_bwd: produces dH partials; returns their layout
static int warp_bwd_core(const float* U, const float* Hs, const float* d_out, const float* d_img, const WarpShape& s,
                         float* dU, float* dHs_acc /*[cells,9]*/, void* workspace, const float** parts, int* nparts,
                         int* part_stride, cudaStream_t st, const FusedImgLoss* fl = nullptr, float* d_out_scratch = nullptr,
                         bool zero_dU = true)
{
    const size_t ncell = (size_t)s.N * s.gh * s.gw;
    const int mode = impl_mode();
    // the one-tile-per-CTA kernels serve every backward they can take (MGW_IMPL=tma and =pipe: or fail), the generic kernels the rest
    const bool tma_ok = mode != 1 && workspace && tma_bwd_supported(s) && aligned(U, 16) && (!dU || aligned(dU, 16)) &&
                        (!d_img || aligned(d_img, 8));
    bool own_fill = false;          // the tile backward then runs NEXT TO the fill up to its first access to dU (programmatic launch)
    if (dU && zero_dU) {
        // the library's own fill (evict_last: the lines are still in L2 when the reductions arrive) where its 16-byte granularity
        // fits, the driver's memset otherwise (odd sizes only occur on the generic path)
        const size_t bytes = sizeof(float) * (size_t)s.N * s.H * s.W * s.C;
        if (bytes % 16 == 0 && aligned(dU, 16)) { TRY(launch_fill_zero(dU, bytes, true, st)); own_fill = true; }
        else TRY(check_memset(cudaMemsetAsync(dU, 0, bytes, st), "memset dU"));
    }
    if (!tma_ok && mode >= 2)
        return set_error(MGW_ERR_UNSUPPORTED, "TMA path required (MGW_IMPL=tma|pipe) but shape/alignment/workspace does not allow it");
    if (tma_ok) {
        int np = 0;
        TRY(launch_warp_bwd_tma(U, Hs, d_out, d_img, s, dU, (float*)workspace, &np, fl, st, own_fill));
        *parts = (const float*)workspace; *nparts = np; *part_stride = 8;
        return MGW_OK;
    }
    TRY(check_memset(cudaMemsetAsync(dHs_acc, 0, sizeof(float) * ncell * 9, st), "memset dHs"));
    if (fl) {       // generic path: materialise d_out of the fused loss first
        if (!d_out_scratch) return set_error(MGW_ERR_INVALID, "fused img_loss backward: workspace too small for the generic path");
        TRY(launch_img_loss_bwd(fl->out, fl->y, fl->black, fl->sums, fl->kscale * 0.5f * (float)s.N, fl->kscale_dev, s.N, s.H, s.W, s.C, d_out_scratch, st,
                                d_out /* a second gradient on `output`, nullable */));
        d_out = d_out_scratch;
    }
    TRY(launch_warp_bwd_generic(U, Hs, d_out, d_img, s, false, dU, dHs_acc, st));
    *parts = dHs_acc; *nparts = 1; *part_stride = 9;
    return MGW_OK;
}

static int warp_bwd_impl(const float* U, const float* Hs, const float* d_out, const float* d_img, int N, int H, int W, int C,
                         int gh, int gw, float* dU, float* dHs, void* workspace, void* stream, bool zero_dU)
{
    REQUIRE(U && Hs && d_out, "mgw_warp_bwd: null pointer");
    REQUIRE(dHs || (workspace && impl_mode() != 1 && tma_bwd_supported(WarpShape{N, H, W, C, H, W, gh, gw})),
            "mgw_warp_bwd: dHs may only be NULL when a tile family serves the shape (the per-tile partials then stay in the workspace)");
    TRY(validate_mesh_shape("mgw_warp_bwd", N, H, W, C, gh, gw));
    REQUIRE(!d_img || aligned(d_img, 8), "mgw_warp_bwd: d_img must be 8-byte aligned");
    const WarpShape s{N, H, W, C, H, W, gh, gw};
    cudaStream_t st = (cudaStream_t)stream;
    const float* parts; int np, ps;
    TRY(warp_bwd_core(U, Hs, d_out, d_img, s, dU, dHs, workspace, &parts, &np, &ps, st, nullptr, nullptr, zero_dU));
    if (parts != dHs && dHs) {                    // dHs == NULL: the per-tile partials stay in the workspace (kernel timing)
        const int ncell = N * gh * gw;
        reduce_parts_kernel<<<(ncell * 9 + 127) / 128, 128, 0, st>>>(parts, np, ncell, dHs);
        TRY(check_launch("reduce_parts"));
    }
    return MGW_OK;
}

int mgw_warp_bwd(const float* U, const float* Hs, const float* d_out, const float* d_img, int N, int H, int W, int C,
                 int gh, int gw, float* dU, float* dHs, void* workspace, void* stream)
{
    return warp_bwd_impl(U, Hs, d_out, d_img, N, H, W, C, gh, gw, dU, dHs, workspace, stream, true);
}

int mgw_warp_bwd_acc(const float* U, const float* Hs, const float* d_out, const float* d_img, int N, int H, int W, int C,
                     int gh, int gw, float* dU, float* dHs, void* workspace, void* stream)
{
    return warp_bwd_impl(U, Hs, d_out, d_img, N, H, W, C, gh, gw, dU, dHs, workspace, stream, false);
}

int mgw_mesh_warp_fwd(const float* U, const float* theta, int N, int H, int W, int C, int gh, int gw, float* Hs,
                      float* out, float* black, float* img, void* stream)
{
    REQUIRE(U && theta && Hs, "mgw_mesh_warp_fwd: null pointer");
    TRY(validate_mesh_shape("mgw_mesh_warp_fwd", N, H, W, C, gh, gw));
    TRY(launch_solve_h_fwd(theta, N, gh, gw, Hs, (cudaStream_t)stream));
    return mgw_warp_fwd(U, Hs, N, H, W, C, gh, gw, out, black, img, nullptr, stream);
}

size_t mgw_mesh_warp_bwd_workspace_bytes(int N, int H, int W, int C, int gh, int gw)
{
    return align_up(sizeof(float) * (size_t)N * gh * gw * 9, 256) + mgw_warp_bwd_workspace_bytes(N, H, W, C, gh, gw);
}

static int mesh_warp_bwd_impl(const float* U, const float* theta, const float* Hs, const float* d_out, const float* d_img,
                              int N, int H, int W, int C, int gh, int gw, float* dU, float* dtheta, void* workspace, void* stream,
                              bool zero_dU)
{
    REQUIRE(U && theta && Hs && d_out && dtheta && workspace, "mgw_mesh_warp_bwd: null pointer");
    TRY(validate_mesh_shape("mgw_mesh_warp_bwd", N, H, W, C, gh, gw));
    REQUIRE(aligned(workspace, 256), "mgw_mesh_warp_bwd: workspace must be 256-byte aligned");
    const WarpShape s{N, H, W, C, H, W, gh, gw};
    cudaStream_t st = (cudaStream_t)stream;
    float* dHs_acc = (float*)workspace;
    const size_t off = align_up(sizeof(float) * (size_t)N * gh * gw * 9, 256);
    void* tma_ws = mgw_warp_bwd_workspace_bytes(N, H, W, C, gh, gw) ? (void*)((char*)workspace + off) : nullptr;
    const float* parts; int np, ps;
    TRY(warp_bwd_core(U, Hs, d_out, d_img, s, dU, dHs_acc, tma_ws, &parts, &np, &ps, st, nullptr, nullptr, zero_dU));
    return launch_solve_h_bwd(theta, Hs, parts, np, ps, N, gh, gw, dtheta, st, ps == 8);
}

int mgw_mesh_warp_bwd(const float* U, const float* theta, const float* Hs, const float* d_out, const float* d_img,
                      int N, int H, int W, int C, int gh, int gw, float* dU, float* dtheta, void* workspace, void* stream)
{
    return mesh_warp_bwd_impl(U, theta, Hs, d_out, d_img, N, H, W, C, gh, gw, dU, dtheta, workspace, stream, true);
}

int mgw_mesh_warp_bwd_acc(const float* U, const float* theta, const float* Hs, const float* d_out, const float* d_img,
                          int N, int H, int W, int C, int gh, int gw, float* dU, float* dtheta, void* workspace, void* stream)
{
    return mesh_warp_bwd_impl(U, theta, Hs, d_out, d_img, N, H, W, C, gh, gw, dU, dtheta, workspace, stream, false);
}

int mgw_mesh_warp_img_loss_fwd(const float* U, const float* theta, const float* y, int N, int H, int W, int C, int gh, int gw,
                               float* Hs, float* out, float* black, float* img, float* sums, void* stream)
{
    REQUIRE(U && theta && y && Hs && out && black && sums, "mgw_mesh_warp_img_loss_fwd: null pointer");
    TRY(validate_mesh_shape("mgw_mesh_warp_img_loss_fwd", N, H, W, C, gh, gw));
    REQUIRE(!img || aligned(img, 8), "mgw_mesh_warp_img_loss_fwd: img must be 8-byte aligned");
    cudaStream_t st = (cudaStream_t)stream;
    const WarpShape s{N, H, W, C, H, W, gh, gw};
    TRY(launch_solve_h_fwd(theta, N, gh, gw, Hs, st));
    int rc = MGW_OK;
    if (use_tma_fwd(s, U, out, black, img, &rc)) {
        TRY(check_memset(cudaMemsetAsync(sums, 0, sizeof(float) * 2 * N, st), "memset sums"));
        return launch_warp_fwd_tma(U, Hs, s, out, black, img, y, sums, st);
    }
    if (rc != MGW_OK) return rc;
    TRY(launch_warp_fwd_generic(U, Hs, s, false, out, black, img, nullptr, st));
    return launch_img_loss_fwd(out, y, black, N, H, W, C, sums, st);
}

size_t mgw_mesh_warp_img_loss_bwd_workspace_bytes(int N, int H, int W, int C, int gh, int gw)
{
    // worst case, whatever kernel family ends up serving the call: the generic family materialises d_out in the scratch part.
    // (The size must not depend on anything that can change between this query and the call.)
    const size_t base = mgw_mesh_warp_bwd_workspace_bytes(N, H, W, C, gh, gw);
    return align_up(base, 256) + sizeof(float) * (size_t)N * H * W * C;
}

int mgw_mesh_warp_img_loss_bwd(const float* U, const float* theta, const float* Hs, const float* out, const float* y,
                               const float* black, const float* sums, float upstream, const float* upstream_dev, float batch, const float* d_img,
                               const float* d_out_extra, int N, int H, int W, int C, int gh, int gw, float* dU, float* dtheta,
                               void* workspace, void* stream)
{
    REQUIRE(U && theta && Hs && out && y && black && sums && dtheta && workspace, "mgw_mesh_warp_img_loss_bwd: null pointer");
    TRY(validate_mesh_shape("mgw_mesh_warp_img_loss_bwd", N, H, W, C, gh, gw));
    REQUIRE(aligned(workspace, 256) && batch > 0.0f, "mgw_mesh_warp_img_loss_bwd: workspace must be 256-byte aligned, batch > 0");
    const WarpShape s{N, H, W, C, H, W, gh, gw};
    cudaStream_t st = (cudaStream_t)stream;
    float* dHs_acc = (float*)workspace;
    const size_t off = align_up(sizeof(float) * (size_t)N * gh * gw * 9, 256);
    const size_t tma_bytes = mgw_warp_bwd_workspace_bytes(N, H, W, C, gh, gw);
    void* tma_ws = tma_bytes ? (void*)((char*)workspace + off) : nullptr;
    const size_t base = align_up(mgw_mesh_warp_bwd_workspace_bytes(N, H, W, C, gh, gw), 256);
    float* scratch = (float*)((char*)workspace + base);
    const FusedImgLoss fl{out, y, black, sums, upstream * 2.0f / batch, upstream_dev};
    const float* parts; int np, ps;
    TRY(warp_bwd_core(U, Hs, d_out_extra, d_img, s, dU, dHs_acc, tma_ws, &parts, &np, &ps, st, &fl, scratch));
    return launch_solve_h_bwd(theta, Hs, parts, np, ps, N, gh, gw, dtheta, st, ps == 8);
}

int mgw_feature_loss_dh(const float* matches, const float* mask, const float* img, const float* Hs, const float* facc, float upstream,
                        const float* upstream_dev, int N, int M, int H, int W, int gh, int gw, float* dH_part, void* stream)
{
    REQUIRE(matches && mask && img && Hs && facc && dH_part, "mgw_feature_loss_dh: null pointer");
    REQUIRE(N > 0 && N <= 65535 && M > 0 && H > 1 && W > 1 && gh > 0 && gw > 0 && gh <= H && gw <= W, "mgw_feature_loss_dh: bad sizes");
    REQUIRE(aligned(matches, 16) && aligned(img, 8), "mgw_feature_loss_dh: alignment");
    return launch_feature_dh(matches, mask, img, Hs, facc, upstream, upstream_dev, N, M, H, W, gh, gw, dH_part, (cudaStream_t)stream);
}

int mgw_loss_ratio_sum(const float* sums, int N, int clamp, float scale, float* out, void* stream)
{
    REQUIRE(sums && out && N > 0, "mgw_loss_ratio_sum: null pointer or N <= 0");
    return launch_ratio_sum(sums, N, clamp != 0, scale, out, (cudaStream_t)stream);
}

// ------------------------------------------------------------------------------------------------ one training pass
// coef (host, 11 floats) = PassCoef: v[4], img, feat, regu, theta_share, grid_theta_share, inv_batch, gate
static mgw::PassCoef pass_coef(const float* c)
{
    mgw::PassCoef p;
    for (int k = 0; k < 4; ++k) p.v[k] = c[k];
    p.img = c[4]; p.feat = c[5]; p.regu = c[6]; p.theta_share = c[7]; p.grid_theta_share = c[8]; p.inv_batch = c[9]; p.gate = c[10];
    return p;
}

int mgw_train_pass_fwd(const float* head, const float* U, const float* y, const float* matches, const float* mask, const float* regu_dev,
                       const float* coef, int N, int H, int W, int C, int gh, int gw, int M, float do_crop_rate, float* pts1, float* pts2,
                       float* Hs, float* out, float* black, float* img, float* acc, float* warpped, float* result, void* stream)
{
    REQUIRE(head && U && y && matches && mask && coef && pts1 && pts2 && Hs && out && black && img && acc && result,
            "mgw_train_pass_fwd: null pointer");
    TRY(validate_mesh_shape("mgw_train_pass_fwd", N, H, W, C, gh, gw));
    REQUIRE(M > 0 && N <= 65535 && do_crop_rate > 0.0f, "mgw_train_pass_fwd: need M > 0, N <= 65535, do_crop_rate > 0");
    REQUIRE(aligned(matches, 16) && aligned(img, 8) && (!warpped || aligned(warpped, 8)), "mgw_train_pass_fwd: alignment");
    cudaStream_t st = (cudaStream_t)stream;
    const WarpShape s{N, H, W, C, H, W, gh, gw};
    const PassCoef pc = pass_coef(coef);
    TRY(launch_vertices_fwd(head, N, gh, gw, do_crop_rate, pts2, pts1, st));                 // get_4_pts          :29-71
    TRY(launch_solve_h_fwd(pts2, N, gh, gw, Hs, st));                                        // get_Hs             st3:144-198
    float* vsums = acc + 4 * (size_t)N;
    TRY(check_memset(cudaMemsetAsync(acc, 0, sizeof(float) * (4 * (size_t)N + 4), st), "memset acc"));     // img [N,2] | feature [N,2] | vertex [4]
    int rc = MGW_OK;
    if (use_tma_fwd(s, U, out, black, img, &rc)) {                                           // transformer + img_loss  :332,:347-352
        TRY(launch_warp_fwd_tma(U, Hs, s, out, black, img, y, acc, st));
    } else {
        if (rc != MGW_OK) return rc;
        TRY(launch_warp_fwd_generic(U, Hs, s, false, out, black, img, nullptr, st));
        TRY(launch_img_loss_fwd(out, y, black, N, H, W, C, acc, st));
    }
    TRY(launch_feature_acc_fwd(matches, mask, img, N, M, H, W, warpped, acc + 2 * (size_t)N, st));      // feature_loss  :335-343
    TRY(launch_vertex_losses_fwd(head, pts1, pts2, N, gh, gw, do_crop_rate, vsums, nullptr, st, true));  // :139-210,:246
    return launch_objective_fwd(acc, acc + 2 * (size_t)N, vsums, regu_dev, N, pc, result, st);           // :308-317,:354-359
}

static size_t pass_bwd_offsets(int N, int H, int W, int C, int gh, int gw, size_t* extra, size_t* dp2, size_t* dp1)
{
    size_t off = mgw::align_up(mgw_mesh_warp_img_loss_bwd_workspace_bytes(N, H, W, C, gh, gw), 256);
    *extra = off; off += mgw::align_up(sizeof(float) * (size_t)N * gh * gw * 8, 256);
    *dp2 = off; off += mgw::align_up(sizeof(float) * (size_t)N * (gh + 1) * (gw + 1) * 2, 256);
    *dp1 = off; off += mgw::align_up(sizeof(float) * (size_t)N * gh * gw * 8, 256);
    return off;
}

size_t mgw_train_pass_bwd_workspace_bytes(int N, int H, int W, int C, int gh, int gw)
{
    size_t a, b, c;
    return pass_bwd_offsets(N, H, W, C, gh, gw, &a, &b, &c);
}

int mgw_train_pass_bwd(const float* head, const float* pts1, const float* pts2, const float* U, const float* y, const float* matches,
                       const float* mask, const float* Hs, const float* out, const float* black, const float* img, const float* acc,
                       const float* g_total_dev, const float* d_out_extra, const float* coef, int N, int H, int W, int C, int gh, int gw,
                       int M, float do_crop_rate, float* dU, float* d_head, void* workspace, void* stream)
{
    REQUIRE(head && pts1 && pts2 && U && y && matches && mask && Hs && out && black && img && acc && coef && d_head && workspace,
            "mgw_train_pass_bwd: null pointer");
    TRY(validate_mesh_shape("mgw_train_pass_bwd", N, H, W, C, gh, gw));
    REQUIRE(M > 0 && N <= 65535 && do_crop_rate > 0.0f, "mgw_train_pass_bwd: need M > 0, N <= 65535, do_crop_rate > 0");
    REQUIRE(aligned(workspace, 256) && aligned(matches, 16) && aligned(img, 8), "mgw_train_pass_bwd: alignment");
    cudaStream_t st = (cudaStream_t)stream;
    const WarpShape s{N, H, W, C, H, W, gh, gw};
    const PassCoef pc = pass_coef(coef);
    size_t o_extra, o_dp2, o_dp1;
    pass_bwd_offsets(N, H, W, C, gh, gw, &o_extra, &o_dp2, &o_dp1);
    float* extra = (float*)((char*)workspace + o_extra);
    float* d_pts2 = (float*)((char*)workspace + o_dp2);
    float* d_pts1 = (float*)((char*)workspace + o_dp1);
    // feature_loss backward straight to one dH partial per cell (no dense d(flow map))
    TRY(launch_feature_dh(matches, mask, img, Hs, acc + 2 * (size_t)N, pc.gate * pc.feat * (float)N * pc.inv_batch, g_total_dev, N, M, H, W, gh, gw,
                          extra, st));
    // warp backward with the img_loss gradient formed in registers (+ the gradient of another consumer of `output`)
    float* dHs_acc = (float*)workspace;
    const size_t off = align_up(sizeof(float) * (size_t)N * gh * gw * 9, 256);
    const size_t tma_bytes = mgw_warp_bwd_workspace_bytes(N, H, W, C, gh, gw);
    void* tma_ws = tma_bytes ? (void*)((char*)workspace + off) : nullptr;
    const size_t base = align_up(mgw_mesh_warp_bwd_workspace_bytes(N, H, W, C, gh, gw), 256);
    float* scratch = (float*)((char*)workspace + base);
    const FusedImgLoss fl{out, y, black, acc, pc.gate * pc.img * 2.0f * pc.inv_batch, g_total_dev};
    const float* parts; int np, ps;
    TRY(warp_bwd_core(U, Hs, d_out_extra, nullptr, s, dU, dHs_acc, tma_ws, &parts, &np, &ps, st, &fl, scratch));
    TRY(launch_solve_h_bwd(pts2, Hs, parts, np, ps, N, gh, gw, d_pts2, st, ps == 8, extra));
    // vertex regularisers: d_pts2 += consistency term, d_pts1 = black_pos + distortion terms; then back through get_4_pts with
    // the id term on the head itself
    const float vc[4] = {pc.v[0], pc.gate * pc.v[1], pc.gate * pc.v[2], pc.gate * pc.v[3]};
    TRY(launch_vertex_losses_bwd_coef(pts1, pts2, N, gh, gw, do_crop_rate, vc, g_total_dev, d_pts1, d_pts2, st));
    return launch_vertices_bwd(head, d_pts2, d_pts1, N, gh, gw, do_crop_rate, d_head, st, pc.v[0], g_total_dev);
}

int mgw_fill_zero(void* p, size_t bytes, int keep_in_l2, void* stream)
{
    REQUIRE(p && aligned(p, 16) && bytes % 16 == 0, "mgw_fill_zero: pointer and size must be multiples of 16 bytes");
    if (bytes == 0) return MGW_OK;
    return launch_fill_zero(p, bytes, keep_in_l2 != 0, (cudaStream_t)stream);
}

int mgw_u8_to_train_f32(const uint8_t* src, float* dst, size_t n, void* stream)
{
    REQUIRE(src && dst, "mgw_u8_to_train_f32: null pointer");
    if (n == 0) return MGW_OK;
    return launch_u8_to_train(src, dst, n, (cudaStream_t)stream);
}

int mgw_train_f32_to_u8(const float* src, uint8_t* dst, size_t n, void* stream)
{
    REQUIRE(src && dst, "mgw_train_f32_to_u8: null pointer");
    if (n == 0) return MGW_OK;
    return launch_train_to_u8(src, dst, n, (cudaStream_t)stream);
}

int mgw_interp_fwd(const float* im, const float* x, const float* y, int N, int IH, int IW, int C, int OH, int OW,
                   float* out, void* stream)
{
    REQUIRE(im && x && y && out, "mgw_interp_fwd: null pointer");
    REQUIRE(N > 0 && IH > 0 && IW > 0 && C > 0 && OH > 0 && OW > 0, "mgw_interp_fwd: bad sizes");
    return launch_interp_fwd(im, x, y, N, IH, IW, C, OH, OW, out, (cudaStream_t)stream);
}

int mgw_interp_bwd(const float* im, const float* x, const float* y, const float* d_out, int N, int IH, int IW, int C,
                   int OH, int OW, float* d_im, float* dx, float* dy, void* stream)
{
    REQUIRE(im && x && y && d_out, "mgw_interp_bwd: null pointer");
    REQUIRE(N > 0 && IH > 0 && IW > 0 && C > 0 && OH > 0 && OW > 0, "mgw_interp_bwd: bad sizes");
    cudaStream_t st = (cudaStream_t)stream;
    if (d_im) TRY(check_memset(cudaMemsetAsync(d_im, 0, sizeof(float) * (size_t)N * IH * IW * C, st), "memset d_im"));
    return launch_interp_bwd(im, x, y, d_out, N, IH, IW, C, OH, OW, d_im, dx, dy, st);
}

int mgw_homography_warp_fwd(const float* U, const float* theta, int N, int H, int W, int C, int OH, int OW, float* out,
                            float* black, float* img, void* stream)
{
    REQUIRE(U && theta, "mgw_homography_warp_fwd: null pointer");
    REQUIRE(N > 0 && H > 0 && W > 0 && C > 0 && OH > 1 && OW > 1, "mgw_homography_warp_fwd: bad sizes");
    REQUIRE(!img || aligned(img, 8), "mgw_homography_warp_fwd: img must be 8-byte aligned");
    const WarpShape s{N, H, W, C, OH, OW, 1, 1};
    return launch_warp_fwd_generic(U, theta, s, true, out, black, img, nullptr, (cudaStream_t)stream);
}

int mgw_homography_warp_bwd(const float* U, const float* theta, const float* d_out, int N, int H, int W, int C, int OH,
                            int OW, float* dU, float* dtheta, void* stream)
{
    REQUIRE(U && theta && d_out && dtheta, "mgw_homography_warp_bwd: null pointer");
    REQUIRE(N > 0 && H > 0 && W > 0 && C > 0 && OH > 1 && OW > 1, "mgw_homography_warp_bwd: bad sizes");
    const WarpShape s{N, H, W, C, OH, OW, 1, 1};
    cudaStream_t st = (cudaStream_t)stream;
    if (dU) TRY(check_memset(cudaMemsetAsync(dU, 0, sizeof(float) * (size_t)N * H * W * C, st), "memset dU"));
    // dtheta doubles as the dHn accumulator ([N,9]); finished in place
    TRY(check_memset(cudaMemsetAsync(dtheta, 0, sizeof(float) * (size_t)N * 9, st), "memset dtheta"));
    TRY(launch_warp_bwd_generic(U, theta, d_out, nullptr, s, true, dU, dtheta, st));
    return launch_homography_finish_bwd(theta, dtheta, N, dtheta, st);
}

size_t mgw_remap_bundle_u8_workspace_bytes(int N, int H, int W)
{
    return (N > 0 && H >= 4 && W >= 4) ? remap_bundle_workspace_bytes(N, H, W) : 0;
}

int mgw_remap_bundle_u8(const uint8_t* img, const float* xy, int N, int H, int W, int C, uint8_t* dst, void* workspace, void* stream)
{
    REQUIRE(img && xy && dst && workspace, "mgw_remap_bundle_u8: null pointer");
    REQUIRE(N > 0 && H >= 8 && W >= 8, "mgw_remap_bundle_u8: need N > 0, H >= 8, W >= 8 (got N=%d H=%d W=%d)", N, H, W);
    REQUIRE(H <= 32767 && W <= 32767 && (long long)N * H * W < (1LL << 31), "mgw_remap_bundle_u8: image too large");
    REQUIRE(aligned(xy, 8) && aligned(workspace, 8), "mgw_remap_bundle_u8: xy and workspace must be 8-byte aligned");
    return launch_remap_bundle_u8(img, xy, N, H, W, C, dst, workspace, (cudaStream_t)stream);
}

size_t mgw_remap_bundle_frame_workspace_bytes(int S, int h, int w, int H, int W)
{
    (void)H; (void)W;       // the workspace holds the /4 maps, whose size is the network's
    return mgw_remap_bundle_u8_workspace_bytes(S, h, w);
}

// The batch calls' order: sizes and format, then S = 0, then pointers.  H, W <= 32767: OpenCV clamps the taps to int16.
int mgw_remap_bundle_frame(const uint8_t* src, int format, const float* xy, int S, int h, int w, int H, int W, uint8_t* dst,
                           void* workspace, void* stream)
{
    REQUIRE(S >= 0 && S <= 65535 && h >= 8 && w >= 8 && H >= 1 && W >= 1 && H <= 32767 && W <= 32767 &&
            (format == MGW_BGR24 || (H % 2 == 0 && W % 2 == 0)) && (long long)S * H * W * 3 < (1LL << 31) &&
            (long long)S * h * w < (1LL << 31),
            "mgw_remap_bundle_frame: bad sizes (S=%d maps %dx%d frame %dx%d; h, w >= 8, H and W even for YUV)", S, h, w, H, W);
    REQUIRE(format == MGW_BGR24 || format == MGW_YUV420_NV12 || format == MGW_YUV420_I420, "mgw_remap_bundle_frame: unknown format %d",
            format);
    if (S == 0) return MGW_OK;
    REQUIRE(src && xy && dst && workspace, "mgw_remap_bundle_frame: null pointer");
    REQUIRE(aligned(xy, 8) && aligned(workspace, 8), "mgw_remap_bundle_frame: xy and workspace must be 8-byte aligned");
    return launch_remap_bundle(src, format, 3, xy, S, h, w, H, W, dst, workspace, (cudaStream_t)stream);
}

// mgw_remap_bundle_frame's checks in its order, with H and W even for every source (a 4:2:0 result) and dst_format one of the two
// YUV layouts (MGW_BGR24 is mgw_remap_bundle_frame)
int mgw_remap_bundle_frame_yuv420(const uint8_t* src, int format, const float* xy, int S, int h, int w, int H, int W, int dst_format,
                                  uint8_t* dst, void* workspace, void* stream)
{
    REQUIRE(S >= 0 && S <= 65535 && h >= 8 && w >= 8 && H >= 2 && W >= 2 && H <= 32766 && W <= 32766 && H % 2 == 0 && W % 2 == 0 &&
            (long long)S * H * W * 3 < (1LL << 31) && (long long)S * h * w < (1LL << 31),
            "mgw_remap_bundle_frame_yuv420: bad sizes (S=%d maps %dx%d frame %dx%d; h, w >= 8, H and W even)", S, h, w, H, W);
    REQUIRE(format == MGW_BGR24 || format == MGW_YUV420_NV12 || format == MGW_YUV420_I420,
            "mgw_remap_bundle_frame_yuv420: unknown format %d", format);
    REQUIRE(dst_format == MGW_YUV420_NV12 || dst_format == MGW_YUV420_I420,
            "mgw_remap_bundle_frame_yuv420: unknown destination format %d (NV12 or I420; BGR is mgw_remap_bundle_frame)", dst_format);
    if (S == 0) return MGW_OK;
    REQUIRE(src && xy && dst && workspace, "mgw_remap_bundle_frame_yuv420: null pointer");
    REQUIRE(aligned(xy, 8) && aligned(workspace, 8), "mgw_remap_bundle_frame_yuv420: xy and workspace must be 8-byte aligned");
    return launch_remap_bundle_yuv420(src, format, xy, S, h, w, H, W, dst_format, dst, workspace, (cudaStream_t)stream);
}

// mgw_remap_bundle_frame's checks over the capacity, in the batch calls' order; the capacity is even when either format is YUV
int mgw_remap_bundle_frame_mixed(const uint8_t* src, int format, int S, int max_h, int max_w, const int32_t* sizes, const float* xy,
                                 int h, int w, int dst_format, uint8_t* dst, void* workspace, void* stream)
{
    const auto known = [](int f) { return f == MGW_BGR24 || f == MGW_YUV420_NV12 || f == MGW_YUV420_I420; };
    REQUIRE(known(format), "mgw_remap_bundle_frame_mixed: unknown format %d", format);
    REQUIRE(known(dst_format), "mgw_remap_bundle_frame_mixed: unknown destination format %d", dst_format);
    REQUIRE(S >= 0 && S <= 65535 && h >= 8 && w >= 8 && max_h >= 1 && max_w >= 1 && max_h <= 32767 && max_w <= 32767 &&
            ((format == MGW_BGR24 && dst_format == MGW_BGR24) || (max_h % 2 == 0 && max_w % 2 == 0)) &&
            (long long)S * max_h * max_w * 3 < (1LL << 31) && (long long)S * h * w < (1LL << 31),
            "mgw_remap_bundle_frame_mixed: bad sizes (S=%d maps %dx%d capacity %dx%d; h, w >= 8, capacity even for YUV)", S, h, w,
            max_h, max_w);
    if (S == 0) return MGW_OK;
    REQUIRE(src && sizes && xy && dst && workspace, "mgw_remap_bundle_frame_mixed: null pointer");
    REQUIRE(aligned(xy, 8) && aligned(workspace, 8) && aligned(sizes, 8),
            "mgw_remap_bundle_frame_mixed: xy, workspace and sizes must be 8-byte aligned");
    return launch_remap_bundle_mixed(src, format, S, max_h, max_w, sizes, xy, h, w, dst_format, dst, workspace, (cudaStream_t)stream);
}

// The address a kernel reaches the `bytes` bytes at p through: device or managed memory as it is, pinned host memory through its
// mapped device address.  Both ends are looked up, so a buffer that runs past its allocation is refused; pageable memory has no
// device address.
static int device_address(const char* fn, const char* what, const void* p, size_t bytes, const void** dev)
{
    const char* q[2] = {static_cast<const char*>(p), static_cast<const char*>(p) + bytes - 1};
    const char* d[2];
    for (int k = 0; k < 2; ++k) {
        cudaPointerAttributes a;
        const cudaError_t e = cudaPointerGetAttributes(&a, q[k]);
        if (e != cudaSuccess) {
            cudaGetLastError();
            return set_error(MGW_ERR_CUDA, "%s: %s: %s", fn, what, cudaGetErrorString(e));
        }
        REQUIRE(a.type != cudaMemoryTypeUnregistered, "%s: %s is pageable host memory (pin it: cudaHostAlloc / cudaHostRegister)", fn, what);
        REQUIRE(a.devicePointer, "%s: %s has no device address", fn, what);
        d[k] = static_cast<const char*>(a.devicePointer);
    }
    REQUIRE(d[1] == d[0] + (bytes - 1), "%s: %s is not one mapped range of %zu bytes", fn, what, bytes);
    *dev = d[0];
    return MGW_OK;
}

// The batch calls' order: format and sizes, then S = 0, then pointers and alignment; then where src and dst live
int mgw_copy_slots_mixed(const uint8_t* src, uint8_t* dst, int format, int S, int max_h, int max_w, const int32_t* sizes, void* stream)
{
    REQUIRE(format == MGW_BGR24 || format == MGW_YUV420_NV12 || format == MGW_YUV420_I420, "mgw_copy_slots_mixed: unknown format %d",
            format);
    const long long stride = format == MGW_BGR24 ? 3LL * max_h * max_w : 3LL * max_h * max_w / 2;
    REQUIRE(S >= 0 && S <= 65535 && max_h >= 1 && max_w >= 1 && max_h <= 32767 && max_w <= 32767 &&
            (format == MGW_BGR24 || (max_h % 2 == 0 && max_w % 2 == 0)) && S * stride < (1LL << 31),
            "mgw_copy_slots_mixed: bad sizes (S=%d capacity %dx%d; capacity even for YUV, S * frame_bytes(capacity) < 2^31)", S, max_h,
            max_w);
    if (S == 0) return MGW_OK;
    REQUIRE(src && dst && sizes, "mgw_copy_slots_mixed: null pointer");
    REQUIRE(aligned(src, 16) && aligned(dst, 16), "mgw_copy_slots_mixed: src and dst must be 16-byte aligned");
    REQUIRE(aligned(sizes, 8), "mgw_copy_slots_mixed: sizes must be 8-byte aligned");
    const size_t bytes = (size_t)(S * stride);
    const void *s_dev, *d_dev;
    TRY(device_address("mgw_copy_slots_mixed", "src", src, bytes, &s_dev));
    TRY(device_address("mgw_copy_slots_mixed", "dst", dst, bytes, &d_dev));
    return launch_copy_slots_mixed(static_cast<const uint8_t*>(s_dev), static_cast<uint8_t*>(const_cast<void*>(d_dev)), format, S, max_h,
                                   max_w, sizes, (cudaStream_t)stream);
}

int mgw_stream_assemble(const float* frames, const float* masks, int depth, int head, const int* taps, int ntaps, int use_masks,
                        const float* cur, int H, int W, float* in_x, void* stream)
{
    REQUIRE(frames && taps && cur && in_x && (masks || !use_masks), "mgw_stream_assemble: null pointer");
    REQUIRE(depth > 0 && head >= 0 && head < depth && H > 0 && W > 0 && (long long)H * W < (1LL << 31), "mgw_stream_assemble: bad sizes");
    return launch_stream_assemble(frames, masks, depth, head, taps, ntaps, use_masks, cur, H, W, in_x, (cudaStream_t)stream);
}

int mgw_stream_push(float* frames, float* masks, int depth, int slot, const float* img, const float* black, int H, int W,
                    float* frame_out, int out_stride, void* stream)
{
    REQUIRE(img && black && (frames || frame_out), "mgw_stream_push: null pointer");
    REQUIRE(depth > 0 && slot >= 0 && slot < depth && H > 0 && W > 0 && (long long)H * W < (1LL << 31) && out_stride >= 1,
            "mgw_stream_push: bad sizes");
    return launch_stream_push(frames, masks, depth, slot, img, black, H, W, frame_out, out_stride, (cudaStream_t)stream);
}

int mgw_resize_linear_u8(const uint8_t* img, int H, int W, int C, const int32_t* xtab, const int32_t* ytab, int out_h, int out_w,
                         uint8_t* dst, void* stream)
{
    REQUIRE(img && dst, "mgw_resize_linear_u8: null pointer");
    REQUIRE(H > 0 && W > 0 && out_h > 0 && out_w > 0 && (long long)H * W * 4 < (1LL << 31) && (long long)out_h * out_w < (1LL << 29),
            "mgw_resize_linear_u8: bad sizes");
    REQUIRE((!xtab || aligned(xtab, 16)) && (!ytab || aligned(ytab, 16)), "mgw_resize_linear_u8: tables must be 16-byte aligned");
    return launch_resize_linear_u8(img, 1, H, W, C, xtab, ytab, out_h, out_w, dst, (cudaStream_t)stream);
}

int mgw_cvt_img2train_u8(const uint8_t* bgr, int H, int W, const int32_t* kx, const int32_t* x0, const int32_t* xn, int ksx,
                         const int32_t* ky, const int32_t* y0, const int32_t* yn, int ksy, int out_h, int out_w, uint8_t* tmp,
                         float* out, void* stream)
{
    REQUIRE(bgr && kx && x0 && xn && ky && y0 && yn && tmp && out, "mgw_cvt_img2train_u8: null pointer");
    REQUIRE(H > 0 && W > 0 && out_h > 0 && out_w > 0 && ksx > 0 && ksy > 0 && (long long)H * out_w < (1LL << 31) &&
            (long long)H * W < (1LL << 29), "mgw_cvt_img2train_u8: bad sizes");
    return launch_cvt_img2train_u8(bgr, 1, H, W, kx, x0, xn, ksx, ky, y0, yn, ksy, out_h, out_w, tmp, out, (cudaStream_t)stream);
}

int mgw_warp_rev_bundle_u8(const uint8_t* img, const double* Hs_cvt, int N, int H, int W, int C, int gh, int gw, uint8_t* dst,
                           void* stream)
{
    REQUIRE(img && Hs_cvt && dst, "mgw_warp_rev_bundle_u8: null pointer");
    REQUIRE(N > 0 && H > 0 && W > 0 && gh > 0 && gw > 0 && gh <= H && gw <= W && (long long)N * H * W < (1LL << 31),
            "mgw_warp_rev_bundle_u8: bad sizes");
    return launch_warp_rev_bundle_u8(img, Hs_cvt, N, H, W, C, gh, gw, dst, (cudaStream_t)stream);
}

int mgw_vertex_losses_fwd(const float* theta, const float* pts1, const float* pts2, int N, int gh, int gw, float do_crop_rate,
                          float* sums, float* black_err, void* stream)
{
    REQUIRE(sums && (theta || pts1 || pts2), "mgw_vertex_losses_fwd: null pointer");
    REQUIRE(!black_err || pts1, "mgw_vertex_losses_fwd: black_err needs pts1");
    REQUIRE(N > 0 && gh > 0 && gw > 0 && do_crop_rate > 0.0f && (long long)N * (gh + 1) * (gw + 1) * 2 < (1LL << 31),
            "mgw_vertex_losses_fwd: bad sizes");
    return launch_vertex_losses_fwd(theta, pts1, pts2, N, gh, gw, do_crop_rate, sums, black_err, (cudaStream_t)stream);
}

int mgw_vertex_losses_bwd(const float* theta, const float* pts1, const float* pts2, int N, int gh, int gw, float do_crop_rate,
                          const float* f, float* d_theta, float* d_pts1, float* d_pts2,
                          void* stream)
{
    REQUIRE(f && (!d_theta || theta) && (!d_pts1 || pts1) && (!d_pts2 || pts2) && (d_theta || d_pts1 || d_pts2),
            "mgw_vertex_losses_bwd: a gradient was requested without its input");
    REQUIRE(N > 0 && gh > 0 && gw > 0 && do_crop_rate > 0.0f && (long long)N * (gh + 1) * (gw + 1) * 2 < (1LL << 31),
            "mgw_vertex_losses_bwd: bad sizes");
    return launch_vertex_losses_bwd(theta, pts1, pts2, N, gh, gw, do_crop_rate, f, d_theta, d_pts1, d_pts2,
                                    (cudaStream_t)stream);
}

int mgw_black_accumulate(const float* black, int32_t* all_black, int n, void* stream)
{
    REQUIRE(black && all_black, "mgw_black_accumulate: null pointer");
    REQUIRE(n > 0, "mgw_black_accumulate: bad sizes");
    return launch_black_accumulate(black, all_black, n, (cudaStream_t)stream);
}

size_t mgw_crop_rect_workspace_bytes(int H, int W) { return (H > 0 && W > 0) ? crop_rect_workspace_bytes(H, W) : 0; }

int mgw_crop_rect(const int32_t* all_black, int H, int W, int step, void* workspace, int32_t* rect, void* stream)
{
    REQUIRE(all_black && workspace && rect, "mgw_crop_rect: null pointer");
    REQUIRE(H > 0 && W > 0 && step > 0 && (long long)H * W < (1LL << 31), "mgw_crop_rect: bad sizes");
    return launch_crop_rect(all_black, H, W, step, workspace, rect, (cudaStream_t)stream);
}

int mgw_stream_assemble_dev(const float* frames, const float* masks, int depth, const int32_t* head_dev, const int* taps, int ntaps,
                            int use_masks, const float* cur, int H, int W, float* in_x, void* stream)
{
    REQUIRE(frames && cur && in_x && taps && head_dev && (masks || !use_masks), "mgw_stream_assemble_dev: null pointer");
    REQUIRE(depth > 0 && H > 0 && W > 0 && (long long)H * W < (1LL << 31), "mgw_stream_assemble_dev: bad sizes");
    return launch_stream_assemble(frames, masks, depth, 0, taps, ntaps, use_masks, cur, H, W, in_x, (cudaStream_t)stream,
                                  reinterpret_cast<const int*>(head_dev));
}

int mgw_stream_push_dev(float* frames, float* masks, int depth, int32_t* head_dev, const float* img, const float* black, int H, int W,
                        void* stream)
{
    REQUIRE(img && black && frames && head_dev, "mgw_stream_push_dev: null pointer");
    REQUIRE(depth > 0 && H > 0 && W > 0 && (long long)H * W < (1LL << 31), "mgw_stream_push_dev: bad sizes");
    TRY(launch_stream_push(frames, masks, depth, 0, img, black, H, W, nullptr, 1, (cudaStream_t)stream, reinterpret_cast<const int*>(head_dev)));
    return launch_stream_advance(reinterpret_cast<int*>(head_dev), depth, (cudaStream_t)stream);
}

// Batched deploy calls: S streams (frames) of one size, the stream index in gridDim.y (hence S <= 65535).  The sizes are checked
// first: S = 0 returns MGW_OK before the pointers are looked at (an empty batch may come with null buffers) and launches nothing.
int mgw_cvt_img2train_u8_batch(const uint8_t* bgr, int S, int H, int W, const int32_t* kx, const int32_t* x0, const int32_t* xn, int ksx,
                               const int32_t* ky, const int32_t* y0, const int32_t* yn, int ksy, int out_h, int out_w, uint8_t* tmp,
                               float* out, void* stream)
{
    REQUIRE(S >= 0 && S <= 65535 && H > 0 && W > 0 && out_h > 0 && out_w > 0 && ksx > 0 && ksy > 0 &&
            (long long)S * H * out_w < (1LL << 31) && (long long)S * out_h * out_w < (1LL << 31) && (long long)S * H * W < (1LL << 29),
            "mgw_cvt_img2train_u8_batch: bad sizes (S=%d H=%d W=%d out %dx%d)", S, H, W, out_h, out_w);
    if (S == 0) return MGW_OK;
    REQUIRE(bgr && kx && x0 && xn && ky && y0 && yn && tmp && out, "mgw_cvt_img2train_u8_batch: null pointer");
    return launch_cvt_img2train_u8(bgr, S, H, W, kx, x0, xn, ksx, ky, y0, yn, ksy, out_h, out_w, tmp, out, (cudaStream_t)stream);
}

int mgw_resize_linear_u8_batch(const uint8_t* img, int S, int H, int W, int C, const int32_t* xtab, const int32_t* ytab, int out_h,
                               int out_w, uint8_t* dst, void* stream)
{
    REQUIRE(S >= 0 && S <= 65535 && H > 0 && W > 0 && out_h > 0 && out_w > 0 && (long long)S * H * W * 4 < (1LL << 31) &&
            (long long)S * out_h * out_w < (1LL << 29), "mgw_resize_linear_u8_batch: bad sizes (S=%d H=%d W=%d out %dx%d)", S, H, W,
            out_h, out_w);
    REQUIRE(C == 1 || C == 3 || C == 4, "mgw_resize_linear_u8_batch: C must be 1, 3 or 4 (got %d)", C);
    if (S == 0) return MGW_OK;
    REQUIRE(img && dst, "mgw_resize_linear_u8_batch: null pointer");
    REQUIRE((W == 2 * out_w && H == 2 * out_h) || (xtab && ytab), "mgw_resize_linear_u8_batch: coefficient tables are required");
    REQUIRE((!xtab || aligned(xtab, 16)) && (!ytab || aligned(ytab, 16)), "mgw_resize_linear_u8_batch: tables must be 16-byte aligned");
    return launch_resize_linear_u8(img, S, H, W, C, xtab, ytab, out_h, out_w, dst, (cudaStream_t)stream);
}

// YUV 4:2:0 frames [S,3H/2,W]: the BGR batch calls' checks in the same order, their 32-bit index limit taken over the YUV bytes
static int validate_yuv420(const char* fn, int format, int S, int H, int W, int out_h, int out_w)
{
    REQUIRE(S >= 0 && S <= 65535 && H > 0 && W > 0 && H % 2 == 0 && W % 2 == 0 && out_h > 0 && out_w > 0 &&
            (long long)S * (H + H / 2) * W < (1LL << 31) && (long long)S * H * out_w < (1LL << 31) && (long long)S * out_h * out_w < (1LL << 29),
            "%s: bad sizes (S=%d H=%d W=%d out %dx%d; H and W must be even)", fn, S, H, W, out_h, out_w);
    REQUIRE(format == MGW_YUV420_NV12 || format == MGW_YUV420_I420, "%s: unknown format %d", fn, format);
    return MGW_OK;
}

int mgw_cvt_img2train_yuv420_batch(const uint8_t* yuv, int format, int S, int H, int W, const int32_t* kx, const int32_t* x0,
                                   const int32_t* xn, int ksx, const int32_t* ky, const int32_t* y0, const int32_t* yn, int ksy, int out_h,
                                   int out_w, uint8_t* tmp, float* out, void* stream)
{
    TRY(validate_yuv420("mgw_cvt_img2train_yuv420_batch", format, S, H, W, out_h, out_w));
    REQUIRE(ksx > 0 && ksy > 0, "mgw_cvt_img2train_yuv420_batch: bad sizes (ksx=%d ksy=%d)", ksx, ksy);
    if (S == 0) return MGW_OK;
    REQUIRE(yuv && kx && x0 && xn && ky && y0 && yn && tmp && out, "mgw_cvt_img2train_yuv420_batch: null pointer");
    return launch_cvt_img2train_u8(yuv, S, H, W, kx, x0, xn, ksx, ky, y0, yn, ksy, out_h, out_w, tmp, out, (cudaStream_t)stream, format);
}

int mgw_resize_linear_yuv420_batch(const uint8_t* yuv, int format, int S, int H, int W, const int32_t* xtab, const int32_t* ytab,
                                   int out_h, int out_w, uint8_t* dst, void* stream)
{
    TRY(validate_yuv420("mgw_resize_linear_yuv420_batch", format, S, H, W, out_h, out_w));
    if (S == 0) return MGW_OK;
    REQUIRE(yuv && dst, "mgw_resize_linear_yuv420_batch: null pointer");
    REQUIRE((W == 2 * out_w && H == 2 * out_h) || (xtab && ytab), "mgw_resize_linear_yuv420_batch: coefficient tables are required");
    REQUIRE((!xtab || aligned(xtab, 16)) && (!ytab || aligned(ytab, 16)), "mgw_resize_linear_yuv420_batch: tables must be 16-byte aligned");
    return launch_resize_linear_u8(yuv, S, H, W, 3, xtab, ytab, out_h, out_w, dst, (cudaStream_t)stream, format);
}

// Per-slot source geometry: the capacity (max_h, max_w) takes the place of the uniform batch's H, W in its size checks (every
// slot's region and tmp rows are laid out for it); the 8-byte alignment of sizes is that of the int2 each block loads.
static int validate_mixed(const char* fn, int format, int S, int max_h, int max_w, int out_h, int out_w)
{
    REQUIRE(format == MGW_BGR24 || format == MGW_YUV420_NV12 || format == MGW_YUV420_I420, "%s: unknown format %d", fn, format);
    if (format != MGW_BGR24) return validate_yuv420(fn, format, S, max_h, max_w, out_h, out_w);
    REQUIRE(S >= 0 && S <= 65535 && max_h > 0 && max_w > 0 && out_h > 0 && out_w > 0 && (long long)S * max_h * max_w < (1LL << 29) &&
            (long long)S * max_h * out_w < (1LL << 31) && (long long)S * out_h * out_w < (1LL << 29),
            "%s: bad sizes (S=%d capacity %dx%d out %dx%d)", fn, S, max_h, max_w, out_h, out_w);
    return MGW_OK;
}

int mgw_cvt_img2train_mixed(const uint8_t* src, int format, int S, int max_h, int max_w, const int32_t* sizes, const int32_t* kx,
                            const int32_t* x0, const int32_t* xn, int ksx, const int32_t* ky, const int32_t* y0, const int32_t* yn, int ksy,
                            int out_h, int out_w, uint8_t* tmp, float* out, void* stream)
{
    TRY(validate_mixed("mgw_cvt_img2train_mixed", format, S, max_h, max_w, out_h, out_w));
    REQUIRE(ksx > 0 && ksy > 0, "mgw_cvt_img2train_mixed: bad sizes (ksx=%d ksy=%d)", ksx, ksy);
    if (S == 0) return MGW_OK;
    REQUIRE(src && sizes && kx && x0 && xn && ky && y0 && yn && tmp && out, "mgw_cvt_img2train_mixed: null pointer");
    REQUIRE(aligned(sizes, 8), "mgw_cvt_img2train_mixed: sizes must be 8-byte aligned");
    return launch_cvt_img2train_mixed(src, format, S, max_h, max_w, sizes, kx, x0, xn, ksx, ky, y0, yn, ksy, out_h, out_w, tmp, out,
                                      (cudaStream_t)stream);
}

int mgw_resize_linear_mixed(const uint8_t* src, int format, int S, int max_h, int max_w, const int32_t* sizes, const int32_t* xtab,
                            const int32_t* ytab, int out_h, int out_w, uint8_t* dst, void* stream)
{
    TRY(validate_mixed("mgw_resize_linear_mixed", format, S, max_h, max_w, out_h, out_w));
    if (S == 0) return MGW_OK;
    REQUIRE(src && sizes && xtab && ytab && dst, "mgw_resize_linear_mixed: null pointer");
    REQUIRE(aligned(xtab, 16) && aligned(ytab, 16), "mgw_resize_linear_mixed: tables must be 16-byte aligned");
    REQUIRE(aligned(sizes, 8), "mgw_resize_linear_mixed: sizes must be 8-byte aligned");
    return launch_resize_linear_mixed(src, format, S, max_h, max_w, sizes, xtab, ytab, out_h, out_w, dst, (cudaStream_t)stream);
}

static_assert(sizeof(mgw_planes) == 48 && offsetof(mgw_planes, pitch) == 24, "mgw_planes: 48-byte entries, pitches at 24");

// Per-slot planes: the uniform calls' size limits at (H, W) for the format (validate_mixed with the frame size as the capacity);
// a table is 16-byte aligned, the alignment of the two vector loads of each entry
int mgw_cvt_img2train_planes(const void* src, int format, int S, int H, int W, const int32_t* kx, const int32_t* x0, const int32_t* xn,
                             int ksx, const int32_t* ky, const int32_t* y0, const int32_t* yn, int ksy, int out_h, int out_w, uint8_t* tmp,
                             float* out, void* stream)
{
    TRY(validate_mixed("mgw_cvt_img2train_planes", format, S, H, W, out_h, out_w));
    REQUIRE(ksx > 0 && ksy > 0, "mgw_cvt_img2train_planes: bad sizes (ksx=%d ksy=%d)", ksx, ksy);
    if (S == 0) return MGW_OK;
    REQUIRE(src && kx && x0 && xn && ky && y0 && yn && tmp && out, "mgw_cvt_img2train_planes: null pointer");
    REQUIRE(aligned(src, 16), "mgw_cvt_img2train_planes: the planes table must be 16-byte aligned");
    return launch_cvt_img2train_planes(static_cast<const mgw_planes*>(src), format, S, H, W, kx, x0, xn, ksx, ky, y0, yn, ksy, out_h, out_w,
                                       tmp, out, (cudaStream_t)stream);
}

int mgw_resize_linear_planes(const void* src, int format, int S, int H, int W, const int32_t* xtab, const int32_t* ytab, int out_h,
                             int out_w, uint8_t* dst, void* stream)
{
    TRY(validate_mixed("mgw_resize_linear_planes", format, S, H, W, out_h, out_w));
    if (S == 0) return MGW_OK;
    REQUIRE(src && dst, "mgw_resize_linear_planes: null pointer");
    REQUIRE((W == 2 * out_w && H == 2 * out_h) || (xtab && ytab), "mgw_resize_linear_planes: coefficient tables are required");
    REQUIRE((!xtab || aligned(xtab, 16)) && (!ytab || aligned(ytab, 16)), "mgw_resize_linear_planes: tables must be 16-byte aligned");
    REQUIRE(aligned(src, 16), "mgw_resize_linear_planes: the planes table must be 16-byte aligned");
    return launch_resize_linear_planes(static_cast<const mgw_planes*>(src), format, S, H, W, xtab, ytab, out_h, out_w, dst,
                                       (cudaStream_t)stream);
}

// mgw_remap_bundle_frame_mixed's checks at the frame size: H and W even when either format is YUV
int mgw_remap_bundle_frame_planes(const void* src, int format, const float* xy, int S, int h, int w, int H, int W, const void* dst,
                                  int dst_format, void* workspace, void* stream)
{
    const auto known = [](int f) { return f == MGW_BGR24 || f == MGW_YUV420_NV12 || f == MGW_YUV420_I420; };
    REQUIRE(known(format), "mgw_remap_bundle_frame_planes: unknown format %d", format);
    REQUIRE(known(dst_format), "mgw_remap_bundle_frame_planes: unknown destination format %d", dst_format);
    REQUIRE(S >= 0 && S <= 65535 && h >= 8 && w >= 8 && H >= 1 && W >= 1 && H <= 32767 && W <= 32767 &&
            ((format == MGW_BGR24 && dst_format == MGW_BGR24) || (H % 2 == 0 && W % 2 == 0)) &&
            (long long)S * H * W * 3 < (1LL << 31) && (long long)S * h * w < (1LL << 31),
            "mgw_remap_bundle_frame_planes: bad sizes (S=%d maps %dx%d frame %dx%d; h, w >= 8, H and W even for YUV)", S, h, w, H, W);
    if (S == 0) return MGW_OK;
    REQUIRE(src && xy && dst && workspace, "mgw_remap_bundle_frame_planes: null pointer");
    REQUIRE(aligned(src, 16) && aligned(dst, 16), "mgw_remap_bundle_frame_planes: the planes tables must be 16-byte aligned");
    REQUIRE(aligned(xy, 8) && aligned(workspace, 8), "mgw_remap_bundle_frame_planes: xy and workspace must be 8-byte aligned");
    return launch_remap_bundle_planes(static_cast<const mgw_planes*>(src), format, xy, S, h, w, H, W, static_cast<const mgw_planes*>(dst),
                                      dst_format, workspace, (cudaStream_t)stream);
}

static int validate_streams(const char* fn, int S, int depth, int H, int W, int nch)
{
    REQUIRE(S >= 0 && S <= 65535 && depth > 0 && H > 0 && W > 0 && (long long)S * depth * H * W < (1LL << 31) &&
            (long long)S * H * W * nch < (1LL << 31), "%s: bad sizes (S=%d depth=%d H=%d W=%d)", fn, S, depth, H, W);
    return MGW_OK;
}

int mgw_streams_assemble(const float* frames, const float* masks, int S, int depth, const int32_t* heads_dev, const int* taps, int ntaps,
                         int use_masks, const float* cur, int H, int W, float* in_x, void* stream)
{
    REQUIRE(taps || ntaps == 0, "mgw_streams_assemble: null pointer");
    REQUIRE(ntaps >= 0 && ntaps <= 32, "mgw_streams_assemble: at most 32 taps (got %d)", ntaps);
    for (int k = 0; k < ntaps; ++k)
        REQUIRE(taps[k] >= 1 && taps[k] <= depth, "mgw_streams_assemble: tap %d outside [1, depth = %d]", taps[k], depth);
    TRY(validate_streams("mgw_streams_assemble", S, depth, H, W, (use_masks ? 2 : 1) * ntaps + 1));
    if (S == 0) return MGW_OK;
    REQUIRE(frames && cur && in_x && heads_dev && (masks || !use_masks), "mgw_streams_assemble: null pointer");
    return launch_stream_assemble(frames, masks, depth, 0, taps, ntaps, use_masks, cur, H, W, in_x, (cudaStream_t)stream,
                                  reinterpret_cast<const int*>(heads_dev), S);
}

int mgw_streams_push(float* frames, float* masks, int S, int depth, int32_t* heads_dev, const float* img, const float* black, int H, int W,
                     void* stream)
{
    TRY(validate_streams("mgw_streams_push", S, depth, H, W, 1));
    if (S == 0) return MGW_OK;
    REQUIRE(img && black && frames && heads_dev, "mgw_streams_push: null pointer");
    TRY(launch_stream_push(frames, masks, depth, 0, img, black, H, W, nullptr, 1, (cudaStream_t)stream,
                           reinterpret_cast<const int*>(heads_dev), S));
    return launch_stream_advance(reinterpret_cast<int*>(heads_dev), depth, (cudaStream_t)stream, S);
}

int mgw_img_loss_fwd(const float* out, const float* y, const float* black, int N, int H, int W, int C, float* sums, void* stream)
{
    REQUIRE(out && y && black && sums, "mgw_img_loss_fwd: null pointer");
    REQUIRE(N > 0 && H > 0 && W > 0 && C > 0, "mgw_img_loss_fwd: bad sizes");
    return launch_img_loss_fwd(out, y, black, N, H, W, C, sums, (cudaStream_t)stream);
}

int mgw_img_loss_bwd(const float* out, const float* y, const float* black, const float* sums, float upstream,
                     const float* upstream_dev, int N,
                     int H, int W, int C, float* d_out, void* stream)
{
    REQUIRE(out && y && black && sums && d_out, "mgw_img_loss_bwd: null pointer");
    REQUIRE(N > 0 && H > 0 && W > 0 && C > 0, "mgw_img_loss_bwd: bad sizes");
    return launch_img_loss_bwd(out, y, black, sums, upstream, upstream_dev, N, H, W, C, d_out, (cudaStream_t)stream);
}

int mgw_feature_loss_fwd(const float* matches, const float* mask, const float* img, int N, int M, int H, int W,
                         float* warpped, float* per_sample, void* stream)
{
    REQUIRE(matches && mask && img && per_sample, "mgw_feature_loss_fwd: null pointer");
    REQUIRE(N > 0 && M > 0 && H > 0 && W > 0, "mgw_feature_loss_fwd: bad sizes");
    REQUIRE(aligned(matches, 16) && aligned(img, 8) && (!warpped || aligned(warpped, 8)), "mgw_feature_loss_fwd: alignment");
    return launch_feature_loss_fwd(matches, mask, img, N, M, H, W, warpped, per_sample, (cudaStream_t)stream);
}

int mgw_feature_loss_bwd(const float* matches, const float* mask, const float* img, float upstream, const float* upstream_dev,
                         int N, int M, int H,
                         int W, float* d_img, void* stream)
{
    REQUIRE(matches && mask && img && d_img, "mgw_feature_loss_bwd: null pointer");
    REQUIRE(N > 0 && M > 0 && H > 0 && W > 0, "mgw_feature_loss_bwd: bad sizes");
    REQUIRE(aligned(matches, 16) && aligned(img, 8), "mgw_feature_loss_bwd: alignment");
    return launch_feature_loss_bwd(matches, mask, img, upstream, upstream_dev, N, M, H, W, d_img, (cudaStream_t)stream);
}

int mgw_temp_loss_fwd(const float* out1, const float* black1, const float* out2, const float* black2, const float* flow,
                      int N, int H, int W, int C, float* sums, void* stream)
{
    REQUIRE(out1 && black1 && out2 && black2 && flow && sums, "mgw_temp_loss_fwd: null pointer");
    REQUIRE(N > 0 && H > 0 && W > 0 && C > 0 && (long long)H * W * C < (1LL << 31), "mgw_temp_loss_fwd: bad sizes");
    REQUIRE(aligned(flow, 8), "mgw_temp_loss_fwd: flow must be 8-byte aligned");
    return launch_temp_loss_fwd(out1, black1, out2, black2, flow, N, H, W, C, sums, (cudaStream_t)stream);
}

int mgw_temp_loss_bwd(const float* out1, const float* black1, const float* out2, const float* black2, const float* flow,
                      const float* sums, float upstream, const float* upstream_dev, int N, int H, int W, int C, float* d_out1,
                      float* d_out2, void* stream)
{
    REQUIRE(out1 && black1 && out2 && black2 && flow && sums && d_out1 && d_out2, "mgw_temp_loss_bwd: null pointer");
    REQUIRE(N > 0 && H > 0 && W > 0 && C > 0 && (long long)H * W * C < (1LL << 31), "mgw_temp_loss_bwd: bad sizes");
    REQUIRE(aligned(flow, 8), "mgw_temp_loss_bwd: flow must be 8-byte aligned");
    return launch_temp_loss_bwd(out1, black1, out2, black2, flow, sums, upstream, upstream_dev, N, H, W, C, d_out1, d_out2, (cudaStream_t)stream);
}

}  // extern "C"

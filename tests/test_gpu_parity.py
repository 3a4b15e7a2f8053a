"""GPU parity tests proper: every check goes through the C ABI (ctypes) on cuda:0 and compares with
(a) the golden vectors = outputs of the unmodified reference sources, and (b) the C oracle.

Bars (BASELINE.json north_star): cell index and in-bounds masks bit-exact; warped pixels <= 1e-5 abs fp32
(and in fact bit-exact given the reference's Hs); gradients <= 1e-4 relative (max-norm), arbitrated by the fp64
run of the reference where the reference's own fp32 noise is larger than that (SURVEY.md 7, hard part 2).
"""
import numpy as np
import pytest
import torch

import c_oracle
from conftest import (FULL_MESH_CASES, MESH_CASES, SMALL_MESH_CASES, TMA_MESH_CASES, bits_equal, golden_black, golden_inputs,
                      load_golden, relmax)

pytestmark = pytest.mark.gpu

IMPLS = ['generic', 'auto']


@pytest.fixture(scope='module')
def mgw():
    import dovs_b200
    assert torch.cuda.is_available(), 'GPU tests need a CUDA device; there is no CPU fallback'
    yield dovs_b200
    dovs_b200.set_impl('auto')


def dev(a):
    return torch.tensor(np.ascontiguousarray(a), device='cuda')


def grad_ok(got, ref32, f64=None, tol=1e-4):
    """<= tol vs the fp32 reference, or -- when fp64 truth exists -- no worse than 2x the reference's own error."""
    e_ref = relmax(got, ref32)
    if e_ref <= tol:
        return True, e_ref
    if f64 is not None:
        e64, r64 = relmax(got, f64), relmax(ref32, f64)
        return e64 <= max(tol, 2 * r64), e64
    return False, e_ref


# ------------------------------------------------------------------ stage 1: H solve
@pytest.mark.parametrize('name', MESH_CASES)
def test_solve_h(mgw, name):
    g = load_golden(name)
    Hs = mgw.ops.solve_h_fwd(dev(g['theta'])).cpu().numpy()
    assert bits_equal(Hs, c_oracle.solve_h(g['theta'])).all(), 'CUDA solve must be bit-identical to the C oracle'
    assert np.abs(Hs - g['ref_Hs']).max() < 1e-5
    if 'f64_Hs' in g:
        assert np.abs(Hs - g['f64_Hs']).max() <= 2 * np.abs(g['ref_Hs'] - g['f64_Hs']).max() + 1e-6


# ------------------------------------------------------------------ stage 2: per-pixel, given the reference's Hs
@pytest.mark.parametrize('impl', IMPLS)
@pytest.mark.parametrize('name', MESH_CASES)
def test_warp_given_reference_hs_bit_exact(mgw, name, impl):
    mgw.set_impl(impl)
    g = load_golden(name)
    U, _, _ = golden_inputs(name, g)
    out, black, img, cell = mgw.ops.warp_fwd(dev(U), dev(g['ref_Hs']), want_cell=(impl == 'generic'))
    assert bits_equal(img.cpu().numpy(), g['ref_img']).all(), 'x_map / y_map'
    assert (black.cpu().numpy() == golden_black(g)).all(), 'black_pix'
    assert bits_equal(out.cpu().numpy(), g['ref_out']).all(), 'output_img'
    if cell is not None:
        assert (cell.cpu().numpy() == c_oracle.warp(U, g['ref_Hs'], want_out=False)[3]).all(), 'cell index'


# ------------------------------------------------------------------ end to end forward
@pytest.mark.parametrize('impl', IMPLS)
@pytest.mark.parametrize('name', MESH_CASES)
def test_transformer_forward(mgw, name, impl):
    mgw.set_impl(impl)
    g = load_golden(name)
    U, _, _ = golden_inputs(name, g)
    out, black, img = mgw.transformer(dev(U), dev(g['theta']))
    out, black, img = out.cpu().numpy(), black.cpu().numpy(), img.cpu().numpy()
    # bit-identical to the C oracle end to end
    o_out, o_black, o_img, _ = c_oracle.warp(U, c_oracle.solve_h(g['theta']))
    assert bits_equal(out, o_out).all() and (black == o_black).all() and bits_equal(img, o_img).all()
    # versus the reference: Hs differs at the 1e-6 level (different LU), so compare to tolerance
    fin = np.isfinite(g['ref_out']).all(-1) & (np.abs(g['ref_img']).max(-1) < 4)
    assert np.abs(img - g['ref_img'])[fin].max() < 2e-5
    rb = golden_black(g)
    knife = (np.abs(np.abs(g['ref_img']) - 1).min(-1) < 2e-5)          # |coord| within a few ulp of the +-1 edge
    assert ((black != rb) & ~knife & fin).sum() == 0
    if str(g['kind']) == 'smooth':
        assert np.abs(out - g['ref_out'])[fin].max() < 1e-5


# ------------------------------------------------------------------ backward
BWD_CASES = SMALL_MESH_CASES[:5] + ['mesh_tma_ragged', 'mesh_tma_c1', 'mesh_tma_c4_g22'] + FULL_MESH_CASES


@pytest.mark.parametrize('impl', IMPLS)
@pytest.mark.parametrize('name', BWD_CASES)
def test_warp_backward_given_reference_hs(mgw, name, impl):
    """stage K3: with the reference's own Hs the taps are identical, so dU / dHs differ from the reference's autograd
    only by fp32 summation order."""
    mgw.set_impl(impl)
    g = load_golden(name)
    U, d_out, d_img = golden_inputs(name, g)
    dU, dHs = mgw.ops.warp_bwd(dev(U), dev(g['ref_Hs']), dev(d_out), dev(d_img))
    assert relmax(dHs.cpu().numpy()[..., :8], g['ref_dHs'][..., :8]) < 1e-4
    assert (dHs.cpu().numpy()[..., 8] == 0).all()
    if 'ref_dU' in g:
        assert relmax(dU.cpu().numpy(), g['ref_dU']) < 1e-4
    # d_img = None and dU skipped are the same numbers minus those terms
    dU0, dHs0 = mgw.ops.warp_bwd(dev(U), dev(g['ref_Hs']), dev(d_out), dev(np.zeros_like(d_img)), want_dU=False)
    dU1, dHs1 = mgw.ops.warp_bwd(dev(U), dev(g['ref_Hs']), dev(d_out), None)
    assert dU0 is None and relmax(dHs0.cpu().numpy(), dHs1.cpu().numpy()) < 5e-5      # two runs of fp32 atomics (generic path)


@pytest.mark.parametrize('name', BWD_CASES)
def test_solve_h_backward(mgw, name):
    """stage K4: dtheta from (theta, Hs, dHs) against fp64 autograd of the oracle's solve (the reference's own fp32
    inverse is the less accurate side here; its distance from fp64 is printed next to ours)."""
    import mesh_warp_ref as ref
    g = load_golden(name)
    th64 = torch.tensor(g['theta'], dtype=torch.float64, requires_grad=True)
    H64 = ref.solve_h(th64)
    up = torch.tensor(g['ref_dHs'], dtype=torch.float64)
    up[..., 8] = 0
    (H64 * up).sum().backward()
    got = mgw.ops.solve_h_bwd(dev(g['theta']), dev(g['ref_Hs']), dev(g['ref_dHs'])).cpu().numpy()
    e = relmax(got, th64.grad.numpy())
    assert e < 2e-5, 'dtheta (K4) rel err vs fp64 %.3g' % e


@pytest.mark.parametrize('impl', IMPLS)
@pytest.mark.parametrize('name', BWD_CASES)
def test_transformer_backward_end_to_end(mgw, name, impl):
    """autograd through transformer(): <= 1e-4 relative on smooth images.  On white-noise images the gradient is a
    discontinuous function of Hs (a 1e-6 change of H moves taps across pixel boundaries): the reference's own fp32
    result is then ~1e-2 away from its fp64 run, so the bar there is 'no worse than 4x the reference's own error'."""
    mgw.set_impl(impl)
    g = load_golden(name)
    U, d_out, d_img = golden_inputs(name, g)
    Ut = dev(U).requires_grad_(True)
    th = dev(g['theta']).requires_grad_(True)
    out, black, img = mgw.transformer(Ut, th)
    ((out * dev(d_out)).sum() + (img * dev(d_img)).sum()).backward()
    got = th.grad.cpu().numpy()
    e64, r64 = relmax(got, g['f64_dtheta']), relmax(g['ref_dtheta'], g['f64_dtheta'])
    smooth = str(g['kind']) == 'smooth'
    assert e64 <= (max(1e-4, 2 * r64) if smooth else max(1e-4, 4 * r64)), 'dtheta: ours %.3g, reference %.3g (vs fp64)' % (e64, r64)
    if 'f64_dU' in g:
        eu, ru = relmax(Ut.grad.cpu().numpy(), g['f64_dU']), relmax(g['ref_dU'], g['f64_dU'])
        assert eu <= max(1e-4, 4 * ru), 'dU: ours %.3g, reference %.3g (vs fp64)' % (eu, ru)


@pytest.mark.parametrize('name', TMA_MESH_CASES + FULL_MESH_CASES)
def test_tma_path_is_taken_and_matches_generic(mgw, name):
    """set_impl('tma') errors out instead of falling back; TMA forward == generic forward bit for bit."""
    g = load_golden(name)
    U, d_out, d_img = golden_inputs(name, g)
    Ud, Hd = dev(U), dev(g['ref_Hs'])
    mgw.set_impl('generic')
    o_g, b_g, i_g, _ = mgw.ops.warp_fwd(Ud, Hd)
    dU_g, dH_g = mgw.ops.warp_bwd(Ud, Hd, dev(d_out), dev(d_img))
    mgw.set_impl('tma')
    o_t, b_t, i_t, _ = mgw.ops.warp_fwd(Ud, Hd)
    dU_t, dH_t = mgw.ops.warp_bwd(Ud, Hd, dev(d_out), dev(d_img))
    only_img = mgw.ops.warp_fwd(Ud, Hd, want_out=False, want_black=False)[2]
    assert torch.equal(o_g.view(torch.int32), o_t.view(torch.int32)) and torch.equal(b_g, b_t)
    assert torch.equal(i_g.view(torch.int32), i_t.view(torch.int32)) and torch.equal(only_img.view(torch.int32), i_t.view(torch.int32))
    s0 = 1 if 'fold' in name else 0      # a folded cell scatters 1e5-weighted terms: order-dependent garbage in any implementation
    assert relmax(dU_t[s0:].cpu().numpy(), dU_g[s0:].cpu().numpy()) < 2e-5      # fixed-point (tile) vs fp32 atomics (generic)
    if 'fold' not in name:
        assert relmax(dH_t.cpu().numpy(), dH_g.cpu().numpy()) < 5e-5      # (the generic dH is a sum of fp32 atomics)
    dU_n, dH_n = mgw.ops.warp_bwd(Ud, Hd, dev(d_out), None, want_dU=False)      # the no-dU / no-d_img variant of the kernel
    assert dU_n is None and torch.isfinite(dH_n).all() or 'fold' in name
    mgw.set_impl('auto')


@pytest.mark.parametrize('name', TMA_MESH_CASES + FULL_MESH_CASES)
def test_pipe_path_is_taken_and_matches_generic(mgw, name):
    """set_impl('pipe') (forward as a persistent warp-specialised pipeline) errors out instead of falling back; == generic bit for bit."""
    g = load_golden(name)
    U, d_out, d_img = golden_inputs(name, g)
    Ud, Hd = dev(U), dev(g['ref_Hs'])
    mgw.set_impl('generic')
    o_g, b_g, i_g, _ = mgw.ops.warp_fwd(Ud, Hd)
    dU_g, dH_g = mgw.ops.warp_bwd(Ud, Hd, dev(d_out), dev(d_img))
    mgw.set_impl('pipe')
    o_t, b_t, i_t, _ = mgw.ops.warp_fwd(Ud, Hd)
    assert torch.equal(o_g.view(torch.int32), o_t.view(torch.int32)) and torch.equal(b_g, b_t)
    assert torch.equal(i_g.view(torch.int32), i_t.view(torch.int32))
    # the backward under 'pipe' runs the tile kernels (fixed-point shared accumulation, 16-byte reductions) vs fp32 atomics (generic)
    dU_t, dH_t = mgw.ops.warp_bwd(Ud, Hd, dev(d_out), dev(d_img))
    s0 = 1 if 'fold' in name else 0      # a folded cell scatters 1e5-weighted terms: order-dependent garbage in any implementation
    assert relmax(dU_t[s0:].cpu().numpy(), dU_g[s0:].cpu().numpy()) < 2e-5
    if 'fold' not in name:
        assert relmax(dH_t.cpu().numpy(), dH_g.cpu().numpy()) < 5e-5
    dU_r, dH_r = mgw.ops.warp_bwd(Ud, Hd, dev(d_out), dev(d_img))               # run to run: dH partials are deterministic
    assert torch.equal(dH_r, dH_t)
    with pytest.raises(mgw.MgwError):                                          # the pipeline serves the full call only
        mgw.ops.warp_fwd(Ud, Hd, want_black=False, want_img=False)
    o_r = mgw.ops.warp_fwd(Ud, Hd)[0]                                          # run to run
    assert torch.equal(o_r.view(torch.int32), o_t.view(torch.int32))
    mgw.set_impl('auto')


def _random_shapes():
    rng = np.random.RandomState(2024)
    shapes = []
    for _ in range(14):
        gh, gw = int(rng.choice([1, 2, 3, 4])), int(rng.choice([1, 2, 3, 4, 6]))
        c = int(rng.choice([1, 3, 4]))
        n = int(rng.choice([1, 2, 3]))
        h = int(rng.randint(max(24, 9 * gh), 200))
        w = 4 * int(rng.randint(max(16, 9 * gw), 70))
        shapes.append((n, h, w, c, gh, gw, float(rng.choice([0.0, 0.03, 0.08, 0.2])), int(rng.randint(1 << 30))))
    return shapes


@pytest.mark.parametrize('shape', _random_shapes(), ids=lambda s: '%dx%dx%dx%d_g%dx%d_s%g' % s[:7])
def test_random_shapes_all_kernel_families_agree(mgw, shape):
    """whatever family `auto` picks for a shape (pipeline, tiles, generic -- ragged meshes, tiles shifted onto their
    neighbours, boxes that overflow, clamped and folded vertices), the forward equals the generic kernels bit for bit and
    the backward agrees to rounding."""
    import synth
    n, h, w, c, gh, gw, sigma, seed = shape
    U = dev(synth.noise_image(n, h, w, c, seed))
    th = dev(synth.random_mesh(n, gh, gw, sigma, seed + 1))
    go = dev(synth.randn((n, h, w, c), seed + 2)); gi = dev(synth.randn((n, h, w, 2), seed + 3, 0.1))
    mgw.set_impl('generic')
    o_g, b_g, i_g, Hs = mgw.ops.mesh_warp_fwd(U, th)
    dU_g, dH_g = mgw.ops.warp_bwd(U, Hs, go, gi)
    mgw.set_impl('auto')
    o_a, b_a, i_a, Hs_a = mgw.ops.mesh_warp_fwd(U, th)
    dU_a, dH_a = mgw.ops.warp_bwd(U, Hs, go, gi)
    assert torch.equal(Hs, Hs_a)
    fin = torch.isfinite(o_g)
    assert torch.equal(o_g.view(torch.int32)[fin], o_a.view(torch.int32)[fin]) and torch.equal(torch.isfinite(o_a), fin)
    assert torch.equal(b_g, b_a)
    fi = torch.isfinite(i_g)
    assert torch.equal(i_g.view(torch.int32)[fi], i_a.view(torch.int32)[fi])
    # gradients at the SAME Hs, before the adjoint solve (which amplifies fp32 summation noise by the conditioning of the
    # cell's 8x8 system, in any implementation); folded cells (sigma 0.2) scatter order-dependent garbage everywhere
    if sigma <= 0.08 and torch.isfinite(dU_g).all() and torch.isfinite(dH_g).all():
        assert relmax(dU_a.cpu().numpy(), dU_g.cpu().numpy()) < 5e-5
        assert relmax(dH_a.cpu().numpy(), dH_g.cpu().numpy()) < 5e-5


def test_tma_rejects_shapes_it_cannot_serve(mgw):
    g = load_golden('mesh_ragged_c1')            # 50 x 70: row pitch not a multiple of 16 bytes
    U, _, _ = golden_inputs('mesh_ragged_c1', g)
    mgw.set_impl('tma')
    with pytest.raises(mgw.MgwError):
        mgw.ops.warp_fwd(dev(U), dev(g['ref_Hs']))
    mgw.set_impl('auto')


def test_backward_accumulates_into_callers_dU(mgw):
    """mgw_warp_bwd_acc / mgw_mesh_warp_bwd_acc: dU += gradient, never zero-filled by the library."""
    g = load_golden('mesh_tma_fold_clamp_shift')
    U, d_out, d_img = golden_inputs('mesh_tma_fold_clamp_shift', g)
    Ud, Hd, th = dev(U[1:]), dev(g['ref_Hs'][1:]), dev(g['theta'][1:])
    go, gi = dev(d_out[1:]), dev(d_img[1:])
    for impl in IMPLS:
        mgw.set_impl(impl)
        dU, dHs = mgw.ops.warp_bwd(Ud, Hd, go, gi)
        buf = torch.full_like(Ud, 3.0)
        dU2, dHs2 = mgw.ops.warp_bwd(Ud, Hd, go, gi, accumulate_into=buf)
        assert dU2.data_ptr() == buf.data_ptr() and relmax(dHs2.cpu().numpy(), dHs.cpu().numpy()) < 5e-5
        assert relmax((buf - 3.0).cpu().numpy(), dU.cpu().numpy()) < 5e-5
        buf = torch.full_like(Ud, -1.0)
        dU3, dth3 = mgw.ops.mesh_warp_bwd(Ud, th, mgw.ops.solve_h_fwd(th), go, gi, accumulate_into=buf)
        dU4, dth4 = mgw.ops.mesh_warp_bwd(Ud, th, mgw.ops.solve_h_fwd(th), go, gi)
        assert relmax((buf + 1.0).cpu().numpy(), dU4.cpu().numpy()) < 5e-5 and relmax(dth3.cpu().numpy(), dth4.cpu().numpy()) < 5e-5
    mgw.set_impl('auto')


@pytest.mark.parametrize('name', ['mesh_full_noise_s05', 'mesh_tma_ragged', 'mesh_tma_c1'])
def test_backward_workspace_needs_no_initialisation(mgw, name):
    """the dH partial slots are all written (uniform mesh) or zero-filled by the library (ragged): a NaN-filled workspace
    must give the same dtheta as a zeroed one."""
    from dovs_b200._lib import lib, check
    g = load_golden(name)
    U, d_out, d_img = golden_inputs(name, g)
    Ud, th, go, gi = dev(U), dev(g['theta']), dev(d_out), dev(d_img)
    Hs = mgw.ops.solve_h_fwd(th)
    n, h, w, c = Ud.shape
    gh, gw = Hs.shape[1:3]
    nbytes = lib.mgw_mesh_warp_bwd_workspace_bytes(n, h, w, c, gh, gw)
    res = []
    for fill in (0.0, float('nan')):
        ws = torch.full((nbytes // 4 + 64,), fill, device='cuda')
        dU, dth = torch.empty_like(Ud), torch.empty_like(th)
        check(lib.mgw_mesh_warp_bwd(Ud.data_ptr(), th.data_ptr(), Hs.data_ptr(), go.data_ptr(), gi.data_ptr(), n, h, w, c, gh, gw,
                                    dU.data_ptr(), dth.data_ptr(), ws.data_ptr(), torch.cuda.current_stream().cuda_stream), 'bwd')
        res.append(dth.clone())
    assert torch.isfinite(res[1]).all() and torch.equal(res[0], res[1])


def test_backward_without_dU_and_without_dimg(mgw):
    g = load_golden('mesh_smooth_s03')
    U, d_out, _ = golden_inputs('mesh_smooth_s03', g)
    th = dev(g['theta']).requires_grad_(True)
    out, _, _ = mgw.transformer(dev(U), th)           # U does not require grad: dU is skipped (reference: U is a placeholder)
    (out * dev(d_out)).sum().backward()
    th2 = dev(g['theta']).requires_grad_(True)
    Ut = dev(U).requires_grad_(True)
    out2, _, _ = mgw.transformer(Ut, th2)
    (out2 * dev(d_out)).sum().backward()
    assert relmax(th.grad.cpu().numpy(), th2.grad.cpu().numpy()) < 5e-5      # two runs of the generic path's fp32 atomics


# ------------------------------------------------------------------ interpolate
@pytest.mark.parametrize('name', ['interp_same', 'interp_resize_c1'])
def test_interpolate(mgw, name):
    g = load_golden(name)
    oh, ow = g['x'].shape[1:3]
    it, xt, yt = dev(g['im']).requires_grad_(True), dev(g['x']).requires_grad_(True), dev(g['y']).requires_grad_(True)
    out = mgw.interpolate(it, xt, yt, (oh, ow))
    assert bits_equal(out.detach().cpu().numpy(), g['ref_out']).all()
    (out * dev(g['d_out'])).sum().backward()
    for got, key in ((it.grad, 'dim'), (xt.grad, 'dx'), (yt.grad, 'dy')):
        ok, e = grad_ok(got.cpu().numpy(), g['ref_' + key], g['f64_' + key], tol=1e-5)
        assert ok, '%s rel err %.3g' % (key, e)


# ------------------------------------------------------------------ single homography
@pytest.mark.parametrize('name', ['homog_s05', 'homog_c1_s10'])
def test_homography_transformer(mgw, name):
    g = load_golden(name)
    n, h, w, c = g['U'].shape
    Ut, th = dev(g['U']).requires_grad_(True), dev(g['theta']).requires_grad_(True)
    out, black = mgw.spatial_transformer.transformer(Ut, th, (h, w))
    assert bits_equal(out.detach().cpu().numpy(), g['ref_out']).all()
    assert (black.cpu().numpy() == g['ref_black']).all()
    (out * dev(g['d_out'])).sum().backward()
    ok, e = grad_ok(Ut.grad.cpu().numpy(), g['ref_dU'], g['f64_dU'])
    assert ok, 'dU %.3g' % e
    ok, e = grad_ok(th.grad.cpu().numpy(), g['ref_dtheta'], g['f64_dtheta'])
    assert ok, 'dtheta %.3g' % e


def test_homography_out_size_differs_from_input(mgw):
    """the reference breaks here (spatial_transformer.py:184); we follow the C oracle."""
    g = load_golden('homog_s05')
    out, black = mgw.spatial_transformer.transformer(dev(g['U']), dev(g['theta']), (40, 72))
    o_out, o_black, _ = c_oracle.homography_warp(g['U'], g['theta'], (40, 72))
    assert bits_equal(out.cpu().numpy(), o_out).all() and (black.cpu().numpy() == o_black).all()


def test_north_star_signature_dispatches_mesh(mgw):
    g = load_golden('mesh_smooth_s03')
    U, _, _ = golden_inputs('mesh_smooth_s03', g)
    out, black, img = mgw.spatial_transformer.transformer(dev(U), dev(g['theta']), (U.shape[1], U.shape[2]))
    out3, _, _ = mgw.spatial_transformer3.transformer(dev(U), dev(g['theta']))
    assert torch.equal(out, out3)
    named = mgw.spatial_transformer3.named_outputs(dev(U), dev(g['theta']))
    assert set(named) == {'output_img', 'black_pix', 'Hs', 'x_map', 'y_map'}
    assert named['x_map'].shape == (U.shape[0], U.shape[1], U.shape[2], 1)


# ------------------------------------------------------------------ vertices + losses
def test_vertices_and_losses(mgw):
    g = load_golden('losses')
    gh, gw = (int(v) for v in g['grid'])
    n, h, w, _ = g['x1'].shape
    hd, hd2 = dev(g['head']).requires_grad_(True), dev(g['head2']).requires_grad_(True)
    pts1, pts2 = mgw.get_4_pts(hd, n, (gh, gw))
    _, pts2b = mgw.get_4_pts(hd2, n, (gh, gw))
    assert bits_equal(pts1.detach().cpu().numpy(), g['ref_pts1']).all()
    assert bits_equal(pts2.detach().cpu().numpy(), g['ref_pts2']).all()
    out1, black1, img1 = mgw.transformer(dev(g['x1']), pts2)
    out2, black2, img2 = mgw.transformer(dev(g['x2']), pts2b)
    fl, warpped = mgw.feature_loss(dev(g['matches']), dev(g['mask']), img1)
    il = mgw.img_loss(out1, dev(g['y1']), black1)
    tl = mgw.temp_loss(out1, black1, out2, black2, dev(g['flow']))
    assert np.abs(warpped.cpu().numpy() - g['ref_stable_warpped']).max() < 2e-5
    for nm, l in (('feature', fl), ('img', il), ('temp', tl)):
        want = float(g['ref_%s_loss' % nm])
        assert abs(float(l) - want) <= 2e-5 * max(1.0, abs(want)), (nm, float(l), want)
        gr = torch.autograd.grad(l, [hd, hd2], retain_graph=True, allow_unused=True)
        for k, t in (('dhead', gr[0]), ('dhead2', gr[1])):
            ref32, f64 = g['ref_%s_%s' % (k, nm)], g['f64_%s_%s' % (k, nm)]
            got = np.zeros_like(ref32) if t is None else t.cpu().numpy()
            if np.abs(ref32).max() == 0:
                assert np.abs(got).max() == 0, (nm, k)
            else:
                ok, e = grad_ok(got, ref32, f64, tol=2e-4)
                assert ok, '%s %s rel err %.3g' % (nm, k, e)


@pytest.mark.parametrize('impl', IMPLS)
@pytest.mark.parametrize('shape', [(2, 96, 160, 3), (2, 48, 64, 1)])
def test_fused_img_loss_equals_unfused(mgw, impl, shape):
    """transformer_img_loss (loss sums inside the warp kernel, d_out formed in registers) == transformer + img_loss, and
    == the oracle port's fp64 autograd at the same inputs."""
    import mesh_warp_ref as ref
    import synth
    mgw.set_impl(impl)
    n, h, w, c = shape
    U, y = synth.smooth_image(n, h, w, c, 700), synth.smooth_image(n, h, w, c, 701)
    theta = synth.random_mesh(n, 4, 4, 0.05, 702)
    d_img = synth.randn((n, h, w, 2), 703, 1e-4)
    Ua, ta = dev(U).requires_grad_(True), dev(theta).requires_grad_(True)
    loss_f, out_f, black_f, img_f = mgw.transformer_img_loss(Ua, ta, dev(y))
    (loss_f * 3.0 + (img_f * dev(d_img)).sum()).backward()
    Ub, tb = dev(U).requires_grad_(True), dev(theta).requires_grad_(True)
    out_u, black_u, img_u = mgw.transformer(Ub, tb)
    loss_u = mgw.img_loss(out_u, dev(y), black_u)
    (loss_u * 3.0 + (img_u * dev(d_img)).sum()).backward()
    assert torch.equal(out_f, out_u) and torch.equal(black_f, black_u) and torch.equal(img_f, img_u)
    assert abs(float(loss_f) - float(loss_u)) <= 1e-5 * abs(float(loss_u))
    assert relmax(ta.grad.cpu().numpy(), tb.grad.cpu().numpy()) < 1e-4
    assert relmax(Ua.grad.cpu().numpy(), Ub.grad.cpu().numpy()) < 1e-4
    # fused loss with ANOTHER gradient on the output takes the unfused backward and must still be right
    Uc, tc = dev(U).requires_grad_(True), dev(theta).requires_grad_(True)
    loss_c, out_c, _, _ = mgw.transformer_img_loss(Uc, tc, dev(y))
    (loss_c * 3.0 + (out_c * dev(d_img[..., :1]).expand_as(out_c)).sum()).backward()
    Ud, td = dev(U).requires_grad_(True), dev(theta).requires_grad_(True)
    out_d, black_d, _ = mgw.transformer(Ud, td)
    (mgw.img_loss(out_d, dev(y), black_d) * 3.0 + (out_d * dev(d_img[..., :1]).expand_as(out_d)).sum()).backward()
    assert relmax(tc.grad.cpu().numpy(), td.grad.cpu().numpy()) < 1e-4
    # and against the oracle (fp64 port) for the loss value
    o64, b64, _, _ = ref.transformer(torch.tensor(U, dtype=torch.float64), torch.tensor(theta, dtype=torch.float64))
    l64 = float(ref.img_loss(o64, torch.tensor(y, dtype=torch.float64), b64))
    assert abs(float(loss_f) - l64) <= 2e-5 * abs(l64)


# ------------------------------------------------------------------ full-size properties (config #2: 32 x 288 x 512 x 3)
@pytest.fixture(scope='module')
def full():
    import synth
    n, h, w, c = 32, 288, 512, 3
    return dict(U=synth.noise_image(n, h, w, c, 900), theta=synth.random_mesh(n, 4, 4, 0.05, 901),
                d_out=synth.randn((n, h, w, c), 902), d_img=synth.randn((n, h, w, 2), 903, 0.1))


@pytest.mark.parametrize('impl', IMPLS)
def test_full_size_properties(mgw, full, impl):
    mgw.set_impl(impl)
    U, th = dev(full['U']), dev(full['theta'])
    out, black, img, Hs = mgw.ops.mesh_warp_fwd(U, th)
    # (1) the C oracle on a slice of the batch: bit-exact
    for n in (0, 17, 31):
        o_out, o_black, o_img, _ = c_oracle.warp(full['U'][n:n + 1], c_oracle.solve_h(full['theta'][n:n + 1]))
        assert bits_equal(out[n:n + 1].cpu().numpy(), o_out).all()
        assert (black[n:n + 1].cpu().numpy() == o_black).all() and bits_equal(img[n:n + 1].cpu().numpy(), o_img).all()
    # (2) batch independence and determinism: sample n alone == sample n inside the batch, bit for bit
    o1, b1, i1, _ = mgw.ops.mesh_warp_fwd(U[5:6].contiguous(), th[5:6].contiguous())
    assert torch.equal(o1, out[5:6]) and torch.equal(b1, black[5:6]) and torch.equal(i1, img[5:6])
    o2 = mgw.ops.mesh_warp_fwd(U, th)[0]
    assert torch.equal(o2, out)
    # (3) linearity in U (bilinear sampling is linear): warp(U) + warp(V) == warp(U+V) to rounding
    V = torch.flip(U, dims=[0])
    lhs = mgw.ops.warp_fwd(U + V, Hs)[0]
    rhs = out + mgw.ops.warp_fwd(V, Hs)[0]
    assert (lhs - rhs).abs().max().item() < 2e-5
    # (4) adjoint identity of the backward at full size: <warp(U), G> == <U, dU(G)>
    G = dev(full['d_out'])
    dU, dHs = mgw.ops.warp_bwd(U, Hs, G, dev(full['d_img']))
    lhs = (out.double() * G.double()).sum().item()
    rhs = (U.double() * dU.double()).sum().item()
    assert abs(lhs - rhs) <= 1e-5 * max(abs(lhs), (out.double() * G.double()).abs().sum().item() * 1e-2)
    # (5) dtheta by central differences in fp64-ish (directional derivative along a random direction)
    dU2, dth = mgw.ops.mesh_warp_bwd(U[:2].contiguous(), th[:2].contiguous(), Hs[:2].contiguous(), G[:2].contiguous(), None)
    assert torch.isfinite(dth).all() and torch.isfinite(dU2).all()


# ------------------------------------------------------------------ deploy side: warpRevBundle2
@pytest.mark.parametrize('tag', ['net', 'ragged', 'identity'])
def test_deploy_remap_byte_exact(mgw, tag):
    """mgw_remap_bundle_u8 == the reference's warpRevBundle2 (OpenCV plain path) byte for byte; numpy in -> numpy out."""
    g = load_golden('deploy_remap')
    img, xm, ym, ref = g[tag + '_img'], g[tag + '_x_map'], g[tag + '_y_map'], g[tag + '_ref_dst']
    dst = mgw.warpRevBundle2(img, xm, ym)
    assert isinstance(dst, np.ndarray) and dst.dtype == np.uint8 and np.array_equal(dst, ref)
    # batched, on the device, straight from the operator's interleaved x/y maps; sample independence
    xy = dev(np.stack([xm, ym], -1)[None].repeat(3, 0))
    xy[1] = torch.flip(xy[1], dims=[0])
    im3 = torch.tensor(img, device='cuda')[None].repeat(3, 1, 1, 1)
    out3 = mgw.ops.remap_bundle_u8(im3, xy)
    assert np.array_equal(out3[0].cpu().numpy(), ref) and np.array_equal(out3[2].cpu().numpy(), ref)
    import deploy_ref
    assert np.array_equal(out3[1].cpu().numpy(), deploy_ref.warp_rev_bundle2(img, xy[1, ..., 0].cpu().numpy(), xy[1, ..., 1].cpu().numpy()))
    # one channel, and coordinates that are NaN / far outside: constant border 0 like cv2.remap
    xy1 = dev(np.stack([xm, ym], -1)[None].copy())
    xy1[0, :4, :4, 0] = float('nan'); xy1[0, 4:8, :4, 1] = 1e30
    g1 = mgw.ops.remap_bundle_u8(torch.tensor(img[None, ..., :1].copy(), device='cuda'), xy1)
    want = deploy_ref.warp_rev_bundle2(img[..., :1], np.nan_to_num(xy1[0, ..., 0].cpu().numpy(), nan=-1e30), xy1[0, ..., 1].cpu().numpy())
    assert np.array_equal(g1[0].cpu().numpy(), want)


def test_deploy_warp_rev_bundle_byte_exact(mgw):
    """warpRevBundle (mgw_warp_rev_bundle_u8) == the reference's function on OpenCV (fixture), and C = 1 / 4, batched, against
    the restatement"""
    import deploy_ref
    g = load_golden('deploy_warp_rev_bundle')
    for n in sorted(k[:-4] for k in g if k.endswith('_dst')):
        gh, gw = (int(v) for v in g[n + '_grid'])
        got = mgw.warpRevBundle(g[n + '_img'], g[n + '_Hs'], grid=(gh, gw))
        assert isinstance(got, np.ndarray) and np.array_equal(got, g[n + '_dst']), n
    assert np.array_equal(mgw.deploy.warpRev(g['strong_img'], g['warprev_theta']), g['warprev_out'])       # warpRev (:113-117)
    # CUDA tensors in -> CUDA tensor out
    got = mgw.warpRevBundle(torch.as_tensor(g['ragged_img']).cuda(), torch.as_tensor(g['ragged_Hs']).cuda(), grid=(3, 4))
    assert got.is_cuda and np.array_equal(got.cpu().numpy(), g['ragged_dst'])
    # other channel counts and a batch through the op
    r = np.random.RandomState(9)
    for c in (1, 4):
        h, w, gh, gw = 60, 88, 2, 4
        imgs = r.randint(0, 256, (2, h, w, c)).astype(np.uint8)
        Hs = [g['strong_Hs'].reshape(2, 2, 9)[[0, 1]][:, [0, 1, 0, 1]], g['ragged_Hs'].reshape(3, 4, 9)[:2]]
        Hc = np.stack([deploy_ref.cvt_theta_mat_bundle(Hs[k], h, w, gh, gw) for k in range(2)])
        got = mgw.ops.warp_rev_bundle_u8(torch.as_tensor(imgs).cuda(), torch.as_tensor(Hc).cuda(), gh, gw).cpu().numpy()
        for k in range(2):
            want = deploy_ref.warp_rev_bundle(np.repeat(imgs[k], 3, -1)[..., :3] if c == 1 else imgs[k][..., :3], Hs[k], gh, gw)
            assert np.array_equal(got[k][..., 0], want[..., 0]), (c, k)


def test_cvt_img2train_exact(mgw):
    """deploy.cvt_img2train (mgw_cvt_img2train_u8) == the reference's config.py function on OpenCV + Pillow (fixture), and a
    1080p frame against the restatement"""
    import deploy_ref
    g = load_golden('deploy_cvt_img2train')
    for n in sorted(k[:-4] for k in g if k.endswith('_out')):
        h, w, cr = g[n + '_cfg']
        cr = 1 if cr == 1 else float(cr)
        out = mgw.deploy.cvt_img2train(g[n + '_img'], cr, height=int(h), width=int(w))
        assert out.is_cuda and out.dtype == torch.float32 and out.shape == (1, int(h), int(w), 1)
        assert np.array_equal(out.cpu().numpy(), g[n + '_out'].astype(np.float32)), n
        assert np.array_equal(mgw.deploy.cvt_img2train(g[n + '_img'], cr, height=int(h), width=int(w), as_numpy=True), g[n + '_out']), n
    img = np.random.RandomState(4).randint(0, 256, (1080, 1920, 3)).astype(np.uint8)
    want = deploy_ref.cvt_img2train(img, 288, 512).astype(np.float32)
    assert np.array_equal(mgw.deploy.cvt_img2train(img).cpu().numpy(), want)


def test_cv2_resize_byte_exact(mgw):
    """deploy.cv2_resize (mgw_resize_linear_u8) == cv2.resize of the uint8 frame (fixture made by OpenCV), and the deploy loop's
    own size (1080p -> 512x288) against the restatement"""
    import deploy_ref
    g = load_golden('deploy_cv2_resize')
    for n in sorted(k[:-4] for k in g if k.endswith('_dst')):
        want = g[n + '_dst']
        img = g[n + '_img']
        got = mgw.deploy.cv2_resize(img if img.ndim == 3 else img[..., None], (want.shape[1], want.shape[0]))
        assert np.array_equal(got.reshape(want.shape), want), n
    img = np.random.RandomState(6).randint(0, 256, (1080, 1920, 3)).astype(np.uint8)
    got = mgw.deploy.cv2_resize(torch.as_tensor(img).cuda(), (512, 288))
    assert got.is_cuda and np.array_equal(got.cpu().numpy(), deploy_ref.resize_linear_u8(img, 512, 288))


def test_deploy_stream_state_exact(mgw):
    """StreamState (device rings, mgw_stream_assemble / mgw_stream_push) == the reference's per-frame list handling."""
    import deploy_ref
    g = load_golden('deploy_stream')
    st = mgw.StreamState(g['first'])
    for k in range(g['cur_frames'].shape[0]):
        in_x = st.assemble(g['cur_frames'][k])
        assert np.array_equal(in_x.cpu().numpy(), g['in_x'][k])
        for _ in range(int(g['refine'])):
            img, black = deploy_ref.stream_fake_net(in_x.cpu().numpy(), k)
            img_d, black_d = dev(img), dev(black)
            st.refeed(in_x, img_d, black_d)
        assert np.array_equal(in_x.cpu().numpy(), g['tmp_in_x'][k])
        st.push(img_d, black_d)
    fr, mk = st.history()
    assert np.array_equal(fr.cpu().numpy()[..., None], g['final_frames']) and np.array_equal(mk.cpu().numpy()[..., None], g['final_masks'])


def test_vertex_regularisers_match_the_reference(mgw):
    """id / black_pos / distortion / consistency (mgw_vertex_losses_fwd/bwd) against the reference's own functions (fixture):
    values 1e-5 relative, gradients 1e-4 of the largest entry (north_star tolerances; observed ~1e-6)."""
    g = load_golden('vertex_losses')

    def close(a, b, tol):
        a, b = np.asarray(a.detach().cpu() if torch.is_tensor(a) else a, np.float64), np.asarray(b, np.float64)
        assert a.shape == b.shape, (a.shape, b.shape)
        return np.abs(a - b).max() <= tol * max(np.abs(b).max(), 1e-30) + 1e-12

    for gi, (gh, gw) in enumerate(g['grids']):
        gh, gw = int(gh), int(gw)
        head = dev(g['g%d_head' % gi]).requires_grad_(True)
        raw = dev(g['g%d_raw' % gi]).requires_grad_(True)
        pts1, pts2 = mgw.get_4_pts(head, grid=(gh, gw))
        pts1.retain_grad(); pts2.retain_grad()
        idl, _, dist, cons = mgw.vertex_losses(head, pts1, pts2)
        black = mgw.get_black_pos_loss(raw)
        assert mgw.get_black_pos_loss(pts1).item() == 0.0            # clamped vertices cannot overshoot (get_4_pts :58)
        for tag in ('ref', 'f64'):
            k = 'g%d_%s_' % (gi, tag)
            assert close(idl, g[k + 'id'], 1e-5) and close(black, g[k + 'black'], 1e-5), (gh, gw, tag)
            assert close(dist, g[k + 'dist'], 1e-5) and close(cons, g[k + 'cons'], 1e-5), (gh, gw, tag)
        assert np.array_equal(mgw.get_black_pos(raw).cpu().numpy(), g['g%d_ref_black_err' % gi])
        k = 'g%d_f64_' % gi
        assert close(torch.autograd.grad(idl, head, retain_graph=True)[0], g[k + 'did_dhead'], 1e-6)
        assert close(torch.autograd.grad(black, raw)[0], g[k + 'dblack_draw'], 1e-5)
        gd = torch.autograd.grad(dist, [head, pts1], retain_graph=True)
        assert close(gd[0], g[k + 'ddist_dhead'], 1e-5) and close(gd[1], g[k + 'ddist_dpts1'], 1e-5), (gh, gw)
        if cons.requires_grad and np.abs(g[k + 'dcons_dpts2']).max() > 0:
            gc = torch.autograd.grad(cons, [head, pts2], retain_graph=True)
            assert close(gc[0], g[k + 'dcons_dhead'], 1e-5) and close(gc[1], g[k + 'dcons_dpts2'], 1e-5), (gh, gw)
        # the named single-term entry points are the same numbers
        assert float(mgw.get_distortion_loss(pts1)) == float(dist) and float(mgw.get_consistency_loss(pts2)) == float(cons)


def test_total_loss_and_schedule(mgw):
    """total_loss (s_net_bundle_nobm.py:354-359) and loss_gates (train_bundle_nobm.py:219-236) against the restatement; the
    gradient of the whole head-only part reaches the head through ONE vertex-loss backward + mgw_vertices_bwd."""
    import vertex_loss_ref as V
    for i in (0, 100, 101, 999, 1000, 4999, 5000, 10 ** 6 + 1):
        gates = mgw.loss_gates(i)
        assert (gates['use_theta'], gates['use_temp'], gates['use_black'], gates['theta_only']) == V.loss_gates(i)
    g = load_golden('vertex_losses')
    head_np, raw = g['g0_head'], g['g0_raw']
    head = dev(head_np).requires_grad_(True)
    pts1, pts2 = mgw.get_4_pts(head, grid=(4, 4))
    img_l, feat_l = torch.tensor(0.37, device='cuda'), torch.tensor(0.011, device='cuda')
    total, parts = mgw.total_loss(head, pts1, pts2, img_l, feat_l, regu_loss=0.5, use_black_loss=1.0, use_theta_only=0.0)
    p1, p2 = g['g0_f64_pts1'], g['g0_f64_pts2']
    idl, gid = V.id_loss(head_np.astype(np.float64))
    bl, _, _ = V.black_pos_loss(p1)
    dl, gd1 = V.distortion_loss(p1, 4, 4)
    cl, gc2 = V.consistency_loss(p2, 4, 4)
    m = mgw.losses.V2_93_MULS
    want = V.total_loss(idl * m['id_mul'], idl * m['id_mul'], 0.37, 0.5, bl, dl, cl, 0.011, 0.0, m)
    assert abs(float(total) - want) <= 1e-5 * abs(want)
    assert abs(float(parts['consistency_loss']) - cl * m['consistency_mul']) <= 1e-5 * abs(cl * m['consistency_mul'])
    (dh,) = torch.autograd.grad(total, head)
    want_dh = (gid * m['id_mul'] * (m['theta_mul'] + m['grid_theta_mul']) + g['g0_f64_ddist_dhead'] * m['distortion_mul'] +
               g['g0_f64_dcons_dhead'] * m['consistency_mul'])
    assert np.abs(dh.cpu().numpy() - want_dh).max() <= 1e-5 * np.abs(want_dh).max()
    # theta_only = 1 switches everything but the id terms off
    t1, _ = mgw.total_loss(head, pts1, pts2, img_l, feat_l, use_theta_only=1.0)
    assert abs(float(t1) - idl * m['id_mul'] * (m['theta_mul'] + m['grid_theta_mul'])) <= 1e-6 * float(t1)


def test_stabnet_train_objective_flows_end_to_end(mgw):
    """StabNet carrier + this library's path: two passes + temp loss (train_bundle_nobm.py:107-141); the objective is finite,
    every parameter receives a gradient, and the image-side parts equal the standalone entry points."""
    import synth
    torch.manual_seed(1)
    n, h, w = 2, 64, 96
    net = mgw.StabNet(in_ch=13, grid=(4, 4)).cuda()

    def batch(seed):
        return dict(x=dev(synth.smooth_image(n, h, w, 13, seed)), y=dev(synth.smooth_image(n, h, w, 1, seed + 1)),
                    matches=dev(synth.uniform((n, 30, 4), -1, 1, seed + 2)), mask=dev((synth.uniform((n, 30), 0, 1, seed + 3) < 0.5).astype(np.float32)))

    b1, b2 = batch(10), batch(20)
    flow = dev(synth.uniform((n, h, w, 2), -1, 1, 30))
    total, ret1, ret2, t_loss = mgw.train_losses(net, b1, b2, flow, mgw.loss_gates(6000))
    assert torch.isfinite(total) and ret1['output'].shape == (n, h, w, 1) and ret1['black_pix'].shape == (n, h, w, 1)
    total.backward()
    missing = [k for k, p in net.named_parameters() if p.grad is None or not torch.isfinite(p.grad).all()]
    assert not missing, missing
    assert float(net.backbone.conv1.weight.grad.abs().max()) > 0
    # parts: the fused img_loss inside equals the standalone op on the same warped output
    x = b1['x'][..., 12:13].contiguous()
    out, black, _ = mgw.transformer(x, ret1['pts2'].detach())
    il = mgw.img_loss(out, b1['y'], black)
    assert abs(float(il) * mgw.losses.V2_93_MULS['img_mul'] - float(ret1['img_loss'])) <= 1e-5 * abs(float(ret1['img_loss']))
    # theta_only (iterations <= 100): only the id terms reach the objective
    t0, r1, _, _ = mgw.train_losses(net, b1, b2, flow, mgw.loss_gates(50))
    want = float(r1['theta_loss'] + r1['grid_theta_loss']) * 1.0
    assert torch.isfinite(t0) and float(t0) < float(total) and want > 0


def test_loss_backwards_take_the_upstream_from_the_device(mgw):
    """upstream_dev of the loss backwards: the same gradients as the by-value upstream, and a whole objective
    (warp + img/feature/temp/vertex losses, forward and backward) enqueues without a single host synchronisation."""
    import synth
    n, h, w = 3, 48, 64
    U, y = dev(synth.smooth_image(n, h, w, 1, 1)), dev(synth.smooth_image(n, h, w, 1, 2))
    th = dev(synth.random_mesh(n, 4, 4, 0.05, 3))
    out, black, img, Hs, sums = mgw.ops.mesh_warp_img_loss_fwd(U, th, y)
    up = torch.tensor([0.37], device='cuda')
    a = mgw.ops.img_loss_bwd(out, y, black, sums, 0.37)
    b = mgw.ops.img_loss_bwd(out, y, black, sums, up)
    assert torch.allclose(a, b, rtol=1e-6, atol=0)
    a = mgw.ops.mesh_warp_img_loss_bwd(U, th, Hs, out, y, black, sums, 0.37, float(n))
    b = mgw.ops.mesh_warp_img_loss_bwd(U, th, Hs, out, y, black, sums, up, float(n))
    assert torch.allclose(a[1], b[1], rtol=1e-5, atol=1e-7) and torch.allclose(a[0], b[0], rtol=1e-5, atol=1e-7)
    matches = dev(synth.uniform((n, 20, 4), -1, 1, 4)); mask = dev((synth.uniform((n, 20), 0, 1, 5) < 0.6).astype(np.float32))
    assert torch.allclose(mgw.ops.feature_loss_bwd(matches, mask, img, 0.37), mgw.ops.feature_loss_bwd(matches, mask, img, up), rtol=1e-6, atol=0)
    ts = mgw.ops.temp_loss_fwd(out, black, out, black, img)
    a, b = mgw.ops.temp_loss_bwd(out, black, out, black, img, ts, 0.37), mgw.ops.temp_loss_bwd(out, black, out, black, img, ts, up)
    assert torch.allclose(a[0], b[0], rtol=1e-6, atol=0) and torch.allclose(a[1], b[1], rtol=1e-5, atol=1e-9)

    head = dev(synth.randn((n, 50), 6, 0.05)).requires_grad_(True)
    flow = dev(synth.uniform((n, h, w, 2), -1, 1, 7))

    def objective():
        tot, rets = 0, []
        for _ in range(2):
            p1, p2 = mgw.get_4_pts(head, grid=(4, 4))
            il, o, bl, fl = mgw.transformer_img_loss(U, p2, y)
            ftl, _ = mgw.feature_loss(matches, mask, fl)
            t, _ = mgw.total_loss(head, p1, p2, il, ftl)
            tot = tot + t
            rets.append((o, bl))
        tot = tot + 500.0 * mgw.temp_loss(rets[0][0], rets[0][1], rets[1][0], rets[1][1], flow)
        tot.backward()
        return tot

    objective()                                   # warm-up (allocations, lazy initialisation)
    head.grad = None
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode('error')
    try:
        tot = objective()
    finally:
        torch.cuda.set_sync_debug_mode('default')
    assert torch.isfinite(tot) and torch.isfinite(head.grad).all() and float(head.grad.abs().max()) > 0


@pytest.mark.parametrize('impl', ['auto', 'generic'])
def test_no_kernel_writes_outside_its_buffers(mgw, impl):
    """Every output and the workspace of the warp calls sit between guard bands filled with a NaN pattern inside one big
    allocation; after forward + backward (TMA stores, TMA reduce-adds, red.v4 drains, fixed-point scatter) the guards are
    intact and nothing inside the buffers was left unwritten.  (compute-sanitizer is not available on this pool.)"""
    import synth
    from dovs_b200._lib import lib, check
    mgw.set_impl(impl)
    try:
        for (n, h, w, c, gh, gw) in [(2, 48, 64, 3, 4, 4), (1, 288, 512, 3, 4, 4), (3, 50, 70, 1, 2, 3), (2, 96, 128, 4, 4, 4),
                                     (2, 72, 96, 1, 4, 4), (1, 40, 36, 2, 1, 1)]:
            G = 8192                                            # guard floats (32 KB) around every buffer
            sizes = dict(Hs=n * gh * gw * 9, out=n * h * w * c, black=n * h * w, img=n * h * w * 2, dU=n * h * w * c,
                         dtheta=n * (gh + 1) * (gw + 1) * 2,
                         ws=(lib.mgw_mesh_warp_bwd_workspace_bytes(n, h, w, c, gh, gw) + 3) // 4 + 64)
            offs, total = {}, G
            for k, v in sizes.items():
                offs[k] = total
                total += (v + 63) // 64 * 64 + G                 # 256-byte aligned starts
            pool = torch.full((total,), float('nan'), device='cuda')
            pool.view(torch.int32).fill_(0x7fc0dead)            # a recognisable quiet NaN
            view = {k: pool[offs[k]:offs[k] + sizes[k]] for k in sizes}
            U = dev(synth.noise_image(n, h, w, c, 1)); th = dev(synth.random_mesh(n, gh, gw, 0.06, 2))
            d_out = dev(synth.randn((n, h, w, c), 3)); d_img = dev(synth.randn((n, h, w, 2), 4))
            st = torch.cuda.current_stream().cuda_stream
            P = lambda t: t.data_ptr()
            check(lib.mgw_mesh_warp_fwd(P(U), P(th), n, h, w, c, gh, gw, P(view['Hs']), P(view['out']), P(view['black']), P(view['img']), st), 'fwd')
            check(lib.mgw_mesh_warp_bwd(P(U), P(th), P(view['Hs']), P(d_out), P(d_img), n, h, w, c, gh, gw, P(view['dU']), P(view['dtheta']),
                                        P(view['ws']), st), 'bwd')
            torch.cuda.synchronize()
            raw = pool.view(torch.int32)
            mask = torch.ones(total, dtype=torch.bool, device='cuda')
            for k in sizes:
                mask[offs[k]:offs[k] + sizes[k]] = False
            assert bool((raw[mask] == 0x7fc0dead).all()), ('guard band overwritten', impl, (n, h, w, c, gh, gw))
            for k in ('Hs', 'out', 'black', 'img', 'dU', 'dtheta'):
                assert not bool((view[k].view(torch.int32) == 0x7fc0dead).any()), ('unwritten output', k, impl, (n, h, w, c))
            # and the guarded results are the ordinary ones
            o, b, i, Hs = mgw.ops.mesh_warp_fwd(U, th)
            assert torch.equal(o.reshape(-1), view['out']) and torch.equal(b.reshape(-1), view['black']) and torch.equal(i.reshape(-1), view['img'])
    finally:
        mgw.set_impl('auto')


def test_deploy_crop_exact(mgw):
    """CropState (mgw_black_accumulate / mgw_crop_rect) == the reference's loops (fixture) and the restatement (larger sizes)."""
    import deploy_ref
    g = load_golden('deploy_crop')
    for name in sorted(k[:-4] for k in g if k.endswith('_ans')):
        ab = torch.as_tensor(g[name + '_all_black'].astype(np.int32)).cuda()
        rect = mgw.ops.crop_rect(ab).cpu().tolist()
        want = g[name + '_ans'].tolist()
        assert rect == (want if want else [-1, -1, -1, -1]), name
    crop = mgw.CropState(44, 70)
    crop.all_black.copy_(torch.as_tensor(g['all_corners_black_all_black'].astype(np.int32)))
    with pytest.raises(IndexError):
        crop.rect()
    # accumulation: the reference's own `all_black` after 40 frames x 2 refine passes of the stream fixture
    s = load_golden('deploy_stream')
    h, w = s['first'].shape
    crop, ref = mgw.CropState(h, w), deploy_ref.StreamStateRef(s['first'])
    for k in range(s['cur_frames'].shape[0]):
        in_x = ref.assemble(s['cur_frames'][k])
        for _ in range(int(s['refine'])):
            img, black = deploy_ref.stream_fake_net(in_x, k)
            crop.add(dev(black))
            in_x[..., -1] = ref.frame_of(img, black)
        ref.push(img, black)
    assert np.array_equal(crop.all_black.cpu().numpy().astype(np.int64), s['all_black'])
    # full-size and ragged masks against the restatement, several steps
    r = np.random.RandomState(3)
    for (H, W, step, dens) in [(288, 512, 10, 0.0005), (288, 512, 10, 0.0), (287, 509, 7, 0.002), (33, 31, 1, 0.05), (2, 2, 10, 0.0),
                               (720, 1280, 10, 0.0002)]:
        ab = (r.random_sample((H, W)) < dens).astype(np.int64) * 3
        ab[:min(3, H), :] += r.randint(0, 2, (min(3, H), W))
        ab[:, -2:] += 1
        got = mgw.ops.crop_rect(torch.as_tensor(ab.astype(np.int32)).cuda(), step).cpu().tolist()
        want = deploy_ref.crop_rect(ab, step)
        assert got == (want if want else [-1, -1, -1, -1]), (H, W, step)
        frame = torch.arange(H * W * 3, device='cuda').reshape(H, W, 3)
        if want:
            c = mgw.CropState(H, W); c.all_black.copy_(torch.as_tensor(ab.astype(np.int32)))
            assert torch.equal(c.cut(frame, step), frame[want[0]:want[2] + 1, want[1]:want[3] + 1, :])


def test_empty_batch_is_a_no_op(mgw):
    """N = 0 (an empty shard): empty outputs of the right shapes, no launch, and backward through them works"""
    l0 = mgw.launch_count()
    U = torch.zeros(0, 48, 64, 3, device='cuda', requires_grad=True)
    th = torch.zeros(0, 5, 5, 2, device='cuda', requires_grad=True)
    out, black, img = mgw.transformer(U, th)
    assert out.shape == (0, 48, 64, 3) and black.shape == (0, 48, 64) and img.shape == (0, 48, 64, 2)
    (out.sum() + img.sum()).backward()
    assert th.grad.shape == th.shape and U.grad.shape == U.shape
    o2, b2 = mgw.spatial_transformer.transformer(U, torch.zeros(0, 9, device='cuda'), (24, 32))
    assert o2.shape == (0, 24, 32, 3) and b2.shape == (0, 48, 64)
    o3 = mgw.interpolate(U, torch.zeros(0, 24, 32, 1, device='cuda'), torch.zeros(0, 24, 32, 1, device='cuda'), (24, 32))
    assert o3.shape == (0, 24, 32, 3)
    assert mgw.launch_count() == l0
    with pytest.raises(RuntimeError):
        mgw.transformer(torch.zeros(0, 8, 8, 3), torch.zeros(0, 5, 5, 2))          # still no CPU path


def test_deploy_stream_state_device_head_and_graph_replay(mgw):
    """StreamState(device_head=True): same histories and inputs as the host-head rings, and a frame (assemble + push) captured
    ONCE in a CUDA graph replays correctly for every later frame"""
    import deploy_ref
    g = load_golden('deploy_stream')
    h, w = g['first'].shape
    st = mgw.StreamState(g['first'], device_head=True)
    cur = torch.empty((h, w), device='cuda'); img_b = torch.empty((h, w), device='cuda'); blk_b = torch.empty((h, w), device='cuda')
    in_x_buf = torch.empty((1, h, w, 13), device='cuda')
    graph = None
    side = torch.cuda.Stream()
    for k in range(g['cur_frames'].shape[0]):
        cur.copy_(dev(g['cur_frames'][k]))
        # the stand-in network of the fixture needs in_x on the host; its last refine pass decides what is pushed
        in_x = st.assemble(cur)
        assert np.array_equal(in_x.cpu().numpy(), g['in_x'][k])
        x_np = in_x.cpu().numpy()
        for _ in range(int(g['refine'])):
            img, black = deploy_ref.stream_fake_net(x_np, k)
            x_np[..., -1] = (img.reshape(h, w) + black.reshape(h, w) * np.float32(-1))
        img_b.copy_(dev(img).reshape(h, w)); blk_b.copy_(dev(black).reshape(h, w))
        if k < 3:
            st.push(img_b, blk_b)
            if k == 2:                                   # capture "assemble into a static buffer + push" once
                torch.cuda.synchronize()
                graph = torch.cuda.CUDAGraph()
                snap = (st.frames.clone(), st.masks.clone(), st.head_dev.clone())
                with torch.cuda.graph(graph):
                    st.assemble(cur, out=in_x_buf)
                    st.push(img_b, blk_b)
                st.frames.copy_(snap[0]); st.masks.copy_(snap[1]); st.head_dev.copy_(snap[2])      # capture does not run anything
        else:
            graph.replay()
            assert np.array_equal(in_x_buf.cpu().numpy(), g['in_x'][k])
    fr, mk = st.history()
    assert np.array_equal(fr.cpu().numpy()[..., None], g['final_frames']) and np.array_equal(mk.cpu().numpy()[..., None], g['final_masks'])


def test_errors_are_loud(mgw):
    with pytest.raises(RuntimeError):
        mgw.transformer(torch.zeros(1, 8, 8, 3), torch.zeros(1, 5, 5, 2))          # CPU tensors: no fallback
    with pytest.raises(TypeError):
        mgw.transformer(torch.zeros(1, 8, 8, 3, device='cuda', dtype=torch.float64), torch.zeros(1, 5, 5, 2, device='cuda'))
    with pytest.raises(ValueError):
        mgw.transformer(torch.zeros(1, 8, 8, 3, device='cuda'), torch.zeros(2, 5, 5, 2, device='cuda'))
    with pytest.raises(mgw.MgwError):
        mgw.ops.warp_fwd(torch.zeros(1, 2, 2, 3, device='cuda'), torch.zeros(1, 4, 4, 9, device='cuda'))   # gh > H

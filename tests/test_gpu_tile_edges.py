"""The edges the training hot path's correctness arguments cover, driven to those edges.

  * The tile backward (mgw_warp_tma.cu, warp_bwd_tma_kernel) sums dU per tile in int32 shared memory, one power-of-two
    scale per tile from max|d_out|.  Its headroom argument: a word receives at most one term per pixel of the tile, each
    term rounds to at most 2^kBits, so kTerms * 2^kBits must stay below 2^31.  A constant map sends every pixel of every
    tile onto ONE source word with weight 1, and d_out just below a power of two makes every term round UP to exactly
    2^kBits: the worst case of that argument, for every compiled variant.
  * The same accumulator's quantisation contract, element by element: every term is within 2^-kBits of its tile's max|d_out|.
  * The persistent forward pipeline (mgw_warp_pipe.cu) hands tile records from its producer warp to the consumers through a
    16-slot ring filled 8 tiles at a time; MGW_PIPE_GRID shrinks the grid so that one call wraps that ring many times.
  * The tiled temp_loss backward (mgw_loss_tile.cu) has the same fixed-point accumulator with 768 terms and 21 bits.

References are fp64: an explicit bilinear scatter at the kernels' own fp32 sample positions (the forward's x/y maps, which
the generic kernels produce bit-identically to the C oracle), the oracle port's autograd for temp_loss, and the generic
kernels themselves for the bit-exact forward.
"""
import numpy as np
import pytest
import torch

import mesh_warp_ref as ref
import synth

pytestmark = pytest.mark.gpu


@pytest.fixture(scope='module')
def mgw():
    import dovs_b200
    assert torch.cuda.is_available(), 'GPU tests need a CUDA device; there is no CPU fallback'
    yield dovs_b200
    dovs_b200.set_impl('auto')


def dev(a):
    return torch.tensor(np.ascontiguousarray(a), device='cuda')


# ------------------------------------------------------------------ fp64 reference of the backward's dU scatter
def scatter64(img, g, H, W, q_pix=None):
    """dU of the bilinear warp for upstream g [N,H,W,C] at the fp32 sample points img [N,H,W,2] (normalised x/y maps), in fp64.
    The tap coordinates and weights are formed in fp32 exactly as the kernels form them (spatial_transformer3.py:81-93,114-121);
    only their products with g and the sums are exact.  A pixel with a clipped tap contributes nothing: clipping collapses a
    tap pair onto one word with weights of opposite sign (mgw_device.cuh, taps_scatter).
    Returns (dU, sum of |terms|, number of terms, sum of q_pix over the terms) per word; q_pix [N,H,W] is a per-pixel budget."""
    N, _, _, C = g.shape
    f32 = np.float32
    x = (img[..., 0] + f32(1)) * f32(W) * f32(0.5)
    y = (img[..., 1] + f32(1)) * f32(H) * f32(0.5)
    with np.errstate(invalid='ignore'):
        fx, fy = np.floor(x), np.floor(y)
        ok = np.isfinite(x) & np.isfinite(y) & (fx >= 0) & (fx <= W - 2) & (fy >= 0) & (fy <= H - 2)
    n, r, c = np.nonzero(ok)
    x, y, fx, fy = x[ok], y[ok], fx[ok], fy[ok]
    ax, bx = ((fx + f32(1)) - x).astype(np.float64), (x - fx).astype(np.float64)
    ay, by = ((fy + f32(1)) - y).astype(np.float64), (y - fy).astype(np.float64)
    x0, y0 = fx.astype(np.int64), fy.astype(np.int64)
    gv = g[n, r, c].astype(np.float64)                                       # [P, C]
    qv = np.zeros(len(n)) if q_pix is None else q_pix[n, r, c]
    size = N * H * W * C
    out, absum, cnt, qsum = (np.zeros(size) for _ in range(4))
    ch = np.arange(C)
    for dy, dx, w in ((0, 0, ax * ay), (1, 0, ax * by), (0, 1, bx * ay), (1, 1, bx * by)):
        word = (((n * H + y0 + dy) * W + x0 + dx) * C)[:, None] + ch[None, :]
        term = w[:, None] * gv
        live = np.broadcast_to((w > 0)[:, None], term.shape)
        np.add.at(out, word.ravel(), term.ravel())
        np.add.at(absum, word.ravel(), np.abs(term).ravel())
        np.add.at(cnt, word.ravel(), live.ravel().astype(np.float64))
        np.add.at(qsum, word.ravel(), (live * qv[:, None]).ravel())
    shp = (N, H, W, C)
    return out.reshape(shp), absum.reshape(shp), cnt.reshape(shp), qsum.reshape(shp)


def tile_quantum(g, TH, TW, kbits):
    """per pixel: 2^-kBits of its tile's max|d_out| over all channels (tiles = mesh cells here), the rounding budget of one term"""
    N, H, W, C = g.shape
    m = np.abs(g).max(-1).reshape(N, H // TH, TH, W // TW, TW).max((2, 4))
    return np.repeat(np.repeat(m, TH, 1), TW, 2) * 2.0 ** -kbits


def bound_violations(got, want, tol):
    """elements outside |got - want| <= tol, and elements whose sign differs where |want| > tol"""
    got = np.asarray(got, np.float64)
    err = np.abs(got - want)
    far = err > tol
    flipped = (np.abs(want) > tol) & (np.sign(got) != np.sign(want))
    msg = []
    if far.any():
        i = np.unravel_index(np.argmax(err - tol), err.shape)
        msg.append('%d outside the bound, worst at %s: got %r, fp64 %r, bound %.3g' % (far.sum(), i, got[i], want[i], tol[i]))
    if flipped.any():
        i = np.unravel_index(np.argmax(np.where(flipped, np.abs(want), 0)), want.shape)
        msg.append('%d with the wrong sign, e.g. at %s: got %r, fp64 %r' % (flipped.sum(), i, got[i], want[i]))
    return '; '.join(msg)


# ------------------------------------------------------------------ A. fixed-point headroom of every compiled tile backward
# (MGW_TILE, TW, TH): TH = K * threads / TW.  kTerms = TH * TW terms can reach one word; kBits = 30 - floor(log2 kTerms) keeps
# kTerms * 2^kBits below 2^31 (2^-kBits of the tile's max|d_out| is the rounding budget of one term).
VARIANTS = [('64x6', 64, 24), ('64x3x512', 64, 24), ('64x3', 64, 12), ('32x3', 32, 24), ('32x2', 32, 16), ('32x1', 32, 8)]
VARIANT_C = [(v, c) for v in VARIANTS for c in (1, 3, 4) if not (c == 4 and v[1] == 64)]      # no 64-wide tiles at C = 4


def kbits_of(TH, TW):
    return 30 - int(np.floor(np.log2(TH * TW)))


def constant_map_hs(n, gh, gw, xn, yn):
    """every cell's homography sends every pixel to the one normalised point (xn, yn): z = 1, x = xn, y = yn"""
    hs = np.zeros((n, gh, gw, 9), np.float32)
    hs[..., 2], hs[..., 5], hs[..., 8] = xn, yn, 1.0
    return hs


def d_out_values():
    """+-nextafter(2^k, 0): every term of the tile rounds up to exactly 2^kBits; +-2^k: exactly 2^(kBits-1)"""
    vals = []
    for k in (-6, 1, 9):
        v = np.float32(2.0 ** k)
        vals += [np.nextafter(v, np.float32(0)), -np.nextafter(v, np.float32(0)), v, -v]
    return vals


def collapse_case(H, W, C, frac, v, seed):
    U = synth.noise_image(1, H, W, C, seed)
    # the image centre, or half a pixel right of and below it (then four words share each term: weights of about 1/4)
    xn, yn = (np.float32(1.0 / W), np.float32(1.0 / H)) if frac else (np.float32(0), np.float32(0))
    return U, constant_map_hs(1, 4, 4, xn, yn), np.full((1, H, W, C), v, np.float32)


def dU_bound(img, g, TH, TW, H, W, tiles):
    """fp64 dU and the element-wise budget: 2^-kBits of the tile's max|d_out| per term, 2^-22 of the absolute sum for the fp32
    tap weights, and one fp32 rounding of the absolute sum per draining tile plus one"""
    want, absum, _, qsum = scatter64(img, g, H, W, tile_quantum(g, TH, TW, kbits_of(TH, TW)))
    return want, qsum + absum * (2.0 ** -22 + (tiles + 1) * 2.0 ** -24)


@pytest.mark.parametrize('variant,c', VARIANT_C, ids=['%s-c%d' % (v[0], c) for v, c in VARIANT_C])
def test_tile_backward_headroom_when_every_pixel_hits_one_word(mgw, monkeypatch, variant, c):
    """4 x 4 mesh whose cells are exactly one tile of the forced variant; every pixel maps onto one source point.  dU there is
    H*W*d_out: the int32 sum of a tile holds kTerms terms that round up to 2^kBits each and must neither wrap nor lose its sign."""
    tile, TW, TH = variant
    H, W = 4 * TH, 4 * TW
    monkeypatch.setenv('MGW_TILE', tile)
    failures = []
    for frac in (False, True):
        for v in d_out_values():
            U, Hs, g = collapse_case(H, W, c, frac, v, 7)
            Ud, Hd = dev(U), dev(Hs)
            mgw.set_impl('generic')
            img = mgw.ops.warp_fwd(Ud, Hd, want_out=False, want_black=False)[2].cpu().numpy()
            mgw.set_impl('tma')                                      # the tile kernels or an error, never the generic ones
            dU, _ = mgw.ops.warp_bwd(Ud, Hd, dev(g))
            want, tol = dU_bound(img, g, TH, TW, H, W, 16)
            bad = bound_violations(dU.cpu().numpy(), want, tol)
            if bad:
                failures.append('%s point, d_out %r: %s' % ('fractional' if frac else 'integer', float(v), bad))
    mgw.set_impl('auto')
    assert not failures, '\n'.join(failures)


def test_mesh_warp_bwd_headroom_and_dtheta(mgw, monkeypatch):
    """the same collapse through mgw_mesh_warp_bwd (the tile backward feeding the adjoint solve): dU within the bound of the
    fp64 scatter, dtheta equal to the generic family's to summation-order rounding"""
    TW, TH, c = 32, 16, 3
    H, W = 4 * TH, 4 * TW
    monkeypatch.setenv('MGW_TILE', '32x2')
    U, Hs, g = collapse_case(H, W, c, False, np.nextafter(np.float32(2), np.float32(0)), 8)
    Ud, Hd, gd = dev(U), dev(Hs), dev(g)
    theta = dev(synth.identity_mesh(1, 4, 4))
    mgw.set_impl('generic')
    img = mgw.ops.warp_fwd(Ud, Hd, want_out=False, want_black=False)[2].cpu().numpy()
    _, dth_g = mgw.ops.mesh_warp_bwd(Ud, theta, Hd, gd)
    mgw.set_impl('tma')
    dU, dth_t = mgw.ops.mesh_warp_bwd(Ud, theta, Hd, gd)
    mgw.set_impl('auto')
    want, tol = dU_bound(img, g, TH, TW, H, W, 16)
    bad = bound_violations(dU.cpu().numpy(), want, tol)
    assert not bad, bad
    # (the generic family sums dHs with fp32 atomics; the adjoint solve amplifies that noise by the cells' conditioning)
    a, b = dth_t.cpu().double(), dth_g.cpu().double()
    assert torch.isfinite(a).all() and (a - b).abs().max() <= 1e-3 * b.abs().max(), ((a - b).abs().max(), b.abs().max())


# ------------------------------------------------------------------ B. quantisation under a high dynamic range of d_out
@pytest.mark.parametrize('variant,c', VARIANT_C, ids=['%s-c%d' % (v[0], c) for v, c in VARIANT_C])
def test_tile_backward_quantum_per_element(mgw, monkeypatch, variant, c):
    """a smooth mesh (sigma 0.05) and d_out whose magnitude spans 1e-4 .. 1e4 inside every tile: each element of dU is within
    2^-kBits of its tiles' max|d_out| per term of the fp64 scatter (the small terms of a tile may vanish, nothing more)"""
    tile, TW, TH = variant
    n, H, W = 2, 4 * TH, 4 * TW
    monkeypatch.setenv('MGW_TILE', tile)
    U = synth.smooth_image(n, H, W, c, 30)
    theta = dev(synth.random_mesh(n, 4, 4, 0.05, 31))
    r = np.random.RandomState(32)
    g = (r.standard_normal((n, H, W, c)) * 10.0 ** r.uniform(-4, 4, (n, H, W, 1))).astype(np.float32)
    gi = synth.randn((n, H, W, 2), 33, 0.1)                        # staged next to d_out in the plain variant; no effect on dU
    Ud = dev(U)
    Hs = mgw.ops.solve_h_fwd(theta)
    mgw.set_impl('generic')
    img = mgw.ops.warp_fwd(Ud, Hs, want_out=False, want_black=False)[2].cpu().numpy()
    mgw.set_impl('tma')
    dU, _ = mgw.ops.warp_bwd(Ud, Hs, dev(g), dev(gi))
    mgw.set_impl('auto')
    want, absum, cnt, qsum = scatter64(img, g, H, W, tile_quantum(g, TH, TW, kbits_of(TH, TW)))
    # tiles whose box does not hold every tap add some terms by fp32 atomics: one rounding of the absolute sum per term
    tol = qsum + absum * (2.0 ** -22 + (2 * cnt + 1) * 2.0 ** -24)
    bad = bound_violations(dU.cpu().numpy(), want, tol)
    assert not bad, bad


# ------------------------------------------------------------------ C. persistent forward beyond one record round
# (name, N, H, W, gh, gw): cells of 24 x 32 / 44 x 36 take the 32 x 24 tiles ("big"), cells of 8 x 32 / 20 x 36 the 32 x 8 ones
# ("small"); 44 and 20 rows / 36 columns make every cell's last tile row and column shift back onto its neighbour.
PIPE_SHAPES = [('big', 7, 168, 224, 7, 7),              # 343 tiles
               ('big-shifted', 3, 132, 180, 3, 5),      # 180 tiles
               ('small', 7, 88, 224, 11, 7),            # 539 tiles
               ('small-shifted', 5, 60, 216, 3, 6)]     # 540 tiles
PIPE_GRIDS = ['1', '2', '3', '5', '37', None]


def same_bits(a, b):
    """bit-identical, NaN payloads aside"""
    return bool(((a.view(torch.int32) == b.view(torch.int32)) | (torch.isnan(a) & torch.isnan(b))).all())


def pipe_vs_generic(mgw, monkeypatch, U, theta, grids):
    mgw.set_impl('generic')
    want = mgw.ops.mesh_warp_fwd(U, theta)
    mgw.set_impl('pipe')                                            # the pipeline or an error, never a fallback
    failures = []
    for grid in grids:
        if grid is None:
            monkeypatch.delenv('MGW_PIPE_GRID', raising=False)
        else:
            monkeypatch.setenv('MGW_PIPE_GRID', grid)
        got = mgw.ops.mesh_warp_fwd(U, theta)
        torch.cuda.synchronize()
        for name, a, b in zip(('out', 'black', 'img', 'Hs'), got, want):
            if not same_bits(a, b):
                failures.append('grid %s: %s differs from the generic kernels in %d elements'
                                % (grid or 'default', name, int((a.view(torch.int32) != b.view(torch.int32)).sum())))
    monkeypatch.delenv('MGW_PIPE_GRID', raising=False)
    mgw.set_impl('auto')
    return failures


@pytest.mark.parametrize('c', [1, 3, 4])
@pytest.mark.parametrize('shape', PIPE_SHAPES, ids=[s[0] for s in PIPE_SHAPES])
def test_pipe_forward_many_rounds_per_cta(mgw, monkeypatch, shape, c):
    """grids of 1, 2, 3, 5 and 37 CTAs run tens to hundreds of tiles per CTA through the record ring (more than 16 per CTA
    wraps it); folded and clamped cells (sigma 0.2) leave tiles incomplete.  The whole batch equals the generic kernels
    bit for bit."""
    _, n, h, w, gh, gw = shape
    U = dev(synth.noise_image(n, h, w, c, 40 + c))
    theta = dev(synth.random_mesh(n, gh, gw, 0.2, 41 + c))
    failures = pipe_vs_generic(mgw, monkeypatch, U, theta, PIPE_GRIDS)
    assert not failures, '\n'.join(failures)


def test_pipe_forward_production_batch(mgw, monkeypatch):
    """128 x 288 x 512 x 3 on the default grid: 24 576 tiles, more than 16 per CTA on any GPU of up to 1536 CTAs"""
    n, h, w, c = 128, 288, 512, 3
    U = dev(synth.noise_image(n, h, w, c, 50))
    theta = dev(synth.random_mesh(n, 4, 4, 0.05, 51))
    failures = pipe_vs_generic(mgw, monkeypatch, U, theta, [None])
    assert not failures, '\n'.join(failures)


# ------------------------------------------------------------------ D. temp_loss tile backward: a whole tile onto one point
@pytest.mark.parametrize('c', [3, 4])                                # (the tiled backward serves C >= 3)
def test_temp_loss_tile_backward_collapse(mgw, c):
    """a constant flow sends all 768 pixels of every 32 x 24 tile to one point; out1 - out2 is chosen so that the gradient
    sits just below a power of two (every fixed-point term rounds up to 2^21).  d_out2 against the fp64 port, both signs."""
    n, H, W = 2, 48, 64
    f32 = np.float32
    k = f32(2) / ((f32(H * W) + f32(1e-8)) * f32(n))                 # mgw_loss_tile.cu: upstream * 2 / ((sum m + 1e-8) * N)
    top = f32(2.0 ** -11)                                            # = 1.5 / (H * W * n)
    a = f32(1.5)
    while k * a >= top:                                              # the largest |out1 - out2| <= 1.5 with g1 below 2^-11
        a = np.nextafter(a, f32(0))
    failures = []
    for sx, sy in ((0, 0), (2.0 ** -7, 2.0 ** -5)):                  # source (32, 24), or (32.25, 24.75)
        flow = np.zeros((n, H, W, 2), np.float32)
        flow[..., 0], flow[..., 1] = sx, sy
        for sign in (1, -1):
            out1 = np.full((n, H, W, c), sign * a, np.float32)
            out2 = np.zeros((n, H, W, c), np.float32)
            black = np.zeros((n, H, W), np.float32)
            o1, o2 = dev(out1).requires_grad_(True), dev(out2).requires_grad_(True)
            mgw.temp_loss(o1, dev(black), o2, dev(black), dev(flow)).backward()
            t1, t2 = (torch.tensor(x, dtype=torch.float64, requires_grad=True) for x in (out1, out2))
            b64 = torch.tensor(black, dtype=torch.float64)
            ref.temp_loss(t1, b64, t2, b64, torch.tensor(flow, dtype=torch.float64)).backward()
            g1 = o1.grad.cpu().numpy()
            want = t2.grad.numpy()
            # d_out2 = -sum of g1 * w: 2^-21 of the tile's max|g1| per term, the fp32 g1 against the fp64 one (a few ulps),
            # one rounding per draining tile (4 per image) and one more
            q = np.abs(g1).max() * 2.0 ** -21
            terms = H * W
            tol = q * terms + np.abs(want) * (2.0 ** -21 + 5 * 2.0 ** -24)
            tag = 'flow (%g, %g), sign %+d' % (sx, sy, sign)
            e1 = np.abs(g1 - t1.grad.numpy()).max() / np.abs(t1.grad.numpy()).max()
            if not e1 < 2.0 ** -20:
                failures.append('%s: d_out1 differs from fp64 by %.3g relative' % (tag, e1))
            bad = bound_violations(o2.grad.cpu().numpy(), want, np.where(want != 0, tol, 0.0))
            if bad:
                failures.append('%s: d_out2 %s' % (tag, bad))
    assert not failures, '\n'.join(failures)

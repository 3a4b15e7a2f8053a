"""CPU: warpRevBundle2 at any output size -- the numpy restatement (oracle/remap_frame_ref.py) against the fixture and live cv2, the
argument checks of mgw_remap_bundle_frame (decided before anything reaches the device), and deploy.scale_rect."""
import os
import sys

import numpy as np
import pytest

from conftest import ROOT, load_golden

sys.path.insert(0, os.path.join(ROOT, 'oracle'))
import deploy_ref  # noqa: E402
import remap_frame_ref as M  # noqa: E402

MGW_OK, MGW_ERR_INVALID = 0, -1
BGR, NV12, I420 = 0, 1, 2
FAKE = 1 << 20          # a non-null, 16-byte aligned address: never dereferenced, every call below fails or returns before a launch


@pytest.fixture(scope='module')
def golden():
    return load_golden('deploy_remap_frame')


@pytest.fixture(scope='module')
def mgw():
    import dovs_b200
    return dovs_b200


@pytest.fixture(scope='module')
def cv2_plain():
    cv2 = pytest.importorskip('cv2')
    prev = cv2.useOptimized()
    cv2.setUseOptimized(False)
    yield cv2
    cv2.setUseOptimized(prev)


def _cases():
    for tag, _, _, _, outs in M.CASES:
        for out in outs:
            yield tag, out


@pytest.mark.parametrize('tag,out', list(_cases()), ids=['%s_%dx%d' % (t, o[0], o[1]) for t, o in _cases()])
def test_restatement_equals_fixture(golden, tag, out):
    dst = M.warp_rev_bundle2_sized(golden[tag + '_frame'], *M.fixture_maps(golden, tag), out)
    np.testing.assert_array_equal(dst, golden['%s_%dx%d_dst' % (tag, out[0], out[1])])


def test_fixture_records_the_optimised_path(golden):
    for tag, out in _cases():
        name = '%s_%dx%d' % (tag, out[0], out[1])
        assert 0 <= float(golden[name + '_opt_diff_frac']) < 0.01 and 0 <= int(golden[name + '_opt_diff_max']) <= 16, name


@pytest.mark.parametrize('out', [(288, 512), (1080, 1920), (37, 61)])
def test_restatement_equals_live_cv2_on_a_1080p_frame(cv2_plain, out):
    rs = np.random.RandomState(5)
    frame = rs.randint(0, 256, (1080, 1920, 3)).astype(np.uint8)
    xm, ym = M.smooth_mesh(288, 512, 11)
    np.testing.assert_array_equal(M.warp_rev_bundle2_sized(frame, xm, ym, out), M.cv2_sized(frame, xm, ym, out))


def test_at_the_maps_size_it_is_warp_rev_bundle2(golden):
    frame, (xm, ym) = golden['net_frame'], M.fixture_maps(golden, 'net')
    small = deploy_ref.resize_linear_u8(frame, 512, 288)
    np.testing.assert_array_equal(M.warp_rev_bundle2_sized(frame, xm, ym, (288, 512)), deploy_ref.warp_rev_bundle2(small, xm, ym))
    np.testing.assert_array_equal(M.warp_rev_bundle2_sized(small, xm, ym, (288, 512)), deploy_ref.warp_rev_bundle2(small, xm, ym))


# ---- mgw_remap_bundle_frame argument checks, in the batch calls' order
def call(lib, S, h=288, w=512, H=1080, W=1920, fmt=BGR, src=FAKE, xy=FAKE, dst=FAKE, ws=FAKE):
    return lib.mgw_remap_bundle_frame(src, fmt, xy, S, h, w, H, W, dst, ws, None)


def test_empty_batch_returns_ok_without_a_launch(mgw):
    lib = mgw._lib.lib
    n0 = lib.mgw_launch_count()
    for fmt in (BGR, NV12, I420):
        assert call(lib, 0, fmt=fmt, src=None, xy=None, dst=None, ws=None) == MGW_OK
    assert lib.mgw_launch_count() == n0


def test_bad_sizes_and_format_are_rejected_before_an_empty_batch_returns(mgw):
    lib = mgw._lib.lib
    for S in (0, 2):
        for kw in (dict(S=-1), dict(S=65536, h=8, w=8, H=1, W=1), dict(h=7), dict(w=7), dict(H=0), dict(W=0), dict(H=32768),
                   dict(W=32768), dict(H=-2)):
            args = dict(S=S)
            args.update(kw)
            assert call(lib, **args) == MGW_ERR_INVALID, kw
            assert b'bad sizes' in lib.mgw_last_error()
        for fmt in (NV12, I420):                # a YUV frame has an even size
            for H, W in ((1081, 1920), (1080, 1921)):
                assert call(lib, S, H=H, W=W, fmt=fmt) == MGW_ERR_INVALID
                assert b'bad sizes' in lib.mgw_last_error()
        for fmt in (3, -1):
            assert call(lib, S, fmt=fmt) == MGW_ERR_INVALID
            assert b'unknown format' in lib.mgw_last_error()
    assert call(lib, 0, H=1081, W=1921, src=None, xy=None, dst=None, ws=None) == MGW_OK      # BGR takes odd sizes
    # the 32-bit index limits: S*H*W*3 < 2^31 (345 frames of 1080p fit, 346 do not) and S*h*w < 2^31
    assert call(lib, 346, src=None) == MGW_ERR_INVALID and b'bad sizes' in lib.mgw_last_error()
    assert call(lib, 345, src=None) == MGW_ERR_INVALID and b'null pointer' in lib.mgw_last_error()
    assert call(lib, 2, h=32768, w=32768, H=8, W=8) == MGW_ERR_INVALID and b'bad sizes' in lib.mgw_last_error()


def test_null_pointers_then_alignment(mgw):
    lib = mgw._lib.lib
    for fmt in (BGR, NV12, I420):
        for kw in (dict(src=None), dict(xy=None), dict(dst=None), dict(ws=None)):
            assert call(lib, 2, fmt=fmt, **kw) == MGW_ERR_INVALID
            assert b'null pointer' in lib.mgw_last_error()
        for kw in (dict(xy=FAKE + 4), dict(ws=FAKE + 4)):
            assert call(lib, 2, fmt=fmt, **kw) == MGW_ERR_INVALID
            assert b'8-byte aligned' in lib.mgw_last_error()
        assert call(lib, 2, fmt=fmt, xy=FAKE + 4, src=None) == MGW_ERR_INVALID
        assert b'null pointer' in lib.mgw_last_error()


def test_workspace_is_the_quarter_maps(mgw):
    lib = mgw._lib.lib
    for S, h, w, H, W in ((1, 288, 512, 1080, 1920), (64, 288, 512, 2160, 3840), (5, 36, 64, 37, 61)):
        assert lib.mgw_remap_bundle_frame_workspace_bytes(S, h, w, H, W) == lib.mgw_remap_bundle_u8_workspace_bytes(S, h, w)
        assert lib.mgw_remap_bundle_frame_workspace_bytes(S, h, w, H, W) == 8 * S * (h // 4) * (w // 4)


# ---- scale_rect
def _brute(rect, from_size, to_size):
    """the definition evaluated in exact rationals: output row R is kept iff top <= (R+0.5)*h/OH - 0.5 <= bottom"""
    from fractions import Fraction as F
    (h, w), (OH, OW) = from_size, to_size
    t, l, b, r = rect

    def kept(lo, hi, n, N):
        ks = [R for R in range(N) if lo <= (R + F(1, 2)) * F(n, N) - F(1, 2) <= hi]
        return ks

    rows, cols = kept(t, b, h, OH), kept(l, r, w, OW)
    return rows, cols


def test_scale_rect_is_the_identity_at_equal_sizes(mgw):
    rs = np.random.RandomState(0)
    for _ in range(200):
        h, w = rs.randint(1, 600, 2)
        t, b = sorted(rs.randint(0, h, 2)); l, r = sorted(rs.randint(0, w, 2))
        assert mgw.deploy.scale_rect([t, l, b, r], (h, w), (h, w)) == [t, l, b, r]


def test_scale_rect_agrees_with_its_definition_and_stays_in_bounds(mgw):
    rs = np.random.RandomState(1)
    sizes = [((288, 512), (1080, 1920)), ((288, 512), (720, 1280)), ((288, 512), (37, 61)), ((288, 512), (2160, 3840)),
             ((36, 64), (101, 203)), ((7, 5), (3, 11))]
    for frm, to in sizes:
        for _ in range(60):
            t, b = sorted(rs.randint(0, frm[0], 2)); l, r = sorted(rs.randint(0, frm[1], 2))
            got = mgw.deploy.scale_rect([t, l, b, r], frm, to)
            assert 0 <= got[0] < to[0] and 0 <= got[2] < to[0] and 0 <= got[1] < to[1] and 0 <= got[3] < to[1]
            rows, cols = _brute((t, l, b, r), frm, to)
            if rows:
                assert (got[0], got[2]) == (rows[0], rows[-1]), (frm, to, t, b)
            else:                               # no output row centre inside: empty, or one row where the clamp meets it
                assert got[0] >= got[2]
            if cols:
                assert (got[1], got[3]) == (cols[0], cols[-1]), (frm, to, l, r)
            else:
                assert got[1] >= got[3]


def test_scale_rect_is_monotone(mgw):
    frm, to = (288, 512), (1080, 1920)
    prev = None
    for k in range(0, 140):
        cur = mgw.deploy.scale_rect([k, k, 287 - k, 511 - k], frm, to)
        if prev is not None:
            assert cur[0] >= prev[0] and cur[1] >= prev[1] and cur[2] <= prev[2] and cur[3] <= prev[3]
        prev = cur
    # a larger rectangle maps to a larger one, edge by edge
    for t in range(0, 288, 7):
        a = mgw.deploy.scale_rect([t, 0, 287, 511], frm, to)
        b = mgw.deploy.scale_rect([min(t + 1, 287), 0, 287, 511], frm, to)
        assert b[0] >= a[0]

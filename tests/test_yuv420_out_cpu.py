"""CPU: stabilised frames handed out as YUV 4:2:0 -- the numpy restatement of cv2.cvtColor(COLOR_BGR2YUV_I420)
(oracle/yuv420_out_ref.bgr_to_i420) against the fixture and live cv2, the argument checks of mgw_remap_bundle_frame_yuv420 (decided
before anything reaches the device), and the Python front end's checks of out_size / out_format."""
import numpy as np
import pytest

import yuv420_out_ref as O
import yuv420_ref as Y
from conftest import load_golden

MGW_OK, MGW_ERR_INVALID = 0, -1
BGR, NV12, I420 = 0, 1, 2
FAKE = 1 << 20          # a non-null, 16-byte aligned address: never dereferenced, every call below fails or returns before a launch


@pytest.fixture(scope='module')
def golden():
    return load_golden('deploy_yuv420_out')


@pytest.fixture(scope='module')
def mgw():
    import dovs_b200
    return dovs_b200


def fixture_names(g):
    return sorted(k[:-4] for k in g if k.endswith('_bgr'))


def test_fixture_covers_the_sizes(golden):
    assert fixture_names(golden) == ['block_288x512', 'random_2x2', 'random_6x10', 'random_90x158']


def test_restatement_equals_fixture(golden):
    for name in fixture_names(golden):
        bgr, want = golden[name + '_bgr'], golden[name + '_i420']
        H, W, _ = bgr.shape
        assert want.shape == (H * 3 // 2, W), name
        np.testing.assert_array_equal(O.bgr_to_i420(bgr), want, err_msg=name)


@pytest.mark.parametrize('optimised', [False, True])
def test_restatement_equals_live_cv2_at_1080p(optimised):
    cv2 = pytest.importorskip('cv2')
    rs = np.random.RandomState(7)
    frame = rs.randint(0, 256, (1080, 1920, 3)).astype(np.uint8)
    frame[:8] = 0
    frame[8:16] = 255                         # the extremes of every channel
    prev = cv2.useOptimized()
    try:
        cv2.setUseOptimized(optimised)
        want = cv2.cvtColor(frame, cv2.COLOR_BGR2YUV_I420)
    finally:
        cv2.setUseOptimized(prev)
    np.testing.assert_array_equal(O.bgr_to_i420(frame), want)


def test_chroma_is_the_top_left_pixel_not_the_average():
    bgr = np.zeros((2, 2, 3), np.uint8)
    bgr[0, 0] = (255, 0, 0)                   # a blue top-left pixel in a black block
    i420 = O.bgr_to_i420(bgr)
    assert i420[2, 0] == O.bgr_to_i420(np.full((2, 2, 3), (255, 0, 0), np.uint8))[2, 0] == 240
    assert i420[2, 1] == 110


def test_nv12_layout_of_the_fixture(golden):
    for name in fixture_names(golden):
        i420 = golden[name + '_i420']
        nv12 = O.bgr_to_yuv420(golden[name + '_bgr'], 'nv12')
        np.testing.assert_array_equal(nv12, Y.i420_to_nv12(i420))
        H, W = i420.shape[0] // 3 * 2, i420.shape[1]
        assert nv12.shape == i420.shape
        np.testing.assert_array_equal(nv12[:H], i420[:H])
        uv = nv12[H:].reshape(H // 2, W // 2, 2)
        _, U, V = Y.planes(i420, 'i420')
        np.testing.assert_array_equal(uv[..., 0], U)
        np.testing.assert_array_equal(uv[..., 1], V)
        for p, q in zip(Y.planes(nv12, 'nv12'), Y.planes(i420, 'i420')):
            np.testing.assert_array_equal(p, q)


# ---- mgw_remap_bundle_frame_yuv420 argument checks, in the batch calls' order
def call(lib, S, h=288, w=512, H=1080, W=1920, fmt=BGR, dst_fmt=NV12, src=FAKE, xy=FAKE, dst=FAKE, ws=FAKE):
    return lib.mgw_remap_bundle_frame_yuv420(src, fmt, xy, S, h, w, H, W, dst_fmt, dst, ws, None)


def test_empty_batch_returns_ok_without_a_launch(mgw):
    lib = mgw._lib.lib
    n0 = lib.mgw_launch_count()
    for fmt in (BGR, NV12, I420):
        for dst_fmt in (NV12, I420):
            assert call(lib, 0, fmt=fmt, dst_fmt=dst_fmt, src=None, xy=None, dst=None, ws=None) == MGW_OK
    assert lib.mgw_launch_count() == n0


def test_bad_sizes_and_formats_are_rejected_before_an_empty_batch_returns(mgw):
    lib = mgw._lib.lib
    for S in (0, 2):
        for kw in (dict(S=-1), dict(S=65536, h=8, w=8, H=2, W=2), dict(h=7), dict(w=7), dict(H=0), dict(W=0), dict(H=32768),
                   dict(W=32768), dict(H=-2)):
            args = dict(S=S)
            args.update(kw)
            assert call(lib, **args) == MGW_ERR_INVALID, kw
            assert b'bad sizes' in lib.mgw_last_error()
        for fmt in (BGR, NV12, I420):           # a 4:2:0 result has an even size, whatever the source
            for H, W in ((1081, 1920), (1080, 1921), (1, 2), (2, 1), (32767, 2)):
                assert call(lib, S, H=H, W=W, fmt=fmt) == MGW_ERR_INVALID, (fmt, H, W)
                assert b'bad sizes' in lib.mgw_last_error()
        for fmt in (3, -1):
            assert call(lib, S, fmt=fmt) == MGW_ERR_INVALID
            assert b'unknown format' in lib.mgw_last_error()
        for dst_fmt in (BGR, 3, -1):            # BGR is mgw_remap_bundle_frame's result
            assert call(lib, S, dst_fmt=dst_fmt) == MGW_ERR_INVALID, dst_fmt
            assert b'unknown destination format' in lib.mgw_last_error()
    # sizes are checked before the formats
    assert call(lib, 2, H=1081, fmt=3, dst_fmt=BGR) == MGW_ERR_INVALID and b'bad sizes' in lib.mgw_last_error()
    assert call(lib, 2, fmt=3, dst_fmt=BGR) == MGW_ERR_INVALID and b'unknown format' in lib.mgw_last_error()
    assert call(lib, 0, H=2, W=2, src=None, xy=None, dst=None, ws=None) == MGW_OK
    assert call(lib, 0, H=32766, W=32766, src=None, xy=None, dst=None, ws=None) == MGW_OK
    # the 32-bit index limits: S*H*W*3 < 2^31 (345 frames of 1080p fit, 346 do not) and S*h*w < 2^31
    assert call(lib, 346, src=None) == MGW_ERR_INVALID and b'bad sizes' in lib.mgw_last_error()
    assert call(lib, 345, src=None) == MGW_ERR_INVALID and b'null pointer' in lib.mgw_last_error()
    assert call(lib, 2, h=32768, w=32768, H=8, W=8) == MGW_ERR_INVALID and b'bad sizes' in lib.mgw_last_error()


def test_null_pointers_then_alignment(mgw):
    lib = mgw._lib.lib
    for fmt in (BGR, NV12, I420):
        for dst_fmt in (NV12, I420):
            for kw in (dict(src=None), dict(xy=None), dict(dst=None), dict(ws=None)):
                assert call(lib, 2, fmt=fmt, dst_fmt=dst_fmt, **kw) == MGW_ERR_INVALID
                assert b'null pointer' in lib.mgw_last_error()
            for kw in (dict(xy=FAKE + 4), dict(ws=FAKE + 4)):
                assert call(lib, 2, fmt=fmt, dst_fmt=dst_fmt, **kw) == MGW_ERR_INVALID
                assert b'8-byte aligned' in lib.mgw_last_error()
            assert call(lib, 2, fmt=fmt, dst_fmt=dst_fmt, xy=FAKE + 4, src=None) == MGW_ERR_INVALID
            assert b'null pointer' in lib.mgw_last_error()


# ---- the Python front end: decided before anything is allocated on a device
def test_stream_batch_rejects_odd_sizes_and_unknown_formats(mgw):
    for fmt in ('nv12', 'i420'):
        for out in ((1081, 1920), (1080, 1921), (37, 61)):
            with pytest.raises(ValueError, match='even size'):
                mgw.StreamBatch(2, (1080, 1920), out_size=out, out_format=fmt, device='cpu')
        with pytest.raises(ValueError, match='even size'):          # no out_size: the network's size is the output's
            mgw.StreamBatch(2, (1080, 1920), height=287, width=512, out_format=fmt, device='cpu')
        with pytest.raises(ValueError, match='even size'):
            mgw.MixedStreamBatch(2, (1080, 1920), height=288, width=511, out_format=fmt, device='cpu')
    for bad in ('rgb', 'yuv', 'NV12', None):
        with pytest.raises(ValueError, match='out_format'):
            mgw.StreamBatch(2, (1080, 1920), out_format=bad, device='cpu')
        with pytest.raises(ValueError, match='out_format'):
            mgw.MixedStreamBatch(2, (1080, 1920), out_format=bad, device='cpu')

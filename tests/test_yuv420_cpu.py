"""CPU: YUV 4:2:0 input (NV12 / I420).  The numpy restatement of cv2.cvtColor(COLOR_YUV2BGR_NV12 / _I420) against the fixture
made by OpenCV and against live OpenCV, and the argument checks of the two YUV batch entry points, every one of which is decided
before anything reaches the device (so they run without a GPU: an empty batch is a no-op, bad arguments are errors)."""
import numpy as np
import pytest

import yuv420_ref
from conftest import load_golden

MGW_OK, MGW_ERR_INVALID = 0, -1
NV12, I420 = 1, 2
FAKE = 1 << 20          # a non-null, 16-byte aligned address: never dereferenced, every call below fails or returns before a launch


def fixture_cases(g):
    return sorted(k[:-4] for k in g if k.endswith('_yuv'))


def test_restatement_matches_the_fixture():
    g = load_golden('deploy_yuv420')
    names = fixture_cases(g)
    assert len(names) == 2 * 2 * len(yuv420_ref.SIZES)                  # both formats, random and limited-range content
    for n in names:
        fmt = n.split('_')[0]
        assert np.array_equal(yuv420_ref.yuv420_to_bgr(g[n + '_yuv'], fmt), g[n + '_bgr']), n


def test_fixture_covers_both_clamps_and_the_unclamped_path():
    g = load_golden('deploy_yuv420')
    rnd = np.concatenate([g[n + '_bgr'].reshape(-1) for n in fixture_cases(g) if '_random_' in n])
    assert (rnd == 0).any() and (rnd == 255).any()
    for n in fixture_cases(g):
        if '_limited_' in n:
            y = yuv420_ref.planes(g[n + '_yuv'], n.split('_')[0])[0]
            assert y.min() >= 16 and y.max() <= 235, n


def test_fixture_resize_is_the_existing_restatement():
    """the stored cv2.resize of the converted frames is what deploy_ref.resize_linear_u8 (the BGR path's oracle) computes"""
    import deploy_ref
    g = load_golden('deploy_yuv420')
    names = [n for n in fixture_cases(g) if n + '_resized' in g]
    assert len(names) == 8
    for n in names:
        want = g[n + '_resized']
        assert np.array_equal(deploy_ref.resize_linear_u8(g[n + '_bgr'], want.shape[1], want.shape[0]), want), n


@pytest.mark.parametrize('optimized', [True, False])
def test_restatement_matches_live_opencv(optimized):
    cv2 = pytest.importorskip('cv2')
    codes = {'nv12': cv2.COLOR_YUV2BGR_NV12, 'i420': cv2.COLOR_YUV2BGR_I420}
    rs = np.random.RandomState(7)
    prev = cv2.useOptimized()
    try:
        cv2.setUseOptimized(optimized)
        for H, W in ((720, 1278), (288, 512), (6, 10), (2, 2)):
            frames = [yuv420_ref.random_frame(rs, H, W), yuv420_ref.limited_frame(H, W, 3)]
            for fmt in ('nv12', 'i420'):
                for yuv in frames:
                    assert np.array_equal(yuv420_ref.yuv420_to_bgr(yuv, fmt), cv2.cvtColor(yuv, codes[fmt])), (H, W, fmt)
    finally:
        cv2.setUseOptimized(prev)


# ---- argument checks of mgw_cvt_img2train_yuv420_batch / mgw_resize_linear_yuv420_batch
@pytest.fixture(scope='module')
def lib():
    import dovs_b200
    return dovs_b200._lib.lib


def cvt(lib, S, H, W, fmt=NV12, out_h=288, out_w=512, ptr=FAKE):
    return lib.mgw_cvt_img2train_yuv420_batch(ptr, fmt, S, H, W, ptr, ptr, ptr, 5, ptr, ptr, ptr, 5, out_h, out_w, ptr, ptr, None)


def resize(lib, S, H, W, fmt=NV12, out_h=288, out_w=512, ptr=FAKE, tab=FAKE):
    return lib.mgw_resize_linear_yuv420_batch(ptr, fmt, S, H, W, tab, tab, out_h, out_w, ptr, None)


def test_version(lib):
    assert lib.mgw_version() == 102


def test_empty_batch_returns_ok_without_a_launch(lib):
    n0 = lib.mgw_launch_count()
    for fmt in (NV12, I420):
        assert cvt(lib, 0, 1080, 1920, fmt, ptr=None) == MGW_OK
        assert resize(lib, 0, 1080, 1920, fmt, ptr=None, tab=None) == MGW_OK
    assert lib.mgw_launch_count() == n0


def test_bad_format_is_rejected(lib):
    for fn in (cvt, resize):
        for fmt in (0, 3, -1):
            assert fn(lib, 2, 96, 128, fmt) == MGW_ERR_INVALID
            assert b'unknown format' in lib.mgw_last_error()
        assert fn(lib, 0, 96, 128, 0, ptr=None) == MGW_ERR_INVALID           # checked before an empty batch returns


def test_odd_sizes_are_rejected(lib):
    for fn in (cvt, resize):
        for H, W in ((97, 128), (96, 127), (1, 2), (2, 1)):
            assert fn(lib, 2, H, W) == MGW_ERR_INVALID, (fn.__name__, H, W)
            assert b'bad sizes' in lib.mgw_last_error()
        assert fn(lib, 0, 97, 128, ptr=None) == MGW_ERR_INVALID              # checked before an empty batch returns
        for H, W in ((0, 128), (96, 0), (-2, 128)):
            assert fn(lib, 2, H, W) == MGW_ERR_INVALID


def test_sizes_past_the_32_bit_index_limits_are_rejected(lib):
    # 1080p 4:2:0 frames are 3 110 400 bytes: S*(3H/2)*W must stay below 2^31, so 690 frames fit and 691 do not
    for fn in (cvt, resize):
        assert fn(lib, 691, 1080, 1920) == MGW_ERR_INVALID
        assert b'bad sizes' in lib.mgw_last_error()
        assert fn(lib, 65536, 2, 2, out_h=1, out_w=1) == MGW_ERR_INVALID        # the stream index is gridDim.y
        assert fn(lib, -1, 48, 64) == MGW_ERR_INVALID
        assert fn(lib, 2, 48, 64, out_h=0) == MGW_ERR_INVALID
    assert cvt(lib, 2, 96, 128, out_h=1 << 15, out_w=1 << 15) == MGW_ERR_INVALID   # the output's limit, as for the BGR batch


def test_null_pointers_and_tables(lib):
    for fmt in (NV12, I420):
        assert cvt(lib, 2, 96, 128, fmt, ptr=None) == MGW_ERR_INVALID
        assert b'null pointer' in lib.mgw_last_error()
        assert resize(lib, 2, 96, 128, fmt, ptr=None) == MGW_ERR_INVALID
        assert b'null pointer' in lib.mgw_last_error()
        assert resize(lib, 2, 96, 128, fmt, tab=FAKE + 4) == MGW_ERR_INVALID          # tables must be 16-byte aligned
        assert b'16-byte aligned' in lib.mgw_last_error()
        assert resize(lib, 2, 96, 128, fmt, tab=None) == MGW_ERR_INVALID              # tables are needed unless 2x2 decimation
        assert b'tables are required' in lib.mgw_last_error()


# ---- the Python front end refuses malformed YUV frames before anything reaches the device
def test_python_front_end_rejects_malformed_frames():
    import dovs_b200
    d = dovs_b200.deploy
    good = np.zeros((144, 128), np.uint8)
    for fn in (lambda x, f='nv12': d.cvt_img2train(x, src_format=f), lambda x, f='nv12': d.cv2_resize(x, (64, 48), src_format=f)):
        for bad in (np.zeros((145, 128), np.uint8),            # rows not a multiple of 3
                    np.zeros((144, 127), np.uint8),            # odd W
                    np.zeros((144, 128), np.float32),          # dtype
                    np.zeros((144, 128, 3), np.uint8)[None],   # a BGR batch is not a YUV batch
                    np.zeros((0, 128), np.uint8)):
            with pytest.raises(ValueError):
                fn(bad)
        with pytest.raises(ValueError):
            fn(good, 'nv21')
    with pytest.raises(ValueError):
        dovs_b200.StreamBatch(2, (97, 128), src_format='i420', device='cpu')      # odd H
    with pytest.raises(ValueError):
        dovs_b200.StreamBatch(2, (96, 128), src_format='yv12', device='cpu')

"""CPU: the per-slot source geometry calls (mgw_cvt_img2train_mixed, mgw_resize_linear_mixed) refuse bad arguments before anything
reaches the device, and the padded per-slot tables of deploy.mixed_slot_tables are the uniform tables at the slot's size."""
import numpy as np
import pytest

MGW_OK, MGW_ERR_INVALID = 0, -1
BGR, NV12, I420 = 0, 1, 2
FAKE = 1 << 20          # a non-null, 16-byte aligned address: never dereferenced, every call below fails or returns before a launch


@pytest.fixture(scope='module')
def mgw():
    import dovs_b200
    return dovs_b200


def cvt(lib, S, mh, mw, fmt=BGR, out_h=288, out_w=512, ptr=FAKE, sizes=FAKE, ks=5):
    return lib.mgw_cvt_img2train_mixed(ptr, fmt, S, mh, mw, sizes, ptr, ptr, ptr, ks, ptr, ptr, ptr, ks, out_h, out_w, ptr, ptr, None)


def resize(lib, S, mh, mw, fmt=BGR, out_h=288, out_w=512, ptr=FAKE, sizes=FAKE, tab=FAKE):
    return lib.mgw_resize_linear_mixed(ptr, fmt, S, mh, mw, sizes, tab, tab, out_h, out_w, ptr, None)


def test_empty_batch_returns_ok_without_a_launch(mgw):
    lib = mgw._lib.lib
    n0 = lib.mgw_launch_count()
    for fmt in (BGR, NV12, I420):
        assert cvt(lib, 0, 1080, 1920, fmt, ptr=None, sizes=None) == MGW_OK
        assert resize(lib, 0, 1080, 1920, fmt, ptr=None, sizes=None, tab=None) == MGW_OK
    assert lib.mgw_launch_count() == n0


def test_bad_capacity_and_format_are_rejected(mgw):
    lib = mgw._lib.lib
    for fn in (cvt, resize):
        for fmt in (3, -1):
            assert fn(lib, 2, 96, 128, fmt) == MGW_ERR_INVALID
            assert b'unknown format' in lib.mgw_last_error()
            assert fn(lib, 0, 96, 128, fmt, ptr=None, sizes=None) == MGW_ERR_INVALID     # checked before an empty batch returns
        for fmt in (BGR, NV12, I420):
            for mh, mw in ((0, 128), (96, 0), (-2, 128)):
                assert fn(lib, 2, mh, mw, fmt) == MGW_ERR_INVALID, (fn.__name__, fmt, mh, mw)
                assert b'bad sizes' in lib.mgw_last_error()
            assert fn(lib, 2, 96, 128, fmt, out_h=0) == MGW_ERR_INVALID
            assert fn(lib, -1, 96, 128, fmt) == MGW_ERR_INVALID
            assert fn(lib, 65536, 2, 2, fmt, out_h=1, out_w=1) == MGW_ERR_INVALID        # the slot index is gridDim.y
        for fmt in (NV12, I420):                                                         # a YUV capacity is even
            for mh, mw in ((97, 128), (96, 127)):
                assert fn(lib, 2, mh, mw, fmt) == MGW_ERR_INVALID
                assert fn(lib, 0, mh, mw, fmt, ptr=None, sizes=None) == MGW_ERR_INVALID
    assert cvt(lib, 2, 96, 128, ks=0) == MGW_ERR_INVALID


def test_sizes_past_the_32_bit_index_limits_are_rejected(mgw):
    lib = mgw._lib.lib
    for fn in (cvt, resize):
        # BGR: S*max_h*max_w < 2^29 -- 64 slots of a 2160x3840 capacity fit, 65 do not
        assert fn(lib, 65, 2160, 3840) == MGW_ERR_INVALID
        assert b'bad sizes' in lib.mgw_last_error()
        # YUV 4:2:0: S*(3max_h/2)*max_w < 2^31 -- 690 slots of 1080p fit, 691 do not
        for fmt in (NV12, I420):
            assert fn(lib, 691, 1080, 1920, fmt) == MGW_ERR_INVALID
            assert b'bad sizes' in lib.mgw_last_error()


def test_null_pointers_and_alignment(mgw):
    lib = mgw._lib.lib
    for fmt in (BGR, NV12, I420):
        for fn in (cvt, resize):
            assert fn(lib, 2, 96, 128, fmt, ptr=None) == MGW_ERR_INVALID
            assert b'null pointer' in lib.mgw_last_error()
            assert fn(lib, 2, 96, 128, fmt, sizes=None) == MGW_ERR_INVALID
            assert b'null pointer' in lib.mgw_last_error()
            assert fn(lib, 2, 96, 128, fmt, sizes=FAKE + 4) == MGW_ERR_INVALID           # sizes are read as one int2
            assert b'8-byte aligned' in lib.mgw_last_error()
        assert resize(lib, 2, 96, 128, fmt, tab=FAKE + 8) == MGW_ERR_INVALID             # tables are read as int4
        assert b'16-byte aligned' in lib.mgw_last_error()
        # the tables are required even where every slot could take the 2x2 shortcut (96x128 -> 48x64)
        assert resize(lib, 2, 96, 128, fmt, out_h=48, out_w=64, tab=None) == MGW_ERR_INVALID
        assert b'null pointer' in lib.mgw_last_error()


def test_padded_tables_are_the_uniform_tables(mgw):
    d = mgw.deploy
    cap = (1920, 1920)
    for (H, W), cr, (h, w) in [((1080, 1920), 1, (288, 512)), ((720, 1280), 1, (288, 512)), ((1920, 1080), 0.9, (288, 512)),
                               ((576, 1024), 1, (288, 512)), ((240, 426), 1, (288, 512)), ((91, 157), 0.8, (72, 128)),
                               ((1920, 1920), 1, (288, 512))]:
        kx, x0, xn, ky, y0, yn, xtab, ytab = d.mixed_slot_tables((H, W), cap, h, w, cr)
        ukx, ux0, uxn, uky, uy0, uyn = d._cvt_windows(H, W, h, w, cr)
        for pad, u in ((kx, ukx), (ky, uky)):
            assert pad.dtype == np.int32 and pad.shape[1] >= u.shape[1]
            assert np.array_equal(pad[:, :u.shape[1]], u) and not pad[:, u.shape[1]:].any(), (H, W, cr)
        for a, b in ((x0, ux0), (xn, uxn), (y0, uy0), (yn, uyn)):
            assert np.array_equal(a, b), (H, W, cr)
        assert np.array_equal(xtab, d._cv_linear_table(w, W, True)) and np.array_equal(ytab, d._cv_linear_table(h, H, False))
        rh, rw, _, _ = d._resample_size(h, w, cr)
        assert kx.shape == (w, d._pil_ksize(cap[1], rw)) and ky.shape == (h, d._pil_ksize(cap[0], rh))
    with pytest.raises(ValueError):
        d.mixed_slot_tables((1080, 1921), (1080, 1920))
    with pytest.raises(ValueError):
        d.mixed_slot_tables((0, 64), (1080, 1920))


@pytest.mark.parametrize('crop_rate', [1, 0.9, 0.8])
def test_no_slot_needs_a_longer_window_than_the_capacity(mgw, crop_rate):
    d = mgw.deploy
    for h, w in ((288, 512), (72, 128)):
        rh, rw, _, _ = d._resample_size(h, w, crop_rate)
        for cap_h, cap_w in ((1080, 1920), (1920, 1920), (2160, 3840), (97, 131)):
            ksx, ksy = d._pil_ksize(cap_w, rw), d._pil_ksize(cap_h, rh)
            for H in range(1, cap_h + 1, 7):
                assert d._pil_ksize(H, rh) <= ksy, (H, cap_h, crop_rate)
            for W in range(1, cap_w + 1, 7):
                assert d._pil_ksize(W, rw) <= ksx, (W, cap_w, crop_rate)
            # and the Pillow windows themselves are no longer than the length they are built for
            for n in (1, cap_w // 3, cap_w):
                kk, _, count = d._pil_bilinear_windows(n, rw)
                assert kk.shape[1] <= ksx and count.max() <= ksx


def test_mixed_stream_batch_rejects_bad_frames_without_a_gpu(mgw):
    mb = mgw.MixedStreamBatch(2, (96, 128), height=24, width=40, device='cpu')
    import torch
    for bad in (np.zeros((97, 128, 3), np.uint8), np.zeros((96, 129, 3), np.uint8), np.zeros((48, 64, 3), np.float32),
                np.zeros((48, 64), np.uint8), np.zeros((0, 64, 3), np.uint8)):
        with pytest.raises(ValueError):
            mb.join(0, bad)
    with pytest.raises(ValueError):
        mb.step(torch.zeros((2, 96 * 128 * 3 + 1), dtype=torch.uint8), None)           # pool shape
    with pytest.raises(ValueError):
        mb.step(torch.zeros(mb.pool_shape, dtype=torch.float32), None)                 # pool dtype
    with pytest.raises(ValueError):
        mb.slot_frame(torch.zeros(mb.pool_shape, dtype=torch.uint8), 0)                # slot 0 has not joined
    yb = mgw.MixedStreamBatch(2, (96, 128), height=24, width=40, device='cpu', src_format='nv12')
    for bad in (np.zeros((144, 127), np.uint8), np.zeros((145, 128), np.uint8), np.zeros((147, 128), np.uint8),
                np.zeros((96, 128, 3), np.uint8)):
        with pytest.raises(ValueError):
            yb.join(0, bad)
    with pytest.raises(ValueError):
        mgw.MixedStreamBatch(2, (97, 128), src_format='i420', device='cpu')            # odd YUV capacity

"""CPU: the per-slot warp (mgw_remap_bundle_frame_mixed) refuses bad arguments before anything reaches the device, in the batch
calls' order, and deploy.mixed_slot_tables(out_size=) gives the uniform resize tables at the slot's size for that output size."""
import numpy as np
import pytest

MGW_OK, MGW_ERR_INVALID = 0, -1
BGR, NV12, I420 = 0, 1, 2
FAKE = 1 << 20          # a non-null, 16-byte aligned address: never dereferenced, every call below fails or returns before a launch


@pytest.fixture(scope='module')
def mgw():
    import dovs_b200
    return dovs_b200


def remap(lib, S, mh, mw, fmt=BGR, dst_fmt=BGR, h=288, w=512, src=FAKE, sizes=FAKE, xy=FAKE, dst=FAKE, ws=FAKE):
    return lib.mgw_remap_bundle_frame_mixed(src, fmt, S, mh, mw, sizes, xy, h, w, dst_fmt, dst, ws, None)


def test_empty_batch_returns_ok_without_a_launch(mgw):
    lib = mgw._lib.lib
    n0 = lib.mgw_launch_count()
    for fmt in (BGR, NV12, I420):
        for dst_fmt in (BGR, NV12, I420):
            assert remap(lib, 0, 1080, 1920, fmt, dst_fmt, src=None, sizes=None, xy=None, dst=None, ws=None) == MGW_OK
    assert lib.mgw_launch_count() == n0


def test_unknown_formats_and_odd_yuv_capacity_are_rejected_before_an_empty_batch(mgw):
    lib = mgw._lib.lib
    for bad in (3, -1):
        for S in (2, 0):
            assert remap(lib, S, 96, 128, fmt=bad) == MGW_ERR_INVALID
            assert b'unknown format' in lib.mgw_last_error()
            assert remap(lib, S, 96, 128, dst_fmt=bad) == MGW_ERR_INVALID
            assert b'unknown destination format' in lib.mgw_last_error()
    for fmt, dst_fmt in ((NV12, BGR), (I420, BGR), (BGR, NV12), (BGR, I420), (NV12, I420)):
        for mh, mw in ((97, 128), (96, 127)):
            for S in (2, 0):
                assert remap(lib, S, mh, mw, fmt, dst_fmt) == MGW_ERR_INVALID, (fmt, dst_fmt, mh, mw, S)
                assert b'bad sizes' in lib.mgw_last_error()
    # BGR on both sides takes any capacity
    n0 = lib.mgw_launch_count()
    assert remap(lib, 0, 97, 127) == MGW_OK and lib.mgw_launch_count() == n0


def test_bad_capacity_and_map_sizes_are_rejected(mgw):
    lib = mgw._lib.lib
    for fmt, dst_fmt in ((BGR, BGR), (NV12, NV12), (I420, BGR), (BGR, I420)):
        for mh, mw in ((0, 128), (96, 0), (-2, 128), (32768, 128), (96, 32768)):
            assert remap(lib, 2, mh, mw, fmt, dst_fmt) == MGW_ERR_INVALID, (fmt, dst_fmt, mh, mw)
            assert b'bad sizes' in lib.mgw_last_error()
        for h, w in ((7, 512), (288, 7), (0, 0)):
            assert remap(lib, 2, 96, 128, fmt, dst_fmt, h=h, w=w) == MGW_ERR_INVALID
            assert b'bad sizes' in lib.mgw_last_error()
        assert remap(lib, -1, 96, 128, fmt, dst_fmt) == MGW_ERR_INVALID
        assert remap(lib, 65536, 8, 8, fmt, dst_fmt, h=8, w=8) == MGW_ERR_INVALID         # the slot index is gridDim.y
        assert b'bad sizes' in lib.mgw_last_error()


def test_sizes_past_the_32_bit_index_limits_are_rejected(mgw):
    lib = mgw._lib.lib
    n0 = lib.mgw_launch_count()
    for fmt, dst_fmt in ((BGR, BGR), (NV12, NV12), (I420, BGR)):
        # S*max_h*max_w*3 < 2^31: 345 slots of a 1080p capacity fit, 346 do not; the largest capacity side fits alone
        assert remap(lib, 346, 1080, 1920, fmt, dst_fmt) == MGW_ERR_INVALID
        assert b'bad sizes' in lib.mgw_last_error()
        assert remap(lib, 345, 1080, 1920, fmt, dst_fmt, src=None) == MGW_ERR_INVALID
        assert b'null pointer' in lib.mgw_last_error()                                    # the sizes passed
        assert remap(lib, 1, 32766, 21844, fmt, dst_fmt, src=None) == MGW_ERR_INVALID
        assert b'null pointer' in lib.mgw_last_error()
        assert remap(lib, 1, 32766, 21848, fmt, dst_fmt) == MGW_ERR_INVALID
        assert b'bad sizes' in lib.mgw_last_error()
    # S*h*w < 2^31 for the maps
    assert remap(lib, 2, 96, 128, h=32768, w=32768) == MGW_ERR_INVALID
    assert b'bad sizes' in lib.mgw_last_error()
    assert lib.mgw_launch_count() == n0


def test_null_pointers_and_alignment(mgw):
    lib = mgw._lib.lib
    n0 = lib.mgw_launch_count()
    for fmt, dst_fmt in ((BGR, BGR), (NV12, I420), (I420, BGR), (BGR, NV12)):
        for arg in ('src', 'sizes', 'xy', 'dst', 'ws'):
            assert remap(lib, 2, 96, 128, fmt, dst_fmt, **{arg: None}) == MGW_ERR_INVALID, arg
            assert b'null pointer' in lib.mgw_last_error()
        for arg, off in (('xy', 4), ('ws', 4), ('sizes', 4)):                             # float2 maps, int2 sizes
            assert remap(lib, 2, 96, 128, fmt, dst_fmt, **{arg: FAKE + off}) == MGW_ERR_INVALID, arg
            assert b'8-byte aligned' in lib.mgw_last_error()
    assert lib.mgw_launch_count() == n0


def test_slot_tables_for_an_output_size(mgw):
    d = mgw.deploy
    cap = (1920, 1920)
    for (H, W), out in [((1080, 1920), (1080, 1920)), ((720, 1280), (1080, 1920)), ((1920, 1080), (720, 1280)),
                        ((91, 157), (64, 96)), ((576, 1024), (288, 512)), ((123, 77), (123, 77))]:
        tabs = d.mixed_slot_tables((H, W), cap, 288, 512, 1, out_size=out)
        xtab, ytab = tabs[6], tabs[7]
        assert xtab.dtype == np.int32 and xtab.shape == (out[1], 4) and ytab.shape == (out[0], 4)
        assert np.array_equal(xtab, d._cv_linear_table(out[1], W, True)), (H, W, out)
        assert np.array_equal(ytab, d._cv_linear_table(out[0], H, False)), (H, W, out)
        # the front-end tables do not depend on the output size
        for a, b in zip(tabs[:6], d.mixed_slot_tables((H, W), cap, 288, 512, 1)[:6]):
            assert np.array_equal(a, b)
    # the default is the network's size, as before
    a, b = d.mixed_slot_tables((720, 1280), cap), d.mixed_slot_tables((720, 1280), cap, out_size=(288, 512))
    assert all(np.array_equal(x, y) for x, y in zip(a, b))


def test_mixed_stream_batch_output_modes_without_a_gpu(mgw):
    import torch
    for bad in ('src', 'Source', (0, 64), (64, 32768)):
        with pytest.raises(ValueError):
            mgw.MixedStreamBatch(2, (96, 128), height=24, width=40, device='cpu', out_size=bad)
    with pytest.raises(ValueError):                                                      # an odd capacity cannot hold YUV results
        mgw.MixedStreamBatch(2, (97, 128), height=24, width=40, device='cpu', out_size='source', out_format='nv12')
    mb = mgw.MixedStreamBatch(2, (96, 128), height=24, width=40, device='cpu', out_size='source', out_format='i420')
    assert mb.out_pool_shape == (2, 96 * 128 * 3 // 2) and tuple(mb.colour.shape) == mb.out_pool_shape and mb.small is None
    assert mb.out_size == 'source' and mb.xtab is None
    with pytest.raises(ValueError):
        mb.join(0, np.zeros((91, 128, 3), np.uint8))                                     # odd size with a YUV result
    with pytest.raises(ValueError):
        mb.slot_output(torch.zeros(mb.out_pool_shape, dtype=torch.uint8), 0)             # slot 0 has not joined
    bgr = mgw.MixedStreamBatch(2, (97, 127), height=24, width=40, device='cpu', out_size='source')
    assert bgr.out_pool_shape == (2, 97 * 127 * 3)
    common = mgw.MixedStreamBatch(2, (96, 128), height=24, width=40, device='cpu', out_size=(96, 128))
    assert tuple(common.small.shape) == (2, 96, 128, 3) and tuple(common.colour.shape) == (2, 96, 128, 3)
    assert tuple(common.xtab.shape) == (2, 128, 4) and tuple(common.ytab.shape) == (2, 96, 4)
    with pytest.raises(ValueError):
        common.slot_output(common.colour, 0)                                             # only with out_size='source'
    net = mgw.MixedStreamBatch(2, (96, 128), height=24, width=40, device='cpu')
    assert tuple(net.small.shape) == (2, 24, 40, 3) and tuple(net.xtab.shape) == (2, 40, 4)

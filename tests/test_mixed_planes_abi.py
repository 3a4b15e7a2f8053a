"""CPU: the mixed plane-table calls (mgw_cvt_img2train_mixed_planes, mgw_resize_linear_mixed_planes,
mgw_remap_bundle_frame_mixed_planes) refuse bad arguments before anything reaches the device, in the _mixed calls' order and
without the pool's limits; deploy.MixedPlaneTable checks each slot's planes at the slot's own size and writes that size into the
entry's reserved words; and a uniform batch refuses a mixed table (and a mixed batch a uniform one)."""
import numpy as np
import pytest

MGW_OK, MGW_ERR_INVALID = 0, -1
BGR, NV12, I420 = 0, 1, 2
FMTS = (BGR, NV12, I420)
FAKE = 1 << 20          # a non-null, 16-byte aligned address: never dereferenced, every call below fails or returns before a launch


@pytest.fixture(scope='module')
def mgw():
    import dovs_b200
    return dovs_b200


def cvt(lib, S, mh, mw, fmt=BGR, src=FAKE, sizes=FAKE, tabs=FAKE, tmp=FAKE, out=FAKE, ks=3, out_h=288, out_w=512):
    return lib.mgw_cvt_img2train_mixed_planes(src, fmt, S, mh, mw, sizes, tabs, tabs, tabs, ks, tabs, tabs, tabs, ks, out_h, out_w, tmp,
                                              out, None)


def resize(lib, S, mh, mw, fmt=BGR, src=FAKE, sizes=FAKE, xtab=FAKE, ytab=FAKE, dst=FAKE, out_h=288, out_w=512):
    return lib.mgw_resize_linear_mixed_planes(src, fmt, S, mh, mw, sizes, xtab, ytab, out_h, out_w, dst, None)


def remap(lib, S, mh, mw, fmt=BGR, dst_fmt=BGR, h=288, w=512, src=FAKE, sizes=FAKE, xy=FAKE, dst=FAKE, ws=FAKE):
    return lib.mgw_remap_bundle_frame_mixed_planes(src, fmt, S, mh, mw, sizes, xy, h, w, dst, dst_fmt, ws, None)


def err(lib, rc, what):
    return rc == MGW_ERR_INVALID and what in lib.mgw_last_error()


def test_formats_then_sizes_then_empty_batch(mgw):
    lib = mgw._lib.lib
    n0 = lib.mgw_launch_count()
    for bad in (3, -1):
        for S in (2, 0):
            assert err(lib, cvt(lib, S, 96, 128, bad, ks=0), b'unknown format')           # the format comes before the sizes
            assert err(lib, resize(lib, S, 96, 128, bad, out_w=0), b'unknown format')
            assert err(lib, remap(lib, S, 96, 128, fmt=bad, h=0), b'unknown format')
            assert err(lib, remap(lib, S, 96, 128, dst_fmt=bad, h=0), b'unknown destination format')
    for S in (2, 0):                                                           # bad sizes are refused before S = 0 returns
        for fmt in (NV12, I420):
            for mh, mw in ((97, 128), (96, 127)):
                assert err(lib, cvt(lib, S, mh, mw, fmt), b'bad sizes')
                assert err(lib, resize(lib, S, mh, mw, fmt), b'bad sizes')
        for fmt, dst_fmt in ((NV12, BGR), (BGR, NV12), (BGR, I420), (I420, NV12)):
            for mh, mw in ((97, 128), (96, 127)):
                assert err(lib, remap(lib, S, mh, mw, fmt, dst_fmt), b'bad sizes'), (fmt, dst_fmt, mh, mw, S)
    for fmt in FMTS:
        for mh, mw in ((0, 128), (96, 0), (-2, 128)):
            assert err(lib, cvt(lib, 2, mh, mw, fmt), b'bad sizes')
            assert err(lib, resize(lib, 2, mh, mw, fmt), b'bad sizes')
        for mh, mw in ((0, 128), (96, 0), (32768, 128), (96, 32768)):
            assert err(lib, remap(lib, 2, mh, mw, fmt, fmt), b'bad sizes')
        for S in (-1, 65536):                                                  # the slot index is gridDim.y
            assert err(lib, cvt(lib, S, 8, 8, fmt, out_h=8, out_w=8), b'bad sizes')
            assert err(lib, resize(lib, S, 8, 8, fmt, out_h=8, out_w=8), b'bad sizes')
            assert err(lib, remap(lib, S, 8, 8, fmt, fmt, h=8, w=8), b'bad sizes')
        assert err(lib, cvt(lib, 2, 96, 128, fmt, ks=0), b'bad sizes')
        assert err(lib, cvt(lib, 2, 96, 128, fmt, out_h=0), b'bad sizes')
        assert err(lib, resize(lib, 2, 96, 128, fmt, out_w=0), b'bad sizes')
        for h, w in ((7, 512), (288, 7)):
            assert err(lib, remap(lib, 2, 96, 128, fmt, fmt, h=h, w=w), b'bad sizes')
        assert cvt(lib, 0, 96, 128, fmt, src=None, sizes=None, tabs=None, tmp=None, out=None) == MGW_OK
        assert resize(lib, 0, 96, 128, fmt, src=None, sizes=None, xtab=None, ytab=None, dst=None) == MGW_OK
        for dst_fmt in FMTS:
            assert remap(lib, 0, 96, 128, fmt, dst_fmt, src=None, sizes=None, xy=None, dst=None, ws=None) == MGW_OK
    assert remap(lib, 0, 97, 127) == MGW_OK                                   # BGR on both sides takes an odd capacity
    assert lib.mgw_launch_count() == n0


def test_limits_bound_one_frame_and_the_outputs_not_a_pool(mgw):
    """there is no pool: S*max_h*max_w may exceed the _mixed calls' pool limits, while one frame, tmp, out and xy stay bounded"""
    lib = mgw._lib.lib
    n0 = lib.mgw_launch_count()
    # 300 BGR slots of 1080x1920: S*max_h*max_w > 2^29 (refused by mgw_cvt_img2train_mixed), accepted here up to the pointers
    assert err(lib, lib.mgw_cvt_img2train_mixed(FAKE, BGR, 300, 1080, 1920, FAKE, FAKE, FAKE, FAKE, 3, FAKE, FAKE, FAKE, 3, 288, 512, FAKE,
                                                FAKE, None), b'bad sizes')
    assert err(lib, cvt(lib, 300, 1080, 1920, src=None), b'null pointer')
    assert err(lib, resize(lib, 300, 1080, 1920, src=None), b'null pointer')
    assert err(lib, cvt(lib, 700, 2160, 3840, NV12, src=None), b'null pointer')  # S*(3H/2)*W > 2^31
    assert err(lib, remap(lib, 400, 1080, 1920, src=None), b'null pointer')   # S*max_h*max_w*3 > 2^31
    assert err(lib, remap(lib, 400, 1080, 1920, NV12, NV12, src=None), b'null pointer')
    # one frame: the capacity's limits at S = 1
    assert err(lib, cvt(lib, 1, 1 << 14, 1 << 15, out_h=8, out_w=8), b'bad sizes')          # max_h*max_w = 2^29 (BGR)
    assert err(lib, cvt(lib, 1, (1 << 14) - 2, 1 << 15, out_h=8, out_w=8, src=None), b'null pointer')
    assert err(lib, resize(lib, 1, 1 << 15, 1 << 16, NV12, out_h=8, out_w=8), b'bad sizes')  # (3H/2)*W > 2^31 (YUV)
    # tmp [S,max_h,out_w] < 2^31 bytes, out [S,out_h,out_w] < 2^29 elements, xy [S,h,w] < 2^31
    assert err(lib, cvt(lib, 3900, 1080, 512, out_h=8), b'bad sizes')          # 3900 * 1080 * 512 > 2^31
    assert err(lib, cvt(lib, 3800, 1080, 512, out_h=8, src=None), b'null pointer')
    assert err(lib, resize(lib, 3700, 96, 128), b'bad sizes')                 # 3700 * 288 * 512 > 2^29
    assert err(lib, resize(lib, 3600, 96, 128, src=None), b'null pointer')
    assert err(lib, remap(lib, 14600, 96, 128), b'bad sizes')                 # 14600 * 288 * 512 > 2^31
    assert err(lib, remap(lib, 14500, 96, 128, src=None), b'null pointer')
    assert lib.mgw_launch_count() == n0


def test_pointers_then_alignment(mgw):
    lib = mgw._lib.lib
    n0 = lib.mgw_launch_count()
    for fmt in FMTS:
        for arg in ('src', 'sizes', 'tabs', 'tmp', 'out'):
            assert err(lib, cvt(lib, 2, 96, 128, fmt, **{arg: None}), b'null pointer'), arg
        for arg in ('src', 'sizes', 'xtab', 'ytab', 'dst'):
            assert err(lib, resize(lib, 2, 96, 128, fmt, **{arg: None}), b'null pointer'), arg
        # null before any alignment; sizes (8 bytes) before the table (16 bytes)
        assert err(lib, cvt(lib, 2, 96, 128, fmt, src=FAKE + 8, sizes=None), b'null pointer')
        assert err(lib, cvt(lib, 2, 96, 128, fmt, src=FAKE + 8, sizes=FAKE + 4), b'sizes must be 8-byte aligned')
        assert err(lib, cvt(lib, 2, 96, 128, fmt, src=FAKE + 8), b'16-byte aligned')
        assert err(lib, resize(lib, 2, 96, 128, fmt, xtab=FAKE + 4), b'tables must be 16-byte aligned')
        assert err(lib, resize(lib, 2, 96, 128, fmt, src=FAKE + 8, sizes=FAKE + 4), b'sizes must be 8-byte aligned')
        for off in (4, 8):
            assert err(lib, resize(lib, 2, 96, 128, fmt, src=FAKE + off), b'planes table must be 16-byte aligned')
        for dst_fmt in FMTS:
            for arg in ('src', 'sizes', 'xy', 'dst', 'ws'):
                assert err(lib, remap(lib, 2, 96, 128, fmt, dst_fmt, **{arg: None}), b'null pointer'), arg
            for arg in ('xy', 'ws', 'sizes'):
                assert err(lib, remap(lib, 2, 96, 128, fmt, dst_fmt, src=FAKE + 8, **{arg: FAKE + 4}), b'8-byte aligned'), arg
            for arg in ('src', 'dst'):
                assert err(lib, remap(lib, 2, 96, 128, fmt, dst_fmt, **{arg: FAKE + 8}), b'planes tables must be 16-byte aligned'), arg
    assert lib.mgw_launch_count() == n0


def entries(t):
    return t.host.numpy().view(np.dtype([('plane', '<u8', (3,)), ('pitch', '<i4', (3,)), ('reserved', '<i4', (3,))])).reshape(t.S)


def test_set_writes_the_slot_size_into_the_reserved_words(mgw):
    t = mgw.MixedPlaneTable(3, 'nv12', (2160, 3840), device='cpu')
    assert not isinstance(t, mgw.PlaneTable) and t.capacity == (2160, 3840) and tuple(t.host.shape) == (3, 6)
    t.set(1, ((0x4000_0000, 1536), (0x4000_0000 + 1536 * 720, 1536)), (720, 1280))     # NVDEC layout of a 720p surface
    t.set(0, ((0x10, 3840), (0x20, 3840)), (2160, 3840))
    e = entries(t)
    assert list(e[1]['plane'][:2]) == [0x4000_0000, 0x4000_0000 + 1536 * 720] and list(e[1]['pitch'][:2]) == [1536, 1536]
    assert list(e[1]['reserved']) == [720, 1280, 0] and list(e[0]['reserved']) == [2160, 3840, 0]
    raw = t.host.numpy()[1]                                                   # C layout: reserved[0] at byte 36, reserved[1] at 40
    assert raw[4] >> 32 == 720 and raw[5] & 0xffffffff == 1280
    assert not e[2]['plane'].any() and not e[2]['reserved'].any()
    t.clear(1)
    assert not entries(t)[1]['plane'].any() and not entries(t)[1]['reserved'].any()
    t.upload()
    assert np.array_equal(t.device.numpy(), t.host.numpy())
    bgr = mgw.MixedPlaneTable(1, 'bgr', (9, 7), device='cpu')
    bgr.set(0, ((0x1000, 15),), (3, 5))                                        # odd BGR sizes; planes checked at 5 columns
    assert list(entries(bgr)[0]['reserved']) == [3, 5, 0] and entries(bgr)[0]['pitch'][0] == 15


def test_set_checks_planes_at_the_slot_size(mgw):
    import torch
    t = mgw.MixedPlaneTable(2, 'i420', (96, 128), device='cpu')
    y, u = torch.zeros(48, 64, dtype=torch.uint8), torch.zeros(24, 32, dtype=torch.uint8)
    t.set(0, (y, u, u), (48, 64))                                               # covers the slot's size, not the capacity: fine
    assert list(entries(t)[0]['pitch']) == [64, 32, 32]
    with pytest.raises(ValueError, match='cover'):
        t.set(0, (y[:47], u, u), (48, 64))                                      # a plane too short
    with pytest.raises(ValueError, match='cover'):
        t.set(0, (y[:, :62], u, u), (48, 64))                                   # a plane too narrow
    with pytest.raises(ValueError, match='cover'):
        t.set(0, (y, u, u), (50, 64))                                           # the same planes at a larger size
    with pytest.raises(ValueError, match='below'):
        t.set(0, ((0x1000, 64), (0x2000, 31), (0x3000, 32)), (48, 64))
    with pytest.raises(ValueError, match='missing'):
        t.set(0, ((0x1000, 64), (0x2000, 32), (0, 32)), (48, 64))
    with pytest.raises(ValueError, match='planes'):
        t.set(0, ((0x1000, 64),), (48, 64))
    for bad in ((98, 128), (96, 130), (0, 64), (48, 0), (47, 64), (48, 63)):   # above the capacity, empty, odd for YUV
        with pytest.raises(ValueError, match='capacity'):
            t.set(1, ((0x1000, 128), (0x2000, 64), (0x3000, 64)), bad)
    with pytest.raises(ValueError, match='slot'):
        t.set(2, ((0x1000, 64), (0x2000, 32), (0x3000, 32)), (48, 64))
    e = entries(t)
    assert list(e[0]['reserved']) == [48, 64, 0] and not e[1]['plane'].any()   # nothing written by a refusal
    for bad in (dict(fmt='yuyv'), dict(capacity=(95, 128)), dict(capacity=(0, 128)), dict(S=0), dict(S=65536)):
        kw = dict(S=2, fmt='nv12', capacity=(96, 128), device='cpu')
        kw.update(bad)
        with pytest.raises(ValueError):
            mgw.MixedPlaneTable(**kw)


def test_pool_table_describes_each_slot_at_its_size(mgw):
    import torch
    cap = (96, 128)
    pool = torch.zeros(3, 96 * 3 // 2 * 128, dtype=torch.uint8)
    t = mgw.MixedPlaneTable.pool(pool, 'i420', cap, [(48, 64), None, (96, 128)])
    e, base, row = entries(t), pool.data_ptr(), pool.shape[1]
    assert list(e[0]['plane']) == [base, base + 48 * 64, base + 48 * 64 + 24 * 32] and list(e[0]['pitch']) == [64, 32, 32]
    assert list(e[0]['reserved']) == [48, 64, 0] and not e[1]['plane'].any()
    assert e[2]['plane'][0] == base + 2 * row and list(e[2]['reserved']) == [96, 128, 0]
    assert np.array_equal(t.device.numpy(), t.host.numpy())                    # uploaded
    with pytest.raises(ValueError):
        mgw.MixedPlaneTable.pool(pool, 'nv12', (96, 130), [None] * 3)           # not a pool of that capacity
    with pytest.raises(ValueError):
        mgw.MixedPlaneTable.pool(pool, 'i420', cap, [None] * 2)


def test_batches_refuse_the_other_kind_of_table(mgw):
    import torch
    net = lambda x: None                                                     # noqa: E731 -- never reached
    sb = mgw.StreamBatch(2, (96, 128), height=24, width=40, device='cpu', src_format='nv12')
    mixed = mgw.MixedPlaneTable(2, 'nv12', (96, 128), device='cpu')
    with pytest.raises(ValueError, match='PlaneTable'):
        sb.step_planes(mixed, net)
    with pytest.raises(ValueError, match='PlaneTable'):
        sb.capture_planes(mixed, net)
    with pytest.raises(ValueError, match='PlaneTable'):
        sb.step_planes(mgw.PlaneTable(2, 'nv12', (96, 128), device='cpu'), net, mgw.MixedPlaneTable(2, 'bgr', (24, 40), device='cpu'))

    for out_size in ('source', None):
        mb = mgw.MixedStreamBatch(2, (96, 128), height=24, width=40, device='cpu', src_format='nv12', out_size=out_size)
        for run in (mb.step_planes, mb.capture_planes):
            with pytest.raises(TypeError):
                run(mgw.PlaneTable(2, 'nv12', (96, 128), device='cpu'), net)
            with pytest.raises(TypeError):
                run(torch.zeros(2, 6, dtype=torch.int64), net)
            for bad in (mgw.MixedPlaneTable(2, 'i420', (96, 128), device='cpu'), mgw.MixedPlaneTable(3, 'nv12', (96, 128), device='cpu'),
                        mgw.MixedPlaneTable(2, 'nv12', (96, 130), device='cpu')):
                with pytest.raises(ValueError, match='must describe'):
                    run(bad, net)
    mb = mgw.MixedStreamBatch(2, (96, 128), height=24, width=40, device='cpu', src_format='nv12', out_size='source', out_format='i420')
    with pytest.raises(TypeError):                                            # 'source' writes a mixed table
        mb.step_planes(mixed, net, mgw.PlaneTable(2, 'i420', (96, 128), device='cpu'))
    with pytest.raises(ValueError, match='must describe'):
        mb.step_planes(mixed, net, mgw.MixedPlaneTable(2, 'nv12', (96, 128), device='cpu'))
    mb = mgw.MixedStreamBatch(2, (96, 128), height=24, width=40, device='cpu', src_format='nv12', out_size=(48, 64))
    with pytest.raises(ValueError, match='PlaneTable'):                       # a common output size writes a uniform table
        mb.step_planes(mixed, net, mgw.MixedPlaneTable(2, 'bgr', (48, 64), device='cpu'))
    with pytest.raises(ValueError, match='must describe'):
        mb.step_planes(mixed, net, mgw.PlaneTable(2, 'bgr', (96, 128), device='cpu'))

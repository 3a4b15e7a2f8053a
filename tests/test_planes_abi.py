"""CPU: the plane-table calls (mgw_cvt_img2train_planes, mgw_resize_linear_planes, mgw_remap_bundle_frame_planes) refuse bad
arguments before anything reaches the device, in the batch calls' order; the ctypes mirror of mgw_planes matches the header; and
deploy.PlaneTable packs (address, pitch) pairs into that layout and refuses entries a slot could not be read from."""
import ctypes
import os
import re

import numpy as np
import pytest

MGW_OK, MGW_ERR_INVALID = 0, -1
BGR, NV12, I420 = 0, 1, 2
FMTS = (BGR, NV12, I420)
FAKE = 1 << 20          # a non-null, 16-byte aligned address: never dereferenced, every call below fails or returns before a launch
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope='module')
def mgw():
    import dovs_b200
    return dovs_b200


def cvt(lib, S, H, W, fmt=BGR, src=FAKE, tmp=FAKE, out=FAKE, tabs=FAKE, ks=3, out_h=288, out_w=512):
    return lib.mgw_cvt_img2train_planes(src, fmt, S, H, W, tabs, tabs, tabs, ks, tabs, tabs, tabs, ks, out_h, out_w, tmp, out, None)


def resize(lib, S, H, W, fmt=BGR, src=FAKE, xtab=FAKE, ytab=FAKE, dst=FAKE, out_h=288, out_w=512):
    return lib.mgw_resize_linear_planes(src, fmt, S, H, W, xtab, ytab, out_h, out_w, dst, None)


def remap(lib, S, H, W, fmt=BGR, dst_fmt=BGR, h=288, w=512, src=FAKE, xy=FAKE, dst=FAKE, ws=FAKE):
    return lib.mgw_remap_bundle_frame_planes(src, fmt, xy, S, h, w, H, W, dst, dst_fmt, ws, None)


def test_struct_matches_the_header(mgw):
    P = mgw._lib.mgw_planes
    assert ctypes.sizeof(P) == 48
    assert P.plane.offset == 0 and P.pitch.offset == 24 and P.reserved.offset == 36
    hdr = re.sub(r'/\*.*?\*/', '', open(os.path.join(ROOT, 'include', 'mgw.h')).read(), flags=re.S)
    m = re.search(r'typedef struct \{([^}]*)\} mgw_planes;', hdr)
    assert m and re.sub(r'\s+', ' ', m.group(1)).strip() == 'uint64_t plane[3]; int32_t pitch[3]; int32_t reserved[3];'
    assert mgw.ops.PLANES_ENTRY_BYTES == 48
    assert mgw.deploy._PLANES_DTYPE.itemsize == 48 and mgw.deploy._PLANES_DTYPE.fields['pitch'][1] == 24


def test_empty_batch_returns_ok_without_a_launch(mgw):
    lib = mgw._lib.lib
    n0 = lib.mgw_launch_count()
    for fmt in FMTS:
        assert cvt(lib, 0, 1080, 1920, fmt, src=None, tmp=None, out=None, tabs=None) == MGW_OK
        assert resize(lib, 0, 1080, 1920, fmt, src=None, xtab=None, ytab=None, dst=None) == MGW_OK
        for dst_fmt in FMTS:
            assert remap(lib, 0, 1080, 1920, fmt, dst_fmt, src=None, xy=None, dst=None, ws=None) == MGW_OK
    assert lib.mgw_launch_count() == n0


def test_unknown_formats_are_rejected_before_an_empty_batch(mgw):
    lib = mgw._lib.lib
    for bad in (3, -1):
        for S in (2, 0):
            assert cvt(lib, S, 96, 128, bad) == MGW_ERR_INVALID and b'unknown format' in lib.mgw_last_error()
            assert resize(lib, S, 96, 128, bad) == MGW_ERR_INVALID and b'unknown format' in lib.mgw_last_error()
            assert remap(lib, S, 96, 128, fmt=bad) == MGW_ERR_INVALID and b'unknown format' in lib.mgw_last_error()
            assert remap(lib, S, 96, 128, dst_fmt=bad) == MGW_ERR_INVALID
            assert b'unknown destination format' in lib.mgw_last_error()


def test_bad_and_odd_sizes_are_rejected_before_an_empty_batch(mgw):
    lib = mgw._lib.lib
    for S in (2, 0):
        for fmt in (NV12, I420):
            for H, W in ((97, 128), (96, 127)):
                assert cvt(lib, S, H, W, fmt) == MGW_ERR_INVALID and b'bad sizes' in lib.mgw_last_error()
                assert resize(lib, S, H, W, fmt) == MGW_ERR_INVALID and b'bad sizes' in lib.mgw_last_error()
        for fmt, dst_fmt in ((NV12, BGR), (I420, BGR), (BGR, NV12), (BGR, I420), (NV12, I420), (I420, NV12)):
            for H, W in ((97, 128), (96, 127)):
                assert remap(lib, S, H, W, fmt, dst_fmt) == MGW_ERR_INVALID, (fmt, dst_fmt, H, W, S)
                assert b'bad sizes' in lib.mgw_last_error()
    for fmt in FMTS:
        for H, W in ((0, 128), (96, 0), (-2, 128)):
            assert cvt(lib, 2, H, W, fmt) == MGW_ERR_INVALID and b'bad sizes' in lib.mgw_last_error()
            assert resize(lib, 2, H, W, fmt) == MGW_ERR_INVALID and b'bad sizes' in lib.mgw_last_error()
        for H, W in ((0, 128), (96, 0), (32768, 128), (96, 32768)):
            assert remap(lib, 2, H, W, fmt, fmt) == MGW_ERR_INVALID and b'bad sizes' in lib.mgw_last_error()
        for S in (-1, 65536):                                                  # the slot index is gridDim.y
            assert cvt(lib, S, 8, 8, fmt, out_h=8, out_w=8) == MGW_ERR_INVALID and b'bad sizes' in lib.mgw_last_error()
            assert resize(lib, S, 8, 8, fmt, out_h=8, out_w=8) == MGW_ERR_INVALID and b'bad sizes' in lib.mgw_last_error()
            assert remap(lib, S, 8, 8, fmt, fmt, h=8, w=8) == MGW_ERR_INVALID and b'bad sizes' in lib.mgw_last_error()
        assert cvt(lib, 2, 96, 128, fmt, ks=0) == MGW_ERR_INVALID and b'bad sizes' in lib.mgw_last_error()
        assert cvt(lib, 2, 96, 128, fmt, out_h=0) == MGW_ERR_INVALID
        assert resize(lib, 2, 96, 128, fmt, out_w=0) == MGW_ERR_INVALID
        for h, w in ((7, 512), (288, 7)):
            assert remap(lib, 2, 96, 128, fmt, fmt, h=h, w=w) == MGW_ERR_INVALID and b'bad sizes' in lib.mgw_last_error()
    # BGR on both sides of the warp takes any size; the 32-bit limits of the uniform calls hold
    n0 = lib.mgw_launch_count()
    assert remap(lib, 0, 97, 127) == MGW_OK
    assert remap(lib, 346, 1080, 1920) == MGW_ERR_INVALID and b'bad sizes' in lib.mgw_last_error()
    assert remap(lib, 345, 1080, 1920, src=None) == MGW_ERR_INVALID and b'null pointer' in lib.mgw_last_error()
    assert cvt(lib, 259, 1080, 1920) == MGW_ERR_INVALID and b'bad sizes' in lib.mgw_last_error()       # S*H*W < 2^29 for BGR
    assert cvt(lib, 258, 1080, 1920, src=None) == MGW_ERR_INVALID and b'null pointer' in lib.mgw_last_error()
    assert lib.mgw_launch_count() == n0


def test_null_pointers_and_alignment(mgw):
    lib = mgw._lib.lib
    n0 = lib.mgw_launch_count()
    for fmt in FMTS:
        for arg in ('src', 'tmp', 'out', 'tabs'):
            assert cvt(lib, 2, 96, 128, fmt, **{arg: None}) == MGW_ERR_INVALID and b'null pointer' in lib.mgw_last_error(), arg
        for arg in ('src', 'dst'):
            assert resize(lib, 2, 96, 128, fmt, **{arg: None}) == MGW_ERR_INVALID and b'null pointer' in lib.mgw_last_error(), arg
        assert resize(lib, 2, 96, 128, fmt, xtab=None) == MGW_ERR_INVALID and b'tables are required' in lib.mgw_last_error()
        assert resize(lib, 2, 96, 128, fmt, xtab=FAKE + 4) == MGW_ERR_INVALID and b'16-byte aligned' in lib.mgw_last_error()
        for off in (4, 8):                                                     # the table: 16-byte vector loads
            assert cvt(lib, 2, 96, 128, fmt, src=FAKE + off) == MGW_ERR_INVALID and b'16-byte aligned' in lib.mgw_last_error()
            assert resize(lib, 2, 96, 128, fmt, src=FAKE + off) == MGW_ERR_INVALID and b'16-byte aligned' in lib.mgw_last_error()
        for dst_fmt in FMTS:
            for arg in ('src', 'xy', 'dst', 'ws'):
                assert remap(lib, 2, 96, 128, fmt, dst_fmt, **{arg: None}) == MGW_ERR_INVALID, arg
                assert b'null pointer' in lib.mgw_last_error()
            for arg in ('src', 'dst'):
                assert remap(lib, 2, 96, 128, fmt, dst_fmt, **{arg: FAKE + 8}) == MGW_ERR_INVALID, arg
                assert b'16-byte aligned' in lib.mgw_last_error()
            for arg in ('xy', 'ws'):
                assert remap(lib, 2, 96, 128, fmt, dst_fmt, **{arg: FAKE + 4}) == MGW_ERR_INVALID, arg
                assert b'8-byte aligned' in lib.mgw_last_error()
    assert lib.mgw_launch_count() == n0


def entries(t):
    return t.host.numpy().view(np.dtype([('plane', '<u8', (3,)), ('pitch', '<i4', (3,)), ('reserved', '<i4', (3,))])).reshape(t.S)


def test_plane_table_packs_address_pitch_pairs(mgw):
    PT = mgw.PlaneTable
    t = PT(4, 'i420', (1080, 1920), device='cpu')
    assert tuple(t.host.shape) == (4, 6) and t.host.dtype.itemsize == 8 and tuple(t.device.shape) == (4, 6)
    assert not entries(t)['plane'].any()                                      # every slot starts idle
    t.set(2, ((0x7000_0000_1000, 1923), (0x7000_0100_0000, 960), (0x7100_0000_0003, 1001)))
    t.set(0, ((0x10, 1920), (0x20, 960), (0x30, 960)))
    e = entries(t)
    assert list(e[2]['plane']) == [0x7000_0000_1000, 0x7000_0100_0000, 0x7100_0000_0003] and list(e[2]['pitch']) == [1923, 960, 1001]
    assert list(e[0]['plane']) == [0x10, 0x20, 0x30] and not e[0]['reserved'].any()
    raw = t.host.numpy()[2]                                                   # the C layout: 3 addresses, then the pitches at byte 24
    assert raw[0] == 0x7000_0000_1000 and raw[3] == 1923 | (960 << 32) and raw[4] == 1001
    assert not e[1]['plane'].any() and not e[3]['plane'].any()
    t.clear(2)
    assert not entries(t)[2]['plane'].any() and not entries(t)[2]['pitch'].any() and entries(t)[0]['plane'][0] == 0x10
    t.upload()
    assert np.array_equal(t.device.numpy(), t.host.numpy())

    nv = PT(2, 'nv12', (1080, 1920), device='cpu')
    pitch = 2048
    nv.set(1, ((0x4000_0000, pitch), (0x4000_0000 + pitch * 1088, pitch)))     # NVDEC: chroma at row 1088 of the surface
    assert list(entries(nv)[1]['plane'][:2]) == [0x4000_0000, 0x4000_0000 + pitch * 1088] and entries(nv)[1]['plane'][2] == 0
    bgr = PT(1, 'bgr', (7, 5), device='cpu')
    bgr.set(0, ((0x1000, 15),))
    assert entries(bgr)[0]['pitch'][0] == 15


def test_plane_table_rejects_entries_a_slot_cannot_be_read_from(mgw):
    PT = mgw.PlaneTable
    t = PT(2, 'nv12', (1080, 1920), device='cpu')
    with pytest.raises(ValueError, match='planes'):
        t.set(0, ((0x1000, 1920),))                                          # NV12 has two planes
    with pytest.raises(ValueError, match='missing'):
        t.set(0, ((0x1000, 1920), (0, 1920)))
    with pytest.raises(ValueError, match='below'):
        t.set(0, ((0x1000, 1919), (0x2000, 1920)))                           # a Y row is 1920 bytes
    with pytest.raises(ValueError, match='below'):
        t.set(0, ((0x1000, 1920), (0x2000, 960)))                            # so is an interleaved UV row
    with pytest.raises(ValueError, match='slot'):
        t.set(2, ((0x1000, 1920), (0x2000, 1920)))
    assert not entries(t)['plane'].any()                                      # nothing was written
    i420 = PT(1, 'i420', (1080, 1920), device='cpu')
    with pytest.raises(ValueError, match='below'):
        i420.set(0, ((0x1000, 1920), (0x2000, 960), (0x3000, 959)))
    bgr = PT(1, 'bgr', (1080, 1920), device='cpu')
    with pytest.raises(ValueError, match='below'):
        bgr.set(0, ((0x1000, 1920 * 3 - 1),))
    with pytest.raises(ValueError, match='below'):
        bgr.set(0, ((0x1000, 1 << 31),))
    for bad in (dict(fmt='yuyv'), dict(size=(1079, 1920)), dict(S=0), dict(S=65536)):
        kw = dict(S=2, fmt='nv12', size=(1080, 1920), device='cpu')
        kw.update(bad)
        with pytest.raises(ValueError):
            PT(**kw)


def test_stream_batch_planes_entry_points_check_their_tables(mgw):
    import torch
    sb = mgw.StreamBatch(2, (96, 128), height=24, width=40, device='cpu', src_format='nv12')
    net = lambda x: None                                                     # noqa: E731 -- never reached
    with pytest.raises(ValueError, match='PlaneTable'):
        sb.step_planes(torch.zeros(2, 6, dtype=torch.int64), net)
    with pytest.raises(ValueError, match='must describe'):
        sb.step_planes(mgw.PlaneTable(2, 'i420', (96, 128), device='cpu'), net)
    with pytest.raises(ValueError, match='must describe'):
        sb.step_planes(mgw.PlaneTable(3, 'nv12', (96, 128), device='cpu'), net)
    with pytest.raises(ValueError, match='must describe'):
        sb.capture_planes(mgw.PlaneTable(2, 'nv12', (96, 130), device='cpu'), net)
    mb = mgw.MixedStreamBatch(2, (96, 128), height=24, width=40, device='cpu')
    with pytest.raises(TypeError):
        mb.step_planes(mgw.PlaneTable(2, 'bgr', (96, 128), device='cpu'), net)
    with pytest.raises(TypeError):
        mb.capture_planes(mgw.PlaneTable(2, 'bgr', (96, 128), device='cpu'), net)

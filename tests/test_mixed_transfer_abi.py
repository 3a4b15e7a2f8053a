"""CPU: the exact-bytes pool transfer (mgw_copy_slots_mixed, ops.copy_slots_mixed, MixedStreamBatch.capture(exact_bytes=True))
refuses bad arguments before anything reaches the device, in the batch calls' order."""
import pytest

MGW_OK, MGW_ERR_INVALID = 0, -1
BGR, NV12, I420 = 0, 1, 2
FAKE = 1 << 20          # a non-null, 16-byte aligned address: never dereferenced, every call below fails or returns before a launch


@pytest.fixture(scope='module')
def mgw():
    import dovs_b200
    return dovs_b200


def copy(lib, S, mh, mw, fmt=BGR, src=FAKE, dst=FAKE, sizes=FAKE):
    return lib.mgw_copy_slots_mixed(src, dst, fmt, S, mh, mw, sizes, None)


def test_empty_batch_returns_ok_without_a_launch(mgw):
    lib = mgw._lib.lib
    n0 = lib.mgw_launch_count()
    for fmt in (BGR, NV12, I420):
        assert copy(lib, 0, 1080, 1920, fmt, src=None, dst=None, sizes=None) == MGW_OK
        assert copy(lib, 0, 1080, 1920, fmt, src=FAKE + 1, dst=FAKE + 3, sizes=FAKE + 4) == MGW_OK
    assert lib.mgw_launch_count() == n0


def test_unknown_format_and_odd_yuv_capacity_are_rejected_before_an_empty_batch(mgw):
    lib = mgw._lib.lib
    n0 = lib.mgw_launch_count()
    for bad in (3, -1):
        for S in (2, 0):
            assert copy(lib, S, 96, 128, bad) == MGW_ERR_INVALID
            assert b'unknown format' in lib.mgw_last_error()
    # the format is checked first: an unknown one is named even with bad sizes
    assert copy(lib, -1, 0, 0, 3) == MGW_ERR_INVALID and b'unknown format' in lib.mgw_last_error()
    for fmt in (NV12, I420):
        for mh, mw in ((97, 128), (96, 127), (1, 1)):
            for S in (2, 0):
                assert copy(lib, S, mh, mw, fmt) == MGW_ERR_INVALID, (fmt, mh, mw, S)
                assert b'bad sizes' in lib.mgw_last_error()
    # BGR takes any capacity
    assert copy(lib, 0, 97, 127) == MGW_OK and copy(lib, 0, 1, 1) == MGW_OK
    assert lib.mgw_launch_count() == n0


def test_bad_capacity_and_slot_counts_are_rejected(mgw):
    lib = mgw._lib.lib
    n0 = lib.mgw_launch_count()
    for fmt in (BGR, NV12, I420):
        for mh, mw in ((0, 128), (96, 0), (-2, 128), (96, -2), (32768, 128), (96, 32768)):
            assert copy(lib, 2, mh, mw, fmt) == MGW_ERR_INVALID, (fmt, mh, mw)
            assert b'bad sizes' in lib.mgw_last_error()
        assert copy(lib, -1, 96, 128, fmt) == MGW_ERR_INVALID
        assert b'bad sizes' in lib.mgw_last_error()
        assert copy(lib, 65536, 2, 2, fmt) == MGW_ERR_INVALID                             # the slot index is gridDim.y
        assert b'bad sizes' in lib.mgw_last_error()
        assert copy(lib, 65535, 2, 2, fmt, src=None) == MGW_ERR_INVALID
        assert b'null pointer' in lib.mgw_last_error()                                    # the sizes passed
    assert lib.mgw_launch_count() == n0


def test_pools_past_the_32_bit_limit_are_rejected(mgw):
    lib = mgw._lib.lib
    n0 = lib.mgw_launch_count()
    # S * frame_bytes(capacity) < 2^31: 345 BGR slots of a 1080p capacity fit and 346 do not; 690 / 691 for YUV 4:2:0
    for fmt, fit in ((BGR, 345), (NV12, 690), (I420, 690)):
        assert copy(lib, fit + 1, 1080, 1920, fmt) == MGW_ERR_INVALID
        assert b'bad sizes' in lib.mgw_last_error()
        assert copy(lib, fit, 1080, 1920, fmt, dst=None) == MGW_ERR_INVALID
        assert b'null pointer' in lib.mgw_last_error()
    # one BGR slot: 32767 x 21846 x 3 < 2^31 <= 32767 x 21847 x 3; the largest even YUV capacity fits alone
    assert copy(lib, 1, 32767, 21846, BGR, sizes=None) == MGW_ERR_INVALID and b'null pointer' in lib.mgw_last_error()
    assert copy(lib, 1, 32767, 21847, BGR) == MGW_ERR_INVALID and b'bad sizes' in lib.mgw_last_error()
    assert copy(lib, 1, 32766, 32766, NV12, sizes=None) == MGW_ERR_INVALID and b'null pointer' in lib.mgw_last_error()
    assert lib.mgw_launch_count() == n0


def test_null_pointers_and_alignment(mgw):
    lib = mgw._lib.lib
    n0 = lib.mgw_launch_count()
    for fmt in (BGR, NV12, I420):
        for arg in ('src', 'dst', 'sizes'):
            assert copy(lib, 2, 96, 128, fmt, **{arg: None}) == MGW_ERR_INVALID, arg
            assert b'null pointer' in lib.mgw_last_error()
        for arg in ('src', 'dst'):
            for off in (1, 4, 8):
                assert copy(lib, 2, 96, 128, fmt, **{arg: FAKE + off}) == MGW_ERR_INVALID, (arg, off)
                assert b'16-byte aligned' in lib.mgw_last_error()
        for off in (1, 4):                                                                # int2 sizes
            assert copy(lib, 2, 96, 128, fmt, sizes=FAKE + off) == MGW_ERR_INVALID
            assert b'8-byte aligned' in lib.mgw_last_error()
        # a null pointer is named before a misaligned one
        assert copy(lib, 2, 96, 128, fmt, src=FAKE + 1, sizes=None) == MGW_ERR_INVALID
        assert b'null pointer' in lib.mgw_last_error()
    assert lib.mgw_launch_count() == n0


def test_python_errors_before_the_call(mgw):
    import torch
    ops = mgw.ops
    n0 = mgw.launch_count()
    sizes = torch.zeros((2, 2), dtype=torch.int32)
    a, b = torch.zeros((2, 96, 128, 3), dtype=torch.uint8), torch.zeros((2, 96, 128, 3), dtype=torch.uint8)
    for bad in ('rgb', 'NV12', None):
        with pytest.raises(ValueError, match='format'):
            ops.copy_slots_mixed(a, b, bad, sizes)
    with pytest.raises(ValueError, match='pageable'):                                    # both pageable
        ops.copy_slots_mixed(a, b, 'bgr', sizes)
    for other in (torch.zeros((2, 96, 127, 3), dtype=torch.uint8), torch.zeros((3, 96, 128, 3), dtype=torch.uint8),
                  torch.zeros((2, 96 * 128 * 3), dtype=torch.uint8)):
        with pytest.raises(ValueError, match='one shape'):
            ops.copy_slots_mixed(a, other, 'bgr', sizes)
    with pytest.raises(ValueError):                                                      # a pool of another format's shape
        ops.copy_slots_mixed(a, b, 'nv12', sizes)
    with pytest.raises(ValueError):                                                      # a flat pool does not give the capacity
        ops.copy_slots_mixed(a.view(2, -1), b.view(2, -1), 'bgr', sizes)
    with pytest.raises(ValueError):
        ops.copy_slots_mixed(a, b, 'bgr', sizes[:1])
    with pytest.raises(ValueError):
        ops.copy_slots_mixed(a, b.float(), 'bgr', sizes)
    y = torch.zeros((2, 144, 128), dtype=torch.uint8)
    with pytest.raises(ValueError, match='pageable'):
        ops.copy_slots_mixed(y, y.clone(), 'i420', sizes)
    assert mgw.launch_count() == n0


def test_exact_bytes_capture_needs_pinned_host_buffers(mgw):
    import torch
    for out in ('source', None):
        mb = mgw.MixedStreamBatch(2, (96, 128), height=24, width=40, device='cpu', out_size=out)
        pool = torch.zeros(mb.pool_shape, dtype=torch.uint8)
        with pytest.raises(ValueError, match='pinned'):
            mb.capture(pool, None, upload_from=torch.zeros(mb.pool_shape, dtype=torch.uint8), exact_bytes=True)
        with pytest.raises(ValueError, match='pinned'):
            mb.capture(pool, None, download_to=torch.zeros(tuple(mb.colour.shape), dtype=torch.uint8), exact_bytes=True)

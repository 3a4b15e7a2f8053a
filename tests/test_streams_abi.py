"""CPU: argument checks of the batched deploy entry points (mgw_*_batch, mgw_streams_*).  Every check below is decided before
anything reaches the device, so it runs without a GPU: an empty batch is a no-op, bad sizes and taps are errors."""
import ctypes

import pytest

MGW_OK, MGW_ERR_INVALID = 0, -1
FAKE = 1 << 20          # a non-null, 16-byte aligned address: never dereferenced, every call below fails or returns before a launch


@pytest.fixture(scope='module')
def lib():
    import dovs_b200
    return dovs_b200._lib.lib


def taps(*t):
    return (ctypes.c_int * len(t))(*t)


def cvt(lib, S, H, W, out_h=288, out_w=512, ptr=FAKE):
    return lib.mgw_cvt_img2train_u8_batch(ptr, S, H, W, ptr, ptr, ptr, 5, ptr, ptr, ptr, 5, out_h, out_w, ptr, ptr, None)


def resize(lib, S, H, W, C=3, out_h=288, out_w=512, ptr=FAKE, tab=FAKE):
    return lib.mgw_resize_linear_u8_batch(ptr, S, H, W, C, tab, tab, out_h, out_w, ptr, None)


def assemble(lib, S, depth, H, W, t=(1, 2, 4, 8, 16, 32), ptr=FAKE):
    return lib.mgw_streams_assemble(ptr, ptr, S, depth, ptr, taps(*t), len(t), 1, ptr, H, W, ptr, None)


def push(lib, S, depth, H, W, ptr=FAKE):
    return lib.mgw_streams_push(ptr, ptr, S, depth, ptr, ptr, ptr, H, W, None)


def test_empty_batch_returns_ok_without_a_launch(lib):
    n0 = lib.mgw_launch_count()
    assert cvt(lib, 0, 1080, 1920, ptr=None) == MGW_OK
    assert resize(lib, 0, 1080, 1920, ptr=None, tab=None) == MGW_OK
    assert assemble(lib, 0, 32, 288, 512, ptr=None) == MGW_OK
    assert push(lib, 0, 32, 288, 512, ptr=None) == MGW_OK
    assert lib.mgw_launch_count() == n0


def test_sizes_past_the_32_bit_index_limits_are_rejected(lib):
    # 1080p BGR frames: S*H*W must stay below 2^29 (byte offsets of the 3-channel frames): 258 frames fit, 259 do not
    assert cvt(lib, 259, 1080, 1920) == MGW_ERR_INVALID
    assert b'bad sizes' in lib.mgw_last_error()
    assert resize(lib, 259, 1080, 1920) == MGW_ERR_INVALID
    # rings: S*depth*H*W < 2^31 floats; 288x512 with depth 32 allows 455 streams
    assert assemble(lib, 456, 32, 288, 512) == MGW_ERR_INVALID
    assert push(lib, 456, 32, 288, 512) == MGW_ERR_INVALID
    # the stream index is gridDim.y
    assert push(lib, 65536, 1, 1, 1) == MGW_ERR_INVALID
    for fn in (cvt, resize):
        assert fn(lib, -1, 48, 64) == MGW_ERR_INVALID
    assert assemble(lib, -1, 32, 48, 64) == MGW_ERR_INVALID


def test_bad_arguments_are_rejected(lib):
    assert assemble(lib, 2, 32, 48, 64, t=(1, 33)) == MGW_ERR_INVALID
    assert b'tap 33' in lib.mgw_last_error()
    assert assemble(lib, 2, 32, 48, 64, t=(0,)) == MGW_ERR_INVALID
    assert assemble(lib, 2, 32, 48, 64, ptr=None) == MGW_ERR_INVALID
    assert push(lib, 2, 32, 48, 64, ptr=None) == MGW_ERR_INVALID
    assert cvt(lib, 2, 96, 128, ptr=None) == MGW_ERR_INVALID
    assert resize(lib, 2, 96, 128, ptr=None) == MGW_ERR_INVALID
    assert resize(lib, 2, 96, 128, C=2) == MGW_ERR_INVALID
    assert resize(lib, 2, 96, 128, tab=FAKE + 4) == MGW_ERR_INVALID                 # tables must be 16-byte aligned
    assert resize(lib, 2, 96, 128, tab=None) == MGW_ERR_INVALID                     # tables are needed unless 2x2 decimation
    assert b'tables are required' in lib.mgw_last_error()

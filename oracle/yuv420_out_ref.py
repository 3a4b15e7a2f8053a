"""TEST INFRASTRUCTURE -- numpy restatement of cv2.cvtColor(COLOR_BGR2YUV_I420), the inverse of yuv420_ref.yuv420_to_bgr, and the
generator of tests/golden/deploy_yuv420_out.npz, made from OpenCV alone (no reference sources needed):

    python oracle/yuv420_out_ref.py        # rewrites tests/golden/deploy_yuv420_out.npz

OpenCV 4.13 (color_yuv.simd.hpp), BT.601 limited range in 20-bit fixed point; the plain C++ path and the optimised path give the
same bytes.  Y of every pixel; U and V of the TOP-LEFT pixel of each 2x2 block only (the four pixels are not averaged):
  Y = (269484 R + 528482 G + 102760 B + (16 << 20) + (1 << 19)) >> 20
  U = (-155188 R - 305135 G + 460324 B + (128 << 20) + (1 << 19)) >> 20
  V = (460324 R - 385875 G - 74448 B + (128 << 20) + (1 << 19)) >> 20
Every sum lies in [16 << 20, 241 << 20): nothing saturates.  Odd sizes are an error.  The layout is yuv420_ref's (I420: Y, U, V
planes; NV12 is yuv420_ref.i420_to_nv12 of it -- OpenCV has no BGR -> NV12 code).  Only tests/ may import this module.
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
import yuv420_ref  # noqa: E402

OUT = os.path.join(os.path.dirname(HERE), 'tests', 'golden', 'deploy_yuv420_out.npz')
SIZES = ((2, 2), (6, 10), (90, 158))       # random bytes; 90x158: W not a multiple of 4
BLOCK = (288, 512)                         # a block frame (remap_frame_ref.block_frame): compresses well


def bgr_to_i420(bgr):
    """cv2.cvtColor(bgr, COLOR_BGR2YUV_I420) of a BGR uint8 frame [H,W,3], H and W even -> [3H/2,W] uint8 (Y, U, V planes)"""
    bgr = np.ascontiguousarray(bgr, np.uint8)
    H, W, _ = bgr.shape
    assert H % 2 == 0 and W % 2 == 0, bgr.shape
    b, g, r = (bgr[..., k].astype(np.int64) for k in range(3))
    Y = (269484 * r + 528482 * g + 102760 * b + (16 << 20) + (1 << 19)) >> 20
    b, g, r = b[::2, ::2], g[::2, ::2], r[::2, ::2]
    U = (-155188 * r - 305135 * g + 460324 * b + (128 << 20) + (1 << 19)) >> 20
    V = (460324 * r - 385875 * g - 74448 * b + (128 << 20) + (1 << 19)) >> 20
    return np.concatenate([Y.reshape(-1), U.reshape(-1), V.reshape(-1)]).astype(np.uint8).reshape(H * 3 // 2, W)


def bgr_to_yuv420(bgr, fmt):
    """bgr_to_i420 in fmt 'i420' or 'nv12' (U and V interleaved)"""
    i420 = bgr_to_i420(bgr)
    if fmt == 'i420':
        return i420
    assert fmt == 'nv12', fmt
    return yuv420_ref.i420_to_nv12(i420)


def gen_cases():
    """cv2.cvtColor(COLOR_BGR2YUV_I420) of BGR frames straight from OpenCV: random bytes at small sizes and a block frame at the
    network's size.  The plain C++ path makes the stored bytes and the optimised path must agree."""
    import cv2
    import remap_frame_ref
    rng = np.random.RandomState(4200)
    frames = {'random_%dx%d' % s: rng.randint(0, 256, s + (3,)).astype(np.uint8) for s in SIZES}
    frames['block_%dx%d' % BLOCK] = remap_frame_ref.block_frame(BLOCK[0], BLOCK[1], rng)
    fx = {}
    for name, bgr in frames.items():
        try:
            cv2.setUseOptimized(False)
            i420 = cv2.cvtColor(bgr, cv2.COLOR_BGR2YUV_I420)
        finally:
            cv2.setUseOptimized(True)
        assert np.array_equal(i420, cv2.cvtColor(bgr, cv2.COLOR_BGR2YUV_I420)), name
        fx[name + '_bgr'], fx[name + '_i420'] = bgr, i420
    fx['cv2_version'] = np.array(cv2.__version__)
    return fx


if __name__ == '__main__':
    np.savez_compressed(OUT, **gen_cases())
    print('%s %.1f KB' % (OUT, os.path.getsize(OUT) / 1024))

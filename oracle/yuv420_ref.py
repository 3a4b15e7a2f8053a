"""TEST INFRASTRUCTURE -- numpy restatement of cv2.cvtColor(COLOR_YUV2BGR_NV12 / COLOR_YUV2BGR_I420) and the generator of
tests/golden/deploy_yuv420.npz, made from OpenCV alone (no reference sources needed):

    python oracle/yuv420_ref.py            # rewrites tests/golden/deploy_yuv420.npz

The conversion lives in a third-party dependency (OpenCV 4.13 here, color_yuv.simd.hpp); the plain C++ path and the optimised
path give the same bytes.  A frame is [3H/2, W] uint8 with H and W even: the Y plane, then
  NV12: H/2 rows of W bytes of interleaved U,V;
  I420: the U plane, then the V plane, H/2 x W/2 bytes each, contiguous (byte offsets H*W and H*W + H*W/4, not row offsets).
One chroma sample per 2x2 block, no chroma interpolation; BT.601 limited range in 20-bit fixed point:
  u = U-128, v = V-128, y = max(0, Y-16)*CY
  R = sat8((y + 2^19 + CVR*v) >> 20), G = sat8((y + 2^19 + CVG*v + CUG*u) >> 20), B = sat8((y + 2^19 + CUB*u) >> 20)
Every sum fits int32.  cv2.VideoCapture converts with FFmpeg's swscale instead, which is not byte-identical to this.
Only tests/ may import this module.
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
OUT = os.path.join(os.path.dirname(HERE), 'tests', 'golden', 'deploy_yuv420.npz')

CY, CUB, CUG, CVG, CVR = 1220542, 2116026, -409993, -852492, 1673527

FORMATS = ('nv12', 'i420')
SIZES = ((2, 2), (6, 10), (36, 64), (90, 158), (72, 128))      # 90x158: W not a multiple of 4; 72x128: the resize's 2x2 shortcut
RESIZE = {(72, 128): (36, 64), (90, 158): (36, 64)}            # (H, W) -> (h, w) of the stored cv2.resize of the BGR frame


def planes(yuv, fmt):
    """(Y [H,W], U [H/2,W/2], V [H/2,W/2]) of a frame [3H/2,W] in OpenCV's layout"""
    yuv = np.ascontiguousarray(yuv, np.uint8)
    rows, W = yuv.shape
    assert rows % 3 == 0 and W % 2 == 0, yuv.shape
    H = rows // 3 * 2
    Y, c = yuv[:H], yuv[H:].reshape(-1)
    if fmt == 'nv12':
        uv = c.reshape(H // 2, W // 2, 2)
        return Y, uv[..., 0], uv[..., 1]
    assert fmt == 'i420', fmt
    n = (H // 2) * (W // 2)
    return Y, c[:n].reshape(H // 2, W // 2), c[n:].reshape(H // 2, W // 2)


def yuv420_to_bgr(yuv, fmt):
    """cv2.cvtColor(yuv, COLOR_YUV2BGR_NV12 / _I420) -> BGR uint8 [H,W,3]; fmt 'nv12' or 'i420'"""
    Y, U, V = planes(yuv, fmt)
    u = np.repeat(np.repeat(U.astype(np.int64) - 128, 2, 0), 2, 1)
    v = np.repeat(np.repeat(V.astype(np.int64) - 128, 2, 0), 2, 1)
    y = np.maximum(Y.astype(np.int64) - 16, 0) * CY + (1 << 19)
    b = (y + CUB * u) >> 20
    g = (y + CVG * v + CUG * u) >> 20
    r = (y + CVR * v) >> 20
    return np.clip(np.stack([b, g, r], -1), 0, 255).astype(np.uint8)


def i420_to_nv12(yuv):
    """the same picture with the U and V planes interleaved"""
    Y, U, V = planes(yuv, 'i420')
    return np.concatenate([Y.reshape(-1), np.stack([U.reshape(-1), V.reshape(-1)], -1).reshape(-1)]).reshape(yuv.shape)


def random_frame(rng, H, W):
    return rng.randint(0, 256, (H * 3 // 2, W)).astype(np.uint8)


def limited_frame(H, W, seed):
    """a limited-range I420 frame: cv2's BGR2YUV_I420 of a smooth image (synth.smooth_image)"""
    import cv2
    sys.path.insert(0, HERE)
    import synth
    bgr = ((synth.smooth_image(1, H, W, 3, seed)[0] + 0.5) * 255).astype(np.uint8)
    return cv2.cvtColor(bgr, cv2.COLOR_BGR2YUV_I420)


def gen_yuv420_cases():
    """cv2.cvtColor of small 4:2:0 frames straight from OpenCV: random bytes (the saturating clamps) and limited-range frames (the
    non-saturating path), both formats.  The plain C++ path makes the stored bytes and the optimised path must agree.  The RESIZE
    sizes also carry cv2.resize of the BGR frame (plain path): the 2x2 shortcut and the linear path."""
    import cv2
    codes = {'nv12': cv2.COLOR_YUV2BGR_NV12, 'i420': cv2.COLOR_YUV2BGR_I420}
    fx = {}
    rng = np.random.RandomState(420)
    for H, W in SIZES:
        i420 = limited_frame(H, W, H * 1000 + W)
        content = {'random': {f: random_frame(rng, H, W) for f in FORMATS}, 'limited': {'i420': i420, 'nv12': i420_to_nv12(i420)}}
        for kind, frames in content.items():
            for fmt, yuv in frames.items():
                name = '%s_%s_%dx%d' % (fmt, kind, H, W)
                try:
                    cv2.setUseOptimized(False)
                    bgr = cv2.cvtColor(yuv, codes[fmt])
                    resized = cv2.resize(bgr, RESIZE[(H, W)][::-1]) if (H, W) in RESIZE else None
                finally:
                    cv2.setUseOptimized(True)
                assert np.array_equal(bgr, cv2.cvtColor(yuv, codes[fmt])), name
                fx[name + '_yuv'], fx[name + '_bgr'] = yuv, bgr
                if resized is not None:
                    fx[name + '_resized'] = resized
    return fx


if __name__ == '__main__':
    np.savez_compressed(OUT, **gen_yuv420_cases())
    print('%s %.1f KB' % (OUT, os.path.getsize(OUT) / 1024))

"""TEST INFRASTRUCTURE -- warpRevBundle2 at any output size, and the generator of tests/golden/deploy_remap_frame.npz, made from
OpenCV alone (no reference sources needed):

    python oracle/remap_frame_ref.py       # rewrites tests/golden/deploy_remap_frame.npz

The reference resizes the colour frame to the network's size before it warps it (deploy_bundle.py:301).  The maps are normalised
coordinates and are decimated to a (h/4, w/4) grid before they are upsampled, so the same network output warps the frame at any
size; only the size the frame is resized to becomes a parameter (OH, OW):

    frame_o = cv2.resize(frame, (OW, OH))                            # skipped when (OH, OW) is the frame's size
    xs = cv2.resize(cv2.resize(x_map, (w // 4, h // 4)), (OW, OH))   # (h, w) = the maps' size
    ys = cv2.resize(cv2.resize(y_map, (w // 4, h // 4)), (OW, OH))
    dst = cv2.remap(frame_o, (xs + 1) / 2 * OW, (ys + 1) / 2 * OH, cv2.INTER_LINEAR)        # fp32, constant border 0

At (OH, OW) == (h, w) this is warpRevBundle2(cv2.resize(frame, (w, h)), x_map, y_map).  A YUV 4:2:0 frame is first converted as
cv2.cvtColor(COLOR_YUV2BGR_NV12 / _I420) converts it.  Restated with the pieces of deploy_ref (OpenCV's plain C++ path,
cv2.setUseOptimized(False)) and yuv420_ref.  Only tests/ may import this module.
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
import deploy_ref as R          # noqa: E402
import yuv420_ref as Y          # noqa: E402

OUT = os.path.join(os.path.dirname(HERE), 'tests', 'golden', 'deploy_remap_frame.npz')
f32 = np.float32


def warp_rev_bundle2_sized(frame, x_map, y_map, out_size, src_format='bgr'):
    """the stabilised frame [OH,OW,3] (BGR) of a frame of any size (BGR [H,W,3] or YUV 4:2:0 [3H/2,W]) and maps [h,w]"""
    if src_format != 'bgr':
        frame = Y.yuv420_to_bgr(frame, src_format)
    OH, OW = (int(v) for v in out_size)
    h, w = x_map.shape
    f = frame if frame.shape[:2] == (OH, OW) else R.resize_linear_u8(frame, OW, OH)
    xs = R.resize_linear(R.resize_linear(np.asarray(x_map, f32), w // 4, h // 4), OW, OH)
    ys = R.resize_linear(R.resize_linear(np.asarray(y_map, f32), w // 4, h // 4), OW, OH)
    xp = ((xs + f32(1)) / f32(2) * f32(OW)).astype(f32)
    yp = ((ys + f32(1)) / f32(2) * f32(OH)).astype(f32)
    return R.remap_linear_u8(f, xp, yp)


def cv2_sized(frame, x_map, y_map, out_size):
    """the same expression evaluated by cv2 (BGR frame); the caller picks OpenCV's path"""
    import cv2
    OH, OW = (int(v) for v in out_size)
    h, w = x_map.shape
    f = frame if frame.shape[:2] == (OH, OW) else cv2.resize(frame, (OW, OH))
    xs = cv2.resize(cv2.resize(x_map, (w // 4, h // 4)), (OW, OH))
    ys = cv2.resize(cv2.resize(y_map, (w // 4, h // 4)), (OW, OH))
    return cv2.remap(f, ((xs + 1) / 2 * OW).astype(f32), ((ys + 1) / 2 * OH).astype(f32), cv2.INTER_LINEAR)


def smooth_mesh(h, w, seed, noise=0.01):
    """maps near the identity with a smooth warp and a little noise, as the network emits them"""
    rs = np.random.RandomState(seed)
    yy, xx = np.meshgrid(np.linspace(-1, 1, h), np.linspace(-1, 1, w), indexing='ij')
    xm = (xx * 0.93 + 0.02 * np.sin(3 * yy) + noise * rs.standard_normal((h, w))).astype(f32)
    ym = (yy * 0.95 + 0.03 * np.cos(2 * xx) + noise * rs.standard_normal((h, w))).astype(f32)
    return xm, ym


def block_frame(H, W, rng):
    """a BGR frame of 16x16 blocks of one random colour each: sharp edges and flat areas, and it compresses well, so the fixture
    stays small"""
    blocks = rng.randint(0, 256, ((H + 15) // 16, (W + 15) // 16, 3)).astype(np.uint8)
    return np.ascontiguousarray(np.repeat(np.repeat(blocks, 16, 0), 16, 1)[:H, :W])


def wild_mesh(h, w, seed):
    """maps far outside [-1, 1] with NaN and +-Inf entries (the constant border, cvRound's INT_MIN)"""
    rs = np.random.RandomState(seed)
    xm = (rs.standard_normal((h, w)) * 3).astype(f32)
    ym = (rs.standard_normal((h, w)) * 3).astype(f32)
    for m in (xm, ym):
        idx = rs.randint(0, h * w, 12)
        m.reshape(-1)[idx[:4]] = np.nan
        m.reshape(-1)[idx[4:8]] = np.inf
        m.reshape(-1)[idx[8:]] = -np.inf
    return xm, ym


# (tag, maps (h, w), mesh, frame (H, W), outputs): outputs equal to, smaller and larger than the frame, odd sizes and the 2x2
# decimation of the frame resize (OpenCV's INTER_AREA shortcut).  The 288x512 maps are a noise-free smooth mesh stored as float16
# (every float16 is exact in float32), which keeps the fixture small; the 36x64 maps carry the noise and the non-finite values.
CASES = (
    ('net', (288, 512), 'half', (180, 320), ((180, 320), (288, 512), (90, 160), (37, 61))),
    ('small', (36, 64), 'smooth', (72, 128), ((72, 128), (36, 64), (101, 203))),
    ('wild', (36, 64), 'wild', (60, 96), ((60, 96), (30, 48), (45, 77))),
)


def fixture_maps(g, tag):
    """a case's x_map, y_map from the fixture as the float32 maps the network hands out"""
    return g[tag + '_x_map'].astype(f32), g[tag + '_y_map'].astype(f32)


def gen_cases():
    import cv2
    fx = {}
    rng = np.random.RandomState(2024)
    for tag, (h, w), kind, (H, W), outs in CASES:
        if kind == 'wild':
            xm, ym = wild_mesh(h, w, h * 7 + w)
        else:
            xm, ym = smooth_mesh(h, w, h * 7 + w, noise=0.0 if kind == 'half' else 0.01)
        if kind == 'half':
            xm, ym = xm.astype(np.float16), ym.astype(np.float16)
        frame = block_frame(H, W, rng)
        frame[:H // 8] = rng.randint(0, 256, (H // 8, W, 3))           # random bytes in the top eighth: every clamp of the blend
        fx[tag + '_x_map'], fx[tag + '_y_map'], fx[tag + '_frame'] = xm, ym, frame
        xm, ym = xm.astype(f32), ym.astype(f32)
        for OH, OW in outs:
            name = '%s_%dx%d' % (tag, OH, OW)
            try:
                cv2.setUseOptimized(False)
                dst = cv2_sized(frame, xm, ym, (OH, OW))
                cv2.setUseOptimized(True)
                dst_opt = cv2_sized(frame, xm, ym, (OH, OW))
            finally:
                cv2.setUseOptimized(True)
            fx[name + '_dst'] = dst
            fx[name + '_opt_diff_frac'] = np.float64(np.mean(dst != dst_opt))
            fx[name + '_opt_diff_max'] = np.int64(np.abs(dst.astype(int) - dst_opt.astype(int)).max())
    fx['cv2_version'] = np.array(cv2.__version__)
    return fx


if __name__ == '__main__':
    np.savez_compressed(OUT, **gen_cases())
    print('%s %.1f KB' % (OUT, os.path.getsize(OUT) / 1024))

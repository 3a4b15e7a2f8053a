"""GPU: stabilised frames handed out as YUV 4:2:0 (mgw_remap_bundle_frame_yuv420, ops.remap_bundle_frame(out_format=...),
deploy.warpRevBundle2(dst_format=...), StreamBatch / MixedStreamBatch(out_format=...)).  Every comparison is bit-exact: the result
must be cv2.cvtColor(COLOR_BGR2YUV_I420) of the BGR result -- OpenCV's bytes in tests/golden/deploy_remap_frame.npz, or the BGR
call's output -- converted by the numpy restatement oracle/yuv420_out_ref.bgr_to_i420 (and yuv420_ref.i420_to_nv12 for NV12)."""
import numpy as np
import pytest
import torch

import remap_frame_ref as M
import yuv420_out_ref as O
import yuv420_ref as Y
from conftest import load_golden
from test_gpu_remap_frame import cuda, frames_for, xy_of
from test_gpu_streams import fake_net_batch, identity_mesh, rect_or_none

pytestmark = pytest.mark.gpu

OUT_FORMATS = ('nv12', 'i420')


@pytest.fixture(scope='module')
def mgw():
    import dovs_b200
    assert torch.cuda.is_available(), 'GPU tests need a CUDA device; there is no CPU fallback'
    return dovs_b200


def yuv_of(bgr, fmt):
    """the restatement of one BGR frame [H,W,3] (numpy) as a 4:2:0 frame [3H/2,W] in fmt"""
    return O.bgr_to_yuv420(bgr, fmt)


def yuv_batch(bgr, fmt):
    """the restatement of a BGR batch [S,H,W,3] (tensor) -> [S,3H/2,W] numpy"""
    return np.stack([yuv_of(f, fmt) for f in bgr.cpu().numpy()])


def test_every_even_fixture_case(mgw):
    """slot k of a batch of 5 (and a batch of 1) holds the fixture's frame resized to the output size; its 4:2:0 result is the
    conversion of OpenCV's BGR bytes"""
    g = load_golden('deploy_remap_frame')
    rs = np.random.RandomState(70)
    n = 0
    for tag, _, _, _, outs in M.CASES:
        xm, ym = M.fixture_maps(g, tag)
        frame = cuda(g[tag + '_frame'])
        for OH, OW in outs:
            if OH % 2 or OW % 2:
                continue
            want = g['%s_%dx%d_dst' % (tag, OH, OW)]
            src = frame if tuple(frame.shape[:2]) == (OH, OW) else mgw.deploy.cv2_resize(frame, (OW, OH))
            for S in (1, 5):
                batch = cuda(rs.randint(0, 256, (S, OH, OW, 3)).astype(np.uint8))
                xy = cuda(rs.uniform(-1.2, 1.2, (S,) + xm.shape + (2,)).astype(np.float32))
                k = min(3, S - 1)
                batch[k], xy[k] = src, xy_of(xm, ym)
                for fmt in OUT_FORMATS:
                    got = mgw.ops.remap_bundle_frame(batch, 'bgr', xy, out_format=fmt)
                    assert got.shape == (S, OH * 3 // 2, OW)
                    assert np.array_equal(got[k].cpu().numpy(), yuv_of(want, fmt)), (tag, OH, OW, S, fmt)
            n += 1
    assert n == 7


# (frame (H, W), maps (h, w), mesh): the network's size, 1080p read directly, 720p, W not a multiple of 4, the smallest frame
SIZES = (((288, 512), (288, 512), 'smooth'), ((1080, 1920), (288, 512), 'smooth'), ((720, 1280), (288, 512), 'wild'),
         ((90, 158), (36, 64), 'wild'), ((2, 2), (36, 64), 'smooth'), ((90, 158), (36, 64), 'smooth'))


@pytest.mark.parametrize('src_fmt', ['bgr', 'nv12', 'i420'])
def test_yuv_out_equals_the_converted_bgr_out(mgw, src_fmt):
    rs = np.random.RandomState(71)
    for (H, W), (h, w), mesh in SIZES:
        S = 2 if H >= 720 else 3
        src = frames_for(rs, src_fmt, S, H, W)
        maps = M.wild_mesh(h, w, H + W) if mesh == 'wild' else M.smooth_mesh(h, w, H + W)
        xy = xy_of(*maps)[None].repeat(S, 1, 1, 1).contiguous()
        xy[S - 1] = cuda(rs.uniform(-1.3, 1.3, (h, w, 2)).astype(np.float32))
        bgr = mgw.ops.remap_bundle_frame(src, src_fmt, xy)
        for fmt in OUT_FORMATS:
            out = torch.full((S, H * 3 // 2, W), 7, device='cuda', dtype=torch.uint8)
            got = mgw.ops.remap_bundle_frame(src, src_fmt, xy, out=out, out_format=fmt)
            assert got.data_ptr() == out.data_ptr()
            assert np.array_equal(got.cpu().numpy(), yuv_batch(bgr, fmt)), (src_fmt, fmt, H, W, mesh)


def test_unaligned_destination(mgw):
    """a destination that starts 1 byte off a word: every store falls back to bytes and the result is the same"""
    rs = np.random.RandomState(72)
    S, H, W = 3, 90, 160
    src = frames_for(rs, 'bgr', S, H, W)
    xy = xy_of(*M.smooth_mesh(36, 64, 1))[None].repeat(S, 1, 1, 1).contiguous()
    for fmt in OUT_FORMATS:
        want = mgw.ops.remap_bundle_frame(src, 'bgr', xy, out_format=fmt)
        buf = torch.zeros(S * H * 3 // 2 * W + 1, device='cuda', dtype=torch.uint8)
        got = mgw.ops.remap_bundle_frame(src, 'bgr', xy, out=buf[1:].view(S, H * 3 // 2, W), out_format=fmt)
        assert torch.equal(got, want) and int(buf[0]) == 0, fmt


def test_warp_rev_bundle2_dst_format(mgw):
    rs = np.random.RandomState(73)
    frame = rs.randint(0, 256, (1080, 1920, 3)).astype(np.uint8)
    xm, ym = M.smooth_mesh(288, 512, 74)
    bgr = mgw.deploy.warpRevBundle2(frame, xm, ym)
    small = rs.randint(0, 256, (288, 512, 3)).astype(np.uint8)
    small_bgr = mgw.deploy.warpRevBundle2(small, xm, ym)          # the maps' size: the network-size call
    nv12_src = Y.random_frame(rs, 1080, 1920)
    nv12_bgr = mgw.deploy.warpRevBundle2(nv12_src, xm, ym, src_format='nv12')
    for fmt in OUT_FORMATS:
        got = mgw.deploy.warpRevBundle2(frame, xm, ym, dst_format=fmt)
        assert isinstance(got, np.ndarray) and got.shape == (1620, 1920)
        assert np.array_equal(got, yuv_of(bgr, fmt)), fmt
        assert np.array_equal(mgw.deploy.warpRevBundle2(small, xm, ym, dst_format=fmt), yuv_of(small_bgr, fmt)), fmt
        assert np.array_equal(mgw.deploy.warpRevBundle2(nv12_src, xm, ym, src_format='nv12', dst_format=fmt), yuv_of(nv12_bgr, fmt))
        two = mgw.deploy.warpRevBundle2(cuda(np.stack([frame, frame])), cuda(np.stack([xm, xm])), cuda(np.stack([ym, ym])),
                                        dst_format=fmt)
        assert two.is_cuda and two.shape == (2, 1620, 1920) and np.array_equal(two[1].cpu().numpy(), got), fmt
    with pytest.raises(ValueError):
        mgw.deploy.warpRevBundle2(frame, xm, ym, dst_format='rgb')
    with pytest.raises(ValueError):
        mgw.deploy.warpRevBundle2(frame[:1079], xm, ym, dst_format='nv12')


# ---- StreamBatch(out_format=...) against the BGR batch, step by step
@pytest.mark.parametrize('src_fmt,out', [(f, o) for f in ('bgr', 'nv12') for o in ('default', (720, 1280), 'src')])
def test_stream_batch_out_format(mgw, src_fmt, out):
    S, H, W, h, w, refine = 3, 360, 640, 72, 128, 1
    out_size = None if out == 'default' else (H, W) if out == 'src' else out
    OH, OW = (h, w) if out_size is None else out_size
    net, _ = fake_net_batch(mgw, identity_mesh())
    mk = lambda fmt: mgw.StreamBatch(S, (H, W), height=h, width=w, refine=refine, src_format=src_fmt, out_size=out_size,  # noqa: E731
                                     out_format=fmt)
    ref, sbs = mk('bgr'), {fmt: mk(fmt) for fmt in OUT_FORMATS}
    for fmt, sb in sbs.items():
        assert sb.colour.shape == (S, OH * 3 // 2, OW) and (sb.small is None) == (out == 'src'), fmt
    rs = np.random.RandomState(75)
    joins, leaves = {0: [0, 1, 2], 9: [1], 17: [0], 30: [2]}, {8: [1], 16: [0], 29: [2], 39: [0, 1, 2]}
    for k in range(40):
        for s in joins.get(k, []):
            first = frames_for(rs, src_fmt, 1, H, W)[0]
            ref.join(s, first)
            for sb in sbs.values():
                sb.join(s, first)
        raw = frames_for(rs, src_fmt, S, H, W)
        bgr = ref.step(raw, net)
        for fmt, sb in sbs.items():
            got = sb.step(raw, net)
            assert got.data_ptr() == sb.colour.data_ptr()
            assert np.array_equal(got.cpu().numpy(), yuv_batch(bgr, fmt)), (k, fmt)
        for s in leaves.get(k, []):
            want = rect_or_none(lambda: ref.leave(s))
            for sb in sbs.values():
                assert rect_or_none(lambda: sb.leave(s)) == want, (k, s)
    for sb in sbs.values():
        for a, b in ((sb.frames, ref.frames), (sb.masks, ref.masks), (sb.heads_dev, ref.heads_dev), (sb.all_black, ref.all_black)):
            assert torch.equal(a, b)


@pytest.mark.parametrize('src_fmt,out,fmt', [('nv12', 'src', 'nv12'), ('bgr', 'default', 'i420'), ('bgr', (720, 1280), 'nv12')])
def test_stream_batch_out_format_graph_replay_equals_eager(mgw, src_fmt, out, fmt):
    S, H, W, h, w = 3, 360, 640, 72, 128
    out_size = None if out == 'default' else (H, W) if out == 'src' else out
    OH, OW = (h, w) if out_size is None else out_size
    net, _ = fake_net_batch(mgw, identity_mesh())
    eager, graphed = (mgw.StreamBatch(S, (H, W), height=h, width=w, refine=2, src_format=src_fmt, out_size=out_size, out_format=fmt)
                      for _ in range(2))
    rs = np.random.RandomState(76)
    host_in = torch.empty((S,) + graphed.frame_shape, dtype=torch.uint8).pin_memory()
    host_out = torch.empty((S, OH * 3 // 2, OW), dtype=torch.uint8).pin_memory()
    raw_dev = torch.zeros((S,) + graphed.frame_shape, device='cuda', dtype=torch.uint8)
    with pytest.raises(ValueError):
        graphed.capture(raw_dev, net, download_to=torch.empty((S, OH, OW, 3), dtype=torch.uint8).pin_memory())
    firsts = frames_for(rs, src_fmt, S, H, W)
    for s in range(S):
        eager.join(s, firsts[s]); graphed.join(s, firsts[s])
    graph = graphed.capture(raw_dev, net, upload_from=host_in, download_to=host_out)
    for k in range(10):
        if k == 5:
            assert rect_or_none(lambda: eager.leave(1)) == rect_or_none(lambda: graphed.leave(1))
            first = frames_for(rs, src_fmt, 1, H, W)[0]
            eager.join(1, first); graphed.join(1, first)
        raw = frames_for(rs, src_fmt, S, H, W).cpu()
        host_in.copy_(raw)
        graph.replay()
        torch.cuda.synchronize()
        assert torch.equal(host_out.cuda(), eager.step(raw.cuda(), net)), k
    for a, b in ((eager.frames, graphed.frames), (eager.masks, graphed.masks), (eager.heads_dev, graphed.heads_dev),
                 (eager.all_black, graphed.all_black), (eager.in_x, graphed.in_x)):
        assert torch.equal(a, b)


def test_mixed_stream_batch_i420(mgw):
    """two source sizes in one MixedStreamBatch: the I420 output is the conversion of the BGR batch's, at the network's size"""
    S, cap, h, w = 2, (120, 200), 48, 80
    net, _ = fake_net_batch(mgw, identity_mesh())
    rs = np.random.RandomState(77)
    ref = mgw.MixedStreamBatch(S, cap, height=h, width=w, refine=2)
    mb = mgw.MixedStreamBatch(S, cap, height=h, width=w, refine=2, out_format='i420')
    assert mb.colour.shape == (S, h * 3 // 2, w)
    pools = [torch.zeros(b.pool_shape, device='cuda', dtype=torch.uint8) for b in (ref, mb)]
    sizes = {0: (120, 200), 1: (72, 128)}
    for s, sz in sizes.items():
        first = frames_for(rs, 'bgr', 1, *sz)[0]
        ref.join(s, first); mb.join(s, first)
    for k in range(8):
        for s, sz in sizes.items():
            f = frames_for(rs, 'bgr', 1, *sz)[0]
            for b, pool in zip((ref, mb), pools):
                b.slot_frame(pool, s).copy_(f)
        bgr = ref.step(pools[0], net)
        assert np.array_equal(mb.step(pools[1], net).cpu().numpy(), yuv_batch(bgr, 'i420')), k
    for s in range(S):
        assert rect_or_none(lambda: ref.leave(s)) == rect_or_none(lambda: mb.leave(s))


def test_errors(mgw):
    S, H, W, h, w = 2, 60, 80, 24, 40
    src = torch.zeros((S, H, W, 3), device='cuda', dtype=torch.uint8)
    xy = torch.zeros((S, h, w, 2), device='cuda')
    with pytest.raises(ValueError):
        mgw.ops.remap_bundle_frame(src, 'bgr', xy, out_format='yuv')
    with pytest.raises(ValueError):
        mgw.ops.remap_bundle_frame(src[:, :59].contiguous(), 'bgr', xy, out_format='nv12')
    with pytest.raises(ValueError):                       # a BGR-shaped out for a 4:2:0 result
        mgw.ops.remap_bundle_frame(src, 'bgr', xy, out=torch.empty_like(src), out_format='i420')

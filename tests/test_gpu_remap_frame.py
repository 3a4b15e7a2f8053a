"""GPU: warpRevBundle2 at any output size (mgw_remap_bundle_frame, deploy.warpRevBundle2 on frames of any size, StreamBatch's
out_size).  Every comparison is bit-exact: against OpenCV's bytes in tests/golden/deploy_remap_frame.npz, the numpy restatement
oracle/remap_frame_ref.py, and the network-size call mgw_remap_bundle_u8 where the sizes meet."""
import numpy as np
import pytest
import torch

import remap_frame_ref as M
import yuv420_ref
from conftest import load_golden
from test_gpu_streams import fake_net_batch, identity_mesh, rect_or_none, slot_history

pytestmark = pytest.mark.gpu

FORMATS = ('nv12', 'i420')


@pytest.fixture(scope='module')
def mgw():
    import dovs_b200
    assert torch.cuda.is_available(), 'GPU tests need a CUDA device; there is no CPU fallback'
    return dovs_b200


def cuda(a):
    return torch.as_tensor(np.ascontiguousarray(a)).cuda()


def xy_of(xm, ym):
    return torch.stack([cuda(xm), cuda(ym)], -1)


def yuv_frames(rs, S, H, W):
    return cuda(np.stack([yuv420_ref.random_frame(rs, H, W) for _ in range(S)]))


def to_bgr(yuv, fmt):
    return cuda(np.stack([yuv420_ref.yuv420_to_bgr(f, fmt) for f in yuv.cpu().numpy()]))


def fixture_cases():
    for tag, _, _, _, outs in M.CASES:
        for out in outs:
            yield tag, out


def test_every_fixture_case(mgw):
    """slot 2 of a batch of 5 (and a batch of 1) holds the fixture's frame resized to the output size, as the reference resizes
    it; its result is OpenCV's"""
    g = load_golden('deploy_remap_frame')
    rs = np.random.RandomState(60)
    for tag, (OH, OW) in fixture_cases():
        frame = cuda(g[tag + '_frame'])
        want = g['%s_%dx%d_dst' % (tag, OH, OW)]
        src = frame if tuple(frame.shape[:2]) == (OH, OW) else mgw.deploy.cv2_resize(frame, (OW, OH))
        xm, ym = M.fixture_maps(g, tag)
        for S in (1, 5):
            batch = cuda(rs.randint(0, 256, (S, OH, OW, 3)).astype(np.uint8))
            xy = cuda(rs.uniform(-1.2, 1.2, (S,) + xm.shape + (2,)).astype(np.float32))
            k = min(2, S - 1)
            batch[k] = src
            xy[k] = xy_of(xm, ym)
            got = mgw.ops.remap_bundle_frame(batch, 'bgr', xy)
            assert got.shape == (S, OH, OW, 3)
            assert np.array_equal(got[k].cpu().numpy(), want), (tag, OH, OW, S)


def test_at_the_maps_size_it_is_remap_bundle_u8(mgw):
    rs = np.random.RandomState(61)
    for S, h, w in ((1, 288, 512), (5, 288, 512), (3, 36, 64), (2, 100, 196), (4, 9, 13)):
        img = cuda(rs.randint(0, 256, (S, h, w, 3)).astype(np.uint8))
        xy = cuda(rs.uniform(-1.3, 1.3, (S, h, w, 2)).astype(np.float32))
        assert torch.equal(mgw.ops.remap_bundle_frame(img, 'bgr', xy), mgw.ops.remap_bundle_u8(img, xy)), (S, h, w)


@pytest.mark.parametrize('fmt', FORMATS)
def test_yuv_equals_bgr_on_the_converted_frames(mgw, fmt):
    rs = np.random.RandomState(62)
    cases = [(1080, 1920, 288, 512)] + [(OH - OH % 2, OW - OW % 2, 36, 64) for _, (OH, OW) in fixture_cases()]
    for H, W, h, w in cases:
        for S in (1, 5):
            yuv = yuv_frames(rs, S, H, W)
            xm, ym = M.smooth_mesh(h, w, H + W + S)
            xy = xy_of(xm, ym)[None].repeat(S, 1, 1, 1).contiguous()
            xy[S - 1] = cuda(rs.uniform(-1.3, 1.3, (h, w, 2)).astype(np.float32))
            got = mgw.ops.remap_bundle_frame(yuv, fmt, xy)
            assert torch.equal(got, mgw.ops.remap_bundle_frame(to_bgr(yuv, fmt), 'bgr', xy)), (fmt, H, W, S)


def test_warp_rev_bundle2_on_a_1080p_frame(mgw):
    rs = np.random.RandomState(63)
    frame = rs.randint(0, 256, (1080, 1920, 3)).astype(np.uint8)
    xm, ym = M.smooth_mesh(288, 512, 64)
    got = mgw.deploy.warpRevBundle2(frame, xm, ym)
    assert isinstance(got, np.ndarray) and got.shape == (1080, 1920, 3)
    assert np.array_equal(got, M.warp_rev_bundle2_sized(frame, xm, ym, (1080, 1920)))
    # the network's [1,h,w,1] maps, a batch, and the YUV formats
    assert np.array_equal(mgw.deploy.warpRevBundle2(frame, xm[None, ..., None], ym[None, ..., None]), got)
    two = mgw.deploy.warpRevBundle2(cuda(np.stack([frame, frame])), cuda(np.stack([xm, xm])), cuda(np.stack([ym, ym])))
    assert torch.equal(two[1].cpu(), torch.as_tensor(got))
    for fmt in FORMATS:
        yuv = yuv420_ref.random_frame(rs, 1080, 1920)
        assert np.array_equal(mgw.deploy.warpRevBundle2(yuv, xm, ym, src_format=fmt),
                              M.warp_rev_bundle2_sized(yuv, xm, ym, (1080, 1920), src_format=fmt)), fmt
    # a frame at the maps' size is the network-size call
    small = rs.randint(0, 256, (288, 512, 3)).astype(np.uint8)
    import deploy_ref
    assert np.array_equal(mgw.deploy.warpRevBundle2(small, xm, ym), deploy_ref.warp_rev_bundle2(small, xm, ym))


# ---- StreamBatch(out_size=...)
def recording_net(mgw, base):
    net, _ = fake_net_batch(mgw, base)
    last = {}

    def rec(in_x):
        out, black, xy = net(in_x)
        last['xy'] = xy.clone()
        return out, black, xy
    return rec, last


def frames_for(rs, fmt, S, H, W):
    if fmt == 'bgr':
        return cuda(rs.randint(0, 256, (S, H, W, 3)).astype(np.uint8))
    return yuv_frames(rs, S, H, W)


@pytest.mark.parametrize('fmt,out', [('bgr', 'src'), ('nv12', 'src'), ('i420', 'src'), ('bgr', (720, 1280)), ('nv12', (720, 1280))])
def test_stream_batch_out_size(mgw, fmt, out):
    S, H, W, h, w, refine = 4, 360, 640, 72, 128, 2
    OH, OW = (H, W) if out == 'src' else out
    base = identity_mesh()
    sb = mgw.StreamBatch(S, (H, W), height=h, width=w, refine=refine, src_format=fmt, out_size=(OH, OW))
    ref = mgw.StreamBatch(S, (H, W), height=h, width=w, refine=refine, src_format=fmt)
    assert (sb.small is None) == (out == 'src') and sb.colour.shape == (S, OH, OW, 3)
    net, last = recording_net(mgw, base)
    rs = np.random.RandomState(65)
    joins, leaves = {0: [0, 1], 5: [2], 9: [1]}, {7: [1]}
    for k in range(12):
        for s in leaves.get(k, []):
            assert rect_or_none(lambda: sb.leave(s)) == rect_or_none(lambda: ref.leave(s)), (k, s)
        for s in joins.get(k, []):
            first = frames_for(rs, fmt, 1, H, W)[0]
            sb.join(s, first); ref.join(s, first)
        raw = frames_for(rs, fmt, S, H, W)
        got = sb.step(raw, net).clone()
        xy = last['xy']
        ref.step(raw, net)
        assert got.shape == (S, OH, OW, 3)
        for s in range(S):
            frame = raw[s] if out == 'src' else mgw.deploy.cv2_resize(raw[s], (OW, OH), src_format=fmt)
            want = mgw.deploy.warpRevBundle2(frame, xy[s, ..., 0], xy[s, ..., 1], src_format=fmt if out == 'src' else 'bgr')
            assert torch.equal(got[s], want), (k, s)
        assert torch.equal(sb.in_x, ref.in_x), k
    # one slot of the last step against the numpy restatement
    frame = raw[0].cpu().numpy()
    xs, ys = xy[0, ..., 0].cpu().numpy(), xy[0, ..., 1].cpu().numpy()
    assert np.array_equal(got[0].cpu().numpy(), M.warp_rev_bundle2_sized(frame, xs, ys, (OH, OW), src_format=fmt))
    for t, u in ((sb.frames, ref.frames), (sb.masks, ref.masks), (sb.heads_dev, ref.heads_dev), (sb.all_black, ref.all_black)):
        assert torch.equal(t, u)
    for s in range(S):
        fa, ma = slot_history(sb, s)
        fb, mb = slot_history(ref, s)
        assert torch.equal(fa, fb) and torch.equal(ma, mb), s
        assert rect_or_none(lambda: sb.leave(s)) == rect_or_none(lambda: ref.leave(s)), s


@pytest.mark.parametrize('fmt,out', [('nv12', 'src'), ('bgr', (720, 1280))])
def test_stream_batch_out_size_graph_replay_equals_eager(mgw, fmt, out):
    S, H, W, h, w = 3, 360, 640, 72, 128
    OH, OW = (H, W) if out == 'src' else out
    base = identity_mesh()
    eager = mgw.StreamBatch(S, (H, W), height=h, width=w, refine=2, src_format=fmt, out_size=(OH, OW))
    graphed = mgw.StreamBatch(S, (H, W), height=h, width=w, refine=2, src_format=fmt, out_size=(OH, OW))
    net, _ = fake_net_batch(mgw, base)
    rs = np.random.RandomState(66)
    shape = graphed.frame_shape
    host_in = torch.empty((S,) + shape, dtype=torch.uint8).pin_memory()
    host_out = torch.empty((S, OH, OW, 3), dtype=torch.uint8).pin_memory()
    raw_dev = torch.zeros((S,) + shape, device='cuda', dtype=torch.uint8)
    firsts = frames_for(rs, fmt, S, H, W)
    for s in range(S):
        eager.join(s, firsts[s]); graphed.join(s, firsts[s])
    graph = graphed.capture(raw_dev, net, upload_from=host_in, download_to=host_out)
    for k in range(12):
        if k == 4:
            assert rect_or_none(lambda: eager.leave(2)) == rect_or_none(lambda: graphed.leave(2))
        if k in (4, 8):
            first = frames_for(rs, fmt, 1, H, W)[0]
            eager.join(k // 4 - 1, first); graphed.join(k // 4 - 1, first)
        raw = frames_for(rs, fmt, S, H, W).cpu()
        host_in.copy_(raw)
        graph.replay()
        torch.cuda.synchronize()
        want = eager.step(raw.cuda(), net)
        assert torch.equal(host_out.cuda(), want), k
    for t, u in ((eager.frames, graphed.frames), (eager.masks, graphed.masks), (eager.heads_dev, graphed.heads_dev),
                 (eager.all_black, graphed.all_black), (eager.in_x, graphed.in_x)):
        assert torch.equal(t, u)


def test_errors(mgw):
    S, H, W, h, w = 2, 60, 80, 24, 40
    for bad in ((0, 80), (60, 0), (32768, 80), (60, 32768), (-1, 5)):
        with pytest.raises(ValueError):
            mgw.StreamBatch(S, (H, W), height=h, width=w, out_size=bad)
    sb = mgw.StreamBatch(S, (H, W), height=h, width=w, out_size=(H, W))
    net, _ = fake_net_batch(mgw, identity_mesh())
    raw = torch.zeros((S, H, W, 3), device='cuda', dtype=torch.uint8)
    with pytest.raises(ValueError):
        sb.capture(raw, net, download_to=torch.empty((S, h, w, 3), dtype=torch.uint8).pin_memory())
    with pytest.raises(ValueError):
        mgw.deploy.warpRevBundle2(np.zeros((H, W, 3), np.uint8), np.zeros((7, 9), np.float32), np.zeros((7, 10), np.float32))
    with pytest.raises(ValueError):
        mgw.ops.remap_bundle_frame(raw, 'yuv', torch.zeros((S, h, w, 2), device='cuda'))

"""GPU: YUV 4:2:0 input (NV12 / I420) through cvt_img2train, cv2_resize and StreamBatch.  Every comparison is bit-exact: a YUV
call must give what the BGR call gives on the frame cv2.cvtColor(COLOR_YUV2BGR_NV12 / _I420) makes of it (the numpy restatement
oracle/yuv420_ref.py, pinned against OpenCV by tests/golden/deploy_yuv420.npz)."""
import numpy as np
import pytest
import torch

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


def yuv_frames(rs, S, H, W):
    return torch.as_tensor(np.stack([yuv420_ref.random_frame(rs, H, W) for _ in range(S)])).cuda()


def to_bgr(yuv, fmt):
    """[S,3H/2,W] -> [S,H,W,3] by the restatement (cv2.cvtColor), on the device"""
    return torch.as_tensor(np.stack([yuv420_ref.yuv420_to_bgr(f, fmt) for f in yuv.cpu().numpy()])).cuda()


def cvt_cases():
    """(H, W, h, w, crop_rate): the fixture sizes, 1080p, and the output / crop-rate configurations of the BGR fixture (its
    source sizes rounded down to even)"""
    cases = [(H, W, 36, 64, 1) for H, W in yuv420_ref.SIZES] + [(1080, 1920, 288, 512, 1), (1080, 1920, 288, 512, 0.9)]
    g = load_golden('deploy_cvt_img2train')
    for n in sorted(k[:-4] for k in g if k.endswith('_out')):
        h, w, cr = g[n + '_cfg']
        H, W = g[n + '_img'].shape[:2]
        cases.append((H - H % 2, W - W % 2, int(h), int(w), 1 if cr == 1 else float(cr)))
    return cases


@pytest.mark.parametrize('fmt', FORMATS)
def test_fused_cvt_img2train_equals_bgr_call(mgw, fmt):
    rs = np.random.RandomState(40)
    for H, W, h, w, cr in cvt_cases():
        for S in (1, 5):
            yuv = yuv_frames(rs, S, H, W)
            bgr = to_bgr(yuv, fmt)
            got = mgw.deploy.cvt_img2train(yuv, cr, height=h, width=w, src_format=fmt)
            assert got.shape == (S, h, w, 1)
            assert torch.equal(got, mgw.deploy.cvt_img2train(bgr, cr, height=h, width=w)), (fmt, H, W, h, w, cr, S)
        one = mgw.deploy.cvt_img2train(yuv[2], cr, height=h, width=w, src_format=fmt)        # a single frame [3H/2,W]
        assert torch.equal(one, mgw.deploy.cvt_img2train(bgr[2], cr, height=h, width=w)), (fmt, H, W)
    # numpy in, the reference's float64 out
    yuv = yuv420_ref.random_frame(rs, 90, 158)
    got = mgw.deploy.cvt_img2train(yuv, 1, height=36, width=64, as_numpy=True, src_format=fmt)
    assert np.array_equal(got, mgw.deploy.cvt_img2train(yuv420_ref.yuv420_to_bgr(yuv, fmt), 1, height=36, width=64, as_numpy=True))


def resize_cases():
    """(H, W, h, w): the 2x2 shortcut (72x128 -> 36x64, 576x1024 -> 288x512), down- and up-scaling, W not a multiple of 4, 1080p"""
    return [(72, 128, 36, 64), (576, 1024, 288, 512), (1080, 1920, 288, 512), (90, 158, 36, 64), (36, 64, 37, 41), (6, 10, 36, 64),
            (2, 2, 3, 5), (720, 1278, 288, 512)]


@pytest.mark.parametrize('fmt', FORMATS)
def test_fused_cv2_resize_equals_bgr_call(mgw, fmt):
    rs = np.random.RandomState(41)
    for H, W, h, w in resize_cases():
        for S in (1, 5):
            yuv = yuv_frames(rs, S, H, W)
            bgr = to_bgr(yuv, fmt)
            got = mgw.deploy.cv2_resize(yuv, (w, h), src_format=fmt)
            assert got.shape == (S, h, w, 3)
            assert torch.equal(got, mgw.deploy.cv2_resize(bgr, (w, h))), (fmt, H, W, h, w, S)
        assert torch.equal(mgw.deploy.cv2_resize(yuv[1], (w, h), src_format=fmt), mgw.deploy.cv2_resize(bgr[1], (w, h)))
    yuv = yuv420_ref.random_frame(rs, 36, 64)                                                  # numpy in -> numpy out
    assert np.array_equal(mgw.deploy.cv2_resize(yuv, (40, 20), src_format=fmt),
                          mgw.deploy.cv2_resize(yuv420_ref.yuv420_to_bgr(yuv, fmt), (40, 20)))


def test_batch_slot_against_the_fixture(mgw):
    """slot 3 of a batch of 5 holds a fixture frame: its results are the BGR calls' on the BGR frame OpenCV made of it, and its
    resize is OpenCV's own where the fixture stores one"""
    g = load_golden('deploy_yuv420')
    rs = np.random.RandomState(42)
    for n in sorted(k[:-4] for k in g if k.endswith('_yuv')):
        fmt = n.split('_')[0]
        yuv_np, bgr_np = g[n + '_yuv'], g[n + '_bgr']
        H, W = bgr_np.shape[:2]
        batch = yuv_frames(rs, 5, H, W)
        batch[3] = torch.as_tensor(yuv_np).cuda()
        bgr = torch.as_tensor(bgr_np).cuda()
        got = mgw.deploy.cvt_img2train(batch, 0.9, height=24, width=40, src_format=fmt)
        assert torch.equal(got[3:4], mgw.deploy.cvt_img2train(bgr, 0.9, height=24, width=40)), n
        got = mgw.deploy.cv2_resize(batch, (64, 36), src_format=fmt)
        assert torch.equal(got[3], mgw.deploy.cv2_resize(bgr, (64, 36))), n
        if n + '_resized' in g:
            assert np.array_equal(got[3].cpu().numpy(), g[n + '_resized']), n


def test_1080p_against_the_restatement(mgw):
    """seeded 1080p frames: the fused calls against the numpy restatement followed by the BGR oracle (deploy_ref)"""
    import deploy_ref
    rs = np.random.RandomState(43)
    for fmt in FORMATS:
        yuv = yuv420_ref.random_frame(rs, 1080, 1920)
        bgr = yuv420_ref.yuv420_to_bgr(yuv, fmt)
        got = mgw.deploy.cv2_resize(torch.as_tensor(yuv).cuda(), (512, 288), src_format=fmt)
        assert np.array_equal(got.cpu().numpy(), deploy_ref.resize_linear_u8(bgr, 512, 288)), fmt
        got = mgw.deploy.cvt_img2train(torch.as_tensor(yuv).cuda(), src_format=fmt, as_numpy=True)
        assert np.array_equal(got, deploy_ref.cvt_img2train(bgr, 288, 512)), fmt


# ---- StreamBatch: a YUV batch against a BGR batch fed the converted frames
@pytest.mark.parametrize('fmt', FORMATS)
def test_stream_batch_yuv_equals_bgr_batch(mgw, fmt):
    S, H, W, h, w, refine, cr = 4, 180, 320, 72, 128, 2, 0.9
    base = identity_mesh()
    yb = mgw.StreamBatch(S, (H, W), height=h, width=w, crop_rate=cr, refine=refine, src_format=fmt)
    bb = mgw.StreamBatch(S, (H, W), height=h, width=w, crop_rate=cr, refine=refine)
    net, _ = fake_net_batch(mgw, base)
    rs = np.random.RandomState(44)
    # slot 0: steps 0-11; slot 1: steps 0-6, then a second video from step 9; slot 2: from step 5; slot 3: never joined
    joins, leaves = {0: [0, 1], 5: [2], 9: [1]}, {7: [1]}
    for k in range(12):
        for s in leaves.get(k, []):
            assert rect_or_none(lambda: yb.leave(s)) == rect_or_none(lambda: bb.leave(s)), (k, s)
        for s in joins.get(k, []):
            first = yuv_frames(rs, 1, H, W)
            yb.join(s, first[0])
            bb.join(s, to_bgr(first, fmt)[0])
        raw = yuv_frames(rs, S, H, W)
        got = yb.step(raw, net).clone()
        want = bb.step(to_bgr(raw, fmt), net)
        assert torch.equal(got, want), k
        assert torch.equal(yb.in_x, bb.in_x), k
    for t, u in ((yb.frames, bb.frames), (yb.masks, bb.masks), (yb.heads_dev, bb.heads_dev), (yb.all_black, bb.all_black)):
        assert torch.equal(t, u)
    for s in range(S):
        fy, my = slot_history(yb, s)
        fb, mb = slot_history(bb, s)
        assert torch.equal(fy, fb) and torch.equal(my, mb), s
        assert rect_or_none(lambda: yb.leave(s)) == rect_or_none(lambda: bb.leave(s)), s
    assert int(yb.all_black.sum()) > 0


def test_stream_batch_yuv_graph_replay_equals_eager(mgw):
    """an NV12 step captured once with the upload of the [S,3H/2,W] pinned buffer and the download inside the graph, replayed for
    12 steps with joins and a leave between replays == the same schedule run eagerly"""
    S, H, W, h, w, fmt = 3, 120, 200, 48, 80, 'nv12'
    base = identity_mesh()
    eager = mgw.StreamBatch(S, (H, W), height=h, width=w, refine=2, src_format=fmt)
    graphed = mgw.StreamBatch(S, (H, W), height=h, width=w, refine=2, src_format=fmt)
    net, _ = fake_net_batch(mgw, base)
    rs = np.random.RandomState(45)
    host_in = torch.empty((S, H * 3 // 2, W), dtype=torch.uint8).pin_memory()
    host_out = torch.empty((S, h, w, 3), dtype=torch.uint8).pin_memory()
    raw_dev = torch.zeros((S, H * 3 // 2, W), device='cuda', dtype=torch.uint8)
    firsts = yuv_frames(rs, S, H, W)
    for s in range(S):
        eager.join(s, firsts[s]); graphed.join(s, firsts[s])
    graph = graphed.capture(raw_dev, net, upload_from=host_in, download_to=host_out)
    for t, u in ((eager.frames, graphed.frames), (eager.masks, graphed.masks), (eager.heads_dev, graphed.heads_dev),
                 (eager.all_black, graphed.all_black)):
        assert torch.equal(t, u)                                         # capturing changed nothing
    for k in range(12):
        if k == 4:
            assert rect_or_none(lambda: eager.leave(2)) == rect_or_none(lambda: graphed.leave(2))
        if k in (4, 8):
            first = yuv_frames(rs, 1, H, W)[0]
            eager.join(k // 4 - 1, first); graphed.join(k // 4 - 1, first)
        raw = np.stack([yuv420_ref.random_frame(rs, H, W) for _ in range(S)])
        host_in.copy_(torch.as_tensor(raw))
        graph.replay()
        torch.cuda.synchronize()
        want = eager.step(torch.as_tensor(raw).cuda(), net)
        assert torch.equal(host_out.cuda(), want), k
    for t, u in ((eager.frames, graphed.frames), (eager.masks, graphed.masks), (eager.heads_dev, graphed.heads_dev),
                 (eager.all_black, graphed.all_black), (eager.in_x, graphed.in_x)):
        assert torch.equal(t, u)
    for s in range(S):
        assert rect_or_none(lambda: eager.leave(s)) == rect_or_none(lambda: graphed.leave(s))


def test_yuv_errors(mgw):
    S, H, W, h, w = 2, 60, 80, 24, 40
    u8 = dict(device='cuda', dtype=torch.uint8)
    d = mgw.deploy
    for fn in (lambda x, f='nv12': d.cvt_img2train(x, height=h, width=w, src_format=f),
               lambda x, f='nv12': d.cv2_resize(x, (w, h), src_format=f)):
        for bad in (torch.zeros((91, W), **u8),                       # rows not a multiple of 3
                    torch.zeros((90, W + 1), **u8),                   # odd W
                    torch.zeros((90, W), device='cuda'),              # dtype
                    torch.zeros((S, H, W, 3), **u8)):                 # a BGR batch
            with pytest.raises(ValueError):
                fn(bad)
        with pytest.raises(ValueError):
            fn(torch.zeros((90, W), **u8), 'yuv')
    with pytest.raises(ValueError):
        mgw.ops.cvt_img2train_yuv420_batch(torch.zeros((S, 90, W), **u8), 'nv21', d._cvt_tables(H, W, h, w, 1, torch.device('cuda')), h, w)
    with pytest.raises(ValueError):
        mgw.ops.resize_linear_yuv420_batch(torch.zeros((S, 91, W), **u8), 'nv12', None, None, 30, 40)
    sb = mgw.StreamBatch(S, (H, W), height=h, width=w, src_format='i420')
    net, _ = fake_net_batch(mgw, identity_mesh())
    with pytest.raises(ValueError):
        sb.step(torch.zeros((S, H, W, 3), **u8), net)                  # a BGR batch into a YUV StreamBatch
    with pytest.raises(ValueError):
        sb.step(torch.zeros((S + 1, 90, W), **u8), net)
    with pytest.raises(ValueError):
        sb.join(0, torch.zeros((H, W, 3), **u8))
    sb.join(0, torch.zeros((h, w), device='cuda'))                        # a network frame is still accepted
    with pytest.raises(ValueError):
        mgw.StreamBatch(S, (H + 1, W), height=h, width=w, src_format='nv12')
    # an empty batch launches nothing
    n0 = mgw.launch_count()
    tabs = d._cvt_tables(H, W, h, w, 1, torch.device('cuda'))
    assert mgw.ops.cvt_img2train_yuv420_batch(torch.zeros((0, 90, W), **u8), 'nv12', tabs, h, w).shape == (0, h, w)
    assert mgw.ops.resize_linear_yuv420_batch(torch.zeros((0, 90, W), **u8), 'i420', None, None, 30, 40).shape == (0, 30, 40, 3)
    assert mgw.launch_count() == n0

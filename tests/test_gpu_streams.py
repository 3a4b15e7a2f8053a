"""GPU: several videos at once (deploy.StreamBatch and the batched deploy kernels).  Every comparison is bit-exact: a batched
frame or stream must equal the single-frame / single-stream call on the same data, and a stream of a batch must reproduce the
reference's own per-frame list handling (fixture)."""
import numpy as np
import pytest
import torch

from conftest import load_golden

pytestmark = pytest.mark.gpu


@pytest.fixture(scope='module')
def mgw():
    import dovs_b200
    assert torch.cuda.is_available(), 'GPU tests need a CUDA device; there is no CPU fallback'
    return dovs_b200


def frames(rs, shape):
    return torch.as_tensor(rs.randint(0, 256, shape).astype(np.uint8)).cuda()


# ---- batched front end: cvt_img2train and cv2_resize over [S,H,W,C]
def test_batched_cvt_img2train_equals_per_frame_calls(mgw):
    g = load_golden('deploy_cvt_img2train')
    cases = [((1080, 1920), 288, 512, 1)]
    for n in sorted(k[:-4] for k in g if k.endswith('_out')):
        h, w, cr = g[n + '_cfg']
        cases.append((g[n + '_img'].shape[:2], int(h), int(w), 1 if cr == 1 else float(cr)))
    rs = np.random.RandomState(20)
    for (H, W), h, w, cr in cases:
        for S in (1, 5):
            bgr = frames(rs, (S, H, W, 3))
            got = mgw.deploy.cvt_img2train(bgr, cr, height=h, width=w)
            assert got.shape == (S, h, w, 1)
            for s in range(S):
                assert torch.equal(got[s:s + 1], mgw.deploy.cvt_img2train(bgr[s], cr, height=h, width=w)), (H, W, h, w, cr, S, s)
    # one slot of a batch against the fixtures made by OpenCV + Pillow
    for n in sorted(k[:-4] for k in g if k.endswith('_out')):
        h, w, cr = g[n + '_cfg']
        img = torch.as_tensor(g[n + '_img']).cuda()
        bgr = frames(rs, (5,) + tuple(img.shape))
        bgr[3] = img
        got = mgw.deploy.cvt_img2train(bgr, 1 if cr == 1 else float(cr), height=int(h), width=int(w))
        assert np.array_equal(got[3:4].cpu().numpy(), g[n + '_out'].astype(np.float32)), n


def test_batched_cv2_resize_equals_per_frame_calls(mgw):
    g = load_golden('deploy_cv2_resize')
    sizes = [((1080, 1920), (288, 512))]
    sizes += [(g[n + '_img'].shape[:2], g[n + '_dst'].shape[:2]) for n in sorted(k[:-4] for k in g if k.endswith('_dst'))]
    rs = np.random.RandomState(21)
    for (H, W), (h, w) in sizes:
        for C in (1, 3, 4):
            for S in (1, 5):
                img = frames(rs, (S, H, W, C))
                got = mgw.deploy.cv2_resize(img, (w, h))
                assert got.shape == (S, h, w, C)
                for s in range(S):
                    assert torch.equal(got[s], mgw.deploy.cv2_resize(img[s], (w, h))), (H, W, h, w, C, S, s)
    for n in sorted(k[:-4] for k in g if k.endswith('_dst')):
        want, img = g[n + '_dst'], g[n + '_img']
        img = torch.as_tensor(img if img.ndim == 3 else img[..., None]).cuda()
        batch = frames(rs, (5,) + tuple(img.shape))
        batch[1] = img
        got = mgw.deploy.cv2_resize(batch, (want.shape[1], want.shape[0]))
        assert np.array_equal(got[1].cpu().numpy().reshape(want.shape), want), n


# ---- StreamBatch against independent single-stream pipelines
def identity_mesh(gh=4, gw=4):
    ys, xs = torch.meshgrid(torch.linspace(-1, 1, gh + 1), torch.linspace(-1, 1, gw + 1), indexing='ij')
    return torch.stack([xs, ys], -1)[None].cuda()


def fake_net_one(mgw, x, base):
    """deterministic stand-in for the network + multi-grid warp of ONE stream (x [1,h,w,nch], device only, no host sync):
    the frame to warp mixes the current frame and a history tap, the mesh is moved by pixels of the input"""
    h, w = x.shape[1:3]
    img = (0.7 * x[..., -1:] + 0.3 * x[..., 6:7]).contiguous()
    d = x[0, :h // 2:h // 10, :w // 2:w // 10, -1][:5, :5]
    theta = (base + 0.06 * torch.stack([d, -d], -1)[None]).contiguous()
    out, black, xy, _ = mgw.ops.mesh_warp_fwd(img, theta)
    return out, black, xy


def fake_net_batch(mgw, base, record=None):
    """the same stand-in applied slot by slot to a batched input; record: list that receives a copy of the first input
    of every step (the assembled in_x, before the refine passes overwrite its last channel)"""
    state = {'first': True}

    def net(in_x):
        if record is not None and state['first']:
            record.append(in_x.clone())
        state['first'] = False
        outs = [fake_net_one(mgw, in_x[s:s + 1], base) for s in range(in_x.shape[0])]
        return tuple(torch.cat(t, 0) for t in zip(*outs))

    def new_step():
        state['first'] = True
    return net, new_step


class OnePipeline:
    """one video the single-stream way: StreamState + CropState + cv2_resize + warpRevBundle2"""

    def __init__(self, mgw, first_bgr, h, w, crop_rate, refine, base):
        self.mgw, self.h, self.w, self.cr, self.refine, self.base = mgw, h, w, crop_rate, refine, base
        cur = mgw.deploy.cvt_img2train(first_bgr, crop_rate, height=h, width=w)
        self.st, self.crop = mgw.StreamState(cur.reshape(h, w)), mgw.CropState(h, w)

    def step(self, raw):
        mgw, h, w = self.mgw, self.h, self.w
        cur = mgw.deploy.cvt_img2train(raw, self.cr, height=h, width=w)
        in_x = self.st.assemble(cur.reshape(h, w))
        assembled = in_x.clone()
        for _ in range(self.refine):
            out, black, xy = fake_net_one(mgw, in_x, self.base)
            self.crop.add(black)
            self.st.refeed(in_x, out, black)
        self.st.push(out, black)
        small = mgw.deploy.cv2_resize(raw, (w, h))
        colour = mgw.deploy.warpRevBundle2(small, xy[0, ..., 0], xy[0, ..., 1])
        return assembled, in_x, colour


def rect_or_none(fn):
    try:
        return fn()
    except IndexError:
        return None


def slot_history(sb, s):
    head = int(sb.heads_dev[s].item())
    order = [(head + 1 + k) % sb.depth for k in range(sb.depth)]
    return sb.frames[s][order], sb.masks[s][order]


def test_stream_batch_equals_independent_pipelines(mgw):
    S, H, W, h, w, refine, cr = 4, 180, 320, 72, 128, 2, 0.9
    base = identity_mesh()
    sb = mgw.StreamBatch(S, (H, W), height=h, width=w, crop_rate=cr, refine=refine)
    rec = []
    net, new_step = fake_net_batch(mgw, base, rec)
    rs = np.random.RandomState(30)
    # slot 0: steps 0-11; slot 1: steps 0-6, then a second video from step 9; slot 2: from step 5; slot 3: never joined
    joins, leaves = {0: [0, 1], 5: [2], 9: [1]}, {7: [1]}
    pipes, steps_run = {}, 0
    for k in range(12):
        raw = frames(rs, (S, H, W, 3))
        for s in leaves.get(k, []):
            p = pipes.pop(s)
            assert rect_or_none(lambda: sb.leave(s)) == rect_or_none(p.crop.rect), (k, s)
            fr, mk = slot_history(sb, s)
            f0, m0 = p.st.history()
            assert torch.equal(fr, f0) and torch.equal(mk, m0) and torch.equal(sb.all_black[s], p.crop.all_black), (k, s)
        for s in joins.get(k, []):
            first = frames(rs, (H, W, 3))
            sb.join(s, first)
            pipes[s] = OnePipeline(mgw, first, h, w, cr, refine, base)
        new_step()
        colour = sb.step(raw, net).clone()
        steps_run += 1
        for s, p in pipes.items():
            assembled, refined, want = p.step(raw[s])
            assert torch.equal(rec[-1][s:s + 1], assembled), (k, s)
            assert torch.equal(sb.in_x[s:s + 1], refined), (k, s)
            assert torch.equal(colour[s], want), (k, s)
    assert len(rec) == steps_run
    for s, p in pipes.items():
        fr, mk = slot_history(sb, s)
        f0, m0 = p.st.history()
        assert torch.equal(fr, f0) and torch.equal(mk, m0), s
        assert torch.equal(sb.all_black[s], p.crop.all_black), s
        assert int(sb.all_black[s].sum()) > 0, s
        assert rect_or_none(lambda: sb.leave(s)) == rect_or_none(p.crop.rect), s


def test_stream_batch_slot_reproduces_the_reference(mgw):
    """slot 1 of a batch fed the stream fixture's frames == the reference's own list handling (as test_deploy_stream_state_exact
    and test_deploy_crop_exact check for one stream)"""
    import deploy_ref
    g = load_golden('deploy_stream')
    h, w = g['first'].shape
    S, slot = 3, 1
    sb = mgw.StreamBatch(S, (h, w), height=h, width=w, refine=int(g['refine']))
    rs = np.random.RandomState(31)
    for s in range(S):
        sb.join(s, torch.as_tensor(g['first']).cuda() if s == slot else frames(rs, (h, w, 3)))
    rec, k_now = [], {'k': 0, 'first': True}

    def net(in_x):
        if k_now['first']:
            rec.append(in_x.clone())
            k_now['first'] = False
        x = in_x.cpu().numpy()
        img, black = [], []
        for s in range(S):
            if s == slot:
                i, b = deploy_ref.stream_fake_net(x[s:s + 1], k_now['k'])
            else:
                i, b = 0.5 * x[s:s + 1, ..., -1:], (x[s:s + 1, ..., 0] > 0.25).astype(np.float32)
            img.append(i.reshape(1, h, w, 1)); black.append(b.reshape(1, h, w))
        return (torch.as_tensor(np.concatenate(img)).cuda(), torch.as_tensor(np.concatenate(black)).cuda(),
                torch.zeros((S, h, w, 2), device='cuda'))

    for k in range(g['cur_frames'].shape[0]):
        k_now['k'], k_now['first'] = k, True
        cur = torch.as_tensor(rs.random_sample((S, h, w)).astype(np.float32) - 0.5).cuda()
        cur[slot] = torch.as_tensor(g['cur_frames'][k]).cuda()
        sb.advance(cur, net)
        assert np.array_equal(rec[-1][slot:slot + 1].cpu().numpy(), g['in_x'][k]), k
        assert np.array_equal(sb.in_x[slot:slot + 1].cpu().numpy(), g['tmp_in_x'][k]), k
    fr, mk = slot_history(sb, slot)
    assert np.array_equal(fr.cpu().numpy()[..., None], g['final_frames']) and np.array_equal(mk.cpu().numpy()[..., None], g['final_masks'])
    assert np.array_equal(sb.all_black[slot].cpu().numpy().astype(np.int64), g['all_black'])


def test_stream_batch_graph_replay_equals_eager(mgw):
    """one step captured once (with the upload and the download inside the graph), replayed for 12 steps with joins and a
    leave between replays == the same schedule run eagerly on a second batch"""
    S, H, W, h, w = 3, 120, 200, 48, 80
    base = identity_mesh()
    eager = mgw.StreamBatch(S, (H, W), height=h, width=w, refine=2)
    graphed = mgw.StreamBatch(S, (H, W), height=h, width=w, refine=2)
    net, _ = fake_net_batch(mgw, base)
    rs = np.random.RandomState(32)
    host_in = torch.empty((S, H, W, 3), dtype=torch.uint8).pin_memory()
    host_out = torch.empty((S, h, w, 3), dtype=torch.uint8).pin_memory()
    raw_dev = torch.zeros((S, H, W, 3), device='cuda', dtype=torch.uint8)
    for s in range(S):
        first = frames(rs, (H, W, 3))
        eager.join(s, first); graphed.join(s, first)
    graph = graphed.capture(raw_dev, net, upload_from=host_in, download_to=host_out)
    for t, u in ((eager.frames, graphed.frames), (eager.masks, graphed.masks), (eager.heads_dev, graphed.heads_dev),
                 (eager.all_black, graphed.all_black)):
        assert torch.equal(t, u)                                         # capturing changed nothing
    for k in range(12):
        if k == 4:
            assert rect_or_none(lambda: eager.leave(2)) == rect_or_none(lambda: graphed.leave(2))
        if k in (4, 8):
            first = frames(rs, (H, W, 3))
            eager.join(k // 4 - 1, first); graphed.join(k // 4 - 1, first)
        raw = rs.randint(0, 256, (S, H, W, 3)).astype(np.uint8)
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


def test_stream_batch_errors(mgw):
    from dovs_b200._lib import check, lib
    S, H, W, h, w = 2, 60, 80, 24, 40
    sb = mgw.StreamBatch(S, (H, W), height=h, width=w)
    net, _ = fake_net_batch(mgw, identity_mesh())
    with pytest.raises(ValueError):
        sb.step(torch.zeros((S + 1, H, W, 3), device='cuda', dtype=torch.uint8), net)      # batch size
    with pytest.raises(ValueError):
        sb.step(torch.zeros((S, H, W + 1, 3), device='cuda', dtype=torch.uint8), net)      # source size
    with pytest.raises(ValueError):
        sb.join(0, torch.zeros((H, W, 4), device='cuda', dtype=torch.uint8))
    with pytest.raises(ValueError):
        sb.advance(torch.zeros((S, h, w), device='cuda'), lambda x: (torch.zeros((S, h, w, 1), device='cuda'),
                                                                      torch.zeros((S, h, w), device='cuda'),
                                                                      torch.zeros((S, h, w + 1, 2), device='cuda')))
    for bad in (-1, S, 1.0):
        with pytest.raises(ValueError):
            sb.join(bad, torch.zeros((H, W, 3), device='cuda', dtype=torch.uint8))
        with pytest.raises(ValueError):
            sb.leave(bad)
    with pytest.raises(ValueError):
        mgw.StreamBatch(S, (H, W), height=h, width=w, taps=(1, 2, 33))
    with pytest.raises(ValueError):
        mgw.ops.streams_assemble(sb.frames, sb.masks, sb.heads_dev, sb.taps, torch.zeros((S, h + 1, w), device='cuda'))
    with pytest.raises(ValueError):
        mgw.ops.streams_push(sb.frames, sb.masks, sb.heads_dev[:1], sb.cur, sb.cur)
    with pytest.raises(mgw.MgwError, match='tap 33'):
        mgw.ops.streams_assemble(sb.frames, sb.masks, sb.heads_dev, (1, 33), sb.cur)
    # S x frame size past the 32-bit index limits: refused before anything is launched
    kx, x0, xn, ky, y0, yn = mgw.deploy._cvt_tables(1080, 1920, 288, 512, 1, torch.device('cuda'))
    p = sb.frames.data_ptr()
    with pytest.raises(mgw.MgwError, match='bad sizes'):
        check(lib.mgw_cvt_img2train_u8_batch(p, 300, 1080, 1920, kx.data_ptr(), x0.data_ptr(), xn.data_ptr(), kx.shape[1], ky.data_ptr(),
                                             y0.data_ptr(), yn.data_ptr(), ky.shape[1], 288, 512, p, p, None), 'cvt')
    with pytest.raises(mgw.MgwError, match='bad sizes'):
        check(lib.mgw_streams_push(p, p, 500, 32, sb.heads_dev.data_ptr(), p, p, 288, 512, None), 'push')
    # an empty batch launches nothing
    n0 = mgw.launch_count()
    e = mgw.ops.cvt_img2train_u8_batch(torch.zeros((0, 1080, 1920, 3), device='cuda', dtype=torch.uint8), (kx, x0, xn, ky, y0, yn), 288, 512)
    assert e.shape == (0, 288, 512)
    assert mgw.ops.resize_linear_u8_batch(torch.zeros((0, 96, 128, 3), device='cuda', dtype=torch.uint8), None, None, 48, 64).shape == (0, 48, 64, 3)
    z = torch.zeros((0, 32, h, w), device='cuda')
    hd = torch.zeros((0,), device='cuda', dtype=torch.int32)
    assert mgw.ops.streams_assemble(z, z, hd, sb.taps, torch.zeros((0, h, w), device='cuda')).shape == (0, h, w, 13)
    mgw.ops.streams_push(z, z, hd, torch.zeros((0, h, w), device='cuda'), torch.zeros((0, h, w), device='cuda'))
    assert mgw.launch_count() == n0

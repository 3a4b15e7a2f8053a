"""GPU: videos of different source sizes in one batch (deploy.MixedStreamBatch and the per-slot geometry calls).  Every comparison
is bit-exact: each slot of a mixed call must equal the uniform batch call at that slot's size, and each slot of a MixedStreamBatch
its own single-stream pipeline."""
import numpy as np
import pytest
import torch

import yuv420_ref
from conftest import load_golden
from test_gpu_streams import fake_net_batch, fake_net_one, identity_mesh, rect_or_none, slot_history

pytestmark = pytest.mark.gpu


@pytest.fixture(scope='module')
def mgw():
    import dovs_b200
    assert torch.cuda.is_available(), 'GPU tests need a CUDA device; there is no CPU fallback'
    return dovs_b200


def frame(rs, fmt, H, W):
    """one random source frame as a uint8 CUDA tensor: BGR [H,W,3] or YUV 4:2:0 [3H/2,W]"""
    f = rs.randint(0, 256, (H, W, 3)).astype(np.uint8) if fmt == 'bgr' else yuv420_ref.random_frame(rs, H, W)
    return torch.as_tensor(f).cuda()


def frame_bytes(fmt, H, W):
    return H * W * 3 if fmt == 'bgr' else H * W * 3 // 2


def cap_shape(fmt, H, W):
    return (H, W, 3) if fmt == 'bgr' else (H * 3 // 2, W)


class MixedCall:
    """the arguments of one mixed call: a pool with `slack` bytes past the last region, sizes and stacked per-slot tables"""

    def __init__(self, mgw, fmt, cap, frames, sizes, h, w, cr, slack=0, table_sizes=None):
        S, fb = len(sizes), frame_bytes(fmt, *cap)
        self.flat = torch.zeros(S * fb + slack, device='cuda', dtype=torch.uint8)
        self.pool = self.flat[:S * fb].view((S,) + cap_shape(fmt, *cap))
        for s, f in enumerate(frames):
            if f is not None:
                self.flat[s * fb:s * fb + f.numel()] = f.reshape(-1)
        self.sizes = torch.tensor(sizes, dtype=torch.int32).reshape(S, 2).cuda()
        tabs = [mgw.deploy.mixed_slot_tables(ts, cap, h, w, cr) for ts in (table_sizes or sizes)]
        stacked = [torch.as_tensor(np.stack(t)).cuda() for t in zip(*tabs)]
        self.tables, self.xtab, self.ytab = tuple(stacked[:6]), stacked[6], stacked[7]
        self.fmt, self.h, self.w = fmt, h, w

    def cvt(self, mgw, **kw):
        return mgw.ops.cvt_img2train_mixed(self.pool, self.fmt, self.sizes, self.tables, self.h, self.w, **kw)

    def resize(self, mgw, **kw):
        return mgw.ops.resize_linear_mixed(self.pool, self.fmt, self.sizes, self.xtab, self.ytab, self.h, self.w, **kw)


def uniform(mgw, f, fmt, h, w, cr):
    """the uniform batch calls at the frame's own size (a batch of one)"""
    cur = mgw.deploy.cvt_img2train(f[None], cr, height=h, width=w, src_format=fmt)
    return cur.reshape(h, w), mgw.deploy.cv2_resize(f[None], (w, h), src_format=fmt)[0]


# ---- the front end: one mixed call against the uniform calls slot by slot
BIG_BGR = [(1080, 1920), (720, 1280), (1920, 1080), (576, 1024), (240, 426), (91, 157), (123, 77), (480, 854)]
BIG_YUV = [(1080, 1920), (720, 1280), (1920, 1080), (576, 1024), (240, 426), (90, 158), (6, 10), (480, 854)]


def front_end_cases(fmt):
    """(slot sizes, h, w, crop_rate): the production sizes at 288x512 with crop_rate 1 and 0.9 (576x1024 takes the 2x2
    shortcut), and every output / crop-rate configuration of the cvt_img2train fixture with its source sizes"""
    big = BIG_BGR if fmt == 'bgr' else BIG_YUV
    cases = [(big, 288, 512, 1), (big, 288, 512, 0.9)]
    g = load_golden('deploy_cvt_img2train')
    fixture = [g[n + '_img'].shape[:2] for n in sorted(k[:-4] for k in g if k.endswith('_out'))]
    fixture = [(H - H % 2, W - W % 2) if fmt != 'bgr' else (H, W) for H, W in fixture]
    for n in sorted(k[:-4] for k in g if k.endswith('_out')):
        h, w, cr = g[n + '_cfg']
        cases.append((fixture + [(96, 128), (36, 64)], int(h), int(w), 1 if cr == 1 else float(cr)))
    return cases


@pytest.mark.parametrize('fmt', ['bgr', 'nv12', 'i420'])
def test_mixed_front_end_equals_uniform_calls(mgw, fmt):
    rs = np.random.RandomState(50)
    for sizes, h, w, cr in front_end_cases(fmt):
        largest = (max(s[0] for s in sizes), max(s[1] for s in sizes))
        for cap in (largest, (largest[0] + 2, largest[1] + 6)):           # the capacity equal to the largest slot, and larger
            frames = [frame(rs, fmt, H, W) for H, W in sizes]
            mc = MixedCall(mgw, fmt, cap, frames, sizes, h, w, cr)
            out, dst = mc.cvt(mgw), mc.resize(mgw)
            for s, f in enumerate(frames):
                want_cur, want_small = uniform(mgw, f, fmt, h, w, cr)
                assert torch.equal(out[s], want_cur), (fmt, sizes[s], cap, h, w, cr)
                assert torch.equal(dst[s], want_small), (fmt, sizes[s], cap, h, w, cr)


def test_mixed_slot_reproduces_the_fixtures(mgw):
    """one slot of a mixed batch against the fixtures made by OpenCV + Pillow"""
    rs = np.random.RandomState(51)
    g = load_golden('deploy_cvt_img2train')
    for n in sorted(k[:-4] for k in g if k.endswith('_out')):
        h, w, cr = g[n + '_cfg']
        img = torch.as_tensor(g[n + '_img']).cuda()
        H, W = img.shape[:2]
        sizes = [(H + 5, W + 3), (H, W), (H // 2 + 1, W // 2 + 1)]
        frames = [frame(rs, 'bgr', *sizes[0]), img, frame(rs, 'bgr', *sizes[2])]
        mc = MixedCall(mgw, 'bgr', (H + 8, W + 8), frames, sizes, int(h), int(w), 1 if cr == 1 else float(cr))
        assert np.array_equal(mc.cvt(mgw)[1].cpu().numpy(), g[n + '_out'][0, ..., 0].astype(np.float32)), n
    g = load_golden('deploy_cv2_resize')
    for n in sorted(k[:-4] for k in g if k.endswith('_dst')):
        want, img = g[n + '_dst'], g[n + '_img']
        if img.ndim != 3 or img.shape[2] != 3:
            continue                                                        # the mixed resize is BGR
        H, W = img.shape[:2]
        sizes = [(H + 4, W + 2), (H, W)]
        mc = MixedCall(mgw, 'bgr', (H + 4, W + 4), [frame(rs, 'bgr', *sizes[0]), torch.as_tensor(img).cuda()], sizes,
                       want.shape[0], want.shape[1], 1)
        assert np.array_equal(mc.resize(mgw)[1].cpu().numpy(), want), n
    g = load_golden('deploy_yuv420')
    for n in sorted(k[:-8] for k in g if k.endswith('_resized')):
        fmt, want, yuv = n.split('_')[0], g[n + '_resized'], torch.as_tensor(g[n + '_yuv']).cuda()
        H, W = yuv.shape[0] // 3 * 2, yuv.shape[1]
        sizes = [(H + 2, W + 4), (H, W)]
        mc = MixedCall(mgw, fmt, (H + 4, W + 4), [frame(rs, fmt, *sizes[0]), yuv], sizes, want.shape[0], want.shape[1], 1)
        assert np.array_equal(mc.resize(mgw)[1].cpu().numpy(), want), n


@pytest.mark.parametrize('fmt', ['bgr', 'nv12', 'i420'])
def test_idle_slots_write_nothing(mgw, fmt):
    """slots of size 0, above the capacity or (YUV) odd leave out / tmp / dst as they were.  The pool and every output have
    slack past their end, so that a slot that read or wrote past its region would show up here as changed bytes"""
    rs = np.random.RandomState(52)
    cap, h, w = (96, 160), 36, 64
    sizes = [(90, 158), (0, 0), (0, 64), (98, 160), (96, 166), (72, 128)]
    if fmt != 'bgr':
        sizes += [(91, 128), (90, 127)]
    active = {0, 5}
    fb = frame_bytes(fmt, *cap)
    frames = [frame(rs, fmt, *sz) if s in active else None for s, sz in enumerate(sizes)]
    mc = MixedCall(mgw, fmt, cap, frames, sizes, h, w, 1, slack=4 * fb, table_sizes=[cap] * len(sizes))
    mc.flat[mc.pool.numel():] = torch.as_tensor(rs.randint(0, 256, 4 * fb).astype(np.uint8)).cuda()
    for s in set(range(len(sizes))) - active:
        mc.flat[s * fb:(s + 1) * fb] = torch.as_tensor(rs.randint(0, 256, fb).astype(np.uint8)).cuda()
    for s in active:                                                        # active slots use their own tables
        own = MixedCall(mgw, fmt, cap, [None], [sizes[s]], h, w, 1)
        for t, o in zip(mc.tables + (mc.xtab, mc.ytab), own.tables + (own.xtab, own.ytab)):
            t[s] = o[0]
    S, slack = len(sizes), 4096
    out_buf = torch.full((S * h * w + slack,), 7.25, device='cuda')
    tmp_buf = torch.full((S * cap[0] * w + slack,), 0xA5, device='cuda', dtype=torch.uint8)
    dst_buf = torch.full((S * h * w * 3 + slack,), 0x5A, device='cuda', dtype=torch.uint8)
    out, tmp = out_buf[:S * h * w].view(S, h, w), tmp_buf[:S * cap[0] * w].view(S, cap[0], w)
    dst = dst_buf[:S * h * w * 3].view(S, h, w, 3)
    mc.cvt(mgw, out=out, tmp=tmp)
    mc.resize(mgw, out=dst)
    for s in range(S):
        if s in active:
            want_cur, want_small = uniform(mgw, frames[s], fmt, h, w, 1)
            assert torch.equal(out[s], want_cur) and torch.equal(dst[s], want_small), (fmt, sizes[s])
        else:
            assert bool((out[s] == 7.25).all()) and bool((tmp[s] == 0xA5).all()) and bool((dst[s] == 0x5A).all()), (fmt, sizes[s])
    assert bool((out_buf[S * h * w:] == 7.25).all()) and bool((tmp_buf[S * cap[0] * w:] == 0xA5).all())
    assert bool((dst_buf[S * h * w * 3:] == 0x5A).all())


# ---- MixedStreamBatch against independent single-stream pipelines
class OnePipeline:
    """one video the single-stream way at its own size: StreamState + CropState + cv2_resize + warpRevBundle2"""

    def __init__(self, mgw, first, fmt, h, w, crop_rate, refine, base):
        self.mgw, self.fmt, self.h, self.w, self.cr, self.refine, self.base = mgw, fmt, h, w, crop_rate, refine, base
        cur = mgw.deploy.cvt_img2train(first, crop_rate, height=h, width=w, src_format=fmt)
        self.st, self.crop = mgw.StreamState(cur.reshape(h, w)), mgw.CropState(h, w)

    def step(self, raw):
        mgw, h, w = self.mgw, self.h, self.w
        cur = mgw.deploy.cvt_img2train(raw, self.cr, height=h, width=w, src_format=self.fmt)
        in_x = self.st.assemble(cur.reshape(h, w))
        assembled = in_x.clone()
        for _ in range(self.refine):
            out, black, xy = fake_net_one(mgw, in_x, self.base)
            self.crop.add(black)
            self.st.refeed(in_x, out, black)
        self.st.push(out, black)
        small = mgw.deploy.cv2_resize(raw, (w, h), src_format=self.fmt)
        colour = mgw.deploy.warpRevBundle2(small, xy[0, ..., 0], xy[0, ..., 1])
        return assembled, in_x, colour


def check_slot_state(mb, s, p, where):
    fr, mk = slot_history(mb, s)
    f0, m0 = p.st.history()
    assert torch.equal(fr, f0) and torch.equal(mk, m0) and torch.equal(mb.all_black[s], p.crop.all_black), where
    assert rect_or_none(lambda: mb.leave(s)) == rect_or_none(p.crop.rect), where


@pytest.mark.parametrize('fmt', ['bgr', 'nv12'])
def test_mixed_stream_batch_equals_independent_pipelines(mgw, fmt):
    cap, h, w, refine, cr = (150, 256), 48, 80, 2, 0.9
    # slot 0: 120x200 throughout; slot 1: 96x160 for steps 0-5, then 150x96 portrait from step 7 (a re-join at another size);
    # slot 2: 150x256 (the capacity) from step 3; slot 3: 96x160 (the 2x2 shortcut) from step 2, leaves at step 9; slot 4: idle
    first_sizes = {(0, 0): (120, 200), (0, 1): (96, 160), (2, 3): (96, 160), (3, 2): (150, 256), (7, 1): (150, 96)}
    leaves = {6: [1], 9: [3]}
    base = identity_mesh()
    mb = mgw.MixedStreamBatch(5, cap, height=h, width=w, crop_rate=cr, refine=refine, src_format=fmt)
    rec = []
    net, new_step = fake_net_batch(mgw, base, rec)
    rs = np.random.RandomState(53)
    pool = torch.zeros(mb.pool_shape, device='cuda', dtype=torch.uint8)
    pipes, size_of = {}, {}
    for k in range(12):
        for s in leaves.get(k, []):
            check_slot_state(mb, s, pipes.pop(s), (k, s))
        for (kk, s), sz in first_sizes.items():
            if kk == k:
                first = frame(rs, fmt, *sz)
                mb.join(s, first)
                pipes[s], size_of[s] = OnePipeline(mgw, first, fmt, h, w, cr, refine, base), sz
        for s in pipes:
            mb.slot_frame(pool, s).copy_(frame(rs, fmt, *size_of[s]))
        new_step()
        colour = mb.step(pool, net).clone()
        for s, p in pipes.items():
            assembled, refined, want = p.step(mb.slot_frame(pool, s))
            assert torch.equal(rec[-1][s:s + 1], assembled), (fmt, k, s)
            assert torch.equal(mb.in_x[s:s + 1], refined), (fmt, k, s)
            assert torch.equal(colour[s], want), (fmt, k, s)
        assert not mb.cur[4].any() and not mb.small[4].any()                 # the idle slot fed zeros
    for s, p in pipes.items():
        assert int(mb.all_black[s].sum()) > 0, s
        check_slot_state(mb, s, p, ('end', s))


def test_uniform_sizes_equal_stream_batch(mgw):
    """every slot at one size: a mixed batch (capacity equal to that size, and larger) == StreamBatch, byte for byte"""
    S, H, W, h, w = 3, 90, 160, 36, 64
    base = identity_mesh()
    net, _ = fake_net_batch(mgw, base)
    rs = np.random.RandomState(54)
    sb = mgw.StreamBatch(S, (H, W), height=h, width=w, refine=2)
    mbs = [mgw.MixedStreamBatch(S, cap, height=h, width=w, refine=2) for cap in ((H, W), (H + 30, W + 50))]
    pools = [torch.zeros(mb.pool_shape, device='cuda', dtype=torch.uint8) for mb in mbs]
    for s in range(S):
        first = frame(rs, 'bgr', H, W)
        sb.join(s, first)
        for mb in mbs:
            mb.join(s, first)
    for k in range(6):
        raw = torch.stack([frame(rs, 'bgr', H, W) for _ in range(S)])
        want = sb.step(raw, net).clone()
        for mb, pool in zip(mbs, pools):
            for s in range(S):
                mb.slot_frame(pool, s).copy_(raw[s])
            assert torch.equal(mb.step(pool, net), want), k
            for a, b in ((mb.frames, sb.frames), (mb.masks, sb.masks), (mb.heads_dev, sb.heads_dev), (mb.all_black, sb.all_black),
                         (mb.in_x, sb.in_x), (mb.cur, sb.cur), (mb.small, sb.small)):
                assert torch.equal(a, b), k


def test_mixed_graph_replay_equals_eager(mgw):
    """one capture with the whole-pool upload and the download inside the graph, replayed 12 times, with a slot re-joining at a
    new size and an idle slot joining between replays == the same schedule run eagerly"""
    S, cap, h, w = 3, (120, 200), 48, 80
    base = identity_mesh()
    net, _ = fake_net_batch(mgw, base)
    rs = np.random.RandomState(55)
    eager = mgw.MixedStreamBatch(S, cap, height=h, width=w, refine=2, src_format='i420')
    graphed = mgw.MixedStreamBatch(S, cap, height=h, width=w, refine=2, src_format='i420')
    host_in = torch.zeros(graphed.pool_shape, dtype=torch.uint8).pin_memory()
    host_out = torch.empty((S, h, w, 3), dtype=torch.uint8).pin_memory()
    pool_g = torch.zeros(graphed.pool_shape, device='cuda', dtype=torch.uint8)
    pool_e = torch.zeros(eager.pool_shape, device='cuda', dtype=torch.uint8)
    sizes = {0: (120, 200), 1: (72, 128)}
    for s, sz in sizes.items():
        first = frame(rs, 'i420', *sz)
        eager.join(s, first); graphed.join(s, first)
    graph = graphed.capture(pool_g, net, upload_from=host_in, download_to=host_out)
    for k in range(12):
        if k in (4, 8):
            s, sz = (1, (100, 60)) if k == 4 else (2, (60, 100))
            first = frame(rs, 'i420', *sz)
            eager.join(s, first); graphed.join(s, first)
            sizes[s] = sz
        for s, sz in sizes.items():
            graphed.slot_frame(host_in, s).copy_(frame(rs, 'i420', *sz).cpu())
        graph.replay()
        torch.cuda.synchronize()
        pool_e.copy_(host_in)
        want = eager.step(pool_e, net)
        assert torch.equal(host_out.cuda(), want), k
    for a, b in ((eager.frames, graphed.frames), (eager.masks, graphed.masks), (eager.heads_dev, graphed.heads_dev),
                 (eager.all_black, graphed.all_black), (eager.in_x, graphed.in_x)):
        assert torch.equal(a, b)
    for s in range(S):
        assert rect_or_none(lambda: eager.leave(s)) == rect_or_none(lambda: graphed.leave(s))


def test_mixed_errors(mgw):
    from dovs_b200._lib import check, lib
    mb = mgw.MixedStreamBatch(2, (96, 160), height=24, width=40)
    yb = mgw.MixedStreamBatch(2, (96, 160), height=24, width=40, src_format='nv12')
    net, _ = fake_net_batch(mgw, identity_mesh())
    for bad in (torch.zeros((98, 160, 3), device='cuda', dtype=torch.uint8),         # above the capacity
                torch.zeros((96, 162, 3), device='cuda', dtype=torch.uint8),
                torch.zeros((48, 64, 3), device='cuda', dtype=torch.float32),        # dtype
                torch.zeros((48, 64, 4), device='cuda', dtype=torch.uint8)):
        with pytest.raises(ValueError):
            mb.join(0, bad)
    for bad in (torch.zeros((72, 63), device='cuda', dtype=torch.uint8),             # odd W
                torch.zeros((73, 64), device='cuda', dtype=torch.uint8),             # 3H/2 rows: not a multiple of 3
                torch.zeros((147, 160), device='cuda', dtype=torch.uint8)):          # H = 98 above the capacity
        with pytest.raises(ValueError):
            yb.join(0, bad)
    for bad in (torch.zeros((2, 96 * 160 * 3 - 1), device='cuda', dtype=torch.uint8),
                torch.zeros((3, 96 * 160 * 3), device='cuda', dtype=torch.uint8),
                torch.zeros((2, 96 * 160 * 3), device='cuda', dtype=torch.int32)):
        with pytest.raises(ValueError):
            mb.step(bad, net)
    with pytest.raises(ValueError):
        mb.slot_frame(torch.zeros(mb.pool_shape, dtype=torch.uint8), 1)             # slot 1 never joined
    mb.join(1, torch.zeros((50, 70, 3), device='cuda', dtype=torch.uint8))
    assert tuple(mb.slot_frame(torch.zeros(mb.pool_shape, dtype=torch.uint8), 1).shape) == (50, 70, 3)
    with pytest.raises(ValueError):
        mb.slot_frame(torch.zeros((2, 10), dtype=torch.uint8), 1)
    # the C calls: bad sizes and a misaligned `sizes` are refused before anything is launched
    p, sz = mb.frames.data_ptr(), mb.sizes.data_ptr()
    kx, x0, xn, ky, y0, yn = (t.data_ptr() for t in mb.tables)
    with pytest.raises(mgw.MgwError, match='bad sizes'):
        check(lib.mgw_cvt_img2train_mixed(p, 0, 65, 2160, 3840, sz, kx, x0, xn, 5, ky, y0, yn, 5, 24, 40, p, p, None), 'cvt')
    with pytest.raises(mgw.MgwError, match='bad sizes'):
        check(lib.mgw_resize_linear_mixed(p, 1, 2, 97, 160, sz, p, p, 24, 40, p, None), 'resize')
    with pytest.raises(mgw.MgwError, match='8-byte aligned'):
        check(lib.mgw_resize_linear_mixed(p, 0, 2, 96, 160, sz + 4, p, p, 24, 40, p, None), 'resize')
    with pytest.raises(ValueError):
        mgw.ops.resize_linear_mixed(mb.frames.new_zeros((2, 96, 160, 3), dtype=torch.uint8), 'bgr', mb.sizes[:1], mb.xtab, mb.ytab, 24, 40)
    n0 = mgw.launch_count()
    empty = torch.zeros((0, 96, 160, 3), device='cuda', dtype=torch.uint8)
    z = lambda *s: torch.zeros(s, device='cuda', dtype=torch.int32)
    assert mgw.ops.cvt_img2train_mixed(empty, 'bgr', z(0, 2), (z(0, 40, 5), z(0, 40), z(0, 40), z(0, 24, 5), z(0, 24), z(0, 24)),
                                       24, 40).shape == (0, 24, 40)
    assert mgw.ops.resize_linear_mixed(empty, 'bgr', z(0, 2), z(0, 40, 4), z(0, 24, 4), 24, 40).shape == (0, 24, 40, 3)
    assert mgw.launch_count() == n0

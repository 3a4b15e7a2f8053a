"""GPU: a batch of one size read from decoder-style surfaces and written into encoder-style surfaces through plane tables
(mgw_*_planes, StreamBatch.step_planes / capture_planes).  Every comparison is bit-exact against the packed batch calls on the
same frames; every byte of a surface outside its planes' used bytes, and every byte of an idle slot, keeps its sentinel."""
import numpy as np
import pytest
import torch

import remap_frame_ref as M
from test_gpu_streams import fake_net_batch, identity_mesh, rect_or_none

pytestmark = pytest.mark.gpu

FORMATS = ('bgr', 'nv12', 'i420')
SENTINEL = 0xA7
LAYOUTS = ('nvdec', 'odd', 'split')


@pytest.fixture(scope='module')
def mgw():
    import dovs_b200
    assert torch.cuda.is_available(), 'GPU tests need a CUDA device; there is no CPU fallback'
    return dovs_b200


def plane_rows(fmt, H, W):
    if fmt == 'bgr':
        return [(H, 3 * W)]
    if fmt == 'nv12':
        return [(H, W), (H // 2, W)]
    return [(H, W), (H // 2, W // 2), (H // 2, W // 2)]


def packed_shape(fmt, H, W):
    return (H, W, 3) if fmt == 'bgr' else (H * 3 // 2, W)


class Surface:
    """one frame's planes in allocations of their own, laid out as
      nvdec  one allocation, pitch rounded up to 512 bytes (2048 at 1920), each plane after the previous one's coded rows
             (the height rounded up to 16: the chroma of a 1080p surface starts at row 1088)
      odd    one allocation starting 1 byte past an aligned address, pitch = row bytes + 3, 5 bytes between the planes
      split  every plane in an allocation of its own, pitch = row bytes + 1 (I420's U and V apart)
    every byte outside the planes' used bytes holds SENTINEL"""

    def __init__(self, fmt, H, W, layout):
        self.fmt, self.H, self.W, self.layout = fmt, H, W, layout
        self.rows = plane_rows(fmt, H, W)
        self.allocs, self.views, self.pitches = [], [], []
        if layout == 'split':
            for n, nb in self.rows:
                a = torch.full((n * (nb + 1) + 64,), SENTINEL, dtype=torch.uint8, device='cuda')
                self.allocs.append(a)
                self.views.append((a, 0, n, nb, nb + 1))
        else:
            if layout == 'nvdec':
                p0 = -(-self.rows[0][1] // 512) * 512
                pitches = [p0] + [p0 if fmt == 'nv12' else p0 // 2] * (len(self.rows) - 1)
                coded = [-(-n // 16) * 16 if k == 0 else -(-H // 16) * 16 // 2 for k, (n, _) in enumerate(self.rows)]
                gap, start = 0, 0
            else:
                pitches = [nb + 3 for _, nb in self.rows]
                coded = [n for n, _ in self.rows]
                gap, start = 5, 1
            total = start + sum(c * p + gap for c, p in zip(coded, pitches)) + 64
            a = torch.full((total,), SENTINEL, dtype=torch.uint8, device='cuda')
            self.allocs.append(a)
            off = start
            for (n, nb), c, p in zip(self.rows, coded, pitches):
                self.views.append((a, off, n, nb, p))
                off += c * p + gap

    def plane_view(self, k):
        a, off, n, nb, p = self.views[k]
        return a[off:off + n * p].view(n, p)[:, :nb]

    def planes(self):
        """pitched views for nvdec / odd, raw (address, pitch) pairs for split"""
        if self.layout == 'split':
            return [(a.data_ptr() + off, p) for a, off, n, nb, p in self.views]
        return [self.plane_view(k) for k in range(len(self.views))]

    def write(self, frame):
        flat, off = frame.reshape(-1), 0
        for k, (n, nb) in enumerate(self.rows):
            self.plane_view(k).copy_(flat[off:off + n * nb].view(n, nb))
            off += n * nb

    def read(self):
        return torch.cat([self.plane_view(k).reshape(-1) for k in range(len(self.rows))]).view(packed_shape(self.fmt, self.H, self.W))

    def untouched_outside(self):
        for a in self.allocs:
            mask = torch.ones_like(a, dtype=torch.bool)
            for b, off, n, nb, p in self.views:
                if b is a:
                    mask[off:off + n * p].view(n, p)[:, :nb] = False
            if not bool((a[mask] == SENTINEL).all()):
                return False
        return True

    def all_sentinel(self):
        return all(bool((a == SENTINEL).all()) for a in self.allocs)


def surfaces(S, fmt, H, W, seed):
    """S surfaces with the layouts in turn, allocated in a permuted slot order"""
    order = np.random.RandomState(seed).permutation(S)
    out = [None] * S
    for s in order:
        out[s] = Surface(fmt, H, W, LAYOUTS[s % len(LAYOUTS)])
    return out


def table_of(mgw, fmt, H, W, surfs, idle=()):
    t = mgw.PlaneTable(len(surfs), fmt, (H, W))
    for s, sf in enumerate(surfs):
        t.set(s, sf.planes())
    # entries PlaneTable.set() refuses, written into the mirror directly: the device must treat them as idle slots
    e = t.host.numpy().view(mgw.deploy._PLANES_DTYPE).reshape(t.S)
    last = len(plane_rows(fmt, H, W)) - 1
    for s, kind in idle:
        if kind == 'null':
            e['plane'][s, last] = 0                                    # the last plane the format needs is missing
        else:
            e['pitch'][s, last] = plane_rows(fmt, H, W)[last][1] - 1     # its pitch is one byte short of its rows
    t.upload()
    return t


def random_frames(gen, fmt, S, H, W):
    return torch.randint(0, 256, (S,) + packed_shape(fmt, H, W), dtype=torch.uint8, device='cuda', generator=gen)


def maps(h, w, seed, wild):
    xm, ym = M.wild_mesh(h, w, seed) if wild else M.smooth_mesh(h, w, seed)
    return torch.stack([torch.as_tensor(np.ascontiguousarray(xm)), torch.as_tensor(np.ascontiguousarray(ym))], -1).cuda()


# ---- the front end against the packed batch calls
@pytest.mark.parametrize('fmt', FORMATS)
@pytest.mark.parametrize('H,W', [(1080, 1920), (90, 158)])
def test_front_end_equals_packed_calls(mgw, fmt, H, W):
    d, ops = mgw.deploy, mgw.ops
    S, h, w = 7, 48, 80
    idle = [(5, 'null'), (6, 'short')]
    gen = torch.Generator(device='cuda')
    gen.manual_seed(80 + H)
    frames = random_frames(gen, fmt, S, H, W)
    surfs = surfaces(S, fmt, H, W, 1)
    for s, sf in enumerate(surfs):
        sf.write(frames[s])
    table = table_of(mgw, fmt, H, W, surfs, idle)
    tabs = d._cvt_tables(H, W, h, w, 1, 'cuda')
    if fmt == 'bgr':
        want = ops.cvt_img2train_u8_batch(frames, tabs, h, w)
    else:
        want = ops.cvt_img2train_yuv420_batch(frames, fmt, tabs, h, w)
    out = torch.full((S, h, w), 7.0, device='cuda')
    tmp = torch.full((S, H, w), SENTINEL, dtype=torch.uint8, device='cuda')
    ops.cvt_img2train_planes(table.device, fmt, (H, W), tabs, h, w, out=out, tmp=tmp)
    assert torch.equal(out[:5], want[:5]), fmt
    assert bool((out[5:] == 7.0).all()) and bool((tmp[5:] == SENTINEL).all())
    # cv2.resize: the general path and the 2x2 INTER_AREA shortcut
    for oh, ow in ((72, 128), (H // 2, W // 2), (H + 6, W + 10)):
        xt, yt = d._resize_tables(H, W, oh, ow, 'cuda')
        if fmt == 'bgr':
            want = ops.resize_linear_u8_batch(frames, xt, yt, oh, ow)
        else:
            want = ops.resize_linear_yuv420_batch(frames, fmt, xt, yt, oh, ow)
        dst = torch.full((S, oh, ow, 3), SENTINEL, dtype=torch.uint8, device='cuda')
        ops.resize_linear_planes(table.device, fmt, (H, W), xt, yt, oh, ow, out=dst)
        assert torch.equal(dst[:5], want[:5]), (fmt, oh, ow)
        assert bool((dst[5:] == SENTINEL).all())
    for s, sf in enumerate(surfs):
        assert torch.equal(sf.read(), frames[s]) and sf.untouched_outside()      # the sources are only read


# ---- the warp against the packed warp, all nine format pairs
@pytest.mark.parametrize('src_fmt', FORMATS)
@pytest.mark.parametrize('dst_fmt', FORMATS)
def test_warp_equals_packed_warp(mgw, src_fmt, dst_fmt):
    ops = mgw.ops
    yuv = src_fmt != 'bgr' or dst_fmt != 'bgr'
    gen = torch.Generator(device='cuda')
    gen.manual_seed(81)
    for (H, W), (h, w) in (((1080, 1920), (288, 512)), (((90, 158) if yuv else (91, 157)), (36, 64)), (((6, 10) if yuv else (7, 9)), (8, 8))):
        S = 8
        idle_src, idle_dst = [(6, 'null')], [(7, 'short')]
        frames = random_frames(gen, src_fmt, S, H, W)
        src = surfaces(S, src_fmt, H, W, 2)
        for s, sf in enumerate(src):
            sf.write(frames[s])
        dst = surfaces(S, dst_fmt, H, W, 3)
        st, dt = table_of(mgw, src_fmt, H, W, src, idle_src), table_of(mgw, dst_fmt, H, W, dst, idle_dst)
        xy = torch.stack([maps(h, w, 200 + s, wild=s % 2 == 1) for s in range(S)]).contiguous()
        ops.remap_bundle_frame_planes(st.device, src_fmt, xy, (H, W), dt.device, dst_fmt)
        want = ops.remap_bundle_frame(frames, src_fmt, xy, out_format=dst_fmt)
        for s in range(6):
            assert torch.equal(dst[s].read(), want[s]), (src_fmt, dst_fmt, H, W, s, dst[s].layout)
            assert dst[s].untouched_outside(), (src_fmt, dst_fmt, H, W, s)
        for s in (6, 7):
            assert dst[s].all_sentinel(), (src_fmt, dst_fmt, H, W, s)                # idle: nothing written
        for s, sf in enumerate(src):
            assert torch.equal(sf.read(), frames[s]) and sf.untouched_outside()


def test_packed_table_is_the_packed_call(mgw):
    """a contiguous batch described by PlaneTable.packed gives the packed call's bytes"""
    ops = mgw.ops
    gen = torch.Generator(device='cuda')
    gen.manual_seed(82)
    S, H, W, h, w = 3, 90, 158, 36, 64
    for fmt, dfmt in (('bgr', 'i420'), ('nv12', 'bgr'), ('i420', 'nv12')):
        frames = random_frames(gen, fmt, S, H, W)
        xy = torch.stack([maps(h, w, 300 + s, wild=s == 1) for s in range(S)]).contiguous()
        want = ops.remap_bundle_frame(frames, fmt, xy, out_format=dfmt)
        got = torch.full_like(want, SENTINEL)
        ops.remap_bundle_frame_planes(mgw.PlaneTable.packed(frames, fmt).device, fmt, xy, (H, W), mgw.PlaneTable.packed(got, dfmt).device,
                                      dfmt)
        assert torch.equal(got, want), (fmt, dfmt)


# ---- StreamBatch.step_planes against StreamBatch.step on the packed frames
CASES = [('nv12', None, 'bgr', False), ('bgr', 'src', 'nv12', True), ('i420', (96, 160), 'i420', True),
         ('nv12', 'src', 'bgr', True), ('i420', 'src', 'i420', False), ('bgr', (72, 100), 'bgr', True)]


@pytest.mark.parametrize('fmt,out,out_format,pitched_out', CASES)
def test_step_planes_equals_step(mgw, fmt, out, out_format, pitched_out):
    S, size, h, w, refine = 3, (120, 200), 48, 80, 2
    out_size = size if out == 'src' else out
    base = identity_mesh()
    net, _ = fake_net_batch(mgw, base)
    kw = dict(height=h, width=w, refine=refine, src_format=fmt, out_size=out_size, out_format=out_format)
    ref, sb = mgw.StreamBatch(S, size, **kw), mgw.StreamBatch(S, size, **kw)
    OH, OW = sb.out_size
    gen = torch.Generator(device='cuda')
    gen.manual_seed(83)
    src = surfaces(S, fmt, *size, 4)
    src_t = table_of(mgw, fmt, *size, src)
    dst = surfaces(S, out_format, OH, OW, 5) if pitched_out else None
    dst_t = table_of(mgw, out_format, OH, OW, dst) if pitched_out else None
    # slot 0 from step 0; slot 1 steps 0-19, then a second video from step 25; slot 2 from step 10
    joins, leaves = {0: [0, 1], 10: [2], 25: [1]}, {20: [1]}
    for k in range(40):
        for s in leaves.get(k, []):
            assert rect_or_none(lambda: sb.leave(s)) == rect_or_none(lambda: ref.leave(s)), (k, s)
        raw = random_frames(gen, fmt, S, *size)
        for s in joins.get(k, []):
            sb.join(s, raw[s]); ref.join(s, raw[s])
        for s in range(S):
            src[s].write(raw[s])
        want = ref.step(raw, net)
        got = sb.step_planes(src_t, net, dst_t)
        if pitched_out:
            assert got is dst_t
            for s in range(S):
                assert torch.equal(dst[s].read(), want[s]), (k, s)
        else:
            assert got.data_ptr() == sb.colour.data_ptr() and torch.equal(got, want), k
    for s in range(S):
        assert rect_or_none(lambda: sb.leave(s)) == rect_or_none(lambda: ref.leave(s)), s
    assert torch.equal(sb.frames, ref.frames) and torch.equal(sb.all_black, ref.all_black)
    if pitched_out:
        assert all(d.untouched_outside() for d in dst)


# ---- one captured graph following a rotating surface pool
@pytest.mark.parametrize('fmt,out,out_format', [('nv12', 'src', 'nv12'), ('i420', None, 'bgr'), ('bgr', (96, 160), 'i420')])
def test_capture_planes_follows_rotating_surfaces(mgw, fmt, out, out_format):
    S, size, h, w, refine, K = 3, (120, 200), 48, 80, 2, 3
    out_size = size if out == 'src' else out
    base = identity_mesh()
    net, _ = fake_net_batch(mgw, base)
    kw = dict(height=h, width=w, refine=refine, src_format=fmt, out_size=out_size, out_format=out_format)
    ref, sb = mgw.StreamBatch(S, size, **kw), mgw.StreamBatch(S, size, **kw)
    OH, OW = sb.out_size
    gen = torch.Generator(device='cuda')
    gen.manual_seed(84)
    pool = [surfaces(S, fmt, *size, 10 + i) for i in range(K)]                 # a decoder's surface pool, K surfaces per slot
    outs = [surfaces(S, out_format, OH, OW, 20 + i) for i in range(K)]         # an encoder's input surfaces
    src_t, dst_t = mgw.PlaneTable(S, fmt, size), mgw.PlaneTable(S, out_format, (OH, OW))

    def point(k):
        for s in range(S):
            src_t.set(s, pool[(k + s) % K][s].planes())
            dst_t.set(s, outs[(2 * k + s) % K][s].planes())

    first = random_frames(gen, fmt, S, *size)
    for s in range(S):
        sb.join(s, first[s]); ref.join(s, first[s])
    point(0)
    graph = sb.capture_planes(src_t, net, dst_t)
    for k in range(12):
        if k == 6:                                                             # slot 1 leaves and a new video joins between replays
            assert rect_or_none(lambda: sb.leave(1)) == rect_or_none(lambda: ref.leave(1))
            new = random_frames(gen, fmt, 1, *size)[0]
            sb.join(1, new); ref.join(1, new)
        raw = random_frames(gen, fmt, S, *size)
        src_t.uploaded.synchronize()                                           # the previous replay has copied the mirrors
        dst_t.uploaded.synchronize()
        point(k)
        for s in range(S):
            pool[(k + s) % K][s].write(raw[s])
        graph.replay()
        want = ref.step(raw, net)
        torch.cuda.synchronize()
        for s in range(S):
            d = outs[(2 * k + s) % K][s]
            assert torch.equal(d.read(), want[s]), (k, s)
    for a, b in ((sb.frames, ref.frames), (sb.masks, ref.masks), (sb.heads_dev, ref.heads_dev), (sb.all_black, ref.all_black)):
        assert torch.equal(a, b)
    for s in range(S):
        assert rect_or_none(lambda: sb.leave(s)) == rect_or_none(lambda: ref.leave(s))
    assert all(d.untouched_outside() for o in outs for d in o)


# ---- an idle slot inside a StreamBatch
@pytest.mark.parametrize('fmt,out,out_format', [('nv12', 'src', 'nv12'), ('bgr', (72, 100), 'i420')])
def test_cleared_slot_is_idle_between_replays(mgw, fmt, out, out_format):
    """a slot cleared between replays of one capture_planes graph writes nothing into its destination surface while the other
    slots stay equal to step() on the packed frames.  At out_size == src_size clearing the source entry is enough; through the
    resize (out_size != src_size) the destination entry is cleared as well, as StreamBatch.step_planes documents."""
    S, size, h, w = 3, (120, 200), 48, 80
    out_size = size if out == 'src' else out
    net, _ = fake_net_batch(mgw, identity_mesh())
    kw = dict(height=h, width=w, refine=1, src_format=fmt, out_size=out_size, out_format=out_format)
    ref, sb = mgw.StreamBatch(S, size, **kw), mgw.StreamBatch(S, size, **kw)
    OH, OW = sb.out_size
    gen = torch.Generator(device='cuda')
    gen.manual_seed(85)
    src, dst = surfaces(S, fmt, *size, 30), surfaces(S, out_format, OH, OW, 31)
    src_t, dst_t = table_of(mgw, fmt, *size, src), table_of(mgw, out_format, OH, OW, dst)
    first = random_frames(gen, fmt, S, *size)
    for s in range(S):
        sb.join(s, first[s]); ref.join(s, first[s])
    graph = sb.capture_planes(src_t, net, dst_t)
    kept = None
    for k in range(10):
        raw = random_frames(gen, fmt, S, *size)
        if k == 5:
            src_t.uploaded.synchronize(); dst_t.uploaded.synchronize()
            src_t.clear(1)
            if out != 'src':
                dst_t.clear(1)
            kept = [a.clone() for a in dst[1].allocs]
        for s in range(S):
            src[s].write(raw[s])
        graph.replay()
        want = ref.step(raw, net)
        torch.cuda.synchronize()
        for s in (0, 2):
            assert torch.equal(dst[s].read(), want[s]), (k, s)
        if kept is None:
            assert torch.equal(dst[1].read(), want[1]), k
        else:
            assert all(torch.equal(a, b) for a, b in zip(dst[1].allocs, kept)), k       # not a byte written

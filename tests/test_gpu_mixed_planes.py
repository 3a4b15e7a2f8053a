"""GPU: a batch of videos of different sizes read from decoder-style surfaces and written into encoder-style surfaces through
mixed plane tables (mgw_*_mixed_planes, MixedStreamBatch.step_planes / capture_planes).  Every comparison is bit-exact against
the _mixed calls (or MixedStreamBatch.step) on the packed pool of the same frames; every byte of a surface outside its planes'
used bytes, every tmp / out row and every surface byte of an idle slot keeps its sentinel."""
import pytest
import torch

from test_gpu_mixed import MixedCall, frame_bytes
from test_gpu_planes import SENTINEL, Surface, maps, random_frames
from test_gpu_streams import fake_net_batch, identity_mesh, rect_or_none

pytestmark = pytest.mark.gpu

FORMATS = ('bgr', 'nv12', 'i420')
LAYOUTS = ('nvdec', 'odd', 'split')
SIZES_BGR = [(1080, 1920), (720, 1280), (1920, 1080), (91, 157), (123, 77), (7, 9)]
SIZES_YUV = [(1080, 1920), (720, 1280), (1920, 1080), (90, 158), (6, 10), (480, 854)]
IDLE = ('never', 'cleared', 'stale', 'null', 'short')     # size 0 / entry cleared / entry of another size / a plane 0 / a short pitch


@pytest.fixture(scope='module')
def mgw():
    import dovs_b200
    assert torch.cuda.is_available(), 'GPU tests need a CUDA device; there is no CPU fallback'
    return dovs_b200


def frame(gen, fmt, H, W):
    return random_frames(gen, fmt, 1, H, W)[0]


def mixed_table(mgw, fmt, cap, surfs, idle=None):
    """the MixedPlaneTable of one Surface per slot (None: cleared) at the surface's size; idle {slot: kind} damages entries the
    way set() refuses (written into the mirror directly) or as a caller can: cleared, or an entry of another size"""
    t = mgw.MixedPlaneTable(len(surfs), fmt, cap)
    for s, sf in enumerate(surfs):
        if sf is not None:
            t.set(s, sf.planes(), (sf.H, sf.W))
    e = t.host.numpy().view(mgw.deploy._PLANES_DTYPE).reshape(t.S)
    for s, kind in (idle or {}).items():
        last = len(surfs[s].rows) - 1
        if kind == 'cleared':
            t.clear(s)
        elif kind == 'stale':
            e['reserved'][s, 0] -= 2                                       # names a frame two rows shorter than sizes[s]
        elif kind == 'null':
            e['plane'][s, last] = 0
        elif kind == 'short':
            e['pitch'][s, last] = surfs[s].rows[last][1] - 1
    t.upload()
    return t


def slots(sizes):
    """the active sizes followed by one slot of each idle kind (their frames at a valid size, 'never' at size 0)"""
    idle_size = (6, 10)
    all_sizes = list(sizes) + [idle_size] * len(IDLE)
    idle = {len(sizes) + k: kind for k, kind in enumerate(IDLE)}
    return all_sizes, idle


# ---- the front end against the _mixed calls on the packed pool
@pytest.mark.parametrize('fmt', FORMATS)
def test_front_end_equals_mixed_calls(mgw, fmt):
    sizes = SIZES_BGR if fmt == 'bgr' else SIZES_YUV
    # a capacity both 1080p orientations fit, then one that only landscape 1080p fits, exactly
    for cap, h, w in (((1920, 1920), 48, 80), ((1080, 1920), 36, 64)):
        act = [sz for sz in sizes if sz[0] <= cap[0] and sz[1] <= cap[1]]
        all_sizes, idle = slots(act)
        S = len(all_sizes)
        gen = torch.Generator(device='cuda')
        gen.manual_seed(90 + cap[0])
        frames = [frame(gen, fmt, *sz) for sz in all_sizes]
        surfs = [Surface(fmt, *sz, LAYOUTS[s % 3]) for s, sz in enumerate(all_sizes)]
        for sf, f in zip(surfs, frames):
            sf.write(f)
        table = mixed_table(mgw, fmt, cap, surfs, idle)
        call_sizes = [(0, 0) if idle.get(s) == 'never' else sz for s, sz in enumerate(all_sizes)]
        mc = MixedCall(mgw, fmt, cap, frames, call_sizes, h, w, 1, table_sizes=all_sizes)
        want = mc.cvt(mgw)
        out = torch.full((S, h, w), 7.0, device='cuda')
        tmp = torch.full((S, cap[0], w), SENTINEL, dtype=torch.uint8, device='cuda')
        mgw.ops.cvt_img2train_mixed_planes(table.device, fmt, mc.sizes, cap, mc.tables, h, w, out=out, tmp=tmp)
        n = len(act)
        assert torch.equal(out[:n], want[:n]), (fmt, cap)
        assert bool((out[n:] == 7.0).all()) and bool((tmp[n:] == SENTINEL).all()), (fmt, cap)
        want = mc.resize(mgw)
        dst = torch.full((S, h, w, 3), SENTINEL, dtype=torch.uint8, device='cuda')
        mgw.ops.resize_linear_mixed_planes(table.device, fmt, mc.sizes, cap, mc.xtab, mc.ytab, h, w, out=dst)
        assert torch.equal(dst[:n], want[:n]) and bool((dst[n:] == SENTINEL).all()), (fmt, cap)
        for sf, f in zip(surfs, frames):
            assert torch.equal(sf.read(), f) and sf.untouched_outside()          # the sources are only read


def test_resize_shortcut_per_slot(mgw):
    """the 2x2 INTER_AREA shortcut is chosen per slot: one slot at twice the output size, one not"""
    gen = torch.Generator(device='cuda')
    gen.manual_seed(91)
    for fmt in FORMATS:
        cap, h, w, sizes = (120, 200), 48, 80, [(96, 160), (120, 200), (60, 100)]
        frames = [frame(gen, fmt, *sz) for sz in sizes]
        surfs = [Surface(fmt, *sz, LAYOUTS[s]) for s, sz in enumerate(sizes)]
        for sf, f in zip(surfs, frames):
            sf.write(f)
        mc = MixedCall(mgw, fmt, cap, frames, sizes, h, w, 1)
        got = mgw.ops.resize_linear_mixed_planes(mixed_table(mgw, fmt, cap, surfs).device, fmt, mc.sizes, cap, mc.xtab, mc.ytab, h, w)
        assert torch.equal(got, mc.resize(mgw)), fmt


# ---- the warp against the _mixed warp on the packed pool, all nine format pairs
@pytest.mark.parametrize('src_fmt', FORMATS)
@pytest.mark.parametrize('dst_fmt', FORMATS)
def test_warp_equals_mixed_warp(mgw, src_fmt, dst_fmt):
    yuv = src_fmt != 'bgr' or dst_fmt != 'bgr'
    act = SIZES_YUV if yuv else SIZES_BGR
    cap, (h, w) = (1920, 1920), (288, 512)
    all_sizes, idle = slots(act)
    S = len(all_sizes)
    gen = torch.Generator(device='cuda')
    gen.manual_seed(92)
    frames = [frame(gen, src_fmt, *sz) for sz in all_sizes]
    src = [Surface(src_fmt, *sz, LAYOUTS[s % 3]) for s, sz in enumerate(all_sizes)]
    dst = [Surface(dst_fmt, *sz, LAYOUTS[(s + 1) % 3]) for s, sz in enumerate(all_sizes)]
    for sf, f in zip(src, frames):
        sf.write(f)
    # the idle kinds on the source side, and a stale and a short destination entry of two more slots (0 and 1 stay active)
    dst_idle = {len(act) - 1: 'stale', len(act) - 2: 'short'}
    st, dt = mixed_table(mgw, src_fmt, cap, src, idle), mixed_table(mgw, dst_fmt, cap, dst, dst_idle)
    call_sizes = [(0, 0) if idle.get(s) == 'never' else sz for s, sz in enumerate(all_sizes)]
    pool = torch.zeros((S, frame_bytes(src_fmt, *cap)), dtype=torch.uint8, device='cuda')
    for s, f in enumerate(frames):
        pool[s, :f.numel()] = f.reshape(-1)
    sizes = torch.tensor(call_sizes, dtype=torch.int32).cuda()
    xy = torch.stack([maps(h, w, 400 + s, wild=s % 2 == 1) for s in range(S)]).contiguous()
    cap_shape = (cap[0], cap[1], 3) if src_fmt == 'bgr' else (cap[0] * 3 // 2, cap[1])
    want = mgw.ops.remap_bundle_frame_mixed(pool.view((S,) + cap_shape), src_fmt, sizes, xy, dst_fmt)
    got = mgw.ops.remap_bundle_frame_mixed_planes(st.device, src_fmt, sizes, xy, cap, dt.device, dst_fmt)
    assert got is dt.device
    torch.cuda.synchronize()
    for s, sz in enumerate(all_sizes):
        if s in idle or s in dst_idle:
            assert dst[s].all_sentinel(), (src_fmt, dst_fmt, s, idle.get(s), dst_idle.get(s))        # idle: not a byte written
        else:
            n = frame_bytes(dst_fmt, *sz)
            assert torch.equal(dst[s].read().reshape(-1), want[s, :n]), (src_fmt, dst_fmt, sz, dst[s].layout)
            assert dst[s].untouched_outside(), (src_fmt, dst_fmt, sz)
    for sf, f in zip(src, frames):
        assert torch.equal(sf.read(), f) and sf.untouched_outside()


def test_pool_table_is_the_mixed_call(mgw):
    """pools described by MixedPlaneTable.pool give the _mixed call's bytes, including the bytes past each slot it leaves alone"""
    gen = torch.Generator(device='cuda')
    gen.manual_seed(93)
    cap, (h, w), sizes = (120, 200), (36, 64), [(120, 200), (60, 100), (90, 158), None]
    for fmt, dfmt in (('bgr', 'i420'), ('nv12', 'bgr'), ('i420', 'nv12')):
        S = len(sizes)
        pool = torch.randint(0, 256, (S, frame_bytes(fmt, *cap)), dtype=torch.uint8, device='cuda', generator=gen)
        sz = torch.tensor([s or (0, 0) for s in sizes], dtype=torch.int32).cuda()
        xy = torch.stack([maps(h, w, 500 + s, wild=s == 1) for s in range(S)]).contiguous()
        cap_shape = (cap[0], cap[1], 3) if fmt == 'bgr' else (cap[0] * 3 // 2, cap[1])
        want = torch.full((S, frame_bytes(dfmt, *cap)), SENTINEL, dtype=torch.uint8, device='cuda')
        mgw.ops.remap_bundle_frame_mixed(pool.view((S,) + cap_shape), fmt, sz, xy, dfmt, out=want)
        got = torch.full_like(want, SENTINEL)
        mgw.ops.remap_bundle_frame_mixed_planes(mgw.MixedPlaneTable.pool(pool, fmt, cap, sizes).device, fmt, sz, xy, cap,
                                                mgw.MixedPlaneTable.pool(got, dfmt, cap, sizes).device, dfmt)
        assert torch.equal(got, want), (fmt, dfmt)


# ---- MixedStreamBatch.step_planes against MixedStreamBatch.step on the packed pool
CASES = [('nv12', 'source', 'nv12', True), ('bgr', 'source', 'bgr', False), ('i420', 'source', 'i420', True),
         ('nv12', None, 'bgr', True), ('bgr', (96, 160), 'i420', False), ('i420', (72, 100), 'nv12', True)]


@pytest.mark.parametrize('fmt,out,out_format,pitched_out', CASES)
def test_step_planes_equals_step(mgw, fmt, out, out_format, pitched_out):
    S, cap, h, w, refine = 3, (150, 256), 48, 80, 2
    net, _ = fake_net_batch(mgw, identity_mesh())
    kw = dict(height=h, width=w, refine=refine, src_format=fmt, out_size=out, out_format=out_format)
    ref, mb = mgw.MixedStreamBatch(S, cap, **kw), mgw.MixedStreamBatch(S, cap, **kw)
    gen = torch.Generator(device='cuda')
    gen.manual_seed(94)
    odd = (91, 157) if fmt == 'bgr' and out_format == 'bgr' else (90, 158)
    src_t = mgw.MixedPlaneTable(S, fmt, cap)
    if out == 'source':
        dst_t = mgw.MixedPlaneTable(S, out_format, cap) if pitched_out else None
    else:
        OH, OW = mb.out_size
        dst = [Surface(out_format, OH, OW, LAYOUTS[s]) for s in range(S)]
        dst_t = mgw.PlaneTable(S, out_format, (OH, OW)) if pitched_out else None
        if pitched_out:
            for s in range(S):
                dst_t.set(s, dst[s].planes())
            dst_t.upload()
    pool = torch.zeros(ref.pool_shape, dtype=torch.uint8, device='cuda')
    src, outs, size_of = [None] * S, [None] * S, {}
    # slot 0 from step 0; slot 1 steps 0-19, then a second video at another size from step 25; slot 2 (the capacity) from step 10
    joins, leaves = {0: {0: (120, 200), 1: odd}, 10: {2: cap}, 25: {1: (144, 96)}}, {20: [1]}
    for k in range(40):
        for s in leaves.get(k, []):
            assert rect_or_none(lambda: mb.leave(s)) == rect_or_none(lambda: ref.leave(s)), (k, s)
        for s, sz in joins.get(k, {}).items():
            first = frame(gen, fmt, *sz)
            mb.join(s, first); ref.join(s, first)
            size_of[s] = sz
            src[s] = Surface(fmt, *sz, LAYOUTS[(s + k) % 3])                  # the decoder's surface at the new size
            src_t.set(s, src[s].planes(), sz)
            if out == 'source' and pitched_out:
                outs[s] = Surface(out_format, *sz, LAYOUTS[(s + k + 1) % 3])
                dst_t.set(s, outs[s].planes(), sz)
        if k in joins:
            src_t.upload()
            if out == 'source' and pitched_out:
                dst_t.upload()
        for s, sz in size_of.items():
            f = frame(gen, fmt, *sz)
            ref.slot_frame(pool, s).copy_(f)
            src[s].write(f)
        want = ref.step(pool, net)
        got = mb.step_planes(src_t, net, dst_t)
        assert got is (mb.colour if dst_t is None else dst_t)
        for s in size_of:
            if out == 'source':
                g = outs[s].read() if pitched_out else mb.slot_output(mb.colour, s)
                assert torch.equal(g, ref.slot_output(want, s)), (k, s)
            elif pitched_out:
                assert torch.equal(dst[s].read(), want[s]), (k, s)
            else:
                assert torch.equal(mb.colour[s], want[s]), (k, s)
    for s in range(S):
        assert rect_or_none(lambda: mb.leave(s)) == rect_or_none(lambda: ref.leave(s)), s
    for a, b in ((mb.frames, ref.frames), (mb.masks, ref.masks), (mb.all_black, ref.all_black), (mb.cur, ref.cur)):
        assert torch.equal(a, b)
    assert all(sf.untouched_outside() for sf in src + outs if sf is not None)
    if out != 'source' and pitched_out:
        assert all(sf.untouched_outside() for sf in dst)


# ---- one captured graph over a rotating surface pool, with a re-join at another size between replays
@pytest.mark.parametrize('fmt,out,out_format,own_out', [('nv12', 'source', 'nv12', False), ('bgr', 'source', 'i420', True),
                                                         ('i420', (96, 160), 'bgr', False)])
def test_capture_planes_follows_rotating_surfaces(mgw, fmt, out, out_format, own_out):
    """eager = MixedStreamBatch.step on the packed pool.  At replay 6 slot 1 joins again at another size while its entries still
    name surfaces of the old size: for replays 6 and 7 the slot is idle (not a byte of its surfaces written; through the resize
    its destination entry is cleared as step_planes documents) and the other slots stay exact.  At replay 8 it joins again,
    its entries are set at the new size, and from then on it equals eager and its own StreamBatch at that size."""
    S, cap, h, w, K = 3, (150, 256), 48, 80, 3
    base = identity_mesh()
    net, _ = fake_net_batch(mgw, base)
    kw = dict(height=h, width=w, refine=2, src_format=fmt, out_size=out, out_format=out_format)
    eager, mb = mgw.MixedStreamBatch(S, cap, **kw), mgw.MixedStreamBatch(S, cap, **kw)
    gen = torch.Generator(device='cuda')
    gen.manual_seed(95)
    sizes = {0: (120, 200), 1: (96, 160), 2: cap}
    new_size = (150, 96)
    source = out == 'source'
    OH, OW = (None, None) if source else mb.out_size

    def surfaces_at(f, sz, seed):
        return [Surface(f, *sz, LAYOUTS[(seed + i) % 3]) for i in range(K)]       # K surfaces of one slot, rotating
    pool = {s: surfaces_at(fmt, sz, s) for s, sz in sizes.items()}
    outs = {s: surfaces_at(out_format, sz if source else (OH, OW), s + 1) for s, sz in sizes.items()}
    src_t = mgw.MixedPlaneTable(S, fmt, cap)
    if own_out:
        dst_t = None
    else:
        dst_t = mgw.MixedPlaneTable(S, out_format, cap) if source else mgw.PlaneTable(S, out_format, (OH, OW))
    cur_size = dict(sizes)                                                   # the size the slot's entries name

    def point(k, slots):
        for s in slots:
            src_t.set(s, pool[s][(k + s) % K].planes(), cur_size[s])
            if dst_t is not None:
                o = outs[s][(2 * k + s) % K].planes()
                if source:
                    dst_t.set(s, o, cur_size[s])
                else:
                    dst_t.set(s, o)

    packed = torch.zeros(eager.pool_shape, dtype=torch.uint8, device='cuda')
    for s, sz in sizes.items():
        first = frame(gen, fmt, *sz)
        mb.join(s, first); eager.join(s, first)
    point(0, range(S))
    graph = mb.capture_planes(src_t, net, dst_t)
    own = None
    for k in range(12):
        if k in (6, 8):
            first = frame(gen, fmt, *new_size)
            mb.join(1, first); eager.join(1, first)
            sizes[1] = new_size
            if k == 8:                                                        # re-join, set the new surfaces, then replay
                own = mgw.StreamBatch(1, new_size, height=h, width=w, refine=2, src_format=fmt,
                                      out_size=new_size if source else out, out_format=out_format)
                own.join(0, first)
        frames = {s: frame(gen, fmt, *sz) for s, sz in sizes.items()}
        src_t.uploaded.synchronize()                                           # the previous replay has copied the mirrors
        if dst_t is not None:
            dst_t.uploaded.synchronize()
        if k == 6:
            # slot 1's entries keep naming old-size surfaces: stale.  Through the resize the warp reads self.small, so the
            # destination entry is cleared to leave the slot's surface alone
            if not source and dst_t is not None:
                dst_t.clear(1)
            kept = [a.clone() for o in outs[1] for a in o.allocs]
            kept_row = mb.colour[1].clone()
        if k == 8:
            pool[1] = surfaces_at(fmt, new_size, 5)
            if source:
                outs[1] = surfaces_at(out_format, new_size, 6)
            cur_size[1] = new_size
        point(k, [0, 2] if k in (6, 7) else range(S))
        for s, f in frames.items():
            eager.slot_frame(packed, s).copy_(f)
            if k in (6, 7) and s == 1:
                continue                                                     # the decoder has no surface at the new size yet
            pool[s][(k + s) % K].write(f)
        graph.replay()
        want = eager.step(packed, net)
        torch.cuda.synchronize()
        for s in range(S):
            if own_out:
                got = mb.slot_output(mb.colour, s) if (s != 1 or k not in (6, 7)) else None
            else:
                got = outs[s][(2 * k + s) % K].read() if (s != 1 or k not in (6, 7)) else None
            ref = eager.slot_output(want, s) if source else want[s]
            if got is not None:
                assert torch.equal(got, ref), (k, s)
        if k in (6, 7):
            assert all(torch.equal(a, b) for a, b in zip((a for o in outs[1] for a in o.allocs), kept)), k    # not a byte written
            if own_out:
                # the batch's own output table follows the join to the new size: the stale source entry alone idles the slot
                assert torch.equal(mb.colour[1], kept_row), k
        if own is not None:
            o = own.step(eager.slot_frame(packed, 1)[None].contiguous(), net)[0]
            got = mb.slot_output(mb.colour, 1) if own_out else outs[1][(2 * k + 1) % K].read()
            assert torch.equal(got, o), k
    for a, b in ((mb.frames, eager.frames), (mb.masks, eager.masks), (mb.heads_dev, eager.heads_dev), (mb.all_black, eager.all_black)):
        assert torch.equal(a, b)
    for s in range(S):
        assert rect_or_none(lambda: mb.leave(s)) == rect_or_none(lambda: eager.leave(s))
    assert all(sf.untouched_outside() for o in list(outs.values()) + list(pool.values()) for sf in o)

"""GPU: videos of different source sizes in one batch, each stabilised at its own resolution (mgw_remap_bundle_frame_mixed,
MixedStreamBatch(out_size='source' | (OH, OW))).  Every comparison is bit-exact: each slot of the per-slot warp must equal the
uniform warp on that slot's frame alone, and each slot of a MixedStreamBatch its own StreamBatch at its own size."""
import numpy as np
import pytest
import torch

import remap_frame_ref as M
from test_gpu_streams import fake_net_batch, identity_mesh, rect_or_none

pytestmark = pytest.mark.gpu

FORMATS = ('bgr', 'nv12', 'i420')
SENTINEL = 0xA7


@pytest.fixture(scope='module')
def mgw():
    import dovs_b200
    assert torch.cuda.is_available(), 'GPU tests need a CUDA device; there is no CPU fallback'
    return dovs_b200


def frame_shape(fmt, H, W):
    return (H, W, 3) if fmt == 'bgr' else (H * 3 // 2, W)


def frame_bytes(fmt, H, W):
    return H * W * 3 if fmt == 'bgr' else H * W * 3 // 2


def random_frame(gen, fmt, H, W):
    """random bytes on the device: any bytes are a valid BGR or YUV 4:2:0 frame"""
    return torch.randint(0, 256, frame_shape(fmt, H, W), dtype=torch.uint8, device='cuda', generator=gen)


def maps(h, w, seed, wild):
    xm, ym = M.wild_mesh(h, w, seed) if wild else M.smooth_mesh(h, w, seed)
    return torch.stack([torch.as_tensor(np.ascontiguousarray(xm)), torch.as_tensor(np.ascontiguousarray(ym))], -1).cuda()


# ---- the call against the uniform call, slot by slot
SIZES_BGR = [(1080, 1920), (720, 1280), (1920, 1080), (576, 1024), (91, 157), (123, 77), (90, 166)]
SIZES_YUV = [(1080, 1920), (720, 1280), (1920, 1080), (576, 1024), (90, 158), (6, 10), (480, 854)]


@pytest.mark.parametrize('src_fmt', FORMATS)
@pytest.mark.parametrize('dst_fmt', FORMATS)
def test_mixed_warp_equals_uniform_warp(mgw, src_fmt, dst_fmt):
    """every active slot's bytes are the uniform call's on its frame alone; bytes past a slot's result, the regions of idle slots
    (size 0, above the capacity, odd with either format YUV) and the bytes past the pool keep the sentinel"""
    yuv = src_fmt != 'bgr' or dst_fmt != 'bgr'
    sizes = list(SIZES_YUV if yuv else SIZES_BGR)
    largest = (max(s[0] for s in sizes), max(s[1] for s in sizes))
    gen = torch.Generator(device='cuda')
    gen.manual_seed(70)
    for cap, (h, w) in ((largest, (288, 512)), ((largest[0] + 4, largest[1] + 6), (36, 64))):
        idle = [(0, 0), (0, 64), (cap[0] + 2, 64), (64, cap[1] + 2)] + ([(91, 128), (90, 127)] if yuv else [])
        all_sizes = sizes + idle
        S, fb, db = len(all_sizes), frame_bytes(src_fmt, *cap), frame_bytes(dst_fmt, *cap)
        pool = torch.randint(0, 256, (S, fb), dtype=torch.uint8, device='cuda', generator=gen)
        frames = [random_frame(gen, src_fmt, *sz) for sz in sizes]
        for s, f in enumerate(frames):
            pool[s, :f.numel()] = f.reshape(-1)
        xy = torch.stack([maps(h, w, 100 + s, wild=s % 2 == 1) for s in range(S)]).contiguous()
        sz = torch.tensor(all_sizes, dtype=torch.int32).cuda()
        slack = 4096
        flat = torch.full((S * db + slack,), SENTINEL, dtype=torch.uint8, device='cuda')
        out = flat[:S * db].view(S, db)
        got = mgw.ops.remap_bundle_frame_mixed(pool.view((S,) + frame_shape(src_fmt, *cap)), src_fmt, sz, xy, dst_fmt, out=out)
        assert got.data_ptr() == out.data_ptr() and tuple(got.shape) == (S, db)
        for s, f in enumerate(frames):
            want = mgw.ops.remap_bundle_frame(f[None].contiguous(), src_fmt, xy[s:s + 1].contiguous(), out_format=dst_fmt).reshape(-1)
            n = want.numel()
            assert torch.equal(out[s, :n], want), (src_fmt, dst_fmt, sizes[s], cap)
            assert bool((out[s, n:] == SENTINEL).all()), (src_fmt, dst_fmt, sizes[s], cap)
        for s in range(len(sizes), S):
            assert bool((out[s] == SENTINEL).all()), (src_fmt, dst_fmt, all_sizes[s], cap)
        assert bool((flat[S * db:] == SENTINEL).all())


# ---- MixedStreamBatch against one StreamBatch per video
class OwnBatch:
    """one video in a StreamBatch of one slot at its own size (the reference for one slot of a MixedStreamBatch)"""

    def __init__(self, mgw, first, fmt, size, out, out_format, h, w, refine, base):
        self.sb = mgw.StreamBatch(1, size, height=h, width=w, refine=refine, src_format=fmt,
                                  out_size=size if out == 'source' else out, out_format=out_format)
        self.sb.join(0, first)
        self.net, _ = fake_net_batch(mgw, base)

    def step(self, raw):
        return self.sb.step(raw[None].contiguous(), self.net)[0]


def run_against_own_batches(mgw, fmt, out, out_format, sizes_at, steps=8):
    """sizes_at: {step: {slot: size}} joins (a slot that joins again takes a new size); returns nothing, asserts every step"""
    cap, h, w, refine = (150, 256), 48, 80, 2
    base = identity_mesh()
    S = 5
    mb = mgw.MixedStreamBatch(S, cap, height=h, width=w, refine=refine, src_format=fmt, out_size=out, out_format=out_format)
    net, _ = fake_net_batch(mgw, base)
    gen = torch.Generator(device='cuda')
    gen.manual_seed(71)
    pool = torch.zeros(mb.pool_shape, device='cuda', dtype=torch.uint8)
    own, size_of = {}, {}
    for k in range(steps):
        for s, sz in sizes_at.get(k, {}).items():
            if s in own:
                assert rect_or_none(lambda: mb.leave(s)) == rect_or_none(lambda: own[s].sb.leave(0)), (k, s)
            first = random_frame(gen, fmt, *sz)
            mb.join(s, first)
            own[s], size_of[s] = OwnBatch(mgw, first, fmt, sz, out, out_format, h, w, refine, base), sz
        for s in own:
            mb.slot_frame(pool, s).copy_(random_frame(gen, fmt, *size_of[s]))
        colour = mb.step(pool, net)
        for s, o in own.items():
            want = o.step(mb.slot_frame(pool, s))
            got = mb.slot_output(colour, s) if out == 'source' else colour[s]
            assert torch.equal(got, want), (fmt, out, out_format, k, s, size_of[s])
    for s, o in own.items():
        assert rect_or_none(lambda: mb.leave(s)) == rect_or_none(lambda: o.sb.leave(0)), s


@pytest.mark.parametrize('fmt,out_format', [('bgr', 'bgr'), ('nv12', 'nv12'), ('i420', 'bgr')])
def test_source_size_output_equals_own_stream_batches(mgw, fmt, out_format):
    # slot 0: 120x200; slot 1: 96x160, then 150x96 portrait from step 4 (a re-join at another size); slot 2: the capacity
    # from step 1; slot 3: odd 91x157 (BGR only; 90x158 otherwise) from step 2; slot 4: idle
    odd = (91, 157) if fmt == 'bgr' and out_format == 'bgr' else (90, 158)
    run_against_own_batches(mgw, fmt, 'source', out_format,
                            {0: {0: (120, 200), 1: (96, 160)}, 1: {2: (150, 256)}, 2: {3: odd}, 4: {1: (150, 96)}})


@pytest.mark.parametrize('fmt,out_format', [('bgr', 'bgr'), ('nv12', 'i420')])
def test_common_output_size_equals_own_stream_batches(mgw, fmt, out_format):
    # slot 1 has the output's size (StreamBatch then reads the frame itself, the mixed batch resizes it 1:1), slot 2 is the
    # capacity (a downscale), slot 3 an upscale; slot 0 re-joins at another size
    run_against_own_batches(mgw, fmt, (96, 160), out_format,
                            {0: {0: (120, 200), 1: (96, 160), 2: (150, 256)}, 1: {3: (60, 100)}, 3: {0: (144, 240)}}, steps=6)


def test_common_output_at_the_capacity(mgw):
    """out_size equal to the capacity still resizes every slot (1:1 for a slot of the capacity's size)"""
    run_against_own_batches(mgw, 'bgr', (150, 256), 'bgr', {0: {0: (150, 256), 1: (96, 160)}}, steps=3)


# ---- graph replay
@pytest.mark.parametrize('fmt,out_format', [('nv12', 'nv12'), ('bgr', 'i420')])
def test_source_output_graph_replay_equals_eager(mgw, fmt, out_format):
    """one capture with the whole-pool upload and the whole-output-pool download inside the graph, replayed 10 times, with a slot
    re-joining at a new size and an idle slot joining between replays == the same schedule run eagerly, and the re-joined slot
    == its own StreamBatch at the new size"""
    S, cap, h, w = 3, (120, 200), 48, 80
    base = identity_mesh()
    net, _ = fake_net_batch(mgw, base)
    gen = torch.Generator(device='cuda')
    gen.manual_seed(72)
    kw = dict(height=h, width=w, refine=2, src_format=fmt, out_size='source', out_format=out_format)
    eager, graphed = mgw.MixedStreamBatch(S, cap, **kw), mgw.MixedStreamBatch(S, cap, **kw)
    host_in = torch.zeros(graphed.pool_shape, dtype=torch.uint8).pin_memory()
    host_out = torch.zeros(graphed.out_pool_shape, dtype=torch.uint8).pin_memory()
    pool_g = torch.zeros(graphed.pool_shape, device='cuda', dtype=torch.uint8)
    pool_e = torch.zeros(eager.pool_shape, device='cuda', dtype=torch.uint8)
    sizes = {0: (120, 200), 1: (72, 128)}
    for s, sz in sizes.items():
        first = random_frame(gen, fmt, *sz)
        eager.join(s, first); graphed.join(s, first)
    graph = graphed.capture(pool_g, net, upload_from=host_in, download_to=host_out)
    own = None
    for k in range(10):
        if k in (3, 6):
            s, sz = (1, (100, 60)) if k == 3 else (2, (60, 100))
            first = random_frame(gen, fmt, *sz)
            eager.join(s, first); graphed.join(s, first)
            sizes[s] = sz
            if s == 1:
                own = OwnBatch(mgw, first, fmt, sz, 'source', out_format, h, w, 2, base)
        for s, sz in sizes.items():
            graphed.slot_frame(host_in, s).copy_(random_frame(gen, fmt, *sz).cpu())
        graph.replay()
        torch.cuda.synchronize()
        pool_e.copy_(host_in)
        colour = eager.step(pool_e, net)
        for s in sizes:
            assert torch.equal(graphed.slot_output(host_out, s).cuda(), eager.slot_output(colour, s)), (k, s)
        if own is not None:
            assert torch.equal(graphed.slot_output(host_out, 1).cuda(), own.step(eager.slot_frame(pool_e, 1))), k
    for a, b in ((eager.frames, graphed.frames), (eager.masks, graphed.masks), (eager.heads_dev, graphed.heads_dev),
                 (eager.all_black, graphed.all_black), (eager.in_x, graphed.in_x)):
        assert torch.equal(a, b)
    for s in range(S):
        assert rect_or_none(lambda: eager.leave(s)) == rect_or_none(lambda: graphed.leave(s))


# ---- Python-level errors
def test_errors(mgw):
    for bad in ('src', (0, 64), (64, 32768)):
        with pytest.raises(ValueError):
            mgw.MixedStreamBatch(2, (96, 160), height=24, width=40, out_size=bad)
    yb = mgw.MixedStreamBatch(2, (96, 160), height=24, width=40, out_size='source', out_format='nv12')
    with pytest.raises(ValueError):
        yb.join(0, torch.zeros((91, 160, 3), device='cuda', dtype=torch.uint8))        # odd size with a YUV result
    with pytest.raises(ValueError):
        yb.join(0, torch.zeros((96, 159, 3), device='cuda', dtype=torch.uint8))
    yb.join(0, torch.zeros((90, 158, 3), device='cuda', dtype=torch.uint8))
    assert tuple(yb.slot_output(yb.colour, 0).shape) == (135, 158)
    net, _ = fake_net_batch(mgw, identity_mesh())
    pool = torch.zeros(yb.pool_shape, device='cuda', dtype=torch.uint8)
    for bad in (torch.empty((2, 24, 40, 3), dtype=torch.uint8).pin_memory(),
                torch.empty((2, 96 * 160 * 3), dtype=torch.uint8).pin_memory()):
        with pytest.raises(ValueError):
            yb.capture(pool, net, download_to=bad)
    with pytest.raises(ValueError):
        yb.slot_output(torch.zeros((2, 10), dtype=torch.uint8), 0)
    # the op: a YUV result needs an even capacity, xy must match the pool, out must be the output pool
    sz = torch.zeros((2, 2), device='cuda', dtype=torch.int32)
    xy = torch.zeros((2, 24, 40, 2), device='cuda')
    odd = torch.zeros((2, 97, 160, 3), device='cuda', dtype=torch.uint8)
    with pytest.raises(ValueError):
        mgw.ops.remap_bundle_frame_mixed(odd, 'bgr', sz, xy, 'i420')
    with pytest.raises(ValueError):
        mgw.ops.remap_bundle_frame_mixed(odd, 'bgr', sz, xy[:1], 'bgr')
    with pytest.raises(ValueError):
        mgw.ops.remap_bundle_frame_mixed(odd, 'bgr', sz, xy, 'bgr', out=torch.zeros((2, 10), device='cuda', dtype=torch.uint8))
    n0 = mgw.launch_count()
    assert mgw.ops.remap_bundle_frame_mixed(odd, 'bgr', sz, xy, 'bgr').shape == (2, 97 * 160 * 3)   # idle slots: one K5a + K5b
    assert mgw.launch_count() == n0 + 2
    empty = torch.zeros((0, 96, 160, 3), device='cuda', dtype=torch.uint8)
    n0 = mgw.launch_count()
    assert mgw.ops.remap_bundle_frame_mixed(empty, 'bgr', sz[:0], xy[:0], 'nv12').shape == (0, 96 * 160 * 3 // 2)
    assert mgw.launch_count() == n0

"""GPU: the exact-bytes transfer of a pool of per-slot frames (mgw_copy_slots_mixed, ops.copy_slots_mixed) and
MixedStreamBatch.capture(exact_bytes=True).  Every comparison is bit-exact, and every byte the copy must not touch is checked
against a sentinel."""
import pytest
import torch

from test_gpu_mixed_out import frame_bytes, frame_shape, random_frame
from test_gpu_streams import fake_net_batch, identity_mesh, rect_or_none

pytestmark = pytest.mark.gpu

SENTINEL = 0x5C
SLACK = 4096


@pytest.fixture(scope='module')
def mgw():
    import dovs_b200
    assert torch.cuda.is_available(), 'GPU tests need a CUDA device; there is no CPU fallback'
    return dovs_b200


def pool_view(fmt, S, cap):
    return (S,) + frame_shape(fmt, *cap)


def buffer(where, shape, fill=None, gen=None):
    """a pool-shaped uint8 buffer at the start of a larger one ('host' = pinned, 'dev'), and the larger one: the bytes past the
    pool show an overrun"""
    n = 1
    for d in shape:
        n *= d
    if fill is None:
        flat = torch.randint(0, 256, (n + SLACK,), dtype=torch.uint8, device='cuda', generator=gen)
    else:
        flat = torch.full((n + SLACK,), fill, dtype=torch.uint8, device='cuda')
    if where == 'host':
        flat = flat.cpu().pin_memory()
    return flat[:n].view(shape), flat


def slot_sizes(fmt, cap):
    """active sizes from the smallest frame to the capacity (odd widths for BGR), then idle ones: size 0, above the capacity,
    odd with YUV"""
    H, W = cap
    if fmt == 'bgr':
        active = [(1, 1), (1, W), (H, 1), (33, 65), (H, W), (50, 101), (H - 1, W - 2)]
        idle = [(0, 0), (0, 5), (H + 1, 10), (10, W + 1)]
    else:
        active = [(2, 2), (2, W), (H, 2), (40, 66), (H, W), (50, 102), (H - 2, W - 4)]
        idle = [(0, 0), (0, 4), (H + 2, 4), (4, W + 2), (3, 4), (4, 5), (5, 5)]
    sizes = active + idle
    order = [4, 9, 0, 6, 10, 1, 2, 7, 3, 5, 8] + list(range(11, len(sizes)))        # active and idle slots interleaved
    return [sizes[i] for i in order], len(active)


CAPACITIES = {'bgr': [(97, 127), (96, 128)], 'nv12': [(96, 130), (98, 130)], 'i420': [(96, 130), (98, 130)]}


@pytest.mark.parametrize('direction', ['h2d', 'd2h', 'd2d'])
@pytest.mark.parametrize('fmt', ['bgr', 'nv12', 'i420'])
def test_copy_moves_exactly_each_active_slots_bytes(mgw, direction, fmt):
    """each active slot's first frame_bytes(size) bytes arrive; every other byte of dst, and past it, keeps the sentinel.  Of the
    two capacities one has a stride that is a multiple of 16 and one does not, so slots start at every misalignment"""
    gen = torch.Generator(device='cuda')
    gen.manual_seed(80)
    src_where, dst_where = {'h2d': ('host', 'dev'), 'd2h': ('dev', 'host'), 'd2d': ('dev', 'dev')}[direction]
    strides = set()
    for cap in CAPACITIES[fmt]:
        sizes, _ = slot_sizes(fmt, cap)
        S, stride = len(sizes), frame_bytes(fmt, *cap)
        strides.add(stride % 16 == 0)
        src, _ = buffer(src_where, pool_view(fmt, S, cap), gen=gen)
        dst, dst_flat = buffer(dst_where, pool_view(fmt, S, cap), fill=SENTINEL)
        sz = torch.tensor(sizes, dtype=torch.int32, device='cuda')
        n0 = mgw.launch_count()
        assert mgw.ops.copy_slots_mixed(src, dst, fmt, sz) is dst
        assert mgw.launch_count() == n0 + 1
        torch.cuda.synchronize()
        got, want = dst_flat.cpu(), src.reshape(S, stride).cpu()
        rows = got[:S * stride].view(S, stride)
        for s, (H, W) in enumerate(sizes):
            active = 0 < H <= cap[0] and 0 < W <= cap[1] and (fmt == 'bgr' or (H % 2 == 0 and W % 2 == 0))
            n = frame_bytes(fmt, H, W) if active else 0
            assert torch.equal(rows[s, :n], want[s, :n]), (direction, fmt, cap, (H, W))
            assert bool((rows[s, n:] == SENTINEL).all()), (direction, fmt, cap, (H, W))
        assert bool((got[S * stride:] == SENTINEL).all())
    assert strides == {True, False}


def test_pageable_memory_is_refused_before_a_launch(mgw):
    """the pointer reaches the argument check only: nothing is launched, so nothing touches it"""
    lib = mgw._lib.lib
    S, cap = 2, (96, 128)
    dev = torch.zeros((S, 96 * 128 * 3), dtype=torch.uint8, device='cuda')
    pageable = torch.zeros((S, 96 * 128 * 3), dtype=torch.uint8)
    pinned = torch.zeros((S, 96 * 128 * 3), dtype=torch.uint8).pin_memory()
    sz = torch.tensor([[96, 128], [10, 10]], dtype=torch.int32, device='cuda')
    assert pageable.data_ptr() % 16 == 0
    st = torch.cuda.current_stream().cuda_stream
    n0 = lib.mgw_launch_count()
    for src, dst in ((pageable, dev), (dev, pageable), (pinned, pageable), (pageable, pinned)):
        assert lib.mgw_copy_slots_mixed(src.data_ptr(), dst.data_ptr(), 0, S, cap[0], cap[1], sz.data_ptr(), st) == -1
        assert b'pageable' in lib.mgw_last_error()
    assert lib.mgw_launch_count() == n0
    with pytest.raises(ValueError, match='pageable'):
        mgw.ops.copy_slots_mixed(pageable.view(S, 96, 128, 3), dev.view(S, 96, 128, 3), 'bgr', sz)
    assert lib.mgw_launch_count() == n0


def test_capture_in_the_default_global_mode(mgw):
    """the pointer check runs while a stream is captured in torch's default (global) mode, and the replayed copy follows the
    sizes and the bytes of each replay"""
    fmt, cap, S = 'nv12', (96, 130), 3
    gen = torch.Generator(device='cuda')
    gen.manual_seed(81)
    src, _ = buffer('host', pool_view(fmt, S, cap), gen=gen)
    dst, _ = buffer('dev', pool_view(fmt, S, cap), fill=SENTINEL)
    sz = torch.tensor([[96, 130], [0, 0], [40, 66]], dtype=torch.int32, device='cuda')
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, capture_error_mode='global'):
        mgw.ops.copy_slots_mixed(src, dst, fmt, sz)
    stride = frame_bytes(fmt, *cap)
    for sizes in ([[96, 130], [0, 0], [40, 66]], [[20, 30], [96, 130], [40, 66]]):
        sz.copy_(torch.tensor(sizes, dtype=torch.int32))
        src.copy_(torch.randint(0, 256, src.shape, dtype=torch.uint8, device='cuda', generator=gen).cpu())
        dst.fill_(SENTINEL)
        g.replay()
        torch.cuda.synchronize()
        got, want = dst.reshape(S, stride).cpu(), src.reshape(S, stride)
        for s, (H, W) in enumerate(sizes):
            n = frame_bytes(fmt, H, W)
            assert torch.equal(got[s, :n], want[s, :n]) and bool((got[s, n:] == SENTINEL).all()), (sizes, s)


# ---- MixedStreamBatch.capture(exact_bytes=True): the same schedule eagerly, with the whole-pool graph, with the exact one
CASES = [('bgr', 'source', 'bgr'), ('nv12', 'source', 'nv12'), ('i420', 'source', 'bgr'), ('bgr', None, 'bgr'),
         ('nv12', (60, 100), 'i420')]


@pytest.mark.parametrize('fmt,out,out_format', CASES)
def test_exact_bytes_graph_replay_equals_eager_and_whole_pool(mgw, fmt, out, out_format):
    S, cap, h, w, refine = 4, (120, 200), 48, 80, 2
    yuv = fmt != 'bgr' or out_format != 'bgr'
    net, _ = fake_net_batch(mgw, identity_mesh())
    gen = torch.Generator(device='cuda')
    gen.manual_seed(82)
    kw = dict(height=h, width=w, refine=refine, src_format=fmt, out_size=out, out_format=out_format)
    eager, exact, whole = (mgw.MixedStreamBatch(S, cap, **kw) for _ in range(3))
    host_in = torch.zeros(exact.pool_shape, dtype=torch.uint8).pin_memory()
    out_shape = tuple(exact.colour.shape)
    out_x = torch.full(out_shape, SENTINEL, dtype=torch.uint8).pin_memory()
    out_w = torch.zeros(out_shape, dtype=torch.uint8).pin_memory()
    pool_e = torch.zeros(eager.pool_shape, device='cuda', dtype=torch.uint8)
    pool_x = torch.full(exact.pool_shape, SENTINEL, device='cuda', dtype=torch.uint8)
    pool_w = torch.zeros(whole.pool_shape, device='cuda', dtype=torch.uint8)
    batches = (eager, exact, whole)

    def join(s, size):
        first = random_frame(gen, fmt, *size)
        for b in batches:
            b.join(s, first)

    sizes = {0: (120, 200), 1: (72, 128)}
    for s, size in sizes.items():
        join(s, size)
    g_x = exact.capture(pool_x, net, upload_from=host_in, download_to=out_x, exact_bytes=True)
    g_w = whole.capture(pool_w, net, upload_from=host_in, download_to=out_w)
    # slot 1 re-joins at a new size, idle slot 2 joins, slot 0 leaves (and keeps running), slot 3 stays idle
    rejoin, late = ((100, 60), (60, 100)) if yuv else ((101, 61), (61, 99))
    up_extent, down_extent = [0] * S, [0] * S
    for k in range(10):
        if k == 3:
            join(1, rejoin); sizes[1] = rejoin
        if k == 5:
            join(2, late); sizes[2] = late
        if k == 7:
            rects = [rect_or_none(lambda: b.leave(0)) for b in batches]
            assert rects[0] == rects[1] == rects[2], rects
        for s, size in sizes.items():
            exact.slot_frame(host_in, s).copy_(random_frame(gen, fmt, *size).cpu())
            up_extent[s] = max(up_extent[s], frame_bytes(fmt, *size))
            down_extent[s] = max(down_extent[s], frame_bytes(out_format, *size))
        g_x.replay()
        g_w.replay()
        torch.cuda.synchronize()
        pool_e.copy_(host_in)
        colour = eager.step(pool_e, net)
        for s in sizes:
            want = eager.slot_output(colour, s) if out == 'source' else colour[s]
            got_x = exact.slot_output(out_x, s) if out == 'source' else out_x[s]
            got_w = whole.slot_output(out_w, s) if out == 'source' else out_w[s]
            assert torch.equal(got_x.cuda(), want) and torch.equal(got_w.cuda(), want), (fmt, out, out_format, k, s)
            assert torch.equal(exact.slot_frame(pool_x, s), eager.slot_frame(pool_e, s)), (k, s)
        # what the exact transfers must not touch: past each slot's largest frame so far, and the idle slot's rows
        px = pool_x.cpu()
        for s in range(S):
            assert bool((px[s, up_extent[s]:] == SENTINEL).all()), ('pool', k, s)
            if out == 'source':
                assert bool((out_x[s, down_extent[s]:] == SENTINEL).all()), ('host output pool', k, s)
    for a, b, c in zip(*((bt.frames, bt.masks, bt.heads_dev, bt.all_black, bt.in_x) for bt in batches)):
        assert torch.equal(a, b) and torch.equal(a, c)
    for s in range(S):
        rects = [rect_or_none(lambda: bt.leave(s)) for bt in batches]
        assert rects[0] == rects[1] == rects[2], (s, rects)


def test_exact_bytes_capture_errors(mgw):
    mb = mgw.MixedStreamBatch(2, (96, 160), height=24, width=40, out_size='source')
    net, _ = fake_net_batch(mgw, identity_mesh())
    pool = torch.zeros(mb.pool_shape, device='cuda', dtype=torch.uint8)
    for bad in (torch.zeros(mb.pool_shape, device='cuda', dtype=torch.uint8), torch.zeros(mb.pool_shape, dtype=torch.uint8)):
        with pytest.raises(ValueError, match='pinned'):
            mb.capture(pool, net, upload_from=bad, exact_bytes=True)
    with pytest.raises(ValueError, match='upload_from must be'):
        mb.capture(pool, net, upload_from=torch.zeros((2, 10), dtype=torch.uint8).pin_memory(), exact_bytes=True)
    with pytest.raises(ValueError, match='download_to must be'):
        mb.capture(pool, net, download_to=torch.zeros((2, 10), dtype=torch.uint8).pin_memory(), exact_bytes=True)

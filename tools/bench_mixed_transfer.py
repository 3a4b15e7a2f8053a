"""Exact-bytes transfers for a MixedStreamBatch: the per-slot copy kernel (mgw_copy_slots_mixed, ops.copy_slots_mixed) that
moves each slot's own frame bytes across PCIe, against the copy engine's whole-pool copies.  S = 64, BGR, network 288x512,
refine = 1, arms alternated in rounds in one process.
  1 copy:    the copy alone, CUDA events around --calls back-to-back calls.  (i) 64 x 1080p at a 1080p capacity, every slot
             full, so both arms move the same bytes: the kernel against cudaMemcpyAsync of the same pool (torch copy_ from / to
             pinned memory), host to device and device to host, in GB/s.  (ii) bench_mixed.py's workloads 2 and 3: the kernel
             on each slot's bytes against the whole-pool DMA, both directions.
  2 network: host to host at the network's output size, bench_mixed.py's legs (b) fixed mesh and (c) StabNet carrier, for
             workloads 2 and 3: the mixed batch with the whole-pool upload, with exact_bytes=True, and the per-size batches.
  3 source:  host to host (b) at out_size='source' (bench_mixed_fullres.py), workloads 2 and 3, the same three arms: the
             exact-bytes arm moves each slot's frame both ways.
Prints one JSON object (the GPU's name and power limit included); --out also writes it to a file."""
import argparse, json, os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, 'oracle')); sys.path.insert(0, os.path.join(ROOT, 'tools'))
import numpy as np, torch
import dovs_b200 as mgw
import bench_mixed as bm
import bench_mixed_fullres as bf
from bench_streams import gpu_info

dev = 'cuda'
WORKLOADS = {'2': ('2_few_sizes', bm.FEW, (1920, 1920)), '3': ('3_fragmented_16_sizes', bm.FRAGMENTED, (2160, 3840))}


def frame_bytes(H, W):
    return 3 * H * W


def back_to_back(fn, calls):
    """CUDA-event time of one call, from `calls` calls in a row (after 3 warm-up calls), in us"""
    for _ in range(3):
        fn()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(calls):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) * 1e3 / calls


def copy_alone(sizes, cap, calls, rounds):
    """kernel (each slot's bytes) and DMA (the whole pool) in both directions between a pinned host pool and a device pool"""
    S = len(sizes)
    shape = (S, cap[0], cap[1], 3)
    host = torch.randint(0, 256, shape, dtype=torch.uint8).pin_memory()
    pool = torch.zeros(shape, dtype=torch.uint8, device=dev)
    sz = torch.tensor(sizes, dtype=torch.int32, device=dev)
    arms = {'kernel_h2d': lambda: mgw.ops.copy_slots_mixed(host, pool, 'bgr', sz),
            'dma_h2d': lambda: pool.copy_(host, non_blocking=True),
            'kernel_d2h': lambda: mgw.ops.copy_slots_mixed(pool, host, 'bgr', sz),
            'dma_d2h': lambda: host.copy_(pool, non_blocking=True)}
    ts = {k: [] for k in arms}
    for _ in range(rounds):
        for k, fn in arms.items():
            ts[k].append(back_to_back(fn, calls))
    exact, whole = sum(frame_bytes(*s) for s in sizes), host.numel()
    out = {'slots': S, 'capacity': list(cap), 'bytes_exact': exact, 'bytes_whole_pool': whole, 'calls_per_timing': calls}
    for k, t in ts.items():
        us = float(np.median(t))
        moved = exact if k.startswith('kernel') else whole
        out[k] = {'us_per_call': us, 'bytes': moved, 'GB_per_s': moved / us / 1e3, 'us_per_round': t}
    for d in ('h2d', 'd2h'):
        out['kernel_over_dma_time_' + d] = out['kernel_' + d]['us_per_call'] / out['dma_' + d]['us_per_call']
    del host, pool
    torch.cuda.empty_cache()
    return out


class ExactNet:
    """the mixed batch of a bench_mixed.Mixed arm, captured with exact_bytes=True (same buffers, another graph)"""

    def __init__(self, mixed, sizes):
        self.m, self.S = mixed, mixed.S
        self.h2d_bytes = sum(frame_bytes(*s) for s in sizes)

    def graph(self, net, io):
        kw = dict(upload_from=self.m.pool_h, download_to=self.m.out_h, exact_bytes=True) if io else {}
        return [self.m.mb.capture(self.m.pool_d, net(self.m.mb), **kw)]


class ExactSource(ExactNet):
    """the same for a bench_mixed_fullres.Mixed arm (out_size='source'): each slot's frame up and its result down"""

    def __init__(self, mixed, sizes):
        super().__init__(mixed, sizes)
        self.d2h_bytes = self.h2d_bytes


def ratios(r, keys):
    per = r['per_size_stream_batches']
    return {arm: {k: r[arm][k]['frames_per_s'] / per[k]['frames_per_s'] for k in keys} for arm in ('mixed_whole_pool', 'mixed_exact_bytes')}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--calls', type=int, default=50, help='back-to-back calls per copy timing')
    ap.add_argument('--reps', type=int, default=100, help='timed replays per host-to-host measurement (StabNet takes a sixth, '
                                                          'source resolution a quarter)')
    ap.add_argument('--rounds', type=int, default=3)
    ap.add_argument('--parts', default='1,2,3')
    ap.add_argument('--workloads', default='2,3')
    ap.add_argument('--out')
    a = ap.parse_args()
    assert torch.cuda.is_available(), 'bench_mixed_transfer.py measures on the GPU; there is nothing to measure without one'
    torch.backends.cudnn.benchmark = True
    rs = np.random.RandomState(0)
    gen = torch.Generator(device=dev)
    gen.manual_seed(0)
    torch.manual_seed(0)
    res = {'gpu': gpu_info(), 'source': 'BGR uint8', 'network_size': '%dx%d' % (bm.h, bm.w), 'refine': 1, 'S': 64,
           'method': 'arms alternated in rounds in one process; copy: median over rounds of the CUDA-event time of --calls '
                     'back-to-back calls; host to host: bench_mixed.py / bench_mixed_fullres.py legs, percentiles over all rounds',
           'calls': a.calls, 'reps': a.reps, 'rounds': a.rounds,
           '1_copy_alone': {}, '2_host_to_host_network_size': {}, '3_host_to_host_source_size': {}}
    parts, todo = set(a.parts.split(',')), [k for k in a.workloads.split(',') if k in WORKLOADS]

    def emit(final=False):
        if final:
            print(json.dumps(res, indent=1))
        if a.out:
            with open(a.out, 'w') as f:
                json.dump(res, f, indent=1)
    if '1' in parts:
        res['1_copy_alone']['64x1080p_full_slots'] = copy_alone([(1080, 1920)] * 64, (1080, 1920), a.calls, a.rounds)
        emit()
        for k in todo:
            name, groups, cap = WORKLOADS[k]
            res['1_copy_alone'][name] = copy_alone([sz for sz, n in groups for _ in range(n)], cap, a.calls, a.rounds)
            emit()
    model = mgw.StabNet(in_ch=13, grid=(4, 4)).to(dev).eval().to(memory_format=torch.channels_last) if '2' in parts else None
    for k in todo:
        name, groups, cap = WORKLOADS[k]
        sizes = [sz for sz, n in groups for _ in range(n)]
        if '2' in parts:
            mixed = bm.Mixed(groups, cap, rs)
            arms = {'mixed_whole_pool': mixed, 'mixed_exact_bytes': ExactNet(mixed, sizes), 'per_size_stream_batches': bm.PerSize(groups, rs)}
            r = bm.workload(name, arms, ('b', 'c'), model, a.rounds, a.reps)
            r['over_per_size_frames_per_s'] = ratios(r, ('b_host_to_host_fixed_mesh', 'c_host_to_host_stabnet'))
            r['capacity'] = list(cap)
            res['2_host_to_host_network_size'][name] = r
            emit()
            del arms, mixed
            torch.cuda.empty_cache()
        if '3' in parts:
            mixed = bf.Mixed(groups, cap, 'bgr', 'bgr', gen)
            arms = {'mixed_whole_pool': mixed, 'mixed_exact_bytes': ExactSource(mixed, sizes),
                    'per_size_stream_batches': bf.PerSize(groups, 'bgr', 'bgr', gen)}
            r = bf.workload(name, arms, ('b',), a.rounds, a.reps)
            r['over_per_size_frames_per_s'] = ratios(r, ('b_host_to_host_fixed_mesh',))
            r['capacity'] = list(cap)
            res['3_host_to_host_source_size'][name] = r
            emit()
            del arms, mixed
            torch.cuda.empty_cache()
    emit(final=True)


if __name__ == '__main__':
    main()

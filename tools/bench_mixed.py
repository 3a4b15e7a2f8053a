"""Videos of different source sizes in one batch: deploy.MixedStreamBatch against one StreamBatch per distinct size, S = 64 streams.

The bench_streams.py method: one CUDA graph per step (per batch), refine = 1, arms timed alternately in rounds in one process.
  (a) device time of one step with the frames resident on the device and a fixed mesh in place of the network (the library's
      share of a step); the per-size arm replays its graphs back to back between the two events;
  (b) host-to-host time per step with the upload and the download inside the graphs (pinned host buffers), fixed mesh: the mixed
      batch uploads its whole pool (capacity bytes per slot), the per-size batches exactly their frames;
  (c) the same with the StabNet carrier (torch / cuDNN ResNet-50, random init, fp32) as the network, in frames/s.
Workloads (BGR sources, network 288x512):
  1 overhead:   64 x 1080p; MixedStreamBatch at capacity 1080p and 2160p against StreamBatch(64, 1080p); (a) only;
  2 few sizes:  24 x 1080p, 24 x 720p, 8 x 480x854, 8 x 1920x1080 (portrait), capacity 1920x1920; (a), (b), (c);
  3 fragmented: 16 sizes x 4 streams from 240x426 (upscaled to the network size) to 2160x3840, capacity 2160x3840; (a), (b), (c).
Prints one JSON object (the GPU's name and power limit included); --out also writes it to a file."""
import argparse, json, os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, 'oracle')); sys.path.insert(0, os.path.join(ROOT, 'tools'))
import numpy as np, torch
import dovs_b200 as mgw
from bench_streams import dev_time, fixed_mesh_net, gpu_info, host_times, stabnet_net, summary

dev = 'cuda'
h, w = 288, 512

FEW = [((1080, 1920), 24), ((720, 1280), 24), ((480, 854), 8), ((1920, 1080), 8)]
FRAGMENTED = [((H, W), 4) for H, W in [(240, 426), (270, 480), (360, 640), (480, 640), (480, 854), (540, 960), (576, 1024), (640, 360),
                                       (720, 1280), (960, 540), (1080, 1080), (1080, 1440), (1080, 1920), (1280, 720), (1440, 2560),
                                       (2160, 3840)]]


def rand_frame(rs, H, W):
    return torch.as_tensor(rs.randint(0, 256, (H, W, 3)).astype(np.uint8))


class Mixed:
    """one MixedStreamBatch holding every stream of a workload"""

    def __init__(self, groups, cap, rs):
        sizes = [sz for sz, n in groups for _ in range(n)]
        self.S = len(sizes)
        self.mb = mgw.MixedStreamBatch(self.S, cap, height=h, width=w, refine=1)
        self.pool_h = torch.zeros(self.mb.pool_shape, dtype=torch.uint8).pin_memory()
        for s, sz in enumerate(sizes):
            self.mb.join(s, rand_frame(rs, *sz).to(dev))
            self.mb.slot_frame(self.pool_h, s).copy_(rand_frame(rs, *sz))
        self.pool_d = self.pool_h.to(dev)
        self.out_h = torch.empty((self.S, h, w, 3), dtype=torch.uint8).pin_memory()
        self.h2d_bytes = self.pool_h.numel()

    def graph(self, net, io):
        kw = dict(upload_from=self.pool_h, download_to=self.out_h) if io else {}
        return [self.mb.capture(self.pool_d, net(self.mb), **kw)]


class PerSize:
    """one StreamBatch per distinct size, their graphs replayed back to back"""

    def __init__(self, groups, rs):
        self.S = sum(n for _, n in groups)
        self.parts = []
        for (H, W), n in groups:
            sb = mgw.StreamBatch(n, (H, W), height=h, width=w, refine=1)
            for s in range(n):
                sb.join(s, rand_frame(rs, H, W).to(dev))
            raw_h = torch.stack([rand_frame(rs, H, W) for _ in range(n)]).pin_memory()
            self.parts.append((sb, raw_h, raw_h.to(dev), torch.empty((n, h, w, 3), dtype=torch.uint8).pin_memory()))
        self.h2d_bytes = sum(p[1].numel() for p in self.parts)

    def graph(self, net, io):
        return [sb.capture(raw_d, net(sb), **(dict(upload_from=raw_h, download_to=out_h) if io else {}))
                for sb, raw_h, raw_d, out_h in self.parts]


def replay_all(graphs):
    def fn():
        for g in graphs:
            g.replay()
    return fn


def alternate(arms, legs, rounds, reps):
    """arms: name -> {leg: graphs}; per round and leg every arm in turn.  (a) device time of the step, (b)/(c) host-to-host"""
    res = {name: {leg: [] for leg in legs} for name in arms}
    for _ in range(rounds):
        for leg in legs:
            for name, graphs in arms.items():
                fn = replay_all(graphs[leg])
                if leg == 'a':
                    res[name][leg].append(dev_time(fn, reps))
                else:
                    res[name][leg].append(host_times(fn, reps if leg == 'b' else max(reps // 6, 20)))
    out = {}
    for name, r in res.items():
        S = arms[name]['S']
        o = {}
        if 'a' in r:
            a = float(np.median(r['a']))
            o.update(a_us_device_step_fixed_mesh_resident=a, a_us_device_per_frame=a / S, a_us_per_round=r['a'])
        for leg, key in (('b', 'b_host_to_host_fixed_mesh'), ('c', 'c_host_to_host_stabnet')):
            if leg in r:
                o[key] = summary([t for ts in r[leg] for t in ts], S)
                o[key]['us_p50_per_round'] = [float(np.percentile(ts, 50)) for ts in r[leg]]
        out[name] = o
    return out


def workload(name, arms, legs, model, rounds, reps):
    graphs = {}
    with torch.no_grad():
        for arm_name, arm in arms.items():
            g = {'S': arm.S}
            if 'a' in legs:
                g['a'] = arm.graph(fixed_mesh_net, False)
            if 'b' in legs:
                g['b'] = arm.graph(fixed_mesh_net, True)
            if 'c' in legs:
                g['c'] = arm.graph(lambda sb: stabnet_net(model), True)
            graphs[arm_name] = g
        r = alternate(graphs, legs, rounds, reps)
    for arm_name, arm in arms.items():
        r[arm_name]['bytes_pcie_per_frame'] = {'h2d': arm.h2d_bytes / arm.S, 'd2h_colour': h * w * 3,
                                               'total': arm.h2d_bytes / arm.S + h * w * 3}
    print(json.dumps({name: r}), file=sys.stderr)
    return r


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--reps', type=int, default=200, help='timed replays per measurement (the StabNet leg takes a sixth)')
    ap.add_argument('--rounds', type=int, default=5)
    ap.add_argument('--workloads', default='1,2,3')
    ap.add_argument('--out')
    a = ap.parse_args()
    assert torch.cuda.is_available(), 'bench_mixed.py measures on the GPU; there is nothing to measure without one'
    torch.backends.cudnn.benchmark = True
    rs = np.random.RandomState(0)
    torch.manual_seed(0)
    model = mgw.StabNet(in_ch=13, grid=(4, 4)).to(dev).eval().to(memory_format=torch.channels_last)
    res = {'gpu': gpu_info(), 'source': 'BGR uint8', 'network_size': '%dx%d' % (h, w), 'refine': 1, 'S': 64,
           'method': 'one CUDA graph per batch and step; arms alternated in rounds of --reps replays; (a) median of the per-round '
                     'medians, (b)/(c) percentiles over all rounds', 'reps': a.reps, 'rounds': a.rounds, 'workloads': {}}
    todo = set(a.workloads.split(','))

    def emit(final=False):
        """the result so far (after every workload, so that an interrupted run keeps what it measured)"""
        out = dict(res, workloads=dict(res['workloads']))
        for k in ('1_overhead_64x1080p', '2_few_sizes', '3_fragmented_16_sizes'):
            out['workloads'].setdefault(k, 'not measured')
        if final:
            print(json.dumps(out, indent=1))
        if a.out:
            with open(a.out, 'w') as f:
                json.dump(out, f, indent=1)
    if '1' in todo:
        groups = [((1080, 1920), 64)]
        arms = {'mixed_capacity_1080p': Mixed(groups, (1080, 1920), rs), 'mixed_capacity_2160p': Mixed(groups, (2160, 3840), rs),
                'stream_batch_1080p': PerSize(groups, rs)}
        res['workloads']['1_overhead_64x1080p'] = workload('1', arms, ('a',), model, a.rounds, a.reps)
        res['workloads']['1_overhead_64x1080p']['legs_not_measured'] = ['b', 'c']
        emit()
        del arms
        torch.cuda.empty_cache()
    for key, groups, cap in (('2', FEW, (1920, 1920)), ('3', FRAGMENTED, (2160, 3840))):
        if key not in todo:
            continue
        arms = {'mixed': Mixed(groups, cap, rs), 'per_size_stream_batches': PerSize(groups, rs)}
        r = workload(key, arms, ('a', 'b', 'c'), model, a.rounds, a.reps)
        r['groups'] = [{'size': list(sz), 'streams': n} for sz, n in groups]
        r['capacity'] = list(cap)
        r['per_size_graphs'] = len(groups)
        mix, per = r['mixed'], r['per_size_stream_batches']
        r['mixed_over_per_size'] = {
            'a_device_step': mix['a_us_device_step_fixed_mesh_resident'] / per['a_us_device_step_fixed_mesh_resident'],
            'b_frames_per_s': mix['b_host_to_host_fixed_mesh']['frames_per_s'] / per['b_host_to_host_fixed_mesh']['frames_per_s'],
            'c_frames_per_s': mix['c_host_to_host_stabnet']['frames_per_s'] / per['c_host_to_host_stabnet']['frames_per_s'],
            'h2d_bytes': mix['bytes_pcie_per_frame']['h2d'] / per['bytes_pcie_per_frame']['h2d']}
        res['workloads'][{'2': '2_few_sizes', '3': '3_fragmented_16_sizes'}[key]] = r
        emit()
        del arms
        torch.cuda.empty_cache()
    emit(final=True)


if __name__ == '__main__':
    main()

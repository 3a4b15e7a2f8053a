"""Videos of different source sizes in one batch, each stabilised at its own resolution: MixedStreamBatch(out_size='source')
against StreamBatch(out_size=own size), S = 64 streams, network 288x512, refine = 1.

The bench_mixed.py method: one CUDA graph per step (per batch), a fixed mesh in place of the network, arms timed alternately in
rounds in one process.
  (a) device time of one step with the frames resident on the device; the per-size arm replays its graphs back to back;
  call: the warp alone (mgw_remap_bundle_frame_mixed, or mgw_remap_bundle_frame per batch), CUDA events around eager calls;
  (b) host-to-host time per step with the upload and the download inside the graphs (pinned host buffers): the mixed batch
      copies its whole input pool and its whole output pool (capacity bytes per slot both ways), the per-size batches exactly
      their frames.
Workloads:
  1 overhead:   64 x 1080p, BGR -> BGR and NV12 -> NV12; MixedStreamBatch at capacity 1080p and 2160p against
                StreamBatch(64, 1080p, out_size=1080p); (a) and call;
  2 few sizes:  bench_mixed.py's workload 2 (BGR), capacity 1920x1920, against one StreamBatch(out_size=own size) per size; (a), (b);
  3 fragmented: bench_mixed.py's workload 3 (BGR), capacity 2160x3840, likewise; (a), (b).
Prints one JSON object (the GPU's name and power limit included); --out also writes it to a file."""
import argparse, json, os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, 'oracle')); sys.path.insert(0, os.path.join(ROOT, 'tools'))
import numpy as np, torch
import dovs_b200 as mgw
from bench_mixed import FEW, FRAGMENTED
from bench_streams import dev_time, fixed_mesh_net, gpu_info, host_times, summary

dev = 'cuda'
h, w = 288, 512


def frame_shape(fmt, H, W):
    return (H, W, 3) if fmt == 'bgr' else (H * 3 // 2, W)


def rand_frame(gen, fmt, H, W):
    return torch.randint(0, 256, frame_shape(fmt, H, W), dtype=torch.uint8, device=dev, generator=gen)


def near_identity_maps(S):
    """the maps a stabiliser hands out: the identity moved by a smooth warp of a few pixels"""
    ys, xs = torch.meshgrid(torch.linspace(-1, 1, h), torch.linspace(-1, 1, w), indexing='ij')
    xy = torch.stack([xs + 0.01 * torch.sin(3 * ys), ys + 0.01 * torch.cos(2 * xs)], -1)
    return xy[None].repeat(S, 1, 1, 1).contiguous().to(dev)


class Mixed:
    """one MixedStreamBatch(out_size='source') holding every stream of a workload"""

    def __init__(self, groups, cap, fmt, out_fmt, gen):
        sizes = [sz for sz, n in groups for _ in range(n)]
        self.S, self.fmt, self.out_fmt = len(sizes), fmt, out_fmt
        self.mb = mgw.MixedStreamBatch(self.S, cap, height=h, width=w, refine=1, src_format=fmt, out_size='source', out_format=out_fmt)
        self.pool_h = torch.zeros(self.mb.pool_shape, dtype=torch.uint8).pin_memory()
        for s, sz in enumerate(sizes):
            self.mb.join(s, rand_frame(gen, fmt, *sz))
            self.mb.slot_frame(self.pool_h, s).copy_(rand_frame(gen, fmt, *sz).cpu())
        self.pool_d = self.pool_h.to(dev)
        self.out_h = torch.zeros(self.mb.out_pool_shape, dtype=torch.uint8).pin_memory()
        self.h2d_bytes, self.d2h_bytes = self.pool_h.numel(), self.out_h.numel()
        self.xy = near_identity_maps(self.S)

    def graph(self, net, io):
        kw = dict(upload_from=self.pool_h, download_to=self.out_h) if io else {}
        return [self.mb.capture(self.pool_d, net(self.mb), **kw)]

    def call(self):
        pool = self.pool_d.view((self.S,) + self.mb.frame_shape)
        return lambda: mgw.ops.remap_bundle_frame_mixed(pool, self.fmt, self.mb.sizes, self.xy, self.out_fmt, out=self.mb.colour,
                                                        workspace=self.mb.remap_ws)


class PerSize:
    """one StreamBatch(out_size=own size) per distinct size, their graphs replayed back to back"""

    def __init__(self, groups, fmt, out_fmt, gen):
        self.S, self.fmt, self.out_fmt = sum(n for _, n in groups), fmt, out_fmt
        self.parts = []
        for (H, W), n in groups:
            sb = mgw.StreamBatch(n, (H, W), height=h, width=w, refine=1, src_format=fmt, out_size=(H, W), out_format=out_fmt)
            for s in range(n):
                sb.join(s, rand_frame(gen, fmt, H, W))
            raw_h = torch.stack([rand_frame(gen, fmt, H, W) for _ in range(n)]).cpu().pin_memory()
            out_h = torch.zeros(tuple(sb.colour.shape), dtype=torch.uint8).pin_memory()
            self.parts.append((sb, raw_h, raw_h.to(dev), out_h, near_identity_maps(n)))
        self.h2d_bytes = sum(p[1].numel() for p in self.parts)
        self.d2h_bytes = sum(p[3].numel() for p in self.parts)

    def graph(self, net, io):
        return [sb.capture(raw_d, net(sb), **(dict(upload_from=raw_h, download_to=out_h) if io else {}))
                for sb, raw_h, raw_d, out_h, _ in self.parts]

    def call(self):
        def fn():
            for sb, _, raw_d, _, xy in self.parts:
                mgw.ops.remap_bundle_frame(raw_d, self.fmt, xy, out=sb.colour, workspace=sb.remap_ws, out_format=self.out_fmt)
        return fn


def replay_all(graphs):
    def fn():
        for g in graphs:
            g.replay()
    return fn


def workload(name, arms, legs, rounds, reps):
    """per round and leg every arm in turn: 'a' and 'call' device time (CUDA events), 'b' host to host"""
    fns = {}
    with torch.no_grad():
        for arm_name, arm in arms.items():
            f = {}
            if 'a' in legs:
                f['a'] = replay_all(arm.graph(fixed_mesh_net, False))
            if 'call' in legs:
                f['call'] = arm.call()
            if 'b' in legs:
                f['b'] = replay_all(arm.graph(fixed_mesh_net, True))
            fns[arm_name] = f
        res = {n: {leg: [] for leg in legs} for n in arms}
        for _ in range(rounds):
            for leg in legs:
                for arm_name in arms:
                    if leg == 'b':
                        res[arm_name][leg].append(host_times(fns[arm_name][leg], max(reps // 4, 10)))
                    else:
                        res[arm_name][leg].append(dev_time(fns[arm_name][leg], reps))
    out = {}
    for arm_name, arm in arms.items():
        r, S, o = res[arm_name], arm.S, {}
        if 'a' in r:
            a = float(np.median(r['a']))
            o.update(a_us_device_step_fixed_mesh_resident=a, a_us_device_per_frame=a / S, a_us_per_round=r['a'])
        if 'call' in r:
            c = float(np.median(r['call']))
            o.update(call_us_remap_alone=c, call_us_per_frame=c / S, call_us_per_round=r['call'])
        if 'b' in r:
            o['b_host_to_host_fixed_mesh'] = summary([t for ts in r['b'] for t in ts], S)
            o['b_host_to_host_fixed_mesh']['us_p50_per_round'] = [float(np.percentile(ts, 50)) for ts in r['b']]
        o['bytes_pcie_per_frame'] = {'h2d': arm.h2d_bytes / S, 'd2h': arm.d2h_bytes / S, 'total': (arm.h2d_bytes + arm.d2h_bytes) / S}
        out[arm_name] = o
    print(json.dumps({name: out}), file=sys.stderr)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--reps', type=int, default=100, help='timed replays per device measurement (host to host takes a quarter)')
    ap.add_argument('--rounds', type=int, default=3)
    ap.add_argument('--workloads', default='1,2,3')
    ap.add_argument('--out')
    a = ap.parse_args()
    assert torch.cuda.is_available(), 'bench_mixed_fullres.py measures on the GPU; there is nothing to measure without one'
    gen = torch.Generator(device=dev)
    gen.manual_seed(0)
    torch.manual_seed(0)
    res = {'gpu': gpu_info(), 'network_size': '%dx%d' % (h, w), 'refine': 1, 'S': 64, 'output': 'each slot at its source size',
           'method': 'one CUDA graph per batch and step, fixed mesh; arms alternated in rounds of --reps replays; (a) and call: median '
                     'of the per-round medians of CUDA-event times, (b) percentiles over all rounds', 'reps': a.reps,
           'rounds': a.rounds, 'workloads': {}}
    todo = set(a.workloads.split(','))

    def emit(final=False):
        if final:
            print(json.dumps(res, indent=1))
        if a.out:
            with open(a.out, 'w') as f:
                json.dump(res, f, indent=1)
    if '1' in todo:
        groups = [((1080, 1920), 64)]
        for fmt in ('bgr', 'nv12'):
            arms = {'mixed_capacity_1080p': Mixed(groups, (1080, 1920), fmt, fmt, gen),
                    'mixed_capacity_2160p': Mixed(groups, (2160, 3840), fmt, fmt, gen),
                    'stream_batch_1080p': PerSize(groups, fmt, fmt, gen)}
            r = workload('1_' + fmt, arms, ('a', 'call'), a.rounds, a.reps)
            base = r['stream_batch_1080p']
            r['over_stream_batch'] = {n: {'a_device_step': r[n]['a_us_device_step_fixed_mesh_resident'] /
                                          base['a_us_device_step_fixed_mesh_resident'],
                                          'call': r[n]['call_us_remap_alone'] / base['call_us_remap_alone']}
                                      for n in ('mixed_capacity_1080p', 'mixed_capacity_2160p')}
            res['workloads']['1_overhead_64x1080p_%s_to_%s' % (fmt, fmt)] = r
            emit()
            del arms
            torch.cuda.empty_cache()
    for key, groups, cap in (('2', FEW, (1920, 1920)), ('3', FRAGMENTED, (2160, 3840))):
        if key not in todo:
            continue
        arms = {'mixed': Mixed(groups, cap, 'bgr', 'bgr', gen), 'per_size_stream_batches': PerSize(groups, 'bgr', 'bgr', gen)}
        r = workload(key, arms, ('a', 'b'), a.rounds, a.reps)
        r['groups'] = [{'size': list(sz), 'streams': n} for sz, n in groups]
        r['capacity'] = list(cap)
        r['per_size_graphs'] = len(groups)
        mix, per = r['mixed'], r['per_size_stream_batches']
        r['mixed_over_per_size'] = {
            'a_device_step': mix['a_us_device_step_fixed_mesh_resident'] / per['a_us_device_step_fixed_mesh_resident'],
            'b_frames_per_s': mix['b_host_to_host_fixed_mesh']['frames_per_s'] / per['b_host_to_host_fixed_mesh']['frames_per_s'],
            'pcie_bytes': mix['bytes_pcie_per_frame']['total'] / per['bytes_pcie_per_frame']['total']}
        res['workloads'][{'2': '2_few_sizes', '3': '3_fragmented_16_sizes'}[key]] = r
        emit()
        del arms
        torch.cuda.empty_cache()
    emit(final=True)


if __name__ == '__main__':
    main()

#!/usr/bin/env python
"""Benchmark of the multi-grid warp hot path (BASELINE.json: warp Mpix/s fwd & fwd+bwd; achieved HBM GB/s).

    python bench.py [--gpus N] [--steps K] [--warmup W]          # B200 arm (one process per GPU under torchrun)
    python bench.py --impl reference [...]                       # the reference arm: CPU port on the host cores
    python bench.py --dump-outputs DIR [...]                     # also write the last timed step's outputs to DIR/<name>.npy

A step = one forward + backward of spatial_transformer3.transformer over one batch of synthetic frames at
BASELINE.json configs[1]: 32 x 288 x 512 x 3 fp32 per GPU, 4x4 mesh (weak scaling: every rank gets its own 32).
Rank 0 prints ONE JSON line.  Besides the contract's fields the line carries `sustained` (>= 1 s of graph replay of the same
step with its own clock record), `configs` (the other BASELINE.json configurations: #1 single frame, #3 the warp stage inside
a StabNet-shaped forward, #4 1080p stream latency with uint8 frames over PCIe, #5 the 256-clip data-parallel step with the
all-reduce overlapped and synchronous), `e2e_u8_fused` (a second end-to-end leg: uint8 frames over PCIe, loss fused onto the
warp) and, on one GPU, `dU_double_buffered` (the same step when the caller owns two dU buffers: the zero-fill of the next step's
buffer runs next to this step's backward).  See DESIGN.md "Measurement" for how every field is obtained.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for _p in (ROOT, os.path.join(ROOT, 'oracle')):
    if _p not in sys.path:
        sys.path.insert(0, _p)

import numpy as np   # noqa: E402
import torch         # noqa: E402

H, W, C, GH, GW = 288, 512, 3, 4, 4
FWD_BYTES_PER_PX = 8 * C + 12      # read U 4C, write out 4C, black 4, x/y maps 8        (SURVEY.md 8d)
BWD_BYTES_PER_PX = 12 * C + 8      # read d_out 4C, U 4C, write dU 4C, read d_img 8
METRIC = 'warp_fwd_bwd_mpix_per_s'
# where the zero-fill of dU sits in the step (see make_step): 'pipelined' = dU double-buffered, the fill of the buffer step i+1
# accumulates into runs next to step i's backward (mgw_mesh_warp_bwd_acc); 'fused' = inside the plain backward call, behind the forward
# 'pipelined_tail' = the same double buffering with the fill AFTER the backward, next to the join of the all-reduce (tuning aid).
# The headline step keeps the fill inside the call ('fused') at every GPU count, so that the weak-scaling figures compare the same
# schedule; the double-buffered form is reported next to it on one GPU (`dU_double_buffered`: 122.8 vs 126.9 us).  In a 32-frame
# step that also carries the NCCL all-reduce and the head-gradient GEMM one more concurrent kernel costs more than it hides (2 GPUs:
# 145.0 us next to the backward, 148.5 us after it, 137.0 us with the fill inside the call); config #5's 64+ frames per rank gain.
FILL_MODE = os.environ.get('BENCH_FILL', '')
PIPELINED = ('pipelined', 'pipelined_tail')


def fill_mode_for(world, frames_per_rank):
    return FILL_MODE or 'fused'


def peaks():
    try:
        with open(os.path.join(ROOT, 'MEASURED_PEAKS.json')) as f:
            return float(json.load(f)['hbm_gbs']), 'measured (MEASURED_PEAKS.json)'
    except Exception:      # noqa: BLE001
        return 6650.0, 'fallback (B200_PROFILING.md)'


def synth_inputs(n, seed=0):
    import synth
    return dict(U=synth.noise_image(n, H, W, C, 900 + seed), theta=synth.random_mesh(n, GH, GW, 0.05, 901 + seed),
                d_out=synth.randn((n, H, W, C), 902 + seed), d_img=synth.randn((n, H, W, 2), 903 + seed, 0.1))


DUMP_BYTES = 60 << 20      # --dump-outputs writes at most this much


def dump_outputs(path, outputs):
    """Writes the arrays one step handed its caller as path/<name>.npy (float32).  Every array is cut to the same frames: a
    fixed, seeded sample of the batch, as many as fit in DUMP_BYTES.  Returns the frame indices."""
    n = next(iter(outputs.values())).shape[0]
    per_frame = sum(t[0].numel() * t.element_size() for t in outputs.values())
    k = max(1, min(n, DUMP_BYTES // per_frame))
    frames = np.sort(np.random.RandomState(0).choice(n, k, replace=False))
    idx = torch.as_tensor(frames, device=next(iter(outputs.values())).device)
    os.makedirs(path, exist_ok=True)
    for name, t in outputs.items():
        np.save(os.path.join(path, name + '.npy'), t.index_select(0, idx).float().cpu().numpy())
    return frames.tolist()


class ClockSampler:
    """nvidia-smi clocks/throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ('index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,'
         'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap')

    def __init__(self, index):
        self.index, self.lines, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(['nvidia-smi', '-i', str(self.index), '--query-gpu=' + self.Q, '--format=csv,noheader,nounits',
                                          '-lms', '100'], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:      # noqa: BLE001
            self.proc = None
        return self

    def _pump(self):
        for ln in self.proc.stdout:
            self.lines.append(ln.strip())

    def stop(self):
        if self.proc is None:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, pw, reasons = [], [], [], set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(',')]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2])); pw.append(float(f[3]))
            except ValueError:
                continue
            for name, v in zip(('hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap'), f[5:9]):
                if v.lower().startswith('active'):
                    reasons.add(name)
        return {'sm_mhz': float(np.median(sm)) if sm else None, 'sm_max_mhz': max(mx) if mx else None,
                'power_w_max': max(pw) if pw else None, 'samples': len(sm), 'reasons': sorted(reasons)}


def cpu_port_step(inp, n):
    """one fwd+bwd of the oracle's torch-CPU port on the first n frames; returns seconds."""
    import mesh_warp_ref as ref
    U = torch.tensor(inp['U'][:n], requires_grad=True)
    th = torch.tensor(inp['theta'][:n], requires_grad=True)
    g_out, g_img = torch.tensor(inp['d_out'][:n]), torch.tensor(inp['d_img'][:n])
    t0 = time.perf_counter()
    out, black, img, _ = ref.transformer(U, th)
    torch.autograd.backward([out, img], [g_out, g_img])
    return time.perf_counter() - t0


def run_reference(args):
    """reference arm: the reference's CPU implementation of the path = the oracle port (TensorFlow is absent and the
    reference is pure Python that cannot travel), all host threads, bounded sample per step."""
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    torch.set_num_threads(os.cpu_count() or 1)
    ns = args.cpu_sample
    inp = synth_inputs(ns)
    for _ in range(max(args.warmup, 1)):
        cpu_port_step(inp, ns)
    steps = args.steps
    t = sum(cpu_port_step(inp, ns) for _ in range(steps))
    val = ns * H * W * steps / t / 1e6
    sample = '%d of 32 frames of configs[1] per step (fwd+bwd, dU+dtheta), %d steps' % (ns, steps)
    print(json.dumps({
        'impl': 'reference', 'metric': METRIC, 'value': val, 'unit': 'Mpix/s', 'n_gpus': args.gpus, 'steps': steps,
        'warmup': args.warmup, 'ms_per_step': 1e3 * t / steps, 'higher_is_better': True, 'scaling': 'weak',
        'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
        'config': {'workload': 'configs[1]: %d x %dx%dx%d fp32 frames per GPU, %dx%d mesh warp forward+backward (dU + dtheta)' % (32, H, W, C, GH, GW),
                   'sample': '%d of the 32 frames per step' % ns},
        'cpu_baseline': {'value': val, 'unit': 'Mpix/s', 'cores': torch.get_num_threads(), 'kind': 'port', 'sample': sample},
        'e2e': {'value': val, 'unit': 'Mpix/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
        'note': 'oracle/mesh_warp_ref.py (torch-CPU restatement of the reference graph); TensorFlow is not installable here',
    }))


def pin_to_gpu_cores(local):
    """run this rank on the host cores next to its GPU (NUMA-local staging buffers); returns the cpu count or None."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(local)
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (os.cpu_count() + 63) // 64)
        cpus = [64 * i + b for i, wd in enumerate(words) for b in range(64) if (wd >> b) & 1]
        cpus = [c for c in cpus if c in os.sched_getaffinity(0)]
        if cpus:
            os.sched_setaffinity(0, cpus)
            return len(cpus)
    except Exception:      # noqa: BLE001
        pass
    return None


def main():
    sys.dont_write_bytecode = True      # the benchmark writes nothing into the tree it runs from (which may be read-only)
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=50)
    ap.add_argument('--warmup', type=int, default=5)
    ap.add_argument('--impl', default='b200', choices=['b200', 'reference'])
    ap.add_argument('--batch', type=int, default=32, help='frames per GPU')
    ap.add_argument('--cpu-sample', type=int, default=32, help='frames per CPU-baseline step (of the 32-frame batch)')
    ap.add_argument('--no-cpu-baseline', action='store_true', help='skip the CPU leg (profiling runs)')
    ap.add_argument('--no-configs', action='store_true', help='skip the sub-records of the other BASELINE configs and the sustained leg')
    ap.add_argument('--kernel-impl', default='auto', choices=['auto', 'generic', 'tma', 'pipe'])
    ap.add_argument('--no-graph', action='store_true', help='launch the step eagerly instead of replaying CUDA graphs')
    ap.add_argument('--no-l2-keep', action='store_true', help='zero-fill dU without the L2 evict_last policy')
    ap.add_argument('--dump-outputs', metavar='DIR', help='write what the last timed step returned (out, black, img, Hs, dU, dtheta; '
                                                          'a seeded sample of its frames) to DIR/<name>.npy')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.impl == 'reference':
        return run_reference(args)

    import dovs_b200 as mgw
    from dovs_b200 import ops
    import torch.distributed as dist
    assert torch.cuda.is_available(), 'bench.py needs a CUDA device: the product has no CPU path'
    rank, world, local = mgw.parallel.init_from_env()
    torch.manual_seed(rank)          # the torch-generated inputs (mesh-head features, config #3) are the same from run to run
    assert world == args.gpus or world == 1, 'launch with torchrun --nproc-per-node %d' % args.gpus
    ncores = pin_to_gpu_cores(local)
    dev = torch.device('cuda', local)
    torch.cuda.set_device(dev)
    mgw.set_impl(args.kernel_impl)
    n, K, Wm = args.batch, args.steps, max(args.warmup, 3)
    P = n * H * W
    keep = not args.no_l2_keep

    # --- inputs: 3 rotating sets so that no step finds its inputs in L2 (each set is 151 MB, L2 is 126 MB)
    base = synth_inputs(n, seed=rank)
    R = 3
    sets = []
    for k in range(R):
        sets.append({key: torch.tensor(np.roll(v, k, axis=0), device=dev) for key, v in base.items()})
    feats = torch.randn(n, 512, device=dev)
    reducer = mgw.parallel.MeshHeadGradReducer(512, 2 * (GH + 1) * (GW + 1), dev, nbuf=R)

    def make_step(sets, feats, reducer, sync_reduce=False, fill_mode=None):
        """the step over rotating input sets: K1, K2 (PDL), zero-fill of dU on a side branch, K3, K4 (PDL); with more than one
        rank the head gradient + all-reduce of the PREVIOUS step (overlapped form) or of THIS step (synchronous form)."""
        nset = len(sets)
        fill_mode = fill_mode or fill_mode_for(world, sets[0]['U'].shape[0])
        # 'pipelined' double-buffers dU: step i accumulates into buffer i % 2 (mgw_mesh_warp_bwd_acc) while the zero-fill of the
        # buffer step i+1 will use runs next to its backward on a side branch -- one fill per step inside the timed region, every
        # step's dU complete and correct (tests/test_gpu_configs.py::test_double_buffered_dU_pipeline)
        dU_bufs = [torch.zeros_like(sets[0]['U']) for _ in range(2 if fill_mode in PIPELINED else 1)]
        dU_buf = dU_bufs[0]
        ngraph = nset * 2 if (fill_mode in PIPELINED and nset % 2) else nset
        dth_slots = [torch.zeros_like(sets[0]['theta']) for _ in range(nset)]
        side = torch.cuda.Stream(device=dev)

        def step_eager(i):
            s = sets[i % nset]
            cur = torch.cuda.current_stream()
            # dU of the step is zero-filled by the library's own kernel (evict_last: its lines are still in L2 when the backward's
            # reductions arrive), INSIDE the timed step.  Placement is a tuning aid (BENCH_FILL): after_fwd = between forward
            # and backward on the main stream; with_k1 = on a side branch next to K1, joined before K2; side = on a side branch next
            # to the whole forward; serial = before K1; none = no fill (wrong dU, timing only); fused (default) = no fill here at
            # all: the plain backward entry point zero-fills dU itself (under the backward pipeline's own shadow when that runs)
            if fill_mode == 'serial':
                ops.fill_zero(dU_buf, keep_in_l2=keep)
            if fill_mode in ('side', 'with_k1'):
                side.wait_stream(cur)
                with torch.cuda.stream(side):
                    ops.fill_zero(dU_buf, keep_in_l2=keep)
            if fill_mode == 'with_k1':
                Hs = ops.solve_h_fwd(s['theta'])
                cur.wait_stream(side)
                out, black, img, _ = ops.warp_fwd(s['U'], Hs)
            else:
                out, black, img, Hs = ops.mesh_warp_fwd(s['U'], s['theta'])
            if world > 1 and not sync_reduce:
                # head gradient (features^T . dtheta) and all-reduce of the PREVIOUS step on a high-priority side stream, forked
                # right AFTER the forward and BEFORE the zero-fill: the persistent forward kernel owns every SM with a static tile
                # schedule (a CTA displaced by the NCCL kernel would finish late), the fill's 64-thread blocks leave the SMs
                # nearly empty, so the GEMM and the NCCL kernel become resident at once
                reducer.launch(slot=(i - 1) % nset, features=feats, dtheta=dth_slots[(i - 1) % nset])
            if fill_mode == 'race':     # timing experiment only (WRONG dU): the fill next to the backward, no ordering between them
                side.wait_stream(cur)
                with torch.cuda.stream(side):
                    ops.fill_zero(dU_buf, keep_in_l2=keep)
            if fill_mode == 'pipelined':
                side.wait_stream(cur)
                with torch.cuda.stream(side):
                    ops.fill_zero(dU_bufs[(i + 1) % 2], keep_in_l2=False)
            if fill_mode == 'after_fwd':
                ops.fill_zero(dU_buf, keep_in_l2=keep)
            if fill_mode == 'side':
                cur.wait_stream(side)
            if fill_mode == 'fused':
                dU, dtheta = ops.mesh_warp_bwd(s['U'], s['theta'], Hs, s['d_out'], s['d_img'], dU_out=dU_buf, dtheta_out=dth_slots[i % nset])
            elif fill_mode in PIPELINED:
                dU, dtheta = ops.mesh_warp_bwd(s['U'], s['theta'], Hs, s['d_out'], s['d_img'], accumulate_into=dU_bufs[i % 2],
                                               dtheta_out=dth_slots[i % nset])
            else:
                dU, dtheta = ops.mesh_warp_bwd(s['U'], s['theta'], Hs, s['d_out'], s['d_img'], accumulate_into=dU_buf,
                                               dtheta_out=dth_slots[i % nset])
            if fill_mode in ('race', 'pipelined'):
                cur.wait_stream(side)
            if world > 1 and sync_reduce:
                reducer.launch(slot=i % nset, features=feats, dtheta=dth_slots[i % nset])
            if fill_mode == 'pipelined_tail':           # next to the all-reduce the step is about to wait for
                side.wait_stream(cur)
                with torch.cuda.stream(side):
                    ops.fill_zero(dU_bufs[(i + 1) % 2], keep_in_l2=False)
                cur.wait_stream(side)
            if world > 1:
                reducer.wait()                          # join: fork and join both lie inside the step (CUDA-graph capturable)
            return dict(out=out, black=black, img=img, Hs=Hs, dU=dU, dtheta=dtheta)

        graphs = None
        captured = []         # what the capture of graph i returned: every replay of graph i rewrites these tensors
        if not args.no_graph:
            # The step is launch-bound on the host once NCCL is in it (a dozen launches for ~100 us of GPU work): capture one
            # CUDA graph per rotating input set and replay.  Same kernels, same work; eager launches if capture is not possible.
            try:
                for i in range(ngraph):
                    step_eager(i)
                if world > 1:
                    reducer.wait()
                torch.cuda.synchronize()
                graphs = []
                for i in range(ngraph):
                    gph = torch.cuda.CUDAGraph()
                    # thread_local: the NCCL watchdog thread polls CUDA events while we capture
                    with torch.cuda.graph(gph, capture_error_mode='thread_local'):
                        captured.append(step_eager(i))
                    graphs.append(gph)
                torch.cuda.synchronize()
            except Exception as e:      # noqa: BLE001
                sys.stderr.write('CUDA graph capture failed (%s); running eager\n' % e)
                graphs = None
                torch.cuda.synchronize()

        # the steps follow each other whatever index the caller passes (the dU buffers alternate); 'eager' = what the last
        # eager step() returned
        state = {'k': 0, 'eager': None}

        def step(_i):
            k = state['k']
            state['k'] = k + 1
            if graphs is not None:
                graphs[k % ngraph].replay()
            else:
                state['eager'] = step_eager(k)

        def last_outputs():
            """the tensors the last call of step() wrote (calls of step_eager outside step() do not change them)"""
            return captured[(state['k'] - 1) % ngraph] if graphs is not None else state['eager']
        return step, step_eager, graphs, dU_buf, last_outputs

    def timed(fn, steps, warm, before_stop=None):
        for i in range(warm):
            fn(i)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(steps):
            fn(i)
        if world > 1:
            reducer.wait()
        if before_stop is not None:
            before_stop()
        e1.record()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item())

    step, step_eager, graphs, dU_buf, last_outputs = make_step(sets, feats, reducer)
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
        time.sleep(0.3)
    l0 = mgw.launch_count()
    step_eager(0)
    if world > 1:
        reducer.wait()
    launches_per_step = mgw.launch_count() - l0          # kernels of OUR library per step (replayed as-is under the graph)
    fill_mode = fill_mode_for(world, n)
    if fill_mode in PIPELINED:
        step_eager(1)                                    # an even number of steps: the dU buffers are back in phase
        if world > 1:
            reducer.wait()
    ms_total = timed(step, K, Wm)
    launches_timed = launches_per_step * K
    clocks = sampler.stop() if rank == 0 else None
    dumped = None
    if args.dump_outputs and rank == 0:      # before the legs below reuse dU_buf and replay the step again
        dumped = {'dir': args.dump_outputs, 'frames': dump_outputs(args.dump_outputs, last_outputs())}

    # --- the same step sustained: >= 1 s of replay (the K-step figure above lasts a few milliseconds)
    sustained = None
    if not args.no_configs:
        ks = max(K, int(1.2e3 / max(ms_total / K, 1e-3)))
        sm2 = ClockSampler(local).start() if rank == 0 else None
        if rank == 0:
            time.sleep(0.2)
        ms_s = timed(step, ks, 3)
        sustained = {'ms_per_step': ms_s / ks, 'steps': ks, 'seconds': ms_s * 1e-3, 'value': P * world * ks / (ms_s * 1e-3) / 1e6,
                     'unit': 'Mpix/s', 'clocks': sm2.stop() if rank == 0 else None}

    # --- the same step with dU double-buffered: the zero-fill of the buffer step i+1 accumulates into runs next to step i's backward
    # (mgw_mesh_warp_bwd_acc): what a training loop that owns two dU buffers gets.  One GPU only (see FILL_MODE above).
    double_buffered = None
    if not args.no_configs and fill_mode == 'fused' and world == 1:
        step_db, _, _, _, _ = make_step(sets, feats, reducer, fill_mode='pipelined')
        ms_db = timed(step_db, K, Wm) / K
        double_buffered = {'ms_per_step': ms_db, 'value': P / (ms_db * 1e-3) / 1e6, 'unit': 'Mpix/s',
                           'note': 'one zero-fill per step inside the timed region, of the buffer the NEXT step accumulates into, next to '
                                   'this step\'s backward; every step\'s dU complete (tests: test_double_buffered_dU_pipeline)'}
        del step_db

    # --- per-kernel timings (same rotation, CUDA events around the single C-ABI call)
    Hs_sets = [ops.solve_h_fwd(s['theta']) for s in sets]
    ms_fwd = timed(lambda i: ops.warp_fwd(sets[i % R]['U'], Hs_sets[i % R]), K, Wm)

    from dovs_b200._lib import lib, check
    ws_k3 = torch.empty(max(lib.mgw_warp_bwd_workspace_bytes(n, H, W, C, GH, GW), 256) // 4 + 64, device=dev)

    def bwd_call(i):
        # the backward KERNEL alone (dHs = NULL: the per-tile dH partials stay in the workspace, K4 sums them in the step), behind
        # the zero-fill exactly as in the step
        s = sets[i % R]
        ops.fill_zero(dU_buf, keep_in_l2=keep)
        check(lib.mgw_warp_bwd_acc(s['U'].data_ptr(), Hs_sets[i % R].data_ptr(), s['d_out'].data_ptr(), s['d_img'].data_ptr(), n, H, W, C, GH, GW,
                                   dU_buf.data_ptr(), None, ws_k3.data_ptr(), torch.cuda.current_stream().cuda_stream), 'mgw_warp_bwd_acc')
    ms_bwd_fill = timed(bwd_call, K, Wm)
    ms_fill = timed(lambda i: ops.fill_zero(dU_buf, keep_in_l2=keep), K, Wm)
    ms_bwd = ms_bwd_fill - ms_fill
    ms_fwd_full = timed(lambda i: ops.mesh_warp_fwd(sets[i % R]['U'], sets[i % R]['theta']), K, Wm)

    # --- end to end through the public API with HOST (pinned) buffers: H2D of the step's inputs and D2H of its result
    # Two staging sets and a copy stream: the H2D of step i+1 runs under the kernels of step i (the step is PCIe-bound:
    # 151 MB per step); every step still copies ITS inputs from pinned host memory and returns ITS dtheta to the host, and
    # the host waits for the result of step i-1 before it enqueues step i+1's copy (bounded run-ahead, as a training loop has).
    def e2e_leg(host, compute, res_shape):
        stages = [{k: torch.empty_like(v, device=dev) for k, v in host.items()} for _ in range(2)]
        res_host = [torch.empty(res_shape).pin_memory() for _ in range(2)]
        copy_stream = torch.cuda.Stream(device=dev)
        ev_copied = [torch.cuda.Event() for _ in range(2)]
        ev_free = [torch.cuda.Event() for _ in range(2)]
        ev_res = [torch.cuda.Event() for _ in range(2)]
        state = {'n': 0}

        def issue_h2d(j):
            b = j % 2
            with torch.cuda.stream(copy_stream):
                copy_stream.wait_event(ev_free[b])              # the step that last used this staging set has finished
                for k in host:
                    stages[b][k].copy_(host[k], non_blocking=True)
                ev_copied[b].record(copy_stream)

        def e2e_step(i):
            j = state['n']
            b = j % 2
            cur = torch.cuda.current_stream()
            if j == 0:
                for e in ev_free:
                    e.record(cur)
                issue_h2d(0)
            issue_h2d(j + 1)                                    # next step's inputs travel while this step computes
            cur.wait_event(ev_copied[b])
            res = compute(stages[b])
            res_host[b].copy_(res, non_blocking=True)
            ev_res[b].record(cur)
            ev_free[b].record(cur)
            if j > 0:
                ev_res[1 - b].synchronize()                     # the caller reads the previous step's result on the host
            state['n'] = j + 1

        Ke = max(3, min(K, 20))
        # the copy issued ahead by the last step is waited for inside the timed region: K steps pay for K copies
        ms = timed(e2e_step, Ke, 3, before_stop=lambda: torch.cuda.current_stream().wait_stream(copy_stream))
        return ms / Ke, Ke, sum(v.numel() * v.element_size() for v in host.values()), res_host[0].numel() * 4

    def compute_main(st):
        Ut, th = st['U'].requires_grad_(True), st['theta'].requires_grad_(True)
        out, black, img = mgw.transformer(Ut, th)
        torch.autograd.backward([out, img], [st['d_out'], st['d_img']])
        g = th.grad
        Ut.grad = None; th.grad = None
        Ut.requires_grad_(False); th.requires_grad_(False)
        return g
    host_main = {k: torch.tensor(v).pin_memory() for k, v in base.items()}
    ms_e2e, Ke, h2d, d2h = e2e_leg(host_main, compute_main, (n, GH + 1, GW + 1, 2))

    # second leg: what a training step really moves -- uint8 frames (the reference's frames are uint8: config.py:6-21), widened on
    # the device exactly as config.py:19 does, img_loss fused onto the warp (s_net_bundle_nobm.py:332,347-352): no upstream
    # gradient tensor crosses PCIe
    e2e_u8 = None
    if not args.no_configs:
        rs = np.random.RandomState(7 + rank)
        host_u8 = {'U': torch.tensor(rs.randint(0, 256, (n, H, W, C)).astype(np.uint8)).pin_memory(),
                   'y': torch.tensor(rs.randint(0, 256, (n, H, W, C)).astype(np.uint8)).pin_memory(),
                   'theta': torch.tensor(base['theta']).pin_memory()}
        Uf, yf = torch.empty((n, H, W, C), device=dev), torch.empty((n, H, W, C), device=dev)

        def compute_u8(st):
            ops.u8_to_train(st['U'], out=Uf); ops.u8_to_train(st['y'], out=yf)
            th = st['theta'].requires_grad_(True)
            loss, out, black, img = mgw.transformer_img_loss(Uf, th, yf)
            loss.backward()
            g = th.grad
            th.grad = None
            th.requires_grad_(False)
            return g
        ms2, Ke2, h2d2, d2h2 = e2e_leg(host_u8, compute_u8, (n, GH + 1, GW + 1, 2))
        e2e_u8 = {'value': P * world / (ms2 * 1e-3) / 1e6, 'unit': 'Mpix/s', 'ms_per_step': ms2, 'steps': Ke2, 'h2d_bytes_per_step': h2d2,
                  'd2h_bytes_per_step': d2h2, 'h2d_gbs_per_rank': h2d2 / (ms2 * 1e-3) / 1e9,
                  'workload': 'uint8 U and target frames over PCIe, exact on-device v/255-0.5, fused transformer+img_loss forward+backward (dtheta)'}

    configs = None
    if not args.no_configs:
        configs = other_configs(mgw, ops, dev, rank, world, timed, make_step, keep)

    if rank != 0:
        finish(world)
        return
    peak, peak_src = peaks()
    pix_per_step = P * world
    value = pix_per_step * K / (ms_total * 1e-3) / 1e6
    gbs_fwd = FWD_BYTES_PER_PX * P / (ms_fwd / K * 1e-3) / 1e9
    gbs_bwd = BWD_BYTES_PER_PX * P / (ms_bwd / K * 1e-3) / 1e9
    gbs_step = (FWD_BYTES_PER_PX + BWD_BYTES_PER_PX) * P / (ms_total / K * 1e-3) / 1e9
    traffic = None
    try:
        with open(os.path.join(ROOT, 'profiles', 'traffic.json')) as f:
            traffic = json.load(f)
    except Exception:      # noqa: BLE001
        pass
    dominant = 'warp_bwd' if ms_bwd >= ms_fwd else 'warp_fwd'
    roof = {
        'warp_fwd': {'bound': 'hbm', 'achieved': gbs_fwd, 'peak': peak, 'unit': 'GB/s', 'frac': gbs_fwd / peak,
                     'traffic': (traffic or {}).get('warp_fwd'), 'us_per_launch': 1e3 * ms_fwd / K,
                     'algorithmic_bytes_per_launch': FWD_BYTES_PER_PX * P},
        'warp_bwd': {'bound': 'hbm', 'achieved': gbs_bwd, 'peak': peak, 'unit': 'GB/s', 'frac': gbs_bwd / peak,
                     'traffic': (traffic or {}).get('warp_bwd'), 'us_per_launch': 1e3 * ms_bwd / K,
                     'algorithmic_bytes_per_launch': BWD_BYTES_PER_PX * P,
                     'note': 'mgw_warp_bwd_acc with dHs = NULL (the backward kernel alone: K4 sums its dH partials in the step) timed back to '
                             'back with the zero-fill of dU as in the step, minus the zero-fill timed alone (%.1f us)' % (1e3 * ms_fill / K)},
    }
    line = {
        'metric': METRIC, 'value': value, 'unit': 'Mpix/s', 'n_gpus': world, 'steps': K, 'warmup': Wm,
        'ms_per_step': ms_total / K, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32',
        'data': 'synthetic',
        'config': {'workload': 'configs[1]: %d x %dx%dx%d fp32 frames per GPU, %dx%d mesh warp forward+backward (dU + dtheta)' % (n, H, W, C, GH, GW),
                   'l2': 'inputs rotate over %d sets of 151 MB (> 126 MB L2)' % R, 'kernel_impl': args.kernel_impl,
                   'launch': 'cuda graph replay' if graphs is not None else 'eager',
                   'dU_zero_fill': {'pipelined': 'one fill per step inside the timed region; dU double-buffered: the fill of the buffer step i+1 '
                                                 'accumulates into (mgw_mesh_warp_bwd_acc) runs next to the backward of step i',
                                    'pipelined_tail': 'one fill per step inside the timed region; dU double-buffered: the fill of the buffer '
                                                      'step i+1 accumulates into (mgw_mesh_warp_bwd_acc) runs after the backward of step i, '
                                                      'next to the wait for the all-reduce',
                                    'fused': 'inside the backward call (mgw_mesh_warp_bwd), between forward and backward; the backward kernel is launched '
                                             'programmatically behind it and waits for it (griddepcontrol.wait) before its first access to dU'}.get(fill_mode, fill_mode),
                   'parallelism': ('dp%d (batch-sharded, 100 KB mesh-head grad all-reduce of step i-1 overlapped with step i; the '
                                   'synchronous form is in configs.config5)' % world) if world > 1 else 'single GPU',
                   'host_cores_pinned_per_rank': ncores},
        'fwd_mpix_per_s': pix_per_step * K / (ms_fwd_full * 1e-3) / 1e6,
        'step_hbm_gbs': gbs_step, 'step_hbm_frac_of_measured': gbs_step / peak, 'step_hbm_frac_of_8tbs': gbs_step / 8000.0,
        'roofline': dict(roof[dominant], kernel=dominant, peak_source=peak_src), 'roofline_kernels': roof,
        'e2e': {'value': pix_per_step / (ms_e2e * 1e-3) / 1e6, 'unit': 'Mpix/s', 'h2d_bytes_per_step': h2d,
                'd2h_bytes_per_step': d2h, 'ms_per_step': ms_e2e, 'steps': Ke, 'h2d_gbs_per_rank': h2d / (ms_e2e * 1e-3) / 1e9},
        'gpu_launches': launches_timed, 'clocks': clocks,
    }
    if double_buffered is not None:
        line['dU_double_buffered'] = double_buffered
    if sustained is not None:
        line['sustained'] = sustained
    if e2e_u8 is not None:
        line['e2e_u8_fused'] = e2e_u8
    if configs is not None:
        line['configs'] = configs
    if dumped is not None:
        line['dump_outputs'] = dumped
    if world == 1 and not args.no_cpu_baseline:
        torch.set_num_threads(os.cpu_count() or 1)
        ns = args.cpu_sample
        cpu_port_step(base, ns)
        ts, t_start = [], time.perf_counter()
        while len(ts) < 3 or (time.perf_counter() - t_start < 12 and len(ts) < 200):
            ts.append(cpu_port_step(base, ns))
        line['cpu_baseline'] = {'value': ns * H * W / float(np.mean(ts)) / 1e6, 'unit': 'Mpix/s', 'cores': torch.get_num_threads(),
                                'kind': 'port', 'sample': '%d of %d frames of the same workload, fwd+bwd, mean of %d runs (%.1f s of CPU work)'
                                % (ns, n, len(ts), sum(ts))}
    print(json.dumps(line))
    finish(world)


def other_configs(mgw, ops, dev, rank, world, timed, make_step, keep):
    """sub-records for the BASELINE.json configurations that are not the headline (bounded: a few seconds in total)."""
    import synth
    from dovs_b200._lib import lib, check
    res = {}
    flush = torch.empty(48 * 1024 * 1024, device=dev)

    def dev_us(fn, reps=30, flush_l2=True):
        for _ in range(3):
            fn()
        ts = []
        for _ in range(reps):
            if flush_l2:
                flush.zero_()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(); fn(); e1.record(); torch.cuda.synchronize()
            ts.append(e0.elapsed_time(e1) * 1e3)
        return float(np.median(ts))

    if rank == 0:
        # ---- config #1: single 288x512x3 frame, forward (K1 + K2)
        U1 = torch.tensor(synth.noise_image(1, H, W, C, 1), device=dev)
        th1 = torch.tensor(synth.random_mesh(1, GH, GW, 0.05, 2), device=dev)
        t1 = dev_us(lambda: ops.mesh_warp_fwd(U1, th1))
        res['config1_single_frame_fwd'] = {'us_device': t1, 'mpix_per_s': H * W / t1}

        # ---- config #3: the warp stage inside a StabNet-shaped forward (torch ResNet-50-v2 carrier, random init, batch 16, 13 channels)
        try:
            net = mgw.StabNet(in_ch=13).to(dev).eval()
            x13 = torch.randn(16, H, W, 13, device=dev) * 0.2
            with torch.no_grad():
                def fwd3():
                    theta = net(x13)
                    _, pts2 = mgw.get_4_pts(theta, 16)
                    return mgw.transformer(x13[..., 12:13].contiguous(), pts2)
                t_all = dev_us(fwd3, 10, flush_l2=False)
                theta = net(x13)
                _, pts2 = mgw.get_4_pts(theta, 16)
                x1 = x13[..., 12:13].contiguous()
                t_warp = dev_us(lambda: mgw.transformer(x1, pts2), 30)
            res['config3_stabnet_fwd_b16'] = {'ms_forward': t_all * 1e-3, 'us_warp_stage': t_warp, 'warp_share': t_warp / t_all,
                                              'note': 'backbone = torch/cuDNN carrier (parity unpinned); the warp stage is this library (C = 1)'}
            del net, x13
        except Exception as e:      # noqa: BLE001
            res['config3_stabnet_fwd_b16'] = {'error': str(e)[:200]}

        # ---- config #4: 1080p stream, batch 1, per-frame latency host-to-host.  Frames are uint8 (config.py:6-21,
        # deploy_bundle.py:301): H2D uint8 -> v/255-0.5 on the device -> K1 + K2 -> (x+0.5)*255 -> uint8 -> D2H, one CUDA graph
        Hh, Ww = 1080, 1920
        fr_h = torch.randint(0, 256, (1, Hh, Ww, 3), dtype=torch.uint8).pin_memory()
        out_h = torch.empty((1, Hh, Ww, 3), dtype=torch.uint8).pin_memory()
        th4 = torch.tensor(synth.random_mesh(1, GH, GW, 0.03, 4), device=dev)
        fr_d = torch.empty((1, Hh, Ww, 3), device=dev, dtype=torch.uint8)
        f32_d, o32_d = torch.empty((1, Hh, Ww, 3), device=dev), torch.empty((1, Hh, Ww, 3), device=dev)
        bl_d, xy_d, Hs_d = torch.empty((1, Hh, Ww), device=dev), torch.empty((1, Hh, Ww, 2), device=dev), torch.empty((1, GH, GW, 9), device=dev)
        ou_d = torch.empty((1, Hh, Ww, 3), device=dev, dtype=torch.uint8)
        PP = lambda x: x.data_ptr()      # noqa: E731
        s4 = torch.cuda.Stream(device=dev)
        with torch.cuda.stream(s4):
            def kernels():
                ops.u8_to_train(fr_d, out=f32_d)
                check(lib.mgw_mesh_warp_fwd(PP(f32_d), PP(th4), 1, Hh, Ww, 3, GH, GW, PP(Hs_d), PP(o32_d), PP(bl_d), PP(xy_d),
                                            torch.cuda.current_stream().cuda_stream), 'fwd')
                ops.train_to_u8(o32_d, out=ou_d)

            def frame():
                fr_d.copy_(fr_h, non_blocking=True)
                kernels()
                out_h.copy_(ou_d, non_blocking=True)
            for _ in range(3):
                frame()
            s4.synchronize()
            g4 = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g4, stream=s4):
                frame()
            gk = torch.cuda.CUDAGraph()
            with torch.cuda.graph(gk, stream=s4):
                kernels()
            us_dev = dev_us(gk.replay, 100, flush_l2=False)
            lat = []
            for _ in range(1000):
                t0 = time.perf_counter()
                g4.replay()
                s4.synchronize()
                lat.append((time.perf_counter() - t0) * 1e6)
        res['config4_1080p_stream'] = {'us_device_kernels': us_dev, 'us_p50_host_to_host': float(np.percentile(lat, 50)),
                                       'us_p99_host_to_host': float(np.percentile(lat, 99)), 'frames': 1000,
                                       'bytes_h2d_per_frame': fr_h.numel(), 'bytes_d2h_per_frame': out_h.numel(),
                                       'note': 'uint8 frames over PCIe, u8->fp32->warp->u8 on the device, H2D + 4 kernels + D2H as ONE CUDA graph'}
        del f32_d, o32_d, xy_d

    # ---- config #5: data-parallel train step, batch 256 clips sharded over the ranks (256/N per rank), mesh-head all-reduce
    nb = 256 // world
    base5 = synth_inputs(32, seed=50 + rank)
    rep = (nb + 31) // 32
    set5 = [{k: torch.tensor(np.concatenate([np.roll(v, j, axis=0) for j in range(rep)])[:nb], device=dev) for k, v in base5.items()}]
    feats5 = torch.randn(nb, 512, device=dev)
    red5 = mgw.parallel.MeshHeadGradReducer(512, 2 * (GH + 1) * (GW + 1), dev, nbuf=2)
    rec5 = {'frames_per_rank': nb, 'global_batch': nb * world,
            'l2': 'one input set of %.0f MB per rank (> 126 MB L2)' % (nb * 151.0 / 32)}
    for name, sync in (('overlapped', False), ('synchronous', True)):
        if world == 1 and sync:
            continue
        mode5 = FILL_MODE or ('pipelined' if nb >= 64 else 'fused')
        rec5['dU_zero_fill'] = mode5
        step5, _, _, _, _ = make_step(set5 * 2, feats5, red5, sync_reduce=sync, fill_mode=mode5)
        k5 = 20
        ms5 = timed(step5, k5, 3)
        rec5['ms_per_step_' + name] = ms5 / k5
        rec5['mpix_per_s_' + name] = nb * world * H * W * k5 / (ms5 * 1e-3) / 1e6
    if world == 1:
        rec5['note'] = 'one rank: no collective; ms_per_step_overlapped is the 256-frame step on one GPU'
    res['config5_dp_train_step_256'] = rec5
    return res


def finish(world):
    """multi-rank teardown: CUDA graphs that captured NCCL kernels are still alive, and destroying the process group under
    them can hang; flush and leave (exit code 0) once every rank is done."""
    sys.stdout.flush()
    sys.stderr.flush()
    if world > 1:
        import torch.distributed as dist
        torch.cuda.synchronize()
        dist.barrier()
        torch.cuda.synchronize()
        os._exit(0)


if __name__ == '__main__':
    main()

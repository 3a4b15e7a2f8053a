"""bench.py --dump-outputs: the same seeded sample of frames of every output, as float32, within its byte budget (CPU); on the
GPU, what the last timed step of the benchmark computed."""
import importlib.util
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from conftest import bits_equal, relmax

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def load_bench():
    spec = importlib.util.spec_from_file_location('bench', os.path.join(ROOT, 'bench.py'))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def test_dump_outputs_sample_and_budget(tmp_path, monkeypatch):
    bench = load_bench()
    n, h, w, c = 9, 6, 10, 3
    g = torch.Generator().manual_seed(0)
    outs = dict(out=torch.randn(n, h, w, c, generator=g), black=torch.rand(n, h, w, generator=g),
                img=torch.randn(n, h, w, 2, generator=g), Hs=torch.randn(n, 2, 2, 9, generator=g),
                dU=torch.randn(n, h, w, c, generator=g), dtheta=torch.randn(n, 3, 3, 2, generator=g))
    per_frame = sum(t[0].numel() * 4 for t in outs.values())
    monkeypatch.setattr(bench, 'DUMP_BYTES', 4 * per_frame + 1)
    frames = bench.dump_outputs(str(tmp_path / 'a'), outs)
    assert len(frames) == 4 and frames == sorted(set(frames)) and all(0 <= f < n for f in frames)
    assert bench.dump_outputs(str(tmp_path / 'b'), outs) == frames
    total = 0
    for name, t in outs.items():
        a, b = np.load(tmp_path / 'a' / (name + '.npy')), np.load(tmp_path / 'b' / (name + '.npy'))
        assert a.dtype == np.float32 and np.array_equal(a, t.numpy()[frames]) and np.array_equal(a, b), name
        total += a.nbytes
    assert total <= bench.DUMP_BYTES
    # a batch smaller than the budget is written whole
    monkeypatch.setattr(bench, 'DUMP_BYTES', 100 * per_frame)
    assert bench.dump_outputs(str(tmp_path / 'c'), outs) == list(range(n))


@pytest.mark.gpu
def test_bench_dumps_the_last_timed_step(tmp_path):
    """a short run (graph replay, 3 rotating input sets): the dump equals the step recomputed on the inputs of the last timed
    step -- warmup max(3, W) + K steps, so the last one used set (max(3, W) + K - 1) % 3 = np.roll(inputs, that, axis=0)"""
    import dovs_b200 as mgw
    steps, warmup, n = 5, 3, 4
    r = subprocess.run([sys.executable, 'bench.py', '--gpus', '1', '--steps', str(steps), '--warmup', str(warmup), '--batch', str(n),
                        '--no-configs', '--no-cpu-baseline', '--dump-outputs', str(tmp_path)],
                       cwd=ROOT, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-3000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line['steps'] == steps and line['config']['launch'] == 'cuda graph replay'
    assert line['dump_outputs']['frames'] == list(range(n))
    bench = load_bench()
    k = (warmup + steps - 1) % 3
    s = {key: torch.tensor(np.roll(v, k, axis=0), device='cuda') for key, v in bench.synth_inputs(n).items()}
    out, black, img, Hs = mgw.ops.mesh_warp_fwd(s['U'], s['theta'])
    dU, dtheta = mgw.ops.mesh_warp_bwd(s['U'], s['theta'], Hs, s['d_out'], s['d_img'])
    for name, want in dict(out=out, black=black, img=img, Hs=Hs, dtheta=dtheta).items():
        assert bits_equal(np.load(tmp_path / (name + '.npy')), want.cpu().numpy()).all(), name
    # the reductions into dU arrive in any order: fp32 summation noise
    assert relmax(np.load(tmp_path / 'dU.npy'), dU.cpu().numpy()) <= 2e-6

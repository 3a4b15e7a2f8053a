"""Stabilising videos of different sizes straight from decoder surfaces: MixedStreamBatch.capture_planes (mixed plane tables)
against the route without them, strided copies into the packed pool around MixedStreamBatch.step.

S = 64 NV12 sources, each in its own surface in NVDEC's layout (pitch rounded up to 512 bytes, the chroma plane at the coded
height, rows rounded up to 16), out_size='source' with NV12 output into pitched encoder surfaces of the same layout, a fixed mesh
in place of the network (tools/bench_streams.fixed_mesh_net), refine 1.  The workloads are tools/bench_mixed.py's:
  few_sizes    24 x 1080p, 24 x 720p, 8 x 480x854, 8 x 1920x1080 (portrait), capacity 1920x1920
  fragmented   16 sizes x 4 streams from 240x426 to 2160x3840, capacity 2160x3840
Arms, each captured as one CUDA graph:
  (A) capture_planes: the two table uploads, then the step reading the source surfaces and writing the encoder surfaces;
  (B) per slot and plane one strided copy (torch copy_ of the pitched view, one cudaMemcpyAsync each) into the packed pool,
      MixedStreamBatch.step, then per slot and plane one strided copy out of the output pool into the encoder surfaces.
Before timing, one replay of each arm on the same frames must give the same output bytes.  The arms are then timed alternately in
--rounds rounds (device time of one replay, CUDA events, median).  Reported per workload and arm: us per step and per frame, and
the copy operations and HBM bytes that (A) removes, counted from shapes (each copy reads and writes its bytes once).
Prints one JSON object (the GPU's name and power limit included); --out also writes it to a file."""
import argparse, json, os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, 'tools'))

h, w = 288, 512
FEW = [((1080, 1920), 24), ((720, 1280), 24), ((480, 854), 8), ((1920, 1080), 8)]
FRAGMENTED = [((H, W), 4) for H, W in [(240, 426), (270, 480), (360, 640), (480, 640), (480, 854), (540, 960), (576, 1024), (640, 360),
                                       (720, 1280), (960, 540), (1080, 1080), (1080, 1440), (1080, 1920), (1280, 720), (1440, 2560),
                                       (2160, 3840)]]


def nvdec_surface(torch, H, W):
    """one NV12 surface as NVDEC lays it out: (allocation, Y view [H,W], UV view [H/2,W])"""
    pitch, coded = -(-W // 512) * 512, -(-H // 16) * 16
    a = torch.zeros(pitch * (coded + coded // 2), dtype=torch.uint8, device='cuda')
    y = a[:pitch * H].view(H, pitch)[:, :W]
    uv = a[pitch * coded:pitch * coded + pitch * (H // 2)].view(H // 2, pitch)[:, :W]
    return a, y, uv


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--reps', type=int, default=200)
    ap.add_argument('--rounds', type=int, default=5)
    ap.add_argument('--workloads', default='few_sizes,fragmented')
    ap.add_argument('--out')
    a = ap.parse_args()
    sys.path.insert(0, ROOT)
    import numpy as np, torch
    assert torch.cuda.is_available(), 'bench_mixed_planes.py measures on the GPU; there is nothing to measure without one'
    import dovs_b200 as mgw
    from bench_streams import dev_time, fixed_mesh_net, gpu_info
    res = {'gpu': gpu_info(), 'source': 'nv12, one NVDEC-layout surface per stream (pitch rounded to 512, chroma at the coded height)',
           'output': "out_size='source', nv12 into NVDEC-layout encoder surfaces", 'network_size': '%dx%d' % (h, w), 'refine': 1,
           'net': 'fixed mesh (tools/bench_streams.fixed_mesh_net)', 'reps': a.reps, 'rounds': a.rounds, 'per_workload': {}}
    gen = torch.Generator(device='cuda')
    gen.manual_seed(0)
    todo = a.workloads.split(',')
    for name, groups, cap in (('few_sizes', FEW, (1920, 1920)), ('fragmented', FRAGMENTED, (2160, 3840))):
        if name not in todo:
            continue
        sizes = [sz for sz, n in groups for _ in range(n)]
        S = len(sizes)
        src = [nvdec_surface(torch, *sz) for sz in sizes]
        dst = [nvdec_surface(torch, *sz) for sz in sizes]
        for (_, y, uv), (H, W) in zip(src, sizes):
            y.copy_(torch.randint(0, 256, (H, W), dtype=torch.uint8, device='cuda', generator=gen))
            uv.copy_(torch.randint(0, 256, (H // 2, W), dtype=torch.uint8, device='cuda', generator=gen))
        kw = dict(height=h, width=w, refine=1, src_format='nv12', out_size='source', out_format='nv12')
        ma, mb = mgw.MixedStreamBatch(S, cap, **kw), mgw.MixedStreamBatch(S, cap, **kw)
        pool = torch.zeros(mb.pool_shape, dtype=torch.uint8, device='cuda')
        st, dt = mgw.MixedPlaneTable(S, 'nv12', cap), mgw.MixedPlaneTable(S, 'nv12', cap)
        for s, (H, W) in enumerate(sizes):
            first = torch.cat([src[s][1], src[s][2]])
            ma.join(s, first); mb.join(s, first)
            st.set(s, (src[s][1], src[s][2]), (H, W))
            dt.set(s, (dst[s][1], dst[s][2]), (H, W))
        with torch.no_grad():
            g_a = ma.capture_planes(st, fixed_mesh_net(ma), dt)

            def copies_in():
                for s, (H, W) in enumerate(sizes):
                    f = mb.slot_frame(pool, s)
                    f[:H].copy_(src[s][1]); f[H:].copy_(src[s][2])

            def copies_out():
                for s, (H, W) in enumerate(sizes):
                    o = mb.slot_output(mb.colour, s)
                    dst[s][1].copy_(o[:H]); dst[s][2].copy_(o[H:])
            net_b = fixed_mesh_net(mb)                          # built outside the capture: it copies a host mesh to the device
            g_b = mb._record(lambda: mb.step(pool, net_b), copies_in, copies_out, warm_upload=True)
            # one replay of each on the same frames and state: the same output bytes
            g_a.replay(); torch.cuda.synchronize()
            got = [torch.cat([d[1].reshape(-1), d[2].reshape(-1)]) for d in dst]
            for d in dst:
                d[0].zero_()
            g_b.replay(); torch.cuda.synchronize()
            for s in range(S):
                assert torch.equal(got[s], torch.cat([dst[s][1].reshape(-1), dst[s][2].reshape(-1)])), (name, s, sizes[s])
            del got
            ta, tb = [], []
            per = max(a.reps // a.rounds, 10)
            for _ in range(a.rounds):
                ta.append(dev_time(g_a.replay, per))
                tb.append(dev_time(g_b.replay, per))
        t_a, t_b = float(np.median(ta)), float(np.median(tb))
        frame_bytes = sum(H * W * 3 // 2 for H, W in sizes)
        r = {'S': S, 'capacity': '%dx%d' % cap, 'sizes': {'%dx%d' % sz: n for sz, n in groups},
             'A_capture_planes': {'us_per_step': t_a, 'us_per_frame': t_a / S, 'us_per_round': ta},
             'B_copies_and_step': {'us_per_step': t_b, 'us_per_frame': t_b / S, 'us_per_round': tb},
             'A_over_B_time': t_a / t_b, 'A_faster': t_a < t_b,
             'removed_by_A': {'copy_operations_per_step': 4 * S, 'hbm_bytes_per_step': 4 * frame_bytes,
                              'hbm_bytes_per_frame': 4 * frame_bytes / S}}
        res['per_workload'][name] = r
        print(json.dumps({name: r}), file=sys.stderr)
        del g_a, g_b, ma, mb, pool, src, dst, st, dt
        torch.cuda.empty_cache()
    print(json.dumps(res, indent=1))
    if a.out:
        with open(a.out, 'w') as f:
            json.dump(res, f, indent=1)


if __name__ == '__main__':
    main()

"""Stabilising straight from decoder surfaces: StreamBatch.capture_planes (plane tables) against today's route of strided copies
into the packed batch around StreamBatch.step.

S = 64 1080p NV12 sources in the NVDEC layout (one allocation per surface, pitch 2048, the chroma plane at row 1088), a fixed mesh
in place of the network (tools/bench_fullres.py's leg (a)), refine 1.  Cases:
  bgr_288x512     the network-size BGR output in StreamBatch.colour (no copies out in either arm)
  nv12_1080p      1080p NV12 output into pitched encoder surfaces of the same layout
  nv12_1080p_half the same with every other slot idle: (A) clears both table entries, so the front end and the warp skip the slot;
                  (B) copies only the active slots' planes, and the step still computes every slot
Arms, each captured as one CUDA graph:
  (A) capture_planes: the two table uploads, then the step reading and writing the surfaces;
  (B) per slot and plane one strided copy (torch copy_ of the pitched view) into the packed [S,3H/2,W] batch, StreamBatch.step,
      then per slot and plane one strided copy out of StreamBatch.colour into the pitched surfaces.
Before timing, one replay of each arm on the same frames must give the same output bytes.  The arms are then timed alternately in
--rounds rounds (device time of one replay, CUDA events, median).  Reported per case and arm: us per step and per frame, and the
copy operations and HBM bytes that (A) removes, counted from shapes (each copy reads and writes its bytes once).
Prints one JSON object (the GPU's name and power limit included); --out also writes it to a file."""
import argparse, json, os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, 'tools'))

H, W, h, w = 1080, 1920, 288, 512
PITCH, CODED = 2048, 1088


def nvdec_surface(torch, fmt, Hs, Ws):
    """one NV12 surface as NVDEC lays it out: (allocation, Y view [Hs,Ws], UV view [Hs/2,Ws]) with pitch PITCH"""
    a = torch.zeros(PITCH * (CODED + CODED // 2), dtype=torch.uint8, device='cuda')
    y = a[:PITCH * Hs].view(Hs, PITCH)[:, :Ws]
    uv = a[PITCH * CODED:PITCH * CODED + PITCH * (Hs // 2)].view(Hs // 2, PITCH)[:, :Ws]
    return a, y, uv


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--streams', type=int, default=64)
    ap.add_argument('--reps', type=int, default=200)
    ap.add_argument('--rounds', type=int, default=5)
    ap.add_argument('--out')
    a = ap.parse_args()
    sys.path.insert(0, ROOT)
    import numpy as np, torch
    assert torch.cuda.is_available(), 'bench_planes.py measures on the GPU; there is nothing to measure without one'
    import dovs_b200 as mgw
    from bench_streams import dev_time, fixed_mesh_net, gpu_info
    S = a.streams
    res = {'gpu': gpu_info(), 'source': 'nv12 %dx%d, NVDEC layout (pitch %d, chroma at row %d)' % (H, W, PITCH, CODED), 'S': S,
           'network_size': '%dx%d' % (h, w), 'refine': 1, 'net': 'fixed mesh (tools/bench_streams.fixed_mesh_net)', 'per_case': {}}
    gen = torch.Generator(device='cuda')
    gen.manual_seed(0)
    src = [nvdec_surface(torch, 'nv12', H, W) for _ in range(S)]
    for _, y, uv in src:
        y.copy_(torch.randint(0, 256, (H, W), dtype=torch.uint8, device='cuda', generator=gen))
        uv.copy_(torch.randint(0, 256, (H // 2, W), dtype=torch.uint8, device='cuda', generator=gen))
    for case, out_size, out_format, half in (('bgr_288x512', None, 'bgr', False), ('nv12_1080p', (H, W), 'nv12', False),
                                             ('nv12_1080p_half', (H, W), 'nv12', True)):
        active = [s for s in range(S) if not half or s % 2 == 0]
        pitched_out = out_format == 'nv12'
        dst = [nvdec_surface(torch, 'nv12', H, W) for _ in range(S)] if pitched_out else None
        kw = dict(height=h, width=w, refine=1, src_format='nv12', out_size=out_size, out_format=out_format)
        sa, sb = mgw.StreamBatch(S, (H, W), **kw), mgw.StreamBatch(S, (H, W), **kw)
        raw = torch.zeros((S, H * 3 // 2, W), dtype=torch.uint8, device='cuda')
        for s in range(S):
            raw[s, :H].copy_(src[s][1]); raw[s, H:].copy_(src[s][2])
            sa.join(s, raw[s]); sb.join(s, raw[s])
        st = mgw.PlaneTable(S, 'nv12', (H, W))
        dt = mgw.PlaneTable(S, 'nv12', (H, W)) if pitched_out else None
        for s in range(S):
            if s in active:
                st.set(s, (src[s][1], src[s][2]))
                if dt is not None:
                    dt.set(s, (dst[s][1], dst[s][2]))
        with torch.no_grad():
            g_a = sa.capture_planes(st, fixed_mesh_net(sa), dt)

            def copies_in():
                for s in active:
                    raw[s, :H].copy_(src[s][1]); raw[s, H:].copy_(src[s][2])

            def copies_out():
                for s in active:
                    dst[s][1].copy_(sb.colour[s, :H]); dst[s][2].copy_(sb.colour[s, H:])
            net_b = fixed_mesh_net(sb)                          # built outside the capture: it copies a host mesh to the device
            g_b = sb._record(lambda: sb.step(raw, net_b), copies_in, copies_out if pitched_out else None, warm_upload=True)
            # one replay of each on the same frames and state: the same output bytes
            g_a.replay(); g_b.replay(); torch.cuda.synchronize()
            for s in active:
                got = torch.cat([dst[s][1].reshape(-1), dst[s][2].reshape(-1)]) if pitched_out else sa.colour[s].reshape(-1)
                want = sb.colour[s].reshape(-1)
                assert torch.equal(got, want), (case, s)
                if pitched_out:
                    dst[s][1].zero_(); dst[s][2].zero_()
            ta, tb = [], []
            per = max(a.reps // a.rounds, 10)
            for _ in range(a.rounds):
                ta.append(dev_time(g_a.replay, per))
                tb.append(dev_time(g_b.replay, per))
        t_a, t_b = float(np.median(ta)), float(np.median(tb))
        frame = H * W * 3 // 2
        n_in, n_out = 2 * len(active), (2 * len(active) if pitched_out else 0)
        removed = 2 * frame * len(active) + (2 * frame * len(active) if pitched_out else 0)
        r = {'active_slots': len(active), 'output': '%s %s%s' % (out_format, 'x'.join(map(str, sa.out_size)),
                                                                ' into pitched surfaces' if pitched_out else ' in StreamBatch.colour'),
             'A_capture_planes': {'us_per_step': t_a, 'us_per_frame': t_a / len(active), 'us_per_round': ta},
             'B_copies_and_step': {'us_per_step': t_b, 'us_per_frame': t_b / len(active), 'us_per_round': tb},
             'A_over_B_time': t_a / t_b, 'A_faster': t_a < t_b,
             'removed_by_A': {'copy_operations_per_step': n_in + n_out, 'hbm_bytes_per_step': removed,
                              'hbm_bytes_per_frame': removed / len(active)}}
        res['per_case'][case] = r
        print(json.dumps({case: r}), file=sys.stderr)
        del g_a, g_b, sa, sb, raw, dst, st, dt
        torch.cuda.empty_cache()
    print(json.dumps(res, indent=1))
    if a.out:
        with open(a.out, 'w') as f:
            json.dump(res, f, indent=1)


if __name__ == '__main__':
    main()

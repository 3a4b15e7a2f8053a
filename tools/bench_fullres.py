"""Stabilised video at any output size: deploy.StreamBatch(out_size=...) on 1080p sources, BGR and NV12, S in 1, 16, 64, outputs
288x512 (the network's size, the default path), 720x1280 and 1080x1920 (the source's size: no resize, the warp reads the source).

Per (format, S, output):
  (a) device time of one replayed step with the frames resident and a fixed mesh in place of the network (tools/bench_streams.py's
      leg (a));
  (b) host-to-host time per step with the upload of the raw frames and the download of the [S,OH,OW,3] colour frames inside the
      graph (pinned host buffers), and the bytes each frame moves over PCIe;
  the remap call alone (mgw_remap_bundle_frame: the /4 maps and the warp at the output size, with a smooth mesh near the
  identity) from CUDA events around many back-to-back launches, with its algorithmic HBM bytes (colour frames read once and written once, maps read once), the share of
  the B200's 7.7 TB/s those bytes take in that time, and the bound that applies (bytes; the call does no tensor-core work).  At
  S = 1 the frames fit in the 126 MB L2, so that row is an L2 figure, not an HBM one.
--ab-parent DIR: also times leg (a) of today's 288x512 path at S = 1 and 64 with this tree's library and with the library of the
tree in DIR (the parent build), alternately in rounds, each arm in its own process (the library is loaded once per process).
--out-formats bgr,nv12,i420: instead, StreamBatch(out_format=...) per (source format, S, output in 288x512 and 1080x1920): legs
(a) and (b) -- (b) with the [S,OH,OW,3] or [S,3OH/2,OW] download inside the graph -- and the remap call alone (its output written
at 3 or 1.5 bytes per pixel), each out_format's arm timed alternately with the others in the same process, in rounds.
Prints one JSON object (the GPU's name and power limit included); --out also writes it to a file."""
import argparse, json, os, subprocess, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, 'tools'))

H, W, h, w = 1080, 1920, 288, 512
OUTS = ((288, 512), (720, 1280), (1080, 1920))
HBM_BYTES_PER_S = 7.7e12


def frame_bytes(fmt, Hs, Ws):
    return Hs * Ws * 3 if fmt == 'bgr' else Hs * Ws * 3 // 2


def ab_leg(root, S_list, reps):
    """leg (a) of the default 288x512 path, with the package of `root`: one JSON line {S: us}"""
    sys.path.insert(0, root); sys.path.insert(0, os.path.join(root, 'oracle'))
    import numpy as np, torch
    import dovs_b200 as mgw, synth
    rs, res = np.random.RandomState(0), {}
    for S in S_list:
        sb = mgw.StreamBatch(S, (H, W), height=h, width=w, refine=1)
        for s in range(S):
            sb.join(s, torch.as_tensor(rs.randint(0, 256, (H, W, 3)).astype(np.uint8)).cuda())
        raw = torch.as_tensor(rs.randint(0, 256, (S, H, W, 3)).astype(np.uint8)).cuda()
        th = torch.tensor(synth.random_mesh(S, 4, 4, 0.03, 4), device='cuda')
        cur = sb.cur.view(S, h, w, 1)
        with torch.no_grad():
            g = sb.capture(raw, lambda in_x: mgw.transformer(cur, th))
        for _ in range(20):
            g.replay()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ts = []
        for _ in range(reps):
            e0.record(); g.replay(); e1.record(); torch.cuda.synchronize()
            ts.append(e0.elapsed_time(e1) * 1e3)
        res[str(S)] = float(np.median(ts))
    print(json.dumps(res))


def remap_call(mgw, torch, np, fmt, S, OH, OW, rs, out_format='bgr'):
    """(one mgw_remap_bundle_frame call as a closure, the source format it reads, its algorithmic HBM bytes)"""
    direct = (OH, OW) == (H, W)
    src_fmt = fmt if direct else 'bgr'
    shape = ((S, OH, OW, 3) if src_fmt == 'bgr' else (S, OH * 3 // 2, OW))
    src = torch.randint(0, 256, shape, device='cuda', dtype=torch.uint8, generator=torch.Generator('cuda').manual_seed(int(rs.randint(1 << 30))))
    # a smooth mesh near the identity, as the network emits it (random maps would turn the taps into scattered gathers)
    ys, xs = torch.meshgrid(torch.linspace(-1, 1, h, device='cuda'), torch.linspace(-1, 1, w, device='cuda'), indexing='ij')
    xy = torch.stack([0.93 * xs + 0.02 * torch.sin(3 * ys), 0.95 * ys + 0.03 * torch.cos(2 * xs)], -1)[None].repeat(S, 1, 1, 1).contiguous()
    out_bytes = frame_bytes(out_format, OH, OW)
    out = torch.empty((S, out_bytes), device='cuda', dtype=torch.uint8).view((S, OH, OW, 3) if out_format == 'bgr' else (S, OH * 3 // 2, OW))
    ws = torch.empty(mgw.ops.remap_bundle_workspace_floats(S, h, w), device='cuda')
    call = lambda: mgw.ops.remap_bundle_frame(src, src_fmt, xy, out=out, workspace=ws, out_format=out_format)      # noqa: E731
    nbytes = S * (out_bytes + frame_bytes(src_fmt, OH, OW)) + S * h * w * 8 + S * (h // 4) * (w // 4) * 8 * 2
    return call, src_fmt, nbytes


def time_launches(torch, call, launches):
    """mean device time of one call over `launches` back-to-back calls"""
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(launches):
        call()
    e1.record(); torch.cuda.synchronize()
    return e0.elapsed_time(e1) * 1e3 / launches


def remap_report(t, src_fmt, nbytes, S):
    return {'us': t, 'source_read': src_fmt, 'algorithmic_bytes': nbytes, 'GB_per_s': nbytes / t / 1e3,
            'share_of_7.7TB_per_s': nbytes / HBM_BYTES_PER_S / (t * 1e-6), 'bound': 'HBM bytes' if S > 1 else 'bytes (L2 resident at S = 1)'}


def remap_alone(mgw, torch, np, fmt, S, OH, OW, rs, launches=50, rounds=5):
    """mean device time of one mgw_remap_bundle_frame call over `launches` back-to-back calls (median of `rounds`)"""
    call, src_fmt, nbytes = remap_call(mgw, torch, np, fmt, S, OH, OW, rs)
    for _ in range(5):
        call()
    t = float(np.median([time_launches(torch, call, launches) for _ in range(rounds)]))
    return remap_report(t, src_fmt, nbytes, S)


def out_formats_main(a, mgw, torch, np, res):
    """--out-formats: per (source format, S, output) one StreamBatch per out_format, timed alternately in a.rounds rounds"""
    from bench_streams import dev_time, fixed_mesh_net, host_times, summary
    ofs = a.out_formats.split(',')
    res['out_formats'] = ofs
    rs = np.random.RandomState(0)
    for fmt in a.formats.split(','):
        for S in [int(v) for v in a.streams.split(',')]:
            for OH, OW in ((h, w), (H, W)):
                key = '%s_S%d_%dx%d' % (fmt, S, OH, OW)
                fshape = (H, W, 3) if fmt == 'bgr' else (H * 3 // 2, W)
                raw_d = torch.randint(0, 256, (S,) + fshape, device='cuda', dtype=torch.uint8)
                raw_h = raw_d.cpu().pin_memory()
                arms = {}
                with torch.no_grad():
                    for of in ofs:
                        sb = mgw.StreamBatch(S, (H, W), height=h, width=w, refine=1, src_format=fmt,
                                             out_size=None if (OH, OW) == (h, w) else (OH, OW), out_format=of)
                        for s in range(S):
                            sb.join(s, raw_d[s])
                        out_h = torch.empty(sb.colour.shape, dtype=torch.uint8).pin_memory()
                        net = fixed_mesh_net(sb)
                        arms[of] = dict(sb=sb, out_h=out_h, g_res=sb.capture(raw_d, net), g_io=sb.capture(raw_d, net, upload_from=raw_h, download_to=out_h),
                                        remap=remap_call(mgw, torch, np, fmt, S, OH, OW, rs, out_format=of), dev=[], host=[], remap_us=[])
                    per = max(a.reps // a.rounds, 5)
                    for _ in range(a.rounds):
                        for of, arm in arms.items():
                            arm['dev'].append(dev_time(arm['g_res'].replay, per))
                            arm['host'] += host_times(arm['g_io'].replay, per)
                            call = arm['remap'][0]
                            for _ in range(3):
                                call()
                            arm['remap_us'].append(time_launches(torch, call, 50))
                r = {}
                for of, arm in arms.items():
                    t = float(np.median(arm['dev']))
                    d2h = frame_bytes(of, OH, OW)
                    r[of] = {'a_us_device_step_fixed_mesh_resident': t, 'a_us_device_per_frame': t / S,
                             'b_host_to_host_fixed_mesh': summary(arm['host'], S),
                             'bytes_pcie_per_frame': {'h2d_raw': frame_bytes(fmt, H, W), 'd2h_colour': d2h, 'total': frame_bytes(fmt, H, W) + d2h},
                             'remap_call_alone': remap_report(float(np.median(arm['remap_us'])), arm['remap'][1], arm['remap'][2], S)}
                if 'bgr' in r:
                    for of in ofs:
                        if of != 'bgr':
                            r[of]['vs_bgr_out'] = {
                                'host_to_host_frames_per_s_ratio': r[of]['b_host_to_host_fixed_mesh']['frames_per_s'] / r['bgr']['b_host_to_host_fixed_mesh']['frames_per_s'],
                                'device_step_time_ratio': r[of]['a_us_device_step_fixed_mesh_resident'] / r['bgr']['a_us_device_step_fixed_mesh_resident'],
                                'remap_call_time_ratio': r[of]['remap_call_alone']['us'] / r['bgr']['remap_call_alone']['us']}
                del arms, raw_h, raw_d
                torch.cuda.empty_cache()
                res['per_case'][key] = r
                print(json.dumps({key: r}), file=sys.stderr)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--streams', default='1,16,64')
    ap.add_argument('--formats', default='bgr,nv12')
    ap.add_argument('--reps', type=int, default=100)
    ap.add_argument('--ab-parent', help='a tree of the parent commit with its library built')
    ap.add_argument('--ab-rounds', type=int, default=4)
    ap.add_argument('--ab-leg', help=argparse.SUPPRESS)
    ap.add_argument('--out-formats', help='e.g. bgr,nv12,i420: compare the output formats (outputs 288x512 and 1080x1920)')
    ap.add_argument('--rounds', type=int, default=5, help='--out-formats: alternation rounds (reps are split over them)')
    ap.add_argument('--out')
    a = ap.parse_args()
    if a.ab_leg:
        return ab_leg(a.ab_leg, (1, 64), a.reps)
    sys.path.insert(0, ROOT)
    import numpy as np, torch
    assert torch.cuda.is_available(), 'bench_fullres.py measures on the GPU; there is nothing to measure without one'
    import dovs_b200 as mgw
    from bench_streams import dev_time, fixed_mesh_net, gpu_info, host_times, summary
    res = {'gpu': gpu_info(), 'source': '%dx%d' % (H, W), 'network_size': '%dx%d' % (h, w), 'refine': 1, 'per_case': {}}
    rs = np.random.RandomState(0)
    for fmt in ([] if a.out_formats else a.formats.split(',')):
        for S in [int(v) for v in a.streams.split(',')]:
            for OH, OW in OUTS:
                key = '%s_S%d_%dx%d' % (fmt, S, OH, OW)
                fshape = (H, W, 3) if fmt == 'bgr' else (H * 3 // 2, W)
                sb = mgw.StreamBatch(S, (H, W), height=h, width=w, refine=1, src_format=fmt,
                                     out_size=None if (OH, OW) == (h, w) else (OH, OW))
                for s in range(S):
                    sb.join(s, torch.as_tensor(rs.randint(0, 256, fshape).astype(np.uint8)).cuda())
                raw_h = torch.as_tensor(rs.randint(0, 256, (S,) + fshape).astype(np.uint8)).pin_memory()
                raw_d = raw_h.cuda()
                out_h = torch.empty((S, OH, OW, 3), dtype=torch.uint8).pin_memory()
                r = {}
                with torch.no_grad():
                    net = fixed_mesh_net(sb)
                    g_res = sb.capture(raw_d, net)
                    t = dev_time(g_res.replay, a.reps)
                    r['a_us_device_step_fixed_mesh_resident'] = t
                    r['a_us_device_per_frame'] = t / S
                    g_io = sb.capture(raw_d, net, upload_from=raw_h, download_to=out_h)
                    r['b_host_to_host_fixed_mesh'] = summary(host_times(g_io.replay, a.reps), S)
                    r['bytes_pcie_per_frame'] = {'h2d_raw': frame_bytes(fmt, H, W), 'd2h_colour': OH * OW * 3,
                                                 'total': frame_bytes(fmt, H, W) + OH * OW * 3}
                    del g_res, g_io
                    r['remap_call_alone'] = remap_alone(mgw, torch, np, fmt, S, OH, OW, rs)
                del sb, raw_h, raw_d, out_h
                torch.cuda.empty_cache()
                res['per_case'][key] = r
                print(json.dumps({key: r}), file=sys.stderr)
    if a.out_formats:
        out_formats_main(a, mgw, torch, np, res)
    if a.ab_parent:
        arms = {'this_build': ROOT, 'parent_build': os.path.abspath(a.ab_parent)}
        rounds = {k: [] for k in arms}
        for _ in range(a.ab_rounds):
            for name, root in arms.items():
                p = subprocess.run([sys.executable, os.path.abspath(__file__), '--ab-leg', root, '--reps', str(a.reps * 3)],
                                   capture_output=True, text=True, cwd=root, timeout=900)
                if p.returncode != 0:
                    raise RuntimeError('%s arm failed: %s' % (name, p.stderr[-2000:]))
                rounds[name].append(json.loads(p.stdout.strip().splitlines()[-1]))
        res['ab_288x512_a_us_device_step_per_round'] = rounds
        res['ab_288x512_a_us_device_step_median'] = {k: {S: float(np.median([r[S] for r in v])) for S in ('1', '64')}
                                                     for k, v in rounds.items()}
    print(json.dumps(res, indent=1))
    if a.out:
        with open(a.out, 'w') as f:
            json.dump(res, f, indent=1)


if __name__ == '__main__':
    main()

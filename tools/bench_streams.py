"""Several videos at once: deploy.StreamBatch advancing S 1080p streams per step, one CUDA graph per step, for S in 1, 4, 16, 64.

Per S:
  (a) device time of one replayed step with the frames resident on the device and a fixed mesh in place of the network
      (cvt_img2train, ring assembly, the multi-grid warp on the current frame, black accumulation, re-feed, ring push,
      cv2.resize of the colour frame, warpRevBundle2): the library's share of a step;
  (b) host-to-host time per step with the upload of the raw 1080p BGR frames and the download of the stabilised 512x288 colour
      frames inside the graph (pinned host buffers): p50, p99 and frames/s; beside it the two copies alone;
  (c) the same with the StabNet carrier (torch / cuDNN ResNet-50, random init, fp32) as the network at batch S;
  and the bytes each frame moves over PCIe.
First the S = 1 step against the single-stream graph loop of tools/bench_configs.py (one stream, one refine pass, fixed mesh; that
loop has no refine re-feed, so it is also timed with one), timed alternately in rounds.  refine = 1 throughout.
--src-format nv12 / i420: the same legs (a), (b), (c) with YUV 4:2:0 frames [S,1620,1920] uploaded instead of BGR (half the bytes;
the conversion runs inside the kernels that read the source), no single-stream comparison, and at S = 1 and S = 64 the BGR batch's
(a) and (b) timed alternately with the YUV batch's in rounds, in the same process.
Prints one JSON object (the GPU's name and power limit included); --out also writes it to a file."""
import argparse, json, os, subprocess, sys, time
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, 'oracle'))
import numpy as np, torch
import synth, dovs_b200 as mgw

dev = 'cuda'
H, W, h, w = 1080, 1920, 288, 512


def gpu_info():
    try:
        q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'], capture_output=True,
                           text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception as e:      # noqa: BLE001
        q = 'nvidia-smi unavailable: %s' % e
    return {'device': torch.cuda.get_device_name(0), 'nvidia_smi_name_power_limit_max_sm_clock': q}


def dev_time(fn, reps):
    for _ in range(5):
        fn()
    ts = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); fn(); e1.record(); torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1) * 1e3)
    return float(np.median(ts))


def host_times(fn, reps):
    for _ in range(5):
        fn(); torch.cuda.synchronize()
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter(); fn(); torch.cuda.synchronize(); ts.append((time.perf_counter() - t0) * 1e6)
    return ts


def summary(ts, S):
    p50 = float(np.percentile(ts, 50))
    return {'us_p50': p50, 'us_p99': float(np.percentile(ts, 99)), 'frames_per_s': S * 1e6 / p50}


def fixed_mesh_net(sb):
    """the warp of the current frame with a fixed mesh; with refine = 1 the current frame is the last channel of in_x, read
    here from the batch's cvt_img2train output (no copy, as tools/bench_configs.py's loop warps its `cur`)"""
    S = sb.S
    th = torch.tensor(synth.random_mesh(S, 4, 4, 0.03, 4), device=dev)
    cur = sb.cur.view(S, h, w, 1)

    def net(in_x):
        return mgw.transformer(cur, th)
    return net


def stabnet_net(model):
    def net(in_x):
        theta = model(in_x)
        _, pts2 = mgw.get_4_pts(theta, grid=(4, 4))
        return mgw.transformer(in_x[..., -1:].contiguous(), pts2)
    return net


def frame_shape(fmt):
    return (H, W, 3) if fmt == 'bgr' else (H * 3 // 2, W)


def make_batch(S, rs, fmt='bgr'):
    sb = mgw.StreamBatch(S, (H, W), height=h, width=w, refine=1, src_format=fmt)
    for s in range(S):
        sb.join(s, torch.as_tensor(rs.randint(0, 256, frame_shape(fmt)).astype(np.uint8)).to(dev))
    raw_h = torch.as_tensor(rs.randint(0, 256, (S,) + frame_shape(fmt)).astype(np.uint8)).pin_memory()
    raw_d = raw_h.to(dev)
    out_h = torch.empty((S, h, w, 3), dtype=torch.uint8).pin_memory()
    return sb, raw_h, raw_d, out_h


def single_stream_graph(rs, refeed=False):
    """tools/bench_configs.py's whole-deploy-loop graph (one stream, device head, upload and download inside the graph);
    refeed: plus the refine re-feed of the network input (StreamState.refeed), which StreamBatch runs after every pass"""
    th = torch.tensor(synth.random_mesh(1, 4, 4, 0.03, 4), device=dev)
    first = mgw.deploy.cvt_img2train(torch.as_tensor(rs.randint(0, 256, (H, W, 3)).astype(np.uint8)).to(dev))
    raw_h = torch.as_tensor(rs.randint(0, 256, (H, W, 3)).astype(np.uint8)).pin_memory()
    raw_d = torch.empty((H, W, 3), device=dev, dtype=torch.uint8)
    out_hh = torch.empty((h, w, 3), dtype=torch.uint8).pin_memory()
    st_g = mgw.StreamState(first.reshape(h, w), device_head=True)
    crop = mgw.CropState(h, w)
    in_x_g = torch.empty((1, h, w, 13), device=dev)

    def graph_frame():
        raw_d.copy_(raw_h, non_blocking=True)
        cur = mgw.deploy.cvt_img2train(raw_d)
        st_g.assemble(cur.reshape(h, w), out=in_x_g)
        out, black, img = mgw.transformer(cur, th)
        if refeed:
            st_g.refeed(in_x_g, out, black)
        st_g.push(out.reshape(h, w), black.reshape(h, w))
        crop.add(black)
        small = mgw.deploy.cv2_resize(raw_d, (w, h))
        dst = mgw.ops.remap_bundle_u8(small.reshape(1, h, w, 3), img)
        out_hh.copy_(dst[0], non_blocking=True)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        for _ in range(3):
            graph_frame()
    torch.cuda.current_stream().wait_stream(s)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        graph_frame()
    return g


def yuv_vs_bgr_rounds(S, rs, fmt, rounds, reps):
    """(a) and (b) of a YUV batch and of a BGR batch at the same S, alternately in rounds: per round and format the device step
    with the frames resident and the host-to-host p50 with the copies inside the graph"""
    arms = {}
    for f in (fmt, 'bgr'):
        sb, raw_h, raw_d, out_h = make_batch(S, rs, f)
        net = fixed_mesh_net(sb)
        arms[f] = (sb.capture(raw_d, net), sb.capture(raw_d, net, upload_from=raw_h, download_to=out_h), sb, raw_h, raw_d, out_h)
    out = {f: {'a_us_device_step_per_round': [], 'b_us_p50_host_to_host_per_round': []} for f in arms}
    for _ in range(rounds):
        for f, (g_res, g_io, *_) in arms.items():
            out[f]['a_us_device_step_per_round'].append(dev_time(g_res.replay, reps))
            out[f]['b_us_p50_host_to_host_per_round'].append(float(np.percentile(host_times(g_io.replay, reps), 50)))
    for f in out:
        a_med, b_med = float(np.median(out[f]['a_us_device_step_per_round'])), float(np.median(out[f]['b_us_p50_host_to_host_per_round']))
        out[f].update(a_us_device_per_frame_median=a_med / S, b_frames_per_s_median=S * 1e6 / b_med)
    del arms
    torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--streams', default='1,4,16,64')
    ap.add_argument('--reps', type=int, default=300, help='timed replays per measurement (the StabNet leg takes a sixth)')
    ap.add_argument('--ab-rounds', type=int, default=6)
    ap.add_argument('--src-format', default='bgr', choices=('bgr', 'nv12', 'i420'))
    ap.add_argument('--out')
    a = ap.parse_args()
    assert torch.cuda.is_available(), 'bench_streams.py measures on the GPU; there is nothing to measure without one'
    torch.backends.cudnn.benchmark = True
    fmt = a.src_format
    raw_bytes = int(np.prod(frame_shape(fmt)))
    res = {'gpu': gpu_info(), 'source': '%dx%d %s uint8' % (H, W, fmt.upper()), 'network_size': '%dx%d' % (h, w), 'refine': 1,
           'bytes_pcie_per_frame': {'h2d_raw_' + fmt: raw_bytes, 'd2h_colour': h * w * 3, 'total': raw_bytes + h * w * 3}, 'per_S': {}}
    rs = np.random.RandomState(0)
    torch.manual_seed(0)
    model = mgw.StabNet(in_ch=13, grid=(4, 4)).to(dev).eval().to(memory_format=torch.channels_last)
    if fmt != 'bgr':
        measure_format(a, res, rs, model, fmt)
        return emit(res, a.out)
    # S = 1 against the single-stream loop, alternately
    sb, raw_h, raw_d, out_h = make_batch(1, rs)
    with torch.no_grad():
        g_batch = sb.capture(raw_d, fixed_mesh_net(sb), upload_from=raw_h, download_to=out_h)
        arms = (('single_stream_loop', single_stream_graph(rs)), ('single_stream_loop_plus_refeed', single_stream_graph(rs, True)),
                ('stream_batch_S1', g_batch))
        rounds = {name: [] for name, _ in arms}
        for _ in range(a.ab_rounds):
            for name, g in arms:
                rounds[name].append(float(np.percentile(host_times(g.replay, a.reps), 50)))
                rounds[name + '_device'] = rounds.get(name + '_device', []) + [dev_time(g.replay, a.reps)]
    res['S1_vs_single_stream_loop_us_p50_host_to_host_per_round'] = rounds
    del sb, raw_h, raw_d, out_h, g_batch, arms
    torch.cuda.empty_cache()
    for S in [int(v) for v in a.streams.split(',')]:
        res['per_S'][str(S)] = legs(S, rs, model, a.reps)
    emit(res, a.out)


def legs(S, rs, model, reps, fmt='bgr'):
    """(a), (b) with the copies alone and the upload rate, (c) for one S"""
    r = {}
    raw_bytes = int(np.prod(frame_shape(fmt)))
    sb, raw_h, raw_d, out_h = make_batch(S, rs, fmt)
    with torch.no_grad():
        net = fixed_mesh_net(sb)
        g_res = sb.capture(raw_d, net)
        t = dev_time(g_res.replay, reps)
        r['a_us_device_step_fixed_mesh_resident'] = t
        r['a_us_device_per_frame'] = t / S
        g_io = sb.capture(raw_d, net, upload_from=raw_h, download_to=out_h)
        r['b_host_to_host_fixed_mesh'] = summary(host_times(g_io.replay, reps), S)

        def copies():
            raw_d.copy_(raw_h, non_blocking=True); out_h.copy_(sb.colour, non_blocking=True)
        r['b_host_to_host_copies_only'] = summary(host_times(copies, reps), S)
        r['h2d_GB_per_s'] = S * raw_bytes / (dev_time(lambda: raw_d.copy_(raw_h, non_blocking=True), reps) * 1e3)
        del g_res, g_io
        g_net = sb.capture(raw_d, stabnet_net(model), upload_from=raw_h, download_to=out_h)
        reps_c = max(reps // 6, 20)
        r['c_host_to_host_stabnet'] = summary(host_times(g_net.replay, reps_c), S)
        r['c_us_device_step_stabnet'] = dev_time(g_net.replay, reps_c)
        del g_net
    del sb, raw_h, raw_d, out_h
    torch.cuda.empty_cache()
    print(json.dumps({S: r}), file=sys.stderr)
    return r


def measure_format(a, res, rs, model, fmt):
    """--src-format nv12 / i420: every leg with YUV input, and the BGR batch alongside at S = 1 and S = 64"""
    res['bytes_pcie_per_frame_bgr'] = {'h2d_raw_bgr': H * W * 3, 'd2h_colour': h * w * 3, 'total': H * W * 3 + h * w * 3}
    res['yuv_vs_bgr_alternating'] = {}
    for S in [int(v) for v in a.streams.split(',')]:
        res['per_S'][str(S)] = legs(S, rs, model, a.reps, fmt)
        if S in (1, 64):
            with torch.no_grad():
                res['yuv_vs_bgr_alternating'][str(S)] = yuv_vs_bgr_rounds(S, rs, fmt, a.ab_rounds, a.reps)
            print(json.dumps({'alternating': {S: res['yuv_vs_bgr_alternating'][str(S)]}}), file=sys.stderr)


def emit(res, out):
    print(json.dumps(res, indent=1))
    if out:
        with open(out, 'w') as f:
            json.dump(res, f, indent=1)


if __name__ == '__main__':
    main()

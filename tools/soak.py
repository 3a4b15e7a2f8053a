"""Randomised agreement soak (GPU): many random shapes / meshes, `auto` (forward: pipeline / TMA tiles; backward: TMA tiles)
against the generic kernels -- forward bit for bit, backward to rounding -- plus the no-dU and fused-loss variants against their unfused forms.
usage: soak.py [cases] [seed].  Not part of the test suite (minutes of GPU time at a few hundred cases)."""
import os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, 'oracle'))
import numpy as np, torch
import synth, dovs_b200 as mgw
from dovs_b200 import ops

cases = int(sys.argv[1]) if len(sys.argv) > 1 else 200
rng = np.random.RandomState(int(sys.argv[2]) if len(sys.argv) > 2 else 0)
dev = lambda a: torch.tensor(a, device='cuda')


def relmax(a, b):
    a, b = a.double(), b.double()
    return float((a - b).abs().max() / b.abs().max().clamp_min(1e-30))


worst = dict(dU=0.0, dH=0.0, dth_nodu=0.0, fused=0.0)
fams = {}
for it in range(cases):
    c = int(rng.choice([1, 3, 4]))
    gh, gw = int(rng.randint(1, 7)), int(rng.randint(1, 7))
    if rng.rand() < 0.7:                 # shapes the TMA families can take: W and the cell width multiples of 4
        w = int(rng.randint(1, 10)) * 4 * gw * int(rng.choice([1, 2, 4, 8]))
        w = min(w, 768)
        w -= w % (4 * gw)
        w = max(w, 4 * gw)
    else:
        w = int(rng.randint(max(gw, 8), 300))
    h = int(rng.randint(max(gh, 6), 320))
    n = int(rng.randint(1, 5))
    sigma = float(rng.choice([0.0, 0.02, 0.05, 0.08, 0.2]))
    seed = int(rng.randint(1 << 30))
    U = dev(synth.noise_image(n, h, w, c, seed))
    th = dev(synth.random_mesh(n, gh, gw, sigma, seed + 1))
    go = dev(synth.randn((n, h, w, c), seed + 2)); gi = dev(synth.randn((n, h, w, 2), seed + 3, 0.1))
    y = dev(synth.noise_image(n, h, w, c, seed + 4))
    tag = (n, h, w, c, gh, gw, sigma, seed)
    mgw.set_impl('generic')
    o_g, b_g, i_g, Hs = ops.mesh_warp_fwd(U, th)
    dU_g, dH_g = ops.warp_bwd(U, Hs, go, gi)
    mgw.set_impl('auto')
    l0 = mgw.launch_count()
    o_a, b_a, i_a, Hs_a = ops.mesh_warp_fwd(U, th)
    dU_a, dH_a = ops.warp_bwd(U, Hs, go, gi)
    _, dH_n = ops.warp_bwd(U, Hs, go, gi, want_dU=False)
    assert torch.equal(Hs, Hs_a), tag
    fin = torch.isfinite(o_g)
    assert torch.equal(torch.isfinite(o_a), fin) and torch.equal(o_g.view(torch.int32)[fin], o_a.view(torch.int32)[fin]), ('out', tag)
    assert torch.equal(b_g, b_a), ('black', tag)
    fi = torch.isfinite(i_g)
    assert torch.equal(i_g.view(torch.int32)[fi], i_a.view(torch.int32)[fi]), ('img', tag)
    if sigma <= 0.08 and torch.isfinite(dU_g).all() and torch.isfinite(dH_g).all():
        e1, e2, e3 = relmax(dU_a, dU_g), relmax(dH_a, dH_g), relmax(dH_n, dH_g)
        worst['dU'] = max(worst['dU'], e1); worst['dH'] = max(worst['dH'], e2); worst['dth_nodu'] = max(worst['dth_nodu'], e3)
        assert e1 < 5e-5 and e2 < 5e-5 and e3 < 5e-5, ('bwd', tag, e1, e2, e3)
        # fused img_loss pair against the unfused one
        out, black, img, Hs2, sums = ops.mesh_warp_img_loss_fwd(U, th, y)
        assert torch.equal(out.view(torch.int32)[fin], o_g.view(torch.int32)[fin]) and torch.equal(black, b_g), ('fused fwd', tag)
        dUf, dthf = ops.mesh_warp_img_loss_bwd(U, th, Hs2, out, y, black, sums, 1.0, float(n), gi)
        d_out = ops.img_loss_bwd(out, y, black, sums, 1.0)
        dUu, dthu = ops.mesh_warp_bwd(U, th, Hs2, d_out, gi)
        if torch.isfinite(dthu).all() and float(dthu.abs().max()) > 0:
            e4 = relmax(dUf, dUu)
            worst['fused'] = max(worst['fused'], e4)
            assert e4 < 5e-5, ('fused bwd', tag, e4)
    if it % 25 == 0:
        print(it, tag, {k: '%.1e' % v for k, v in worst.items()}, flush=True)
print('soak ok: %d cases' % cases, {k: '%.2e' % v for k, v in worst.items()})

"""Thin host wrappers over the C ABI: torch tensors are only carriers of device memory and the current stream.

Every function takes/returns contiguous fp32 CUDA tensors in the reference's layouts (NHWC images,
mesh [N,gh+1,gw+1,2], Hs [N,gh,gw,9]).  No computation happens in Python and nothing falls back to torch.
"""
import torch

from ._lib import check, lib


def _chk(t, name, dtype=torch.float32):
    if not isinstance(t, torch.Tensor):
        raise TypeError('%s must be a torch.Tensor' % name)
    if not t.is_cuda:
        raise RuntimeError('%s must live on a CUDA device: this library has no CPU path' % name)
    if t.dtype != dtype:
        raise TypeError('%s must be %s (got %s)' % (name, dtype, t.dtype))
    return t if t.is_contiguous() else t.contiguous()


def _chk_out(t, name, dtype=torch.float32):
    """a tensor the kernel WRITES in place: a silent .contiguous() copy would swallow the update, so anything but a
    contiguous CUDA tensor of the right dtype is an error"""
    if not isinstance(t, torch.Tensor):
        raise TypeError('%s must be a torch.Tensor' % name)
    if not t.is_cuda:
        raise RuntimeError('%s must live on a CUDA device: this library has no CPU path' % name)
    if t.dtype != dtype:
        raise TypeError('%s must be %s (got %s)' % (name, dtype, t.dtype))
    if not t.is_contiguous():
        raise ValueError('%s is written in place and must be contiguous' % name)
    return t


def _p(t):
    return None if t is None else t.data_ptr()


def _up(upstream):
    """upstream gradient as (host factor, device pointer): a CUDA tensor is read by the kernel itself (no host sync); a pair
    (host factor, CUDA tensor) is their product, formed inside the kernel"""
    if isinstance(upstream, tuple):
        f, t = _up(upstream[1])
        return f * float(upstream[0]), t
    if isinstance(upstream, torch.Tensor) and upstream.is_cuda:
        t = upstream.detach().reshape(-1)[:1].to(torch.float32).contiguous()
        return 1.0, t
    return float(upstream), None


def _st():
    return torch.cuda.current_stream().cuda_stream


def _mesh_dims(U, grid_tensor, what):
    n, h, w, c = U.shape
    if grid_tensor.dim() != 4 or grid_tensor.shape[0] != n:
        raise ValueError('%s has shape %s, batch %d expected' % (what, tuple(grid_tensor.shape), n))
    return n, h, w, c


def vertices_fwd(head, gh, gw, do_crop_rate=0.8, want_pts1=True):
    head = _chk(head, 'head')
    n = head.shape[0]
    if head.numel() != n * 2 * (gh + 1) * (gw + 1):
        raise ValueError('head must be [N, %d]' % (2 * (gh + 1) * (gw + 1)))
    pts2 = torch.empty((n, gh + 1, gw + 1, 2), device=head.device, dtype=torch.float32)
    pts1 = torch.empty((n, gh, gw, 8), device=head.device, dtype=torch.float32) if want_pts1 else None
    with torch.cuda.device(head.device):
        check(lib.mgw_vertices_fwd(_p(head), n, gh, gw, do_crop_rate, _p(pts2), _p(pts1), _st()), 'mgw_vertices_fwd')
    return pts1, pts2


def vertices_bwd(head, d_pts2, d_pts1, gh, gw, do_crop_rate=0.8):
    head = _chk(head, 'head')
    d_pts2 = None if d_pts2 is None else _chk(d_pts2, 'd_pts2')
    d_pts1 = None if d_pts1 is None else _chk(d_pts1, 'd_pts1')
    d_head = torch.empty_like(head)
    with torch.cuda.device(head.device):
        check(lib.mgw_vertices_bwd(_p(head), _p(d_pts2), _p(d_pts1), head.shape[0], gh, gw, do_crop_rate, _p(d_head), _st()),
              'mgw_vertices_bwd')
    return d_head


def solve_h_fwd(theta):
    theta = _chk(theta, 'theta')
    n, gh1, gw1, two = theta.shape
    assert two == 2
    Hs = torch.empty((n, gh1 - 1, gw1 - 1, 9), device=theta.device, dtype=torch.float32)
    with torch.cuda.device(theta.device):
        check(lib.mgw_solve_h_fwd(_p(theta), n, gh1 - 1, gw1 - 1, _p(Hs), _st()), 'mgw_solve_h_fwd')
    return Hs


def solve_h_bwd(theta, Hs, dHs):
    theta, Hs, dHs = _chk(theta, 'theta'), _chk(Hs, 'Hs'), _chk(dHs, 'dHs')
    n, gh, gw, _ = Hs.shape
    dtheta = torch.empty_like(theta)
    with torch.cuda.device(theta.device):
        check(lib.mgw_solve_h_bwd(_p(theta), _p(Hs), _p(dHs), n, gh, gw, _p(dtheta), _st()), 'mgw_solve_h_bwd')
    return dtheta


def warp_fwd(U, Hs, want_out=True, want_black=True, want_img=True, want_cell=False):
    U, Hs = _chk(U, 'U'), _chk(Hs, 'Hs')
    n, h, w, c = _mesh_dims(U, Hs, 'Hs')
    gh, gw = Hs.shape[1:3]
    dev = U.device
    out = torch.empty((n, h, w, c), device=dev, dtype=torch.float32) if want_out else None
    black = torch.empty((n, h, w), device=dev, dtype=torch.float32) if want_black else None
    img = torch.empty((n, h, w, 2), device=dev, dtype=torch.float32) if want_img else None
    cell = torch.empty((n, h, w), device=dev, dtype=torch.int32) if want_cell else None
    with torch.cuda.device(dev):
        check(lib.mgw_warp_fwd(_p(U), _p(Hs), n, h, w, c, gh, gw, _p(out), _p(black), _p(img), _p(cell), _st()), 'mgw_warp_fwd')
    return out, black, img, cell


def _workspace(nbytes, dev):
    return torch.empty((max(nbytes, 256) + 255) // 256 * 64, device=dev, dtype=torch.float32) if nbytes else None


def _acc_target(U, accumulate_into):
    """dU buffer of the accumulate variants: the caller's tensor, added to in place (never zero-filled by the library)."""
    dU = _chk_out(accumulate_into, 'accumulate_into')
    if dU.shape != U.shape or dU.device != U.device:
        raise ValueError('accumulate_into must have the shape and device of U')
    return dU


def warp_bwd(U, Hs, d_out, d_img=None, want_dU=True, accumulate_into=None):
    """accumulate_into: a [N,H,W,C] tensor that receives dU += gradient (mgw_warp_bwd_acc); otherwise dU is a fresh tensor."""
    U, Hs, d_out = _chk(U, 'U'), _chk(Hs, 'Hs'), _chk(d_out, 'd_out')
    d_img = None if d_img is None else _chk(d_img, 'd_img')
    n, h, w, c = _mesh_dims(U, Hs, 'Hs')
    gh, gw = Hs.shape[1:3]
    acc = accumulate_into is not None
    dU = _acc_target(U, accumulate_into) if acc else (torch.empty_like(U) if want_dU else None)
    dHs = torch.empty_like(Hs)
    ws = _workspace(lib.mgw_warp_bwd_workspace_bytes(n, h, w, c, gh, gw), U.device)
    fn = lib.mgw_warp_bwd_acc if acc else lib.mgw_warp_bwd
    with torch.cuda.device(U.device):
        check(fn(_p(U), _p(Hs), _p(d_out), _p(d_img), n, h, w, c, gh, gw, _p(dU), _p(dHs), _p(ws), _st()), 'mgw_warp_bwd')
    return dU, dHs


def mesh_warp_fwd(U, theta, want_out=True, want_black=True, want_img=True):
    U, theta = _chk(U, 'U'), _chk(theta, 'theta')
    n, h, w, c = _mesh_dims(U, theta, 'theta')
    gh, gw = theta.shape[1] - 1, theta.shape[2] - 1
    if theta.shape[3] != 2 or gh < 1 or gw < 1:
        raise ValueError('theta must be [N, gh+1, gw+1, 2] mesh vertices, got %s' % (tuple(theta.shape),))
    dev = U.device
    Hs = torch.empty((n, gh, gw, 9), device=dev, dtype=torch.float32)
    out = torch.empty((n, h, w, c), device=dev, dtype=torch.float32) if want_out else None
    black = torch.empty((n, h, w), device=dev, dtype=torch.float32) if want_black else None
    img = torch.empty((n, h, w, 2), device=dev, dtype=torch.float32) if want_img else None
    with torch.cuda.device(dev):
        check(lib.mgw_mesh_warp_fwd(_p(U), _p(theta), n, h, w, c, gh, gw, _p(Hs), _p(out), _p(black), _p(img), _st()),
              'mgw_mesh_warp_fwd')
    return out, black, img, Hs


def mesh_warp_bwd(U, theta, Hs, d_out, d_img=None, want_dU=True, accumulate_into=None, dtheta_out=None, dU_out=None):
    """dtheta_out / dU_out: optional preallocated tensors to receive dtheta / dU (static buffers for CUDA-graph pipelines);
    accumulate_into: dU += gradient into the caller's tensor instead (never zero-filled by the library)."""
    U, theta, Hs, d_out = _chk(U, 'U'), _chk(theta, 'theta'), _chk(Hs, 'Hs'), _chk(d_out, 'd_out')
    d_img = None if d_img is None else _chk(d_img, 'd_img')
    n, h, w, c = _mesh_dims(U, theta, 'theta')
    gh, gw = Hs.shape[1:3]
    acc = accumulate_into is not None
    if acc:
        dU = _acc_target(U, accumulate_into)
    elif dU_out is not None:
        dU = _acc_target(U, dU_out)
    else:
        dU = torch.empty_like(U) if want_dU else None
    if dtheta_out is not None:
        dtheta = _chk(dtheta_out, 'dtheta_out')
        if dtheta.shape != theta.shape or not dtheta_out.is_contiguous():
            raise ValueError('dtheta_out must be a contiguous tensor of the shape of theta')
    else:
        dtheta = torch.empty_like(theta)
    ws = _workspace(lib.mgw_mesh_warp_bwd_workspace_bytes(n, h, w, c, gh, gw), U.device)
    fn = lib.mgw_mesh_warp_bwd_acc if acc else lib.mgw_mesh_warp_bwd
    with torch.cuda.device(U.device):
        check(fn(_p(U), _p(theta), _p(Hs), _p(d_out), _p(d_img), n, h, w, c, gh, gw, _p(dU), _p(dtheta), _p(ws), _st()),
              'mgw_mesh_warp_bwd')
    return dU, dtheta


def mesh_warp_img_loss_fwd(U, theta, y, want_img=True):
    """transformer(U, theta) with the img_loss partial sums accumulated inside the warp kernel -> (out, black, img, Hs, sums[N,2])."""
    U, theta, y = _chk(U, 'U'), _chk(theta, 'theta'), _chk(y, 'y')
    n, h, w, c = _mesh_dims(U, theta, 'theta')
    if tuple(y.shape) != (n, h, w, c):
        raise ValueError('y must have the shape of U')
    gh, gw = theta.shape[1] - 1, theta.shape[2] - 1
    dev = U.device
    Hs = torch.empty((n, gh, gw, 9), device=dev, dtype=torch.float32)
    out = torch.empty((n, h, w, c), device=dev, dtype=torch.float32)
    black = torch.empty((n, h, w), device=dev, dtype=torch.float32)
    img = torch.empty((n, h, w, 2), device=dev, dtype=torch.float32) if want_img else None
    sums = torch.empty((n, 2), device=dev, dtype=torch.float32)
    with torch.cuda.device(dev):
        check(lib.mgw_mesh_warp_img_loss_fwd(_p(U), _p(theta), _p(y), n, h, w, c, gh, gw, _p(Hs), _p(out), _p(black), _p(img),
                                             _p(sums), _st()), 'mgw_mesh_warp_img_loss_fwd')
    return out, black, img, Hs, sums


def mesh_warp_img_loss_bwd(U, theta, Hs, out, y, black, sums, upstream, batch, d_img=None, want_dU=True, d_out_extra=None):
    U, theta, Hs, out, y, black, sums = (_chk(t, nm) for t, nm in ((U, 'U'), (theta, 'theta'), (Hs, 'Hs'), (out, 'out'), (y, 'y'),
                                                                   (black, 'black'), (sums, 'sums')))
    d_img = None if d_img is None else _chk(d_img, 'd_img')
    d_out_extra = None if d_out_extra is None else _chk(d_out_extra, 'd_out_extra')
    if d_out_extra is not None and d_out_extra.shape != U.shape:
        raise ValueError('d_out_extra must have the shape of U')
    up = _up(upstream)
    n, h, w, c = _mesh_dims(U, theta, 'theta')
    gh, gw = Hs.shape[1:3]
    dU = torch.empty_like(U) if want_dU else None
    dtheta = torch.empty_like(theta)
    ws = _workspace(lib.mgw_mesh_warp_img_loss_bwd_workspace_bytes(n, h, w, c, gh, gw), U.device)
    with torch.cuda.device(U.device):
        check(lib.mgw_mesh_warp_img_loss_bwd(_p(U), _p(theta), _p(Hs), _p(out), _p(y), _p(black), _p(sums), up[0], _p(up[1]),
                                             float(batch), _p(d_img), _p(d_out_extra), n, h, w, c, gh, gw, _p(dU), _p(dtheta), _p(ws), _st()),
              'mgw_mesh_warp_img_loss_bwd')
    return dU, dtheta


def feature_loss_dh(matches, mask, img, Hs, upstream):
    """mgw_feature_loss_dh: d(feature_loss)/dH as one partial per cell [N,gh,gw,8] (what the warp backward would form from the dense
    d_img of feature_loss_bwd)."""
    matches, mask, img, Hs = _chk(matches, 'matches'), _chk(mask, 'mask'), _chk(img, 'img'), _chk(Hs, 'Hs')
    n, h, w, _ = img.shape
    gh, gw = Hs.shape[1:3]
    up = _up(upstream)
    facc = torch.stack([torch.zeros_like(mask[:, 0]), mask.sum(1)], 1).contiguous()
    part = torch.empty((n, gh, gw, 8), device=img.device, dtype=torch.float32)
    with torch.cuda.device(img.device):
        check(lib.mgw_feature_loss_dh(_p(matches), _p(mask), _p(img), _p(Hs), _p(facc), up[0], _p(up[1]), n, matches.shape[1], h, w, gh, gw,
                                      _p(part), _st()), 'mgw_feature_loss_dh')
    return part


def loss_ratio_sum(sums, scale, clamp=False):
    """scale * sum_n sums[n,0] / (sums[n,1] + 1e-8)  (clamp: / max(sums[n,1], 1)) -> 0-dim tensor, one launch"""
    sums = _chk(sums, 'sums')
    if sums.dim() != 2 or sums.shape[1] != 2:
        raise ValueError('sums [N,2] expected')
    out = torch.empty(1, device=sums.device, dtype=torch.float32)
    with torch.cuda.device(sums.device):
        check(lib.mgw_loss_ratio_sum(_p(sums), sums.shape[0], int(bool(clamp)), float(scale), _p(out), _st()), 'mgw_loss_ratio_sum')
    return out[0]


def _coef_array(coef):
    import ctypes
    if len(coef) != 11:
        raise ValueError('coef: 11 floats expected (see include/mgw.h, mgw_train_pass_fwd)')
    return (ctypes.c_float * 11)(*[float(c) for c in coef])


def train_pass_fwd(head, U, y, matches, mask, coef, gh, gw, do_crop_rate=0.8, regu=None, want_warpped=True):
    """mgw_train_pass_fwd: head -> get_4_pts -> transformer + img_loss -> feature_loss -> vertex terms -> total, 7 launches.
    -> dict(pts1, pts2, Hs, out, black, img, acc, warpped, result)."""
    head, U, y, matches, mask = (_chk(t, nm) for t, nm in ((head, 'head'), (U, 'U'), (y, 'y'), (matches, 'matches'), (mask, 'mask')))
    n, h, w, c = U.shape
    if tuple(y.shape) != (n, h, w, c):
        raise ValueError('y must have the shape of U')
    if head.shape[0] != n or head.numel() != n * 2 * (gh + 1) * (gw + 1):
        raise ValueError('head has shape %s for a %dx%d grid, batch %d' % (tuple(head.shape), gh, gw, n))
    if matches.dim() != 3 or matches.shape[0] != n or matches.shape[2] != 4 or tuple(mask.shape) != tuple(matches.shape[:2]):
        raise ValueError('matches [N,M,4] / mask [N,M] expected, got %s / %s' % (tuple(matches.shape), tuple(mask.shape)))
    m = matches.shape[1]
    regu = None if regu is None else _chk(regu.reshape(-1)[:1], 'regu')
    dev = U.device
    f = lambda *shape: torch.empty(shape, device=dev, dtype=torch.float32)      # noqa: E731
    r = dict(pts1=f(n, gh, gw, 8), pts2=f(n, gh + 1, gw + 1, 2), Hs=f(n, gh, gw, 9), out=f(n, h, w, c), black=f(n, h, w), img=f(n, h, w, 2),
             acc=f(4 * n + 4), warpped=f(n, m, 2) if want_warpped else None, result=f(9))
    with torch.cuda.device(dev):
        check(lib.mgw_train_pass_fwd(_p(head), _p(U), _p(y), _p(matches), _p(mask), _p(regu), _coef_array(coef), n, h, w, c, gh, gw, m,
                                     float(do_crop_rate), _p(r['pts1']), _p(r['pts2']), _p(r['Hs']), _p(r['out']), _p(r['black']),
                                     _p(r['img']), _p(r['acc']), _p(r['warpped']), _p(r['result']), _st()),
              'mgw_train_pass_fwd')
    return r


def train_pass_bwd(head, U, y, matches, mask, fwd, coef, gh, gw, do_crop_rate=0.8, g_total=None, d_out_extra=None, want_dU=False):
    """mgw_train_pass_bwd -> (d_head, dU or None); fwd = the dict train_pass_fwd returned; g_total: device scalar or None (= 1)."""
    n, h, w, c = U.shape
    m = matches.shape[1]
    g = None if g_total is None else _chk(g_total.detach().reshape(-1)[:1], 'g_total')
    extra = None if d_out_extra is None else _chk(d_out_extra, 'd_out_extra')
    if extra is not None and tuple(extra.shape) != (n, h, w, c):
        raise ValueError('d_out_extra must have the shape of U')
    d_head = torch.empty_like(head)
    dU = torch.empty_like(U) if want_dU else None
    ws = _workspace(lib.mgw_train_pass_bwd_workspace_bytes(n, h, w, c, gh, gw), U.device)
    with torch.cuda.device(U.device):
        check(lib.mgw_train_pass_bwd(_p(head), _p(fwd['pts1']), _p(fwd['pts2']), _p(U), _p(y), _p(matches), _p(mask), _p(fwd['Hs']),
                                     _p(fwd['out']), _p(fwd['black']), _p(fwd['img']), _p(fwd['acc']), _p(g), _p(extra),
                                     _coef_array(coef), n, h, w, c, gh, gw, m, float(do_crop_rate), _p(dU), _p(d_head), _p(ws), _st()),
              'mgw_train_pass_bwd')
    return d_head, dU


def interp_fwd(im, x, y, out_size):
    im, x, y = _chk(im, 'im'), _chk(x, 'x'), _chk(y, 'y')
    n, ih, iw, c = im.shape
    oh, ow = int(out_size[0]), int(out_size[1])
    if x.numel() != n * oh * ow or y.numel() != n * oh * ow:
        raise ValueError('x and y must hold N*out_h*out_w coordinates')
    out = torch.empty((n, oh, ow, c), device=im.device, dtype=torch.float32)
    with torch.cuda.device(im.device):
        check(lib.mgw_interp_fwd(_p(im), _p(x), _p(y), n, ih, iw, c, oh, ow, _p(out), _st()), 'mgw_interp_fwd')
    return out


def interp_bwd(im, x, y, d_out, out_size, want_dim=True, want_dxy=True):
    im, x, y, d_out = _chk(im, 'im'), _chk(x, 'x'), _chk(y, 'y'), _chk(d_out, 'd_out')
    n, ih, iw, c = im.shape
    oh, ow = int(out_size[0]), int(out_size[1])
    d_im = torch.empty_like(im) if want_dim else None
    dx = torch.empty_like(x) if want_dxy else None
    dy = torch.empty_like(y) if want_dxy else None
    with torch.cuda.device(im.device):
        check(lib.mgw_interp_bwd(_p(im), _p(x), _p(y), _p(d_out), n, ih, iw, c, oh, ow, _p(d_im), _p(dx), _p(dy), _st()),
              'mgw_interp_bwd')
    return d_im, dx, dy


def homography_warp_fwd(U, theta, out_size, want_img=False):
    U, theta = _chk(U, 'U'), _chk(theta, 'theta')
    n, h, w, c = U.shape
    if theta.numel() != n * 9:
        raise ValueError('theta must be [N, 9]')
    oh, ow = int(out_size[0]), int(out_size[1])
    out = torch.empty((n, oh, ow, c), device=U.device, dtype=torch.float32)
    black = torch.empty((n, oh, ow), device=U.device, dtype=torch.float32)
    img = torch.empty((n, oh, ow, 2), device=U.device, dtype=torch.float32) if want_img else None
    with torch.cuda.device(U.device):
        check(lib.mgw_homography_warp_fwd(_p(U), _p(theta), n, h, w, c, oh, ow, _p(out), _p(black), _p(img), _st()),
              'mgw_homography_warp_fwd')
    return out, black, img


def homography_warp_bwd(U, theta, d_out, out_size, want_dU=True):
    U, theta, d_out = _chk(U, 'U'), _chk(theta, 'theta'), _chk(d_out, 'd_out')
    n, h, w, c = U.shape
    oh, ow = int(out_size[0]), int(out_size[1])
    dU = torch.empty_like(U) if want_dU else None
    dtheta = torch.empty((n, 9), device=U.device, dtype=torch.float32)
    with torch.cuda.device(U.device):
        check(lib.mgw_homography_warp_bwd(_p(U), _p(theta), _p(d_out), n, h, w, c, oh, ow, _p(dU), _p(dtheta), _st()),
              'mgw_homography_warp_bwd')
    return dU, dtheta.reshape(theta.shape)


def img_loss_fwd(out, y, black):
    out, y, black = _chk(out, 'out'), _chk(y, 'y'), _chk(black, 'black')
    n, h, w, c = out.shape
    sums = torch.empty((n, 2), device=out.device, dtype=torch.float32)
    with torch.cuda.device(out.device):
        check(lib.mgw_img_loss_fwd(_p(out), _p(y), _p(black), n, h, w, c, _p(sums), _st()), 'mgw_img_loss_fwd')
    return sums


def img_loss_bwd(out, y, black, sums, upstream):
    out, y, black, sums = _chk(out, 'out'), _chk(y, 'y'), _chk(black, 'black'), _chk(sums, 'sums')
    n, h, w, c = out.shape
    d_out = torch.empty_like(out)
    up = _up(upstream)
    with torch.cuda.device(out.device):
        check(lib.mgw_img_loss_bwd(_p(out), _p(y), _p(black), _p(sums), up[0], _p(up[1]), n, h, w, c, _p(d_out), _st()),
              'mgw_img_loss_bwd')
    return d_out


def feature_loss_fwd(matches, mask, img, want_warpped=True):
    matches, mask, img = _chk(matches, 'matches'), _chk(mask, 'mask'), _chk(img, 'img')
    n, m, _ = matches.shape
    _, h, w, _ = img.shape
    warpped = torch.empty((n, m, 2), device=img.device, dtype=torch.float32) if want_warpped else None
    per = torch.empty((n,), device=img.device, dtype=torch.float32)
    with torch.cuda.device(img.device):
        check(lib.mgw_feature_loss_fwd(_p(matches), _p(mask), _p(img), n, m, h, w, _p(warpped), _p(per), _st()),
              'mgw_feature_loss_fwd')
    return per, warpped


def feature_loss_bwd(matches, mask, img, upstream, d_img=None):
    matches, mask, img = _chk(matches, 'matches'), _chk(mask, 'mask'), _chk(img, 'img')
    n, m, _ = matches.shape
    _, h, w, _ = img.shape
    if d_img is None:
        d_img = torch.zeros_like(img)
    up = _up(upstream)
    with torch.cuda.device(img.device):
        check(lib.mgw_feature_loss_bwd(_p(matches), _p(mask), _p(img), up[0], _p(up[1]), n, m, h, w, _p(d_img), _st()),
              'mgw_feature_loss_bwd')
    return d_img


def temp_loss_fwd(out1, black1, out2, black2, flow):
    out1, black1, out2, black2, flow = (_chk(t, nm) for t, nm in ((out1, 'out1'), (black1, 'black1'), (out2, 'out2'),
                                                                     (black2, 'black2'), (flow, 'flow')))
    n, h, w, c = out1.shape
    sums = torch.empty((n, 2), device=out1.device, dtype=torch.float32)
    with torch.cuda.device(out1.device):
        check(lib.mgw_temp_loss_fwd(_p(out1), _p(black1), _p(out2), _p(black2), _p(flow), n, h, w, c, _p(sums), _st()),
              'mgw_temp_loss_fwd')
    return sums


def temp_loss_bwd(out1, black1, out2, black2, flow, sums, upstream):
    out1, black1, out2, black2, flow, sums = (_chk(t, nm) for t, nm in ((out1, 'out1'), (black1, 'black1'), (out2, 'out2'),
                                                                           (black2, 'black2'), (flow, 'flow'), (sums, 'sums')))
    n, h, w, c = out1.shape
    d1, d2 = torch.empty_like(out1), torch.empty_like(out2)
    up = _up(upstream)
    with torch.cuda.device(out1.device):
        check(lib.mgw_temp_loss_bwd(_p(out1), _p(black1), _p(out2), _p(black2), _p(flow), _p(sums), up[0], _p(up[1]), n, h, w, c,
                                    _p(d1), _p(d2), _st()), 'mgw_temp_loss_bwd')
    return d1, d2


def remap_bundle_u8(img, xy, out=None, workspace=None):
    """deploy_bundle.py:136-146 on the device: img [N,H,W,C] uint8, xy [N,H,W,2] fp32 (x_map,y_map interleaved, the `img`
    output of warp_fwd) -> [N,H,W,C] uint8.  One C-ABI call (two launches).  out / workspace: optional preallocated result and
    fp32 scratch of remap_bundle_workspace_floats(N, H, W) (static buffers for CUDA-graph capture)."""
    img, xy = _chk(img, 'img', torch.uint8), _chk(xy, 'xy')
    if img.dim() != 4 or xy.dim() != 4 or xy.shape[3] != 2 or xy.shape[:3] != img.shape[:3]:
        raise ValueError('img must be [N,H,W,C] uint8 and xy [N,H,W,2] (got %s, %s)' % (tuple(img.shape), tuple(xy.shape)))
    n, h, w, c = img.shape
    dst = _out(out, tuple(img.shape), img.device, torch.uint8, 'out')
    ws = (torch.empty(remap_bundle_workspace_floats(n, h, w), device=img.device, dtype=torch.float32) if workspace is None
          else _chk_out(workspace, 'workspace'))
    if ws.numel() < remap_bundle_workspace_floats(n, h, w):
        raise ValueError('workspace needs %d floats' % remap_bundle_workspace_floats(n, h, w))
    with torch.cuda.device(img.device):
        check(lib.mgw_remap_bundle_u8(_p(img), _p(xy), n, h, w, c, _p(dst), _p(ws), _st()), 'mgw_remap_bundle_u8')
    return dst


def remap_bundle_workspace_floats(n, h, w):
    return max(lib.mgw_remap_bundle_u8_workspace_bytes(n, h, w) // 4, 2)


def stream_assemble(frames, masks, head, taps, cur, use_masks=True):
    """deploy_bundle.py:259-274 on the device: frames / masks [depth,H,W] rings (newest entry at slot `head`), cur [H,W]
    -> in_x [1,H,W,nch] = [masks[-i] for i in taps] + [frames[-i] for i in taps] + [cur]."""
    import ctypes
    frames, cur = _chk(frames, 'frames'), _chk(cur, 'cur')
    masks = _chk(masks, 'masks') if use_masks else None
    depth, h, w = frames.shape
    nch = (2 if use_masks else 1) * len(taps) + 1
    in_x = torch.empty((1, h, w, nch), device=frames.device, dtype=torch.float32)
    arr = (ctypes.c_int * len(taps))(*[int(t) for t in taps])
    with torch.cuda.device(frames.device):
        check(lib.mgw_stream_assemble(_p(frames), _p(masks), depth, int(head), arr, len(taps), 1 if use_masks else 0, _p(cur), h, w,
                                      _p(in_x), _st()), 'mgw_stream_assemble')
    return in_x


def stream_push(frames, masks, slot, img, black, refeed_into=None):
    """deploy_bundle.py:292-295,319-328: frame = img + black*(-1) -> frames[slot], black -> masks[slot]; refeed_into: an
    assembled in_x [1,H,W,nch] whose LAST channel receives the frame (the refine loop).  frames/masks None: re-feed only."""
    img, black = _chk(img, 'img'), _chk(black, 'black')
    frames = None if frames is None else _chk_out(frames, 'frames')
    masks = None if masks is None else _chk_out(masks, 'masks')
    ref = frames if frames is not None else refeed_into
    depth, h, w = (frames.shape if frames is not None else (1, refeed_into.shape[1], refeed_into.shape[2]))
    fo, stride = None, 1
    if refeed_into is not None:
        refeed_into = _chk_out(refeed_into, 'refeed_into')
        stride = refeed_into.shape[-1]
        fo = refeed_into.data_ptr() + 4 * (stride - 1)
    with torch.cuda.device(ref.device):
        check(lib.mgw_stream_push(_p(frames), _p(masks), depth, int(slot), _p(img), _p(black), h, w, fo, stride, _st()), 'mgw_stream_push')


def u8_to_train(frame, out=None):
    """config.py:19 on the device: uint8 tensor (any shape) -> float32 v * (1/255) - 0.5, exact."""
    frame = _chk(frame, 'frame', torch.uint8)
    out = torch.empty(frame.shape, device=frame.device, dtype=torch.float32) if out is None else _chk_out(out, 'out')
    if out.numel() != frame.numel():
        raise ValueError('out has %d elements, frame %d' % (out.numel(), frame.numel()))
    with torch.cuda.device(frame.device):
        check(lib.mgw_u8_to_train_f32(_p(frame), _p(out), frame.numel(), _st()), 'mgw_u8_to_train_f32')
    return out


def train_to_u8(x, out=None):
    """cvt_train2img (deploy_bundle.py:75) on the device: float32 -> uint8 ((x + 0.5) * 255, truncated)."""
    x = _chk(x, 'x')
    out = torch.empty(x.shape, device=x.device, dtype=torch.uint8) if out is None else _chk_out(out, 'out', torch.uint8)
    if out.numel() != x.numel():
        raise ValueError('out has %d elements, x %d' % (out.numel(), x.numel()))
    with torch.cuda.device(x.device):
        check(lib.mgw_train_f32_to_u8(_p(x), _p(out), x.numel(), _st()), 'mgw_train_f32_to_u8')
    return out


def fill_zero(t, keep_in_l2=False):
    """zero-fill of a contiguous CUDA tensor by the library's own kernel; keep_in_l2: evict_last policy (dU before *_bwd_acc)."""
    if not (isinstance(t, torch.Tensor) and t.is_cuda and t.is_contiguous()):
        raise ValueError('fill_zero needs a contiguous CUDA tensor')
    nbytes = t.numel() * t.element_size()
    if nbytes % 16 or t.data_ptr() % 16:
        raise ValueError('fill_zero needs a 16-byte aligned tensor whose size is a multiple of 16 bytes')
    with torch.cuda.device(t.device):
        check(lib.mgw_fill_zero(_p(t), nbytes, 1 if keep_in_l2 else 0, _st()), 'mgw_fill_zero')
    return t


def black_accumulate(all_black, black):
    """deploy_bundle.py:291: all_black = all_black + np.round(black).astype(np.int64), in place on the device (int32 counts)."""
    black, all_black = _chk(black, 'black'), _chk_out(all_black, 'all_black', torch.int32)
    if black.numel() != all_black.numel():
        raise ValueError('black has %d pixels, all_black %d' % (black.numel(), all_black.numel()))
    with torch.cuda.device(black.device):
        check(lib.mgw_black_accumulate(_p(black), _p(all_black), black.numel(), _st()), 'mgw_black_accumulate')
    return all_black


def crop_rect(all_black, step=10):
    """deploy_bundle.py:344-365: [top, left, bottom, right] (inclusive, int32 device tensor) of the largest never-black
    rectangle anchored on the `step` lattice of the top-left quadrant; -1s when there is none."""
    all_black = _chk(all_black, 'all_black', torch.int32)
    h, w = all_black.shape
    ws = torch.empty(lib.mgw_crop_rect_workspace_bytes(h, w), device=all_black.device, dtype=torch.uint8)
    rect = torch.empty(4, device=all_black.device, dtype=torch.int32)
    with torch.cuda.device(all_black.device):
        check(lib.mgw_crop_rect(_p(all_black), h, w, int(step), _p(ws), _p(rect), _st()), 'mgw_crop_rect')
    return rect


def vertex_losses_fwd(theta, pts1, pts2, gh, gw, do_crop_rate=0.8, want_black_err=False):
    """sums[4] of mgw_vertex_losses_fwd (id, black_pos, distortion, consistency); inputs may be None (term skipped)."""
    theta = None if theta is None else _chk(theta, 'theta')
    pts1 = None if pts1 is None else _chk(pts1, 'pts1')
    pts2 = None if pts2 is None else _chk(pts2, 'pts2')
    ref = next(t for t in (theta, pts1, pts2) if t is not None)
    n = ref.shape[0]
    for t, cnt, name in ((theta, 2 * (gh + 1) * (gw + 1), 'theta'), (pts1, gh * gw * 8, 'pts1'), (pts2, 2 * (gh + 1) * (gw + 1), 'pts2')):
        if t is not None and (t.shape[0] != n or t.numel() != n * cnt):
            raise ValueError('%s has shape %s for a %dx%d grid, batch %d' % (name, tuple(t.shape), gh, gw, n))
    sums = torch.empty(4, device=ref.device, dtype=torch.float32)
    err = torch.empty((n, gh, gw, 8), device=ref.device, dtype=torch.float32) if want_black_err else None
    with torch.cuda.device(ref.device):
        check(lib.mgw_vertex_losses_fwd(_p(theta), _p(pts1), _p(pts2), n, gh, gw, do_crop_rate, _p(sums), _p(err), _st()),
              'mgw_vertex_losses_fwd')
    return (sums, err) if want_black_err else sums


def vertex_losses_bwd(theta, pts1, pts2, gh, gw, f, do_crop_rate=0.8, need=(True, True, True)):
    """f [4] (device) = d(total)/d(sums[k]) -> (d_theta, d_pts1, d_pts2), None where not needed."""
    f = _chk(f, 'f')
    ref = next(t for t in (theta, pts1, pts2) if t is not None)
    outs = [torch.empty_like(t) if (t is not None and nd) else None for t, nd in zip((theta, pts1, pts2), need)]
    with torch.cuda.device(ref.device):
        check(lib.mgw_vertex_losses_bwd(_p(theta), _p(pts1), _p(pts2), ref.shape[0], gh, gw, do_crop_rate, _p(f),
                                        _p(outs[0]), _p(outs[1]), _p(outs[2]), _st()), 'mgw_vertex_losses_bwd')
    return tuple(outs)


def warp_rev_bundle_u8(img, Hs_cvt, gh, gw):
    """deploy_bundle.py:148-173 on the device: img [N,H,W,C] uint8, Hs_cvt [N,gh,gw,9] float64 (pixel-space homographies of
    cvt_theta_mat_bundle) -> [N,H,W,C] uint8, every cell cut from the frame warped by its own homography."""
    img, Hs_cvt = _chk(img, 'img', torch.uint8), _chk(Hs_cvt, 'Hs_cvt', torch.float64)
    n, h, w, c = img.shape
    if Hs_cvt.numel() != n * gh * gw * 9:
        raise ValueError('Hs_cvt has %d elements for batch %d and a %dx%d grid' % (Hs_cvt.numel(), n, gh, gw))
    dst = torch.empty_like(img)
    with torch.cuda.device(img.device):
        check(lib.mgw_warp_rev_bundle_u8(_p(img), _p(Hs_cvt), n, h, w, c, gh, gw, _p(dst), _st()), 'mgw_warp_rev_bundle_u8')
    return dst


def cvt_img2train_u8(bgr, tables, out_h, out_w):
    """config.py:6-21 on the device: bgr [H,W,3] uint8, tables = (kx, x0, xn, ky, y0, yn) int32 device tensors (Pillow's
    coefficient windows, see deploy.cvt_img2train) -> [out_h,out_w] fp32 in [-0.5, 0.5]."""
    bgr = _chk(bgr, 'bgr', torch.uint8)
    kx, x0, xn, ky, y0, yn = (_chk(t, 'table', torch.int32) for t in tables)
    h, w, c = bgr.shape
    if c != 3 or kx.shape[0] != out_w or ky.shape[0] != out_h:
        raise ValueError('bgr must be [H,W,3] and the tables must cover the %dx%d output' % (out_h, out_w))
    tmp = torch.empty((h, out_w), device=bgr.device, dtype=torch.uint8)
    out = torch.empty((out_h, out_w), device=bgr.device, dtype=torch.float32)
    with torch.cuda.device(bgr.device):
        check(lib.mgw_cvt_img2train_u8(_p(bgr), h, w, _p(kx), _p(x0), _p(xn), kx.shape[1], _p(ky), _p(y0), _p(yn), ky.shape[1],
                                       out_h, out_w, _p(tmp), _p(out), _st()), 'mgw_cvt_img2train_u8')
    return out


def resize_linear_u8(img, xtab, ytab, out_h, out_w):
    """cv2.resize(img, (out_w, out_h)) for a uint8 [H,W,C] frame on the device; xtab / ytab: int32 [out,4] tables
    {i0, i1, a0, a1} (see deploy.cv2_resize), None for the exact 2x2 decimation."""
    img = _chk(img, 'img', torch.uint8)
    h, w, c = img.shape
    xtab = None if xtab is None else _chk(xtab, 'xtab', torch.int32)
    ytab = None if ytab is None else _chk(ytab, 'ytab', torch.int32)
    dst = torch.empty((out_h, out_w, c), device=img.device, dtype=torch.uint8)
    with torch.cuda.device(img.device):
        check(lib.mgw_resize_linear_u8(_p(img), h, w, c, _p(xtab), _p(ytab), out_h, out_w, _p(dst), _st()), 'mgw_resize_linear_u8')
    return dst


def stream_assemble_dev(frames, masks, head_dev, taps, cur, use_masks=True, out=None):
    """stream_assemble with the ring head read on the device (head_dev: int32 [1]); `out`: optional preallocated in_x
    (static buffers for CUDA-graph capture of the frame loop)."""
    import ctypes
    frames, cur, head_dev = _chk(frames, 'frames'), _chk(cur, 'cur'), _chk(head_dev, 'head_dev', torch.int32)
    masks = _chk(masks, 'masks') if use_masks else None
    depth, h, w = frames.shape
    nch = (2 if use_masks else 1) * len(taps) + 1
    in_x = out if out is not None else torch.empty((1, h, w, nch), device=frames.device, dtype=torch.float32)
    if tuple(in_x.shape) != (1, h, w, nch) or not in_x.is_contiguous():
        raise ValueError('out must be a contiguous [1,%d,%d,%d] tensor' % (h, w, nch))
    arr = (ctypes.c_int * len(taps))(*[int(t) for t in taps])
    with torch.cuda.device(frames.device):
        check(lib.mgw_stream_assemble_dev(_p(frames), _p(masks), depth, _p(head_dev), arr, len(taps), 1 if use_masks else 0, _p(cur),
                                          h, w, _p(in_x), _st()), 'mgw_stream_assemble_dev')
    return in_x


def stream_push_dev(frames, masks, head_dev, img, black):
    """stream_push into the slot after the device-resident head, then head = (head + 1) % depth on the device."""
    frames, img, black, head_dev = _chk_out(frames, 'frames'), _chk(img, 'img'), _chk(black, 'black'), _chk_out(head_dev, 'head_dev', torch.int32)
    masks = None if masks is None else _chk_out(masks, 'masks')
    depth, h, w = frames.shape
    with torch.cuda.device(frames.device):
        check(lib.mgw_stream_push_dev(_p(frames), _p(masks), depth, _p(head_dev), _p(img), _p(black), h, w, _st()), 'mgw_stream_push_dev')


# ---- several videos of one size at once (deploy.StreamBatch): one launch per stage for all S streams, each stream's result
# bit-identical to the single-stream call on its slice.  `out` / `tmp`: optional preallocated buffers (CUDA-graph capture).
def _out(out, shape, dev, dtype, name):
    if out is None:
        return torch.empty(shape, device=dev, dtype=dtype)
    out = _chk_out(out, name, dtype)
    if tuple(out.shape) != tuple(shape):
        raise ValueError('%s must be %s (got %s)' % (name, tuple(shape), tuple(out.shape)))
    return out


def cvt_img2train_u8_batch(bgr, tables, out_h, out_w, out=None, tmp=None):
    """cvt_img2train_u8 for bgr [S,H,W,3] uint8 (one size, shared tables) -> [S,out_h,out_w] fp32."""
    bgr = _chk(bgr, 'bgr', torch.uint8)
    kx, x0, xn, ky, y0, yn = (_chk(t, 'table', torch.int32) for t in tables)
    if bgr.dim() != 4 or bgr.shape[3] != 3 or kx.shape[0] != out_w or ky.shape[0] != out_h:
        raise ValueError('bgr must be [S,H,W,3] and the tables must cover the %dx%d output (got %s)' % (out_h, out_w, tuple(bgr.shape)))
    s, h, w, _ = bgr.shape
    tmp = _out(tmp, (s, h, out_w), bgr.device, torch.uint8, 'tmp')
    out = _out(out, (s, out_h, out_w), bgr.device, torch.float32, 'out')
    with torch.cuda.device(bgr.device):
        check(lib.mgw_cvt_img2train_u8_batch(_p(bgr), s, h, w, _p(kx), _p(x0), _p(xn), kx.shape[1], _p(ky), _p(y0), _p(yn), ky.shape[1],
                                             out_h, out_w, _p(tmp), _p(out), _st()), 'mgw_cvt_img2train_u8_batch')
    return out


def resize_linear_u8_batch(img, xtab, ytab, out_h, out_w, out=None):
    """resize_linear_u8 for img [S,H,W,C] uint8 (one size, shared tables) -> [S,out_h,out_w,C]."""
    img = _chk(img, 'img', torch.uint8)
    if img.dim() != 4:
        raise ValueError('img must be [S,H,W,C] (got %s)' % (tuple(img.shape),))
    s, h, w, c = img.shape
    xtab = None if xtab is None else _chk(xtab, 'xtab', torch.int32)
    ytab = None if ytab is None else _chk(ytab, 'ytab', torch.int32)
    dst = _out(out, (s, out_h, out_w, c), img.device, torch.uint8, 'out')
    with torch.cuda.device(img.device):
        check(lib.mgw_resize_linear_u8_batch(_p(img), s, h, w, c, _p(xtab), _p(ytab), out_h, out_w, _p(dst), _st()),
              'mgw_resize_linear_u8_batch')
    return dst


YUV420_FORMATS = {'nv12': 1, 'i420': 2}          # MGW_YUV420_NV12, MGW_YUV420_I420


def _yuv420_dims(yuv, fmt):
    """yuv [S,3H/2,W] uint8 in OpenCV's 4:2:0 layout -> (format constant, S, H, W)"""
    if fmt not in YUV420_FORMATS:
        raise ValueError('YUV 4:2:0 format must be one of %s (got %r)' % (sorted(YUV420_FORMATS), fmt))
    # 3H/2 rows: a row count that is a multiple of 3 is exactly an even H
    if yuv.dim() != 3 or yuv.shape[1] % 3 != 0 or yuv.shape[2] % 2 != 0:
        raise ValueError('yuv must be [S,3H/2,W] with H and W even (got %s)' % (tuple(yuv.shape),))
    s, rows, w = yuv.shape
    return YUV420_FORMATS[fmt], s, rows // 3 * 2, w


def cvt_img2train_yuv420_batch(yuv, fmt, tables, out_h, out_w, out=None, tmp=None):
    """cvt_img2train_u8_batch of the BGR frames cv2.cvtColor(COLOR_YUV2BGR_NV12 / _I420) makes of yuv [S,3H/2,W] uint8
    (fmt 'nv12' / 'i420'), converted inside the kernel -> [S,out_h,out_w] fp32."""
    yuv = _chk(yuv, 'yuv', torch.uint8)
    code, s, h, w = _yuv420_dims(yuv, fmt)
    kx, x0, xn, ky, y0, yn = (_chk(t, 'table', torch.int32) for t in tables)
    if kx.shape[0] != out_w or ky.shape[0] != out_h:
        raise ValueError('the tables must cover the %dx%d output' % (out_h, out_w))
    tmp = _out(tmp, (s, h, out_w), yuv.device, torch.uint8, 'tmp')
    out = _out(out, (s, out_h, out_w), yuv.device, torch.float32, 'out')
    with torch.cuda.device(yuv.device):
        check(lib.mgw_cvt_img2train_yuv420_batch(_p(yuv), code, s, h, w, _p(kx), _p(x0), _p(xn), kx.shape[1], _p(ky), _p(y0), _p(yn),
                                                 ky.shape[1], out_h, out_w, _p(tmp), _p(out), _st()), 'mgw_cvt_img2train_yuv420_batch')
    return out


def resize_linear_yuv420_batch(yuv, fmt, xtab, ytab, out_h, out_w, out=None):
    """resize_linear_u8_batch of the BGR frames cv2.cvtColor makes of yuv [S,3H/2,W] uint8 (fmt 'nv12' / 'i420'), converted
    inside the kernel -> [S,out_h,out_w,3] BGR."""
    yuv = _chk(yuv, 'yuv', torch.uint8)
    code, s, h, w = _yuv420_dims(yuv, fmt)
    xtab = None if xtab is None else _chk(xtab, 'xtab', torch.int32)
    ytab = None if ytab is None else _chk(ytab, 'ytab', torch.int32)
    dst = _out(out, (s, out_h, out_w, 3), yuv.device, torch.uint8, 'out')
    with torch.cuda.device(yuv.device):
        check(lib.mgw_resize_linear_yuv420_batch(_p(yuv), code, s, h, w, _p(xtab), _p(ytab), out_h, out_w, _p(dst), _st()),
              'mgw_resize_linear_yuv420_batch')
    return dst


def _streams_dims(frames, heads_dev, what):
    if frames.dim() != 4:
        raise ValueError('%s must be [S,depth,H,W] rings (got %s)' % (what, tuple(frames.shape)))
    s, depth, h, w = frames.shape
    if tuple(heads_dev.shape) != (s,):
        raise ValueError('heads_dev must be [%d] (got %s)' % (s, tuple(heads_dev.shape)))
    return s, depth, h, w


def streams_assemble(frames, masks, heads_dev, taps, cur, use_masks=True, out=None):
    """stream_assemble_dev for S streams: frames / masks [S,depth,H,W], heads_dev int32 [S], cur [S,H,W] -> in_x [S,H,W,nch]."""
    import ctypes
    frames, cur, heads_dev = _chk(frames, 'frames'), _chk(cur, 'cur'), _chk(heads_dev, 'heads_dev', torch.int32)
    s, depth, h, w = _streams_dims(frames, heads_dev, 'frames')
    masks = _chk(masks, 'masks') if use_masks else None
    if (masks is not None and masks.shape != frames.shape) or tuple(cur.shape) != (s, h, w):
        raise ValueError('masks must have the shape of frames and cur must be [%d,%d,%d]' % (s, h, w))
    nch = (2 if use_masks else 1) * len(taps) + 1
    in_x = _out(out, (s, h, w, nch), frames.device, torch.float32, 'out')
    arr = (ctypes.c_int * len(taps))(*[int(t) for t in taps])
    with torch.cuda.device(frames.device):
        check(lib.mgw_streams_assemble(_p(frames), _p(masks), s, depth, _p(heads_dev), arr, len(taps), 1 if use_masks else 0, _p(cur),
                                       h, w, _p(in_x), _st()), 'mgw_streams_assemble')
    return in_x


def streams_push(frames, masks, heads_dev, img, black):
    """stream_push_dev for S streams: frame = img + black*(-1) and black [S,H,W] into the slot after each stream's head, then
    every head advances."""
    frames, heads_dev = _chk_out(frames, 'frames'), _chk_out(heads_dev, 'heads_dev', torch.int32)
    img, black = _chk(img, 'img'), _chk(black, 'black')
    masks = None if masks is None else _chk_out(masks, 'masks')
    s, depth, h, w = _streams_dims(frames, heads_dev, 'frames')
    if (masks is not None and masks.shape != frames.shape) or img.numel() != s * h * w or black.numel() != s * h * w:
        raise ValueError('masks must have the shape of frames and img / black %d x %d x %d pixels' % (s, h, w))
    with torch.cuda.device(frames.device):
        check(lib.mgw_streams_push(_p(frames), _p(masks), s, depth, _p(heads_dev), _p(img), _p(black), h, w, _st()), 'mgw_streams_push')


# ---- several videos of different source sizes at once (deploy.MixedStreamBatch): per-slot source geometry
SRC_FORMATS = {'bgr': 0, 'nv12': 1, 'i420': 2}    # MGW_BGR24, MGW_YUV420_NV12, MGW_YUV420_I420


def _mixed_dims(pool, fmt, sizes):
    """pool [S,max_h,max_w,3] (BGR) or [S,3max_h/2,max_w] (YUV 4:2:0) uint8: slot s's frame lies at the start of pool[s] in its
    own size sizes[s] (int32 device [S,2]) -> (format constant, S, max_h, max_w)"""
    if fmt not in SRC_FORMATS:
        raise ValueError('source format must be one of %s (got %r)' % (sorted(SRC_FORMATS), fmt))
    if fmt == 'bgr':
        if pool.dim() != 4 or pool.shape[3] != 3:
            raise ValueError('a BGR pool must be [S,max_h,max_w,3] (got %s)' % (tuple(pool.shape),))
        s, mh, mw, _ = pool.shape
    else:
        code, s, mh, mw = _yuv420_dims(pool, fmt)
    if tuple(sizes.shape) != (s, 2):
        raise ValueError('sizes must be [%d,2] (got %s)' % (s, tuple(sizes.shape)))
    return SRC_FORMATS[fmt], s, mh, mw


def cvt_img2train_mixed(pool, fmt, sizes, tables, out_h, out_w, out=None, tmp=None):
    """cvt_img2train of every slot of a pool at the slot's own size -> [S,out_h,out_w] fp32; tables = (kx [S,out_w,ksx], x0, xn
    [S,out_w], ky [S,out_h,ksy], y0, yn [S,out_h]) int32 (deploy.mixed_slot_tables per slot).  Idle slots (size 0, above the
    capacity, odd for YUV) leave their rows of out / tmp [S,max_h,out_w] untouched."""
    pool, sizes = _chk(pool, 'pool', torch.uint8), _chk(sizes, 'sizes', torch.int32)
    code, s, mh, mw = _mixed_dims(pool, fmt, sizes)
    kx, x0, xn, ky, y0, yn = (_chk(t, 'table', torch.int32) for t in tables)
    if (kx.dim() != 3 or tuple(kx.shape[:2]) != (s, out_w) or ky.dim() != 3 or tuple(ky.shape[:2]) != (s, out_h) or
            any(tuple(t.shape) != (s, out_w) for t in (x0, xn)) or any(tuple(t.shape) != (s, out_h) for t in (y0, yn))):
        raise ValueError('the tables must be [%d,%d,ksx], [%d,%d] x2, [%d,%d,ksy], [%d,%d] x2' % (s, out_w, s, out_w, s, out_h, s, out_h))
    tmp = _out(tmp, (s, mh, out_w), pool.device, torch.uint8, 'tmp')
    out = _out(out, (s, out_h, out_w), pool.device, torch.float32, 'out')
    with torch.cuda.device(pool.device):
        check(lib.mgw_cvt_img2train_mixed(_p(pool), code, s, mh, mw, _p(sizes), _p(kx), _p(x0), _p(xn), kx.shape[2], _p(ky), _p(y0),
                                          _p(yn), ky.shape[2], out_h, out_w, _p(tmp), _p(out), _st()), 'mgw_cvt_img2train_mixed')
    return out


def resize_linear_mixed(pool, fmt, sizes, xtab, ytab, out_h, out_w, out=None):
    """cv2.resize of every slot of a pool at the slot's own size -> [S,out_h,out_w,3] BGR; xtab [S,out_w,4], ytab [S,out_h,4]
    int32 (also for slots that take the 2x2 shortcut).  Idle slots leave their rows of out untouched."""
    pool, sizes = _chk(pool, 'pool', torch.uint8), _chk(sizes, 'sizes', torch.int32)
    code, s, mh, mw = _mixed_dims(pool, fmt, sizes)
    xtab, ytab = _chk(xtab, 'xtab', torch.int32), _chk(ytab, 'ytab', torch.int32)
    if tuple(xtab.shape) != (s, out_w, 4) or tuple(ytab.shape) != (s, out_h, 4):
        raise ValueError('xtab / ytab must be [%d,%d,4] / [%d,%d,4]' % (s, out_w, s, out_h))
    dst = _out(out, (s, out_h, out_w, 3), pool.device, torch.uint8, 'out')
    with torch.cuda.device(pool.device):
        check(lib.mgw_resize_linear_mixed(_p(pool), code, s, mh, mw, _p(sizes), _p(xtab), _p(ytab), out_h, out_w, _p(dst), _st()),
              'mgw_resize_linear_mixed')
    return dst


def dst_frame_bytes(out_format, H, W):
    """bytes of one result frame: 3*H*W for 'bgr', 3H/2*W for YUV 4:2:0"""
    return H * W * 3 if out_format == 'bgr' else H * W * 3 // 2


def remap_bundle_frame_mixed(pool, fmt, sizes, xy, out_format='bgr', out=None, workspace=None):
    """warpRevBundle2 of every slot of a pool at the slot's own size (remap_bundle_frame of the slot's frame alone, with xy[s]):
    pool as for cvt_img2train_mixed, xy [S,h,w,2] fp32 -> the output pool [S, dst_frame_bytes(capacity)] uint8, slot s's result
    at the start of its row, BGR [H_s,W_s,3] or YUV 4:2:0 [3H_s/2,W_s] for out_format 'nv12' / 'i420' (the capacity must then be
    even).  Bytes past a slot's result, and the rows of idle slots (size 0, above the capacity, odd with either format YUV), are
    left as they were.  out / workspace: optional preallocated output pool and fp32 scratch of remap_bundle_workspace_floats(S, h, w)."""
    pool, sizes, xy = _chk(pool, 'pool', torch.uint8), _chk(sizes, 'sizes', torch.int32), _chk(xy, 'xy')
    code, s, mh, mw = _mixed_dims(pool, fmt, sizes)
    if out_format not in SRC_FORMATS:
        raise ValueError('out_format must be one of %s (got %r)' % (sorted(SRC_FORMATS), out_format))
    if out_format != 'bgr' and (mh % 2 or mw % 2):
        raise ValueError('a %s result needs an even capacity (got %dx%d)' % (out_format, mh, mw))
    if xy.dim() != 4 or xy.shape[0] != s or xy.shape[3] != 2:
        raise ValueError('xy must be [%d,h,w,2] (got %s)' % (s, tuple(xy.shape)))
    h, w = int(xy.shape[1]), int(xy.shape[2])
    dst = _out(out, (s, dst_frame_bytes(out_format, mh, mw)), pool.device, torch.uint8, 'out')
    ws = (torch.empty(remap_bundle_workspace_floats(s, h, w), device=pool.device, dtype=torch.float32) if workspace is None
          else _chk_out(workspace, 'workspace'))
    if ws.numel() < remap_bundle_workspace_floats(s, h, w):
        raise ValueError('workspace needs %d floats' % remap_bundle_workspace_floats(s, h, w))
    with torch.cuda.device(pool.device):
        check(lib.mgw_remap_bundle_frame_mixed(_p(pool), code, s, mh, mw, _p(sizes), _p(xy), h, w, SRC_FORMATS[out_format], _p(dst),
                                               _p(ws), _st()), 'mgw_remap_bundle_frame_mixed')
    return dst


def copy_slots_mixed(src, dst, fmt, sizes):
    """Each slot's own frame bytes of a pool, and nothing else, from src to dst: slot s's first frame_bytes(sizes[s]) bytes of
    src[s] go to dst[s] (3*H_s*W_s for 'bgr', 3H_s/2*W_s for 'nv12' / 'i420'); bytes past them and the rows of idle slots (size 0,
    above the capacity, odd for YUV) are neither read nor written.  src and dst have one shape, that of the pools of
    cvt_img2train_mixed ([S,max_h,max_w,3] for 'bgr', [S,3max_h/2,max_w] for YUV 4:2:0, which gives the capacity), and each is
    a contiguous CUDA tensor or a pinned CPU tensor: the kernel reads or writes pinned host memory across PCIe itself, so this
    one call is an upload, a download or a device copy, and inside a captured graph it follows the sizes of the replay.
    One C-ABI call (mgw_copy_slots_mixed)."""
    if fmt not in SRC_FORMATS:
        raise ValueError('format must be one of %s (got %r)' % (sorted(SRC_FORMATS), fmt))
    for name, t in (('src', src), ('dst', dst)):
        if not isinstance(t, torch.Tensor) or t.dtype != torch.uint8:
            raise ValueError('%s must be a uint8 tensor' % name)
    if tuple(src.shape) != tuple(dst.shape):
        raise ValueError('src and dst must have one shape (got %s and %s)' % (tuple(src.shape), tuple(dst.shape)))
    code, s, mh, mw = _mixed_dims(src, fmt, sizes)
    for name, t in (('src', src), ('dst', dst)):
        if not t.is_cuda and not t.is_pinned():
            raise ValueError('%s is pageable host memory: the copy reaches host memory through its device address, which only pinned '
                             'memory has' % name)
        if not t.is_contiguous():
            raise ValueError('%s must be contiguous' % name)
    sizes = _chk(sizes, 'sizes', torch.int32)
    with torch.cuda.device(sizes.device):
        check(lib.mgw_copy_slots_mixed(_p(src), _p(dst), code, s, mh, mw, _p(sizes), _st()), 'mgw_copy_slots_mixed')
    return dst


# ---- warpRevBundle2 at the frame's own size
def remap_bundle_frame(src, src_format, xy, out=None, workspace=None, out_format='bgr'):
    """warpRevBundle2 of frames at any size: src [S,H,W,3] uint8 ('bgr') or [S,3H/2,W] ('nv12' / 'i420'), xy [S,h,w,2] fp32 (the
    operator's x_map,y_map at the network size) -> [S,H,W,3] BGR: the /4 maps resized to (W, H) and scaled by (W, H), then
    cv2.remap of the frame.  At (H, W) == (h, w) with 'bgr' this is remap_bundle_u8.  One C-ABI call (two launches).
    out_format 'nv12' / 'i420' (H and W even): the result is [S,3H/2,W] YUV 4:2:0 instead, cv2.cvtColor(COLOR_BGR2YUV_I420) of
    the BGR result (U and V interleaved for NV12), converted inside the warp (mgw_remap_bundle_frame_yuv420).
    out / workspace: optional preallocated result and fp32 scratch of remap_bundle_workspace_floats(S, h, w) (CUDA-graph capture)."""
    src, xy = _chk(src, 'src', torch.uint8), _chk(xy, 'xy')
    if src_format not in SRC_FORMATS:
        raise ValueError('source format must be one of %s (got %r)' % (sorted(SRC_FORMATS), src_format))
    if out_format not in SRC_FORMATS:
        raise ValueError('out_format must be one of %s (got %r)' % (sorted(SRC_FORMATS), out_format))
    if src_format == 'bgr':
        if src.dim() != 4 or src.shape[3] != 3:
            raise ValueError('a BGR batch must be [S,H,W,3] (got %s)' % (tuple(src.shape),))
        s, H, W = int(src.shape[0]), int(src.shape[1]), int(src.shape[2])
    else:
        _, s, H, W = _yuv420_dims(src, src_format)
    if xy.dim() != 4 or xy.shape[0] != s or xy.shape[3] != 2:
        raise ValueError('xy must be [%d,h,w,2] (got %s)' % (s, tuple(xy.shape)))
    h, w = int(xy.shape[1]), int(xy.shape[2])
    if out_format != 'bgr' and (H % 2 or W % 2):
        raise ValueError('a %s result needs an even size (got %dx%d)' % (out_format, H, W))
    dst = _out(out, (s, H, W, 3) if out_format == 'bgr' else (s, H * 3 // 2, W), src.device, torch.uint8, 'out')
    ws = (torch.empty(remap_bundle_workspace_floats(s, h, w), device=src.device, dtype=torch.float32) if workspace is None
          else _chk_out(workspace, 'workspace'))
    if ws.numel() < remap_bundle_workspace_floats(s, h, w):
        raise ValueError('workspace needs %d floats' % remap_bundle_workspace_floats(s, h, w))
    with torch.cuda.device(src.device):
        if out_format == 'bgr':
            check(lib.mgw_remap_bundle_frame(_p(src), SRC_FORMATS[src_format], _p(xy), s, h, w, H, W, _p(dst), _p(ws), _st()),
                  'mgw_remap_bundle_frame')
        else:
            check(lib.mgw_remap_bundle_frame_yuv420(_p(src), SRC_FORMATS[src_format], _p(xy), s, h, w, H, W, SRC_FORMATS[out_format],
                                                    _p(dst), _p(ws), _st()), 'mgw_remap_bundle_frame_yuv420')
    return dst


# ---- a batch of one size whose frames lie in decoder / encoder surfaces (deploy.StreamBatch.step_planes): per-slot planes
PLANES_ENTRY_BYTES = 48          # sizeof(mgw_planes)


def _planes_table(t, name):
    """a device table of mgw_planes: a contiguous CUDA tensor, uint8 [S,48] or int64 [S,6] (deploy.PlaneTable.device) -> S"""
    if not isinstance(t, torch.Tensor) or not t.is_cuda:
        raise ValueError('%s must be a CUDA tensor holding a table of mgw_planes' % name)
    if t.dtype not in (torch.uint8, torch.int64) or t.dim() != 2 or t.shape[1] * t.element_size() != PLANES_ENTRY_BYTES:
        raise ValueError('%s must be uint8 [S,%d] or int64 [S,%d] (got %s %s)' % (name, PLANES_ENTRY_BYTES, PLANES_ENTRY_BYTES // 8,
                                                                                  t.dtype, tuple(t.shape)))
    if not t.is_contiguous():
        raise ValueError('%s must be contiguous' % name)
    return int(t.shape[0])


def cvt_img2train_planes(table, fmt, size, tables, out_h, out_w, out=None, tmp=None):
    """cvt_img2train of S frames of one size (H, W) = size, each described by its entry of the planes table (fmt 'bgr', 'nv12' or
    'i420') -> [S,out_h,out_w] fp32, byte for byte the uniform batch call on the packed frames; the uniform tables.  Idle slots
    (a missing plane or a short pitch) leave their rows of out / tmp [S,H,out_w] untouched.  One C-ABI call."""
    if fmt not in SRC_FORMATS:
        raise ValueError('source format must be one of %s (got %r)' % (sorted(SRC_FORMATS), fmt))
    s, (h, w) = _planes_table(table, 'table'), (int(size[0]), int(size[1]))
    kx, x0, xn, ky, y0, yn = (_chk(t, 'table', torch.int32) for t in tables)
    if kx.shape[0] != out_w or ky.shape[0] != out_h:
        raise ValueError('the tables must cover the %dx%d output' % (out_h, out_w))
    tmp = _out(tmp, (s, h, out_w), table.device, torch.uint8, 'tmp')
    out = _out(out, (s, out_h, out_w), table.device, torch.float32, 'out')
    with torch.cuda.device(table.device):
        check(lib.mgw_cvt_img2train_planes(_p(table), SRC_FORMATS[fmt], s, h, w, _p(kx), _p(x0), _p(xn), kx.shape[1], _p(ky), _p(y0),
                                           _p(yn), ky.shape[1], out_h, out_w, _p(tmp), _p(out), _st()), 'mgw_cvt_img2train_planes')
    return out


def resize_linear_planes(table, fmt, size, xtab, ytab, out_h, out_w, out=None):
    """cv2.resize of S frames of one size described by the planes table -> [S,out_h,out_w,3] BGR, contiguous (the uniform
    tables; None / None for the 2x2 shortcut).  Idle slots leave their rows of out untouched.  One C-ABI call."""
    if fmt not in SRC_FORMATS:
        raise ValueError('source format must be one of %s (got %r)' % (sorted(SRC_FORMATS), fmt))
    s, (h, w) = _planes_table(table, 'table'), (int(size[0]), int(size[1]))
    xtab = None if xtab is None else _chk(xtab, 'xtab', torch.int32)
    ytab = None if ytab is None else _chk(ytab, 'ytab', torch.int32)
    dst = _out(out, (s, out_h, out_w, 3), table.device, torch.uint8, 'out')
    with torch.cuda.device(table.device):
        check(lib.mgw_resize_linear_planes(_p(table), SRC_FORMATS[fmt], s, h, w, _p(xtab), _p(ytab), out_h, out_w, _p(dst), _st()),
              'mgw_resize_linear_planes')
    return dst


def remap_bundle_frame_planes(src_table, src_format, xy, size, dst_table, dst_format, workspace=None):
    """warpRevBundle2 of S frames of one size (H, W) = size from the surfaces of src_table into those of dst_table (dst_format
    'bgr', 'nv12' or 'i420'; H and W even when either format is YUV), xy [S,h,w,2] fp32.  Each active slot's used bytes are
    remap_bundle_frame's on the packed frame; pitch padding, bytes between planes and idle slots are not written.  workspace:
    optional fp32 scratch of remap_bundle_workspace_floats(S, h, w).  Returns dst_table.  One C-ABI call (two launches)."""
    for name, f in (('source format', src_format), ('dst_format', dst_format)):
        if f not in SRC_FORMATS:
            raise ValueError('%s must be one of %s (got %r)' % (name, sorted(SRC_FORMATS), f))
    s, (H, W) = _planes_table(src_table, 'src_table'), (int(size[0]), int(size[1]))
    if _planes_table(dst_table, 'dst_table') != s:
        raise ValueError('src_table and dst_table must have one entry per slot (got %d and %d)' % (s, dst_table.shape[0]))
    xy = _chk(xy, 'xy')
    if xy.dim() != 4 or xy.shape[0] != s or xy.shape[3] != 2:
        raise ValueError('xy must be [%d,h,w,2] (got %s)' % (s, tuple(xy.shape)))
    h, w = int(xy.shape[1]), int(xy.shape[2])
    ws = (torch.empty(remap_bundle_workspace_floats(s, h, w), device=xy.device, dtype=torch.float32) if workspace is None
          else _chk_out(workspace, 'workspace'))
    if ws.numel() < remap_bundle_workspace_floats(s, h, w):
        raise ValueError('workspace needs %d floats' % remap_bundle_workspace_floats(s, h, w))
    if not (src_table.device == dst_table.device == xy.device == ws.device):
        raise ValueError('src_table, dst_table, xy and workspace must be on one device (got %s, %s, %s, %s)'
                         % (src_table.device, dst_table.device, xy.device, ws.device))
    with torch.cuda.device(xy.device):
        check(lib.mgw_remap_bundle_frame_planes(_p(src_table), SRC_FORMATS[src_format], _p(xy), s, h, w, H, W, _p(dst_table),
                                                SRC_FORMATS[dst_format], _p(ws), _st()), 'mgw_remap_bundle_frame_planes')
    return dst_table

"""Deploy-side helpers with the reference's names (deploy_bundle.py).

    img_warped = warpRevBundle2(cv2.resize(frame, (width, height)), xmap, ymap)      # reference deploy_bundle.py:301

`warpRevBundle2` keeps the reference signature -- one uint8 frame [H,W,3] and the operator's x_map / y_map [H,W] -- and
accepts numpy arrays (as the reference's caller passes; the result comes back as a numpy array) or CUDA tensors (batched
[N,H,W,C] / [N,H,W] too; the result stays on the device).  The work is one C-ABI call, mgw_remap_bundle_u8; a frame of
another size than the maps (1080p with the network's 288x512 maps) is stabilised at its own size by mgw_remap_bundle_frame.

StreamBatch runs the whole per-frame loop for S videos of one size at once: one set of launches per frame, capturable as one
CUDA graph, every video's result bit-identical to its own StreamState / CropState pipeline.  MixedStreamBatch does the same for
videos of different source sizes up to a capacity.
"""
import numpy as np
import torch

from . import ops

__all__ = ['warpRevBundle2', 'warpRevBundle', 'warpRev', 'cvt_theta_mat_bundle', 'cvt_img2train', 'cv2_resize', 'StreamState', 'CropState', 'StreamBatch',
           'MixedStreamBatch', 'mixed_slot_tables', 'scale_rect', 'PlaneTable', 'MixedPlaneTable']


def warpRevBundle2(img, x_map, y_map, device=None, src_format='bgr', dst_format='bgr'):
    """The frame img, of any size, stabilised at its own size with the operator's x_map / y_map (network size): the reference's
    expression with the size the colour frame is resized to taken from the frame instead of the network.  A frame at the maps'
    size is exactly the reference's warpRevBundle2.  img: [H,W,C] or [N,H,W,C] uint8 BGR, or for src_format 'nv12' / 'i420' a
    YUV 4:2:0 frame [3H/2,W] or batch [N,3H/2,W] (read as the BGR frame cv2.cvtColor makes of it; the result is BGR [H,W,3]).
    dst_format 'nv12' / 'i420' (3-channel frames of even size): the result is YUV 4:2:0 [3H/2,W] ([N,3H/2,W]) for a video
    encoder, cv2.cvtColor(COLOR_BGR2YUV_I420) of the BGR result (U and V interleaved for NV12), converted inside the warp."""
    as_numpy = isinstance(img, np.ndarray)
    dev = torch.device(device) if device is not None else (torch.device('cuda') if as_numpy else img.device)

    def to_dev(a, dtype):
        t = torch.as_tensor(np.ascontiguousarray(a)) if isinstance(a, np.ndarray) else a
        return t.to(device=dev, dtype=dtype)

    xm, ym = to_dev(x_map, torch.float32), to_dev(y_map, torch.float32)
    yuv = _yuv420_frames(img, src_format)
    if yuv is not None:
        im, single, H, W = yuv
        im = im.to(device=dev).contiguous()
    else:
        im = to_dev(img, torch.uint8)
        single = im.dim() == 3
        if single:
            im = im.unsqueeze(0)
        H, W = int(im.shape[1]), int(im.shape[2])
    n = int(im.shape[0])
    if yuv is None and dst_format == 'bgr' and xm.numel() == n * H * W:
        # the maps have the frame's size: the reference's call
        xy = torch.stack([xm.reshape(n, H, W), ym.reshape(n, H, W)], dim=-1)
        dst = ops.remap_bundle_u8(im, xy)
    else:
        shape = list(xm.shape)
        while len(shape) > 2 and shape[-1] == 1:        # [1,h,w,1] as the network hands it out
            shape.pop()
        if len(shape) < 2 or xm.numel() != n * shape[-2] * shape[-1] or ym.numel() != xm.numel():
            raise ValueError('x_map / y_map must be [h,w] maps, one per frame (got %s for %d frames)' % (tuple(xm.shape), n))
        h, w = shape[-2], shape[-1]
        xy = torch.stack([xm.reshape(n, h, w), ym.reshape(n, h, w)], dim=-1)
        dst = ops.remap_bundle_frame(im.contiguous(), src_format, xy, out_format=dst_format)
    if single:
        dst = dst[0]
    return dst.cpu().numpy() if as_numpy else dst


def scale_rect(rect, from_size, to_size):
    """A crop rectangle [top, left, bottom, right] (inclusive, as leave() / CropState.rect() give it on the network's lattice
    from_size = (h, w)) carried to an output of to_size = (OH, OW) pixels with the centre alignment of the maps: output row R is
    kept iff top <= (R + 0.5) * h / OH - 0.5 <= bottom (columns alike), in integers and clamped to the output.  The identity at
    equal sizes."""
    t, l, b, r = (int(v) for v in rect)
    (h, w), (OH, OW) = (int(v) for v in from_size), (int(v) for v in to_size)

    def first(lo, n, N):            # ceil(((2 lo + 1) N - n) / (2 n))
        return min(max(-((n - (2 * lo + 1) * N) // (2 * n)), 0), N - 1)

    def last(hi, n, N):             # floor(((2 hi + 1) N - n) / (2 n))
        return min(max(((2 * hi + 1) * N - n) // (2 * n), 0), N - 1)

    return [first(t, h, OH), first(l, w, OW), last(b, h, OH), last(r, w, OW)]


def _pil_bilinear_windows(in_size, out_size):
    """Pillow's precompute_coeffs + normalize_coeffs_8bpc (src/libImaging/Resample.c) for BILINEAR, in the same double
    arithmetic: per output sample the first source index, the window length and the 22-bit fixed-point weights."""
    import math
    scale = in_size / float(out_size)
    filterscale = max(scale, 1.0)
    support = 1.0 * filterscale
    ksize = _pil_ksize(in_size, out_size)
    first = np.zeros(out_size, np.int32)
    count = np.zeros(out_size, np.int32)
    kk = np.zeros((out_size, ksize), np.int32)
    ss = 1.0 / filterscale
    for xx in range(out_size):
        center = (xx + 0.5) * scale
        xmin = max(int(center - support + 0.5), 0)
        xmax = min(int(center + support + 0.5), in_size) - xmin
        w = [max(1.0 - abs((x + xmin - center + 0.5) * ss), 0.0) for x in range(xmax)]
        ww = 0.0
        for v in w:
            ww += v
        for x, v in enumerate(w):
            v = v / ww if ww != 0.0 else v
            kk[xx, x] = int(v * (1 << 22) + 0.5)
        first[xx], count[xx] = xmin, xmax
    return kk, first, count


def _pil_ksize(in_size, out_size):
    """the window length of _pil_bilinear_windows: 2*ceil(max(in/out, 1)) + 1, which does not decrease as in_size grows"""
    import math
    return int(math.ceil(1.0 * max(in_size / float(out_size), 1.0))) * 2 + 1


def _cv_linear_table(n_out, n_in, horizontal):
    """resize.cpp: fx = (float)((d + 0.5) * scale - 0.5), s = floor(fx), fx -= s; horizontally a tap outside the row is folded
    onto the border with weight 0, vertically the row indices are clamped and the weights kept; 11-bit weights cvRound(w*2048)"""
    f32 = np.float32
    scale = 1.0 / (n_out / float(n_in))
    tab = np.zeros((n_out, 4), np.int32)
    for d in range(n_out):
        f = f32((d + 0.5) * scale - 0.5)
        s0 = int(np.floor(f))
        f = f32(f - f32(s0))
        if horizontal:
            if s0 < 0:
                s0, f = 0, f32(0)
            if s0 >= n_in - 1:
                s0, f = n_in - 1, f32(0)
            i0, i1 = s0, min(s0 + 1, n_in - 1)
        else:
            i0, i1 = min(max(s0, 0), n_in - 1), min(max(s0 + 1, 0), n_in - 1)
        tab[d] = (i0, i1, int(np.rint(f32(f32(1) - f) * f32(2048))), int(np.rint(f * f32(2048))))
    return tab


_CVT_TABLES = {}
_RESIZE_TABLES = {}


def _resize_tables(H, W, oh, ow, device):
    key = (H, W, oh, ow, str(device))
    if key not in _RESIZE_TABLES:
        if W == 2 * ow and H == 2 * oh:
            _RESIZE_TABLES[key] = (None, None)
        else:
            _RESIZE_TABLES[key] = (torch.as_tensor(_cv_linear_table(ow, W, True)).to(device),
                                   torch.as_tensor(_cv_linear_table(oh, H, False)).to(device))
    return _RESIZE_TABLES[key]


def _yuv420_frames(img, src_format):
    """src_format 'bgr' -> None.  'nv12' / 'i420': img is a YUV 4:2:0 frame [3H/2,W] or a batch [S,3H/2,W] (uint8, OpenCV's
    layout) -> (the frames as a uint8 tensor [S,3H/2,W] where they are, single, H, W).  Anything else is a ValueError."""
    if src_format == 'bgr':
        return None
    if src_format not in ops.YUV420_FORMATS:
        raise ValueError("src_format must be 'bgr', 'nv12' or 'i420' (got %r)" % (src_format,))
    is_np = isinstance(img, np.ndarray)
    if not is_np and not isinstance(img, torch.Tensor) or img.dtype != (np.uint8 if is_np else torch.uint8):
        raise ValueError('a %s frame must be a uint8 array or tensor (got %s)' % (src_format, getattr(img, 'dtype', type(img))))
    shape = tuple(img.shape)
    if len(shape) not in (2, 3) or shape[-2] % 3 != 0 or shape[-2] == 0 or shape[-1] % 2 != 0 or shape[-1] == 0:
        raise ValueError('a %s frame must be [3H/2,W] or [S,3H/2,W] with H and W even (got %s)' % (src_format, shape))
    t = torch.as_tensor(np.ascontiguousarray(img)) if is_np else img
    return (t.unsqueeze(0) if len(shape) == 2 else t), len(shape) == 2, shape[-2] // 3 * 2, shape[-1]


def cv2_resize(img, dsize, device='cuda', src_format='bgr'):
    """cv2.resize(img, dsize) for a uint8 frame [H,W,C] (reference deploy_bundle.py:301 resizes the unstable colour frame to the
    network size before warpRevBundle2), byte-exact with OpenCV's INTER_LINEAR; dsize = (width, height) as in OpenCV.
    A batch [S,H,W,C] of frames of one size gives [S,height,width,C], each frame as its own call would (one launch).
    src_format 'nv12' / 'i420': img is a YUV 4:2:0 frame [3H/2,W] (or a batch [S,3H/2,W]) in OpenCV's layout, and the result
    is the BGR call's on cv2.cvtColor(img, COLOR_YUV2BGR_NV12 / _I420), [height,width,3] ([S,height,width,3]), with the
    conversion done inside the kernel.  numpy in -> numpy out; a CUDA frame stays on the device."""
    as_numpy = isinstance(img, np.ndarray)
    ow, oh = int(dsize[0]), int(dsize[1])
    yuv = _yuv420_frames(img, src_format)
    if yuv is not None:
        yuv, single, H, W = yuv
        yuv = yuv.to(device=device if as_numpy else img.device).contiguous()
        xtab, ytab = _resize_tables(H, W, oh, ow, yuv.device)
        dst = ops.resize_linear_yuv420_batch(yuv, src_format, xtab, ytab, oh, ow)
        dst = dst[0] if single else dst
        return dst.cpu().numpy() if as_numpy else dst
    im = (torch.as_tensor(np.ascontiguousarray(img)) if as_numpy else img).to(device=device if as_numpy else img.device, dtype=torch.uint8)
    H, W = int(im.shape[-3]), int(im.shape[-2])
    xtab, ytab = _resize_tables(H, W, oh, ow, im.device)
    if im.dim() == 4:
        dst = ops.resize_linear_u8_batch(im.contiguous(), xtab, ytab, oh, ow)
    else:
        dst = ops.resize_linear_u8(im.contiguous(), xtab, ytab, oh, ow)
    return dst.cpu().numpy() if as_numpy else dst


def _resample_size(height, width, crop_rate):
    """(h, w, dh, dw): the size cvt_img2train resizes to and the offset of the centre crop"""
    if crop_rate != 1:
        h = int(height / crop_rate); dh = int((h - height) / 2)
        w = int(width / crop_rate); dw = int((w - width) / 2)
        return h, w, dh, dw
    return height, width, 0, 0


def _cvt_windows(H, W, height, width, crop_rate):
    """cvt_img2train's tables (kx, x0, xn, ky, y0, yn) for an H x W source, numpy int32"""
    h, w, dh, dw = _resample_size(height, width, crop_rate)
    kx, x0, xn = _pil_bilinear_windows(W, w)
    ky, y0, yn = _pil_bilinear_windows(H, h)
    return kx[dw:dw + width], x0[dw:dw + width], xn[dw:dw + width], ky[dh:dh + height], y0[dh:dh + height], yn[dh:dh + height]


def _cvt_tables(H, W, height, width, crop_rate, device):
    key = (H, W, height, width, float(crop_rate), str(device))
    if key not in _CVT_TABLES:
        tabs = _cvt_windows(H, W, height, width, crop_rate)
        _CVT_TABLES[key] = tuple(torch.as_tensor(np.ascontiguousarray(t)).to(device) for t in tabs)
    return _CVT_TABLES[key]


def mixed_slot_tables(src_size, max_src_size, height=288, width=512, crop_rate=1, out_size=None):
    """One slot's tables for the per-slot calls (ops.cvt_img2train_mixed / ops.resize_linear_mixed), numpy int32:
    (kx [width,ksx], x0, xn [width], ky [height,ksy], y0, yn [height], xtab [OW,4], ytab [OH,4]).  They are the uniform
    tables at the slot's size src_size = (H, W), with the Pillow windows zero-padded to the lengths ksx, ksy of the capacity
    max_src_size; xtab / ytab resize to out_size = (OH, OW) (default: the network's (height, width)) and are given even where
    the slot takes the 2x2 shortcut."""
    (H, W), (mh, mw) = (int(v) for v in src_size), (int(v) for v in max_src_size)
    if not (0 < H <= mh and 0 < W <= mw):
        raise ValueError('source size %dx%d outside the capacity %dx%d' % (H, W, mh, mw))
    rh, rw, _, _ = _resample_size(height, width, crop_rate)
    kx, x0, xn, ky, y0, yn = _cvt_windows(H, W, height, width, crop_rate)
    ksx, ksy = _pil_ksize(mw, rw), _pil_ksize(mh, rh)
    if kx.shape[1] > ksx or ky.shape[1] > ksy:
        raise ValueError('a %dx%d source needs longer windows than its capacity %dx%d' % (H, W, mh, mw))
    kxp, kyp = np.zeros((width, ksx), np.int32), np.zeros((height, ksy), np.int32)
    kxp[:, :kx.shape[1]], kyp[:, :ky.shape[1]] = kx, ky
    oh, ow = (height, width) if out_size is None else (int(out_size[0]), int(out_size[1]))
    return (kxp, np.ascontiguousarray(x0), np.ascontiguousarray(xn), kyp, np.ascontiguousarray(y0), np.ascontiguousarray(yn),
            _cv_linear_table(ow, W, True), _cv_linear_table(oh, H, False))


def cvt_img2train(img, crop_rate=1, height=288, width=512, device='cuda', as_numpy=False, src_format='bgr'):
    """reference config.py:6-21 (`height`, `width` are its config globals): one BGR uint8 frame [H,W,3] -> the network's frame
    format, exact: cv2 BGR2GRAY, Pillow resize(BILINEAR) (to (width, height), or to the 1/crop_rate larger size followed by
    the centre crop), v * (1/255) - 0.5.  Returns a CUDA fp32 tensor [1,height,width,1]; as_numpy=True gives the reference's
    float64 numpy array (same values: the network's placeholder casts to fp32).  The coefficient tables are built once per
    shape on the host and kept on the device.  A batch [S,H,W,3] of frames of one size gives [S,height,width,1], each frame
    as its own call would (one pair of launches for the batch).
    src_format 'nv12' / 'i420': img is a YUV 4:2:0 frame [3H/2,W] (or a batch [S,3H/2,W]) in OpenCV's layout, as video
    decoders emit it, and the result is the BGR call's on cv2.cvtColor(img, COLOR_YUV2BGR_NV12 / _I420): the conversion runs
    inside the kernel, and the gray frame is BGR2GRAY of the converted frame (not the Y plane)."""
    yuv = _yuv420_frames(img, src_format)
    if yuv is not None:
        yuv, _, H, W = yuv
        yuv = yuv.to(device=device).contiguous()
        tabs = _cvt_tables(H, W, height, width, crop_rate, yuv.device)
        out = ops.cvt_img2train_yuv420_batch(yuv, src_format, tabs, height, width).reshape(-1, height, width, 1)
    else:
        im = (torch.as_tensor(np.ascontiguousarray(img)) if isinstance(img, np.ndarray) else img).to(device=device, dtype=torch.uint8)
        H, W = int(im.shape[-3]), int(im.shape[-2])
        tabs = _cvt_tables(H, W, height, width, crop_rate, im.device)
        if im.dim() == 4:
            out = ops.cvt_img2train_u8_batch(im.contiguous(), tabs, height, width).reshape(-1, height, width, 1)
        else:
            out = ops.cvt_img2train_u8(im.contiguous(), tabs, height, width).reshape(1, height, width, 1)
    if not as_numpy:
        return out
    v = np.rint((out.cpu().numpy().astype(np.float64) + 0.5) * 255)          # the resampled byte, recovered exactly
    return v * (1. / 255) - 0.5


def cvt_theta_mat_bundle(Hs, height, width, grid_h, grid_w):
    """reference deploy_bundle.py:121-134 with its own numpy expressions (float64 on the host: 16 3x3 products), so that the
    pixel-space homographies the kernel receives are the reference's bit for bit; height / width / grid are its config globals."""
    from numpy.linalg import inv
    scale_mat = np.eye(3)
    scale_mat[0, 0] = width / 2.
    scale_mat[0, 2] = width / 2.
    scale_mat[1, 1] = height / 2.
    scale_mat[1, 2] = height / 2.
    Hs = np.asarray(Hs).reshape((grid_h, grid_w, 3, 3))
    return np.matmul(np.matmul(scale_mat, Hs), inv(scale_mat))


def warpRevBundle(img, Hs, grid=(4, 4), device=None):
    """reference deploy_bundle.py:148-173: one uint8 frame [H,W,3] and the operator's Hs ([gh,gw,9] or anything that reshapes to
    it, as `Hs[0]` of the reference's fetch) -> the frame with every mesh cell warped by its own homography
    (cv2.warpPerspective, WARP_INVERSE_MAP | INTER_LINEAR, byte-exact).  numpy in -> numpy out; a CUDA frame stays on the device."""
    as_numpy = isinstance(img, np.ndarray)
    dev = torch.device(device) if device is not None else (torch.device('cuda') if as_numpy else img.device)
    im = (torch.as_tensor(np.ascontiguousarray(img)) if as_numpy else img).to(device=dev, dtype=torch.uint8)
    h, w = im.shape[-3], im.shape[-2]
    gh, gw = int(grid[0]), int(grid[1])
    Hs_np = Hs.detach().cpu().numpy() if isinstance(Hs, torch.Tensor) else np.asarray(Hs)
    Hc = torch.as_tensor(np.ascontiguousarray(cvt_theta_mat_bundle(Hs_np, h, w, gh, gw), dtype=np.float64)).to(dev)
    dst = ops.warp_rev_bundle_u8(im.reshape(1, h, w, -1).contiguous(), Hc.reshape(1, gh, gw, 9), gh, gw)[0]
    return dst.cpu().numpy() if as_numpy else dst


def warpRev(img, theta, device=None):
    """reference deploy_bundle.py:100-118: cv2.warpPerspective(img, cvt_theta_mat(theta), WARP_INVERSE_MAP | INTER_LINEAR) for one
    3x3 homography in normalised coordinates -- the 1x1-grid case of warpRevBundle."""
    return warpRevBundle(img, np.asarray(theta.detach().cpu() if isinstance(theta, torch.Tensor) else theta).reshape(1, 1, 9),
                         grid=(1, 1), device=device)


class StreamState:
    """The per-video state of deploy_bundle.py on the device: the last `depth` stabilised frames and their black masks
    (the reference's before_frames / before_masks lists, :221-224) as rings, the 13-channel network input assembled from
    the index taps in one launch (:259-274), the refine re-feed (:292-295) and the per-frame update (:319-328).

        st = StreamState(first_frame)                    # first_frame: [H,W] fp32 (cvt_img2train output)
        for frame in video:
            in_x = st.assemble(frame)                    # [1,H,W,13] = 6 masks + 6 frames + current
            for _ in range(refine):
                img, black = net(in_x)                   # the network + the multi-grid warp
                st.refeed(in_x, img, black)              # in_x[..., -1] = img - black
            st.push(img, black)
    """

    def __init__(self, first_frame, depth=32, taps=(1, 2, 4, 8, 16, 32), use_masks=True, device='cuda', device_head=False):
        """device_head=True keeps the ring head in device memory: assemble / push then take no per-frame launch parameter, so the
        whole frame loop can be captured in one CUDA graph and replayed (the host-side `head` is not maintained in that mode)."""
        f = torch.as_tensor(first_frame, dtype=torch.float32).to(device)
        h, w = f.shape
        self.frames = f.reshape(1, h, w).repeat(depth, 1, 1).contiguous()
        self.masks = torch.zeros((depth, h, w), device=f.device, dtype=torch.float32)
        self.depth, self.taps, self.use_masks, self.head = depth, tuple(int(t) for t in taps), use_masks, depth - 1
        self.head_dev = torch.full((1,), depth - 1, device=f.device, dtype=torch.int32) if device_head else None

    def assemble(self, cur, out=None):
        cur = torch.as_tensor(cur, dtype=torch.float32).to(self.frames.device).reshape(self.frames.shape[1:]).contiguous()
        if self.head_dev is not None:
            return ops.stream_assemble_dev(self.frames, self.masks, self.head_dev, self.taps, cur, self.use_masks, out=out)
        return ops.stream_assemble(self.frames, self.masks, self.head, self.taps, cur, self.use_masks)

    def refeed(self, in_x, img, black):
        ops.stream_push(None, None, 0, img.reshape(self.frames.shape[1:]).contiguous(), black.reshape(self.frames.shape[1:]).contiguous(),
                        refeed_into=in_x)

    def push(self, img, black):
        img, black = img.reshape(self.frames.shape[1:]).contiguous(), black.reshape(self.frames.shape[1:]).contiguous()
        if self.head_dev is not None:
            ops.stream_push_dev(self.frames, self.masks, self.head_dev, img, black)
            return
        self.head = (self.head + 1) % self.depth
        ops.stream_push(self.frames, self.masks, self.head, img, black)

    def history(self):
        """(frames, masks) oldest first, as the reference's lists hold them"""
        head = int(self.head_dev.item()) if self.head_dev is not None else self.head
        order = [(head + 1 + k) % self.depth for k in range(self.depth)]
        return self.frames[order], self.masks[order]


def _crop_rect(all_black, step):
    r = [int(v) for v in ops.crop_rect(all_black, step).cpu()]
    if r[0] < 0:
        raise IndexError('no black-free rectangle: every lattice corner has been black (the reference fails on ans[3] here)')
    return r


class CropState:
    """The crop bookkeeping of deploy_bundle.py: `all_black` (:240) gathers every black mask the network produced (:291),
    and after the last frame the largest never-black rectangle on the 10-pixel corner lattice (:344-365) is cut out of
    every output frame (:368-370).

        crop = CropState(height, width)
        ... crop.add(black) after every network evaluation ...
        top, left, bottom, right = crop.rect()
        cut = crop.cut(frame)                            # frame[top:bottom+1, left:right+1, :]
    """

    def __init__(self, height, width, device='cuda'):
        self.all_black = torch.zeros((height, width), device=device, dtype=torch.int32)

    def add(self, black):
        ops.black_accumulate(self.all_black, black)

    def rect(self, step=10):
        return _crop_rect(self.all_black, step)

    def cut(self, frame, step=10):
        t, l, b, r = self.rect(step)
        return frame[..., t:b + 1, l:r + 1, :]


_PLANES_DTYPE = np.dtype([('plane', '<u8', (3,)), ('pitch', '<i4', (3,)), ('reserved', '<i4', (3,))])     # mgw_planes, 48 bytes


def _plane_rows(fmt, H, W):
    """(rows, row bytes) of each plane of an H x W frame in fmt"""
    if fmt == 'bgr':
        return [(H, 3 * W)]
    if fmt == 'nv12':
        return [(H, W), (H // 2, W)]
    return [(H, W), (H // 2, W // 2), (H // 2, W // 2)]


def _packed_planes(fmt, base, H, W):
    """the (address, pitch) pairs of an H x W frame packed at address base: each plane after the previous one, pitch = row bytes"""
    planes, off = [], 0
    for rows, nbytes in _plane_rows(fmt, H, W):
        planes.append((base + off, nbytes))
        off += rows * nbytes
    return planes


class _PlaneMirror:
    """What PlaneTable and MixedPlaneTable share: the pinned host mirror of S mgw_planes entries, the device table, the checks of
    one entry's planes against a frame size, clear() and upload()."""

    def __init__(self, S, fmt, size, device, what):
        """S entries of fmt for frames up to size (H, W); what names the size in the error"""
        S, H, W = int(S), int(size[0]), int(size[1])
        if fmt not in ops.SRC_FORMATS:
            raise ValueError("fmt must be 'bgr', 'nv12' or 'i420' (got %r)" % (fmt,))
        if not 1 <= S <= 65535 or not (1 <= H <= 32767 and 1 <= W <= 32767) or (fmt != 'bgr' and (H % 2 or W % 2)):
            raise ValueError('%s needs 1 <= S <= 65535 and a %s in [1, 32767], even for %s (got S=%d, %dx%d)'
                             % (type(self).__name__, what, fmt, S, H, W))
        dev = torch.device(device)
        self.S, self.fmt = S, fmt
        self.host = torch.zeros((S, ops.PLANES_ENTRY_BYTES // 8), dtype=torch.int64, pin_memory=dev.type == 'cuda')
        self.device = torch.zeros((S, ops.PLANES_ENTRY_BYTES // 8), dtype=torch.int64, device=dev)
        self.uploaded = torch.cuda.Event(external=True) if dev.type == 'cuda' else None
        self._entries = self.host.numpy().view(_PLANES_DTYPE).reshape(S)
        self._keep = [None] * S

    def _slot(self, slot):
        if not isinstance(slot, (int, np.integer)) or not 0 <= slot < self.S:
            raise ValueError('slot %r outside [0, %d)' % (slot, self.S))
        return int(slot)

    def _write(self, slot, planes, H, W, reserved):
        """entry `slot` = the planes of an H x W frame (checked as set() documents) and the words `reserved`, into the mirror"""
        s = self._slot(slot)
        rows = _plane_rows(self.fmt, H, W)
        if len(planes) != len(rows):
            raise ValueError('a %s frame has %d planes (got %d)' % (self.fmt, len(rows), len(planes)))
        addr, pitch = [0, 0, 0], [0, 0, 0]
        for k, (p, (n, nbytes)) in enumerate(zip(planes, rows)):
            if isinstance(p, torch.Tensor):
                if p.dtype != torch.uint8 or p.device != self.device.device:
                    raise ValueError('plane %d must be a uint8 tensor on %s (got %s on %s)' % (k, self.device.device, p.dtype, p.device))
                if p.dim() == 3 and self.fmt == 'bgr' and p.shape[2] == 3 and p.stride(2) == 1 and p.stride(1) == 3:
                    cover = p.shape[0] >= n and p.shape[1] * 3 >= nbytes
                else:
                    cover = p.dim() == 2 and p.stride(1) == 1 and p.shape[0] >= n and p.shape[1] >= nbytes
                if not cover:
                    raise ValueError('plane %d must cover %d rows of %d bytes with unit column stride (got %s, strides %s)'
                                     % (k, n, nbytes, tuple(p.shape), p.stride()))
                a, q = p.data_ptr(), p.stride(0)
            else:
                a, q = int(p[0]), int(p[1])
            if a == 0:
                raise ValueError('plane %d of slot %d is missing (address 0)' % (k, s))
            if not nbytes <= q < 2 ** 31:
                raise ValueError('plane %d of slot %d: pitch %d is below its %d row bytes (or above 2^31)' % (k, s, q, nbytes))
            addr[k], pitch[k] = a, q
        self._entries[s] = (addr, pitch, reserved)
        self._keep[s] = [p for p in planes if isinstance(p, torch.Tensor)]

    def clear(self, slot):
        """Slot `slot` becomes idle: the plane-table calls read and write nothing for it (after the next upload())."""
        s = self._slot(slot)
        self._entries[s] = ((0, 0, 0), (0, 0, 0), (0, 0, 0))
        self._keep[s] = None

    def upload(self):
        """One cudaMemcpyAsync of the host mirror into the device table on the current stream, then the event `uploaded`."""
        self.device.copy_(self.host, non_blocking=True)
        if self.uploaded is not None:
            self.uploaded.record()


class PlaneTable(_PlaneMirror):
    """Where the S frames of a batch of one size lie: per slot the device address and row pitch of each plane, as a decoder or an
    encoder hands its surfaces out.  A pinned host mirror (host, int64 [S,6], one include/mgw.h mgw_planes per row) that set() /
    clear() edit, and the device table (device) that the plane-table calls read, refreshed by upload().

        src = PlaneTable(S, 'nv12', (1080, 1920))
        src.set(0, (y_plane, uv_plane))                 # pitched uint8 CUDA views: [1080,>=1920] and [540,>=1920]
        src.set(1, ((y_addr, pitch), (uv_addr, pitch))) # or raw (address, pitch) pairs from any decoder binding
        src.clear(2)                                    # slot 2 is idle: nothing is read or written for it
        src.upload()

    fmt 'bgr': one plane of H rows of 3W bytes; 'nv12': Y (H rows of W) and interleaved UV (H/2 rows of W); 'i420': Y, U and V
    (H/2 rows of W/2 each).  Pitches are in bytes, need no alignment, and planes need not be adjacent.  set() checks each entry:
    every plane present and its pitch at least its row bytes.  The table holds addresses only: the caller keeps the surfaces
    alive (views passed to set() are referenced until the slot is set again or cleared).

    upload() is one cudaMemcpyAsync of the mirror on the current stream, followed by the event `uploaded`.  Inside a captured
    graph (StreamBatch.capture_planes) the copy is recorded and reads the mirror at every replay, so the mirror must not be edited
    while a replay that reads it is in flight: wait for `uploaded` (uploaded.synchronize()) after replaying before the next edit,
    or alternate two tables, each with its own graph."""

    def __init__(self, S, fmt, size, device='cuda'):
        super().__init__(S, fmt, size, device, 'size')
        self.size = (int(size[0]), int(size[1]))

    @classmethod
    def packed(cls, batch, fmt):
        """The table of a contiguous batch [S,H,W,3] ('bgr') or [S,3H/2,W] ('nv12' / 'i420'): pitches are the row bytes.
        Uploaded on the current stream."""
        if fmt == 'bgr':
            S, H, W = int(batch.shape[0]), int(batch.shape[1]), int(batch.shape[2])
        else:
            S, H, W = int(batch.shape[0]), int(batch.shape[1]) // 3 * 2, int(batch.shape[2])
        if not batch.is_contiguous() or batch.dtype != torch.uint8:
            raise ValueError('a packed batch must be a contiguous uint8 tensor')
        t = cls(S, fmt, (H, W), device=batch.device)
        base, frame = batch.data_ptr(), batch[0].numel()
        for s in range(S):
            t.set(s, _packed_planes(fmt, base + s * frame, H, W))
        t._keep = [batch] * S
        t.upload()
        return t

    def set(self, slot, planes):
        """Slot `slot`'s frame: one plane for 'bgr', two for 'nv12', three for 'i420', each a pitched uint8 view on the device
        ([rows, >= row bytes] with unit column stride, or [H,W,3] for 'bgr'; the pitch is its row stride) or an (address, pitch)
        pair.  Edits the host mirror only (see upload())."""
        self._write(slot, planes, *self.size, (0, 0, 0))


class MixedPlaneTable(_PlaneMirror):
    """PlaneTable for a MixedStreamBatch: the S frames have sizes of their own up to the capacity (H, W), and each entry names
    the size of the frame it describes (mgw_planes.reserved[0], reserved[1] = height, width).  The mixed plane-table calls read
    slot s only when its entry's size equals the batch's sizes[s]; otherwise the slot is idle.  host / device / uploaded, clear()
    and upload() are PlaneTable's, and so is the rule on editing the mirror while a captured replay may still copy it.

        src = MixedPlaneTable(S, 'nv12', (2160, 3840))
        src.set(0, (y_plane, uv_plane), (1080, 1920))  # slot 0's surface holds a 1080p frame
        src.set(1, ((y_addr, pitch), (uv_addr, pitch)), (720, 1280))
        src.upload()

    A slot that joins the batch again at another size stays idle until its entries are set at the new size and uploaded: a
    stale entry can only stop the slot, never let it read or write past the surface it names.  Not a PlaneTable: a uniform
    batch (StreamBatch.step_planes) refuses it."""

    def __init__(self, S, fmt, capacity, device='cuda'):
        super().__init__(S, fmt, capacity, device, 'capacity')
        self.capacity = (int(capacity[0]), int(capacity[1]))

    @classmethod
    def pool(cls, buf, fmt, capacity, sizes):
        """The table of a pool-shaped buffer buf (contiguous uint8, S rows of frame_bytes(capacity) bytes, e.g. MixedStreamBatch's
        pool or its output pool): slot s's frame lies packed at the start of its row at sizes[s] = (H_s, W_s), or is idle for
        None.  Uploaded on the current stream."""
        H, W = int(capacity[0]), int(capacity[1])
        if not isinstance(buf, torch.Tensor) or buf.dtype != torch.uint8 or not buf.is_contiguous():
            raise ValueError('a pool must be a contiguous uint8 tensor')
        S = int(buf.shape[0])
        if len(sizes) != S or buf[0].numel() != ops.dst_frame_bytes(fmt, H, W):
            raise ValueError('a %s pool of capacity %dx%d is [%d, %d] bytes with one size per slot (got %s and %d sizes)'
                             % (fmt, H, W, S, ops.dst_frame_bytes(fmt, H, W), tuple(buf.shape), len(sizes)))
        t = cls(S, fmt, (H, W), device=buf.device)
        row = buf[0].numel()
        for s, size in enumerate(sizes):
            if size is not None:
                t.set(s, _packed_planes(fmt, buf.data_ptr() + s * row, *size), size)
        t._keep = [buf] * S
        t.upload()
        return t

    def set(self, slot, planes, size):
        """Slot `slot`'s frame of size (H_s, W_s) = size: within the capacity, even for 'nv12' / 'i420'.  planes as for
        PlaneTable.set, each checked against that size; the size goes into the entry's reserved[0:2].  Edits the host mirror only."""
        H, W = int(size[0]), int(size[1])
        if not (1 <= H <= self.capacity[0] and 1 <= W <= self.capacity[1]) or (self.fmt != 'bgr' and (H % 2 or W % 2)):
            raise ValueError('a slot of a %s table of capacity %dx%d takes a size within it, even for YUV (got %dx%d)'
                             % ((self.fmt,) + self.capacity + (H, W)))
        self._write(slot, planes, H, W, (H, W, 0))


class StreamBatch:
    """S videos of one source size stabilised side by side.  Slot s holds what StreamState + CropState hold for one video (the
    history rings, a device-resident ring head, `all_black`), and one step advances every slot by one frame with one set of
    launches: the deploy loop of deploy_bundle.py:259-328 for all slots at once, each slot bit-identical to its own pipeline.

        sb = StreamBatch(4, (1080, 1920))               # 4 slots of 1080p BGR frames, network size 288x512
        sb.join(0, first_bgr)                           # slot 0 starts a video: [1080,1920,3] uint8
        for raw in frames:                              # raw: [4,1080,1920,3] uint8 on the device, one frame per slot
            colour = sb.step(raw, net)                  # [4,288,512,3] uint8: the stabilised frames
        top, left, bottom, right = sb.leave(0)          # slot 0's video ends: its crop rectangle

    src_format='nv12' or 'i420' takes the frames as video decoders emit them, YUV 4:2:0 [3H/2,W] uint8 in OpenCV's layout
    (src_size stays the picture's (H, W)): step() then takes [S,3H/2,W], join() a frame of that format, and every result is the
    BGR batch's on the frames cv2.cvtColor(COLOR_YUV2BGR_NV12 / _I420) makes of them -- half the bytes to upload, and the
    conversion runs inside the two kernels that read the source frame.

    net(in_x) takes the assembled input [S,h,w,nch] and returns (out [S,h,w,1], black [S,h,w], xy [S,h,w,2]): the network plus
    the multi-grid warp (out / black / img of the transformer), as StreamState's `net` does for one video.

    Every slot is computed at every step.  A slot that carries no video (never joined, or left and not joined again) runs on
    whatever frame the caller puts there and its output means nothing: the caller decides which slots carry a video and
    ignores the others.  All buffers are allocated here and never reallocated, so a step can be captured once as a CUDA graph
    (capture()) and replayed; join / leave between replays act on the same buffers.

    out_size=(OH, OW) sets the size of the stabilised colour frames (default: the network's (height, width), the reference's
    output).  The network's maps warp the frame resized to that size; at out_size == src_size nothing is resized and the warp
    reads the source batch (BGR or YUV 4:2:0) itself, so a 1080p video comes out at 1080p.  crop_rate does not act on the colour
    frames, as in the reference; scale_rect() carries leave()'s rectangle to output pixels.

    out_format='nv12' or 'i420' hands the stabilised frames out as a video encoder takes them: self.colour, step() and the
    captured download are YUV 4:2:0 [S,3OH/2,OW] uint8, cv2.cvtColor(COLOR_BGR2YUV_I420) of the BGR frames (U and V interleaved
    for NV12), converted inside the warp -- half the bytes to download.  The output size must then be even."""

    def __init__(self, S, src_size, height=288, width=512, depth=32, taps=(1, 2, 4, 8, 16, 32), use_masks=True, crop_rate=1, refine=1,
                 device='cuda', src_format='bgr', out_size=None, out_format='bgr'):
        S, H, W, h, w = int(S), int(src_size[0]), int(src_size[1]), int(height), int(width)
        if S < 1 or refine < 1:
            raise ValueError('StreamBatch needs S >= 1 and refine >= 1 (got S=%d, refine=%d)' % (S, refine))
        out = (h, w) if out_size is None else (int(out_size[0]), int(out_size[1]))
        if not (1 <= out[0] <= 32767 and 1 <= out[1] <= 32767):
            raise ValueError('out_size %s: each side in [1, 32767]' % (tuple(out_size),))
        if out_format not in ('bgr',) + tuple(ops.YUV420_FORMATS):
            raise ValueError("out_format must be 'bgr', 'nv12' or 'i420' (got %r)" % (out_format,))
        if out_format != 'bgr' and (out[0] % 2 or out[1] % 2):
            raise ValueError('a %s output needs an even size (got %dx%d)' % (out_format, out[0], out[1]))
        if src_format == 'bgr':
            self.frame_shape = (H, W, 3)
        elif src_format in ops.YUV420_FORMATS:
            if H % 2 or W % 2:
                raise ValueError('a %s source needs an even size (got %dx%d)' % (src_format, H, W))
            self.frame_shape = (H * 3 // 2, W)
        else:
            raise ValueError("src_format must be 'bgr', 'nv12' or 'i420' (got %r)" % (src_format,))
        self.src_format = src_format
        self.taps = tuple(int(t) for t in taps)
        if not 1 <= len(self.taps) <= 32 or any(t < 1 or t > depth for t in self.taps):
            raise ValueError('taps %s: 1 to 32 distances in [1, depth = %d]' % (self.taps, depth))
        dev = torch.device(device)
        self.S, self.src_size, self.height, self.width, self.depth = S, (H, W), h, w, int(depth)
        self.out_size, self.out_format = out, out_format
        # the remap reads the source batch itself when the output has its size; None keeps the network-size path as it was
        self._direct = out_size is not None and out == (H, W)
        self.use_masks, self.crop_rate, self.refine = bool(use_masks), crop_rate, int(refine)
        self.nch = (2 if use_masks else 1) * len(self.taps) + 1
        f32 = dict(device=dev, dtype=torch.float32)
        self.frames = torch.zeros((S, depth, h, w), **f32)
        self.masks = torch.zeros((S, depth, h, w), **f32)
        self.heads_dev = torch.full((S,), depth - 1, device=dev, dtype=torch.int32)
        self.all_black = torch.zeros((S, h, w), device=dev, dtype=torch.int32)
        # per-step buffers: the network frames, the horizontal pass of cvt_img2train, the network input, the resized and the
        # stabilised colour frames, the /4 maps of warpRevBundle2
        self.cur = torch.empty((S, h, w), **f32)
        self.cvt_tmp = torch.empty((S, H, w), device=dev, dtype=torch.uint8)
        self.in_x = torch.empty((S, h, w, self.nch), **f32)
        self.small = None if self._direct else torch.empty((S,) + out + (3,), device=dev, dtype=torch.uint8)
        self.colour = torch.empty((S,) + out + (3,) if out_format == 'bgr' else (S, out[0] * 3 // 2, out[1]), device=dev,
                                  dtype=torch.uint8)
        self.remap_ws = torch.empty(ops.remap_bundle_workspace_floats(S, h, w), **f32)
        self._init_front_end(dev)

    def _init_front_end(self, dev):
        """the coefficient tables of the two stages that read the source frame: the uniform ones of src_size"""
        (H, W), h, w = self.src_size, self.height, self.width
        self._cvt = _cvt_tables(H, W, h, w, self.crop_rate, dev)
        self._resize = _resize_tables(H, W, self.out_size[0], self.out_size[1], dev)

    def _slot(self, slot):
        if not isinstance(slot, (int, np.integer)) or not 0 <= slot < self.S:
            raise ValueError('slot %r outside [0, %d)' % (slot, self.S))
        return int(slot)

    def join(self, slot, first):
        """A new video starts in `slot`: its first frame (a uint8 frame in the batch's format -- BGR [H,W,3], or YUV 4:2:0
        [3H/2,W] --, or a network frame [h,w] fp32 already in cvt_img2train's format) fills the frames ring, the masks ring and all_black are zeroed and the head is reset -- what
        StreamState(first) and CropState() construct for one video."""
        s = self._slot(slot)
        dev = self.frames.device
        f = torch.as_tensor(np.ascontiguousarray(first)) if isinstance(first, np.ndarray) else first
        if f.dtype == torch.uint8:
            if tuple(f.shape) != self.frame_shape:
                raise ValueError('first frame must be %s uint8 (got %s)' % (list(self.frame_shape), tuple(f.shape)))
            f = cvt_img2train(f.to(dev), self.crop_rate, self.height, self.width, src_format=self.src_format).reshape(self.height, self.width)
        elif tuple(f.shape) != (self.height, self.width):
            raise ValueError('a network frame must be [%d,%d] (got %s)' % (self.height, self.width, tuple(f.shape)))
        self.frames[s].copy_(f.to(device=dev, dtype=torch.float32).expand(self.depth, self.height, self.width))
        self.masks[s].zero_()
        self.heads_dev[s].fill_(self.depth - 1)
        self.all_black[s].zero_()

    def leave(self, slot, step=10):
        """The video in `slot` has ended: its crop rectangle [top, left, bottom, right] (CropState.rect).  The slot's state is
        left as it is until the next join."""
        return _crop_rect(self.all_black[self._slot(slot)], step)

    def advance(self, cur, net):
        """One frame of every slot from network frames cur [S,h,w] (cvt_img2train's format): input assembly from the rings,
        `refine` x (net, black accumulation, re-feed of the current-frame channel), ring push.  Returns the last xy [S,h,w,2]."""
        S, h, w, nch = self.S, self.height, self.width, self.nch
        masks = self.masks if self.use_masks else None
        in_x = ops.streams_assemble(self.frames, masks, self.heads_dev, self.taps, cur, self.use_masks, out=self.in_x)
        for _ in range(self.refine):
            out, black, xy = net(in_x)
            if out.numel() != S * h * w or black.numel() != S * h * w or tuple(xy.shape) != (S, h, w, 2):
                raise ValueError('net must return out [S,h,w,1], black [S,h,w] and xy [S,h,w,2] (S=%d, %dx%d)' % (S, h, w))
            ops.black_accumulate(self.all_black, black)
            ops.stream_push(None, None, 0, out.reshape(S * h, w), black.reshape(S * h, w), refeed_into=in_x.view(1, S * h, w, nch))
        ops.streams_push(self.frames, self.masks, self.heads_dev, out.reshape(S, h, w), black.reshape(S, h, w))
        return xy

    def step(self, raw_bgr, net):
        """One frame of every slot from raw_bgr [S,H,W,3] uint8 on the device ([S,3H/2,W] for a YUV 4:2:0 batch): cvt_img2train,
        advance(), cv2_resize of the colour frames to out_size (none at out_size == src_size) and warpRevBundle2 with the last xy.
        Returns the stabilised colour frames [S,OH,OW,3] uint8 BGR, or [S,3OH/2,OW] YUV 4:2:0 for out_format 'nv12' / 'i420'
        (self.colour, overwritten by the next step)."""
        raw = ops._chk(raw_bgr, 'raw_bgr', torch.uint8)
        if tuple(raw.shape) != (self.S,) + self.frame_shape:
            raise ValueError('raw_bgr must be %s uint8 (got %s)' % ([self.S] + list(self.frame_shape), tuple(raw.shape)))
        h, w = self.height, self.width
        if self.src_format == 'bgr':
            cur = ops.cvt_img2train_u8_batch(raw, self._cvt, h, w, out=self.cur, tmp=self.cvt_tmp)
        else:
            cur = ops.cvt_img2train_yuv420_batch(raw, self.src_format, self._cvt, h, w, out=self.cur, tmp=self.cvt_tmp)
        xy = self.advance(cur, net)
        if self._direct:
            return ops.remap_bundle_frame(raw, self.src_format, xy, out=self.colour, workspace=self.remap_ws, out_format=self.out_format)
        oh, ow = self.out_size
        if self.src_format == 'bgr':
            small = ops.resize_linear_u8_batch(raw, self._resize[0], self._resize[1], oh, ow, out=self.small)
        else:
            small = ops.resize_linear_yuv420_batch(raw, self.src_format, self._resize[0], self._resize[1], oh, ow, out=self.small)
        return self._warp_small(small, xy)

    def _warp_small(self, small, xy):
        """warpRevBundle2 of the resized colour frames small [S,OH,OW,3] into self.colour"""
        if self.out_size == (self.height, self.width) and self.out_format == 'bgr':
            return ops.remap_bundle_u8(small, xy, out=self.colour, workspace=self.remap_ws)
        return ops.remap_bundle_frame(small, 'bgr', xy, out=self.colour, workspace=self.remap_ws, out_format=self.out_format)

    def capture(self, raw_bgr, net, upload_from=None, download_to=None):
        """Records step(raw_bgr, net) as a CUDA graph and returns it: graph.replay() runs one step on whatever raw_bgr holds and
        leaves the frames in self.colour.  upload_from / download_to: optional host buffers (raw_bgr's shape / self.colour's:
        [S,H,W,3] or, for a YUV 4:2:0 batch, [S,3H/2,W] / [S,OH,OW,3] or, for a YUV 4:2:0 output, [S,3OH/2,OW]; uint8, pinned)
        copied into raw_bgr before and out of self.colour after the step, inside the graph.  One eager step runs first
        on a side stream as a warm-up (a network may select algorithms or allocate on its first call); the state it changed
        is restored, so capturing leaves every slot as it was."""
        if download_to is not None and tuple(download_to.shape) != tuple(self.colour.shape):
            raise ValueError('download_to must be %s (got %s)' % (list(self.colour.shape), tuple(download_to.shape)))
        upload = None if upload_from is None else lambda: raw_bgr.copy_(upload_from, non_blocking=True)
        download = None if download_to is None else lambda: download_to.copy_(self.colour, non_blocking=True)
        return self._capture(raw_bgr, net, upload, download)

    def _capture(self, raw_bgr, net, upload, download):
        """capture() with the transfers as callables (or None) recorded before and after the step"""
        return self._record(lambda: self.step(raw_bgr, net), upload, download)

    def _record(self, run, upload, download, warm_upload=False):
        """run() (one step) as a CUDA graph with upload / download (callables or None) recorded before and after it, after one
        eager warm-up run on a side stream (with the upload first when warm_upload) whose state changes are undone"""
        state = (self.frames, self.masks, self.heads_dev, self.all_black)
        snap = [t.clone() for t in state]
        side = torch.cuda.Stream(device=self.frames.device)
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            if warm_upload and upload is not None:
                upload()
            run()
        torch.cuda.current_stream().wait_stream(side)
        for t, v in zip(state, snap):
            t.copy_(v)
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            if upload is not None:
                upload()
            run()
            if download is not None:
                download()
        return graph

    def _check_table(self, table, fmt, size, name):
        if not isinstance(table, PlaneTable):
            raise ValueError('%s must be a PlaneTable' % name)
        if (table.S, table.fmt, table.size) != (self.S, fmt, tuple(size)):
            raise ValueError('%s must describe %d %s frames of %dx%d (got %d %s frames of %dx%d)'
                             % ((name, self.S, fmt) + tuple(size) + (table.S, table.fmt) + table.size))
        if table.device.device != self.frames.device:
            raise ValueError('%s lives on %s, the batch on %s' % (name, table.device.device, self.frames.device))

    def _packed_table(self, attr, buf, fmt):
        """the table of one of the batch's own buffers (self.colour / self.small), built and uploaded once"""
        t = getattr(self, attr, None)
        if t is None:
            t = PlaneTable.packed(buf, fmt)
            setattr(self, attr, t)
        return t

    def step_planes(self, src_table, net, dst_table=None):
        """step() on frames that lie wherever the decoder put them: src_table (a PlaneTable of src_format and src_size, uploaded)
        gives each slot's source planes and pitches, and the stabilised frames are written into the surfaces of dst_table (a
        PlaneTable of out_format and out_size), or into self.colour when dst_table is None.  Every slot's frames and rings are
        those of step() on the packed frames; join, leave, the crop and the rings behave as in step().  At out_size == src_size
        the warp reads the source planes itself, otherwise cv2.resize writes them into self.small first.
        A slot whose source entry is empty (PlaneTable.clear) is idle in the front end: its network frame keeps what it held; with
        out_size == src_size the warp also writes nothing for it, and with a resize its destination is only left alone when its
        dst_table entry is cleared as well.  Returns self.colour (dst_table None) or dst_table."""
        self._check_table(src_table, self.src_format, self.src_size, 'src_table')
        dst = self._packed_table('_colour_table', self.colour, self.out_format) if dst_table is None else dst_table
        self._check_table(dst, self.out_format, self.out_size, 'dst_table')
        h, w = self.height, self.width
        cur = ops.cvt_img2train_planes(src_table.device, self.src_format, self.src_size, self._cvt, h, w, out=self.cur, tmp=self.cvt_tmp)
        xy = self.advance(cur, net)
        if self._direct:
            ops.remap_bundle_frame_planes(src_table.device, self.src_format, xy, self.src_size, dst.device, self.out_format,
                                          workspace=self.remap_ws)
        else:
            oh, ow = self.out_size
            ops.resize_linear_planes(src_table.device, self.src_format, self.src_size, self._resize[0], self._resize[1], oh, ow,
                                     out=self.small)
            ops.remap_bundle_frame_planes(self._packed_table('_small_table', self.small, 'bgr').device, 'bgr', xy, self.out_size,
                                          dst.device, self.out_format, workspace=self.remap_ws)
        return self.colour if dst_table is None else dst_table

    def capture_planes(self, src_table, net, dst_table=None):
        """Records step_planes(src_table, net, dst_table) as a CUDA graph with the uploads of both tables at its head: edit the
        tables' host mirrors (set / clear) between replays and each replay reads the surfaces they name then -- one graph follows a
        decoder's rotating surface pool and an encoder's input surfaces.  A replay's upload reads the mirror when the replay runs,
        so do not edit a mirror before the replay that reads it has copied it: wait for the table's event (table.uploaded.
        synchronize(), recorded right after the copy inside the graph), or alternate two tables, each captured in its own graph.
        join / leave between replays act as with capture()."""
        self._check_table(src_table, self.src_format, self.src_size, 'src_table')
        return self._record_planes(src_table, net, dst_table)

    def _record_planes(self, src_table, net, dst_table):
        """step_planes(src_table, net, dst_table) as a CUDA graph with the uploads of the tables at its head"""
        tables = (src_table,) if dst_table is None else (src_table, dst_table)

        def upload():
            for t in tables:
                t.upload()
        return self._record(lambda: self.step_planes(src_table, net, dst_table), upload, None, warm_upload=True)


class MixedStreamBatch(StreamBatch):
    """A StreamBatch whose slots carry videos of different source sizes, up to the capacity max_src_size = (H, W).  Every size
    is resized to the same network frame, so everything after the front end is the StreamBatch's; the two kernels that read the
    source frame take each slot's size and tables from device memory.  Every slot is bit-identical to its own pipeline at its
    own size (and so to a StreamBatch of that size).

        mb = MixedStreamBatch(4, (1080, 1920))          # capacity 1080p, BGR
        pool = torch.empty(mb.pool_shape, dtype=torch.uint8, device='cuda')
        mb.join(0, first_720p)                          # [720,1280,3] uint8: slot 0 is now a 720p video
        mb.join(1, first_1080p)
        for ...:
            mb.slot_frame(pool, 0).copy_(next_720p)     # each slot's frame goes to the start of its region of the pool
            mb.slot_frame(pool, 1).copy_(next_1080p)
            colour = mb.step(pool, net)                 # [4,288,512,3] uint8

    pool: [S, frame_bytes(max_src_size)] uint8 (frame_bytes = 3*H*W for BGR, 3H/2*W for YUV 4:2:0); slot s's frame lies contiguous
    at the start of pool[s], BGR [H_s,W_s,3] or YUV [3H_s/2,W_s].  slot_frame() gives that view of any pool-shaped buffer (device
    or pinned host).  capture(pool, net, upload_from=, download_to=) is StreamBatch.capture: the upload inside the graph copies
    the whole pool, capacity bytes per slot whatever the slots' sizes.  capture(..., exact_bytes=True) records the transfers as
    one kernel each (ops.copy_slots_mixed) that moves every slot's frame at its size at replay and nothing else: the bytes past
    each slot's frame, and idle slots' rows, are not copied in either direction.  A slot can join again at another size
    between replays of a captured graph: join writes the slot's size and tables with stream-ordered device copies, and the graph reads them.
    Slots that never joined are idle: the front end writes nothing for them and the network sees zero frames.  A slot that left
    keeps its size and runs on whatever its region holds, as in StreamBatch.

    out_size sets the size of the stabilised colour frames, and out_format ('bgr', 'nv12', 'i420') their format, as in
    StreamBatch:
      None       the network's (height, width) for every slot: self.colour is [S,h,w,3] (or [S,3h/2,w]).
      (OH, OW)   one size for every slot: each slot is resized to it with its own tables and warped; self.colour is [S,OH,OW,3]
                 (or [S,3OH/2,OW]), each slot bit-identical to StreamBatch(1, (H_s, W_s), out_size=(OH, OW)).
      'source'   each slot at its own size: the warp reads the pool itself and writes the output pool self.colour, of shape
                 out_pool_shape = [S, dst_frame_bytes(capacity)] (3*H*W for BGR, 3H/2*W for YUV 4:2:0), slot s's frame at the
                 start of its row; slot_output() gives that view of any buffer of that shape (device, or a pinned host buffer
                 that capture(download_to=) fills -- the download copies the whole output pool, or with exact_bytes=True
                 each slot's frame).  Each slot is bit-identical
                 to StreamBatch(1, (H_s, W_s), out_size=(H_s, W_s)).  With a YUV out_format, join() refuses a frame of odd size.
    leave() gives the rectangle on the network's lattice; in output pixels it is scale_rect(mb.leave(s), (h, w),
    mb.slot_sizes[s]) for 'source', or scale_rect(mb.leave(s), (h, w), (OH, OW)) for a common size."""

    def __init__(self, S, max_src_size, height=288, width=512, depth=32, taps=(1, 2, 4, 8, 16, 32), use_masks=True, crop_rate=1,
                 refine=1, device='cuda', src_format='bgr', out_size=None, out_format='bgr'):
        if isinstance(out_size, str) and out_size != 'source':
            raise ValueError("out_size must be None, (OH, OW) or 'source' (got %r)" % (out_size,))
        self._source_out = out_size == 'source'
        # 'source': StreamBatch sizes its checks and its result at the capacity, which holds the output pool's bytes
        super().__init__(S, max_src_size, height, width, depth, taps, use_masks, crop_rate, refine, device, src_format,
                         out_size=tuple(max_src_size) if self._source_out else out_size, out_format=out_format)
        if self._source_out:
            self.out_size = 'source'
            self.colour = self.colour.view(self.S, -1)
            self.out_pool_shape = tuple(self.colour.shape)
            # the output pool's planes for step_planes, every slot idle until it joins (join writes its entry on the device)
            self._colour_mtable = MixedPlaneTable.pool(self.colour, self.out_format, self.src_size, [None] * self.S)
        elif self._direct:
            # a common output size equal to the capacity: the slots still go through the per-slot resize
            self._direct = False
            self.small = torch.zeros((self.S,) + self.out_size + (3,), device=self.frames.device, dtype=torch.uint8)

    def _init_front_end(self, dev):
        """per-slot sizes and tables, all zero (every slot idle) until a slot joins"""
        (H, W), h, w = self.src_size, self.height, self.width
        rh, rw, _, _ = _resample_size(h, w, self.crop_rate)
        i32 = dict(device=dev, dtype=torch.int32)
        self.pool_shape = (self.S, int(np.prod(self.frame_shape)))
        self.sizes = torch.zeros((self.S, 2), **i32)
        self.tables = (torch.zeros((self.S, w, _pil_ksize(W, rw)), **i32), torch.zeros((self.S, w), **i32),
                       torch.zeros((self.S, w), **i32), torch.zeros((self.S, h, _pil_ksize(H, rh)), **i32),
                       torch.zeros((self.S, h), **i32), torch.zeros((self.S, h), **i32))
        if self._source_out:
            self.xtab = self.ytab = None                    # the warp reads the pool: no resize
        else:
            oh, ow = self.out_size
            self.xtab, self.ytab = torch.zeros((self.S, ow, 4), **i32), torch.zeros((self.S, oh, 4), **i32)
        self.slot_sizes = [None] * self.S
        self.cur.zero_()
        if self.small is not None:
            self.small.zero_()

    def _frame_size(self, f):
        if not isinstance(f, torch.Tensor) or f.dtype != torch.uint8:
            raise ValueError('a source frame must be a uint8 array or tensor (got %s)' % (getattr(f, 'dtype', type(f)),))
        if self.src_format == 'bgr':
            if f.dim() != 3 or f.shape[2] != 3:
                raise ValueError('a BGR frame must be [H,W,3] (got %s)' % (tuple(f.shape),))
            H, W = int(f.shape[0]), int(f.shape[1])
        else:
            if f.dim() != 2 or f.shape[0] % 3 or f.shape[1] % 2:
                raise ValueError('a %s frame must be [3H/2,W] with H and W even (got %s)' % (self.src_format, tuple(f.shape)))
            H, W = int(f.shape[0]) // 3 * 2, int(f.shape[1])
        if not (0 < H <= self.src_size[0] and 0 < W <= self.src_size[1]):
            raise ValueError('a %dx%d frame does not fit the capacity %dx%d' % (H, W, self.src_size[0], self.src_size[1]))
        return H, W

    def _frame_shape_of(self, H, W):
        return (H, W, 3) if self.src_format == 'bgr' else (H * 3 // 2, W)

    def join(self, slot, first):
        """A new video starts in `slot` at the size of its first frame (BGR [H,W,3] or YUV 4:2:0 [3H/2,W] uint8, up to the
        capacity): the slot's size and tables are written, then everything StreamBatch.join does, with the first frame converted
        by cvt_img2train at its own size."""
        s = self._slot(slot)
        f = torch.as_tensor(np.ascontiguousarray(first)) if isinstance(first, np.ndarray) else first
        H, W = self._frame_size(f)
        if self._source_out and self.out_format != 'bgr' and (H % 2 or W % 2):
            raise ValueError('a %s output needs an even size (got a %dx%d frame)' % (self.out_format, H, W))
        # host-built tables (about 15 ms at 2160x3840), copied into the slot's rows on the current stream; nothing is kept per size
        tabs = mixed_slot_tables((H, W), self.src_size, self.height, self.width, self.crop_rate,
                                 out_size=None if self._source_out else self.out_size)
        dsts = (self.sizes,) + self.tables + (() if self._source_out else (self.xtab, self.ytab))
        for dst, src in zip(dsts, (np.array([H, W], np.int32),) + tabs):
            dst[s].copy_(torch.as_tensor(src))
        self.slot_sizes[s] = (H, W)
        if self._source_out:
            # the output pool's entry at the new size, by a stream-ordered copy from pageable memory (as sizes): no wait on a replay
            ct = self._colour_mtable
            ct.set(s, _packed_planes(self.out_format, self.colour[s].data_ptr(), H, W), (H, W))
            ct.device[s].copy_(torch.as_tensor(ct.host[s].numpy().copy()))
        cur = cvt_img2train(f.to(self.frames.device), self.crop_rate, self.height, self.width, src_format=self.src_format)
        super().join(s, cur.reshape(self.height, self.width))

    def slot_frame(self, buf, slot):
        """The view of slot `slot`'s current frame inside a pool-shaped buffer buf [S, frame_bytes(capacity)] uint8 (the pool on
        the device, or a pinned host buffer that is uploaded into it): BGR [H_s,W_s,3] or YUV [3H_s/2,W_s] at the slot's size."""
        s = self._slot(slot)
        if self.slot_sizes[s] is None:
            raise ValueError('slot %d carries no video' % s)
        if tuple(buf.shape) != self.pool_shape or buf.dtype != torch.uint8:
            raise ValueError('buf must be %s uint8 (got %s %s)' % (list(self.pool_shape), tuple(buf.shape), buf.dtype))
        shape = self._frame_shape_of(*self.slot_sizes[s])
        return buf[s, :int(np.prod(shape))].view(shape)

    def slot_output(self, buf, slot):
        """out_size='source': the view of slot `slot`'s stabilised frame inside a buffer buf of out_pool_shape uint8 (self.colour,
        or a pinned host buffer it is downloaded into): BGR [H_s,W_s,3] or YUV 4:2:0 [3H_s/2,W_s] at the slot's size."""
        if not self._source_out:
            raise ValueError("slot_output needs out_size='source' (the output is self.colour[slot])")
        s = self._slot(slot)
        if self.slot_sizes[s] is None:
            raise ValueError('slot %d carries no video' % s)
        if tuple(buf.shape) != self.out_pool_shape or buf.dtype != torch.uint8:
            raise ValueError('buf must be %s uint8 (got %s %s)' % (list(self.out_pool_shape), tuple(buf.shape), buf.dtype))
        H, W = self.slot_sizes[s]
        shape = (H, W, 3) if self.out_format == 'bgr' else (H * 3 // 2, W)
        return buf[s, :int(np.prod(shape))].view(shape)

    def step(self, pool, net):
        """One frame of every slot from pool [S, frame_bytes(capacity)] uint8 on the device: cvt_img2train and cv2.resize of each
        slot at its own size (no resize for out_size='source'), and the StreamBatch step around them.  Returns the stabilised
        colour frames (self.colour, overwritten by the next step): [S,OH,OW,3] uint8 BGR, or [S,3OH/2,OW] YUV 4:2:0 for out_format
        'nv12' / 'i420', with (OH, OW) the network's size by default; the output pool out_pool_shape for out_size='source'."""
        if not isinstance(pool, torch.Tensor) or pool.dtype != torch.uint8 or tuple(pool.shape) != self.pool_shape:
            raise ValueError('pool must be a %s uint8 tensor (got %s %s)' % (list(self.pool_shape), tuple(getattr(pool, 'shape', ())),
                                                                           getattr(pool, 'dtype', type(pool))))
        pool = ops._chk(pool, 'pool', torch.uint8).view((self.S,) + self.frame_shape)
        h, w = self.height, self.width
        cur = ops.cvt_img2train_mixed(pool, self.src_format, self.sizes, self.tables, h, w, out=self.cur, tmp=self.cvt_tmp)
        xy = self.advance(cur, net)
        if self._source_out:
            return ops.remap_bundle_frame_mixed(pool, self.src_format, self.sizes, xy, self.out_format, out=self.colour,
                                                workspace=self.remap_ws)
        oh, ow = self.out_size
        small = ops.resize_linear_mixed(pool, self.src_format, self.sizes, self.xtab, self.ytab, oh, ow, out=self.small)
        return self._warp_small(small, xy)

    def _check_mixed_table(self, table, fmt, name):
        if not isinstance(table, MixedPlaneTable):
            raise TypeError('%s must be a MixedPlaneTable: a PlaneTable describes frames of one size (StreamBatch.step_planes)' % name)
        if (table.S, table.fmt, table.capacity) != (self.S, fmt, self.src_size):
            raise ValueError('%s must describe %d %s frames of capacity %dx%d (got %d %s frames of capacity %dx%d)'
                             % ((name, self.S, fmt) + self.src_size + (table.S, table.fmt) + table.capacity))
        if table.device.device != self.frames.device:
            raise ValueError('%s lives on %s, the batch on %s' % (name, table.device.device, self.frames.device))

    def step_planes(self, src_table, net, dst_table=None):
        """step() on frames that lie wherever the decoder put them: src_table is a MixedPlaneTable of src_format and the batch's
        capacity (uploaded), whose entry s names slot s's surface at the slot's current size; a uniform PlaneTable is a TypeError.
        Every slot's frames and rings are those of step() on the packed pool; join, leave, the crop and the rings are step()'s.
          'source'    the warp reads the source planes and writes each slot at its own size into dst_table, a MixedPlaneTable of
                      out_format and the capacity whose entries carry the slots' sizes, or into the output pool self.colour
                      (dst_table None: the batch keeps that pool's table, and join updates a slot's entry on the device).
          None / (OH, OW)  each slot is resized into self.small at its own size, then warped into dst_table, a PlaneTable of
                      out_format and out_size, or into self.colour.
        A slot is idle in the front end when its source entry is cleared, or names another size than the slot's (after a join at
        a new size, until the entry is set at that size): its network frame keeps what it held.  With 'source' the warp then
        writes nothing for it either, and a destination entry of another size idles it too; through the resize its destination
        is left alone only when its dst_table entry is cleared as well.  Returns self.colour (dst_table None) or dst_table."""
        self._check_mixed_table(src_table, self.src_format, 'src_table')
        h, w = self.height, self.width
        if self._source_out:
            dst = self._colour_mtable if dst_table is None else dst_table
            self._check_mixed_table(dst, self.out_format, 'dst_table')
        else:
            dst = self._packed_table('_colour_table', self.colour, self.out_format) if dst_table is None else dst_table
            self._check_table(dst, self.out_format, self.out_size, 'dst_table')
        cur = ops.cvt_img2train_mixed_planes(src_table.device, self.src_format, self.sizes, self.src_size, self.tables, h, w,
                                             out=self.cur, tmp=self.cvt_tmp)
        xy = self.advance(cur, net)
        if self._source_out:
            ops.remap_bundle_frame_mixed_planes(src_table.device, self.src_format, self.sizes, xy, self.src_size, dst.device,
                                                self.out_format, workspace=self.remap_ws)
        else:
            oh, ow = self.out_size
            ops.resize_linear_mixed_planes(src_table.device, self.src_format, self.sizes, self.src_size, self.xtab, self.ytab, oh, ow,
                                           out=self.small)
            ops.remap_bundle_frame_planes(self._packed_table('_small_table', self.small, 'bgr').device, 'bgr', xy, self.out_size,
                                          dst.device, self.out_format, workspace=self.remap_ws)
        return self.colour if dst_table is None else dst_table

    def capture_planes(self, src_table, net, dst_table=None):
        """StreamBatch.capture_planes for a MixedPlaneTable: step_planes(src_table, net, dst_table) as a CUDA graph with the uploads
        of both tables at its head.  A slot may join again at another size between replays: it is idle until its entries are set
        at the new size and uploaded by the next replay (the batch's own output pool table follows the join by itself)."""
        self._check_mixed_table(src_table, self.src_format, 'src_table')
        return self._record_planes(src_table, net, dst_table)

    def capture(self, pool, net, upload_from=None, download_to=None, exact_bytes=False):
        """StreamBatch.capture of step(pool, net).  exact_bytes=False copies the whole pool up (and, for out_size='source', the
        whole output pool down).  exact_bytes=True records the transfers as ops.copy_slots_mixed, which moves each slot's frame at
        the size it has at replay and nothing else: upload_from (pool_shape) and download_to (out_pool_shape for 'source') must
        then be pinned host tensors.  The bytes past each slot's frame, and idle slots' rows, are not copied in either direction:
        the device pool and the host output pool keep what they held there.  A uniform output ([S,OH,OW,3] or [S,3OH/2,OW]) is
        downloaded whole either way: it has no bytes but the frames."""
        if not exact_bytes:
            return super().capture(pool, net, upload_from, download_to)
        for name, t, shape in (('upload_from', upload_from, self.pool_shape),
                               ('download_to', download_to, tuple(self.colour.shape))):
            if t is None:
                continue
            if not isinstance(t, torch.Tensor) or t.is_cuda or not t.is_pinned():
                raise ValueError('%s must be a pinned host tensor with exact_bytes=True' % name)
            if tuple(t.shape) != shape:
                raise ValueError('%s must be %s (got %s)' % (name, list(shape), tuple(t.shape)))
        upload = download = None
        if upload_from is not None:
            src_view = (self.S,) + self.frame_shape
            def upload():
                ops.copy_slots_mixed(upload_from.view(src_view), pool.view(src_view), self.src_format, self.sizes)
        if download_to is not None:
            if self._source_out:
                H, W = self.src_size                        # the output pool's capacity
                out_view = (self.S, H, W, 3) if self.out_format == 'bgr' else (self.S, H * 3 // 2, W)
                def download():
                    ops.copy_slots_mixed(self.colour.view(out_view), download_to.view(out_view), self.out_format, self.sizes)
            else:
                def download():
                    download_to.copy_(self.colour, non_blocking=True)
        return self._capture(pool, net, upload, download)

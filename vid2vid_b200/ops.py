"""Stand-alone operators: thin Python wrappers over group (1) of the C ABI, mirroring the reference's
operator surface (same class names / argument meaning / output-ownership rules):

  Correlation / Resample2d / ChannelNorm  <- models/flownet2_pytorch/networks/*_package/*.py
  resample(image, flow)                   <- BaseModel.resample (models/base_model.py:189-196)
  onehot_edges / avgpool3s2 / fg_mask     <- Vid2VidModelG.encode_input / build_pyr / compute_mask
  face_window / crop_concat               <- Vid2VidModelD.get_face_region + the face crop (--add_face_disc)

CUDA fp32 contiguous tensors only; errors from the library raise RuntimeError (the reference's
wrapper raises via AT_ERROR, correlation_cuda.cc:81-83).  No CPU fallback.
"""
import ctypes as C

import torch
import torch.nn as nn

from . import _lib as L


def _chk(*ts):
    for t in ts:
        if t is None:
            continue
        if not t.is_cuda or t.dtype != torch.float32:
            raise RuntimeError('vid2vid_b200 ops need CUDA float32 tensors (no CPU fallback)')
        if not t.is_contiguous():
            raise RuntimeError('vid2vid_b200 ops need contiguous tensors')   # resample2d.py:9-10, channelnorm.py:9


def _ck(rc):
    L.check(rc)
    L.LAUNCHES[0] += 1


def _on(t):
    """Context for a launch on tensor t's device (correlation.py:21 `with torch.cuda.device_of(input1)`); pair it with
    _st(t), the caller's current stream on THAT device."""
    return torch.cuda.device_of(t)


def _st(t):
    return C.c_void_p(torch.cuda.current_stream(t.device).cuda_stream)


def _p(t):
    return C.c_void_p(t.data_ptr()) if t is not None else C.c_void_p(None)


def correlation(input1, input2, pad_size=20, kernel_size=1, max_displacement=20, stride1=1, stride2=2,
                corr_multiply=1):
    """CorrelationFunction.forward (correlation.py:18-30)."""
    _chk(input1, input2)
    n, c, h, w = input1.shape
    oc, oh, ow = C.c_int(), C.c_int(), C.c_int()
    L.check(L.lib().v2v_correlation_out_shape(h, w, pad_size, kernel_size, max_displacement, stride1, stride2,
                                              C.byref(oc), C.byref(oh), C.byref(ow)))
    out = torch.empty((n, oc.value, oh.value, ow.value), device=input1.device, dtype=torch.float32)
    with torch.cuda.device_of(input1):
        _ck(L.lib().v2v_correlation_forward(_p(input1), _p(input2), _p(out), n, c, h, w, pad_size, kernel_size,
                                                max_displacement, stride1, stride2, corr_multiply, _st(input1)))
    return out


class Correlation(nn.Module):
    """correlation.py:47-61."""

    def __init__(self, pad_size=0, kernel_size=0, max_displacement=0, stride1=1, stride2=2, corr_multiply=1):
        super().__init__()
        self.pad_size, self.kernel_size, self.max_displacement = pad_size, kernel_size, max_displacement
        self.stride1, self.stride2, self.corr_multiply = stride1, stride2, corr_multiply

    def forward(self, input1, input2):
        return correlation(input1.contiguous(), input2.contiguous(), self.pad_size, self.kernel_size,
                           self.max_displacement, self.stride1, self.stride2, self.corr_multiply)


def resample2d(input1, input2, kernel_size=1):
    """Resample2dFunction.forward (resample2d.py:8-21)."""
    _chk(input1, input2)
    _, d, ih, iw = input1.shape
    b, _, h, w = input2.shape
    out = torch.empty((b, d, h, w), device=input1.device, dtype=torch.float32)
    with torch.cuda.device_of(input1):
        _ck(L.lib().v2v_resample2d_forward(_p(input1), _p(input2), _p(out), b, d, h, w, ih, iw, kernel_size, _st(input1)))
    return out


class Resample2d(nn.Module):
    """resample2d.py:38-46."""

    def __init__(self, kernel_size=1):
        super().__init__()
        self.kernel_size = kernel_size

    def forward(self, input1, input2):
        return resample2d(input1.contiguous(), input2.contiguous(), self.kernel_size)


def channelnorm(input1, norm_deg=2):
    """ChannelNormFunction.forward (channelnorm.py:7-17)."""
    _chk(input1)
    b, c, h, w = input1.shape
    out = torch.empty((b, 1, h, w), device=input1.device, dtype=torch.float32)
    with torch.cuda.device_of(input1):
        _ck(L.lib().v2v_channelnorm_forward(_p(input1), _p(out), b, c, h, w, norm_deg, _st(input1)))
    return out


class ChannelNorm(nn.Module):
    """channelnorm.py:31-38."""

    def __init__(self, norm_deg=2):
        super().__init__()
        self.norm_deg = norm_deg

    def forward(self, input1):
        return channelnorm(input1.contiguous(), self.norm_deg)


def _resample_fwd(image, flow, align_corners):
    image, flow = image.contiguous(), flow.contiguous()
    _chk(image, flow)
    b, c, h, w = image.shape
    out = torch.empty_like(image)
    with _on(image):
        _ck(L.lib().v2v_resample_forward(_p(image), _p(flow), _p(out), b, c, h, w, int(align_corners), _st(image)))
    return out


class ResampleFunction(torch.autograd.Function):
    """resample with gradients wrt image and flow (the warp losses differentiate through it, vid2vid_model_D.py:123)."""

    @staticmethod
    def forward(ctx, image, flow, align_corners):
        image, flow = image.detach().contiguous(), flow.detach().contiguous()
        ctx.save_for_backward(image, flow)
        ctx.ac = int(align_corners)
        return _resample_fwd(image, flow, align_corners)

    @staticmethod
    def backward(ctx, g):
        image, flow = ctx.saved_tensors
        b, c, h, w = image.shape
        g = g.contiguous()
        gi = torch.zeros_like(image) if ctx.needs_input_grad[0] else None
        gf = torch.empty_like(flow) if ctx.needs_input_grad[1] else None
        _ck(L.lib().v2v_resample_backward(_p(image), _p(flow), _p(g), _p(gi), _p(gf), b, c, h, w, ctx.ac, L.current_stream_ptr()))
        return gi, gf, None


def resample(image, flow, align_corners=False):
    """BaseModel.resample / BaseNetwork.resample (base_model.py:189-196, networks.py:108-115)."""
    if torch.is_grad_enabled() and (image.requires_grad or flow.requires_grad):
        return ResampleFunction.apply(image, flow, align_corners)
    return _resample_fwd(image, flow, align_corners)


def onehot_edges(label_map, inst_map, label_nc, use_instance):
    """encode_input + get_edges (vid2vid_model_G.py:86-112, base_model.py:146-152).
    label_map / inst_map: (b, t, 1, H, W) float ids -> (b, t, label_nc [+1], H, W)."""
    label_map = label_map.contiguous()
    inst = inst_map.contiguous() if use_instance else None
    _chk(label_map, inst)
    b, t, _, h, w = label_map.shape
    out = torch.empty((b, t, label_nc + int(bool(use_instance)), h, w), device=label_map.device, dtype=torch.float32)
    with _on(label_map):
        _ck(L.lib().v2v_onehot_edges(_p(label_map), _p(inst), _p(out), b * t, label_nc, int(bool(use_instance)), h, w, _st(label_map)))
    return out


class AvgPool3s2Function(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x):
        ctx.shape = x.shape
        return _avgpool3s2_fwd(x.detach())

    @staticmethod
    def backward(ctx, g):
        h, w = ctx.shape[-2:]
        g = g.contiguous()
        gin = torch.empty(ctx.shape, device=g.device, dtype=torch.float32)
        _ck(L.lib().v2v_avgpool3s2_backward(_p(g), _p(gin), gin.numel() // (h * w), h, w, L.current_stream_ptr()))
        return gin


def avgpool3s2(x):
    """AvgPool2d(3, stride=2, padding=1, count_include_pad=False) over the last two dims (autograd-aware)."""
    if torch.is_grad_enabled() and x.requires_grad:
        return AvgPool3s2Function.apply(x)
    return _avgpool3s2_fwd(x)


def _avgpool3s2_fwd(x):
    x = x.contiguous()
    _chk(x)
    h, w = x.shape[-2:]
    planes = x.numel() // (h * w)
    out = torch.empty(tuple(x.shape[:-2]) + ((h - 1) // 2 + 1, (w - 1) // 2 + 1), device=x.device, dtype=torch.float32)
    with _on(x):
        _ck(L.lib().v2v_avgpool3s2(_p(x), _p(out), planes, h, w, _st(x)))
    return out


def fg_mask(real_As, ts, fg_labels):
    """compute_mask (vid2vid_model_G.py:322-330): (b, T, C, h, w) -> (b, 1, h, w)."""
    real_As = real_As.contiguous()
    _chk(real_As)
    b, T, c, h, w = real_As.shape
    out = torch.empty((b, 1, h, w), device=real_As.device, dtype=torch.float32)
    arr = (C.c_int * len(fg_labels))(*fg_labels)
    with _on(real_As):
        _ck(L.lib().v2v_fg_mask(_p(real_As), _p(out), b, T, c, h, w, ts, arr, len(fg_labels), _st(real_As)))
    return out


# ------------------------------------------------------------------------------------------------ training losses
def _scalar_ws(dev):
    return torch.zeros(1, device=dev, dtype=torch.float64), torch.empty(1, device=dev, dtype=torch.float32)


class L1LossFunction(torch.autograd.Function):
    """mean |a*m - b*m| (MaskedL1Loss, networks.py:804-812) / mean |a - b| (nn.L1Loss) with m = None; b may be None (= 0)."""

    @staticmethod
    def forward(ctx, a, b, mask):
        a = a.detach().contiguous()
        b = b.detach().contiguous() if b is not None else None
        mask = mask.detach().contiguous() if mask is not None else None
        _chk(a, b, mask)
        a4 = a if a.dim() == 4 else a.reshape(-1, a.shape[-3], a.shape[-2], a.shape[-1])
        ctx.dims = a4.shape
        ws, out = _scalar_ws(a.device)
        n, c, h, w = a4.shape
        _ck(L.lib().v2v_l1_loss_forward(_p(a), _p(b), _p(mask), n, c, h, w, C.c_void_p(ws.data_ptr()), _p(out), L.current_stream_ptr()))
        ctx.save_for_backward(a, b, mask)
        return out.reshape(())

    @staticmethod
    def backward(ctx, g):
        a, b, mask = ctx.saved_tensors
        n, c, h, w = ctx.dims
        g = g.reshape(1).contiguous().float()
        ga = torch.empty_like(a) if ctx.needs_input_grad[0] else None
        gb = torch.empty_like(b) if (b is not None and ctx.needs_input_grad[1]) else None
        if ga is None and gb is None:
            return None, None, None
        _ck(L.lib().v2v_l1_loss_backward(_p(a), _p(b), _p(mask), n, c, h, w, _p(g), _p(ga), _p(gb), L.current_stream_ptr()))
        return ga, gb, None


def l1_loss(a, b=None, mask=None):
    return L1LossFunction.apply(a, b, mask)


class MseConstFunction(torch.autograd.Function):
    """mean (x - target)^2 against a constant label: GANLoss with use_lsgan (networks.py:764-774)."""

    @staticmethod
    def forward(ctx, x, target):
        x = x.detach().contiguous()
        _chk(x)
        ctx.t = float(target)
        ws, out = _scalar_ws(x.device)
        _ck(L.lib().v2v_mse_const_forward(_p(x), x.numel(), ctx.t, C.c_void_p(ws.data_ptr()), _p(out), L.current_stream_ptr()))
        ctx.save_for_backward(x)
        return out.reshape(())

    @staticmethod
    def backward(ctx, g):
        (x,) = ctx.saved_tensors
        g = g.reshape(1).contiguous().float()
        gx = torch.empty_like(x)
        _ck(L.lib().v2v_mse_const_backward(_p(x), x.numel(), ctx.t, _p(g), _p(gx), L.current_stream_ptr()))
        return gx, None


def mse_to_const(x, target):
    return MseConstFunction.apply(x, target)


# ------------------------------------------------------------------------------------------------ face discriminator
FACE_WINDOW_WORDS = 10      # {found, ys, ye, xs, xe} + the kernel's accumulators (include/v2v_b200.h)


def face_window_buffer(device):
    """Device buffer for face_window(..., buf=): zeroed once here, left reusable by every call."""
    return torch.zeros(FACE_WINDOW_WORDS, device=device, dtype=torch.int32)


def face_half(fine_size):
    """Half the side of the face window: the reference's fineSize // 32 * 8 (vid2vid_model_D.py:224-225) halved."""
    return fine_size // 32 * 8 // 2


def face_window(real_A, fine_size, openpose_only=False, buf=None):
    """Vid2VidModelD.get_face_region (vid2vid_model_D.py:215-230) on the device: real_A (N, C, H, W) -> int32 tensor
    {found, ys, ye, xs, xe} (all zero when no face pixel exists).  One launch, no host synchronisation; `buf` (from
    face_window_buffer) avoids allocating and zeroing a buffer per call, and the result is a view into it."""
    real_A = real_A.contiguous()
    _chk(real_A)
    n, c, h, w = real_A.shape
    half = face_half(fine_size)
    if c < 3:
        raise ValueError('face_window needs at least 3 input channels, got %d' % c)
    if 2 * half > h or 2 * half > w:
        raise ValueError('face window %dx%d (fineSize %d) is larger than the %dx%d frame' % (2 * half, 2 * half, fine_size, h, w))
    if buf is None:
        buf = face_window_buffer(real_A.device)
    if buf.dtype != torch.int32 or buf.device != real_A.device or buf.numel() != FACE_WINDOW_WORDS or not buf.is_contiguous():
        raise RuntimeError('face_window: buf must be a contiguous int32 tensor of %d words on the input device' % FACE_WINDOW_WORDS)
    with _on(real_A):
        _ck(L.lib().v2v_face_window(_p(real_A), n, c, h, w, int(bool(openpose_only)), half, half, _p(buf), _st(real_A)))
    return buf[:5]


def _chk_win(win, dev):
    if win.dtype != torch.int32 or win.device != dev or win.numel() < 5 or not win.is_contiguous():
        raise RuntimeError('crop window must be a contiguous int32 device tensor {found, ys, ye, xs, xe}')


class CropConcatFunction(torch.autograd.Function):
    """cat(a[:, :, ys:ys+L, xs:xs+L], b[..same..], dim=1) with the window read on the device; the gradient goes to b only
    (a is the condition real_A, which needs none)."""

    @staticmethod
    def forward(ctx, a, b, win, size):
        a, b = a.detach().contiguous(), b.detach().contiguous()
        _chk(a, b)
        _chk_win(win, a.device)
        n, ca, h, w = a.shape
        cb = b.shape[1]
        if b.shape[0] != n or tuple(b.shape[2:]) != (h, w):
            raise RuntimeError('crop_concat: a %s and b %s differ in batch or frame size' % (tuple(a.shape), tuple(b.shape)))
        if size > h or size > w:
            raise ValueError('crop window %dx%d is larger than the %dx%d frame' % (size, size, h, w))
        out = torch.empty((n, ca + cb, size, size), device=a.device, dtype=torch.float32)
        with _on(a):
            _ck(L.lib().v2v_crop_concat_forward(_p(a), ca, _p(b), cb, n, h, w, _p(win), size, size, _p(out), _st(a)))
        ctx.save_for_backward(win)
        ctx.dims = (ca, cb, n, h, w, size)
        return out

    @staticmethod
    def backward(ctx, g):
        if not ctx.needs_input_grad[1]:
            return None, None, None, None
        (win,) = ctx.saved_tensors
        ca, cb, n, h, w, size = ctx.dims
        g = g.contiguous()
        gb = torch.empty((n, cb, h, w), device=g.device, dtype=torch.float32)
        _ck(L.lib().v2v_crop_backward(_p(g), ca, cb, n, h, w, _p(win), size, size, _p(gb), L.current_stream_ptr()))
        return None, gb, None, None


def crop_concat(a, b, win, size):
    """The face discriminator's input (vid2vid_model_D.py:152-153 + compute_loss_D's cat): (N, Ca+Cb, size, size)."""
    return CropConcatFunction.apply(a, b, win, size)

"""Boundary hygiene on the GPU box (SURVEY 8b): the reference-side bindings INTEGRATION.md shows are executed for real.

  b1  the reference-shaped pybind stubs `correlation_cuda.forward(in1, in2, rbot1, rbot2, out, ...) -> 1`,
      `resample2d_cuda.forward`, `channelnorm_cuda.forward` (INTEGRATION.md section 1) bound to libv2v_b200.so, checked
      against the C oracle, and then installed under the UNMODIFIED reference FlowNet2 (copied to oracle/_ref): the
      reference's own Python graph (its nn.Conv2d layers run by PyTorch on the GPU, TF32 off) with our three native ops
      must agree with our FlowNet2 (all convolutions on tcgen05).
  b2  the one-line `networks` swap of INTEGRATION.md section 2: the reference's own Vid2VidModelG (encode_input, build_pyr,
      compute_mask and the frame loop are the reference's code) with vid2vid_b200.networks supplying netG0..2, against our
      Vid2VidModelG on identical weights and inputs.
"""
import ctypes
import fractions
import json
import math
import os
import sys
import types

import numpy as np
import pytest
import torch

from oracle import flowops
from oracle import ref_shim
from vid2vid_b200 import _lib as L

pytestmark = pytest.mark.gpu
# b1's second half and b2 run the reference's own Python modules, which oracle/make_ref.py copies into oracle/_ref/ only where
# the reference tree is present
needs_reference = pytest.mark.skipif(not ref_shim.available(), reason='no reference tree (oracle/make_ref.py)')
GOLD = os.path.join(os.path.dirname(__file__), 'golden')


def _ref_on_path():
    """The reference importable WITHOUT the CPU shims of ref_shim.install() (this process owns a GPU)."""
    if not hasattr(fractions, 'gcd'):
        fractions.gcd = math.gcd
    if ref_shim.REF_ROOT not in sys.path:
        sys.path.insert(0, ref_shim.REF_ROOT)


def _stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def _p(t):
    return ctypes.c_void_p(t.data_ptr())


def _check(rc):
    if rc:
        raise RuntimeError(L.lib().v2v_last_error().decode())      # the reference raises via AT_ERROR


# ---- INTEGRATION.md section 1, verbatim in spirit: reference-shaped entry points over the C ABI
def corr_forward(in1, in2, rbot1, rbot2, out, pad, k, max_disp, s1, s2, corr_type):
    n, c, h, w = in1.size()
    oc, oh, ow = ctypes.c_int(), ctypes.c_int(), ctypes.c_int()
    _check(L.lib().v2v_correlation_out_shape(h, w, pad, k, max_disp, s1, s2, ctypes.byref(oc), ctypes.byref(oh), ctypes.byref(ow)))
    out.resize_(n, oc.value, oh.value, ow.value)                   # correlation_cuda.cc:36-42 resizes the caller's tensor
    _check(L.lib().v2v_correlation_forward(_p(in1), _p(in2), _p(out), n, c, h, w, pad, k, max_disp, s1, s2, corr_type, _stream()))
    return 1


def res_forward(in1, flow, out, kernel_size):
    _, d, ih, iw = in1.size()
    b, _, h, w = flow.size()
    _check(L.lib().v2v_resample2d_forward(_p(in1), _p(flow), _p(out), b, d, h, w, ih, iw, kernel_size, _stream()))
    return 1


def cn_forward(inp, out, norm_deg):
    b, c, h, w = inp.size()
    _check(L.lib().v2v_channelnorm_forward(_p(inp), _p(out), b, c, h, w, norm_deg, _stream()))
    return 1


def test_reference_shaped_operator_stubs_vs_c_oracle():
    g = torch.Generator().manual_seed(2)
    a, b = torch.randn(2, 64, 24, 40, generator=g).cuda(), torch.randn(2, 64, 24, 40, generator=g).cuda()
    out = a.new()
    assert corr_forward(a, b, a.new(), b.new(), out, 20, 1, 20, 1, 2, 1) == 1
    ref = flowops.correlation(a.cpu().numpy(), b.cpu().numpy(), 20, 1, 20, 1, 2)
    assert out.shape == ref.shape and np.abs(out.cpu().numpy() - ref).max() < 1e-5
    img, flow = torch.rand(2, 3, 32, 48, generator=g).cuda(), (torch.randn(2, 2, 32, 48, generator=g) * 3).cuda()
    o = torch.zeros_like(img)
    assert res_forward(img, flow, o, 1) == 1
    assert np.array_equal(o.cpu().numpy(), flowops.resample2d(img.cpu().numpy(), flow.cpu().numpy(), 1))
    n = torch.zeros(2, 1, 32, 48).cuda()
    assert cn_forward(img, n, 2) == 1
    assert np.array_equal(n.cpu().numpy(), flowops.channelnorm(img.cpu().numpy(), 2))
    with pytest.raises(RuntimeError):
        corr_forward(a, b, a.new(), b.new(), a.new(), 20, 3, 20, 1, 2, 1)      # unsupported kernel_size -> exception, like AT_ERROR


@needs_reference
def test_reference_flownet2_with_our_native_ops_vs_our_flownet2():
    _ref_on_path()
    for name, fn in (('correlation_cuda', corr_forward), ('resample2d_cuda', res_forward), ('channelnorm_cuda', cn_forward)):
        m = types.ModuleType(name)
        m.forward = fn
        sys.modules[name] = m
    from models.flownet2_pytorch.networks.correlation_package import correlation as ref_corr   # noqa (reference module)

    def forward(self, input1, input2):      # the legacy autograd Function wrapper does not run on current PyTorch
        out = input1.new()
        sys.modules['correlation_cuda'].forward(input1, input2, input1.new(), input2.new(), out, self.pad_size, self.kernel_size,
                                                self.max_displacement, self.stride1, self.stride2, self.corr_multiply)
        return out
    ref_corr.Correlation.forward = forward
    from models.flownet2_pytorch import models as ref_models   # noqa (reference module)
    from oracle import flownet2_oracle as FO
    from vid2vid_b200 import flownet as FN
    keys = json.load(open(os.path.join(GOLD, 'flownet2_keys.json')))
    sd = FO.det_state_dict(keys, seed=7)
    ref = ref_models.FlowNet2().eval().cuda()
    ref.load_state_dict(sd)
    ours = FN.FlowNet2()
    ours.load_state_dict(sd)
    ours = ours.cuda()
    g = torch.Generator().manual_seed(8)
    base = torch.rand(1, 3, 128, 192, generator=g)
    pair = torch.stack([base, torch.roll(base, shifts=(1, 2), dims=(2, 3)) * 0.9 + 0.05], 2).cuda()
    tf32 = torch.backends.cudnn.allow_tf32
    torch.backends.cudnn.allow_tf32 = False
    try:
        with torch.no_grad():
            r = ref(pair)
            o = ours(pair)
    finally:
        torch.backends.cudnn.allow_tf32 = tf32
    d = (r - o).abs()
    print('reference FlowNet2 (PyTorch convs + our ops) vs ours: max|d|=%.3e mean|d|=%.3e ref max %.3f' % (d.max(), d.mean(), r.abs().max()))
    assert d.max().item() <= 2e-3 * max(1.0, r.abs().max().item())


@needs_reference
def test_reference_model_G_with_networks_swapped_in():
    _ref_on_path()
    import models.vid2vid_model_G as ref_G          # noqa (reference module)
    import vid2vid_b200.networks as our_networks
    from vid2vid_b200.model_g import Vid2VidModelG as OurG
    from vid2vid_b200.utils import det_fill_, make_opt, synth_label_sequence
    opt = make_opt(label_nc=35, use_instance=True, fg=True, fg_labels=[26], n_scales_spatial=2, ngf=32, n_blocks=4, n_downsample_G=2,
                   use_single_G=True, loadSize=512, dataroot='datasets/Cityscapes/', gpu_ids=[0], no_first_img=True)
    old = ref_G.networks
    ref_G.networks = our_networks                    # <- the one-line substitution of INTEGRATION.md section 2
    try:
        class M(ref_G.Vid2VidModelG):
            def load_network(self, *a, **k):
                return None

            def load_single_G(self):
                return None
        ref = M()
        ref.initialize(opt)
        ours = OurG()
        opt2 = make_opt(**vars(opt))
        opt2.use_single_G = False
        ours.initialize(opt2)
        for s in range(2):
            det_fill_(getattr(ref, 'netG%d' % s), seed=40 + s)
            getattr(ours, 'netG%d' % s).load_state_dict(getattr(ref, 'netG%d' % s).state_dict())
            assert isinstance(getattr(ref, 'netG%d' % s), our_networks._Planned)
            # The reference driver knows nothing of our "the one-hot input is exact in bf16" hint (model_g.py sets it on the
            # finest scale and the plan then skips the all-zero lo half: same value, different tiling and summation order).
            # With random weights the recurrence amplifies a 1e-6 difference ~30x per frame (DESIGN.md section 4), so the two
            # drivers are compared on identical kernels: then they must agree bit for bit.
            getattr(ours, 'netG%d' % s).input_exact_bf16 = False
        seq = synth_label_sequence(5, 128, 256, label_nc=35, block=8, seed=3).cuda()
        for t in range(3):
            A = seq[:, t:t + 3]
            fr, _ = ref.inference(A, None, A)
            fo, _ = ours.inference(A, None, A)
            d = (fr - fo).abs()
            print('frame %d reference driver + our networks vs our driver: max|d|=%.3e' % (t, d.max().item()))
            assert torch.isfinite(fr).all() and d.max().item() == 0.0
    finally:
        ref_G.networks = old

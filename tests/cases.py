"""Seeded synthetic cases shared by oracle/make_golden.py (which runs the *reference* on them
and writes tests/golden/<case>.npz) and by the parity tests (which rebuild the same weights
and inputs from the seeds and compare the oracle / the CUDA path with the stored outputs).

Weights never travel: `det_fill_` regenerates them from (seed, parameter name, shape)."""
import glob
import os

import numpy as np
import torch

from vid2vid_b200.utils import make_opt, synth_label_sequence

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden')
GEN_OUT_NAMES = ['img_final', 'flow', 'weight', 'img_raw', 'img_feat', 'flow_feat', 'img_fg_feat']


def load_golden(name):
    """tests/golden/<name>.npz and its continuation parts <name>.1.npz, ... (files stay under 1 MB) as one dict."""
    out = dict(np.load(os.path.join(GOLD, name + '.npz')))
    for path in sorted(glob.glob(os.path.join(GOLD, glob.escape(name) + '.[0-9]*.npz'))):
        out.update(np.load(path))
    return out


def onehot_input(label_nc, h, w, seed, block=4, n_frames=3):
    """(1, n_frames*(label_nc+1), h, w) one-hot + edge input, plus the label sequence."""
    lab = synth_label_sequence(n_frames, h, w, label_nc=label_nc, block=block, seed=seed)
    oh = torch.zeros(1, n_frames, label_nc, h, w)
    oh.scatter_(2, lab.long(), 1.0)
    t = lab
    edge = torch.zeros(t.size(), dtype=torch.bool)
    edge[..., :, 1:] |= (t[..., :, 1:] != t[..., :, :-1])
    edge[..., :, :-1] |= (t[..., :, 1:] != t[..., :, :-1])
    edge[..., 1:, :] |= (t[..., 1:, :] != t[..., :-1, :])
    edge[..., :-1, :] |= (t[..., 1:, :] != t[..., :-1, :])
    real_A = torch.cat([oh, edge.float()], dim=2)
    return real_A.view(1, -1, h, w), lab


def gen_inputs(label_nc, h, w, seed, fg_label=2, block=4):
    g = torch.Generator().manual_seed(seed + 77)
    inp, lab = onehot_input(label_nc, h, w, seed, block)
    # low-pass noise (SURVEY 8d): coarse U(-1,1) field, bilinearly upsampled
    coarse = torch.rand(1, 6, max(2, h // 8), max(2, w // 8), generator=g) * 2 - 1
    img_prev = torch.nn.functional.interpolate(coarse, size=(h, w), mode='bilinear', align_corners=False)
    mask = (lab[:, -1] == fg_label).float()
    return inp, img_prev, mask


def pin_inputs(nc, h, w, seed=0):
    """Inputs of the reference pins of tests/test_oracle_vs_reference.py (encode_input of a 3-frame label clip)."""
    from oracle import generator_oracle as GO
    g = torch.Generator().manual_seed(seed)
    lab = synth_label_sequence(3, h, w, label_nc=nc - 1, block=4, seed=seed)
    real_A = GO.encode_input(lab, lab, nc - 1, True)
    inp = real_A.view(1, -1, h, w)
    img_prev = torch.rand(1, 6, h, w, generator=g) * 2 - 1
    mask = (lab[:, -1] == 2).float()
    return inp, img_prev, mask


# (fg, no_flow, n_downsample_G) of the CompositeGenerator pins
PIN_COMPOSITE = [(True, False, 3), (False, False, 2), (True, True, 3)]


def pin_inference_opt():
    return make_opt(label_nc=5, use_instance=True, fg=True, fg_labels=[2], n_scales_spatial=2, ngf=8, n_blocks=2,
                    n_blocks_local=1, use_single_G=True, n_downsample_G=2, gpu_ids=[], dataroot='City')


def pin_train_opt(no_first_img):
    return make_opt(label_nc=5, use_instance=True, fg=True, fg_labels=[2], n_scales_spatial=2, ngf=8, n_blocks=2,
                    n_blocks_local=1, n_downsample_G=2, gpu_ids=[0], n_gpus_gen=1, isTrain=True, no_first_img=no_first_img,
                    max_frames_per_gpu=2, batchSize=1, dataroot='City')


def pin_train_clip(opt):
    """(label clip, real frames) of the training-forward pin: two calls of two frames each."""
    T = 2 * 2 + opt.n_frames_G - 1
    seq = synth_label_sequence(T, 32, 64, label_nc=5, block=4, seed=4)
    real = torch.rand(1, T, 3, 32, 64, generator=torch.Generator().manual_seed(6)) * 2 - 1
    return seq, real


def pin_objective(outs):
    """One scalar from every output of a generator: sum of <output, seeded random cotangent>."""
    g = torch.Generator().manual_seed(9)
    cot = [torch.randn(o.shape, generator=g) if o is not None else None for o in outs]
    return sum((o * c).sum() for o, c in zip(outs, cot) if o is not None)


# det_fill_ seeds of the spatial and the first temporal discriminator of the loss pins
PIN_SEED_D, PIN_SEED_D_T = 50, 51


def pin_loss_opt(**kw):
    opt = make_opt(label_nc=35, use_instance=True, isTrain=True, gpu_ids=[0], n_gpus_gen=1, no_vgg=True, **kw)
    opt.add_face_disc = False
    opt.debug = True
    opt.load_pretrain = ''
    return opt


def _rand(shape, g, lo=-1.0, hi=1.0):
    return torch.rand(shape, generator=g) * (hi - lo) + lo


def pin_spatial_loss_inputs(with_raw):
    """tensors_list of Vid2VidModelD.forward(0, ...): real_B, fake_B, fake_B_raw, real_A, real_B_prev, fake_B_prev, flow,
    weight, flow_ref, conf_ref."""
    g = torch.Generator().manual_seed(1)
    h, w = 48, 64
    real_B, fake_B, real_B_prev, fake_B_prev = (_rand((1, 3, h, w), g) for _ in range(4))
    fake_B_raw = _rand((1, 3, h, w), g) if with_raw else None
    real_A = (_rand((1, 36, h, w), g) > 0.8).float()
    flow, flow_ref = _rand((1, 2, h, w), g, -3, 3), _rand((1, 2, h, w), g, -3, 3)
    weight = _rand((1, 1, h, w), g, 0, 1)
    conf = (_rand((1, 1, h, w), g) > 0).float()
    return [real_B, fake_B, fake_B_raw, real_A, real_B_prev, fake_B_prev, flow, weight, flow_ref, conf]


def pin_temporal_loss_inputs(opt):
    """tensors_list of Vid2VidModelD.forward(1, ...): real_B, fake_B, flow_ref, conf_ref."""
    g = torch.Generator().manual_seed(2)
    h, w, tD = 48, 64, opt.n_frames_D
    real_B, fake_B = _rand((1, tD, 3, h, w), g), _rand((1, tD, 3, h, w), g)
    flow_ref = _rand((1, tD - 1, 2, h, w), g, -40, 40)
    conf = (_rand((1, tD - 1, 1, h, w), g) > 0).float()
    return [real_B, fake_B, flow_ref, conf]


FLOWNET2_PIN_SIZES = ((64, 64), (70, 64))


def flownet2_pin_inputs():
    """Inputs of the FlowNet2 pins: a batch-2 frame pair, sub-network inputs and wrapper frame pairs (one needs the resize)."""
    g = torch.Generator().manual_seed(3)
    i = dict(pair=torch.rand(2, 3, 2, 64, 64, generator=g), x6=torch.rand(1, 6, 64, 128, generator=g) - 0.5,
             x12=torch.rand(1, 12, 64, 128, generator=g) - 0.5,
             xf=torch.rand(1, 11, 64, 64, generator=torch.Generator().manual_seed(1)))
    for h, w in FLOWNET2_PIN_SIZES:
        i['im1_%d' % h] = torch.rand(1, 3, h, w, generator=g)
        i['im2_%d' % h] = torch.roll(i['im1_%d' % h], shifts=(1, 1), dims=(2, 3))
    return i


# state of the BaseModel schedule pins (options of train_options.py read by the schedules)
SCHEDULE_OPT = dict(name='run', lr=2e-4, niter=10, niter_decay=10, beta1=0.5, max_frames_backpropagate=4, max_frames_per_gpu=8)
SCHEDULE_EPOCHS = (11, 15, 20)
SCHEDULE_RATIOS = (1, 2, 3, 4, 5)


# name -> dict(kind, args...) ; every entry is a reference forward whose outputs are stored.
CASES = {
    # CompositeGenerator, full structure (nd 3, 9 blocks, fg) at toy width
    'g0_small': dict(kind='composite', label_nc=35, ngf=16, nd=3, n_blocks=9, fg=True, no_flow=False,
                     h=32, w=64, seed=11),
    'g0_small_ac': dict(kind='composite', label_nc=35, ngf=16, nd=3, n_blocks=9, fg=True, no_flow=False,
                        h=32, w=64, seed=11, align_corners=True),
    'g0_nofg_nd2': dict(kind='composite', label_nc=5, ngf=32, nd=2, n_blocks=4, fg=False, no_flow=False,
                        h=24, w=40, seed=12),
    'g0_noflow': dict(kind='composite', label_nc=5, ngf=16, nd=3, n_blocks=3, fg=True, no_flow=True,
                      h=32, w=32, seed=13),
    # CompositeLocalGenerator scale 1 / 2
    'gl_small_s1': dict(kind='compositeLocal', label_nc=35, ngf=16, nd=3, n_blocks_local=3, fg=True,
                        scale=1, h=32, w=64, seed=14),
    'gl_small_s2': dict(kind='compositeLocal', label_nc=5, ngf=8, nd=3, n_blocks_local=2, fg=True,
                        scale=2, h=48, w=80, seed=15),
    # first-frame generators (InstanceNorm)
    'global_small': dict(kind='global', input_nc=35, ngf=16, nd=3, n_blocks=4, h=32, w=64, seed=16),
    'local_small': dict(kind='local', input_nc=35, ngf=8, nd=3, n_blocks=3, n_blocks_local=3,
                        h=64, w=64, seed=17),
    # discriminator towers
    'D_small': dict(kind='D', input_nc=39, ndf=16, n_layers=3, num_D=3, batch=2, h=64, w=96, seed=18),
    # BASELINE config 1: full-width CompositeGenerator forward at 256x128 (W x H)
    'cfg1': dict(kind='composite', label_nc=35, ngf=128, nd=3, n_blocks=9, fg=True, no_flow=False,
                 h=128, w=256, seed=21, block=8, subsample=8),
    # Vid2VidModelG.inference, 3 scales, --fg --use_single_G, 4 generated frames
    'infer_s3': dict(kind='inference', label_nc=35, ngf=16, nd=2, n_blocks=4, n_blocks_local=2,
                     n_scales=3, h=128, w=256, n_gen=4, seed=31, flow_weight_scale=0.05),
}


def inference_opt(c):
    return make_opt(label_nc=c['label_nc'], use_instance=True, fg=True, fg_labels=[2],
                    n_scales_spatial=c['n_scales'], ngf=c['ngf'], n_blocks=c['n_blocks'],
                    n_blocks_local=c['n_blocks_local'], use_single_G=True, n_downsample_G=c['nd'],
                    gpu_ids=[], dataroot='City')


def build_module(c):
    """Our (vid2vid_b200.networks) module for a case, constructed like the reference constructs its own
    in oracle/make_golden.py."""
    from vid2vid_b200 import networks as NW
    kind = c['kind']
    if kind in ('composite', 'compositeLocal'):
        nc = 3 * (c['label_nc'] + 1)
        opt = make_opt(ngf=c['ngf'], n_blocks=c.get('n_blocks', 9), n_blocks_local=c.get('n_blocks_local', 3),
                       fg=c['fg'], no_flow=c.get('no_flow', False), n_downsample_G=c['nd'], gpu_ids=[])
        return NW.define_G(nc, 3, 6, c['ngf'], kind, c['nd'], 'batch', c.get('scale', 0), [], opt)
    if kind in ('global', 'local'):
        opt = make_opt(n_blocks=c['n_blocks'], n_blocks_local=c.get('n_blocks_local', 3), gpu_ids=[])
        return NW.define_G(c['input_nc'], 3, 0, c['ngf'], kind, c['nd'], 'instance', 0, [], opt)
    if kind == 'D':
        return NW.define_D(c['input_nc'], c['ndf'], c['n_layers'], 'batch', c['num_D'], True, [])
    raise ValueError(kind)


# module configurations whose state_dict key/shape lists are pinned in tests/golden/state_dict_keys.json
KEY_CASES = {
    'G0_street': dict(kind='composite', label_nc=35, ngf=128, nd=3, n_blocks=9, fg=True, no_flow=False),
    'G1_street': dict(kind='compositeLocal', label_nc=35, ngf=64, nd=3, n_blocks_local=3, fg=True, scale=1),
    'G2_street': dict(kind='compositeLocal', label_nc=35, ngf=32, nd=3, n_blocks_local=3, fg=True, scale=2),
    'G0_noflow_nofg': dict(kind='composite', label_nc=5, ngf=16, nd=2, n_blocks=5, fg=False, no_flow=True),
    'single_512': dict(kind='global', input_nc=35, ngf=64, nd=3, n_blocks=9),
    'single_2048': dict(kind='local', input_nc=35, ngf=32, nd=4, n_blocks=9, n_blocks_local=3),
    'D_img': dict(kind='D', input_nc=39, ndf=64, n_layers=3, num_D=3),
}


def condition_flow_heads(net, scale):
    """Random N(0,0.02) flow heads times the x20*2^s output scale give noise-like multi-pixel flows, which turn the
    warp into an error amplifier no trained model has; the inference case shrinks the flow-head weights instead."""
    import torch
    with torch.no_grad():
        if hasattr(net, 'model_final_flow'):
            net.model_final_flow[1].weight.mul_(scale)
            net.model_final_flow[1].bias.mul_(scale)

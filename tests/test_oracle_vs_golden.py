"""Pins oracle/generator_oracle.py against the committed fixtures (outputs of the unmodified
reference, oracle/make_golden.py).  CPU-only; this is the check that travels to the GPU box."""

import numpy as np
import pytest
import torch

import cases as C
from oracle import generator_oracle as GO
from oracle.make_golden import coarse_feats
from vid2vid_b200.utils import det_fill_, synth_label_sequence
from vid2vid_b200 import networks as NW



def load(name):
    return C.load_golden(name)


def close(a, gold, tol=3e-5):
    a = a.detach().numpy()
    assert a.shape == gold.shape, (a.shape, gold.shape)
    # relative to the output's magnitude where it exceeds 1 (flow is in pixels, x20 head scale): the CPU convolutions sum in
    # an order that depends on the host's vector ISA and thread count (3.3e-5 on flows of ~8 px seen between two hosts)
    assert np.abs(a - gold).max() <= tol * max(1.0, float(np.abs(gold).max())), np.abs(a - gold).max()


def build_state_dict(c):
    """Our modules reproduce the reference's state_dict keys/shapes exactly, so a state dict
    filled by det_fill_ on OUR module equals the one make_golden filled on the reference's."""
    return det_fill_(C.build_module(c), seed=c["seed"]).state_dict()


@pytest.mark.parametrize('name', ['g0_small', 'g0_small_ac', 'g0_nofg_nd2', 'g0_noflow', 'gl_small_s1',
                                  'gl_small_s2'])
def test_generators(name):
    c = C.CASES[name]
    gold = load(name)
    sd = build_state_dict(c)
    inp, img_prev, mask = C.gen_inputs(c['label_nc'], c['h'], c['w'], c['seed'], block=c.get('block', 4))
    with torch.no_grad():
        if c['kind'] == 'composite':
            out = GO.composite_generator(sd, inp, img_prev, mask, False, n_downsampling=c['nd'],
                                         n_blocks=c['n_blocks'], use_fg_model=c['fg'], no_flow=c['no_flow'],
                                         align_corners=c.get('align_corners', False))
        else:
            out = GO.composite_local_generator(sd, inp, img_prev, mask, *coarse_feats(c), False,
                                               n_blocks_local=c['n_blocks_local'], use_fg_model=c['fg'],
                                               scale=c['scale'])
    for nme, t in zip(C.GEN_OUT_NAMES, out):
        if t is None:
            assert nme not in gold
        else:
            close(t, gold[nme])


def test_single_generators_and_D():
    for name in ('global_small', 'local_small'):
        c = C.CASES[name]
        sd = build_state_dict(c)
        lab = synth_label_sequence(1, c['h'], c['w'], label_nc=c['input_nc'], block=4, seed=c['seed'])
        x = torch.zeros(1, c['input_nc'], c['h'], c['w']).scatter_(1, lab[:, 0].long(), 1.0)
        with torch.no_grad():
            if c['kind'] == 'global':
                o = GO.global_generator(sd, x, n_downsampling=c['nd'], n_blocks=c['n_blocks'])
            else:
                o = GO.local_enhancer(sd, x, n_downsample_global=c['nd'], n_blocks_global=c['n_blocks'],
                                      n_blocks_local=c['n_blocks_local'])
        close(o, load(name)['out'])
    c = C.CASES['D_small']
    sd = build_state_dict(c)
    g = torch.Generator().manual_seed(c['seed'] + 1)
    x = torch.randn(c['batch'], c['input_nc'], c['h'], c['w'], generator=g)
    gold = load('D_small')
    with torch.no_grad():
        res = GO.multiscale_discriminator(sd, x, num_D=c['num_D'], n_layers=c['n_layers'])
    for i, tower in enumerate(res):
        for j, t in enumerate(tower):
            close(t, gold['t%d_l%d' % (i, j)], 1e-4)


def test_inference_sequence():
    c = C.CASES['infer_s3']
    opt = C.inference_opt(c)
    gold = load('infer_s3')
    nets = [det_fill_(NW.build_netG(opt, s), seed=c['seed'] + s) for s in range(c['n_scales'])]
    for n_ in nets:
        C.condition_flow_heads(n_, c['flow_weight_scale'])
    sds = [n_.state_dict() for n_ in nets]
    single = det_fill_(NW.GlobalGenerator(c['label_nc'], 3, 16, 2, opt.n_blocks, NW.get_norm_layer('instance')),
                       seed=c['seed'] + 100).state_dict()
    orc = GO.ModelGOracle(opt, sds, single, 'global', 2)
    tG = opt.n_frames_G
    seq = synth_label_sequence(c['n_gen'] + tG - 1, c['h'], c['w'], label_nc=c['label_nc'], block=8, seed=c['seed'])
    with torch.no_grad():
        for t in range(c['n_gen']):
            A = seq[:, t:t + tG]
            fake_B, _ = orc.inference(A, A)
            close(fake_B, gold['fake_B_%d' % t], 1e-4)
    for si in range(c['n_scales']):
        close(orc.fake_B_prev[si], gold['prev_state_%d' % si], 1e-4)

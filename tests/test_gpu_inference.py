"""GPU parity of Vid2VidModelG.inference (multi-scale, --fg --use_single_G) against the reference fixture
and the oracle driver."""

import numpy as np
import pytest
import torch

import cases as C
from vid2vid_b200 import networks as NW
from vid2vid_b200.model_g import Vid2VidModelG
from vid2vid_b200.utils import det_fill_, synth_label_sequence

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize('mode', ['precise', 'fast'])
def test_inference_sequence_vs_reference_fixture(mode):
    NW.set_default_precision(mode)
    try:
        _inference_sequence(mode)
    finally:
        NW.set_default_precision('precise')


def _inference_sequence(mode):
    lim_mean, lim_max, lim_state = (0.02, 0.35, 0.03) if mode == 'fast' else (2e-4, 3e-3, 3e-4)
    c = C.CASES['infer_s3']
    opt = C.inference_opt(c)
    opt.gpu_ids = [0]
    gold = C.load_golden('infer_s3')
    m = Vid2VidModelG()
    m.use_single_G = False
    opt.use_single_G = False               # build without touching checkpoints/, then attach the seeded nets
    m.initialize(opt)
    opt.use_single_G = True
    m.use_single_G = True
    m.netG_i = det_fill_(NW.define_G(c['label_nc'], 3, 0, 16, 'global', 2, 'instance', 0, [], opt), seed=c['seed'] + 100).cuda()
    for s in range(c['n_scales']):
        det_fill_(getattr(m, 'netG%d' % s), seed=c['seed'] + s)
        C.condition_flow_heads(getattr(m, 'netG%d' % s), c['flow_weight_scale'])
    tG = opt.n_frames_G
    seq = synth_label_sequence(c['n_gen'] + tG - 1, c['h'], c['w'], label_nc=c['label_nc'], block=8, seed=c['seed'])
    worst = 0.0
    for t in range(c['n_gen']):
        A = seq[:, t:t + tG]
        fake_B, real_A = m.inference(A, None, A)
        d = np.abs(fake_B.cpu().numpy() - gold['fake_B_%d' % t])
        print('frame %d: max|d|=%.4f mean|d|=%.5f' % (t, d.max(), d.mean()))
        worst = max(worst, d.mean())
        assert torch.isfinite(fake_B).all()
        # recurrent generation: errors feed back through fake_B_prev; stated tolerance on [-1,1] images
        assert d.mean() < lim_mean and d.max() < lim_max
    for si in range(c['n_scales']):
        d = np.abs(m.fake_B_prev[si].cpu().numpy() - gold['prev_state_%d' % si])
        assert d.mean() < lim_state

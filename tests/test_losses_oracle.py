"""Pins oracle/losses_oracle.py (SURVEY 8 row a13: warp / flow / GAN / feature-matching losses of the training step)
against the unmodified reference Vid2VidModelD.forward (models/vid2vid_model_D.py:92-197) on CPU, --no_vgg, through its
outputs on seeded inputs (tests/golden/ref_losses.npz, written by `python -m oracle.make_golden losses`)."""
import os

import numpy as np
import pytest
import torch

import cases
from oracle import losses_oracle as LO
from vid2vid_b200 import networks as NW
from vid2vid_b200.utils import det_fill_

GOLD = np.load(os.path.join(os.path.dirname(__file__), 'golden', 'ref_losses.npz'))


def _netD_sd(opt, input_nc, seed):
    """The discriminator Vid2VidModelD.initialize builds (vid2vid_model_D.py:28-38), filled as the pins fill the reference's."""
    return det_fill_(NW.define_D(input_nc, opt.ndf, opt.n_layers_D, opt.norm, opt.num_D, not opt.no_ganFeat, []), seed=seed).state_dict()


def _ref(key, n):
    return [torch.from_numpy(GOLD['%s_%d' % (key, i)]) for i in range(n)]


@pytest.mark.parametrize('no_first_img,with_raw', [(False, True), (True, False)])
def test_spatial_losses_match_reference(no_first_img, with_raw):
    opt = cases.pin_loss_opt(n_scales_spatial=2, no_first_img=no_first_img)
    sd = _netD_sd(opt, opt.label_nc + 1 + opt.output_nc, cases.PIN_SEED_D)
    with torch.no_grad():
        ours = LO.spatial_losses(sd, *cases.pin_spatial_loss_inputs(with_raw), lambda_F=opt.lambda_F, lambda_T=opt.lambda_T,
                                 lambda_feat=opt.lambda_feat, n_scales_spatial=opt.n_scales_spatial, no_first_img=no_first_img,
                                 num_D=opt.num_D, n_layers_D=opt.n_layers_D, norm=opt.norm)
    names = ['G_VGG', 'G_GAN', 'G_GAN_Feat', 'D_real', 'D_fake', 'G_Warp', 'F_Flow', 'F_Warp', 'W']
    ref = _ref('spatial_%d' % no_first_img, len(names))
    assert len(ours) == len(names)
    for n, a, b in zip(names, ours, ref):
        # (G_VGG under --no_vgg and W without --no_first_img are zeros_like(weight): H*W rows of zeros in both)
        assert a.shape == b.shape, (n, a.shape, b.shape)
        assert torch.allclose(a, b, rtol=1e-4, atol=1e-6), (n, float(a.abs().max()), float(b.abs().max()))
        if n in ('G_GAN', 'G_GAN_Feat', 'D_real', 'D_fake', 'G_Warp', 'F_Flow', 'F_Warp'):
            assert a.shape == (1, 1) and float(a) > 0


def test_temporal_losses_match_reference():
    opt = cases.pin_loss_opt()
    tD = opt.n_frames_D
    sd = _netD_sd(opt, opt.output_nc * tD + 2 * (tD - 1), cases.PIN_SEED_D_T)
    with torch.no_grad():
        ours = LO.temporal_losses(sd, *cases.pin_temporal_loss_inputs(opt), n_frames_D=tD, output_nc=3,
                                  lambda_feat=opt.lambda_feat, num_D=opt.num_D, n_layers_D=opt.n_layers_D, norm=opt.norm)
    names = ['G_T_GAN', 'G_T_GAN_Feat', 'D_T_real', 'D_T_fake', 'G_T_Warp']
    assert len(ours) == len(names)
    for n, a, b in zip(names, ours, _ref('temporal', len(names))):
        assert torch.allclose(a, b, rtol=1e-4, atol=1e-6), (n, float(a), float(b))

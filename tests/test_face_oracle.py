"""Pins tests/face_oracle.py (the face discriminator of the pose training step, --add_face_disc) against the unmodified
reference Vid2VidModelD on CPU through its stored outputs (tests/golden/ref_face.npz and ref_face_keys.json, written by
`python tools/make_face_golden.py`): the face window as exact integers, the 13 spatial losses to the tolerance of
tests/test_losses_oracle.py, and the netD_f state_dict layout."""
import json
import os

import numpy as np
import pytest
import torch

import face_oracle as FC
from vid2vid_b200 import networks as NW
from vid2vid_b200.utils import det_fill_

GOLD_DIR = os.path.join(os.path.dirname(__file__), 'golden')
GOLD = np.load(os.path.join(GOLD_DIR, 'ref_face.npz'))


def _netD_f(opt):
    return NW.define_D(6 + opt.output_nc, opt.ndf, opt.n_layers_D, opt.norm, max(1, opt.num_D - 2), not opt.no_ganFeat, [])


@pytest.mark.parametrize('name', list(FC.FACE_CASES))
def test_face_region_matches_reference(name):
    _, openpose = FC.FACE_CASES[name]
    win = FC.face_region(FC.face_case_real_A(name), FC.FACE_FINE, openpose)
    ref = [int(v) for v in GOLD['%s_window' % name]]
    assert (list(win) if win is not None else [-1] * 4) == ref


def test_face_cases_cover_every_border():
    wins = {n: [int(v) for v in GOLD['%s_window' % n]] for n in FC.FACE_CASES}
    L = FC.FACE_FINE // 32 * 8
    assert wins['top'][0] == 0 and wins['left'][2] == 0
    assert wins['bottom'][1] == FC.FACE_H - 1 and wins['right'][3] == FC.FACE_W - 1        # the reference's h - 1 / w - 1
    assert wins['none'] == [-1] * 4
    for n, w in wins.items():
        if n != 'none':
            assert w[1] - w[0] == L and w[3] - w[2] == L, n


@pytest.mark.parametrize('name', list(FC.FACE_CASES))
def test_spatial_losses_with_face_match_reference(name):
    _, openpose = FC.FACE_CASES[name]
    opt = FC.face_opt(openpose_only=openpose)
    sd = det_fill_(NW.define_D(6 + opt.output_nc, opt.ndf, opt.n_layers_D, opt.norm, opt.num_D, True, []), seed=FC.FACE_SEED_D)
    sd_f = det_fill_(_netD_f(opt), seed=FC.FACE_SEED_D_F)
    with torch.no_grad():
        ours = FC.spatial_losses(sd.state_dict(), sd_f.state_dict(), *FC.face_case_inputs(name), fine_size=opt.fineSize,
                                 openpose_only=openpose, lambda_F=opt.lambda_F, lambda_T=opt.lambda_T, lambda_feat=opt.lambda_feat,
                                 n_scales_spatial=opt.n_scales_spatial, no_first_img=opt.no_first_img, num_D=opt.num_D,
                                 n_layers_D=opt.n_layers_D, norm=opt.norm)
    assert len(ours) == len(FC.SPATIAL_LOSS_NAMES) == 13
    for n, a in zip(FC.SPATIAL_LOSS_NAMES, ours):
        b = torch.from_numpy(GOLD['%s_%s' % (name, n)])
        assert a.shape == b.shape, (n, a.shape, b.shape)
        assert torch.allclose(a, b, rtol=1e-4, atol=1e-6), (n, float(a.abs().max()), float(b.abs().max()))
        if n in FC.FACE_LOSS_NAMES:
            assert (float(a) == 0) == (name == 'none'), (n, float(a))


def test_netD_f_state_dict_layout_matches_reference():
    ref = json.load(open(os.path.join(GOLD_DIR, 'ref_face_keys.json')))
    ours = [[k, list(v.shape)] for k, v in _netD_f(FC.face_opt()).state_dict().items()]
    assert ours == ref

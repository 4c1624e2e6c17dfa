"""Pins oracle/flownet2_oracle.py (SURVEY 8 rows a14 / a15: the reference flow network behind the training targets).
  * against the committed fixtures tests/golden/flownet2_small.npz and flownet2_pins.npz: outputs of the unmodified
    reference modules (models/flownet2_pytorch/models.py, models/flownet.py) on seeded inputs, with weights regenerated
    from (seed, key, shape).  The three native ops are CUDA-only in the reference and were supplied by
    oracle/flowops_oracle.c there, so this pins the network wiring, layer hyper-parameters and the wrapper logic, not
    those ops.  CPU only."""
import json
import os

import numpy as np
import torch

import cases
from oracle import flownet2_oracle as FO

GOLD = os.path.join(os.path.dirname(__file__), 'golden')


def _close(a, b, name, tol=2e-4):
    a, b = torch.as_tensor(a).float(), torch.as_tensor(b).float()
    assert a.shape == b.shape, (name, a.shape, b.shape)
    scale = max(1.0, float(b.abs().max()))
    err = float((a - b).abs().max())
    assert err <= tol * scale, '%s: max |d| = %.3e (scale %.2f)' % (name, err, scale)


def test_flownet2_oracle_vs_golden():
    keys = json.load(open(os.path.join(GOLD, 'flownet2_keys.json')))
    assert len(keys) == 220 and sum(int(np.prod(s)) for _, s in keys) == 162518834      # models.py:16 parameter count
    g = np.load(os.path.join(GOLD, 'flownet2_small.npz'))
    sd = FO.det_state_dict(keys, seed=7)
    with torch.no_grad():
        flow = FO.flownet2(sd, torch.from_numpy(g['pair']))
        wflow, wconf = FO.flow_and_conf(sd, torch.from_numpy(g['im1']), torch.from_numpy(g['im2']))
    _close(flow, g['flow'], 'FlowNet2 flow')
    _close(wflow, g['wflow'], 'wrapper flow (80 -> 64 rows and back)')
    # the confidence is a thresholded mask: allow the few pixels that sit on the 0.02 threshold to flip
    assert float(np.abs(wconf.numpy() - g['wconf']).mean()) < 2e-3


def test_flownet2_oracle_vs_reference_random_init():
    keys = json.load(open(os.path.join(GOLD, 'flownet2_keys.json')))
    sd = FO.det_state_dict(keys, seed=3)
    g = np.load(os.path.join(GOLD, 'flownet2_pins.npz'))
    i = cases.flownet2_pin_inputs()
    with torch.no_grad():
        _close(FO.flownet2(sd, i['pair']), g['flow'], 'FlowNet2 (batch 2, 64x64)')
        # sub-networks on their own inputs (eval mode returns a 1-tuple)
        _close(FO.flownet_c(sd, 'flownetc.', i['x6']), g['flownetc'], 'FlowNetC')
        _close(FO.flownet_s(sd, 'flownets_1.', i['x12']), g['flownets_1'], 'FlowNetS')
        _close(FO.flownet_sd(sd, 'flownets_d.', i['x6']), g['flownets_d'], 'FlowNetSD')
        _close(FO.flownet_fusion(sd, 'flownetfusion.', i['xf']), g['flownetfusion'], 'FlowNetFusion')
    # the vid2vid wrapper (models/flownet.py:43-58), un-resized and resized paths
    for h, w in cases.FLOWNET2_PIN_SIZES:
        with torch.no_grad():
            of, oc = FO.flow_and_conf(sd, i['im1_%d' % h], i['im2_%d' % h])
        _close(of, g['wflow_%d' % h], 'wrapper flow %dx%d' % (h, w))
        assert float(np.abs(oc.numpy() - g['wconf_%d' % h]).mean()) < 2e-3

"""GPU parity of the generator modules (the nn.Module boundary, SURVEY 8b2) through the C-ABI plan
runtime: against the committed reference fixtures (tests/golden, fp32 reference outputs), against the
oracle on the same seeded inputs, and against the bf16-rounding emulation (kernel exactness)."""
import os

import numpy as np
import pytest
import torch

import cases as C
from oracle.make_golden import coarse_feats
from vid2vid_b200.utils import det_fill_, synth_label_sequence

pytestmark = pytest.mark.gpu

# Stated tolerances against the fp32 reference (DESIGN.md 4), (max |d|, mean |d|); images and masks live in [-1,1] / [0,1],
# features are O(1) (rms ~0.7), flow is in pixels and carries the x20*2^s head scale.
#   precise (split-bf16 x3, the product default): fp32-class -- images 5e-3, features 1e-3, flow 0.02 px ABSOLUTE.
#   fast (bf16 operands): flow limits are relative to the reference rms.
TOLS = {
    'precise': {'img_final': (5e-3, 3e-4), 'img_raw': (5e-3, 3e-4), 'weight': (1e-3, 1e-4), 'flow': (0.02, 0.004),
                'img_feat': (1e-3, 1e-4), 'flow_feat': (1e-3, 1e-4), 'img_fg_feat': (1e-3, 1e-4), 'out': (2e-3, 2e-4)},
    'fast': {'img_final': (0.30, 0.02), 'img_raw': (0.15, 0.015), 'weight': (0.08, 0.01), 'flow': (0.15, 0.03),
             'img_feat': (0.5, 0.03), 'flow_feat': (0.5, 0.03), 'img_fg_feat': (0.5, 0.03), 'out': (0.12, 0.015)},
}
TOL = dict(TOLS['precise'])
MODE = ['precise']


@pytest.fixture(autouse=True, params=['precise', 'fast'])
def mode(request):
    from vid2vid_b200 import networks as NW
    old = NW.DEFAULT_PRECISION
    NW.set_default_precision(request.param)
    MODE[0] = request.param
    TOL.clear()
    TOL.update(TOLS[request.param])
    yield request.param
    NW.set_default_precision(old)


def load(name):
    return C.load_golden(name)


def report(name, key, out, gold):
    d = np.abs(out - gold)
    rms = np.sqrt((gold ** 2).mean())
    print('%-12s %-12s max|d|=%.4f mean|d|=%.5f  ref rms=%.3f' % (name, key, d.max(), d.mean(), rms))
    if key == 'flow' and MODE[0] == 'fast':
        return d.max() / rms, d.mean() / rms
    return d.max(), d.mean()


@pytest.mark.parametrize('name', ['g0_small', 'g0_small_ac', 'g0_nofg_nd2', 'g0_noflow', 'gl_small_s1', 'gl_small_s2'])
def test_generator_vs_reference_fixture(name):
    c = C.CASES[name]
    gold = load(name)
    net = det_fill_(C.build_module(c), seed=c['seed']).cuda()
    net.align_corners = c.get('align_corners', False)
    inp, img_prev, mask = (t.cuda() for t in C.gen_inputs(c['label_nc'], c['h'], c['w'], c['seed'], block=c.get('block', 4)))
    coarse = tuple(t.cuda() for t in coarse_feats(c)) if c['kind'] == 'compositeLocal' else (None, None, None)
    with torch.no_grad():
        out = net(inp, img_prev, mask, *coarse, False)
    bad = []
    for key, t in zip(C.GEN_OUT_NAMES, out):
        if t is None:
            assert key not in gold
            continue
        assert torch.isfinite(t).all(), key
        mx, mn = report(name, key, t.cpu().numpy(), gold[key])
        if mx > TOL[key][0] or mn > TOL[key][1]:
            bad.append((key, mx, mn))
    assert not bad, bad


def test_cfg1_full_width_generator():
    """BASELINE config 1: CompositeGenerator(ngf 128, nd 3, 9 blocks, fg) at 256x128."""
    c = C.CASES['cfg1']
    gold = load('cfg1')
    net = det_fill_(C.build_module(c), seed=c['seed']).cuda()
    inp, img_prev, mask = (t.cuda() for t in C.gen_inputs(c['label_nc'], c['h'], c['w'], c['seed'], block=c['block']))
    with torch.no_grad():
        out = net(inp, img_prev, mask, None, None, None, False)
    ss = c['subsample']
    bad = []
    for key, t in zip(C.GEN_OUT_NAMES, out):
        t = t.cpu()
        if key + '_sub' in gold:
            mx, mn = report('cfg1', key, t[:, :, ::ss, ::ss].numpy(), gold[key + '_sub'])
            cm = np.abs(t.mean(dim=(2, 3)).numpy() - gold[key + '_cmean']).max()
            assert cm < (0.02 if MODE[0] == 'fast' else 2e-3 * (20 if key == 'flow' else 1)), (key, cm)
        else:
            mx, mn = report('cfg1', key, t.numpy(), gold[key])
        if mx > TOL[key][0] or mn > TOL[key][1]:
            bad.append((key, mx, mn))
    assert not bad, bad


@pytest.mark.parametrize('name', ['global_small', 'local_small'])
def test_first_frame_generators(name):
    c = C.CASES[name]
    net = det_fill_(C.build_module(c), seed=c['seed']).cuda()
    lab = synth_label_sequence(1, c['h'], c['w'], label_nc=c['input_nc'], block=4, seed=c['seed'])
    x = torch.zeros(1, c['input_nc'], c['h'], c['w']).scatter_(1, lab[:, 0].long(), 1.0).cuda()
    with torch.no_grad():
        out = net(x)
    mx, mn = report(name, 'out', out.cpu().numpy(), load(name)['out'])
    assert mx <= TOL['out'][0] and mn <= TOL['out'][1]


def test_generator_simt_vs_umma_same_plan():
    """The tcgen05 kernel and the SIMT cross-check kernel evaluate the same lowered plan."""
    c = C.CASES['g0_small']
    inp, img_prev, mask = (t.cuda() for t in C.gen_inputs(c['label_nc'], c['h'], c['w'], c['seed']))
    outs = []
    for impl in ('umma', 'simt'):
        os.environ['V2V_CONV_IMPL'] = impl
        try:
            net = det_fill_(C.build_module(c), seed=c['seed']).cuda()
            with torch.no_grad():
                outs.append(net(inp, img_prev, mask, None, None, None, False))
        finally:
            os.environ.pop('V2V_CONV_IMPL', None)
    for key, a, b in zip(C.GEN_OUT_NAMES, *outs):
        d = (a - b).abs()
        print('%-12s umma-vs-simt max|d|=%.4f mean|d|=%.5f' % (key, d.max().item(), d.mean().item()))
        lim = 0.03 * b.pow(2).mean().sqrt().item() if key == 'flow' else (2e-2 if key == 'img_final' else 1e-2)
        if MODE[0] == 'precise':
            lim = 0.004 if key == 'flow' else 1e-4
        assert d.mean().item() < lim, key


def test_multiscale_discriminator_vs_reference_fixture():
    """MultiscaleDiscriminator (SURVEY 8 a12): all 5 layer outputs of all 3 towers, batch 2, BatchNorm train mode."""
    c = C.CASES['D_small']
    gold = load('D_small')
    net = det_fill_(C.build_module(c), seed=c['seed']).cuda()
    g = torch.Generator().manual_seed(c['seed'] + 1)
    x = torch.randn(c['batch'], c['input_nc'], c['h'], c['w'], generator=g).cuda()
    with torch.no_grad():
        res = net(x)
        res2 = net(x)
    bad = []
    for i, tower in enumerate(res):
        for j, t in enumerate(tower):
            assert torch.equal(t, res2[i][j])
            gk = gold['t%d_l%d' % (i, j)]
            d = np.abs(t.cpu().numpy() - gk)
            rms = np.sqrt((gk ** 2).mean())
            print('D tower %d layer %d: max|d|=%.4f mean|d|=%.5f ref rms=%.3f' % (i, j, d.max(), d.mean(), rms))
            # bf16 operands, <= 5 layers deep: mean error within 2 %% of the layer's rms (precise: 1e-4)
            if d.mean() > (0.02 if MODE[0] == 'fast' else 1e-4) * max(rms, 0.05):
                bad.append((i, j, d.mean(), rms))
    assert not bad, bad


def test_cfg2_full_size_vs_oracle():
    """BASELINE config 2 geometry (full-width CompositeGenerator, 512x256): CUDA path vs the CPU oracle on the same
    seeded inputs (the oracle needs a few seconds here)."""
    from oracle import generator_oracle as GO
    c = dict(C.CASES['cfg1'], h=256, w=512, seed=41)
    net = det_fill_(C.build_module(c), seed=c['seed'])
    sd = {k: v.clone() for k, v in net.state_dict().items()}
    inp, img_prev, mask = C.gen_inputs(c['label_nc'], c['h'], c['w'], c['seed'], block=8)
    with torch.no_grad():
        ref = GO.composite_generator(sd, inp, img_prev, mask, False, n_downsampling=3, n_blocks=9, use_fg_model=True, no_flow=False)
        net = net.cuda()
        out = net(inp.cuda(), img_prev.cuda(), mask.cuda(), None, None, None, False)
    bad = []
    for key, o, r in zip(C.GEN_OUT_NAMES, out, ref):
        mx, mn = report('cfg2', key, o.cpu().numpy(), r.numpy())
        if mx > TOL[key][0] * (1.5 if MODE[0] == 'fast' else 1.0) or mn > TOL[key][1]:
            bad.append((key, mx, mn))
    assert not bad, bad


def test_cfg4_finest_scale_properties():
    """BASELINE config 4 geometry, finest scale (CompositeLocalGenerator ngf 32 at 2048x1024) -- too large for the CPU
    oracle inside a test, so size-independent properties are checked: finite outputs in range, bit-identical CUDA-graph
    replay, per-channel statistics of a train-mode BatchNorm + ReLU output, and agreement of the fused warp/composite
    with the stand-alone resample operator on the generator's own flow."""
    from vid2vid_b200 import ops
    c = dict(kind='compositeLocal', label_nc=35, ngf=32, nd=3, n_blocks_local=3, fg=True, scale=2, h=1024, w=2048, seed=51)
    net = det_fill_(C.build_module(c), seed=c['seed']).cuda()
    inp, img_prev, mask = (t.cuda() for t in C.gen_inputs(c['label_nc'], c['h'], c['w'], c['seed'], block=32))
    g = torch.Generator().manual_seed(7)
    coarse = [torch.randn(1, ch, 512, 1024, generator=g).cuda() for ch in (64, 64, 32)]
    with torch.no_grad():
        out = net(inp, img_prev, mask, *coarse, False)
        out2 = net(inp, img_prev, mask, *coarse, False)
    img_final, flow, weight, img_raw, img_feat, flow_feat, fg_feat = out
    for a, b in zip(out, out2):
        assert torch.equal(a, b)
    for t in out:
        assert torch.isfinite(t).all()
    assert img_final.abs().max() <= 1.0 + 1e-5 and img_raw.abs().max() <= 1.0 + 1e-5
    assert weight.min() >= 0 and weight.max() <= 1
    # img_feat = ReLU(BatchNorm(deconv)): gamma ~ 1, beta small -> per-channel mean of max(z,0), z ~ N(beta, 1): ~0.4
    m = img_feat.mean(dim=(0, 2, 3))
    assert (m > 0.2).all() and (m < 0.7).all(), m
    assert (img_feat >= 0).all()
    # composite identity: img_final = fg*mask + (raw_nofg*w + warp*(1-w))*(1-mask); check the non-fg region via resample
    warp = ops.resample(img_prev[:, -3:].contiguous(), flow, align_corners=False)
    sel = (mask.expand_as(img_final) == 0)
    recon = img_raw * weight + warp * (1 - weight)
    d = (recon - img_final).abs()[sel]
    assert d.max().item() < 1e-5, d.max().item()


def test_running_statistics_update_once_per_forward():
    """nn.BatchNorm2d's train-mode side effect happens exactly once per layer per forward -- also for the layer whose raw
    output feeds two normalise passes (CompositeLocalGenerator: model_down_img's last norm is applied with the img and the
    flow coarse features, networks.py:298-305) -- and moves running_mean towards the batch mean."""
    import torch.nn as nn
    c = C.CASES['gl_small_s1']
    net = det_fill_(C.build_module(c), seed=c['seed']).cuda()
    inp, img_prev, mask = (t.cuda() for t in C.gen_inputs(c['label_nc'], c['h'], c['w'], c['seed']))
    coarse = tuple(t.cuda() for t in coarse_feats(c))
    with torch.no_grad():
        net(inp, img_prev, mask, *coarse, False)
        torch.cuda.synchronize()
        bns = [(n, m) for n, m in net.named_modules() if isinstance(m, nn.BatchNorm2d)]
        assert len(bns) > 10
        for n, m in bns:
            assert int(m.num_batches_tracked.item()) == 1, (n, int(m.num_batches_tracked.item()))
            assert m.running_mean.abs().max().item() > 0 and torch.isfinite(m.running_var).all(), n
        net(inp, img_prev, mask, *coarse, False)
        torch.cuda.synchronize()
        for n, m in bns:
            assert int(m.num_batches_tracked.item()) == 2, n

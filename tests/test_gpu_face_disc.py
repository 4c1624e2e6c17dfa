"""The face discriminator of the pose training step (--add_face_disc) on the GPU: the face_window / crop_concat kernels against
the CPU oracle and torch, Vid2VidModelD.forward(0, ...) with the face terms against tests/face_oracle.py (itself pinned to the
reference by tests/test_face_oracle.py), one pose training step's losses and gradients against oracle autograd, and six
Trainer steps on a pose clip.  Reads only the fixtures under tests/golden/ and oracle/."""
import json
import os

import numpy as np
import pytest
import torch

import face_oracle as FC
from oracle import flownet2_oracle as FO
from oracle import generator_oracle as GO
from vid2vid_b200 import flownet as FN
from vid2vid_b200 import ops
from vid2vid_b200.model_d import Vid2VidModelD
from vid2vid_b200.model_g import Vid2VidModelG
from vid2vid_b200.trainer import Trainer
from vid2vid_b200.utils import det_fill_, make_opt, synth_pose_sequence

pytestmark = pytest.mark.gpu

GOLD_DIR = os.path.join(os.path.dirname(__file__), 'golden')
GOLD = np.load(os.path.join(GOLD_DIR, 'ref_face.npz'))


def _win(real_A, fine, openpose):
    w = ops.face_window(real_A.cuda(), fine, openpose).cpu().tolist()
    o = FC.face_region(real_A, fine, openpose)
    return w, ([1] + list(o) if o is not None else [0] * 5)


# ------------------------------------------------------------------------------------------------ face_window
@pytest.mark.parametrize('name', list(FC.FACE_CASES))
def test_face_window_matches_oracle_and_reference(name):
    _, openpose = FC.FACE_CASES[name]
    ours, orc = _win(FC.face_case_real_A(name), FC.FACE_FINE, openpose)
    assert ours == orc
    ref = [int(v) for v in GOLD['%s_window' % name]]
    assert ours[1:] == (ref if ref[0] >= 0 else [0] * 4)


@pytest.mark.parametrize('H,W,N,seed', [(37, 53, 2, 1), (61, 129, 3, 2), (100, 77, 1, 3), (16, 16, 2, 4)])
def test_face_window_odd_sizes_and_one_face_in_three(H, W, N, seed):
    fine = 64                                                        # a 16x16 window
    g = torch.Generator().manual_seed(seed)
    for trial in range(6):
        real_A = torch.rand(N, 6, H, W, generator=g) * 1.7 - 0.85
        k = int(torch.randint(0, N, (1,), generator=g))              # the only image with face pixels
        n_px = int(torch.randint(1, 12, (1,), generator=g))
        ys = torch.randint(0, H, (n_px,), generator=g)
        xs = torch.randint(0, W, (n_px,), generator=g)
        real_A[k, 2, ys, xs] = 0.95
        ours, orc = _win(real_A, fine, False)
        assert ours == orc, (trial, ours, orc)
        assert ours[0] == 1 and ours[2] - ours[1] == 16 and ours[4] - ours[3] == 16


def test_face_window_fp32_thresholds():
    """Pixels exactly at the fp32 thresholds are not face pixels (strict comparisons on float32 values, as torch makes them)."""
    f32 = lambda v: float(np.float32(v))
    H, W = 40, 48
    real_A = torch.zeros(2, 6, H, W)
    real_A[0, 2, 5, 7] = f32(0.9)                                    # channel 2 == 0.9f: not a face
    assert _win(real_A, 64, False) == ([0] * 5, [0] * 5)
    real_A[1, 2, 30, 40] = torch.nextafter(torch.tensor(f32(0.9)), torch.tensor(1.0))
    ours, orc = _win(real_A, 64, False)
    assert ours == orc and ours[0] == 1
    face = (0.2, -1.0, -0.6)
    op = torch.zeros(2, 6, H, W)
    boundary = [(0, f32(0.19)), (0, f32(0.21)), (1, f32(-0.99)), (2, f32(-0.61)), (2, f32(-0.59))]
    for i, (c, v) in enumerate(boundary):
        px = list(face)
        px[c] = v
        for cc in range(3):
            op[i % 2, cc, 3 + 6 * i, 2 + 8 * i] = px[cc]
    assert _win(op, 64, True) == ([0] * 5, [0] * 5)
    for cc in range(3):
        op[1, cc, 35, 44] = face[cc]
    ours, orc = _win(op, 64, True)
    assert ours == orc and ours[0] == 1


def test_face_window_buffer_is_reusable():
    buf = ops.face_window_buffer('cuda')
    for name in ('interior', 'none', 'bottom', 'openpose', 'right'):
        _, openpose = FC.FACE_CASES[name]
        real_A = FC.face_case_real_A(name)
        got = ops.face_window(real_A.cuda(), FC.FACE_FINE, openpose, buf=buf).cpu().tolist()
        assert got == _win(real_A, FC.FACE_FINE, openpose)[1], name
        assert buf[5:].cpu().tolist() == [0] * 5


def test_face_window_rejects_frames_smaller_than_the_window():
    with pytest.raises(ValueError):
        ops.face_window(torch.zeros(1, 6, 31, 64, device='cuda'), 128, False)


# ------------------------------------------------------------------------------------------------ crop kernels
@pytest.mark.parametrize('name', ['interior', 'bottom', 'right', 'top'])
def test_crop_concat_forward_backward_bit_identical_to_torch(name):
    _, openpose = FC.FACE_CASES[name]
    real_A = FC.face_case_real_A(name).cuda()
    g = torch.Generator().manual_seed(5)
    b = torch.randn(2, 3, FC.FACE_H, FC.FACE_W, generator=g).cuda().requires_grad_(True)
    win = ops.face_window(real_A, FC.FACE_FINE, openpose)
    _, ys, ye, xs, xe = win.cpu().tolist()
    size = ye - ys
    out = ops.crop_concat(real_A, b, win, size)
    b2 = b.detach().clone().requires_grad_(True)
    ref = torch.cat((real_A[:, :, ys:ye, xs:xe], b2[:, :, ys:ye, xs:xe]), dim=1)
    assert torch.equal(out, ref)
    cot = torch.randn(ref.shape, generator=g).cuda()
    (out * cot).sum().backward()
    (ref * cot).sum().backward()
    assert torch.equal(b.grad, b2.grad)


# ------------------------------------------------------------------------------------------------ losses
def _model_D(openpose=False, **kw):
    opt = FC.face_opt(openpose_only=openpose, **kw)
    D = Vid2VidModelD().initialize(opt)
    det_fill_(D.netD, seed=FC.FACE_SEED_D)
    det_fill_(D.netD_f, seed=FC.FACE_SEED_D_F)
    return opt, D


def _oracle_losses(opt, D, inputs, openpose):
    sd = {k: v.detach().cpu() for k, v in D.netD.state_dict().items()}
    sd_f = {k: v.detach().cpu() for k, v in D.netD_f.state_dict().items()}
    return FC.spatial_losses(sd, sd_f, *inputs, fine_size=opt.fineSize, openpose_only=openpose, lambda_F=opt.lambda_F,
                             lambda_T=opt.lambda_T, lambda_feat=opt.lambda_feat, n_scales_spatial=opt.n_scales_spatial,
                             no_first_img=opt.no_first_img, num_D=opt.num_D, n_layers_D=opt.n_layers_D, norm=opt.norm)


@pytest.mark.parametrize('name', ['interior', 'bottom', 'left', 'one_of_two', 'openpose'])
def test_spatial_losses_with_face_vs_oracle(name):
    _, openpose = FC.FACE_CASES[name]
    opt, D = _model_D(openpose)
    assert D.loss_names[9:] == FC.FACE_LOSS_NAMES
    inputs = FC.face_case_inputs(name)
    with torch.no_grad():
        ref = _oracle_losses(opt, D, inputs, openpose)
        ours = D(0, [t.cuda() for t in inputs])
    assert len(ours) == 13
    for n, a, r in zip(D.loss_names, ours, ref):
        a, r = float(a.mean()), float(r.mean())
        print('%-13s ours %.6f oracle %.6f' % (n, a, r))
        assert abs(a - r) <= 2e-3 * max(1.0, abs(r)), n
        if n in FC.FACE_LOSS_NAMES:
            assert r > 0


def test_no_face_gives_zero_face_losses_and_leaves_netD_f_alone():
    opt, D = _model_D()
    inputs = FC.face_case_inputs('none')
    stats = {k: v.clone() for k, v in D.netD_f.state_dict().items() if 'running' in k or 'num_batches' in k}
    with torch.no_grad():
        ref = _oracle_losses(opt, D, inputs, False)
        ours = D(0, [t.cuda() for t in inputs])
    for n, a, r in zip(D.loss_names, ours, ref):
        if n in FC.FACE_LOSS_NAMES:
            assert torch.count_nonzero(a) == 0 and a.shape == (1, 1), n
        else:
            assert abs(float(a.mean()) - float(r.mean())) <= 2e-3 * max(1.0, abs(float(r.mean()))), n
    for k, v in D.netD_f.state_dict().items():
        if k in stats:
            assert torch.equal(v, stats[k]), k


# ------------------------------------------------------------------------------------------------ training step
def _pose_setup(H=64, W=128, seed=3, T=8):
    opt = make_opt(label_nc=0, input_nc=6, use_instance=False, fg=True, fg_labels=[2], no_first_img=True, n_scales_spatial=2, ngf=16,
                   n_downsample_G=2, n_blocks=4, n_blocks_local=2, num_D=3, ndf=16, n_scales_temporal=2, isTrain=True, no_vgg=True,
                   gpu_ids=[0], n_frames_total=12, add_face_disc=True, fineSize=128, dataroot='datasets/pose/')
    G = Vid2VidModelG().initialize(opt)
    D = Vid2VidModelD().initialize(opt)
    for s in range(2):
        det_fill_(getattr(G, 'netG%d' % s), seed=seed + s)
        net = getattr(G, 'netG%d' % s)
        if hasattr(net, 'model_final_flow'):          # few-pixel flows, as tests/cases.condition_flow_heads makes them
            with torch.no_grad():
                net.model_final_flow[1].weight.mul_(0.05)
                net.model_final_flow[1].bias.mul_(0.05)
    det_fill_(D.netD, seed=seed + 10)
    det_fill_(D.netD_f, seed=seed + 30)
    for s in range(2):
        det_fill_(getattr(D, 'netD_T%d' % s), seed=seed + 20 + s)
    flow = FN.FlowNet().initialize(opt)
    keys = json.load(open(os.path.join(GOLD_DIR, 'flownet2_keys.json')))
    flow.flowNet.load_state_dict({k: v.cuda() for k, v in FO.det_state_dict(keys, seed=3).items()})
    A = synth_pose_sequence(T, H, W, seed=seed, block=8, face_size=8)
    g = torch.Generator().manual_seed(seed)
    coarse = torch.rand(T, 3, H // 8, W // 8, generator=g) * 2 - 1
    B = torch.nn.functional.interpolate(coarse, size=(H, W), mode='bilinear', align_corners=False).view(1, T, 3, H, W)
    return opt, G, D, flow, A, B


class _RecordingFlow:
    """The FlowNet of the step, keeping its outputs so that the oracle sees the same flow_ref / conf_ref."""

    def __init__(self, net):
        self.net, self.calls = net, []

    def __call__(self, a, b):
        out = self.net(a, b)
        self.calls.append(out)
        return out


def _rel_check(ours, ref, what, lim_each, lim_median):
    rels = []
    gmax = max(r.abs().max().item() for r in ref.values())
    for k, r in ref.items():
        if r.abs().max().item() < 1e-9 or (k.endswith('.bias') and ours[k].abs().max().item() == 0 and r.abs().max().item() < 1e-5 * gmax):
            continue          # conv bias in front of a norm layer: exactly zero here, rounding noise in the oracle
        rel = ((ours[k] - r).norm() / r.norm()).item()
        rels.append(rel)
        assert rel <= lim_each, (what, k, rel)
    rels.sort()
    print('%s gradients: %d tensors, median rel L2 %.2e, max %.2e' % (what, len(rels), rels[len(rels) // 2], rels[-1]))
    assert rels[len(rels) // 2] <= lim_median, what


def test_pose_training_step_losses_and_gradients_vs_oracle():
    opt, G, D, flow, A, B = _pose_setup()
    rec = _RecordingFlow(flow)
    tr = Trainer(opt, G, D, rec, world=1)
    tG = opt.n_frames_G
    tr.losses(A[:, :tG].cuda(), B[:, :tG].cuda(), None)                    # first call: raw-only frame, primes fake_B_prev
    prev_pyr = [p.detach().cpu() for p in tr.fake_B_prev_last]
    rec.calls.clear()
    a, b = A[:, 1:1 + tG], B[:, 1:1 + tG]
    loss_G, loss_D, loss_D_T, ld, _ = tr.losses(a.cuda(), b.cuda(), None)
    assert not loss_D_T and float(ld['W']) > 0 and float(ld['D_f_real']) > 0
    tr.grads.zero()
    loss_G.backward()
    gG = {'%d.%s' % (s, n): q.grad.detach().cpu().double().clone() for s in range(2) for n, q in getattr(G, 'netG%d' % s).named_parameters()}
    tr.grads.zero(1)
    loss_D.backward()
    gD = {n: p.grad.detach().cpu().double().clone() for n, p in D.netD.named_parameters()}
    gDf = {n: p.grad.detach().cpu().double().clone() for n, p in D.netD_f.named_parameters()}
    flow_ref, conf_ref = (t.cpu() for t in rec.calls[0])

    # ---- oracle on the CPU, same inputs, same previous frames, same reference flow
    leaf = lambda k: k.split('.')[-1] in ('weight', 'bias')
    sds = [{k: v.detach().cpu().clone().requires_grad_(v.dtype.is_floating_point and leaf(k))
            for k, v in getattr(G, 'netG%d' % s).state_dict().items()} for s in range(2)]
    sdD = {k: v.detach().cpu().clone().requires_grad_(leaf(k)) for k, v in D.netD.state_dict().items()}
    sdDf = {k: v.detach().cpu().clone().requires_grad_(leaf(k)) for k, v in D.netD_f.state_dict().items()}
    orc = GO.ModelGOracle(opt, sds)
    fake_B, raws, flows, weights, real_A, real_Bp, _ = orc.train_forward(a, b, None, prev_pyr, n_frames_load=1)
    real_B_prev, real_B = real_Bp[:, :-1], real_Bp[:, 1:]
    fake_B_prev = prev_pyr[0][:, -1:]
    m = lambda t: t.reshape(-1, *t.shape[2:])
    lo = FC.spatial_losses(sdD, sdDf, m(real_B), m(fake_B), m(raws), m(real_A), m(real_B_prev), m(fake_B_prev), m(flows), m(weights),
                           m(flow_ref), m(conf_ref), fine_size=opt.fineSize, lambda_F=opt.lambda_F, lambda_T=opt.lambda_T,
                           lambda_feat=opt.lambda_feat, n_scales_spatial=2, no_first_img=True, num_D=opt.num_D,
                           n_layers_D=opt.n_layers_D, norm=opt.norm)
    od = dict(zip(D.loss_names, [torch.mean(x) for x in lo]))
    for n in D.loss_names:
        ours, ref = float(ld[n]), float(od[n])
        print('%-13s ours %.6f oracle %.6f' % (n, ours, ref))
        assert abs(ours - ref) <= 2e-3 * max(1.0, abs(ref)), n
    oG = sum(od[k] for k in ('G_GAN', 'G_GAN_Feat', 'G_VGG', 'G_Warp', 'F_Flow', 'F_Warp', 'W', 'G_f_GAN', 'G_f_GAN_Feat'))
    oD = (od['D_fake'] + od['D_real']) * 0.5 + (od['D_f_fake'] + od['D_f_real']) * 0.5
    oG.backward(retain_graph=True)
    ref_gG = {'%d.%s' % (s, k): v.grad.double().clone() for s in range(2) for k, v in sds[s].items() if v.grad is not None}
    for v in list(sdD.values()) + list(sdDf.values()):
        v.grad = None
    oD.backward()
    _rel_check(gG, ref_gG, 'G', 0.15, 3e-2)
    _rel_check(gD, {k: v.grad.double() for k, v in sdD.items() if v.grad is not None}, 'D', 0.1, 2e-2)
    _rel_check(gDf, {k: v.grad.double() for k, v in sdDf.items() if v.grad is not None}, 'D_f', 0.1, 2e-2)


def test_pose_training_steps_update_netD_f_and_save_it(tmp_path):
    opt, G, D, flow, A, B = _pose_setup(seed=5)
    opt.checkpoints_dir = str(tmp_path)
    tr = Trainer(opt, G, D, flow, world=1)
    tG = opt.n_frames_G
    before = {n: p.detach().clone() for n, p in D.netD_f.named_parameters()}
    for i in range(6):
        a, b = A[:, i:i + tG].cuda(), B[:, i:i + tG].cuda()
        ld, ldT = tr.step(a, b, None)
        assert all(np.isfinite(v) for v in ld.values()), ld
        assert set(FC.FACE_LOSS_NAMES) <= set(ld)
        print('step %d: G_f_GAN %.4f D_f_real %.4f D_f_fake %.4f W %.4f temporal scales %d' % (
            i, ld['G_f_GAN'], ld['D_f_real'], ld['D_f_fake'], ld['W'], len(ldT)))
    moved = max((p.detach() - before[n]).abs().max().item() for n, p in D.netD_f.named_parameters())
    assert moved > 0
    flat = tr.grads.flat
    lo, hi = flat.data_ptr(), flat.data_ptr() + flat.numel() * flat.element_size()
    for n, p in D.netD_f.named_parameters():
        assert p.grad is not None and lo <= p.grad.data_ptr() < hi and p.grad._base is flat, n
    D.save('latest')
    path = os.path.join(str(tmp_path), opt.name, 'latest_net_D_f.pth')
    sd = torch.load(path)
    ref = json.load(open(os.path.join(GOLD_DIR, 'ref_face_keys.json')))
    assert [[k, list(v.shape)] for k, v in sd.items()] == ref

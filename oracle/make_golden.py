"""TEST INFRASTRUCTURE.  Generates tests/golden/*.npz by running the UNMODIFIED reference
(imported from /root/reference through oracle/ref_shim.py) on the seeded cases of
tests/cases.py.  Run in the build container:   python -m oracle.make_golden [case ...]

The fixtures are what pins oracle/generator_oracle.py and the CUDA path on the GPU box,
where the reference tree does not exist.
"""
import os
import sys

import numpy as np
import torch

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), '..'))
sys.path.insert(0, ROOT)
from oracle import ref_shim                                     # noqa: E402
sys.path.insert(0, os.path.join(ROOT, 'tests'))
import cases as C                                               # noqa: E402
from vid2vid_b200.utils import make_opt, det_fill_, synth_label_sequence   # noqa: E402

OUT = os.path.join(ROOT, 'tests', 'golden')


def _np(t):
    return t.detach().cpu().numpy().astype(np.float32)


def coarse_feats(c):
    g = torch.Generator().manual_seed(c['seed'] + 5)
    h2, w2, ngf = c['h'] // 2, c['w'] // 2, c['ngf']
    return (torch.randn(1, 2 * ngf, h2, w2, generator=g), torch.randn(1, 2 * ngf, h2, w2, generator=g),
            torch.randn(1, ngf, h2, w2, generator=g))


def run_case(name, c):
    N = ref_shim.networks()
    kind = c['kind']
    out = {}
    torch.manual_seed(0)
    if c.get('align_corners'):
        # original PyTorch-0.4 semantics (SURVEY App. B #2): force the flag the reference omits
        import torch.nn.functional as F
        orig = F.grid_sample
        F.grid_sample = lambda *a, **k: orig(*a, **{**k, 'align_corners': True})
    try:
        with torch.no_grad():
            if kind in ('composite', 'compositeLocal'):
                nc = 3 * (c['label_nc'] + 1)
                opt = make_opt(ngf=c['ngf'], n_blocks=c.get('n_blocks', 9), n_blocks_local=c.get('n_blocks_local', 3),
                               fg=c['fg'], no_flow=c.get('no_flow', False), n_downsample_G=c['nd'], gpu_ids=[])
                net = det_fill_(N.define_G(nc, 3, 6, c['ngf'], kind, c['nd'], 'batch', c.get('scale', 0), [], opt),
                                seed=c['seed'])
                inp, img_prev, mask = C.gen_inputs(c['label_nc'], c['h'], c['w'], c['seed'], block=c.get('block', 4))
                if kind == 'composite':
                    res = net(inp, img_prev, mask, None, None, None, False)
                else:
                    res = net(inp, img_prev, mask, *coarse_feats(c), False)
                ss = c.get('subsample', 1)
                for nme, t in zip(C.GEN_OUT_NAMES, res):
                    if t is None:
                        continue
                    if ss > 1 and t.shape[1] > 3:     # big feature maps: keep a strided sample + channel means
                        out[nme + '_sub'] = _np(t[:, :, ::ss, ::ss])
                        out[nme + '_cmean'] = _np(t.mean(dim=(2, 3)))
                    else:
                        out[nme] = _np(t)
            elif kind in ('global', 'local'):
                opt = make_opt(n_blocks=c['n_blocks'], n_blocks_local=c.get('n_blocks_local', 3), gpu_ids=[])
                net = det_fill_(N.define_G(c['input_nc'], 3, 0, c['ngf'], kind, c['nd'], 'instance', 0, [], opt),
                                seed=c['seed'])
                g = torch.Generator().manual_seed(c['seed'] + 1)
                lab = synth_label_sequence(1, c['h'], c['w'], label_nc=c['input_nc'], block=4, seed=c['seed'])
                x = torch.zeros(1, c['input_nc'], c['h'], c['w']).scatter_(1, lab[:, 0].long(), 1.0)
                out['out'] = _np(net(x))
            elif kind == 'D':
                net = det_fill_(N.define_D(c['input_nc'], c['ndf'], c['n_layers'], 'batch', c['num_D'], True, []),
                                seed=c['seed'])
                g = torch.Generator().manual_seed(c['seed'] + 1)
                x = torch.randn(c['batch'], c['input_nc'], c['h'], c['w'], generator=g)
                for i, tower in enumerate(net(x)):
                    for j, t in enumerate(tower):
                        out['t%d_l%d' % (i, j)] = _np(t)
            elif kind == 'inference':
                opt = C.inference_opt(c)
                single = det_fill_(N.define_G(c['label_nc'], 3, 0, 16, 'global', 2, 'instance', 0, [], opt),
                                   seed=c['seed'] + 100)
                m = ref_shim.make_model_G(opt, single)
                for s in range(c['n_scales']):
                    det_fill_(getattr(m, 'netG%d' % s), seed=c['seed'] + s)
                    C.condition_flow_heads(getattr(m, 'netG%d' % s), c['flow_weight_scale'])
                tG = opt.n_frames_G
                seq = synth_label_sequence(c['n_gen'] + tG - 1, c['h'], c['w'], label_nc=c['label_nc'], block=8,
                                           seed=c['seed'])
                for t in range(c['n_gen']):
                    A = seq[:, t:t + tG]
                    fake_B, real_A = m.inference(A, None, A)
                    out['fake_B_%d' % t] = _np(fake_B)
                for si in range(c['n_scales']):
                    out['prev_state_%d' % si] = _np(m.fake_B_prev[si])
            else:
                raise ValueError(kind)
    finally:
        if c.get('align_corners'):
            F.grid_sample = orig
    _save(name, out)


def dump_keys():
    """state_dict key / shape lists of the reference modules -> tests/golden/state_dict_keys.json."""
    import json
    N = ref_shim.networks()
    out = {}
    for name, c in C.KEY_CASES.items():
        kind = c['kind']
        if kind in ('composite', 'compositeLocal'):
            opt = make_opt(ngf=c['ngf'], n_blocks=c.get('n_blocks', 9), n_blocks_local=c.get('n_blocks_local', 3),
                           fg=c['fg'], no_flow=c.get('no_flow', False), n_downsample_G=c['nd'], gpu_ids=[])
            net = N.define_G(3 * (c['label_nc'] + 1), 3, 6, c['ngf'], kind, c['nd'], 'batch', c.get('scale', 0), [], opt)
        elif kind in ('global', 'local'):
            opt = make_opt(n_blocks=c['n_blocks'], n_blocks_local=c.get('n_blocks_local', 3), gpu_ids=[])
            net = N.define_G(c['input_nc'], 3, 0, c['ngf'], kind, c['nd'], 'instance', 0, [], opt)
        else:
            net = N.define_D(c['input_nc'], c['ndf'], c['n_layers'], 'batch', c['num_D'], True, [])
        out[name] = [[k, list(v.shape)] for k, v in net.state_dict().items()]
    with open(os.path.join(OUT, 'state_dict_keys.json'), 'w') as f:
        json.dump(out, f)
    print('state_dict_keys.json', {k: len(v) for k, v in out.items()})


def flownet2_golden():
    """Reference FlowNet2 (with the op stand-ins of ref_shim.install_flownet2_ops) and the FlowNet wrapper's
    compute_flow_and_conf on seeded inputs, with the deterministic weights of flownet2_oracle.det_state_dict ->
    tests/golden/flownet2_keys.json + flownet2_small.npz."""
    import json
    import types
    from oracle import flownet2_oracle as FO
    F2 = ref_shim.flownet2_class()
    net = F2().eval()
    keys = [[k, list(v.shape)] for k, v in net.state_dict().items()]
    with open(os.path.join(OUT, 'flownet2_keys.json'), 'w') as f:
        json.dump(keys, f)
    net.load_state_dict(FO.det_state_dict(keys, seed=7))
    g = torch.Generator().manual_seed(11)
    pair = torch.rand(1, 3, 2, 64, 128, generator=g)
    base = torch.rand(1, 3, 80, 64, generator=g)                    # height 80: exercises the resize-to-64 path
    im1, im2 = base, torch.roll(base, shifts=(1, 2), dims=(2, 3)) * 0.9 + 0.05
    from models.flownet import FlowNet                              # noqa (reference module)
    from models.flownet2_pytorch.networks.resample2d_package.resample2d import Resample2d   # noqa
    stub = types.SimpleNamespace(flowNet=net, resample=Resample2d())
    stub.norm = lambda t: FlowNet.norm(stub, t)
    with torch.no_grad():
        flow = net(pair)
        wflow, wconf = FlowNet.compute_flow_and_conf(stub, im1, im2)
    out = dict(pair=_np(pair), flow=_np(flow), im1=_np(im1), im2=_np(im2), wflow=_np(wflow), wconf=_np(wconf))
    path = os.path.join(OUT, 'flownet2_small.npz')
    np.savez_compressed(path, **out)
    print('flownet2_small %7.1f KB flow rms %.3f wflow rms %.3f conf mean %.3f' % (
        os.path.getsize(path) / 1024, float(flow.pow(2).mean().sqrt()), float(wflow.pow(2).mean().sqrt()), float(wconf.mean())))


def _put(out, prefix, ts):
    """Stores the non-None tensors of `ts` as prefix_<index> (a missing key stands for a None output)."""
    for i, t in enumerate(ts):
        if t is not None:
            out['%s_%d' % (prefix, i)] = _np(t)


def _save(name, out, limit=900 * 1024):
    """np.savez_compressed to tests/golden/<name>.npz, continued in <name>.1.npz, <name>.2.npz, ... so that no file is much
    larger than `limit` bytes (cases.load_golden reads the parts back as one dict)."""
    import io
    parts, size = [{}], 0
    for k, v in out.items():
        b = io.BytesIO()
        np.savez_compressed(b, v=v)
        if parts[-1] and size + len(b.getvalue()) > limit:
            parts.append({})
            size = 0
        parts[-1][k] = v
        size += len(b.getvalue())
    os.makedirs(OUT, exist_ok=True)
    for i, part in enumerate(parts):
        path = os.path.join(OUT, name + ('.%d' % i if i else '') + '.npz')
        np.savez_compressed(path, **part)
        print('%-16s %7.1f KB, %d arrays' % (os.path.basename(path), os.path.getsize(path) / 1024, len(part)))


def generator_pins():
    """The reference side of tests/test_oracle_vs_reference.py -> tests/golden/ref_pins.npz (generator / discriminator outputs,
    Vid2VidModelG inference), ref_train.npz (Vid2VidModelG training forward) and ref_grads.npz (parameter / input gradients
    of the coarse generator)."""
    N = ref_shim.networks()
    out = {}
    with torch.no_grad():
        for fg, no_flow, nd in C.PIN_COMPOSITE:
            opt = make_opt(ngf=8, n_blocks=3, fg=fg, no_flow=no_flow, n_downsample_G=nd, gpu_ids=[])
            net = det_fill_(N.define_G(18, 3, 6, 8, 'composite', nd, 'batch', 0, [], opt), seed=1)
            inp, img_prev, mask = C.pin_inputs(6, 16, 32)
            _put(out, 'composite_%d_%d_%d' % (fg, no_flow, nd), net(inp, img_prev, mask, None, None, None, False))

        opt = make_opt(ngf=8, n_blocks_local=2, fg=True, gpu_ids=[])
        net = det_fill_(N.define_G(18, 3, 6, 4, 'compositeLocal', 3, 'batch', 1, [], opt), seed=2)
        inp, img_prev, mask = C.pin_inputs(6, 16, 32)
        g = torch.Generator().manual_seed(5)
        c1, c2, c3 = (torch.randn(1, c, 8, 16, generator=g) for c in (8, 8, 4))
        _put(out, 'composite_local', net(inp, img_prev, mask, c1, c2, c3, False))

        opt = make_opt(n_blocks=2, n_blocks_local=2, gpu_ids=[])
        x = torch.rand(1, 5, 32, 64, generator=torch.Generator().manual_seed(3))
        out['global'] = _np(det_fill_(N.define_G(5, 3, 0, 8, 'global', 2, 'instance', 0, [], opt), seed=3)(x))
        out['local'] = _np(det_fill_(N.define_G(5, 3, 0, 4, 'local', 2, 'instance', 0, [], opt), seed=4)(x))

        net = det_fill_(N.define_D(9, 8, 3, 'batch', 2, True, []), seed=5)
        x = torch.randn(2, 9, 32, 48, generator=torch.Generator().manual_seed(6))
        for i, tower in enumerate(net(x)):
            _put(out, 'D_%d' % i, tower)

    opt = C.pin_inference_opt()
    single = det_fill_(N.define_G(5, 3, 0, 8, 'global', 2, 'instance', 0, [], opt), seed=9)
    m = ref_shim.make_model_G(opt, single)
    det_fill_(m.netG0, seed=10)
    det_fill_(m.netG1, seed=11)
    seq = synth_label_sequence(5, 32, 64, label_nc=5, block=4, seed=3)
    for t in range(3):
        A = seq[:, t:t + 3]
        _put(out, 'infer_%d' % t, m.inference(A, None, A))
    _save('ref_pins', out)

    out = {}
    for no_first_img in (False, True):
        opt = C.pin_train_opt(no_first_img)
        m = ref_shim.make_model_G(opt)
        assert m.n_frames_load == 2
        det_fill_(m.netG0, seed=20)
        det_fill_(m.netG1, seed=21)
        C.condition_flow_heads(m.netG0, 0.05)
        C.condition_flow_heads(m.netG1, 0.05)
        seq, real = C.pin_train_clip(opt)
        prev = None
        for call in range(2):
            sl = slice(call * 2, call * 2 + 2 + opt.n_frames_G - 1)
            with torch.no_grad():
                r = m.forward(seq[:, sl].contiguous(), real[:, sl].contiguous(), seq[:, sl].contiguous(), prev)
            # real_B is the input clip from frame tG - 2 on: checked here, not stored
            assert torch.equal(r[5], real[:, sl][:, opt.n_frames_G - 2:])
            _put(out, 'train_%d_%d' % (no_first_img, call), r[:5])
            _put(out, 'train_%d_%d_prev' % (no_first_img, call), r[6])
            prev = r[6]
    _save('ref_train', out)

    out = {}
    opt = make_opt(ngf=8, n_blocks=2, fg=True, n_downsample_G=2, gpu_ids=[])
    net = det_fill_(N.define_G(18, 3, 6, 8, 'composite', 2, 'batch', 0, [], opt), seed=31)
    C.condition_flow_heads(net, 0.05)
    inp, img_prev, mask = C.pin_inputs(6, 16, 32, seed=2)
    x, p = inp.clone().requires_grad_(True), img_prev.clone().requires_grad_(True)
    res = net(x, p, mask, None, None, None, False)
    C.pin_objective(res).backward()
    for k, v in net.named_parameters():
        out['grad.' + k] = _np(v.grad)
    out['grad_input'], out['grad_img_prev'] = _np(x.grad), _np(p.grad)
    _save('ref_grads', out)


def loss_pins():
    """The reference Vid2VidModelD.forward (spatial and temporal losses, --no_vgg) on the seeded inputs of
    tests/test_losses_oracle.py, discriminators filled by det_fill_ -> tests/golden/ref_losses.npz."""
    ref_shim.install()
    from models.vid2vid_model_D import Vid2VidModelD          # noqa (reference module)
    out = {}
    for key, kw in (('spatial_0', dict(n_scales_spatial=2, no_first_img=False)), ('spatial_1', dict(n_scales_spatial=2, no_first_img=True)),
                    ('temporal', {})):
        opt = C.pin_loss_opt(**kw)
        m = Vid2VidModelD()
        m.initialize(opt)
        det_fill_(m.netD, seed=C.PIN_SEED_D)
        det_fill_(m.netD_T0, seed=C.PIN_SEED_D_T)
        with torch.no_grad():
            if key == 'temporal':
                ref = m.forward(1, C.pin_temporal_loss_inputs(opt))
            else:
                ref = m.forward(0, C.pin_spatial_loss_inputs(with_raw=not opt.no_first_img))
        _put(out, key, ref)
    _save('ref_losses', out)


def flownet2_pins():
    """The reference FlowNet2 at batch 2, its four sub-networks on their own inputs and the FlowNet wrapper at 64x64 and
    70x64, with the deterministic weights of flownet2_oracle.det_state_dict(seed=3) -> tests/golden/flownet2_pins.npz."""
    import json
    import types
    from oracle import flownet2_oracle as FO
    F2 = ref_shim.flownet2_class()
    keys = json.load(open(os.path.join(OUT, 'flownet2_keys.json')))
    net = F2().eval()
    net.load_state_dict(FO.det_state_dict(keys, seed=3))
    from models.flownet import FlowNet                                                        # noqa (reference module)
    from models.flownet2_pytorch.networks.resample2d_package.resample2d import Resample2d     # noqa
    stub = types.SimpleNamespace(flowNet=net, resample=Resample2d())
    stub.norm = lambda t: FlowNet.norm(stub, t)
    i = C.flownet2_pin_inputs()
    out = {}
    with torch.no_grad():
        out['flow'] = _np(net(i['pair']))
        out['flownetc'] = _np(net.flownetc(i['x6'])[0])
        out['flownets_1'] = _np(net.flownets_1(i['x12'])[0])
        out['flownets_d'] = _np(net.flownets_d(i['x6'])[0])
        out['flownetfusion'] = _np(net.flownetfusion(i['xf']))
        for h, w in C.FLOWNET2_PIN_SIZES:
            rf, rc = FlowNet.compute_flow_and_conf(stub, i['im1_%d' % h], i['im2_%d' % h])
            out['wflow_%d' % h], out['wconf_%d' % h] = _np(rf), _np(rc)
    _save('flownet2_pins', out)


def schedule_pins():
    """The reference BaseModel's learning-rate / training-batch schedules and save_network file on the state of
    tests/test_host_schedule.py -> tests/golden/base_model_schedule.json."""
    import json
    import tempfile
    import types
    import torch.nn as nn
    ref_shim.install()
    from models.base_model import BaseModel                     # noqa (reference module)
    with tempfile.TemporaryDirectory() as tmp:
        opt = types.SimpleNamespace(**C.SCHEDULE_OPT, checkpoints_dir=tmp)
        m = BaseModel()
        m.opt, m.old_lr, m.n_scales = opt, opt.lr, 2
        m.netG0, m.netG1 = nn.Linear(3, 2), nn.Linear(2, 2)
        m.optimizer_G = torch.optim.Adam(list(m.netG1.parameters()), lr=opt.lr, betas=(opt.beta1, 0.999))
        m.n_gpus, m.n_frames_per_gpu, m.n_frames_load, m.n_frames_bp = 1, 1, 1, 1
        m.finetune_all = False
        m.save_dir = os.path.join(tmp, opt.name)
        os.makedirs(m.save_dir)
        out = {'lr': [], 'batch': []}
        for epoch in C.SCHEDULE_EPOCHS:
            m.update_learning_rate(epoch, 'G')
            out['lr'].append([m.old_lr, [g['lr'] for g in m.optimizer_G.param_groups]])
        for ratio in C.SCHEDULE_RATIOS:
            m.update_training_batch(ratio)
            out['batch'].append([m.n_frames_bp, m.n_frames_per_gpu, m.n_frames_load])
        m.update_fixed_params()
        out['finetune_all'] = m.finetune_all
        out['n_params_G'] = sum(p.numel() for g in m.optimizer_G.param_groups for p in g['params'])
        out['lr_after_fix'] = m.optimizer_G.param_groups[0]['lr']
        m.save_network(m.netG1, 'G1', 'latest', [])
        files = os.listdir(m.save_dir)
        out['saved_files'] = files
        out['saved_keys'] = list(torch.load(os.path.join(m.save_dir, files[0])))
    with open(os.path.join(OUT, 'base_model_schedule.json'), 'w') as f:
        json.dump(out, f, indent=1)
    print('base_model_schedule.json', out)


PINS = {'pins': generator_pins, 'losses': loss_pins, 'flownet2_pins': flownet2_pins, 'schedule': schedule_pins}

if __name__ == '__main__':
    names = sys.argv[1:] or (list(C.CASES) + ['keys'] + list(PINS))
    for n in names:
        if n == 'keys':
            dump_keys()
        elif n == 'flownet2':
            flownet2_golden()
        elif n in PINS:
            PINS[n]()
        else:
            run_case(n, C.CASES[n])

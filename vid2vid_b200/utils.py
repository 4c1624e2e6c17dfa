"""Small host-side helpers shared by the modules, the tests and bench.py.

Nothing here touches the GPU.  `make_opt` mirrors the argparse namespace the
reference builds in options/base_options.py:11-128 + options/test_options.py:4-15
(only the fields the generator / discriminator hot path reads).
"""
import zlib
from types import SimpleNamespace

import torch


def make_opt(**kw):
    """Option namespace with the reference's defaults (options/base_options.py:14-84)."""
    opt = SimpleNamespace(
        # base_options.py:14-20
        dataroot='datasets/Cityscapes/', batchSize=1, loadSize=512, fineSize=512,
        input_nc=3, label_nc=0, output_nc=3,
        # base_options.py:22-26
        netG='composite', ngf=128, ndf=64, n_blocks=9, n_downsample_G=3,
        gpu_ids=[0], n_gpus_gen=1, name='synthetic', dataset_mode='temporal',
        checkpoints_dir='./checkpoints', norm='batch',
        # base_options.py:43-59
        use_instance=False, label_feat=False, feat_num=3, n_blocks_local=3,
        n_local_enhancers=1, n_frames_G=3, n_scales_spatial=1, no_first_img=False,
        use_single_G=False, fg=False, fg_labels=[26], no_flow=False,
        openpose_only=False, densepose_only=False, add_face_disc=False,
        load_pretrain='', debug=True, fp16=False,
        # test_options.py
        which_epoch='latest', use_real_img=False, isTrain=False,
        # train_options.py (subset read by Vid2VidModelD)
        num_D=2, n_layers_D=3, n_frames_D=3, n_scales_temporal=3, no_ganFeat=False,
        no_vgg=True, lambda_feat=10.0, lambda_F=10.0, lambda_T=10.0,
        gan_mode='ls', continue_train=False, niter_fix_global=0, lr=0.0002,
        beta1=0.5, TTUR=False, max_frames_per_gpu=1, n_frames_total=30,
        max_frames_backpropagate=1,
        # not a reference option: random-initialised networks (no checkpoints exist offline); False = the reference's behaviour
        synthetic_weights=True,
    )
    for k, v in kw.items():
        setattr(opt, k, v)
    return opt


def det_fill_(module, seed=0):
    """Fill every parameter/buffer of `module` with values that depend only on
    (seed, tensor name, shape) -- not on construction order or RNG history -- so the
    reference modules (oracle side) and ours can be given identical random weights.

    Distributions follow the reference's initialiser (models/networks.py:15-21):
    conv weights N(0, 0.02), norm gamma N(1, 0.02); biases get small non-zero values
    so that affine shifts are exercised.
    """
    sd = module.state_dict()
    with torch.no_grad():
        for name, t in sd.items():
            g = torch.Generator().manual_seed((seed * 1000003 + zlib.crc32(name.encode())) & 0x7FFFFFFF)
            leaf = name.rsplit('.', 1)[-1]
            if leaf == 'num_batches_tracked':
                t.zero_()
            elif leaf == 'running_mean':
                t.zero_()
            elif leaf == 'running_var':
                t.fill_(1.0)
            elif t.dim() >= 2:
                t.copy_(torch.randn(t.shape, generator=g) * 0.02)
            elif leaf == 'weight':          # norm gamma
                t.copy_(1.0 + torch.randn(t.shape, generator=g) * 0.02)
            else:                           # conv bias / norm beta
                t.copy_(torch.randn(t.shape, generator=g) * 0.05)
    return module


def synth_label_sequence(n_frames, H, W, label_nc=35, block=8, seed=0, drift=1):
    """Blocky synthetic label maps (SURVEY 8d): ids U{0..label_nc-1} on a coarse grid,
    nearest-upsampled by `block`, shifted by `drift` coarse cells per frame so consecutive
    frames differ.  Returns float tensor (1, n_frames, 1, H, W) of label ids (the
    reference feeds label ids as floats, data/test_dataset.py / vid2vid_model_G.py:95)."""
    g = torch.Generator().manual_seed(seed)
    gh, gw = (H + block - 1) // block, (W + block - 1) // block
    base = torch.randint(0, label_nc, (gh, gw + drift * n_frames), generator=g)
    frames = []
    for t in range(n_frames):
        m = base[:, t * drift: t * drift + gw]
        m = m.repeat_interleave(block, 0).repeat_interleave(block, 1)[:H, :W]
        frames.append(m)
    return torch.stack(frames).float().view(1, n_frames, 1, H, W)


def synth_pose_sequence(n_frames, H, W, seed=0, block=8, face=True, openpose=False, face_size=6, face_yx=None, drift=1):
    """Synthetic pose-style input clip (label_nc 0, input_nc 6): U(-1,1) blobs on a zero background -- each coarse cell of a
    block-pixel grid carries one with probability 0.3, drifting `drift` cells per frame -- plus a `face_size`-pixel "face"
    patch drifting one pixel per frame from `face_yx` (default: a seeded interior position).  The face is channel 2 = 0.95,
    or with `openpose` the openpose face colour (0.2, -1, -0.6) in channels 0-2; these are what the face detector of
    Vid2VidModelD.get_face_region looks for, so blob values in channel 2 are capped at 0.85 to keep them out of it.
    Returns float tensor (1, n_frames, 6, H, W)."""
    g = torch.Generator().manual_seed(seed)
    gh, gw = (H + block - 1) // block, (W + block - 1) // block
    vals = torch.rand(6, gh, gw + drift * n_frames, generator=g) * 2 - 1
    vals = vals * (torch.rand(1, gh, gw + drift * n_frames, generator=g) < 0.3).float()
    vals[2].clamp_(max=0.85)
    if face_yx is None:
        face_yx = (int(torch.randint(0, max(1, H - face_size - n_frames), (1,), generator=g)),
                   int(torch.randint(0, max(1, W - face_size - n_frames), (1,), generator=g)))
    colour = (0.2, -1.0, -0.6) if openpose else (None, None, 0.95)
    frames = []
    for t in range(n_frames):
        f = vals[:, :, t * drift: t * drift + gw].repeat_interleave(block, 1).repeat_interleave(block, 2)[:, :H, :W].clone()
        if face:
            y0, x0 = min(face_yx[0] + t, H - face_size), min(face_yx[1] + t, W - face_size)
            for c, v in enumerate(colour):
                if v is not None:
                    f[c, y0:y0 + face_size, x0:x0 + face_size] = v
        frames.append(f)
    return torch.stack(frames).view(1, n_frames, 6, H, W)

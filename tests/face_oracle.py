"""TEST INFRASTRUCTURE.  CPU restatement of the face discriminator of the pose training step (Vid2VidModelD with
--add_face_disc, models/vid2vid_model_D.py:38-40,148-158,215-230,253-255) on top of oracle/losses_oracle.py, and the seeded
cases its reference fixtures are made from (tests/golden/ref_face*.npz, written by `python tools/make_face_golden.py`).
Pinned against those fixtures in tests/test_face_oracle.py; the GPU tests compare the CUDA path with it."""
import torch

from oracle import generator_oracle as GO
from oracle import losses_oracle as LO
from vid2vid_b200.utils import make_opt, synth_pose_sequence

FACE_LOSS_NAMES = ['G_f_GAN', 'G_f_GAN_Feat', 'D_f_real', 'D_f_fake']
SPATIAL_LOSS_NAMES = ['G_VGG', 'G_GAN', 'G_GAN_Feat', 'D_real', 'D_fake', 'G_Warp', 'F_Flow', 'F_Warp', 'W'] + FACE_LOSS_NAMES
FACE_WEIGHT = 2                     # vid2vid_model_D.py:149


def face_region(real_A, fine_size, openpose_only=False):
    """get_face_region: the bounding box of the face pixels over all images of real_A (N, C, H, W), its centre clamped so a
    window of fine_size // 32 * 8 pixels fits -- up to the reference's `h - 1`, which leaves a window clamped to the bottom or
    right edge one pixel short of the frame.  Returns (ys, ye, xs, xe) or None when there is no face pixel."""
    _, _, h, w = real_A.shape
    c0, c1, c2 = real_A[:, 0], real_A[:, 1], real_A[:, 2]
    if openpose_only:
        face = (c0 > 0.19) & (c0 < 0.21) & (c1 < -0.99) & (c2 > -0.61) & (c2 < -0.59)
    else:
        face = c2 > 0.9
    idx = face.nonzero()
    if idx.shape[0] == 0:
        return None
    half = fine_size // 32 * 8 // 2
    ys, ye = int(idx[:, 1].min()), int(idx[:, 1].max())
    xs, xe = int(idx[:, 2].min()), int(idx[:, 2].max())
    yc = max(half, min(h - 1 - half, (ys + ye) // 2))
    xc = max(half, min(w - 1 - half, (xs + xe) // 2))
    return yc - half, yc + half, xc - half, xc + half


def face_losses(sd_D_f, real_A, real_B, fake_B, *, fine_size, openpose_only=False, num_D=2, n_layers_D=3, norm='batch',
                lambda_feat=10.0, no_ganFeat=False):
    """[G_f_GAN, G_f_GAN_Feat, D_f_real, D_f_fake] (each a 0-dim tensor) and the window, or None for both when no face is
    found.  netD_f has max(1, num_D - 2) towers; feature matching still weights by 1 / num_D (GAN_and_FM_loss reads
    opt.num_D)."""
    win = face_region(real_A, fine_size, openpose_only)
    if win is None:
        return None, None
    ys, ye, xs, xe = win
    crop = lambda t: t[:, :, ys:ye, xs:xe]
    d = dict(num_D=max(1, num_D - 2), n_layers=n_layers_D, norm=norm, getIntermFeat=True)
    pred_real = GO.multiscale_discriminator(sd_D_f, torch.cat((crop(real_A), crop(real_B)), 1), **d)
    pred_fake = GO.multiscale_discriminator(sd_D_f, torch.cat((crop(real_A), crop(fake_B)), 1), **d)
    g_gan, g_fm = LO.gan_and_fm_loss(pred_real, pred_fake, n_layers_D=n_layers_D, num_D=num_D, lambda_feat=lambda_feat,
                                     no_ganFeat=no_ganFeat)
    return [g_gan * FACE_WEIGHT, g_fm * FACE_WEIGHT, LO.gan_loss(pred_real, True), LO.gan_loss(pred_fake, False)], win


def spatial_losses(sd_D, sd_D_f, real_B, fake_B, fake_B_raw, real_A, real_B_prev, fake_B_prev, flow, weight, flow_ref, conf_ref, *,
                   fine_size, openpose_only=False, **kw):
    """Vid2VidModelD.forward(0, ...) with --add_face_disc: losses_oracle.spatial_losses' nine terms followed by the four face
    terms (zeros_like(D_real) when there is no face), each (1, 1) -- the reference's 13-entry loss list."""
    base = LO.spatial_losses(sd_D, real_B, fake_B, fake_B_raw, real_A, real_B_prev, fake_B_prev, flow, weight, flow_ref, conf_ref,
                             **kw)
    keep = {k: kw[k] for k in ('num_D', 'n_layers_D', 'norm', 'lambda_feat', 'no_ganFeat') if k in kw}
    face, _ = face_losses(sd_D_f, real_A, real_B, fake_B, fine_size=fine_size, openpose_only=openpose_only, **keep)
    if face is None:
        face = [torch.zeros_like(base[3])] * 4
    return base + [t.reshape(-1, 1) for t in face]


# ------------------------------------------------------------------------------------------------ pinned cases
# det_fill_ seeds of netD / netD_f of the face pins
FACE_SEED_D, FACE_SEED_D_F = 60, 61
FACE_H, FACE_W = 64, 96
FACE_FINE = 128                     # a 32x32 window

# name -> (per-image face top-left (y, x) or None for an image without a face, openpose colour)
FACE_CASES = {
    'interior': ([(20, 40), (22, 43)], False),
    'top': ([(0, 40), (1, 44)], False),
    'bottom': ([(FACE_H - 6, 30), (FACE_H - 7, 33)], False),
    'left': ([(25, 0), (28, 1)], False),
    'right': ([(25, FACE_W - 6), (30, FACE_W - 7)], False),
    'one_of_two': ([None, (30, 50)], False),
    'none': ([None, None], False),
    'openpose': ([(14, 60), (18, 66)], True),
}


def face_opt(openpose_only=False, **kw):
    """Options of the face pins: the pose configuration (label_nc 0, input_nc 6) with --add_face_disc, three image-D towers
    (so netD_f has one) and a 32-pixel face window."""
    opt = make_opt(label_nc=0, input_nc=6, use_instance=False, isTrain=True, gpu_ids=[0], n_gpus_gen=1, no_vgg=True, ndf=16,
                   num_D=3, fineSize=FACE_FINE, add_face_disc=True, openpose_only=openpose_only, no_first_img=True, **kw)
    opt.debug = True
    opt.load_pretrain = ''
    return opt


def face_case_real_A(name):
    """real_A (2, 6, H, W) of a pinned case: one synthetic pose frame per image."""
    faces, openpose = FACE_CASES[name]
    imgs = []
    for i, yx in enumerate(faces):
        seq = synth_pose_sequence(1, FACE_H, FACE_W, seed=100 + i, face=yx is not None, openpose=openpose, face_yx=yx)
        imgs.append(seq[0, 0])
    return torch.stack(imgs)


def face_case_inputs(name):
    """tensors_list of Vid2VidModelD.forward(0, ...) for a pinned case: real_B, fake_B, fake_B_raw, real_A, real_B_prev,
    fake_B_prev, flow, weight, flow_ref, conf_ref."""
    g = torch.Generator().manual_seed(7)
    n, h, w = 2, FACE_H, FACE_W
    rnd = lambda c, lo=-1.0, hi=1.0: torch.rand((n, c, h, w), generator=g) * (hi - lo) + lo
    real_B, fake_B, fake_B_raw, real_B_prev, fake_B_prev = (rnd(3) for _ in range(5))
    flow, flow_ref = rnd(2, -3, 3), rnd(2, -3, 3)
    weight = rnd(1, 0, 1)
    conf = (rnd(1) > 0).float()
    return [real_B, fake_B, fake_B_raw, face_case_real_A(name), real_B_prev, fake_B_prev, flow, weight, flow_ref, conf]

"""Times the pose2body training step (BASELINE config 5: scripts/pose/train_512p.sh at H512 x W256 on one GPU, one clip per step)
with and without --add_face_disc, and the face discriminator's own pieces:
  * ms per step of both configurations, measured in alternating blocks of K steps (CUDA events, synchronised at block ends);
  * netD_f forward + backward: the three netD_f passes of compute_loss_D on a 128x128 face window and their backward;
  * the face_window kernel on the step's real_A;
  * the host time Vid2VidModelD spends waiting for the window event (the read of `found`).
    python tools/time_train_pose.py [out.json]      (prints the JSON result, and also writes it to out.json when given)"""
import json
import os
import subprocess
import sys
import time

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), '..'))
sys.path.insert(0, ROOT)
import torch                                                            # noqa: E402

from vid2vid_b200 import flownet as FN                                  # noqa: E402
from vid2vid_b200 import ops                                            # noqa: E402
from vid2vid_b200.model_d import Vid2VidModelD                          # noqa: E402
from vid2vid_b200.model_g import Vid2VidModelG                          # noqa: E402
from vid2vid_b200.trainer import Trainer                                # noqa: E402
from vid2vid_b200.utils import make_opt, synth_pose_sequence            # noqa: E402

H, W = 512, 256
K, ROUNDS = int(os.environ.get('POSE_STEPS', '8')), int(os.environ.get('POSE_ROUNDS', '4'))


def build(face):
    opt = make_opt(label_nc=0, input_nc=6, n_scales_spatial=2, num_D=3, fineSize=512, loadSize=768, no_first_img=True, fg=True,
                   fg_labels=[2], add_face_disc=face, isTrain=True, no_vgg=True, gpu_ids=[0], n_frames_total=12, lr=0.0001,
                   dataroot='datasets/pose')
    torch.manual_seed(1234)
    G = Vid2VidModelG().initialize(opt)
    D = Vid2VidModelD().initialize(opt)
    F = FN.FlowNet().initialize(opt)
    return opt, Trainer(opt, G, D, F, world=1)


def main():
    out_path = sys.argv[1] if len(sys.argv) > 1 else None
    torch.cuda.set_device(0)
    arms = {'no_face': build(False), 'face': build(True)}
    opt = arms['face'][0]
    tG = opt.n_frames_G
    # warm-up reaches the steady state: every temporal scale active (tD**s * (tD - 1) + 1 frames for scale s)
    warm = opt.n_frames_D ** (opt.n_scales_temporal - 1) * (opt.n_frames_D - 1) + 3
    T = warm + ROUNDS * K + tG + 2
    A = synth_pose_sequence(T, H, W, seed=0, block=32, face_size=24).cuda()
    g = torch.Generator().manual_seed(77)
    coarse = torch.rand(T, 3, H // 16, W // 16, generator=g) * 2 - 1
    B = torch.nn.functional.interpolate(coarse, size=(H, W), mode='bilinear', align_corners=False).view(1, T, 3, H, W).cuda()
    pos = {k: 0 for k in arms}

    def steps(k, n, waits=None):
        """n steps issued back to back (the loss values are read once, after the last one)."""
        tr = arms[k][1]
        for _ in range(n):
            t = pos[k]
            pend = tr.step_async(A[:, t:t + tG], B[:, t:t + tG], None)
            pos[k] += 1
            if waits is not None and tr.modelD.add_face_disc:
                waits.append(tr.modelD.face_wait_s * 1e3)
        return pend.get()

    for k in arms:
        ld, ldT = steps(k, warm)
        print('%-8s warm-up done: %d temporal scales active, losses %s' % (k, len(ldT), sorted(ld)))
    times = {k: [] for k in arms}
    waits = []
    for r in range(ROUNDS):
        for k in (('no_face', 'face') if r % 2 == 0 else ('face', 'no_face')):
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            ld, _ = steps(k, K, waits)
            e1.record()
            torch.cuda.synchronize()
            times[k].append(e0.elapsed_time(e1) / K)
            assert all(v == v for v in ld.values()), ld
    res = {'workload': 'pose2body training step, H512 x W256, input_nc 6, n_scales_spatial 2, num_D 3, n_scales_temporal %d, '
                       '--no_first_img --fg --fg_labels 2, fineSize 512 (128x128 face window), one clip, ngf %d, ndf %d'
                       % (opt.n_scales_temporal, opt.ngf, opt.ndf),
           'steps_per_block': K, 'blocks': ROUNDS}
    for k in arms:
        v = sorted(times[k])
        res['step_ms_%s' % k] = {'median': v[len(v) // 2], 'min': v[0], 'max': v[-1], 'blocks': times[k]}
    res['face_overhead_pct'] = 100 * (res['step_ms_face']['median'] / res['step_ms_no_face']['median'] - 1)
    w = sorted(waits)
    res['host_wait_ms_face_window_event'] = {'median': w[len(w) // 2], 'max': w[-1], 'n': len(w)}

    # the face discriminator on its own: three netD_f passes on the window (compute_loss_D) + the backward of both losses
    D = arms['face'][1].modelD
    t = pos['face']
    real_A = A[0, t + tG - 1:t + tG].contiguous()
    real_B = B[0, t + tG - 1:t + tG].contiguous()
    fake_B = (real_B * 0.9).requires_grad_(True)
    win = ops.face_window(real_A, opt.fineSize, False)
    assert int(win[0]) == 1

    def dface():
        d_real, d_fake, g_gan, g_fm = D.compute_loss_D_face(real_A, real_B, fake_B, win)
        (g_gan + g_fm + (d_real + d_fake) * 0.5).backward()
    n = 20
    for _ in range(3):
        dface()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n):
        dface()
    e1.record()
    torch.cuda.synchronize()
    res['netD_f_fwd_bwd_ms'] = e0.elapsed_time(e1) / n

    buf = ops.face_window_buffer(real_A.device)
    for _ in range(10):
        ops.face_window(real_A, opt.fineSize, False, buf=buf)
    n = 1000
    torch.cuda.synchronize()
    e0.record()
    for _ in range(n):
        ops.face_window(real_A, opt.fineSize, False, buf=buf)
    e1.record()
    torch.cuda.synchronize()
    res['face_window_kernel_us'] = e0.elapsed_time(e1) / n * 1e3
    res['face_window_note'] = 'back-to-back launches on a (1, 6, 512, 256) real_A (3.1 MB, L2-resident after the first)'

    res['device'] = torch.cuda.get_device_name(0)
    try:
        res['nvidia_smi'] = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                                           capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError) as e:
        res['nvidia_smi'] = 'unavailable: %s' % e
    res['date'] = time.strftime('%Y-%m-%d')
    if out_path:
        os.makedirs(os.path.dirname(os.path.abspath(out_path)), exist_ok=True)
        with open(out_path, 'w') as f:
            json.dump(res, f, indent=1)
    print(json.dumps(res, indent=1))


if __name__ == '__main__':
    main()

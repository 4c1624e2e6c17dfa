"""Vid2VidModelD on the B200 engine: the discriminator-side model of the training step (models/vid2vid_model_D.py:13-272)
with the same initialize(opt) / forward(scale_T, tensors_list) / get_losses / loss_names / save, the towers running through
the plan runtime (forward on tcgen05, hand-written backward kernels) and every loss term through libv2v_b200.so (masked L1,
LSGAN, feature matching, the two resample warps).  With --add_face_disc (the pose scripts at 512p and above) a face
discriminator netD_f sees a fixed window around the face pixels of real_A: the window is found on the device
(ops.face_window) and cropped there (ops.crop_concat), and the host reads back only whether a face exists.  The VGG
perceptual term needs downloaded weights and is outside the hot path (DESIGN.md section 5): `--no_vgg` is required, as in
the oracle and the reference pin."""
import time

import torch
import torch.nn as nn

from .base_model import HostScheduleMixin
from . import networks, ops


def _adam(params, **kw):
    """torch.optim.Adam as the reference builds it; on CUDA parameters the fused multi-tensor implementation (same arithmetic,
    a few dozen launches for ~1000 parameter tensors instead of several hundred)."""
    params = list(params)
    if params and all(p.is_cuda for p in params):
        try:
            return torch.optim.Adam(params, fused=True, **kw)
        except (TypeError, RuntimeError):
            pass
    return torch.optim.Adam(params, **kw)


class Vid2VidModelD(HostScheduleMixin, nn.Module):
    def name(self):
        return 'Vid2VidModelD'

    def initialize(self, opt):
        """vid2vid_model_D.py:17-91."""
        self.opt = opt
        self.isTrain = opt.isTrain
        self.gpu_ids = opt.gpu_ids
        self.tD = opt.n_frames_D
        self.output_nc = opt.output_nc
        if not opt.no_vgg:
            raise NotImplementedError('VGG loss needs downloaded weights; run with --no_vgg (DESIGN.md section 5)')
        dev = torch.device('cuda', self.gpu_ids[0] if len(self.gpu_ids) else torch.cuda.current_device())
        self.device_ = dev
        self.input_nc = (opt.label_nc if opt.label_nc != 0 else opt.input_nc) + (1 if opt.use_instance else 0)
        self.netD = networks.define_D(self.input_nc + opt.output_nc, opt.ndf, opt.n_layers_D, opt.norm, opt.num_D,
                                      not opt.no_ganFeat, []).to(dev)
        self.add_face_disc = bool(getattr(opt, 'add_face_disc', False))
        if self.add_face_disc:                                                                          # :38-40
            self.netD_f = networks.define_D(self.input_nc + opt.output_nc, opt.ndf, opt.n_layers_D, opt.norm,
                                            max(1, opt.num_D - 2), not opt.no_ganFeat, []).to(dev)
            self._face_buf = ops.face_window_buffer(dev)
            self._face_host = torch.zeros(5, dtype=torch.int32, pin_memory=True)
            self._face_event = torch.cuda.Event()
            self.face_wait_s = 0.0          # host time spent in the last wait for the face window (tools/time_train_pose.py)
        nc_t = opt.output_nc * opt.n_frames_D + 2 * (opt.n_frames_D - 1)
        for s in range(opt.n_scales_temporal):
            setattr(self, 'netD_T' + str(s), networks.define_D(nc_t, opt.ndf, opt.n_layers_D, opt.norm, opt.num_D,
                                                                not opt.no_ganFeat, []).to(dev))
        self.old_lr = opt.lr
        self.loss_names = ['G_VGG', 'G_GAN', 'G_GAN_Feat', 'D_real', 'D_fake', 'G_Warp', 'F_Flow', 'F_Warp', 'W']
        self.loss_names_T = ['G_T_GAN', 'G_T_GAN_Feat', 'D_T_real', 'D_T_fake', 'G_T_Warp']
        if self.add_face_disc:
            self.loss_names += ['G_f_GAN', 'G_f_GAN_Feat', 'D_f_real', 'D_f_fake']                             # :73-74
        beta1, beta2, lr = (0, 0.9, opt.lr * 2) if opt.TTUR else (opt.beta1, 0.999, opt.lr)        # :78-84
        params_D = list(self.netD.parameters()) + (list(self.netD_f.parameters()) if self.add_face_disc else [])
        self.optimizer_D = _adam(params_D, lr=lr, betas=(beta1, beta2))
        for s in range(opt.n_scales_temporal):
            setattr(self, 'optimizer_D_T' + str(s), _adam(list(getattr(self, 'netD_T' + str(s)).parameters()), lr=opt.lr,
                                                                       betas=(opt.beta1, 0.999)))
        return self

    # ------------------------------------------------------------------ criteria (models/networks.py:731-812)
    @staticmethod
    def criterionGAN(preds, target_is_real):
        """GANLoss.__call__ with use_lsgan (networks.py:764-774): sum over towers of MSE(last output, 1 or 0)."""
        label = 1.0 if target_is_real else 0.0
        total = 0
        for tower in preds:
            total = total + ops.mse_to_const(tower[-1], label)
        return total

    def resample(self, image, flow):
        """BaseModel.resample (base_model.py:189-196)."""
        return ops.resample(image, flow, align_corners=networks._Planned.align_corners)

    def GAN_and_FM_loss(self, pred_real, pred_fake):
        """vid2vid_model_D.py:199-213."""
        loss_G_GAN = self.criterionGAN(pred_fake, True)
        loss_G_GAN_Feat = torch.zeros_like(loss_G_GAN)
        if not self.opt.no_ganFeat:
            w = (4.0 / (self.opt.n_layers_D + 1)) * (1.0 / self.opt.num_D) * self.opt.lambda_feat
            for i in range(min(len(pred_fake), self.opt.num_D)):
                for j in range(len(pred_fake[i]) - 1):
                    loss_G_GAN_Feat = loss_G_GAN_Feat + w * ops.l1_loss(pred_fake[i][j], pred_real[i][j].detach())
        return loss_G_GAN, loss_G_GAN_Feat

    def compute_loss_D(self, netD, real_A, real_B, fake_B):
        """vid2vid_model_D.py:166-177."""
        real_AB = torch.cat((real_A, real_B), dim=1) if real_A is not None else real_B
        fake_AB = torch.cat((real_A, fake_B), dim=1) if real_A is not None else fake_B
        return self._loss_D_on(netD, real_AB, fake_AB)

    def _loss_D_on(self, netD, real_AB, fake_AB):
        pred_real = netD.forward(real_AB)
        pred_fake = netD.forward(fake_AB.detach())
        loss_D_real = self.criterionGAN(pred_real, True)
        loss_D_fake = self.criterionGAN(pred_fake, False)
        pred_fake = netD.forward(fake_AB)
        loss_G_GAN, loss_G_GAN_Feat = self.GAN_and_FM_loss(pred_real, pred_fake)
        return loss_D_real, loss_D_fake, loss_G_GAN, loss_G_GAN_Feat

    def compute_loss_D_T(self, real_B, fake_B, flow_ref, conf_ref, scale_T):
        """vid2vid_model_D.py:179-197."""
        netD_T = getattr(self, 'netD_T' + str(scale_T))
        real_B = real_B.reshape(-1, self.output_nc * self.tD, self.height, self.width)
        fake_B = fake_B.reshape(-1, self.output_nc * self.tD, self.height, self.width)
        if flow_ref is not None:
            flow_ref = flow_ref.reshape(-1, 2 * (self.tD - 1), self.height, self.width)
            real_B = torch.cat([real_B, flow_ref], dim=1)
            fake_B = torch.cat([fake_B, flow_ref], dim=1)
        return self.compute_loss_D(netD_T, None, real_B, fake_B)

    # ------------------------------------------------------------------ face discriminator
    def face_window_async(self, real_A):
        """get_face_region (vid2vid_model_D.py:215-230) without stalling the host: the window is computed on the device and
        copied to pinned memory behind an event; face_found() waits for that event only."""
        win = ops.face_window(real_A, self.opt.fineSize, getattr(self.opt, 'openpose_only', False), buf=self._face_buf)
        self._face_host.copy_(win, non_blocking=True)
        self._face_event.record(torch.cuda.current_stream(real_A.device))
        return win

    def face_found(self):
        t0 = time.perf_counter()
        self._face_event.synchronize()
        self.face_wait_s = time.perf_counter() - t0
        return bool(self._face_host[0])

    def compute_loss_D_face(self, real_A, real_B, fake_B, win):
        """vid2vid_model_D.py:150-155: netD_f on the face window of (real_A, real_B) / (real_A, fake_B), the generator terms
        weighted by face_weight = 2.  Feature matching keeps GAN_and_FM_loss's 1 / opt.num_D weight, as the reference does.
        `win` lives in the model's window buffer, which the next forward(0, ...) overwrites: back-propagate these losses before
        that call, as the training step does."""
        size = 2 * ops.face_half(self.opt.fineSize)
        real_AB = ops.crop_concat(real_A, real_B, win, size)
        fake_AB = ops.crop_concat(real_A, fake_B, win, size)
        d_real, d_fake, g_gan, g_fm = self._loss_D_on(self.netD_f, real_AB, fake_AB)
        return d_real, d_fake, g_gan * 2, g_fm * 2

    # ------------------------------------------------------------------ forward
    def forward(self, scale_T, tensors_list, dummy_bs=0):
        """vid2vid_model_D.py:93-164 (one process per GPU: no dummy padding).  Returns the reference's loss lists, each
        entry a (1, 1) tensor."""
        opt = self.opt
        if scale_T > 0:
            real_B, fake_B, flow_ref, conf_ref = tensors_list
            self.height, self.width = real_B.shape[-2:]
            d_real, d_fake, g_gan, g_fm = self.compute_loss_D_T(real_B, fake_B, flow_ref / 20 if flow_ref is not None else None,
                                                                conf_ref, scale_T - 1)
            return [t.reshape(-1, 1) for t in (g_gan, g_fm, d_real, d_fake, torch.zeros_like(g_gan))]
        real_B, fake_B, fake_B_raw, real_A, real_B_prev, fake_B_prev, flow, weight, flow_ref, conf_ref = tensors_list
        self.height, self.width = real_B.shape[-2:]
        win = self.face_window_async(real_A) if self.add_face_disc else None       # read back after the netD launches
        if flow is not None:
            loss_F_Flow = ops.l1_loss(flow, flow_ref, conf_ref) * (opt.lambda_F / (2 ** (opt.n_scales_spatial - 1)))     # :121
            loss_F_Warp = ops.l1_loss(self.resample(real_B_prev, flow), real_B, conf_ref) * opt.lambda_T                 # :123-124
            loss_W = torch.zeros_like(weight)
            if opt.no_first_img:
                loss_W = ops.l1_loss(weight, None, conf_ref)                                                             # :128-130
        else:
            loss_F_Flow = loss_F_Warp = loss_W = torch.zeros_like(conf_ref)
        loss_G_VGG = torch.zeros_like(loss_W)
        loss_D_real, loss_D_fake, loss_G_GAN, loss_G_GAN_Feat = self.compute_loss_D(self.netD, real_A, real_B, fake_B)
        fake_B_warp_ref = self.resample(fake_B_prev, flow_ref)
        loss_G_Warp = ops.l1_loss(fake_B, fake_B_warp_ref.detach(), conf_ref) * opt.lambda_T                            # :139-140
        if fake_B_raw is not None:
            r = self.compute_loss_D(self.netD, real_A, real_B, fake_B_raw)
            loss_D_real, loss_D_fake = loss_D_real + r[0], loss_D_fake + r[1]
            loss_G_GAN, loss_G_GAN_Feat = loss_G_GAN + r[2], loss_G_GAN_Feat + r[3]
        losses = [loss_G_VGG, loss_G_GAN, loss_G_GAN_Feat, loss_D_real, loss_D_fake, loss_G_Warp, loss_F_Flow, loss_F_Warp, loss_W]
        if self.add_face_disc:                                                                                       # :148-158
            if self.face_found():
                d_f_real, d_f_fake, g_f_gan, g_f_fm = self.compute_loss_D_face(real_A, real_B, fake_B, win)
            else:             # no face: netD_f does not run (its running statistics stay put)
                d_f_real = d_f_fake = g_f_gan = g_f_fm = torch.zeros_like(loss_D_real)
            losses += [g_f_gan, g_f_fm, d_f_real, d_f_fake]
        return [t.reshape(-1, 1) for t in losses]

    def save(self, label):
        """vid2vid_model_D.py:266-272."""
        self.save_network(self.netD, 'D', label, self.gpu_ids)
        for s in range(self.opt.n_scales_temporal):
            self.save_network(getattr(self, 'netD_T' + str(s)), 'D_T' + str(s), label, self.gpu_ids)
        if self.add_face_disc:
            self.save_network(self.netD_f, 'D_f', label, self.gpu_ids)

    def get_all_skipped_frames(self, frames_all, real_B, fake_B, flow_ref, conf_ref, t_scales, tD, n_frames_load, i, flowNet):
        """vid2vid_model_D.py:232-247: the temporally sub-sampled real / fake / flow groups of every temporal scale (dense form;
        --sparse_D is not implemented, DESIGN.md section 9)."""
        from .trainer import get_skipped_flows, get_skipped_frames
        if getattr(self.opt, 'sparse_D', False):
            raise NotImplementedError('--sparse_D is out of scope (DESIGN.md section 9)')
        real_B_all, fake_B_all, flow_ref_all, conf_ref_all = frames_all
        real_sk = fake_sk = flow_sk = conf_sk = None
        if t_scales > 0:
            real_B_all, real_sk = get_skipped_frames(real_B_all, real_B, t_scales, tD)
            fake_B_all, fake_sk = get_skipped_frames(fake_B_all, fake_B, t_scales, tD)
            flow_ref_all, conf_ref_all, flow_sk, conf_sk = get_skipped_flows(flowNet, flow_ref_all, conf_ref_all, real_sk, flow_ref, conf_ref,
                                                                              t_scales, tD)
        return (real_B_all, fake_B_all, flow_ref_all, conf_ref_all), (real_sk, fake_sk, flow_sk, conf_sk)

    def get_losses(self, loss_dict, loss_dict_T, t_scales):
        """vid2vid_model_D.py:243-259."""
        loss_D = (loss_dict['D_fake'] + loss_dict['D_real']) * 0.5
        loss_G = loss_dict['G_GAN'] + loss_dict['G_GAN_Feat'] + loss_dict['G_VGG']
        loss_G = loss_G + loss_dict['G_Warp'] + loss_dict['F_Flow'] + loss_dict['F_Warp'] + loss_dict['W']
        if self.add_face_disc:                                                                                       # :253-255
            loss_G = loss_G + loss_dict['G_f_GAN'] + loss_dict['G_f_GAN_Feat']
            loss_D = loss_D + (loss_dict['D_f_fake'] + loss_dict['D_f_real']) * 0.5
        loss_D_T = []
        t_scales_act = min(t_scales, len(loss_dict_T))
        for s in range(t_scales_act):
            loss_G = loss_G + loss_dict_T[s]['G_T_GAN'] + loss_dict_T[s]['G_T_GAN_Feat'] + loss_dict_T[s]['G_T_Warp']
            loss_D_T.append((loss_dict_T[s]['D_T_fake'] + loss_dict_T[s]['D_T_real']) * 0.5)
        return loss_G, loss_D, loss_D_T, t_scales_act

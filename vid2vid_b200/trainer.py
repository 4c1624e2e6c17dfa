"""The training step of train.py:50-93 on the B200 engine, one process per GPU.

  * `FlatGrads`: every parameter's .grad is a view into ONE flat fp32 buffer laid out [G | D | D_T0 | ...] (D holds netD and,
    with --add_face_disc, netD_f: the two share optimizer_D as in vid2vid_model_D.py:76-85); a step issues a
    single NCCL all-reduce(SUM) / world over it (SURVEY 8e) -- the replacement of DataParallel's per-forward parameter
    broadcast + per-backward reduce-to-GPU-0 (models/models.py:10-59).  Batch statistics stay per rank, as under DataParallel.
  * `Trainer.step`: generator forward (Vid2VidModelG.forward), reference flow (FlowNet, no grad), image / temporal
    discriminator losses (Vid2VidModelD.forward) and the three backward passes in the reference's order
    (loss_G, loss_D, loss_D_T*; train.py:83-90), then the all-reduce and the Adam steps.
  * the temporal-discriminator frame bookkeeping (get_skipped_frames / get_skipped_flows, vid2vid_model_D.py:267-301).
All tensor math runs in libv2v_b200.so (plan runtime forward / backward, loss kernels); torch supplies autograd bookkeeping,
tensor views / concatenation, torch.optim.Adam (the reference's optimizer) and torch.distributed.
"""
import torch
import torch.distributed as dist


# ------------------------------------------------------------------------------------------------ gradient exchange
class FlatGrads:
    """One flat gradient buffer over several parameter groups; group g occupies [offsets[g], offsets[g + 1])."""

    def __init__(self, groups):
        self.groups = [list(g) for g in groups]
        params = [p for g in self.groups for p in g]
        dev = params[0].device
        self.numel = sum(p.numel() for p in params)
        self.flat = torch.zeros(self.numel, device=dev, dtype=torch.float32)
        self.offsets = [0]
        off = 0
        for g in self.groups:
            for p in g:
                p.grad = self.flat[off:off + p.numel()].view_as(p)         # autograd accumulates in place into the view
                off += p.numel()
            self.offsets.append(off)

    def zero(self, group=None):
        if group is None:
            self.flat.zero_()
        else:
            self.flat[self.offsets[group]:self.offsets[group + 1]].zero_()

    def all_reduce_mean(self, world):
        """The step's single collective: average the gradients over the ranks (NCCL on GPUs, gloo in the CPU tests)."""
        if world > 1:
            dist.all_reduce(self.flat, op=dist.ReduceOp.SUM)
            self.flat.div_(world)


# ------------------------------------------------------------------------------------------------ temporal bookkeeping
def get_skipped_frames(B_all, B, t_scales, tD):
    """vid2vid_model_D.py:267-282: keep the running history B_all (b, T, ...) and return, per temporal scale s, the groups of
    tD frames sampled every tD**s frames that end in the newly generated frames."""
    B_all = torch.cat([B_all.detach(), B], dim=1) if B_all is not None else B
    B_skipped = [None] * t_scales
    for s in range(t_scales):
        tDs = tD ** s
        span = tDs * (tD - 1)
        n_groups = min(B_all.size(1) - span, B.size(1))
        if n_groups > 0:
            for t in range(0, n_groups, tD):
                skip = B_all[:, (-span - t - 1):-t:tDs].contiguous() if t != 0 else B_all[:, -span - 1::tDs].contiguous()
                B_skipped[s] = torch.cat([B_skipped[s], skip]) if B_skipped[s] is not None else skip
    max_prev = tD ** (t_scales - 1) * (tD - 1)
    if B_all.size(1) > max_prev:
        B_all = B_all[:, -max_prev:]
    return B_all, B_skipped


def get_skipped_flows(flowNet, flow_ref_all, conf_ref_all, real_B_skipped, flow_ref, conf_ref, t_scales, tD):
    """vid2vid_model_D.py:285-296: scale 0 reuses the flows already computed; coarser temporal scales re-run FlowNet2 on the
    skipped real frames."""
    flow_skipped, conf_skipped = [None] * t_scales, [None] * t_scales
    flow_ref_all, flow = get_skipped_frames(flow_ref_all, flow_ref, 1, tD)
    conf_ref_all, conf = get_skipped_frames(conf_ref_all, conf_ref, 1, tD)
    if flow[0] is not None:
        flow_skipped[0], conf_skipped[0] = flow[0][:, 1:], conf[0][:, 1:]
    for s in range(1, t_scales):
        if real_B_skipped[s] is not None and real_B_skipped[s].size(1) == tD:
            flow_skipped[s], conf_skipped[s] = flowNet(real_B_skipped[s][:, 1:], real_B_skipped[s][:, :-1])
    return flow_ref_all, conf_ref_all, flow_skipped, conf_skipped


def _merge(t):
    """train.py `reshape`: (b, t, c, h, w) -> (b*t, c, h, w)."""
    if t is None:
        return None
    return t.contiguous().view(-1, *t.shape[2:])


# ------------------------------------------------------------------------------------------------ the step
class Trainer:
    def __init__(self, opt, modelG, modelD, flowNet, world=1):
        self.opt, self.modelG, self.modelD, self.flowNet, self.world = opt, modelG, modelD, flowNet, world
        self.tG, self.tD, self.t_scales = opt.n_frames_G, opt.n_frames_D, opt.n_scales_temporal
        params_D = list(modelD.netD.parameters())
        if getattr(modelD, 'add_face_disc', False):
            params_D += list(modelD.netD_f.parameters())     # each rank's window comes from its own shard, as per replica
        groups = [[p for s in range(modelG.n_scales) for p in getattr(modelG, 'netG' + str(s)).parameters()], params_D]
        groups += [list(getattr(modelD, 'netD_T' + str(s)).parameters()) for s in range(self.t_scales)]
        self.grads = FlatGrads(groups)
        self.reset_clip()
        self.timing = {}

    def reset_clip(self):
        """Start of a new training sequence (train.py:57-58)."""
        self.fake_B_prev_last = None
        self.frames_all = (None, None, None, None)

    def losses(self, input_A, input_B, inst_A):
        """Forward half of train.py:62-81 for the next n_frames_load frames: returns (loss_G, loss_D, [loss_D_T...], dicts)."""
        G, D = self.modelG, self.modelD
        fake_B, fake_B_raw, flow, weight, real_A, real_Bp, fake_B_last = G(input_A, input_B, inst_A, self.fake_B_prev_last)
        real_B_prev, real_B = real_Bp[:, :-1], real_Bp[:, 1:]
        flow_ref, conf_ref = self.flowNet(real_B, real_B_prev)
        fake_B_prev = G.compute_fake_B_prev(real_B_prev, self.fake_B_prev_last, fake_B)
        self.fake_B_prev_last = fake_B_last
        losses = D(0, [_merge(t) for t in (real_B, fake_B, fake_B_raw, real_A, real_B_prev, fake_B_prev, flow, weight, flow_ref, conf_ref)])
        loss_dict = dict(zip(D.loss_names, [torch.mean(x) for x in losses]))
        # temporal discriminators (train.py:70-78)
        real_all, fake_all, flow_all, conf_all = self.frames_all
        real_sk = fake_sk = flow_sk = conf_sk = [None] * max(self.t_scales, 1)
        if self.t_scales > 0:
            real_all, real_sk = get_skipped_frames(real_all, real_B, self.t_scales, self.tD)
            fake_all, fake_sk = get_skipped_frames(fake_all, fake_B, self.t_scales, self.tD)
            flow_all, conf_all, flow_sk, conf_sk = get_skipped_flows(self.flowNet, flow_all, conf_all, real_sk, flow_ref, conf_ref,
                                                                     self.t_scales, self.tD)
        self.frames_all = (real_all, fake_all, flow_all, conf_all)
        loss_dict_T = []
        for s in range(self.t_scales):
            if real_sk[s] is not None:
                lt = D(s + 1, [real_sk[s], fake_sk[s], flow_sk[s], conf_sk[s]])
                loss_dict_T.append(dict(zip(D.loss_names_T, [torch.mean(x) for x in lt])))
        loss_G, loss_D, loss_D_T, t_act = D.get_losses(loss_dict, loss_dict_T, self.t_scales)
        return loss_G, loss_D, loss_D_T, loss_dict, loss_dict_T

    def step_async(self, input_A, input_B, inst_A):
        """One iteration of train.py's inner loop on this rank's shard of the batch; returns the PendingLosses of the step."""
        G, D = self.modelG, self.modelD
        loss_G, loss_D, loss_D_T, loss_dict, loss_dict_T = self.losses(input_A, input_B, inst_A)
        # backward passes in the reference's order (train.py:83-90): the generator loss also back-propagates through the
        # discriminators, whose gradients from it are discarded (each optimizer zero_grad()s before its own backward)
        self.grads.zero()
        loss_G.backward()
        for g in range(1, len(self.grads.groups)):
            self.grads.zero(g)
        loss_D.backward()
        for lt in loss_D_T:
            lt.backward()
        # ONE collective per step over [G | D | D_T...], then the optimizers
        self.grads.all_reduce_mean(self.world)
        G.optimizer_G.step()
        D.optimizer_D.step()
        for s in range(len(loss_D_T)):
            getattr(D, 'optimizer_D_T' + str(s)).step()
        # ONE device -> host read per step: the loss values of all dictionaries stacked, copied to pinned host memory
        # asynchronously; PendingLosses.get() waits for that copy only
        keys = [(None, k) for k in loss_dict] + [(i, k) for i, d in enumerate(loss_dict_T) for k in d]
        vals = torch.stack([(loss_dict if i is None else loss_dict_T[i])[k].detach().reshape(()).float() for i, k in keys])
        return PendingLosses(keys, vals, len(loss_dict_T))

    def step(self, input_A, input_B, inst_A):
        """One iteration of train.py's inner loop on this rank's shard of the batch -> (loss dict, [temporal loss dicts]) as
        Python floats (blocks until the step has finished on the GPU, as reading `v.data.item()` in train.py:104 does)."""
        return self.step_async(input_A, input_B, inst_A).get()


class PendingLosses:
    """Loss values of a step on their way to the host.  The reference reads them every print_freq steps (train.py:102-107); a
    training loop that reads every step can do so one step late -- issue step n + 1, then get() step n -- so that the host
    never waits for the GPU and the GPU never waits for the host."""

    def __init__(self, keys, vals, n_T):
        self.keys, self.n_T = keys, n_T
        self.host = torch.empty(vals.shape, dtype=torch.float32, pin_memory=vals.is_cuda)
        self.host.copy_(vals, non_blocking=True)
        self.event = None
        if vals.is_cuda:
            self.event = torch.cuda.Event()
            self.event.record(torch.cuda.current_stream(vals.device))

    def get(self):
        if self.event is not None:
            self.event.synchronize()
        out, out_T = {}, [dict() for _ in range(self.n_T)]
        for (i, k), v in zip(self.keys, self.host.tolist()):
            (out if i is None else out_T[i])[k] = v
        return out, out_T

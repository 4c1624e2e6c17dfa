"""CPU: the host-side checkpoint / schedule helpers (vid2vid_b200/base_model.py) against what the reference's BaseModel
(models/base_model.py:43-48,154-181) did on the same state (tests/golden/base_model_schedule.json, written by
`python -m oracle.make_golden schedule`)."""
import json
import os
import types

import torch
import torch.nn as nn

import cases
from vid2vid_b200.base_model import HostScheduleMixin

REF = json.load(open(os.path.join(os.path.dirname(__file__), 'golden', 'base_model_schedule.json')))


class _Ours(HostScheduleMixin):
    pass


def _state(opt, cls):
    m = cls()
    m.opt = opt
    m.old_lr = opt.lr
    m.n_scales = 2
    m.netG0, m.netG1 = nn.Linear(3, 2), nn.Linear(2, 2)
    m.optimizer_G = torch.optim.Adam(list(m.netG1.parameters()), lr=opt.lr, betas=(opt.beta1, 0.999))
    m.n_gpus, m.n_frames_per_gpu, m.n_frames_load, m.n_frames_bp = 1, 1, 1, 1
    m.finetune_all = False
    return m


def _opt(tmp):
    return types.SimpleNamespace(checkpoints_dir=str(tmp), **cases.SCHEDULE_OPT)


def test_schedules_match_the_reference(tmp_path):
    opt = _opt(tmp_path)
    ours = _state(opt, _Ours)
    for epoch, (old_lr, lrs) in zip(cases.SCHEDULE_EPOCHS, REF['lr'], strict=True):
        ours.update_learning_rate(epoch, 'G')
        assert ours.old_lr == old_lr
        assert [g['lr'] for g in ours.optimizer_G.param_groups] == lrs
    for ratio, batch in zip(cases.SCHEDULE_RATIOS, REF['batch'], strict=True):     # train.py:121-123: every niter_step epochs
        ours.update_training_batch(ratio)
        assert [ours.n_frames_bp, ours.n_frames_per_gpu, ours.n_frames_load] == batch
    assert ours.n_frames_per_gpu == 8
    ours.update_fixed_params()
    assert ours.finetune_all and REF['finetune_all']
    n_ours = sum(p.numel() for g in ours.optimizer_G.param_groups for p in g['params'])
    assert n_ours == REF['n_params_G'] == sum(p.numel() for m in (ours.netG0, ours.netG1) for p in m.parameters())
    assert ours.optimizer_G.param_groups[0]['lr'] == REF['lr_after_fix'] == ours.old_lr


def test_save_network_writes_the_reference_file_and_keeps_the_parameters_in_place(tmp_path):
    opt = _opt(tmp_path)
    ours = _state(opt, _Ours)
    ptrs = [p.data_ptr() for p in ours.netG1.parameters()]
    path = ours.save_network(ours.netG1, 'G1', 'latest', [])
    assert [os.path.basename(path)] == REF['saved_files'] and os.path.dirname(path) == os.path.join(opt.checkpoints_dir, opt.name)
    a, b = torch.load(path), ours.netG1.state_dict()
    assert list(a) == REF['saved_keys'] and all(torch.equal(a[k], b[k]) and a[k].device.type == 'cpu' for k in a)
    assert ptrs == [p.data_ptr() for p in ours.netG1.parameters()]          # no .cpu() / .cuda() round trip of the module

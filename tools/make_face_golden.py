"""Writes the reference fixtures of the face discriminator: runs the unmodified reference Vid2VidModelD with --add_face_disc
(through oracle/ref_shim.py, on CPU) on the seeded cases of tests/face_oracle.py and stores
  tests/golden/ref_face.npz      per case: the reference's get_face_region window and the 13 spatial losses of forward(0, ...)
  tests/golden/ref_face_keys.json  the reference netD_f state_dict keys and shapes.
Needs the reference tree (V2V_REFERENCE_ROOT or the default of ref_shim).   python tools/make_face_golden.py"""
import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), '..'))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tests'))
from oracle import ref_shim                                   # noqa: E402
import face_oracle as FC                                      # noqa: E402
from vid2vid_b200.utils import det_fill_                      # noqa: E402

OUT = os.path.join(ROOT, 'tests', 'golden')


def face_pins():
    ref_shim.install()
    from models.vid2vid_model_D import Vid2VidModelD          # noqa (reference module)
    out, keys = {}, None
    for name, (_, openpose) in FC.FACE_CASES.items():
        opt = FC.face_opt(openpose_only=openpose)
        m = Vid2VidModelD()
        m.initialize(opt)
        det_fill_(m.netD, seed=FC.FACE_SEED_D)
        det_fill_(m.netD_f, seed=FC.FACE_SEED_D_F)
        keys = [[k, list(v.shape)] for k, v in m.netD_f.state_dict().items()]
        inputs = FC.face_case_inputs(name)
        win = m.get_face_region(inputs[3])
        out['%s_window' % name] = np.array([-1] * 4 if win[0] is None else win, dtype=np.int64)
        with torch.no_grad():
            losses = m.forward(0, inputs)
        assert len(losses) == len(FC.SPATIAL_LOSS_NAMES)
        for n, t in zip(FC.SPATIAL_LOSS_NAMES, losses):
            out['%s_%s' % (name, n)] = t.detach().cpu().numpy().astype(np.float32)
        print('%-10s window %s D_f_real %.5f G_f_GAN %.5f' % (name, win, float(losses[11].mean()), float(losses[9].mean())))
    np.savez_compressed(os.path.join(OUT, 'ref_face.npz'), **out)
    with open(os.path.join(OUT, 'ref_face_keys.json'), 'w') as f:
        json.dump(keys, f)
    print('ref_face.npz %.1f KB, netD_f %d tensors' % (os.path.getsize(os.path.join(OUT, 'ref_face.npz')) / 1024, len(keys)))


if __name__ == '__main__':
    face_pins()

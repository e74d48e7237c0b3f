"""Generates the fixtures that pin the oracle and this package's model to the original PointContrast code (run where the
original project's `pretrain/pointcontrast` package can be imported, see tests/refload.py):

    python tests/golden/make_reference_fixtures.py

  reference_res16unet34c_structure.json -- the original `model/res16unet.py` Res16UNet34C built on the CPU oracle: every
      module (name, class, kernel offsets, stride, bias, BatchNorm momentum / eps) and every state-dict entry (name, shape);
  reference_losses.npz -- the original loss code on the inputs that tests/test_oracle_reference.py draws:
      `HardestContrastiveLossTrainer.contrastive_hardest_negative_loss` (pos / neg loss per `num_pos`) and
      `PointNCELossTrainer._train_iter` on a small stand-in model (loss and the stand-in's weight gradient per `npos`).
"""
import json
import os
import sys
import types

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

from oracle import me_cpu                                   # noqa: E402
from tests import refload                                   # noqa: E402
from tests.helpers import model_structure                   # noqa: E402
from tests.test_oracle_reference import HARDEST_NUM_POS, NCE_NPOS, StandIn, hardest_inputs, nce_batch   # noqa: E402

GOLDEN = os.path.dirname(os.path.abspath(__file__))


def structure():
    pkg = refload.load_reference_model_module(me_cpu.install)
    net = pkg.load_model("Res16UNet34C")(3, 32, refload.default_config(), D=3)
    return model_structure(net)


def hardest(tr):
    obj = tr.HardestContrastiveLossTrainer.__new__(tr.HardestContrastiveLossTrainer)
    obj.pos_thresh, obj.neg_thresh = 0.1, 1.4
    F0, F1, pairs = hardest_inputs()
    out = {}
    for num_pos in HARDEST_NUM_POS:
        np.random.seed(7)
        pos, neg = obj.contrastive_hardest_negative_loss(F0, F1, pairs, num_pos=num_pos, num_hn_samples=256)
        out[f"hardest_{num_pos}"] = np.array([float(pos), float(neg)])
    return out


def point_nce(tr):
    # the original `_train_iter` moves its inputs and model with hard-coded `.cuda()` calls: identity on the CPU here
    torch.Tensor.cuda = lambda self, *a, **k: self
    torch.nn.Module.cuda = lambda self, *a, **k: self
    batch = nce_batch()
    inp = {k: (torch.from_numpy(v) if isinstance(v, np.ndarray) else v) for k, v in batch.items()}
    inp["pcd0"], inp["pcd1"] = inp["sinput0_C"], inp["sinput1_C"]                  # only .shape[0] is read

    class It:
        def next(self):
            return inp

    out = {}
    for npos in NCE_NPOS:
        net = StandIn()
        obj = tr.PointNCELossTrainer.__new__(tr.PointNCELossTrainer)
        obj.model, obj.cur_device, obj.T, obj.npos = net, "cpu", 0.4, npos
        obj.optimizer = types.SimpleNamespace(zero_grad=lambda: None, step=lambda: None)
        obj.config = refload.Cfg(misc=dict(num_gpus=1))
        torch.manual_seed(11); np.random.seed(12)
        out[f"nce_{npos}_loss"] = np.float64(obj._train_iter(It(), [tr.AverageMeter(), tr.Timer(), tr.Timer()]))
        out[f"nce_{npos}_grad"] = net.lin.weight.grad.numpy().copy()
    return out


def main():
    path = os.path.join(GOLDEN, "reference_res16unet34c_structure.json")
    with open(path, "w") as f:
        json.dump(structure(), f, separators=(",", ":"))
        f.write("\n")
    print("wrote", path, os.path.getsize(path), "bytes")
    tr = refload.load_reference_trainer_module(me_cpu.install)
    path = os.path.join(GOLDEN, "reference_losses.npz")
    np.savez_compressed(path, **hardest(tr), **point_nce(tr))
    print("wrote", path, os.path.getsize(path), "bytes")


if __name__ == "__main__":
    main()

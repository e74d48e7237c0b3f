"""The oracle against the original PointContrast code: its model graph and its two losses, as recorded from that code in
tests/golden/ by tests/golden/make_reference_fixtures.py."""
import os
import types

import numpy as np
import torch

from oracle import loss_cpu, me_cpu
from tests import refload
from tests.helpers import GOLDEN, model_backend, model_structure, reference_structure

HARDEST_NUM_POS = (1024, 5000)
NCE_NPOS = (64, 1 << 20)                             # with and without the npos subsample (`lib/ddp_trainer.py:411-415`)


def hardest_inputs():
    g = torch.Generator().manual_seed(0)
    N0, N1, P = 700, 650, 3000
    F0 = torch.nn.functional.normalize(torch.randn(N0, 32, generator=g, dtype=torch.float64), dim=1)
    F1 = torch.nn.functional.normalize(torch.randn(N1, 32, generator=g, dtype=torch.float64), dim=1)
    F1[:300] = F0[:300] + 0.05 * torch.randn(300, 32, generator=g, dtype=torch.float64)
    rng = np.random.default_rng(0)
    i0 = np.sort(rng.integers(0, 300, P))
    pairs = torch.from_numpy(np.stack([i0, np.clip(i0 + rng.integers(-1, 2, P), 0, N1 - 1)], 1))
    return F0, F1, pairs


class StandIn(torch.nn.Module):
    """Stand-in for Res16UNet in the PointInfoNCE check: per-row features from (feats, coords)."""
    def __init__(self):
        super().__init__()
        torch.manual_seed(0)
        self.lin = torch.nn.Linear(7, 32).double()

    def forward(self, s):
        x = torch.cat([s.F.double(), torch.sin(s.C.double() * 0.37)], 1)
        return types.SimpleNamespace(F=torch.nn.functional.normalize(self.lin(x), dim=1))


def nce_batch():
    from pointcontrast_b200 import synth
    return synth.collate_pairs([synth.synth_pair(3, scale=0.1), synth.synth_pair(4, scale=0.1)])


def _recorded():
    return np.load(os.path.join(GOLDEN, "reference_losses.npz"))


def test_reference_res16unet34c_builds_on_oracle():
    """The original Res16UNet34C as recorded on the oracle, and this package's model file built on the oracle: the same modules,
    kernel offsets, strides, BatchNorm settings and state-dict layout."""
    ref = reference_structure()
    assert ref["n_params"] == 37_847_808
    classes = [m["class"] for m in ref["modules"]]
    assert (classes.count("MinkowskiConvolution"), classes.count("MinkowskiConvolutionTranspose"),
            classes.count("MinkowskiBatchNorm")) == (59, 4, 62)
    moms = sorted(m["momentum"] for m in ref["modules"] if m["class"] == "MinkowskiBatchNorm")
    assert moms.count(0.1) == 46 and moms.count(0.05) == 16          # SURVEY 8a row B1
    sd = dict((k, tuple(s)) for k, s in ref["state_dict"])
    assert sd["conv0p1s1.kernel"] == (27, 3, 32)
    assert sd["final.kernel"] == (1, 96, 32) and sd["final.bias"] == (1, 32)
    assert sd["block2.0.downsample.0.kernel"] == (1, 32, 64)
    assert "bn0.bn.running_mean" in sd and "block8.1.norm2.bn.weight" in sd
    with model_backend(me_cpu) as mod:
        net = mod.Res16UNet34C(3, 32, refload.default_config(), D=3)
    assert model_structure(net) == ref


def test_hardest_loss_oracle_matches_reference_function():
    rec = _recorded()
    F0, F1, pairs = hardest_inputs()
    N0, N1, P = len(F0), len(F1), len(pairs)
    for num_pos in HARDEST_NUM_POS:
        ref_pos, ref_neg = (torch.tensor(v, dtype=torch.float64) for v in rec[f"hardest_{num_pos}"])
        np.random.seed(7)
        sel0 = np.random.choice(N0, 256, replace=False)
        sel1 = np.random.choice(N1, 256, replace=False)
        pos_sel = np.random.choice(P, num_pos, replace=False) if P > num_pos else None
        pos, neg = loss_cpu.hardest_contrastive_loss(F0, F1, pairs.numpy(), sel0, sel1, pos_sel)
        assert torch.allclose(pos, ref_pos, rtol=1e-12) and torch.allclose(neg, ref_neg, rtol=1e-12)


def test_point_nce_oracle_matches_reference_train_iter():
    """Rows L1 + L2: the original `PointNCELossTrainer._train_iter` (`lib/ddp_trainer.py:380-440`, `NCESoftmaxLoss` from
    `lib/criterion.py`) run on the CPU with a small stand-in model -- its loss and the stand-in's weight gradient, recorded --
    against `loss_cpu.select_positives` + `point_nce_loss` fed with the same RNG draws."""
    rec = _recorded()
    batch = nce_batch()
    inp = {k: (torch.from_numpy(v) if isinstance(v, np.ndarray) else v) for k, v in batch.items()}
    nq = len(np.unique(batch["correspondences"][:, 0]))
    for npos in NCE_NPOS:
        ref_loss, ref_grad = float(rec[f"nce_{npos}_loss"]), torch.from_numpy(rec[f"nce_{npos}_grad"])
        torch.manual_seed(11); np.random.seed(12)
        uniform = torch.distributions.Uniform(0, 1).sample([nq])
        sampled = np.random.choice(nq, npos, replace=False) if npos < nq else None
        net = StandIn()
        F0 = net(me_cpu.SparseTensor(inp["sinput0_F"], coords=inp["sinput0_C"])).F
        F1 = net(me_cpu.SparseTensor(inp["sinput1_F"], coords=inp["sinput1_C"])).F
        q, k = loss_cpu.select_positives(batch["correspondences"], uniform, npos, sampled)
        assert len(q) == min(npos, nq)
        loss = loss_cpu.point_nce_loss(F0, F1, q, k, 0.4)
        loss.backward()
        assert abs(float(loss) - ref_loss) < 1e-12 * abs(ref_loss), (float(loss), ref_loss)
        assert torch.allclose(net.lin.weight.grad, ref_grad, rtol=1e-10, atol=1e-14)

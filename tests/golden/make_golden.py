"""Generates tests/golden/c0_res16unet34c.npz and c0_res16unet34c_features.npz (run where the original project's
`pretrain/pointcontrast` package can be imported, see tests/refload.py):

    python tests/golden/make_golden.py

The REFERENCE's own model graph (`pretrain/pointcontrast/model/res16unet.py` of the original project, imported unmodified)
is executed on the CPU oracle (oracle/me_cpu.py, fp64) for BASELINE config C0: one synthetic scene pair (~4k voxels
per view), Res16UNet34C, PointInfoNCE (T = 0.4, npos = 4096), deterministic weights (tests/helpers.det_init).
Stored: the inputs, per-point output features of both views, the loss, the chosen positive indices, the gradient
norm of every parameter, slices of three gradients, and -- because the backward pass of this network is ill-conditioned
(BatchNorm backward cancels the common-mode part of the gradient; DESIGN.md "Numerics") -- the relative error that the
SAME graph run in plain fp32 has against fp64, per parameter (`grad_relerr_f32`): the floor of any fp32 implementation.  tests/test_gpu_model.py replays it on the GPU.
"""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

from oracle import loss_cpu, me_cpu          # noqa: E402
from pointcontrast_b200 import synth         # noqa: E402
from tests import refload                    # noqa: E402
from tests.helpers import det_init           # noqa: E402


def run(pkg, batch, dtype):
    net = pkg.load_model("Res16UNet34C")(3, 32, refload.default_config(), D=3)
    det_init(net, seed=0)
    net = net.to(dtype).train()
    F = []
    for v in ("0", "1"):
        st = me_cpu.SparseTensor(torch.from_numpy(batch[f"sinput{v}_F"]).to(dtype),
                                 coords=torch.from_numpy(batch[f"sinput{v}_C"]))
        F.append(net(st).F)
    return net, F


def main():
    torch.set_num_threads(os.cpu_count())
    pkg = refload.load_reference_model_module(me_cpu.install)
    batch = synth.collate_pairs([synth.synth_pair(0, scale=0.24)])
    net, F = run(pkg, batch, torch.float64)
    rng = np.random.default_rng(123)
    pairs = batch["correspondences"]
    nq = len(np.unique(pairs[:, 0]))
    uniform = rng.random(nq).astype(np.float32)
    sampled = rng.choice(nq, 4096, replace=False) if nq > 4096 else None
    q_rows, k_rows = loss_cpu.select_positives(pairs, uniform, 4096, sampled)
    loss = loss_cpu.point_nce_loss(F[0], F[1], q_rows, k_rows, 0.4)
    loss.backward()
    # the same graph in plain fp32: the noise floor ANY fp32 implementation (the reference included) has on this problem
    net32, F32 = run(pkg, batch, torch.float32)
    loss_cpu.point_nce_loss(F32[0], F32[1], q_rows, k_rows, 0.4).backward()
    f32_err = np.array([float((p32.grad.double() - p.grad).norm() / p.grad.norm())
                        for (_, p), (_, p32) in zip(net.named_parameters(), net32.named_parameters())])
    f32_feat_err = float((F32[0].double() - F[0]).abs().max() / F[0].pow(2).mean().sqrt())
    names = [n for n, _ in net.named_parameters()]
    gnorm = np.array([float(p.grad.norm()) for _, p in net.named_parameters()])
    sd = dict(net.named_parameters())
    bn_rm = np.stack([float(m.running_mean.abs().sum()) for m in net.modules() if isinstance(m, torch.nn.BatchNorm1d)])
    out = dict(C0=batch["sinput0_C"], C1=batch["sinput1_C"], X0=batch["sinput0_F"], X1=batch["sinput1_F"],
               F0=F[0].detach().numpy().astype(np.float32), F1=F[1].detach().numpy().astype(np.float32),
               q_rows=q_rows.numpy(), k_rows=k_rows.numpy(), loss=np.float64(loss.item()), grad_norms=gnorm,
               param_names=np.array(names), g_conv0=sd["conv0p1s1.kernel"].grad.numpy().astype(np.float32),
               g_final=sd["final.kernel"].grad.numpy().astype(np.float32),
               g_b8=sd["block8.1.conv2.kernel"].grad.numpy()[13].astype(np.float32), bn_running_mean_l1=bn_rm,
               grad_relerr_f32=f32_err, feat_relerr_f32=np.float64(f32_feat_err))
    feats = {k: out.pop(k) for k in ("F0", "F1")}           # a file of their own: each file stays under 1 MB
    for name, arrays in (("c0_res16unet34c.npz", out), ("c0_res16unet34c_features.npz", feats)):
        path = os.path.join(ROOT, "tests", "golden", name)
        np.savez_compressed(path, **arrays)
        print("wrote", path, os.path.getsize(path), "bytes")
    print("loss", loss.item(), "N0", len(batch["sinput0_C"]))


if __name__ == "__main__":
    main()

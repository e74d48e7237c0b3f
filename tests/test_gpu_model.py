"""Whole-network parity on the GPU (BASELINE config C0): Res16UNet34C + PointInfoNCE, forward and backward.
  * against the committed golden vectors, produced by the REFERENCE's model file running on the fp64 oracle
    (tests/golden/make_golden.py);
  * against the oracle run live with this repo's own model wiring (needs no reference tree).
Tolerance: 1e-3 relative (north star) on per-point features, the loss and -- with the ReLU decisions pinned, see
test_small_scene_all_gradients_with_pinned_relu_decisions -- every parameter gradient.  Against an oracle taking its own ReLU
decisions the gradients of ANY finite-precision evaluation sit a few coin flips away (the same graph in plain fp32 on the CPU:
2e-5 .. 7e-3 from fp64 depending on the thread count; stored in the golden file as `grad_relerr_f32`), so the golden-file test
holds them to max(1e-3, 10 x that fp32 figure); the individual backward kernels are held to 1e-3 in tests/test_gpu_ops.py."""
import os

import numpy as np
import pytest
import torch

from oracle import loss_cpu
from oracle import me_cpu as OR
from tests import refload
from tests.helpers import det_init, load_c0_golden, max_rel_err, model_backend, rel_err

pytestmark = pytest.mark.gpu


def _grad_tol(floor, factor):
    """Gradient tolerance: max(1e-3, factor x the network-wide fp32 floor).  The floor is the relative error of the SAME
    graph evaluated in plain fp32 on the CPU against fp64 (worst parameter): 5e-3 .. 1e-2 on these problems, at any scene
    size we could afford to evaluate in fp64 (measured up to 24k voxels/view)."""
    floor = np.asarray(floor, np.float64)
    return np.full_like(floor, max(1e-3, factor * float(floor.max())))


def _gpu_net(seed=0, normalize=True):
    from pointcontrast_b200.model import load_model
    cfg = refload.default_config()
    cfg["net"]["normalize_feature"] = normalize
    net = load_model("Res16UNet34C")(3, 32, cfg, D=3)
    det_init(net, seed)
    return net.cuda().train()


def test_c0_against_reference_graph_golden():
    from pointcontrast_b200 import losses, me
    g = load_c0_golden()
    net = _gpu_net(0)
    F = []
    for v in ("0", "1"):
        st = me.SparseTensor(torch.from_numpy(g["X" + v]), coords=torch.from_numpy(g["C" + v])).to("cuda")
        F.append(net(st).F)
    assert "_fused_runner" in net.__dict__                  # a training-mode call takes the fused executor
    assert max_rel_err(F[0], torch.from_numpy(g["F0"])) < 1e-3 and max_rel_err(F[1], torch.from_numpy(g["F1"])) < 1e-3
    loss = losses.point_nce_loss(F[0], F[1], torch.from_numpy(g["q_rows"]).cuda(), torch.from_numpy(g["k_rows"]).cuda(), 0.4)
    assert abs(float(loss.detach()) - float(g["loss"])) / float(g["loss"]) < 1e-3
    loss.backward()
    names = [n for n, _ in net.named_parameters()]
    assert names == list(g["param_names"])
    gn = np.array([float(p.grad.norm()) for _, p in net.named_parameters()])
    rel = np.abs(gn - g["grad_norms"]) / (g["grad_norms"] + 1e-30)
    tol = _grad_tol(g["grad_relerr_f32"], 10)
    bad = np.nonzero(rel > tol)[0]
    assert len(bad) == 0, [(names[i], rel[i], tol[i]) for i in bad[:5]]
    sd = dict(net.named_parameters())
    t = dict(zip(names, tol))
    assert rel_err(sd["conv0p1s1.kernel"].grad, torch.from_numpy(g["g_conv0"])) < t["conv0p1s1.kernel"]
    assert rel_err(sd["final.kernel"].grad, torch.from_numpy(g["g_final"])) < t["final.kernel"]
    assert rel_err(sd["block8.1.conv2.kernel"].grad[13], torch.from_numpy(g["g_b8"])) < t["block8.1.conv2.kernel"]
    rm = np.array([float(m.running_mean.abs().sum()) for m in net.modules() if isinstance(m, torch.nn.BatchNorm1d)])
    assert (np.abs(rm - g["bn_running_mean_l1"]) / (g["bn_running_mean_l1"] + 1e-30)).max() < 1e-3


_SMALL = {}


def _small_problem():
    """Two small scene pairs, the deterministic weights, the positive draw and the fp64 oracle's own (unpinned) result."""
    if _SMALL:
        return _SMALL
    from pointcontrast_b200 import synth
    batch = synth.collate_pairs([synth.synth_pair(3, scale=0.12), synth.synth_pair(4, scale=0.1)])
    rng = np.random.default_rng(0)
    pairs = batch["correspondences"]
    nq = len(np.unique(pairs[:, 0]))
    q, k = loss_cpu.select_positives(pairs, rng.random(nq).astype(np.float32), 4096,
                                     rng.choice(nq, 4096, replace=False) if nq > 4096 else None)
    _SMALL.update(batch=batch, q=q, k=k)
    return _SMALL


def _oracle_run(state, batch, q, k, dtype, masks=None):
    """Forward + PointInfoNCE + backward of the oracle; with `masks` (one bool [n, C] per ReLU call: view 0's calls, then view 1's)
    the ReLU decisions are replayed instead of taken (tests/helpers.py pinned_relu)."""
    import contextlib
    from tests.helpers import pinned_relu
    flips = []
    with (pinned_relu(OR, masks, flips) if masks is not None else contextlib.nullcontext()):
        with model_backend(OR) as mod:
            onet = mod.Res16UNet34C(3, 32, refload.default_config(), D=3).to(dtype)
            onet.load_state_dict({n: v.to(dtype).cpu() if v.dtype.is_floating_point else v.cpu() for n, v in state.items()})
            onet.train()
            Fo = [onet(OR.SparseTensor(torch.from_numpy(batch[f"sinput{v}_F"]).to(dtype),
                                       coords=torch.from_numpy(batch[f"sinput{v}_C"]))).F for v in "01"]
    lo = loss_cpu.point_nce_loss(Fo[0], Fo[1], q, k, 0.4)
    lo.backward()
    return onet, Fo, lo, flips


@pytest.mark.parametrize("path", ["fused_pair", "fused_views", "modular_simt"])
def test_small_scene_all_gradients_with_pinned_relu_decisions(path):
    """Every one of the 187 parameter gradients, tensor by tensor, against the fp64 oracle -- at the north-star tolerance (1e-3).

    ReLU is the network's one discontinuous operator.  A pre-activation that is zero to within rounding falls on either side in ANY
    finite precision: the oracle itself in fp32 disagrees with its fp64 run on 2 of the 3.0 million ReLU entries of this problem, and
    those two entries alone put its gradients 5e-3 (median) .. 7e-3 (max) away from fp64 -- or 2e-5 away when a different thread count
    happens to round them the other way (one flipped entry on a stride-16 level moves every upstream gradient by
    ~1/sqrt(rows x channels) of its norm).  So the gradient comparison replays, in the fp64 oracle, the ReLU decisions the GPU pass
    took (the sign of each unit's stored output, which is what its backward pass masks with); everything else -- convolutions,
    BatchNorm statistics and backward, weight / data gradients, normalisation, loss -- is then held to 1e-3.  The decisions themselves
    are checked separately: they may differ from the fp64 oracle's only on a handful of entries (< 1e-4 of them).

    paths: the stacked-pair fused executor (what `forward_pair` / the trainer / bench.py run), the fused executor one view at a time
    (`net(sparse_tensor)`), and the modular per-operator surface on the exact-fp32 SIMT kernels."""
    from pointcontrast_b200 import fused, losses, me
    P = _small_problem()
    batch, q, k = P["batch"], P["q"], P["k"]
    net = _gpu_net(1)
    state = {n: v.clone() for n, v in net.state_dict().items()}
    if "natural" not in P:
        P["natural"] = _oracle_run(state, batch, q, k, torch.float64)
    onet, Fo, lo, _ = P["natural"]
    dev = torch.device("cuda")
    T = {n: torch.from_numpy(batch[n]) for n in ("sinput0_F", "sinput0_C", "sinput1_F", "sinput1_C")}
    cap, hooks = [], []
    try:
        if path == "modular_simt":
            me.FORCE_SIMT = True
            for mod in net.modules():
                if isinstance(mod, me.MinkowskiReLU):
                    hooks.append(mod.register_forward_hook(lambda m, i, o: cap.append((o.F.shape[0], o.F.detach() > 0))))
        else:
            fused.CAPTURE_RELU = cap
        if path == "fused_pair":
            F = list(net.forward_pair(T["sinput0_F"], T["sinput0_C"], T["sinput1_F"], T["sinput1_C"], dev))
        else:
            F = [net(me.SparseTensor(T[f"sinput{v}_F"], coords=T[f"sinput{v}_C"]).to("cuda")).F for v in "01"]
        l = losses.point_nce_loss(F[0], F[1], q.cuda(), k.cuda(), 0.4)
        l.backward()
    finally:
        me.FORCE_SIMT = False
        fused.CAPTURE_RELU = None
        for h in hooks:
            h.remove()
    assert len(cap) in (55, 110)
    if len(cap) == 55:                     # stacked: rows of view 0, then rows of view 1, in every unit
        masks = [m[:n0].cpu() for n0, m in cap] + [m[n0:].cpu() for n0, m in cap]
    else:
        masks = [m.cpu() for _, m in cap]
    pnet, Fp, lp, flips = _oracle_run(state, batch, q, k, torch.float64, masks)
    entries = sum(m.numel() for m in masks)
    assert max_rel_err(F[0], Fo[0]) < 1e-3 and max_rel_err(F[1], Fo[1]) < 1e-3          # features: against the oracle's own decisions
    assert abs(float(l.detach()) - float(lo.detach())) / abs(float(lo.detach())) < 1e-3
    assert abs(float(l.detach()) - float(lp.detach())) / abs(float(lp.detach())) < 1e-3
    names = [n for n, _ in net.named_parameters()]
    err = np.array([rel_err(p.grad, po.grad) for (_, p), (_, po) in zip(net.named_parameters(), pnet.named_parameters())])
    err_nat = np.array([rel_err(p.grad, po.grad) for (_, p), (_, po) in zip(net.named_parameters(), onet.named_parameters())])
    order = np.argsort(-err)
    report = [(names[i], float(err[i])) for i in order[:8]]
    if os.environ.get("PCB_REPORT_DIR"):
        import json
        json.dump({"path": path, "relu_entries": entries, "relu_flips_vs_fp64": int(sum(flips)),
                   "flips_by_call": [(i, f, int(masks[i].numel())) for i, f in enumerate(flips) if f],
                   "pinned_err_max": float(err.max()), "pinned_err_median": float(np.median(err)),
                   "unpinned_err_max": float(err_nat.max()), "unpinned_err_median": float(np.median(err_nat)), "worst_pinned": report},
                  open(os.path.join(os.environ["PCB_REPORT_DIR"], f"grad_pinned_{path}.json"), "w"), indent=1)
    assert sum(flips) <= 1e-4 * entries, (sum(flips), entries)
    assert (err <= 1e-3).all(), report
    assert err_nat.max() < 5e-2               # unpinned: a few coin flips; bounded, not meaningful beyond that
    for (n, b), (_, bo) in zip(net.named_buffers(), onet.named_buffers()):
        if b.dtype.is_floating_point:
            assert rel_err(b, bo) < 1e-3, n


def test_eval_mode_forward_matches_oracle_semseg_shape():
    """BASELINE config 5 shape: eval-mode BatchNorm, no L2 normalisation, 13 output classes, forward only."""
    from pointcontrast_b200 import me, synth
    from pointcontrast_b200.model import load_model
    sc = synth.synth_scene(0, scale=0.3, voxel=0.05, n_raw=60_000)
    cfg = refload.default_config(); cfg["net"]["normalize_feature"] = False
    net = load_model("Res16UNet34C")(3, 13, cfg, D=3)
    det_init(net, 2)
    for m in net.modules():
        if isinstance(m, torch.nn.BatchNorm1d):
            m.running_mean.uniform_(-0.1, 0.1); m.running_var.uniform_(0.5, 1.5)
    net = net.cuda().eval()
    with model_backend(OR) as mod:
        onet = mod.Res16UNet34C(3, 13, cfg, D=3).double()
        onet.load_state_dict({k: v.double().cpu() for k, v in net.state_dict().items()})
        onet.eval()
        with torch.no_grad():
            yo = onet(OR.SparseTensor(torch.from_numpy(sc["feats"]).double(), coords=torch.from_numpy(sc["coords"]))).F
    with torch.no_grad():
        y = net(me.SparseTensor(torch.from_numpy(sc["feats"]), coords=torch.from_numpy(sc["coords"])).to("cuda")).F
    assert y.shape == (len(sc["coords"]), 13) and max_rel_err(y, yo) < 1e-3


def test_fused_executor_matches_modular_path():
    """One-autograd-node fused executor (pointcontrast_b200/fused.py) vs the per-module ME-style path: same kernels, so
    features, every parameter gradient and the BatchNorm running statistics agree to fp32 rounding."""
    from pointcontrast_b200 import fused, losses, me, synth
    batch = synth.collate_pairs([synth.synth_pair(5, scale=0.15), synth.synth_pair(6, scale=0.12)])
    rng = np.random.default_rng(1)
    pairs = batch["correspondences"]
    nq = len(np.unique(pairs[:, 0]))
    q, k = loss_cpu.select_positives(pairs, rng.random(nq).astype(np.float32), 4096,
                                     rng.choice(nq, 4096, replace=False) if nq > 4096 else None)
    out = {}
    saved_fmt = me.FWD_FP16
    me.FWD_FP16 = False          # same operand format on both sides (the modular kernels split to bf16 hi/lo): this test is about the wiring
    for mode in (True, False):
        fused.ENABLED = mode
        try:
            net = _gpu_net(4)
            F = [net(me.SparseTensor(torch.from_numpy(batch[f"sinput{v}_F"]), coords=torch.from_numpy(batch[f"sinput{v}_C"])).to("cuda")).F
                 for v in "01"]
            loss = losses.point_nce_loss(F[0], F[1], q.cuda(), k.cuda(), 0.4)
            loss.backward()
            out[mode] = (F[0].detach(), F[1].detach(), float(loss.detach()), {n: p.grad.clone() for n, p in net.named_parameters()},
                         {n: b.clone() for n, b in net.named_buffers()})
        finally:
            fused.ENABLED = True
            if not mode:
                me.FWD_FP16 = saved_fmt
    a, b = out[True], out[False]
    assert max_rel_err(a[0], b[0]) < 1e-5 and max_rel_err(a[1], b[1]) < 1e-5 and abs(a[2] - b[2]) < 1e-5 * abs(b[2])
    worst = max((rel_err(a[3][n], b[3][n]), n) for n in b[3])
    assert worst[0] < 2e-4, worst
    for n in b[4]:
        if b[4][n].dtype.is_floating_point:
            assert rel_err(a[4][n], b[4][n]) < 1e-5, n
        else:
            assert (a[4][n] == b[4][n]).all(), n


def test_stacked_pair_pass_matches_two_forwards():
    """`forward_pair` with fused.PAIR: both views in one stacked pass (view 1's batch indices shifted, BatchNorm statistics
    per view through the row-segmented kernels) vs the reference's two forward calls: features, loss, every parameter
    gradient and the running statistics.  The passes differ only in fp32 summation order (split points of the small
    levels, one weight-gradient reduction instead of two); the network amplifies that to ~2e-4 on the features (each pass
    is ~3e-4 from the fp64 oracle, `__graft_entry__.smoke`) and the ill-conditioned backward further (see _grad_tol)."""
    from pointcontrast_b200 import fused, losses, synth
    batch = synth.collate_pairs([synth.synth_pair(5, scale=0.15), synth.synth_pair(6, scale=0.12)])
    rng = np.random.default_rng(1)
    pairs = batch["correspondences"]
    nq = len(np.unique(pairs[:, 0]))
    q, k = loss_cpu.select_positives(pairs, rng.random(nq).astype(np.float32), 4096,
                                     rng.choice(nq, 4096, replace=False) if nq > 4096 else None)
    out = {}
    saved = fused.PAIR
    for mode in (True, False):
        fused.PAIR = mode
        try:
            net = _gpu_net(4)
            F0, F1 = net.forward_pair(torch.from_numpy(batch["sinput0_F"]), torch.from_numpy(batch["sinput0_C"]),
                                      torch.from_numpy(batch["sinput1_F"]), torch.from_numpy(batch["sinput1_C"]), torch.device("cuda"))
            assert F0.shape[0] == len(batch["sinput0_C"]) and F1.shape[0] == len(batch["sinput1_C"])
            loss = losses.point_nce_loss(F0, F1, q.cuda(), k.cuda(), 0.4)
            loss.backward()
            out[mode] = (F0.detach(), F1.detach(), float(loss.detach()), {n: p.grad.clone() for n, p in net.named_parameters()},
                         {n: b.clone() for n, b in net.named_buffers()})
        finally:
            fused.PAIR = saved
    a, b = out[True], out[False]
    errs = sorted((rel_err(a[3][n], b[3][n]), n) for n in b[3])
    stats = max((rel_err(a[4][n], b[4][n]), n) for n in b[4] if b[4][n].dtype.is_floating_point)
    report = {"F0": max_rel_err(a[0], b[0]), "F1": max_rel_err(a[1], b[1]), "loss": abs(a[2] - b[2]) / abs(b[2]),
              "grad_worst": errs[-1], "grad_median": errs[len(errs) // 2], "running_stats_worst": stats}
    if os.environ.get("PCB_REPORT_DIR"):
        import json
        json.dump(report, open(os.path.join(os.environ["PCB_REPORT_DIR"], "stacked_vs_two_forwards.json"), "w"), indent=1)
    assert report["F0"] < 1e-3 and report["F1"] < 1e-3 and report["loss"] < 1e-5, report
    # measured (gpurun_out r44): features 1.9e-4 / 2.1e-4, loss 6e-8, gradients median 1.2e-2 / worst 1.6e-2, running
    # statistics 1.2e-5.  The gradient spread is the tensor-core path's own distance from fp64 on these tiny scenes
    # (median 2.3e-2, worst 3.5e-2 against a plain-fp32 floor of 3e-3 / 6e-3: test_small_scene_against_live_oracle...).
    assert errs[-1][0] < 5e-2 and errs[len(errs) // 2][0] < 3e-2, report
    assert stats[0] < 1e-3, report
    for n in b[4]:
        if not b[4][n].dtype.is_floating_point:
            assert (a[4][n] == b[4][n]).all(), n

"""Parity AT THE BENCHMARKED SHAPE (BASELINE configs[1]: ~41k / ~36k voxels per view, 2.5 cm; `bench.py` workload c1).

The small-scene tests (test_gpu_ops.py, test_gpu_model.py) only ever reach the offset-split + reduce mode of the
tensor-core convolution (`conv_splits` > 1 below ~38k output rows); the stride-1 / stride-2 layers of the benchmark, which
carry ~75 % of its bytes, run the DIRECT mode (TMEM -> Y epilogue with bias / accumulate, no partial sums).  This file
holds that mode, and the whole network at full C1 size, to the fp64 oracle:

  * one 96->96 and one 128->96 HYBRID 3x3x3 convolution at ~48k rows through the C ABI (`pcb_conv_forward_split`,
    `pcb_conv_wgrad_split`): forward with bias, forward with PCB_CONV_ACCUMULATE, data gradient, weight gradient;
  * ONE full-size scene pair through `forward_pair` (stacked pass, fused executor) + PointInfoNCE: per-point features,
    loss, every parameter gradient, per-offset kernel-map sizes of every level (`lib/ddp_trainer.py:392-426`);
  * the same features through the hardest-contrastive loss (`lib/ddp_trainer.py:186-238,290-308`).

Tolerances: 1e-3 relative on features and losses (north star); parameter gradients max(1e-3, 10 x the fp32-CPU floor of
the same graph), as in test_gpu_model.py.
"""
import numpy as np
import pytest
import torch

from oracle import loss_cpu
from oracle import me_cpu as OR
from tests import refload
from tests.helpers import det_init, max_rel_err, model_backend, rel_err, surface_coords

pytestmark = pytest.mark.gpu
TOL = 1e-3


def _split(x, flags=0):
    from pointcontrast_b200._lib import check, lib, ptr, stream
    n, C = x.shape
    planes = torch.empty(2, n * C, dtype=torch.bfloat16, device="cuda")
    check(lib.pcb_split_rows(ptr(x), C, n, C, planes[0].data_ptr(), planes[1].data_ptr(), C, flags, stream()))
    return planes


@pytest.mark.parametrize("cin,cout", [(96, 96), (128, 96)])
def test_direct_epilogue_conv_at_c1_rows(cin, cout):
    from pointcontrast_b200 import me
    from pointcontrast_b200._lib import check, lib, ptr, stream
    rng = np.random.default_rng(cin + cout)
    coords = surface_coords(rng, 60000, batches=2, extent=150)
    n = len(coords)
    assert n >= 40000
    # direct mode: no partial-sum workspace is requested for these shapes (conv_splits == 1), both role assignments
    assert lib.pcb_conv_forward_ws_bytes(27, n, cin, cout) == 256 and lib.pcb_conv_forward_ws_bytes(27, n, cout, cin) == 256
    g = torch.Generator().manual_seed(cin * 3 + cout)
    st = me.SparseTensor(torch.zeros(n, 1, device="cuda"), coords=torch.from_numpy(coords))
    kg = me.KernelGenerator(3, 1, 1, region_type=me.RegionType.HYBRID, axis_types=[me.RegionType.HYPERCUBE] * 3, dimension=3)
    plan = st.coords_man.conv_plan(st.coords_key, st.coords_key, kg, False)
    # fp64 oracle with autograd
    okg = OR.KernelGenerator(3, 1, 1, region_type=OR.RegionType.HYBRID, axis_types=[OR.RegionType.HYPERCUBE] * 3, dimension=3)
    oconv = OR.MinkowskiConvolution(in_channels=cin, out_channels=cout, kernel_size=3, stride=1, dilation=1, has_bias=True,
                                    kernel_generator=okg, dimension=3).double()
    W = oconv.kernel.detach().float()
    bias = oconv.bias.detach().float().reshape(-1)
    with torch.no_grad():
        oconv.kernel.copy_(W.double()); oconv.bias.copy_(bias.double()[None])
    x = torch.randn(n, cin, generator=g, dtype=torch.float64)
    dy = torch.randn(n, cout, generator=g, dtype=torch.float64)
    xo = x.clone().requires_grad_(True)
    yo = oconv(OR.SparseTensor(xo, coords=torch.from_numpy(coords))).F
    yo.backward(dy)
    # CUDA path through the C ABI
    Wd = W.cuda()
    ft = torch.zeros(lib.pcb_weight_tile_bytes(27, cin, cout, 0), dtype=torch.uint8, device="cuda")
    dt = torch.zeros(lib.pcb_weight_tile_bytes(27, cin, cout, 1), dtype=torch.uint8, device="cuda")
    check(lib.pcb_weight_tile(ptr(Wd), 27, cin, cout, ptr(ft), ptr(dt), 0, stream()))
    ws = torch.empty(256, dtype=torch.uint8, device="cuda")
    X = x.float().cuda(); DY = dy.float().cuda()
    Xs, DYs = _split(X), _split(DY)
    tbl = plan.fwd_tbl
    y = torch.empty(n, cout, device="cuda")
    check(lib.pcb_conv_forward_split(Xs[0].data_ptr(), Xs[1].data_ptr(), cin, ptr(tbl), tbl.shape[1], None, 27, n, cin, cout, ptr(ft),
                                     ptr(bias.cuda()), ptr(y), cout, ptr(ws), 256, 0, stream()))
    assert max_rel_err(y, yo) < TOL and rel_err(y, yo) < TOL / 10
    # accumulate onto existing contents, no bias
    base = torch.randn(n, cout, generator=g)
    y2 = base.clone().cuda()
    check(lib.pcb_conv_forward_split(Xs[0].data_ptr(), Xs[1].data_ptr(), cin, ptr(tbl), tbl.shape[1], None, 27, n, cin, cout, ptr(ft),
                                     None, ptr(y2), cout, ptr(ws), 256, 4, stream()))
    assert max_rel_err(y2 - base.cuda(), yo.detach() - bias.double()[None]) < TOL
    # data gradient: the same kernel on the data-gradient tiles and the opposite-offset permutation of the table
    dx = torch.empty(n, cin, device="cuda")
    check(lib.pcb_conv_forward_split(DYs[0].data_ptr(), DYs[1].data_ptr(), cout, ptr(plan.dg_tbl), plan.dg_tbl.shape[1],
                                     me._c_int_array(plan.dg_kmap), 27, n, cout, cin, ptr(dt), None, ptr(dx), cin, ptr(ws), 256, 0, stream()))
    assert max_rel_err(dx, xo.grad) < TOL and rel_err(dx, xo.grad) < TOL / 10
    # weight gradient (accumulated onto a non-zero buffer, as the fused executor does into the flat gradient)
    dW = torch.full((27, cin, cout), 0.125, device="cuda")
    wsb = lib.pcb_conv_wgrad_split_ws_bytes(27, n, cin, cout)
    wws = torch.empty(wsb, dtype=torch.uint8, device="cuda")
    check(lib.pcb_conv_wgrad_split(Xs[0].data_ptr(), Xs[1].data_ptr(), cin, DYs[0].data_ptr(), DYs[1].data_ptr(), cout, ptr(plan.wg_tbl),
                                   plan.wg_tbl.shape[1], 27, n, cin, cout, ptr(dW), 0, ptr(wws), wsb, 4, stream()))
    torch.cuda.synchronize()
    assert max_rel_err(dW - 0.125, oconv.kernel.grad) < TOL and rel_err(dW - 0.125, oconv.kernel.grad) < TOL / 10
    # fp16 hi/lo activation planes x fp16 weight tiles (the fused executor's forward format, PCB_FWD_FP16): 2^-22 products
    ft16 = torch.zeros_like(ft); dt16 = torch.zeros_like(dt)
    check(lib.pcb_weight_tile(ptr(Wd), 27, cin, cout, ptr(ft16), ptr(dt16), 16, stream()))
    assert torch.equal(dt16, dt)                                   # the data-gradient tiles stay bf16
    Xs16 = _split(X, 8)
    y16 = torch.empty(n, cout, device="cuda")
    check(lib.pcb_conv_forward_split(Xs16[0].data_ptr(), Xs16[1].data_ptr(), cin, ptr(tbl), tbl.shape[1], None, 27, n, cin, cout, ptr(ft16),
                                     ptr(bias.cuda()), ptr(y16), cout, ptr(ws), 256, 8 | 16, stream()))
    e_bf16, e_fp16 = rel_err(y, yo), rel_err(y16, yo)
    # measured: 4.8e-6 (bf16 hi/lo) vs 2.1e-6 (fp16 hi/lo: what is left is the fp32 accumulation over 27 x Cin terms)
    assert e_fp16 < 0.6 * e_bf16 and max_rel_err(y16, yo) < 1e-4, (e_bf16, e_fp16)
    # (tcgen05.mma rejects mixed fp16 x bf16 operands -- profiles/probes/mixed_fmt_probe.cu -- so the weight gradient keeps reading
    #  the bf16 planes of the activations, checked above)

# ----------------------------------------------------------------------------------------------- one full C1 pair
def _oracle(state, batch, dtype, masks=None, flips=None):
    import contextlib
    from tests.helpers import pinned_relu
    with (pinned_relu(OR, masks, flips) if masks is not None else contextlib.nullcontext()), model_backend(OR) as mod:
        onet = mod.Res16UNet34C(3, 32, refload.default_config(), D=3).to(dtype)
        onet.load_state_dict({k: (v.to(dtype) if v.dtype.is_floating_point else v) for k, v in state.items()})
        onet.train()
        Fo = [onet(OR.SparseTensor(torch.from_numpy(batch[f"sinput{v}_F"]).to(dtype), coords=torch.from_numpy(batch[f"sinput{v}_C"]))).F
              for v in "01"]
    return onet, Fo


@pytest.fixture(scope="module")
def c1():
    """One full-size pair on the GPU (stacked pass + PointInfoNCE + backward) and on the fp64 oracle, twice: taking its own ReLU
    decisions, and replaying the GPU pass's (tests/test_gpu_model.py::test_small_scene_all_gradients_with_pinned_relu_decisions)."""
    from pointcontrast_b200 import fused, losses, synth
    from pointcontrast_b200.model import load_model
    assert fused.PAIR
    batch = synth.collate_pairs([synth.synth_pair(0, scale=0.9)])
    assert len(batch["sinput0_C"]) > 38000 and len(batch["sinput1_C"]) > 34000
    net = load_model("Res16UNet34C")(3, 32, refload.default_config(), D=3)
    det_init(net, 5)
    state = {k: v.clone() for k, v in net.state_dict().items()}
    net = net.cuda().train()
    rng = np.random.default_rng(7)
    pairs = batch["correspondences"]
    nq = len(np.unique(pairs[:, 0]))
    q, k = loss_cpu.select_positives(pairs, rng.random(nq).astype(np.float32), 4096, rng.choice(nq, 4096, replace=False))
    fused.CAPTURE_RELU = cap = []
    try:
        F0, F1 = net.forward_pair(torch.from_numpy(batch["sinput0_F"]), torch.from_numpy(batch["sinput0_C"]),
                                  torch.from_numpy(batch["sinput1_F"]), torch.from_numpy(batch["sinput1_C"]), torch.device("cuda"))
    finally:
        fused.CAPTURE_RELU = None
    assert "_fused_runner" in net.__dict__ and len(cap) == 55
    masks = [m[:n0].cpu() for n0, m in cap] + [m[n0:].cpu() for n0, m in cap]
    loss = losses.point_nce_loss(F0, F1, q.cuda(), k.cuda(), 0.4)
    loss.backward()
    torch.cuda.synchronize()
    onet, Fo = _oracle(state, batch, torch.float64)
    lo = loss_cpu.point_nce_loss(Fo[0], Fo[1], q, k, 0.4)
    lo.backward()
    flips = []
    pnet, Fp = _oracle(state, batch, torch.float64, masks, flips)
    loss_cpu.point_nce_loss(Fp[0], Fp[1], q, k, 0.4).backward()
    return dict(batch=batch, net=net, F=(F0.detach(), F1.detach()), loss=float(loss.detach()), onet=onet, Fo=[f.detach() for f in Fo],
                lo=float(lo.detach()), pnet=pnet, flips=flips, relu_entries=sum(m.numel() for m in masks),
                flip_sizes=[int(m.numel()) for m in masks], rng=rng)


def test_c1_pair_features_and_loss(c1):
    assert max_rel_err(c1["F"][0], c1["Fo"][0]) < TOL and max_rel_err(c1["F"][1], c1["Fo"][1]) < TOL
    assert abs(c1["loss"] - c1["lo"]) / abs(c1["lo"]) < TOL


def test_c1_pair_every_parameter_gradient(c1):
    """All 187 parameter gradients of the full-size pair at the north-star tolerance, the fp64 oracle replaying the GPU pass's ReLU
    decisions; those decisions may differ from the oracle's own on < 1e-4 of the entries (pre-activations within rounding of zero)."""
    import json
    import os
    net, onet, pnet = c1["net"], c1["onet"], c1["pnet"]
    names = [n for n, _ in net.named_parameters()]
    err = np.array([rel_err(p.grad, po.grad) for (_, p), (_, po) in zip(net.named_parameters(), pnet.named_parameters())])
    err_nat = np.array([rel_err(p.grad, po.grad) for (_, p), (_, po) in zip(net.named_parameters(), onet.named_parameters())])
    order = np.argsort(-err)
    flips = c1["flips"]
    report = {"relu_entries": c1["relu_entries"], "relu_flips_vs_fp64": int(sum(flips)),
              "flips_by_call": [(i, f, c1["flip_sizes"][i]) for i, f in enumerate(flips) if f],
              "pinned_err_max": float(err.max()), "pinned_err_median": float(np.median(err)),
              "unpinned_err_max": float(err_nat.max()), "unpinned_err_median": float(np.median(err_nat)),
              "worst_pinned": [(names[i], float(err[i])) for i in order[:8]]}
    if os.environ.get("PCB_REPORT_DIR"):
        json.dump(report, open(os.path.join(os.environ["PCB_REPORT_DIR"], "c1_grad_report.json"), "w"), indent=1)
    assert sum(flips) <= 1e-4 * c1["relu_entries"], report
    assert (err <= 1e-3).all(), report
    assert err_nat.max() < 5e-2, report
    for (n, b), (_, bo) in zip(net.named_buffers(), onet.named_buffers()):        # BatchNorm running statistics after view 0, view 1
        if b.dtype.is_floating_point:
            assert rel_err(b, bo) < 1e-3, n


def test_c1_pair_kernel_map_sizes_per_offset(c1):
    """|M_k| of every level / kernel of the STACKED coordinate manager == view 0's + view 1's on the oracle (bit-exact)."""
    from pointcontrast_b200 import fused, me
    b = c1["batch"]
    s, n0 = fused.stack_views(torch.from_numpy(b["sinput0_F"]), torch.from_numpy(b["sinput0_C"]), torch.from_numpy(b["sinput1_F"]),
                              torch.from_numpy(b["sinput1_C"]), torch.device("cuda"))
    cm, key = s.coords_man, s.coords_key
    ocms = [OR.CoordsManager(3), OR.CoordsManager(3)]
    okeys = [ocm.initialize(b[f"sinput{v}_C"], [1, 1, 1]) for v, ocm in zip("01", ocms)]
    hyb = me.KernelGenerator(3, 1, 1, region_type=me.RegionType.HYBRID, axis_types=[me.RegionType.HYPERCUBE] * 3, dimension=3)
    ohyb = OR.KernelGenerator(3, 1, 1, region_type=OR.RegionType.HYBRID, axis_types=[OR.RegionType.HYPERCUBE] * 3, dimension=3)
    k2 = me.KernelGenerator([2, 2, 2], 2, 1, dimension=3)
    ok2 = OR.KernelGenerator([2, 2, 2], 2, 1, dimension=3)
    for level in range(5):
        got = cm.conv_plan(key, key, hyb, False).pair_counts()
        ref = [sum(len(ocm.get_kernel_map(ok, ok, ohyb, False)[kk][0]) for ocm, ok in zip(ocms, okeys)) for kk in range(27)]
        assert got == ref, level
        assert cm.num_rows(key) == sum(len(ocm.levels[ok.ts]) for ocm, ok in zip(ocms, okeys))
        if level == 4:
            break
        nkey = cm.stride(key, [2, 2, 2])
        onkeys = [ocm.stride(ok, [2, 2, 2]) for ocm, ok in zip(ocms, okeys)]
        got = cm.conv_plan(key, nkey, k2, False).pair_counts()
        ref = [sum(len(ocm.get_kernel_map(ok, onk, ok2, False)[kk][0]) for ocm, ok, onk in zip(ocms, okeys, onkeys)) for kk in range(8)]
        assert got == ref, level
        key, okeys = nkey, onkeys


def test_c1_pair_hardest_contrastive_loss(c1):
    """`HardestContrastiveLossTrainer` loss (`lib/ddp_trainer.py:186-238`) on the full-size features: GPU kernels
    (`pcb_pdist_rowmin` + device-side false-negative mask) vs the oracle's restatement on the oracle's fp64 features."""
    from pointcontrast_b200 import losses
    b = c1["batch"]
    rng = np.random.default_rng(11)
    pairs = b["correspondences"]
    N0, N1 = len(b["sinput0_C"]), len(b["sinput1_C"])
    sel0 = rng.choice(N0, 1024, replace=False); sel1 = rng.choice(N1, 1024, replace=False)
    pos_sel = rng.choice(len(pairs), 4096, replace=False)
    f0o, f1o = c1["Fo"][0].clone().requires_grad_(True), c1["Fo"][1].clone().requires_grad_(True)
    po, no = loss_cpu.hardest_contrastive_loss(f0o, f1o, pairs, sel0, sel1, pos_sel)
    (po + no).backward()
    f0, f1 = c1["F"][0].clone().requires_grad_(True), c1["F"][1].clone().requires_grad_(True)
    p, n_ = losses.hardest_contrastive_loss(f0, f1, torch.from_numpy(pairs).cuda(), torch.from_numpy(sel0).cuda(),
                                            torch.from_numpy(sel1).cuda(), torch.from_numpy(pos_sel).cuda())
    (p + n_).backward()
    assert abs(float(p) - float(po)) <= TOL * max(abs(float(po)), 1e-3) and abs(float(n_) - float(no)) <= TOL * abs(float(no))
    # the hardest negative of a positive may switch between near-tied candidates under 3e-4 feature noise: gradients to 1e-2
    assert rel_err(f0.grad, f0o.grad) < 1e-2 and rel_err(f1.grad, f1o.grad) < 1e-2


def test_fused_reduce_statistics_match_separate_pass(c1):
    """BatchNorm statistics from the offset-split convolutions' reduction pass (default on the small levels) vs a separate
    column-statistics pass over z everywhere (PCB_UNIT_SEPARATE_STATS): same numbers up to fp32 summation order."""
    from pointcontrast_b200 import fused
    from pointcontrast_b200.model import load_model
    b = c1["batch"]
    outs = {}
    for sep in (False, True):
        fused.SEPARATE_STATS = sep
        try:
            net = load_model("Res16UNet34C")(3, 32, refload.default_config(), D=3)
            det_init(net, 5)
            net = net.cuda().train()
            F0, F1 = net.forward_pair(torch.from_numpy(b["sinput0_F"]), torch.from_numpy(b["sinput0_C"]), torch.from_numpy(b["sinput1_F"]),
                                      torch.from_numpy(b["sinput1_C"]), torch.device("cuda"))
            outs[sep] = (F0.detach(), F1.detach(), {n: v.clone() for n, v in net.named_buffers() if v.dtype.is_floating_point})
        finally:
            fused.SEPARATE_STATS = False
    assert max_rel_err(outs[False][0], outs[True][0]) < 2e-5 and max_rel_err(outs[False][1], outs[True][1]) < 2e-5
    for n in outs[True][2]:
        assert rel_err(outs[False][2][n], outs[True][2][n]) < 1e-5, n
    assert torch.equal(outs[False][0], c1["F"][0])            # the default path is the one the other tests of this file checked

"""Semantic-segmentation evaluation on the GPU (`downstream/semseg/lib/test.py::test`, SURVEY.md 8f-5): pcb_seg_eval against the
numpy oracle (oracle/seg_metrics_cpu.py), its determinism and accumulation, SegmentationMeter without host synchronisation,
semseg.test against the original code's recorded 4-tuple, and evaluation of Res16UNet34C end to end."""
import numpy as np
import pytest
import torch

from oracle import seg_metrics_cpu as SM
from tests import refload
from tests.helpers import det_init
from tests.semseg_eval_common import FIXTURE, IGNORE, NUM_LABELS, StandInLoader, StandInModel, fixture_batches, make_batch

pytestmark = pytest.mark.gpu


def _seg_eval(x, t, C, hist=None, ignore=IGNORE):
    """One pcb_seg_eval call on device tensors; returns pred, hist, stats, ap, prob (device)."""
    from pointcontrast_b200 import _lib
    n = x.shape[0]
    pred = torch.empty(n, dtype=torch.int32, device="cuda")
    hist = torch.zeros(C, C, dtype=torch.int64, device="cuda") if hist is None else hist
    stats = torch.empty(4, dtype=torch.float64, device="cuda")
    ap = torch.empty(C, dtype=torch.float64, device="cuda")
    prob = torch.empty(n, C, dtype=torch.float32, device="cuda")
    ws = torch.empty(int(_lib.lib.pcb_seg_eval_ws_bytes(n, C)), dtype=torch.uint8, device="cuda")
    _lib.check(_lib.lib.pcb_seg_eval(x.data_ptr(), t.data_ptr(), n, C, ignore, pred.data_ptr(), hist.data_ptr(), stats.data_ptr(),
                                     ap.data_ptr(), prob.data_ptr(), ws.data_ptr(), ws.numel(), _lib.stream()))
    return pred, hist, stats, ap, prob


def _inputs(n, C, seed):
    """make_batch's ties and ignored rows, plus one absent class and one out-of-range target (when n allows)."""
    x, t = make_batch(seed, n, C) if n >= 4 * C else (np.random.default_rng(seed).normal(size=(n, C)).astype(np.float32),
                                                       np.random.default_rng(seed).integers(0, C, n))
    if n >= 4 * C:
        t[t == C - 1] = IGNORE                                 # class C-1 has no positive
        t[C] = C + 3                                           # out of range: an ignored row
    return x, t


@pytest.mark.parametrize("n,C", [(1, 13), (1000, 13), (107_750, 13), (50_000, 20), (3000, 64), ((1 << 20) + 3, 13)])
def test_seg_eval_matches_oracle(n, C):
    x, t = _inputs(n, C, seed=n + C)
    xd, td = torch.from_numpy(x).cuda(), torch.from_numpy(t).cuda()
    pred, hist, stats, ap, prob = _seg_eval(xd, td, C)
    torch.cuda.synchronize()
    assert torch.equal(pred.long(), xd.argmax(1))
    ok = SM.valid_rows(t, C, IGNORE)
    p = pred.cpu().numpy()
    assert (hist.cpu().numpy() == SM.fast_hist(p[ok], t[ok], C)).all()
    st = stats.cpu().numpy()
    assert st[1] == ok.sum() and st[2] == (p[ok] == t[ok]).sum() and st[3] == n
    if ok.any():
        ce = SM.cross_entropy(x, t, IGNORE)
        assert abs(st[0] / st[1] - ce) <= 1e-6 * abs(ce)
    ref_prob = torch.softmax(xd, 1)
    torch.testing.assert_close(prob, ref_prob, rtol=1e-6, atol=1e-30)
    ap_own = SM.average_precision(prob.cpu().numpy(), t, IGNORE)
    a = ap.cpu().numpy()
    assert (np.isnan(a) == np.isnan(ap_own)).all()
    np.testing.assert_allclose(a, ap_own, rtol=1e-12, atol=1e-14)
    ap_torch = SM.average_precision(ref_prob.cpu().numpy(), t, IGNORE)
    assert (np.isnan(a) == np.isnan(ap_torch)).all()
    np.testing.assert_allclose(a, ap_torch, rtol=0, atol=1e-5)
    if n >= 4 * C:
        assert np.isnan(a[C - 1]) and not np.isnan(a[:C - 1]).any()


def test_seg_eval_is_deterministic_and_accumulates():
    x, t = _inputs(107_750, 13, seed=5)
    xd, td = torch.from_numpy(x).cuda(), torch.from_numpy(t).cuda()
    _, h1, s1, a1, _ = _seg_eval(xd, td, 13)
    h1 = h1.clone()
    _, h2, s2, a2, _ = _seg_eval(xd, td, 13, hist=h1.clone())
    assert torch.equal(s1, s2) and torch.equal(a1.isnan(), a2.isnan()) and torch.equal(a1.nan_to_num(), a2.nan_to_num())
    assert torch.equal(h2, 2 * h1)


def test_seg_eval_all_rows_ignored():
    x, _ = _inputs(5000, 13, seed=6)
    t = np.full(5000, IGNORE, dtype=np.int64)
    h0 = torch.arange(169, dtype=torch.int64, device="cuda").reshape(13, 13)
    _, h, st, ap, _ = _seg_eval(torch.from_numpy(x).cuda(), torch.from_numpy(t).cuda(), 13, hist=h0.clone())
    st = st.cpu()
    assert st[1] == 0 and st[2] == 0 and st[0] == 0
    assert torch.isnan(st[0] / st[1]) and torch.isnan(st[2] * 100 / st[1]) and ap.isnan().all()
    assert torch.equal(h, h0)


def test_meter_update_never_synchronises():
    from pointcontrast_b200 import semseg
    batches = [(torch.from_numpy(x).cuda(), torch.from_numpy(t).cuda()) for x, t in fixture_batches()[:3]]
    m = semseg.SegmentationMeter(NUM_LABELS, IGNORE)
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        preds = [m.update(x, t) for x, t in batches]
    finally:
        torch.cuda.set_sync_debug_mode("default")
    s = m.summary()
    e = SM.evaluate([(x.cpu().numpy(), t.cpu().numpy()) for x, t in batches], NUM_LABELS, IGNORE)
    for p, (x, _) in zip(preds, batches):
        assert torch.equal(p.long(), x.argmax(1))
    assert (s["hist"] == e["hist"]).all()
    assert abs(s["score"] - e["score"]) <= 1e-12 * abs(e["score"]) and abs(s["loss"] - e["loss"]) <= 1e-6 * abs(e["loss"])
    assert abs(s["mAP"] - e["mAP"]) < 1e-3 and abs(s["mIoU"] - e["mIoU"]) <= 1e-12 * abs(e["mIoU"])


def _test_config(freq=2):
    return refload.Cfg(data=dict(ignore_label=IGNORE, return_transformation=False), net=dict(wrapper_type=None),
                       augmentation=dict(normalize_color=True),
                       test=dict(save_prediction=False, test_original_pointcloud=False, evaluate_original_pointcloud=False, test_stat_freq=freq))


def test_semseg_test_reproduces_the_reference_loop():
    """The original `lib/test.py::test` 4-tuple recorded on the same batches: precision@1 to the fp32 rounding of the original's
    `precision_at_one`, mIoU to fp64 rounding (integer histogram), loss to 1e-6, mAP to 1e-3 percent (the original ranks by torch's
    softmax, the kernel by its own: probabilities a few ulp apart can split or merge a tie)."""
    from pointcontrast_b200 import semseg
    batches = fixture_batches()
    loss, score, mAP, mIoU = semseg.test(StandInModel(batches), StandInLoader(batches), _test_config())
    rl, rs, rm, ri = np.load(FIXTURE)["test"]
    assert abs(score - rs) <= 1e-6 * abs(rs) and abs(mIoU - ri) <= 1e-12 * abs(ri)
    assert abs(loss - rl) <= 1e-6 * abs(rl) and abs(mAP - rm) < 1e-3


class _Capture(torch.nn.Module):
    def __init__(self, net):
        super().__init__()
        self.net = net
        self.outputs = []

    def forward(self, x):
        out = self.net(x)
        self.outputs.append(out.F.clone())
        return out


class _Loader:
    def __init__(self, batches):
        self.batches = batches
        self.dataset = type("D", (), {"NUM_LABELS": NUM_LABELS})()

    def __len__(self):
        return len(self.batches)

    def __iter__(self):
        return iter([(c, f.clone(), t) for c, f, t in self.batches])


def test_evaluation_end_to_end():
    from pointcontrast_b200 import me, semseg, synth
    from pointcontrast_b200.model import load_model
    mcfg = refload.default_config(); mcfg["net"]["normalize_feature"] = False
    rng = np.random.default_rng(11)
    batches = []
    for s in (0, 1):
        sc = synth.synth_scene(s, scale=0.25, voxel=0.05, n_raw=40_000)
        t = rng.integers(0, NUM_LABELS, len(sc["coords"])); t[rng.random(len(t)) < 0.1] = IGNORE
        feats = (torch.from_numpy(sc["feats"]) + 0.5) * 255.0                 # colours; test() normalises them
        batches.append((torch.from_numpy(sc["coords"]), feats, torch.from_numpy(t)))
    net = load_model("Res16UNet34C")(3, NUM_LABELS, mcfg, D=3)
    det_init(net, 4)
    net = net.cuda().eval()
    with torch.no_grad():
        logits = [net(me.SparseTensor(f / 255. - 0.5, c).to("cuda")).F.clone() for c, f, _ in batches]
    cap = _Capture(net)
    got = semseg.test(cap, _Loader(batches), _test_config(freq=100))
    for a, b in zip(cap.outputs, logits):
        assert torch.equal(a, b)                                                # the eval executor is deterministic
    e = SM.evaluate([(x.cpu().numpy(), t.numpy()) for x, (_, _, t) in zip(logits, batches)], NUM_LABELS, IGNORE)
    want = (e["loss"], e["score"], e["mAP"], e["mIoU"])
    for g, w, tol in zip(got, want, (1e-6, 1e-9, 1e-3, 1e-9)):
        assert abs(g - w) <= tol * max(1.0, abs(w)), (got, want)
    cfg = refload.Cfg(dict(_test_config(freq=100)), optimizer=dict(optimizer="SGD", lr=0.01, sgd_momentum=0.9, sgd_dampening=0.1,
                                                                   weight_decay=1e-4, iter_size=1, scheduler="PolyLR", max_iter=100,
                                                                   poly_power=0.9))
    tr = semseg.SegmentationTrainer(net, cfg)
    net.train()
    miou = tr.validate(_Loader(batches))
    assert miou == got[3] and net.training

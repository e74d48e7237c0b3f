"""Semantic-segmentation evaluation without a GPU: the numpy oracle (oracle/seg_metrics_cpu.py) against scikit-learn and against the
original evaluation code's recorded outputs (tests/golden/semseg_eval_reference.npz), the argument checks of pcb_seg_eval, and the
host-side refusals of semseg.test / SegmentationMeter."""
import numpy as np
import pytest
import torch

from oracle import seg_metrics_cpu as SM
from tests import refload
from tests.semseg_eval_common import FIXTURE, IGNORE, NUM_LABELS, StandInLoader, fixture_batches, make_batch


def _random_batch(seed, n=20_000, C=13):
    x, t = make_batch(seed, n, C)
    x[:500] = 0.0                                              # one more all-tied block
    return SM.softmax(x).astype(np.float32), t, x


def test_oracle_ap_equals_scikit_learn():
    sk = pytest.importorskip("sklearn.metrics")
    prob, t, _ = _random_batch(3)
    ap = SM.average_precision(prob, t, IGNORE)
    for c in range(prob.shape[1]):
        ref = sk.average_precision_score(t == c, prob[:, c])
        assert abs(ap[c] - ref) < 1e-12, c


def test_oracle_ap_is_nan_for_a_class_without_positives():
    prob, t, x = _random_batch(4, n=3000)
    t[t == 5] = IGNORE
    t[0] = 7                                                   # out-of-range targets are ignored rows too
    t[1] = -1
    ap = SM.average_precision(prob, t, IGNORE)
    assert np.isnan(ap[5]) and not np.isnan(np.delete(ap, 5)).any()
    m = SM.evaluate([(x, t, prob)], NUM_LABELS, IGNORE)
    assert np.isnan(m["ap_class"][5]) and np.isnan(m["acc"][5]) and m["ious"][5] == 0 and np.isfinite(m["mAP"])
    allign = np.full_like(t, IGNORE)
    b = SM.batch_metrics(x, allign, NUM_LABELS, IGNORE, prob)
    assert np.isnan(b["loss"]) and np.isnan(b["score"]) and np.isnan(b["ap"]).all() and b["hist"].sum() == 0


def test_oracle_reproduces_the_reference_fixture():
    """The original code's own outputs.  Its loss and precision@1 are computed in fp32 (nn.CrossEntropyLoss on fp32 logits,
    `correct.float().sum(0).mul(100 / count)`), so those agree to fp32 rounding; histogram, IoU and AP to 1e-12."""
    ref = np.load(FIXTURE)
    batches = fixture_batches()
    for b, (x, t) in enumerate(batches):
        m = SM.batch_metrics(x, t, NUM_LABELS, IGNORE, ref[f"prob_{b}"])
        assert (m["hist"] == ref[f"hist_{b}"]).all()
        np.testing.assert_allclose(SM.per_class_iu(m["hist"]), ref[f"iu_{b}"], rtol=1e-12, atol=0)
        np.testing.assert_allclose(m["ap"], ref[f"ap_{b}"], rtol=1e-12, atol=1e-15)
        assert abs(m["score"] - ref[f"score_{b}"]) <= 1e-6 * abs(ref[f"score_{b}"])
        assert abs(m["loss"] - ref[f"loss_{b}"]) <= 1e-6 * abs(ref[f"loss_{b}"])
    e = SM.evaluate([(x, t, ref[f"prob_{b}"]) for b, (x, t) in enumerate(batches)], NUM_LABELS, IGNORE)
    loss, score, mAP, mIoU = ref["test"]
    assert abs(e["loss"] - loss) <= 1e-6 * abs(loss) and abs(e["score"] - score) <= 1e-6 * abs(score)
    assert abs(e["mAP"] - mAP) <= 1e-12 * abs(mAP) and abs(e["mIoU"] - mIoU) <= 1e-12 * abs(mIoU)


def test_seg_eval_argument_errors_do_not_need_a_gpu():
    from pointcontrast_b200 import _lib
    L = _lib.lib
    big = 1 << 40
    for n, C in ((100, 1), (100, 65), (0, 13), ((1 << 31) // 13 + 1, 13)):
        rc = L.pcb_seg_eval(big, big, n, C, 255, None, big, big, big, None, big, 1 << 40, None)
        assert rc == 2 and b"bad argument" in L.pcb_last_error(), (n, C)
    assert L.pcb_seg_eval(None, big, 100, 13, 255, None, big, big, big, None, big, 1 << 40, None) == 2    # logits
    assert L.pcb_seg_eval(big, big, 100, 13, 255, None, None, big, big, None, big, 1 << 40, None) == 2     # hist
    assert L.pcb_seg_eval(big, big, 100, 13, 255, None, big, big, big, None, big, 16, None) == 2          # workspace too small
    assert L.pcb_seg_eval_ws_bytes(200_000, 13) > L.pcb_seg_eval_ws_bytes(100_000, 13) >= 3 * 8 * 13 * 100_000


def test_semseg_test_refuses_unsupported_options_before_touching_a_device():
    from pointcontrast_b200 import semseg
    loader = StandInLoader(fixture_batches()[:1])

    def cfg(**over):
        c = refload.Cfg(data=dict(ignore_label=IGNORE), net=dict(wrapper_type=None), augmentation=dict(normalize_color=True),
                        test=dict(save_prediction=False, test_original_pointcloud=False, evaluate_original_pointcloud=False, test_stat_freq=10))
        for k, v in over.items():
            a, b = k.split("__")
            c[a][b] = v
        return c

    class NoModel:
        def eval(self):
            raise AssertionError("touched the model")

    for over in (dict(net__wrapper_type="CRF"), dict(test__save_prediction=True), dict(test__test_original_pointcloud=True),
                 dict(test__evaluate_original_pointcloud=True)):
        with pytest.raises(NotImplementedError):
            semseg.test(NoModel(), loader, cfg(**over))
    with pytest.raises(NotImplementedError):
        semseg.test(NoModel(), loader, cfg(), has_gt=False)


def test_segmentation_meter_has_no_cpu_path():
    from pointcontrast_b200 import _lib, semseg
    with pytest.raises(_lib.PcbError):
        semseg.SegmentationMeter(NUM_LABELS, IGNORE, device="cpu")
    m = semseg.SegmentationMeter(NUM_LABELS, IGNORE) if torch.cuda.is_available() else object.__new__(semseg.SegmentationMeter)
    with pytest.raises(_lib.PcbError):
        m.update(torch.zeros(4, NUM_LABELS), torch.zeros(4, dtype=torch.int64))

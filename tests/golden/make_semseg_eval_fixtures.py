"""Generates semseg_eval_reference.npz: the original semantic-segmentation evaluation code on the batches of
tests/semseg_eval_common.py (run where the original project's `downstream/semseg` package and scikit-learn can be imported):

    python tests/golden/make_semseg_eval_fixtures.py [path/to/downstream/semseg]

Per batch b: the softmax the original loop ranks by (prob_b, torch on the CPU), and the original `lib/utils.py` / `lib/test.py`
helpers' outputs: fast_hist (hist_b), per_class_iu of that histogram (iu_b), precision_at_one (score_b), average_precision (ap_b),
nn.CrossEntropyLoss (loss_b).  `test` = the 4-tuple (loss, precision@1, mAP, mIoU) returned by the original `lib/test.py::test`,
driven on the CPU by a stand-in model that returns the stored logits.  Every class has a positive in every batch, so the
scikit-learn version's convention for a class without positives does not enter.
"""
import os
import sys
import types

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

from oracle import me_cpu                                    # noqa: E402
from tests import refload                                    # noqa: E402
from tests.semseg_eval_common import (FIXTURE, IGNORE, NUM_LABELS, StandInLoader, StandInModel,   # noqa: E402
                                      fixture_batches)


def load_reference(semseg_dir):
    """lib.utils / lib.test of the original semseg package.  Its lib/__init__.py imports open3d and lib/utils.py imports omegaconf and
    lib.pc_utils (plyfile, pandas), none of which the evaluation uses: stubbed.  MinkowskiEngine is the CPU oracle."""
    me_cpu.install()
    for k in [k for k in sys.modules if k == "lib" or k.startswith("lib.")]:
        del sys.modules[k]
    sys.modules.setdefault("open3d", types.ModuleType("open3d"))
    om = types.ModuleType("omegaconf")
    om.OmegaConf = object
    sys.modules["omegaconf"] = om
    pc = types.ModuleType("lib.pc_utils")
    pc.colorize_pointcloud = pc.save_point_cloud = None
    sys.modules["lib.pc_utils"] = pc
    sys.path.insert(0, semseg_dir)
    try:
        import lib.test as ref_test
        import lib.utils as ref_utils
    finally:
        sys.path.remove(semseg_dir)
    return ref_utils, ref_test


def main(semseg_dir):
    ref_utils, ref_test = load_reference(semseg_dir)
    batches = fixture_batches()
    out = {}
    for b, (x, t) in enumerate(batches):
        assert all(((t == c).sum() > 0) for c in range(NUM_LABELS))
        logits = torch.from_numpy(x)
        pred = ref_utils.get_prediction(None, logits, None).int()
        target = torch.from_numpy(t)
        prob = torch.nn.functional.softmax(logits, dim=1)
        hist = ref_utils.fast_hist(pred.numpy().flatten(), t.flatten(), NUM_LABELS)
        out[f"prob_{b}"] = prob.numpy()
        out[f"hist_{b}"] = hist.astype(np.int64)
        out[f"iu_{b}"] = ref_utils.per_class_iu(hist)
        out[f"score_{b}"] = np.float64(ref_utils.precision_at_one(pred, target))
        out[f"ap_{b}"] = ref_test.average_precision(prob.numpy(), t)
        out[f"loss_{b}"] = np.float64(torch.nn.CrossEntropyLoss(ignore_index=IGNORE)(logits, target.long()))
    cfg = refload.Cfg(misc=dict(is_cuda=False), data=dict(ignore_label=IGNORE, return_transformation=False),
                      net=dict(wrapper_type=None), augmentation=dict(normalize_color=True),
                      test=dict(save_prediction=False, test_original_pointcloud=False, evaluate_original_pointcloud=False, test_stat_freq=2),
                      train=dict(empty_cache_freq=1))
    torch.cuda.empty_cache = lambda: None                    # the loop calls it; there is no device here
    out["test"] = np.array(ref_test.test(StandInModel(batches), StandInLoader(batches), cfg), dtype=np.float64)
    np.savez_compressed(FIXTURE, **out)
    print(FIXTURE, out["test"])


if __name__ == "__main__":
    main(sys.argv[1] if len(sys.argv) > 1 else "/root/reference/downstream/semseg")

"""Semantic-segmentation finetune step on the same backbone (SURVEY.md 8f-1): mirror of `downstream/semseg/lib/train.py:46-232`
(the optimisation step of the loop, not its logging / validation / tensorboard shell), `lib/solvers.py:27-83` (SGD with
dampening, PolyLR) and `lib/utils.py:19-43` (lenient loading of pretraining checkpoints into a model with a different head).

    model = load_model("Res16UNet34C")(3, num_labels, config, D=3)           # `normalize_feature` False: logits
    load_state_with_same_shape(model, torch.load("weights.pth")["state_dict"])   # PointContrast backbone, fresh `final` layer
    trainer = SegmentationTrainer(model, config)
    loss = trainer.train_step([(coords, feats, target), ...])                 # len == config.optimizer.iter_size

Everything numerical runs on libpcb200: the fused executor (the 13 / 20-class head on the exact fp32 kernels), the cross-entropy
kernels (`pcb_ce_forward_backward`), the flat SGD kernel with dampening.

Evaluation (SURVEY.md 8f-5) mirrors `downstream/semseg/lib/test.py::test` and `lib/train.py::validate`:

    loss, score, mAP, mIoU = test(model, val_loader, config)        # or trainer.validate(val_loader) -> mIoU

with every metric (prediction, cross-entropy, precision@1, confusion histogram, per-class average precision) computed on the device
by `pcb_seg_eval` and folded across batches by `SegmentationMeter` without a host round trip.
"""
import logging
import time
import warnings

import numpy as np
import torch

from . import _lib, losses, me as ME
from .optim import FlatSGD, PolyLR


def load_state_with_same_shape(model, weights):
    """`downstream/semseg/lib/utils.py:19-43`: keep the checkpoint entries whose name and shape match the model (drops a `final`
    head of another width), stripping the `module.` / `encoder.` prefixes.  Returns the filtered dict AND loads it (strict=False)."""
    state = model.state_dict()
    first = next(iter(weights))
    if first.startswith("module."):
        weights = {k.partition("module.")[2]: v for k, v in weights.items()}
    if next(iter(weights)).startswith("encoder."):
        weights = {k.partition("encoder.")[2]: v for k, v in weights.items()}
    filtered = {k: v for k, v in weights.items() if k in state and v.size() == state[k].size()}
    logging.info("Loading weights:" + ", ".join(filtered.keys()))
    model.load_state_dict(filtered, strict=False)
    ME.bump_weights_epoch()
    return filtered


def initialize_optimizer(params, config):
    """`lib/solvers.py:47-57` (SGD branch; the hot path's optimiser)."""
    if config.optimizer != "SGD":
        raise ValueError("Optimizer type not supported")
    return FlatSGD(params, lr=config.lr, momentum=config.sgd_momentum, dampening=config.sgd_dampening, weight_decay=config.weight_decay)


def initialize_scheduler(optimizer, config, last_step=-1):
    """`lib/solvers.py:66-83`."""
    if config.scheduler == "PolyLR":
        return PolyLR(optimizer, max_iter=config.max_iter, power=config.poly_power, last_step=last_step)
    if config.scheduler == "StepLR":
        return torch.optim.lr_scheduler.StepLR(optimizer, step_size=config.step_size, gamma=config.step_gamma, last_epoch=last_step)
    if config.scheduler == "ExpLR":
        return torch.optim.lr_scheduler.LambdaLR(optimizer, lambda s: config.exp_gamma ** (s / config.exp_step_size), last_step)
    raise ValueError("Scheduler not supported")


class SegmentationTrainer:
    def __init__(self, model, config, device=None):
        self.device = torch.device(device) if device is not None else torch.device("cuda", torch.cuda.current_device())
        self.model = model.to(self.device)
        self.config = config
        self.optimizer = initialize_optimizer(self.model.parameters(), config.optimizer)
        self.scheduler = initialize_scheduler(self.optimizer, config.optimizer)
        self.ignore_label = config.data.ignore_label
        self.iter_size = config.optimizer.iter_size
        self.curr_iter = 1

    def train_step(self, sub_batches, shift_coords=True):
        """One optimiser step = `iter_size` sub-batches of (coords int32 [N,4], feats fp32 [N,3], target int [N]), gradients
        accumulated (`lib/train.py:97-160`).  Returns the summed (already 1/iter_size-scaled) loss as a device scalar."""
        assert len(sub_batches) == self.iter_size
        self.model.train()
        self.optimizer.zero_grad()
        total = None
        for coords, feats, target in sub_batches:
            if shift_coords:          # `lib/train.py:110`: even/odd-coordinate invariance (shifts the batch column too: SURVEY.md appendix B)
                coords = coords.clone()
                coords[:, :3] += (torch.rand(3) * 100).type_as(coords)
            sinput = ME.SparseTensor(feats, coords).to(self.device)
            soutput = self.model(sinput)
            loss = losses.cross_entropy(soutput.F, target.to(self.device, non_blocking=True), self.ignore_label) / self.iter_size
            loss.backward()
            total = loss.detach() if total is None else total + loss.detach()
        self.optimizer.step()
        self.scheduler.step()
        self.curr_iter += 1
        return total

    def validate(self, data_loader, transform_data_fn=None):
        """`lib/train.py:30-35,201-210`: `test()` on the validation loader, then back to training mode.  Returns the mIoU."""
        try:
            return test(self.model, data_loader, self.config, transform_data_fn)[3]
        finally:
            self.model.train()


def per_class_iu(hist):
    """`lib/utils.py:136-138`: diag / (rowsum + colsum - diag), 0/0 -> NaN."""
    with np.errstate(divide="ignore", invalid="ignore"):
        return np.diag(hist) / (hist.sum(1) + hist.sum(0) - np.diag(hist))


class SegmentationMeter:
    """Device accumulators of the reference's evaluation loop (`lib/test.py:119-149`): the confusion histogram, the n-weighted
    loss and precision@1 sums (`AverageMeter`, weight = every row of the batch, ignored ones included) and the per-class sum and count
    of the non-NaN batch APs (`np.nanmean(aps, 0)`).

    A row is valid when 0 <= target < C and target != ignore_label; invalid rows count in no loss, precision or histogram term and
    are negatives for every class in the AP.  (The reference's precision@1 is called with its default ignore label 255 instead of
    the configured one, `test.py:139`; for its configs, where both are 255, that is the same rule.)  The AP of a batch is scikit-learn's
    uninterpolated average precision with equal scores ranked as one group, and NaN for a class without a positive row in the batch
    (what the reference's scikit-learn returned; current releases return 0.0) -- such batches are left out of that class's mean.

    `update` never synchronises with the host; `summary` does the one device-to-host read."""

    def __init__(self, num_labels, ignore_label=255, device=None):
        self.num_labels = int(num_labels)
        self.ignore_label = int(ignore_label)
        self.device = torch.device(device) if device is not None else torch.device("cuda", torch.cuda.current_device())
        self._ws = None
        self.reset()

    def reset(self):
        C, dev = self.num_labels, self.device
        if dev.type != "cuda":
            raise _lib.PcbError("SegmentationMeter runs on a CUDA device only (no CPU fallback)")
        self.hist = torch.zeros(C, C, dtype=torch.int64, device=dev)
        self.sums = torch.zeros(3, dtype=torch.float64, device=dev)           # sum loss_b n_b, sum score_b n_b, sum n_b
        self.last = torch.full((2,), float("nan"), dtype=torch.float64, device=dev)   # loss_b, score_b of the latest batch
        self.ap_sum = torch.zeros(C, dtype=torch.float64, device=dev)
        self.ap_count = torch.zeros(C, dtype=torch.float64, device=dev)

    def update(self, logits, target):
        """Folds in one batch: logits [n, C] fp32, target [n] integer (both on the meter's device).  Returns pred [n] int32 (device),
        the first maximal class of each row."""
        _lib.require_cuda(logits)
        _lib.require_cuda(target)
        n, C = logits.shape
        if C != self.num_labels:
            raise ValueError(f"logits have {C} classes, the meter {self.num_labels}")
        logits = logits.detach().float().contiguous()
        target = target.detach().to(torch.int64).contiguous()
        dev = logits.device
        pred = torch.empty(n, dtype=torch.int32, device=dev)
        stats = torch.empty(4, dtype=torch.float64, device=dev)
        ap = torch.empty(C, dtype=torch.float64, device=dev)
        need = int(_lib.lib.pcb_seg_eval_ws_bytes(n, C))
        if self._ws is None or self._ws.numel() < need:
            self._ws = torch.empty(need, dtype=torch.uint8, device=dev)
        _lib.check(_lib.lib.pcb_seg_eval(_lib.ptr(logits), _lib.ptr(target), n, C, self.ignore_label, _lib.ptr(pred), _lib.ptr(self.hist),
                                         _lib.ptr(stats), _lib.ptr(ap), None, _lib.ptr(self._ws), self._ws.numel(),
                                         _lib.stream()))
        loss_b = stats[0] / stats[1]                    # NaN when no row is valid, as nn.CrossEntropyLoss
        score_b = stats[2] * 100.0 / stats[1]
        self.last = torch.stack([loss_b, score_b])
        self.sums += torch.stack([loss_b * stats[3], score_b * stats[3], stats[3]])
        ok = ~torch.isnan(ap)
        self.ap_sum += torch.where(ok, ap, torch.zeros_like(ap))
        self.ap_count += ok.to(torch.float64)
        return pred

    def summary(self):
        """One device-to-host read.  Returns a dict: loss, score (precision@1 in %), mAP, mIoU, mAcc, and per class ious, ap_class,
        acc (%), hist (int64 [C, C]); loss_val / score_val are the latest batch's values."""
        C = self.num_labels
        host = torch.cat([self.sums, self.last, self.ap_sum, self.ap_count, self.hist.flatten().to(torch.float64)]).cpu().numpy()
        sums, last = host[:3], host[3:5]
        ap_sum, ap_count = host[5:5 + C], host[5 + C:5 + 2 * C]
        hist = host[5 + 2 * C:].reshape(C, C).astype(np.int64)
        with np.errstate(divide="ignore", invalid="ignore"), warnings.catch_warnings():
            warnings.simplefilter("ignore", category=RuntimeWarning)
            ap_class = ap_sum / ap_count * 100.0
            iu = per_class_iu(hist)
            acc = np.diag(hist) / hist.sum(1) * 100.0
            return dict(loss=sums[0] / sums[2], score=sums[1] / sums[2], loss_val=last[0], score_val=last[1], mAP=float(np.nanmean(ap_class)),
                        mIoU=float(np.nanmean(iu) * 100.0), mAcc=float(np.nanmean(acc)), ious=iu * 100.0, ap_class=ap_class, acc=acc, hist=hist)


def _cfg(config, path, default=None):
    node = config
    for k in path.split("."):
        try:
            node = getattr(node, k)
        except (AttributeError, KeyError):
            return default
    return node


def print_info(iteration, max_iteration, data_time, iter_time, s, dataset=None):
    """`lib/test.py:25-52`: the running metrics (`s` = SegmentationMeter.summary()), per class in the dataset's order."""
    reorder = getattr(dataset, "reorder_result", lambda x: x)
    ious, ap_class = reorder(s["ious"]), reorder(s["ap_class"])
    class_names = dataset.get_classnames() if hasattr(dataset, "get_classnames") else None
    with warnings.catch_warnings():
        warnings.simplefilter("ignore", category=RuntimeWarning)
        msg = "{}/{}: Data time: {:.4f}, Iter time: {:.4f}".format(iteration + 1, max_iteration, data_time, iter_time)
        msg += "\tLoss {:.3f} (AVG: {:.3f})\tScore {:.3f} (AVG: {:.3f})\tmIOU {:.3f} mAP {:.3f} mAcc {:.3f}\n".format(
            s["loss_val"], s["loss"], s["score_val"], s["score"], np.nanmean(ious), np.nanmean(ap_class), s["mAcc"])
    if class_names is not None:
        msg += "\nClasses: " + " ".join(class_names) + "\n"
    msg += "IOU: " + " ".join("{:.03f}".format(i) for i in ious) + "\n"
    msg += "mAP: " + " ".join("{:.03f}".format(i) for i in ap_class) + "\n"
    msg += "mAcc: " + " ".join("{:.03f}".format(i) for i in s["acc"]) + "\n"
    logging.info(msg)


def test(model, data_loader, config, transform_data_fn=None, has_gt=True):
    """`downstream/semseg/lib/test.py:62-196`: evaluates `model` over `data_loader` (batches of (coords, feats, target) or, with
    `data.return_transformation`, (coords, feats, target, transformation)) and returns (loss, precision@1, mAP, mIoU) -- loss and
    precision averaged over batches weighted by their row count, mAP the mean over classes of the per-class mean of the batch APs,
    mIoU from the accumulated confusion histogram (percent).  Metric definitions: `SegmentationMeter`.

    Logs the running metrics every `test.test_stat_freq` batches and at the end.  Saving predictions, evaluation on the original
    point cloud, wrapper models and test sets without labels are not supported."""
    if not has_gt:
        raise NotImplementedError("test() without ground truth")
    if _cfg(config, "net.wrapper_type") is not None:
        raise NotImplementedError("net.wrapper_type")
    for key in ("test.save_prediction", "test.test_original_pointcloud", "test.evaluate_original_pointcloud"):
        if _cfg(config, key, False):
            raise NotImplementedError(key)
    device = torch.device("cuda", torch.cuda.current_device())
    dataset = data_loader.dataset
    meter = SegmentationMeter(dataset.NUM_LABELS, _cfg(config, "data.ignore_label", 255), device)
    normalize_color = _cfg(config, "augmentation.normalize_color", True)
    stat_freq = _cfg(config, "test.test_stat_freq", 100)
    logging.info("===> Start testing")
    t_start = time.time()
    data_iter = iter(data_loader)
    max_iter = len(data_loader)
    model.eval()
    data_time = iter_time = 0.0
    with torch.no_grad():
        for iteration in range(max_iter):
            t0 = time.time()
            batch = next(data_iter)
            coords, feats, target = batch[:3]
            data_time = time.time() - t0
            t0 = time.time()
            if normalize_color:
                feats[:, :3] = feats[:, :3] / 255. - 0.5
            output = model(ME.SparseTensor(feats, coords).to(device)).F
            meter.update(output, target.to(device, non_blocking=True))
            iter_time = time.time() - t0
            if iteration % stat_freq == 0 and iteration > 0:
                print_info(iteration, max_iter, data_time, iter_time, meter.summary(), dataset)
    s = meter.summary()
    print_info(max_iter - 1, max_iter, data_time, iter_time, s, dataset)
    logging.info("Finished test. Elapsed time: {:.4f}".format(time.time() - t_start))
    return s["loss"], s["score"], s["mAP"], s["mIoU"]

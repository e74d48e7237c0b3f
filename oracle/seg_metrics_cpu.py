"""numpy restatement of the semantic-segmentation evaluation of `downstream/semseg/lib/test.py:55-196` and `lib/utils.py:117-133`:
the per-batch metrics (prediction, cross-entropy, precision@1, confusion histogram, per-class average precision) and the loop that
folds batches together.  The reference for pcb_seg_eval / semseg.SegmentationMeter; product code never imports it.

Conventions (the same as the kernels'):
  - a row is valid when 0 <= target < C and target != ignore_label.  Invalid rows count in no loss, precision or histogram term and
    are negatives for every class in the average precision (`label_binarize` gives them an all-zero row).
  - average precision is scikit-learn's uninterpolated one, equal scores ranked as one group: with TP_g / FP_g the counts up to the
    end of tie group g and P the positives, AP = sum_g (TP_g - TP_{g-1}) / P * TP_g / (TP_g + FP_g).  A class without a positive
    gets NaN (0/0 recall, what the reference's scikit-learn returned and what its `np.nanmean` over batches relies on).
"""
import numpy as np


def valid_rows(target, num_labels, ignore_label):
    target = np.asarray(target)
    return (target >= 0) & (target < num_labels) & (target != ignore_label)


def fast_hist(pred, label, n):
    """`lib/utils.py:131-133`: hist[label, pred] over 0 <= label < n."""
    label = np.asarray(label).astype(np.int64)
    pred = np.asarray(pred).astype(np.int64)
    k = (label >= 0) & (label < n)
    return np.bincount(n * label[k] + pred[k], minlength=n ** 2).reshape(n, n)


def per_class_iu(hist):
    with np.errstate(divide="ignore", invalid="ignore"):
        return np.diag(hist) / (hist.sum(1) + hist.sum(0) - np.diag(hist))


def softmax(logits):
    x = np.asarray(logits, dtype=np.float64)
    e = np.exp(x - x.max(1, keepdims=True))
    return e / e.sum(1, keepdims=True)


def cross_entropy(logits, target, ignore_label):
    """Mean cross-entropy over the valid rows in fp64; NaN when there are none."""
    x = np.asarray(logits, dtype=np.float64)
    ok = valid_rows(target, x.shape[1], ignore_label)
    m = x.max(1)
    lse = m + np.log(np.exp(x - m[:, None]).sum(1))
    t = np.asarray(target)[ok].astype(np.int64)
    with np.errstate(invalid="ignore"):
        return float(np.sum(lse[ok] - x[ok, t]) / ok.sum())


def precision_at_one(pred, target, num_labels, ignore_label):
    """100 * #(pred == target) / #valid; NaN when no row is valid.  (`lib/utils.py:117-128` is called by the reference's test loop with
    its default ignore label 255 rather than the configured one, `test.py:139`; here the configured one applies.)"""
    ok = valid_rows(target, num_labels, ignore_label)
    if not ok.any():
        return float("nan")
    return 100.0 * float(np.sum(np.asarray(pred)[ok] == np.asarray(target)[ok])) / float(ok.sum())


def average_precision(prob, target, ignore_label=255):
    """Per-class AP of the scores prob[:, c] against target == c (tie-grouped, NaN for a class without positives)."""
    prob = np.asarray(prob)
    n, C = prob.shape
    target = np.asarray(target)
    ok = valid_rows(target, C, ignore_label)
    out = np.full(C, np.nan)
    for c in range(C):
        y = ok & (target == c)
        P = int(y.sum())
        if P == 0:
            continue
        order = np.argsort(-prob[:, c], kind="stable")
        s, yy = prob[order, c], y[order]
        tp = np.cumsum(yy)
        ends = np.r_[np.nonzero(s[1:] != s[:-1])[0], n - 1]
        tpg = tp[ends].astype(np.float64)
        prev = np.r_[0.0, tpg[:-1]]
        out[c] = float(np.sum((tpg - prev) / P * tpg / (ends + 1)))
    return out


def batch_metrics(logits, target, num_labels, ignore_label, prob=None):
    """One batch: pred, loss, score, hist, ap (on `prob` if given, else the fp64 softmax of the logits)."""
    logits = np.asarray(logits)
    target = np.asarray(target)
    pred = logits.argmax(1)
    ok = valid_rows(target, num_labels, ignore_label)
    hist = fast_hist(pred[ok], target[ok], num_labels)
    return dict(pred=pred, loss=cross_entropy(logits, target, ignore_label), score=precision_at_one(pred, target, num_labels, ignore_label),
                hist=hist, ap=average_precision(softmax(logits) if prob is None else prob, target, ignore_label))


def evaluate(batches, num_labels, ignore_label):
    """The reference's test loop (`lib/test.py:62-196`) over an iterable of (logits, target[, prob]) batches.  loss and score are
    averaged with weight n_b = all rows of the batch (`test.py:133`), NaNs propagating as in `AverageMeter`."""
    hist = np.zeros((num_labels, num_labels), dtype=np.int64)
    loss_sum = score_sum = 0.0
    count = 0
    aps = []
    for b in batches:
        logits, target = b[0], b[1]
        m = batch_metrics(logits, target, num_labels, ignore_label, b[2] if len(b) > 2 else None)
        n = len(target)
        loss_sum += m["loss"] * n
        score_sum += m["score"] * n
        count += n
        hist += m["hist"]
        aps.append(m["ap"])
    with np.errstate(divide="ignore", invalid="ignore"):
        import warnings
        with warnings.catch_warnings():
            warnings.simplefilter("ignore", category=RuntimeWarning)
            ap_class = np.nanmean(np.array(aps), 0) * 100.0
            ious = per_class_iu(hist) * 100.0
            acc = np.diag(hist) / hist.sum(1) * 100.0
            return dict(loss=loss_sum / count, score=score_sum / count, mAP=float(np.nanmean(ap_class)),
                        mIoU=float(np.nanmean(per_class_iu(hist)) * 100.0), mAcc=float(np.nanmean(acc)), ious=ious, ap_class=ap_class,
                        acc=acc, hist=hist)

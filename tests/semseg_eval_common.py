"""Inputs shared by the semantic-segmentation evaluation tests and tests/golden/make_semseg_eval_fixtures.py: seeded logit / target
batches with exact ties (constant rows, duplicated rows, logit gaps that make probabilities underflow to 0 or round to 1) and ~10 %
ignored rows, and the stand-ins that drive an evaluation loop with them: a model returning the stored logits, a loader, a dataset."""
import os
import types

import numpy as np
import torch

NUM_LABELS = 13
IGNORE = 255
FIXTURE = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "semseg_eval_reference.npz")
BATCH_ROWS = (1500, 2200, 3000, 1800)


def make_batch(seed, n, C=NUM_LABELS, ignore=IGNORE):
    """fp32 logits [n, C] and int64 targets [n] with every class present among the valid rows."""
    rng = np.random.default_rng(seed)
    t = rng.integers(0, C, n)
    t[:C] = np.arange(C)                                      # every class has a positive
    x = rng.normal(0.0, 2.0, (n, C)).astype(np.float32)
    x[np.arange(n), t] += 1.5                                 # scores that carry some signal
    ign = rng.random(n) < 0.1
    ign[:C] = False
    t[ign] = ignore
    rows = rng.permutation(np.arange(C, n))
    k = n // 30
    x[rows[:k]] = np.float32(0.75)                            # constant rows: every probability 1/C, one big tie group per class
    x[rows[k:2 * k]] = x[rows[2 * k:3 * k]]                   # duplicated rows
    gap = rows[3 * k:4 * k]
    x[gap] = 0.0
    x[gap, rng.integers(0, C, len(gap))] = 110.0              # exp(-110) underflows: probabilities exactly 0 and 1
    return x, t.astype(np.int64)


def fixture_batches():
    return [make_batch(1000 + i, n) for i, n in enumerate(BATCH_ROWS)]


def batch_coords(n):
    """Distinct voxel coordinates (batch, x, y, z) for n rows."""
    i = np.arange(n)
    return torch.from_numpy(np.stack([np.zeros(n), i % 64, i // 64, np.zeros(n)], 1).astype(np.int32))


class StandInDataset:
    NUM_LABELS = NUM_LABELS

    def reorder_result(self, result):
        return result

    def get_classnames(self):
        return [f"c{i}" for i in range(NUM_LABELS)]


class StandInLoader:
    """Yields (coords, feats, target) per batch; offers both the iterator protocol and the Python-2 `.next()`."""

    def __init__(self, batches):
        self.batches = batches
        self.dataset = StandInDataset()
        self._i = 0

    def __len__(self):
        return len(self.batches)

    def __iter__(self):
        self._i = 0
        return self

    def __next__(self):
        if self._i >= len(self.batches):
            raise StopIteration
        x, t = self.batches[self._i]
        self._i += 1
        return batch_coords(len(t)), torch.full((len(t), 3), 128.0), torch.from_numpy(t)

    next = __next__


class StandInModel(torch.nn.Module):
    """Returns the stored logits of the next batch as `.F`, on the device of the input features."""

    def __init__(self, batches):
        super().__init__()
        self.logits = [torch.from_numpy(x) for x, _ in batches]
        self.calls = 0

    def forward(self, sinput):
        x = self.logits[self.calls % len(self.logits)].to(sinput.F.device)
        self.calls += 1
        return types.SimpleNamespace(F=x)

"""TEST INFRASTRUCTURE ONLY -- CPU oracle for the two contrastive losses (see oracle/me_cpu.py header).

The reference draws its random subsets from process-global RNGs (`lib/ddp_trainer.py:199-200,203,404,413`).
For parity the draws are *injected*: every function here takes the already-chosen indices.

PINNED against the reference's own unmodified code (tests/test_oracle_reference.py, against its outputs recorded in tests/golden/):
  * `hardest_contrastive_loss` == `HardestContrastiveLossTrainer.contrastive_hardest_negative_loss`
    (`lib/ddp_trainer.py:186-238`), same numpy RNG draws, rtol 1e-12;
  * `select_positives` + `point_nce_loss` == the loss and gradients of `PointNCELossTrainer._train_iter`
    (`lib/ddp_trainer.py:380-440` + `lib/criterion.py:10-19`) executed on the CPU with its hard-coded `.cuda()` calls
    patched to identity and a stand-in model, same torch / numpy RNG draws, rtol 1e-12.
"""
import numpy as np
import torch
import torch.nn.functional as F


def select_positives(pos_pairs, uniform, npos=None, sampled_inds=None):
    """`lib/ddp_trainer.py:400-415`.  pos_pairs int [P,2] grouped by column 0; `uniform` = the U(0,1) draw per
    unique query (`:404`); `sampled_inds` = the np.random.choice(|q|, npos) draw (`:413`) or None.
    Returns (q_rows into F0, k_rows into F1) as int64 tensors."""
    pos_pairs = torch.as_tensor(pos_pairs).long()
    q_unique, count = pos_pairs[:, 0].unique(return_counts=True)
    off = torch.floor(torch.as_tensor(uniform, dtype=torch.float32) * count).long()
    cums = torch.cat([torch.zeros(1, dtype=torch.long), torch.cumsum(count, 0)[:-1]])
    k_sel = pos_pairs[:, 1][off + cums]
    if npos is not None and npos < len(q_unique):
        si = torch.as_tensor(sampled_inds).long()
        q_unique, k_sel = q_unique[si], k_sel[si]
    return q_unique, k_sel


def point_nce_loss(F0, F1, q_rows, k_rows, T):
    """`lib/ddp_trainer.py:409-426`: logits = q k^T / T ; CrossEntropy(logits, arange) (one direction)."""
    q = F0[q_rows]
    k = F1[k_rows]
    logits = torch.mm(q, k.t()) / T
    labels = torch.arange(q.shape[0])
    return F.cross_entropy(logits, labels)


def _hash(a, b, M):
    """`lib/ddp_trainer.py:39-51` for the two-column case: a + b*M in int64."""
    return np.asarray(a, np.int64) + np.asarray(b, np.int64) * np.int64(M)


def hardest_contrastive_loss(F0, F1, pos_pairs, sel0, sel1, pos_sel, pos_thresh=0.1, neg_thresh=1.4):
    """`lib/ddp_trainer.py:186-238` with the three np.random.choice draws injected
    (`sel0`,`sel1` = hard-negative candidate rows `:199-200`; `pos_sel` = positive subsample `:203` or None)."""
    N0, N1 = len(F0), len(F1)
    pos_pairs = np.asarray(pos_pairs, np.int64)
    hash_seed = max(N0, N1)
    sample = pos_pairs if pos_sel is None else pos_pairs[np.asarray(pos_sel)]
    i0 = torch.from_numpy(sample[:, 0]).long()
    i1 = torch.from_numpy(sample[:, 1]).long()
    sel0 = np.asarray(sel0, np.int64)
    sel1 = np.asarray(sel1, np.int64)
    subF0, subF1 = F0[torch.from_numpy(sel0)], F1[torch.from_numpy(sel1)]
    posF0, posF1 = F0[i0], F1[i1]

    def pdist(A, B):          # `:182-184`
        return torch.sqrt(((A.unsqueeze(1) - B.unsqueeze(0)) ** 2).sum(2) + 1e-7)

    D01min, D01ind = pdist(posF0, subF1).min(1)
    D10min, D10ind = pdist(posF1, subF0).min(1)
    pos_keys = _hash(pos_pairs[:, 0], pos_pairs[:, 1], hash_seed)
    neg0 = _hash(sample[:, 0], sel1[D01ind.numpy()], hash_seed)
    neg1 = _hash(sel0[D10ind.numpy()], sample[:, 1], hash_seed)
    mask0 = torch.from_numpy(~np.isin(neg0, pos_keys))
    mask1 = torch.from_numpy(~np.isin(neg1, pos_keys))
    pos_loss = F.relu(((posF0 - posF1) ** 2).sum(1) - pos_thresh)
    neg0l = F.relu(neg_thresh - D01min[mask0]) ** 2
    neg1l = F.relu(neg_thresh - D10min[mask1]) ** 2
    return pos_loss.mean(), (neg0l.mean() + neg1l.mean()) / 2

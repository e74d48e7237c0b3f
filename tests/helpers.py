"""Shared helpers for the parity tests."""
import contextlib
import json
import math
import os

import numpy as np
import torch

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def load_c0_golden():
    """tests/golden/c0_res16unet34c.npz with the per-point features of tests/golden/c0_res16unet34c_features.npz, as one dict
    (two files keep each under 1 MB)."""
    g = dict(np.load(os.path.join(GOLDEN, "c0_res16unet34c.npz")))
    g.update(np.load(os.path.join(GOLDEN, "c0_res16unet34c_features.npz")))
    return g


def model_structure(net):
    """Module tree and state-dict layout of a Res16UNet built on any MinkowskiEngine-compatible module, as JSON data: every
    module's name and class, a convolution's kernel offsets, stride and bias flag, a BatchNorm's momentum and eps."""
    mods = []
    for name, m in net.named_modules():
        d = {"name": name, "class": type(m).__name__}
        if getattr(m, "kernel_generator", None) is not None:
            d.update(offsets=np.asarray(m.kernel_generator.offsets).tolist(), stride=[int(s) for s in m.stride], has_bias=bool(m.has_bias))
        if isinstance(getattr(m, "bn", None), torch.nn.BatchNorm1d):
            d.update(momentum=float(m.bn.momentum), eps=float(m.bn.eps))
        mods.append(d)
    return {"n_params": sum(p.numel() for p in net.parameters()), "modules": mods,
            "state_dict": [[k, list(v.shape)] for k, v in net.state_dict().items()]}


def reference_structure():
    """`model_structure` of the original project's Res16UNet34C (tests/golden/make_reference_fixtures.py)."""
    with open(os.path.join(GOLDEN, "reference_res16unet34c_structure.json")) as f:
        return json.load(f)


def rand_coords(rng, n, lo=-20, hi=21, batches=2):
    c = np.stack([rng.integers(0, batches, n), rng.integers(lo, hi, n), rng.integers(lo, hi, n),
                  rng.integers(lo, hi, n)], 1)
    c = np.unique(c, axis=0).astype(np.int32)
    return c[rng.permutation(len(c))]


def surface_coords(rng, n, batches=2, extent=40):
    """Voxels near a few random planes: the neighbour statistics of real scans (about half of 27 present)."""
    out = []
    for b in range(batches):
        per = n // batches
        pts = []
        for _ in range(3):
            nrm = rng.normal(size=3); nrm /= np.linalg.norm(nrm)
            u = np.cross(nrm, [1.0, 0.3, 0.2]); u /= np.linalg.norm(u)
            v = np.cross(nrm, u)
            ab = rng.uniform(-extent, extent, size=(per, 2))
            p = ab[:, :1] * u + ab[:, 1:] * v + nrm * rng.normal(0, 0.4, size=(per, 1)) + rng.uniform(-5, 5, 3)
            pts.append(p)
        c = np.floor(np.concatenate(pts)).astype(np.int32)
        c = np.unique(c, axis=0)[:per]
        out.append(np.concatenate([np.full((len(c), 1), b, np.int32), c], 1))
    return np.concatenate(out)


def det_init(model, seed=0):
    """Deterministic, architecture-independent parameter fill (same values for any backend of the same model)."""
    with torch.no_grad():
        for i, (name, p) in enumerate(model.named_parameters()):
            g = torch.Generator().manual_seed(seed * 100003 + i)
            if name.endswith("kernel"):
                stdv = 1.0 / math.sqrt(p.shape[0] * p.shape[1])
                v = (torch.rand(p.shape, generator=g, dtype=torch.float64) * 2 - 1) * stdv
            elif name.endswith("bn.weight"):
                v = 1.0 + 0.2 * (torch.rand(p.shape, generator=g, dtype=torch.float64) - 0.5)
            else:
                v = 0.2 * (torch.rand(p.shape, generator=g, dtype=torch.float64) - 0.5)
            p.copy_(v.to(p.dtype))


@contextlib.contextmanager
def model_backend(me_module):
    """Build / run pointcontrast_b200.model.res16unet on another MinkowskiEngine-compatible module (the oracle)."""
    from pointcontrast_b200.model import res16unet
    old = res16unet.ME
    res16unet.ME = me_module
    try:
        yield res16unet
    finally:
        res16unet.ME = old


@contextlib.contextmanager
def pinned_relu(me_module, masks, flips):
    """Run the oracle with the ReLU decisions of another run: the i-th MinkowskiReLU call multiplies by masks[i] (bool [n, C]) instead of
    testing the sign itself; flips[i] = number of entries where the oracle's own sign test disagrees.  ReLU is the one discontinuous
    operator of the network: a pre-activation that is zero to within rounding falls on either side in any finite precision (the fp32
    CPU oracle against the fp64 one: 2 entries of 3 million at C0 size), and a single flipped entry on a deep level changes every upstream
    gradient by ~1/sqrt(rows x channels) of its norm.  Pinning the decisions separates that coin from the arithmetic being tested."""
    cls = me_module.MinkowskiReLU
    old = cls.forward
    it = iter(masks)

    def forward(self, x):
        m = next(it)
        assert m.shape == x.F.shape, (m.shape, x.F.shape)
        flips.append(int(((x.F > 0) != m).sum()))
        return me_module.SparseTensor(x.F * m.to(x.F.dtype), coords_key=x.coords_key, coords_manager=x.coords_man)

    cls.forward = forward
    try:
        yield
    finally:
        cls.forward = old


def rel_err(a, b):
    a = a.detach().double().cpu(); b = b.detach().double().cpu()
    return float((a - b).norm() / (b.norm() + 1e-300))


def max_rel_err(a, b):
    """max |a-b| scaled by the RMS of the reference: the 'per-point feature' metric."""
    a = a.detach().double().cpu(); b = b.detach().double().cpu()
    return float((a - b).abs().max() / (b.pow(2).mean().sqrt() + 1e-300))


def table_to_pairs(tbl):
    """Dense neighbour table [K, n_out] -> ME-style per-offset (in_rows, out_rows), ascending out row."""
    tbl = tbl.cpu().numpy()
    out = []
    for k in range(tbl.shape[0]):
        j = np.nonzero(tbl[k] >= 0)[0]
        out.append((tbl[k][j].astype(np.int64), j.astype(np.int64)))
    return out

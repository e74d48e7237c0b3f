"""CPU-side checks: the C-ABI library loads and exports every symbol include/pcb200.h declares, the host-side mirror of
the MinkowskiEngine interface behaves like the oracle where no GPU is needed, and there is no CPU compute path."""
import ctypes
import os
import re

import numpy as np
import pytest
import torch

from oracle import me_cpu as OR
from tests import refload

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_declared_symbol():
    from pointcontrast_b200 import _lib
    hdr = open(os.path.join(ROOT, "include", "pcb200.h")).read()
    hdr = re.sub(r"/\*.*?\*/", "", hdr, flags=re.S)
    declared = sorted(set(re.findall(r"\b(pcb_[a-z0-9_]+)\s*\(", hdr)))
    assert len(declared) >= 20
    handle = ctypes.CDLL(os.path.join(ROOT, "pointcontrast_b200", "libpcb200.so"))
    for name in declared:
        assert hasattr(handle, name), f"{name} declared in pcb200.h but not exported"
    assert sorted(_lib.EXPORTS) == declared
    assert b"sm_100a" in _lib.lib.pcb_version()


def test_library_has_sm100a_code_and_tensor_core_instructions():
    import shutil
    import subprocess
    if not shutil.which("cuobjdump"):
        pytest.skip("cuobjdump not on PATH")
    so = os.path.join(ROOT, "pointcontrast_b200", "libpcb200.so")
    out = subprocess.run(["cuobjdump", "-lelf", so], capture_output=True, text=True).stdout
    assert "sm_100a" in out
    sass = subprocess.run(["cuobjdump", "-sass", so], capture_output=True, text=True).stdout
    # Blackwell-native evidence (B200_PROFILING.md): tcgen05.mma -> UTCHMMA, tcgen05.ld -> LDTM, TMA bulk copy -> UBLKCP, commit -> UTCBAR,
    # programmatic dependent launch -> ACQBULK; and NO legacy mma.sync (" HMMA.") tensor-core path left in the library
    for mnemonic in ("UTCHMMA", "LDTM", "UBLKCP", "UTCBAR", "ACQBULK"):
        assert mnemonic in sass, mnemonic
    assert " HMMA." not in sass and "HGMMA" not in sass


def test_argument_errors_do_not_need_a_gpu():
    from pointcontrast_b200 import _lib
    rc = _lib.lib.pcb_hash_build(None, 10, None, None, 24, None, None)      # capacity not a power of two
    assert rc == 2 and b"bad argument" in _lib.lib.pcb_last_error()
    with pytest.raises(_lib.PcbError):
        _lib.check(rc)
    assert _lib.lib.pcb_conv_wgrad_ws_bytes(27, 100000, 96, 96) > 27 * 96 * 96 * 4
    assert _lib.lib.pcb_nce_ws_bytes(4096) >= 4096 * 4096 * 4


def test_offset_tables_match_oracle():
    from pointcontrast_b200 import me
    for ks in ([3, 3, 3], [2, 2, 2], [1, 1, 1]):
        a = me.KernelGenerator(ks, 1, 1, dimension=3).offsets
        b = OR.KernelGenerator(ks, 1, 1, dimension=3).offsets
        assert (a == b).all()
    a = me.KernelGenerator(3, 1, 1, region_type=me.RegionType.HYBRID, axis_types=[me.RegionType.HYPERCUBE] * 3, dimension=3)
    b = OR.KernelGenerator(3, 1, 1, region_type=OR.RegionType.HYBRID, axis_types=[OR.RegionType.HYPERCUBE] * 3, dimension=3)
    assert (a.offsets == b.offsets).all() and a.kernel_volume == 27
    assert [m.value for m in me.RegionType] == [0, 1, 2, 3]


def test_own_model_matches_reference_model_structure():
    """This package's Res16UNet34C on its own MinkowskiEngine surface against the original model file's, as recorded in
    tests/golden/reference_res16unet34c_structure.json: the same modules in the same order (classes, kernel offsets, strides,
    biases, BatchNorm momentum / eps) and the same state-dict layout."""
    from pointcontrast_b200.model import load_model
    from tests.helpers import model_structure, reference_structure
    net = load_model("Res16UNet34C")(3, 32, refload.default_config(), D=3)
    own, ref = model_structure(net), reference_structure()
    assert own["state_dict"] == ref["state_dict"]
    assert [m["name"] for m in own["modules"]] == [m["name"] for m in ref["modules"]]
    for m1, m2 in zip(own["modules"], ref["modules"]):
        assert m1 == m2, m1["name"]
    assert own["n_params"] == ref["n_params"] == 37_847_808


def test_no_cpu_compute_path():
    from pointcontrast_b200 import _lib, losses, me
    st = me.SparseTensor(torch.zeros(4, 32), coords=torch.tensor([[0, 0, 0, i] for i in range(4)], dtype=torch.int32))
    with pytest.raises(_lib.PcbError):
        me.MinkowskiConvolution(32, 32, kernel_size=3, dimension=3)(st)
    with pytest.raises(_lib.PcbError):
        me.MinkowskiBatchNorm(32)(st)
    with pytest.raises(_lib.PcbError):
        losses.point_nce_loss(torch.zeros(4, 32), torch.zeros(4, 32), torch.arange(4), torch.arange(4), 0.4)
    with pytest.raises(_lib.PcbError):
        losses.pdist_rowmin(torch.zeros(4, 32), torch.zeros(4, 32))


def test_product_code_never_imports_the_oracle():
    pkg = os.path.join(ROOT, "pointcontrast_b200")
    for dp, _, fs in os.walk(pkg):
        for f in fs:
            if f.endswith(".py"):
                src = open(os.path.join(dp, f)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle\b", src, flags=re.M), f


def test_golden_fixture_is_consistent_with_the_oracle():
    """The committed golden file replays on the oracle with THIS repo's model wiring (own graph == reference graph)."""
    from tests.helpers import det_init, load_c0_golden, max_rel_err, model_backend
    g = load_c0_golden()
    with model_backend(OR) as mod:
        net = mod.Res16UNet34C(3, 32, refload.default_config(), D=3)
        det_init(net, 0)                   # fp32 parameter values (what the GPU model holds), evaluated in fp64
        net = net.double().train()
        torch.set_num_threads(os.cpu_count())
        with torch.no_grad():
            F0 = net(OR.SparseTensor(torch.from_numpy(g["X0"]).double(), coords=torch.from_numpy(g["C0"]))).F
    assert max_rel_err(F0, torch.from_numpy(g["F0"])) < 1e-6

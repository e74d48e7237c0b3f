"""ctypes binding of libpcb200.so (include/pcb200.h).  There is NO fallback: if the library is missing or a call
fails, this raises."""
import ctypes as C
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
_PATH = os.path.join(_HERE, "libpcb200.so")


class PcbError(RuntimeError):
    pass


def _load():
    if not os.path.exists(_PATH):
        raise ImportError(
            f"{_PATH} not found: the CUDA extension is not built. Run `python -m pointcontrast_b200.build` "
            "(needs nvcc; there is no CPU fallback).")
    return C.CDLL(_PATH)


lib = _load()

_p, _i, _l, _f, _sz = C.c_void_p, C.c_int, C.c_int64, C.c_float, C.c_size_t
_SIGS = {
    "pcb_last_error": (C.c_char_p, []),
    "pcb_version": (C.c_char_p, []),
    "pcb_launch_count": (C.c_uint64, []),
    "pcb_set_device": (_i, [_i]),
    "pcb_coords_pack": (_i, [_p, _l, _p, _p, _p]),
    "pcb_coords_unpack": (_i, [_p, _l, _p, _p]),
    "pcb_hash_build": (_i, [_p, _l, _p, _p, _l, _p, _p]),
    "pcb_coords_stride_ws_bytes": (_sz, [_l]),
    "pcb_coords_stride": (_i, [_p, _l, C.c_int32, _p, _p, C.POINTER(C.c_int64), _p, _sz, _p]),
    "pcb_voxelize_ws_bytes": (_sz, [_l]),
    "pcb_voxelize": (_i, [_p, _l, _f, _p, _p, C.POINTER(C.c_int64), _p, _sz, _p]),
    "pcb_radius_pairs_ws_bytes": (_sz, [_l, _l]),
    "pcb_radius_pairs": (_i, [_p, _l, _p, _l, _f, _p, _l, C.POINTER(C.c_int64), _p, _sz, _p]),
    "pcb_kernel_map": (_i, [_p, _l, _p, _p, _l, _p, _i, _p, _p]),
    "pcb_kernel_map_count": (_i, [_p, _i, _l, _p, _p]),
    "pcb_weight_prep": (_i, [_p, _i, _i, _i, _p, _p, _p, _p, _p]),
    "pcb_conv_forward_ws_bytes": (_sz, [_i, _l, _i, _i]),
    "pcb_conv_forward": (_i, [_p, _i, _p, _l, _p, _i, _l, _i, _i, _p, _p, _p, _p, _p, _i, _p, _sz, _i, _p]),
    "pcb_gather_sum": (_i, [_p, _i, _p, _l, _p, _i, _l, _i, _p, _i, _p, _p]),
    "pcb_conv_wgrad_ws_bytes": (_sz, [_i, _l, _i, _i]),
    "pcb_conv_wgrad": (_i, [_p, _i, _p, _i, _p, _l, _i, _l, _i, _i, _p, _i, _p, _sz, _i, _p]),
    "pcb_weight_tile_bytes": (_sz, [_i, _i, _i, _i]),
    "pcb_weight_tile": (_i, [_p, _i, _i, _i, _p, _p, _i, _p]),
    "pcb_tile_desc_fill": (_i, [_p, _p, _i, _i, _i, _p, _p, _i, _l]),
    "pcb_weight_tile_batch": (_i, [_p, _i, _l, _p]),
    "pcb_conv_forward_split": (_i, [_p, _p, _i, _p, _l, _p, _i, _l, _i, _i, _p, _p, _p, _i, _p, _sz, _i, _p]),
    "pcb_conv_wgrad_split_ws_bytes": (_sz, [_i, _l, _i, _i]),
    "pcb_conv_wgrad_split": (_i, [_p, _p, _i, _p, _p, _i, _p, _l, _i, _l, _i, _i, _p, _i, _p, _sz, _i, _p]),
    "pcb_bn_ws_bytes": (_sz, [_l, _i]),
    "pcb_bn_stats": (_i, [_p, _l, _i, _f, _f, _p, _p, _p, _p, _p, _sz, _p]),
    "pcb_bn_apply": (_i, [_p, _l, _i, _p, _p, _p, _p, _p, _i, _p, _p]),
    "pcb_bn_backward": (_i, [_p, _p, _l, _i, _p, _p, _p, _p, _p, _p, _p, _sz, _p]),
    "pcb_bn_stats_seg": (_i, [_p, _i, _l, _l, _i, _f, _f, _p, _p, _p, _p, _p, _sz, _p]),
    "pcb_bn_apply_seg": (_i, [_p, _i, _l, _l, _i, _p, _p, _p, _p, _p, _i, _i, _p, _i, _p, _p, _i, _p, _p, _p]),
    "pcb_bn_backward_seg": (_i, [_p, _i, _p, _i, _p, _i, _l, _l, _i, _p, _p, _p, _p, _i, _p, _p, _i, _p, _i, _i, _p, _p, _i, _p, _sz,
                                 _p]),
    "pcb_split_rows": (_i, [_p, _i, _l, _i, _p, _p, _i, _i, _p]),
    "pcb_nce_ws_bytes": (_sz, [_l]),
    "pcb_nce_forward_backward": (_i, [_p, _p, _l, _i, _f, _p, _p, _p, _p, _sz, _p]),
    "pcb_l2norm_forward": (_i, [_p, _l, _i, _p, _p, _p]),
    "pcb_l2norm_backward": (_i, [_p, _p, _p, _l, _i, _p, _p]),
    "pcb_pdist_rowmin": (_i, [_p, _l, _p, _l, _i, _p, _p, _p, _p]),
    "pcb_sgd_step": (_i, [_p, _p, _p, _l, _f, _f, _f, _f, _i, _f, _p]),
    "pcb_ce_ws_bytes": (_sz, [_l]),
    "pcb_ce_forward_backward": (_i, [_p, _p, _l, _i, _l, _f, _p, _p, _p, _sz, _p]),
    "pcb_seg_eval_ws_bytes": (_sz, [_l, _i]),
    "pcb_seg_eval": (_i, [_p, _p, _l, _i, _l, _p, _p, _p, _p, _p, _p, _sz, _p]),
    "pcb_profile_enable": (_i, [_i]),
    "pcb_profile_read": (_i, [_p, _p, _i, C.POINTER(C.c_int)]),
    "pcb_unit_ws_bytes": (_sz, [_i, _l, _l, _i, _i]),
    "pcb_unit_forward": (_i, [_p, _p]),
    "pcb_unit_backward": (_i, [_p, _p]),
}


class PcbTileDesc(C.Structure):
    """`struct pcb_tile_desc` of include/pcb200.h."""
    _fields_ = [("W", _p), ("fwd", _p), ("dgrad", _p), ("K", C.c_int32), ("Cin", C.c_int32), ("Cout", C.c_int32), ("flags", C.c_int32),
                ("bn_f", C.c_int32), ("bn_d", C.c_int32), ("start", _l)]


class PcbUnit(C.Structure):
    """`struct pcb_unit` of include/pcb200.h (field for field)."""
    _fields_ = [
        ("n_in", _l), ("n_out", _l), ("n0", _l),
        ("K", C.c_int32), ("Cin", C.c_int32), ("Cout", C.c_int32), ("relu", C.c_int32),
        ("fwd_tbl", _p), ("fwd_stride", _l), ("fwd_kmap", _p),
        ("dg_tbl", _p), ("dg_stride", _l), ("dg_kmap", _p),
        ("wg_tbl", _p), ("wg_stride", _l), ("wg_gather_x", C.c_int32),
        ("W", _p), ("wt_fwd", _p), ("wt_dg", _p), ("dW", _p),
        ("gamma", _p), ("beta", _p), ("running_mean", _p), ("running_var", _p), ("dgamma", _p), ("dbeta", _p),
        ("eps", _f), ("momentum", _f),
        ("mean", _p), ("invstd", _p),
        ("x_p", _p), ("x_ld", C.c_int32), ("x_hi", _p), ("x_lo", _p), ("x_lds", C.c_int32), ("x_bhi", _p), ("x_blo", _p),
        ("z_p", _p), ("z_ld", C.c_int32),
        ("out_p", _p), ("out_ld", C.c_int32), ("out_hi", _p), ("out_lo", _p), ("out_lds", C.c_int32), ("out_bhi", _p), ("out_blo", _p),
        ("res_p", _p), ("res_ld", C.c_int32),
        ("g_p", _p), ("g_ld", C.c_int32),
        ("dz_p", _p), ("dz_hi", _p), ("dz_lo", _p), ("dz_ld", C.c_int32),
        ("gin_p", _p), ("gin_ld", C.c_int32), ("gin_mode", C.c_int32),
        ("gres_p", _p), ("gres_ld", C.c_int32), ("gres_mode", C.c_int32),
        ("ws", _p), ("ws_bytes", _sz),
        ("flags", C.c_int32),
    ]
EXPORTS = sorted(_SIGS)
for _name, (_res, _args) in _SIGS.items():
    _fn = getattr(lib, _name)          # AttributeError here == the library does not export a declared symbol
    _fn.restype = _res
    _fn.argtypes = _args


def check(rc):
    if rc != 0:
        raise PcbError(f"libpcb200 error {rc}: {lib.pcb_last_error().decode()}")


def ptr(t):
    """Device (or None) pointer of a contiguous tensor."""
    if t is None:
        return None
    assert t.is_contiguous(), "libpcb200 needs contiguous tensors"
    return t.data_ptr()


_cur_dev = [-1]


def stream():
    """Current torch stream handle; also keeps the library's CUDA runtime on torch's current device."""
    d = torch.cuda.current_device()
    if d != _cur_dev[0]:
        check(lib.pcb_set_device(d))
        _cur_dev[0] = d
    return torch.cuda.current_stream().cuda_stream


def require_cuda(t):
    if not t.is_cuda:
        raise PcbError("pointcontrast_b200 ops run on CUDA tensors only (no CPU fallback); got a CPU tensor")


def launch_count():
    return int(lib.pcb_launch_count())

"""ctypes binding of libpsg_b200.so -- the C ABI declared in include/psg_b200.h.

The library is the product; there is no Python or CPU fallback.  Importing this module on a
machine where the shared object has not been built raises, and every call checks the returned
status code and raises ``PsgError`` on anything but PSG_OK.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libpsg_b200.so")

PSG_OK, PSG_EINVAL, PSG_EUNSUPPORTED, PSG_EWORKSPACE, PSG_ECUDA = 0, -1, -2, -3, -4
_ERR = {PSG_EINVAL: "invalid argument", PSG_EUNSUPPORTED: "unsupported configuration",
        PSG_EWORKSPACE: "workspace too small", PSG_ECUDA: "CUDA launch failed"}


class PsgError(RuntimeError):
    pass


class MlpDesc(C.Structure):
    _fields_ = [("cin", C.c_int), ("cout", C.c_int), ("w_host", C.c_void_p), ("b_host", C.c_void_p)]


class SaDesc(C.Structure):
    _fields_ = [("npoint", C.c_int), ("nbranch", C.c_int), ("radius", C.c_double * 2), ("nsample", C.c_int * 2),
                ("nlayers", C.c_int * 2), ("mlp", (MlpDesc * 3) * 2)]


class FpDesc(C.Structure):
    _fields_ = [("d1", C.c_int), ("d2", C.c_int), ("nlayers", C.c_int), ("mlp", MlpDesc * 3)]


class NetDesc(C.Structure):
    _fields_ = [("in_channels", C.c_int), ("num_classes", C.c_int), ("sa", SaDesc * 4), ("fp", FpDesc * 4),
                ("conv1", MlpDesc), ("conv2", MlpDesc), ("mlp_mode", C.c_int)]


class NuBuffers(C.Structure):
    _fields_ = [("w", C.c_void_p), ("adam_m", C.c_void_p), ("adam_v", C.c_void_p), ("adv", C.c_void_p),
                ("base", C.c_void_p), ("images", C.c_void_p), ("mask", C.c_void_p), ("labels", C.c_void_p),
                ("cost", C.c_void_p), ("status", C.c_void_p), ("scratch", C.c_void_p),
                ("field_c0", C.c_int), ("field_nc", C.c_int), ("box_lo", C.c_float * 8), ("box_hi", C.c_float * 8)]


_vp, _i, _i64, _f, _sz, _d = C.c_void_p, C.c_int, C.c_int64, C.c_float, C.c_size_t, C.c_double

# name -> (restype, argtypes); status-returning functions are wrapped with a check
_PROTOS = {
    "psg_version": (_i, []),
    "psg_launch_count": (_i64, []),
    "psg_fps_workspace": (_sz, [_i, _i]),
    "psg_fps": (_i, [_vp, _i, _i, _i, _i, _vp, _vp, _vp, _vp, _sz, _vp]),
    "psg_square_distance": (_i, [_vp, _vp, _i, _i, _i, _vp, _vp]),
    "psg_ball_query": (_i, [_vp, _i, _i, _i, _vp, _i, _i, C.POINTER(C.c_double), C.POINTER(C.c_int), _vp, _vp, _vp]),
    "psg_ball_grid_workspace": (_sz, [_i, _i]),
    "psg_ball_query_grid": (_i, [_vp, _i, _i, _i, _vp, _i, _i, C.POINTER(C.c_double), C.POINTER(C.c_int), _vp, _vp, _vp, _sz, _vp]),
    "psg_three_nn": (_i, [_vp, _i, _i, _i, _vp, _i, _vp, _vp, _vp, _vp]),
    "psg_index_points": (_i, [_vp, _vp, _i, _i, _i, _i64, _vp, _vp]),
    "psg_pack_channels_first": (_i, [_vp, _i64, _i64, _i64, _i, _i, _i, _vp, _i, _i, _vp, _vp]),
    "psg_unpack_channels_first": (_i, [_vp, _i, _i, _i, _i, _i, _vp, _i, _vp]),
    "psg_group_points": (_i, [_vp, _i, _i, _vp, _i, _i, _vp, _vp, _i, _i, _i, _vp, _i, _vp]),
    "psg_group_max": (_i, [_vp, _i, _i64, _i, _i, _vp, _i, _i, _vp, _vp]),
    "psg_group_max_backward": (_i, [_vp, _i, _i, _vp, _i, _i, _vp, _i64, _i, _i, _vp, _i, _vp]),
    "psg_interpolate": (_i, [_vp, _i, _i, _vp, _vp, _i64, _i, _i, _vp, _i, _i, _vp]),
    "psg_csr_workspace": (_sz, [_i64, _i, _i]),
    "psg_csr_build_by_source": (_i, [_vp, _i64, _i, _i, _i, _vp, _vp, _vp, _vp]),
    "psg_segment_sum": (_i, [_vp, _i, _i, _i64, _i, _vp, _vp, _vp, _i, _i, _i64, _i, _vp, _i, _i, _i, _vp]),
    "psg_mlp_create": (_vp, [_vp, _vp, _i, _i]),
    "psg_mlp_destroy": (None, [_vp]),
    "psg_mlp_create_device": (_vp, [_i, _i]),
    "psg_mlp_load": (_i, [_vp, _vp, _vp, _vp]),
    "psg_bn_workspace": (_sz, [_i]),
    "psg_bn_train_forward": (_i, [_vp, _i, _i64, _i, _vp, _vp, _vp, _vp, _f, _f, _vp, _i, _i, _vp, _vp, _vp, _sz, _vp]),
    "psg_bn_train_backward": (_i, [_vp, _i, _vp, _i, _vp, _i, _i64, _i, _vp, _vp, _vp, _vp, _vp, _vp, _i, _vp, _sz, _vp]),
    "psg_wgrad_workspace": (_sz, [_i, _i, _i64]),
    "psg_conv_wgrad": (_i, [_vp, _i, _i, _vp, _i, _i, _i, _vp, _i, _i, _i, _i64, _vp, _vp, _i, _vp, _sz, _vp]),
    "psg_log_softmax_rows": (_i, [_vp, _i, _i64, _i, _vp, _vp]),
    "psg_dlogits_from_dlogp": (_i, [_vp, _i, _vp, _i64, _i, _vp, _i, _vp]),
    "psg_nll_workspace": (_sz, []),
    "psg_nll_loss": (_i, [_vp, _vp, _vp, _i64, _i, _vp, _vp, _vp, _sz, _vp]),
    "psg_nll_loss_backward": (_i, [_vp, _vp, _i64, _i, _vp, _vp, _vp, _vp]),
    "psg_tl_mul": (_i, [_vp, _i, _vp, _i, _i64, _i, _f, _vp]),
    "psg_adam_step": (_i, [_vp, _vp, _vp, _vp, _i64, _f, _f, _f, _f, _f, _i, _vp]),
    "psg_mlp_forward": (_i, [_vp, _vp, _i, _i, _i, _vp, _i, _i, _i, _i64, _vp, _i, _i, _i, _vp]),
    "psg_mlp_backward": (_i, [_vp, _vp, _i, _i64, _vp, _i, _vp, _i, _i, _vp]),
    "psg_dense_knn": (_i, [_vp, _i, _i, _i, _i, _vp, _vp, _vp]),
    "psg_pairwise_distance": (_i, [_vp, _i, _i, _i, _vp, _vp]),
    "psg_net_create": (_vp, [C.POINTER(NetDesc)]),
    "psg_net_destroy": (None, [_vp]),
    "psg_net_set_mlp_mode": (_i, [_vp, _i]),
    "psg_net_workspace": (_sz, [_vp, _i, _i, _i]),
    "psg_net_bind": (_i, [_vp, _i, _i, _i, _vp, _sz]),
    "psg_net_set_input": (_i, [_vp, _vp, _i64, _i64, _i64, _vp]),
    "psg_net_copy_input": (_i, [_vp, _vp, _vp]),
    "psg_debug_l2_stream": (_i, [_vp, _i64, _i, _i, _i, _i, _vp]),
    "psg_net_geometry": (_i, [_vp, _vp, _i, _vp]),
    "psg_net_read_geometry": (_i, [_vp, _i, _i, _i, _i, _vp, _sz, _vp]),
    "psg_net_forward": (_i, [_vp, _i, _vp, _vp, _vp]),
    "psg_net_loss_grad": (_i, [_vp, _i, _vp, _vp, _i, _f, _f, _vp, _vp]),
    "psg_net_backward": (_i, [_vp, _i, _vp, _vp]),
    "psg_net_pgd_update": (_i, [_vp, _vp, _vp, _vp, _i, _i, _f, _f, _f, _f, _vp]),
    "psg_nb_attack": (_i, [_vp, _vp, _vp, _vp, _vp, _i, _i, _i, _f, _f, _f, _vp]),
    "psg_net_pgd_update_l2": (_i, [_vp, _vp, _vp, _vp, _i, _i, _f, _f, _f, _f, _vp]),
    "psg_nb_attack_l2": (_i, [_vp, _vp, _vp, _vp, _vp, _i, _i, _i, _f, _f, _f, _vp]),
    "psg_nu_scratch_floats": (_sz, [_i, _i]),
    "psg_nu_init": (_i, [_vp, C.POINTER(NuBuffers), _vp]),
    "psg_nu_step": (_i, [_vp, C.POINTER(NuBuffers), _i, _i, _i, _i, _f, _f, _f, _f, _f, _i, _d, _d, _i, _i, _vp, _vp]),
    "psg_net_set_xyz_grad": (_i, [_vp, _i]),
    "psg_clamp": (_i, [_vp, _i64, _f, _f, _vp]),
    "psg_add_vote": (_i, [_vp, _vp, _vp, _i64, _i, _vp, _i64, _vp]),
    "psg_set_option": (_i, [C.c_char_p, _i]),
    "psg_prof_enable": (_i, [_i]),
    "psg_prof_ncat": (_i, []),
    "psg_prof_name": (C.c_char_p, [_i]),
    "psg_prof_collect": (_i, [C.POINTER(C.c_double), C.POINTER(C.c_int64)]),
    "psg_confusion_matrix": (_i, [_vp, _vp, _vp, _i, _i64, _i, _vp, _vp]),
    "psg_debug_trace": (_i, [_vp, _i]),
    "psg_scene_minmax_workspace": (_sz, []),
    "psg_scene_minmax": (_i, [_vp, _i64, _i, _vp, _vp, _sz, _vp]),
    "psg_scene_chunks": (_i64, [_i64]),
    "psg_scene_cell_counts": (_i, [_vp, _i64, _i, _vp, _i, _vp, _vp, _vp]),
    "psg_scene_cell_fill": (_i, [_vp, _i64, _i, _vp, _i, _vp, _vp, _vp, _vp]),
    "psg_scene_gather": (_i, [_vp, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i, _i64, _i, _vp, _vp, _vp, _vp, _vp, _vp]),
}

EXPORTS = tuple(_PROTOS)


def _load():
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} is missing: build it with ./build.sh (or __graft_entry__.build()). "
            "pointsecguard_b200 has no CPU or pure-PyTorch fallback.")
    return C.CDLL(LIB_PATH)


_cdll = _load()


def _wrap(name, restype, argtypes):
    fn = getattr(_cdll, name)
    fn.restype = restype
    fn.argtypes = argtypes
    if restype is not _i or name in ("psg_version", "psg_prof_ncat"):
        return fn

    def checked(*args):
        rc = fn(*args)
        if rc != PSG_OK:
            raise PsgError(f"{name} failed: {_ERR.get(rc, rc)} ({rc})")
        return rc

    checked.__name__ = name
    return checked


for _n, (_r, _a) in _PROTOS.items():
    globals()[_n] = _wrap(_n, _r, _a)


# ---- device discipline -----------------------------------------------------------------------------
# The C library launches on the CURRENT CUDA device and on the stream it is handed.  Every Python entry point of the
# package therefore runs with the device of its tensors made current, and asks torch for that device's current stream
# (a model on cuda:1 while cuda:0 is current would otherwise launch on cuda:0's stream with cuda:1's pointers).
def on_device_of(fn):
    """Decorator: run ``fn`` with the CUDA device of its first CUDA-tensor argument made current."""
    import functools

    import torch

    @functools.wraps(fn)
    def wrapped(*args, **kwargs):
        for a in args:
            if isinstance(a, torch.Tensor) and a.is_cuda:
                if a.device.index == torch.cuda.current_device():
                    break
                with torch.cuda.device(a.device):
                    return fn(*args, **kwargs)
        return fn(*args, **kwargs)

    return wrapped

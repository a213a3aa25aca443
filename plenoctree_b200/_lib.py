"""ctypes binding of libplenoctree_b200.so (the C ABI in include/plenoctree_b200.h).

There is no fallback: if the shared library is missing the import raises, and every compute entry
point fails when no sm_100 device is present.
"""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("POB_LIB_PATH") or os.path.join(_HERE, "libplenoctree_b200.so")   # override: kernel A/B experiments

PREC_FP16 = 1
PREC_FP16X3 = 3

_c = ctypes
_vp, _i, _i64, _u32, _fp = _c.c_void_p, _c.c_int, _c.c_int64, _c.c_uint32, _c.c_void_p

# name -> (restype, argtypes); must list every symbol the header declares
SIGNATURES = {
    "pob_abi_version": (_i, []),
    "pob_last_error": (_c.c_char_p, []),
    "pob_sm_count": (_i, []),
    "pob_launch_count": (_c.c_longlong, []),
    "pob_timing_enable": (None, [_i]),
    "pob_timing_read": (_i, [_vp, _vp]),
    "pob_param_count": (_i64, [_i]),
    "pob_packed_bytes": (_i64, [_i]),
    "pob_pack_weights": (_i, [_fp, _i, _vp, _vp]),
    "pob_eval_points_raw": (_i, [_vp, _i, _fp, _i64, _fp, _fp, _i, _vp]),
    "pob_debug_trace_fwd": (_i, [_vp, _i, _fp, _i64, _fp, _vp, _vp, _vp, _vp, _vp]),
    "pob_debug_trace_bwd": (_i, [_vp, _i, _i64, _fp, _fp, _vp, _vp, _vp, _vp, _vp]),
    "pob_eval_points": (_i, [_vp, _i, _fp, _fp, _i64, _fp, _i, _vp]),
    "pob_eval_cells_mean": (_i, [_vp, _i, _fp, _i64, _i, _fp, _i, _vp]),
    "pob_eval_grid": (_i, [_vp, _i, _i, _i, _i, _i, _i, _c.POINTER(_c.c_float), _c.POINTER(_c.c_float),
                           _fp, _fp, _i, _vp]),
    "pob_eval_points_raw_host": (_i, [_vp, _i, _fp, _i64, _fp, _fp, _i]),
    "pob_sample_coarse": (_i, [_fp, _fp, _i, _i, _fp, _vp]),
    "pob_draw_uniforms": (_i, [_c.c_uint64, _c.c_float, _fp, _fp, _i64, _fp, _i64, _fp, _i64, _c.c_float, _vp]),
    "pob_composite": (_i, [_fp, _fp, _fp, _i, _i, _i, _fp, _fp, _fp, _fp, _vp]),
    "pob_composite_bwd": (_i, [_fp, _fp, _fp, _fp, _fp, _i, _i, _i, _c.c_float, _fp, _fp, _vp]),
    "pob_sample_pdf": (_i, [_fp, _fp, _fp, _i, _i, _i, _i, _fp, _vp]),
    "pob_workspace_bytes": (_i64, [_vp, _i]),
    "pob_render_rays": (_i, [_vp, _vp, _vp, _fp, _fp, _fp, _i, _fp, _fp, _fp, _i, _fp, _fp, _fp, _vp, _i, _vp]),
    "pob_loss_and_grad": (_i, [_vp, _vp, _vp, _vp, _fp, _fp, _fp, _fp, _i, _fp, _fp, _fp, _i, _fp, _fp, _fp, _fp,
                               _vp, _vp]),
    "pob_adam_update": (_i, [_i, _i, _fp, _fp, _fp, _fp, _c.c_float, _c.c_float, _fp, _c.c_float, _c.c_float,
                             _vp, _vp, _vp]),
    "pob_octree_render": (_i, [_vp, _vp, _fp, _fp, _fp, _i64, _vp, _i, _i, _fp, _vp, _vp]),
    "pob_octree_render_backward": (_i, [_vp, _vp, _fp, _fp, _fp, _i64, _vp, _i, _i, _fp, _fp, _vp]),
    "pob_octree_train_persp": (_i, [_vp, _vp, _vp, _i, _i, _fp, _c.c_float, _fp, _vp, _fp, _vp]),
    "pob_octree_sgd_step": (_i, [_fp, _fp, _i64, _c.c_float, _vp]),
    "pob_octree_adam_step": (_i, [_fp, _fp, _fp, _fp, _i64, _c.c_float, _c.c_float, _c.c_float, _vp]),
    "pob_octree_query": (_i, [_vp, _fp, _i64, _vp, _vp]),
    "pob_grid_weight_render": (_i, [_fp, _i, _vp, _i, _i, _i, _c.POINTER(_c.c_float), _c.POINTER(_c.c_float),
                                    _vp, _fp, _vp, _vp]),
    "pob_umma_probe": (_i, [_vp, _u32, _vp, _u32, _u32, _vp, _vp, _vp, _vp, _i, _u32, _i, _fp, _vp]),
    "pob_umma_probe_pair": (_i, [_vp, _u32, _vp, _u32, _u32, _vp, _vp, _vp, _vp, _i, _u32, _i, _fp, _vp]),
}


class RenderConfig(_c.Structure):
    _fields_ = [("sh_deg", _i), ("num_coarse_samples", _i), ("num_fine_samples", _i), ("white_bkgd", _i),
                ("max_rays", _i), ("sparsity_npoints", _i), ("sigma_noise_coarse_dev", _vp),
                ("sigma_noise_fine_dev", _vp)]


class TrainHParams(_c.Structure):
    _fields_ = [("sparsity_weight", _c.c_float), ("sparsity_length", _c.c_float), ("loss_scale", _c.c_float)]


class Octree(_c.Structure):
    _fields_ = [("data_dev", _vp), ("child_dev", _vp), ("n_nodes", _i64), ("N", _i), ("data_dim", _i),
                ("basis_dim", _i), ("format", _i), ("offset", _c.c_float * 3), ("invradius", _c.c_float * 3)]


class OctreeOpts(_c.Structure):
    _fields_ = [("step_size", _c.c_float), ("background_brightness", _c.c_float), ("sigma_thresh", _c.c_float),
                ("stop_thresh", _c.c_float)]


class Camera(_c.Structure):
    _fields_ = [("c2w", _c.c_float * 12), ("fx", _c.c_float), ("fy", _c.c_float), ("width", _c.c_float),
                ("height", _c.c_float)]


class PobError(RuntimeError):
    pass


def _load():
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} not found: build it with `python -m plenoctree_b200.build` "
            "(there is no CPU fallback)")
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    return lib


lib = _load()


def check(rc):
    if rc != 0:
        raise PobError(lib.pob_last_error().decode())


def ptr(t):
    """device/host pointer of a torch tensor or numpy array (None -> NULL)."""
    if t is None:
        return None
    if hasattr(t, "data_ptr"):
        return t.data_ptr()
    return t.ctypes.data


def stream_ptr():
    import torch
    return torch.cuda.current_stream().cuda_stream

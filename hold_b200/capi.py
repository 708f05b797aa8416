"""ctypes binding of libhold_b200.so (include/hold_b200.h).

PyTorch is used for device memory and streams only; every arithmetic step of the path runs in the
library's sm_100a kernels.  There is no fallback: if the library is missing or no B200 is visible the
import of the product path raises.
"""
from __future__ import annotations

import ctypes as C
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libhold_b200.so")

MAX_NODES, MAX_LAYERS = 4, 9
KIND_HAND, KIND_OBJECT = 0, 1
MLP_FP32, MLP_TC = 0, 1

fp = C.c_void_p  # device pointers travel as void*


class NodeCfg(C.Structure):
    _fields_ = [("kind", C.c_int32), ("class_id", C.c_int32), ("n_samples_eval", C.c_int32), ("n_samples", C.c_int32),
                ("n_samples_extra", C.c_int32), ("beta_iters", C.c_int32), ("max_total_iters", C.c_int32),
                ("mlp_mode", C.c_int32), ("eps", C.c_float), ("add_tiny", C.c_float), ("near", C.c_float),
                ("bounding_sphere", C.c_float), ("beta_min", C.c_float)]


class MlpWeights(C.Structure):
    _fields_ = [("n_layers", C.c_int32), ("in_dim", C.c_int32 * MAX_LAYERS), ("out_dim", C.c_int32 * MAX_LAYERS),
                ("weight_v", fp * MAX_LAYERS), ("weight_g", fp * MAX_LAYERS), ("bias", fp * MAX_LAYERS)]


class ManoModel(C.Structure):
    _fields_ = [("v_template", fp), ("shapedirs", fp), ("posedirs", fp), ("J_regressor", fp), ("lbs_weights", fp),
                ("hands_mean", fp), ("parents_host", C.POINTER(C.c_int32)), ("tip_ids_host", C.POINTER(C.c_int32))]


class NodePose(C.Structure):
    _fields_ = [("tfs", fp), ("posed_verts", fp), ("pose_cond", fp), ("time_code", fp), ("embed_w", fp), ("beta_param", fp)]


class Factors(C.Structure):
    _fields_ = [("color", fp), ("normal", fp), ("density", fp), ("z_vals", fp), ("sdf", fp), ("canonical_pts", fp)]


class RenderOut(C.Structure):
    _fields_ = [("fg_rgb", fp), ("mask_prob", fp), ("normal", fp), ("depth", fp), ("fg_semantics", fp), ("bg_weights", fp),
                ("fg_weights", fp)]


class EwArgs(C.Structure):
    _fields_ = [("in0", fp), ("in1", fp), ("in2", fp), ("out0", fp), ("out1", fp), ("ld_in0", C.c_int32), ("ld_in1", C.c_int32),
                ("ld_in2", C.c_int32), ("ld_out0", C.c_int32), ("ld_out1", C.c_int32), ("ncols", C.c_int32), ("aux", C.c_int32)]


class SamplerRand(C.Structure):
    _fields_ = [("jitter", fp), ("u", fp), ("extra_idx", fp)]


EXPORTS = {
    "hold_version": (C.c_int, []),
    "hold_last_error": (C.c_char_p, []),
    "hold_ctx_create": (C.c_int, [C.POINTER(C.c_void_p), C.c_int]),
    "hold_ctx_destroy": (C.c_int, [C.c_void_p]),
    "hold_ctx_check": (C.c_int, [C.c_void_p, C.c_void_p]),
    "hold_ctx_launch_count": (C.c_int64, [C.c_void_p]),
    "hold_node_configure": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(NodeCfg)]),
    "hold_node_set_weights": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(MlpWeights), C.POINTER(MlpWeights), fp, fp, C.c_void_p]),
    "hold_node_set_rig": (C.c_int, [C.c_void_p, C.c_int, fp, fp, C.c_void_p]),
    "hold_mano_lbs": (C.c_int, [C.c_void_p, C.POINTER(ManoModel), C.c_int, fp, fp, fp, fp, fp, fp, fp, fp, fp, C.c_void_p]),
    "hold_object_tf": (C.c_int, [C.c_void_p, C.c_int, fp, fp, fp, C.c_float, fp, fp, C.c_int, fp, fp, C.c_void_p]),
    "hold_inverse_warp_bwd": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, fp, C.POINTER(NodePose), C.c_void_p, fp, fp, fp, C.c_void_p]),
    "hold_mise_create": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_float, C.POINTER(C.c_void_p), C.c_void_p]),
    "hold_mise_query": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.POINTER(C.c_int), C.c_void_p]),
    "hold_mise_update": (C.c_int, [C.c_void_p, fp, C.c_int, C.c_void_p]),
    "hold_mise_to_dense": (C.c_int, [C.c_void_p, fp, C.c_void_p]),
    "hold_mc_mark": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, fp, C.c_float, C.c_void_p, C.c_void_p, C.c_void_p]),
    "hold_mc_emit": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, fp, C.c_float, C.c_void_p, C.c_void_p, C.c_void_p, fp, C.c_void_p, C.c_void_p]),
    "hold_mise_destroy": (C.c_int, [C.c_void_p]),
    "hold_mesh_sdf": (C.c_int, [C.c_void_p, C.c_int, C.c_int, fp, C.c_int, fp, C.c_int, C.c_int, C.c_void_p, fp, C.c_void_p, C.c_void_p]),
    "hold_off_in_surface": (C.c_int, [C.c_void_p, C.c_int, C.c_int, fp, C.c_float, C.c_void_p, C.c_void_p, C.c_void_p]),
    "hold_mano_lbs_bwd": (C.c_int, [C.c_void_p, C.POINTER(ManoModel), C.c_int] + [fp] * 12 + [C.c_void_p]),
    "hold_object_tf_bwd": (C.c_int, [C.c_void_p, C.c_int, fp, fp, fp, C.c_float, fp, fp, C.c_int] + [fp] * 6 + [C.c_void_p]),
    "hold_camera_rays": (C.c_int, [C.c_void_p, C.c_int, C.c_int, fp, fp, fp, fp, fp, C.c_void_p]),
    "hold_sample": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, fp, fp, C.POINTER(NodePose), C.POINTER(SamplerRand), fp, fp, C.c_void_p]),
    "hold_sampler_round": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int] + [fp] * 11 + [C.POINTER(C.c_int32), C.c_void_p]),
    "hold_shade": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, fp, fp, C.POINTER(NodePose), C.POINTER(Factors), C.c_void_p]),
    "hold_composite": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.POINTER(Factors), C.POINTER(C.c_int32), C.POINTER(RenderOut), C.POINTER(RenderOut), C.c_void_p]),
    "hold_composite_bwd": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.POINTER(Factors), C.POINTER(C.c_int32), C.POINTER(RenderOut), C.POINTER(RenderOut), C.POINTER(Factors), C.c_void_p]),
    "hold_render_fg": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(C.c_int32), C.c_int, C.c_int, fp, fp, C.POINTER(NodePose), C.POINTER(Factors), C.POINTER(RenderOut), C.POINTER(RenderOut), fp, C.c_void_p]),
    "hold_bg_set_weights": (C.c_int, [C.c_void_p, C.POINTER(MlpWeights), C.POINTER(MlpWeights), C.c_int, C.c_void_p]),
    "hold_background": (C.c_int, [C.c_void_p, C.c_int, C.c_int, fp, fp, fp, fp, fp, fp, fp, fp, C.c_void_p]),
    "hold_sdf_eval": (C.c_int, [C.c_void_p, C.c_int, C.c_int, fp, fp, fp, fp, fp, C.c_void_p]),
    "hold_linear": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, fp, C.c_int, C.c_int, C.c_int, fp, fp, C.c_int, C.c_int, C.c_void_p]),
    "hold_wgrad": (C.c_int, [C.c_void_p, C.c_int, fp, C.c_int, C.c_int, fp, C.c_int, C.c_int, fp, fp, fp, C.c_int, C.c_void_p]),
    "hold_pow2_scale": (C.c_int, [C.c_void_p, C.c_int, C.c_int, fp, C.c_int, fp, C.c_void_p]),
    "hold_train_ew": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.POINTER(EwArgs), C.c_void_p]),
    "hold_rgb_eval": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, fp, fp, fp, fp, fp, fp, C.c_void_p]),
    "hold_forward_warp": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, fp, C.POINTER(NodePose), fp, fp, fp, C.c_void_p]),
    "hold_inverse_warp": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, fp, C.POINTER(NodePose), fp, fp, fp, C.c_void_p]),
    "hold_train_glue_sizes": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_int64), C.POINTER(C.c_int64)]),
    "hold_normal_density": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int] + [fp] * 8 + [C.c_void_p]),
    "hold_normal_density_bwd": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int] + [fp] * 11 + [C.c_void_p]),
    "hold_bg_inputs": (C.c_int, [C.c_void_p, C.c_int, C.c_float, fp, fp, fp, fp, C.c_void_p]),
    "hold_bg_integrate": (C.c_int, [C.c_void_p, C.c_int, C.c_float, fp, C.c_int, fp, fp, fp, fp, fp, C.c_void_p]),
    "hold_bg_integrate_bwd": (C.c_int, [C.c_void_p, C.c_int, C.c_float, fp, C.c_int, fp, fp, fp, fp, fp, fp, fp, fp, C.c_void_p]),
}

_lib = None


def lib():
    """The loaded library.  Loading needs only libcudart, so this also works on a GPU-less box
    (symbol/ABI checks); any compute entry point fails there with HOLD_E_CUDA."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(f"{LIB_PATH} is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                               "(hold_b200 has no CPU/PyTorch fallback)")
        _lib = C.CDLL(LIB_PATH)
        for name, (res, args) in EXPORTS.items():
            f = getattr(_lib, name)
            f.restype, f.argtypes = res, args
    return _lib


class HoldError(RuntimeError):
    pass


def check(rc: int):
    if rc != 0:
        raise HoldError(f"hold_b200 error {rc}: {lib().hold_last_error().decode()}")


def ptr(t):
    """Device pointer of a contiguous fp32/int32/uint8 CUDA tensor (None -> NULL)."""
    if t is None:
        return None
    assert t.is_cuda and t.is_contiguous(), "hold_b200 takes contiguous CUDA tensors"
    return C.c_void_p(t.data_ptr())


def stream_ptr():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


class Context:
    """One hold_ctx per (process, device)."""

    def __init__(self, device: int | None = None):
        if not torch.cuda.is_available():
            raise HoldError("no CUDA device visible: hold_b200 has no CPU fallback")
        self.device = torch.cuda.current_device() if device is None else device
        h = C.c_void_p()
        check(lib().hold_ctx_create(C.byref(h), self.device))
        self.h = h
        self._keep = {}  # python-side references to tensors the library reads lazily (none today)

    def close(self):
        if getattr(self, "h", None):
            lib().hold_ctx_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def check(self):
        check(lib().hold_ctx_check(self.h, stream_ptr()))

    @property
    def launches(self) -> int:
        return int(lib().hold_ctx_launch_count(self.h))


def mlp_weights(sd: dict, n_layers: int) -> tuple[MlpWeights, list]:
    """Pack a reference-format state_dict (`lin<k>.weight_v/weight_g/bias`, or plain `.weight`) of CUDA tensors."""
    w = MlpWeights()
    w.n_layers = n_layers
    keep = []
    for l in range(n_layers):
        if f"lin{l}.weight_v" in sd:
            v, g = sd[f"lin{l}.weight_v"], sd[f"lin{l}.weight_g"]
        else:
            v, g = sd[f"lin{l}.weight"], None
        b = sd[f"lin{l}.bias"]
        v = v.detach().float().contiguous()
        b = b.detach().float().contiguous()
        g = None if g is None else g.detach().float().contiguous()
        keep += [v, g, b]
        w.out_dim[l], w.in_dim[l] = v.shape[0], v.shape[1]
        w.weight_v[l] = v.data_ptr()
        w.weight_g[l] = g.data_ptr() if g is not None else None
        w.bias[l] = b.data_ptr()
    return w, keep
TC_READY = True  # tcgen05 MLP path built into libhold_b200.so

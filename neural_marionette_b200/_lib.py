"""ctypes binding of the nm_b200 C ABI (include/nm_b200.h).

There is no CPU fallback: if the shared library is missing or a call fails the
caller gets an exception.  PyTorch only supplies device memory (``data_ptr``)
and the current CUDA stream.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "csrc", "libnm_b200.so")

_vp, _i, _f, _d, _sz, _ll = C.c_void_p, C.c_int, C.c_float, C.c_double, C.c_size_t, C.c_longlong


class HsvrnnWeights(C.Structure):
    _fields_ = [(n, _vp) for n in (
        "post0_wt", "post0_b", "post2_wt", "post2_b",
        "prior0_wt", "prior0_b", "prior2_wt", "prior2_b",
        "root0_wt", "root0_b", "root2_wt", "root2_b",
        "joint0_wt", "joint0_b", "joint2_wt", "joint2_b",
        "gru_ih_wt", "gru_hh_wt", "gru_ih_b", "gru_hh_b")]


class HsvrnnGrads(C.Structure):
    _fields_ = [(n, _vp) for n in (
        "post0_w", "post0_b", "post2_w", "post2_b", "prior0_w", "prior0_b", "prior2_w", "prior2_b",
        "root0_w", "root0_b", "root2_w", "root2_b", "joint0_w", "joint0_b", "joint2_w", "joint2_b",
        "gru_ih_w", "gru_hh_w", "gru_ih_b", "gru_hh_b", "init_state", "offset_param")]


# name -> (restype, argtypes); every symbol declared in include/nm_b200.h
PROTOTYPES = {
    "nm_last_error": (C.c_char_p, []),
    "nm_version": (_i, []),
    "nm_device_supported": (_i, []),
    "nm_voxelize": (_i, [_vp, _i, _i, _i, _i, _vp, _vp, _vp]),
    "nm_normalize_voxelize_workspace_bytes": (_sz, [_i]),
    "nm_normalize_voxelize": (_i, [_vp, _i, _i, _i, _i, _f, _d, _d, _vp, _vp, _vp, _vp, _vp]),
    "nm_pack_conv_weights": (_i, [_vp, _vp, _i, _i, _i, _vp]),
    "nm_conv3d_tc": (_i, [_vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _i, _i, _vp, _vp]),
    "nm_conv3d_stats_chunks": (_i, [_i, _i, _i, _i, _i, _i, _i, _i]),
    "nm_conv3d_can_fuse_input": (_i, [_i, _i, _i, _i, _i, _i, _i, _i]),
    "nm_conv3d_up2x_supported": (_i, [_i, _i, _i, _i, _i, _i]),
    "nm_conv3d_tc_up2x": (_i, [_vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _vp, _vp, _i, _vp, _vp]),
    "nm_conv_transpose3d_pw_supported": (_i, [_i, _i, _i, _i, _i, _i]),
    "nm_conv_transpose3d_pw_stats_chunks": (_i, [_i, _i, _i, _i, _i, _i]),
    "nm_conv_transpose3d_pw_packed_bytes": (_sz, [_i, _i]),
    "nm_pack_conv_transpose3d_pw_weights": (_i, [_vp, _i, _i, _vp, _vp]),
    "nm_conv_transpose3d_pw": (_i, [_vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _vp, _vp]),
    "nm_conv3d_pw_supported": (_i, [_i, _i, _i, _i, _i, _i, _i, _i]),
    "nm_conv3d_pw_dual_supported": (_i, [_i, _i, _i, _i, _i, _i, _i, _i]),
    "nm_conv3d_pw_stats_chunks": (_i, [_i, _i, _i, _i, _i, _i, _i, _i]),
    "nm_conv3d_pw_packed_bytes": (_sz, [_i, _i, _i]),
    "nm_pack_conv_pw_weights": (_i, [_vp, _i, _i, _i, _vp, _vp]),
    "nm_conv3d_pw": (_i, [_vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _i, _i, _vp, _vp, _i, _vp, _vp, _vp, _vp, _vp]),
    "nm_conv3d_tc_fused": (_i, [_vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _i, _i, _vp, _vp, _i, _vp, _vp]),
    "nm_groupnorm_finalize": (_i, [_vp, _i, _i, _i, _i, _i, _vp, _vp, _f, _vp, _vp, _vp, _vp, _vp]),
    "nm_conv3d_direct": (_i, [_vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _i, _i, _i, _vp]),
    "nm_conv_transpose3d_k2s2": (_i, [_vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _vp]),
    "nm_first_conv_tables_bytes": (_sz, [_i]),
    "nm_first_conv_prepare": (_i, [_vp, _i, _vp, _vp]),
    "nm_first_conv_stats_chunks": (_i, [_i]),
    "nm_first_conv_k5": (_i, [_vp, _vp, _vp, _vp, _i, _i, _i, _vp, _vp, _vp]),
    "nm_gn_workspace_bytes": (_sz, [_i, _i, _i]),
    "nm_groupnorm_scale_shift": (_i, [_vp, _i, _i, _i, _i, _vp, _vp, _f, _vp, _vp, _vp, _vp, _vp, _vp]),
    "nm_affine_act": (_i, [_vp, _vp, _vp, _i, _vp, _vp, _vp, _vp, _i, _i, _i, _vp]),
    "nm_upsample2x": (_i, [_vp, _vp, _vp, _i, _vp, _i, _i, _i, _i, _i, _vp]),
    "nm_ndhwc_to_ncdhw_f32": (_i, [_vp, _vp, _i, _i, _i, _ll, _vp]),
    "nm_ncdhw_f32_to_ndhwc": (_i, [_vp, _vp, _i, _i, _i, _vp]),
    "nm_mean_over_frames": (_i, [_vp, _vp, _i, _i, _ll, _vp]),
    "nm_final_recon_workspace_bytes": (_sz, [_i]),
    "nm_final_recon": (_i, [_vp, _vp, _vp, _vp, _f, _vp, _vp, _i, _f, _f, _vp, _vp, _vp, _vp, _i, _i, _i, _vp]),
    "nm_chamfer_workspace_bytes": (_sz, [_i]),
    "nm_chamfer_vol_fit": (_i, [_vp, _vp, _vp, _i, _i, _i, _vp, _vp, _vp]),
    "nm_heatmap_head": (_i, [_vp, _vp, _vp, _i, _i, _i, _i, _i, _vp, _i, _f, _f, _f, _vp, _vp, _f, _vp, _vp, _vp, _vp,
                             _vp]),
    "nm_gaussian_render": (_i, [_vp, _i, _i, _i, _vp, _f, _vp, _vp]),
    "nm_decoder_adjust_workspace_bytes": (_sz, [_i, _i]),
    "nm_decoder_adjust": (_i, [_vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _vp, _f, _vp, _vp, _vp]),
    "nm_hsvrnn_step": (_i, [C.POINTER(HsvrnnWeights), _vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i,
                            _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "nm_hsvrnn_step_record": (_i, [C.POINTER(HsvrnnWeights), _vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i,
                                   _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "nm_hsvrnn_backward_workspace_bytes": (_sz, [_i, _i]),
    "nm_hsvrnn_step_backward": (_i, [C.POINTER(HsvrnnWeights), C.POINTER(HsvrnnWeights)] + [_vp] * 10 + [_i, _i, _i] +
                                [_vp] * 11),
    "nm_hsvrnn_weight_grads": (_i, [_vp] * 9 + [_i, _i, _i, C.POINTER(HsvrnnGrads), _vp]),
    "nm_hsvrnn_decode_pose": (_i, [C.POINTER(HsvrnnWeights), _vp, _vp, _vp, _vp, _i, _i, _vp, _vp, _vp]),
    "nm_hsvrnn_bone_offsets": (_i, [_vp, _vp, _vp, _i, _i, _i, _vp, _vp]),
    "nm_voxel_chamfer_workspace_bytes": (_sz, [_i, _i]),
    "nm_voxel_chamfer": (_i, [_vp, _vp, _i, _i, _i, _vp, _vp, _vp, _vp, _vp]),
    "nm_semantic_nearest": (_i, [_vp, _vp, _i, _i, _i, _f, _vp, _vp, _vp]),
    "nm_skin_weights": (_i, [_vp, _i, _vp, _vp, _i, _i, _f, _f, _vp, _vp, _vp, _vp]),
    "nm_retarget_fk": (_i, [_vp, _vp, _vp, _vp, _vp, _i, _i, _i, _vp, _vp]),
    "nm_linear_blend_skinning": (_i, [_vp, _i, _vp, _vp, _vp, _vp, _i, _i, _vp, _vp]),
    "nm_conv3d_k3_wgrad_workspace_bytes": (_sz, [_i, _i, _i, _i, _i, _i]),
    "nm_conv3d_k3_wgrad": (_i, [_vp, _vp, _i, _i, _i, _i, _i, _i, _f, _vp, _vp, _vp]),
    "nm_conv3d_k3_wgrad_tc_supported": (_i, [_i, _i, _i, _i, _i, _i]),
    "nm_conv3d_k3_wgrad_tc_workspace_bytes": (_sz, [_i, _i, _i, _i, _i, _i]),
    "nm_conv3d_k3_wgrad_tc": (_i, [_vp, _vp, _i, _i, _i, _i, _i, _i, _f, _vp, _vp, _vp]),
    "nm_groupnorm_backward_workspace_bytes": (_sz, [_i, _i, _i]),
    "nm_groupnorm_backward": (_i, [_vp, _vp, _vp, _vp, _i, _ll, _i, _i, _f, _i, _f, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "nm_conv3d_wgrad_gather_workspace_bytes": (_sz, [_i, _i, _i, _i, _i, _i, _i, _i]),
    "nm_conv3d_wgrad_gather": (_i, [_vp, _vp, _i, _i, _i, _i, _i, _i, _i, _i, _f, _vp, _vp, _vp]),
    "nm_depth_to_space2": (_i, [_vp, _vp, _i, _i, _i, _i, _i, _i, _i, _vp]),
    "nm_upsample2x_backward_workspace_bytes": (_sz, [_i, _i, _i, _i, _i]),
    "nm_upsample2x_backward": (_i, [_vp, _vp, _i, _i, _i, _i, _i, _vp, _vp]),
    "nm_final_recon_backward_workspace_bytes": (_sz, [_i]),
    "nm_final_recon_backward": (_i, [_vp, _vp, _vp, _vp, _f, _vp, _vp, _i, _f, _f, _vp, _vp, _vp, _f, _vp, _vp, _vp, _vp, _i, _i,
                                     _i, _vp]),
    "nm_final_recon_backward_fused_workspace_bytes": (_sz, [_i, _ll, _i, _i]),
    "nm_final_recon_backward_fused": (_i, [_vp, _vp, _vp, _vp, _f, _vp, _f, _vp, _vp, _vp, _f, _vp, _vp, _vp, _vp, _i, _vp, _vp,
                                           _vp, _vp, _vp, _vp, _vp, _i, _ll, _i, _vp]),
    "nm_heatmap_head_backward_workspace_bytes": (_sz, [_i, _i, _i]),
    "nm_heatmap_head_backward": (_i, [_vp, _vp, _vp, _i, _i, _i, _i, _i, _vp, _i, _f, _f, _f, _vp, _vp, _vp, _vp, _vp, _vp, _vp,
                                      _vp, _vp, _f, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "nm_decoder_adjust_backward_workspace_bytes": (_sz, [_i, _i]),
    "nm_decoder_adjust_backward": (_i, [_vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _vp, _f, _f, _vp, _vp, _vp, _vp, _vp, _vp]),
    "nm_chamfer_vol_fit_backward_workspace_bytes": (_sz, [_i, _i]),
    "nm_chamfer_vol_fit_backward": (_i, [_vp, _vp, _vp, _vp, _i, _i, _i, _vp, _vp, _vp]),
    "nm_first_conv_wgrad_workspace_bytes": (_sz, [_i, _i]),
    "nm_first_conv_wgrad": (_i, [_vp, _vp, _vp, _i, _i, _i, _f, _vp, _vp, _vp]),
    "nm_grad_nonfinite": (_i, [_vp, _ll, _vp, _vp]),
    "nm_adam_step": (_i, [_vp, _vp, _vp, _vp, _ll, _f, _f, _f, _f, _i, _f, _vp, _vp]),
    "nm_adam_step_dev": (_i, [_vp, _vp, _vp, _vp, _ll, _f, _f, _f, _f, _vp, _f, _vp, _vp]),
}

_lib = None
CALLS = 0   # C-ABI calls that enqueue kernels (bench.py reports the delta over its timed region)


class NmError(RuntimeError):
    pass


def build(verbose: bool = False) -> str:
    """Compile csrc/*.cu for sm_100a into csrc/libnm_b200.so (nvcc cross-compiles without a GPU)."""
    script = os.path.join(_HERE, "csrc", "build.sh")
    out = subprocess.run(["bash", script], capture_output=True, text=True)
    if out.returncode != 0:
        raise NmError("building libnm_b200.so failed:\n" + out.stdout + out.stderr)
    if verbose:
        print(out.stdout.strip())
    return LIB_PATH


def lib() -> C.CDLL:
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise NmError(f"{LIB_PATH} is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                          "(there is no CPU fallback)")
        handle = C.CDLL(LIB_PATH)
        for name, (res, args) in PROTOTYPES.items():
            fn = getattr(handle, name)
            fn.restype = res
            fn.argtypes = args
        _lib = handle
    return _lib


def ptr(t):
    """Device pointer of a tensor (None -> NULL).  The tensor must be contiguous."""
    if t is None:
        return None
    assert t.is_contiguous(), "nm_b200 kernels take dense tensors"
    return t.data_ptr()


def stream():
    return torch.cuda.current_stream().cuda_stream


def call(name: str, *args):
    """Invoke an int-returning entry point and raise on failure."""
    global CALLS
    CALLS += 1
    handle = lib()
    rc = getattr(handle, name)(*args)
    if rc != 0:
        raise NmError(f"{name} failed ({rc}): {handle.nm_last_error().decode()}")


_QUERY_CACHE = {}


def query(name: str, *args):
    """Shape queries (`*_supported`, `*_chunks`, `*_bytes`): pure functions of their integer arguments, memoised - the
    launch-bound hour-glass levels make several of them per layer and per step."""
    key = (name, args)
    hit = _QUERY_CACHE.get(key)
    if hit is None:
        hit = _QUERY_CACHE[key] = getattr(lib(), name)(*args)
    return hit

"""ctypes binding of include/diffuscene_b200.h (the C ABI of the CUDA engine).

This is exactly the stub a reference maintainer would add (INTEGRATION.md): load the shared library,
declare argtypes, pass raw device pointers (`tensor.data_ptr()`) and the CUDA stream handle.
There is no fallback: if the library is missing it is built with nvcc; if that fails, import fails.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Dict, List, Optional, Tuple

from . import build as _build

DS_PREC_FP32, DS_PREC_BF16 = 0, 1
DS_GEMM_AUTO, DS_GEMM_SIMT, DS_GEMM_TCGEN05 = 0, 1, 2
DS_MEAN_EPS, DS_MEAN_X0, DS_MEAN_V = 0, 1, 2
MEAN_TYPES = {"eps": DS_MEAN_EPS, "x0": DS_MEAN_X0, "v": DS_MEAN_V}


class DsConfig(C.Structure):
    _fields_ = [(n, C.c_int32) for n in (
        "dim", "channels", "seperate_all", "objectness_dim", "class_dim", "translation_dim", "size_dim",
        "angle_dim", "objfeat_dim", "cond_dim", "text_condition", "text_dim", "n_stages", "num_objects",
        "num_timesteps", "precision", "gemm_backend", "device", "fuse_level", "train")] + [("reserved", C.c_int32 * 6)]


class DsSchedule(C.Structure):
    _fields_ = [("T", C.c_int32), ("mean_type", C.c_int32)] + [(n, C.POINTER(C.c_float)) for n in (
        "sqrt_ac", "sqrt_1mac", "sqrt_recip_ac", "sqrt_recipm1_ac", "coef1", "coef2", "sigma", "alphas_cumprod",
        "loss_weight")]


class DsSampleArgs(C.Structure):
    _fields_ = [
        ("batch", C.c_int32), ("clip_denoised", C.c_int32), ("num_steps", C.c_int32), ("ddim", C.c_int32),
        ("ddim_eta", C.c_float), ("seed", C.c_uint64), ("scene_offset", C.c_uint64),
        ("x_init_dev", C.c_void_p), ("noise_dev", C.c_void_p), ("partial_dev", C.c_void_p),
        ("num_partial", C.c_int32), ("partial_noise_dev", C.c_void_p), ("traj_freq", C.c_int32),
        ("traj_dev", C.c_void_p), ("use_graph", C.c_int32), ("ddim_times", C.POINTER(C.c_int32)),
        ("chunk_scenes", C.c_int32), ("reserved", C.c_int32 * 5)]


_lib = None


def lib_path() -> str:
    return _build.LIB_PATH


def load(rebuild: bool = False):
    """Load (building first if needed) the shared library and declare its prototypes."""
    global _lib
    if _lib is not None and not rebuild:
        return _lib
    path = _build.build(force=rebuild)
    lib = C.CDLL(path)
    H = C.c_void_p
    p = C.c_void_p
    sig = {
        "ds_create": (C.c_int, [C.POINTER(DsConfig), C.POINTER(H)]),
        "ds_destroy": (C.c_int, [H]),
        "ds_last_error": (C.c_char_p, []),
        "ds_version": (C.c_char_p, []),
        "ds_load_weight": (C.c_int, [H, C.c_char_p, p, C.c_int64]),
        "ds_commit_weights": (C.c_int, [H]),
        "ds_expected_weight_count": (C.c_int, [H]),
        "ds_expected_weight": (C.c_int, [H, C.c_int, C.POINTER(C.c_char_p), C.POINTER(C.c_int64)]),
        "ds_set_schedule": (C.c_int, [H, C.POINTER(DsSchedule)]),
        "ds_set_context": (C.c_int, [H, p, C.c_int32, C.c_int32, p]),
        "ds_set_context_cross": (C.c_int, [H, p, C.c_int32, C.c_int32, p]),
        "ds_denoise_forward": (C.c_int, [H, p, p, p, C.c_int32, p]),
        "ds_denoise_forward_host": (C.c_int, [H, p, p, p, C.c_int32]),
        "ds_sample_loop": (C.c_int, [H, C.POINTER(DsSampleArgs), p, p]),
        "ds_sample_loop_host": (C.c_int, [H, C.POINTER(DsSampleArgs), p]),
        "ds_traj_count": (C.c_int, [C.c_int32, C.c_int32]),
        "ds_p_sample_step": (C.c_int, [H, p, p, p, C.c_int32, p, C.c_int32, p]),
        "ds_q_sample": (C.c_int, [H, p, p, p, p, C.c_int32, p]),
        "ds_p_losses": (C.c_int, [H, p, p, p, C.c_int32, C.c_int32, p, p, p, C.c_int32, p]),
        "ds_train_param_count": (C.c_int64, [H]),
        "ds_train_step": (C.c_int, [H, p, p, p, p, p, C.c_int32, C.c_int32, C.c_int32, C.c_int32, p, C.c_float, p, p, p, p,
                                    C.c_int32, p]),
        "ds_train_set_context_cross": (C.c_int, [H, p, C.c_int32, C.c_int32, p]),
        "ds_train_set_buckets": (C.c_int, [H, p, C.c_int32, p]),
        "ds_train_phase_ms": (C.c_int, [H, p]),
        "ds_sumsq": (C.c_int, [p, C.c_int64, p, p]),
        "ds_adam_step": (C.c_int, [p, p, p, p, C.c_int64, C.c_float, C.c_float, C.c_float, C.c_float, C.c_int32, p,
                                   C.c_float, p]),
        "ds_retrieve_objects": (C.c_int, [p, C.c_int32, p, p, C.c_int32, C.c_int32, p, p, p, C.c_int32, C.c_int32, p, p]),
        "ds_plan_describe": (C.c_int, [C.POINTER(DsConfig), C.c_char_p, C.c_int64]),
        "ds_plan_export_json": (C.c_int, [C.POINTER(DsConfig), C.c_int32, C.c_char_p, C.c_int64]),
        "ds_enable_taps": (C.c_int, [H, C.c_int32]),
        "ds_read_tap": (C.c_int, [H, C.c_char_p, p, C.c_int64, C.POINTER(C.c_int32), C.POINTER(C.c_int32)]),
        "ds_launch_count": (C.c_int64, [H]),
        "ds_graph_build_count": (C.c_int64, [H]),
        "ds_gnt_weight_row": (C.c_int32, [C.c_int32]),
        "ds_profile_ops": (C.c_int, [H, C.c_int32, C.c_char_p, C.c_int64, p, C.c_int32]),
        "ds_test_gemm_trace": (C.c_int, [p, p, p, p, p, C.c_int32, C.c_int32, C.c_int32, C.c_int32, p, p, C.c_int32, p, p]),
        "ds_test_gemm_bf16": (C.c_int, [C.c_int, p, p, p, p, C.c_int32, C.c_int32, C.c_int32, C.c_int32, p]),
    }
    for name, (res, args) in sig.items():
        fn = getattr(lib, name)      # AttributeError here == a symbol of the header is missing
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


EXPORTED = ["ds_create", "ds_destroy", "ds_last_error", "ds_version", "ds_load_weight", "ds_commit_weights",
            "ds_expected_weight_count", "ds_expected_weight", "ds_set_schedule", "ds_set_context",
            "ds_set_context_cross", "ds_denoise_forward", "ds_denoise_forward_host", "ds_sample_loop",
            "ds_sample_loop_host", "ds_traj_count", "ds_p_sample_step", "ds_q_sample", "ds_p_losses", "ds_retrieve_objects",
            "ds_train_param_count", "ds_train_step", "ds_train_set_context_cross", "ds_train_set_buckets", "ds_train_phase_ms", "ds_sumsq", "ds_adam_step",
            "ds_plan_describe", "ds_plan_export_json", "ds_enable_taps", "ds_read_tap", "ds_launch_count", "ds_graph_build_count", "ds_gnt_weight_row", "ds_profile_ops",
            "ds_test_gemm_bf16", "ds_test_gemm_trace"]


class DsError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__("diffuscene_b200 error %d: %s" % (code, msg))
        self.code = code


def check(rc: int):
    if rc < 0:
        raise DsError(rc, load().ds_last_error().decode(errors="replace"))
    return rc


def make_config(spec, num_objects: int, num_timesteps: int, precision: int = DS_PREC_BF16,
                gemm_backend: int = DS_GEMM_AUTO, device: int = 0, fuse_level: int = 0, train: int = 0) -> DsConfig:
    """DsConfig from a diffuscene_b200.weights.NetSpec."""
    c = DsConfig()
    c.dim, c.channels, c.seperate_all = spec.dim, spec.channels, int(spec.seperate_all)
    c.objectness_dim, c.class_dim = spec.objectness_dim, spec.class_dim
    c.translation_dim, c.size_dim, c.angle_dim = spec.translation_dim, spec.size_dim, spec.angle_dim
    c.objfeat_dim, c.cond_dim = spec.objfeat_dim, spec.cond_dim
    c.text_condition, c.text_dim = int(spec.text_condition), spec.text_dim
    c.n_stages, c.num_objects, c.num_timesteps = spec.n_stages, num_objects, num_timesteps
    c.precision, c.gemm_backend, c.device, c.fuse_level = precision, gemm_backend, device, fuse_level
    c.train = int(train)
    return c


def plan_describe(cfg: DsConfig) -> str:
    lib = load()
    buf = C.create_string_buffer(1 << 20)
    check(lib.ds_plan_describe(C.byref(cfg), buf, len(buf)))
    return buf.value.decode()


def plan_export(cfg: DsConfig, no_reuse: bool = False) -> dict:
    import json
    lib = load()
    buf = C.create_string_buffer(1 << 22)
    check(lib.ds_plan_export_json(C.byref(cfg), int(no_reuse), buf, len(buf)))
    return json.loads(buf.value.decode())


def plan_expected_weights(cfg: DsConfig) -> List[Tuple[str, int]]:
    txt = plan_describe(cfg)
    lines = txt.split("weights:\n", 1)[1].strip().split("\n")
    return [(l.rsplit(" ", 1)[0], int(l.rsplit(" ", 1)[1])) for l in lines]

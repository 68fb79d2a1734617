"""ctypes binding of libgnca.so (C ABI declared in include/gnca.h).  There is no CPU fallback: if the
library is missing every operator raises (build it with `python -m graph_neural_cellular_automata_b200.build`
or `__graft_entry__.build()`)."""
from __future__ import annotations

import ctypes as C
import os
from typing import Optional

_PKG = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_PKG, "lib", "libgnca.so")

GNCA_F_GRAPH, GNCA_F_TORUS, GNCA_F_HIDDEN_ONLY, GNCA_F_ALIVE_TO_ALIVE, GNCA_F_GROUPNORM = 1, 2, 4, 8, 16
GNCA_MAX_K = 64
GNCA_ERR_ARG, GNCA_ERR_UNSUPPORTED, GNCA_ERR_WORKSPACE = -1, -2, -3
GNCA_VERSION = 106


class GncaModel(C.Structure):
    _fields_ = [("C", C.c_int32), ("hidden", C.c_int32), ("d_model", C.c_int32), ("flags", C.c_uint32),
                ("update_gain", C.c_float), ("alpha_thr", C.c_float), ("graph_alpha_thr", C.c_float),
                ("gn_eps", C.c_float)]


class GncaLayout(C.Structure):
    _fields_ = [(n, C.c_int64) for n in ("w1", "b1", "w2", "gamma", "beta", "wm", "bm", "wq", "bq", "wk", "bk",
                                          "scaling", "total", "packed_total")]


class GncaSchedule(C.Structure):
    _fields_ = [("T", C.c_int32), ("k", C.c_int32), ("fire_rate", C.c_void_p), ("message_gain", C.c_void_p),
                ("offsets", C.c_void_p), ("steps", C.c_void_p), ("fire_u", C.c_void_p),
                ("philox_seed", C.c_uint64), ("philox_offset", C.c_uint64), ("damage", C.c_void_p),
                ("damage_step", C.c_int32), ("max_offset", C.c_int32), ("damage_layout", C.c_int32),
                ("reserved_", C.c_int32)]


class GncaDamage(C.Structure):
    _fields_ = [("kind", C.c_int32), ("size", C.c_int32), ("softness", C.c_float), ("p", C.c_float),
                ("alpha_thr", C.c_float), ("reserved_", C.c_int32), ("pos", C.c_void_p), ("rand", C.c_void_p)]


EXPORTS = {
    # name: (restype, argtypes)
    "gnca_version": (C.c_int, []),
    "gnca_damage_plane": (C.c_int, [C.POINTER(GncaDamage), C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p,
                                    C.POINTER(C.c_int32), C.c_void_p]),
    "gnca_apply_plane": (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p]),
    "gnca_error_string": (C.c_char_p, [C.c_int]),
    "gnca_launch_count": (C.c_ulonglong, []),
    "gnca_profile_enable": (C.c_int, [C.c_int]),
    "gnca_profile_read": (C.c_int, [C.c_int, C.POINTER(C.c_double), C.POINTER(C.c_ulonglong)]),
    "gnca_param_layout": (C.c_int, [C.POINTER(GncaModel), C.POINTER(GncaLayout)]),
    "gnca_pack_weights": (C.c_int, [C.POINTER(GncaModel), C.c_void_p, C.c_void_p, C.c_void_p]),
    "gnca_perception_fwd": (C.c_int, [C.c_int] * 4 + [C.c_void_p] * 3),
    "gnca_perception_bwd": (C.c_int, [C.c_int] * 4 + [C.c_void_p] * 3),
    "gnca_alive_mask": (C.c_int, [C.c_int] * 4 + [C.c_void_p, C.c_float, C.c_void_p, C.c_void_p]),
    "gnca_step_workspace_bytes": (C.c_size_t, [C.POINTER(GncaModel), C.c_int, C.c_int, C.c_int]),
    "gnca_step_fwd": (C.c_int, [C.POINTER(GncaModel), C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p,
                                C.c_void_p, C.c_float, C.POINTER(C.c_int32), C.c_int, C.c_float,
                                C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "gnca_step_bwd": (C.c_int, [C.POINTER(GncaModel), C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p,
                                C.c_void_p, C.c_float, C.POINTER(C.c_int32), C.c_int, C.c_float,
                                C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                C.c_void_p, C.c_size_t, C.c_void_p]),
    "gnca_graph_fwd": (C.c_int, [C.POINTER(GncaModel), C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p,
                                 C.POINTER(C.c_int32), C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t,
                                 C.c_void_p]),
    "gnca_graph_bwd": (C.c_int, [C.POINTER(GncaModel), C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p,
                                 C.POINTER(C.c_int32), C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                 C.c_size_t, C.c_void_p]),
    "gnca_rollout_workspace_bytes": (C.c_size_t, [C.POINTER(GncaModel), C.c_int, C.c_int, C.c_int, C.c_int]),
    "gnca_rollout_fwd": (C.c_int, [C.POINTER(GncaModel), C.c_void_p, C.c_int, C.c_int, C.c_int,
                                   C.POINTER(GncaSchedule), C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                   C.c_void_p, C.c_size_t, C.c_int, C.c_void_p]),
    "gnca_record_frames": (C.c_int, [C.c_int, C.c_int]),
    "gnca_rollout_record": (C.c_int, [C.POINTER(GncaModel), C.c_void_p, C.c_int, C.c_int, C.c_int,
                                      C.POINTER(GncaSchedule), C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p,
                                      C.c_void_p, C.c_size_t, C.c_int, C.c_void_p]),
    "gnca_metrics_scratch_bytes": (C.c_size_t, [C.POINTER(GncaModel), C.c_int, C.c_int, C.c_int, C.c_int, C.c_int]),
    "gnca_rollout_metrics": (C.c_int, [C.POINTER(GncaModel), C.c_void_p, C.c_int, C.c_int, C.c_int,
                                       C.POINTER(GncaSchedule), C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_float,
                                       C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t, C.c_int,
                                       C.c_void_p]),
    "gnca_rollout_record_models": (C.c_int, [C.POINTER(GncaModel), C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int,
                                             C.POINTER(GncaSchedule), C.c_void_p, C.c_void_p, C.c_int, C.c_void_p,
                                             C.c_void_p, C.c_size_t, C.c_int, C.c_void_p]),
    "gnca_rollout_metrics_models": (C.c_int, [C.POINTER(GncaModel), C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int,
                                              C.POINTER(GncaSchedule), C.c_void_p, C.c_void_p, C.c_int, C.c_void_p,
                                              C.c_float, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p,
                                              C.c_size_t, C.c_int, C.c_void_p]),
    "gnca_ssim_rgb_scratch_bytes": (C.c_size_t, [C.c_int, C.c_int, C.c_int]),
    "gnca_ssim_rgb": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p,
                                C.c_size_t, C.c_void_p]),
    "gnca_metrics_ssim_scratch_bytes": (C.c_size_t, [C.POINTER(GncaModel), C.c_int, C.c_int, C.c_int, C.c_int,
                                                     C.c_int]),
    "gnca_rollout_metrics_ssim": (C.c_int, [C.POINTER(GncaModel), C.c_void_p, C.c_int, C.c_int, C.c_int,
                                            C.POINTER(GncaSchedule), C.c_void_p, C.c_void_p, C.c_int, C.c_void_p,
                                            C.c_float, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t,
                                            C.c_void_p, C.c_size_t, C.c_int, C.c_void_p]),
    "gnca_rollout_metrics_ssim_models": (C.c_int, [C.POINTER(GncaModel), C.c_void_p, C.c_int, C.c_int, C.c_int,
                                                   C.c_int, C.POINTER(GncaSchedule), C.c_void_p, C.c_void_p, C.c_int,
                                                   C.c_void_p, C.c_float, C.c_void_p, C.c_void_p, C.c_void_p,
                                                   C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t, C.c_int,
                                                   C.c_void_p]),
    "gnca_rollout_metrics_targets": (C.c_int, [C.POINTER(GncaModel), C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int,
                                               C.POINTER(GncaSchedule), C.c_void_p, C.c_void_p, C.c_int, C.c_void_p,
                                               C.c_float, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t,
                                               C.c_void_p, C.c_size_t, C.c_int, C.c_void_p]),
    "gnca_rollout_bwd": (C.c_int, [C.POINTER(GncaModel), C.c_void_p, C.c_int, C.c_int, C.c_int,
                                   C.POINTER(GncaSchedule), C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                   C.c_void_p, C.c_void_p, C.c_size_t, C.c_int, C.c_void_p]),
    "gnca_rollout_bwd_frames": (C.c_int, [C.POINTER(GncaModel), C.c_void_p, C.c_int, C.c_int, C.c_int,
                                          C.POINTER(GncaSchedule), C.c_void_p, C.c_void_p, C.c_void_p, C.c_int,
                                          C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t,
                                          C.c_int, C.c_void_p]),
    "gnca_ckpt_segment_bytes": (C.c_size_t, [C.POINTER(GncaModel), C.c_int, C.c_int, C.c_int, C.c_int]),
    "gnca_rollout_bwd_ckpt": (C.c_int, [C.POINTER(GncaModel), C.c_void_p, C.c_int, C.c_int, C.c_int,
                                        C.POINTER(GncaSchedule), C.c_void_p, C.c_int, C.c_void_p, C.c_void_p,
                                        C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t,
                                        C.c_void_p]),
    "gnca_bptt_bytes": (C.c_size_t, [C.POINTER(GncaModel), C.c_int, C.c_int, C.c_int, C.c_int]),
    "gnca_rollout_fwd_bptt": (C.c_int, [C.POINTER(GncaModel), C.c_void_p, C.c_int, C.c_int, C.c_int,
                                        C.POINTER(GncaSchedule), C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                        C.c_size_t, C.c_void_p, C.c_size_t, C.c_void_p]),
    "gnca_rollout_bwd_bptt": (C.c_int, [C.POINTER(GncaModel), C.c_void_p, C.c_int, C.c_int, C.c_int,
                                        C.POINTER(GncaSchedule), C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p,
                                        C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "gnca_rollout_fwd_bptt_record": (C.c_int, [C.POINTER(GncaModel), C.c_void_p, C.c_int, C.c_int, C.c_int,
                                               C.POINTER(GncaSchedule), C.c_void_p, C.c_void_p, C.c_int, C.c_void_p,
                                               C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t, C.c_void_p]),
    "gnca_rollout_bwd_bptt_frames": (C.c_int, [C.POINTER(GncaModel), C.c_void_p, C.c_int, C.c_int, C.c_int,
                                               C.POINTER(GncaSchedule), C.c_void_p, C.c_size_t, C.c_int, C.c_void_p,
                                               C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t,
                                               C.c_void_p]),
    "gnca_bptt_zp_bytes": (C.c_size_t, [C.POINTER(GncaModel), C.c_int, C.c_int, C.c_int, C.c_int]),
    "gnca_rollout_fwd_bptt_zp": (C.c_int, [C.POINTER(GncaModel), C.c_void_p, C.c_int, C.c_int, C.c_int,
                                           C.POINTER(GncaSchedule), C.c_void_p, C.c_void_p, C.c_int, C.c_void_p,
                                           C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t, C.c_void_p]),
    "gnca_rollout_bwd_bptt_zp": (C.c_int, [C.POINTER(GncaModel), C.c_void_p, C.c_int, C.c_int, C.c_int,
                                           C.POINTER(GncaSchedule), C.c_void_p, C.c_size_t, C.c_int, C.c_void_p,
                                           C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t,
                                           C.c_void_p]),
    "gnca_rollout_workspace_models_bytes": (C.c_size_t, [C.POINTER(GncaModel), C.c_int, C.c_int, C.c_int, C.c_int,
                                                         C.c_int]),
    **{name: (C.c_int, [C.POINTER(GncaModel), C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(GncaSchedule),
                        C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t, C.c_void_p])
       for name in ("gnca_rollout_fwd_bptt_models", "gnca_rollout_fwd_bptt_zp_models")},
    **{name: (C.c_int, [C.POINTER(GncaModel), C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(GncaSchedule),
                        C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t,
                        C.c_void_p])
       for name in ("gnca_rollout_bwd_bptt_models", "gnca_rollout_bwd_bptt_zp_models")},
    "gnca_bptt_ckpt_bytes": (C.c_size_t, [C.POINTER(GncaModel), C.c_int, C.c_int, C.c_int, C.c_int]),
    "gnca_rollout_fwd_bptt_ckpt": (C.c_int, [C.POINTER(GncaModel), C.c_void_p, C.c_int, C.c_int, C.c_int,
                                             C.POINTER(GncaSchedule), C.c_void_p, C.c_void_p, C.c_int, C.c_void_p,
                                             C.c_void_p, C.c_size_t, C.c_void_p]),
    "gnca_rollout_bwd_bptt_ckpt": (C.c_int, [C.POINTER(GncaModel), C.c_void_p, C.c_int, C.c_int, C.c_int,
                                             C.POINTER(GncaSchedule), C.c_void_p, C.c_int, C.c_void_p, C.c_void_p,
                                             C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t, C.c_void_p]),
    "gnca_rollout_bwd_bptt_ckpt_frames": (C.c_int, [C.POINTER(GncaModel), C.c_void_p, C.c_int, C.c_int, C.c_int,
                                                    C.POINTER(GncaSchedule), C.c_void_p, C.c_int, C.c_int, C.c_void_p,
                                                    C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t,
                                                    C.c_void_p, C.c_size_t, C.c_void_p]),
    "gnca_host_sample_indices": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p]),
    "gnca_host_sample_offsets_words": (C.c_int, [C.c_char_p, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_int,
                                                 C.c_void_p, C.POINTER(C.c_int32)]),
    "gnca_loss_premult_rgba": (C.c_int, [C.c_int] * 4 + [C.c_void_p] * 4 + [C.c_float, C.c_void_p]),
    "gnca_loss_premult_rgba_targets": (C.c_int, [C.c_int] * 4 + [C.c_void_p] * 2 + [C.c_int] + [C.c_void_p] * 2
                                       + [C.c_float, C.c_void_p]),
    "gnca_normalize_adam": (C.c_int, [C.c_void_p] * 4 + [C.POINTER(C.c_int64), C.POINTER(C.c_int32), C.c_int, C.c_int,
                                      C.c_float, C.c_float, C.c_float, C.c_float, C.c_float, C.c_int64, C.c_void_p]),
    "gnca_apply_mask": (C.c_int, [C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p]),
}

_lib: Optional[C.CDLL] = None


class GncaError(RuntimeError):
    pass


def load() -> C.CDLL:
    """Load libgnca.so and bind every symbol include/gnca.h declares.  Raises (never falls back)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise GncaError(f"{LIB_PATH} is missing: build it with `python -m graph_neural_cellular_automata_b200.build` "
                        "(needs nvcc). There is no CPU/PyTorch fallback for the graph-NCA step.")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in EXPORTS.items():
        fn = getattr(lib, name)          # AttributeError if the .so does not export a declared symbol
        fn.restype, fn.argtypes = res, args
    if lib.gnca_version() != GNCA_VERSION:
        raise GncaError(f"libgnca.so version {lib.gnca_version()} != binding version {GNCA_VERSION}; rebuild")
    _lib = lib
    return lib


def check(code: int, what: str) -> None:
    if code != 0:
        msg = load().gnca_error_string(code).decode()
        raise GncaError(f"{what} failed: {msg} (code {code})")

"""CPU checks of the checkpointed-BPTT C ABI (gnca_ckpt_segment_bytes, gnca_rollout_bwd_ckpt): the symbols, the segment
size formula, and argument errors that return their code before any kernel is launched."""
import ctypes as C
import os
import re

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def lib():
    from graph_neural_cellular_automata_b200 import _lib, build
    build.build(verbose=False)
    return _lib.load()


def _desc(C_=16):
    from graph_neural_cellular_automata_b200 import functional as GF
    return GF.make_model_desc(C_, 128, 16, graph=True, torus=True, hidden_only=True, alive_to_alive=True,
                              groupnorm=True, update_gain=0.05, alpha_thr=0.12, graph_alpha_thr=0.12)


def test_symbols_are_exported_and_bound(lib):
    from graph_neural_cellular_automata_b200 import _lib
    header = open(os.path.join(ROOT, "include", "gnca.h")).read()
    assert re.search(r"\bsize_t gnca_ckpt_segment_bytes\(", header)
    assert re.search(r"\bint gnca_rollout_bwd_ckpt\(", header)
    for name in ("gnca_ckpt_segment_bytes", "gnca_rollout_bwd_ckpt"):
        assert name in _lib.EXPORTS
        assert getattr(lib, name).argtypes == _lib.EXPORTS[name][1]


def _al(v):
    return (v + 255) // 256 * 256


@pytest.mark.parametrize("C_,B,H,W,every", [(16, 4, 40, 40, 1), (16, 4, 40, 40, 5), (32, 16, 256, 256, 32),
                                            (4, 3, 7, 9, 3), (8, 1, 1, 1, 2)])
def test_segment_bytes_formula(lib, C_, B, H, W, every):
    n = B * C_ * H * W * 4
    want = _al((every - 1) * n) + _al(every * n) + _al(every * B * 2 * 4)
    assert lib.gnca_ckpt_segment_bytes(C.byref(_desc(C_)), B, H, W, every) == want


@pytest.mark.parametrize("B,H,W,every", [(0, 40, 40, 4), (2, 0, 40, 4), (2, 40, -1, 4), (2, 40, 40, 0),
                                         (2, 40, 40, -2)])
def test_segment_bytes_zero_on_bad_arguments(lib, B, H, W, every):
    assert lib.gnca_ckpt_segment_bytes(C.byref(_desc()), B, H, W, every) == 0
    assert lib.gnca_ckpt_segment_bytes(None, 2, 40, 40, 4) == 0


P = C.c_void_p(256)        # never dereferenced: every call below fails its argument checks first
BIG = 1 << 40


def _call(lib, sched, *, every=2, ckpt=P, gT=P, g0=P, gparams=P, packed=P, segment=P, seg_bytes=BIG, ws=P,
          ws_bytes=BIG):
    return lib.gnca_rollout_bwd_ckpt(C.byref(_desc()), packed, 2, 40, 40, C.byref(sched), ckpt, every, None, gT, g0,
                                     gparams, segment, seg_bytes, ws, ws_bytes, None)


CASES = {
    "every0": ("ARG", dict(every=0)),
    "every_neg": ("ARG", dict(every=-3)),
    "null_ckpt": ("ARG", dict(ckpt=None)),
    "null_gT": ("ARG", dict(gT=None)),
    "null_g0": ("ARG", dict(g0=None)),
    "null_gparams": ("ARG", dict(gparams=None)),
    "null_packed": ("ARG", dict(packed=None)),
    "null_segment": ("ARG", dict(segment=None)),
    "null_workspace": ("ARG", dict(ws=None)),
    "T_neg": ("ARG", {}),
    "segment_small": ("WORKSPACE", dict(seg_bytes=1024)),
    "workspace_small": ("WORKSPACE", dict(ws_bytes=1024)),
    "k65": ("UNSUPPORTED", {}),
    "k_neg": ("UNSUPPORTED", {}),
}


@pytest.mark.parametrize("case", list(CASES))
def test_argument_errors_do_not_launch(lib, case):
    from graph_neural_cellular_automata_b200 import _lib
    code, kw = CASES[case]
    p = C.c_void_p(512)
    sched = _lib.GncaSchedule(4, 8, p, p, p, None, None, 0, 0, None, 0, 4, 0, 0)
    if case == "k65":
        sched.k = _lib.GNCA_MAX_K + 1
    elif case == "k_neg":
        sched.k = -1
    elif case == "T_neg":
        sched.T = -1
    before = lib.gnca_launch_count()
    assert _call(lib, sched, **kw) == getattr(_lib, f"GNCA_ERR_{code}")
    assert lib.gnca_launch_count() == before


def test_segment_one_byte_short_is_rejected(lib):
    from graph_neural_cellular_automata_b200 import _lib
    p = C.c_void_p(512)
    sched = _lib.GncaSchedule(4, 8, p, p, p, None, None, 0, 0, None, 0, 4, 0, 0)
    need = lib.gnca_ckpt_segment_bytes(C.byref(_desc()), 2, 40, 40, 3)
    before = lib.gnca_launch_count()
    assert _call(lib, sched, every=3, seg_bytes=need - 1) == _lib.GNCA_ERR_WORKSPACE
    assert lib.gnca_launch_count() == before

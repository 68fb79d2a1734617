"""CPU checks of the differentiable-frames C ABI (gnca_rollout_fwd_bptt_record, gnca_rollout_bwd_frames,
gnca_rollout_bwd_bptt_frames): the symbols, the version, and argument errors that return their code before any kernel
is launched."""
import ctypes as C
import os
import re

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NEW = ("gnca_rollout_fwd_bptt_record", "gnca_rollout_bwd_frames", "gnca_rollout_bwd_bptt_frames")


@pytest.fixture(scope="module")
def lib():
    from graph_neural_cellular_automata_b200 import _lib, build
    build.build(verbose=False)
    return _lib.load()


def _desc():
    from graph_neural_cellular_automata_b200 import functional as GF
    return GF.make_model_desc(16, 128, 16, graph=True, torus=True, hidden_only=True, alive_to_alive=True,
                              groupnorm=True, update_gain=0.05, alpha_thr=0.12, graph_alpha_thr=0.12)


def test_new_symbols_are_exported_and_bound(lib):
    from graph_neural_cellular_automata_b200 import _lib
    header = open(os.path.join(ROOT, "include", "gnca.h")).read()
    for name in NEW:
        assert name in _lib.EXPORTS
        assert re.search(r"\bint " + name + r"\(", header), name
        assert getattr(lib, name).argtypes == _lib.EXPORTS[name][1]


def test_version_is_106_in_header_binding_and_library(lib):
    from graph_neural_cellular_automata_b200 import _lib
    header = open(os.path.join(ROOT, "include", "gnca.h")).read()
    assert re.search(r"#define GNCA_VERSION (\d+)", header).group(1) == "106"
    assert _lib.GNCA_VERSION == 106
    assert lib.gnca_version() == 106


P = C.c_void_p(256)        # never dereferenced: every call below fails its argument checks first


def _call(lib, fn, desc, sched, *, every=2, frames=P, gT=P, bptt=P):
    if fn == "gnca_rollout_fwd_bptt_record":
        return lib.gnca_rollout_fwd_bptt_record(C.byref(desc), P, 2, 40, 40, C.byref(sched), P, P, every, frames, bptt,
                                                1 << 30, P, 1 << 30, None)
    if fn == "gnca_rollout_bwd_frames":
        return lib.gnca_rollout_bwd_frames(C.byref(desc), P, 2, 40, 40, C.byref(sched), P, None, None, every, frames,
                                           gT, P, P, P, 1 << 30, 0, None)
    return lib.gnca_rollout_bwd_bptt_frames(C.byref(desc), P, 2, 40, 40, C.byref(sched), bptt, 1 << 30, every, frames,
                                            gT, P, P, P, 1 << 30, None)


# case: (error code, arguments); which entry points the case applies to
CASES = {
    "every0": ("ARG", dict(every=0), NEW),
    "every_neg": ("ARG", dict(every=-3), NEW),
    "null_frames": ("ARG", dict(frames=None), NEW[:1]),   # a NULL frame gradient is the plain backward, not an error
    "null_gT": ("ARG", dict(gT=None), NEW[1:]),
    "null_bptt": ("ARG", dict(bptt=None), (NEW[0], NEW[2])),
    "k65": ("UNSUPPORTED", {}, NEW),
    "k_neg": ("UNSUPPORTED", {}, NEW),
    "T_neg": ("ARG", {}, NEW),
}


@pytest.mark.parametrize("fn,case", [(fn, case) for case, (_, _, fns) in CASES.items() for fn in fns])
def test_argument_errors_do_not_launch(lib, fn, case):
    from graph_neural_cellular_automata_b200 import _lib
    code, kw, _ = CASES[case]
    p = C.c_void_p(512)
    sched = _lib.GncaSchedule(4, 8, p, p, p, None, None, 0, 0, None, 0, 4, 0, 0)
    if case == "k65":
        sched.k = _lib.GNCA_MAX_K + 1
    elif case == "k_neg":
        sched.k = -1
    elif case == "T_neg":
        sched.T = -1
    before = lib.gnca_launch_count()
    assert _call(lib, fn, _desc(), sched, **kw) == getattr(_lib, f"GNCA_ERR_{code}")
    assert lib.gnca_launch_count() == before

"""CPU checks of frame gradients on the checkpointed resident BPTT: the C ABI of gnca_rollout_bwd_bptt_ckpt_frames
(symbol, argument errors that return before any launch) and the host-side plan of
record_rollout(..., differentiable=True, bptt_budget=...) (bptt_plan(..., every=S))."""
import ctypes as C
import os
import re

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NAME = "gnca_rollout_bwd_bptt_ckpt_frames"


@pytest.fixture(scope="module")
def lib():
    from graph_neural_cellular_automata_b200 import _lib, build
    build.build(verbose=False)
    return _lib.load()


def _desc(C_=16, torus=True, graph=True):
    from graph_neural_cellular_automata_b200 import functional as GF
    return GF.make_model_desc(C_, 128, 16, graph=graph, torus=torus, hidden_only=True, alive_to_alive=True,
                              groupnorm=True, update_gain=0.05, alpha_thr=0.12, graph_alpha_thr=0.12)


def test_symbol_is_exported_and_bound(lib):
    from graph_neural_cellular_automata_b200 import _lib
    header = open(os.path.join(ROOT, "include", "gnca.h")).read()
    assert re.search(rf"\bint {NAME}\(", header)
    assert getattr(lib, NAME).argtypes == _lib.EXPORTS[NAME][1]
    assert lib.gnca_version() == 106


P = C.c_void_p(256)        # never dereferenced: every call below fails its argument checks first
BIG = 1 << 40


def _sched(case):
    from graph_neural_cellular_automata_b200 import _lib
    p = C.c_void_p(512)
    s = _lib.GncaSchedule(8, 8, p, p, p, None, None, 0, 0, None, 0, 4, 0, 0)
    if case == "k65":
        s.k = _lib.GNCA_MAX_K + 1
    elif case == "T_neg":
        s.T = -1
    elif case == "null_fire_rate":
        s.fire_rate = None
    elif case == "null_gain":
        s.message_gain = None
    elif case == "null_offsets":
        s.offsets = None
    return s


def _bwd(lib, sched, *, every=2, ckpt_every=4, frames=P, g_frames=P, gT=P, g0=P, gparams=P, packed=P, segment=P,
         seg_bytes=BIG, ws=P, ws_bytes=BIG, model="torus"):
    d = {"torus": _desc(), "zeropad": _desc(torus=False), None: None}[model]
    return lib.gnca_rollout_bwd_bptt_ckpt_frames(C.byref(d) if d is not None else None, packed, 2, 40, 40,
                                                 C.byref(sched), frames, every, ckpt_every, g_frames, gT, g0, gparams,
                                                 segment, seg_bytes, ws, ws_bytes, None)


CASES = {
    "null_model": ("ARG", dict(model=None)),
    "null_packed": ("ARG", dict(packed=None)),
    "null_frames": ("ARG", dict(frames=None)),
    "null_gT": ("ARG", dict(gT=None)),
    "null_g0": ("ARG", dict(g0=None)),
    "null_gparams": ("ARG", dict(gparams=None)),
    "null_segment": ("ARG", dict(segment=None)),
    "null_workspace": ("ARG", dict(ws=None)),
    "null_fire_rate": ("ARG", {}),
    "null_gain": ("ARG", {}),
    "null_offsets": ("ARG", {}),
    "T_neg": ("ARG", {}),
    "every0": ("ARG", dict(every=0)),
    "every_neg": ("ARG", dict(every=-2)),
    "ckpt_every0": ("ARG", dict(ckpt_every=0)),
    "ckpt_every_neg": ("ARG", dict(ckpt_every=-4)),
    "ckpt_every_not_multiple": ("ARG", dict(every=2, ckpt_every=3)),
    "ckpt_every_below_every": ("ARG", dict(every=4, ckpt_every=2)),
    "segment_small": ("WORKSPACE", dict(seg_bytes=1024)),
    "workspace_small": ("WORKSPACE", dict(ws_bytes=1024)),
    "k65": ("UNSUPPORTED", {}),
    "zeropad_model": ("UNSUPPORTED", dict(model="zeropad")),
}


@pytest.mark.parametrize("case", list(CASES))
def test_argument_errors_do_not_launch(lib, case):
    from graph_neural_cellular_automata_b200 import _lib
    code, kw = CASES[case]
    before = lib.gnca_launch_count()
    assert _bwd(lib, _sched(case), **kw) == getattr(_lib, f"GNCA_ERR_{code}")
    assert lib.gnca_launch_count() == before


def test_segment_is_sized_for_ckpt_every(lib):
    """the segment holds the records of ckpt_every steps, not of every: one byte short of that is rejected"""
    from graph_neural_cellular_automata_b200 import _lib
    d = _desc()
    need = lib.gnca_bptt_ckpt_bytes(C.byref(d), 2, 40, 40, 6)
    assert need > lib.gnca_bptt_ckpt_bytes(C.byref(d), 2, 40, 40, 2)
    before = lib.gnca_launch_count()
    assert _bwd(lib, _sched(""), every=2, ckpt_every=6, seg_bytes=need - 1) == _lib.GNCA_ERR_WORKSPACE
    assert lib.gnca_launch_count() == before


# ---- bptt_plan(..., every=S) ------------------------------------------------------------------------------------------
def _plan(d, B, H, W, T, budget, every, impl="auto", k=0):
    from graph_neural_cellular_automata_b200.rollout import IMPL, _bptt_plan
    return _bptt_plan(d, B, H, W, T, budget, IMPL[impl], k, every=every)


def _res(lib, d, B, H, W, K):
    return lib.gnca_bptt_ckpt_bytes(C.byref(d), B, H, W, K)


def _stream(lib, d, B, H, W, K):
    return lib.gnca_ckpt_segment_bytes(C.byref(d), B, H, W, K)


def test_plan_keeps_records_when_they_fit(lib):
    from graph_neural_cellular_automata_b200.rollout import _record_bytes
    d = _desc()
    nrec = _record_bytes(lib, d, 32, 40, 40, 64)
    assert _plan(d, 32, 40, 40, 64, nrec, 8) == ("records", None, nrec)
    assert _plan(d, 32, 40, 40, 64, nrec - 1, 8)[0] == "resident_ckpt"


@pytest.mark.parametrize("T,S,budget", [(64, 8, 1 << 30), (300, 20, 2 << 30), (1000, 10, 3 << 30),
                                        (1000, 50, 4 << 30), (13, 4, 300 << 20), (100, 7, 600 << 20),
                                        (12, 5, 600 << 20)])
def test_plan_takes_the_largest_resident_multiple_of_every(lib, T, S, budget):
    d = _desc()
    path, K, nb = _plan(d, 32, 40, 40, T, budget, S)
    assert path == "resident_ckpt" and K % S == 0 and S <= K <= -(-T // S) * S, (path, K)
    assert nb == _res(lib, d, 32, 40, 40, K) <= budget
    assert all(_res(lib, d, 32, 40, 40, k) > budget for k in range(K + S, -(-T // S) * S + 1, S))


def test_plan_1000_steps_frames_every_50(lib):
    """B = 32, 40x40: the records of T = 1000 (72.9 GB) exceed BPTT_MAX_BYTES, and one resident segment of 50 steps takes
    3.40 GiB.  4 GiB holds it; 3 GiB does not, so there the frames are the checkpoints of the streaming kernels."""
    d = _desc()
    assert _plan(d, 32, 40, 40, 1000, 4 << 30, 50) == ("resident_ckpt", 50, _res(lib, d, 32, 40, 40, 50))
    assert 3 << 30 < _res(lib, d, 32, 40, 40, 50) <= 4 << 30
    assert _plan(d, 32, 40, 40, 1000, 3 << 30, 50) == ("streaming_ckpt", 50, _stream(lib, d, 32, 40, 40, 50))


def test_plan_one_segment_when_it_fits(lib):
    """K never exceeds the first multiple of S that covers T: a larger K would only grow the segment buffer"""
    from graph_neural_cellular_automata_b200.rollout import _record_bytes
    d = _desc()
    T, S = 22, 4                 # the record buffer is sized for 64 steps: one 24-step segment is smaller
    budget = _record_bytes(lib, d, 4, 40, 40, T) - 1
    assert _res(lib, d, 4, 40, 40, 24) <= budget
    assert _plan(d, 4, 40, 40, T, budget, S) == ("resident_ckpt", 24, _res(lib, d, 4, 40, 40, 24))


@pytest.mark.parametrize("case", ["zeropad", "large_grid", "impl_streaming", "k17"])
def test_plan_streaming_branch(lib, case):
    from graph_neural_cellular_automata_b200.rollout import RESIDENT_MAX_K
    d, B, H, W, T, S, impl, k = _desc(), 4, 40, 40, 12, 3, "auto", 0
    if case == "zeropad":
        d = _desc(torus=False)
    elif case == "large_grid":
        d, B, H, W = _desc(32), 2, 256, 256
    elif case == "impl_streaming":
        impl = "streaming"
    else:
        k = RESIDENT_MAX_K + 1
    dense = _plan(d, B, H, W, T, 1 << 50, S, impl, k)
    assert dense[0] == "dense"
    seg = _stream(lib, d, B, H, W, S)
    assert seg < dense[2]
    assert _plan(d, B, H, W, T, dense[2] - 1, S, impl, k) == ("streaming_ckpt", S, seg)
    assert _plan(d, B, H, W, T, seg, S, impl, k) == ("streaming_ckpt", S, seg)


def test_plan_resident_before_streaming(lib):
    d = _desc()
    T, S = 40, 5
    budget = _res(lib, d, 8, 40, 40, S)
    assert _stream(lib, d, 8, 40, 40, S) < budget           # streaming would fit too; resident comes first
    assert _plan(d, 8, 40, 40, T, budget, S) == ("resident_ckpt", S, budget)
    assert _plan(d, 8, 40, 40, T, budget - 1, S)[0] == "streaming_ckpt"


def test_plan_names_the_smallest_budget(lib):
    d = _desc()
    B, T, S = 8, 50, 5
    smallest = min(_res(lib, d, B, 40, 40, S), _stream(lib, d, B, 40, 40, S))
    msg = (f"record_rollout: bptt_budget={smallest - 1} bytes is too small for this recording (B={B}, 40x40, T={T}, "
           f"every={S}); the smallest budget that works is {smallest} bytes")
    with pytest.raises(ValueError, match=f"^{re.escape(msg)}$"):
        _plan(d, B, 40, 40, T, smallest - 1, S)
    assert _plan(d, B, 40, 40, T, smallest, S)[2] == smallest


def test_plan_impl_resident(lib):
    d = _desc()
    assert _plan(d, 8, 40, 40, 100, 1 << 40, 10, "resident")[0] == "records"
    path, K, _ = _plan(d, 8, 40, 40, 100, 400 << 20, 10, "resident")
    assert path == "resident_ckpt" and K % 10 == 0
    with pytest.raises(ValueError, match="record_rollout: impl='resident'"):
        _plan(_desc(torus=False), 8, 40, 40, 100, 1 << 40, 10, "resident")
    # T = 0: no record buffer, so impl='resident' takes one checkpoint segment
    assert _plan(d, 4, 40, 40, 0, 1 << 40, 3, "resident") == ("resident_ckpt", 3, _res(lib, d, 4, 40, 40, 3))


@pytest.mark.parametrize("T,budget", [(64, 1 << 30), (1000, 3 << 30), (13, 400 << 20), (12, 1 << 40), (50, 8 << 30)])
def test_plan_without_every_is_unchanged(lib, T, budget):
    """no `every`: the rollout() plan, checkpoints every K steps on top of the segment"""
    from graph_neural_cellular_automata_b200.rollout import bptt_plan

    class _M:
        def model_desc(self):
            return _desc()
    d = _desc()
    plan = _plan(d, 32, 40, 40, T, budget, None)
    assert bptt_plan(_M(), 32, 40, 40, T, budget, k=0) == plan
    if plan[0] == "resident_ckpt":
        K = plan[1]
        assert plan[2] == (T // K + 1) * 32 * 16 * 40 * 40 * 4 + _res(lib, d, 32, 40, 40, K)


def test_public_bptt_plan_every():
    from graph_neural_cellular_automata_b200.rollout import bptt_plan

    class _M:
        def model_desc(self):
            return _desc()
    path, K, _ = bptt_plan(_M(), 32, 40, 40, 1000, 4 << 30, every=50)
    assert path == "resident_ckpt" and K % 50 == 0
    with pytest.raises(ValueError, match="every"):
        bptt_plan(_M(), 32, 40, 40, 1000, 3 << 30, every=0)
    with pytest.raises(TypeError):
        bptt_plan(_M(), 32, 40, 40, 1000, 3 << 30, "auto", 0, 50)         # keyword only

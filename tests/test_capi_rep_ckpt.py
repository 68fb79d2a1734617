"""CPU checks of the checkpointed resident BPTT: the C ABI (gnca_bptt_ckpt_bytes, gnca_rollout_fwd_bptt_ckpt,
gnca_rollout_bwd_bptt_ckpt) -- symbols, the segment size, argument errors that return before any launch -- and the
host-side path choice of rollout(..., bptt_budget=...) (bptt_plan)."""
import ctypes as C
import os
import re

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NAMES = ("gnca_bptt_ckpt_bytes", "gnca_rollout_fwd_bptt_ckpt", "gnca_rollout_bwd_bptt_ckpt")


@pytest.fixture(scope="module")
def lib():
    from graph_neural_cellular_automata_b200 import _lib, build
    build.build(verbose=False)
    return _lib.load()


def _desc(C_=16, torus=True, graph=True, hidden=128):
    from graph_neural_cellular_automata_b200 import functional as GF
    return GF.make_model_desc(C_, hidden, 16, graph=graph, torus=torus, hidden_only=True, alive_to_alive=True,
                              groupnorm=True, update_gain=0.05, alpha_thr=0.12, graph_alpha_thr=0.12)


def test_symbols_are_exported_and_bound(lib):
    from graph_neural_cellular_automata_b200 import _lib
    header = open(os.path.join(ROOT, "include", "gnca.h")).read()
    for name in NAMES:
        assert re.search(rf"\b(size_t|int) {name}\(", header), name
        assert name in _lib.EXPORTS
        assert getattr(lib, name).argtypes == _lib.EXPORTS[name][1]


def _al(v):
    return (v + 255) // 256 * 256


@pytest.mark.parametrize("B,H,W,every", [(32, 40, 40, 1), (32, 40, 40, 8), (4, 40, 40, 13), (1, 8, 4, 3),
                                         (7, 32, 64, 64)])
def test_segment_bytes_are_records_of_every_steps_plus_two_states(lib, B, H, W, every):
    d = _desc()
    n = B * 16 * H * W * 4
    want = _al(lib.gnca_bptt_bytes(C.byref(d), B, H, W, every)) + _al(n) + _al(n)
    assert lib.gnca_bptt_ckpt_bytes(C.byref(d), B, H, W, every) == want
    # the records of `every` steps: per step and cell one 100-float record and one 256-float h | gh row
    assert lib.gnca_bptt_bytes(C.byref(d), B, H, W, every) >= every * B * H * W * (100 + 256) * 4


@pytest.mark.parametrize("case", ["zeropad", "C32", "hidden64", "too_large", "W_not_4", "bad_B", "bad_every",
                                  "every_neg", "null_model"])
def test_segment_bytes_zero_where_not_supported(lib, case):
    d, B, H, W, every = _desc(), 4, 40, 40, 4
    if case == "zeropad":
        d = _desc(torus=False)
    elif case == "C32":
        d = _desc(32)
    elif case == "hidden64":
        d = _desc(hidden=64)
    elif case == "too_large":
        H = W = 64
    elif case == "W_not_4":
        W = 42
    elif case == "bad_B":
        B = 0
    elif case == "bad_every":
        every = 0
    elif case == "every_neg":
        every = -1
    assert lib.gnca_bptt_ckpt_bytes(None if case == "null_model" else C.byref(d), B, H, W, every) == 0


def test_classic_model_is_eligible(lib):
    assert lib.gnca_bptt_ckpt_bytes(C.byref(_desc(graph=False, torus=False)), 4, 40, 40, 4) > 0


P = C.c_void_p(256)        # never dereferenced: every call below fails its argument checks first
BIG = 1 << 40


def _sched(case):
    from graph_neural_cellular_automata_b200 import _lib
    p = C.c_void_p(512)
    s = _lib.GncaSchedule(4, 8, p, p, p, None, None, 0, 0, None, 0, 4, 0, 0)
    if case == "k65":
        s.k = _lib.GNCA_MAX_K + 1
    elif case == "k_neg":
        s.k = -1
    elif case == "T_neg":
        s.T = -1
    elif case == "null_fire_rate":
        s.fire_rate = None
    elif case == "null_offsets":
        s.offsets = None
    return s


def _bwd(lib, sched, *, every=2, ckpt=P, gT=P, g0=P, gparams=P, packed=P, segment=P, seg_bytes=BIG, ws=P,
         ws_bytes=BIG, model=True, **_):
    return lib.gnca_rollout_bwd_bptt_ckpt(C.byref(_desc()) if model else None, packed, 2, 40, 40, C.byref(sched), ckpt,
                                          every, gT, g0, gparams, segment, seg_bytes, ws, ws_bytes, None)


def _fwd(lib, sched, *, every=2, ckpt=P, x0=P, xT=P, packed=P, ws=P, ws_bytes=BIG, model=True, **_):
    return lib.gnca_rollout_fwd_bptt_ckpt(C.byref(_desc()) if model else None, packed, 2, 40, 40, C.byref(sched), x0,
                                          xT, every, ckpt, ws, ws_bytes, None)


CASES = {
    "every0": ("ARG", dict(every=0)),
    "every_neg": ("ARG", dict(every=-3)),
    "null_model": ("ARG", dict(model=False)),
    "null_ckpt": ("ARG", dict(ckpt=None)),
    "null_packed": ("ARG", dict(packed=None)),
    "null_workspace": ("ARG", dict(ws=None)),
    "null_fire_rate": ("ARG", {}),
    "null_offsets": ("ARG", {}),
    "T_neg": ("ARG", {}),
    "workspace_small": ("WORKSPACE", dict(ws_bytes=1024)),
    "k65": ("UNSUPPORTED", {}),
    "k_neg": ("UNSUPPORTED", {}),
}
BWD_ONLY = {
    "null_gT": ("ARG", dict(gT=None)),
    "null_g0": ("ARG", dict(g0=None)),
    "null_gparams": ("ARG", dict(gparams=None)),
    "null_segment": ("ARG", dict(segment=None)),
    "segment_small": ("WORKSPACE", dict(seg_bytes=1024)),
}
FWD_ONLY = {
    "null_x0": ("ARG", dict(x0=None)),
    "null_xT": ("ARG", dict(xT=None)),
}


@pytest.mark.parametrize("case", list(CASES) + list(BWD_ONLY))
def test_backward_argument_errors_do_not_launch(lib, case):
    from graph_neural_cellular_automata_b200 import _lib
    code, kw = {**CASES, **BWD_ONLY}[case]
    before = lib.gnca_launch_count()
    assert _bwd(lib, _sched(case), **kw) == getattr(_lib, f"GNCA_ERR_{code}")
    assert lib.gnca_launch_count() == before


@pytest.mark.parametrize("case", list(CASES) + list(FWD_ONLY))
def test_forward_argument_errors_do_not_launch(lib, case):
    from graph_neural_cellular_automata_b200 import _lib
    code, kw = {**CASES, **FWD_ONLY}[case]
    before = lib.gnca_launch_count()
    assert _fwd(lib, _sched(case), **kw) == getattr(_lib, f"GNCA_ERR_{code}")
    assert lib.gnca_launch_count() == before


def test_segment_one_byte_short_is_rejected(lib):
    from graph_neural_cellular_automata_b200 import _lib
    need = lib.gnca_bptt_ckpt_bytes(C.byref(_desc()), 2, 40, 40, 3)
    before = lib.gnca_launch_count()
    assert _bwd(lib, _sched(""), every=3, seg_bytes=need - 1) == _lib.GNCA_ERR_WORKSPACE
    assert lib.gnca_launch_count() == before


# ---- bptt_plan ---------------------------------------------------------------------------------------------------------
def _plan(lib, d, B, H, W, T, budget, impl="auto"):
    from graph_neural_cellular_automata_b200.rollout import IMPL, _bptt_plan
    return _bptt_plan(d, B, H, W, T, budget, IMPL[impl])


def _ckpt_total(lib, d, B, H, W, T, K, resident):
    f = lib.gnca_bptt_ckpt_bytes if resident else lib.gnca_ckpt_segment_bytes
    return (T // K + 1) * B * d.C * H * W * 4 + f(C.byref(d), B, H, W, K)


def test_plan_keeps_records_when_they_fit(lib):
    from graph_neural_cellular_automata_b200.rollout import _record_bytes
    d = _desc()
    nrec = _record_bytes(lib, d, 32, 40, 40, 64)
    assert nrec >= lib.gnca_bptt_bytes(C.byref(d), 32, 40, 40, 64)
    assert _plan(lib, d, 32, 40, 40, 64, nrec) == ("records", None, nrec)
    assert _plan(lib, d, 32, 40, 40, 64, nrec - 1)[0] == "resident_ckpt"


@pytest.mark.parametrize("T,budget", [(64, 1 << 30), (400, 4 << 30), (448, 2 << 30), (1000, 3 << 30), (1000, 1200 << 20),
                                      (13, 400 << 20)])
def test_plan_takes_the_largest_resident_stride_that_fits(lib, T, budget):
    d = _desc()
    path, K, nb = _plan(lib, d, 32, 40, 40, T, budget)
    assert path == "resident_ckpt" and 1 <= K <= T
    assert nb == _ckpt_total(lib, d, 32, 40, 40, T, K, True) <= budget
    assert all(_ckpt_total(lib, d, 32, 40, 40, T, k, True) > budget for k in range(K + 1, T + 1))


def test_plan_1000_steps_beyond_the_record_limit(lib):
    from graph_neural_cellular_automata_b200.rollout import BPTT_MAX_BYTES
    d = _desc()
    assert lib.gnca_bptt_bytes(C.byref(d), 32, 40, 40, 1000) > BPTT_MAX_BYTES
    # without records the budget-free path is the dense history (6.6 GB): it fits 8 GB ...
    dense = _plan(lib, d, 32, 40, 40, 1000, 8 << 30)
    assert dense[0] == "dense" and 6.5e9 < dense[2] < 6.8e9
    # ... and below it the resident checkpoints take over
    assert _plan(lib, d, 32, 40, 40, 1000, 4 << 30)[0] == "resident_ckpt"


@pytest.mark.parametrize("case", ["zeropad", "large_grid", "impl_streaming"])
def test_plan_streaming_branch(lib, case):
    d, B, H, W, T, impl = _desc(), 4, 40, 40, 12, "auto"
    if case == "zeropad":
        d = _desc(torus=False)
    elif case == "large_grid":
        d, B, H, W = _desc(32), 2, 256, 256
    else:
        impl = "streaming"
    dense = _plan(lib, d, B, H, W, T, 1 << 50, impl)
    assert dense[0] == "dense"
    budget = dense[2] // 2
    path, K, nb = _plan(lib, d, B, H, W, T, budget, impl)
    assert path == "streaming_ckpt" and K < T
    assert nb == _ckpt_total(lib, d, B, H, W, T, K, False) <= budget
    assert all(_ckpt_total(lib, d, B, H, W, T, k, False) > budget for k in range(K + 1, T + 1))


def test_plan_impl_resident(lib):
    d = _desc()
    assert _plan(lib, d, 8, 40, 40, 100, 1 << 40, "resident")[0] == "records"
    assert _plan(lib, d, 8, 40, 40, 100, 100 << 20, "resident")[0] == "resident_ckpt"
    with pytest.raises(ValueError, match="resident"):
        _plan(lib, _desc(torus=False), 8, 40, 40, 100, 1 << 40, "resident")


def test_plan_names_the_smallest_budget(lib):
    d = _desc()
    T = 50
    smallest = min(min(_ckpt_total(lib, d, 8, 40, 40, T, k, True), _ckpt_total(lib, d, 8, 40, 40, T, k, False))
                   for k in range(1, T + 1))
    with pytest.raises(ValueError, match=f"smallest budget that works is {smallest} bytes"):
        _plan(lib, d, 8, 40, 40, T, smallest - 1)
    assert _plan(lib, d, 8, 40, 40, T, smallest)[2] == smallest


def test_plan_T0(lib):
    d = _desc()
    path, every, nb = _plan(lib, d, 4, 40, 40, 0, 1 << 30)
    assert path == "dense" and every is None and nb == 4 * 16 * 40 * 40 * 4


def test_public_bptt_plan_argument_checks():
    from graph_neural_cellular_automata_b200.rollout import bptt_plan

    class _M:
        def model_desc(self):
            return _desc()
    assert bptt_plan(_M(), 4, 40, 40, 12, 1 << 40)[0] == "records"
    with pytest.raises(ValueError):
        bptt_plan(_M(), 4, 40, 40, 12, 1 << 40, impl="banded")
    with pytest.raises(ValueError):
        bptt_plan(_M(), 4, 40, 40, 12, -1)


def test_trainer_config_reads_the_budget():
    from graph_neural_cellular_automata_b200.training.trainer import TrainConfig
    base = {"training": {"batch_size": 8, "pool_size": 64, "nca_steps_min": 48, "nca_steps_max": 80,
                         "learning_rate": 2e-4, "weight_decay": 1e-5}}
    assert TrainConfig().bptt_budget_bytes is None
    assert TrainConfig.from_reference_config(base).bptt_budget_bytes is None
    base["training"]["bptt_budget_bytes"] = 3 << 30
    assert TrainConfig.from_reference_config(base).bptt_budget_bytes == 3 << 30


def test_plan_leaves_resident_out_above_16_offsets(lib):
    from graph_neural_cellular_automata_b200.rollout import IMPL, RESIDENT_MAX_K, _bptt_plan
    d = _desc()
    assert _bptt_plan(d, 8, 40, 40, 100, 1 << 40, IMPL["auto"], RESIDENT_MAX_K)[0] == "records"
    # more offsets than the resident kernels take: the budget-free path is the dense history, the fallback streaming
    assert _bptt_plan(d, 8, 40, 40, 100, 1 << 40, IMPL["auto"], RESIDENT_MAX_K + 1)[0] == "dense"
    assert _bptt_plan(d, 8, 40, 40, 100, 100 << 20, IMPL["auto"], RESIDENT_MAX_K + 1)[0] == "streaming_ckpt"
    with pytest.raises(ValueError, match="offsets per step"):
        _bptt_plan(d, 8, 40, 40, 100, 1 << 40, IMPL["resident"], RESIDENT_MAX_K + 1)


def test_public_bptt_plan_reads_k_from_the_model():
    from graph_neural_cellular_automata_b200.rollout import bptt_plan

    class _Graph:
        num_neighbors, offsets = 24, [(0, 1)] * 40

    class _M:
        _is_graph, graph = True, _Graph()

        def model_desc(self):
            return _desc()
    assert bptt_plan(_M(), 8, 40, 40, 100, 100 << 20)[0] == "streaming_ckpt"
    assert bptt_plan(_M(), 8, 40, 40, 100, 100 << 20, k=8)[0] == "resident_ckpt"

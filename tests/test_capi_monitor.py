"""CPU checks of the monitoring rollout's C ABI (gnca_metrics_scratch_bytes / gnca_rollout_metrics) and of the argument
checks of rollout.monitor_rollout: the symbols, the scratch size, and argument errors that return before any launch."""
import ctypes as C

import pytest


@pytest.fixture(scope="module")
def lib():
    from graph_neural_cellular_automata_b200 import _lib, build
    build.build(verbose=False)
    return _lib.load()


def _desc(C_=16, graph=True):
    from graph_neural_cellular_automata_b200 import functional as GF
    return GF.make_model_desc(C_, 128, 16 if graph else 0, graph=graph, torus=True, hidden_only=graph,
                              alive_to_alive=graph, groupnorm=True, update_gain=0.05, alpha_thr=0.12,
                              graph_alpha_thr=0.12)


def test_symbols_exist(lib):
    assert hasattr(lib, "gnca_metrics_scratch_bytes") and hasattr(lib, "gnca_rollout_metrics")


@pytest.mark.parametrize("B,H,W,T,every", [(2, 40, 40, 10, 3), (128, 256, 256, 1000, 10), (16, 256, 256, 200, 1),
                                           (1, 8, 8, 0, 1), (4, 40, 40, 5, 9)])
def test_scratch_bytes_cover_every_family(lib, B, H, W, T, every):
    """one partial of 4 doubles per (frame, sample, rank <= 8) for the cluster kernels, and per (sample, block of 4096
    cells) of one frame for the streaming path"""
    F = T // every + 1
    need = max(F * B * 8, B * -(-H * W // 4096)) * 4 * 8
    assert lib.gnca_metrics_scratch_bytes(C.byref(_desc()), B, H, W, T, every) == need


@pytest.mark.parametrize("case", ["B0", "H0", "W0", "T_neg", "every0", "every_neg", "C3", "null_model"])
def test_scratch_bytes_zero_on_bad_arguments(lib, case):
    args = dict(B=2, H=40, W=40, T=10, every=2)
    desc = _desc()
    if case == "C3":
        desc = _desc(3, graph=False)
    elif case == "null_model":
        desc = None
    elif case == "T_neg":
        args["T"] = -1
    elif case == "every_neg":
        args["every"] = -1
    else:
        args[{"B0": "B", "H0": "H", "W0": "W", "every0": "every"}[case]] = 0
    d = C.byref(desc) if desc is not None else None
    assert lib.gnca_metrics_scratch_bytes(d, args["B"], args["H"], args["W"], args["T"], args["every"]) == 0


def _metrics(lib, desc, sched, *, every=2, eps=0.05, target=16, sums=16, counts=16, scratch=16, scratch_bytes=1 << 30):
    p = C.c_void_p(256)        # never dereferenced: every call below fails its argument checks first
    opt = lambda v: C.c_void_p(v) if v else None
    return lib.gnca_rollout_metrics(C.byref(desc), p, 2, 40, 40, C.byref(sched), p, p, every, opt(target), eps,
                                    opt(sums), opt(counts), opt(scratch), scratch_bytes, p, 1 << 30, 0, None)


@pytest.mark.parametrize("case,code", [("every0", "ARG"), ("every_neg", "ARG"), ("eps_neg", "ARG"), ("eps_nan", "ARG"),
                                       ("no_target", "ARG"), ("no_sums", "ARG"), ("no_counts", "ARG"),
                                       ("no_scratch", "ARG"), ("C3", "ARG"), ("T_neg", "ARG"),
                                       ("small_scratch", "WORKSPACE"), ("k65", "UNSUPPORTED"),
                                       ("k_neg", "UNSUPPORTED")])
def test_rollout_metrics_argument_errors_do_not_launch(lib, case, code):
    from graph_neural_cellular_automata_b200 import _lib
    p = C.c_void_p(512)
    sched = _lib.GncaSchedule(4, 8, p, p, p, None, None, 0, 0, None, 0, 4, 0, 0)
    desc = _desc(3, graph=False) if case == "C3" else _desc()
    kw = {}
    if case == "every0":
        kw["every"] = 0
    elif case == "every_neg":
        kw["every"] = -2
    elif case == "eps_neg":
        kw["eps"] = -0.01
    elif case == "eps_nan":
        kw["eps"] = float("nan")
    elif case.startswith("no_"):
        kw[case[3:]] = 0
    elif case == "small_scratch":
        kw["scratch_bytes"] = lib.gnca_metrics_scratch_bytes(C.byref(desc), 2, 40, 40, 4, 2) - 8
    elif case == "k65":
        sched.k = _lib.GNCA_MAX_K + 1
    elif case == "k_neg":
        sched.k = -1
    elif case == "T_neg":
        sched.T = -1
    before = lib.gnca_launch_count()
    assert _metrics(lib, desc, sched, **kw) == getattr(_lib, f"GNCA_ERR_{code}")
    assert lib.gnca_launch_count() == before


def test_monitor_rollout_rejects_bad_arguments_on_the_host():
    """Python-side checks that run before the library is asked for anything (no GPU needed)."""
    import torch
    import graph_neural_cellular_automata_b200 as G
    from graph_neural_cellular_automata_b200.rollout import Schedule, monitor_rollout
    g = G.NeuralCAGraph(16, update_hidden=128, img_size=8, graph_zero_padded_shift=False)
    x0 = torch.zeros(1, 16, 8, 8)
    tgt = torch.zeros(4, 8, 8)
    s = Schedule(T=2, k=0, fire_rate=torch.ones(2), message_gain=torch.zeros(2), offsets=None)
    for every in (0, -1):
        with pytest.raises(ValueError, match="every"):
            monitor_rollout(g, x0, s, tgt, every=every)
    for eps in (-0.1, float("nan")):
        with pytest.raises(ValueError, match="eps"):
            monitor_rollout(g, x0, s, tgt, every=1, eps=eps)
    with pytest.raises(ValueError, match="impl"):
        monitor_rollout(g, x0, s, tgt, every=1, impl="fastest")
    for bad in (torch.zeros(3, 8, 8), torch.zeros(4, 8, 9), torch.zeros(1, 4, 8, 8), torch.zeros(4, 64)):
        with pytest.raises(ValueError, match="target"):
            monitor_rollout(g, x0, s, bad, every=1)
    with pytest.raises(ValueError, match="channels"):
        monitor_rollout(g, torch.zeros(1, 8, 8, 8), s, tgt, every=1)
    with pytest.raises(RuntimeError, match="CUDA"):
        monitor_rollout(g, x0, s, tgt, every=1)          # CPU input: no fallback

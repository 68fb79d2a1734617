"""CPU checks of the recording rollout's C ABI (gnca_record_frames / gnca_rollout_record): the frame count, and
argument errors that return their code before any kernel is launched."""
import ctypes as C

import pytest


@pytest.fixture(scope="module")
def lib():
    from graph_neural_cellular_automata_b200 import _lib, build
    build.build(verbose=False)
    return _lib.load()


def _desc(graph=True):
    from graph_neural_cellular_automata_b200 import functional as GF
    return GF.make_model_desc(16, 128, 16 if graph else 0, graph=graph, torus=True, hidden_only=graph,
                              alive_to_alive=graph, groupnorm=True, update_gain=0.05, alpha_thr=0.12,
                              graph_alpha_thr=0.12)


@pytest.mark.parametrize("T,every,frames", [(0, 1, 1), (0, 5, 1), (1, 1, 2), (12, 5, 3), (12, 3, 5), (12, 12, 2),
                                            (12, 13, 1), (1000, 50, 21), (1000, 1, 1001), (7, 2, 4)])
def test_record_frames(lib, T, every, frames):
    assert lib.gnca_record_frames(T, every) == frames == T // every + 1


@pytest.mark.parametrize("T,every", [(5, 0), (5, -3), (-1, 1)])
def test_record_frames_rejects_bad_arguments(lib, T, every):
    from graph_neural_cellular_automata_b200 import _lib
    assert lib.gnca_record_frames(T, every) == _lib.GNCA_ERR_ARG


def _record(lib, desc, sched, *, every=2, frames=16, attn=0):
    p = C.c_void_p(256)        # never dereferenced: every call below fails its argument checks first
    return lib.gnca_rollout_record(C.byref(desc), p, 2, 40, 40, C.byref(sched), p, p, every,
                                   C.c_void_p(frames) if frames else None, C.c_void_p(attn) if attn else None, p,
                                   1 << 30, 0, None)


@pytest.mark.parametrize("case,code", [("every0", "ARG"), ("every_neg", "ARG"), ("no_frames", "ARG"),
                                       ("classic_attention", "ARG"), ("k65", "UNSUPPORTED"), ("k_neg", "UNSUPPORTED"),
                                       ("T_neg", "ARG")])
def test_rollout_record_argument_errors_do_not_launch(lib, case, code):
    from graph_neural_cellular_automata_b200 import _lib
    p = C.c_void_p(512)
    sched = _lib.GncaSchedule(4, 8, p, p, p, None, None, 0, 0, None, 0, 4, 0, 0)
    desc = _desc(graph=case != "classic_attention")
    kw = {}
    if case == "every0":
        kw["every"] = 0
    elif case == "every_neg":
        kw["every"] = -2
    elif case == "no_frames":
        kw["frames"] = 0
    elif case == "classic_attention":
        sched.k = 0
        kw["attn"] = 1024
    elif case == "k65":
        sched.k = _lib.GNCA_MAX_K + 1
    elif case == "k_neg":
        sched.k = -1
    elif case == "T_neg":
        sched.T = -1
    before = lib.gnca_launch_count()
    assert _record(lib, desc, sched, **kw) == getattr(_lib, f"GNCA_ERR_{code}")
    assert lib.gnca_launch_count() == before


def test_record_rollout_rejects_bad_arguments_on_the_host():
    """Python-side checks that run before the library is asked for anything (no GPU needed)."""
    import torch
    import graph_neural_cellular_automata_b200 as G
    from graph_neural_cellular_automata_b200.rollout import Schedule, record_rollout
    g = G.NeuralCAGraph(16, update_hidden=128, img_size=8, graph_zero_padded_shift=False)
    c = G.NeuralCA(16, update_hidden=128, img_size=8)
    x0 = torch.zeros(1, 16, 8, 8)
    s = Schedule(T=2, k=0, fire_rate=torch.ones(2), message_gain=torch.zeros(2), offsets=None)
    with pytest.raises(ValueError):
        record_rollout(g, x0, s, every=0)
    with pytest.raises(ValueError):
        record_rollout(c, x0, s, every=1, attention=True)
    with pytest.raises(RuntimeError):
        record_rollout(g, x0, s, every=1)          # CPU input: no fallback

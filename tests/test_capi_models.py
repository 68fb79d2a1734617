"""CPU checks of the model-stacked rollouts (gnca_rollout_record_models / gnca_rollout_metrics_models) and of the
list-of-models checks of rollout.record_rollout / monitor_rollout: the symbols, argument errors that return before any
launch, and the Python ValueErrors raised before any GPU work."""
import ctypes as C

import pytest


@pytest.fixture(scope="module")
def lib():
    from graph_neural_cellular_automata_b200 import _lib, build
    build.build(verbose=False)
    return _lib.load()


def _desc(C_=16):
    from graph_neural_cellular_automata_b200 import functional as GF
    return GF.make_model_desc(C_, 128, 16, graph=True, torus=True, hidden_only=True, alive_to_alive=True,
                              groupnorm=True, update_gain=0.05, alpha_thr=0.12, graph_alpha_thr=0.12)


def test_symbols_exist(lib):
    assert hasattr(lib, "gnca_rollout_record_models") and hasattr(lib, "gnca_rollout_metrics_models")


def _sched():
    from graph_neural_cellular_automata_b200 import _lib
    p = C.c_void_p(512)
    return _lib.GncaSchedule(4, 8, p, p, p, None, None, 0, 0, None, 0, 4, 0, 0)


def _record(lib, desc, sched, *, n_models=3, B=6, every=2, frames=16, packed=16, impl=0):
    p = C.c_void_p(256)        # never dereferenced: every call below fails its argument checks first
    opt = lambda v: C.c_void_p(v) if v else None
    return lib.gnca_rollout_record_models(C.byref(desc), opt(packed), n_models, B, 40, 40, C.byref(sched), p, p, every,
                                          opt(frames), p, 1 << 30, impl, None)


def _metrics(lib, desc, sched, *, n_models=3, B=6, every=2, eps=0.05, target=16, sums=16, packed=16, impl=0,
             scratch_bytes=1 << 30):
    p = C.c_void_p(256)
    opt = lambda v: C.c_void_p(v) if v else None
    return lib.gnca_rollout_metrics_models(C.byref(desc), opt(packed), n_models, B, 40, 40, C.byref(sched), p, p,
                                           every, opt(target), eps, opt(sums), p, p, scratch_bytes, p, 1 << 30, impl,
                                           None)


# case -> (expected code, keyword arguments, schedule edit)
CASES = {
    "n_models0": ("ARG", {"n_models": 0}, None),
    "n_models_neg": ("ARG", {"n_models": -2}, None),
    "B_not_multiple": ("ARG", {"n_models": 4, "B": 6}, None),
    "B0": ("ARG", {"B": 0}, None),
    "every0": ("ARG", {"every": 0}, None),
    "every_neg": ("ARG", {"every": -3}, None),
    "no_packed": ("ARG", {"packed": 0}, None),
    "impl_neg": ("ARG", {"impl": -1}, None),
    "impl4": ("ARG", {"impl": 4}, None),
    "T_neg": ("ARG", {}, ("T", -1)),
    "no_fire_rate": ("ARG", {}, ("fire_rate", None)),
    "no_message_gain": ("ARG", {}, ("message_gain", None)),
    "no_offsets": ("ARG", {}, ("offsets", None)),
    "streaming": ("UNSUPPORTED", {"impl": 1}, None),
    "k65": ("UNSUPPORTED", {}, ("k", 65)),
    "k_neg": ("UNSUPPORTED", {}, ("k", -1)),
}


@pytest.mark.parametrize("fn", ["record", "metrics"])
@pytest.mark.parametrize("case", list(CASES))
def test_argument_errors_do_not_launch(lib, fn, case):
    from graph_neural_cellular_automata_b200 import _lib
    code, kw, edit = CASES[case]
    sched = _sched()
    if edit is not None:
        setattr(sched, *edit)
    before = lib.gnca_launch_count()
    rc = (_record if fn == "record" else _metrics)(lib, _desc(), sched, **kw)
    assert rc == getattr(_lib, f"GNCA_ERR_{code}"), (case, rc)
    assert lib.gnca_launch_count() == before


@pytest.mark.parametrize("case,code", [("no_frames", "ARG"), ("no_target", "ARG"), ("no_sums", "ARG"),
                                       ("eps_neg", "ARG"), ("eps_nan", "ARG"), ("C3", "ARG"),
                                       ("small_scratch", "WORKSPACE")])
def test_per_call_argument_errors_do_not_launch(lib, case, code):
    """the checks of gnca_rollout_record / gnca_rollout_metrics, with the scratch sized for the total batch"""
    from graph_neural_cellular_automata_b200 import _lib
    sched = _sched()
    before = lib.gnca_launch_count()
    if case == "no_frames":
        rc = _record(lib, _desc(), sched, frames=0)
    elif case == "C3":
        rc = _metrics(lib, _desc(3), sched)
    elif case == "small_scratch":
        need = lib.gnca_metrics_scratch_bytes(C.byref(_desc()), 6, 40, 40, 4, 2)
        rc = _metrics(lib, _desc(), sched, scratch_bytes=need - 8)
    else:
        kw = {"no_target": {"target": 0}, "no_sums": {"sums": 0}, "eps_neg": {"eps": -0.5},
              "eps_nan": {"eps": float("nan")}}[case]
        rc = _metrics(lib, _desc(), sched, **kw)
    assert rc == getattr(_lib, f"GNCA_ERR_{code}"), (case, rc)
    assert lib.gnca_launch_count() == before


def _graph(torus=True, **kw):
    import graph_neural_cellular_automata_b200 as G
    args = dict(update_hidden=128, img_size=8, graph_zero_padded_shift=not torus)
    args.update(kw)
    return G.NeuralCAGraph(16, **args)


def test_record_rollout_rejects_bad_stacks_on_the_host():
    """The list-of-models checks run before the library is asked for anything: CPU models and states reach them."""
    import torch
    from graph_neural_cellular_automata_b200.rollout import Schedule, record_rollout
    g, h = _graph(), _graph()
    x0 = torch.zeros(4, 16, 8, 8)
    s = Schedule(T=2, k=0, fire_rate=torch.ones(2), message_gain=torch.zeros(2), offsets=None)
    with pytest.raises(ValueError, match="empty"):
        record_rollout([], x0, s, every=1)
    for kw, name in (({"differentiable": True}, "differentiable"), ({"attention": True}, "attention"),
                     ({"checkpoint": True, "differentiable": True}, "differentiable"),
                     ({"bptt_budget": 1 << 30}, "bptt_budget")):
        with pytest.raises(ValueError, match=name):
            record_rollout([g, h], x0, s, every=1, **kw)
    with pytest.raises(ValueError, match="streaming"):
        record_rollout([g, h], x0, s, every=1, impl="streaming")
    with pytest.raises(ValueError, match="multiple"):
        record_rollout([g, h, g], x0, s, every=1)
    with pytest.raises(ValueError, match="update_gain"):
        record_rollout([g, _graph(update_gain=0.2)], x0, s, every=1)
    with pytest.raises(ValueError, match="flags"):
        record_rollout([g, _graph(torus=False)], x0, s, every=1)
    with pytest.raises(ValueError, match="d_model"):
        record_rollout([g, _graph(graph_d_model=8)], x0, s, every=1)
    with pytest.raises(ValueError, match="graph.offsets or num_neighbors"):
        record_rollout([g, _graph(graph_num_neighbors=4)], x0, s, every=1)
    with pytest.raises(ValueError, match="meta"):
        record_rollout([g, _graph().to("meta")], x0, s, every=1)
    with pytest.raises(ValueError, match="x0 on meta"):
        record_rollout([g, h], x0.to("meta"), s, every=1)
    with pytest.raises(ValueError, match="every"):
        record_rollout([g, h], x0, s, every=0)
    with pytest.raises(RuntimeError, match="CUDA"):
        record_rollout([g, h], x0, s, every=1)          # a valid stack on CPU: no fallback
    with pytest.raises(RuntimeError, match="CUDA"):
        record_rollout((g,), x0, s, every=1)            # a tuple is a list of models too


def test_monitor_rollout_rejects_bad_stacks_on_the_host():
    import torch
    from graph_neural_cellular_automata_b200.rollout import Schedule, monitor_rollout
    g, h = _graph(), _graph()
    x0 = torch.zeros(4, 16, 8, 8)
    tgt = torch.zeros(4, 8, 8)
    s = Schedule(T=2, k=0, fire_rate=torch.ones(2), message_gain=torch.zeros(2), offsets=None)
    with pytest.raises(ValueError, match="empty"):
        monitor_rollout([], x0, s, tgt, every=1)
    with pytest.raises(ValueError, match="streaming"):
        monitor_rollout([g, h], x0, s, tgt, every=1, impl="streaming")
    with pytest.raises(ValueError, match="multiple"):
        monitor_rollout([g, h, g], x0, s, tgt, every=1)
    with pytest.raises(ValueError, match="alpha_thr"):
        monitor_rollout([g, _graph(alpha_thr=0.3)], x0, s, tgt, every=1)
    with pytest.raises(ValueError, match="graph.offsets or num_neighbors"):
        monitor_rollout([g, _graph(graph_num_neighbors=4)], x0, s, tgt, every=1)
    with pytest.raises(ValueError, match="target"):
        monitor_rollout([g, h], x0, s, torch.zeros(3, 8, 8), every=1)
    with pytest.raises(RuntimeError, match="CUDA"):
        monitor_rollout([g, h], x0, s, tgt, every=1)

"""CPU checks of training a stack of models: the stacked resident BPTT entry points (gnca_rollout_fwd_bptt_models,
gnca_rollout_bwd_bptt_models and their _zp forms), their workspace query, the list-of-models checks of
rollout.rollout, the record-buffer size of a stack, and the PopulationTrainer configuration errors -- all raised or
returned before any launch."""
import ctypes as C

import pytest

FWD = ("gnca_rollout_fwd_bptt_models", "gnca_rollout_fwd_bptt_zp_models")
BWD = ("gnca_rollout_bwd_bptt_models", "gnca_rollout_bwd_bptt_zp_models")


@pytest.fixture(scope="module")
def lib():
    from graph_neural_cellular_automata_b200 import _lib, build
    build.build(verbose=False)
    return _lib.load()


def _desc(torus=True):
    from graph_neural_cellular_automata_b200 import functional as GF
    return GF.make_model_desc(16, 128, 16, graph=True, torus=torus, hidden_only=True, alive_to_alive=True,
                              groupnorm=True, update_gain=0.05, alpha_thr=0.12, graph_alpha_thr=0.12)


def _sched():
    from graph_neural_cellular_automata_b200 import _lib
    p = C.c_void_p(512)
    return _lib.GncaSchedule(4, 8, p, p, p, None, None, 0, 0, None, 0, 4, 0, 0)


def test_symbols_exist(lib):
    for name in FWD + BWD + ("gnca_rollout_workspace_models_bytes",):
        assert hasattr(lib, name)


def _call(lib, name, desc, sched, *, n_models=3, B=6, packed=16, x0=16, gT=16, g0=16, gparams=16, bptt=16,
          bptt_bytes=1 << 40, ws=16, ws_bytes=1 << 40):
    opt = lambda v: C.c_void_p(v) if v else None
    if name in FWD:
        return getattr(lib, name)(C.byref(desc), opt(packed), n_models, B, 40, 40, C.byref(sched), opt(x0), opt(x0),
                                  opt(bptt), bptt_bytes, opt(ws), ws_bytes, None)
    return getattr(lib, name)(C.byref(desc), opt(packed), n_models, B, 40, 40, C.byref(sched), opt(bptt), bptt_bytes,
                              opt(gT), opt(g0), opt(gparams), opt(ws), ws_bytes, None)


# case -> (expected code, keyword arguments, schedule edit, entry points it applies to)
CASES = {
    "n_models0": ("ARG", {"n_models": 0}, None, FWD + BWD),
    "n_models_neg": ("ARG", {"n_models": -2}, None, FWD + BWD),
    "B_not_multiple": ("ARG", {"n_models": 4, "B": 6}, None, FWD + BWD),
    "B0": ("ARG", {"B": 0}, None, FWD + BWD),
    "T_neg": ("ARG", {}, ("T", -1), FWD + BWD),
    "no_packed": ("ARG", {"packed": 0}, None, FWD + BWD),
    "no_bptt": ("ARG", {"bptt": 0}, None, FWD + BWD),
    "no_workspace": ("ARG", {"ws": 0}, None, FWD + BWD),
    "no_x0": ("ARG", {"x0": 0}, None, FWD),
    "no_gT": ("ARG", {"gT": 0}, None, BWD),
    "no_g0": ("ARG", {"g0": 0}, None, BWD),
    "no_gparams": ("ARG", {"gparams": 0}, None, BWD),
    "no_fire_rate": ("ARG", {}, ("fire_rate", None), FWD + BWD),
    "no_message_gain": ("ARG", {}, ("message_gain", None), FWD + BWD),
    "no_offsets": ("ARG", {}, ("offsets", None), FWD + BWD),
    "k65": ("UNSUPPORTED", {}, ("k", 65), FWD + BWD),
    "small_bptt": ("WORKSPACE", {"bptt_bytes": 64}, None, FWD + BWD),
    "small_workspace": ("WORKSPACE", {"ws_bytes": 64}, None, FWD + BWD),
}


@pytest.mark.parametrize("name,case", [(n, c) for c, v in CASES.items() for n in v[3]])
def test_argument_errors_do_not_launch(lib, name, case):
    from graph_neural_cellular_automata_b200 import _lib
    code, kw, edit, _ = CASES[case]
    sched = _sched()
    if edit is not None:
        setattr(sched, *edit)
    # the _zp entry points take the zero-padded graph shift, the others torus / classic models
    desc = _desc(torus="_zp_" not in name)
    before = lib.gnca_launch_count()
    rc = _call(lib, name, desc, sched, **kw)
    assert rc == getattr(_lib, f"GNCA_ERR_{code}"), (case, rc)
    assert lib.gnca_launch_count() == before


@pytest.mark.parametrize("name", FWD + BWD)
def test_wrong_model_kind_is_unsupported(lib, name):
    """the plain pair has no zero-pad buffer and the _zp pair no torus one: GNCA_ERR_UNSUPPORTED, no fallback"""
    from graph_neural_cellular_automata_b200 import _lib
    before = lib.gnca_launch_count()
    assert _call(lib, name, _desc(torus="_zp_" in name), _sched()) == _lib.GNCA_ERR_UNSUPPORTED
    assert lib.gnca_launch_count() == before


def test_workspace_grows_with_n_models(lib):
    """at least one weight-gradient partial per model; up to 296 models the single-model workspace holds them"""
    from graph_neural_cellular_automata_b200 import functional as GF
    d = _desc()
    total = GF.param_layout(d).total
    for B, H in ((300, 40), (1200, 8)):
        one = lib.gnca_rollout_workspace_bytes(C.byref(d), B, H, H, 8)
        for M in (1, 150, 300):
            assert lib.gnca_rollout_workspace_models_bytes(C.byref(d), M, B, H, H, 8) == one
    # 1200 one-sample models on 8x8: the backward's scratch (GZ, RG, affine partials) plus 1200 partials is the largest
    B, HW = 1200, 64
    rep = (B * HW * (16 + 64) + B * 8 * 2 * 16 + 1200 * total) * 4 + 1024
    assert lib.gnca_rollout_workspace_models_bytes(C.byref(d), 1200, B, 8, 8, 8) == rep > one
    assert lib.gnca_rollout_workspace_models_bytes(C.byref(d), 0, 300, 40, 40, 8) == 0
    assert lib.gnca_rollout_workspace_models_bytes(None, 1, 300, 40, 40, 8) == 0


def _graph(torus=True, **kw):
    import graph_neural_cellular_automata_b200 as G
    args = dict(update_hidden=128, img_size=8, graph_zero_padded_shift=not torus)
    args.update(kw)
    return G.NeuralCAGraph(16, **args)


def test_rollout_rejects_bad_stacks_on_the_host():
    """The list-of-models checks of rollout() run before the library is asked for anything."""
    import torch
    from graph_neural_cellular_automata_b200.rollout import Schedule, rollout
    g, h = _graph(), _graph()
    x0 = torch.zeros(4, 16, 8, 8)
    s = Schedule(T=2, k=0, fire_rate=torch.ones(2), message_gain=torch.zeros(2), offsets=None)
    with pytest.raises(ValueError, match="empty"):
        rollout([], x0, s)
    for kw, name in (({"checkpoint_every": 1}, "checkpoint_every"), ({"bptt_budget": 1 << 30}, "bptt_budget"),
                     ({"return_history": True}, "return_history")):
        with pytest.raises(ValueError, match=name):
            rollout([g, h], x0, s, **kw)
    for impl in ("streaming", "banded"):
        with pytest.raises(ValueError, match=impl):
            rollout([g, h], x0, s, impl=impl)
    with pytest.raises(ValueError, match="multiple"):
        rollout([g, h, g], x0, s)
    with pytest.raises(ValueError, match="flags"):
        rollout([g, _graph(torus=False)], x0, s)
    with pytest.raises(ValueError, match="graph.offsets or num_neighbors"):
        rollout([g, _graph(graph_num_neighbors=4)], x0, s)
    with pytest.raises(RuntimeError, match="CUDA"):
        rollout([g, h], x0, s)                         # a valid stack on CPU: no fallback


def test_stack_bptt_bytes():
    """A stack keeps the single-model records of the whole batch, and raises, naming the bytes, where the single-model
    call would fall back to the dense streaming history."""
    from graph_neural_cellular_automata_b200 import _lib
    from graph_neural_cellular_automata_b200.rollout import BPTT_MAX_BYTES, _record_bytes, stack_bptt_bytes
    lib = _lib.load()
    for torus in (True, False):
        d = _desc(torus)
        nb, zp = stack_bptt_bytes(d, 12, 40, 40, 64, 8)
        assert zp == (not torus)
        assert nb == _record_bytes(lib, d, 12, 40, 40, 64, lib.gnca_bptt_zp_bytes if zp else lib.gnca_bptt_bytes) > 0
        assert stack_bptt_bytes(d, 12, 40, 40, 0, 8)[0] > 0          # T = 0 still takes a (tiny) buffer
        # 4 * 32 samples over 400 steps at 40x40: more records than BPTT_MAX_BYTES
        raw = (lib.gnca_bptt_zp_bytes if zp else lib.gnca_bptt_bytes)(C.byref(d), 128, 40, 40, 400)
        assert raw > BPTT_MAX_BYTES
        with pytest.raises(ValueError, match=f"{raw} bytes"):
            stack_bptt_bytes(d, 128, 40, 40, 400, 8)
        with pytest.raises(ValueError, match="resident BPTT"):
            stack_bptt_bytes(d, 4, 40, 42, 8, 8)                     # W % 4 != 0
        with pytest.raises(ValueError, match="resident BPTT"):
            stack_bptt_bytes(d, 4, 40, 40, 8, 17)                    # more offsets than the resident kernels take


def test_population_trainer_config_errors():
    import torch
    from graph_neural_cellular_automata_b200.training.population import PopulationTrainer
    from graph_neural_cellular_automata_b200.training.trainer import TrainConfig
    g, h = _graph(), _graph()
    tgt = torch.zeros(4, 8, 8)
    ok = dict(fire="philox", batch_size=2, pool_size=4)
    for kw, match in (({"fire": "torch"}, "philox"), ({"bptt_budget_bytes": 1 << 30}, "bptt_budget"),
                      ({"rollout_impl": "streaming"}, "rollout_impl"), ({"rollout_impl": "banded"}, "rollout_impl")):
        with pytest.raises(ValueError, match=match):
            PopulationTrainer([g, h], tgt, TrainConfig(**{**ok, **kw}))
    with pytest.raises(ValueError, match="learning rates"):
        PopulationTrainer([g, h], tgt, TrainConfig(**ok), learning_rates=[1e-3])
    with pytest.raises(ValueError, match="empty"):
        PopulationTrainer([], tgt, TrainConfig(**ok))
    with pytest.raises(ValueError, match="flags"):
        PopulationTrainer([g, _graph(torus=False)], tgt, TrainConfig(**ok))


def test_population_trainer_rejects_more_than_one_rank(monkeypatch):
    import torch
    from graph_neural_cellular_automata_b200.training import population
    from graph_neural_cellular_automata_b200.training.trainer import TrainConfig

    class TwoRanks(population.Shard):
        def __init__(self, global_batch):
            super().__init__(global_batch, rank=0, world=2)
    monkeypatch.setattr(population, "Shard", TwoRanks)
    with pytest.raises(ValueError, match="one rank"):
        population.PopulationTrainer([_graph(), _graph()], torch.zeros(4, 8, 8),
                                     TrainConfig(fire="philox", batch_size=2, pool_size=4))

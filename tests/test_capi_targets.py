"""CPU checks of per-model targets: gnca_rollout_metrics_targets and gnca_loss_premult_rgba_targets argument errors,
and the shape, count and device errors of monitor_rollout, premult_loss and PopulationTrainer with a [M, 4, H, W]
target -- all raised or returned before any launch."""
import ctypes as C

import pytest
import torch


@pytest.fixture(scope="module")
def lib():
    from graph_neural_cellular_automata_b200 import _lib, build
    build.build(verbose=False)
    return _lib.load()


def _desc(torus=True):
    from graph_neural_cellular_automata_b200 import functional as GF
    return GF.make_model_desc(16, 128, 16, graph=True, torus=torus, hidden_only=True, alive_to_alive=True,
                              groupnorm=True, update_gain=0.05, alpha_thr=0.12, graph_alpha_thr=0.12)


def _graph(**kw):
    import graph_neural_cellular_automata_b200 as G
    return G.NeuralCAGraph(16, update_hidden=128, img_size=8, graph_zero_padded_shift=False, **kw)


def test_symbols_exist(lib):
    for name in ("gnca_rollout_metrics_targets", "gnca_loss_premult_rgba_targets"):
        assert hasattr(lib, name)


# case -> (expected code, keyword arguments): the checks of the new entry point, then those it shares with the
# _models calls
METRICS_CASES = {
    "no_targets": ("ARG", {"targets": 0}),
    "n_models0": ("ARG", {"n_models": 0}),
    "n_models_neg": ("ARG", {"n_models": -1}),
    "B_not_multiple": ("ARG", {"n_models": 4, "B": 6}),
    "B0": ("ARG", {"B": 0}),
    "every0": ("ARG", {"every": 0}),
    "eps_neg": ("ARG", {"eps": -0.01}),
    "no_sums": ("ARG", {"sums": 0}),
    "no_counts": ("ARG", {"counts": 0}),
    "no_scratch": ("ARG", {"scratch": 0}),
    "ssim_H6": ("ARG", {"H": 6}),
    "impl4": ("ARG", {"impl": 4}),
    "streaming": ("UNSUPPORTED", {"impl": 1}),
    "small_scratch": ("WORKSPACE", {"scratch_bytes": 8}),
}


@pytest.mark.parametrize("ssim", [False, True])
@pytest.mark.parametrize("case", list(METRICS_CASES))
def test_rollout_metrics_targets_argument_errors_do_not_launch(lib, case, ssim):
    from graph_neural_cellular_automata_b200 import _lib
    code, kw = METRICS_CASES[case]
    ssim = ssim or case == "ssim_H6"                 # H < 7 is an error of the SSIM only
    p = C.c_void_p(512)          # never dereferenced: every call below fails its argument checks first
    sched = _lib.GncaSchedule(4, 8, p, p, p, None, None, 0, 0, None, 0, 4, 0, 0)
    a = dict(n_models=3, B=6, H=40, W=40, every=2, eps=0.05, targets=16, sums=16, counts=16, ssim=16 if ssim else 0,
             scratch=16, scratch_bytes=1 << 30, impl=0)
    a.update(kw)
    opt = lambda v: C.c_void_p(v) if v else None
    before = lib.gnca_launch_count()
    rc = lib.gnca_rollout_metrics_targets(C.byref(_desc()), p, a["n_models"], a["B"], a["H"], a["W"], C.byref(sched),
                                          p, p, a["every"], opt(a["targets"]), a["eps"], opt(a["sums"]),
                                          opt(a["counts"]), opt(a["ssim"]), opt(a["scratch"]), a["scratch_bytes"], p,
                                          1 << 30, a["impl"], None)
    assert rc == getattr(_lib, f"GNCA_ERR_{code}"), rc
    assert lib.gnca_launch_count() == before


@pytest.mark.parametrize("n_targets,B,C_,x,tgt,per,code", [
    (0, 4, 16, 16, 16, 16, "ARG"), (-1, 4, 16, 16, 16, 16, "ARG"), (3, 4, 16, 16, 16, 16, "ARG"),
    (5, 4, 16, 16, 16, 16, "ARG"), (2, 4, 16, 0, 16, 16, "ARG"), (2, 4, 16, 16, 0, 16, "ARG"),
    (2, 4, 16, 16, 16, 0, "ARG"), (2, 0, 16, 16, 16, 16, "ARG"), (2, 4, 3, 16, 16, 16, "ARG")])
def test_loss_targets_argument_errors_do_not_launch(lib, n_targets, B, C_, x, tgt, per, code):
    from graph_neural_cellular_automata_b200 import _lib
    opt = lambda v: C.c_void_p(v) if v else None
    before = lib.gnca_launch_count()
    rc = lib.gnca_loss_premult_rgba_targets(B, C_, 8, 8, opt(x), opt(tgt), n_targets, opt(per), None, 1.0, None)
    assert rc == getattr(_lib, f"GNCA_ERR_{code}")
    assert lib.gnca_launch_count() == before


def test_monitor_rollout_target_errors():
    """a [M', 4, H, W] target with M' != M names both counts; a single model keeps rejecting a 4-D target; the
    spatial shape is checked; a CPU tensor is refused without a fallback"""
    from graph_neural_cellular_automata_b200.rollout import Schedule, monitor_rollout
    g, h = _graph(), _graph()
    x0 = torch.zeros(4, 16, 8, 8)
    s = Schedule(T=2, k=0, fire_rate=torch.ones(2), message_gain=torch.zeros(2), offsets=None)
    for n in (1, 3, 4):
        with pytest.raises(ValueError, match=f"{n} targets for 2 models"):
            monitor_rollout([g, h], x0, s, torch.zeros(n, 4, 8, 8), every=1)
        with pytest.raises(ValueError, match=f"{n} targets for 2 models"):
            monitor_rollout([g, h], x0, s, torch.zeros(n, 4, 8, 8), every=1, ssim=True)
    for bad in (torch.zeros(2, 3, 8, 8), torch.zeros(2, 4, 8, 9), torch.zeros(2, 4, 64), torch.zeros(1, 2, 4, 8, 8)):
        with pytest.raises(ValueError, match="target"):
            monitor_rollout([g, h], x0, s, bad, every=1)
    for bad in (torch.zeros(1, 4, 8, 8), torch.zeros(2, 4, 8, 8)):
        with pytest.raises(ValueError, match=r"target must be \[4, 8, 8\]"):
            monitor_rollout(g, x0[:2], s, bad, every=1)
    with pytest.raises(RuntimeError, match="CUDA"):
        monitor_rollout([g, h], x0, s, torch.zeros(2, 4, 8, 8), every=1)


def test_premult_loss_target_errors():
    from graph_neural_cellular_automata_b200.training.trainer import premult_loss
    x = torch.zeros(6, 16, 8, 8)
    for bad in (torch.zeros(4, 4, 8, 8), torch.zeros(5, 4, 8, 8), torch.zeros(2, 3, 8, 8), torch.zeros(2, 4, 8, 9),
                torch.zeros(0, 4, 8, 8)):
        with pytest.raises(ValueError, match="target"):
            premult_loss(x, bad, 1.0)
    with pytest.raises(RuntimeError, match="CUDA"):
        premult_loss(x, torch.zeros(3, 4, 8, 8), 1.0)        # CPU target: no fallback


def test_population_trainer_target_count():
    from graph_neural_cellular_automata_b200.training.population import PopulationTrainer
    from graph_neural_cellular_automata_b200.training.trainer import TrainConfig
    g, h = _graph(), _graph()
    for n in (1, 3):
        with pytest.raises(ValueError, match=f"{n} targets for 2 models"):
            PopulationTrainer([g, h], torch.zeros(n, 4, 8, 8), TrainConfig(fire="philox", batch_size=2, pool_size=4))

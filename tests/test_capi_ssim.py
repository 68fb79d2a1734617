"""CPU checks of SSIM: the fp64 oracle (oracle/ssim_oracle.py) pinned by an independent formulation and closed forms,
and the C ABI (gnca_ssim_rgb, gnca_rollout_metrics_ssim[_models] and their scratch queries) and Python wrappers'
argument errors, which return before any launch."""
import ctypes as C

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import ssim_oracle as SO


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


def _pool_ssim(state, target):
    """the same definition through avg_pool2d windows, in float64"""
    pred, tgt = SO.images(state, target)
    x = torch.from_numpy(pred)
    y = torch.from_numpy(tgt)[None].expand_as(x)
    m = lambda a: F.avg_pool2d(a, 7, stride=1)
    ux, uy = m(x), m(y)
    vx = (m(x * x) - ux * ux) * 49 / 48
    vy = (m(y * y) - uy * uy) * 49 / 48
    vxy = (m(x * y) - ux * uy) * 49 / 48
    S = (2 * ux * uy + SO.C1) * (2 * vxy + SO.C2) / ((ux ** 2 + uy ** 2 + SO.C1) * (vx + vy + SO.C2))
    return S.mean(dim=(1, 2, 3)).numpy()


@pytest.mark.parametrize("B,Cc,H,W", [(3, 16, 40, 40), (2, 4, 7, 7), (2, 32, 7, 40), (1, 8, 41, 37)])
def test_oracle_matches_pooled_formulation(B, Cc, H, W):
    g = torch.Generator().manual_seed(H * W + Cc)
    x = torch.rand(B, Cc, H, W, generator=g) * 1.4 - 0.2
    x[:, :, : H // 3] *= 0.01                              # near-flat windows next to textured ones
    tgt = torch.rand(4, H, W, generator=g)
    np.testing.assert_allclose(SO.ssim_rgb(x, tgt), _pool_ssim(x, tgt), rtol=0, atol=1e-12)


def test_oracle_identical_images_give_one():
    g = torch.Generator().manual_seed(1)
    x = torch.rand(2, 4, 20, 13, generator=g)
    x[:, 3] = 1.0
    tgt = torch.cat([x[0, :3], torch.ones(1, 20, 13)])
    assert abs(SO.ssim_rgb(x[:1], tgt)[0] - 1.0) < 1e-15


@pytest.mark.parametrize("a,b", [(0.3, 0.7), (0.0, 0.5), (1.0, 1.0), (0.05, 0.9)])
def test_oracle_constant_images(a, b):
    x = torch.zeros(1, 4, 9, 11)
    x[:, :3] = a
    x[:, 3] = 1.0
    tgt = torch.full((4, 9, 11), b)
    a, b = float(torch.tensor(a)), float(torch.tensor(b))      # the fp32 values the images hold
    assert abs(SO.ssim_rgb(x, tgt)[0] - (2 * a * b + SO.C1) / (a * a + b * b + SO.C1)) < 1e-12


@pytest.mark.parametrize("H,W", [(6, 40), (40, 6), (6, 6)])
def test_oracle_rejects_grids_below_the_window(H, W):
    with pytest.raises(ValueError):
        SO.ssim_rgb(torch.zeros(1, 4, H, W), torch.zeros(4, H, W))


def test_symbols_exist(lib):
    for s in ("gnca_ssim_rgb", "gnca_ssim_rgb_scratch_bytes", "gnca_metrics_ssim_scratch_bytes",
              "gnca_rollout_metrics_ssim", "gnca_rollout_metrics_ssim_models"):
        assert hasattr(lib, s)


@pytest.mark.parametrize("B,H,W", [(1, 7, 7), (3, 40, 40), (16, 256, 256), (2, 41, 37)])
def test_ssim_rgb_scratch_bytes(lib, B, H, W):
    """one double per (sample, block of 1024 cells)"""
    assert lib.gnca_ssim_rgb_scratch_bytes(B, H, W) == B * -(-H * W // 1024) * 8


@pytest.mark.parametrize("B,H,W", [(0, 40, 40), (2, 6, 40), (2, 40, 6), (-1, 40, 40)])
def test_ssim_rgb_scratch_bytes_zero_on_bad_arguments(lib, B, H, W):
    assert lib.gnca_ssim_rgb_scratch_bytes(B, H, W) == 0


@pytest.mark.parametrize("B,H,W,T,every", [(2, 40, 40, 10, 3), (128, 256, 256, 1000, 10), (16, 256, 256, 200, 1),
                                           (1, 7, 8, 0, 1), (148, 40, 40, 1000, 10)])
def test_metrics_ssim_scratch_bytes(lib, B, H, W, T, every):
    """the metrics scratch, then one double per (frame, sample, rank <= 8) or per (sample, block) of one frame"""
    d = C.byref(_desc())
    F_ = T // every + 1
    met = lib.gnca_metrics_scratch_bytes(d, B, H, W, T, every)
    assert met > 0
    assert lib.gnca_metrics_ssim_scratch_bytes(d, B, H, W, T, every) == met + max(F_ * B * 8,
                                                                                  B * -(-H * W // 1024)) * 8


@pytest.mark.parametrize("case", ["B0", "H6", "W6", "T_neg", "every0", "C3", "null_model"])
def test_metrics_ssim_scratch_bytes_zero_on_bad_arguments(lib, case):
    a = dict(B=2, H=40, W=40, T=10, every=2)
    desc = _desc(3, graph=False) if case == "C3" else _desc()
    if case == "B0":
        a["B"] = 0
    elif case == "H6":
        a["H"] = 6
    elif case == "W6":
        a["W"] = 6
    elif case == "T_neg":
        a["T"] = -1
    elif case == "every0":
        a["every"] = 0
    d = None if case == "null_model" else C.byref(desc)
    assert lib.gnca_metrics_ssim_scratch_bytes(d, a["B"], a["H"], a["W"], a["T"], a["every"]) == 0


@pytest.mark.parametrize("case,code", [("no_x", "ARG"), ("no_target", "ARG"), ("no_ssim", "ARG"), ("no_scratch", "ARG"),
                                       ("B0", "ARG"), ("C3", "ARG"), ("H6", "ARG"), ("W6", "ARG"),
                                       ("small_scratch", "WORKSPACE")])
def test_ssim_rgb_argument_errors_do_not_launch(lib, case, code):
    from graph_neural_cellular_automata_b200 import _lib
    a = dict(x=256, target=256, ssim=256, scratch=256, B=2, C=16, H=40, W=40)
    a["scratch_bytes"] = lib.gnca_ssim_rgb_scratch_bytes(2, 40, 40)
    if case.startswith("no_"):
        a[case[3:]] = 0
    elif case == "B0":
        a["B"] = 0
    elif case == "C3":
        a["C"] = 3
    elif case in ("H6", "W6"):
        a[case[0]] = 6
    elif case == "small_scratch":
        a["scratch_bytes"] -= 8
    opt = lambda v: C.c_void_p(v) if v else None
    before = lib.gnca_launch_count()
    rc = lib.gnca_ssim_rgb(opt(a["x"]), a["B"], a["C"], a["H"], a["W"], opt(a["target"]), opt(a["ssim"]),
                           opt(a["scratch"]), a["scratch_bytes"], None)
    assert rc == getattr(_lib, f"GNCA_ERR_{code}")
    assert lib.gnca_launch_count() == before


CASES = [("every0", "ARG"), ("eps_neg", "ARG"), ("no_target", "ARG"), ("no_sums", "ARG"), ("no_counts", "ARG"),
         ("no_ssim", "ARG"), ("no_scratch", "ARG"), ("C3", "ARG"), ("T_neg", "ARG"), ("H6", "ARG"), ("W6", "ARG"),
         ("small_scratch", "WORKSPACE"), ("met_scratch_only", "WORKSPACE"), ("k65", "UNSUPPORTED"),
         ("k_neg", "UNSUPPORTED")]


@pytest.mark.parametrize("models", [False, True])
@pytest.mark.parametrize("case,code", CASES)
def test_rollout_metrics_ssim_argument_errors_do_not_launch(lib, case, code, models):
    from graph_neural_cellular_automata_b200 import _lib
    p = C.c_void_p(512)          # never dereferenced: every call below fails its argument checks first
    sched = _lib.GncaSchedule(4, 8, p, p, p, None, None, 0, 0, None, 0, 4, 0, 0)
    desc = _desc(3, graph=False) if case == "C3" else _desc()
    a = dict(every=2, eps=0.05, target=16, sums=16, counts=16, ssim=16, scratch=16, H=40, W=40, scratch_bytes=1 << 30)
    if case == "every0":
        a["every"] = 0
    elif case == "eps_neg":
        a["eps"] = -0.01
    elif case.startswith("no_"):
        a[case[3:]] = 0
    elif case in ("H6", "W6"):
        a[case[0]] = 6
    elif case == "small_scratch":
        a["scratch_bytes"] = lib.gnca_metrics_ssim_scratch_bytes(C.byref(desc), 2, 40, 40, 4, 2) - 8
    elif case == "met_scratch_only":
        a["scratch_bytes"] = lib.gnca_metrics_scratch_bytes(C.byref(desc), 2, 40, 40, 4, 2)
    elif case == "k65":
        sched.k = _lib.GNCA_MAX_K + 1
    elif case == "k_neg":
        sched.k = -1
    elif case == "T_neg":
        sched.T = -1
    opt = lambda v: C.c_void_p(v) if v else None
    tail = (a["every"], opt(a["target"]), a["eps"], opt(a["sums"]), opt(a["counts"]), opt(a["ssim"]),
            opt(a["scratch"]), a["scratch_bytes"], p, 1 << 30, 0, None)
    before = lib.gnca_launch_count()
    if models:
        rc = lib.gnca_rollout_metrics_ssim_models(C.byref(desc), p, 2, 2, a["H"], a["W"], C.byref(sched), p, p, *tail)
    else:
        rc = lib.gnca_rollout_metrics_ssim(C.byref(desc), p, 2, a["H"], a["W"], C.byref(sched), p, p, *tail)
    assert rc == getattr(_lib, f"GNCA_ERR_{code}")
    assert lib.gnca_launch_count() == before


def test_rollout_metrics_ssim_models_stack_errors(lib):
    """n_models < 1 or not dividing B, and the streaming impl, before any launch"""
    from graph_neural_cellular_automata_b200 import _lib
    p = C.c_void_p(512)
    sched = _lib.GncaSchedule(4, 8, p, p, p, None, None, 0, 0, None, 0, 4, 0, 0)
    d = C.byref(_desc())
    before = lib.gnca_launch_count()
    for n, B, impl, code in [(0, 2, 0, "ARG"), (3, 4, 0, "ARG"), (2, 4, 1, "UNSUPPORTED"), (2, 4, 4, "ARG")]:
        rc = lib.gnca_rollout_metrics_ssim_models(d, p, n, B, 40, 40, C.byref(sched), p, p, 2, p, 0.05, p, p, p, p,
                                                  1 << 30, p, 1 << 30, impl, None)
        assert rc == getattr(_lib, f"GNCA_ERR_{code}"), (n, B, impl)
    assert lib.gnca_launch_count() == before


def test_host_side_errors():
    """ValueErrors of monitor_rollout(..., ssim=True) and ssim_rgb before the library is asked for anything, and the
    RuntimeError of a CPU tensor"""
    import graph_neural_cellular_automata_b200 as G
    from graph_neural_cellular_automata_b200.rollout import Schedule, monitor_rollout
    from graph_neural_cellular_automata_b200.utils.metrics import ssim_rgb
    g = G.NeuralCAGraph(16, update_hidden=128, img_size=8, graph_zero_padded_shift=False)
    s = Schedule(T=2, k=0, fire_rate=torch.ones(2), message_gain=torch.zeros(2), offsets=None)
    for H, W in ((6, 8), (8, 6), (6, 6)):
        with pytest.raises(ValueError, match="7x7"):
            monitor_rollout(g, torch.zeros(1, 16, H, W), s, torch.zeros(4, H, W), every=1, ssim=True)
        with pytest.raises(ValueError, match="7x7"):
            ssim_rgb(torch.zeros(2, 16, H, W), torch.zeros(4, H, W))
    with pytest.raises(RuntimeError, match="CUDA"):
        monitor_rollout(g, torch.zeros(1, 16, 8, 8), s, torch.zeros(4, 8, 8), every=1, ssim=True)
    for bad_state, bad_tgt in [(torch.zeros(2, 3, 8, 8), torch.zeros(4, 8, 8)), (torch.zeros(16, 8, 8), torch.zeros(4, 8, 8)),
                               (torch.zeros(2, 4, 8, 8), torch.zeros(3, 8, 8)), (torch.zeros(2, 4, 8, 8), torch.zeros(4, 8, 9))]:
        with pytest.raises(ValueError):
            ssim_rgb(bad_state, bad_tgt)
    with pytest.raises(RuntimeError, match="CUDA"):
        ssim_rgb(torch.zeros(2, 4, 8, 8), torch.zeros(4, 8, 8))

"""GPU tests of the monitoring rollout (gnca_rollout_metrics through rollout.monitor_rollout).

The per-frame metrics are pinned to the frames record_rollout keeps on the same impl: the pixel-perfect and alive
counts exactly to the utils.metrics expressions, the squared-error sums to an fp64 recomputation; x_T bit for bit to
the plain rollout; two calls bit for bit to each other.  Models, states and schedules are built here."""
import ctypes as C
import random

import pytest
import torch

from conftest import load_params

pytestmark = pytest.mark.gpu

if torch.cuda.is_available():
    import graph_neural_cellular_automata_b200 as G
    from graph_neural_cellular_automata_b200 import _lib
    from graph_neural_cellular_automata_b200 import functional as GF
    from graph_neural_cellular_automata_b200.rollout import IMPL, make_schedule, monitor_rollout, record_rollout, rollout
    from graph_neural_cellular_automata_b200.utils import metrics as UM

DEV = "cuda"
IMPLS = ["streaming", "resident", "banded"]


def _graph16(torus):
    m = G.NeuralCAGraph(16, update_hidden=128, img_size=40, update_gain=0.05, alpha_thr=0.12, message_gain=0.25,
                        hidden_only=True, graph_zero_padded_shift=not torus)
    missing, unexpected = m.load_state_dict(load_params("weights_graph_ep960.npz"), strict=False)
    assert not missing and not unexpected
    return m.to(DEV)


def _classic16():
    m = G.NeuralCA(16, update_hidden=128, img_size=40, update_gain=0.1, alpha_thr=0.1)
    missing, unexpected = m.load_state_dict(load_params("weights_classic_ep990.npz"), strict=False)
    assert not missing and not unexpected
    return m.to(DEV)


def _random_graph(C_, H, seed=5):
    torch.manual_seed(seed); random.seed(seed)
    m = G.NeuralCAGraph(C_, update_hidden=128, img_size=H, update_gain=0.1, alpha_thr=0.1, message_gain=0.3,
                        hidden_only=True, graph_zero_padded_shift=False)
    with torch.no_grad():
        m.update_net[2].weight.normal_(0, 0.05)
        m.norm.weight.uniform_(0.5, 1.5); m.norm.bias.normal_(0, 0.1)
    return m.to(DEV)


MODELS = {"torus": lambda: _graph16(True), "zeropad": lambda: _graph16(False), "classic": _classic16}


def _blob(B, C_, H, W, seed=0):
    """random state inside a disk (alive cells with a dead border around them)"""
    g = torch.Generator().manual_seed(seed)
    yy, xx = torch.meshgrid(torch.arange(H), torch.arange(W), indexing="ij")
    disk = (((yy - H / 2) ** 2 + (xx - W / 2) ** 2) < (0.3 * min(H, W)) ** 2).float()
    return (torch.rand(B, C_, H, W, generator=g) * disk).to(DEV)


def _target(x0, seed=0):
    """premultiplied RGBA near sample 0 of x0: a mix of cells within eps of it and cells far from it"""
    g = torch.Generator().manual_seed(seed)
    return (UM.premultiply(x0[:1])[0] + 0.03 * torch.randn(4, *x0.shape[2:], generator=g).to(DEV)).contiguous()


def _case_schedule(m, B, H, W, T, *, fire="u", steps=None, damage_step=None, seed=0, philox_offset=0):
    """per-step fire rates and gains (every third gain 0), recorded uniforms or in-kernel Philox, optional damage and
    ragged steps"""
    random.seed(seed)
    graph = getattr(m, "_is_graph", False)
    offs = [m.graph.draw_offsets() for _ in range(T)] if graph else None
    frs = [0.5 + 0.4 * ((7 * t) % 10) / 10 for t in range(T)]
    gains = [0.25 if t % 3 != 1 else 0.0 for t in range(T)] if graph else None
    fu = None
    if fire == "u":
        fu = torch.rand(T, B, H, W, device=DEV, generator=torch.Generator(device=DEV).manual_seed(seed + 1))
    dmg = None
    if damage_step is not None:
        dmg = torch.ones(B, m.n_channels, H, W, device=DEV)
        dmg[:, :, H // 3:H // 3 + H // 4, W // 4:W // 2] = 0.0
        dmg[0, :, H // 2:H // 2 + 3, :] = 0.5
    s = make_schedule(m, B, H, W, T, fire_rate=frs, offsets=offs, fire_u=fu, message_gains=gains, steps=steps,
                      fire="philox", seed=seed + 7, damage=dmg, damage_step=damage_step or 0)
    s.philox_offset = philox_offset
    return s


def _raw(m, x0, s, tgt, every, impl, eps=0.05):
    """gnca_rollout_metrics straight through the C ABI -> (rc, x_T, sums [F,B,2] f64, counts [F,B,2] i32)"""
    lib = _lib.load()
    desc = m.model_desc()
    B, _, H, W = x0.shape
    F = s.T // every + 1
    xT = torch.empty_like(x0)
    sums = torch.full((F, B, 2), float("nan"), dtype=torch.float64, device=DEV)
    counts = torch.full((F, B, 2), -1, dtype=torch.int32, device=DEV)
    scratch = torch.empty(lib.gnca_metrics_scratch_bytes(C.byref(desc), B, H, W, s.T, every), dtype=torch.uint8,
                          device=DEV)
    ws = GF._WS.get(x0.device, lib.gnca_rollout_workspace_bytes(C.byref(desc), B, H, W, s.T))
    cs = s.c_struct()
    rc = lib.gnca_rollout_metrics(C.byref(desc), GF._ptr(m.packed_weights()), B, H, W, C.byref(cs), GF._ptr(x0),
                                  GF._ptr(xT), every, GF._ptr(tgt), eps, GF._ptr(sums), GF._ptr(counts),
                                  GF._ptr(scratch), scratch.numel(), GF._ptr(ws), ws.numel(), IMPL[impl],
                                  GF._stream())
    return rc, xT, sums, counts


def _reference(frames, tgt, thr, eps):
    """the metrics of every frame [F,B,C,H,W] from utils.metrics (counts) and in fp64 (squared-error sums)"""
    F, B = frames.shape[:2]
    x = frames.reshape(F * B, *frames.shape[2:])
    pm = UM.premultiply(x)
    pp = ((pm - tgt.unsqueeze(0)).abs() < eps).all(dim=1).sum(dim=(1, 2)).reshape(F, B)
    alive = (x[:, 3] > thr).sum(dim=(1, 2)).reshape(F, B)
    x64, t64 = x.double(), tgt.double()
    pm64 = torch.cat([x64[:, :3] * x64[:, 3:4], x64[:, 3:4]], dim=1)
    se = ((pm64 - t64.unsqueeze(0)) ** 2).sum(dim=(1, 2, 3)).reshape(F, B)
    sr = ((pm64[:, :3].clamp(0, 1) - t64[:3].clamp(0, 1).unsqueeze(0)) ** 2).sum(dim=(1, 2, 3)).reshape(F, B)
    return pp, alive, se, sr


def _check(m, x0, s, tgt, S, impl, eps=0.05):
    """checks 1-3 of one configuration: frames' metrics, x_T, determinism; skipped where `impl` has no kernel"""
    T = s.T
    B, _, H, W = x0.shape
    HW = H * W
    with torch.no_grad():
        rc, xT, sums, counts = _raw(m, x0, s, tgt, S, impl, eps)
        if rc == _lib.GNCA_ERR_UNSUPPORTED:
            with pytest.raises(_lib.GncaError, match="unsupported"):
                record_rollout(m, x0, s, every=S, impl=impl)
            with pytest.raises(_lib.GncaError, match="unsupported"):
                monitor_rollout(m, x0, s, tgt, every=S, impl=impl, eps=eps)
            pytest.skip(f"{impl}: no kernel for this configuration")
        _lib.check(rc, "gnca_rollout_metrics")
        tr = record_rollout(m, x0, s, every=S, impl=impl)
        xT_plain = rollout(m, x0, s, impl=impl)
        mon = monitor_rollout(m, x0, s, tgt, every=S, impl=impl, eps=eps)
        rc2, xT2, sums2, counts2 = _raw(m, x0, s, tgt, S, impl, eps)
    F = T // S + 1
    assert mon.t == tr.t == [f * S for f in range(F)]
    # the rollout is untouched
    assert torch.equal(xT, xT_plain) and torch.equal(mon.x_T, xT_plain) and torch.equal(tr.x_T, xT_plain)
    # determinism
    assert rc2 == 0 and torch.equal(sums, sums2) and torch.equal(counts, counts2) and torch.equal(xT, xT2)
    # equality with the frames
    pp, alive, se, sr = _reference(tr.states, tgt, float(m.model_desc().alpha_thr), eps)
    assert torch.equal(counts[..., 0].long(), pp), (counts[..., 0], pp)
    assert torch.equal(counts[..., 1].long(), alive), (counts[..., 1], alive)
    assert torch.equal(mon.alive, alive)
    assert torch.equal(torch.round(mon.pixel_perfect.double() * HW).long(), pp)
    assert ((sums[..., 0] - se).abs() <= 1e-6 * se.abs() + 1e-12).all(), (sums[..., 0], se)
    assert ((sums[..., 1] - sr).abs() <= 1e-6 * sr.abs() + 1e-12).all(), (sums[..., 1], sr)
    assert torch.allclose(mon.loss.double(), se / (4 * HW), rtol=1e-6, atol=0)
    psnr64 = 10 * torch.log10(1 / (sr / (3 * HW)))
    assert torch.allclose(mon.psnr.double(), psnr64, rtol=1e-6, atol=1e-5)
    # the utils.metrics functions on the frames, in fp32
    for f in range(F):
        assert torch.allclose(mon.pixel_perfect[f], UM.pixel_perfect(tr.states[f], tgt, eps), rtol=1e-6, atol=0)
        assert torch.allclose(mon.psnr[f], UM.psnr_rgb(tr.states[f], tgt), rtol=1e-5, atol=1e-4)
    for v in (mon.loss, mon.psnr, mon.pixel_perfect, mon.alive, mon.x_T):
        assert not v.requires_grad and v.grad_fn is None
    return mon


# name: T, every, fire, ragged steps, damage step, philox offset
CASES = {
    "S1": (7, 1, "u", None, None, 0),
    "S3_T%S!=0": (10, 3, "u", None, None, 0),
    "S=T": (9, 9, "u", None, None, 0),
    "S>T": (9, 10, "u", None, None, 0),
    "T0": (0, 1, "u", None, None, 0),
    "T0_S3_damage": (0, 3, "u", None, 0, 0),
    "ragged_philox_damage_at_frame": (10, 3, "philox", [10, 4], 6, 0),
    "ragged_u_damage_between_frames": (11, 3, "u", [5, 11], 4, 0),
    "ragged_frozen_on_frame": (12, 4, "u", [8, 3], None, 0),
    "damage_at_frame_S2": (8, 2, "u", None, 2, 0),
    "damage_at_0": (6, 2, "u", None, 0, 0),
    "philox_offset": (10, 3, "philox", [10, 7], 5, 123457),
}


@pytest.mark.parametrize("impl", IMPLS)
@pytest.mark.parametrize("model", list(MODELS))
@pytest.mark.parametrize("case", list(CASES))
def test_metrics_equal_frames(case, model, impl):
    T, S, fire, steps, dstep, poff = CASES[case]
    m = MODELS[model]()
    B, H, W = 2, 40, 40
    x0 = _blob(B, 16, H, W, seed=1)
    s = _case_schedule(m, B, H, W, T, fire=fire, steps=steps, damage_step=dstep, seed=3, philox_offset=poff)
    _check(m, x0, s, _target(x0), S, impl)


@pytest.mark.parametrize("impl", ["auto", "resident"])
@pytest.mark.parametrize("eps", [0.0, 0.02, 0.3])
def test_metrics_eps_and_batch(impl, eps):
    """other tolerances (eps = 0 counts nothing), a larger batch and the auto dispatch"""
    m = MODELS["torus"]()
    B, H, W, T, S = 6, 40, 40, 9, 2
    x0 = _blob(B, 16, H, W, seed=4)
    s = _case_schedule(m, B, H, W, T, fire="philox", steps=[9, 2, 9, 5, 1, 9], damage_step=3, seed=5)
    mon = _check(m, x0, s, _target(x0, seed=1), S, impl, eps=eps)
    if eps == 0.0:
        assert int(mon.pixel_perfect.count_nonzero()) == 0


@pytest.mark.parametrize("impl", ["resident", "banded"])
def test_metrics_c32_banded(impl):
    """C = 32 at 40x40 runs on the banded cluster kernel (the replicated-state kernel is C = 16 only)"""
    m = _random_graph(32, 40)
    B, H, W, T, S = 3, 40, 40, 13, 4
    x0 = _blob(B, 32, H, W, seed=2)
    s = _case_schedule(m, B, H, W, T, fire="philox", steps=[13, 6, 13], damage_step=8, seed=4)
    _check(m, x0, s, _target(x0), S, impl)


@pytest.mark.parametrize("impl", ["streaming", "auto"])
def test_metrics_large_problem_path(impl):
    """256x256x32, B = 16, 20 steps with damage: the balanced tensor-core update (k_update_tc), 16 blocks of
    k_frame_metrics per sample"""
    m = _random_graph(32, 256)
    B, H, W, T, S = 16, 256, 256, 20, 3
    x0 = _blob(B, 32, H, W, seed=3)
    s = _case_schedule(m, B, H, W, T, fire="philox", steps=[20] * 15 + [11], damage_step=9, seed=6,
                       philox_offset=99)
    _check(m, x0, s, _target(x0), S, impl)


def test_monitor_is_inference_only_under_grad():
    m = MODELS["torus"]()
    B, H, W, T = 2, 40, 40, 6
    x0 = _blob(B, 16, H, W, seed=1).requires_grad_(True)
    s = _case_schedule(m, B, H, W, T, seed=2)
    mon = monitor_rollout(m, x0, s, _target(x0.detach()), every=2)
    for v in (mon.loss, mon.psnr, mon.pixel_perfect, mon.alive, mon.x_T):
        assert not v.requires_grad and v.grad_fn is None
    with torch.no_grad():
        assert torch.equal(mon.x_T, rollout(m, x0, s))


def test_monitor_rejects_a_cpu_target():
    m = MODELS["torus"]()
    x0 = _blob(1, 16, 40, 40)
    s = _case_schedule(m, 1, 40, 40, 2)
    with pytest.raises(RuntimeError, match="target"):
        monitor_rollout(m, x0, s, _target(x0).cpu(), every=1)

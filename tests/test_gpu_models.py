"""GPU tests of the model-stacked rollouts: record_rollout / monitor_rollout over a list of same-architecture models
(gnca_rollout_record_models / gnca_rollout_metrics_models).

Model i's block of a stacked call is pinned bit for bit to the single-model call with model i on the whole stacked x0,
with the same schedule and impl: the same batch gives the same cluster configuration, so only the weights differ.
Models are three seeded perturbations of the golden ep960 / ep990 weights, built here."""
import random
import re

import pytest
import torch

from conftest import load_params, rel_err
from oracle import nca_oracle as O

pytestmark = pytest.mark.gpu

if torch.cuda.is_available():
    import graph_neural_cellular_automata_b200 as G
    from graph_neural_cellular_automata_b200 import _lib
    from graph_neural_cellular_automata_b200 import functional as GF
    from graph_neural_cellular_automata_b200.rollout import make_schedule, monitor_rollout, record_rollout
    from graph_neural_cellular_automata_b200.utils import metrics as UM

DEV = "cuda"


def _perturb(m, seed, scale=0.05):
    """model 0 keeps the golden weights; model i > 0 gets seeded relative noise on every weight tensor"""
    if seed == 0:
        return m
    g = torch.Generator().manual_seed(1000 + seed)
    with torch.no_grad():
        for name, p in m.named_parameters():
            if "perception" in name or not p.requires_grad:
                continue
            p.add_(scale * p.abs().mean() * torch.randn(p.shape, generator=g).to(p.device))
    return m


def _graph16(torus, seed):
    m = G.NeuralCAGraph(16, update_hidden=128, img_size=40, update_gain=0.05, alpha_thr=0.12, message_gain=0.25,
                        hidden_only=True, graph_zero_padded_shift=not torus)
    missing, unexpected = m.load_state_dict(load_params("weights_graph_ep960.npz"), strict=False)
    assert not missing and not unexpected
    return _perturb(m, seed).to(DEV)


def _classic16(seed):
    m = G.NeuralCA(16, update_hidden=128, img_size=40, update_gain=0.1, alpha_thr=0.1)
    missing, unexpected = m.load_state_dict(load_params("weights_classic_ep990.npz"), strict=False)
    assert not missing and not unexpected
    return _perturb(m, seed).to(DEV)


def _random_graph32(seed):
    torch.manual_seed(5); random.seed(5)
    m = G.NeuralCAGraph(32, update_hidden=128, img_size=40, update_gain=0.1, alpha_thr=0.1, message_gain=0.3,
                        hidden_only=True, graph_zero_padded_shift=False)
    with torch.no_grad():
        m.update_net[2].weight.normal_(0, 0.05)
        m.norm.weight.uniform_(0.5, 1.5); m.norm.bias.normal_(0, 0.1)
    return _perturb(m, seed, 0.2).to(DEV)


MODELS = {"torus": lambda s: _graph16(True, s), "zeropad": lambda s: _graph16(False, s), "classic": _classic16,
          "c32": _random_graph32}


def _blob(B, C_, H, W, seed=0):
    """random state inside a disk (alive cells with a dead border around them)"""
    g = torch.Generator().manual_seed(seed)
    yy, xx = torch.meshgrid(torch.arange(H), torch.arange(W), indexing="ij")
    disk = (((yy - H / 2) ** 2 + (xx - W / 2) ** 2) < (0.3 * min(H, W)) ** 2).float()
    return (torch.rand(B, C_, H, W, generator=g) * disk).to(DEV)


def _target(x0, seed=0):
    g = torch.Generator().manual_seed(seed)
    return (UM.premultiply(x0[:1])[0] + 0.03 * torch.randn(4, *x0.shape[2:], generator=g).to(DEV)).contiguous()


def _schedule(m, B, H, W, T, *, fire="u", steps=None, damage_step=None, seed=0, philox_offset=0):
    """per-step fire rates and gains (every third gain 0), recorded uniforms or in-kernel Philox, optional damage and
    ragged steps; built on model 0, as a stacked call is"""
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


def _check_stack(models, x0, s, tgt, S, impl):
    """stacked record + monitor against the single-model calls on the whole x0; returns False when the impl has no
    kernel for the configuration (both calls raise)"""
    M = len(models)
    Bt = x0.shape[0]
    B = Bt // M
    with torch.no_grad():
        try:
            single = [(record_rollout(m, x0, s, every=S, impl=impl), monitor_rollout(m, x0, s, tgt, every=S, impl=impl))
                      for m in models]
        except _lib.GncaError as e:
            assert "unsupported" in str(e)
            with pytest.raises(RuntimeError, match="unsupported"):
                record_rollout(models, x0, s, every=S, impl=impl)
            with pytest.raises(RuntimeError, match="unsupported"):
                monitor_rollout(models, x0, s, tgt, every=S, impl=impl)
            return False
        tr = record_rollout(models, x0, s, every=S, impl=impl)
        mon = monitor_rollout(models, x0, s, tgt, every=S, impl=impl)
        tr2 = record_rollout(models, x0, s, every=S, impl=impl)
        mon2 = monitor_rollout(models, x0, s, tgt, every=S, impl=impl)
    F = s.T // S + 1
    assert tr.t == mon.t == [f * S for f in range(F)]
    assert tr.states.shape == (F, Bt, *x0.shape[1:]) and tr.attention is None and mon.loss.shape == (F, Bt)
    # two stacked calls are bit-identical
    assert torch.equal(tr.states, tr2.states) and torch.equal(tr.x_T, tr2.x_T) and torch.equal(mon.x_T, mon2.x_T)
    for a, b in ((mon.loss, mon2.loss), (mon.psnr, mon2.psnr), (mon.pixel_perfect, mon2.pixel_perfect),
                 (mon.alive, mon2.alive)):
        assert torch.equal(a, b)
    for i, (rt, mt) in enumerate(single):
        blk = slice(i * B, (i + 1) * B)
        assert torch.equal(tr.states[:, blk], rt.states[:, blk]), i
        assert torch.equal(tr.x_T[blk], rt.x_T[blk]), i
        assert torch.equal(mon.x_T[blk], rt.x_T[blk]), i
        for a, b in ((mon.loss, mt.loss), (mon.psnr, mt.psnr), (mon.pixel_perfect, mt.pixel_perfect),
                     (mon.alive, mt.alive)):
            assert torch.equal(a[:, blk], b[:, blk]), i
    if s.T > 0:
        # the models differ on the same samples: a kernel that ignored the stride would fail the equalities above
        for i in range(1, M):
            blk = slice(i * B, (i + 1) * B)
            assert not torch.equal(single[i][0].x_T[blk], single[0][0].x_T[blk]), i
    for v in (tr.states, tr.x_T, mon.loss, mon.x_T):
        assert not v.requires_grad and v.grad_fn is None
    return True


# name: T, every, fire, ragged steps (per model, B = 2), damage step, philox offset
CASES = {
    "S1": (7, 1, "u", None, None, 0),
    "S3_T%S!=0": (10, 3, "u", None, None, 0),
    "T0": (0, 2, "u", None, None, 0),
    "ragged_philox_damage_at_frame": (10, 3, "philox", [10, 4], 6, 0),
    "ragged_u_damage_between_frames": (11, 3, "u", [5, 11], 4, 0),
    "philox_offset": (10, 3, "philox", [10, 7], 5, 123457),
}


@pytest.mark.parametrize("impl", ["resident", "banded"])
@pytest.mark.parametrize("model", ["torus", "zeropad", "classic"])
@pytest.mark.parametrize("case", list(CASES))
def test_stack_blocks_equal_single_model_calls(case, model, impl):
    T, S, fire, steps, dstep, poff = CASES[case]
    M, B, H, W = 3, 2, 40, 40
    models = [MODELS[model](i) for i in range(M)]
    x0 = _blob(M * B, 16, H, W, seed=1)
    s = _schedule(models[0], M * B, H, W, T, fire=fire, steps=steps * M if steps else None, damage_step=dstep, seed=3,
                  philox_offset=poff)
    ran = _check_stack(models, x0, s, _target(x0), S, impl)
    if not ran:
        # the banded kernel has no zero-padded shift; T = 0 launches no step and runs everywhere
        assert model == "zeropad" and impl == "banded" and T > 0


@pytest.mark.parametrize("impl", ["resident", "banded"])
def test_stack_c32(impl):
    """C = 32 runs on the banded kernel only (the replicated-state kernel is C = 16)"""
    M, B, H, W, T, S = 3, 2, 40, 40, 13, 4
    models = [MODELS["c32"](i) for i in range(M)]
    x0 = _blob(M * B, 32, H, W, seed=2)
    s = _schedule(models[0], M * B, H, W, T, fire="philox", steps=[13, 6] * M, damage_step=8, seed=4)
    assert _check_stack(models, x0, s, _target(x0), S, impl)


@pytest.mark.parametrize("impl", ["auto", "resident", "banded"])
def test_one_model_stack_equals_the_model(impl):
    m = MODELS["torus"](1)
    B, H, W, T, S = 4, 40, 40, 9, 2
    x0 = _blob(B, 16, H, W, seed=5)
    s = _schedule(m, B, H, W, T, fire="philox", steps=[9, 3, 9, 6], damage_step=4, seed=6)
    tgt = _target(x0)
    with torch.no_grad():
        a, b = record_rollout([m], x0, s, every=S, impl=impl), record_rollout(m, x0, s, every=S, impl=impl)
        c, d = monitor_rollout([m], x0, s, tgt, every=S, impl=impl), monitor_rollout(m, x0, s, tgt, every=S, impl=impl)
    assert torch.equal(a.states, b.states) and torch.equal(a.x_T, b.x_T) and torch.equal(c.x_T, d.x_T)
    for f in ("loss", "psnr", "pixel_perfect", "alive"):
        assert torch.equal(getattr(c, f), getattr(d, f)), f


def test_large_sweep_blocks(monkeypatch, capfd):
    """150 models at B = 1: 150 clusters of 8 one-CTA-per-SM CTAs do not fit 148 SMs at once, so the launch takes a
    smaller cluster (or a second wave); a few blocks against the same-B single-model call"""
    M, H, W, T, S = 150, 40, 40, 20, 5
    base = MODELS["torus"](0)
    models = [base] + [_perturb(_graph16(True, 0), i, 0.03) for i in range(1, M)]
    x0 = _blob(M, 16, H, W, seed=7)
    s = _schedule(base, M, H, W, T, fire="philox", damage_step=10, seed=8)
    tgt = _target(x0)
    monkeypatch.setenv("GNCA_DEBUG", "1")
    with torch.no_grad():
        mon = monitor_rollout(models, x0, s, tgt, every=S, impl="auto")
        tr = record_rollout(models, x0, s, every=S, impl="auto")
    err = capfd.readouterr().err
    nc = [int(v) for v in re.findall(r"replicated fwd: B=150 NC=(\d+)", err)]
    assert nc and all(v < 8 for v in nc), err[-500:]
    monkeypatch.delenv("GNCA_DEBUG")
    with torch.no_grad():
        for i in (0, 1, 77, 149):
            rt = record_rollout(models[i], x0, s, every=S, impl="auto")
            mt = monitor_rollout(models[i], x0, s, tgt, every=S, impl="auto")
            assert torch.equal(tr.states[:, i], rt.states[:, i]) and torch.equal(tr.x_T[i], rt.x_T[i]), i
            assert torch.equal(mon.x_T[i], rt.x_T[i]) and torch.equal(mon.pixel_perfect[:, i], mt.pixel_perfect[:, i])
            assert torch.equal(mon.loss[:, i], mt.loss[:, i]) and torch.equal(mon.alive[:, i], mt.alive[:, i])
    assert not torch.equal(tr.x_T[1], record_rollout(models[0], x0, s, every=S).x_T[1])


@pytest.mark.parametrize("impl", ["resident", "banded"])
def test_stack_member_against_fp64_oracle(impl):
    """model 1 of a three-model stack against the fp64 oracle with model 1's weights: x_T within the DESIGN section 4
    rollout bound (1e-5 rel-Frobenius), alive mask bit-exact"""
    M, B, H, W, T = 3, 2, 40, 40, 16
    models = [MODELS["torus"](i) for i in range(M)]
    x0 = _blob(M * B, 16, H, W, seed=9)
    random.seed(11)
    offs = [models[0].graph.draw_offsets() for _ in range(T)]
    fu = torch.rand(T, M * B, H, W, device=DEV, generator=torch.Generator(device=DEV).manual_seed(12))
    s = make_schedule(models[0], M * B, H, W, T, fire_rate=0.5, offsets=offs, fire_u=fu)
    with torch.no_grad():
        xT = record_rollout(models, x0, s, every=T, impl=impl).x_T
    blk = slice(B, 2 * B)
    p = {k: v.detach().cpu().double() for k, v in models[1].state_dict().items()}
    cfg = O.StepConfig(update_gain=0.05, alpha_thr=0.12, graph=True, message_gain=0.25, hidden_only=True,
                       zero_padded_shift=False)
    with torch.no_grad():
        ref = O.rollout(x0[blk].cpu().double(), p, cfg, [0.5] * T, [fu[t, blk].cpu().double().unsqueeze(1)
                                                                      for t in range(T)], offs)
    assert float((ref[:, 3] > 0.12).double().mean()) > 0.05          # a live pattern
    assert rel_err(xT[blk].cpu(), ref) < 1e-5, rel_err(xT[blk].cpu(), ref)
    assert torch.equal(GF.alive_mask(xT[blk], 0.12).cpu().bool(), O.alive_mask(ref, 0.12).bool())

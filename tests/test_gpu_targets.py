"""GPU tests of per-model targets: monitor_rollout over a model stack with a [M, 4, H, W] target
(gnca_rollout_metrics_targets), premult_loss with one target per block of samples (gnca_loss_premult_rgba_targets),
and PopulationTrainer with a target per model.

Model i's block of a per-model-target call is pinned bit for bit to block i of the stacked call with the shared target
targets[i]; equal targets are pinned to the [4, H, W] call.  The targets are seeded shifts, flips and noise of the
gecko surrogate in tests/golden."""
import os
import random

import numpy as np
import pytest
import torch

from conftest import GOLDEN, load_params, rel_err
from oracle import nca_oracle as O

pytestmark = pytest.mark.gpu

if torch.cuda.is_available():
    import graph_neural_cellular_automata_b200 as G
    from graph_neural_cellular_automata_b200 import _lib
    from graph_neural_cellular_automata_b200.rollout import make_schedule, monitor_rollout, record_rollout, rollout
    from graph_neural_cellular_automata_b200.training.population import PopulationTrainer
    from graph_neural_cellular_automata_b200.training.trainer import TrainConfig, premult_loss

DEV = "cuda"
QKS = ("query", "key", "scaling")


def _perturb(m, seed, scale=0.05):
    if seed == 0:
        return m
    g = torch.Generator().manual_seed(1000 + seed)
    with torch.no_grad():
        for name, p in m.named_parameters():
            if "perception" in name or not p.requires_grad:
                continue
            p.add_(scale * p.abs().mean() * torch.randn(p.shape, generator=g).to(p.device))
    return m


def _graph16(torus, seed=0):
    m = G.NeuralCAGraph(16, update_hidden=128, img_size=40, update_gain=0.05, alpha_thr=0.12, message_gain=0.25,
                        hidden_only=True, graph_zero_padded_shift=not torus)
    missing, unexpected = m.load_state_dict(load_params("weights_graph_ep960.npz"), strict=False)
    assert not missing and not unexpected
    return _perturb(m, seed).to(DEV)


def _classic16(seed=0):
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


def _targets(M, seed=0):
    """[M, 4, 40, 40]: target 0 is the gecko surrogate, the others seeded shifts and flips of it plus noise"""
    base = torch.from_numpy(np.load(os.path.join(GOLDEN, "target_gecko_surrogate.npy"))).float()
    g = torch.Generator().manual_seed(seed)
    out = [base]
    for i in range(1, M):
        t = torch.roll(base, shifts=(int(torch.randint(-5, 6, (1,), generator=g)),
                                     int(torch.randint(-5, 6, (1,), generator=g))), dims=(1, 2))
        if i % 2:
            t = t.flip(2)
        out.append((t + 0.05 * torch.randn(t.shape, generator=g)).clamp(0, 1))
    return torch.stack(out).to(DEV).contiguous()


def _blob(B, C_, H, W, seed=0):
    """random state inside a disk (alive cells with a dead border around them)"""
    g = torch.Generator().manual_seed(seed)
    yy, xx = torch.meshgrid(torch.arange(H), torch.arange(W), indexing="ij")
    disk = (((yy - H / 2) ** 2 + (xx - W / 2) ** 2) < (0.3 * min(H, W)) ** 2).float()
    return (torch.rand(B, C_, H, W, generator=g) * disk).to(DEV)


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


def _fields(mon):
    return [mon.loss, mon.psnr, mon.pixel_perfect, mon.alive] + ([mon.ssim] if mon.ssim is not None else [])


def _check_targets(models, x0, s, targets, S, impl, ssim):
    """per-model-target monitor against the shared-target stacked calls, block by block; False when the impl has no
    kernel for the configuration (every call raises)"""
    M = len(models)
    B = x0.shape[0] // M
    with torch.no_grad():
        try:
            shared = [monitor_rollout(models, x0, s, targets[i], every=S, impl=impl, ssim=ssim) for i in range(M)]
        except _lib.GncaError as e:
            assert "unsupported" in str(e)
            with pytest.raises(RuntimeError, match="unsupported"):
                monitor_rollout(models, x0, s, targets, every=S, impl=impl, ssim=ssim)
            return False
        mon = monitor_rollout(models, x0, s, targets, every=S, impl=impl, ssim=ssim)
        mon2 = monitor_rollout(models, x0, s, targets, every=S, impl=impl, ssim=ssim)
        xT = record_rollout(models, x0, s, every=S, impl=impl).x_T
    assert mon.t == shared[0].t and mon.loss.shape == (s.T // S + 1, M * B)
    for a, b in zip(_fields(mon) + [mon.x_T], _fields(mon2) + [mon2.x_T]):
        assert torch.equal(a, b)                                           # two calls, identical bits
    assert torch.equal(mon.x_T, xT)                                        # x_T of the call without metrics
    for i in range(M):
        blk = slice(i * B, (i + 1) * B)
        for a, b in zip(_fields(mon), _fields(shared[i])):
            assert torch.equal(a[:, blk], b[:, blk]), i
        assert torch.equal(mon.x_T[blk], shared[i].x_T[blk]), i
    # the targets differ: a kernel that ignored the per-model target would fail the block equalities above
    for i in range(1, M):
        blk = slice(i * B, (i + 1) * B)
        assert not torch.equal(shared[i].loss[:, blk], shared[0].loss[:, blk]), i
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


@pytest.mark.parametrize("ssim", [False, True])
@pytest.mark.parametrize("impl", ["auto", "resident", "banded"])
@pytest.mark.parametrize("model", ["torus", "zeropad", "classic"])
@pytest.mark.parametrize("case", list(CASES))
def test_monitor_blocks_equal_shared_target_calls(case, model, impl, ssim):
    T, S, fire, steps, dstep, poff = CASES[case]
    M, B, H, W = 3, 2, 40, 40
    models = [MODELS[model](i) for i in range(M)]
    x0 = _blob(M * B, 16, H, W, seed=1)
    s = _schedule(models[0], M * B, H, W, T, fire=fire, steps=steps * M if steps else None, damage_step=dstep, seed=3,
                  philox_offset=poff)
    ran = _check_targets(models, x0, s, _targets(M), S, impl, ssim)
    if not ran:
        # the banded kernel has no zero-padded shift; T = 0 launches no step and runs everywhere
        assert model == "zeropad" and impl == "banded" and T > 0


@pytest.mark.parametrize("ssim", [False, True])
def test_monitor_c32_banded(ssim):
    """C = 32 runs on the banded kernel only"""
    M, B, H, W, T, S = 3, 2, 40, 40, 13, 4
    models = [MODELS["c32"](i) for i in range(M)]
    x0 = _blob(M * B, 32, H, W, seed=2)
    s = _schedule(models[0], M * B, H, W, T, fire="philox", steps=[13, 6] * M, damage_step=8, seed=4)
    assert _check_targets(models, x0, s, _targets(M, seed=1), S, "banded", ssim)


@pytest.mark.parametrize("ssim", [False, True])
@pytest.mark.parametrize("impl", ["auto", "resident", "banded"])
@pytest.mark.parametrize("T", [0, 9])
def test_monitor_equal_targets_equal_shared_call(T, impl, ssim):
    """rows that are all one target give the [4, H, W] call's bits"""
    M, B, H, W, S = 3, 2, 40, 40, 3
    models = [MODELS["torus"](i) for i in range(M)]
    x0 = _blob(M * B, 16, H, W, seed=5)
    s = _schedule(models[0], M * B, H, W, T, fire="philox", steps=[9, 5] * M, damage_step=4 if T else None, seed=6)
    tgt = _targets(1, seed=2)[0]
    with torch.no_grad():
        a = monitor_rollout(models, x0, s, tgt, every=S, impl=impl, ssim=ssim)
        b = monitor_rollout(models, x0, s, tgt.expand(M, 4, H, W).contiguous(), every=S, impl=impl, ssim=ssim)
        xT = record_rollout(models, x0, s, every=S, impl=impl).x_T
    for u, v in zip(_fields(a) + [a.x_T], _fields(b) + [b.x_T]):
        assert torch.equal(u, v)
    assert torch.equal(b.x_T, xT)


def test_monitor_large_sweep():
    """148 models at B = 1 (one-CTA clusters), each against its own target: sampled blocks against the shared-target
    calls"""
    M, H, W, T, S = 148, 40, 40, 12, 4
    models = [_graph16(True, 0)] + [_perturb(_graph16(True, 0), i, 0.03) for i in range(1, M)]
    x0 = _blob(M, 16, H, W, seed=7)
    s = _schedule(models[0], M, H, W, T, fire="philox", damage_step=5, seed=8)
    targets = _targets(M, seed=3)
    with torch.no_grad():
        mon = monitor_rollout(models, x0, s, targets, every=S, ssim=True)
        for i in (0, 1, 77, 147):
            ref = monitor_rollout(models, x0, s, targets[i], every=S, ssim=True)
            for a, b in zip(_fields(mon), _fields(ref)):
                assert torch.equal(a[:, i], b[:, i]), i


@pytest.mark.parametrize("M,B", [(1, 4), (2, 4), (3, 6), (4, 8)])
def test_premult_loss_blocks(M, B):
    """[M, 4, H, W] against premult_loss block by block with target[i]: per-sample loss and gradient bit-equal"""
    x = _blob(B, 16, 40, 40, seed=11)
    targets = _targets(M, seed=4)
    per, gx = premult_loss(x, targets, 0.37)
    per_model = B // M
    for i in range(M):
        blk = slice(i * per_model, (i + 1) * per_model)
        p_i, g_i = premult_loss(x[blk].contiguous(), targets[i], 0.37)
        assert torch.equal(per[blk], p_i) and torch.equal(gx[blk], g_i), i
    p0, _ = premult_loss(x, targets, 0.37, want_grad=False)
    assert torch.equal(p0, per)
    one = targets[:1]
    assert all(torch.equal(u, v) for u, v in zip(premult_loss(x, one, 0.5), premult_loss(x, one[0], 0.5)))


# ---- PopulationTrainer ----------------------------------------------------------------------------------------------
def _cfg(**kw):
    base = dict(batch_size=4, pool_size=12, nca_steps_min=6, nca_steps_max=12, long_rollout_prob=0.0,
                fire_rate_min=0.5, fire_rate_max=0.9, learning_rate=2e-3, weight_decay=1e-5, reset_worst_prob=0.25,
                random_reseed_prob=0.5, message_gain=0.25, message_every=3, fire="philox", rollout_impl="auto",
                damage={"start_epoch": 0, "prob": 0.7, "kinds": {"circle": 1.0}, "size_min": 4, "size_max": 8})
    base.update(kw)
    return TrainConfig(**base)


def _grow(pool, m):
    with torch.no_grad():
        x = pool.pool
        for _ in range(16):
            x = m(x, fire_rate=0.7)
        pool.pool.copy_(x)


def _train(targets, seeds=(1, 2, 3), iters=3):
    torch.manual_seed(31); random.seed(31); torch.cuda.manual_seed(31)
    models = [_graph16(True, s_) for s_ in seeds]
    tr = PopulationTrainer(models, targets, _cfg())
    for pool in tr.pools:
        _grow(pool, models[0])
    outs = []
    for ep in range(1, iters + 1):
        last = tr.train_step(ep)
        outs.append({"per": last["per_sample"].clone(), "x_T": last["x_T"].clone(), "steps": np.array(last["steps"])})
    return tr, outs, random.getstate()


def test_trainer_equal_targets_equal_shared_target():
    """[M, 4, H, W] with equal rows: bit-identical to the [4, H, W] trainer over three iterations"""
    tgt = _targets(1)[0]
    a, oa, ra = _train(tgt)
    b, ob, rb = _train(tgt.expand(3, 4, 40, 40).contiguous())
    assert ra == rb
    for x, y in zip(oa, ob):
        assert torch.equal(x["per"], y["per"]) and torch.equal(x["x_T"], y["x_T"])
        assert np.array_equal(x["steps"], y["steps"])
    for i in range(3):
        for f in ("flat", "exp_avg", "exp_avg_sq"):
            assert torch.equal(getattr(a.opts[i], f), getattr(b.opts[i], f)), (i, f)
        assert torch.equal(a.pools[i].pool, b.pools[i].pool), i


def test_trainer_per_model_targets():
    """each model's losses are premult_loss of its x_T block against its own target; changing model 1's target leaves
    model 0's trajectory bit-identical"""
    targets = _targets(3, seed=5)
    a, oa, _ = _train(targets)
    B = 4
    for o in oa:
        for i in range(3):
            blk = slice(i * B, (i + 1) * B)
            per, _ = premult_loss(o["x_T"][blk].contiguous(), targets[i], 1.0, want_grad=False)
            assert torch.equal(o["per"][i], per), i
    other = targets.clone()
    other[1] = _targets(2, seed=9)[1]
    b, ob, _ = _train(other)
    for x, y in zip(oa, ob):
        assert torch.equal(x["per"][0], y["per"][0])
        assert not torch.equal(x["per"][1], y["per"][1])
    for f in ("flat", "exp_avg", "exp_avg_sq"):
        assert torch.equal(getattr(a.opts[0], f), getattr(b.opts[0], f)), f
    assert torch.equal(a.pools[0].pool, b.pools[0].pool)
    assert not torch.equal(a.opts[1].flat, b.opts[1].flat)


@pytest.mark.parametrize("model", ["torus", "zeropad"])
def test_member_gradient_against_fp64_oracle(model):
    """model 1 of a three-model stack trained towards its own target (the trainer's loss: premult_loss with per-model
    targets at scale 1/B, then the stacked BPTT) against fp64 oracle autograd with model 1's weights and target 1
    (DESIGN section 4 tolerances)"""
    M, B, H, W, T = 3, 2, 40, 40, 12
    models = [MODELS[model](i) for i in range(M)]
    m = models[1]
    targets = _targets(M, seed=6)
    x0 = _blob(M * B, 16, H, W, seed=9)
    random.seed(11)
    offs = [models[0].graph.draw_offsets() for _ in range(T)]
    frs = [0.5 + 0.1 * (t % 4) for t in range(T)]
    gains = [0.0 if t % 4 == 2 else 0.25 for t in range(T)]
    fu = torch.rand(T, M * B, H, W, device=DEV, generator=torch.Generator(device=DEV).manual_seed(12))
    s = make_schedule(models[0], M * B, H, W, T, fire_rate=frs, offsets=offs, fire_u=fu, message_gains=gains)
    blk = slice(B, 2 * B)
    for q in models:
        q.zero_grad(set_to_none=True)
    x = x0.clone().requires_grad_(True)
    out = rollout(models, x, s)
    per, gx = premult_loss(out.detach(), targets, 1.0 / B)
    out.backward(gx)
    p = {k: v.detach().cpu().double().requires_grad_(v.is_floating_point() and "perception" not in k)
         for k, v in m.state_dict().items()}
    xr = x0[blk].detach().cpu().double().requires_grad_(True)
    ref = xr
    for t in range(T):
        c = O.StepConfig(update_gain=0.05, alpha_thr=0.12, graph=True, message_gain=gains[t], hidden_only=True,
                         zero_padded_shift=model == "zeropad")
        ref = O.nca_step(ref, p, c, frs[t], fu[t, blk].cpu().double().unsqueeze(1), offs[t])
    tgt = targets[1].cpu().double()
    rgb, a = ref[:, :3], ref[:, 3:4]
    loss_b = (torch.cat([rgb * a, a], 1) - tgt).pow(2).mean(dim=(1, 2, 3))
    (loss_b.sum() / B).backward()
    assert float((ref[:, 3] > 0.12).double().mean()) > 0.05          # a live pattern
    assert rel_err(per[blk].cpu(), loss_b.detach()) < 1e-5
    assert rel_err(x.grad[blk].cpu(), xr.grad) < 1e-4, rel_err(x.grad[blk].cpu(), xr.grad)
    for n, q in m.named_parameters():
        gr = p[n].grad
        ours = q.grad.cpu() if q.grad is not None else torch.zeros_like(q.detach().cpu())
        if gr is None or float(gr.abs().max()) < 1e-12:
            assert float(ours.abs().max()) <= 1e-7, n
        elif any(k in n for k in QKS):
            if model == "torus":
                assert float(ours.abs().max()) <= 1e-7, n
            else:
                assert rel_err(ours, gr) < 1e-3 or float((ours - gr.double()).abs().max()) <= 1e-11, n
        else:
            assert rel_err(ours, gr) < 1e-4, (n, rel_err(ours, gr))

"""GPU tests of training a stack of models: rollout(models, ...) with grad (gnca_rollout_fwd_bptt_models /
gnca_rollout_bwd_bptt_models and their _zp forms) and the PopulationTrainer.

Model i's block of a stacked call is pinned to the single-model call of model i on the whole stacked x0, with the same
schedule and dL/dx_T zero outside block i: the same batch gives the same cluster configuration, so x_T and dL/dx0 of the
block are bit-equal; the parameter gradients differ only in the summation order of the weight-gradient pass (the
single-model call sums the records of all M*B samples, most of them zero).  Models are seeded perturbations of the
golden ep960 / ep990 weights, built here."""
import random
import re

import numpy as np
import pytest
import torch

from conftest import load_params, rel_err
from oracle import nca_oracle as O

pytestmark = pytest.mark.gpu

if torch.cuda.is_available():
    import graph_neural_cellular_automata_b200 as G
    from graph_neural_cellular_automata_b200.rollout import make_schedule, record_rollout, rollout
    from graph_neural_cellular_automata_b200.training.population import PopulationTrainer
    from graph_neural_cellular_automata_b200.training.trainer import GraphNCATrainer, TrainConfig, premult_loss
    from graph_neural_cellular_automata_b200.utils import metrics as UM

DEV = "cuda"
PARAM_TOL = 1e-5          # parameter gradients: max |stack - single| <= PARAM_TOL * max |single|, per tensor
QKS = ("query_proj", "key_proj", "scaling")


def _perturb(m, seed, scale=0.05):
    """seed 0 keeps the golden weights; seed i > 0 adds seeded relative noise to every trained weight tensor"""
    if seed:
        g = torch.Generator().manual_seed(1000 + seed)
        with torch.no_grad():
            for name, p in m.named_parameters():
                if "perception" not in name and p.requires_grad:
                    p.add_(scale * p.abs().mean() * torch.randn(p.shape, generator=g).to(p.device))
    return m


def _graph16(torus, seed, scale=0.05):
    m = G.NeuralCAGraph(16, update_hidden=128, img_size=40, update_gain=0.05, alpha_thr=0.12, message_gain=0.25,
                        hidden_only=True, graph_zero_padded_shift=not torus)
    missing, unexpected = m.load_state_dict(load_params("weights_graph_ep960.npz"), strict=False)
    assert not missing and not unexpected
    return _perturb(m, seed, scale).to(DEV)


def _classic16(seed, scale=0.05):
    m = G.NeuralCA(16, update_hidden=128, img_size=40, update_gain=0.1, alpha_thr=0.1)
    missing, unexpected = m.load_state_dict(load_params("weights_classic_ep990.npz"), strict=False)
    assert not missing and not unexpected
    return _perturb(m, seed, scale).to(DEV)


MODELS = {"torus": lambda s: _graph16(True, s), "zeropad": lambda s: _graph16(False, s), "classic": _classic16}


def _blob(B, H, W, seed=0):
    """random state inside a disk (alive cells with a dead border around them)"""
    g = torch.Generator().manual_seed(seed)
    yy, xx = torch.meshgrid(torch.arange(H), torch.arange(W), indexing="ij")
    disk = (((yy - H / 2) ** 2 + (xx - W / 2) ** 2) < (0.3 * min(H, W)) ** 2).float()
    return (torch.rand(B, 16, H, W, generator=g) * disk).to(DEV)


def _schedule(m, B, H, W, T, *, fire="u", steps=None, damage_step=None, seed=0, philox_offset=0):
    """per-step fire rates, every third message gain 0, recorded uniforms or in-kernel Philox, optional damage and
    ragged steps; built on model 0, as a stacked call is"""
    random.seed(seed)
    graph = getattr(m, "_is_graph", False)
    offs = [m.graph.draw_offsets() for _ in range(T)] if graph else None
    frs = [0.5 + 0.4 * ((7 * t) % 10) / 10 for t in range(T)]
    gains = [0.25 if t % 3 != 1 else 0.0 for t in range(T)] if graph else None
    fu = torch.rand(T, B, H, W, device=DEV, generator=torch.Generator(device=DEV).manual_seed(seed + 1)) \
        if fire == "u" else None
    dmg = None
    if damage_step is not None:
        dmg = torch.ones(B, 16, H, W, device=DEV)
        dmg[:, :, H // 3:H // 3 + H // 4, W // 4:W // 2] = 0.0
        dmg[0, :, H // 2:H // 2 + 3, :] = 0.5
    s = make_schedule(m, B, H, W, T, fire_rate=frs, offsets=offs, fire_u=fu, message_gains=gains, steps=steps,
                      fire="philox", seed=seed + 7, damage=dmg, damage_step=damage_step or 0)
    s.philox_offset = philox_offset
    return s


def _grads(m):
    return {n: (p.grad.clone() if p.grad is not None else torch.zeros_like(p)) for n, p in m.named_parameters()
            if p.requires_grad}


def _run(model, x0, s, gT):
    """(x_T, dL/dx0, {model index: parameter gradients}) of L = sum(x_T * gT) through rollout()"""
    models = model if isinstance(model, list) else [model]
    for m in models:
        m.zero_grad(set_to_none=True)
    x = x0.clone().requires_grad_(True)
    xT = rollout(model, x, s)
    (xT * gT).sum().backward()
    return xT.detach(), x.grad, [_grads(m) for m in models]


def _param_err(a, b):
    """largest per-tensor max |a - b| / max |b| (0 when both are exactly zero)"""
    worst = 0.0
    for n in b:
        scale = float(b[n].abs().max())
        d = float((a[n] - b[n]).abs().max())
        if scale == 0.0:
            assert d == 0.0, n
        else:
            worst = max(worst, d / scale)
    return worst


def _check_blocks(models, x0, s, gT, members):
    """stacked call vs the single-model calls of `members` on the whole batch; returns the largest parameter error"""
    M, B = len(models), x0.shape[0] // len(models)
    xT, g0, gp = _run(models, x0, s, gT)
    worst = 0.0
    for i in members:
        blk = slice(i * B, (i + 1) * B)
        gi = torch.zeros_like(gT)
        gi[blk] = gT[blk]
        xs, g0s, gps = _run(models[i], x0, s, gi)
        assert torch.equal(xT[blk], xs[blk]), i
        assert torch.equal(g0[blk], g0s[blk]), i
        err = _param_err(gp[i], gps[0])
        assert err <= PARAM_TOL, (i, err)
        worst = max(worst, err)
    return xT, g0, gp, worst


# name: T, fire, ragged steps (per model, B = 4), damage step, philox offset
CASES = {
    "damage": (16, "u", None, 6, 0),
    "ragged": (18, "u", [18, 5, 11, 1], None, 0),
    "philox_offset": (14, "philox", [14, 9, 14, 3], 7, 123457),
    "recorded_u": (24, "u", None, None, 0),
    "T0": (0, "u", None, None, 0),
}


@pytest.mark.parametrize("model", list(MODELS))
@pytest.mark.parametrize("case", list(CASES))
def test_stack_blocks_equal_single_model_calls(case, model):
    """every case has gain-0 steps (every third step of a graph model)"""
    T, fire, steps, dstep, poff = CASES[case]
    M, B, H, W = 3, 4, 40, 40
    models = [MODELS[model](i) for i in range(M)]
    x0 = _blob(M * B, H, W, seed=1)
    s = _schedule(models[0], M * B, H, W, T, fire=fire, steps=steps * M if steps else None, damage_step=dstep, seed=3,
                  philox_offset=poff)
    gT = torch.randn(M * B, 16, H, W, device=DEV, generator=torch.Generator(device=DEV).manual_seed(5))
    xT, g0, gp, worst = _check_blocks(models, x0, s, gT, range(M))
    print(f"[population] {model} {case}: max parameter-gradient error {worst:.3g} of the per-tensor max")
    if T > 0:
        # the models differ on the same samples: a kernel that ignored the stack would fail the equalities above
        assert not torch.equal(xT[:B], xT[B:2 * B]) or not torch.equal(g0[:B], g0[B:2 * B])
        assert _param_err(gp[1], gp[0]) > 1e-3
    else:
        assert torch.equal(xT, x0) and torch.equal(g0, gT)


@pytest.mark.parametrize("model", list(MODELS))
def test_one_model_stack_equals_the_model(model):
    m = MODELS[model](1)
    B, H, W, T = 4, 40, 40, 12
    x0 = _blob(B, H, W, seed=5)
    s = _schedule(m, B, H, W, T, fire="philox", steps=[12, 3, 12, 7], damage_step=4, seed=6)
    gT = torch.randn(B, 16, H, W, device=DEV, generator=torch.Generator(device=DEV).manual_seed(7))
    xa, ga, pa = _run([m], x0, s, gT)
    xb, gb, pb = _run(m, x0, s, gT)
    assert torch.equal(xa, xb) and torch.equal(ga, gb)
    for n in pb[0]:
        assert torch.equal(pa[0][n], pb[0][n]), n
    with torch.no_grad():
        assert torch.equal(rollout([m], x0, s), record_rollout([m], x0, s, every=T).x_T)


@pytest.mark.parametrize("model", ["torus", "zeropad"])
def test_isolation_and_repeatability(model):
    """perturbing model 2 leaves model 0's block and gradients bit-identical; two stacked calls are bit-identical"""
    M, B, H, W, T = 3, 4, 40, 40, 14
    models = [MODELS[model](i) for i in range(M)]
    x0 = _blob(M * B, H, W, seed=2)
    s = _schedule(models[0], M * B, H, W, T, fire="philox", damage_step=5, seed=4)
    gT = torch.randn(M * B, 16, H, W, device=DEV, generator=torch.Generator(device=DEV).manual_seed(8))
    a = _run(models, x0, s, gT)
    b = _run(models, x0, s, gT)
    assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])
    for i in range(M):
        for n in a[2][i]:
            assert torch.equal(a[2][i][n], b[2][i][n]), (i, n)
    other = [models[0], models[1], _perturb(MODELS[model](0), 9, 0.3)]
    c = _run(other, x0, s, gT)
    assert torch.equal(a[0][:B], c[0][:B]) and torch.equal(a[1][:B], c[1][:B])
    for n in a[2][0]:
        assert torch.equal(a[2][0][n], c[2][0][n]), n
    assert not torch.equal(a[0][2 * B:], c[0][2 * B:])
    with torch.no_grad():
        assert torch.equal(rollout(models, x0, s), record_rollout(models, x0, s, every=T).x_T)


@pytest.mark.parametrize("model", ["torus", "zeropad"])
def test_stack_member_against_fp64_oracle(model):
    """model 1 of a three-model stack against fp64 oracle autograd with model 1's weights (DESIGN section 4: dL/dx0 and
    parameter gradients 1e-4; query / key / scaling 1e-3 under the zero-padded shift, ~0 on the torus)"""
    M, B, H, W, T = 3, 2, 40, 40, 12
    models = [MODELS[model](i) for i in range(M)]
    m = models[1]
    x0 = _blob(M * B, H, W, seed=9)
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
    (out[blk, :4] ** 2).mean().backward()
    p = {k: v.detach().cpu().double().requires_grad_(v.is_floating_point() and "perception" not in k)
         for k, v in m.state_dict().items()}
    xr = x0[blk].detach().cpu().double().requires_grad_(True)
    ref = xr
    for t in range(T):
        c = O.StepConfig(update_gain=0.05, alpha_thr=0.12, graph=True, message_gain=gains[t], hidden_only=True,
                         zero_padded_shift=model == "zeropad")
        ref = O.nca_step(ref, p, c, frs[t], fu[t, blk].cpu().double().unsqueeze(1), offs[t])
    (ref[:, :4] ** 2).mean().backward()
    assert float((ref[:, 3] > 0.12).double().mean()) > 0.05          # a live pattern
    assert rel_err(out[blk].detach().cpu(), ref.detach()) < 1e-5
    assert rel_err(x.grad[blk].cpu(), xr.grad) < 1e-4, rel_err(x.grad[blk].cpu(), xr.grad)
    assert float(x.grad[:B].abs().max()) == 0.0 and float(x.grad[2 * B:].abs().max()) == 0.0
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
    for q in (models[0], models[2]):              # the loss does not reach the other models
        for n, v in q.named_parameters():
            assert v.grad is None or float(v.grad.abs().max()) == 0.0, n


def test_many_models(monkeypatch, capfd):
    """150 models at B = 1: 150 one-CTA clusters of the backward (more than 148 SMs' worth of 2-CTA clusters); two
    sampled members against their single-model calls"""
    M, H, W, T = 150, 40, 40, 8
    models = [_graph16(True, 0)] + [_graph16(True, i, 0.03) for i in range(1, M)]
    x0 = _blob(M, H, W, seed=7)
    s = _schedule(models[0], M, H, W, T, fire="philox", damage_step=3, seed=8)
    gT = torch.randn(M, 16, H, W, device=DEV, generator=torch.Generator(device=DEV).manual_seed(9))
    monkeypatch.setenv("GNCA_DEBUG", "1")
    capfd.readouterr()
    _run(models, x0, s, gT)
    err = capfd.readouterr().err
    nc = [int(v) for v in re.findall(r"resident bwd: B=150 NC=(\d+)", err)]
    assert nc == [1], err[-500:]
    monkeypatch.delenv("GNCA_DEBUG")
    _check_blocks(models, x0, s, gT, (1, 148))


# ---- PopulationTrainer ----------------------------------------------------------------------------------------------
def _cfg(**kw):
    base = dict(batch_size=4, pool_size=12, nca_steps_min=6, nca_steps_max=12, long_rollout_prob=0.0,
                fire_rate_min=0.5, fire_rate_max=0.9, learning_rate=2e-3, weight_decay=1e-5, reset_worst_prob=0.25,
                random_reseed_prob=0.5, message_gain=0.25, message_every=3, fire="philox", rollout_impl="auto",
                damage={"start_epoch": 0, "prob": 0.7, "kinds": {"circle": 1.0}, "size_min": 4, "size_max": 8})
    base.update(kw)
    return TrainConfig(**base)


def _target():
    return (UM.premultiply(_blob(1, 40, 40, seed=3))[0]).contiguous()


def _grow(pool, m):
    with torch.no_grad():
        x = pool.pool
        for _ in range(16):
            x = m(x, fire_rate=0.7)
        pool.pool.copy_(x)


def test_trainer_one_model_equals_graph_trainer():
    """M = 1 consumes the host RNG as GraphNCATrainer(fire="philox") does and gives bit-identical parameters, Adam
    moments, per-sample losses and pool over three iterations"""
    runs = []
    for cls in (GraphNCATrainer, PopulationTrainer):
        torch.manual_seed(21); random.seed(21); torch.cuda.manual_seed(21)
        m = _graph16(True, 1)
        tr = cls([m] if cls is PopulationTrainer else m, _target(), _cfg())
        _grow(tr.pool, m)
        out = []
        for ep in (1, 2, 3):
            last = tr.train_step(ep)
            out.append((last["per_sample"].reshape(-1).clone(), np.array(last["steps"])))
        runs.append((tr, out, random.getstate()))
    (a, oa, ra), (b, ob, rb) = runs
    assert ra == rb                                          # the same host RNG consumption
    for (la, sa), (lb, sb) in zip(oa, ob):
        assert torch.equal(la, lb) and np.array_equal(sa, sb)
    for f in ("flat", "exp_avg", "exp_avg_sq"):
        assert torch.equal(getattr(a.opt, f), getattr(b.opts[0], f)), f
    assert torch.equal(a.pool.pool, b.pools[0].pool)


def test_trainer_three_models():
    """model 0's trajectory does not depend on models 1 and 2; losses are premult_loss of the stacked x_T; a model at
    learning rate 0 keeps its weights"""
    def run(seeds, lrs):
        torch.manual_seed(31); random.seed(31); torch.cuda.manual_seed(31)
        models = [_graph16(True, s_) for s_ in seeds]
        tr = PopulationTrainer(models, _target(), _cfg(), learning_rates=lrs)
        for pool, m in zip(tr.pools, models):
            _grow(pool, models[0])
        w0 = [o.flat.clone() for o in tr.opts]
        outs = []
        for ep in (1, 2):
            last = tr.train_step(ep)
            per, _ = premult_loss(last["x_T"], tr.target, 1.0, want_grad=False)
            assert torch.equal(last["per_sample"].reshape(-1), per)
            assert torch.equal(last["loss"], last["per_sample"].mean(1))
            outs.append(last["per_sample"][0].clone())
        return tr, w0, outs

    a, wa, oa = run([1, 2, 3], [2e-3, 0.0, 1e-3])
    b, wb, ob = run([1, 5, 6], [2e-3, 1e-3, 0.0])
    for x, y in zip(oa, ob):
        assert torch.equal(x, y)
    assert torch.equal(a.opts[0].flat, b.opts[0].flat) and torch.equal(a.opts[0].exp_avg, b.opts[0].exp_avg)
    assert torch.equal(a.pools[0].pool, b.pools[0].pool)
    assert torch.equal(a.opts[1].flat, wa[1]) and torch.equal(b.opts[2].flat, wb[2])     # learning rate 0
    assert not torch.equal(a.opts[2].flat, wa[2]) and not torch.equal(a.opts[0].flat, wa[0])

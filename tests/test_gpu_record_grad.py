"""GPU tests of differentiable frames: record_rollout(..., differentiable=True), one fused BPTT for losses on the strided
frames x_{f*S} and on x_T.

1. gradients against autograd through T fp64 oracle steps (the same offsets, uniforms, fire rates, gains, step counts
   and damage) on every impl, with a distinct weight per frame so that a frame mix-up shows;
2. truncation identity: a loss on frame f alone gives the gradients of rollout() over the first f*S steps;
3. neutral extension: an all-zero frame gradient, or a loss on x_T alone, gives the plain BPTT bit for bit;
4. plumbing of the autograd node; 5. the training shape, C = 32 and the large-problem path."""
import ctypes as C
import random

import pytest
import torch

from conftest import load_params, rel_err
from oracle import nca_oracle as O

pytestmark = pytest.mark.gpu

if torch.cuda.is_available():
    import graph_neural_cellular_automata_b200 as G
    from graph_neural_cellular_automata_b200 import _lib
    from graph_neural_cellular_automata_b200 import functional as GF
    from graph_neural_cellular_automata_b200.rollout import (IMPL, make_schedule, record_rollout, rollout,
                                                             rollout_bwd_raw, rollout_fwd_raw)

DEV = "cuda"
IMPLS = ["streaming", "resident", "banded"]
QKS = ("query_proj", "key_proj", "scaling")


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
    """random state inside a disk (alive cells with a dead border around them), on the host"""
    g = torch.Generator().manual_seed(seed)
    yy, xx = torch.meshgrid(torch.arange(H), torch.arange(W), indexing="ij")
    disk = (((yy - H / 2) ** 2 + (xx - W / 2) ** 2) < (0.3 * min(H, W)) ** 2).float()
    return torch.rand(B, C_, H, W, generator=g) * disk


def _draws(m, B, H, W, T, *, steps=None, damage_step=None, seed=0):
    """the schedule's random draws on the host: offsets, uniforms, per-step fire rates and gains (some 0), damage"""
    random.seed(seed)
    graph = getattr(m, "_is_graph", False)
    d = dict(offs=[m.graph.draw_offsets() for _ in range(T)] if graph else None,
             frs=[0.5 + 0.4 * ((7 * t) % 10) / 10 for t in range(T)],
             gains=[0.25 if t % 3 != 1 else 0.0 for t in range(T)] if graph else None,
             fu=torch.rand(T, B, H, W, generator=torch.Generator().manual_seed(seed + 1)),
             steps=steps, dmg=None, dmg_step=damage_step)
    if damage_step is not None:
        dmg = torch.ones(B, m.n_channels, H, W)
        dmg[:, :, H // 3:H // 3 + H // 4, W // 4:W // 2] = 0.0
        dmg[0, :, H // 2:H // 2 + 3, :] = 0.5
        d["dmg"] = dmg
    return d


def _schedule(m, B, H, W, T, d):
    return make_schedule(m, B, H, W, T, fire_rate=d["frs"], offsets=d["offs"], fire_u=d["fu"].to(DEV),
                         message_gains=d["gains"], steps=d["steps"],
                         damage=d["dmg"].to(DEV) if d["dmg"] is not None else None, damage_step=d["dmg_step"] or 0)


def _ell(x):
    return (x[:, :4] ** 2).mean() + 0.1 * x[:, 4:].mean()


def _weights(F):
    return [1.0 + 0.37 * f for f in range(F)]


def _frame_loss(states, xT):
    """sum_f w_f ell(frame f) + ell(x_T), distinct w_f"""
    w = _weights(states.shape[0])
    return sum(w[f] * _ell(states[f]) for f in range(states.shape[0])) + _ell(xT)


def _step_cfg(m, gain):
    g = getattr(m, "graph", None)
    return O.StepConfig(update_gain=m.update_gain, alpha_thr=m.alpha_thr, graph=g is not None, message_gain=gain,
                        hidden_only=True if g is not None else False,
                        zero_padded_shift=bool(g.zero_padded_shift) if g is not None else False)


def _oracle(m, x0, T, S, d):
    """fp64 autograd through T oracle steps; frame f = x_{f*S} after the damage of its step, frozen samples kept.
    Returns (x0 leaf, params, frames, x_T) after backward of `_frame_loss`."""
    B = x0.shape[0]
    p = {k: v.detach().cpu().double().requires_grad_(v.is_floating_point() and "perception" not in k)
         for k, v in m.state_dict().items()}
    xr = x0.double().requires_grad_(True)
    x, xs = xr, []
    st = torch.tensor(d["steps"]) if d["steps"] is not None else None
    for t in range(T):
        if d["dmg"] is not None and t == d["dmg_step"]:
            x = x * d["dmg"].double()
        xs.append(x)
        mask = st > t if st is not None else torch.ones(B, dtype=torch.bool)
        if not bool(mask.any()):
            continue
        gain = d["gains"][t] if d["gains"] is not None else 0.0
        chosen = d["offs"][t] if d["offs"] is not None else ()
        new = O.nca_step(x[mask], p, _step_cfg(m, gain), d["frs"][t], d["fu"][t][mask].unsqueeze(1).double(), chosen)
        x = x.clone()
        x[mask] = new
    xs.append(x)
    frames = torch.stack([xs[f * S] for f in range(T // S + 1)])
    _frame_loss(frames, x).backward()
    return xr, p, frames, x


def _check_grads(m, xg, xr, p, *, xtol=5e-4):
    """the tolerances of test_gpu_hparams.check_rollout"""
    B = xg.shape[0]
    per = sorted(rel_err(xg.grad[b].cpu(), xr.grad[b]) for b in range(B))
    assert per[B // 2] <= 1e-5, per
    assert rel_err(xg.grad.cpu(), xr.grad) <= xtol, rel_err(xg.grad.cpu(), xr.grad)
    torus = getattr(m, "_is_graph", False) and not m.graph.zero_padded_shift
    for n, q in m.named_parameters():
        gr = p[n].grad
        ours = q.grad.cpu() if q.grad is not None else torch.zeros_like(q.detach().cpu())
        if gr is None or float(gr.abs().max()) < 1e-12:
            assert float(ours.abs().max()) <= 1e-7, n
        elif any(s in n for s in QKS):
            if torus:
                assert float(ours.abs().max()) <= 1e-7, n
            else:
                assert rel_err(ours, gr) < 1e-3, (n, rel_err(ours, gr))
        else:
            assert rel_err(ours, gr) < 1e-4, (n, rel_err(ours, gr))


def _param_grads(m):
    """every parameter's gradient; zeros for the ones the step never reads (their .grad stays None)"""
    return [q.grad.clone() if q.grad is not None else torch.zeros_like(q) for q in m.parameters()]


def _zero_grads(m):
    for q in m.parameters():
        q.grad = None


def _supported_or_skip(m, x0, s, impl):
    """a combination the plain rollout rejects is rejected the same way by the differentiable recording, then skipped"""
    try:
        with torch.no_grad():
            rollout(m, x0, s, impl=impl)
    except _lib.GncaError as e:
        assert "unsupported" in str(e)
        with pytest.raises(_lib.GncaError, match="unsupported"):
            record_rollout(m, x0.clone().requires_grad_(True), s, every=1, impl=impl, differentiable=True)
        pytest.skip(f"{impl}: no kernel for this configuration")


# name: T, every, ragged steps, damage step
CASES = {
    "S1": (7, 1, None, None),
    "S3_T%S!=0": (10, 3, None, None),
    "S=T": (9, 9, None, None),
    "S=T+1": (9, 10, None, None),
    "T0": (0, 1, None, None),
    "ragged_damage_at_frame": (10, 3, [10, 4], 6),
    "ragged_damage_between_frames": (11, 3, [5, 11], 4),
    "damage_at_frame_S2": (8, 2, None, 2),
}


# ---- 1. against the fp64 oracle ------------------------------------------------------------------------------------
@pytest.mark.parametrize("impl", IMPLS)
@pytest.mark.parametrize("model", list(MODELS))
@pytest.mark.parametrize("case", list(CASES))
def test_frame_gradients_vs_oracle(case, model, impl):
    T, S, steps, dstep = CASES[case]
    m = MODELS[model]()
    B, H, W = 2, 40, 40
    x0 = _blob(B, 16, H, W, seed=1)
    d = _draws(m, B, H, W, T, steps=steps, damage_step=dstep, seed=3)
    s = _schedule(m, B, H, W, T, d)
    _supported_or_skip(m, x0.to(DEV), s, impl)
    xr, p, frames_ref, xT_ref = _oracle(m, x0, T, S, d)
    _zero_grads(m)
    xg = x0.to(DEV).requires_grad_(True)
    tr = record_rollout(m, xg, s, every=S, impl=impl, differentiable=True)
    assert tr.t == [f * S for f in range(T // S + 1)]
    assert tr.states.requires_grad and tr.x_T.requires_grad and tr.states.grad_fn is tr.x_T.grad_fn
    assert rel_err(tr.states.detach().cpu(), frames_ref.detach()) < 1e-5
    assert rel_err(tr.x_T.detach().cpu(), xT_ref.detach()) < 1e-5
    _frame_loss(tr.states, tr.x_T).backward()
    _check_grads(m, xg, xr, p)


# ---- 2. truncation identity ----------------------------------------------------------------------------------------
@pytest.mark.parametrize("impl", ["streaming", "resident"])
@pytest.mark.parametrize("T,S,f", [(10, 3, 1), (10, 3, 2), (9, 3, 3)])
def test_loss_on_one_frame_equals_truncated_rollout(T, S, f, impl):
    """A loss on frame f alone has the gradients of rollout() over the first f*S steps with a loss on its x_T.
    In-kernel Philox uniforms, ragged steps (one sample frozen before frame f), damage before frame f."""
    m = _graph16(True)
    B, H, W = 2, 40, 40
    x0 = _blob(B, 16, H, W, seed=4).to(DEV)
    random.seed(11)
    offs = [m.graph.draw_offsets() for _ in range(T)]
    frs = [0.5 + 0.4 * ((7 * t) % 10) / 10 for t in range(T)]
    gains = [0.25 if t % 3 != 1 else 0.0 for t in range(T)]
    dmg = torch.ones(B, 16, H, W, device=DEV)
    dmg[:, :, 10:20, 12:22] = 0.0
    steps = [T, 2]

    def sched(n):
        return make_schedule(m, B, H, W, n, fire_rate=frs[:n], offsets=offs[:n], message_gains=gains[:n], steps=steps,
                             fire="philox", seed=1234, damage=dmg, damage_step=1)

    _zero_grads(m)
    xa = x0.clone().requires_grad_(True)
    tr = record_rollout(m, xa, sched(T), every=S, impl=impl, differentiable=True)
    _ell(tr.states[f]).backward()
    ga = [xa.grad] + _param_grads(m)
    _zero_grads(m)
    xb = x0.clone().requires_grad_(True)
    xT = rollout(m, xb, sched(f * S), impl=impl)
    if impl == "streaming":
        assert torch.equal(tr.states[f].detach(), xT.detach())
    _ell(xT).backward()
    gb = [xb.grad] + _param_grads(m)
    names = ["x0"] + [n for n, _ in m.named_parameters()]
    for n, a, b in zip(names, ga, gb):
        if impl == "streaming":
            # the zero gradient of the steps after frame f propagates as exact zeros, and x + 0 == x
            assert torch.equal(a, b), (n, rel_err(a, b))
        else:
            # the weight-gradient reduction is partitioned over a different record count
            assert rel_err(a, b) <= 1e-6, (n, rel_err(a, b))


# ---- 3. neutral extension ------------------------------------------------------------------------------------------
def _raw_bwd_old(m, hist, s, gT):
    """the plain entry points gnca_rollout_bwd / gnca_rollout_bwd_bptt straight through the C ABI"""
    lib = _lib.load()
    desc = m.model_desc()
    _, B, Cc, H, W = hist.shape
    g0 = torch.empty(B, Cc, H, W, device=DEV)
    gflat = torch.zeros(GF.param_layout(desc).total, device=DEV)
    ws = GF._WS.get(gT.device, lib.gnca_rollout_workspace_bytes(C.byref(desc), B, H, W, s.T))
    cs = s.c_struct()
    p = GF._ptr
    if hist.bptt is not None:
        rc = lib.gnca_rollout_bwd_bptt(C.byref(desc), p(m.packed_weights()), B, H, W, C.byref(cs), p(hist.bptt),
                                       hist.bptt.numel(), p(gT), p(g0), p(gflat), p(ws), ws.numel(), GF._stream())
    else:
        rc = lib.gnca_rollout_bwd(C.byref(desc), p(m.packed_weights()), B, H, W, C.byref(cs), p(hist.x),
                                  p(hist.stats), p(hist.u), p(gT), p(g0), p(gflat), p(ws), ws.numel(), IMPL["streaming"],
                                  GF._stream())
    _lib.check(rc, "plain backward")
    return g0, gflat


@pytest.mark.parametrize("impl", ["streaming", "resident"])
@pytest.mark.parametrize("T,S", [(9, 3), (10, 4)])
def test_zero_frame_gradient_is_the_plain_backward(T, S, impl):
    m = _graph16(True)
    B, H, W = 2, 40, 40
    x0 = _blob(B, 16, H, W, seed=6).to(DEV)
    d = _draws(m, B, H, W, T, steps=[T, 5], damage_step=3, seed=7)
    s = _schedule(m, B, H, W, T, d)
    desc, packed = m.model_desc(), m.packed_weights()
    gT = torch.randn(B, 16, H, W, device=DEV, generator=torch.Generator(device=DEV).manual_seed(3))
    # the resident backward consumes its record buffer: one forward per backward (the forward is deterministic)
    xT_a, hist_a = rollout_fwd_raw(desc, packed, x0, s, history=True, impl=IMPL[impl], keep_x=False, every=S)
    xT_b, hist_b = rollout_fwd_raw(desc, packed, x0, s, history=True, impl=IMPL[impl], keep_x=False)
    assert (hist_a.bptt is not None) == (impl == "resident")
    assert torch.equal(xT_a, xT_b)
    zeros = torch.zeros(T // S + 1, B, 16, H, W, device=DEV)
    g0_a, gp_a = rollout_bwd_raw(desc, packed, hist_a, s, gT, impl=IMPL[impl], g_frames=zeros, every=S)
    g0_b, gp_b = _raw_bwd_old(m, hist_b, s, gT)
    assert torch.equal(g0_a, g0_b)
    assert torch.equal(gp_a, gp_b)


@pytest.mark.parametrize("impl", IMPLS)
def test_loss_on_x_T_only_equals_rollout(impl):
    m = _graph16(True)
    B, H, W, T, S = 2, 40, 40, 10, 3
    x0 = _blob(B, 16, H, W, seed=8).to(DEV)
    d = _draws(m, B, H, W, T, steps=[10, 6], damage_step=4, seed=9)
    s = _schedule(m, B, H, W, T, d)
    _zero_grads(m)
    xa = x0.clone().requires_grad_(True)
    tr = record_rollout(m, xa, s, every=S, impl=impl, differentiable=True)
    _ell(tr.x_T).backward()
    ga = [xa.grad] + _param_grads(m)
    _zero_grads(m)
    xb = x0.clone().requires_grad_(True)
    xT = rollout(m, xb, s, impl=impl)
    assert torch.equal(xT.detach(), tr.x_T.detach())
    _ell(xT).backward()
    gb = [xb.grad] + _param_grads(m)
    for a, b in zip(ga, gb):
        assert torch.equal(a, b)


# ---- 4. plumbing ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("impl", ["streaming", "resident"])
def test_states_only_x_T_only_and_both(impl):
    m = _graph16(True)
    B, H, W, T, S = 2, 40, 40, 8, 4
    x0 = _blob(B, 16, H, W, seed=10).to(DEV)
    s = _schedule(m, B, H, W, T, _draws(m, B, H, W, T, seed=12))
    grads = {}
    for which in ("states", "x_T", "both"):
        _zero_grads(m)
        xg = x0.clone().requires_grad_(True)
        tr = record_rollout(m, xg, s, every=S, impl=impl, differentiable=True)
        ls = sum(w * _ell(tr.states[f]) for f, w in enumerate(_weights(tr.states.shape[0])))
        loss = {"states": ls, "x_T": _ell(tr.x_T), "both": ls + _ell(tr.x_T)}[which]
        loss.backward()
        grads[which] = [xg.grad] + _param_grads(m)
        assert all(torch.isfinite(g).all() for g in grads[which])
    for a, b, c in zip(grads["states"], grads["x_T"], grads["both"]):
        assert rel_err(a + b, c) <= 1e-5, rel_err(a + b, c)
    assert float(grads["states"][0].abs().max()) > 0 and float(grads["x_T"][0].abs().max()) > 0


def test_autograd_grad_wrt_x0_alone():
    m = _graph16(True)
    B, H, W, T, S = 2, 40, 40, 6, 2
    x0 = _blob(B, 16, H, W, seed=13).to(DEV)
    s = _schedule(m, B, H, W, T, _draws(m, B, H, W, T, seed=14))
    xg = x0.clone().requires_grad_(True)
    tr = record_rollout(m, xg, s, every=S, impl="resident", differentiable=True)
    (gx,) = torch.autograd.grad(_frame_loss(tr.states, tr.x_T), xg)
    _zero_grads(m)
    xh = x0.clone().requires_grad_(True)
    tr = record_rollout(m, xh, s, every=S, impl="resident", differentiable=True)
    _frame_loss(tr.states, tr.x_T).backward()
    assert torch.equal(gx, xh.grad)
    # parameters frozen, only x0 requires grad: still one differentiable node
    for q in m.parameters():
        q.requires_grad_(False)
    try:
        xi = x0.clone().requires_grad_(True)
        tr = record_rollout(m, xi, s, every=S, impl="resident", differentiable=True)
        (gi,) = torch.autograd.grad(_frame_loss(tr.states, tr.x_T), xi)
        assert torch.equal(gi, gx)
    finally:
        for q in m.parameters():
            q.requires_grad_(True)


def test_no_grad_and_default_stay_detached():
    m = _graph16(True)
    B, H, W, T, S = 2, 40, 40, 7, 3
    x0 = _blob(B, 16, H, W, seed=15).to(DEV)
    s = _schedule(m, B, H, W, T, _draws(m, B, H, W, T, seed=16))
    ref = record_rollout(m, x0, s, every=S, impl="resident")
    xg = x0.clone().requires_grad_(True)
    with torch.no_grad():
        a = record_rollout(m, xg, s, every=S, impl="resident", differentiable=True)
    b = record_rollout(m, xg, s, every=S, impl="resident")                    # default: detached even with grad on
    for tr in (a, b):
        assert not tr.states.requires_grad and tr.states.grad_fn is None
        assert not tr.x_T.requires_grad and tr.x_T.grad_fn is None
        assert torch.equal(tr.states, ref.states) and torch.equal(tr.x_T, ref.x_T)
    # differentiable with nothing requiring grad: the detached recording as well
    for q in m.parameters():
        q.requires_grad_(False)
    try:
        c = record_rollout(m, x0, s, every=S, impl="resident", differentiable=True)
        assert c.states.grad_fn is None and torch.equal(c.states, ref.states)
    finally:
        for q in m.parameters():
            q.requires_grad_(True)


def test_attention_stays_detached():
    m = _graph16(True)
    B, H, W, T, S = 2, 40, 40, 7, 3
    x0 = _blob(B, 16, H, W, seed=17).to(DEV)
    s = _schedule(m, B, H, W, T, _draws(m, B, H, W, T, seed=18))
    ref = record_rollout(m, x0, s, every=S, attention=True, impl="resident")
    tr = record_rollout(m, x0.clone().requires_grad_(True), s, every=S, attention=True, impl="resident",
                        differentiable=True)
    assert tr.states.requires_grad and not tr.attention.requires_grad
    assert torch.equal(tr.attention, ref.attention)
    assert rel_err(tr.states.detach(), ref.states) < 1e-5


@pytest.mark.parametrize("impl", ["streaming", "resident"])
def test_second_backward_raises(impl):
    m = _graph16(True)
    B, H, W, T, S = 2, 40, 40, 4, 2
    x0 = _blob(B, 16, H, W, seed=19).to(DEV)
    s = _schedule(m, B, H, W, T, _draws(m, B, H, W, T, seed=20))
    tr = record_rollout(m, x0.clone().requires_grad_(True), s, every=S, impl=impl, differentiable=True)
    loss = _frame_loss(tr.states, tr.x_T)
    loss.backward(retain_graph=True)
    with pytest.raises(RuntimeError):
        loss.backward()


# ---- 5. scale and other shapes -------------------------------------------------------------------------------------
def test_training_shape_resident_vs_streaming():
    """B = 32, T = 64, ragged steps in [48, 80), S = 8: the resident BPTT against the streaming one"""
    m = _graph16(True)
    B, H, W, T, S = 32, 40, 40, 64, 8
    x0 = _blob(B, 16, H, W, seed=21).to(DEV)
    steps = torch.randint(48, 80, (B,), generator=torch.Generator().manual_seed(22)).tolist()
    s = make_schedule(m, B, H, W, T, fire_rate=0.5, steps=steps, fire="philox", seed=23)
    out = {}
    for impl in ("resident", "streaming"):
        _zero_grads(m)
        xg = x0.clone().requires_grad_(True)
        tr = record_rollout(m, xg, s, every=S, impl=impl, differentiable=True)
        _frame_loss(tr.states, tr.x_T).backward()
        out[impl] = (xg.grad, dict(zip([n for n, _ in m.named_parameters()], _param_grads(m))))
    (xa, pa), (xb, pb) = out["resident"], out["streaming"]
    per = sorted(rel_err(xa[b], xb[b]) for b in range(B))
    assert per[B // 2] <= 1e-5, per
    assert rel_err(xa, xb) <= 5e-4
    for n in pa:
        if float(pb[n].abs().max()) < 1e-12:
            assert float(pa[n].abs().max()) <= 1e-7, n
        elif not any(q in n for q in QKS):
            assert rel_err(pa[n], pb[n]) < 1e-4, (n, rel_err(pa[n], pb[n]))


def test_c32_torus_banded_vs_oracle():
    """40x40x32: banded forward with a dense history, streaming backward"""
    m = _random_graph(32, 40)
    B, H, W, T, S = 2, 40, 40, 6, 2
    x0 = _blob(B, 32, H, W, seed=24)
    d = _draws(m, B, H, W, T, steps=[6, 3], damage_step=2, seed=25)
    s = _schedule(m, B, H, W, T, d)
    xr, p, _, _ = _oracle(m, x0, T, S, d)
    _zero_grads(m)
    xg = x0.to(DEV).requires_grad_(True)
    tr = record_rollout(m, xg, s, every=S, impl="banded", differentiable=True)
    _frame_loss(tr.states, tr.x_T).backward()
    _check_grads(m, xg, xr, p)


def test_large_problem_path_vs_oracle():
    """256x256x32, B = 5 (B * ceil(HW / 1024) = 320 >= 296 chunks: the forward runs k_update_tc), T = 3, S = 1, against
    the oracle in fp64"""
    m = _random_graph(32, 256)
    B, H, W, T, S = 5, 256, 256, 3, 1
    x0 = _blob(B, 32, H, W, seed=26)
    d = _draws(m, B, H, W, T, damage_step=1, seed=27)
    s = _schedule(m, B, H, W, T, d)
    xr, p, _, _ = _oracle(m, x0, T, S, d)
    _zero_grads(m)
    xg = x0.to(DEV).requires_grad_(True)
    tr = record_rollout(m, xg, s, every=S, impl="auto", differentiable=True)
    _frame_loss(tr.states, tr.x_T).backward()
    _check_grads(m, xg, xr, p)

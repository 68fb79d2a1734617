"""GPU tests of the resident BPTT of the zero-padded graph shift (gnca_rollout_fwd_bptt_zp / gnca_rollout_bwd_bptt_zp):
rollout(), record_rollout(..., differentiable=True) and the trainer take it under impl 'auto' / 'resident'.

Every case that should run the new path checks that it did (the History holds the zero-pad buffer), so a silent
fallback to the dense history fails.  1. against autograd through fp64 oracle steps with the bounds of
test_gpu_hparams.check_rollout, over k, d_model, radius, gains, ragged steps, damage (dense and both plane layouts),
Philox, flags, B, T and grid shape; 2. bit-equality of x_T / frames with the no-grad rollout / recording, and of two
backward runs; 3. the training shape against the streaming BPTT; 4. the configurations it does not cover keep the
dense history; 5. the trainer."""
import random
import types

import pytest
import torch

from conftest import rel_err
from oracle import nca_oracle as O

pytestmark = pytest.mark.gpu

if torch.cuda.is_available():
    import graph_neural_cellular_automata_b200 as G
    from graph_neural_cellular_automata_b200 import rollout as R
    from graph_neural_cellular_automata_b200.rollout import (make_schedule, record_rollout, rollout, rollout_bwd_raw,
                                                             rollout_fwd_raw)

DEV = "cuda"
QKS = ("query_proj", "key_proj", "scaling")


@pytest.fixture
def zp_runs(monkeypatch):
    """the History of every record-path forward: [True] per forward that kept the zero-pad buffer"""
    seen = []
    orig = R._records_fwd_raw

    def spy(*a, **kw):
        out = orig(*a, **kw)
        seen.append(out is not None and out[1].zp and out[1].bptt is not None)
        return out
    monkeypatch.setattr(R, "_records_fwd_raw", spy)
    return seen


def _model(*, k=8, radius=4, d=16, H=40, a2a=True, hidden_only=True, seed=0):
    torch.manual_seed(seed); random.seed(seed)
    m = G.NeuralCAGraph(16, update_hidden=128, img_size=H, update_gain=0.1, alpha_thr=0.1, message_gain=0.4,
                        hidden_only=hidden_only, graph_alive_to_alive=a2a, graph_d_model=d, graph_attention_radius=radius,
                        graph_num_neighbors=k, graph_zero_padded_shift=True)
    with torch.no_grad():
        m.update_net[2].weight.normal_(0, 0.05)
        m.norm.weight.uniform_(0.5, 1.5); m.norm.bias.normal_(0, 0.1)
        m.graph.query_proj.weight.normal_(0, 0.5); m.graph.key_proj.weight.normal_(0, 0.5)
    return m.to(DEV)


def _state(B, H, W, seed=0):
    """an off-centre alive blob, ragged alive sets on every other sample"""
    g = torch.Generator().manual_seed(seed)
    yy, xx = torch.meshgrid(torch.arange(H), torch.arange(W), indexing="ij")
    r = 0.4 * min(H, W)
    disk = (((yy - 0.45 * H) ** 2 + (xx - 0.55 * W) ** 2) < r * r).float()
    x = torch.rand(B, 16, H, W, generator=g) * disk
    x[1::2, 3] *= (torch.rand((B // 2), H, W, generator=g) > 0.4).float()
    return x


def _ell(x):
    return (x[:, :4] ** 2).mean() + 0.1 * x[:, 4:].mean()


def _frame_loss(states, xT):
    return sum((1.0 + 0.37 * f) * _ell(states[f]) for f in range(states.shape[0])) + _ell(xT)


def _cfg(m, gain):
    return O.StepConfig(update_gain=m.update_gain, alpha_thr=m.alpha_thr, graph=True, message_gain=gain,
                        hidden_only=bool(m.hidden_only), alive_to_alive=bool(m.graph.alive_to_alive),
                        zero_padded_shift=True)


def _draws(m, B, H, W, T, *, gains="t%4", steps=None, dmg=None, seed=0):
    random.seed(seed)
    g = float(m.message_gain)
    gl = {"every": [g] * T, "t%3": [g if t % 3 == 0 else 0.0 for t in range(T)],
          "t%4": [0.0 if t % 4 == 2 else g for t in range(T)], "zero": [0.0] * T}[gains]
    return dict(offs=[m.graph.draw_offsets() for _ in range(T)], frs=[0.5 + 0.1 * (t % 4) for t in range(T)], gains=gl,
                fu=torch.rand(T, B, H, W, generator=torch.Generator().manual_seed(seed + 1)), steps=steps, dmg=dmg)


def _schedule(m, B, H, W, T, d, philox=False):
    kw = dict(fire_rate=d["frs"], offsets=d["offs"], message_gains=d["gains"], steps=d["steps"])
    if d["dmg"] is not None:
        kind, step, mask = d["dmg"]
        if kind == "dense":
            kw.update(damage=mask.to(DEV), damage_step=step)
        else:
            kw.update(damage=types.SimpleNamespace(plane=mask.to(DEV), layout=1 if kind == "plane" else 2),
                      damage_step=step)
    if philox:
        return make_schedule(m, B, H, W, T, fire="philox", seed=77, **kw)
    return make_schedule(m, B, H, W, T, fire_u=d["fu"].to(DEV), **kw)


def _dense_damage(d, B, H, W):
    kind, step, mask = d["dmg"]
    if kind == "dense":
        return step, mask
    full = torch.ones(B, 16, H, W)
    if kind == "plane":
        full *= mask[:, None]
    else:
        full[:, 3] = mask
    return step, full


def _oracle(m, x0, T, S, d, fu=None):
    """fp64 autograd through T oracle steps; frame f = x_{f*S} after the damage of its step.  Returns (x0 leaf, params,
    frames, x_T) after the backward of _frame_loss."""
    B, _, H, W = x0.shape
    p = {k: v.detach().cpu().double().requires_grad_(v.is_floating_point() and "perception" not in k)
         for k, v in m.state_dict().items()}
    xr = x0.double().requires_grad_(True)
    x, xs = xr, []
    dstep, dmask = _dense_damage(d, B, H, W) if d["dmg"] is not None else (None, None)
    st = torch.tensor(d["steps"]) if d["steps"] is not None else None
    fu = d["fu"] if fu is None else fu
    for t in range(T):
        if t == dstep:
            x = x * dmask.double()
        xs.append(x)
        mask = st > t if st is not None else torch.ones(B, dtype=torch.bool)
        if not bool(mask.any()):
            continue
        new = O.nca_step(x[mask], p, _cfg(m, d["gains"][t]), d["frs"][t], fu[t][mask].unsqueeze(1).double(),
                         d["offs"][t])
        x = x.clone()
        x[mask] = new
    xs.append(x)
    frames = torch.stack([xs[f * S] for f in range(T // S + 1)])
    _frame_loss(frames, x).backward()
    return xr, p, frames, x


def _check_grads(m, xg, xr, p):
    """the bounds of test_gpu_hparams.check_rollout"""
    B = xg.shape[0]
    per = sorted(rel_err(xg.grad[b].cpu(), xr.grad[b]) for b in range(B))
    assert per[B // 2] <= 1e-5, per
    assert rel_err(xg.grad.cpu(), xr.grad) <= 5e-4, rel_err(xg.grad.cpu(), xr.grad)
    for n, q in m.named_parameters():
        gr = p[n].grad
        ours = q.grad.cpu() if q.grad is not None else torch.zeros_like(q.detach().cpu())
        if gr is None or float(gr.abs().max()) < 1e-12:
            assert float(ours.abs().max()) <= 1e-7, n
        elif any(s in n for s in QKS):
            assert rel_err(ours, gr) < 1e-3, (n, rel_err(ours, gr))
        else:
            assert rel_err(ours, gr) < 1e-4, (n, rel_err(ours, gr))


def _zero_grads(m):
    for q in m.parameters():
        q.grad = None


def _run_vs_oracle(m, B, H, W, T, S, d, zp_runs, *, impl="auto", philox=False):
    s = _schedule(m, B, H, W, T, d, philox)
    x0 = _state(B, H, W, seed=T + B)
    fu = None
    if philox:      # the oracle needs the uniforms of the in-kernel stream
        fu = _philox_uniforms(m, s, B, H, W, T)
    xr, p, frames_ref, xT_ref = _oracle(m, x0, T, S, d, fu)
    _zero_grads(m)
    xg = x0.to(DEV).requires_grad_(True)
    tr = record_rollout(m, xg, s, every=S, impl=impl, differentiable=True)
    assert zp_runs and all(zp_runs), zp_runs
    assert rel_err(tr.x_T.detach().cpu(), xT_ref.detach()) < 1e-5
    _frame_loss(tr.states, tr.x_T).backward()
    _check_grads(m, xg, xr, p)
    return tr


def _philox_uniforms(m, s, B, H, W, T):
    from philox_replica import fire_uniforms
    return torch.as_tensor(fire_uniforms(s.philox_seed, s.philox_offset, T, B, H, W)).float()


# ---- 1. against the fp64 oracle ---------------------------------------------------------------------------------------
@pytest.mark.parametrize("k,d,radius", [(1, 8, 3), (8, 16, 4), (9, 1, 3), (16, 32, 4), (16, 8, 3)],
                         ids=lambda v: str(v))
def test_k_and_d_model(k, d, radius, zp_runs):
    m = _model(k=k, radius=radius, d=d, seed=10 * k + d)
    _run_vs_oracle(m, 4, 40, 40, 6, 2, _draws(m, 4, 40, 40, 6, seed=k + d), zp_runs)


@pytest.mark.parametrize("gains", ["every", "t%3", "zero"])
def test_message_gains(gains, zp_runs):
    m = _model(seed=3)
    _run_vs_oracle(m, 4, 40, 40, 7, 3, _draws(m, 4, 40, 40, 7, gains=gains, seed=3), zp_runs)


@pytest.mark.parametrize("kind", ["dense", "plane", "plane_alpha"])
def test_ragged_steps_and_damage(kind, zp_runs):
    B, H, W, T = 4, 40, 40, 8
    m = _model(seed=4)
    g = torch.Generator().manual_seed(5)
    if kind == "dense":
        mask = (torch.rand(B, 16, H, W, generator=g) > 0.3).float()
    else:
        mask = (torch.rand(B, H, W, generator=g) > 0.3).float()
    mask[..., 10:20, 12:30] = 0.0
    # damage before step 1, a message step: the attention row term of dL/dx_1 is multiplied by the mask too
    d = _draws(m, B, H, W, T, steps=[8, 3, 0, 6], dmg=(kind, 1, mask), seed=4)
    _run_vs_oracle(m, B, H, W, T, 2, d, zp_runs)


def test_philox_fire(zp_runs):
    m = _model(seed=6)
    _run_vs_oracle(m, 4, 40, 40, 6, 2, _draws(m, 4, 40, 40, 6, seed=6), zp_runs, philox=True)


@pytest.mark.parametrize("a2a,hidden_only", [(False, True), (True, False), (False, False)])
def test_flags(a2a, hidden_only, zp_runs):
    m = _model(a2a=a2a, hidden_only=hidden_only, seed=7)
    _run_vs_oracle(m, 4, 40, 40, 6, 2, _draws(m, 4, 40, 40, 6, seed=7), zp_runs)


@pytest.mark.parametrize("B", [1, 4, 9])
def test_batch_sizes(B, zp_runs):
    m = _model(seed=8)
    _run_vs_oracle(m, B, 40, 40, 5, 5, _draws(m, B, 40, 40, 5, seed=B), zp_runs, impl="resident")


def test_small_grid_24x32(zp_runs):
    m = _model(k=8, radius=3, H=24, seed=9)
    _run_vs_oracle(m, 3, 24, 32, 6, 2, _draws(m, 3, 24, 32, 6, seed=9), zp_runs)


def test_one_step_rollout_vs_oracle(zp_runs):
    """T = 1 through rollout() (check_rollout's loss on x_T)"""
    m = _model(seed=11)
    B, H, W, T = 3, 40, 40, 1
    d = _draws(m, B, H, W, T, gains="every", seed=11)
    s = _schedule(m, B, H, W, T, d)
    x0 = _state(B, H, W, seed=11)
    xr, p, _, xT_ref = _oracle(m, x0, T, T, d)
    _zero_grads(m)
    xg = x0.to(DEV).requires_grad_(True)
    out = rollout(m, xg, s, impl="auto")
    assert zp_runs == [True]
    _frame_loss(torch.stack([xg, out]), out).backward()
    _check_grads(m, xg, xr, p)


def test_zero_steps():
    """T = 0: the forward copies x0 to x_T and the frame, the backward gT plus the frame gradient to g0"""
    import ctypes as C
    from graph_neural_cellular_automata_b200 import _lib
    from graph_neural_cellular_automata_b200 import functional as GF
    lib = _lib.load()
    m = _model(seed=12)
    desc, packed = m.model_desc(), m.packed_weights()
    B, H, W = 2, 40, 40
    x0 = _state(B, H, W).to(DEV)
    s = R.Schedule(T=0, k=8, fire_rate=torch.ones(1, device=DEV), message_gain=torch.ones(1, device=DEV),
                   offsets=torch.ones(16, dtype=torch.int8, device=DEV), max_offset=1)
    cs = s.c_struct()
    nb = lib.gnca_bptt_zp_bytes(C.byref(desc), B, H, W, 0)
    assert nb > 0
    bptt = torch.empty(nb, dtype=torch.uint8, device=DEV)
    ws = torch.empty(lib.gnca_rollout_workspace_bytes(C.byref(desc), B, H, W, 0), dtype=torch.uint8, device=DEV)
    xT, frames = torch.empty_like(x0), torch.empty(1, B, 16, H, W, device=DEV)
    p = GF._ptr
    assert lib.gnca_rollout_fwd_bptt_zp(C.byref(desc), p(packed), B, H, W, C.byref(cs), p(x0), p(xT), 1, p(frames),
                                        p(bptt), nb, p(ws), ws.numel(), None) == 0
    gT, gf = torch.randn_like(x0), torch.randn_like(frames)
    g0, gp = torch.empty_like(x0), torch.zeros(GF.param_layout(desc).total, device=DEV)
    assert lib.gnca_rollout_bwd_bptt_zp(C.byref(desc), p(packed), B, H, W, C.byref(cs), p(bptt), nb, 1, p(gf), p(gT),
                                        p(g0), p(gp), p(ws), ws.numel(), None) == 0
    torch.cuda.synchronize()
    assert torch.equal(xT, x0) and torch.equal(frames[0], x0)
    assert torch.equal(g0, gT + gf[0]) and not gp.any()


# ---- 2. bit-equality -------------------------------------------------------------------------------------------------
def test_bit_equal_forward_and_deterministic_backward(zp_runs):
    m = _model(k=12, radius=3, seed=13)
    B, H, W, T, S = 5, 40, 40, 9, 3
    d = _draws(m, B, H, W, T, gains="t%3", steps=[9, 4, 9, 0, 7], seed=13)
    s = _schedule(m, B, H, W, T, d)
    x0 = _state(B, H, W, seed=13).to(DEV)
    with torch.no_grad():
        xT_plain = rollout(m, x0, s, impl="auto")
        rec = record_rollout(m, x0, s, every=S, impl="auto")
    desc, packed = m.model_desc(), m.packed_weights()
    xT, hist = rollout_fwd_raw(desc, packed, x0, s, history=True, impl=0, keep_x=True)
    assert hist.zp
    assert torch.equal(xT, xT_plain)
    assert torch.equal(hist.x[::S], rec.states)
    xg = x0.clone().requires_grad_(True)
    tr = record_rollout(m, xg, s, every=S, impl="auto", differentiable=True)
    assert torch.equal(tr.states.detach(), rec.states) and torch.equal(tr.x_T.detach(), rec.x_T)
    gT = torch.randn_like(x0)
    gf = torch.randn(T // S + 1, B, 16, H, W, device=DEV)
    _, hist = rollout_fwd_raw(desc, packed, x0, s, history=True, impl=0, keep_x=False, every=S)
    a = rollout_bwd_raw(desc, packed, hist, s, gT, g_frames=gf, every=S)
    _, hist = rollout_fwd_raw(desc, packed, x0, s, history=True, impl=0, keep_x=False, every=S)
    b = rollout_bwd_raw(desc, packed, hist, s, gT, g_frames=gf, every=S)
    assert hist.zp and all(zp_runs)
    assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])


# ---- 3. the training shape against the streaming BPTT ----------------------------------------------------------------
def test_training_shape_vs_streaming(zp_runs):
    """B = 32, T = 64, ragged steps in [48, 80), message on t % 3 == 0: the bounds of
    test_gpu_record_grad.test_training_shape_resident_vs_streaming"""
    m = _model(seed=14)
    B, H, W, T, S = 32, 40, 40, 64, 8
    x0 = _state(B, H, W, seed=21).to(DEV)
    steps = torch.randint(48, 80, (B,), generator=torch.Generator().manual_seed(22)).tolist()
    s = make_schedule(m, B, H, W, T, fire_rate=0.5, steps=steps, fire="philox", seed=23, message_every=3)
    out = {}
    for impl in ("auto", "streaming"):
        _zero_grads(m)
        xg = x0.clone().requires_grad_(True)
        tr = record_rollout(m, xg, s, every=S, impl=impl, differentiable=True)
        _frame_loss(tr.states, tr.x_T).backward()
        out[impl] = (xg.grad, {n: (q.grad.clone() if q.grad is not None else torch.zeros_like(q))
                               for n, q in m.named_parameters()})
    assert zp_runs == [True]
    (xa, pa), (xb, pb) = out["auto"], out["streaming"]
    per = sorted(rel_err(xa[b], xb[b]) for b in range(B))
    assert per[B // 2] <= 1e-5, per
    assert rel_err(xa, xb) <= 5e-4
    for n in pa:
        if float(pb[n].abs().max()) < 1e-12:
            assert float(pa[n].abs().max()) <= 1e-7, n
        elif any(q in n for q in QKS):
            assert rel_err(pa[n], pb[n]) < 1e-3, (n, rel_err(pa[n], pb[n]))
        else:
            assert rel_err(pa[n], pb[n]) < 1e-4, (n, rel_err(pa[n], pb[n]))


# ---- 4. what it does not cover keeps the dense history ---------------------------------------------------------------
@pytest.mark.parametrize("case", ["d33", "k17", "short_grid"])
def test_fallbacks_keep_the_dense_history(case, zp_runs):
    """d_model 33 and k = 17 are outside what the buffer is offered for; on a 4x12 grid with offsets of up to 5 rows
    (k = 8, so the buffer is offered) the zero-pad forward itself rejects the schedule before any launch."""
    if case == "d33":
        m, H = _model(d=33, seed=15), 40
    elif case == "k17":
        m, H = _model(k=17, radius=3, seed=15), 40
    else:
        m, H = _model(k=8, radius=5, H=4, seed=15), 4
    W, B, T = 12 if case == "short_grid" else 40, 3, 3
    d = _draws(m, B, H, W, T, seed=15)
    s = _schedule(m, B, H, W, T, d)
    if case == "short_grid":
        _zp_forward_rejects(m, s, B, H, W)
    x0 = _state(B, H, W, seed=15)
    xr, p, _, _ = _oracle(m, x0, T, T, d)
    _zero_grads(m)
    xg = x0.to(DEV).requires_grad_(True)
    xT, hist = rollout_fwd_raw(m.model_desc(), m.packed_weights(), xg.detach(), s, history=True, impl=0)
    assert hist.bptt is None and hist.x is not None and not hist.zp
    out = rollout(m, xg, s, impl="auto")
    assert torch.equal(out.detach(), xT)
    _frame_loss(torch.stack([xg, out]), out).backward()
    _check_grads(m, xg, xr, p)
    assert not any(zp_runs)


def _zp_forward_rejects(m, s, B, H, W):
    """gnca_rollout_fwd_bptt_zp is offered the schedule (a buffer size exists) and returns UNSUPPORTED without a launch"""
    import ctypes as C
    from graph_neural_cellular_automata_b200 import _lib
    from graph_neural_cellular_automata_b200 import functional as GF
    lib = _lib.load()
    desc, packed = m.model_desc(), m.packed_weights()
    assert s.k <= R.RESIDENT_MAX_K and s.max_offset >= H
    nb = lib.gnca_bptt_zp_bytes(C.byref(desc), B, H, W, s.T)
    assert nb > 0
    bptt = torch.empty(nb, dtype=torch.uint8, device=DEV)
    ws = torch.empty(lib.gnca_rollout_workspace_bytes(C.byref(desc), B, H, W, s.T), dtype=torch.uint8, device=DEV)
    x0 = torch.zeros(B, 16, H, W, device=DEV)
    xT = torch.full_like(x0, -1.0)
    cs = s.c_struct()
    torch.cuda.synchronize()
    before = lib.gnca_launch_count()
    rc = lib.gnca_rollout_fwd_bptt_zp(C.byref(desc), GF._ptr(packed), B, H, W, C.byref(cs), GF._ptr(x0), GF._ptr(xT),
                                      0, None, GF._ptr(bptt), nb, GF._ptr(ws), ws.numel(), GF._stream())
    assert rc == _lib.GNCA_ERR_UNSUPPORTED
    assert lib.gnca_launch_count() == before
    torch.cuda.synchronize()
    assert bool((xT == -1.0).all())


def test_budget_keeps_the_dense_history():
    m = _model(seed=16)
    B, H, W, T = 4, 40, 40, 6
    s = _schedule(m, B, H, W, T, _draws(m, B, H, W, T, seed=16))
    x0 = _state(B, H, W, seed=16).to(DEV)
    _, hist = rollout_fwd_raw(m.model_desc(), m.packed_weights(), x0, s, history=True, impl=0, keep_x=False,
                              bptt_budget=1 << 40)
    assert hist.plan[0] == "dense" and hist.bptt is None and not hist.zp


# ---- 5. the trainer --------------------------------------------------------------------------------------------------
def _train_two_steps(impl):
    from graph_neural_cellular_automata_b200.training.trainer import GraphNCATrainer, TrainConfig
    torch.manual_seed(21); random.seed(21)
    m = _model(seed=17)
    cfg = TrainConfig(batch_size=8, pool_size=16, long_rollout_prob=0.5, long_rollout_steps_min=60,
                      long_rollout_steps_max=90, fire_rate_min=0.5, fire_rate_max=0.9,
                      message_every=3, reset_worst_prob=0.25, random_reseed_prob=0.0, damage={}, fire="philox",
                      rollout_impl=impl)
    target = torch.zeros(4, 40, 40)
    target[:, 12:28, 12:28] = 0.8
    tr = GraphNCATrainer(m, target, cfg)
    with torch.no_grad():
        x = tr.pool.pool
        for _ in range(24):
            x = m(x, fire_rate=0.7)
        tr.pool.pool.copy_(x)
    out = []
    for ep in (1, 2):
        r = tr.train_step(ep)
        out.append((r["per_sample"].clone(), r["gflat"].clone()))
    return out, [q.detach().clone() for q in m.parameters()]


def test_trainer_auto_vs_streaming(zp_runs):
    a, pa = _train_two_steps("auto")
    assert len(zp_runs) == 2 and all(zp_runs)
    b, pb = _train_two_steps("streaming")
    for (la, ga), (lb, gb) in zip(a, b):
        assert rel_err(la, lb) <= 1e-5, rel_err(la, lb)
        assert rel_err(ga, gb) <= 1e-3, rel_err(ga, gb)
    for qa, qb in zip(pa, pb):
        assert rel_err(qa, qb) <= 1e-4, rel_err(qa, qb)

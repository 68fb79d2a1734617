"""GPU tests of checkpointed BPTT: rollout(..., checkpoint_every=K) and record_rollout(..., checkpoint=True).

1. the gradients equal the dense streaming BPTT (x_T and, where the dense backward is itself deterministic, dL/dx0 bit
   for bit; sums through float atomics to 1e-6) over checkpoint strides, ragged steps, damage, Philox and T = 0;
2. against autograd through the fp64 oracle; 3. other widths and the large-problem (tensor-core) forward;
4. differentiable frames as checkpoints; 5. memory does not grow with T beyond the checkpoints; 6. plumbing."""
import random

import pytest
import torch

from conftest import load_params, rel_err
from oracle import nca_oracle as O

pytestmark = pytest.mark.gpu

if torch.cuda.is_available():
    import graph_neural_cellular_automata_b200 as G
    from graph_neural_cellular_automata_b200.rollout import make_schedule, record_rollout, rollout

DEV = "cuda"
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


def _random_graph(C_, H, hidden=128, seed=5):
    torch.manual_seed(seed); random.seed(seed)
    m = G.NeuralCAGraph(C_, update_hidden=hidden, img_size=H, update_gain=0.1, alpha_thr=0.1, message_gain=0.3,
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


def _schedule(m, B, H, W, T, d, *, philox=False):
    if philox:
        return make_schedule(m, B, H, W, T, fire_rate=d["frs"], offsets=d["offs"], message_gains=d["gains"],
                             steps=d["steps"], fire="philox", seed=4321,
                             damage=d["dmg"].to(DEV) if d["dmg"] is not None else None, damage_step=d["dmg_step"] or 0)
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


def _grads_of(m, x0, s, **kw):
    """x_T, dL/dx0 and the parameter gradients of ell(x_T) through rollout(m, x0, s, **kw)"""
    _zero_grads(m)
    xg = x0.clone().requires_grad_(True)
    xT = rollout(m, xg, s, **kw)
    _ell(xT).backward()
    return xT.detach(), xg.grad, _param_grads(m)


def _assert_params_close(m, ga, gb, tol=1e-6):
    for (n, _), a, b in zip(m.named_parameters(), ga, gb):
        if float(b.abs().max()) == 0.0:
            assert float(a.abs().max()) == 0.0, n
        else:
            assert rel_err(a, b) <= tol, (n, rel_err(a, b))


# ---- 1. equals the dense streaming BPTT ----------------------------------------------------------------------------
B1, H1, T1 = 4, 40, 10
KS = [1, 3, 5, 10, 11]


def _inside(K):
    """a damage step strictly inside a segment (not a checkpoint) for stride K, T = 10"""
    return K + K // 2 if K + K // 2 < T1 else K // 2


# name: (ragged steps, damage step as a function of K or None, Philox, T); None from the damage function = no such step
CASES = {
    "plain": (None, None, False, T1),
    # sample 0 never steps, sample 3 runs every step; samples 1 and 2 freeze at t = 2 and t = 6: on checkpoint 6 for
    # K = 3, on either side of checkpoint 5 for K = 5
    "ragged": ([0, 2, 6, T1], None, False, T1),
    "damage_t0": (None, lambda K: 0, False, T1),
    "damage_at_ckpt": (None, lambda K: K if K < T1 else None, False, T1),
    "damage_inside": ([T1, 7, 3, T1], lambda K: _inside(K) if K > 1 else None, False, T1),
    "philox": ([T1, 4, T1, 8], lambda K: 4, True, T1),
    "T0": (None, None, False, 0),
}


def test_dense_streaming_dx0_is_deterministic():
    """The bit-equality below rests on the dense backward's dL/dx0 being run-to-run identical on torus and classic
    models: k_bwd_gather writes each cell once, no atomics."""
    for model in ("torus", "classic"):
        m = MODELS[model]()
        x0 = _blob(B1, 16, H1, H1, seed=1).to(DEV)
        s = _schedule(m, B1, H1, H1, T1, _draws(m, B1, H1, H1, T1, steps=[0, 2, 6, T1], damage_step=4, seed=3))
        _, ga, _ = _grads_of(m, x0, s, impl="streaming")
        _, gb, _ = _grads_of(m, x0, s, impl="streaming")
        assert torch.equal(ga, gb), model


@pytest.mark.parametrize("K", KS)
@pytest.mark.parametrize("model", list(MODELS))
@pytest.mark.parametrize("case", list(CASES))
def test_ckpt_equals_dense_streaming(case, model, K):
    steps, dfn, philox, T = CASES[case]
    dstep = dfn(K) if dfn is not None else None
    if dfn is not None and dstep is None:
        pytest.skip(f"no such damage step for K = {K}, T = {T}")
    m = MODELS[model]()
    x0 = _blob(B1, 16, H1, H1, seed=1).to(DEV)
    s = _schedule(m, B1, H1, H1, T, _draws(m, B1, H1, H1, T, steps=steps, damage_step=dstep, seed=3), philox=philox)
    xa, ga, pa = _grads_of(m, x0, s, checkpoint_every=K)
    xb, gb, pb = _grads_of(m, x0, s, impl="streaming")
    assert torch.equal(xa, xb)
    if model == "zeropad":
        assert rel_err(ga, gb) <= 1e-6, rel_err(ga, gb)     # the attention backward sums dL/dx rows with atomics
    else:
        assert torch.equal(ga, gb), rel_err(ga, gb)
    _assert_params_close(m, pa, pb)
    assert float(ga.abs().max()) > 0


# ---- 2. against the fp64 oracle ------------------------------------------------------------------------------------
@pytest.mark.parametrize("model", list(MODELS))
def test_ckpt_vs_oracle(model):
    """frames as checkpoints (S = 3, T = 10: a short last segment), ragged steps, damage on a checkpoint"""
    T, S = 10, 3
    m = MODELS[model]()
    B, H, W = 2, 40, 40
    x0 = _blob(B, 16, H, W, seed=1)
    d = _draws(m, B, H, W, T, steps=[10, 4], damage_step=6, seed=3)
    s = _schedule(m, B, H, W, T, d)
    xr, p, frames_ref, xT_ref = _oracle(m, x0, T, S, d)
    _zero_grads(m)
    xg = x0.to(DEV).requires_grad_(True)
    tr = record_rollout(m, xg, s, every=S, differentiable=True, checkpoint=True)
    assert rel_err(tr.states.detach().cpu(), frames_ref.detach()) < 1e-5
    assert rel_err(tr.x_T.detach().cpu(), xT_ref.detach()) < 1e-5
    _frame_loss(tr.states, tr.x_T).backward()
    _check_grads(m, xg, xr, p)


# ---- 3. widths and the large-problem path --------------------------------------------------------------------------
@pytest.mark.parametrize("C_,hidden", [(4, 128), (8, 128), (32, 128), (16, 64), (16, 256)])
def test_widths_equal_dense_streaming(C_, hidden):
    m = _random_graph(C_, 40, hidden=hidden)
    B, H, T, K = 3, 40, 9, 4
    x0 = _blob(B, C_, H, H, seed=2).to(DEV)
    s = _schedule(m, B, H, H, T, _draws(m, B, H, H, T, steps=[T, 5, 2], damage_step=6, seed=4))
    xa, ga, pa = _grads_of(m, x0, s, checkpoint_every=K)
    xb, gb, pb = _grads_of(m, x0, s, impl="streaming")
    assert torch.equal(xa, xb)
    assert rel_err(ga, gb) <= 1e-6, rel_err(ga, gb)
    _assert_params_close(m, pa, pb)


def test_large_problem_path_equals_dense_streaming():
    """256x256x32, B = 5 (B * ceil(HW / 1024) = 320 >= 296 chunks: the forward and its recomputation run k_update_tc),
    T = 12, K = 5 (a short last segment), damage at t = 5, a checkpoint"""
    m = _random_graph(32, 256)
    B, H, T, K = 5, 256, 12, 5
    x0 = _blob(B, 32, H, H, seed=26).to(DEV)
    s = _schedule(m, B, H, H, T, _draws(m, B, H, H, T, damage_step=5, seed=27))
    xa, ga, pa = _grads_of(m, x0, s, checkpoint_every=K)
    xb, gb, pb = _grads_of(m, x0, s, impl="streaming")
    assert torch.equal(xa, xb)
    assert rel_err(ga, gb) <= 1e-6, rel_err(ga, gb)
    _assert_params_close(m, pa, pb)


# ---- 4. frames as checkpoints --------------------------------------------------------------------------------------
@pytest.mark.parametrize("S", [1, 3, 10, 11])
def test_checkpointed_frames_equal_dense_frames(S):
    m = _graph16(True)
    B, H, T = 3, 40, 10
    x0 = _blob(B, 16, H, H, seed=5).to(DEV)
    s = _schedule(m, B, H, H, T, _draws(m, B, H, H, T, steps=[T, 4, 7], damage_step=3, seed=6))
    out = {}
    for ck in (True, False):
        _zero_grads(m)
        xg = x0.clone().requires_grad_(True)
        if ck:
            tr = record_rollout(m, xg, s, every=S, differentiable=True, checkpoint=True)
        else:
            tr = record_rollout(m, xg, s, every=S, differentiable=True, impl="streaming")
        assert tr.states.grad_fn is tr.x_T.grad_fn
        _frame_loss(tr.states, tr.x_T).backward()
        out[ck] = (tr.states.detach(), tr.x_T.detach(), xg.grad, _param_grads(m))
    (sa, xa, ga, pa), (sb, xb, gb, pb) = out[True], out[False]
    assert torch.equal(sa, sb) and torch.equal(xa, xb)
    assert torch.equal(ga, gb), rel_err(ga, gb)
    _assert_params_close(m, pa, pb)


def test_editing_a_checkpointed_frame_in_place_makes_backward_raise():
    m = _graph16(True)
    B, H, T, S = 2, 40, 6, 2
    x0 = _blob(B, 16, H, H, seed=7).to(DEV)
    s = _schedule(m, B, H, H, T, _draws(m, B, H, H, T, seed=8))
    tr = record_rollout(m, x0.clone().requires_grad_(True), s, every=S, differentiable=True, checkpoint=True)
    loss = tr.states.sum() + _ell(tr.x_T)       # sum() saves no input: only the node's own saved frames can object
    with torch.no_grad():
        tr.states[1].mul_(0.5)
    with pytest.raises(RuntimeError, match="inplace"):
        loss.backward()


# ---- 5. memory ----------------------------------------------------------------------------------------------------
def _peak(m, x0, T, **kw):
    """peak allocated bytes over one forward + loss + backward, above what is allocated before it"""
    B, _, H, W = x0.shape
    s = make_schedule(m, B, H, W, T, fire_rate=0.5, fire="philox", seed=9)
    _zero_grads(m)
    xg = x0.clone().requires_grad_(True)
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    _ell(rollout(m, xg, s, **kw)).backward()
    torch.cuda.synchronize()
    return torch.cuda.max_memory_allocated() - base


def test_memory_does_not_grow_with_T():
    m = _graph16(True)
    B, H, K = 8, 40, 8
    x0 = _blob(B, 16, H, H, seed=10).to(DEV)
    nbytes = x0.numel() * 4                     # 819200: a multiple of the allocator's 512-byte rounding
    for kw in ({"checkpoint_every": K}, {"impl": "streaming"}):
        _peak(m, x0, 16, **kw)                  # warm the workspace cache and the weights
    ck = _peak(m, x0, 64, checkpoint_every=K) - _peak(m, x0, 16, checkpoint_every=K)
    want = (64 // K - 16 // K) * nbytes
    assert want <= ck <= want + (64 << 10), (ck, want)
    dense = _peak(m, x0, 64, impl="streaming") - _peak(m, x0, 16, impl="streaming")
    assert dense >= 2 * 48 * nbytes, (dense, 2 * 48 * nbytes)


# ---- 6. plumbing --------------------------------------------------------------------------------------------------
def test_no_grad_is_plain_inference():
    m = _graph16(True)
    B, H, T = 2, 40, 9
    x0 = _blob(B, 16, H, H, seed=11).to(DEV)
    s = _schedule(m, B, H, H, T, _draws(m, B, H, H, T, steps=[9, 5], damage_step=4, seed=12))
    with torch.no_grad():
        ref = rollout(m, x0, s)
        a = rollout(m, x0.clone().requires_grad_(True), s, checkpoint_every=4)
    assert a.grad_fn is None and torch.equal(a, ref)
    with torch.no_grad():
        tr = record_rollout(m, x0.clone().requires_grad_(True), s, every=4, differentiable=True, checkpoint=True)
    assert tr.states.grad_fn is None and torch.equal(tr.x_T, ref)


def test_invalid_arguments_raise():
    m = _graph16(True)
    B, H, T = 2, 40, 4
    x0 = _blob(B, 16, H, H, seed=13).to(DEV).requires_grad_(True)
    s = _schedule(m, B, H, H, T, _draws(m, B, H, H, T, seed=14))
    with pytest.raises(ValueError, match="return_history"):
        rollout(m, x0, s, checkpoint_every=2, return_history=True)
    for impl in ("resident", "banded"):
        with pytest.raises(ValueError, match="streaming"):
            rollout(m, x0, s, checkpoint_every=2, impl=impl)
        with pytest.raises(ValueError, match="streaming"):
            record_rollout(m, x0, s, every=2, impl=impl, differentiable=True, checkpoint=True)
    for K in (0, -1):
        with pytest.raises(ValueError, match="checkpoint_every"):
            rollout(m, x0, s, checkpoint_every=K)
    with pytest.raises(ValueError, match="differentiable"):
        record_rollout(m, x0, s, every=2, checkpoint=True)


def test_second_backward_raises():
    m = _graph16(True)
    B, H, T = 2, 40, 6
    x0 = _blob(B, 16, H, H, seed=15).to(DEV)
    s = _schedule(m, B, H, H, T, _draws(m, B, H, H, T, seed=16))
    loss = _ell(rollout(m, x0.clone().requires_grad_(True), s, checkpoint_every=4))
    loss.backward(retain_graph=True)
    with pytest.raises(RuntimeError):
        loss.backward()

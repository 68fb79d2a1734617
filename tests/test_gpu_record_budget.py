"""GPU tests of record_rollout(..., differentiable=True, bptt_budget=N): frame gradients on the checkpointed resident
BPTT (gnca_rollout_bwd_bptt_ckpt_frames) and the budget's choice of history.

1. a budget that covers the unbudgeted history is that call, bit for bit;
2. resident checkpoints (the frames) every K = r * S steps against the unbudgeted record path: frames, x_T and dL/dx0
   bit-equal, parameters to 1e-6, over r, T % S, ragged steps, damage, Philox, gain-0 steps, the loss's outputs, T = 0;
3. against autograd through fp64 oracle steps; 4. the streaming fallback is checkpoint=True bit for bit;
5. T = 1000 at B = 32 within the budget; 6. errors and the autograd node.
Every case meant to take the resident checkpoints asserts the plan its forward stored (x_T.grad_fn.plan)."""
import ctypes as C

import pytest
import torch

from conftest import rel_err

pytestmark = pytest.mark.gpu

if torch.cuda.is_available():
    import graph_neural_cellular_automata_b200 as G
    from graph_neural_cellular_automata_b200 import functional as GF
    from graph_neural_cellular_automata_b200.rollout import (BPTT_MAX_BYTES, bptt_plan, make_schedule, record_rollout,
                                                             rollout_bwd_raw, rollout_fwd_raw)
    from test_gpu_rep_ckpt import MODELS, T1000_MAX, T1000_MEDIAN, _blob, _graph16, _schedule
    import test_gpu_record_grad as RG

DEV = "cuda"
# Parameter-gradient distance of the resident checkpoints to checkpoint=True at T = 1000 with a loss on 21 frames and x_T
# (DESIGN section 3.10): measured 1.11e-3 on an NVIDIA B200 (1000 W), against 8.3e-4 for the x_T-only loss that
# T1000_PARAMS bounds.  Both backwards are checked bit for bit or against the fp64 oracle at short T; over 1000 steps
# their summation orders drift apart, and every frame loss adds its own share of the drift to the parameter sums.
T1000_FRAMES_PARAMS = 1.5e-3


def _ell(x):
    return (x[:, :4] ** 2).mean() + 0.1 * x[:, 4:].mean()


def _loss(states, xT, which):
    """a distinct weight per frame, so that a frame taken for its neighbour shows"""
    frames = sum((1.0 + 0.37 * f) * _ell(states[f]) for f in range(states.shape[0]))
    return {"frames": frames, "xT": _ell(xT), "both": frames + _ell(xT)}[which]


def _run(m, x0, s, S, which="both", **kw):
    """frames, x_T, dL/dx0, parameter gradients and the stored plan of one differentiable recording"""
    for q in m.parameters():
        q.grad = None
    xg = x0.clone().requires_grad_(True)
    tr = record_rollout(m, xg, s, every=S, differentiable=True, **kw)
    assert tr.states.grad_fn is tr.x_T.grad_fn
    _loss(tr.states, tr.x_T, which).backward()
    grads = [q.grad.clone() if q.grad is not None else torch.zeros_like(q) for q in m.parameters()]
    return tr.states.detach(), tr.x_T.detach(), xg.grad, grads, getattr(tr.x_T.grad_fn, "plan", None)


def _bit_equal(a, b):
    for x, y in zip(a[:3], b[:3]):
        assert torch.equal(x, y), float((x - y).abs().max())
    for ga, gb in zip(a[3], b[3]):
        assert torch.equal(ga, gb)


def _ckpt_bytes(m, B, H, W, K):
    return G._lib.load().gnca_bptt_ckpt_bytes(C.byref(m.model_desc()), B, H, W, K)


# ---- 1. a budget that covers the unbudgeted history ------------------------------------------------------------------
@pytest.mark.parametrize("model", ["torus", "classic"])
def test_budget_covering_records_is_bit_identical(model):
    m = MODELS[model]()
    B, H, T, S = 4, 40, 12, 3
    x0 = _blob(B, 16, H, H)
    s = _schedule(m, B, H, H, T, steps=[0, 3, 8, T], damage_step=3)
    assert bptt_plan(m, B, H, H, T, 1 << 40, every=S)[0] == "records"
    a = _run(m, x0, s, S, bptt_budget=1 << 40)
    assert a[4][0] == "records"
    _bit_equal(a, _run(m, x0, s, S))


# ---- 2. resident checkpoints against the unbudgeted record path ------------------------------------------------------
# name: model, T, S, K / S, ragged steps, damage step, Philox, loss.  K = r * S is what the budget buys (r = None: one
# segment, K = the first multiple of S that covers T).  T > 16 for one segment: the record buffer is then sized for 64
# steps, so a budget of one segment leaves it out.
CASES = {
    "r1_TmodS0_damage_t0_ragged": ("torus", 12, 3, 1, [0, 3, 8, 12], 0, False, "both"),
    "r2_TmodS2_damage_frame_philox": ("torus", 14, 3, 2, None, 3, True, "both"),
    "r3_classic_damage_on_ckpt_ragged": ("classic", 13, 2, 3, [13, 5, 9, 1], 6, False, "both"),
    "r3_damage_inside_frames_only": ("torus", 15, 2, 3, [15, 4, 11, 7], 7, False, "frames"),
    "r2_TmodS0_xT_only": ("torus", 16, 4, 2, [16, 6, 12, 2], 9, True, "xT"),
    "one_segment_TmodS0": ("torus", 20, 4, None, [20, 8, 13, 3], 9, False, "both"),
    "one_segment_TmodS2_classic_philox": ("classic", 22, 4, None, [22, 0, 17, 9], 4, True, "frames"),
}


@pytest.mark.parametrize("case", list(CASES))
def test_resident_ckpt_equals_unbudgeted_record_path(case):
    model, T, S, r, steps, dmg, philox, which = CASES[case]
    m = MODELS[model]()
    B, H = 4, 40
    K = r * S if r is not None else -(-T // S) * S
    budget = _ckpt_bytes(m, B, H, H, K)
    assert bptt_plan(m, B, H, H, T, budget, every=S) == ("resident_ckpt", K, budget)
    x0 = _blob(B, 16, H, H, seed=1)
    s = _schedule(m, B, H, H, T, steps=steps, damage_step=dmg, philox=philox)
    ref = _run(m, x0, s, S, which)
    assert ref[4] is None                                       # the unbudgeted call: no plan
    got = _run(m, x0, s, S, which, bptt_budget=budget)
    assert got[4] == ("resident_ckpt", K, budget)
    assert torch.equal(got[0], ref[0]) and torch.equal(got[1], ref[1])
    assert torch.equal(got[2], ref[2]), float((got[2] - ref[2]).abs().max())
    assert rel_err(torch.cat([g.flatten() for g in got[3]]), torch.cat([g.flatten() for g in ref[3]])) <= 1e-6


def test_T0_resident():
    """T = 0 has no record buffer, so impl='resident' takes one checkpoint segment: g0 = gT + dL/dframe_0"""
    m = _graph16()
    x0 = _blob(2, 16, 40, 40)
    s = _schedule(m, 2, 40, 40, 0)
    got = _run(m, x0, s, 3, impl="resident", bptt_budget=1 << 40)
    assert got[4] == ("resident_ckpt", 3, _ckpt_bytes(m, 2, 40, 40, 3))
    ref = _run(m, x0, s, 3)
    _bit_equal(got, ref)
    assert torch.equal(got[0][0], x0) and torch.equal(got[1], x0)


# ---- 3. against the fp64 oracle -------------------------------------------------------------------------------------
@pytest.mark.parametrize("T,S,r,steps,dmg", [(10, 2, 2, [10, 5], 2), (9, 3, 1, [4, 9], 6)])
def test_resident_ckpt_vs_oracle(T, S, r, steps, dmg):
    """damage on a frame that is not a checkpoint (t = 2, K = 4) and on a checkpoint (t = 6, K = 3): the frame's
    gradient is added before the mask"""
    m = _graph16()
    B, H = 2, 40
    x0 = RG._blob(B, 16, H, H, seed=1)
    d = RG._draws(m, B, H, H, T, steps=steps, damage_step=dmg, seed=3)
    s = RG._schedule(m, B, H, H, T, d)
    xr, p, frames_ref, xT_ref = RG._oracle(m, x0, T, S, d)
    budget = _ckpt_bytes(m, B, H, H, r * S)
    RG._zero_grads(m)
    xg = x0.to(DEV).requires_grad_(True)
    tr = record_rollout(m, xg, s, every=S, differentiable=True, bptt_budget=budget)
    assert tr.x_T.grad_fn.plan == ("resident_ckpt", r * S, budget)
    assert rel_err(tr.states.detach().cpu(), frames_ref.detach()) < 1e-5
    RG._frame_loss(tr.states, tr.x_T).backward()
    RG._check_grads(m, xg, xr, p)


# ---- 4. the streaming fallback is checkpoint=True --------------------------------------------------------------------
@pytest.mark.parametrize("case", ["k17", "large_grid"])
def test_streaming_fallback_equals_checkpoint(case):
    m = _graph16()
    if case == "k17":
        B, H, W, T, S = 2, 40, 40, 12, 4
        offs = [[(dy, dx) for dy in (-2, -1, 1, 2) for dx in (-2, -1, 0, 1, 2)][:17] for _ in range(T)]
        s = make_schedule(m, B, H, W, T, offsets=offs, fire="philox", seed=7, fire_rate=0.5)
        assert s.k == 17
    else:
        B, H, W, T, S = 2, 48, 48, 10, 5
        assert H * W > 2048
        s = _schedule(m, B, H, W, T, philox=True)
    x0 = _blob(B, 16, H, W, seed=2)
    plan = bptt_plan(m, B, H, W, T, 1 << 40, every=S, k=s.k)
    assert plan[0] == "dense"
    budget = plan[2] - 1
    got = _run(m, x0, s, S, bptt_budget=budget)
    assert got[4][0] == "streaming_ckpt" and got[4][1] == S
    _bit_equal(got, _run(m, x0, s, S, checkpoint=True))


# ---- 5. T = 1000, B = 32 ---------------------------------------------------------------------------------------------
def test_T1000_B32_frames_every_50_within_budget_against_checkpoint():
    """40x40x16, B = 32, T = 1000, a frame every 50 steps.  The record buffer (72.9 GB) is above BPTT_MAX_BYTES; one
    resident segment of 50 steps takes 3.40 GiB, so a 4 GiB budget runs the resident checkpoints and a 3 GiB one the
    streaming checkpoints of checkpoint=True.  The distances between the two are those DESIGN section 3.10 records for
    1000-step drift."""
    m = _graph16()
    B, H, T, S = 32, 40, 1000, 50
    desc, packed = m.model_desc(), m.packed_weights()
    lib = G._lib.load()
    assert lib.gnca_bptt_bytes(C.byref(desc), B, H, H, T) > BPTT_MAX_BYTES
    budget = 4 << 30
    plan = bptt_plan(m, B, H, H, T, budget, every=S)
    assert plan == ("resident_ckpt", S, _ckpt_bytes(m, B, H, H, S)), plan
    assert bptt_plan(m, B, H, H, T, 3 << 30, every=S)[0] == "streaming_ckpt"
    x0 = _blob(B, 16, H, H, seed=4)
    s = _schedule(m, B, H, H, T, steps=[T - 13 * b for b in range(B)], philox=True)
    gen = torch.Generator().manual_seed(5)
    gT = (torch.randn(B, 16, H, H, generator=gen) * 1e-3).to(DEV)
    gF = (torch.randn(T // S + 1, B, 16, H, H, generator=gen) * 1e-3).to(DEV)
    GF._WS.get(x0.device, lib.gnca_rollout_workspace_bytes(C.byref(desc), B, H, H, T))
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    xT, hist = rollout_fwd_raw(desc, packed, x0, s, history=True, keep_x=False, every=S, bptt_budget=budget)
    assert hist.plan == plan
    g0, gflat = rollout_bwd_raw(desc, packed, hist, s, gT, g_frames=gF, every=S)
    torch.cuda.synchronize()
    peak = torch.cuda.max_memory_allocated() - base
    n = B * 16 * H * H * 4
    frames = hist.frames.numel() * 4
    # the frames, the history, the outputs x_T / g0 and the parameter gradient
    assert peak <= budget + frames + 2 * n + gflat.numel() * 4 + (1 << 20), (peak, budget)
    frames_r = hist.frames
    del hist
    xT_c, hist_c = rollout_fwd_raw(desc, packed, x0, s, history=True, keep_x=False, every=S, bptt_budget=3 << 30)
    assert hist_c.plan[0] == "streaming_ckpt"
    g0_c, gflat_c = rollout_bwd_raw(desc, packed, hist_c, s, gT, g_frames=gF, every=S)
    per = sorted(rel_err(g0[b], g0_c[b]) for b in range(B))
    print(f"T=1000 S=50 resident vs streaming checkpoints: frames {rel_err(frames_r, hist_c.frames):.3e}, "
          f"x_T {rel_err(xT, xT_c):.3e}, dL/dx0 per sample median {per[B // 2]:.3e} max {per[-1]:.3e}, "
          f"parameters {rel_err(gflat, gflat_c):.3e}")
    assert rel_err(xT, xT_c) <= 1e-4 and rel_err(frames_r, hist_c.frames) <= 1e-4
    assert per[B // 2] <= T1000_MEDIAN and per[-1] <= T1000_MAX, per
    assert rel_err(gflat, gflat_c) <= T1000_FRAMES_PARAMS, rel_err(gflat, gflat_c)


# ---- 6. errors and the autograd node ---------------------------------------------------------------------------------
def _resident_case():
    m = _graph16()
    x0 = _blob(2, 16, 40, 40)
    s = _schedule(m, 2, 40, 40, 8)
    return m, x0, s, _ckpt_bytes(m, 2, 40, 40, 4)


def test_errors():
    m, x0, s, budget = _resident_case()
    xg = x0.clone().requires_grad_(True)
    with pytest.raises(ValueError, match="checkpoint=True"):
        record_rollout(m, xg, s, every=2, differentiable=True, checkpoint=True, bptt_budget=budget)
    with pytest.raises(ValueError, match="differentiable=True"):
        record_rollout(m, xg, s, every=2, bptt_budget=budget)
    with pytest.raises(ValueError, match="impl"):
        record_rollout(m, xg, s, every=2, differentiable=True, impl="banded", bptt_budget=budget)
    with pytest.raises(ValueError, match=">= 0"):
        record_rollout(m, xg, s, every=2, differentiable=True, bptt_budget=-1)
    with pytest.raises(ValueError, match="smallest budget that works"):
        record_rollout(m, xg, s, every=2, differentiable=True, bptt_budget=1024)
    zp = _graph16(torus=False)
    with pytest.raises(ValueError, match="impl='resident'"):
        record_rollout(zp, xg, _schedule(zp, 2, 40, 40, 8), every=2, differentiable=True, impl="resident",
                       bptt_budget=1 << 40)


def test_in_place_edit_of_a_frame_raises():
    m, x0, s, budget = _resident_case()
    tr = record_rollout(m, x0.clone().requires_grad_(True), s, every=2, differentiable=True, bptt_budget=budget)
    assert tr.x_T.grad_fn.plan[0] == "resident_ckpt"
    loss = tr.states.sum() + _ell(tr.x_T)       # sum() saves no input: only the node's own saved frames can object
    with torch.no_grad():
        tr.states[1].mul_(2.0)
    with pytest.raises(RuntimeError, match="inplace"):
        loss.backward()


def test_second_backward_raises():
    m, x0, s, budget = _resident_case()
    tr = record_rollout(m, x0.clone().requires_grad_(True), s, every=2, differentiable=True, bptt_budget=budget)
    assert tr.x_T.grad_fn.plan[0] == "resident_ckpt"
    loss = tr.states.sum() + _ell(tr.x_T)
    loss.backward(retain_graph=True)
    with pytest.raises(RuntimeError, match="already consumed"):
        loss.backward()


def test_no_grad_is_the_detached_recording():
    m, x0, s, budget = _resident_case()
    with torch.no_grad():
        tr = record_rollout(m, x0.clone().requires_grad_(True), s, every=2, differentiable=True, bptt_budget=budget)
    ref = record_rollout(m, x0, s, every=2)
    assert not tr.states.requires_grad and not tr.x_T.requires_grad
    assert torch.equal(tr.states, ref.states) and torch.equal(tr.x_T, ref.x_T)

"""GPU tests of the checkpointed resident BPTT (gnca_rollout_fwd_bptt_ckpt / gnca_rollout_bwd_bptt_ckpt) and of the
BPTT memory budget of rollout(..., bptt_budget=...) and the trainer.

1. against the unsegmented resident BPTT: x_T and dL/dx0 bit for bit, parameter gradients to 1e-6, over strides,
   ragged steps, damage at t = 0 / inside a segment / on a checkpoint, Philox with an offset and gain-0 steps;
2. the checkpoints equal the frames of the record-writing forward; 3. T = 1000 at B = 32 on the resident kernels within a
   few GB, against the dense streaming BPTT; 4. budget selection; 5. the trainer; 6. errors."""
import ctypes as C
import random

import pytest
import torch

from conftest import load_params, rel_err

pytestmark = pytest.mark.gpu

if torch.cuda.is_available():
    import graph_neural_cellular_automata_b200 as G
    from graph_neural_cellular_automata_b200 import functional as GF
    from graph_neural_cellular_automata_b200.rollout import (_ckpt_bwd_raw, _ckpt_fwd_raw, bptt_plan, make_schedule,
                                                             rollout, rollout_bwd_raw, rollout_fwd_raw)

DEV = "cuda"


def _graph16(torus=True):
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


MODELS = {"torus": _graph16, "classic": _classic16}


def _blob(B, C_, H, W, seed=0):
    """random state inside a disk (alive cells with a dead border around them)"""
    g = torch.Generator().manual_seed(seed)
    yy, xx = torch.meshgrid(torch.arange(H), torch.arange(W), indexing="ij")
    disk = (((yy - H / 2) ** 2 + (xx - W / 2) ** 2) < (0.3 * min(H, W)) ** 2).float()
    return (torch.rand(B, C_, H, W, generator=g) * disk).to(DEV)


def _schedule(m, B, H, W, T, *, steps=None, damage_step=None, philox=False, seed=0):
    """per-step fire rates, gains (0 on t % 3 == 1), offsets, uniforms or Philox (with a nonzero counter offset)"""
    random.seed(seed)
    graph = getattr(m, "_is_graph", False)
    offs = [m.graph.draw_offsets() for _ in range(T)] if graph else None
    frs = [0.5 + 0.4 * ((7 * t) % 10) / 10 for t in range(T)]
    gains = [0.25 if t % 3 != 1 else 0.0 for t in range(T)] if graph else None
    dmg = None
    if damage_step is not None:
        dmg = torch.ones(B, m.n_channels, H, W)
        dmg[:, :, H // 3:H // 3 + H // 4, W // 4:W // 2] = 0.0
        dmg[0, :, H // 2:H // 2 + 3, :] = 0.5
        dmg = dmg.to(DEV)
    kw = dict(fire_rate=frs, offsets=offs, message_gains=gains, steps=steps, damage=dmg,
              damage_step=damage_step or 0)
    if philox:
        s = make_schedule(m, B, H, W, T, fire="philox", seed=4321, **kw)
        s.philox_offset = 987654
        return s
    fu = torch.rand(T, B, H, W, generator=torch.Generator().manual_seed(seed + 1)).to(DEV)
    return make_schedule(m, B, H, W, T, fire_u=fu, **kw)


def _unsegmented(m, x0, s, gT):
    """x_T, dL/dx0 and the flat parameter gradient of the resident BPTT with records (gnca_rollout_fwd/_bwd_bptt)"""
    desc, packed = m.model_desc(), m.packed_weights()
    xT, hist = rollout_fwd_raw(desc, packed, x0, s, history=True, impl=2, keep_x=False)
    assert hist.bptt is not None
    g0, gflat = rollout_bwd_raw(desc, packed, hist, s, gT, impl=2)
    return xT, g0, gflat


def _segmented(m, x0, s, gT, K):
    desc, packed = m.model_desc(), m.packed_weights()
    out = _ckpt_fwd_raw(desc, packed, x0, s, K, resident=True)
    assert out is not None
    xT, ckpt = out
    g0, gflat = _ckpt_bwd_raw(desc, packed, ckpt, s, K, True, gT)
    return xT, g0, gflat, ckpt


# ---- 1. against the unsegmented resident BPTT -----------------------------------------------------------------------
B1, H1, T1 = 4, 40, 12
KS = [1, 3, 8, T1 - 1, T1, T1 + 5]


def _inside(K):
    """a damage step strictly inside a segment, or None when every step starts one (K = 1) or K >= T"""
    if K == 1 or K >= T1:
        return None
    return K + K // 2 if K + K // 2 < T1 else K // 2


# name: (ragged steps, damage step as a function of K, Philox); None from the damage function: no such case
CASES = {
    "plain": (None, None, False),
    # sample 0 never steps, sample 3 runs every step; samples 1 and 2 freeze at t = 3 and t = 8: on a checkpoint for
    # K = 3 and K = 8, inside a segment for the other one
    "ragged": ([0, 3, 8, T1], None, False),
    "damage_t0": (None, lambda K: 0, False),
    "damage_inside": (None, _inside, False),
    "damage_on_ckpt": (None, lambda K: K if K < T1 else None, False),
    "philox_ragged_damage": ([T1, 5, 9, 1], _inside, True),
}


def test_unsegmented_resident_backward_is_deterministic():
    m = _graph16()
    x0 = _blob(B1, 16, H1, H1)
    s = _schedule(m, B1, H1, H1, T1, steps=[0, 3, 8, T1], damage_step=5)
    gT = torch.randn(B1, 16, H1, H1, generator=torch.Generator().manual_seed(3)).to(DEV)
    a = _unsegmented(m, x0, s, gT)
    b = _unsegmented(m, x0, s, gT)
    assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])


@pytest.mark.parametrize("K", KS)
@pytest.mark.parametrize("model", list(MODELS))
@pytest.mark.parametrize("case", list(CASES))
def test_segmented_equals_unsegmented_resident(case, model, K):
    steps, dmg_fn, philox = CASES[case]
    dmg = dmg_fn(K) if dmg_fn is not None else None
    if dmg_fn is not None and dmg is None:
        pytest.skip("no such damage step for this stride")
    m = MODELS[model]()
    x0 = _blob(B1, 16, H1, H1)
    s = _schedule(m, B1, H1, H1, T1, steps=steps, damage_step=dmg, philox=philox)
    gT = torch.randn(B1, 16, H1, H1, generator=torch.Generator().manual_seed(3)).to(DEV)
    xT_u, g0_u, gp_u = _unsegmented(m, x0, s, gT)
    xT_s, g0_s, gp_s, _ = _segmented(m, x0, s, gT, K)
    assert torch.equal(xT_s, xT_u)
    assert torch.equal(g0_s, g0_u), float((g0_s - g0_u).abs().max())
    assert rel_err(gp_s, gp_u) <= 1e-6, rel_err(gp_s, gp_u)


@pytest.mark.parametrize("K", [1, 4, 10])
def test_T0_copies_the_gradient(K):
    m = _graph16()
    x0 = _blob(2, 16, 40, 40)
    s = _schedule(m, 2, 40, 40, 0)
    gT = torch.randn(2, 16, 40, 40, device=DEV)
    xT, g0, gflat, ckpt = _segmented(m, x0, s, gT, K)
    assert torch.equal(xT, x0) and torch.equal(ckpt[0], x0)
    assert torch.equal(g0, gT) and float(gflat.abs().max()) == 0.0


# ---- 2. the recompute reproduces the forward -------------------------------------------------------------------------
@pytest.mark.parametrize("K", [1, 3, 5, 12])
@pytest.mark.parametrize("model", list(MODELS))
def test_checkpoints_equal_record_frames(model, K):
    m = MODELS[model]()
    x0 = _blob(B1, 16, H1, H1, seed=2)
    s = _schedule(m, B1, H1, H1, T1, steps=[T1, 5, 9, 1], damage_step=6, philox=True)
    desc, packed = m.model_desc(), m.packed_weights()
    xT_r, hist = rollout_fwd_raw(desc, packed, x0, s, history=True, impl=2, keep_x=False, every=K)
    assert hist.bptt is not None
    xT_c, ckpt = _ckpt_fwd_raw(desc, packed, x0, s, K, resident=True)
    assert torch.equal(ckpt, hist.frames)
    assert torch.equal(xT_c, xT_r)


# ---- 3. beyond the record buffer's limit -----------------------------------------------------------------------------
T_LONG = 1000


def _long_case(m, B):
    """x0, a ragged Philox schedule (samples run 1000 down to 1000 - 13 (B - 1) steps) and dL/dx_T at 40x40, T = 1000"""
    x0 = _blob(B, 16, 40, 40, seed=4)
    s = _schedule(m, B, 40, 40, T_LONG, steps=[T_LONG - 13 * b for b in range(B)], philox=True)
    gT = (torch.randn(B, 16, 40, 40, generator=torch.Generator().manual_seed(5)) * 1e-3).to(DEV)
    return x0, s, gT


def test_T1000_segmented_equals_unsegmented_resident():
    """T = 1000 with 42-step segments against the unsegmented resident BPTT (its 18.2 GB record buffer at B = 8 allocated
    through the C ABI): x_T and dL/dx0 bit-equal, parameters to 1e-6"""
    m = _graph16()
    B, H, K = 8, 40, 42
    desc, packed = m.model_desc(), m.packed_weights()
    lib = G._lib.load()
    x0, s, gT = _long_case(m, B)
    xT, g0, gflat, _ = _segmented(m, x0, s, gT, K)
    nrec = lib.gnca_bptt_bytes(C.byref(desc), B, H, H, T_LONG)
    ws = GF._WS.get(x0.device, lib.gnca_rollout_workspace_bytes(C.byref(desc), B, H, H, T_LONG))
    cs = s.c_struct()
    bptt = torch.empty(nrec, dtype=torch.uint8, device=DEV)
    xT_u, g0_u = torch.empty_like(x0), torch.empty_like(x0)
    gflat_u = torch.zeros_like(gflat)
    G._lib.check(lib.gnca_rollout_fwd_bptt(C.byref(desc), GF._ptr(packed), B, H, H, C.byref(cs), GF._ptr(x0),
                                           GF._ptr(xT_u), None, GF._ptr(bptt), nrec, GF._ptr(ws), ws.numel(),
                                           GF._stream()), "gnca_rollout_fwd_bptt")
    G._lib.check(lib.gnca_rollout_bwd_bptt(C.byref(desc), GF._ptr(packed), B, H, H, C.byref(cs), GF._ptr(bptt), nrec,
                                           GF._ptr(gT), GF._ptr(g0_u), GF._ptr(gflat_u), GF._ptr(ws), ws.numel(),
                                           GF._stream()), "gnca_rollout_bwd_bptt")
    del bptt
    assert torch.equal(xT, xT_u)
    assert torch.equal(g0, g0_u), float((g0 - g0_u).abs().max())
    assert rel_err(gflat, gflat_u) <= 1e-6, rel_err(gflat, gflat_u)


# Distances of the resident BPTT to the dense streaming BPTT in this case (DESIGN section 3.10): the section 4 bounds
# (median 1e-4, every sample 5e-3, parameters 1e-4) are stated for 64-step rollouts; over 600 - 1000 steps the two
# summation orders drift further apart.  Measured on an NVIDIA B200 (1000 W): x_T 1.49e-5; dL/dx0 per sample median
# 8.12e-4, max 9.05e-3; parameters 8.33e-4, the same in two runs.  The unsegmented resident BPTT has the same distances
# (test above: it is bit-equal to the segmented one).
T1000_MEDIAN, T1000_MAX, T1000_PARAMS = 1e-3, 1.2e-2, 1e-3


def test_T1000_B32_resident_within_budget_against_dense_streaming():
    """40x40x16, B = 32, T = 1000: the record buffer (72.9 GB) is above BPTT_MAX_BYTES, so rollout() without a budget
    takes the dense streaming history.  A 3 GiB budget runs the resident kernels instead, within the budget."""
    m = _graph16()
    B, H = 32, 40
    budget = 3 << 30
    desc, packed = m.model_desc(), m.packed_weights()
    lib = G._lib.load()
    assert lib.gnca_bptt_bytes(C.byref(desc), B, H, H, T_LONG) > (48 << 30)       # above the record buffer's limit
    plan = bptt_plan(m, B, H, H, T_LONG, budget)
    assert plan[0] == "resident_ckpt" and plan[1] < T_LONG and plan[2] <= budget, plan
    x0, s, gT = _long_case(m, B)
    GF._WS.get(x0.device, lib.gnca_rollout_workspace_bytes(C.byref(desc), B, H, H, T_LONG))
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    xT, hist = rollout_fwd_raw(desc, packed, x0, s, history=True, keep_x=False, bptt_budget=budget)
    assert hist.plan == plan
    g0, gflat = rollout_bwd_raw(desc, packed, hist, s, gT)
    torch.cuda.synchronize()
    peak = torch.cuda.max_memory_allocated() - base
    n = B * 16 * H * H * 4
    # the history, the outputs x_T / g0 and the parameter gradient; the segment's temporaries are part of the plan
    assert peak <= budget + 2 * n + gflat.numel() * 4 + (1 << 20), (peak, budget)
    del hist
    xT_d, hist_d = rollout_fwd_raw(desc, packed, x0, s, history=True, impl=1)
    g0_d, gflat_d = rollout_bwd_raw(desc, packed, hist_d, s, gT, impl=1)
    per = sorted(rel_err(g0[b], g0_d[b]) for b in range(B))
    print(f"T=1000 vs dense streaming: x_T {rel_err(xT, xT_d):.3e}, dL/dx0 per sample median {per[B // 2]:.3e} "
          f"max {per[-1]:.3e}, parameters {rel_err(gflat, gflat_d):.3e}")
    assert rel_err(xT, xT_d) <= 1e-4, rel_err(xT, xT_d)
    assert per[B // 2] <= T1000_MEDIAN and per[-1] <= T1000_MAX, per
    assert rel_err(gflat, gflat_d) <= T1000_PARAMS, rel_err(gflat, gflat_d)


# ---- 4. budget selection ---------------------------------------------------------------------------------------------
def _grads_of(m, x0, s, **kw):
    for q in m.parameters():
        q.grad = None
    xg = x0.clone().requires_grad_(True)
    xT = rollout(m, xg, s, **kw)
    ((xT[:, :4] ** 2).mean() + 0.1 * xT[:, 4:].mean()).backward()
    return xT.detach(), xg.grad, [q.grad.clone() if q.grad is not None else torch.zeros_like(q) for q in m.parameters()]


def _bit_equal(a, b):
    assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])
    for ga, gb in zip(a[2], b[2]):
        assert torch.equal(ga, gb)


@pytest.mark.parametrize("model", list(MODELS))
def test_budget_covering_unsegmented_path_is_bit_identical(model):
    m = MODELS[model]()
    x0 = _blob(B1, 16, H1, H1)
    s = _schedule(m, B1, H1, H1, T1, steps=[0, 3, 8, T1], damage_step=0)
    assert bptt_plan(m, B1, H1, H1, T1, 1 << 40)[0] == "records"
    _bit_equal(_grads_of(m, x0, s, bptt_budget=1 << 40), _grads_of(m, x0, s))


def test_budget_below_records_takes_resident_ckpt():
    m = _graph16()
    x0 = _blob(B1, 16, H1, H1)
    s = _schedule(m, B1, H1, H1, T1, steps=[0, 3, 8, T1], damage_step=4)
    full = bptt_plan(m, B1, H1, H1, T1, 1 << 40)[2]
    path, K, nb = bptt_plan(m, B1, H1, H1, T1, full // 3)
    assert path == "resident_ckpt" and 1 <= K < T1 and nb <= full // 3
    a = _grads_of(m, x0, s, bptt_budget=full // 3)
    b = _grads_of(m, x0, s)
    assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])
    for ga, gb in zip(a[2], b[2]):
        if float(gb.abs().max()) == 0.0:
            assert float(ga.abs().max()) == 0.0
        else:
            assert rel_err(ga, gb) <= 1e-6, rel_err(ga, gb)


def test_zeropad_model_takes_streaming_ckpt():
    m = _graph16(torus=False)
    x0 = _blob(B1, 16, H1, H1)
    s = _schedule(m, B1, H1, H1, T1, steps=[0, 3, 8, T1], damage_step=4)
    dense = bptt_plan(m, B1, H1, H1, T1, 1 << 40)
    assert dense[0] == "dense"
    path, K, _ = bptt_plan(m, B1, H1, H1, T1, dense[2] // 2)
    assert path == "streaming_ckpt" and K < T1
    _bit_equal(_grads_of(m, x0, s, bptt_budget=dense[2] // 2), _grads_of(m, x0, s, checkpoint_every=K))


def test_large_grid_takes_streaming_ckpt():
    torch.manual_seed(5); random.seed(5)
    m = G.NeuralCAGraph(32, update_hidden=128, img_size=256, update_gain=0.1, alpha_thr=0.1, message_gain=0.3,
                        hidden_only=True, graph_zero_padded_shift=False)
    with torch.no_grad():
        m.update_net[2].weight.normal_(0, 0.05)
    m = m.to(DEV)
    B, H, T = 2, 256, 6
    x0 = _blob(B, 32, H, H, seed=7)
    s = _schedule(m, B, H, H, T, philox=True)
    assert bptt_plan(m, B, H, H, T, 1 << 40)[0] == "dense"
    lib = G._lib.load()
    desc = m.model_desc()
    # checkpoints + segment of K = 3 (8 states): K = 4, 5, 6 need 9, 11, 13 states
    budget = (T // 3 + 1) * B * 32 * H * H * 4 + lib.gnca_ckpt_segment_bytes(C.byref(desc), B, H, H, 3)
    path, K, _ = bptt_plan(m, B, H, H, T, budget)
    assert (path, K) == ("streaming_ckpt", 3)
    _bit_equal(_grads_of(m, x0, s, bptt_budget=budget), _grads_of(m, x0, s, checkpoint_every=K))


# ---- 5. the trainer --------------------------------------------------------------------------------------------------
def _train_two_steps(budget):
    from graph_neural_cellular_automata_b200.training.trainer import GraphNCATrainer, TrainConfig
    torch.manual_seed(21); random.seed(21)
    m = _graph16()
    cfg = TrainConfig(batch_size=8, pool_size=16, long_rollout_prob=1.0, long_rollout_steps_min=60,
                      long_rollout_steps_max=90, fire_rate_min=0.5, fire_rate_max=0.9, message_every=3,
                      reset_worst_prob=0.25, random_reseed_prob=0.0, damage={}, fire="philox", bptt_budget_bytes=budget)
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
        out.append((r["per_sample"].clone(), None if r["worst"] is None else r["worst"].clone(), int(r["steps"].max())))
    return out, [q.detach().clone() for q in m.parameters()]


def test_trainer_budget_matches_unbudgeted():
    budget = 256 << 20
    a, pa = _train_two_steps(None)
    b, pb = _train_two_steps(budget)
    for (la, wa, Ta), (lb, wb, Tb) in zip(a, b):
        assert Ta == Tb
        plan = bptt_plan(_graph16(), 8, 40, 40, Tb, budget)
        assert plan[0] == "resident_ckpt" and plan[1] < Tb, plan
        assert rel_err(lb, la) <= 1e-6, rel_err(lb, la)
        assert (wa is None) == (wb is None) and (wa is None or torch.equal(wa, wb))
    for qa, qb in zip(pa, pb):
        assert rel_err(qb, qa) <= 1e-6, rel_err(qb, qa)


# ---- 6. errors -------------------------------------------------------------------------------------------------------
def test_budget_errors():
    m = _graph16()
    x0 = _blob(2, 16, 40, 40).requires_grad_(True)
    s = _schedule(m, 2, 40, 40, 8)
    for kw in (dict(impl="banded"), dict(checkpoint_every=2), dict(return_history=True)):
        with pytest.raises(ValueError):
            rollout(m, x0, s, bptt_budget=1 << 30, **kw)
    with pytest.raises(ValueError, match="smallest budget"):
        rollout(m, x0, s, bptt_budget=1024)
    zp = _graph16(torus=False)
    with pytest.raises(ValueError, match="resident"):
        rollout(zp, x0, _schedule(zp, 2, 40, 40, 8), bptt_budget=1 << 30, impl="resident")


def test_second_backward_raises():
    m = _graph16()
    x0 = _blob(2, 16, 40, 40)
    s = _schedule(m, 2, 40, 40, 8)
    full = bptt_plan(m, 2, 40, 40, 8, 1 << 40)[2]
    assert bptt_plan(m, 2, 40, 40, 8, full // 2)[0] == "resident_ckpt"
    xg = x0.clone().requires_grad_(True)
    loss = rollout(m, xg, s, bptt_budget=full // 2).square().mean()
    loss.backward(retain_graph=True)
    with pytest.raises(RuntimeError):
        loss.backward()

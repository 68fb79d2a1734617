"""GPU tests of the recording rollout (gnca_rollout_record through rollout.record_rollout).

Frames are pinned bit for bit to the full history of gnca_rollout_fwd on the same impl (x_hist[::S]); x_T to the plain
rollout; the streaming frames to the sequential module.step loop; every attention map to the map module.step returns
for that frame and step.  Models, states and schedules are built here."""
import ctypes as C
import random

import numpy as np
import pytest
import torch

from conftest import load_params, rel_err

pytestmark = pytest.mark.gpu

if torch.cuda.is_available():
    import graph_neural_cellular_automata_b200 as G
    from graph_neural_cellular_automata_b200 import _lib
    from graph_neural_cellular_automata_b200 import functional as GF
    from graph_neural_cellular_automata_b200.rollout import IMPL, make_schedule, record_rollout, rollout

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


def _random_graph(C, H, seed=5):
    torch.manual_seed(seed); random.seed(seed)
    m = G.NeuralCAGraph(C, update_hidden=128, img_size=H, update_gain=0.1, alpha_thr=0.1, message_gain=0.3,
                        hidden_only=True, graph_zero_padded_shift=False)
    with torch.no_grad():
        m.update_net[2].weight.normal_(0, 0.05)
        m.norm.weight.uniform_(0.5, 1.5); m.norm.bias.normal_(0, 0.1)
    return m.to(DEV)


MODELS = {"torus": lambda: _graph16(True), "zeropad": lambda: _graph16(False), "classic": _classic16}


def _blob(B, C, H, W, seed=0):
    """random state inside a disk (alive cells with a dead border around them)"""
    g = torch.Generator().manual_seed(seed)
    yy, xx = torch.meshgrid(torch.arange(H), torch.arange(W), indexing="ij")
    disk = (((yy - H / 2) ** 2 + (xx - W / 2) ** 2) < (0.3 * min(H, W)) ** 2).float()
    return (torch.rand(B, C, H, W, generator=g) * disk).to(DEV)


def _case_schedule(m, B, H, W, T, *, fire="u", steps=None, damage_step=None, k=None, seed=0):
    """per-step fire rates and gains (some 0), recorded uniforms or in-kernel Philox, optional damage and ragged steps"""
    random.seed(seed)
    graph = getattr(m, "_is_graph", False)
    offs = None
    if graph:
        offs = [m.graph.draw_offsets() for _ in range(T)] if k is None else [[] for _ in range(T)]
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
    return s, dict(offs=offs, frs=frs, gains=gains, fu=fu, dmg=dmg, steps=steps)


def _fwd_full(m, x0, s, impl):
    """gnca_rollout_fwd with the full [T+1] history, straight through the C ABI -> (rc, x_T, x_hist)"""
    lib = _lib.load()
    desc = m.model_desc()
    B, Cc, H, W = x0.shape
    xT = torch.empty_like(x0)
    hist = torch.empty(s.T + 1, B, Cc, H, W, device=DEV)
    ws = GF._WS.get(x0.device, lib.gnca_rollout_workspace_bytes(C.byref(desc), B, H, W, s.T))
    cs = s.c_struct()
    rc = lib.gnca_rollout_fwd(C.byref(desc), GF._ptr(m.packed_weights()), B, H, W, C.byref(cs), GF._ptr(x0),
                              GF._ptr(xT), GF._ptr(hist), None, None, GF._ptr(ws), ws.numel(), IMPL[impl], GF._stream())
    return rc, xT, hist


def _record_or_skip(m, x0, s, impl, every, attention=False):
    """Record on `impl`; a combination gnca_rollout_fwd rejects as unsupported must be rejected by the recording
    rollout too, and is then skipped."""
    rc, xT_full, hist = _fwd_full(m, x0, s, impl)
    if rc == _lib.GNCA_ERR_UNSUPPORTED:
        with pytest.raises(_lib.GncaError, match="unsupported"):
            record_rollout(m, x0, s, every=every, attention=attention, impl=impl)
        pytest.skip(f"{impl}: no kernel for this configuration")
    _lib.check(rc, "gnca_rollout_fwd")
    tr = record_rollout(m, x0, s, every=every, attention=attention, impl=impl)
    return tr, xT_full, hist


def _sequential(m, x0, T, d):
    """x_0..x_T of T module.step calls with the schedule's draws (frozen samples kept, damage before its step)"""
    xs = [x0]
    x = x0
    for t in range(T):
        if d["dmg"] is not None and t == d["dmg_step"]:
            x = x * d["dmg"]
            xs[-1] = x
        kw = dict(fire_u=d["fu"][t].unsqueeze(1))
        if d["offs"] is not None:
            kw.update(chosen=d["offs"][t], message_gain=d["gains"][t])
        y = m.step(x, d["frs"][t], **kw)
        if d["steps"] is not None:
            frozen = torch.tensor([st <= t for st in d["steps"]], device=DEV)
            y = torch.where(frozen[:, None, None, None], x, y)
        x = y
        xs.append(x)
    return xs


# name: T, every, fire, ragged steps, damage step
STATE_CASES = {
    "S1": (7, 1, "u", None, None),
    "S3_T%S!=0": (10, 3, "u", None, None),
    "S=T": (9, 9, "u", None, None),
    "S=T+1": (9, 10, "u", None, None),
    "T0": (0, 1, "u", None, None),
    "T0_S3": (0, 3, "u", None, None),
    "ragged_philox_damage_at_frame": (10, 3, "philox", [10, 4], 6),
    "ragged_u_damage_between_frames": (11, 3, "u", [5, 11], 4),
    "damage_at_frame_S2": (8, 2, "u", None, 2),
}


@pytest.mark.parametrize("impl", IMPLS)
@pytest.mark.parametrize("model", list(MODELS))
@pytest.mark.parametrize("case", list(STATE_CASES))
def test_frames_equal_strided_history(case, model, impl):
    T, S, fire, steps, dstep = STATE_CASES[case]
    m = MODELS[model]()
    B, H, W = 2, 40, 40
    x0 = _blob(B, 16, H, W, seed=1)
    s, d = _case_schedule(m, B, H, W, T, fire=fire, steps=steps, damage_step=dstep, seed=3)
    with torch.no_grad():
        tr, xT_full, hist = _record_or_skip(m, x0, s, impl, S)
        xT_plain = rollout(m, x0, s, impl=impl)
    F = T // S + 1
    assert tr.t == [f * S for f in range(F)]
    assert tuple(tr.states.shape) == (F, B, 16, H, W)
    assert tr.attention is None
    assert torch.equal(tr.states, hist[::S]), case
    assert torch.equal(tr.x_T, xT_full) and torch.equal(tr.x_T, xT_plain)
    assert not tr.states.requires_grad and tr.states.grad_fn is None
    if impl != "streaming":
        # a defect in a kernel's history store moves x_hist and the frames alike: compare with the streaming frames
        with torch.no_grad():
            ref = record_rollout(m, x0, s, every=S, impl="streaming")
        for f in range(F):
            assert rel_err(tr.states[f], ref.states[f]) < 1e-5, (case, f, rel_err(tr.states[f], ref.states[f]))
    if impl == "streaming" and fire == "u":
        d["dmg_step"] = dstep
        with torch.no_grad():
            xs = _sequential(m, x0, T, d)
        for f in range(F):
            assert torch.equal(tr.states[f], xs[f * S]), (case, f)
        assert torch.equal(tr.x_T, xs[T])


@pytest.mark.parametrize("impl", ["resident", "banded"])
def test_frames_c32_banded(impl):
    """C = 32 at 40x40 runs on the banded cluster kernel (the replicated-state kernel is C = 16 only)"""
    m = _random_graph(32, 40)
    B, H, W, T, S = 3, 40, 40, 13, 4
    x0 = _blob(B, 32, H, W, seed=2)
    s, _ = _case_schedule(m, B, H, W, T, fire="philox", steps=[13, 6, 13], damage_step=8, seed=4)
    with torch.no_grad():
        tr, xT_full, hist = _record_or_skip(m, x0, s, impl, S, attention=True)
        xT_plain = rollout(m, x0, s, impl=impl)
    assert torch.equal(tr.states, hist[::S])
    assert torch.equal(tr.x_T, xT_full) and torch.equal(tr.x_T, xT_plain)
    with torch.no_grad():
        ref = record_rollout(m, x0, s, every=S, impl="streaming")
    for f in range(T // S + 1):
        assert rel_err(tr.states[f], ref.states[f]) < 1e-5, (f, rel_err(tr.states[f], ref.states[f]))
    _check_attention(m, tr, s, S)


def test_frames_large_problem_path():
    """256x256x32, B = 5: B * ceil(HW / 1024) = 320 >= 296 chunks, the balanced tensor-core update (k_update_tc)"""
    m = _random_graph(32, 256)
    B, H, W, T, S = 5, 256, 256, 12, 5
    x0 = _blob(B, 32, H, W, seed=3)
    s, _ = _case_schedule(m, B, H, W, T, fire="philox", damage_step=5, seed=6)
    with torch.no_grad():
        tr, xT_full, hist = _record_or_skip(m, x0, s, "streaming", S, attention=True)
        xT_plain = rollout(m, x0, s, impl="auto")
    assert tr.t == [0, 5, 10]
    assert torch.equal(tr.states, hist[::S])
    assert torch.equal(tr.x_T, xT_full) and torch.equal(tr.x_T, xT_plain)
    _check_attention(m, tr, s, S)


def _check_attention(m, tr, s, S):
    T = s.T
    FA = -(-T // S)
    assert tuple(tr.attention.shape) == (FA,) + tuple(tr.states.shape[1:2]) + tuple(tr.states.shape[3:])
    offs = s.offsets.cpu().numpy() if s.offsets is not None else np.zeros((T, 0, 2), np.int8)
    gains = s.message_gain.cpu().numpy()
    frs = s.fire_rate.cpu().numpy()
    B, _, H, W = tr.x_T.shape
    fu = torch.rand(B, 1, H, W, device=DEV)          # the map depends on neither the fire draw nor the gain
    with torch.no_grad():
        for f in range(FA):
            t = f * S
            chosen = [tuple(int(v) for v in o) for o in offs[t]]
            _, ref = m.step(tr.states[f], float(frs[t]), fire_u=fu, chosen=chosen, message_gain=float(gains[t]),
                            return_attention=True)
            assert torch.equal(tr.attention[f], ref), f


@pytest.mark.parametrize("impl", IMPLS)
@pytest.mark.parametrize("model", ["torus", "zeropad"])
@pytest.mark.parametrize("case", ["S1", "S3_ragged_damage", "S4_k0"])
def test_attention_frames_equal_module_step(case, model, impl):
    m = MODELS[model]()
    B, H, W = 2, 40, 40
    x0 = _blob(B, 16, H, W, seed=5)
    if case == "S1":
        T, S, kw = 6, 1, {}
    elif case == "S3_ragged_damage":
        T, S, kw = 11, 3, dict(steps=[11, 4], damage_step=3, fire="philox")
    else:
        T, S, kw = 9, 4, dict(k=0)
    s, _ = _case_schedule(m, B, H, W, T, seed=8, **kw)
    with torch.no_grad():
        tr, _, hist = _record_or_skip(m, x0, s, impl, S, attention=True)
    assert torch.equal(tr.states, hist[::S])
    _check_attention(m, tr, s, S)
    if case == "S4_k0":
        assert not tr.attention.any()


def test_attention_on_classic_model_raises():
    m = _classic16()
    x0 = _blob(2, 16, 40, 40)
    s, _ = _case_schedule(m, 2, 40, 40, 4)
    with pytest.raises(ValueError):
        record_rollout(m, x0, s, every=2, attention=True)


def test_attention_t0_is_empty():
    m = _graph16(True)
    x0 = _blob(2, 16, 40, 40)
    s, _ = _case_schedule(m, 2, 40, 40, 0)
    tr = record_rollout(m, x0, s, every=3, attention=True)
    assert tuple(tr.attention.shape) == (0, 2, 40, 40)
    assert torch.equal(tr.states[0], x0) and torch.equal(tr.x_T, x0)


def test_resident_recording_allocates_no_record_buffer():
    """B = 8, T = 300 on the resident kernel: the BPTT record buffer of this shape is GBs; a recording rollout
    allocates the frames, the attention maps and nothing else of that order"""
    m = _graph16(True)
    B, H, W, T, S = 8, 40, 40, 300, 10
    x0 = _blob(B, 16, H, W, seed=9)
    s = make_schedule(m, B, H, W, T, fire_rate=0.5, seed=11)
    torch.cuda.synchronize()
    with torch.no_grad():
        record_rollout(m, x0, s, every=S, attention=True, impl="resident")         # workspace warm
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    base = torch.cuda.memory_allocated()
    with torch.no_grad():
        tr = record_rollout(m, x0, s, every=S, attention=True, impl="resident")
    torch.cuda.synchronize()
    out_bytes = tr.states.numel() * 4 + tr.attention.numel() * 4 + tr.x_T.numel() * 4
    assert torch.cuda.max_memory_allocated() - base < out_bytes + (64 << 20)
    lib = _lib.load()
    assert lib.gnca_bptt_bytes(C.byref(m.model_desc()), B, H, W, T) > out_bytes + (64 << 20)

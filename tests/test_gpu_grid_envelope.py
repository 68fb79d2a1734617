"""The cluster kernels against the fp64 oracle across the grid shapes `impl="auto"` sends them, not only 40x40.

Replicated-state forward (k_rep_fwd) and resident BPTT (k_rep_bwd) take C = 16, hidden 128, W % 4 == 0, H, W <= 64 and
H * W <= 2048; their setup depends on the grid: the padded plane and one quad of cells per thread, 64-word bitmaps that
are full at 2048 cells and end in a partial word when H * W % 32 != 0, the in-smem `u` buffer that shrinks near 2048
cells (the rest overflows to global memory), the backward's cluster size (H * W % (4 * NC) == 0, so forward and backward
can pick different NC), the per-row sums of the zero-padded shift.  The banded kernel (k_resident_fwd) takes C in
{4, 8, 16, 32}, hidden 128 and W <= 255 with NC | H, bands at least one halo deep and the tile MB stepping 64 -> 32 -> 16
to fit shared memory.

Every case runs the library against autograd through oracle/nca_oracle.py in fp64 with the same fire uniforms, offsets,
per-step fire rates, gains and damage, at the bounds of test_gpu_hparams.check_rollout: state 1e-5 rel-Frobenius, alive
mask bit-exact, dL/dx0 per-sample median 1e-5 and whole tensor 5e-4, parameter gradients 1e-4, query / key / scaling
gradients 1e-3 under the zero-padded shift and <= 1e-7 absolute on the torus.  Every case also reads the launch lines
GNCA_DEBUG=1 prints and asserts which family ran with which cluster size, `ucap` / overflow and MB, so a silent
fallback to another kernel fails the test.  The expected configurations follow from the shared-memory formulas of
rep_smem_bytes, rep_bwd_smem_bytes and resident_smem_bytes with a 227 KB opt-in limit per block (B200)."""
import ctypes as C
import random
import re
from dataclasses import dataclass, field
from typing import List, Optional

import pytest
import torch

from conftest import rel_err
from oracle import nca_oracle as O

pytestmark = pytest.mark.gpu

if torch.cuda.is_available():
    import graph_neural_cellular_automata_b200 as G
    from graph_neural_cellular_automata_b200 import _lib
    from graph_neural_cellular_automata_b200 import functional as GF
    from graph_neural_cellular_automata_b200.rollout import (bptt_plan, make_schedule, monitor_rollout, record_rollout,
                                                             rollout)
    from graph_neural_cellular_automata_b200.utils import metrics as UM

DEV = "cuda"
QKS = ("query_proj", "key_proj", "scaling")
RE_REP = re.compile(r"\[gnca\] replicated fwd: B=(\d+) NC=(\d+) ucap=(\d+) over=(\d+)")
RE_BAND = re.compile(r"\[gnca\] resident fwd: B=(\d+) NC=(\d+) own_rows=(\d+) halo=(\d+) MB=(\d+)")
RE_BWD = re.compile(r"\[gnca\] resident bwd: B=(\d+) NC=(\d+)")


# ---- fixtures and helpers -------------------------------------------------------------------------------------------
@dataclass
class Launches:
    rep: List[tuple] = field(default_factory=list)     # (B, NC, ucap, over) of every k_rep_fwd launch
    band: List[tuple] = field(default_factory=list)    # (B, NC, own_rows, halo, MB) of every k_resident_fwd launch
    bwd: List[tuple] = field(default_factory=list)     # (B, NC) of every k_rep_bwd launch
    text: str = ""


@pytest.fixture
def launches(monkeypatch, capfd):
    """GNCA_DEBUG=1 for the test; calling the fixture's value returns the launch lines printed since the last call"""
    monkeypatch.setenv("GNCA_DEBUG", "1")
    monkeypatch.delenv("GNCA_RESIDENT_NC", raising=False)
    capfd.readouterr()

    def read():
        err = capfd.readouterr().err
        ints = lambda m: tuple(int(v) for v in m.groups())
        return Launches([ints(m) for m in RE_REP.finditer(err)], [ints(m) for m in RE_BAND.finditer(err)],
                        [ints(m) for m in RE_BWD.finditer(err)], err)
    return read


def _model(kind, C=16, *, k=8, radius=3, d=16, seed=0):
    torch.manual_seed(seed); random.seed(seed)
    if kind == "classic":
        m = G.NeuralCA(C, update_hidden=128, img_size=32, update_gain=0.1, alpha_thr=0.1)
    else:
        # at C <= 8 the message reaches the RGBA channels too (hidden_only would leave C = 4 without a message)
        m = G.NeuralCAGraph(C, update_hidden=128, img_size=32, update_gain=0.1, alpha_thr=0.1, message_gain=0.4,
                            hidden_only=C > 8, graph_d_model=d, graph_attention_radius=radius, graph_num_neighbors=k,
                            graph_zero_padded_shift=kind == "zeropad")
    with torch.no_grad():
        m.update_net[2].weight.normal_(0, 0.05)
        m.norm.weight.uniform_(0.5, 1.5); m.norm.bias.normal_(0, 0.1)
    return m.to(DEV)


def _state(B, C, H, W, seed=0):
    """an off-centre alive blob (the torus wrap and the zero-padded rows both matter), ragged alive sets on odd samples"""
    g = torch.Generator().manual_seed(seed)
    yy, xx = torch.meshgrid(torch.arange(H), torch.arange(W), indexing="ij")
    disk = ((((yy - 0.45 * H) / H) ** 2 + ((xx - 0.55 * W) / W) ** 2) < 0.16).float()
    x = torch.rand(B, C, H, W, generator=g) * disk
    x[1::2, 3] *= (torch.rand(B // 2, H, W, generator=g) > 0.4).float()
    return x


def _loss(x):
    return (x[:, :4] ** 2).mean() + (0.1 * x[:, 4:].mean() if x.shape[1] > 4 else 0.0)


def _cfg(m, gain):
    g = getattr(m, "graph", None)
    return O.StepConfig(update_gain=m.update_gain, alpha_thr=m.alpha_thr, graph=g is not None, message_gain=gain,
                        hidden_only=bool(m.hidden_only) if g is not None else False,
                        zero_padded_shift=bool(g.zero_padded_shift) if g is not None else False)


@dataclass
class Draws:
    """the random draws of one rollout, fed to both the library and the oracle"""
    T: int
    chosen: list
    fu: torch.Tensor                  # [T, B, H, W]
    frs: list
    gains: list
    steps: Optional[list]
    dmg: Optional[torch.Tensor]       # [B, C, H, W] multiplicative mask, applied before step dstep
    dstep: int


def _draws(m, B, H, W, T, *, steps=None, dstep=None, seed=1):
    random.seed(seed)
    is_graph = getattr(m, "_is_graph", False)
    chosen = [m.graph.draw_offsets() for _ in range(T)] if is_graph else [()] * T
    fu = torch.rand(T, B, H, W, generator=torch.Generator().manual_seed(seed))
    dmg = None
    if dstep is not None:
        assert steps is None or min(steps) > dstep        # every sample is still running at the damage step
        dmg = torch.ones(B, m.n_channels, H, W)
        dmg[:, :, H // 3:H // 3 + max(1, H // 4), W // 4:W // 2] = 0.0
        dmg[0, :, H // 2:H // 2 + 2, :] = 0.5
    return Draws(T, chosen, fu, [0.5 + 0.1 * (t % 4) for t in range(T)],
                 [0.0 if t % 4 == 2 else 0.4 for t in range(T)], steps, dmg, dstep or 0)


def _schedule(m, B, H, W, dr):
    is_graph = getattr(m, "_is_graph", False)
    return make_schedule(m, B, H, W, dr.T, fire_rate=dr.frs, fire_u=dr.fu.to(DEV),
                         offsets=dr.chosen if is_graph else None, message_gains=dr.gains if is_graph else None,
                         steps=dr.steps, damage=None if dr.dmg is None else dr.dmg.to(DEV), damage_step=dr.dstep)


def _params(m, grads):
    return {k: v.detach().cpu().double().requires_grad_(grads and v.is_floating_point() and "perception" not in k)
            for k, v in m.state_dict().items()}


def _oracle(m, p, x0, dr, every=None, lo=0):
    """fp64 oracle rollout of samples [lo, lo + B) of the draws: (x_T, frames x_{f*every} or None)"""
    B = x0.shape[0]
    ref = x0
    st = torch.tensor(dr.steps[lo:lo + B]) if dr.steps is not None else None
    frames = []
    for t in range(dr.T):
        if dr.dmg is not None and t == dr.dstep:
            ref = ref * dr.dmg[lo:lo + B].double()
        if every and t % every == 0:
            frames.append(ref)
        mask = st > t if st is not None else torch.ones(B, dtype=torch.bool)
        if not bool(mask.any()):
            continue
        new = O.nca_step(ref[mask], p, _cfg(m, dr.gains[t]), dr.frs[t], dr.fu[t, lo:lo + B][mask].unsqueeze(1).double(),
                         dr.chosen[t])
        ref = ref.clone()
        ref[mask] = new
    if every and dr.T % every == 0:
        frames.append(ref)
    return ref, (torch.stack(frames) if every else None)


def _check_state(m, out, ref):
    assert rel_err(out.detach().cpu(), ref.detach()) < 1e-5, rel_err(out.detach().cpu(), ref.detach())
    thr = float(m.alpha_thr)
    assert torch.equal(GF.alive_mask(out.detach(), thr).cpu(), O.alive_mask(ref.detach().float(), thr))


def _check_grads(m, p, xg, xr):
    B = xg.shape[0]
    per = sorted(rel_err(xg.grad[b].cpu(), xr.grad[b]) for b in range(B))
    assert per[B // 2] <= 1e-5, per
    assert rel_err(xg.grad.cpu(), xr.grad) <= 5e-4, rel_err(xg.grad.cpu(), xr.grad)
    is_graph = getattr(m, "_is_graph", False)
    torus = is_graph and not m.graph.zero_padded_shift
    for n, q in m.named_parameters():
        gr = p[n].grad
        ours = q.grad.cpu() if q.grad is not None else torch.zeros_like(q.detach().cpu())
        if gr is None or float(gr.abs().max()) < 1e-12:       # unused (gate_mlp) or a uniform softmax
            assert float(ours.abs().max()) <= 1e-7, n
        elif any(s in n for s in QKS):
            if torus:
                assert float(ours.abs().max()) <= 1e-7, n
            else:
                # a near-uniform softmax leaves query / key gradients of ~1e-10, summed in fp32: 1e-11 absolute there
                assert rel_err(ours, gr) < 1e-3 or float((ours - gr.double()).abs().max()) <= 1e-11, (n, rel_err(ours, gr))
        else:
            assert rel_err(ours, gr) < 1e-4, (n, rel_err(ours, gr))


def check_rollout(m, x0, dr, impl, *, grads=True, bptt_budget=None):
    """library rollout vs the fp64 oracle: x_T, alive mask and, with `grads`, dL/dx0 and every parameter gradient"""
    B, _, H, W = x0.shape
    p = _params(m, grads)
    xr = x0.double().requires_grad_(grads)
    ref, _ = _oracle(m, p, xr, dr)
    for q in m.parameters():
        q.grad = None
    sched = _schedule(m, B, H, W, dr)
    xg = x0.to(DEV).requires_grad_(grads)
    with torch.set_grad_enabled(grads):
        out = rollout(m, xg, sched, impl=impl, bptt_budget=bptt_budget)
    _check_state(m, out, ref)
    if grads:
        _loss(ref).backward()
        _loss(out).backward()
        _check_grads(m, p, xg, xr)
    return sched


def _share(HW, NC):
    return (HW + NC - 1) // NC + 1


def _assert_rep(L, B, NC, ucap, over, what=""):
    """every k_rep_fwd launch had batch B and this configuration, and there was at least one"""
    assert L.rep and all(r == (B, NC, ucap, over) for r in L.rep), (what, L.rep, L.text)


def _assert_bwd(L, B, NC):
    """NC = None: the dense streaming BPTT ran (no k_rep_bwd launch)"""
    if NC is None:
        assert not L.bwd, (L.bwd, L.text)
    else:
        assert L.bwd and all(r == (B, NC) for r in L.bwd), (L.bwd, L.text)


# ---- 1. replicated-state forward + resident BPTT ---------------------------------------------------------------------
# name: kind, H, W, B, T, k, radius, d, ragged steps, damage step, (fwd NC, ucap, overflow), backward NC (None: the
# zero-pad backward does not fit shared memory at the only NC that H * W allows, so the dense streaming BPTT runs)
REP_CASES = {
    "64x32-torus-ragged":      ("torus", 64, 32, 3, 5, 8, 3, 16, [5, 2, 4], None, (8, 193, 64), 8),
    "32x64-zeropad-damage":    ("zeropad", 32, 64, 3, 5, 8, 3, 16, None, 1, (8, 65, 192), 8),
    "64x32-classic":           ("classic", 64, 32, 2, 4, 0, 0, 16, None, None, (8, 193, 64), 8),
    "32x64-torus-damage":      ("torus", 32, 64, 2, 4, 8, 3, 16, [4, 3], 2, (8, 193, 64), 8),
    "36x20-zeropad-ragged":    ("zeropad", 36, 20, 4, 6, 8, 3, 16, [6, 3, 5, 1], None, (8, 91, 0), 4),
    "20x36-torus-damage":      ("torus", 20, 36, 3, 5, 8, 3, 16, [5, 4, 3], 2, (8, 91, 0), 4),
    "20x36-zeropad":           ("zeropad", 20, 36, 3, 4, 8, 3, 16, None, None, (8, 91, 0), 4),
    "36x20-classic-ragged":    ("classic", 36, 20, 3, 5, 0, 0, 16, [5, 1, 3], None, (8, 91, 0), 4),
    "33x60-torus-ragged":      ("torus", 33, 60, 3, 4, 8, 3, 16, [4, 2, 3], None, (8, 249, 0), 1),
    "33x60-zeropad":           ("zeropad", 33, 60, 3, 4, 8, 3, 16, None, None, (8, 121, 128), None),
    "33x60-classic-damage":    ("classic", 33, 60, 2, 4, 0, 0, 16, None, 1, (8, 249, 0), 1),
    "44x44-zeropad-k16-d32":   ("zeropad", 44, 44, 3, 4, 16, 3, 32, None, None, (8, 179, 64), 4),
    "44x44-torus-ragged":      ("torus", 44, 44, 3, 5, 8, 3, 16, [5, 3, 4], 1, (8, 243, 0), 4),
    "64x4-torus":              ("torus", 64, 4, 3, 5, 8, 3, 16, None, None, (8, 33, 0), 8),
    "64x4-zeropad-ragged":     ("zeropad", 64, 4, 3, 5, 8, 3, 16, [5, 2, 4], None, (8, 33, 0), 8),
    "5x8-torus-r2":            ("torus", 5, 8, 4, 5, 8, 2, 16, [5, 3, 5, 2], None, (8, 6, 0), 2),
    "5x8-zeropad-r1":          ("zeropad", 5, 8, 3, 5, 8, 1, 16, None, 2, (8, 6, 0), 2),
    "5x8-classic":             ("classic", 5, 8, 3, 5, 0, 0, 16, None, None, (8, 6, 0), 2),
}


@pytest.mark.parametrize("name", list(REP_CASES))
def test_replicated_grids(name, launches):
    kind, H, W, B, T, k, radius, d, steps, dstep, fwd, bwd_nc = REP_CASES[name]
    m = _model(kind, k=k or 8, radius=radius or 3, d=d, seed=H * W)
    dr = _draws(m, B, H, W, T, steps=steps, dstep=dstep, seed=H + W)
    check_rollout(m, _state(B, 16, H, W, seed=H), dr, "auto")
    L = launches()
    assert not L.band, L.text
    _assert_rep(L, B, *fwd, what=name)
    _assert_bwd(L, B, bwd_nc)


def test_2048_cells_large_batch_overflows_u(launches):
    """B = 40 at 64 x 32: all 40 clusters co-resident only with fewer than 8 CTAs per cluster, where the update buffer
    of a CTA's share of 2048 cells no longer fits shared memory (ucap < share) and the rest goes to global memory"""
    H, W, B = 64, 32, 40
    m = _model("torus", seed=40)
    dr = _draws(m, B, H, W, 3, steps=[3, 2] * 20, seed=40)
    check_rollout(m, _state(B, 16, H, W, seed=40), dr, "auto")
    L = launches()
    assert L.rep and len(set(L.rep)) == 1, L.text
    b, nc, ucap, over = L.rep[0]
    assert b == B and nc in (1, 2, 4) and ucap < _share(H * W, nc) and over == _share(H * W, nc) - ucap > 0, L.rep
    assert L.bwd and len(set(L.bwd)) == 1 and L.bwd[0][0] == B and L.bwd[0][1] < 8, L.bwd


# forced cluster size on a grid with H * W % 32 = 16: (fwd ucap, overflow), backward NC (None: H * W % (4 * NC) != 0, no
# backward configuration, so the records are not written and the dense streaming BPTT runs after the same forward)
FORCED_NC = {1: ((384, 337), 1), 2: ((361, 0), 2), 4: ((181, 0), 4), 8: ((91, 0), None)}


@pytest.mark.parametrize("kind", ["torus", "zeropad"])
@pytest.mark.parametrize("nc", [1, 2, 4, 8])
def test_forced_cluster_size(nc, kind, launches, monkeypatch):
    H, W, B = 36, 20, 3
    monkeypatch.setenv("GNCA_RESIDENT_NC", str(nc))
    m = _model(kind, seed=nc)
    dr = _draws(m, B, H, W, 4, steps=[4, 2, 3], seed=nc)
    check_rollout(m, _state(B, 16, H, W, seed=nc), dr, "auto")
    L = launches()
    (ucap, over), bwd_nc = FORCED_NC[nc]
    _assert_rep(L, B, nc, ucap, over)
    _assert_bwd(L, B, bwd_nc)


# ---- 2. the recent entry points at a 2048-cell grid and at H * W % 32 != 0 ------------------------------------------
ENTRY_GRIDS = {"64x32-torus": ("torus", 64, 32, (8, 193, 64), 8), "36x20-zeropad": ("zeropad", 36, 20, (8, 91, 0), 4),
               "36x20-classic": ("classic", 36, 20, (8, 91, 0), 4)}


@pytest.mark.parametrize("grid", list(ENTRY_GRIDS))
def test_record_rollout_frame_gradients(grid, launches):
    """record_rollout(..., differentiable=True): the frames, x_T and the gradients of a loss on all of them"""
    kind, H, W, fwd, bwd_nc = ENTRY_GRIDS[grid]
    B, T, S = 3, 5, 2
    m = _model(kind, seed=7)
    dr = _draws(m, B, H, W, T, steps=[5, 3, 4], dstep=1, seed=7)
    x0 = _state(B, 16, H, W, seed=7)
    p = _params(m, True)
    xr = x0.double().requires_grad_(True)
    ref, ref_frames = _oracle(m, p, xr, dr, every=S)
    xg = x0.to(DEV).requires_grad_(True)
    tr = record_rollout(m, xg, _schedule(m, B, H, W, dr), every=S, differentiable=True)
    assert tr.t == [0, 2, 4] and tr.states.shape[0] == ref_frames.shape[0] == 3
    for f in range(3):
        _check_state(m, tr.states[f], ref_frames[f])
    _check_state(m, tr.x_T, ref)
    lf = lambda frames, xT: sum(_loss(frames[f]) * (f + 1) for f in range(frames.shape[0])) + _loss(xT)
    lf(ref_frames, ref).backward()
    lf(tr.states, tr.x_T).backward()
    _check_grads(m, p, xg, xr)
    L = launches()
    _assert_rep(L, B, *fwd)
    _assert_bwd(L, B, bwd_nc)


def _target(x0, seed=0):
    g = torch.Generator().manual_seed(seed)
    return (UM.premultiply(x0[:1])[0] + 0.03 * torch.randn(4, *x0.shape[2:], generator=g)).contiguous()


def _check_metrics(mon, frames, tgt, thr, eps, blk=slice(None)):
    """monitor_rollout's counts against utils.metrics on the fp64 oracle frames -- exact, except for the cells whose
    oracle value lies within 1e-5 of a threshold -- and its sums against fp64"""
    F, B = frames.shape[:2]
    HW = frames.shape[-1] * frames.shape[-2]
    x = frames.reshape(F * B, *frames.shape[2:]).detach()
    pm = UM.premultiply(x)
    dist = (pm - tgt.double().unsqueeze(0)).abs()
    pp = (dist < eps).all(dim=1).sum(dim=(1, 2)).reshape(F, B)
    pp_amb = ((dist - eps).abs() < 1e-5).any(dim=1).sum(dim=(1, 2)).reshape(F, B)
    alive = (x[:, 3] > thr).sum(dim=(1, 2)).reshape(F, B)
    alive_amb = ((x[:, 3] - thr).abs() < 1e-5).sum(dim=(1, 2)).reshape(F, B)
    got_pp = torch.round(mon.pixel_perfect[:, blk].double().cpu() * HW).long()
    assert ((got_pp - pp).abs() <= pp_amb).all(), (got_pp, pp, pp_amb)
    assert ((mon.alive[:, blk].cpu() - alive).abs() <= alive_amb).all(), (mon.alive, alive, alive_amb)
    assert int(pp_amb.sum()) + int(alive_amb.sum()) <= 0.01 * F * B * HW      # the exemption stays an exception
    t64 = tgt.double()
    se = ((pm - t64.unsqueeze(0)) ** 2).sum(dim=(1, 2, 3)).reshape(F, B)
    sr = ((pm[:, :3].clamp(0, 1) - t64[:3].clamp(0, 1).unsqueeze(0)) ** 2).sum(dim=(1, 2, 3)).reshape(F, B)
    loss = mon.loss[:, blk].double().cpu()
    assert rel_err(loss * 4 * HW, se) < 1e-4, rel_err(loss * 4 * HW, se)
    psnr = 10 * torch.log10(1 / (sr / (3 * HW)))
    assert torch.allclose(mon.psnr[:, blk].double().cpu(), psnr, rtol=1e-5, atol=1e-4), (mon.psnr, psnr)


@pytest.mark.parametrize("grid", list(ENTRY_GRIDS))
def test_monitor_rollout_against_oracle_frames(grid, launches):
    """per-CTA partials of the frame metrics where band edges fall mid-word (H * W % 32 != 0) and at 2048 cells"""
    kind, H, W, fwd, _ = ENTRY_GRIDS[grid]
    B, T, S, eps = 3, 6, 2, 0.05
    m = _model(kind, seed=8)
    dr = _draws(m, B, H, W, T, steps=[6, 3, 5], dstep=2, seed=8)
    x0 = _state(B, 16, H, W, seed=8)
    ref, ref_frames = _oracle(m, _params(m, False), x0.double(), dr, every=S)
    tgt = _target(x0, seed=8)
    mon = monitor_rollout(m, x0.to(DEV), _schedule(m, B, H, W, dr), tgt.to(DEV), every=S, eps=eps)
    _check_state(m, mon.x_T, ref)
    _check_metrics(mon, ref_frames, tgt, float(m.alpha_thr), eps)
    L = launches()
    _assert_rep(L, B, *fwd)
    assert not L.bwd and not L.band


@pytest.mark.parametrize("grid", ["64x32-torus", "36x20-classic"])
def test_checkpointed_resident_bptt(grid, launches):
    """rollout(..., bptt_budget=N) with N below the records: bptt_plan picks resident checkpoints with K > 1, and every
    segment recomputes its forward and runs its backward on the cluster kernels"""
    kind, H, W, fwd, bwd_nc = ENTRY_GRIDS[grid]
    B, T = 3, 7
    m = _model(kind, seed=9)
    lib = _lib.load()
    desc = m.model_desc()
    budget = (T // 3 + 1) * B * 16 * H * W * 4 + lib.gnca_bptt_ckpt_bytes(C.byref(desc), B, H, W, 3)
    path, K, _ = bptt_plan(m, B, H, W, T, budget)
    assert path == "resident_ckpt" and 1 < K < T, (path, K)
    dr = _draws(m, B, H, W, T, steps=[7, 4, 6], dstep=2, seed=9)
    check_rollout(m, _state(B, 16, H, W, seed=9), dr, "auto", bptt_budget=budget)
    L = launches()
    _assert_rep(L, B, *fwd)
    assert len(L.rep) == 1 + -(-T // K), L.rep          # the checkpointing forward, then one recompute per segment
    _assert_bwd(L, B, bwd_nc)
    assert len(L.bwd) == -(-T // K), L.bwd


@pytest.mark.parametrize("grid", ["64x32-torus", "36x20-zeropad"])
def test_model_stack(grid, launches):
    """record_rollout and monitor_rollout over M = 3 models in one launch: each model's block against its own oracle
    rollout under the shared schedule"""
    kind, H, W, fwd, _ = ENTRY_GRIDS[grid]
    M, B, T, S = 3, 2, 5, 2
    models = [_model(kind, seed=20 + i) for i in range(M)]
    dr = _draws(models[0], M * B, H, W, T, steps=[5, 3, 4, 5, 2, 5], seed=11)
    x0 = _state(M * B, 16, H, W, seed=11)
    tgt = _target(x0, seed=11)
    with torch.no_grad():
        tr = record_rollout(models, x0.to(DEV), _schedule(models[0], M * B, H, W, dr), every=S)
        mon = monitor_rollout(models, x0.to(DEV), _schedule(models[0], M * B, H, W, dr), tgt.to(DEV), every=S)
    for i, m in enumerate(models):
        blk = slice(i * B, (i + 1) * B)
        ref, ref_frames = _oracle(m, _params(m, False), x0[blk].double(), dr, every=S, lo=i * B)
        _check_state(m, tr.x_T[blk], ref)
        _check_state(m, mon.x_T[blk], ref)
        for f in range(ref_frames.shape[0]):
            _check_state(m, tr.states[f, blk], ref_frames[f])
        _check_metrics(mon, ref_frames, tgt, float(m.alpha_thr), 0.05, blk)
    L = launches()
    _assert_rep(L, M * B, *fwd)
    assert len(L.rep) == 2 and not L.band


# ---- 3. the banded kernel ---------------------------------------------------------------------------------------------
# name: kind, C, H, W, B, T, (NC, own rows, MB), seed; the halo is max_offset + 1 (1 for the classic model).  The forward
# is forced to the banded kernel; its backward is the dense streaming BPTT, checked as well.  Prime H is 37 x 24: at
# 37 x 40 x 16 the single band of NC = 1 needs about 244 KB of shared memory, so the grid would go to the streaming
# kernels.  48 x 41 (bands of 6 x 41 cells) and 30 x 30 (NC = 2, bands of 15 x 30) hold a number of cells that is not a
# multiple of 4.  40 x 40 x 4 uses seed 100: with the default draws sample 2 sits so close to a ReLU kink that fp32
# autograd on the oracle itself is 1.6e-3 from fp64 there.
BAND_CASES = {
    "37x24-torus-primeH":      ("torus", 16, 37, 24, 2, 4, (1, 37, 32), 0),
    "37x24-classic-primeH":    ("classic", 16, 37, 24, 2, 4, (1, 37, 64), 0),
    "48x41-torus-oddW":        ("torus", 16, 48, 41, 3, 4, (8, 6, 64), 0),
    "48x41-classic-oddW":      ("classic", 16, 48, 41, 2, 4, (8, 6, 64), 0),
    "30x30-classic":           ("classic", 16, 30, 30, 3, 4, (2, 15, 64), 0),
    "64x64x16-torus":          ("torus", 16, 64, 64, 2, 4, (8, 8, 64), 0),
    "64x64x16-classic":        ("classic", 16, 64, 64, 2, 3, (8, 8, 64), 0),
    "128x128x8-torus":         ("torus", 8, 128, 128, 2, 3, (8, 16, 16), 0),
    "128x128x8-classic":       ("classic", 8, 128, 128, 2, 3, (8, 16, 32), 0),
    "40x40x4-torus":           ("torus", 4, 40, 40, 3, 5, (8, 5, 64), 100),
    "40x40x8-torus":           ("torus", 8, 40, 40, 3, 5, (8, 5, 64), 0),
    "24x24x32-torus":          ("torus", 32, 24, 24, 3, 4, (4, 6, 64), 0),
    "48x48x32-torus":          ("torus", 32, 48, 48, 2, 3, (8, 6, 16), 0),
}


@pytest.mark.parametrize("name", list(BAND_CASES))
def test_banded_grids(name, launches):
    kind, C, H, W, B, T, (nc, own, mb), seed = BAND_CASES[name]
    m = _model(kind, C, seed=C + H + seed)
    dr = _draws(m, B, H, W, T, steps=[T - 1] + [T] * (B - 1), seed=H + W + seed)
    sched = check_rollout(m, _state(B, C, H, W, seed=W + seed), dr, "banded")
    L = launches()
    halo = sched.max_offset + 1
    assert L.band and all(r == (B, nc, own, halo, mb) for r in L.band), (L.band, L.text)
    assert not L.rep and not L.bwd


# ---- 4. just outside the envelope ------------------------------------------------------------------------------------
# name: H, W, T, what `auto` and `resident` run: ("banded", NC, own rows, MB) or None (neither cluster kernel takes the
# grid: `auto` runs the streaming kernels, `resident` raises "unsupported").  The backward is the dense streaming BPTT.
OUTSIDE = {
    "40x42-W%4": (40, 42, 4, ("banded", 8, 5, 64)),
    "48x48-2304cells": (48, 48, 4, ("banded", 8, 6, 64)),
    "68x8-H>64": (68, 8, 4, ("banded", 4, 17, 64)),
    "3x40-H<max_offset": (3, 40, 4, None),
    "96x96x16": (96, 96, 3, None),
}


@pytest.mark.parametrize("impl", ["auto", "resident"])
@pytest.mark.parametrize("name", list(OUTSIDE))
def test_outside_the_envelope(name, impl, launches):
    H, W, T, want = OUTSIDE[name]
    B = 2
    m = _model("torus", radius=4 if H < 4 else 3, seed=H)
    dr = _draws(m, B, H, W, T, steps=[T, T - 1], seed=H)
    x0 = _state(B, 16, H, W, seed=H)
    if want is None and impl == "resident":
        with pytest.raises(_lib.GncaError, match="unsupported"):
            rollout(m, x0.to(DEV).requires_grad_(True), _schedule(m, B, H, W, dr), impl=impl)
        assert not launches().band
        return
    sched = check_rollout(m, x0, dr, impl)
    if H < 4:
        assert sched.max_offset >= H
    L = launches()
    assert not L.rep and not L.bwd, L.text
    if want is None:
        assert not L.band, L.text
    else:
        _, nc, own, mb = want
        assert L.band and all(r == (B, nc, own, sched.max_offset + 1, mb) for r in L.band), (L.band, L.text)


@pytest.mark.parametrize("name", ["40x42-W%4", "48x48-2304cells", "3x40-H<max_offset"])
def test_outside_the_envelope_zeropad(name, launches):
    """the zero-padded shift has no banded kernel: `auto` runs the streaming kernels"""
    H, W, T, _ = OUTSIDE[name]
    B = 2
    m = _model("zeropad", radius=4 if H < 4 else 3, seed=H + 1)
    dr = _draws(m, B, H, W, T, steps=[T, T - 1], seed=H + 1)
    check_rollout(m, _state(B, 16, H, W, seed=H + 1), dr, "auto")
    L = launches()
    assert not L.rep and not L.bwd and not L.band, L.text

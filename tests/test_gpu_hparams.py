"""The kernels at hyper-parameters other than the reference's defaults (k = 8 offsets per step, attention radius 4,
d_model 16, hidden 128): neighbour counts 0 ... 64, radii whose offsets alias on small grids, query / key widths 1 ... 64
and hidden widths 4 ... 256.  The kernels pick code paths by these values (the KP = 16 sender table of the replicated-state
kernels at 8 < k <= 16, the fallback to the banded kernel and the dense BPTT at k > 16, the odd last sender pair of the
tensor-core update, the chunked attention-weight gradient at small hidden widths, the global-memory W1 plan of the
backward at C = 32 with a wide hidden layer).  Every case runs the library against the fp64 oracle with torch autograd for
the gradients, fed the same fire uniforms and offsets.
Tolerances: state 1e-5 (single step: also max_rel), alive masks bit-exact, parameter gradients 1e-4 rel-Frobenius
(query / key / scaling: 1e-3 under the zero-padded shift, <= 1e-7 absolute under the torus), dL/dx0 per-sample median
1e-5 and whole tensor 5e-4 (a state that differs in the 7th digit can put one hidden unit of one cell on the other side of
its ReLU kink)."""
import ctypes as C
import random

import pytest
import torch

from conftest import max_rel, rel_err
from oracle import nca_oracle as O

pytestmark = pytest.mark.gpu

if torch.cuda.is_available():
    import graph_neural_cellular_automata_b200 as G
    from graph_neural_cellular_automata_b200 import _lib
    from graph_neural_cellular_automata_b200 import functional as GF
    from graph_neural_cellular_automata_b200.rollout import make_schedule, rollout

DEV = "cuda"
QKS = ("query_proj", "key_proj", "scaling")


def _model(C, hid=128, *, H=24, k=8, radius=4, d=16, torus=True, classic=False, seed=0):
    torch.manual_seed(seed); random.seed(seed)
    if classic:
        m = G.NeuralCA(C, update_hidden=hid, img_size=H, update_gain=0.1, alpha_thr=0.1)
    else:
        m = G.NeuralCAGraph(C, update_hidden=hid, img_size=H, update_gain=0.1, alpha_thr=0.1, message_gain=0.4,
                            hidden_only=True, graph_d_model=d, graph_attention_radius=radius, graph_num_neighbors=k,
                            graph_zero_padded_shift=not torus)
    with torch.no_grad():
        m.update_net[2].weight.normal_(0, 0.05)
        m.norm.weight.uniform_(0.5, 1.5); m.norm.bias.normal_(0, 0.1)
    return m.to(DEV)


def _state(B, C, H, W, seed=0):
    """An alive blob (off centre, so the torus wrap and the zero-padded rows both matter) with ragged alive sets on every
    other sample."""
    g = torch.Generator().manual_seed(seed)
    yy, xx = torch.meshgrid(torch.arange(H), torch.arange(W), indexing="ij")
    r = 0.4 * min(H, W)
    disk = (((yy - 0.45 * H) ** 2 + (xx - 0.55 * W) ** 2) < r * r).float()
    x = torch.rand(B, C, H, W, generator=g) * disk
    x[1::2, 3] *= (torch.rand((B // 2), H, W, generator=g) > 0.4).float()
    return x


def _loss(x):
    return (x[:, :4] ** 2).mean() + (0.1 * x[:, 4:].mean() if x.shape[1] > 4 else 0.0)


def _cfg(m, gain):
    g = getattr(m, "graph", None)
    return O.StepConfig(update_gain=m.update_gain, alpha_thr=m.alpha_thr, graph=g is not None, message_gain=gain,
                        hidden_only=True if g is not None else False,
                        zero_padded_shift=bool(g.zero_padded_shift) if g is not None else False)


def check_rollout(m, x0, T, impl, *, steps=None, grads=True, seed=1):
    """Library rollout (impl) vs the fp64 oracle: final state, alive mask and, with `grads`, dL/dx0 and every parameter
    gradient of `_loss`.  Offsets (random.sample of the model's ring), fire uniforms, per-step fire rates and message
    gains are drawn here and fed to both."""
    B, Cc, H, W = x0.shape
    is_graph = getattr(m, "_is_graph", False)
    random.seed(seed)
    chosen = [m.graph.draw_offsets() for _ in range(T)] if is_graph else [()] * T
    fu = torch.rand(T, B, H, W, generator=torch.Generator().manual_seed(seed))
    frs = [0.5 + 0.1 * (t % 4) for t in range(T)]
    gains = [0.0 if t % 4 == 2 else 0.4 for t in range(T)]
    p = {k: v.detach().cpu().double().requires_grad_(grads and v.is_floating_point() and "perception" not in k)
         for k, v in m.state_dict().items()}
    xr = x0.double().requires_grad_(grads)
    ref = xr
    st = torch.tensor(steps) if steps is not None else None
    for t in range(T):
        mask = st > t if st is not None else torch.ones(B, dtype=torch.bool)
        if not bool(mask.any()):
            continue
        new = O.nca_step(ref[mask], p, _cfg(m, gains[t]), frs[t], fu[t][mask].unsqueeze(1).double(), chosen[t])
        ref = ref.clone()
        ref[mask] = new
    for q in m.parameters():
        q.grad = None
    sched = make_schedule(m, B, H, W, T, fire_rate=frs, fire_u=fu.to(DEV), offsets=chosen if is_graph else None,
                          message_gains=gains if is_graph else None, steps=steps)
    xg = x0.to(DEV).requires_grad_(grads)
    if grads:
        out = rollout(m, xg, sched, impl=impl)
    else:
        with torch.no_grad():
            out = rollout(m, xg, sched, impl=impl)
    assert rel_err(out.detach().cpu(), ref.detach()) < 1e-5, rel_err(out.detach().cpu(), ref.detach())
    thr = float(m.alpha_thr)
    assert torch.equal(GF.alive_mask(out.detach(), thr).cpu(), O.alive_mask(ref.detach().float(), thr))
    if not grads:
        return
    _loss(ref).backward()
    _loss(out).backward()
    per = sorted(rel_err(xg.grad[b].cpu(), xr.grad[b]) for b in range(B))
    assert per[B // 2] <= 1e-5, per
    assert rel_err(xg.grad.cpu(), xr.grad) <= 5e-4, rel_err(xg.grad.cpu(), xr.grad)
    torus = is_graph and not m.graph.zero_padded_shift
    for n, q in m.named_parameters():
        gr = p[n].grad
        ours = q.grad.cpu() if q.grad is not None else torch.zeros_like(q.detach().cpu())
        if gr is None or float(gr.abs().max()) < 1e-12:       # unused (gate_mlp, the message at k = 0) or uniform softmax
            assert float(ours.abs().max()) <= 1e-7, n
        elif any(s in n for s in QKS):
            if torus:
                assert float(ours.abs().max()) <= 1e-7, n
            else:
                assert rel_err(ours, gr) < 1e-3, (n, rel_err(ours, gr))
        else:
            assert rel_err(ours, gr) < 1e-4, (n, rel_err(ours, gr))


# ---- 1. neighbour count and radius: streaming kernels, forward + BPTT -----------------------------------------------
@pytest.mark.parametrize("torus", [True, False], ids=["torus", "zeropad"])
@pytest.mark.parametrize("k,radius", [(0, 4), (0, 1), (1, 2), (7, 2), (9, 2), (16, 2), (17, 3), (40, 3), (64, 5)],
                         ids=lambda v: str(v))
def test_neighbour_count_streaming(k, radius, torus):
    """k = 0 twice: graph_num_neighbors = 0, and radius 1 (an empty offset ring)."""
    nk = 8 if (k, radius) == (0, 1) else k
    m = _model(16, k=nk, radius=radius, torus=torus, H=24, seed=k + radius)
    assert min(nk, len(m.graph.offsets)) == k
    check_rollout(m, _state(3, 16, 24, 28, seed=k), 3, "streaming", seed=k + 1)


# ---- 2. the resident families at k in (8, 16], and the fallback above 16 --------------------------------------------
@pytest.mark.parametrize("k,B,steps", [(9, 4, None), (12, 4, [6, 2, 0, 5]), (16, 4, None), (16, 9, None)],
                         ids=["k9", "k12-ragged", "k16", "k16-B9"])
def test_resident_torus_k_up_to_16(k, B, steps):
    """k_rep_fwd + k_rep_bwd with the KP = 16 sender table; B = 9 changes the cluster count of the step."""
    m = _model(16, k=k, radius=3, torus=True, H=40, seed=k)
    check_rollout(m, _state(B, 16, 40, 40, seed=k), 6, "resident", steps=steps, seed=k)


@pytest.mark.parametrize("d", [8, 32])
def test_resident_zeropad_forward_k16(d):
    """The ZP instantiation of k_rep_fwd at k = 16 (one warp per offset, pooled query / key over d lanes)."""
    m = _model(16, k=16, radius=3, d=d, torus=False, H=40, seed=d)
    check_rollout(m, _state(4, 16, 40, 40, seed=d), 5, "resident", seed=d)


@pytest.mark.parametrize("k,radius,B", [(9, 3, 4), (24, 3, 8), (24, 5, 4), (64, 5, 8)], ids=lambda v: str(v))
def test_banded_neighbour_count(k, radius, B):
    """k_resident_fwd with k up to 64 (the s_q[MB * k] sender table); radius 5 makes the halo 6 rows, which forces
    fewer than 8 CTAs per cluster at H = 40."""
    m = _model(16, k=k, radius=radius, torus=True, H=40, seed=k + radius)
    check_rollout(m, _state(B, 16, 40, 40, seed=k), 5, "banded", steps=[5, 3] + [5] * (B - 2), seed=k)


@pytest.mark.parametrize("impl", ["resident", "auto"])
def test_k17_falls_back(impl):
    """k > 16: the replicated-state kernel and its BPTT reject the step; the forward falls back to the banded kernel
    (resident) or the streaming kernels (auto) and the backward to the dense streaming BPTT."""
    m = _model(16, k=17, radius=3, torus=True, H=40, seed=17)
    check_rollout(m, _state(4, 16, 40, 40, seed=17), 5, impl, seed=17)


# ---- 3. grids smaller than twice the radius: offsets alias modulo the grid ------------------------------------------
@pytest.mark.parametrize("impl", ["streaming", "resident", "banded"])
@pytest.mark.parametrize("HW", [12, 8])
def test_small_torus_aliasing_offsets(HW, impl):
    m = _model(16, k=12, radius=5, torus=True, H=HW, seed=HW)
    check_rollout(m, _state(3, 16, HW, HW, seed=HW), 4, impl, seed=HW)


def test_zeropad_grid_shorter_than_the_radius():
    """H = 4 with radius 5: every row shift of 4 or more empties the sender row."""
    m = _model(16, k=24, radius=5, torus=False, H=4, seed=4)
    check_rollout(m, _state(3, 16, 4, 12, seed=4), 3, "streaming", seed=4)


# ---- 4. d_model under the zero-padded shift -------------------------------------------------------------------------
@pytest.mark.parametrize("impl", ["streaming", "auto"])
@pytest.mark.parametrize("d", [1, 8, 32, 33, 64])
def test_zeropad_d_model(d, impl):
    """k_attn_weights / k_attn_bwd with [k][d] tables; at d > 32 the ZP resident forward rejects the model and `auto`
    falls back.  Also one step with the attention map against the oracle's."""
    m = _model(16, k=12, radius=3, d=d, torus=False, H=40, seed=d)
    x0 = _state(3, 16, 40, 40, seed=d)
    check_rollout(m, x0, 4, impl, seed=d)
    random.seed(d)
    chosen = m.graph.draw_offsets()
    fu = torch.rand(3, 1, 40, 40)
    p = {k: v.detach().cpu().double() for k, v in m.state_dict().items()}
    ref, attn_ref = O.nca_step(x0.double(), p, _cfg(m, 0.4), 0.6, fu.double(), chosen, return_attention=True)
    with torch.no_grad():
        out, attn = m.step(x0.to(DEV), 0.6, fire_u=fu.to(DEV), chosen=chosen, message_gain=0.4, return_attention=True)
    assert max_rel(out.cpu(), ref) < 1e-5 and rel_err(out.cpu(), ref) < 1e-5
    assert max_rel(attn.cpu(), attn_ref, floor=1e-2) < 1e-4, max_rel(attn.cpu(), attn_ref, floor=1e-2)


# ---- 5. hidden width: the boundary of the staged backward plan and the chunked attention-weight gradient -----------
@pytest.mark.parametrize("hid", [160, 164, 176, 180, 256])
def test_classic_c32_wide_hidden_backward(hid):
    """The classic model's k_bwd_mlp stages W1T and W1 up to hidden 176 at C = 32 and reads them from global memory
    above (the graph model's boundary, 160 / 164, is in test_streaming_backward_other_channel_counts_vs_oracle_autograd)."""
    m = _model(32, hid, classic=True, seed=hid)
    check_rollout(m, _state(3, 32, 24, 28, seed=hid), 3, "streaming", seed=hid)


@pytest.mark.parametrize("hid", [4, 12])
def test_zeropad_k64_chunked_attention_weight_gradient(hid):
    """k = 64 > kcap = 2 * hid * NBP / NB: the dL/dw_i sums of k_bwd_mlp run over several offset chunks."""
    m = _model(16, hid, k=64, radius=5, torus=False, seed=hid)
    check_rollout(m, _state(3, 16, 24, 28, seed=hid), 3, "streaming", seed=hid)


# ---- 6. the large-problem path (k_update_tc, and k_update under GNCA_NO_TC) ------------------------------------------
@pytest.mark.parametrize("kernel", ["tc", "ffma"])
@pytest.mark.parametrize("torus", [True, False], ids=["torus", "zeropad"])
@pytest.mark.parametrize("k", [1, 7, 17, 64])
@pytest.mark.parametrize("C,Hh,B,hid", [(32, 64, 80, 128), (16, 128, 20, 128)], ids=["64x64x32", "128x128x16"])
def test_large_problem_neighbour_count(C, Hh, B, hid, k, torus, kernel, monkeypatch):
    """B * ceil(HW / 1024) >= 296: the balanced update over compacted active cells, senders fetched in pairs (odd k: a
    half-empty last pair).  Samples are independent, so the oracle checks four of them, ragged and not."""
    monkeypatch.delenv("GNCA_NO_TC", raising=False)
    if kernel == "ffma":
        monkeypatch.setenv("GNCA_NO_TC", "1")
    _one_large_step(C, Hh, B, hid, k, torus)


@pytest.mark.parametrize("torus", [True, False], ids=["torus", "zeropad"])
def test_large_problem_hidden_256(torus):
    """hidden 256 at C = 32: no tensor cores (they need hidden 128), the balanced FFMA kernel."""
    _one_large_step(32, 64, 80, 256, 9, torus)


def _one_large_step(C, Hh, B, hid, k, torus):
    m = _model(C, hid, H=Hh, k=k, radius=5, torus=torus, seed=k)
    x = _state(B, C, Hh, Hh, seed=k)
    fu = torch.rand(B, 1, Hh, Hh, generator=torch.Generator().manual_seed(k))
    random.seed(k)
    chosen = m.graph.draw_offsets()
    with torch.no_grad():
        out = m.step(x.to(DEV), 0.5, fire_u=fu.to(DEV), chosen=chosen, message_gain=0.4)
    p = {n: v.detach().cpu().double() for n, v in m.state_dict().items()}
    idx = [0, 1, B // 2, B - 1]
    ref = O.nca_step(x[idx].double(), p, _cfg(m, 0.4), 0.5, fu[idx].double(), chosen)
    assert max_rel(out[idx].cpu(), ref) < 1e-5, max_rel(out[idx].cpu(), ref)
    assert rel_err(out[idx].cpu(), ref) < 1e-5
    assert torch.equal(GF.alive_mask(out, 0.1)[idx].cpu(), O.alive_mask(ref.float(), 0.1))


def test_large_problem_gradients_odd_k():
    """Two steps at k = 7 on the balanced path (64x64x32, B = 80), gradients against fp64 oracle autograd."""
    m = _model(32, 128, H=64, k=7, radius=4, torus=True, seed=70)
    check_rollout(m, _state(80, 32, 64, 64, seed=70), 2, "streaming", seed=70)


# ---- 7. unsupported arguments return before any launch (C ABI) -----------------------------------------------------
def test_out_of_range_k_returns_before_launch():
    """gnca_rollout_bwd / gnca_step_bwd / the BPTT entry points with k outside [0, GNCA_MAX_K] return UNSUPPORTED and
    leave the caller's gradient buffers bit-identical (k indexes GNCA_MAX_K-long tables in the kernels)."""
    lib = _lib.load()
    m = _model(16, k=8, radius=4, torus=True, H=16, seed=3)
    desc, packed = m.model_desc(), m.packed_weights()
    B, H, W, T = 2, 16, 16, 2
    lay = GF.param_layout(desc)
    N = B * 16 * H * W
    hist = _state(B, 16, H, W).to(DEV).unsqueeze(0).expand(T + 1, -1, -1, -1, -1).contiguous()
    gT = torch.ones(B, 16, H, W, device=DEV)
    ws_bytes = max(lib.gnca_rollout_workspace_bytes(C.byref(desc), B, H, W, T),
                   lib.gnca_step_workspace_bytes(C.byref(desc), B, H, W))
    ws = torch.zeros(ws_bytes, dtype=torch.uint8, device=DEV)
    fr = torch.full((T,), 0.5, device=DEV)
    gains = torch.full((T,), 0.4, device=DEV)
    offs = torch.full((T * 65 * 2,), 2, dtype=torch.int8, device=DEV)
    offs_host = (C.c_int32 * (2 * 65))(*([2] * 130))
    sentinel = -12345.0
    g0 = torch.full((N,), sentinel, device=DEV)
    gp = torch.full((lay.total,), sentinel, device=DEV)
    nb = 1 << 20
    bptt = torch.zeros(nb, dtype=torch.uint8, device=DEV)
    p = GF._ptr
    for k in (65, -1):
        s = _lib.GncaSchedule(T=T, k=k, fire_rate=p(fr), message_gain=p(gains), offsets=p(offs), max_offset=2)
        torch.cuda.synchronize()
        before = lib.gnca_launch_count()
        assert lib.gnca_rollout_bwd(C.byref(desc), p(packed), B, H, W, C.byref(s), p(hist), None, None, p(gT), p(g0),
                                    p(gp), p(ws), ws.numel(), 1, None) == _lib.GNCA_ERR_UNSUPPORTED, k
        assert lib.gnca_rollout_fwd_bptt(C.byref(desc), p(packed), B, H, W, C.byref(s), p(hist), p(gT), None, p(bptt),
                                         nb, p(ws), ws.numel(), None) == _lib.GNCA_ERR_UNSUPPORTED, k
        assert lib.gnca_rollout_bwd_bptt(C.byref(desc), p(packed), B, H, W, C.byref(s), p(bptt), nb, p(gT), p(g0),
                                         p(gp), p(ws), ws.numel(), None) == _lib.GNCA_ERR_UNSUPPORTED, k
        assert lib.gnca_launch_count() == before, k
        torch.cuda.synchronize()
        assert bool((g0 == sentinel).all()) and bool((gp == sentinel).all()), k
    before = lib.gnca_launch_count()
    assert lib.gnca_step_bwd(C.byref(desc), p(packed), B, H, W, p(hist), None, 1.0, offs_host, 65, 0.4, p(hist), p(fr),
                             p(gT), p(g0), p(gp), p(ws), ws.numel(), None) == _lib.GNCA_ERR_UNSUPPORTED
    assert lib.gnca_launch_count() == before
    torch.cuda.synchronize()
    assert bool((g0 == sentinel).all()) and bool((gp == sentinel).all())

"""BASELINE configs[4] shape (256x256 grid, 32 channels, hidden 128, torus graph path) on the GPU: one step against the
CPU oracle, and the size-independent properties of the rollout at that shape (the oracle does not finish a 1000-step
rollout of this size in test time): bitwise run-to-run determinism, frozen samples pass through, samples are
independent (a permuted batch gives the permuted result bit for bit), damage at step t == multiply + continue.
All of it runs the streaming kernels in their large-problem (balanced k_update) mode."""
import random

import pytest
import torch

from conftest import max_rel, rel_err
from oracle import nca_oracle as O

pytestmark = pytest.mark.gpu

if torch.cuda.is_available():
    import graph_neural_cellular_automata_b200 as G
    from graph_neural_cellular_automata_b200 import functional as GF
    from graph_neural_cellular_automata_b200.rollout import make_schedule, rollout
    from graph_neural_cellular_automata_b200.utils.damage import circle_mask

DEV = "cuda"
C, H, W, HID = 32, 256, 256, 128


def _model():
    torch.manual_seed(5); random.seed(5)
    m = G.NeuralCAGraph(C, update_hidden=HID, img_size=H, update_gain=0.1, alpha_thr=0.1, message_gain=0.3,
                        hidden_only=True, graph_zero_padded_shift=False)
    with torch.no_grad():
        m.update_net[2].weight.normal_(0, 0.05)
        m.norm.weight.uniform_(0.5, 1.5); m.norm.bias.normal_(0, 0.1)
    p = {k: v.detach().clone() for k, v in m.state_dict().items()}
    return m.to(DEV), p


def _blobs(B):
    yy, xx = torch.meshgrid(torch.arange(H), torch.arange(W), indexing="ij")
    disk = (((yy - H / 2) ** 2 + (xx - W / 2) ** 2) < (0.3 * H) ** 2).float()
    x = torch.rand(B, C, H, W) * disk
    x[1::2, 3] *= (torch.rand((B + 0) // 2, H, W) > 0.4).float()        # ragged alive sets on every other sample
    return x


@pytest.mark.parametrize("kernel", ["tc", "ffma"])
def test_one_step_vs_oracle_at_scale(kernel, monkeypatch):
    """Both k_update variants of the large-problem path: compacted tensor-core tiles (default), the round-1 FFMA kernel
    (GNCA_NO_TC=1)."""
    monkeypatch.delenv("GNCA_NO_TC", raising=False)
    if kernel == "ffma":
        monkeypatch.setenv("GNCA_NO_TC", "1")
    m, p = _model()
    B = 5                                            # 5 * 64 chunks >= 2 * 148 blocks: the balanced large-problem path
    x = _blobs(B)
    fu = torch.rand(B, 1, H, W)
    chosen = random.sample(m.graph.offsets, 8)
    cfg = O.StepConfig(update_gain=0.1, alpha_thr=0.1, graph=True, message_gain=0.3, hidden_only=True,
                       zero_padded_shift=False)
    # fp64 oracle: deterministic, and the accuracy yard-stick of SURVEY 8c-ii (the fp32 CPU oracle's own distance to it
    # varies run to run at this size with the thread count of the box)
    ref = O.nca_step(x.double(), {k: v.double() for k, v in p.items()}, cfg, 0.5, fu.double(), chosen)
    with torch.no_grad():
        out = m.step(x.to(DEV), 0.5, fire_u=fu.to(DEV), chosen=chosen)
    assert max_rel(out.cpu(), ref) < 1e-5, max_rel(out.cpu(), ref)           # 1e-5 relative, single step (north star)
    assert rel_err(out.cpu(), ref) < 1e-5
    assert torch.equal(GF.alive_mask(out, 0.1).cpu(), O.alive_mask(ref.float(), 0.1))  # alive mask bit-exact


def test_rollout_properties_at_scale():
    m, _ = _model()
    B, T, td = 6, 5, 2
    x0 = _blobs(B).to(DEV)
    random.seed(11)
    offs = [m.graph.draw_offsets() for _ in range(T)]
    fu = torch.rand(T, B, H, W, device=DEV)
    D = circle_mask(x0, 40).expand_as(x0).contiguous()
    steps = [T, T, 0, 3, T, 1]                        # sample 2 is frozen from the start, 3 and 5 stop early

    def run(x, f, d, st):
        sched = make_schedule(m, x.shape[0], H, W, T, fire_rate=0.5, offsets=offs, fire_u=f, damage=d, damage_step=td,
                              steps=st)
        with torch.no_grad():
            return rollout(m, x, sched)

    a = run(x0, fu, D, steps)
    # (1) bitwise deterministic run to run
    assert torch.equal(a, run(x0, fu, D, steps))
    # (2) frozen sample: untouched by the steps (train...:306-321 `state[mask] = model(state[mask])`); the damage of the
    #     batch is still applied to it at t = td, as the reference's in-place damage on the whole batch would
    assert torch.equal(a[2], x0[2] * D[2])
    # (3) samples are independent: a permuted batch (inputs, masks, damage, step counts) gives the permuted result
    perm = torch.tensor([3, 0, 5, 1, 4, 2], device=DEV)
    b = run(x0[perm].contiguous(), fu[:, perm].contiguous(), D[perm].contiguous(), [steps[i] for i in perm.tolist()])
    assert torch.equal(b, a[perm])
    # (4) damage at step td == rollout to td, multiply, continue (regeneration protocol)
    full = [T] * B
    whole = run(x0, fu, D, full)
    sched1 = make_schedule(m, B, H, W, td, fire_rate=0.5, offsets=offs[:td], fire_u=fu[:td].contiguous())
    sched2 = make_schedule(m, B, H, W, T - td, fire_rate=0.5, offsets=offs[td:], fire_u=fu[td:].contiguous())
    with torch.no_grad():
        mid = rollout(m, x0, sched1)
        two = rollout(m, (mid * D).contiguous(), sched2)
    assert torch.equal(whole, two)
    # (5) the state stays finite and alive
    assert torch.isfinite(whole).all() and float((whole[:, 3] > 0.1).float().mean()) > 0.01


_EDGE_CASES = [(64, 64, 80, 8), (48, 66, 80, 8), (40, 75, 100, 8), (64, 64, 80, 7), (40, 75, 100, 7)]


@pytest.mark.parametrize("Hh,Ww,B,k", _EDGE_CASES, ids=[f"{h}-{w}-{b}" + ("" if k == 8 else f"-k{k}") for h, w, b, k in _EDGE_CASES])
@pytest.mark.parametrize("kernel", ["tc", "ffma"])
def test_large_problem_path_at_the_grid_edges(Hh, Ww, B, k, kernel, monkeypatch):
    """The blobs of the tests above never touch the border.  Here the whole grid is alive except a dead band in the
    middle: every edge / corner cell runs the zero-halo perception (clamped taps + selects; the 8-byte tap pairs when W is
    even, the scalar taps at W = 75) and the torus wrap of the sender gather in the large-problem kernels.  k = 7 leaves
    the last sender pair of the tensor-core gather half empty."""
    monkeypatch.delenv("GNCA_NO_TC", raising=False)
    if kernel == "ffma":
        monkeypatch.setenv("GNCA_NO_TC", "1")
    torch.manual_seed(9); random.seed(9)
    m = G.NeuralCAGraph(C, update_hidden=HID, img_size=Hh, update_gain=0.1, alpha_thr=0.1, message_gain=0.3,
                        hidden_only=True, graph_zero_padded_shift=False)
    with torch.no_grad():
        m.update_net[2].weight.normal_(0, 0.05)
        m.norm.weight.uniform_(0.5, 1.5); m.norm.bias.normal_(0, 0.1)
    p = {k: v.detach().double() for k, v in m.state_dict().items()}
    m = m.to(DEV)
    x = torch.rand(B, C, Hh, Ww)
    x[:, :, Hh // 2 - 4:Hh // 2 + 4, 5:Ww - 5] = 0.0                  # a dead band, not touching the border
    x[::3, 3] *= (torch.rand((B + 2) // 3, Hh, Ww) > 0.3).float()       # ragged alive sets on every third sample
    fu = torch.rand(B, 1, Hh, Ww)
    chosen = [(4, -4), (-4, 4), (0, 3), (-3, 0), (1, 1), (-2, 4), (4, 0), (0, -4)][:k]   # wraps on every side
    cfg = O.StepConfig(update_gain=0.1, alpha_thr=0.1, graph=True, message_gain=0.3, hidden_only=True,
                       zero_padded_shift=False)
    ref = O.nca_step(x.double(), p, cfg, 0.5, fu.double(), chosen)
    with torch.no_grad():
        out = m.step(x.to(DEV), 0.5, fire_u=fu.to(DEV), chosen=chosen)
    assert max_rel(out.cpu(), ref) < 1e-5, max_rel(out.cpu(), ref)
    assert torch.equal(GF.alive_mask(out, 0.1).cpu(), O.alive_mask(ref.float(), 0.1))


@pytest.mark.parametrize("flags", [dict(hidden_only=False), dict(graph_alive_to_alive=False), dict(use_groupnorm=False),
                                   dict(hidden_only=False, graph_alive_to_alive=False, use_groupnorm=False)])
@pytest.mark.parametrize("Cc", [16, 32])
def test_tensor_core_path_constructor_flags(flags, Cc):
    """The non-default constructor flags (VERDICT r1: compiled into every kernel, exercised only at 40x40) on the
    tensor-core large-problem path, C = 16 and 32: one step against the fp64 oracle."""
    torch.manual_seed(13); random.seed(13)
    Hh, B = 64, 80
    m = G.NeuralCAGraph(Cc, update_hidden=HID, img_size=Hh, update_gain=0.1, alpha_thr=0.1, message_gain=0.3,
                        graph_zero_padded_shift=False, **{"hidden_only": True, **flags})
    with torch.no_grad():
        m.update_net[2].weight.normal_(0, 0.05)
        if flags.get("use_groupnorm", True):
            m.norm.weight.uniform_(0.5, 1.5); m.norm.bias.normal_(0, 0.1)
    p = {k: v.detach().double() for k, v in m.state_dict().items()}
    m = m.to(DEV)
    yy, xx = torch.meshgrid(torch.arange(Hh), torch.arange(Hh), indexing="ij")
    x = torch.rand(B, Cc, Hh, Hh) * (((yy - 30) ** 2 + (xx - 35) ** 2) < 24 ** 2).float()
    x[1::2, 3] *= (torch.rand(B // 2, Hh, Hh) > 0.4).float()
    fu = torch.rand(B, 1, Hh, Hh)
    chosen = random.sample(m.graph.offsets, 8)
    cfg = O.StepConfig(update_gain=0.1, alpha_thr=0.1, graph=True, message_gain=0.3, zero_padded_shift=False,
                       hidden_only=flags.get("hidden_only", True), alive_to_alive=flags.get("graph_alive_to_alive", True),
                       use_groupnorm=flags.get("use_groupnorm", True))
    ref = O.nca_step(x.double(), p, cfg, 0.5, fu.double(), chosen)
    with torch.no_grad():
        out = m.step(x.to(DEV), 0.5, fire_u=fu.to(DEV), chosen=chosen)
    assert max_rel(out.cpu(), ref) < 1e-5, max_rel(out.cpu(), ref)
    assert torch.equal(GF.alive_mask(out, 0.1).cpu(), O.alive_mask(ref.float(), 0.1))


def test_tensor_core_rollout_vs_oracle():
    """Four steps on the tensor-core large-problem path (64x64x32, B = 80) against the fp64 oracle fed the same uniforms and
    offsets: the per-step hand-over k_compact (lists, active bits, sender-alive bits) -> k_update_tc -> k_apply."""
    torch.manual_seed(17); random.seed(17)
    Hh, B, T = 64, 80, 4
    m = G.NeuralCAGraph(C, update_hidden=HID, img_size=Hh, update_gain=0.1, alpha_thr=0.1, message_gain=0.3,
                        hidden_only=True, graph_zero_padded_shift=False)
    with torch.no_grad():
        m.update_net[2].weight.normal_(0, 0.05)
        m.norm.weight.uniform_(0.5, 1.5); m.norm.bias.normal_(0, 0.1)
    p = {k: v.detach().double() for k, v in m.state_dict().items()}
    m = m.to(DEV)
    yy, xx = torch.meshgrid(torch.arange(Hh), torch.arange(Hh), indexing="ij")
    x0 = torch.rand(B, C, Hh, Hh) * (((yy - 30) ** 2 + (xx - 35) ** 2) < 26 ** 2).float()
    x0[::2, 3] *= (torch.rand(B // 2, Hh, Hh) > 0.5).float()
    fu = torch.rand(T, B, Hh, Hh)
    chosen = [random.sample(m.graph.offsets, 8) for _ in range(T)]
    gains = [0.3, 0.0, 0.3, 0.3]
    sched = make_schedule(m, B, Hh, Hh, T, fire_rate=0.5, fire_u=fu.to(DEV), offsets=chosen, message_gains=gains)
    with torch.no_grad():
        out = rollout(m, x0.to(DEV), sched, impl="streaming")
    ref = x0.double()
    for t in range(T):
        cfg = O.StepConfig(update_gain=0.1, alpha_thr=0.1, graph=True, message_gain=gains[t], hidden_only=True,
                           zero_padded_shift=False)
        ref = O.nca_step(ref, p, cfg, 0.5, fu[t].unsqueeze(1).double(), chosen[t])
    assert rel_err(out.cpu(), ref.float()) < 1e-5, rel_err(out.cpu(), ref.float())
    assert torch.equal(GF.alive_mask(out, 0.1).cpu(), O.alive_mask(ref.float(), 0.1))

"""GPU tests of SSIM on the device: utils.metrics.ssim_rgb (gnca_ssim_rgb) against the fp64 oracle, and
monitor_rollout(..., ssim=True) (gnca_rollout_metrics_ssim[_models]) on every kernel family.

The monitor's SSIM is pinned to ssim_rgb on the frames record_rollout keeps on the same impl (the same per-cell
function, only the partition of the sums differs) and to the oracle; every other output is pinned bit for bit to the
call without SSIM.  GNCA_DEBUG launch lines show which family ran.  Models, states and schedules are built here."""
import random
import re

import numpy as np
import pytest
import torch

from conftest import load_params
from oracle import ssim_oracle as SO

pytestmark = pytest.mark.gpu

if torch.cuda.is_available():
    import graph_neural_cellular_automata_b200 as G
    from graph_neural_cellular_automata_b200 import _lib
    from graph_neural_cellular_automata_b200.rollout import make_schedule, monitor_rollout, record_rollout
    from graph_neural_cellular_automata_b200.utils import metrics as UM

DEV = "cuda"
RE_REP = re.compile(r"replicated fwd: B=(\d+) NC=(\d+)")
RE_BAND = re.compile(r"resident fwd: B=(\d+) NC=(\d+) own_rows=(\d+) halo=(\d+)")


def _perturb(m, seed, scale=0.05):
    if seed == 0:
        return m
    g = torch.Generator().manual_seed(1000 + seed)
    with torch.no_grad():
        for name, p in m.named_parameters():
            if "perception" in name or not p.requires_grad:
                continue
            p.add_(scale * p.abs().mean() * torch.randn(p.shape, generator=g).to(p.device))
    return m


def _graph16(torus, seed=0):
    m = G.NeuralCAGraph(16, update_hidden=128, img_size=40, update_gain=0.05, alpha_thr=0.12, message_gain=0.25,
                        hidden_only=True, graph_zero_padded_shift=not torus)
    missing, unexpected = m.load_state_dict(load_params("weights_graph_ep960.npz"), strict=False)
    assert not missing and not unexpected
    return _perturb(m, seed).to(DEV)


def _classic16(seed=0):
    m = G.NeuralCA(16, update_hidden=128, img_size=40, update_gain=0.1, alpha_thr=0.1)
    missing, unexpected = m.load_state_dict(load_params("weights_classic_ep990.npz"), strict=False)
    assert not missing and not unexpected
    return _perturb(m, seed).to(DEV)


def _random_graph(C_, H, seed=5):
    torch.manual_seed(seed); random.seed(seed)
    m = G.NeuralCAGraph(C_, update_hidden=128, img_size=H, update_gain=0.1, alpha_thr=0.1, message_gain=0.3,
                        hidden_only=True, graph_zero_padded_shift=False)
    with torch.no_grad():
        m.update_net[2].weight.normal_(0, 0.05)
        m.norm.weight.uniform_(0.5, 1.5); m.norm.bias.normal_(0, 0.1)
    return m.to(DEV)


MODELS = {"torus": lambda s=0: _graph16(True, s), "zeropad": lambda s=0: _graph16(False, s), "classic": _classic16}


def _blob(B, C_, H, W, seed=0):
    """random state inside a disk (alive cells with a dead border around them)"""
    g = torch.Generator().manual_seed(seed)
    yy, xx = torch.meshgrid(torch.arange(H), torch.arange(W), indexing="ij")
    disk = (((yy - H / 2) ** 2 + (xx - W / 2) ** 2) < (0.3 * min(H, W)) ** 2).float()
    return (torch.rand(B, C_, H, W, generator=g) * disk).to(DEV)


def _target(x0, seed=0):
    g = torch.Generator().manual_seed(seed)
    return (UM.premultiply(x0[:1])[0] + 0.03 * torch.randn(4, *x0.shape[2:], generator=g).to(DEV)).contiguous()


def _schedule(m, B, H, W, T, *, fire="u", steps=None, damage_step=None, seed=0, philox_offset=0):
    """per-step fire rates and gains (every third gain 0), recorded uniforms or in-kernel Philox, optional damage and
    ragged steps"""
    random.seed(seed)
    graph = getattr(m, "_is_graph", False)
    offs = [m.graph.draw_offsets() for _ in range(T)] if graph else None
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
    s.philox_offset = philox_offset
    return s


@pytest.fixture
def launches(monkeypatch, capfd):
    """GNCA_DEBUG=1 for the test; calling the fixture's value returns (replicated, banded) launch tuples since the last
    call"""
    monkeypatch.setenv("GNCA_DEBUG", "1")
    monkeypatch.delenv("GNCA_RESIDENT_NC", raising=False)
    capfd.readouterr()

    def read():
        err = capfd.readouterr().err
        ints = lambda m: tuple(int(v) for v in m.groups())
        return [ints(m) for m in RE_REP.finditer(err)], [ints(m) for m in RE_BAND.finditer(err)]
    return read


def _check(m, x0, s, tgt, S, impl, read, family):
    """monitor(ssim=True) against monitor(ssim=False), ssim_rgb on the record_rollout frames, the oracle, and itself;
    `family` is 'rep', 'band' or 'stream', asserted from the launch lines of the SSIM call"""
    with torch.no_grad():
        read()
        try:
            mon = monitor_rollout(m, x0, s, tgt, every=S, impl=impl, ssim=True)
        except _lib.GncaError as e:
            assert "unsupported" in str(e)
            with pytest.raises(_lib.GncaError, match="unsupported"):
                monitor_rollout(m, x0, s, tgt, every=S, impl=impl)
            pytest.skip(f"{impl}: no kernel for this configuration")
        rep, band = read()
        if s.T > 0:
            assert {"rep": (len(rep), len(band)) == (1, 0), "band": (len(rep), len(band)) == (0, 1),
                    "stream": (len(rep), len(band)) == (0, 0)}[family], (family, rep, band)
        plain = monitor_rollout(m, x0, s, tgt, every=S, impl=impl)
        again = monitor_rollout(m, x0, s, tgt, every=S, impl=impl, ssim=True)
        tr = record_rollout(m, x0, s, every=S, impl=impl)
        on_frames = torch.stack([UM.ssim_rgb(f, tgt) for f in tr.states])
    assert plain.ssim is None and mon.ssim.dtype == torch.float32 and mon.ssim.shape == (len(tr.t), x0.shape[0])
    assert mon.t == plain.t == tr.t
    for f in ("loss", "psnr", "pixel_perfect", "alive", "x_T"):
        assert torch.equal(getattr(mon, f), getattr(plain, f)), f
    assert torch.equal(mon.ssim, again.ssim)
    assert (mon.ssim.double() - on_frames.double()).abs().max().item() <= 1e-12, (mon.ssim, on_frames)
    oracle = np.stack([SO.ssim_rgb(f, tgt) for f in tr.states])
    assert np.abs(mon.ssim.double().cpu().numpy() - oracle).max() <= 1e-5
    return mon


# name: T, every, fire, ragged steps, damage step, philox offset
CASES = {
    "S1": (7, 1, "u", None, None, 0),
    "S3_T%S!=0": (10, 3, "u", None, None, 0),
    "S>T": (9, 10, "u", None, None, 0),
    "T0": (0, 1, "u", None, None, 0),
    "ragged_philox_damage_at_frame": (10, 3, "philox", [10, 4], 6, 0),
    "ragged_u_damage_between_frames": (11, 3, "u", [5, 11], 4, 0),
    "ragged_frozen_on_frame": (12, 4, "u", [8, 3], None, 0),
    "damage_at_0": (6, 2, "u", None, 0, 0),
    "philox_offset": (10, 3, "philox", [10, 7], 5, 123457),
}
FAMILY = {"auto": "rep", "resident": "rep", "banded": "band", "streaming": "stream"}


@pytest.mark.parametrize("impl", ["auto", "resident", "banded", "streaming"])
@pytest.mark.parametrize("model", list(MODELS))
@pytest.mark.parametrize("case", list(CASES))
def test_monitor_ssim(case, model, impl, launches):
    T, S, fire, steps, dstep, poff = CASES[case]
    m = MODELS[model]()
    B, H, W = 2, 40, 40
    x0 = _blob(B, 16, H, W, seed=1)
    s = _schedule(m, B, H, W, T, fire=fire, steps=steps, damage_step=dstep, seed=3, philox_offset=poff)
    _check(m, x0, s, _target(x0), S, impl, launches, FAMILY[impl])


@pytest.mark.parametrize("model,C_,H,W,nc,family", [
    ("c32", 32, 40, 40, None, "band"),            # C = 32: the banded kernel under every cluster impl
    ("classic", 16, 40, 40, None, "band"),        # halo of 1 row: the window rows beyond it come over DSMEM
    ("classic", 16, 16, 24, "8", "band"),         # bands of 2 rows: a window spans three CTAs
    ("classic", 16, 8, 40, "8", "band"),          # bands of 1 row
    ("torus", 16, 32, 64, None, "rep"),           # 2048 cells on the replicated-state kernel
    ("torus", 16, 40, 41, None, "band"),          # odd W
    ("classic", 16, 37, 24, None, "band"),        # prime H: one CTA
])
def test_monitor_ssim_cluster_shapes(model, C_, H, W, nc, family, launches, monkeypatch):
    m = _random_graph(32, H) if model == "c32" else MODELS[model]()
    B, T, S = 3, 13, 4
    x0 = _blob(B, C_, H, W, seed=2)
    s = _schedule(m, B, H, W, T, fire="philox", steps=[13, 6, 13], damage_step=8, seed=4)
    impl = "resident" if family == "rep" else "banded"
    if nc:
        monkeypatch.setenv("GNCA_RESIDENT_NC", nc)
    mon = _check(m, x0, s, _target(x0), S, impl, launches, family)
    if nc:
        monkeypatch.delenv("GNCA_RESIDENT_NC")
        with torch.no_grad():       # the band split does not move a bit of the SSIM beyond the partition of its sums
            other = monitor_rollout(m, x0, s, _target(x0), every=S, impl=impl, ssim=True)
        assert (mon.ssim.double() - other.ssim.double()).abs().max().item() <= 1e-12


@pytest.mark.parametrize("impl", ["streaming", "auto"])
def test_monitor_ssim_large_problem_path(impl, launches):
    """256x256x32, B = 16: the tensor-core update (k_update_tc) with k_frame_ssim at the kept steps"""
    m = _random_graph(32, 256)
    B, H, W, T, S = 16, 256, 256, 12, 5
    x0 = _blob(B, 32, H, W, seed=3)
    s = _schedule(m, B, H, W, T, fire="philox", steps=[12] * 15 + [7], damage_step=6, seed=6, philox_offset=99)
    _check(m, x0, s, _target(x0), S, impl, launches, "stream")


@pytest.mark.parametrize("C_,H,W", [(16, 40, 40), (4, 7, 7), (16, 7, 40), (32, 41, 37), (4, 256, 256),
                                    (32, 256, 256), (16, 40, 7)])
def test_ssim_rgb_against_oracle(C_, H, W):
    g = torch.Generator().manual_seed(C_ + H * W)
    x = torch.rand(3, C_, H, W, generator=g) * 1.3 - 0.15
    x[0, :, : H // 2] *= 1e-3                               # near-flat windows
    x[1] = x[1].round()                                     # saturated values
    tgt = torch.rand(4, H, W, generator=g)
    tgt[:, : H // 3] = 0.5
    got = UM.ssim_rgb(x.to(DEV), tgt.to(DEV))
    assert got.shape == (3,) and got.dtype == torch.float32
    assert np.abs(got.double().cpu().numpy() - SO.ssim_rgb(x, tgt)).max() <= 1e-5
    assert torch.equal(got, UM.ssim_rgb(x.to(DEV), tgt.to(DEV)))


def test_ssim_rgb_on_grown_patterns():
    """40x40 frames of a trained model's rollout, against the oracle; a state equal to the target gives 1"""
    m = MODELS["torus"]()
    x0 = _blob(4, 16, 40, 40, seed=5)
    s = _schedule(m, 4, 40, 40, 24, fire="philox", seed=9)
    with torch.no_grad():
        fr = record_rollout(m, x0, s, every=8).states
    tgt = UM.premultiply(fr[-1][:1])[0].contiguous()
    for f in fr:
        assert np.abs(UM.ssim_rgb(f, tgt).double().cpu().numpy() - SO.ssim_rgb(f, tgt)).max() <= 1e-5
    x = fr[-1][:1].clone()
    x[:, 3] = 1.0
    t1 = UM.premultiply(x)[0].contiguous()
    assert abs(float(UM.ssim_rgb(x, t1)[0]) - 1.0) <= 1e-7


@pytest.mark.parametrize("impl", ["resident", "banded"])
@pytest.mark.parametrize("model", list(MODELS))
def test_monitor_ssim_stack_blocks(model, impl):
    """every block of a three-model stacked call equals that model's single-model call on the same batch"""
    M, B, H, W, T, S = 3, 2, 40, 40, 11, 3
    models = [MODELS[model](i) for i in range(M)]
    x0 = _blob(M * B, 16, H, W, seed=1)
    s = _schedule(models[0], M * B, H, W, T, fire="philox", steps=[11, 5] * M, damage_step=4, seed=3)
    tgt = _target(x0)
    with torch.no_grad():
        try:
            mon = monitor_rollout(models, x0, s, tgt, every=S, impl=impl, ssim=True)
        except _lib.GncaError as e:
            assert "unsupported" in str(e) and model == "zeropad" and impl == "banded"
            return
        plain = monitor_rollout(models, x0, s, tgt, every=S, impl=impl)
        for f in ("loss", "psnr", "pixel_perfect", "alive", "x_T"):
            assert torch.equal(getattr(mon, f), getattr(plain, f)), f
        for i in range(M):
            one = monitor_rollout(models[i], x0, s, tgt, every=S, impl=impl, ssim=True)
            blk = slice(i * B, (i + 1) * B)
            assert torch.equal(mon.ssim[:, blk], one.ssim[:, blk]), i
            assert torch.equal(mon.x_T[blk], one.x_T[blk]), i


def test_monitor_ssim_large_sweep():
    """150 models at B = 1 in one call: two members against their single-model calls"""
    M, H, W, T, S = 150, 40, 40, 20, 5
    base = MODELS["zeropad"]()
    models = [base] + [_perturb(_graph16(False, 0), i, 0.03) for i in range(1, M)]
    x0 = _blob(M, 16, H, W, seed=7)
    s = _schedule(base, M, H, W, T, fire="philox", damage_step=10, seed=8)
    tgt = _target(x0)
    with torch.no_grad():
        mon = monitor_rollout(models, x0, s, tgt, every=S, ssim=True)
        for i in (0, 149):
            one = monitor_rollout(models[i], x0, s, tgt, every=S, ssim=True)
            assert torch.equal(mon.ssim[:, i], one.ssim[:, i]) and torch.equal(mon.x_T[i], one.x_T[i]), i
    assert torch.isfinite(mon.ssim).all() and not torch.equal(mon.ssim[:, 0], mon.ssim[:, 1])

"""The grid-shape envelope of the cluster-resident BPTT, tabulated through the C ABI without a GPU.

gnca_bptt_bytes and gnca_bptt_ckpt_bytes (torus and classic models) and gnca_bptt_zp_bytes (zero-padded graph shift
models) are > 0 exactly when W % 4 == 0, W >= 4, H <= 64, W <= 64 and H * W <= 2048, and 0 for the other model kind.
bptt_plan names the history rollout(..., bptt_budget=N) keeps on the shapes that tests/test_gpu_grid_envelope.py runs,
so its assertions about which kernel family ran rest on these predicates."""
import ctypes as C

import pytest

# both sides of every boundary: W % 4, W >= 4, H <= 64, W <= 64, H * W <= 2048 (2048 = 64 x 32 = 32 x 64 = 1 x 2048
# is out since W > 64), and the grids of the GPU tests
HS = (1, 4, 5, 20, 31, 32, 33, 36, 37, 44, 46, 48, 63, 64, 65, 68, 128)
WS = (1, 2, 3, 4, 5, 6, 8, 20, 24, 32, 36, 40, 41, 42, 44, 60, 61, 64, 65, 68, 128)
EXTRA = ((45, 44), (46, 44), (47, 44), (51, 40), (52, 40), (64, 33), (64, 36), (32, 64), (33, 64), (34, 60), (56, 36),
         (57, 36))


@pytest.fixture(scope="module")
def lib():
    from graph_neural_cellular_automata_b200 import _lib, build
    build.build(verbose=False)
    return _lib.load()


def _desc(kind, C_=16, hidden=128, d=16):
    from graph_neural_cellular_automata_b200 import functional as GF
    return GF.make_model_desc(C_, hidden, d, graph=kind != "classic", torus=kind == "torus", hidden_only=True,
                              alive_to_alive=True, groupnorm=True, update_gain=0.05, alpha_thr=0.12,
                              graph_alpha_thr=0.12)


def _eligible(H, W):
    return W % 4 == 0 and W >= 4 and H <= 64 and W <= 64 and H * W <= 2048


def _al(v):
    return (v + 255) // 256 * 256


def _records(B, H, W, T):
    """records, h | gh rows, three 64-word bitmaps and the statistics of every (t, b): the bitmaps are 64 words whatever
    H * W, so a partial last word and a full 2048-cell bitmap take the same room"""
    HW = H * W
    return _al(T * B * HW * 100 * 4) + T * B * HW * 256 * 4 + T * B * 3 * 64 * 4 + T * B * 2 * 4 + 256


def _shapes():
    return [(H, W) for H in HS for W in WS] + list(EXTRA)


def test_the_table_has_both_sides_of_every_boundary():
    shapes = _shapes()
    inside = [s for s in shapes if _eligible(*s)]
    assert (64, 32) in inside and (32, 64) in inside and (33, 60) in inside and (5, 8) in inside and (64, 4) in inside
    assert any(h * w == 2048 for h, w in inside)
    assert any(h * w % 32 for h, w in inside)
    outside = [s for s in shapes if not _eligible(*s)]
    for reason in (lambda h, w: w % 4, lambda h, w: w < 4, lambda h, w: h > 64 and w <= 64 and w % 4 == 0 and h * w <= 2048,
                   lambda h, w: w > 64 and w % 4 == 0, lambda h, w: h * w > 2048 and h <= 64 and w <= 64 and w % 4 == 0):
        assert any(reason(h, w) for h, w in outside)


@pytest.mark.parametrize("kind", ["torus", "classic", "zeropad"])
@pytest.mark.parametrize("B,T", [(1, 1), (3, 7)])
def test_bptt_buffers_exist_exactly_inside_the_envelope(lib, kind, B, T):
    d = _desc(kind)
    wrong = []
    for H, W in _shapes():
        ok = _eligible(H, W)
        rec = lib.gnca_bptt_bytes(C.byref(d), B, H, W, T)
        ck = lib.gnca_bptt_ckpt_bytes(C.byref(d), B, H, W, T)
        zp = lib.gnca_bptt_zp_bytes(C.byref(d), B, H, W, T)
        if kind == "zeropad":
            got = (rec, ck, zp > 0)
            want = (0, 0, ok)
        else:
            got = (rec, ck > 0, zp)
            want = (_records(B, H, W, T) if ok else 0, ok, 0)
        if got != want:
            wrong.append((H, W, got, want))
    assert not wrong, wrong


@pytest.mark.parametrize("kind", ["torus", "classic"])
def test_ckpt_segment_bytes_at_the_edges(lib, kind):
    """the segment of the checkpointed resident BPTT: the records of K steps, then the carried gradient and x_T"""
    d = _desc(kind)
    for H, W in ((64, 32), (32, 64), (36, 20), (33, 60), (44, 44), (64, 4), (5, 8)):
        N = 3 * 16 * H * W * 4
        for K in (1, 3, 8):
            assert lib.gnca_bptt_ckpt_bytes(C.byref(d), 3, H, W, K) == _al(_records(3, H, W, K)) + 2 * _al(N), (H, W, K)


@pytest.mark.parametrize("case", ["C32", "hidden64", "d33"])
def test_other_models_have_no_resident_bptt_at_any_grid(lib, case):
    kinds = ("torus", "classic", "zeropad")
    for kind in kinds:
        if case == "C32":
            d = _desc(kind, C_=32)
        elif case == "hidden64":
            d = _desc(kind, hidden=64)
        else:
            d = _desc(kind, d=33)
            if kind != "zeropad":
                continue
        for H, W in ((64, 32), (36, 20), (5, 8)):
            assert lib.gnca_bptt_bytes(C.byref(d), 2, H, W, 4) == 0
            assert lib.gnca_bptt_ckpt_bytes(C.byref(d), 2, H, W, 4) == 0
            assert lib.gnca_bptt_zp_bytes(C.byref(d), 2, H, W, 4) == 0


# ---- bptt_plan on the grids of the GPU tests --------------------------------------------------------------------------
def _plan(d, B, H, W, T, budget, impl="auto", k=8):
    from graph_neural_cellular_automata_b200.rollout import IMPL, _bptt_plan
    return _bptt_plan(d, B, H, W, T, budget, IMPL[impl], k)


BIG = 1 << 40


@pytest.mark.parametrize("H,W", [(64, 32), (32, 64), (36, 20), (20, 36), (33, 60), (44, 44), (64, 4), (5, 8)])
@pytest.mark.parametrize("kind", ["torus", "classic", "zeropad"])
def test_plan_inside_the_envelope(lib, H, W, kind):
    """without a binding budget: the records (torus, classic) or the dense history (zero-pad, which has no checkpointed
    resident BPTT); under a budget below the records: the resident checkpoints with K > 1 (torus, classic)"""
    d = _desc(kind)
    B, T = 3, 7
    if kind == "zeropad":
        assert _plan(d, B, H, W, T, BIG)[0] == "dense"
        with pytest.raises(ValueError, match="resident"):
            _plan(d, B, H, W, T, BIG, impl="resident")
        return
    assert _plan(d, B, H, W, T, BIG) == ("records", None, _records(B, H, W, T))
    n = B * 16 * H * W * 4
    budget = (T // 3 + 1) * n + lib.gnca_bptt_ckpt_bytes(C.byref(d), B, H, W, 3)
    path, K, nb = _plan(d, B, H, W, T, budget)
    assert path == "resident_ckpt" and 3 <= K < T and nb <= budget
    assert _plan(d, B, H, W, T, budget, impl="resident")[0] == "resident_ckpt"


@pytest.mark.parametrize("H,W", [(40, 42), (48, 48), (68, 8), (48, 41), (64, 64), (96, 96), (128, 128)])
@pytest.mark.parametrize("kind", ["torus", "classic"])
def test_plan_outside_the_envelope(lib, H, W, kind):
    """grids the resident BPTT does not take: the dense history, the streaming checkpoints under a budget, and a
    ValueError for impl='resident' with a budget"""
    d = _desc(kind)
    B, T = 2, 6
    n = B * 16 * H * W * 4
    assert _plan(d, B, H, W, T, BIG) == ("dense", None, (T + 1) * n + T * n + T * B * 2 * 4)
    path, K, _ = _plan(d, B, H, W, T, 3 * n + lib.gnca_ckpt_segment_bytes(C.byref(d), B, H, W, 3))
    assert path == "streaming_ckpt" and K >= 3
    with pytest.raises(ValueError, match="resident"):
        _plan(d, B, H, W, T, BIG, impl="resident")


def test_plan_more_than_16_offsets_leaves_the_resident_branches_out(lib):
    d = _desc("torus")
    assert _plan(d, 3, 64, 32, 7, BIG, k=17)[0] == "dense"
    assert _plan(d, 3, 64, 32, 7, BIG, k=16)[0] == "records"

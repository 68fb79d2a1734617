"""CPU checks of the resident BPTT of the zero-padded graph shift: the C ABI (gnca_bptt_zp_bytes,
gnca_rollout_fwd_bptt_zp, gnca_rollout_bwd_bptt_zp) -- symbols, the buffer size and where it is 0, argument errors that
return before any launch -- and that the paths it leaves alone (gnca_bptt_bytes, the budget planner) still see no
resident BPTT for zero-pad models."""
import ctypes as C
import os
import re

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NAMES = ("gnca_bptt_zp_bytes", "gnca_rollout_fwd_bptt_zp", "gnca_rollout_bwd_bptt_zp")


@pytest.fixture(scope="module")
def lib():
    from graph_neural_cellular_automata_b200 import _lib, build
    build.build(verbose=False)
    return _lib.load()


def _desc(C_=16, torus=False, graph=True, hidden=128, d=16):
    from graph_neural_cellular_automata_b200 import functional as GF
    return GF.make_model_desc(C_, hidden, d, graph=graph, torus=torus, hidden_only=True, alive_to_alive=True,
                              groupnorm=True, update_gain=0.05, alpha_thr=0.12, graph_alpha_thr=0.12)


def test_symbols_are_exported_and_bound(lib):
    from graph_neural_cellular_automata_b200 import _lib
    header = open(os.path.join(ROOT, "include", "gnca.h")).read()
    for name in NAMES:
        assert re.search(rf"\b(size_t|int) {name}\(", header), name
        assert name in _lib.EXPORTS
        assert getattr(lib, name).argtypes == _lib.EXPORTS[name][1]


def _al(v):
    return (v + 255) // 256 * 256


def _records(B, H, W, T):
    """gnca_bptt_bytes of the same shape on a torus model: records, h | gh rows, bitmaps, statistics"""
    HW = H * W
    return _al(T * B * HW * 100 * 4) + T * B * HW * 256 * 4 + T * B * 3 * 64 * 4 + T * B * 2 * 4 + 256


@pytest.mark.parametrize("B,H,W,T,d", [(32, 40, 40, 64, 16), (4, 40, 40, 1, 1), (1, 8, 4, 0, 32), (9, 24, 32, 13, 8),
                                       (3, 32, 64, 5, 16)])
def test_buffer_bytes(lib, B, H, W, T, d):
    HW, np_ = H * W, 2 * d * 16 + 2 * d + 1
    want = (_al(_records(B, H, W, T)) + _al((T + 1) * B * 16 * HW * 4) + _al(T * B * 16 * 4) + _al(T * B * 16 * H * 4)
            + _al(B * HW * 4) + _al(B * np_ * 4))
    assert lib.gnca_bptt_zp_bytes(C.byref(_desc(d=d)), B, H, W, T) == want
    assert lib.gnca_bptt_bytes(C.byref(_desc(torus=True, d=d)), B, H, W, T) == _records(B, H, W, T)


@pytest.mark.parametrize("case", ["torus", "classic", "C32", "hidden64", "d33", "64x64", "W_not_4", "W_2", "bad_B",
                                  "bad_T", "null_model"])
def test_buffer_bytes_zero_where_not_supported(lib, case):
    d, B, H, W, T = _desc(), 4, 40, 40, 8
    if case == "torus":
        d = _desc(torus=True)
    elif case == "classic":
        d = _desc(graph=False)
    elif case == "C32":
        d = _desc(32)
    elif case == "hidden64":
        d = _desc(hidden=64)
    elif case == "d33":
        d = _desc(d=33)
    elif case == "64x64":
        H = W = 64
    elif case == "W_not_4":
        W = 42
    elif case == "W_2":
        W = 2
    elif case == "bad_B":
        B = 0
    elif case == "bad_T":
        T = -1
    assert lib.gnca_bptt_zp_bytes(None if case == "null_model" else C.byref(d), B, H, W, T) == 0


def test_existing_entry_points_still_exclude_zero_pad(lib):
    """gnca_bptt_bytes and gnca_bptt_ckpt_bytes keep returning 0 for zero-pad models: the records of the torus path and
    its checkpoints do not apply to them."""
    d = _desc()
    assert lib.gnca_bptt_zp_bytes(C.byref(d), 4, 40, 40, 8) > 0
    assert lib.gnca_bptt_bytes(C.byref(d), 4, 40, 40, 8) == 0
    assert lib.gnca_bptt_ckpt_bytes(C.byref(d), 4, 40, 40, 4) == 0


def test_budget_plan_keeps_the_dense_history_for_zero_pad():
    """bptt_plan plans over the dense history and streaming checkpoints only for zero-pad models."""
    from graph_neural_cellular_automata_b200.rollout import _bptt_plan, IMPL
    d = _desc()
    path, every, nbytes = _bptt_plan(d, 32, 40, 40, 64, 1 << 40, IMPL["auto"], 8)
    assert path == "dense" and every is None
    path, every, _ = _bptt_plan(d, 32, 40, 40, 64, nbytes // 4, IMPL["auto"], 8)
    assert path == "streaming_ckpt" and every >= 1


P = C.c_void_p(256)        # never dereferenced: every call below fails its argument checks first
BIG = 1 << 40


def _sched(case):
    from graph_neural_cellular_automata_b200 import _lib
    p = C.c_void_p(512)
    s = _lib.GncaSchedule(4, 8, p, p, p, None, None, 0, 0, None, 0, 4, 0, 0)
    if case == "k65":
        s.k = _lib.GNCA_MAX_K + 1
    elif case == "k_neg":
        s.k = -1
    elif case == "T_neg":
        s.T = -1
    elif case == "null_fire_rate":
        s.fire_rate = None
    elif case == "null_gain":
        s.message_gain = None
    elif case == "null_offsets":
        s.offsets = None
    return s


def _fwd(lib, sched, *, desc=None, every=2, frames=P, x0=P, xT=P, packed=P, bptt=P, bptt_bytes=BIG, ws=P,
         ws_bytes=BIG, model=True, B=2, **_):
    d = desc or _desc()
    return lib.gnca_rollout_fwd_bptt_zp(C.byref(d) if model else None, packed, B, 40, 40, C.byref(sched), x0, xT, every,
                                        frames, bptt, bptt_bytes, ws, ws_bytes, None)


def _bwd(lib, sched, *, desc=None, every=2, g_frames=P, gT=P, g0=P, gparams=P, packed=P, bptt=P, bptt_bytes=BIG,
         ws=P, ws_bytes=BIG, model=True, B=2, **_):
    d = desc or _desc()
    return lib.gnca_rollout_bwd_bptt_zp(C.byref(d) if model else None, packed, B, 40, 40, C.byref(sched), bptt,
                                        bptt_bytes, every, g_frames, gT, g0, gparams, ws, ws_bytes, None)


CASES = {
    "every0": ("ARG", dict(every=0)),
    "every_neg": ("ARG", dict(every=-3)),
    "null_model": ("ARG", dict(model=False)),
    "null_packed": ("ARG", dict(packed=None)),
    "null_bptt": ("ARG", dict(bptt=None)),
    "null_workspace": ("ARG", dict(ws=None)),
    "B0": ("ARG", dict(B=0)),
    "null_gain": ("ARG", {}),
    "null_offsets": ("ARG", {}),
    "T_neg": ("ARG", {}),
    "bptt_small": ("WORKSPACE", dict(bptt_bytes=1024)),
    "workspace_small": ("WORKSPACE", dict(ws_bytes=1024)),
    "k65": ("UNSUPPORTED", {}),
    "k_neg": ("UNSUPPORTED", {}),
    "torus": ("UNSUPPORTED", dict(desc=_desc(torus=True))),
    "classic": ("UNSUPPORTED", dict(desc=_desc(graph=False))),
    "d33": ("UNSUPPORTED", dict(desc=_desc(d=33))),
}
FWD_ONLY = {
    "null_x0": ("ARG", dict(x0=None)),
    "null_xT": ("ARG", dict(xT=None)),
    "null_fire_rate": ("ARG", {}),
}
BWD_ONLY = {
    "null_gT": ("ARG", dict(gT=None)),
    "null_g0": ("ARG", dict(g0=None)),
    "null_gparams": ("ARG", dict(gparams=None)),
}


@pytest.mark.parametrize("case", list(CASES) + list(FWD_ONLY))
def test_forward_argument_errors(lib, case):
    from graph_neural_cellular_automata_b200 import _lib
    code, kw = {**CASES, **FWD_ONLY}[case]
    assert _fwd(lib, _sched(case), **kw) == getattr(_lib, "GNCA_ERR_" + code)


@pytest.mark.parametrize("case", list(CASES) + list(BWD_ONLY))
def test_backward_argument_errors(lib, case):
    from graph_neural_cellular_automata_b200 import _lib
    code, kw = {**CASES, **BWD_ONLY}[case]
    assert _bwd(lib, _sched(case), **kw) == getattr(_lib, "GNCA_ERR_" + code)


def test_every_is_only_checked_with_frames(lib):
    """every <= 0 is an error only when frames (forward) or frame gradients (backward) are given: with neither, the call
    gets as far as the workspace check."""
    from graph_neural_cellular_automata_b200 import _lib
    s = _sched("plain")
    assert _fwd(lib, s, every=0, frames=None, ws_bytes=1024) == _lib.GNCA_ERR_WORKSPACE
    assert _bwd(lib, s, every=0, g_frames=None, ws_bytes=1024) == _lib.GNCA_ERR_WORKSPACE

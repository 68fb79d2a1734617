"""Rollout = T CA steps in ONE library call (gnca_rollout_fwd / gnca_rollout_bwd).

The reference has no rollout function: every script runs a Python `for` over `model(state[mask], fire_rate=fr)`
(train_graph_augmented_nca.py:305-321, test_graph_augmented_regeneration.py:183-194, ...).  The contract of this
extension is "equals T sequential `forward` calls given the same random draws".  A `Schedule` holds those draws
on the device: per-step fire rate, message gain and offsets, per-sample step counts, and the fire uniforms
(either a recorded/pre-drawn tensor or an in-kernel Philox stream).
"""
from __future__ import annotations

import ctypes as C
import random
from dataclasses import dataclass
from typing import List, Optional, Sequence, Tuple, Union

import numpy as np
import torch

from . import _lib
from . import functional as GF
from ._lib import GncaSchedule

Offset = Tuple[int, int]


@dataclass
class Schedule:
    """Device-resident per-step schedule of a rollout (mirror of `gnca_schedule` in include/gnca.h)."""
    T: int
    k: int
    fire_rate: torch.Tensor                 # [T] f32
    message_gain: torch.Tensor              # [T] f32
    offsets: Optional[torch.Tensor]         # [T,k,2] int8
    steps: Optional[torch.Tensor] = None    # [B] int32
    fire_u: Optional[torch.Tensor] = None   # [T,B,H,W] f32 (row b = sample b)
    philox_seed: int = 0
    philox_offset: int = 0
    damage: Optional[torch.Tensor] = None   # multiplicative mask: [B,C,H,W] (layout 0) or a per-cell plane [B,H,W]
    damage_step: int = 0
    damage_layout: int = 0                  # 0 dense, 1 plane on every channel, 2 plane on alpha only (include/gnca.h)
    total_updates: Optional[int] = None     # sum_b steps_b (host int, for throughput accounting)
    max_offset: int = 0                     # max(|dy|,|dx|) over the offsets (halo depth of the resident kernel)

    def c_struct(self) -> GncaSchedule:
        p = lambda t: C.c_void_p(0 if t is None else t.data_ptr())
        return GncaSchedule(self.T, self.k, p(self.fire_rate), p(self.message_gain), p(self.offsets), p(self.steps),
                            p(self.fire_u), C.c_uint64(self.philox_seed), C.c_uint64(self.philox_offset),
                            p(self.damage), self.damage_step, self.max_offset, int(self.damage_layout), 0)


class _PinnedRing:
    """A few reusable pinned staging buffers (pinning memory per call costs ~100 us); a buffer is reused only after
    the event recorded behind its last H2D copy has completed."""

    def __init__(self, slots: int = 8):
        self.slots, self.buf, self.ev, self.i = slots, [None] * slots, [None] * slots, 0

    def get(self, nbytes: int):
        i = self.i
        self.i = (i + 1) % self.slots
        if self.ev[i] is not None:
            self.ev[i].synchronize()
        if self.buf[i] is None or self.buf[i].numel() < nbytes:
            self.buf[i] = torch.empty(max(nbytes, 1 << 14), dtype=torch.uint8).pin_memory()
        return i, self.buf[i]

    def mark(self, i: int):
        ev = torch.cuda.Event()
        ev.record()
        self.ev[i] = ev


_RING = _PinnedRing()
_TORCH_DTYPE = {np.dtype(np.float32): torch.float32, np.dtype(np.int8): torch.int8, np.dtype(np.int32): torch.int32,
                np.dtype(np.uint8): torch.uint8, np.dtype(np.int64): torch.int64}


def _upload(arrs: Sequence[np.ndarray], device) -> List[torch.Tensor]:
    """One pinned staging buffer, one async H2D copy, typed device views."""
    sizes = [a.nbytes for a in arrs]
    offs, o = [], 0
    for s in sizes:
        offs.append(o)
        o += (s + 15) // 16 * 16
    total = max(o, 16)
    on_cuda = torch.device(device).type == "cuda"
    if on_cuda:
        slot, host = _RING.get(total)
    else:
        host = torch.empty(total, dtype=torch.uint8)
    hv = host.numpy()
    for a, off in zip(arrs, offs):
        hv[off:off + a.nbytes].view(a.dtype)[:] = a.reshape(-1)
    if on_cuda:
        dev = torch.empty(total, dtype=torch.uint8, device=device)
        dev.copy_(host[:total], non_blocking=True)
        _RING.mark(slot)
    else:
        dev = host[:total].clone()
    out = []
    for a, off in zip(arrs, offs):
        t = dev[off:off + a.nbytes].view(_TORCH_DTYPE[a.dtype]).view(a.shape)
        out.append(t)
    return out


def make_schedule(model, B: int, H: int, W: int, T: int, *, fire_rate: Union[float, Sequence[float]] = 1.0,
                  message_gains: Optional[Sequence[float]] = None, message_every: int = 1,
                  offsets: Optional[Sequence[Sequence[Offset]]] = None, steps: Optional[Sequence[int]] = None,
                  fire: str = "philox", fire_u: Optional[torch.Tensor] = None, seed: Optional[int] = None,
                  damage: Optional[torch.Tensor] = None, damage_step: int = 0, device=None) -> Schedule:
    """Build the schedule the way T sequential `forward` calls would consume randomness.

    * offsets: drawn with `random.sample(model.graph.offsets, k)` once per step (graph models), exactly like
      graph_augmentation.py:120-121, unless given.
    * fire="torch": one `torch.rand(B,1,H,W)` per step on the model device (bit-identical stream to T forward
      calls with a fixed fire_rate < 1); fire="philox": in-kernel Philox4x32-10 keyed by `seed` (no HBM traffic,
      statistically equivalent, different numbers); or pass recorded `fire_u` [T,B,H,W].
    * damage: a `utils.damage.Damage` (descriptor evaluated to a per-cell plane, applied in-kernel before step
      `damage_step`) or a dense [B,C,H,W] mask tensor.
    * message_gains: per-step `model.message_gain` (the trainer sets gain or 0 per step, train...:312-319);
      default = model.message_gain on steps with t % message_every == 0, else 0.
    """
    device = device or next(model.parameters()).device
    is_graph = bool(getattr(model, "_is_graph", False))
    fr = np.full(T, float(fire_rate), np.float32) if np.isscalar(fire_rate) else np.asarray(fire_rate, np.float32)
    assert fr.shape == (T,)
    if is_graph:
        if offsets is None:
            off = model.graph.draw_offsets_array(T)          # same python-RNG stream as T forward calls
        elif isinstance(offsets, np.ndarray):
            off = offsets.astype(np.int8, copy=False).reshape(T, -1, 2)
        else:
            k_ = len(offsets[0]) if T > 0 else 0
            flat = [v for st in offsets for o in st for v in o]
            off = np.asarray(flat, dtype=np.int8).reshape(T, k_, 2) if k_ > 0 else np.zeros((T, 0, 2), np.int8)
        k = off.shape[1]
        if message_gains is None:
            g = float(model.message_gain)
            message_gains = [g if (message_every <= 1 or t % message_every == 0) else 0.0 for t in range(T)]
    else:
        k, off = 0, np.zeros((T, 0, 2), np.int8)
        message_gains = [0.0] * T
    gains = np.asarray(message_gains, np.float32)
    arrs = [fr, gains, off if off.size else np.zeros(2, np.int8)]
    if steps is not None:
        st = np.asarray(steps, np.int32)
        assert st.shape == (B,)
        arrs.append(st)
        total = int(np.minimum(st, T).clip(min=0).sum())
    else:
        total = B * T
    dev = _upload(arrs, device)
    damage_layout = 0
    if damage is not None and hasattr(damage, "plane"):              # utils.damage.Damage
        damage_layout, damage = int(damage.layout), GF._require_cuda_f32(damage.plane, "damage plane")
        if tuple(damage.shape) != (B, H, W):
            raise ValueError(f"damage plane has shape {tuple(damage.shape)}, expected {(B, H, W)}")
    elif damage is not None:
        damage = GF._require_cuda_f32(damage, "damage")
    sched = Schedule(T=T, k=k, fire_rate=dev[0], message_gain=dev[1], offsets=dev[2] if off.size else None,
                     steps=dev[3] if steps is not None else None, damage=damage, damage_step=int(damage_step),
                     damage_layout=damage_layout,
                     total_updates=total, max_offset=int(np.abs(off).max()) if off.size else 0)
    needs_fire = bool((fr < 1.0).any())
    if fire_u is not None:
        sched.fire_u = GF._require_cuda_f32(fire_u, "fire_u").view(T, B, H, W)
    elif needs_fire and fire == "torch":
        buf = torch.empty(T, B, 1, H, W, dtype=torch.float32, device=device)
        for t in range(T):
            if fr[t] < 1.0:
                torch.rand(B, 1, H, W, out=buf[t])
        sched.fire_u = buf.view(T, B, H, W)
    elif needs_fire:
        if fire != "philox":
            raise ValueError("fire must be 'torch' or 'philox'")
        sched.philox_seed = int(seed if seed is not None else random.getrandbits(63))
    return sched


class History:
    """What the forward keeps for BPTT.  Two formats:
    * records (`bptt`): the replicated-state kernel's per-active-cell records + bitmaps + statistics -- consumed by the
      cluster-resident backward (gnca_rollout_bwd_bptt); `x` is only filled when the caller asked for the history.
      `zp`: the zero-padded graph shift's buffer (gnca_bptt_zp_bytes: the records plus x_t, the attention weights and
      row sums), consumed by gnca_rollout_bwd_bptt_zp;
    * dense: x_t for every step and (optionally) the masked pre-norm update of the active cells + the GroupNorm
      statistics, consumed by the streaming backward (gnca_rollout_bwd).
    `frames` (forward with `every`): x_{f*every} in a buffer of its own, the differentiable states of `record_rollout`.
    `ckpt` (forward with a BPTT budget that called for checkpoints): x_{f*every} only, recomputed segment by segment on
    the resident (`resident`) or the streaming kernels from every (ckpt_every / every)-th of them, so segments are
    `ckpt_every` steps long (default `every`; a multiple of it when the frames of `record_rollout` are the checkpoints);
    `plan` is the bptt_plan result of that forward."""

    def __init__(self, x, u=None, stats=None, bptt=None, shape=None, frames=None, ckpt=None, every=0, resident=False,
                 zp=False, ckpt_every=None):
        self.x, self.u, self.stats, self.bptt, self.frames, self.zp = x, u, stats, bptt, frames, zp
        self.ckpt, self.every, self.resident, self.plan = ckpt, every, resident, None
        self.ckpt_every = ckpt_every or every
        self._shape = tuple(shape) if shape is not None else tuple(x.shape)

    @property
    def shape(self):
        return self._shape

    def __getitem__(self, i):
        return self.x[i]


_QUANT_SLACK_BYTES = 8 << 30        # never over-allocate more than this for the sake of a stable block size


def _round_up_steps(T: int, q: int = 64) -> int:
    return T if T <= 16 else -(-T // q) * q


BPTT_MAX_BYTES = 48 << 30      # above this the record buffer is not worth it: dense history + streaming backward


def _record_bytes(lib, desc, B: int, H: int, W: int, T: int, nbytes=None) -> int:
    """Bytes of the record buffer the resident BPTT forward allocates for T steps, or 0 when `rollout()` takes the dense
    history instead (configuration without records, T = 0, or more than BPTT_MAX_BYTES).  `nbytes`: the size function
    of the buffer (default gnca_bptt_bytes; gnca_bptt_zp_bytes for the zero-padded graph shift)."""
    if T <= 0:
        return 0
    nbytes = nbytes or lib.gnca_bptt_bytes
    nb = nbytes(C.byref(desc), B, H, W, T)
    if not 0 < nb <= BPTT_MAX_BYTES:
        return 0
    # the record buffer is GBs (T*B*H*W*1.4 KB worst case): sized for T rounded up to 64 steps, so that rollouts of
    # slightly different lengths (per-iteration step counts of the trainer) ask the caching allocator for the SAME
    # block instead of a fresh cudaMalloc whenever a new maximum shows up (70 ms for 29 GB in the long regime)
    nb_q = nbytes(C.byref(desc), B, H, W, _round_up_steps(T))
    if nb <= nb_q <= BPTT_MAX_BYTES and nb_q - nb <= _QUANT_SLACK_BYTES:
        nb = nb_q
    return nb


def _dense_steps(T: int, n_state: int) -> int:
    """Steps the dense history is allocated for (T rounded up like the record buffer, within the same slack)."""
    Tq = _round_up_steps(T)
    return T if (Tq - T) * n_state * 4 > _QUANT_SLACK_BYTES else Tq


def _dense_bytes(B: int, Cc: int, H: int, W: int, T: int) -> int:
    """Bytes of the dense history rollout_fwd_raw allocates: x_t of T + 1 steps, u_t and the statistics of T steps."""
    n = B * Cc * H * W
    Tq = _dense_steps(T, n)
    return (Tq + 1) * n * 4 + ((Tq * n * 4 + Tq * B * 2 * 4) if T > 0 else 0)


RESIDENT_MAX_K = 16      # offsets per step the resident kernels take (gnca_rep.cu, rep_bwd_supported)


def _bptt_plan(desc, B: int, H: int, W: int, T: int, budget: int, impl: int, k: int = 0, resident_ok: bool = True,
               every: Optional[int] = None):
    """bptt_plan on a model descriptor, an impl code and the schedule's offsets per step k; `resident_ok=False` leaves
    the resident branches out (the launch found no resident backward for the batch).  `every`: the plan of
    record_rollout(..., bptt_budget=...) with frames every `every` steps."""
    lib = _lib.load()
    n_bytes = B * desc.C * H * W * 4
    who = "rollout" if every is None else "record_rollout"
    resident_ok = resident_ok and k <= RESIDENT_MAX_K
    eligible = resident_ok and lib.gnca_bptt_ckpt_bytes(C.byref(desc), B, H, W, 1) > 0
    if impl == IMPL["resident"] and not eligible:
        raise ValueError(f"{who}: impl='resident' with bptt_budget needs the resident BPTT, which this model / shape "
                         f"does not have (16 channels, hidden 128, classic or torus graph, H*W <= 2048, W % 4 == 0, "
                         f"at most {RESIDENT_MAX_K} offsets per step)")
    nrec = _record_bytes(lib, desc, B, H, W, T) if (impl in (IMPL["auto"], IMPL["resident"]) and resident_ok) else 0
    if nrec:
        today = ("records", None, nrec)
    elif impl == IMPL["resident"]:
        today = None                                   # the dense history belongs to the streaming backward
    else:
        today = ("dense", None, _dense_bytes(B, desc.C, H, W, T))
    if today is not None and today[2] <= budget:
        return today
    branches = []
    if eligible and impl in (IMPL["auto"], IMPL["resident"]):
        branches.append(("resident_ckpt", lambda K: lib.gnca_bptt_ckpt_bytes(C.byref(desc), B, H, W, K)))
    if impl in (IMPL["auto"], IMPL["streaming"]):
        branches.append(("streaming_ckpt", lambda K: lib.gnca_ckpt_segment_bytes(C.byref(desc), B, H, W, K)))
    smallest = today[2] if today is not None else None
    if every is not None:
        # the frames are the checkpoints, so only the segment buffer comes on top of them.  Resident segments span a
        # whole number of frames: the largest such K that fits, from the first multiple of `every` that covers T (one
        # segment) down; streaming segments are one frame interval long (gnca_rollout_bwd_ckpt).
        for path, segment_bytes in branches:
            Ks = range(-(-max(T, 1) // every) * every, 0, -every) if path == "resident_ckpt" else (every,)
            for K in Ks:
                need = segment_bytes(K)
                if need <= budget:
                    return path, K, need
                smallest = need if smallest is None else min(smallest, need)
        raise ValueError(f"record_rollout: bptt_budget={budget} bytes is too small for this recording (B={B}, {H}x{W}, "
                         f"T={T}, every={every}); the smallest budget that works is {smallest} bytes")
    for path, segment_bytes in branches:
        # largest K first: the fewest segment launches (the recompute costs one forward whatever K is)
        for K in range(max(T, 1), 0, -1):
            need = (T // K + 1) * n_bytes + segment_bytes(K)
            if need <= budget:
                return path, K, need
            smallest = need if smallest is None else min(smallest, need)
    raise ValueError(f"rollout: bptt_budget={budget} bytes is too small for this rollout (B={B}, {H}x{W}, T={T}); "
                     f"the smallest budget that works is {smallest} bytes")


def bptt_plan(model, B: int, H: int, W: int, T: int, budget: int, impl: str = "auto", k: Optional[int] = None, *,
              every: Optional[int] = None):
    """Which BPTT history `rollout(..., bptt_budget=budget)` keeps for a B x C x H x W batch over T steps, without
    touching the GPU: `(path, every, bytes)`.

    * "records" / "dense": the history `rollout()` keeps without a budget (resident records, or the dense x_t / u_t
      history of the streaming backward), when it fits; `every` is None.
    * "resident_ckpt": x_{j*every} only, each segment's records recomputed on the resident kernels (models and shapes
      that have the resident BPTT).
    * "streaming_ckpt": x_{j*every} only, recomputed on the streaming kernels (`checkpoint_every`).
    `every` is the largest stride whose checkpoints plus segment buffer fit; `bytes` is what the history takes (the
    rollout workspace comes on top).  ValueError names the smallest budget that works when nothing fits.

    `k`: offsets per step of the schedule (default: what `make_schedule` draws for the model, 0 for a classic model);
    more than RESIDENT_MAX_K leaves the resident branches out, as in rollout().  rollout() takes this plan, except when
    the resident backward finds no cluster launch configuration for the batch at run time: it then plans again
    without the resident branches.

    Zero-padded graph shift models: the plan is over the dense history and streaming checkpoints only.  The resident
    zero-pad BPTT that rollout() takes without a budget (gnca_bptt_zp_bytes) has no checkpointed form, so under a budget
    these models keep the dense history when it fits.

    `every=S` (keyword only): the plan of `record_rollout(..., every=S, differentiable=True, bptt_budget=budget)`, whose
    frames x_{f*S} are returned whatever the plan, so `bytes` counts what the BPTT keeps beyond them and x_T:
    * "records" / "dense": the history record_rollout keeps without a budget, when it fits;
    * ("resident_ckpt", K, segment bytes): the frames are the checkpoints; K is the largest multiple of S whose resident
      segment buffer (gnca_bptt_ckpt_bytes) fits;
    * ("streaming_ckpt", S, segment bytes): the frames are the checkpoints of the streaming kernels, exactly
      record_rollout(..., checkpoint=True).
    Zero-padded graph shift models take the dense history or the streaming checkpoints here too.  ValueError names the
    smallest budget that works when nothing fits."""
    if impl not in ("auto", "resident", "streaming"):
        raise ValueError(f"bptt_plan: impl must be 'auto', 'resident' or 'streaming', got {impl!r}")
    if int(budget) < 0:
        raise ValueError(f"bptt_plan: budget must be >= 0, got {budget}")
    if every is not None and int(every) < 1:
        raise ValueError(f"bptt_plan: every must be >= 1, got {every}")
    if k is None:
        g = getattr(model, "graph", None) if getattr(model, "_is_graph", False) else None
        k = min(g.num_neighbors, len(g.offsets)) if g is not None else 0
    return _bptt_plan(model.model_desc(), int(B), int(H), int(W), int(T), int(budget), IMPL[impl], int(k),
                      every=None if every is None else int(every))


def _ckpt_fwd_raw(desc, packed, x0: torch.Tensor, sched: Schedule, every: int, resident: bool):
    """Checkpointing forward: (x_T, [T // every + 1, B, C, H, W] checkpoints), or None when the resident branch has no
    backward for this launch (nothing was launched)."""
    B, Cc, H, W = x0.shape
    lib = _lib.load()
    xT = torch.empty_like(x0)
    ckpt = torch.empty(sched.T // every + 1, B, Cc, H, W, dtype=torch.float32, device=x0.device)
    ws = GF._WS.get(x0.device, lib.gnca_rollout_workspace_bytes(C.byref(desc), B, H, W, sched.T))
    cs = sched.c_struct()
    if resident:
        rc = lib.gnca_rollout_fwd_bptt_ckpt(C.byref(desc), GF._ptr(packed), B, H, W, C.byref(cs), GF._ptr(x0),
                                            GF._ptr(xT), every, GF._ptr(ckpt), GF._ptr(ws), ws.numel(), GF._stream())
        if rc == _lib.GNCA_ERR_UNSUPPORTED:
            return None
        _lib.check(rc, "gnca_rollout_fwd_bptt_ckpt")
    else:
        _lib.check(lib.gnca_rollout_record(C.byref(desc), GF._ptr(packed), B, H, W, C.byref(cs), GF._ptr(x0),
                                           GF._ptr(xT), every, GF._ptr(ckpt), None, GF._ptr(ws), ws.numel(),
                                           IMPL["streaming"], GF._stream()), "gnca_rollout_record")
    return xT, ckpt


def _ckpt_bwd_raw(desc, packed, ckpt: torch.Tensor, sched: Schedule, every: int, resident: bool, gT: torch.Tensor,
                  gflat=None, g_frames=None, ckpt_every: Optional[int] = None):
    """Backward of _ckpt_fwd_raw: (dL/dx_0, flat parameter gradient), `gflat` accumulated into when given.  `ckpt` holds
    x_{f*every}; segments are `ckpt_every` steps long (default `every`; resident only: a multiple of it, starting at
    every (ckpt_every / every)-th frame).  `g_frames` (optional, the shape of `ckpt`): dL/dx_{f*every}, added at the
    frames' steps."""
    _, B, Cc, H, W = ckpt.shape
    ckpt_every = ckpt_every or every
    lib = _lib.load()
    gT = GF._require_cuda_f32(gT, "grad_output")
    g0 = torch.empty_like(ckpt[0])
    if gflat is None:
        gflat = torch.zeros(GF.param_layout(desc).total, dtype=torch.float32, device=ckpt.device)
    nseg = (lib.gnca_bptt_ckpt_bytes if resident else lib.gnca_ckpt_segment_bytes)(C.byref(desc), B, H, W, ckpt_every)
    segment = torch.empty(nseg, dtype=torch.uint8, device=ckpt.device)
    ws = GF._WS.get(ckpt.device, lib.gnca_rollout_workspace_bytes(C.byref(desc), B, H, W, sched.T))
    cs = sched.c_struct()
    if resident:
        _lib.check(lib.gnca_rollout_bwd_bptt_ckpt_frames(C.byref(desc), GF._ptr(packed), B, H, W, C.byref(cs),
                                                         GF._ptr(ckpt), every, ckpt_every, GF._ptr(g_frames),
                                                         GF._ptr(gT), GF._ptr(g0), GF._ptr(gflat), GF._ptr(segment),
                                                         segment.numel(), GF._ptr(ws), ws.numel(), GF._stream()),
                   "gnca_rollout_bwd_bptt_ckpt_frames")
    else:
        _lib.check(lib.gnca_rollout_bwd_ckpt(C.byref(desc), GF._ptr(packed), B, H, W, C.byref(cs), GF._ptr(ckpt), every,
                                             GF._ptr(g_frames), GF._ptr(gT), GF._ptr(g0), GF._ptr(gflat),
                                             GF._ptr(segment), segment.numel(), GF._ptr(ws), ws.numel(), GF._stream()),
                   "gnca_rollout_bwd_ckpt")
    return g0, gflat


def _budget_fwd_raw(desc, packed, x0: torch.Tensor, sched: Schedule, impl: int, budget: int, keep_u: bool,
                    every: int = 0):
    """The forward of the path bptt_plan picks: (x_T, History, plan).  `every > 0`: the plan of record_rollout, and the
    History carries the frames x_{f*every} (on the checkpoint paths they are the checkpoints)."""
    B, Cc, H, W = x0.shape
    resident_ok = True
    while True:
        plan = _bptt_plan(desc, B, H, W, sched.T, budget, impl, sched.k, resident_ok, every or None)
        path, K, _ = plan
        if path == "records":
            out = _records_fwd_raw(desc, packed, x0, sched, every, keep_x=False)
            if out is not None:
                return out[0], out[1], plan
        elif path == "dense":
            # never the record attempt of rollout_fwd_raw: the plan chose the dense history because the records do not
            # fit or have no backward for this launch, and their buffer alone could exceed the budget
            xT, hist = _dense_fwd_raw(desc, packed, x0, sched, True, impl, keep_u, every)
            return xT, hist, plan
        else:
            resident = path == "resident_ckpt"
            out = _ckpt_fwd_raw(desc, packed, x0, sched, every or K, resident)
            if out is not None:
                xT, ckpt = out
                return xT, History(None, shape=(sched.T + 1, B, Cc, H, W), ckpt=ckpt, every=every or K,
                                   resident=resident, frames=ckpt if every else None, ckpt_every=K), plan
        if impl == IMPL["resident"]:
            raise ValueError(f"{'record_rollout' if every else 'rollout'}: impl='resident' with bptt_budget, but the "
                             "resident backward has no launch configuration for this batch "
                             f"(B={B}, {H}x{W}, k={sched.k})")
        resident_ok = False              # the resident backward does not take this launch: plan without it


def _records_fwd_raw(desc, packed, x0: torch.Tensor, sched: Schedule, every: int, keep_x: bool):
    """Resident BPTT forward with records: (x_T, History), or None when the configuration has no record path.  Zero-padded
    graph shift models keep the buffer of gnca_bptt_zp_bytes instead (History.zp)."""
    B, Cc, H, W = x0.shape
    lib = _lib.load()
    T = sched.T
    nb = _record_bytes(lib, desc, B, H, W, T)
    zp = nb == 0 and sched.k <= RESIDENT_MAX_K
    if zp:
        nb = _record_bytes(lib, desc, B, H, W, T, lib.gnca_bptt_zp_bytes)
    if nb == 0:
        return None
    xT = torch.empty_like(x0)
    ws = GF._WS.get(x0.device, lib.gnca_rollout_workspace_bytes(C.byref(desc), B, H, W, T))
    cs = sched.c_struct()
    bptt = torch.empty(nb, dtype=torch.uint8, device=x0.device)
    if zp:
        # one call for both: the frames (or the full history, every = 1) are copies of the x_t the buffer keeps
        hist = torch.empty(T + 1, B, Cc, H, W, dtype=torch.float32, device=x0.device) if keep_x and every <= 0 else None
        frames = torch.empty(T // every + 1, B, Cc, H, W, dtype=torch.float32, device=x0.device) if every > 0 else None
        out = frames if every > 0 else hist
        rc = lib.gnca_rollout_fwd_bptt_zp(C.byref(desc), GF._ptr(packed), B, H, W, C.byref(cs), GF._ptr(x0),
                                          GF._ptr(xT), every if every > 0 else 1, GF._ptr(out), GF._ptr(bptt), nb,
                                          GF._ptr(ws), ws.numel(), GF._stream())
        if rc == _lib.GNCA_ERR_UNSUPPORTED:
            return None
        _lib.check(rc, "gnca_rollout_fwd_bptt_zp")
        return xT, History(hist, bptt=bptt, shape=(T + 1, B, Cc, H, W), frames=frames, zp=True)
    if every > 0:
        hist = None
        frames = torch.empty(T // every + 1, B, Cc, H, W, dtype=torch.float32, device=x0.device)
        rc = lib.gnca_rollout_fwd_bptt_record(C.byref(desc), GF._ptr(packed), B, H, W, C.byref(cs), GF._ptr(x0),
                                              GF._ptr(xT), every, GF._ptr(frames), GF._ptr(bptt), nb,
                                              GF._ptr(ws), ws.numel(), GF._stream())
    else:
        frames = None
        hist = torch.empty(T + 1, B, Cc, H, W, dtype=torch.float32, device=x0.device) if keep_x else None
        rc = lib.gnca_rollout_fwd_bptt(C.byref(desc), GF._ptr(packed), B, H, W, C.byref(cs), GF._ptr(x0),
                                       GF._ptr(xT), GF._ptr(hist), GF._ptr(bptt), nb, GF._ptr(ws), ws.numel(),
                                       GF._stream())
    if rc == _lib.GNCA_ERR_UNSUPPORTED:
        return None
    _lib.check(rc, "gnca_rollout_fwd_bptt_record" if every > 0 else "gnca_rollout_fwd_bptt")
    return xT, History(hist, bptt=bptt, shape=(T + 1, B, Cc, H, W), frames=frames)


def rollout_fwd_raw(desc, packed, x0: torch.Tensor, sched: Schedule, *, history: bool, impl: int = 0,
                    keep_u: bool = True, keep_x: bool = True, every: int = 0, bptt_budget: Optional[int] = None):
    """gnca_rollout_fwd without autograd: returns (x_T, History or None).  `keep_x=False`: the caller only needs the
    history for the backward (the resident BPTT path then skips storing x_t).  `every > 0` (with `history`): the
    History also carries the frames x_{f*every} of `record_rollout` -- on the record path the forward writes them in
    place of the x_t history (gnca_rollout_fwd_bptt_record), on the dense path they are copied out of it.
    `bptt_budget` (with `history`, without `keep_x`): the history takes at most that many bytes, on the path bptt_plan
    picks (History.plan; with `every`, the plan of bptt_plan(..., every=every), whose checkpoints are the frames); None
    is exactly the call without it."""
    x0 = GF._require_cuda_f32(x0, "x0")
    B, Cc, H, W = x0.shape
    if Cc != desc.C:
        raise ValueError(f"x0 has {Cc} channels, model has {desc.C}")
    if bptt_budget is not None and history:
        xT, hist, plan = _budget_fwd_raw(desc, packed, x0, sched, impl, int(bptt_budget), keep_u, every)
        hist.plan = plan
        return xT, hist
    if history and impl in (0, 2) and sched.T > 0:
        out = _records_fwd_raw(desc, packed, x0, sched, every, keep_x)
        if out is not None:
            return out
    return _dense_fwd_raw(desc, packed, x0, sched, history, impl, keep_u, every)


def _dense_fwd_raw(desc, packed, x0: torch.Tensor, sched: Schedule, history: bool, impl: int, keep_u: bool,
                   every: int):
    """gnca_rollout_fwd with the dense x_t / u_t history (or none): the path of rollout_fwd_raw without records."""
    B, Cc, H, W = x0.shape
    lib = _lib.load()
    T = sched.T
    xT = torch.empty_like(x0)
    nbytes = lib.gnca_rollout_workspace_bytes(C.byref(desc), B, H, W, T)
    ws = GF._WS.get(x0.device, nbytes)
    cs = sched.c_struct()
    hist = uh = sh = None
    if history:
        Tq = _dense_steps(T, B * Cc * H * W)   # same quantised allocation for the dense history (prefix views)
        hist = torch.empty(Tq + 1, B, Cc, H, W, dtype=torch.float32, device=x0.device)[:T + 1]
        if keep_u and T > 0:
            uh = torch.empty(Tq, B, Cc, H, W, dtype=torch.float32, device=x0.device)[:T]
            sh = torch.empty(Tq, B, 2, dtype=torch.float32, device=x0.device)[:T]
    _lib.check(lib.gnca_rollout_fwd(C.byref(desc), GF._ptr(packed), B, H, W, C.byref(cs), GF._ptr(x0), GF._ptr(xT),
                                    GF._ptr(hist), GF._ptr(sh), GF._ptr(uh), GF._ptr(ws), ws.numel(), int(impl),
                                    GF._stream()), "gnca_rollout_fwd")
    if not history:
        return xT, None
    # the frames are a copy: editing them in place cannot corrupt the history the backward reads
    return xT, History(hist, uh, sh, frames=hist[::every].clone() if every > 0 else None)


def rollout_bwd_raw(desc, packed, hist, sched: Schedule, gT: torch.Tensor, *, gflat=None, impl: int = 0,
                    g_frames: Optional[torch.Tensor] = None, every: int = 0):
    """gnca_rollout_bwd without autograd: returns (dL/dx_0, flat parameter gradient in canonical layout).
    `gflat` (optional) is accumulated into.  `g_frames` (optional, [T // every + 1, B, C, H, W]): dL/dx_{f*every} of the
    frames of the forward, added at their steps (gnca_rollout_bwd_frames / gnca_rollout_bwd_bptt_frames)."""
    if not isinstance(hist, History):
        hist = History(hist)
    if hist.ckpt is not None:
        if g_frames is not None:
            g_frames = GF._require_cuda_f32(g_frames, "frame gradients")
            if g_frames.shape != hist.ckpt.shape:
                raise ValueError(f"frame gradients have shape {tuple(g_frames.shape)}, expected "
                                 f"{tuple(hist.ckpt.shape)}")
        return _ckpt_bwd_raw(desc, packed, hist.ckpt, sched, hist.every, hist.resident, gT, gflat, g_frames,
                             hist.ckpt_every)
    _, B, Cc, H, W = hist.shape
    gT = GF._require_cuda_f32(gT, "grad_output")
    lib = _lib.load()
    g0 = torch.empty(B, Cc, H, W, dtype=torch.float32, device=gT.device)
    if gflat is None:
        lay = GF.param_layout(desc)
        gflat = torch.zeros(lay.total, dtype=torch.float32, device=gT.device)
    nbytes = lib.gnca_rollout_workspace_bytes(C.byref(desc), B, H, W, sched.T)
    ws = GF._WS.get(gT.device, nbytes)
    cs = sched.c_struct()
    if g_frames is not None:
        g_frames = GF._require_cuda_f32(g_frames, "frame gradients")
        if tuple(g_frames.shape) != (sched.T // every + 1, B, Cc, H, W):
            raise ValueError(f"frame gradients have shape {tuple(g_frames.shape)}, expected "
                             f"{(sched.T // every + 1, B, Cc, H, W)}")
    if hist.bptt is not None and hist.zp:
        _lib.check(lib.gnca_rollout_bwd_bptt_zp(C.byref(desc), GF._ptr(packed), B, H, W, C.byref(cs), GF._ptr(hist.bptt),
                                                hist.bptt.numel(), every, GF._ptr(g_frames), GF._ptr(gT), GF._ptr(g0),
                                                GF._ptr(gflat), GF._ptr(ws), ws.numel(), GF._stream()),
                   "gnca_rollout_bwd_bptt_zp")
        return g0, gflat
    if hist.bptt is not None:
        _lib.check(lib.gnca_rollout_bwd_bptt_frames(C.byref(desc), GF._ptr(packed), B, H, W, C.byref(cs),
                                                    GF._ptr(hist.bptt), hist.bptt.numel(), every, GF._ptr(g_frames),
                                                    GF._ptr(gT), GF._ptr(g0), GF._ptr(gflat), GF._ptr(ws), ws.numel(),
                                                    GF._stream()), "gnca_rollout_bwd_bptt_frames")
        return g0, gflat
    _lib.check(lib.gnca_rollout_bwd_frames(C.byref(desc), GF._ptr(packed), B, H, W, C.byref(cs), GF._ptr(hist.x),
                                           GF._ptr(hist.stats), GF._ptr(hist.u), every, GF._ptr(g_frames), GF._ptr(gT),
                                           GF._ptr(g0), GF._ptr(gflat), GF._ptr(ws), ws.numel(), int(impl),
                                           GF._stream()), "gnca_rollout_bwd_frames")
    return g0, gflat


def _model_stack(models, x0: Optional[torch.Tensor], what: str, impl: str):
    """(desc, models as a list, M) of a list of same-architecture models: the model-stacked calls of rollout /
    record_rollout / monitor_rollout.  ValueError, before any launch, for an empty list, models that differ in their
    descriptor, graph offsets or neighbour count, or device, models on another device than x0, a batch that is not a
    multiple of M, and impl='streaming' (the streaming kernels stage weights per tile, not per sample).  x0=None checks
    the models only."""
    models = list(models)
    if not models:
        raise ValueError(f"{what}: the list of models is empty")
    if impl == "streaming":
        raise ValueError(f"{what}: a list of models runs on the cluster kernels only; impl='streaming' cannot take it")
    desc = models[0].model_desc()
    dev = next(models[0].parameters()).device
    g0 = getattr(models[0], "graph", None) if getattr(models[0], "_is_graph", False) else None
    for i, m in enumerate(models[1:], 1):
        d = m.model_desc()
        for name, _ in desc._fields_:
            if getattr(d, name) != getattr(desc, name):
                raise ValueError(f"{what}: model {i} differs from model 0 in {name} ({getattr(d, name)} vs "
                                 f"{getattr(desc, name)}); a stack shares one architecture")
        g = getattr(m, "graph", None) if getattr(m, "_is_graph", False) else None
        if g0 is not None and (list(g.offsets) != list(g0.offsets) or g.num_neighbors != g0.num_neighbors):
            raise ValueError(f"{what}: model {i} differs from model 0 in graph.offsets or num_neighbors; a stack "
                             "shares one schedule")
        if next(m.parameters()).device != dev:
            raise ValueError(f"{what}: model {i} is on {next(m.parameters()).device}, model 0 on {dev}")
    M = len(models)
    if x0 is None:
        return desc, models, M
    if dev != x0.device:
        raise ValueError(f"{what}: the models are on {dev}, x0 on {x0.device}")
    if x0.dim() != 4 or x0.shape[0] % M != 0:
        raise ValueError(f"{what}: x0 must be [M*B, C, H, W] with the batch a multiple of the {M} models, got "
                         f"{list(x0.shape)}")
    return desc, models, M


def _stack_packed(models) -> torch.Tensor:
    """[M, packed_total]: the cached packed_weights() of every model, one row each"""
    return torch.stack([m.packed_weights() for m in models])


def stack_bptt_bytes(desc, B: int, H: int, W: int, T: int, k: int = 0) -> Tuple[int, bool]:
    """(bytes, zp) of the record buffer `rollout(models, ...)` allocates for a stack on a B x C x H x W batch (B counts
    the samples of all models) over T steps with k offsets per step; zp: the zero-padded graph shift's buffer
    (gnca_bptt_zp_bytes), else gnca_bptt_bytes.  That is what the single-model call keeps for the same batch, but a
    stack has no dense streaming history to fall back to, so ValueError, naming the bytes, where the single-model call
    would take it: above BPTT_MAX_BYTES, or outside the resident BPTT's envelope."""
    lib = _lib.load()
    zp = bool(desc.flags & _lib.GNCA_F_GRAPH) and not (desc.flags & _lib.GNCA_F_TORUS)
    nbytes = lib.gnca_bptt_zp_bytes if zp else lib.gnca_bptt_bytes
    nb = nbytes(C.byref(desc), B, H, W, T) if k <= RESIDENT_MAX_K else 0
    if nb == 0:
        raise ValueError(f"rollout: a list of models trains on the resident BPTT only, which this model / shape does not "
                         f"have (16 channels, hidden 128, H*W <= 2048, W % 4 == 0, at most {RESIDENT_MAX_K} offsets per "
                         f"step, d_model <= 32 for the zero-padded shift); got B={B}, {H}x{W}, k={k}")
    if nb > BPTT_MAX_BYTES:
        raise ValueError(f"rollout: the records of this stack take {nb} bytes (B={B}, {H}x{W}, T={T}), more than "
                         f"BPTT_MAX_BYTES = {BPTT_MAX_BYTES}; a stack has no streaming backward to fall back to, so "
                         "train fewer models, samples or steps per call")
    return _record_bytes(lib, desc, B, H, W, T, nbytes) or nb, zp


def rollout_models_fwd_raw(desc, packed: torch.Tensor, x0: torch.Tensor, sched: Schedule):
    """Resident BPTT forward of a stack (gnca_rollout_fwd_bptt_models, or its _zp form) without autograd: (x_T, History).
    packed: [M, packed_total]; x0: [M*B, C, H, W], model-major."""
    x0 = GF._require_cuda_f32(x0, "x0")
    B, Cc, H, W = x0.shape
    if Cc != desc.C:
        raise ValueError(f"x0 has {Cc} channels, model has {desc.C}")
    M, T = packed.shape[0], sched.T
    nb, zp = stack_bptt_bytes(desc, B, H, W, T, sched.k)           # errors before any allocation or launch
    lib = _lib.load()
    xT = torch.empty_like(x0)
    ws = GF._WS.get(x0.device, lib.gnca_rollout_workspace_models_bytes(C.byref(desc), M, B, H, W, T))
    bptt = torch.empty(nb, dtype=torch.uint8, device=x0.device)
    name = "gnca_rollout_fwd_bptt_zp_models" if zp else "gnca_rollout_fwd_bptt_models"
    _lib.check(getattr(lib, name)(C.byref(desc), GF._ptr(packed), M, B, H, W, C.byref(sched.c_struct()), GF._ptr(x0),
                                  GF._ptr(xT), GF._ptr(bptt), nb, GF._ptr(ws), ws.numel(), GF._stream()), name)
    return xT, History(None, bptt=bptt, shape=(T + 1, B, Cc, H, W), zp=zp)


def rollout_models_bwd_raw(desc, packed: torch.Tensor, hist: History, sched: Schedule, gT: torch.Tensor):
    """Backward of rollout_models_fwd_raw: (dL/dx_0, [M, param_total] parameter gradients, row i model i's)."""
    M = packed.shape[0]
    _, B, Cc, H, W = hist.shape
    gT = GF._require_cuda_f32(gT, "grad_output")
    lib = _lib.load()
    g0 = torch.empty(B, Cc, H, W, dtype=torch.float32, device=gT.device)
    gflat = torch.zeros(M, GF.param_layout(desc).total, dtype=torch.float32, device=gT.device)
    ws = GF._WS.get(gT.device, lib.gnca_rollout_workspace_models_bytes(C.byref(desc), M, B, H, W, sched.T))
    name = "gnca_rollout_bwd_bptt_zp_models" if hist.zp else "gnca_rollout_bwd_bptt_models"
    _lib.check(getattr(lib, name)(C.byref(desc), GF._ptr(packed), M, B, H, W, C.byref(sched.c_struct()),
                                  GF._ptr(hist.bptt), hist.bptt.numel(), GF._ptr(gT), GF._ptr(g0), GF._ptr(gflat),
                                  GF._ptr(ws), ws.numel(), GF._stream()), name)
    return g0, gflat


class _RolloutFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x0, cfg, *params):
        xT, hist = rollout_fwd_raw(cfg["desc"], cfg["packed"], x0, cfg["schedule"],
                                   history=bool(cfg["need_grad"] or cfg["history"]), impl=cfg["impl"],
                                   keep_x=bool(cfg["history"]))
        ctx.cfg = cfg
        ctx.param_shapes = [p.shape for p in params]
        ctx.hist = hist
        if cfg["history"]:
            ctx.mark_non_differentiable(hist.x)
            return xT, hist.x
        return xT

    @staticmethod
    def backward(ctx, gT, *unused):
        cfg = ctx.cfg
        if ctx.hist is None:
            raise RuntimeError("rollout was run without gradient history")
        g0, gflat = rollout_bwd_raw(cfg["desc"], cfg["packed"], ctx.hist, cfg["schedule"], gT, impl=cfg["impl"])
        offs = GF.segment_offsets(cfg["desc"])
        grads = [gflat[offs[i]:offs[i + 1]].view(ctx.param_shapes[i]) for i in range(len(ctx.param_shapes))]
        ctx.hist = None
        return (g0, None, *grads)


class _CkptFn(torch.autograd.Function):
    """Checkpointed BPTT: the forward keeps x_{j*every} (gnca_rollout_record on the streaming kernels) and returns them
    with x_T; the backward recomputes one segment of `every` steps at a time from them (gnca_rollout_bwd_ckpt)."""

    @staticmethod
    def forward(ctx, x0, cfg, *params):
        x0 = GF._require_cuda_f32(x0, "x0")
        B, Cc, H, W = x0.shape
        desc, sched, every = cfg["desc"], cfg["schedule"], cfg["every"]
        if Cc != desc.C:
            raise ValueError(f"x0 has {Cc} channels, model has {desc.C}")
        lib = _lib.load()
        xT = torch.empty_like(x0)
        ckpt = torch.empty(sched.T // every + 1, B, Cc, H, W, dtype=torch.float32, device=x0.device)
        ws = GF._WS.get(x0.device, lib.gnca_rollout_workspace_bytes(C.byref(desc), B, H, W, sched.T))
        cs = sched.c_struct()
        _lib.check(lib.gnca_rollout_record(C.byref(desc), GF._ptr(cfg["packed"]), B, H, W, C.byref(cs), GF._ptr(x0),
                                           GF._ptr(xT), every, GF._ptr(ckpt), None, GF._ptr(ws), ws.numel(),
                                           IMPL["streaming"], GF._stream()), "gnca_rollout_record")
        ctx.set_materialize_grads(False)          # an unused output passes None: no zero tensor, no frame pass
        ctx.cfg = cfg
        ctx.param_shapes = [p.shape for p in params]
        ctx.consumed = False
        ctx.save_for_backward(ckpt)               # an in-place edit of a returned checkpoint makes the backward raise
        return ckpt, xT

    @staticmethod
    def backward(ctx, g_ckpt, g_xT):
        if ctx.consumed:
            raise RuntimeError("rollout: the checkpoints were already consumed by an earlier backward")
        (ckpt,) = ctx.saved_tensors
        cfg = ctx.cfg
        desc, sched, every = cfg["desc"], cfg["schedule"], cfg["every"]
        _, B, Cc, H, W = ckpt.shape
        lib = _lib.load()
        g_xT = torch.zeros_like(ckpt[0]) if g_xT is None else GF._require_cuda_f32(g_xT, "grad_output")
        if g_ckpt is not None:
            g_ckpt = GF._require_cuda_f32(g_ckpt, "frame gradients")
        g0 = torch.empty_like(ckpt[0])
        gflat = torch.zeros(GF.param_layout(desc).total, dtype=torch.float32, device=ckpt.device)
        segment = torch.empty(lib.gnca_ckpt_segment_bytes(C.byref(desc), B, H, W, every), dtype=torch.uint8,
                              device=ckpt.device)
        ws = GF._WS.get(ckpt.device, lib.gnca_rollout_workspace_bytes(C.byref(desc), B, H, W, sched.T))
        cs = sched.c_struct()
        _lib.check(lib.gnca_rollout_bwd_ckpt(C.byref(desc), GF._ptr(cfg["packed"]), B, H, W, C.byref(cs),
                                             GF._ptr(ckpt), every, GF._ptr(g_ckpt), GF._ptr(g_xT), GF._ptr(g0),
                                             GF._ptr(gflat), GF._ptr(segment), segment.numel(), GF._ptr(ws),
                                             ws.numel(), GF._stream()), "gnca_rollout_bwd_ckpt")
        ctx.consumed = True
        offs = GF.segment_offsets(desc)
        grads = [gflat[offs[i]:offs[i + 1]].view(ctx.param_shapes[i]) for i in range(len(ctx.param_shapes))]
        return (g0, None, *grads)


class _BudgetFn(torch.autograd.Function):
    """rollout(..., bptt_budget=...): the forward keeps the history bptt_plan picks, the backward consumes it once.
    Checkpoints are kept with save_for_backward, so an in-place edit of them makes the backward raise."""

    @staticmethod
    def forward(ctx, x0, cfg, *params):
        xT, hist = rollout_fwd_raw(cfg["desc"], cfg["packed"], x0, cfg["schedule"], history=True, impl=cfg["impl"],
                                   keep_x=False, bptt_budget=cfg["budget"])
        ctx.cfg = cfg
        ctx.param_shapes = [p.shape for p in params]
        cfg["plan"] = hist.plan
        ctx.has_ckpt = hist.ckpt is not None
        if ctx.has_ckpt:
            ctx.save_for_backward(hist.ckpt)
            hist.ckpt = None
        ctx.hist = hist
        return xT

    @staticmethod
    def backward(ctx, gT):
        cfg = ctx.cfg
        if ctx.hist is None:
            raise RuntimeError("rollout: the BPTT history was already consumed by an earlier backward")
        hist = ctx.hist
        if ctx.has_ckpt:
            (hist.ckpt,) = ctx.saved_tensors
        g0, gflat = rollout_bwd_raw(cfg["desc"], cfg["packed"], hist, cfg["schedule"], gT, impl=cfg["impl"])
        ctx.hist = None
        offs = GF.segment_offsets(cfg["desc"])
        grads = [gflat[offs[i]:offs[i + 1]].view(ctx.param_shapes[i]) for i in range(len(ctx.param_shapes))]
        return (g0, None, *grads)


class _RolloutModelsFn(torch.autograd.Function):
    """rollout(models, ...): one node over the stack; params are every model's canonical parameters, model-major."""

    @staticmethod
    def forward(ctx, x0, cfg, *params):
        xT, hist = rollout_models_fwd_raw(cfg["desc"], cfg["packed"], x0, cfg["schedule"])
        ctx.cfg, ctx.hist = cfg, hist
        ctx.param_shapes = [p.shape for p in params]
        return xT

    @staticmethod
    def backward(ctx, gT):
        cfg = ctx.cfg
        if ctx.hist is None:
            raise RuntimeError("rollout: the BPTT history was already consumed by an earlier backward")
        g0, gflat = rollout_models_bwd_raw(cfg["desc"], cfg["packed"], ctx.hist, cfg["schedule"], gT)
        ctx.hist = None
        offs = GF.segment_offsets(cfg["desc"])
        n = len(offs) - 1
        grads = [gflat[j // n, offs[j % n]:offs[j % n + 1]].view(s) for j, s in enumerate(ctx.param_shapes)]
        return (g0, None, *grads)


def _check_checkpoint_impl(impl: str, what: str) -> None:
    if impl in ("resident", "banded"):
        raise ValueError(f"{what}: checkpoints are recomputed with the streaming kernels, so impl={impl!r} cannot "
                         "produce them; use impl='auto' or 'streaming'")


IMPL = {"auto": 0, "streaming": 1, "resident": 2, "banded": 3}


def rollout(model, x0: torch.Tensor, schedule: Schedule, *, checkpoint_every: Optional[int] = None,
            return_history: bool = False, impl: str = "auto", bptt_budget: Optional[int] = None):
    """x_T (and optionally the [T+1,B,C,H,W] history) of T steps from x0 under `schedule`.  Differentiable
    w.r.t. x0 and the model parameters (BPTT stores x_t only and recomputes the rest).

    `checkpoint_every=K` (with grad): the forward keeps only x_{jK} and the backward recomputes each K-step segment
    from its checkpoint on the streaming kernels, so BPTT memory is T/K + 1 states plus one segment instead of the
    2T + 1 states of the dense history.  The gradients equal those of the dense streaming BPTT.  Without grad it
    changes nothing.

    `bptt_budget=N` (bytes, with grad): the BPTT history takes at most N bytes; `bptt_plan` picks the path.  The
    history `rollout()` keeps without a budget is kept unchanged when it fits (bit-identical results); else the
    resident BPTT recomputes segments from checkpoints x_{jK} (same dL/dx_0 as the unsegmented resident BPTT), else
    the streaming kernels do (`checkpoint_every`), each with the largest K that fits.  ValueError when nothing fits.
    `impl="resident"` / `"streaming"` restrict the choice to that backward.

    `model` may be a list of M models of one architecture (same `model_desc()`, graph offsets and neighbour count, one
    device), e.g. the seeds or learning rates of a sweep.  x0 is [M*B, C, H, W], model-major: model i runs samples
    [i*B, (i+1)*B) and x_T keeps that layout.  Build the schedule with `make_schedule(models[0], M*B, ...)`, so that every
    model sees the same offsets, fire draws and damage.  With grad, the M models train in one resident BPTT
    (gnca_rollout_fwd_bptt_models / gnca_rollout_bwd_bptt_models, or their _zp forms): one autograd node whose backward
    gives dL/dx0 and each model's parameter gradients, so `loss.backward()` fills every model's `.grad`.  Model i's
    gradients come from its own samples only.  Without grad it returns x_T, bit-equal to `record_rollout(models,
    ...).x_T`.  The stack keeps the records the single-model call keeps for an M*B batch (T*M*B*H*W*1.4 KB at worst,
    `stack_bptt_bytes`), but has no streaming backward to fall back to: where the single-model call would take the dense
    history (more than BPTT_MAX_BYTES of records, or a model / shape outside the resident BPTT) it raises ValueError
    naming the bytes, before any launch.  `checkpoint_every`, `bptt_budget`, `return_history`, impl='streaming' or
    'banded', and a batch that is not a multiple of M raise ValueError before any launch."""
    if isinstance(model, (list, tuple)):
        for name, on in (("checkpoint_every", checkpoint_every is not None), ("bptt_budget", bptt_budget is not None),
                         ("return_history=True", return_history)):
            if on:
                raise ValueError(f"rollout: {name} does not take a list of models (a stack trains on the resident "
                                 "BPTT only)")
        if impl == "banded":
            raise ValueError("rollout: a list of models trains on the replicated-state kernels; impl='banded' cannot "
                             "take it")
        desc, models, M = _model_stack(model, x0, "rollout", impl)
        if not x0.is_cuda:
            raise RuntimeError(f"rollout: x0 is on {x0.device}; CUDA (sm_100a) only, no CPU fallback")
        ps = [p for m in models for p in m.canonical_params()]
        if not (torch.is_grad_enabled() and (x0.requires_grad or any(p.requires_grad for p in ps))):
            return record_rollout(models, x0, schedule, every=max(schedule.T, 1), impl=impl).x_T
        cfg = {"desc": desc, "packed": _stack_packed(models), "schedule": schedule}
        return _RolloutModelsFn.apply(x0, cfg, *ps)
    if bptt_budget is not None:
        if int(bptt_budget) < 0:
            raise ValueError(f"rollout: bptt_budget must be >= 0 bytes, got {bptt_budget}")
        if checkpoint_every is not None or return_history:
            raise ValueError("rollout: bptt_budget chooses the history itself; it cannot be combined with "
                             "checkpoint_every or return_history")
        if impl not in ("auto", "resident", "streaming"):
            raise ValueError(f"rollout: bptt_budget needs impl 'auto', 'resident' or 'streaming', got {impl!r}")
    if checkpoint_every is not None:
        if int(checkpoint_every) < 1:
            raise ValueError(f"rollout: checkpoint_every must be >= 1, got {checkpoint_every}")
        if return_history:
            raise ValueError("rollout: return_history=True keeps every state; it cannot be combined with checkpoint_every")
        _check_checkpoint_impl(impl, "rollout")
    if not x0.is_cuda:
        raise RuntimeError(f"rollout: x0 is on {x0.device}; CUDA (sm_100a) only, no CPU fallback")
    ps = model.canonical_params()
    need_grad = torch.is_grad_enabled() and (x0.requires_grad or any(p.requires_grad for p in ps))
    if not need_grad and not return_history:        # inference: no autograd node, no history (same C call underneath)
        return rollout_fwd_raw(model.model_desc(), model.packed_weights(), x0, schedule, history=False, impl=IMPL[impl])[0]
    if checkpoint_every is not None:
        cfg = {"desc": model.model_desc(), "packed": model.packed_weights(), "schedule": schedule,
               "every": int(checkpoint_every)}
        return _CkptFn.apply(x0, cfg, *ps)[1]
    if bptt_budget is not None:
        desc = model.model_desc()
        B, _, H, W = x0.shape
        _bptt_plan(desc, B, H, W, schedule.T, int(bptt_budget), IMPL[impl], schedule.k)   # errors before any launch
        cfg = {"desc": desc, "packed": model.packed_weights(), "schedule": schedule, "impl": IMPL[impl],
               "budget": int(bptt_budget)}
        return _BudgetFn.apply(x0, cfg, *ps)
    cfg = {"desc": model.model_desc(), "packed": model.packed_weights(), "schedule": schedule, "need_grad": need_grad,
           "history": bool(return_history), "impl": IMPL[impl]}
    return _RolloutFn.apply(x0, cfg, *ps)


class _RecordFn(torch.autograd.Function):
    """record_rollout(..., differentiable=True): the frames and x_T as the outputs of one node; its backward is one
    BPTT that adds dL/dframe_f at step f * every.  With cfg["budget"] the history is the one bptt_plan(..., every=every)
    picks (ctx.plan); frames that are checkpoints are kept with save_for_backward, so editing one in place makes the
    backward raise."""

    @staticmethod
    def forward(ctx, x0, cfg, *params):
        xT, hist = rollout_fwd_raw(cfg["desc"], cfg["packed"], x0, cfg["schedule"], history=True, impl=cfg["impl"],
                                   keep_x=False, every=cfg["every"], bptt_budget=cfg.get("budget"))
        ctx.set_materialize_grads(False)          # an unused output passes None: no zero tensor, no frame pass
        ctx.cfg = cfg
        ctx.param_shapes = [p.shape for p in params]
        ctx.plan = hist.plan
        frames = hist.frames
        ctx.has_ckpt = hist.ckpt is not None
        if ctx.has_ckpt:
            ctx.save_for_backward(frames)
            hist.ckpt = hist.frames = None
        ctx.hist = hist
        return frames, xT

    @staticmethod
    def backward(ctx, g_states, g_xT):
        cfg = ctx.cfg
        if ctx.hist is None:
            raise RuntimeError("record_rollout: the gradient history was already consumed by an earlier backward")
        hist = ctx.hist
        if ctx.has_ckpt:
            (hist.ckpt,) = ctx.saved_tensors
        if g_xT is None:
            g_xT = torch.zeros_like(hist.ckpt[0] if ctx.has_ckpt else hist.frames[0])
        g0, gflat = rollout_bwd_raw(cfg["desc"], cfg["packed"], hist, cfg["schedule"], g_xT, impl=cfg["impl"],
                                    g_frames=g_states, every=cfg["every"])
        offs = GF.segment_offsets(cfg["desc"])
        grads = [gflat[offs[i]:offs[i + 1]].view(ctx.param_shapes[i]) for i in range(len(ctx.param_shapes))]
        ctx.hist = None
        return (g0, None, *grads)


@dataclass
class Trajectory:
    """What `record_rollout` returns.  `states[f]` is x_{t[f]}, the state step t[f] consumes (after the schedule's
    damage at `damage_step`); `attention[f]` is the attention map of step t[f] for every step t[f] < T (None when not
    asked for); `x_T` is the final state, also when T is not a multiple of the stride."""
    t: List[int]                            # recorded step indices 0, S, 2S, ... <= T
    states: torch.Tensor                    # [F,B,C,H,W], F = T // S + 1
    attention: Optional[torch.Tensor]       # [FA,B,H,W], FA = ceil(T / S)
    x_T: torch.Tensor                       # [B,C,H,W]


def record_rollout(model, x0: torch.Tensor, schedule: Schedule, *, every: int, attention: bool = False,
                   impl: str = "auto", differentiable: bool = False, checkpoint: bool = False,
                   bptt_budget: Optional[int] = None) -> Trajectory:
    """T steps from x0 under `schedule` in one library call (gnca_rollout_record), keeping x_t every `every` steps and,
    with `attention=True`, the attention map `model.step(x_t, ..., return_attention=True)` gives for each kept step
    t < T.  Watching a rollout this way keeps the fused rollout kernels; no gradient history or record buffer is
    allocated, and the outputs are detached.

    `differentiable=True` (with grad mode on and x0 or a parameter requiring grad): `states` and `x_T` are the outputs
    of one autograd node, and a loss on any of them back-propagates to x0 and the parameters through one fused BPTT --
    the gradients of T sequential `model.step` calls with the same schedule.  The BPTT history is the one `rollout()`
    keeps for its backward.  `attention` stays detached (it costs one more, inference-only rollout).  Without grad the
    call is exactly the detached recording.

    `checkpoint=True` (with `differentiable=True`): the recorded frames are the only history.  The backward recomputes
    each `every`-step segment from its frame on the streaming kernels (rollout(..., checkpoint_every=every)), so memory
    is the frames plus one segment.  Editing a returned frame in place makes the backward raise.

    `bptt_budget=N` (bytes, with `differentiable=True`): what the BPTT keeps beyond the returned frames and x_T takes at
    most N bytes, on the path `bptt_plan(..., every=every)` picks.  The history the call keeps without a budget is kept
    when it fits (bit-identical results); else the frames are the checkpoints of the resident BPTT, which recomputes
    segments of the largest multiple of `every` steps whose buffer fits (dL/dx_0 bit-equal to the unbudgeted resident
    path, parameter gradients up to the summation order); else those of the streaming kernels, exactly
    `checkpoint=True`.  ValueError names the smallest budget that works when nothing fits.  Zero-padded graph shift
    models keep the dense history when it fits and otherwise take the streaming checkpoints, as in
    rollout(..., bptt_budget=N).  `impl="resident"` / `"streaming"` restrict the choice to that backward.  Frames that
    are checkpoints make the backward raise when edited in place.  Without grad the call is the detached recording.

    `model` may be a list of M models of one architecture (same `model_desc()`, graph offsets and neighbour count, one
    device), e.g. the saved checkpoints of a training run: one launch runs them side by side (gnca_rollout_record_models),
    each sample's cluster with its own model's weights.  x0 is [M*B, C, H, W], model-major, and the outputs keep their
    fields with the sample axis M*B long: model i's frames are `states[:, i*B:(i+1)*B]`, its final states
    `x_T[i*B:(i+1)*B]`.  Build the schedule with `make_schedule(models[0], M*B, ...)`: every model then sees the same
    offsets, fire draws and damage, which is the controlled experiment a checkpoint comparison wants.  Inference only, on
    the cluster kernels: `differentiable`, `attention`, `checkpoint`, `bptt_budget` and impl='streaming' raise
    ValueError, and a shape neither cluster kernel takes raises the library's RuntimeError."""
    every = int(every)
    if every < 1:
        raise ValueError(f"record_rollout: every must be >= 1, got {every}")
    stack = isinstance(model, (list, tuple))
    if stack:
        for name, on in (("differentiable=True", differentiable), ("attention=True", attention),
                         ("checkpoint=True", checkpoint), ("bptt_budget", bptt_budget is not None)):
            if on:
                raise ValueError(f"record_rollout: {name} does not take a list of models (the stacked call is "
                                 "inference only)")
        desc, models, M = _model_stack(model, x0, "record_rollout", impl)
    if bptt_budget is not None:
        if checkpoint:
            raise ValueError("record_rollout: bptt_budget chooses the history itself; it cannot be combined with "
                             "checkpoint=True")
        if not differentiable:
            raise ValueError("record_rollout: bptt_budget needs differentiable=True")
        if impl not in ("auto", "resident", "streaming"):
            raise ValueError(f"record_rollout: bptt_budget needs impl 'auto', 'resident' or 'streaming', got {impl!r}")
        if int(bptt_budget) < 0:
            raise ValueError(f"record_rollout: bptt_budget must be >= 0 bytes, got {bptt_budget}")
    if checkpoint:
        if not differentiable:
            raise ValueError("record_rollout: checkpoint=True needs differentiable=True")
        _check_checkpoint_impl(impl, "record_rollout")
    if attention and not getattr(model, "_is_graph", False):
        raise ValueError("record_rollout: attention maps need a graph model (NeuralCAGraph)")
    if not x0.is_cuda:
        raise RuntimeError(f"record_rollout: x0 is on {x0.device}; CUDA (sm_100a) only, no CPU fallback")
    if not stack:
        desc = model.model_desc()
    if differentiable:
        ps = model.canonical_params()
        if torch.is_grad_enabled() and (x0.requires_grad or any(p.requires_grad for p in ps)):
            if x0.shape[1] != desc.C:
                raise ValueError(f"x0 has {x0.shape[1]} channels, model has {desc.C}")
            cfg = {"desc": desc, "packed": model.packed_weights(), "schedule": schedule, "impl": IMPL[impl],
                   "every": every}
            if bptt_budget is not None:
                B, _, H, W = x0.shape
                # errors before any launch
                _bptt_plan(desc, B, H, W, schedule.T, int(bptt_budget), IMPL[impl], schedule.k, every=every)
                cfg["budget"] = int(bptt_budget)
            frames, xT = (_CkptFn if checkpoint else _RecordFn).apply(x0, cfg, *ps)
            attn = None
            if attention:
                with torch.no_grad():
                    attn = record_rollout(model, x0, schedule, every=every, attention=True, impl=impl).attention
            return Trajectory(t=list(range(0, schedule.T + 1, every)), states=frames, attention=attn, x_T=xT)
    x0 = GF._require_cuda_f32(x0.detach(), "x0")
    B, Cc, H, W = x0.shape
    if Cc != desc.C:
        raise ValueError(f"x0 has {Cc} channels, model has {desc.C}")
    lib = _lib.load()
    T = schedule.T
    F = lib.gnca_record_frames(T, every)
    if F < 0:
        _lib.check(F, "gnca_record_frames")
    FA = -(-T // every)
    xT = torch.empty_like(x0)
    frames = torch.empty(F, B, Cc, H, W, dtype=torch.float32, device=x0.device)
    attn = torch.empty(FA, B, H, W, dtype=torch.float32, device=x0.device) if attention else None
    ws = GF._WS.get(x0.device, lib.gnca_rollout_workspace_bytes(C.byref(desc), B, H, W, T))
    cs = schedule.c_struct()
    if stack:
        _lib.check(lib.gnca_rollout_record_models(C.byref(desc), GF._ptr(_stack_packed(models)), M, B, H, W,
                                                  C.byref(cs), GF._ptr(x0), GF._ptr(xT), every, GF._ptr(frames),
                                                  GF._ptr(ws), ws.numel(), IMPL[impl], GF._stream()),
                   "gnca_rollout_record_models")
        return Trajectory(t=list(range(0, T + 1, every)), states=frames, attention=None, x_T=xT)
    _lib.check(lib.gnca_rollout_record(C.byref(desc), GF._ptr(model.packed_weights()), B, H, W, C.byref(cs),
                                       GF._ptr(x0), GF._ptr(xT), every, GF._ptr(frames), GF._ptr(attn), GF._ptr(ws),
                                       ws.numel(), IMPL[impl], GF._stream()), "gnca_rollout_record")
    return Trajectory(t=list(range(0, T + 1, every)), states=frames, attention=attn, x_T=xT)


@dataclass
class Monitor:
    """What `monitor_rollout` returns.  Row f of every [F,B] tensor is frame f of `record_rollout(..., every=S)`:
    x_{t[f]}, after the schedule's damage at `damage_step`, frozen for a sample with steps[b] <= t[f].

    "The target" of a column is the call's [4,H,W] target, or, for a stack of M models given a [M,4,H,W] target,
    target[i] for model i's columns i*B:(i+1)*B (B samples per model)."""
    t: List[int]                            # step indices 0, S, 2S, ... <= T
    loss: torch.Tensor                      # [F,B] f32: premultiplied-RGBA MSE against the column's target
    psnr: torch.Tensor                      # [F,B] f32: utils.metrics.psnr_rgb against the column's target
    pixel_perfect: torch.Tensor             # [F,B] f32: utils.metrics.pixel_perfect(frame, target, eps)
    alive: torch.Tensor                     # [F,B] int64: cells with alpha > model.alpha_thr (no dilation)
    x_T: torch.Tensor                       # [B,C,H,W]
    ssim: Optional[torch.Tensor] = None     # [F,B] f32: utils.metrics.ssim_rgb against the column's target
                                            # (monitor_rollout(..., ssim=True))


def monitor_rollout(model, x0: torch.Tensor, schedule: Schedule, target: torch.Tensor, *, every: int,
                    impl: str = "auto", eps: float = 0.05, ssim: bool = False) -> Monitor:
    """Quality curves of a rollout without its states: the T steps of `rollout()` (same `impl` and dispatch, the same
    x_T) in one library call (gnca_rollout_metrics), reducing every `every`-th state against `target` ([4,H,W]
    premultiplied RGBA on x0's device) where the kernel holds it.  Memory is F*B*24 bytes of results plus at most
    F*B*256 bytes of per-CTA partials, instead of the F*B*C*H*W*4 bytes of `record_rollout` frames.  Inference only: the outputs are
    detached and no BPTT buffer is allocated, whatever the grad mode.  PSNR is 10*log10(1 / mse) of the clipped RGB
    from the kernel's sum; a frame equal to the target gives +inf, as utils.metrics.psnr_rgb does.

    `model` may be a list of M models of one architecture, as in `record_rollout`: one launch
    (gnca_rollout_metrics_models), x0 [M*B, C, H, W] model-major, every [F, M*B] curve and x_T with the sample axis M*B
    long, model i's curves at `[:, i*B:(i+1)*B]`.  Build the schedule with `make_schedule(models[0], M*B, ...)` so that
    every model sees the same offsets, fire draws and damage.  impl='streaming' raises ValueError; a shape neither
    cluster kernel takes raises the library's RuntimeError.  With a list, `target` may also be [M, 4, H, W], one
    target per model (gnca_rollout_metrics_targets): model i's curves are measured against target[i], so a target
    sweep (one model trained per image) compares in one call.  A [4, H, W] target is shared by all M; any other count
    of targets raises ValueError.

    ssim=True adds `Monitor.ssim`, the SSIM of every frame against the target as `utils.metrics.ssim_rgb` defines it
    (skimage's structural_similarity on clip(premultiplied RGB, 0, 1), 7x7 uniform windows, data_range 1), computed
    where the kernel holds the frame (gnca_rollout_metrics_ssim[_models]).  The other curves and x_T are those of the
    call without it; H or W below 7 raises ValueError.  Picking the best epoch of a run is one such call over its
    checkpoints::

        mon = monitor_rollout(checkpoints, x0.repeat(M, 1, 1, 1), sched, target, every=10, ssim=True)
        best = int(mon.ssim[-1].view(M, B).mean(1).argmax())   # the epoch whose final frames score highest
    """
    every = int(every)
    if every < 1:
        raise ValueError(f"monitor_rollout: every must be >= 1, got {every}")
    eps = float(eps)
    if not eps >= 0.0:
        raise ValueError(f"monitor_rollout: eps must be >= 0, got {eps}")
    if impl not in IMPL:
        raise ValueError(f"monitor_rollout: impl must be one of {sorted(IMPL)}, got {impl!r}")
    stack = isinstance(model, (list, tuple))
    if stack:
        desc, models, M = _model_stack(model, x0, "monitor_rollout", impl)
    else:
        desc = model.model_desc()
    if x0.dim() != 4:
        raise ValueError(f"monitor_rollout: x0 must be [B, C, H, W], got {list(x0.shape)}")
    B, Cc, H, W = x0.shape
    if Cc != desc.C:
        raise ValueError(f"x0 has {Cc} channels, model has {desc.C}")
    if desc.C < 4:
        raise ValueError(f"monitor_rollout: the metrics read RGBA (channels 0-3); the model has {desc.C} channels")
    per_model = stack and target.dim() == 4
    if per_model and tuple(target.shape[1:]) == (4, H, W) and target.shape[0] != M:
        raise ValueError(f"monitor_rollout: {target.shape[0]} targets for {M} models; a per-model target is "
                         f"[{M}, 4, {H}, {W}]")
    if tuple(target.shape) != ((M, 4, H, W) if per_model else (4, H, W)):
        want = f"[4, {H}, {W}]" + (f" or [{M}, 4, {H}, {W}]" if stack else "")
        raise ValueError(f"monitor_rollout: target must be {want} (premultiplied RGBA), got {list(target.shape)}")
    if ssim and (H < 7 or W < 7):
        raise ValueError(f"monitor_rollout: SSIM needs a 7x7 window inside the grid, got H={H}, W={W}")
    x0 = GF._require_cuda_f32(x0.detach(), "x0")
    target = GF._require_cuda_f32(target.detach(), "target")
    if target.device != x0.device:
        raise ValueError(f"monitor_rollout: target is on {target.device}, x0 on {x0.device}")
    lib = _lib.load()
    T = schedule.T
    F = T // every + 1
    xT = torch.empty_like(x0)
    sums = torch.empty(F, B, 2, dtype=torch.float64, device=x0.device)
    counts = torch.empty(F, B, 2, dtype=torch.int32, device=x0.device)
    scratch_bytes = (lib.gnca_metrics_ssim_scratch_bytes if ssim else lib.gnca_metrics_scratch_bytes)
    scratch = torch.empty(scratch_bytes(C.byref(desc), B, H, W, T, every), dtype=torch.uint8, device=x0.device)
    ws = GF._WS.get(x0.device, lib.gnca_rollout_workspace_bytes(C.byref(desc), B, H, W, T))
    cs = schedule.c_struct()
    ss = torch.empty(F, B, dtype=torch.float64, device=x0.device) if ssim else None
    if per_model:
        _lib.check(lib.gnca_rollout_metrics_targets(
            C.byref(desc), GF._ptr(_stack_packed(models)), M, B, H, W, C.byref(cs), GF._ptr(x0), GF._ptr(xT), every,
            GF._ptr(target), eps, GF._ptr(sums), GF._ptr(counts), GF._ptr(ss), GF._ptr(scratch), scratch.numel(),
            GF._ptr(ws), ws.numel(), IMPL[impl], GF._stream()), "gnca_rollout_metrics_targets")
    elif ssim and stack:
        _lib.check(lib.gnca_rollout_metrics_ssim_models(
            C.byref(desc), GF._ptr(_stack_packed(models)), M, B, H, W, C.byref(cs), GF._ptr(x0), GF._ptr(xT), every,
            GF._ptr(target), eps, GF._ptr(sums), GF._ptr(counts), GF._ptr(ss), GF._ptr(scratch), scratch.numel(),
            GF._ptr(ws), ws.numel(), IMPL[impl], GF._stream()), "gnca_rollout_metrics_ssim_models")
    elif ssim:
        _lib.check(lib.gnca_rollout_metrics_ssim(
            C.byref(desc), GF._ptr(model.packed_weights()), B, H, W, C.byref(cs), GF._ptr(x0), GF._ptr(xT), every,
            GF._ptr(target), eps, GF._ptr(sums), GF._ptr(counts), GF._ptr(ss), GF._ptr(scratch), scratch.numel(),
            GF._ptr(ws), ws.numel(), IMPL[impl], GF._stream()), "gnca_rollout_metrics_ssim")
    elif stack:
        _lib.check(lib.gnca_rollout_metrics_models(C.byref(desc), GF._ptr(_stack_packed(models)), M, B, H, W,
                                                   C.byref(cs), GF._ptr(x0), GF._ptr(xT), every, GF._ptr(target), eps,
                                                   GF._ptr(sums), GF._ptr(counts), GF._ptr(scratch), scratch.numel(),
                                                   GF._ptr(ws), ws.numel(), IMPL[impl], GF._stream()),
                   "gnca_rollout_metrics_models")
    else:
        _lib.check(lib.gnca_rollout_metrics(C.byref(desc), GF._ptr(model.packed_weights()), B, H, W, C.byref(cs),
                                            GF._ptr(x0), GF._ptr(xT), every, GF._ptr(target), eps, GF._ptr(sums),
                                            GF._ptr(counts), GF._ptr(scratch), scratch.numel(), GF._ptr(ws),
                                            ws.numel(), IMPL[impl], GF._stream()), "gnca_rollout_metrics")
    HW = H * W
    return Monitor(t=list(range(0, T + 1, every)), loss=(sums[..., 0] / (4 * HW)).float(),
                   psnr=(10.0 * torch.log10(1.0 / (sums[..., 1] / (3 * HW)))).float(),
                   pixel_perfect=(counts[..., 0].double() / HW).float(), alive=counts[..., 1].long(), x_T=xT,
                   ssim=ss.float() if ssim else None)

"""One training iteration of the graph-NCA trainer (the loop body of train_graph_augmented_nca.py:289-391;
classic variant train_intermediate_loss.py:230-296) on the fused CUDA path.

RNG consumption follows SURVEY Appendix B call for call so that a seeded run draws the same pool indices, damage,
step counts, fire rates, offsets and fire masks as the reference loop.  Per iteration there is ONE host sync (the
per-sample step counts come back to size the schedule; the reference syncs three times per CA step).
"""
from __future__ import annotations

import random
from dataclasses import dataclass, field
from typing import Callable, Dict, Optional

import numpy as np
import torch

from .. import _lib
from .. import functional as GF
from ..rollout import Schedule, make_schedule, rollout_bwd_raw, rollout_fwd_raw
from ..utils.damage import sample_damage_mask
from ..utils.nca_init import trainer_seed
from .dp import Shard, worst_k_indices
from .optim import FusedNormalizedAdam
from .pool import SamplePool

import ctypes as C


@dataclass
class TrainConfig:
    """Knobs read by the reference trainer (configs/config.json `training`, `graph_augmentation`, `damage`)."""
    batch_size: int = 16
    pool_size: int = 1024
    nca_steps_min: int = 48
    nca_steps_max: int = 80
    long_rollout_prob: float = 0.4
    long_rollout_steps_min: int = 200
    long_rollout_steps_max: int = 400
    fire_rate_min: float = 0.5
    fire_rate_max: float = 0.9
    learning_rate: float = 2e-4
    weight_decay: float = 1e-5
    reset_worst_prob: float = 0.10
    random_reseed_prob: float = 0.05
    message_gain: float = 0.25
    message_rate: float = 0.2
    message_every: int = 3
    scheduler_step_size: int = 150
    scheduler_gamma: float = 0.85
    damage: Dict = field(default_factory=dict)
    fire: str = "torch"            # "torch": the reference's torch.rand stream; "philox": in-kernel RNG (fast)
    rollout_impl: str = "auto"
    # data-parallel pool: "replicated" = every rank holds the whole pool and draws the reference's global batch
    # (random.sample over all slots; needs an all-gather of the final states every step), "owner" = rank r owns
    # pool_size / world slots and draws its share of the batch from them (SURVEY 8e: no state traffic at all; the batch is
    # then stratified over the ranks -- same marginal law per slot, not the reference's joint law)
    pool_sharding: str = "replicated"
    # bytes the BPTT history of one iteration may take (rollout.bptt_plan picks the path and checkpoint stride);
    # None keeps the history rollout() keeps without a budget
    bptt_budget_bytes: Optional[int] = None

    @staticmethod
    def from_reference_config(cfg: dict) -> "TrainConfig":
        t, g = cfg["training"], cfg.get("graph_augmentation", {})
        sch = t.get("scheduler") or {}
        return TrainConfig(
            batch_size=int(t["batch_size"]), pool_size=int(t["pool_size"]), nca_steps_min=int(t["nca_steps_min"]),
            nca_steps_max=int(t["nca_steps_max"]), long_rollout_prob=float(t.get("long_rollout_prob", 0.25)),
            long_rollout_steps_min=int(t.get("long_rollout_steps_min", 200)),
            long_rollout_steps_max=int(t.get("long_rollout_steps_max", 400)),
            fire_rate_min=float(t.get("fire_rate_min", 0.5)), fire_rate_max=float(t.get("fire_rate_max", 1.0)),
            learning_rate=float(t["learning_rate"]), weight_decay=float(t["weight_decay"]),
            reset_worst_prob=float(t.get("reset_worst_prob", 0.10)),
            random_reseed_prob=float(t.get("random_reseed_prob", 0.05)),
            message_gain=float(g.get("message_gain", 0.5)), message_rate=float(g.get("message_rate", 1.0)),
            message_every=int(g.get("message_every", 1)), scheduler_step_size=int(sch.get("step_size", 50)),
            scheduler_gamma=float(sch.get("gamma", 0.7)), damage=dict(cfg.get("damage", {})),
            bptt_budget_bytes=None if t.get("bptt_budget_bytes") is None else int(t["bptt_budget_bytes"]))


def scheduled_message_gain(epoch: int, base: float) -> float:
    """train...:277-280"""
    return 0.30 if epoch < 100 else (0.40 if epoch < 200 else base)


def premult_loss(x: torch.Tensor, target: torch.Tensor, scale: float, want_grad: bool = True):
    """Per-sample premultiplied-RGBA MSE (train...:52-61) and d(scale * sum_b loss_b)/dx, one fused kernel.

    `target` is [4, H, W], or [M, 4, H, W] with M dividing the batch: sample b is then measured against
    target[b // (B // M)], the per-model targets of a model-major stack (PopulationTrainer)."""
    stacked = target.dim() == 4
    if stacked:
        B, _, H, W = x.shape
        M = target.shape[0]
        if tuple(target.shape[1:]) != (4, H, W) or M < 1 or B % M:
            raise ValueError(f"premult_loss: target must be [4, {H}, {W}] or [M, 4, {H}, {W}] with M dividing the "
                             f"batch of {B}, got {list(target.shape)}")
        target = GF._require_cuda_f32(target, "target")
    x = GF._require_cuda_f32(x, "x")
    B, Cc, H, W = x.shape
    if stacked and target.device != x.device:
        raise ValueError(f"premult_loss: target is on {target.device}, x on {x.device}")
    per = torch.empty(B, dtype=torch.float32, device=x.device)
    gx = torch.empty_like(x) if want_grad else None
    lib = _lib.load()
    if stacked:
        _lib.check(lib.gnca_loss_premult_rgba_targets(B, Cc, H, W, GF._ptr(x), GF._ptr(target), M, GF._ptr(per),
                                                      GF._ptr(gx), float(scale), GF._stream()),
                   "gnca_loss_premult_rgba_targets")
    else:
        _lib.check(lib.gnca_loss_premult_rgba(B, Cc, H, W, GF._ptr(x), GF._ptr(target.contiguous()), GF._ptr(per),
                                              GF._ptr(gx), float(scale), GF._stream()), "gnca_loss_premult_rgba")
    return per, gx


class GraphNCATrainer:
    """pool sample -> damage -> per-sample-length rollout with per-step fire rate / message gating -> premult
    loss -> BPTT -> (all-reduce) -> per-tensor grad normalisation -> Adam -> worst-k / random reseed -> pool replace."""

    def __init__(self, model, target: torch.Tensor, cfg: TrainConfig, *, seed_fn: Optional[Callable] = None):
        self.model, self.cfg = model, cfg
        self.device = next(model.parameters()).device
        self.target = target.to(self.device).float().contiguous()           # [4,H,W], RGB premultiplied
        self.n_ch, self.img = model.n_channels, model.img_size
        self.seed_fn = seed_fn or (lambda batch_size=1: trainer_seed(self.n_ch, self.img, batch_size, self.device))
        self.shard = Shard(cfg.batch_size)
        self.owner_pool = cfg.pool_sharding == "owner" and self.shard.world > 1
        if cfg.pool_sharding not in ("replicated", "owner"):
            raise ValueError("pool_sharding must be 'replicated' or 'owner'")
        if self.owner_pool and cfg.pool_size % self.shard.world:
            raise ValueError("pool_size must be divisible by the world size for pool_sharding='owner'")
        self.pool = SamplePool(cfg.pool_size // self.shard.world if self.owner_pool else cfg.pool_size, self.seed_fn,
                               device=self.device)
        self.opt = FusedNormalizedAdam(model, lr=cfg.learning_rate, weight_decay=cfg.weight_decay, normalize=True)
        self.is_graph = bool(getattr(model, "_is_graph", False))
        self.last: Dict = {}

    def lr_at(self, epoch: int) -> float:
        """StepLR stepped once per epoch (train...:149-158, scheduler.step() after each epoch), epochs are 1-based."""
        return self.cfg.learning_rate * self.cfg.scheduler_gamma ** ((epoch - 1) // self.cfg.scheduler_step_size)

    def _draw_schedule(self, epoch: int, B: int, state: torch.Tensor):
        """Appendix B, rows 5 ... end of rollout: regime, step counts, then per step (fire rate, gating, offsets,
        fire uniforms).

        fire="torch" replays the reference's draws call for call (device `torch.randint` step counts -> the iteration's ONE
        host sync, one 1-element `uniform_` per step, one `torch.rand` per step, one `random.sample` per step).
        fire="philox" is the production mode: same distributions, but nothing waits for the device -- step counts come
        from the host generator, the T fire rates from one device call, the T offset draws from one block replay of the
        python RNG stream, fire masks from the in-kernel Philox stream; the whole iteration is enqueued asynchronously."""
        cfg, dev = self.cfg, self.device
        fast = cfg.fire == "philox"
        if random.random() < cfg.long_rollout_prob:
            lo, hi = cfg.long_rollout_steps_min, cfg.long_rollout_steps_max
        else:
            lo, hi = cfg.nca_steps_min, cfg.nca_steps_max
        if fast:
            steps_host = torch.randint(lo, hi + 1, (B,)).numpy()              # host generator: no device round trip
        else:
            steps_host = torch.randint(lo, hi + 1, (B,), device=dev).cpu().numpy()   # train...:297-301; the one host sync
        T = int(steps_host.max())
        base_gain = scheduled_message_gain(epoch, cfg.message_gain)
        H = W = self.img
        fr_dev = torch.empty(T, dtype=torch.float32, device=dev)
        gains, offsets = [], []
        fire_u = torch.empty(T, B, 1, H, W, dtype=torch.float32, device=dev) if not fast else None
        interleaved = cfg.message_every <= 1 and cfg.message_rate < 1.0       # random.random() between the offset draws
        if fast:
            fr_dev.uniform_(cfg.fire_rate_min, cfg.fire_rate_max)
        if fast and not interleaved:
            gains = [base_gain if (cfg.message_every <= 1 or t % cfg.message_every == 0) else 0.0 for t in range(T)]
            offsets = self.model.graph.draw_offsets_array(T) if self.is_graph else None
        else:
            for t in range(T):
                if not fast:
                    fr_dev[t:t + 1].uniform_(cfg.fire_rate_min, cfg.fire_rate_max)       # train...:310
                use_graph = True
                if cfg.message_every > 1:
                    use_graph = (t % cfg.message_every == 0)
                elif cfg.message_rate < 1.0:
                    use_graph = random.random() < cfg.message_rate
                gains.append(base_gain if use_graph else 0.0)
                if self.is_graph:
                    offsets.append(self.model.graph.draw_offsets())                   # graph_augmentation.py:121
                if fire_u is not None:
                    act = np.nonzero(steps_host > t)[0]
                    if len(act) == B:
                        torch.rand(B, 1, H, W, out=fire_u[t])                         # ncagraph.py:145
                    else:
                        fire_u[t, torch.as_tensor(act, device=dev)] = torch.rand(len(act), 1, H, W, device=dev)
        sh = self.shard
        sched = make_schedule(self.model, sh.local_batch, H, W, T, fire_rate=[0.0] * T, message_gains=gains,
                              offsets=offsets if self.is_graph else None, steps=steps_host[sh.lo:sh.hi].tolist(),
                              fire="philox", seed=random.getrandbits(63) if fast else 0, device=dev)
        sched.fire_rate = fr_dev                                            # device-resident draws, no .item()
        if fast and sh.world > 1:
            # the in-kernel counter is indexed by the LOCAL sample (t*B_local + b): give every rank its own block range so
            # that the fire masks of the global batch are independent, like the reference's one torch.rand over the batch
            sched.philox_offset = sh.rank * ((T * sh.local_batch * H * W + 3) // 4)
        if fire_u is not None:
            sched.fire_u = fire_u[:, sh.lo:sh.hi].contiguous().view(T, sh.local_batch, H, W)
        return sched, steps_host

    def train_step(self, epoch: int = 1) -> Dict:
        cfg, sh = self.cfg, self.shard
        Bg = cfg.batch_size
        fast = cfg.fire == "philox"
        if self.owner_pool:     # my share of the batch from my own slots (same host-RNG consumption on every rank)
            idx, state = self.pool.sample(sh.local_batch)
            x0 = state.contiguous()
        else:
            idx, state = self.pool.sample(Bg)                               # pool.py:28 (global batch everywhere)
            x0 = None
        # damage.py:101-138 -- the policy draws (gate, kind, size) are batch-level and identical on every rank; with an
        # owner-sharded pool the geometry is drawn for the local samples only
        D = sample_damage_mask(state, cfg.damage, epoch, fast=fast) if cfg.damage else None
        sched, steps_host = self._draw_schedule(epoch, Bg, state)
        if D is not None:                       # applied in-kernel to x_0 (the reference damages before the rollout)
            mine = D if self.owner_pool else D.take(sh.lo, sh.hi)           # per-cell plane [B,H,W]: no [B,C,H,W] mask
            sched.damage, sched.damage_layout, sched.damage_step = mine.plane, mine.layout, 0
        if x0 is None:
            x0 = sh.take(state).contiguous()
        desc, packed = self.model.model_desc(), self.model.packed_weights()
        impl = {"auto": 0, "streaming": 1, "resident": 2, "banded": 3}[cfg.rollout_impl]
        xT, hist = rollout_fwd_raw(desc, packed, x0, sched, history=True, impl=impl, keep_x=False,
                                   bptt_budget=cfg.bptt_budget_bytes)
        per_local, gxT = premult_loss(xT, self.target, 1.0 / Bg)             # loss = mean over the GLOBAL batch
        _, gflat = rollout_bwd_raw(desc, packed, hist, sched, gxT, impl=impl)
        sh.allreduce_sum_(gflat)                                             # the one data-path collective
        self.opt.step(gflat, lr=self.lr_at(epoch))                           # normalise AFTER the all-reduce
        per_global = sh.allgather(per_local)                                 # B floats: global worst-k stays bit-exact
        worst = worst_k_indices(per_global, cfg.reset_worst_prob)            # train...:378-380
        do_reseed = random.random() < cfg.random_reseed_prob
        if do_reseed:      # train...:386-389; fast mode draws the slot on the host (no device round trip)
            rand_idx = int(torch.randint(0, Bg, (1,)).item()) if fast else \
                int(torch.randint(0, Bg, (1,), device=self.device).item())
        else:
            rand_idx = None
        if self.owner_pool:
            # every rank reseeds and stores only ITS samples: no state leaves the GPU.  Membership of the global worst-k /
            # reseed slot in my shard is decided on the device (mask), so the step stays free of host syncs.
            new_states = xT
            n_w = 0 if worst is None else int(worst.numel())
            if n_w > 0 or do_reseed:
                hit = torch.zeros(Bg, dtype=torch.bool, device=self.device)
                if n_w > 0:
                    hit.index_fill_(0, worst, True)      # (hit[worst] = True would stage the scalar through pageable
                if do_reseed:                            #  memory: a hidden stream synchronisation per step)
                    hit[rand_idx:rand_idx + 1].fill_(True)
                mine = hit[sh.lo:sh.hi].view(-1, 1, 1, 1)
                new_states = torch.where(mine, self.seed_fn(sh.local_batch), xT)
        else:
            new_states = sh.allgather(xT)
            if worst is not None and worst.numel() > 0:
                new_states = new_states.clone()
                new_states[worst] = self.seed_fn(len(worst))
            if do_reseed:
                new_states = new_states.clone()
                new_states[rand_idx:rand_idx + 1] = self.seed_fn(1)
        self.pool.replace(idx, new_states)
        self.last = {"per_sample": per_global, "loss": per_global.mean(), "steps": steps_host, "worst": worst,
                     "gflat": gflat, "cell_updates": int(np.minimum(steps_host, sched.T).sum()) * self.img * self.img}
        return self.last

#!/usr/bin/env python
"""bench.py -- graph-NCA cell-updates/s on B200 (BASELINE.json metric), one JSON line on stdout.

Workload (default, BASELINE.json configs[1]): graph-augmented NCA forward rollout, 16 channels, 40x40, batch 8,
96 steps, fire_rate 0.5, torus graph shift, 8 of 72 offsets per step, trained weights (tests/golden fixture),
growth from the single-cell seed.  A "step" of this bench = ONE such rollout (B*T*H*W = 1,228,800 cell-updates).

  value : rollouts timed with CUDA events, x0 / weights / schedule resident in HBM, L2 flushed between iterations.
  e2e   : the same through the public API with HOST buffers: pinned x0 -> H2D, schedule draws (random.sample per
          step, as T forward calls would), rollout, x_T -> D2H.  Wall clock around each call (sync both sides).
  roofline      : dominant kernel, CUDA events around its launches (library hook), fp32-FMA bound; ncu-derived fields
                  (DRAM traffic, pipe utilisation) are read from the tracked capture summary profiles/ncu_r02.json.
  cpu_baseline  : the REFERENCE's own modules (oracle/_ref, staged by oracle/build_ref.py; oracle port if absent) on
                  the host cores (N=1, rank 0);  gpu_eager: the same modules in PyTorch eager on the B200.
  fwd_bwd       : BASELINE configs[2]/[3] through the public trainer API (GraphNCATrainer.train_step: pool draw, damage
                  policy, per-sample randint step counts, per-step U(0.5,0.9) fire rate, msg_every=3, loss, BPTT,
                  NCCL all-reduce, normalise + Adam, worst-k reseed, pool replace), short and long regime separately,
                  weak (32 per GPU) and -- for N > 1 -- strong (global batch 32) scaling; its own roofline, cpu_baseline
                  and gpu_eager.
  --impl reference : the reference modules alone on the host cores, same JSON shape, batch scaled with --gpus.

Other workloads: --workload c1 (classic NCA rollout), c3 / c3l (the training HOT PATH only -- rollout fwd+bwd, loss,
optimiser -- at fixed T=64 / T=300, no pool: a kernel-development line), c4 (c3 with an in-kernel damage mask), c5s
(256x256x32 scale-up slice, streaming kernels), c5 (the full per-GPU share of BASELINE configs[4]: B=128, T=1000,
damage at t=500 -- seconds per rollout: run it with --steps 2 --warmup 1).
"""
from __future__ import annotations

import argparse
import json
import os
import random
import statistics
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
GOLDEN = os.path.join(ROOT, "tests", "golden")

# dense algorithmic work per cell-update (SURVEY 8d / BASELINE.md 4), graph model C=16 hidden=128 k=8
FLOP_FWD_GRAPH_S = 17.9e3
FLOP_FWDBWD_GRAPH_S = 53.6e3
FLOP_FWD_GRAPH_L = 36.7e3
FP32_LANES = 148 * 128 * 2           # FMA lanes x 2 flop


def load_peaks():
    """Measured roofline denominators (driver-written MEASURED_PEAKS.json), else the profiling guide's fallback."""
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            d = json.load(f)
        return {"hbm_gbs": float(d["hbm_gbs"]), "bf16_tflops": float(d["bf16_tflops"]), "source": "MEASURED_PEAKS.json (of measured)"}
    except Exception:
        return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "source": "B200_PROFILING.md fallback (of fallback)"}


PEAKS = load_peaks()


def ncu_capture(workload, kernel):
    """ncu-derived facts of (workload, kernel) from the tracked summary profiles/ncu_r02.json (written by
    scripts/ncu_summary.py from a committed `ncu --set full` capture; each entry names its command, report and commit).
    They describe THAT capture, not this run -- the bench line says so next to the numbers."""
    try:
        with open(os.path.join(ROOT, "profiles", "ncu_r02.json")) as f:
            return json.load(f).get(f"{workload}:{kernel}")
    except Exception:
        return None


def load_weights(name):
    return {k: torch.from_numpy(v) for k, v in np.load(os.path.join(GOLDEN, name)).items()}


def workload_cfg(name):
    if name == "c2":
        return dict(name="c2: graph NCA fwd rollout, seed growth", C=16, H=40, W=40, B=8, T=96, hidden=128,
                    fire_rate=0.5, message_every=1, train=False, flop=FLOP_FWD_GRAPH_S)
    if name == "c3":
        return dict(name="c3: graph NCA training step (fwd+bwd, short regime)", C=16, H=40, W=40, B=32, T=64,
                    hidden=128, fire_rate=0.7, message_every=3, train=True, flop=FLOP_FWDBWD_GRAPH_S)
    if name == "c1":
        return dict(name="c1: classic NCA fwd rollout, seed growth (the reference's CPU-runnable case, here on the GPU)",
                    C=16, H=40, W=40, B=8, T=96, hidden=128, fire_rate=0.5, message_every=1, train=False,
                    flop=17.0e3, classic=True)
    if name == "c4":
        return dict(name="c4: graph NCA training step with damage (fwd+bwd, short regime, damaged batch)", C=16, H=40, W=40,
                    B=32, T=64, hidden=128, fire_rate=0.7, message_every=3, train=True, flop=FLOP_FWDBWD_GRAPH_S,
                    damage=True)
    if name == "c3l":
        return dict(name="c3l: graph NCA training step (fwd+bwd, long regime)", C=16, H=40, W=40, B=32, T=300,
                    hidden=128, fire_rate=0.7, message_every=3, train=True, flop=FLOP_FWDBWD_GRAPH_S)
    if name == "c5s":
        return dict(name="c5 slice: 256x256x32 fwd rollout", C=32, H=256, W=256, B=16, T=20, hidden=128,
                    fire_rate=0.5, message_every=1, train=False, flop=FLOP_FWD_GRAPH_L)
    if name == "c5":      # BASELINE configs[4] per GPU: batch 1024 over 8 GPUs = 128 per GPU, 1000 steps, damage at t = 500
        return dict(name="c5: 256x256x32 regeneration rollout, B=128 per GPU, T=1000, circle damage at t=500", C=32, H=256,
                    W=256, B=128, T=1000, hidden=128, fire_rate=0.5, message_every=1, train=False, flop=FLOP_FWD_GRAPH_L,
                    damage=True, damage_step=500, damage_size=64)
    raise SystemExit(f"unknown workload {name}")


class ClockSampler(threading.Thread):
    """Samples SM clock and throttle reasons while the timed region runs (B200_PROFILING.md clocks line)."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.stop_flag, self.samples, self.reasons = index, False, [], set()
        self.max_mhz = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def run(self):
        if self.nv is None:
            return
        nv = self.nv
        names = {"hw_slowdown": getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8),
                 "hw_thermal_slowdown": getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40),
                 "sw_thermal_slowdown": getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20),
                 "sw_power_cap": getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4)}
        while not self.stop_flag:
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    mask = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    mask = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for k, bit in names.items():
                    if mask & bit:
                        self.reasons.add(k)
            except Exception:
                pass
            time.sleep(0.002)       # the default timed region is ~20 ms: sample densely enough to see it

    def result(self):
        return {"sm_mhz": statistics.median(self.samples) if self.samples else None,
                "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": len(self.samples)}


def cpu_forward_baseline(cfg):
    """cpu_baseline of a forward workload: the reference's modules on all host cores, full workload, best of 2."""
    import bench_ref
    if cfg["C"] != 16 or cfg.get("classic"):
        return None
    r = bench_ref.time_forward(cfg["B"], cfg["T"], cfg["fire_rate"], "cpu", reps=2)
    return {"value": r["value"], "unit": "cell-updates/s", "cores": r["cores"], "kind": r["kind"],
            "sample": f"full workload: B={cfg['B']} T={cfg['T']} {cfg['H']}x{cfg['W']}x{cfg['C']} forward rollout, best of 2, "
                      f"{r['seconds']:.2f} s per rollout, torch CPU {torch.__version__}"}


def gpu_eager_forward(cfg, dev):
    """The reference's modules in PyTorch eager ON THE B200 (like-for-like GPU comparator, BASELINE.md section 3)."""
    import bench_ref
    if cfg["C"] != 16 or cfg.get("classic"):
        return None
    r = bench_ref.time_forward(cfg["B"], cfg["T"], cfg["fire_rate"], dev, reps=3)
    return {"value": r["value"], "unit": "cell-updates/s", "kind": r["kind"] + " modules, torch eager on cuda",
            "ms_per_step": r["seconds"] * 1e3, "sample": f"full workload, best of 3, torch {torch.__version__}"}


def run_reference_arm(args, cfg, rank):
    """`--impl reference`: the reference's own CPU implementation of the path on this box's host cores, on OUR arm's
    config (weak scaling: per-GPU batch x --gpus), rank 0 only."""
    if rank != 0:
        return
    import bench_ref
    threads = os.cpu_count() or 1
    torch.set_num_threads(threads)
    B = cfg["B"] * max(1, args.gpus)
    model, kind = bench_ref.make_reference_graph("cpu")
    random.seed(42); torch.manual_seed(42)
    T = cfg["T"]
    for _ in range(args.warmup):
        bench_ref.forward_rollout(model, B, T, cfg["fire_rate"], "cpu", cfg["message_every"])
    t0 = time.perf_counter()
    for _ in range(args.steps):
        bench_ref.forward_rollout(model, B, T, cfg["fire_rate"], "cpu", cfg["message_every"])
    dt = time.perf_counter() - t0
    updates = B * T * cfg["H"] * cfg["W"]
    val = updates * args.steps / dt
    line = {"impl": "reference", "metric": "graph-NCA cell-updates/s (fwd)", "value": val, "unit": "cell-updates/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": cfg["name"], "B_per_gpu": cfg["B"], "B_total": B, "T": T, "grid": [cfg["H"], cfg["W"]],
                       "channels": cfg["C"],
                       "note": "the reference's own modules (oracle/_ref, staged from /root/reference/src by "
                               "oracle/build_ref.py) on the host cores; oracle port when that directory is absent"},
            "cpu_baseline": {"value": val, "unit": "cell-updates/s", "cores": threads, "kind": kind,
                             "sample": f"full workload per step (B={B} = {cfg['B']} per GPU x {max(1, args.gpus)})"},
            "e2e": {"value": val, "unit": "cell-updates/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


def make_roofline(cfg, kname, ms, n, nprof, updates, clocks, kernels_ms, step_ms, x_numel, T, args, active_frac=None):
    """roofline object of the dominant kernel `kname` (ms over n launches in nprof steps of `updates` cell-updates).
    FFMA kernels (k_rep_*, the FFMA k_update): fp32-FMA bound, dense-equivalent flops.  The tensor-core k_update
    (256x256x32 path): its 3xTF32 MMAs are far from the tensor peak, the step is bound by moving the state -> HBM view
    (SURVEY 8d: 8C bytes per cell and step for the streaming pair) with the tensor view beside it."""
    wl = cfg["name"][:2]
    # algorithmic (dense) flops / launch.  Training step: the credited 3 x forward flops split evenly over its three
    # kernels (forward 17.9 k; data gradients gh, gy, perception^T, message^T 17.9 k; weight gradients 17.8 k per
    # cell-update -- the hidden-layer recompute inside k_rep_bwd is overhead and not credited, SURVEY 8d)
    kflop = cfg["flop"] / 3.0 if cfg["train"] else cfg["flop"]
    flops_per_launch = kflop * updates * nprof / n
    avg_s = ms * 1e-3 / n
    mhz = clocks["sm_max_mhz"] or 1965
    peak32 = FP32_LANES * mhz * 1e6 / 1e12
    ach32 = flops_per_launch / avg_s / 1e12
    cap = ncu_capture(wl, kname) or {}
    cap_note = (f"ncu fields from the committed capture {cap.get('report')} ({cap.get('command')}, commit {cap.get('commit')}); "
                "they describe that capture, not this run") if cap else "no committed ncu capture for this kernel / workload"
    streaming = kname in ("k_update", "k_apply")
    state_bytes = x_numel * 4
    hbm = {"algorithmic_bytes_per_step": int(2 * state_bytes * (T if streaming else 1)),
           "achieved_GBps": 2 * state_bytes * (T if streaming else 1) * nprof / (ms * 1e-3) / 1e9, "peak_GBps": PEAKS["hbm_gbs"]}
    common = {"kernel": kname, "avg_launch_ms": avg_s * 1e3, "launches_per_step": n / nprof,
              "share_of_step": ms / nprof / step_ms, "kernels": kernels_ms,
              "traffic": cap.get("dram_bytes_per_launch"), "ncu": {k: v for k, v in cap.items() if k.endswith("_pct")},
              "ncu_source": cap_note}
    tc = streaming and cfg["C"] in (16, 32) and cfg["hidden"] == 128 and not os.environ.get("GNCA_NO_TC") and \
        cfg["B"] * ((cfg["H"] * cfg["W"] + 1023) // 1024) >= 2 * 148
    if tc and kname == "k_update":
        # k_update_tc per launch: reads x of the step once (the 3x3 / sender re-reads are L2 hits by design), writes u of the
        # active cells; the MLP runs as 3 TF32 passes on the tensor cores
        af = active_frac if active_frac is not None else cap.get("active_fraction", 0.28)
        bytes_launch = state_bytes * (1.0 + af)
        ach = bytes_launch / avg_s / 1e9
        mlp_flop = 2.0 * (3 * cfg["C"] * cfg["hidden"] + cfg["hidden"] * cfg["C"])
        tf32_exec = 3.0 * mlp_flop * af * (updates / T) / avg_s / 1e12
        return {"bound": "hbm", "achieved": ach, "peak": PEAKS["hbm_gbs"], "unit": "GB/s", "frac": ach / PEAKS["hbm_gbs"],
                "peak_source": PEAKS["source"],
                "note": "algorithmic bytes of ONE k_update_tc launch (state read once + u of the active cells written, active "
                        f"fraction {af:.2f}) / its CUDA-event duration; the launch also covers k_compact + k_scan",
                "tensor_view": {"executed_tf32_TFLOPs": tf32_exec, "peak_tf32_TFLOPs": PEAKS["bf16_tflops"] / 2,
                                "frac": tf32_exec / (PEAKS["bf16_tflops"] / 2),
                                "note": "3 TF32 passes x 2*(3C*hid + hid*C) flops x ACTIVE cells; tf32 dense peak taken as half "
                                        "the measured bf16 cuBLAS figure"},
                "fp32_dense_equivalent": {"achieved_TFLOPs": ach32, "ffma_peak_TFLOPs": peak32, "frac": ach32 / peak32},
                "step_hbm_view": hbm, **common}
    return {"bound": "fp32_fma", "achieved": ach32, "peak": peak32, "unit": "TFLOP/s", "frac": ach32 / peak32,
            "peak_source": f"derived: 148 SM x 128 FMA lanes x 2 x {mhz} MHz (MEASURED_PEAKS.json has no fp32 entry; "
                           f"hbm_gbs {PEAKS['hbm_gbs']} measured is far from binding: see hbm_view)",
            "note": "achieved = DENSE algorithmic flops (every cell counted) / measured kernel time; the kernel "
                    "skips cells whose fire*alive mask is 0, so frac is a dense-equivalent figure (the ncu pipe "
                    "utilisation of the committed capture is in `ncu`)",
            "hbm_view": hbm, **common}


def run_workload(cfg, args, world, rank, local_rank, dev, steps, warmup, with_roofline=True):
    """Times one workload: returns dict(value, ms_per_step, e2e, launches, roofline, clocks, data)."""
    import torch.distributed as dist
    import graph_neural_cellular_automata_b200 as G
    from graph_neural_cellular_automata_b200 import _lib
    from graph_neural_cellular_automata_b200.rollout import make_schedule, rollout
    from graph_neural_cellular_automata_b200.utils.nca_init import make_seed
    import ctypes

    lib = _lib.load()
    C_, H, W, B, T = cfg["C"], cfg["H"], cfg["W"], cfg["B"], cfg["T"]
    torch.manual_seed(42 + rank); random.seed(42 + rank)
    if cfg.get("classic"):
        model = G.NeuralCA(C_, update_hidden=cfg["hidden"], img_size=H, update_gain=0.05, alpha_thr=0.12)
        model.load_state_dict(load_weights("weights_classic_ep990.npz"), strict=False)
        data = "synthetic (seed growth; trained classic 40x40 gecko weights shipped as a fixture)"
    else:
        model = G.NeuralCAGraph(C_, update_hidden=cfg["hidden"], img_size=H, update_gain=0.05, alpha_thr=0.12,
                                message_gain=0.25, hidden_only=True, graph_zero_padded_shift=False)
    if cfg.get("classic"):
        pass
    elif C_ == 16:
        model.load_state_dict(load_weights("weights_graph_ep960.npz"), strict=False)
        data = "synthetic (seed growth; trained 40x40 gecko weights shipped as a fixture)"
    else:
        with torch.no_grad():
            model.update_net[2].weight.normal_(0, 0.05)
        data = "synthetic (seeded random weights, zero-mean W2 sigma 0.05)"
    model = model.to(dev)
    if cfg["train"]:
        target = torch.from_numpy(np.load(os.path.join(GOLDEN, "target_gecko_surrogate.npy"))).to(dev)

    def make_x0():
        if C_ == 16 and cfg["train"]:       # pool-like states: seeds grown for a random number of steps
            x = make_seed(C_, H, B, device=dev)
            with torch.no_grad():
                for t in range(48):
                    x = model(x, fire_rate=0.6)
            return x.cpu()
        if C_ == 16:
            return make_seed(C_, H, B, device="cpu")
        x = torch.rand(B, C_, H, W)
        yy, xx = torch.meshgrid(torch.arange(H), torch.arange(W), indexing="ij")
        disk = (((yy - H / 2) ** 2 + (xx - W / 2) ** 2) < (0.3 * H) ** 2).float()
        return x * disk

    x0_host = make_x0().pin_memory()
    x0_dev = x0_host.to(dev)
    xT_host = torch.empty_like(x0_host).pin_memory()
    flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device=dev)   # > 126 MB L2
    updates = B * T * H * W

    if cfg["train"]:
        from graph_neural_cellular_automata_b200.training.trainer import premult_loss
        from graph_neural_cellular_automata_b200.training.optim import FusedNormalizedAdam
        from graph_neural_cellular_automata_b200.rollout import rollout_fwd_raw, rollout_bwd_raw
        opt = FusedNormalizedAdam(model, lr=2e-4, weight_decay=1e-5, normalize=True)
        IMPLN = {"auto": 0, "streaming": 1, "resident": 2, "banded": 3}[args.rollout_impl]

    def one_rollout(x0, sched):
        if cfg["train"]:     # fwd (history) + premult loss + BPTT + grad normalise + Adam: one training iteration's hot path
            desc, packed = model.model_desc(), model.packed_weights()
            xT, hist = rollout_fwd_raw(desc, packed, x0, sched, history=True, impl=IMPLN, keep_x=False)
            per, gxT = premult_loss(xT, target, 1.0 / (B * world))
            _, gflat = rollout_bwd_raw(desc, packed, hist, sched, gxT, impl=IMPLN)
            if world > 1:
                dist.all_reduce(gflat)
            opt.step(gflat)
            return xT
        with torch.no_grad():
            return rollout(model, x0, sched, impl=args.rollout_impl)

    dmg = None
    if cfg.get("damage"):      # one damage kind / size for the batch, per-sample positions (utils/damage.py), applied in-kernel at step 0
        from graph_neural_cellular_automata_b200.utils.damage import circle_mask
        dmg = circle_mask(x0_dev, int(cfg.get("damage_size", 5)))      # a Damage descriptor -> per-cell plane, no [B,C,H,W] mask

    def new_schedule(seed):
        return make_schedule(model, B, H, W, T, fire_rate=cfg["fire_rate"], message_every=cfg["message_every"],
                             fire="philox", seed=seed, damage=dmg, damage_step=int(cfg.get("damage_step", 0)))

    # ---------------- device-resident timing (value) ----------------
    scheds = [new_schedule(1000 + i) for i in range(warmup + steps)]
    torch.cuda.synchronize()
    for i in range(warmup):
        one_rollout(x0_dev, scheds[i])
    torch.cuda.synchronize()
    import gc
    gc.collect()
    gc.freeze()          # no full-heap Python collection on one of N ranks inside the timed region (max over ranks is reported)
    if world > 1:
        dist.barrier()
    sampler = ClockSampler(local_rank)
    sampler.start()
    launches0 = lib.gnca_launch_count()
    evs = []
    torch.cuda.synchronize()
    for i in range(steps):
        flush.fill_(float(i))                        # L2 flush between timed iterations (outside the events)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        xT = one_rollout(x0_dev, scheds[warmup + i])
        e1.record()
        evs.append((e0, e1))
    torch.cuda.synchronize()
    launches = lib.gnca_launch_count() - launches0
    outputs = None
    if args.dump_outputs:        # copied before the e2e / roofline passes below run further steps (training updates weights)
        outputs = {"x_T": xT.detach().clone()}
        if cfg["train"]:
            outputs["weights"] = opt.flat.clone()
    sampler.stop_flag = True
    sampler.join()
    if world > 1:
        dist.barrier()
    dev_ms = sum(a.elapsed_time(b) for a, b in evs)
    t = torch.tensor([dev_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    dev_ms_max = float(t.item())
    value = world * updates * steps / (dev_ms_max * 1e-3)

    # ---------------- end-to-end through the public API with host buffers ----------------
    def e2e_once(seed):
        x0 = x0_host.to(dev, non_blocking=True)
        sched = new_schedule(seed)
        xT = one_rollout(x0, sched)
        xT_host.copy_(xT, non_blocking=True)
        torch.cuda.synchronize()

    if os.environ.get("GNCA_E2E_DEBUG"):
        import time as _t
        for i in range(5):
            t_a = _t.perf_counter(); x0_ = x0_host.to(dev, non_blocking=True); t_b = _t.perf_counter()
            sc_ = new_schedule(7000 + i); t_c = _t.perf_counter(); y_ = one_rollout(x0_, sc_); t_d = _t.perf_counter()
            xT_host.copy_(y_, non_blocking=True); t_e = _t.perf_counter(); torch.cuda.synchronize(); t_f = _t.perf_counter()
            print("[e2e debug] h2d %.3f sched %.3f launch %.3f d2h-call %.3f sync %.3f total %.3f ms" % (
                (t_b - t_a) * 1e3, (t_c - t_b) * 1e3, (t_d - t_c) * 1e3, (t_e - t_d) * 1e3, (t_f - t_e) * 1e3, (t_f - t_a) * 1e3),
                file=sys.stderr)
    import gc
    for i in range(8 if updates < 1e8 else 1):          # second-long rollouts (c5) need no repeated host warm-up
        e2e_once(5000 + i)
    gc.collect()
    gc.freeze()          # the timed loop allocates a handful of small objects per call; do not rescan the rest of the heap
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for i in range(steps):
        e2e_once(6000 + i)
    e2e_s = time.perf_counter() - t0
    t = torch.tensor([e2e_s], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_value = world * updates * steps / float(t.item())
    sched_bytes = T * 4 * 2 + T * 8 * 2
    e2e = {"value": e2e_value, "unit": "cell-updates/s", "h2d_bytes_per_step": int(x0_host.numel() * 4 + sched_bytes),
           "d2h_bytes_per_step": int(xT_host.numel() * 4), "ms_per_step": float(t.item()) / steps * 1e3}

    # ---------------- roofline of the dominant kernel (library event hook), rank 0 ----------------
    roof = None
    if with_roofline:            # every rank runs these iterations (the training step holds a collective); rank 0 reports
        lib.gnca_profile_enable(1)
        nprof = min(steps, 5)
        for i in range(nprof):
            flush.fill_(1.0)
            one_rollout(x0_dev, scheds[warmup + i])
        torch.cuda.synchronize()
        lib.gnca_profile_enable(0)
        per_kernel = {}
        for kid, kname in ((0, "k_update"), (1, "k_apply"), (2, "k_rep_fwd"), (3, "k_rep_wgrad"), (6, "k_rep_bwd")):
            ms, n = ctypes.c_double(0), ctypes.c_ulonglong(0)
            lib.gnca_profile_read(kid, ctypes.byref(ms), ctypes.byref(n))
            if n.value:
                per_kernel[kname] = (ms.value, n.value)
        kernels_ms = {k: {"ms_per_step": v[0] / nprof, "launches_per_step": v[1] / nprof} for k, v in per_kernel.items()}
        if per_kernel:
            kname = max(per_kernel, key=lambda k: per_kernel[k][0])
            ms, n = per_kernel[kname]
            roof = make_roofline(cfg, kname, ms, n, nprof, updates, sampler.result(), kernels_ms, dev_ms_max / steps,
                                 x0_host.numel(), T, args)

    return {"value": value, "ms_per_step": dev_ms_max / steps, "e2e": e2e, "launches": int(launches), "roofline": roof,
            "clocks": sampler.result(), "data": data, "dims": (C_, H, W, B, T), "outputs": outputs}


def dump_outputs(dirname, arrays, limit=64 << 20):
    """Writes each array as DIR/<name>.npy in float32, `limit` bytes in all.  An array larger than its share is stored as
    DIR/<name>_sample.npy: the flat elements at a fixed set of indices (seeded draw, sorted), the same in every run."""
    os.makedirs(dirname, exist_ok=True)
    share = limit // len(arrays)
    for name, t in arrays.items():
        t = t.detach().float()
        if t.numel() * 4 > share:
            idx = torch.randint(t.numel(), (share // 4,), generator=torch.Generator().manual_seed(0)).unique()
            t, name = t.reshape(-1)[idx.to(t.device)], name + "_sample"
        np.save(os.path.join(dirname, name + ".npy"), t.cpu().numpy())


def run_trainer(args, world, rank, local_rank, dev, steps, warmup, regime="short", scaling="weak", per_gpu=32,
                damage=False):
    """BASELINE configs[2] / [3]: the training iteration through the PUBLIC trainer API (GraphNCATrainer.train_step,
    the loop body of train_graph_augmented_nca.py:289-391): pool draw (1024-pool of mixed ages), damage policy
    (configs[3]: the reference's config.json `damage` section at epoch >= 100), per-sample randint step counts
    (short [48,80] / long [200,400]), per-step U(0.5,0.9) fire rate, message on t % 3 == 0, in-kernel Philox fire masks,
    loss, BPTT, NCCL all-reduce of the flat gradient, normalise + Adam, all-gather of losses / states, worst-k reseed,
    pool replace.  weak: `per_gpu` samples per GPU; strong: global batch `per_gpu` split over the ranks."""
    import ctypes
    import torch.distributed as dist
    import graph_neural_cellular_automata_b200 as G
    from graph_neural_cellular_automata_b200 import _lib
    from graph_neural_cellular_automata_b200.rollout import make_schedule, rollout
    from graph_neural_cellular_automata_b200.training.trainer import GraphNCATrainer, TrainConfig

    lib = _lib.load()
    Bg = per_gpu * world if scaling == "weak" else per_gpu
    if Bg % world:
        return None
    torch.manual_seed(1234); random.seed(1234)           # every rank replays the SAME host RNG (training/dp.py)
    model = G.NeuralCAGraph(16, update_hidden=128, img_size=40, update_gain=0.05, alpha_thr=0.12, message_gain=0.25,
                            hidden_only=True, graph_zero_padded_shift=False)
    model.load_state_dict(load_weights("weights_graph_ep960.npz"), strict=False)
    model = model.to(dev)
    target = torch.from_numpy(np.load(os.path.join(GOLDEN, "target_gecko_surrogate.npy"))).to(dev)
    dmg = {}
    if damage:           # /root/reference/configs/config.json `damage` with prob 1 so that every timed step carries the mask
        dmg = {"start_epoch": 100, "prob": 1.0, "kinds": {"square": 0.35, "circle": 0.25, "stripes": 0.1, "alpha_drop": 0.15,
               "saltpepper": 0.05, "gaussian": 0.1}, "size_min": 6, "size_max": 18, "stripe_width": 6, "alpha_thr": 0.2,
               "alpha_dropout_p": 0.15, "salt_pepper_p": 0.02, "gaussian_softness": 0.35}
    # N > 1: the pool is partitioned over the ranks (rank r owns 1024 / N slots and draws its share of the batch from them:
    # no state all-gather; --pool replicated keeps the reference's global draw + all-gather for comparison)
    sharding = "owner" if (world > 1 and args.pool == "owner") else "replicated"
    tcfg = TrainConfig(batch_size=Bg, pool_size=1024, long_rollout_prob=1.0 if regime == "long" else 0.0, fire="philox",
                       rollout_impl=args.rollout_impl, damage=dmg, pool_sharding=sharding)
    tr = GraphNCATrainer(model, target, tcfg)
    # pool of mixed ages (SURVEY 8d C3): every slot rolled 0..160 steps from its seed, no grad
    n_slots = tr.pool.pool.shape[0]
    chunk = min(256, n_slots)
    with torch.no_grad():
        for i0 in range(0, n_slots, chunk):
            ages = [random.randint(0, 160) for _ in range(chunk)]
            sched = make_schedule(model, chunk, 40, 40, max(ages), fire_rate=0.6, steps=ages, fire="philox", seed=77 + i0 + 1000 * rank)
            tr.pool.pool[i0:i0 + chunk] = rollout(model, tr.pool.pool[i0:i0 + chunk].contiguous(), sched)
    flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device=dev)
    for _ in range(warmup):
        tr.train_step(epoch=300)
    torch.cuda.synchronize()
    import gc
    gc.collect()
    gc.freeze()          # as in the forward e2e loop: no full-heap collection on one of N ranks inside a timed all-reduce window
    if world > 1:
        dist.barrier()
    sampler = ClockSampler(local_rank); sampler.start()
    launches0 = lib.gnca_launch_count()
    evs, updates, steps_sum = [], 0, 0
    for i in range(steps):
        flush.fill_(float(i))
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        out = tr.train_step(epoch=300)
        e1.record()
        evs.append((e0, e1))
        updates += out["cell_updates"]; steps_sum += int(out["steps"].max())
    torch.cuda.synchronize()
    launches = lib.gnca_launch_count() - launches0
    sampler.stop_flag = True; sampler.join()
    if world > 1:
        dist.barrier()
    t = torch.tensor([sum(a.elapsed_time(b) for a, b in evs)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    dev_ms = float(t.item())
    # end to end: the same call + the device->host read of the step's result (the loss) inside the wall-clock region
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    t0 = time.perf_counter()
    upd2 = 0
    for i in range(steps):
        out = tr.train_step(epoch=300)
        loss = float(out["loss"])                      # D2H of the step's result
        upd2 += out["cell_updates"]
    torch.cuda.synchronize()
    t = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_s = float(t.item())
    Tavg = steps_sum / steps
    e2e = {"value": upd2 / e2e_s, "unit": "cell-updates/s", "ms_per_step": e2e_s / steps * 1e3,
           "h2d_bytes_per_step": int(Tavg * 24 + Bg // world * 4), "d2h_bytes_per_step": int(Bg * 8 + 4),
           "note": "train_step() + float(loss); the pool lives on the device as in the reference (pool.py keeps device tensors)"}
    # per-kernel device time (library event hook)
    lib.gnca_profile_enable(1)
    nprof = min(steps, 5)
    upd3 = 0
    for i in range(nprof):
        upd3 += tr.train_step(epoch=300)["cell_updates"]
    torch.cuda.synchronize()
    lib.gnca_profile_enable(0)
    per_kernel = {}
    for kid, kname in ((0, "k_update"), (1, "k_apply"), (2, "k_rep_fwd"), (3, "k_rep_wgrad"), (6, "k_rep_bwd")):
        ms, n = ctypes.c_double(0), ctypes.c_ulonglong(0)
        lib.gnca_profile_read(kid, ctypes.byref(ms), ctypes.byref(n))
        if n.value:
            per_kernel[kname] = (ms.value, n.value)
    kernels_ms = {k: {"ms_per_step": v[0] / nprof, "launches_per_step": v[1] / nprof} for k, v in per_kernel.items()}
    roof = None
    if per_kernel:
        kname = max(per_kernel, key=lambda k: per_kernel[k][0])
        ms, n = per_kernel[kname]
        cfg3 = {"name": "c3", "train": True, "flop": FLOP_FWDBWD_GRAPH_S, "C": 16, "H": 40, "W": 40, "hidden": 128, "B": Bg // world}
        roof = make_roofline(cfg3, kname, ms, n, nprof, upd3 / world / nprof, sampler.result(), kernels_ms, dev_ms / steps,
                             Bg // world * 16 * 1600, int(Tavg), args)
    return {"metric": "graph-NCA cell-updates/s (fwd+bwd)", "value": updates / (dev_ms * 1e-3), "unit": "cell-updates/s",
            "ms_per_step": dev_ms / steps, "n_gpus": world, "scaling": scaling, "regime": regime, "e2e": e2e,
            "gpu_launches": int(launches), "steps_timed": steps, "mean_T": Tavg, "clocks": sampler.result(),
            "config": {"workload": "configs[%d]: GraphNCATrainer.train_step, %s regime%s" % (3 if damage else 2, regime,
                                                                                           ", damage policy on every step" if damage else ""),
                       "global_batch": Bg, "B_per_gpu": Bg // world, "pool": 1024, "steps": "randint(48,80)" if regime == "short" else "randint(200,400)",
                       "fire_rate": "U(0.5,0.9) per step", "message_every": 3, "fire_rng": "in-kernel philox (per-rank stream offset)",
                       "pool_sharding": sharding,
                       "parallelism": f"dp{world}: batch sharded, NCCL all-reduce of the 9,169-float gradient + all-gather of the per-sample losses"
                                      + ("" if sharding == "owner" or world == 1 else " and of the final states (replicated pool)")},
            "roofline": roof}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c2")
    ap.add_argument("--rollout-impl", default="auto", choices=["auto", "streaming", "resident", "banded"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--pool", default="owner", choices=["owner", "replicated"],
                    help="N > 1 training: pool partitioned over the ranks (default) or replicated with a state all-gather")
    ap.add_argument("--no-train-extra", action="store_true", help="skip the fwd+bwd (c3) measurement of the default run")
    ap.add_argument("--T", type=int, default=0, help="development: override the number of CA steps per rollout")
    ap.add_argument("--B", type=int, default=0, help="development: override the per-GPU batch")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step computed (rank 0) as DIR/<name>.npy, float32, 64 MB at most")
    args = ap.parse_args()
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    cfg = workload_cfg(args.workload)
    if args.T > 0:
        cfg["T"] = args.T
    if args.B > 0:
        cfg["B"] = args.B

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))

    if args.impl == "reference":
        run_reference_arm(args, cfg, rank)
        return

    import torch.distributed as dist
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    res = run_workload(cfg, args, world, rank, local_rank, dev, args.steps, args.warmup)
    C_, H, W, B, T = res["dims"]
    value, e2e, launches, roof, data = res["value"], res["e2e"], res["launches"], res["roofline"], res["data"]
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, res["outputs"])

    # the other half of the metric ("fwd, fwd+bwd"): BASELINE configs[2] (and, for N > 1, configs[3]) through the trainer
    train = None
    if args.workload == "c2" and not args.no_train_extra:
        ts = args.steps
        train = {"short": run_trainer(args, world, rank, local_rank, dev, ts, 3, "short", "weak"),
                 "long": run_trainer(args, world, rank, local_rank, dev, ts, 3, "long", "weak")}
        if world > 1:    # configs[3]: damage curriculum, global batch 32 sharded 16 / 8 / 4 per GPU (strong) and 32 per GPU (weak)
            train["damage_weak"] = run_trainer(args, world, rank, local_rank, dev, ts, 3, "short", "weak", damage=True)
            train["damage_strong"] = run_trainer(args, world, rank, local_rank, dev, ts, 3, "short", "strong", damage=True)
        else:
            train["damage_weak"] = run_trainer(args, world, rank, local_rank, dev, ts, 3, "short", "weak", damage=True)

    cpu = eager = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline and not cfg["train"] and not cfg.get("classic"):
        cpu = cpu_forward_baseline(cfg)
        eager = gpu_eager_forward(cfg, dev)
        if train is not None:
            import bench_ref
            r = bench_ref.time_train_step("cpu", batch=32, steps=1)
            train["cpu_baseline"] = {"value": r["value"], "unit": "cell-updates/s", "cores": r["cores"], "kind": r["kind"],
                                     "sample": r["sample"] + f"; {r['seconds_per_step']:.1f} s"}
            r = bench_ref.time_train_step(dev, batch=32, steps=3, warmup=1)
            train["gpu_eager"] = {"value": r["value"], "unit": "cell-updates/s", "kind": r["kind"] + " modules + torch.optim.Adam, torch eager on cuda",
                                  "ms_per_step": r["seconds_per_step"] * 1e3, "sample": r["sample"]}

    if rank == 0:
        line = {"metric": "graph-NCA cell-updates/s (%s)" % ("fwd+bwd" if cfg["train"] else "fwd"), "value": value,
                "unit": "cell-updates/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": res["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "f32", "data": data,
                "config": {"workload": cfg["name"], "B_per_gpu": B, "T": T, "grid": [H, W], "channels": C_,
                           "hidden": cfg["hidden"], "fire_rate": cfg["fire_rate"], "offsets_per_step": 8,
                           "graph_shift": "torus", "fire_rng": "in-kernel philox", "rollout_impl": args.rollout_impl,
                           "l2": "flushed between timed iterations (256 MiB fill)", "parallelism": f"dp{world} batch-sharded, no collective"},
                "e2e": e2e, "gpu_launches": int(launches), "clocks": res["clocks"], "roofline": roof,
                "cpu_baseline": cpu, "gpu_eager": eager, "fwd_bwd": train}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()

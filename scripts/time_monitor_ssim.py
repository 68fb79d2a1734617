"""Cost of SSIM curves from one rollout call (monitor_rollout(..., ssim=True)), timed with CUDA events around whole
calls, the arms alternated within each of three rounds (the spread over the rounds is reported).

Arms, per configuration: the plain rollout, monitor_rollout without SSIM, monitor_rollout with SSIM, and
record_rollout followed by utils.metrics.ssim_rgb on every kept frame (the way to get the curve without ssim=True).

1. C2, bench.py's default shape (graph NCA, 16 channels, 40x40, B = 8, T = 96, torus, trained weights, replicated-state
   kernel), a frame every S in {1, 8, 32} steps.
2. The checkpoint sweep of DESIGN 3.12: 148 zero-pad models at B = 1, 40x40, T = 1000, damage at t = 500, S = 10, in
   one stacked call (the record arm is the stacked record_rollout).
3. c5s, 256x256x32, B = 16, T = 200, damage at t = 100 (streaming kernels, tensor-core update), S in {10, 50}.
Peak memory (torch.cuda.max_memory_allocated above what the inputs hold) of every arm.

Prints the card's name, power limit and max SM clock with the numbers and writes them to
profiles/r10_monitor_ssim.json (or --out).  Needs a CUDA device; it has no CPU path.

    python scripts/time_monitor_ssim.py [--reps 10] [--out profiles/r10_monitor_ssim.json]
"""
from __future__ import annotations

import argparse
import json
import os
import random
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import graph_neural_cellular_automata_b200 as G  # noqa: E402
from graph_neural_cellular_automata_b200.rollout import (make_schedule, monitor_rollout, record_rollout,  # noqa: E402
                                                         rollout)
from graph_neural_cellular_automata_b200.utils import metrics as UM  # noqa: E402
from graph_neural_cellular_automata_b200.utils.nca_init import make_seed  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else torch.cuda.get_device_name()


def time_ms(fn, reps, warmup=1):
    """mean wall time of fn() between two CUDA events, over `reps` calls after `warmup` untimed ones"""
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / reps


def peak_bytes(fn):
    """peak allocation of one fn() call above what was allocated before it"""
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    out = fn()
    torch.cuda.synchronize()
    peak = torch.cuda.max_memory_allocated() - base
    del out
    return peak


def record_and_ssim(m, x0, s, tgt, S, impl):
    tr = record_rollout(m, x0, s, every=S, impl=impl)
    return torch.stack([UM.ssim_rgb(f, tgt) for f in tr.states]), tr.x_T


def run_case(m, x0, s, tgt, strides, impl, reps, rounds=3, record=True):
    arms = {"plain": lambda: rollout(m, x0, s, impl=impl)}
    for S in strides:
        arms[f"monitor_S{S}"] = (lambda S=S: monitor_rollout(m, x0, s, tgt, every=S, impl=impl))
        arms[f"monitor_ssim_S{S}"] = (lambda S=S: monitor_rollout(m, x0, s, tgt, every=S, impl=impl, ssim=True))
        if record:
            arms[f"record+ssim_rgb_S{S}"] = (lambda S=S: record_and_ssim(m, x0, s, tgt, S, impl))
    times = {k: [] for k in arms}
    with torch.no_grad():
        for _ in range(rounds):
            for k, fn in arms.items():
                times[k].append(time_ms(fn, reps))
        mem = {k: peak_bytes(fn) for k, fn in arms.items()}
    return times, mem


def c2(reps, params):
    torch.manual_seed(42); random.seed(42)
    m = G.NeuralCAGraph(16, update_hidden=128, img_size=40, update_gain=0.05, alpha_thr=0.12, message_gain=0.25,
                        hidden_only=True, graph_zero_padded_shift=False)
    m.load_state_dict(params, strict=False)
    m = m.cuda()
    B, H, W, T = 8, 40, 40, 96
    with torch.no_grad():
        x0 = make_seed(16, H, B, device="cuda")
        x0 = rollout(m, x0, make_schedule(m, B, H, W, 48, fire_rate=0.6, seed=1), impl="streaming")
        tgt = UM.premultiply(x0[:1])[0].contiguous()
    s = make_schedule(m, B, H, W, T, fire_rate=0.5, seed=2)
    return run_case(m, x0, s, tgt, (1, 8, 32), "resident", reps)


def sweep(reps, params):
    M, H, W, T = 148, 40, 40, 1000
    ms = []
    for i in range(M):
        m = G.NeuralCAGraph(16, update_hidden=128, img_size=H, update_gain=0.05, alpha_thr=0.12, message_gain=0.25,
                            hidden_only=True, graph_zero_padded_shift=True)
        m.load_state_dict(params, strict=False)
        if i:
            g = torch.Generator().manual_seed(i)
            with torch.no_grad():
                for name, p in m.named_parameters():
                    if "perception" not in name and p.requires_grad:
                        p.add_(0.03 * p.abs().mean() * torch.randn(p.shape, generator=g))
        ms.append(m.cuda())
    with torch.no_grad():
        xg = rollout(ms[0], make_seed(16, H, 1, device="cuda"), make_schedule(ms[0], 1, H, W, 64, fire_rate=0.5, seed=1))
    x0 = xg.expand(M, -1, -1, -1).contiguous()
    tgt = UM.premultiply(xg)[0].contiguous()
    dmg = torch.ones(M, 16, H, W, device="cuda")
    dmg[:, :, H // 4:H // 2, H // 4:H // 2] = 0.0
    random.seed(3)
    s = make_schedule(ms[0], M, H, W, T, fire_rate=0.5, seed=4, damage=dmg, damage_step=500)
    return run_case(ms, x0, s, tgt, (10,), "auto", reps)


def c5s(reps):
    torch.manual_seed(5); random.seed(5)
    C, H, B, T = 32, 256, 16, 200
    m = G.NeuralCAGraph(C, update_hidden=128, img_size=H, update_gain=0.1, alpha_thr=0.1, message_gain=0.3,
                        hidden_only=True, graph_zero_padded_shift=False)
    with torch.no_grad():
        m.update_net[2].weight.normal_(0, 0.05)
    m = m.cuda()
    yy, xx = torch.meshgrid(torch.arange(H), torch.arange(H), indexing="ij")
    disk = (((yy - H / 2) ** 2 + (xx - H / 2) ** 2) < (0.3 * H) ** 2).float()
    x0 = (torch.rand(B, C, H, H) * disk).cuda()
    tgt = UM.premultiply(x0[:1])[0].contiguous()
    dmg = torch.ones(B, C, H, H, device="cuda")
    dmg[:, :, H // 3:H // 2, H // 3:H // 2] = 0.0
    s = make_schedule(m, B, H, H, T, fire_rate=0.5, seed=3, damage=dmg, damage_step=100)
    return run_case(m, x0, s, tgt, (10, 50), "streaming", reps)


def report(name, times, mem):
    base = sum(times["plain"]) / len(times["plain"])
    print(name)
    for k, v in times.items():
        mean = sum(v) / len(v)
        spread = (max(v) - min(v)) / mean
        print(f"  {k:24s} {' '.join(f'{x:9.3f}' for x in v)} ms  spread {100 * spread:5.1f} %  ({mean / base:.3f}x plain)"
              f"   peak {mem[k] / 1e6:10.1f} MB")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r10_monitor_ssim.json"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("time_monitor_ssim.py needs a CUDA device")
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from conftest import load_params      # tests/conftest.py: the trained-weight fixture loader
    params = load_params("weights_graph_ep960.npz")
    dev = card()
    res = {"card": dev}
    for name, fn, title in [
            ("c2", lambda: c2(args.reps, params), "C2: 40x40x16, B=8, T=96, torus, resident kernel"),
            ("sweep", lambda: sweep(max(2, args.reps // 5), params),
             "sweep: 148 zero-pad models, B=1, 40x40, T=1000, damage at t=500, one stacked call"),
            ("c5s", lambda: c5s(max(2, args.reps // 5)), "c5s: 256x256x32, B=16, T=200, damage at t=100, streaming")]:
        t, m = fn()
        report(f"[{dev}] {title}: ms per call, three rounds", t, m)
        res[f"{name}_ms"] = t
        res[f"{name}_peak_bytes"] = m
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()

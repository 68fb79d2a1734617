"""Cost of per-frame quality curves from one rollout call (rollout.monitor_rollout / gnca_rollout_metrics), timed with
CUDA events around whole calls, the arms alternated within each of two rounds.

1. C2, bench.py's default shape (graph NCA, 16 channels, 40x40, B = 8, T = 96, torus, trained weights, resident
   kernel): the plain rollout against monitor_rollout every S in {1, 8, 32} steps, and against record_rollout at the
   same S followed by utils.metrics on the frames (the way to get the curve without this entry point).
2. c5s, 256x256x32, B = 16, T = 200, damage at t = 100 (streaming kernels, tensor-core update): the plain rollout
   against monitor_rollout every S in {1, 10, 50}, and record_rollout + utils.metrics at the same S.
3. Peak memory (torch.cuda.max_memory_allocated above what the inputs hold) of monitor_rollout against
   record_rollout + utils.metrics, at every S above.

Prints the card's name and power limit with the numbers and writes them to profiles/r07_monitor.json (or --out).
Needs a CUDA device; it has no CPU path.

    python scripts/time_monitor.py [--reps 20] [--out profiles/r07_monitor.json]
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


def time_ms(fn, reps, warmup=2):
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


def record_and_reduce(m, x0, s, tgt, S, impl):
    """the curve from kept frames: record_rollout, then utils.metrics on each frame"""
    tr = record_rollout(m, x0, s, every=S, impl=impl)
    st = tr.states
    F, B = st.shape[:2]
    pm = UM.premultiply(st.reshape(F * B, *st.shape[2:]))
    loss = ((pm - tgt.unsqueeze(0)) ** 2).mean(dim=(1, 2, 3)).reshape(F, B)
    psnr = torch.stack([UM.psnr_rgb(st[f], tgt) for f in range(F)])
    pp = torch.stack([UM.pixel_perfect(st[f], tgt) for f in range(F)])
    alive = (st[:, :, 3] > m.alpha_thr).sum(dim=(2, 3))
    return loss, psnr, pp, alive, tr.x_T


def run_case(m, x0, s, tgt, strides, impl, reps, rounds=2):
    arms = {"plain": lambda: rollout(m, x0, s, impl=impl)}
    for S in strides:
        arms[f"monitor_S{S}"] = (lambda S=S: monitor_rollout(m, x0, s, tgt, every=S, impl=impl))
        arms[f"record+metrics_S{S}"] = (lambda S=S: record_and_reduce(m, x0, s, tgt, S, impl))
    times = {k: [] for k in arms}
    with torch.no_grad():
        for _ in range(rounds):
            for k, fn in arms.items():
                times[k].append(time_ms(fn, reps))
        mem = {k: peak_bytes(fn) for k, fn in arms.items()}
    return times, mem


def c2(reps):
    from conftest import load_params      # tests/conftest.py: the trained-weight fixture loader
    torch.manual_seed(42); random.seed(42)
    m = G.NeuralCAGraph(16, update_hidden=128, img_size=40, update_gain=0.05, alpha_thr=0.12, message_gain=0.25,
                        hidden_only=True, graph_zero_padded_shift=False)
    m.load_state_dict(load_params("weights_graph_ep960.npz"), strict=False)
    m = m.cuda()
    B, H, W, T = 8, 40, 40, 96
    with torch.no_grad():
        x0 = make_seed(16, H, B, device="cuda")
        grow = make_schedule(m, B, H, W, 48, fire_rate=0.6, seed=1)
        x0 = rollout(m, x0, grow, impl="streaming")
        tgt = UM.premultiply(x0[:1])[0].contiguous()
    s = make_schedule(m, B, H, W, T, fire_rate=0.5, seed=2)
    return run_case(m, x0, s, tgt, (1, 8, 32), "resident", reps)


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
    return run_case(m, x0, s, tgt, (1, 10, 50), "streaming", reps)


def report(name, times, mem):
    base = sum(times["plain"]) / len(times["plain"])
    print(name)
    for k, v in times.items():
        mean = sum(v) / len(v)
        print(f"  {k:22s} {' '.join(f'{x:9.3f}' for x in v)} ms   ({mean / base:.3f}x plain)   peak {mem[k] / 1e6:10.1f} MB")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r07_monitor.json"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("time_monitor.py needs a CUDA device")
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    dev = card()
    t1, m1 = c2(args.reps)
    report(f"[{dev}] C2: 40x40x16, B=8, T=96, torus, resident kernel: ms per call, two rounds", t1, m1)
    t2, m2 = c5s(max(2, args.reps // 10))
    report(f"[{dev}] c5s: 256x256x32, B=16, T=200, damage at t=100, streaming kernels: ms per call, two rounds", t2,
           m2)
    res = {"card": dev, "c2_ms": t1, "c2_peak_bytes": m1, "c5s_ms": t2, "c5s_peak_bytes": m2}
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()

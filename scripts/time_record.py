"""Cost of recording a rollout (rollout.record_rollout / gnca_rollout_record), timed with CUDA events.

1. bench.py's default shape (graph NCA, 16 channels, 40x40, B = 8, T = 96, torus, trained weights, resident kernel):
   the plain rollout against recordings every S in {1, 8, 32} steps, without and with attention maps, and against the
   loop a user runs without this entry point: T calls of model.step(..., return_attention=True).
2. 256x256x32, B = 16, T = 200, damage at t = 100, every 50 steps with attention (streaming kernels).

Prints the card's name and power limit with the numbers, and one JSON line.  Needs a CUDA device; it has no CPU path.

    python scripts/time_record.py [--reps 20]
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
from graph_neural_cellular_automata_b200.rollout import make_schedule, record_rollout, rollout  # noqa: E402
from graph_neural_cellular_automata_b200.utils.nca_init import make_seed  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else torch.cuda.get_device_name()


def time_ms(fn, reps, warmup=3):
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
    s = make_schedule(m, B, H, W, T, fire_rate=0.5, seed=2)
    offs = s.offsets.cpu().numpy()
    chosen = [[tuple(int(v) for v in o) for o in offs[t]] for t in range(T)]
    fu = torch.rand(T, B, 1, H, W, device="cuda")
    out = {}
    with torch.no_grad():
        out["plain"] = time_ms(lambda: rollout(m, x0, s, impl="resident"), reps)
        for S in (1, 8, 32):
            for att in (False, True):
                out[f"S{S}" + ("_attn" if att else "")] = time_ms(
                    lambda: record_rollout(m, x0, s, every=S, attention=att, impl="resident"), reps)

        def step_loop():
            x = x0
            for t in range(T):
                x, _ = m.step(x, 0.5, fire_u=fu[t], chosen=chosen[t], return_attention=True)
        out["step_loop_attn"] = time_ms(step_loop, max(3, reps // 4))
    return out


def large(reps):
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
    dmg = torch.ones(B, C, H, H, device="cuda")
    dmg[:, :, H // 3:H // 2, H // 3:H // 2] = 0.0
    s = make_schedule(m, B, H, H, T, fire_rate=0.5, seed=3, damage=dmg, damage_step=100)
    with torch.no_grad():
        return {"plain": time_ms(lambda: rollout(m, x0, s), reps, warmup=1),
                "S50_attn": time_ms(lambda: record_rollout(m, x0, s, every=50, attention=True), reps, warmup=1)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("time_record.py needs a CUDA device")
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    dev = card()
    r1 = c2(args.reps)
    print(f"[{dev}] 40x40x16, B=8, T=96, torus, resident kernel: ms per rollout call")
    for k, v in r1.items():
        print(f"  {k:16s} {v:9.3f} ms   ({v / r1['plain']:.2f}x plain)")
    r2 = large(max(2, args.reps // 10))
    print(f"[{dev}] 256x256x32, B=16, T=200, damage at t=100, streaming kernels: ms per rollout call")
    for k, v in r2.items():
        print(f"  {k:16s} {v:9.3f} ms   ({v / r2['plain']:.2f}x plain)")
    print(json.dumps({"card": dev, "c2_ms": r1, "large_ms": r2}))


if __name__ == "__main__":
    main()

"""Cost of per-model targets (a target sweep: one model per image).

1. Training: one iteration of the stacked resident BPTT as PopulationTrainer runs it on the device (forward with
   records, premultiplied loss, backward, M normalise + Adam steps) with one target per model ("targets") against the
   same stack with one shared target ("shared"), and against M sequential single-model iterations of
   GraphNCATrainer(fire="philox")'s device work on B samples each, each towards its own target ("sequential").
   40x40x16 torus graph NCA with the trained ep960 weights perturbed by seed, x0 a grown pattern, fire rate 0.5 on the
   Philox stream, T = 64, M in {2, 4, 8}, B per model in {8, 16}.
2. Monitoring: the sweep of DESIGN 3.12 (148 zero-pad models, B = 1, 40x40, T = 1000, damage at t = 500, a frame every
   10 steps), monitor_rollout with a [148, 4, H, W] target against the same call with one [4, H, W] target, with and
   without SSIM.

The arms alternate within each of three rounds after a warm-up of every arm; each is timed with CUDA events.  The
targets are seeded shifts and flips of the gecko surrogate in tests/golden.

With --bench-base DIR (a built tree of the parent commit), it also runs `bench.py --gpus 1` (default workload) and
`bench.py --gpus 1 --workload c3` from this tree and from DIR, alternated over --bench-rounds rounds (default 3) of
--bench-steps timed steps each (default 200: bench's own 20 steps are a window of under 20 ms at the default workload,
where one disturbed run moves the figure by several per cent), and keeps their JSON lines.

Prints the card's name, power limit and max SM clock with the numbers and writes them to
profiles/r11_target_sweep.json (or --out).  Needs a CUDA device; it has no CPU path.

    python scripts/time_target_sweep.py [--bench-base DIR] [--bench-steps N] [--bench-rounds R]
                                        [--out profiles/r11_target_sweep.json]
"""
from __future__ import annotations

import argparse
import json
import os
import random
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import graph_neural_cellular_automata_b200 as G  # noqa: E402
from graph_neural_cellular_automata_b200.rollout import (make_schedule, monitor_rollout, rollout,  # noqa: E402
                                                         rollout_bwd_raw, rollout_fwd_raw, rollout_models_bwd_raw,
                                                         rollout_models_fwd_raw)
from graph_neural_cellular_automata_b200.training.optim import FusedNormalizedAdam  # noqa: E402
from graph_neural_cellular_automata_b200.training.trainer import premult_loss  # noqa: E402
from graph_neural_cellular_automata_b200.utils.nca_init import make_seed  # noqa: E402

H = W = 40


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else torch.cuda.get_device_name()


def models(n, torus, params):
    out = []
    for i in range(n):
        m = G.NeuralCAGraph(16, update_hidden=128, img_size=H, update_gain=0.05, alpha_thr=0.12, message_gain=0.25,
                            hidden_only=True, graph_zero_padded_shift=not torus)
        m.load_state_dict(params, strict=False)
        if i:
            g = torch.Generator().manual_seed(i)
            with torch.no_grad():
                for name, p in m.named_parameters():
                    if "perception" not in name and p.requires_grad:
                        p.add_(0.03 * p.abs().mean() * torch.randn(p.shape, generator=g))
        out.append(m.cuda())
    return out


def targets(M):
    """[M, 4, H, W]: the gecko surrogate, then seeded shifts and flips of it"""
    base = torch.from_numpy(np.load(os.path.join(ROOT, "tests", "golden", "target_gecko_surrogate.npy"))).float()
    g = torch.Generator().manual_seed(0)
    out = [base]
    for i in range(1, M):
        t = torch.roll(base, shifts=(int(torch.randint(-5, 6, (1,), generator=g)),
                                     int(torch.randint(-5, 6, (1,), generator=g))), dims=(1, 2))
        out.append(t.flip(2) if i % 2 else t)
    return torch.stack(out).cuda().contiguous()


def time_ms(fn, reps=1):
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / reps


def alternate(arms, rounds=3, reps=1):
    for fn in arms.values():
        fn()                                               # warm-up: modules, allocator, launch configuration
    times = {k: [] for k in arms}
    for _ in range(rounds):
        for k, fn in arms.items():
            times[k].append(time_ms(fn, reps))
    return times


def train_row(M, B, T, ms, opts, x_grown, tg):
    n = M * B
    desc = ms[0].model_desc()
    x0 = x_grown[:1].expand(n, -1, -1, -1).contiguous()
    random.seed(3)
    s = make_schedule(ms[0], n, H, W, T, fire_rate=0.5, seed=4)
    random.seed(3)
    s_one = make_schedule(ms[0], B, H, W, T, fire_rate=0.5, seed=4)
    tgt_m = tg[:M].contiguous()

    def sequential():
        for i in range(M):
            desc_i, packed = ms[i].model_desc(), ms[i].packed_weights()
            xT, hist = rollout_fwd_raw(desc_i, packed, x0[i * B:(i + 1) * B], s_one, history=True, impl=0,
                                       keep_x=False)
            _, g = premult_loss(xT, tgt_m[i], 1.0 / B)
            _, gflat = rollout_bwd_raw(desc_i, packed, hist, s_one, g, impl=0)
            opts[i].step(gflat, lr=1e-4)

    def stacked(tgt):
        def run():
            packed = torch.stack([m.packed_weights() for m in ms[:M]])
            xT, hist = rollout_models_fwd_raw(desc, packed, x0, s)
            _, g = premult_loss(xT, tgt, 1.0 / B)
            _, gflat = rollout_models_bwd_raw(desc, packed, hist, s, g)
            for i in range(M):
                opts[i].step(gflat[i], lr=1e-4)
        return run

    times = alternate({"shared": stacked(tgt_m[0]), "targets": stacked(tgt_m), "sequential": sequential})
    best = {k: min(v) for k, v in times.items()}
    return {"M": M, "B": B, "T": T, "ms": times, "cell_updates_per_s": {k: n * H * W * T / (v / 1e3)
                                                                         for k, v in best.items()},
            "targets_over_shared": best["targets"] / best["shared"],
            "sequential_over_targets": best["sequential"] / best["targets"]}


def sweep(params):
    M, T, S = 148, 1000, 10
    ms = models(M, False, params)
    with torch.no_grad():
        xg = rollout(ms[0], make_seed(16, H, 1, device="cuda"), make_schedule(ms[0], 1, H, W, 64, fire_rate=0.5, seed=1))
    x0 = xg.expand(M, -1, -1, -1).contiguous()
    tg = targets(M)
    dmg = torch.ones(M, 16, H, W, device="cuda")
    dmg[:, :, H // 4:H // 2, H // 4:H // 2] = 0.0
    random.seed(3)
    s = make_schedule(ms[0], M, H, W, T, fire_rate=0.5, seed=4, damage=dmg, damage_step=500)
    out = {}
    for ssim in (False, True):
        def arm(tgt):
            def run():
                with torch.no_grad():
                    monitor_rollout(ms, x0, s, tgt, every=S, ssim=ssim)
            return run
        out["ssim" if ssim else "metrics"] = alternate({"shared": arm(tg[0]), "targets": arm(tg)}, reps=3)
    return out


def bench_ab(base, rounds, steps):
    """bench.py default and --workload c3 from this tree and from `base`, alternated; the JSON result lines"""
    out = []
    for r in range(rounds):
        for workload in (None, "c3"):
            for name, tree in (("parent", base), ("this", ROOT)):
                cmd = [sys.executable, "bench.py", "--gpus", "1", "--steps", str(steps), "--warmup", "10",
                       "--no-cpu-baseline"]
                if workload:
                    cmd += ["--workload", workload]
                p = subprocess.run(cmd, cwd=tree, capture_output=True, text=True)
                line = [v for v in p.stdout.splitlines() if v.startswith("{")]
                res = json.loads(line[-1]) if line else {"error": p.stderr[-2000:]}
                out.append({"round": r, "tree": name, "workload": workload or "default", "result": res})
                print(f"bench {name:6s} {workload or 'default':7s}: {res.get('value', res.get('error'))}", flush=True)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--ms", default="2,4,8")
    ap.add_argument("--bs", default="8,16")
    ap.add_argument("--T", type=int, default=64)
    ap.add_argument("--bench-base", default=None)
    ap.add_argument("--bench-steps", type=int, default=200)
    ap.add_argument("--bench-rounds", type=int, default=3)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r11_target_sweep.json"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("time_target_sweep.py needs a CUDA device")
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from conftest import load_params      # tests/conftest.py: the trained-weight fixture loader
    params = load_params("weights_graph_ep960.npz")
    Ms = [int(v) for v in args.ms.split(",")]
    Bs = [int(v) for v in args.bs.split(",")]
    dev = card()
    res = {"card": dev, "train_setup": "40x40x16 torus graph NCA, fire rate 0.5 (Philox), T = %d, one training "
           "iteration: forward with records, premultiplied loss, resident BPTT, normalise + Adam" % args.T,
           "train": [], "sweep_setup": "148 zero-pad models, B = 1, 40x40, T = 1000, damage at t = 500, S = 10"}
    pool = models(max(Ms), True, params)
    opts = [FusedNormalizedAdam(m, lr=1e-4, weight_decay=1e-5) for m in pool]
    with torch.no_grad():
        x_grown = rollout(pool[0], make_seed(16, H, 1, device="cuda"),
                          make_schedule(pool[0], 1, H, W, 64, fire_rate=0.5, seed=1))
    tg = targets(max(Ms))
    for B in Bs:
        for M in Ms:
            r = train_row(M, B, args.T, pool, opts, x_grown, tg)
            res["train"].append(r)
            print(f"[{dev}] train M={M} B={B:2d}: " + ", ".join(
                f"{k} {' '.join(f'{v:7.2f}' for v in r['ms'][k])} ms" for k in r["ms"]) +
                f"; targets/shared {r['targets_over_shared']:.3f}, sequential/targets "
                f"{r['sequential_over_targets']:.2f}x", flush=True)
    del pool, opts
    torch.cuda.empty_cache()
    res["sweep"] = sweep(params)
    for k, v in res["sweep"].items():
        print(f"[{dev}] sweep {k}: " + ", ".join(f"{a} {' '.join(f'{t:8.2f}' for t in v[a])} ms" for a in v),
              flush=True)
    if args.bench_base:
        res["bench_ab_setup"] = {"steps": args.bench_steps, "warmup": 10, "rounds": args.bench_rounds}
        res["bench_ab"] = bench_ab(args.bench_base, args.bench_rounds, args.bench_steps)
    res["card_after"] = card()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()

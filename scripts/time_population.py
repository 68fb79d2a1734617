"""Cost of training M models: M sequential single-model training iterations against one stacked iteration.

An iteration is what PopulationTrainer / GraphNCATrainer(fire="philox") run per step on the device: the resident BPTT
forward with records, the premultiplied loss, the backward and the normalise + Adam step.  The sequential arm does that
M times, model by model, on B samples each (rollout_fwd_raw / rollout_bwd_raw, one FusedNormalizedAdam per model); the
stacked arm does it once on M * B samples (rollout_models_fwd_raw / rollout_models_bwd_raw, then the M Adam steps).

Setup: 40x40x16 graph NCA with the trained ep960 weights (torus and zero-padded shift), models perturbed by seed; x0 a
grown pattern; fire rate 0.5 with the in-kernel Philox stream; B per model in {8, 16, 32}, M in {1, 2, 4, 8}; T = 64 and
T = 300 where the stack's records fit (rollout.stack_bptt_bytes).  The arms alternate within each of three rounds after
a warm-up of both, each timed with CUDA events.  Reported per row: the times, cell updates per second
(M * B * H * W * T / time), and the peak memory of each arm.

With --bench-base DIR (a build of the parent commit), it also runs `bench.py --gpus 1` (default workload) and
`bench.py --gpus 1 --workload c3` from this tree and from DIR, alternated over two rounds, and keeps their JSON lines:
whether the single-model path got slower.

Prints the card's name, power limit and max SM clock with the numbers and writes them to
profiles/r09_population.json (or --out).  Needs a CUDA device; it has no CPU path.

    python scripts/time_population.py [--bench-base DIR] [--out profiles/r09_population.json]
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
from graph_neural_cellular_automata_b200.rollout import (make_schedule, rollout, rollout_bwd_raw,  # noqa: E402
                                                         rollout_fwd_raw, rollout_models_bwd_raw,
                                                         rollout_models_fwd_raw, stack_bptt_bytes)
from graph_neural_cellular_automata_b200.training.optim import FusedNormalizedAdam  # noqa: E402
from graph_neural_cellular_automata_b200.training.trainer import premult_loss  # noqa: E402
from graph_neural_cellular_automata_b200.utils import metrics as UM  # noqa: E402
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


def time_ms(fn):
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b)


def peak_bytes(fn):
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    base = torch.cuda.memory_allocated()
    fn()
    torch.cuda.synchronize()
    return torch.cuda.max_memory_allocated() - base


def row(torus, M, B, T, ms, opts, x_grown, tgt, rounds=3):
    n = M * B
    desc = ms[0].model_desc()
    try:
        stack_bptt_bytes(desc, n, H, W, T, 8)
    except ValueError as e:
        return {"model": "torus" if torus else "zeropad", "M": M, "B": B, "T": T, "skipped": str(e)}
    x0 = x_grown[:1].expand(n, -1, -1, -1).contiguous()
    random.seed(3)
    s = make_schedule(ms[0], n, H, W, T, fire_rate=0.5, seed=4)
    random.seed(3)          # the same offsets for the per-model iterations, on B samples each
    s_one = make_schedule(ms[0], B, H, W, T, fire_rate=0.5, seed=4)

    def sequential():
        for i in range(M):
            desc_i, packed = ms[i].model_desc(), ms[i].packed_weights()
            xT, hist = rollout_fwd_raw(desc_i, packed, x0[i * B:(i + 1) * B], s_one, history=True, impl=0,
                                       keep_x=False)
            _, g = premult_loss(xT, tgt, 1.0 / B)
            _, gflat = rollout_bwd_raw(desc_i, packed, hist, s_one, g, impl=0)
            opts[i].step(gflat, lr=1e-4)

    def stacked():
        packed = torch.stack([m.packed_weights() for m in ms[:M]])
        xT, hist = rollout_models_fwd_raw(desc, packed, x0, s)
        _, g = premult_loss(xT, tgt, 1.0 / B)
        _, gflat = rollout_models_bwd_raw(desc, packed, hist, s, g)
        for i in range(M):
            opts[i].step(gflat[i], lr=1e-4)

    arms = {"sequential": sequential, "stacked": stacked}
    for fn in arms.values():
        fn()                                               # warm-up: modules, allocator, launch configuration
    peak = {k: peak_bytes(fn) for k, fn in arms.items()}
    times = {k: [] for k in arms}
    for _ in range(rounds):
        for k, fn in arms.items():
            times[k].append(time_ms(fn))
    cells = n * H * W * T
    return {"model": "torus" if torus else "zeropad", "M": M, "B": B, "T": T, "ms": times, "peak_bytes": peak,
            "cell_updates_per_s": {k: cells / (min(v) / 1e3) for k, v in times.items()},
            "speedup": min(times["sequential"]) / min(times["stacked"])}


def bench_ab(base, rounds=2):
    """bench.py default and --workload c3 from this tree and from `base`, alternated; the JSON result lines"""
    out = []
    for r in range(rounds):
        for workload in (None, "c3"):
            for name, tree in (("parent", base), ("this", ROOT)):
                cmd = [sys.executable, "bench.py", "--gpus", "1", "--steps", "20", "--warmup", "5", "--no-cpu-baseline"]
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
    ap.add_argument("--ms", default="1,2,4,8")
    ap.add_argument("--bs", default="8,16,32")
    ap.add_argument("--ts", default="64,300")
    ap.add_argument("--bench-base", default=None)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r09_population.json"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("time_population.py needs a CUDA device")
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from conftest import load_params      # tests/conftest.py: the trained-weight fixture loader
    params = load_params("weights_graph_ep960.npz")
    Ms = [int(v) for v in args.ms.split(",")]
    Bs = [int(v) for v in args.bs.split(",")]
    Ts = [int(v) for v in args.ts.split(",")]
    dev = card()
    rows = []
    for torus in (True, False):
        pool = models(max(Ms), torus, params)
        opts = [FusedNormalizedAdam(m, lr=1e-4, weight_decay=1e-5) for m in pool]
        with torch.no_grad():
            x_grown = rollout(pool[0], make_seed(16, H, 1, device="cuda"),
                              make_schedule(pool[0], 1, H, W, 64, fire_rate=0.5, seed=1))
        tgt = UM.premultiply(x_grown[:1])[0].contiguous()
        for T in Ts:
            for B in Bs:
                for M in Ms:
                    r = row(torus, M, B, T, pool, opts, x_grown, tgt)
                    rows.append(r)
                    if "skipped" in r:
                        print(f"[{dev}] {r['model']:7s} T={T} M={M} B={B}: skipped ({r['skipped'][:80]})", flush=True)
                        continue
                    print(f"[{dev}] {r['model']:7s} T={T:3d} M={M} B={B:2d}: sequential "
                          f"{' '.join(f'{v:8.2f}' for v in r['ms']['sequential'])} ms, stacked "
                          f"{' '.join(f'{v:8.2f}' for v in r['ms']['stacked'])} ms, {r['speedup']:.2f}x, "
                          f"{r['cell_updates_per_s']['stacked']:.3e} cell-updates/s stacked, peak "
                          f"{r['peak_bytes']['sequential'] / 2**30:.2f} / {r['peak_bytes']['stacked'] / 2**30:.2f} GiB",
                          flush=True)
        del pool, opts
        torch.cuda.empty_cache()
    res = {"card": dev, "setup": "40x40x16 graph NCA, fire rate 0.5 (Philox), one training iteration: forward with "
                                 "records, premultiplied loss, resident BPTT, normalise + Adam", "rows": rows}
    if args.bench_base:
        res["bench_ab"] = bench_ab(args.bench_base)
    res["card_after"] = card()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()

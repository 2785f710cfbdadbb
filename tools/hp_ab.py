#!/usr/bin/env python
"""Per-agent hyper-parameter sets on the GPU: what they cost and what they buy.

cost:    k_run against k_run_hp holding one set (equal to the configuration) on C2 (1 M agents), C4 (2 M), C3 (4 M) and
         Taxi Q(lambda) on the lazy store (102 400): training steps/s from the kernels' CUDA events, the two engines
         alternating chunk by chunk in one process, `--reps` chunks each after a warm-up chunk.
benefit: the 64-point Taxi Q-learning grid (16 384 agents per point, 1000 episodes, `train(n, n/10)`) as ONE engine
         with 64 sets against 64 engines driven through the asynchronous train call on 8 streams; wall time each.
The card's name and power limit are read (nvidia-smi --query-gpu, read-only) in the same process.
    python tools/hp_ab.py --out DIR          (writes DIR/hp_cost.txt and DIR/hp_grid.txt)"""
import argparse
import importlib
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
abi = importlib.import_module("rl-rust_b200._abi")
W = importlib.import_module("rl-rust_b200.workloads")


def card():
    try:
        return subprocess.check_output(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], text=True).strip()
    except Exception as exc:   # noqa: BLE001
        return "nvidia-smi unavailable: %s" % exc


def one_set(h):
    return dict(learning_rate=h["lr"], discount_factor=h["gamma"], lambda_factor=h["lambda_"], initial_epsilon=h["eps0"],
                epsilon_decay=h["eps_decay"], final_epsilon=h["eps_final"], confidence_level=h["ucb_c"], default_value=h["default_q"])


COST = [("c2", 1 << 20, {}), ("c4", 1 << 21, {}), ("c3", 1 << 22, {}),
        ("taxi_qlambda_lazy", 102400, dict(env=3, agent=1, selector=0, policy=0, target=1, n_episodes=1000, chunk=100))]


def cost(reps, lines):
    for name, n, over in COST:
        w = dict(W.WORKLOADS[name]) if name in W.WORKLOADS else dict(over)
        c, h = W.combo(w, 0), W.workload_hyper(w)
        chunk = w["chunk"]
        store = 4 if name == "taxi_qlambda_lazy" else 0
        plain = W.make_engine(c, h, n, store_kind=store)
        hp = W.make_engine(c, h, n, store_kind=store)
        hp.set_hparams([one_set(h)], np.zeros(n, np.uint32))
        rates = {"k_run": [], "k_run_hp": []}
        ep = 0
        for r in range(reps + 1):
            for label, eng in (("k_run", plain), ("k_run_hp", hp)):
                res = eng.train(ep + chunk, max(1, w["n_episodes"] // 10), ep_begin=ep)
                if r:
                    rates[label].append(res["train_steps"] / (res["kernel_ms"] * 1e-3))
            ep += chunk
        a, b = np.array(rates["k_run"]), np.array(rates["k_run_hp"])
        lines.append("%-18s agents=%-8d store=%d  k_run %s  k_run_hp %s  ratio(median) %.4f" % (
            name, n, plain.store_kind(), " ".join("%.4g" % x for x in a), " ".join("%.4g" % x for x in b), np.median(b) / np.median(a)))
        print(lines[-1], flush=True)
        plain.close()
        hp.close()


def grid(lines, points=64, per_point=16384, n_ep=1000, streams=8):
    import torch
    w = W.WORKLOADS["c4"]
    c = W.combo(w, 0)
    h = W.hyper(n_ep)
    lrs = np.geomspace(0.01, 0.5, 8)
    exps = np.linspace(0.2, 0.9, 8)
    sets = [dict(learning_rate=float(lr), initial_epsilon=1.0, epsilon_decay=1.0 / (float(x) * n_ep)) for lr in lrs for x in exps][:points]
    # one engine, 64 sets
    eng = W.make_engine(c, h, points * per_point)
    eng.set_hparams(sets, np.repeat(np.arange(points, dtype=np.uint32), per_point))
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    res = eng.train(n_ep, n_ep // 10)
    t_one = time.perf_counter() - t0
    steps_one = res["train_steps"]
    sums_one = res["sums"]
    eng.close()
    # 64 engines, asynchronous calls on 8 streams
    strm = [torch.cuda.Stream() for _ in range(streams)]
    engines = []
    for g, s in enumerate(sets):
        hs = dict(h, lr=s["learning_rate"], eps_decay=s["epsilon_decay"])
        e = W.make_engine(c, hs, per_point, g * per_point)
        e.set_stream(strm[g % streams].cuda_stream)
        engines.append(e)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for e in engines:
        e.train(n_ep, n_ep // 10, wait=False)
    parts = [e.train_wait()[0] for e in engines]
    t_many = time.perf_counter() - t0
    steps_many = sum(p["train_steps"] for p in parts)
    same = all(np.array_equal(sums_one[:, g].view(np.uint64), parts[g]["sums"].view(np.uint64)) for g in range(points))
    for e in engines:
        e.close()
    lines.append("Taxi Q-learning grid: %d points x %d agents, %d episodes (train(n, n/10))" % (points, per_point, n_ep))
    lines.append("  one engine, %d sets:            %.3f s wall  (%d train steps, %.4g steps/s)" % (points, t_one, steps_one, steps_one / t_one))
    lines.append("  %d engines, async on %d streams: %.3f s wall  (%d train steps, %.4g steps/s)" % (points, streams, t_many, steps_many, steps_many / t_many))
    lines.append("  speed-up %.3fx; per-point sums bit-identical between the two: %s" % (t_many / t_one, same))
    print("\n".join(lines[-4:]), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True, help="directory for hp_cost.txt and hp_grid.txt")
    ap.add_argument("--reps", type=int, default=3)
    a = ap.parse_args()
    os.makedirs(a.out, exist_ok=True)
    head = ["card: %s" % card()]
    print(head[0], flush=True)
    lines = list(head) + ["training steps/s (train_steps / kernel_ms of each chunk), k_run and k_run_hp alternating"]
    cost(a.reps, lines)
    open(os.path.join(a.out, "hp_cost.txt"), "w").write("\n".join(lines) + "\n")
    lines = list(head)
    grid(lines)
    open(os.path.join(a.out, "hp_grid.txt"), "w").write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()

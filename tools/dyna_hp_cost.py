#!/usr/bin/env python
"""Dyna-Q under hyper-parameter sets on the GPU: what the per-set planning count costs and what it buys.

cost:    k_run<..., MODEL> against k_run_hp<..., MODEL> holding one set equal to the configuration and its count (10) on
         bench.py's `dyna` cell (CliffWalking one-step Q-learning, eps-greedy, Basic, 2^20 agents): training steps/s from
         the kernels' CUDA events, the two engines alternating chunk by chunk in one process, `--reps` chunks each after a
         warm-up chunk; medians and their spread (min .. max).
benefit: the CliffWalking grid planning_steps {0, 1, 5, 10, 50} x learning_rate {0.05, 0.1, 0.2, 0.5}, 16 384 agents per
         point, `train(n, n/10)`, as ONE engine with 20 sets and per-set counts against 20 engines (each with its count
         engine-wide) driven through the asynchronous train call on 8 streams; wall time each, and whether the per-point
         sums are bit-identical.
The card's name, power limit and SM clocks are read (nvidia-smi --query-gpu, read-only) in the same process.
    python tools/dyna_hp_cost.py --out DIR          (writes DIR/dyna_hp_cost.txt)"""
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
        return subprocess.check_output(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader"],
                                       text=True).strip()
    except Exception as exc:   # noqa: BLE001
        return "nvidia-smi unavailable: %s" % exc


def one_set(h):
    return dict(learning_rate=h["lr"], discount_factor=h["gamma"], lambda_factor=h["lambda_"], initial_epsilon=h["eps0"],
                epsilon_decay=h["eps_decay"], final_epsilon=h["eps_final"], confidence_level=h["ucb_c"], default_value=h["default_q"])


def cost(reps, lines):
    w = W.WORKLOADS["dyna"]
    c, h = W.combo(w, 0), W.workload_hyper(w)
    n, chunk, k = w["agents_per_gpu"], w["chunk"], w["planning_steps"]
    plain = W.make_engine(c, h, n)                                   # the model engine-wide: k_run<..., MODEL>
    hp = W.make_engine(c, dict(h, planning_steps=0), n)
    hp.set_hparams([one_set(h)], np.zeros(n, np.uint32))
    hp.set_planning_steps(np.array([k], np.uint32))                 # k_run_hp<..., MODEL>
    rates = {"k_run": [], "k_run_hp": []}
    same = True
    ep = 0
    for r in range(reps + 1):
        got = {}
        for label, eng in (("k_run", plain), ("k_run_hp", hp)):
            res = eng.train(ep + chunk, max(1, w["n_episodes"] // 10), ep_begin=ep)
            got[label] = res["sums"].reshape(chunk, 4)
            if r:
                rates[label].append(res["train_steps"] / (res["kernel_ms"] * 1e-3))
        same = same and np.array_equal(got["k_run"].view(np.uint64), got["k_run_hp"].view(np.uint64))
        ep += chunk
    a, b = np.array(rates["k_run"]), np.array(rates["k_run_hp"])
    lines.append("dyna cell: %s, %d agents, %d planning steps, chunks of %d episodes" % (w["desc"], n, k, chunk))
    lines.append("  k_run<..., MODEL>     steps/s %s  median %.4g  spread %.4g .. %.4g" % (" ".join("%.4g" % x for x in a), np.median(a), a.min(), a.max()))
    lines.append("  k_run_hp<..., MODEL>  steps/s %s  median %.4g  spread %.4g .. %.4g" % (" ".join("%.4g" % x for x in b), np.median(b), b.min(), b.max()))
    lines.append("  ratio hp/plain (medians) %.4f, range of chunk ratios %.4f .. %.4f; per-episode sums bit-identical: %s"
                 % (np.median(b) / np.median(a), (b / a).min(), (b / a).max(), same))
    print("\n".join(lines[-4:]), flush=True)
    plain.close()
    hp.close()


def grid(lines, per_point=16384, n_ep=100, streams=8):
    import torch
    w = W.WORKLOADS["dyna"]
    c = W.combo(w, 0)
    h = W.hyper(n_ep)
    steps = [0, 1, 5, 10, 50]
    lrs = [0.05, 0.1, 0.2, 0.5]
    pts = [(k, lr) for k in steps for lr in lrs]
    sets = [dict(learning_rate=lr) for _, lr in pts]
    eng = W.make_engine(c, h, len(pts) * per_point)
    eng.set_hparams(sets, np.repeat(np.arange(len(pts), dtype=np.uint32), per_point))
    eng.set_planning_steps(np.array([k for k, _ in pts], np.uint32))
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    res = eng.train(n_ep, n_ep // 10)
    t_one = time.perf_counter() - t0
    steps_one, sums_one = res["train_steps"], res["sums"]
    eng.close()
    strm = [torch.cuda.Stream() for _ in range(streams)]
    engines = []
    for g, (k, lr) in enumerate(pts):
        e = W.make_engine(c, dict(h, lr=lr, planning_steps=k), per_point, g * per_point)
        e.set_stream(strm[g % streams].cuda_stream)
        engines.append(e)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for e in engines:
        e.train(n_ep, n_ep // 10, wait=False)
    parts = [e.train_wait()[0] for e in engines]
    t_many = time.perf_counter() - t0
    steps_many = sum(p["train_steps"] for p in parts)
    same = all(np.array_equal(sums_one[:, g].view(np.uint64), parts[g]["sums"].view(np.uint64)) for g in range(len(pts)))
    for e in engines:
        e.close()
    lines.append("CliffWalking Dyna-Q grid: planning_steps %s x learning_rate %s = %d points x %d agents, %d episodes (train(n, n/10))"
                 % (steps, lrs, len(pts), per_point, n_ep))
    lines.append("  one engine, %d sets with per-set counts: %.3f s wall  (%d train steps, %.4g steps/s)" % (len(pts), t_one, steps_one, steps_one / t_one))
    lines.append("  %d engines, async on %d streams:          %.3f s wall  (%d train steps, %.4g steps/s)" % (len(pts), streams, t_many, steps_many, steps_many / t_many))
    lines.append("  speed-up %.3fx; per-point sums bit-identical between the two: %s" % (t_many / t_one, same))
    print("\n".join(lines[-4:]), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True, help="directory for dyna_hp_cost.txt")
    ap.add_argument("--reps", type=int, default=3)
    a = ap.parse_args()
    os.makedirs(a.out, exist_ok=True)
    lines = ["card (name, power limit, SM clock, max SM clock): %s" % card(),
             "training steps/s (train_steps / kernel_ms of each chunk), k_run and k_run_hp alternating"]
    print(lines[0], flush=True)
    cost(a.reps, lines)
    grid(lines)
    lines.append("card after the runs: %s" % card())
    open(os.path.join(a.out, "dyna_hp_cost.txt"), "w").write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()

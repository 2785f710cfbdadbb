#!/usr/bin/env python
"""The bootstrap target per hyper-parameter set on the GPU: what it costs and what it buys.

cost:    k_run against k_run_hp holding one set equal to the configuration, its target given through
         rlb_engine_set_targets, on C2 (hybrid store), C4, C3, Taxi Q(lambda) on the lazy store and the `dyna` cell
         (k_run<..., MODEL> against k_run_hp<..., MODEL>): training steps/s from the kernels' CUDA events, the two engines
         alternating chunk by chunk in one process, `--reps` chunks each after a warm-up chunk; medians and the range of
         the chunk ratios.  Then C4 with three contiguous sets, one per target, against plain C4 the same way.
benefit: the Taxi grid target {sarsa, qlearning, expected_sarsa} x learning_rate {0.05, 0.1, 0.2, 0.5} (16 384 agents
         per point, 1000 episodes of train(n, n/10)) as ONE engine of 12 sets against 12 engines; and C5's one-step cells
         (4 envs x {eps-greedy, UCB} x {Basic, Double}, each with its three targets) at 8 192 and 102 400 agents per cell
         as 16 engines of three sets against 48 engines.  Every engine is driven through the asynchronous train call on 8
         streams; wall time each, after checking that every point's per-episode sums are bit-identical between the two
         forms (the separate engines with first_agent_id = g * per).
The card's name, power limit and SM clocks are read (nvidia-smi --query-gpu, read-only) in the same process.
    python tools/target_sets_cost.py --out DIR          (writes DIR/target_sets_cost.txt)"""
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


COST = [("c2", 1 << 20, {}), ("c4", 1 << 21, {}), ("c3", 1 << 22, {}),
        ("taxi_qlambda_lazy", 102400, dict(env=3, agent=1, selector=0, policy=0, target=1, n_episodes=1000, chunk=100)),
        ("dyna", 1 << 20, {})]


def alternate(plain, hp, w, reps):
    """Rates of the two engines over `reps` chunks after a warm-up chunk, alternating; and whether their sums agree."""
    rates, same, ep, chunk = {"plain": [], "hp": []}, True, 0, w["chunk"]
    for r in range(reps + 1):
        got = {}
        for label, eng in (("plain", plain), ("hp", hp)):
            res = eng.train(ep + chunk, max(1, w["n_episodes"] // 10), ep_begin=ep)
            got[label] = res["sums"].reshape(chunk, -1, 4)
            if r:
                rates[label].append(res["train_steps"] / (res["kernel_ms"] * 1e-3))
        if got["hp"].shape == got["plain"].shape:
            same = same and np.array_equal(got["plain"].view(np.uint64), got["hp"].view(np.uint64))
        ep += chunk
    return np.array(rates["plain"]), np.array(rates["hp"]), same


def fmt(name, n, store, a, b, same):
    return ("%-18s agents=%-8d store=%d  k_run %s  k_run_hp %s  ratio(median) %.4f  chunk ratios %.4f .. %.4f%s" % (
        name, n, store, " ".join("%.4g" % x for x in a), " ".join("%.4g" % x for x in b), np.median(b) / np.median(a),
        (b / a).min(), (b / a).max(), "" if same is None else "  sums bit-identical: %s" % same))


def cost(reps, lines):
    for name, n, over in COST:
        w = dict(W.WORKLOADS[name]) if name in W.WORKLOADS else dict(over)
        c, h = W.combo(w, 0), W.workload_hyper(w)
        store = 4 if name == "taxi_qlambda_lazy" else 0
        plain = W.make_engine(c, h, n, store_kind=store)
        hp = W.make_engine(c, dict(h, planning_steps=0), n, store_kind=store)
        hp.set_hparams([one_set(h)], np.zeros(n, np.uint32))
        if w.get("planning_steps"):
            hp.set_planning_steps(np.array([w["planning_steps"]], np.uint32))
        hp.set_targets(np.array([c["target"]], np.int32))
        a, b, same = alternate(plain, hp, w, reps)
        lines.append(fmt(name, n, plain.store_kind(), a, b, same))
        print(lines[-1], flush=True)
        plain.close()
        hp.close()
    # C4 with three contiguous sets, one per target: what the mixed launch runs at against the plain Q-learning kernel
    w = W.WORKLOADS["c4"]
    c, h = W.combo(w, 0), W.workload_hyper(w)
    n = 1 << 21
    plain = W.make_engine(c, h, n)
    hp = W.make_engine(c, h, n)
    hp.set_hparams([one_set(h)] * 3, (np.arange(n) * 3 // n).astype(np.uint32))
    hp.set_targets(np.array([abi.TARGET_SARSA, abi.TARGET_QLEARNING, abi.TARGET_EXPECTED_SARSA], np.int32))
    a, b, _ = alternate(plain, hp, w, reps)
    lines.append(fmt("c4 mixed targets", n, plain.store_kind(), a, b, None) + "  (three sets: sarsa, qlearning, expected_sarsa)")
    print(lines[-1], flush=True)
    plain.close()
    hp.close()


def one_vs_many(cells, per, n_ep, streams, h):
    """cells: [(combo without target, [targets])].  One engine per cell with a set per target against one engine per
    (cell, target); returns (wall one, wall many, train steps each, every point's sums bit-identical)."""
    import torch
    strm = [torch.cuda.Stream() for _ in range(streams)]

    def drive(engines):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for e in engines:
            e.train(n_ep, max(1, n_ep // 10), wait=False)
        parts = [e.train_wait()[0] for e in engines]
        return time.perf_counter() - t0, parts

    grouped = []
    for k, (c, targets, sets) in enumerate(cells):
        e = W.make_engine(dict(c, target=targets[0]), h, len(targets) * per)
        e.set_hparams(sets, np.repeat(np.arange(len(targets), dtype=np.uint32), per))
        e.set_targets(np.array(targets, np.int32))
        e.set_stream(strm[k % streams].cuda_stream)
        grouped.append(e)
    t_one, parts_one = drive(grouped)
    for e in grouped:
        e.close()
    single, j = [], 0
    for c, targets, sets in cells:
        for g, (t, s) in enumerate(zip(targets, sets)):
            hs = dict(h, lr=s["learning_rate"])
            e = W.make_engine(dict(c, target=t), hs, per, g * per)
            e.set_stream(strm[j % streams].cuda_stream)
            single.append(e)
            j += 1
    t_many, parts_many = drive(single)
    for e in single:
        e.close()
    same, j = True, 0
    for k, (c, targets, _) in enumerate(cells):
        for g in range(len(targets)):
            same = same and np.array_equal(parts_one[k]["sums"][:, g].view(np.uint64), parts_many[j]["sums"].view(np.uint64))
            j += 1
    return t_one, t_many, sum(p["train_steps"] for p in parts_one), sum(p["train_steps"] for p in parts_many), same


def benefit(lines, streams=8):
    n_ep = 1000
    h = W.hyper(n_ep)
    taxi = dict(env=3, agent=0, selector=0, policy=0, real=0)
    lrs = [0.05, 0.1, 0.2, 0.5]
    tg = [abi.TARGET_SARSA, abi.TARGET_QLEARNING, abi.TARGET_EXPECTED_SARSA]
    cells = [(taxi, [t for t in tg for _ in lrs], [dict(one_set(h), learning_rate=lr) for _ in tg for lr in lrs])]
    t_one, t_many, s1, s2, same = one_vs_many(cells, 16384, n_ep, streams, h)
    lines.append("Taxi grid target {sarsa, qlearning, expected_sarsa} x learning_rate %s = 12 points x 16384 agents, %d episodes (train(n, n/10))"
                 % (lrs, n_ep))
    lines.append("  one engine, 12 sets with per-set targets: %.3f s wall  (%d train steps, %.4g steps/s)" % (t_one, s1, s1 / t_one))
    lines.append("  12 engines, async on %d streams:          %.3f s wall  (%d train steps, %.4g steps/s)" % (streams, t_many, s2, s2 / t_many))
    lines.append("  speed-up %.3fx; per-point sums bit-identical between the two: %s" % (t_many / t_one, same))
    print("\n".join(lines[-4:]), flush=True)
    c5 = W.WORKLOADS["c5"]
    h5 = W.hyper(c5["n_episodes"], slippery=True)
    combos = sorted({(x["env"], x["selector"], x["policy"]) for x in c5["cells"] if x["agent"] == 0})
    cells = [(dict(env=e, agent=0, selector=s, policy=p, real=0), tg, [one_set(h5)] * 3) for e, s, p in combos]
    for per in (8192, 102400):
        t_one, t_many, s1, s2, same = one_vs_many(cells, per, c5["n_episodes"], streams, h5)
        lines.append("C5 one-step cells: %d (env, selector, policy) x 3 targets, %d agents per cell, %d episodes (train(n, n/10))"
                     % (len(cells), per, c5["n_episodes"]))
        lines.append("  %d engines of three sets, async on %d streams: %.3f s wall  (%d train steps, %.4g steps/s)" % (len(cells), streams, t_one, s1, s1 / t_one))
        lines.append("  %d engines, async on %d streams:              %.3f s wall  (%d train steps, %.4g steps/s)" % (3 * len(cells), streams, t_many, s2, s2 / t_many))
        lines.append("  speed-up %.3fx; per-cell sums bit-identical between the two: %s" % (t_many / t_one, same))
        print("\n".join(lines[-4:]), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True, help="directory for target_sets_cost.txt")
    ap.add_argument("--reps", type=int, default=3)
    a = ap.parse_args()
    os.makedirs(a.out, exist_ok=True)
    lines = ["card (name, power limit, SM clock, max SM clock): %s" % card(),
             "training steps/s (train_steps / kernel_ms of each chunk), k_run and k_run_hp alternating"]
    print(lines[0], flush=True)
    cost(a.reps, lines)
    benefit(lines)
    lines.append("card after the runs: %s" % card())
    open(os.path.join(a.out, "target_sets_cost.txt"), "w").write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()

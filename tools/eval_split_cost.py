"""What the injected evaluate(100) costs the engines whose trace agents keep their tables on chip, and what running it
in k_eval launches of its own saves.

  python tools/eval_split_cost.py --out DIR [--libs name=path,...] [--cases c2,c2_f64,c2_ucb,c5_fl,driver,flN] [--reps 3]

Three parts, each in fresh engines, every timing the median of --reps runs with the libraries alternating run by run
(one subprocess per run: a process binds one librlb):
  (a) evaluate's share of a train chunk: kernel_ms of train(ep, ep + 100, eval_at=100) against eval_at=10**9;
  (b) evaluate rate: agent-steps/s of evaluate(100) after 100 training episodes on the engine's own store, and on a
      one-step engine on the HBM store (store 1) into which the trained tables and agent states were uploaded; the two
      evaluate sums must be bit-identical (the state contract the split relies on);
  (c) kernel_ms per 100-episode chunk of every library named in --libs (e.g. the RLB_EVAL_SPLIT=0 build against the
      default), on C2 f32, C2 f64, C2 with UCB, a C5-size FrozenLake trace cell, a 4 096-agent driver-size engine,
      and the C2 agent at N agents (case flN).
The card, its power limit and SM clock are read in the same run and written beside the numbers.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CASES = {   # name: (real, agents, selector)
    "c2": (0, 1 << 20, 0),
    "c2_f64": (1, 1 << 20, 0),
    "c2_ucb": (0, 1 << 20, 1),
    "c5_fl": (0, 8192, 0),
    "driver": (0, 4096, 0),
}
C2 = dict(env=1, agent=1, selector=0, policy=0, target=0)


def worker(case, part):
    sys.path.insert(0, ROOT)
    import importlib
    import numpy as np
    W = importlib.import_module("rl-rust_b200.workloads")
    real, n, sel = CASES[case] if case in CASES else (0, int(case[2:]), 0)   # flN: the C2 agent, N of them
    c = dict(C2, real=real, selector=sel)
    h = W.hyper(1000, slippery=True)
    out = {}
    if part in ("a", "c"):
        evals = (100, 10 ** 9) if part == "a" else (100,)
        for eval_at in evals:
            with W.make_engine(c, h, n, store_kind=0) as e:
                e.train(100, eval_at, sums=True)                        # warm-up chunk
                ms = 0.0
                for k in range(1, 4):
                    r = e.train(100 * (k + 1), eval_at, ep_begin=100 * k, sums=True)
                    ms += r["kernel_ms"]
                out["kernel_ms_eval_at_%d" % eval_at] = ms / 3
                out["store"] = e.store_kind()
                out["eval_steps_per_chunk"] = r["eval_steps"]
                out["train_steps_per_chunk"] = r["train_steps"]
    else:
        with W.make_engine(c, h, n, store_kind=0) as e:
            e.train(100, 100, sums=False)
            q, counts = e.download_tables()
            st = e.states()
            e.synchronize()
            t0 = time.perf_counter()
            ra = e.evaluate(100, sums=True)
            ta = time.perf_counter() - t0
            out["store"] = e.store_kind()
        with W.make_engine(dict(c, agent=0), h, n, store_kind=1) as g:
            g.upload_tables(q, counts if c["selector"] else None)   # an eps-greedy engine keeps no counts
            g.set_states(st)
            g.synchronize()
            t0 = time.perf_counter()
            rb = g.evaluate(100, sums=True)
            tb = time.perf_counter() - t0
        out.update(steps=int(ra["steps"]), rate_own_store=ra["steps"] / ta, rate_hbm=rb["steps"] / tb,
                   sums_identical=bool(ra["sums"].tobytes() == rb["sums"].tobytes() and ra["steps"] == rb["steps"]))
    print("RESULT " + json.dumps(out), flush=True)


def run(lib, case, part):
    env = dict(os.environ)
    if lib:
        env["RLB_LIB"] = lib
    p = subprocess.run([sys.executable, os.path.abspath(__file__), "--worker", case, part], env=env, capture_output=True, text=True)
    for line in p.stdout.splitlines():
        if line.startswith("RESULT "):
            return json.loads(line[7:])
    raise RuntimeError("worker %s %s %s failed:\n%s" % (lib, case, part, p.stderr[-3000:]))


def med(runs, key):
    vals = [r[key] for r in runs]
    return statistics.median(vals), min(vals), max(vals)


def card():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader"],
                               capture_output=True, text=True).stdout.strip()
    except OSError:
        return "nvidia-smi not available"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=False)
    ap.add_argument("--libs", default="", help="name=path,... A/B of libraries in part (c); empty: the in-tree build only")
    ap.add_argument("--cases", default="c2,c2_f64,c5_fl,driver")
    ap.add_argument("--parts", default="abc")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--base-lib", default="", help="library of parts (a) and (b) (default: the in-tree build)")
    ap.add_argument("--worker", nargs=2, metavar=("CASE", "PART"))
    args = ap.parse_args()
    if args.worker:
        worker(*args.worker)
        return
    cases = [c for c in args.cases.split(",") if c]
    libs = [tuple(s.split("=", 1)) for s in args.libs.split(",") if s] or [("in-tree", "")]
    lines = []

    def say(line):
        lines.append(line)
        print(line, flush=True)

    say("# eval_split_cost: %s" % card())
    say("# medians of %d alternating runs (min .. max), cases %s, libraries %s, base library %s"
        % (args.reps, args.cases, args.libs or "in-tree", args.base_lib or "in-tree"))
    data = {"card": card(), "reps": args.reps}
    for case in cases:
        if "a" in args.parts:
            runs = [run(args.base_lib, case, "a") for _ in range(args.reps)]
            on, lo1, hi1 = med(runs, "kernel_ms_eval_at_100")
            off, lo2, hi2 = med(runs, "kernel_ms_eval_at_1000000000")
            share = 1 - off / on
            data[case + "_a"] = runs
            say("(a) %-7s store %d: chunk kernel_ms eval_at 100 %.2f (%.2f .. %.2f), no evaluate %.2f (%.2f .. %.2f): evaluate share %.1f %%"
                         % (case, runs[0]["store"], on, lo1, hi1, off, lo2, hi2, 100 * share))
        if "b" in args.parts:
            runs = [run(args.base_lib, case, "b") for _ in range(args.reps)]
            own, _, _ = med(runs, "rate_own_store")
            hbm, _, _ = med(runs, "rate_hbm")
            data[case + "_b"] = runs
            say("(b) %-7s evaluate(100): %.3g steps/s on store %d, %.3g on store 1 (one-step, uploaded state); sums bit-identical: %s"
                         % (case, own, runs[0]["store"], hbm, all(r["sums_identical"] for r in runs)))
            if "a" in args.parts:
                say("    predicted gain (a) x (1 - own/hbm): %.1f %%" % (100 * share * (1 - own / hbm)))
        if "c" in args.parts:
            res = {name: [] for name, _ in libs}
            for _ in range(args.reps):
                for name, path in libs:   # alternating library by library
                    res[name].append(run(path, case, "c"))
            data[case + "_c"] = res
            for name, _ in libs:
                m, lo, hi = med(res[name], "kernel_ms_eval_at_100")
                say("(c) %-7s %-10s chunk kernel_ms %.3f (%.3f .. %.3f)" % (case, name, m, lo, hi))
    text = "\n".join(lines) + "\n"
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "eval_split_cost.txt"), "a") as f:
            f.write(text)
        with open(os.path.join(args.out, "eval_split_cost.jsonl"), "a") as f:
            f.write(json.dumps(data) + "\n")


if __name__ == "__main__":
    main()

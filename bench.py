#!/usr/bin/env python
"""bench.py — agent-env steps/sec (updates included) of the fused hot path on N B200s.

A "step" of this bench is one pass of the hot path over one batch: every agent of every GPU
advances CHUNK training episodes of a reference-style run `agent.train(env, n_episodes,
n_episodes/10)` (src/bin/taxi.rs:165-166), including the evaluate(100) the reference injects
after every episode with episode % eval_at == 0 (src/agent.rs:107-113).  After n_episodes the
agent is reset (src/bin/taxi.rs:200) and the next run starts, so any --steps/--warmup works.

metric  = agent-env steps/sec, updates included: one unit is one iteration of the loop at
          src/agent.rs:86-106 (env.step + get_action + update).  Steps spent inside the
          injected evaluate() calls are executed but NOT counted (reported as eval_steps).
value   = whole-job units / device time (CUDA events, max over ranks), outputs left in HBM.
e2e     = the same through the C ABI with HOST buffers: the per-agent episode records
          (reward_history / episode_length of agent.rs:117) and the per-episode sums are
          copied to pinned host memory inside the timed region.

The headline line is BASELINE.json configs[1] ("c2"): FrozenLake 8x8 slippery, Sarsa(lambda),
eps-greedy, Basic, 1 048 576 agents per GPU (weak scaling), f32.  The same JSON line carries
`workloads`: full sub-records (value, e2e, roofline, clocks, config) of
  c4      Taxi one-step Q-learning, eps-greedy — the configuration north_star's 1e11 target is
          stated on: 16 777 216 agents SHARDED over the GPUs (strong scaling; on one GPU the
          2 097 152-agent shard of the 8-GPU job, 16 M agents do not fit 180 GB),
  c3      CliffWalking Expected Sarsa, Double, UCB, 4 194 304 agents per GPU,
  c2_f64  the headline configuration in the reference's own arithmetic (f64).
`--workload X` measures one configuration alone; `--sub ''` drops the sub-records.

`--dump-outputs DIR` writes, for the headline and every sub-record, what the last timed step returned to its caller
(.npy files, at most 64 MB in all) so that two builds can be compared output for output on the same inputs:
  <name>_<dtype>_episode_sums          device leg: per-episode sums [cells, episodes, 4] ([cells, gpus, episodes, 4],
                                       rank 0's gather, on several GPUs)
  <name>_<dtype>_e2e_episode_sums      e2e leg: the same sums, as copied to host memory
  <name>_<dtype>_e2e_episodes          e2e leg: per-agent episode records (ret, td_sum, td_abs_sum, length) of a fixed,
                                       seeded sample of rank 0's agents [cells, episodes, agents, 4]
Each is float64 with its non-finite entries written as 0, beside a float32 <file>_nonfinite of the same shape that marks
them (0 finite, 1 NaN, 2 +inf, 3 -inf).  Non-finite values are the reference's arithmetic, not a fault: under UCB an
unvisited action's bonus is +inf once t >= 55, so Expected Sarsa's target is inf/inf = NaN and c3's TD sums are NaN
(SURVEY.md 8.1 Q9, tests/test_oracle_kat.py::test_ucb_expected_sarsa_nan_quirk).

`--impl reference` times the CPU oracle (the reference cannot be compiled here: no Rust
toolchain) on the host cores, on a bounded sample of the same workload.
"""
import argparse
import importlib
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True   # the bench leaves the tree as it found it (it may be read-only)
DUMP_BYTES = 60 * 10 ** 6        # --dump-outputs: all arrays together, below 64 MB with the .npy headers
DUMP_ELEM_BYTES = 8 + 4          # --dump-outputs: a float64 value and its float32 _nonfinite code
DUMP_SEED = 0x5EED               # --dump-outputs: which agents' episode records are sampled


def save_output(out_dir, name, arr):
    """--dump-outputs: `name`.npy holds `arr` with its non-finite entries set to 0, and `name`_nonfinite.npy says which
    they were (0 finite, 1 NaN, 2 +inf, 3 -inf), so that every file is finite and nothing the path computed is lost."""
    arr = np.asarray(arr, np.float64)
    code = np.zeros(arr.shape, np.float32)
    code[np.isnan(arr)] = 1
    code[np.isposinf(arr)] = 2
    code[np.isneginf(arr)] = 3
    np.save(os.path.join(out_dir, name + ".npy"), np.where(code == 0, arr, 0.0))
    np.save(os.path.join(out_dir, name + "_nonfinite.npy"), code)


def _workloads():
    return importlib.import_module("rl-rust_b200.workloads")


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.p = None

    def start(self):
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                                       "-lms", "200"], stdout=self.f, stderr=subprocess.DEVNULL)
        except OSError:
            self.p = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.p is None:
            return out
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.p.kill()
        self.f.flush()
        self.f.seek(0)
        sm, mx, power, reasons = [], [], [], set()
        for line in self.f.read().splitlines():
            parts = [x.strip() for x in line.split(",")]
            if len(parts) < 9:
                continue
            try:
                sm.append(float(parts[1])); mx.append(float(parts[2])); power.append(float(parts[3]))
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), parts[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        os.unlink(self.f.name)
        if sm:
            out.update(sm_mhz=float(np.median(sm)), sm_max_mhz=float(max(mx)), reasons=sorted(reasons), samples=len(sm),
                       power_w_max=float(max(power)))
        return out


def measured_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            d = json.load(f)
        return float(d["hbm_gbs"]), float(d.get("sm_max_mhz", 1965.0)), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, 1965.0, "fallback (B200_PROFILING.md: 6.65 TB/s, 1965 MHz)"


def kernel_counters(name, dtype, agents_per_gpu):
    """Per-env-step warp instructions and DRAM bytes of k_run for this configuration, from the committed ncu captures
    (profiles/counters.json, written by tools/make_counters.py from the ncu CSVs named there).  Counters taken at
    another agent count of the same configuration are used as per-step figures and flagged."""
    try:
        with open(os.path.join(ROOT, "profiles", "counters.json")) as f:
            table = json.load(f)["kernels"]
    except Exception:
        return None
    exact = [t for t in table if t["workload"] == name and t["dtype"] == dtype and t["agents_per_gpu"] == agents_per_gpu]
    near = [t for t in table if t["workload"] == name and t["dtype"] == dtype]
    if exact:
        return dict(exact[-1], exact_size=True)
    if near:
        return dict(near[-1], exact_size=False)
    return None


# ------------------------------------------------------------------------------------------------ CPU legs
def cpu_sample(w, real, n_agents, n_threads, chunk_begin, chunk_end, sessions=None):
    """Advance `n_agents` oracle sessions by episodes [chunk_begin, chunk_end) on `n_threads` host threads.
    Returns (train_steps, seconds, sessions).  The one place bench.py touches oracle/ (the CPU baseline)."""
    W = _workloads()
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import parity as P
    from oracle import oracle_py as O
    from concurrent.futures import ThreadPoolExecutor
    cfg = P.oracle_config(W.combo(w, real), W.workload_hyper(w))
    if sessions is None:
        sessions = [O.Session(cfg, i) for i in range(n_agents)]
    L = O.lib()
    eval_at = max(1, w["n_episodes"] // 10)
    lens = [np.zeros(chunk_end - chunk_begin, np.uint64) for _ in sessions]

    def work(tid):
        for i in range(tid, len(sessions), n_threads):
            rc = L.oracle_train(sessions[i].h, chunk_begin, chunk_end, eval_at, None, O._p(lens[i]), None, None)   # ctypes drops the GIL
            assert rc == 0
    t0 = time.perf_counter()
    if n_threads == 1:
        work(0)
    else:
        with ThreadPoolExecutor(n_threads) as ex:
            list(ex.map(work, range(n_threads)))
    dt = time.perf_counter() - t0
    return int(sum(int(l.sum()) for l in lens)), dt, sessions


def run_reference_arm(args, name, w, real):
    """`--impl reference`: the reference's CPU implementation of the path.  The Rust crate cannot be built in this
    image, so the C++ oracle (oracle/, a line-by-line port with hash-map tables and the per-step allocations the
    reference makes) stands in, one independent agent stream per host thread."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    cells = [dict(w, **c) for c in w["cells"]] if "cells" in w else [w]
    per_thread = 64 if len(cells) == 1 else 1   # agents per host thread (per cell): each reference step is a few hundred ms of CPU work
    n_agents = cores * per_thread
    chunk, n_ep = w["chunk"], w["n_episodes"]
    sessions = [None] * len(cells)
    k = 0
    times, steps = [], []
    for it in range(args.warmup + args.steps):
        c = k % (n_ep // chunk)
        ts, dt = 0, 0.0
        for ci, cell in enumerate(cells):
            if c == 0 and k > 0:
                for s in sessions[ci]:
                    s.agent_reset()
            ts_, dt_, sessions[ci] = cpu_sample(cell, real, n_agents, cores, c * chunk, (c + 1) * chunk, sessions[ci])
            ts += ts_; dt += dt_
        k += 1
        if it >= args.warmup:
            times.append(dt); steps.append(ts)
    total_t, total_s = sum(times), sum(steps)
    v = total_s / total_t
    line = {
        "impl": "reference", "metric": "agent-env steps/sec (updates incl.)", "value": v, "unit": "agent-steps/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * total_t / max(1, args.steps),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64" if real else "f32", "data": "synthetic",
        "config": {"workload": name + ": " + w["desc"], "agents": n_agents * len(cells), "episodes_per_step": chunk,
                   "n_episodes": n_ep, "eval_at": n_ep // 10},
        "cpu_baseline": {"value": v, "unit": "agent-steps/s", "cores": cores, "kind": "port",
                         "sample": "%d agents (%d per host thread%s) x %d-episode chunks of the same run; C++ oracle, hash-map tables"
                                   % (n_agents * len(cells), per_thread, " per cell" if len(cells) > 1 else "", chunk)},
        "e2e": {"value": v, "unit": "agent-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------ GPU arm
class Job:
    """torch.distributed plumbing of one bench process (rank) plus the library's NCCL communicator."""

    def __init__(self):
        import torch
        import torch.distributed as dist
        self.torch, self.dist = torch, dist
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.rank = int(os.environ.get("RANK", "0"))
        self.local_rank = int(os.environ.get("LOCAL_RANK", "0"))
        torch.cuda.set_device(self.local_rank)
        self.sh = importlib.import_module("rl-rust_b200.sharding")
        self.comm = None
        if self.world > 1:
            dist.init_process_group("nccl", device_id=torch.device("cuda", self.local_rank))
            self.comm = self.sh.make_comm(self.local_rank)   # the library's own communicator (rlb_comm_*), used for the path's gather
        self.stream = torch.cuda.current_stream()
        self.props = torch.cuda.get_device_properties(self.local_rank)

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def allreduce(self, vals, op):
        if self.world == 1:
            return list(vals)
        t = self.torch.tensor(vals, dtype=self.torch.float64, device="cuda")
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX if op == "max" else self.dist.ReduceOp.SUM)
        return t.tolist()

    def close(self):
        if self.comm is not None:
            self.comm.close()
        if self.world > 1:
            self.dist.destroy_process_group()


def measure(job, args, name, w, real, steps, warmup, with_e2e, cpu_agents, cell_streams, outputs=None, dump_bytes=0):
    """One configuration on this job's GPUs: W warm-up steps, K timed steps (device value), the e2e leg, the CPU
    baseline sample.  Returns the record (rank 0) or None.  `outputs` (a dict) receives, on rank 0, what the last
    timed step of each leg returned, at most `dump_bytes` of it (--dump-outputs)."""
    torch = job.torch
    W = _workloads()
    rlb = importlib.import_module("rl-rust_b200")
    world, rank = job.world, job.rank
    real_size = 4 if real == 0 else 8
    dtype = "f32" if real == 0 else "f64"
    # Sharding: a workload with `agents_total` is ONE job of that many agents cut into contiguous shards of global ids
    # (strong scaling); the others run `agents_per_gpu` agents on every GPU (weak scaling).  Either way the Philox counter
    # carries the global id, so every agent's results are independent of the number of GPUs.
    strong = "agents_total" in w and world > 1 and not args.agents_per_gpu
    if strong:
        first_id, N = job.sh.shard_sizes(w["agents_total"], world)[rank]
    else:
        N = args.agents_per_gpu or w["agents_per_gpu"]
        first_id = job.sh.shard(rank, N)
    chunk, n_ep = w["chunk"], w["n_episodes"]
    eval_at = max(1, n_ep // 10)
    chunks_per_run = n_ep // chunk
    cells = [dict(w, **c) for c in w["cells"]] if "cells" in w else [w]
    stream = job.stream
    n_groups = max(1, min(cell_streams, len(cells))) if len(cells) > 1 else 1
    group_streams = [stream] if n_groups == 1 else [torch.cuda.Stream() for _ in range(n_groups)]
    engines = []
    for ci, cell in enumerate(cells):
        e_ = W.make_engine(W.combo(cell, real), W.workload_hyper(cell), N, first_agent_id=first_id, device=job.local_rank, store_kind=args.store)
        e_.set_stream(group_streams[ci % n_groups].cuda_stream)
        engines.append(e_)
    eng = engines[0]
    table_bytes = sum(N * e_.S * e_.T * e_.A * real_size for e_ in engines)   # every env's rows are unpadded (Taxi: 24-byte f32 rows)

    sums_dev = [torch.zeros((chunk, 4), dtype=torch.float64, device="cuda") for _ in cells]
    # rank 0 receives the gathered curves; two buffers take turns so that the e2e leg's device->host copy of step k (on a
    # side stream: a device->host copy on the main stream would queue behind the record copy and stall the next kernel)
    # is never overwritten by the gather of step k + 1
    gathered = [[torch.zeros((world, chunk, 4), dtype=torch.float64, device="cuda") for _ in range(2)] for _ in cells] if (world > 1 and rank == 0) else None
    side = torch.cuda.Stream() if (world > 1 and rank == 0) else None
    rec_size = 16 if real == 0 else 32
    state = {"k": 0}
    acc = {}

    def reset_acc():
        acc.update(train_steps=0, eval_steps=0, kernel_ms=0.0, launches=0, trace_rows=0, alg_bytes=0)

    def account(ci, r):
        acc["train_steps"] += r["train_steps"]; acc["eval_steps"] += r["eval_steps"]
        acc["kernel_ms"] += r["kernel_ms"]; acc["launches"] += 2 * r["kernel_launches"]   # each k_run is followed by one k_episode_sums
        acc["trace_rows"] += r["trace_rows"]
        acc["alg_bytes"] += W.algorithmic_bytes(cells[ci], real_size, r["train_steps"], r["trace_rows"])

    def step(host=None, wait=True, count=True):
        """One step of every cell: enqueue (asynchronous train call; cells on different streams overlap), then wait.
        host = None: outputs stay in HBM (device leg).  host = (sums, records, gathered): pinned host buffers (e2e leg);
        with wait=False the tail of this step's record copy overlaps the next step's kernels and the results are
        accounted when the library reports the call complete (drain)."""
        k = state["k"]
        c = k % chunks_per_run
        for ci, e_ in enumerate(engines):
            if c == 0 and k > 0:
                e_.agent_reset()                                # src/bin/taxi.rs:200
            sums_target = sums_dev[ci] if (host is None or world > 1) else host[0][ci]
            rec_target = None if host is None else host[1][ci][k & 1]
            e_.train((c + 1) * chunk, eval_at, ep_begin=c * chunk, sums_out=sums_target, episodes_out=rec_target, wait=False)
            if world > 1:                                       # the path's one collective: per-episode metrics to rank 0 (rlb_comm, NCCL)
                s_ = group_streams[ci % n_groups]
                g_ = gathered[ci][k & 1] if rank == 0 else None
                job.sh.gather_episode_sums(sums_dev[ci], comm=job.comm, out=g_, stream=s_.cuda_stream)
                if host is not None and rank == 0:              # e2e: the gathered curves land in rank 0's host memory
                    side.wait_stream(s_)
                    with torch.cuda.stream(side):
                        host[2][ci].copy_(g_, non_blocking=True)
        if wait:
            drain(count)
        state["k"] = k + 1

    def drain(count=True):
        for ci, e_ in enumerate(engines):
            for r in e_.train_wait():
                if count:
                    account(ci, r)

    reset_acc()
    for _ in range(warmup):
        step(count=False)
    # Timing rules: a run that saw a hardware / thermal slowdown is rejected and measured once more (sw_power_cap is
    # kept and noted in `clocks.reasons`).  Every rank must take the same decision, so the flag is max-reduced.
    remeasured = False
    for attempt in range(2):
        reset_acc()
        sampler = ClockSampler(job.local_rank)
        sampler.start()
        job.barrier()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t_wall0 = time.perf_counter()
        ev0.record(stream)
        for _ in range(steps):
            step(wait=False)                                    # asynchronous calls, at most two in flight: launches back to back
        for s_ in group_streams[1:] if n_groups > 1 else []:
            stream.wait_stream(s_)
        ev1.record(stream)
        job.barrier()
        t_wall = time.perf_counter() - t_wall0
        drain(count=True)
        clocks = sampler.stop()
        ms = ev0.elapsed_time(ev1)
        slowed = float(any(r in ("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown") for r in clocks.get("reasons", [])))
        slowed = job.allreduce([slowed], "max")[0]
        if not slowed or attempt == 1:
            break
        remeasured = True
    clocks["remeasured_after_slowdown"] = remeasured
    dev = dict(acc)
    dump = outputs is not None and rank == 0
    if dump:   # taken now: the e2e leg's untimed steps write the same device buffers
        prefix = "%s_%s_" % (name, dtype)
        last = (state["k"] - 1) & 1
        outputs[prefix + "episode_sums"] = np.stack([(gathered[ci][last] if world > 1 else sums_dev[ci]).cpu().numpy()
                                                     for ci in range(len(cells))])

    # ---- e2e leg: same steps through the asynchronous C-ABI call with pinned HOST buffers; two record buffers per cell
    # take turns (step k fills buffer k & 1 while the host may still be reading the other)
    e2e = None
    if with_e2e:
        rec_bytes = chunk * N * rec_size
        double_buf = rec_bytes * len(cells) <= 6e9              # beyond that ONE pinned buffer and synchronous steps (no overlap claimed)
        host_sums = [torch.zeros((chunk, 4), dtype=torch.float64).pin_memory() for _ in cells]
        host_recs = []
        for _ in cells:
            b0 = torch.zeros((chunk, N, rec_size // 4), dtype=torch.int32).pin_memory()
            host_recs.append([b0, torch.zeros_like(b0).pin_memory() if double_buf else b0])
        host_gath = [torch.zeros((world, chunk, 4), dtype=torch.float64).pin_memory() for _ in cells] if (world > 1 and rank == 0) else None
        # the e2e leg times the SAME chunks of the run as the device leg did (episode lengths, hence steps per second,
        # change along a run): untimed steps bring the chunk index back to where the device leg started
        while state["k"] % chunks_per_run != warmup % chunks_per_run:
            step(count=False)
        reset_acc()
        job.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(steps):
            step(host=(host_sums, host_recs, host_gath), wait=not double_buf)
        drain(count=True)                                       # the last call's records are on the host when this returns
        if side is not None:
            stream.wait_stream(side)
        for s_ in group_streams[1:] if n_groups > 1 else []:
            stream.wait_stream(s_)
        e1.record(stream)
        job.barrier()
        if dump:
            last = (state["k"] - 1) & 1
            sums = np.stack([(host_gath[ci] if world > 1 else host_sums[ci]).numpy() for ci in range(len(cells))])
            outputs[prefix + "e2e_episode_sums"] = sums
            room = dump_bytes - DUMP_ELEM_BYTES * (outputs[prefix + "episode_sums"].size + sums.size)
            n_sample = max(0, min(N, room // (len(cells) * chunk * 4 * DUMP_ELEM_BYTES)))
            if n_sample:
                idx = np.sort(np.random.default_rng(DUMP_SEED).choice(N, n_sample, replace=False))
                recs = np.stack([host_recs[ci][last].numpy().view(eng.episode_dtype).reshape(chunk, N)[:, idx]
                                 for ci in range(len(cells))])
                outputs[prefix + "e2e_episodes"] = np.stack([recs[f].astype(np.float64) for f in ("ret", "td_sum", "td_abs_sum", "length")], -1)
        e2e = {"ms": e0.elapsed_time(e1), "train_steps": acc["train_steps"], "kernel_ms": acc["kernel_ms"],
               "d2h": len(cells) * (rec_bytes + chunk * 32 + 64) + (len(cells) * world * chunk * 32 if (world > 1 and rank == 0) else 0),
               "h2d": 24 * len(cells), "double_buf": double_buf}
        del host_recs

    # ---- reduce over ranks: max time, sum of units
    ms_max, e2e_ms_max, kernel_ms_max = job.allreduce([ms, e2e["ms"] if e2e else 0.0, dev["kernel_ms"]], "max")
    train_steps, eval_steps, e2e_steps, trace_rows, agents_total = job.allreduce(
        [dev["train_steps"], dev["eval_steps"], e2e["train_steps"] if e2e else 0, dev["trace_rows"], N * len(cells)], "sum")
    store = {1: "hbm", 2: "shared_memory_groups", 3: "hybrid_smem_q_l2_traces", 4: "hbm_lazy_trace_sweeps"}[rlb.abi.lib.rlb_engine_store_kind(eng.h)]
    for e_ in engines:
        e_.close()
    if rank != 0:
        return None

    value = train_steps / (ms_max * 1e-3)
    hbm_peak, sm_max_mhz, peak_src = measured_peaks()
    n_sm = job.props.multi_processor_count
    sm_hz = 1e6 * (clocks.get("sm_mhz") or sm_max_mhz)          # median SM clock sampled during the timed region
    issue_peak = n_sm * 4 * sm_hz                               # warp-instructions / s: 4 schedulers per SM, one issue per clock
    smem_peak = n_sm * 128 * sm_hz                              # bytes / s: 128 B per SM per clock
    n_launch = max(1, dev["launches"] // 2)                     # k_run launches on this rank (each followed by one k_episode_sums)
    kernel_s = dev["kernel_ms"] * 1e-3
    env_steps_rank = dev["train_steps"] + dev["eval_steps"]     # this rank's env transitions inside those launches
    cnt = kernel_counters(name, dtype, N) if len(cells) == 1 else None
    smem_frac = dev["alg_bytes"] / kernel_s / smem_peak if kernel_s > 0 else None
    issue_frac = hbm_frac = traffic = inst_per_launch = None
    if cnt and kernel_s > 0:
        inst_per_launch = cnt["warp_inst_per_env_step"] * env_steps_rank / n_launch
        traffic = cnt["dram_bytes_per_env_step"] * env_steps_rank / n_launch
        issue_frac = inst_per_launch * n_launch / kernel_s / issue_peak
        hbm_frac = traffic * n_launch / kernel_s / (hbm_peak * 1e9)
    # the binding resource is the one closest to its peak; these kernels live on chip, so it is instruction issue
    fracs = {"sm_issue": issue_frac, "smem": smem_frac, "hbm": hbm_frac}
    bound = max((k for k in fracs if fracs[k] is not None), key=lambda k: fracs[k])
    if bound == "sm_issue":
        achieved, peak, unit = inst_per_launch * n_launch / kernel_s, issue_peak, "warp-inst/s"
    elif bound == "smem":
        achieved, peak, unit = dev["alg_bytes"] / kernel_s / 1e9, smem_peak / 1e9, "GB/s"
    else:
        achieved, peak, unit = traffic * n_launch / kernel_s / 1e9, hbm_peak, "GB/s"
    rec = {
        "metric": "agent-env steps/sec (updates incl.)", "value": value, "unit": "agent-steps/s", "n_gpus": world,
        "steps": steps, "warmup": warmup, "ms_per_step": ms_max / max(1, steps), "higher_is_better": True,
        "scaling": "strong" if strong else "weak", "vs_baseline": None, "dtype": dtype, "data": "synthetic",
        "config": {"workload": name + ": " + w["desc"], "agents_per_gpu": N * len(cells), "agents_total": int(agents_total), "cells": len(cells),
                   "episodes_per_step": chunk, "n_episodes": n_ep, "eval_at": eval_at, "table_store": store,
                   "train_steps_timed": train_steps, "eval_steps_executed_not_counted": eval_steps, "env_steps_per_s_incl_eval": (train_steps + eval_steps) / (ms_max * 1e-3),
                   "l2": "inputs larger than L2: %.2f GB of per-agent tables per GPU vs 126 MB L2 (no flush needed)" % (table_bytes / 1e9),
                   "parallelism": ("%d agents sharded over %d GPUs by global id (strong scaling)" % (agents_total, world) if strong
                                   else "agents sharded by global id, %d per GPU (weak scaling)" % N)
                                  + "; one NCCL gather (rlb_comm_gather_episode_sums, ncclSend/ncclRecv) of [episodes,4] metrics per step"
                                  + ("; the %d cells' engines spread over %d CUDA streams by one host thread (asynchronous train calls: their "
                                     "launches overlap, so kernel_share_of_step counts concurrent kernels)" % (len(cells), n_groups) if n_groups > 1 else ""),
                   "wall_s": t_wall},
        "clocks": clocks,
        "gpu_launches": int(dev["launches"]),
        "roofline": {"bound": bound, "kernel": "k_run", "achieved": achieved, "peak": peak, "unit": unit, "frac": fracs[bound],
                     "issue_frac": issue_frac, "smem_frac": smem_frac, "hbm_frac": hbm_frac, "traffic": traffic,
                     "peaks": {"sm_issue_warp_inst_per_s": issue_peak, "smem_gb_s": smem_peak / 1e9, "hbm_gb_s": hbm_peak, "n_sm": n_sm,
                               "sm_mhz_used": sm_hz / 1e6, "source": peak_src + "; SM count from the device, SM clock = median sampled during the timed region"},
                     "warp_inst_per_launch": inst_per_launch, "algorithmic_smem_bytes_per_launch": dev["alg_bytes"] / n_launch,
                     "launch_ms": dev["kernel_ms"] / n_launch, "kernel_share_of_step": dev["kernel_ms"] / ms if ms > 0 else None,
                     "counters": ({k: cnt[k] for k in ("warp_inst_per_env_step", "dram_bytes_per_env_step", "source", "exact_size", "agents_per_gpu")} if cnt else None),
                     "note": "issue_frac = warp instructions (committed ncu capture, per env step) / launch time (CUDA events, this run) / "
                             "(SMs x 4 x clock); smem_frac = SURVEY 8(d) algorithmic bytes / launch time / (SMs x 128 B x clock); "
                             "hbm_frac = ncu dram bytes / launch time / measured HBM copy bandwidth"},
    }
    if e2e:
        rec["e2e"] = {"value": e2e_steps / (e2e_ms_max * 1e-3), "unit": "agent-steps/s", "ms_per_step": e2e_ms_max / max(1, steps),
                      "kernel_ms_per_step": e2e["kernel_ms"] / max(1, steps),
                      "h2d_bytes_per_step": e2e["h2d"], "d2h_bytes_per_step": e2e["d2h"],
                      "note": "C-ABI rlb_agent_train_range_async with pinned HOST buffers: per-agent episode records + per-episode sums copied "
                              "device->host every step (%s; the last copy is waited for inside the timed region); the path has no per-step "
                              "host inputs besides the call's scalar arguments" % ("two host record buffers take turns" if e2e["double_buf"] else "one host record buffer, every step waited for")}
    if world == 1 and cpu_agents:
        ts, dt = 0, 0.0
        for cell in cells:
            ts_, dt_, _ = cpu_sample(cell, real, cpu_agents, 1, 0, n_ep)
            ts += ts_; dt += dt_
        rec["cpu_baseline"] = {"value": ts / dt, "unit": "agent-steps/s", "cores": 1, "kind": "port",
                               "sample": "%d agents%s x one full %d-episode run (eval_at %d), C++ oracle single thread, %.1f s"
                                         % (cpu_agents, " per cell" if len(cells) > 1 else "", n_ep, eval_at, dt)}
    return rec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c2", choices=["c1", "c2", "c3", "c4", "c5", "dyna"])
    ap.add_argument("--agents-per-gpu", type=int, default=0)
    ap.add_argument("--real", default="f32", choices=["f32", "f64"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--store", type=int, default=0, help="table store: 0 auto, 1 HBM, 2 shared memory")
    ap.add_argument("--cell-streams", type=int, default=8,
                    help="multi-cell workloads (c5): CUDA streams the cells' engines are spread over, so that launches too small to "
                         "fill the GPU overlap (1 = back to back on one stream)")
    ap.add_argument("--sub", default=None,
                    help="comma-separated sub-records to add under `workloads` (c4, c3, c2_f64, c1, c5, dyna); default: "
                         "'c4,c3,c2_f64' for the default headline run, none when --workload / --agents-per-gpu / --real is given")
    ap.add_argument("--sub-steps", type=int, default=10, help="timed steps of each sub-record (10 = one whole 1000-episode run)")
    ap.add_argument("--sub-warmup", type=int, default=3)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step computed as DIR/<name>.npy (see the module docstring)")
    args = ap.parse_args()
    W = _workloads()
    w = dict(W.WORKLOADS[args.workload])
    real = 0 if args.real == "f32" else 1
    if args.warmup < 3 and args.impl == "ours":
        print("note: --warmup %d < 3 (timing rules ask for >= 3)" % args.warmup, file=sys.stderr)

    if args.impl == "reference":
        run_reference_arm(args, args.workload, w, real)
        return

    import torch
    rlb = importlib.import_module("rl-rust_b200")
    if not torch.cuda.is_available() or rlb.abi.lib.rlb_device_count() < 1:
        raise SystemExit("bench.py needs a CUDA device: the engine has no CPU path (use --impl reference for the CPU arm)")
    default_run = args.workload == "c2" and not args.agents_per_gpu and args.real == "f32" and args.store == 0
    subs = args.sub if args.sub is not None else ("c4,c3,c2_f64" if default_run else "")
    subs = [s for s in subs.split(",") if s]

    job = Job()
    outputs = {} if args.dump_outputs else None
    dump_bytes = DUMP_BYTES // (1 + len(subs))   # an equal share for every measured configuration
    cpu_agents = 0 if args.no_cpu_baseline else (512 if "cells" not in w else 4)   # ~10 s of single-thread CPU work
    line = measure(job, args, args.workload, w, real, args.steps, args.warmup, not args.no_e2e, cpu_agents, args.cell_streams,
                   outputs, dump_bytes)
    sub_records = {}
    saved_apg = args.agents_per_gpu
    for sname in subs:
        args.agents_per_gpu = 0
        base, _, suffix = sname.partition("_")
        sw = dict(W.WORKLOADS[base])
        sreal = 1 if suffix == "f64" else 0
        # CPU samples of the sub-records are sized for a few seconds each (C3 executes ~6x its training steps in evaluate)
        scpu = 0 if args.no_cpu_baseline else {"c4": 512, "c3": 64, "c2": 256, "c1": 512}.get(base, 0)
        r = measure(job, args, base, sw, sreal, args.sub_steps, max(3, args.sub_warmup), not args.no_e2e, scpu, args.cell_streams,
                    outputs, dump_bytes)
        if r is not None:
            sub_records[sname] = r
    args.agents_per_gpu = saved_apg
    if job.rank == 0:
        if sub_records:
            line["workloads"] = sub_records
        if outputs is not None:
            os.makedirs(args.dump_outputs, exist_ok=True)
            for oname, arr in outputs.items():
                save_output(args.dump_outputs, oname, arr)
        print(json.dumps(line), flush=True)
    job.close()


if __name__ == "__main__":
    main()

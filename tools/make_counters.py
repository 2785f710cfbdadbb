#!/usr/bin/env python
"""Build profiles/counters.json — per-env-step warp instructions and DRAM bytes of the kernels of one bench step, per
bench configuration.

Usage: python tools/make_counters.py TAG  (reads gpurun_out/TAG_<w>_counters.csv + gpurun_out/TAG_<w>_step1.json)

Each pair comes from the SAME command, `python bench.py --workload W [--real R] --steps 1 --warmup 3 --no-e2e
--no-cpu-baseline --sub ''`, run once plainly (the JSON: how many env transitions — training + injected evaluate — the
first timed step executes; the run is deterministic) and once under `ncu --metrics ... -k regex:"k_run|k_eval" -s S -c C`
(the CSV: the counters of that step's launches).  S and C count the step's k_run and k_eval launches: one per step where
the evaluate blocks run inside k_run (-s 3 -c 1), three per C2 step where the on-chip stores run them in k_eval
(-s 9 -c 3; rlb_train_out.kernel_launches).  Counting metrics (`.sum`) are summed over the launches.  bench.py multiplies the per-step figures by the steps it measures.  The CSVs are copied
to profiles/ so that every figure in a bench line can be traced to a committed file."""
import csv, json, os, shutil, sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
tag = sys.argv[1]
out_path = os.path.join(ROOT, "profiles", "counters.json")
try:
    table = json.load(open(out_path))
except Exception:
    table = {"note": "", "kernels": []}
for w in ("c1", "c2", "c3", "c4", "c2_f64", "c4_f64", "c3_f64"):
    c = os.path.join(ROOT, "gpurun_out", "%s_%s_counters.csv" % (tag, w))
    j = os.path.join(ROOT, "gpurun_out", "%s_%s_step1.json" % (tag, w))
    if not (os.path.exists(c) and os.path.exists(j)):
        continue
    m = {}
    for row in csv.reader(open(c)):
        if len(row) >= 15 and row[0].isdigit():   # ID, ..., Section Name, Metric Name, Metric Unit, Metric Value
            try:
                v = float(row[-1].replace(",", ""))
            except ValueError:
                continue
            # one row per launch and metric: counts add up over the step's launches; a rate or ratio keeps the last launch's
            m[row[-3]] = m.get(row[-3], 0.0) + v if row[-3].endswith(".sum") else v
    line = json.loads(open(j).read().strip().splitlines()[-1])
    env_steps = line["config"]["train_steps_timed"] + line["config"]["eval_steps_executed_not_counted"]
    inst = m["smsp__inst_executed.sum"]
    dram = m["dram__bytes_read.sum"] + m["dram__bytes_write.sum"]
    base = w.split("_")[0]
    entry = {"workload": base, "dtype": line["dtype"], "agents_per_gpu": line["config"]["agents_per_gpu"], "tag": tag,
             "env_steps_in_launch": env_steps, "train_steps_in_launch": line["config"]["train_steps_timed"],
             "warp_inst_per_launch": inst, "dram_bytes_per_launch": dram, "launch_ns_under_ncu": m.get("gpu__time_duration.sum"),
             "issue_pct_under_ncu": m.get("sm__inst_issued.avg.pct_of_peak_sustained_active"),
             "threads_per_inst": m.get("smsp__thread_inst_executed_per_inst_executed.ratio"),
             "smem_wavefronts": m.get("l1tex__data_pipe_lsu_wavefronts_mem_shared.sum"),
             "smem_bank_conflicts": m.get("l1tex__data_bank_conflicts_pipe_lsu_mem_shared.sum"),
             "warp_inst_per_env_step": inst / env_steps, "dram_bytes_per_env_step": dram / env_steps,
             "source": "profiles/%s_%s_counters.csv + profiles/%s_%s_step1.json" % (tag, w, tag, w)}
    table["kernels"] = [t for t in table["kernels"] if not (t["workload"] == base and t["dtype"] == entry["dtype"] and t["agents_per_gpu"] == entry["agents_per_gpu"])]
    table["kernels"].append(entry)
    shutil.copy(c, os.path.join(ROOT, "profiles", os.path.basename(c)))
    shutil.copy(j, os.path.join(ROOT, "profiles", os.path.basename(j)))
    print(w, "inst/env-step %.1f" % (32 * entry["warp_inst_per_env_step"]), "per warp-step; dram B/env-step %.2f" % entry["dram_bytes_per_env_step"])
table["note"] = ("ncu counters of the kernels of one bench step (k_run, and k_eval where the engine runs its evaluate blocks apart) "
                 "and the env transitions (training + injected evaluate) they execute, per bench configuration; written by "
                 "tools/make_counters.py; bench.py scales them by the steps it measures")
json.dump(table, open(out_path, "w"), indent=1)

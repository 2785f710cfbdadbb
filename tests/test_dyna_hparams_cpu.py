"""Dyna-Q under hyper-parameter sets without a GPU: the integer perturbation of the planning count, the planning_steps
grid axis and what it rejects, the calls a stubbed engine receives (none without the axis) and the JSON, the binding's
argument checks, the new entry point being declared, exported and bound, and the ptxas budgets of the k_run_hp<..., MODEL>
twins."""
import glob
import importlib
import json
import os
import re
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
abi = importlib.import_module("rl-rust_b200._abi")
driver = importlib.import_module("rl-rust_b200.driver")


def test_integer_perturbation_of_the_planning_count():
    p = driver.pbt_perturb_planning
    assert [p(k, 1.2) for k in (0, 1, 2, 3, 5, 10, 50)] == [1, 2, 3, 4, 6, 12, 60]     # round(k * 1.2), else k + 1
    assert [p(k, 0.8) for k in (0, 1, 2, 3, 5, 10, 50)] == [0, 0, 1, 2, 4, 8, 40]      # round(k * 0.8), else max(0, k - 1)
    assert all(isinstance(p(k, f), int) for k in range(20) for f in driver.PBT_FACTORS)
    rng = np.random.default_rng(3)
    out = driver.pbt_explore(dict(planning_steps=4, learning_rate=0.1), ["planning_steps", "learning_rate"], rng)
    assert out["planning_steps"] in (3, 5) and isinstance(out["planning_steps"], int)
    assert out["learning_rate"] in (pytest.approx(0.08), pytest.approx(0.12))


def test_grid_accepts_the_axis_and_rejects_what_is_not_a_count():
    pts = driver.expand_grid({"planning_steps": [0, 5], "learning_rate": [0.1, 0.2]})
    assert pts == [dict(planning_steps=0, learning_rate=0.1), dict(planning_steps=0, learning_rate=0.2),
                   dict(planning_steps=5, learning_rate=0.1), dict(planning_steps=5, learning_rate=0.2)]
    assert all(type(p["planning_steps"]) is int for p in driver.expand_grid({"planning_steps": [np.int64(3)]}))
    for bad in ([-1], [2.5], [1.0], [True], ["3"]):
        with pytest.raises(ValueError):
            driver.expand_grid({"planning_steps": bad})
    assert "planning_steps" not in driver.SWEEP_FLAGS and "planning_steps" not in driver.DEFAULTS
    hp = driver.point_hparams(dict(driver.DEFAULTS, planning_steps=7), 100)
    assert "planning_steps" not in hp and set(hp) == set(abi.HPARAM_FIELDS)


def test_cli_parses_the_axis():
    ap = driver.sweep_parser("test")
    env, grid, out, kw = driver.parse_sweep_args(ap, ["cliffwalking", "--planning_steps", "0,5,10,50", "--learning_rate", "0.05,0.1"])
    assert env == "cliffwalking" and grid == {"learning_rate": [0.05, 0.1], "planning_steps": [0, 5, 10, 50]}
    assert "planning_steps" not in kw
    _, grid, _, _ = driver.parse_sweep_args(ap, ["cliffwalking", "--grid", "planning_steps=1,2"])
    assert grid == {"planning_steps": [1, 2]}
    for bad in (["--planning_steps", "1,-2"], ["--planning_steps", "1.5"], ["--grid", "planning_steps=x"]):
        with pytest.raises(SystemExit):
            driver.parse_sweep_args(driver.sweep_parser("test"), ["cliffwalking"] + bad)


class StubEngine:
    """Stands in for abi.Engine: every agent of set g returns 100 * learning_rate + planning count of its set per
    episode.  Records the planning counts it is given."""
    made = []

    def __init__(self, env_kind, *, n_agents, **kw):
        self.N, self.kw, self.G = n_agents, kw, 0
        self.planning_calls, self.clones = [], []
        self.planning = None
        StubEngine.made.append(self)

    def set_hparams(self, sets, group):
        self.sets, self.group = [dict(s) for s in sets], np.asarray(group)
        self.G = len(sets)

    def set_planning_steps(self, steps):
        self.planning = None if steps is None else [int(x) for x in steps]
        self.planning_calls.append(self.planning)

    def set_active_sets(self, mask):
        pass

    def retune_hparams(self, sets):
        self.sets = [dict(s) for s in sets]

    def clone_agents(self, src, dst):
        self.clones.append((list(src), list(dst)))

    def _sums(self, n):
        s = np.zeros((n, self.G, 4))
        for g in range(self.G):
            k = float((self.group == g).sum())
            extra = self.planning[g] if self.planning else 0
            s[:, g, 0], s[:, g, 1] = k * 10.0, k * (100.0 * self.sets[g]["learning_rate"] + extra)
        return s

    def train(self, n, eval_at, ep_begin=0):
        return dict(sums=self._sums(n - ep_begin), train_steps=(n - ep_begin) * self.G)

    def evaluate(self, n, sums=True):
        return dict(sums=self._sums(n))

    def close(self):
        pass


def stubbed(monkeypatch):
    monkeypatch.setattr(driver.abi, "Engine", StubEngine)
    StubEngine.made = []


def test_sweep_without_the_axis_makes_no_planning_call(monkeypatch):
    stubbed(monkeypatch)
    res = driver.run_sweep("cliffwalking", {"learning_rate": [0.1, 0.2]}, agents_per_point=2, n_episodes=50, verbose=False)
    assert StubEngine.made[0].planning_calls == []
    assert all(set(p["params"]) == {"learning_rate"} for p in res["points"])
    assert res["grid"] == {"learning_rate": [0.1, 0.2]}


def test_sweep_with_the_axis(monkeypatch, tmp_path):
    stubbed(monkeypatch)
    out = tmp_path / "sweep.json"
    res = driver.main_sweep(["cliffwalking", "--target", "qlearning", "--planning_steps", "0,1,5", "--learning_rate", "0.05,0.1",
                             "-n", "50", "--agents_per_point", "3", "--out", str(out)])
    eng = StubEngine.made[0]
    assert eng.planning_calls == [[0, 1, 5, 0, 1, 5]]                     # after set_hparams, one count per point
    data = json.loads(out.read_text())
    assert [p["params"]["planning_steps"] for p in data["points"]] == [0, 1, 5, 0, 1, 5]
    assert data["grid"]["planning_steps"] == [0, 1, 5]
    assert all("planning_steps" not in p["hparams"] for p in data["points"])
    assert data["ranking"] == res["ranking"] and data["ranking"][0] == 5       # lr 0.1 and 5 replays score highest


def test_pbt_carries_integer_counts(monkeypatch):
    stubbed(monkeypatch)
    grid = {"planning_steps": [0, 2, 10], "learning_rate": [0.1, 0.2]}
    res = driver.run_pbt("cliffwalking", grid, interval=10, fraction=0.34, pbt_seed=7, agents_per_point=2, n_episodes=40, verbose=False)
    eng = StubEngine.made[0]
    assert len(eng.planning_calls) == 1 + 3                                 # grid_engine, then one per chunk boundary
    for step, counts in zip(res["lineage"], eng.planning_calls[1:]):
        for p in step["pairs"]:
            assert type(p["flags"]["planning_steps"]) is int and counts[p["loser"]] == p["flags"]["planning_steps"]
    assert [p["final_params"]["planning_steps"] for p in res["points"]] == eng.planning_calls[-1]
    json.dumps(res)
    with pytest.raises(ValueError):
        driver.run_pbt("cliffwalking", grid, interval=10, agent="traces", agents_per_point=2, n_episodes=40, verbose=False)
    assert len(StubEngine.made) == 1                                        # refused before an engine was built


def test_halving_with_the_axis(monkeypatch):
    stubbed(monkeypatch)
    res = driver.run_halving("cliffwalking", {"planning_steps": [0, 3, 9]}, min_episodes=10, eta=3, agents_per_point=2,
                             n_episodes=30, verbose=False)
    assert StubEngine.made[0].planning_calls == [[0, 3, 9]]
    assert res["ranking"][0] == 2


def test_binding_checks_and_the_symbol():
    hdr = open(os.path.join(ROOT, "include", "rlb.h")).read()
    assert re.search(r"rlb_status rlb_engine_set_planning_steps\(rlb_engine\* e, const uint32_t\* steps, uint32_t n_sets\);", hdr)
    assert "#define RLB_ABI_VERSION 2" in hdr
    assert "rlb_engine_set_planning_steps" in abi.EXPORTS and hasattr(abi.lib, "rlb_engine_set_planning_steps")
    nm = subprocess.run(["nm", "-D", "--defined-only", abi.LIB_PATH], capture_output=True, text=True)
    if nm.returncode == 0:
        assert " rlb_engine_set_planning_steps" in nm.stdout
    fake = abi.Engine.__new__(abi.Engine)       # no device: the checks run before the library is called
    fake.G = 3
    for bad in ([1, 2], [[1, 2, 3]], [1, -1, 2], [1.5, 2, 3], [0, 2 ** 32, 1]):
        with pytest.raises(ValueError):
            fake.set_planning_steps(np.asarray(bad))


def ptxas_record(frag, pattern):
    logs = glob.glob(os.path.join(ROOT, "rl-rust_b200", "build", pattern))
    if not logs:
        import __graft_entry__
        __graft_entry__.build()
        logs = glob.glob(os.path.join(ROOT, "rl-rust_b200", "build", pattern))
    for f in logs:
        txt = open(f).read()
        i = txt.find("Function properties for _ZN3rlb" + frag)
        if i >= 0:
            s = txt[i:i + 600]
            return (int(re.search(r"Used (\d+) registers", s).group(1)), int(re.search(r"(\d+) bytes spill stores", s).group(1)),
                    int(re.search(r"(\d+) bytes stack frame", s).group(1)))
    raise AssertionError("no ptxas record for %s" % frag)


def ctas_per_sm(regs, block=128):
    return 65536 // (((regs + 7) // 8 * 8) * block)    # registers are allocated 8 per thread at a time


# (cell, template arguments): the bench's dyna cell and Taxi's one-step Q-learning cell.  Measured with nvcc 12.9
# (registers, spill bytes, stack bytes): dyna k_run (105, 0, 0), k_run_hp (110, 0, 0); Taxi k_run (111, 0, 0),
# k_run_hp (116, 0, 0).  The twin holds its set's values and count in registers where the plain kernel reads them from
# the parameter bank; neither needs more than 4 CTAs of 128 threads per SM, so the twin keeps its plain twin's occupancy.
MODEL_TWINS = {"dyna CLIFF f32 Basic eps one-step": "ILi2EfLi0ELi0ELb0ELi1ELb1E",
               "TAXI f32 Basic eps one-step": "ILi3EfLi0ELi0ELb0ELi1ELb1E"}


@pytest.mark.parametrize("name", sorted(MODEL_TWINS))
def test_model_hp_twins_keep_their_plain_twins_budget(name):
    args = MODEL_TWINS[name]
    plain = ptxas_record("5k_run" + args, "*_model.ptxas.log")
    twin = ptxas_record("8k_run_hp" + args, "*_model_hp.ptxas.log")
    assert ctas_per_sm(twin[0]) == ctas_per_sm(plain[0]), (name, plain, twin)
    assert twin[1] <= plain[1] + 32 and twin[2] <= plain[2] + 32, (name, plain, twin)

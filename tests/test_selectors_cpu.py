"""The action selector per hyper-parameter set without a GPU: the entry point being declared, exported and bound, the
HpParams layout the step and fused kernels read, the selector grid axis against a single engine-wide name and what both
reject, the calls a stubbed engine receives and the JSON, PBT's inheritance, resampling and call order, its draws
without the axis, the snapshot load order, and the ptxas records of the _hp twins with the position base."""
import glob
import importlib
import inspect
import json
import os
import re
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
abi = importlib.import_module("rl-rust_b200._abi")
driver = importlib.import_module("rl-rust_b200.driver")
snapshot = importlib.import_module("rl-rust_b200.snapshot")
CSRC = os.path.join(ROOT, "rl-rust_b200", "csrc")


def test_entry_point_is_declared_exported_and_bound():
    hdr = open(os.path.join(ROOT, "include", "rlb.h")).read()
    assert re.search(r"rlb_status rlb_engine_set_selectors\(rlb_engine\* e, const int32_t\* selectors, uint32_t n_sets\);", hdr)
    assert "#define RLB_ABI_VERSION 2" in hdr
    assert "rlb_engine_set_selectors" in abi.EXPORTS and hasattr(abi.lib, "rlb_engine_set_selectors")
    nm = subprocess.run(["nm", "-D", "--defined-only", abi.LIB_PATH], capture_output=True, text=True)
    if nm.returncode == 0:
        assert " rlb_engine_set_selectors" in nm.stdout
    fake = abi.Engine.__new__(abi.Engine)       # no device: the checks run before the library is called
    fake.G = 2
    for bad in ([0], [[0, 1]], [0, 2], [-1, 0], [0.0, 1.0], ["eps", "ucb"]):
        with pytest.raises(ValueError):
            fake.set_selectors(np.asarray(bad))


def test_hp_params_layout(tmp_path):
    """HpParams as the kernels read it: pos_base last, after the fields the earlier kernels read at their offsets."""
    src = tmp_path / "hp.cu"
    src.write_text('#include <cstddef>\n#include <cstdio>\n#include "rlb_device.cuh"\nint main() { printf("%zu %zu %zu %zu\\n", '
                   'sizeof(rlb::HpParams), offsetof(rlb::HpParams, n_launch), offsetof(rlb::HpParams, targets), '
                   'offsetof(rlb::HpParams, pos_base)); return 0; }\n')
    exe = str(tmp_path / "hp")
    r = subprocess.run(["nvcc", "-std=c++17", "-I", CSRC, "-I", os.path.join(ROOT, "include"), str(src), "-o", exe],
                       capture_output=True, text=True)
    if r.returncode != 0:
        pytest.skip("nvcc could not build the layout probe: %s" % r.stderr[-400:])
    size, off_n, off_t, off_b = map(int, subprocess.check_output([exe]).split())
    assert (off_n, off_t, off_b, size) == (24, 40, 48, 56)


def test_kernels_use_the_list_and_the_base():
    step = open(os.path.join(CSRC, "rlb_step_agent_kernels.inc")).read()
    assert step.count("    RLB_STEP_AGENT\n") == 6                                  # every kernel of the file takes the list
    assert "if (t_ >= h.n_launch) return;" in step and "h.agents ? (uint64_t)__ldg(h.agents + t_) : t_" in step
    run = open(os.path.join(CSRC, "rlb_run_kernel.inc")).read()
    assert "core.st.init(smem_raw, p, i, pos + h.pos_base, threadIdx.x);" in run
    eng = open(os.path.join(CSRC, "rlb_engine.cu")).read()
    assert "second.pos_base = (e->n_sel_run[0] + 31) / 32 * 32;" in eng
    assert "(e->cfg.n_agents + 31) / 32 * 32 + 32" in eng                       # the scratch covers both launches
    assert "#define RLB_SEL_CONCURRENT 1" in eng


def test_grid_accepts_the_axis_and_rejects_unknown_names():
    pts = driver.expand_grid({"selector": ["eps", "ucb"], "confidence_level": [0.5, 2.0]})
    assert pts == [dict(selector="eps", confidence_level=0.5), dict(selector="eps", confidence_level=2.0),
                   dict(selector="ucb", confidence_level=0.5), dict(selector="ucb", confidence_level=2.0)]
    for bad in (["eps", "greedy"], [0, 1], [None]):
        with pytest.raises(ValueError):
            driver.expand_grid({"selector": bad})
    hp = driver.point_hparams(dict(driver.DEFAULTS, selector="ucb"), 100)
    assert "selector" not in hp and set(hp) == set(abi.HPARAM_FIELDS)
    assert "selector" not in driver.SWEEP_FLAGS and "selector" not in driver.DEFAULTS


def test_cli_axis_against_a_single_engine_wide_name():
    ap = driver.sweep_parser("test")
    env, grid, _, kw = driver.parse_sweep_args(ap, ["taxi", "--selector", "eps,ucb", "--learning_rate", "0.1,0.2"])
    assert grid == {"selector": ["eps", "ucb"], "learning_rate": [0.1, 0.2]} and kw["selector"] == "eps"
    _, grid, _, kw = driver.parse_sweep_args(driver.sweep_parser("test"), ["taxi", "--selector", "ucb", "--learning_rate", "0.1,0.2"])
    assert grid == {"learning_rate": [0.1, 0.2]} and kw["selector"] == "ucb"          # one name: engine-wide
    _, grid, _, kw = driver.parse_sweep_args(driver.sweep_parser("test"), ["taxi", "--grid", "selector=ucb,eps"])
    assert grid == {"selector": ["ucb", "eps"]} and kw["selector"] == "ucb"
    _, grid, _, kw = driver.parse_sweep_args(driver.sweep_parser("test"), ["taxi", "--learning_rate", "0.1"])
    assert kw["selector"] == "eps" and "selector" not in grid                          # the default
    _, grid, _, kw = driver.parse_sweep_args(driver.sweep_parser("test"), ["taxi", "--selector", "eps,ucb", "--target", "sarsa,qlearning"])
    assert grid == {"target": ["sarsa", "qlearning"], "selector": ["eps", "ucb"]}
    for bad in (["--selector", "eps,greedy"], ["--selector", "UCB"], ["--grid", "selector=x"], ["--grid", "selector="], ["--selector", ","]):
        with pytest.raises(SystemExit):
            driver.parse_sweep_args(driver.sweep_parser("test"), ["taxi", "--learning_rate", "0.1"] + bad)


class StubEngine:
    """Stands in for abi.Engine: every agent of set g returns 100 * learning_rate + 10 * its set's selector per episode.
    Records every call that carries selectors, clones and targets, in order."""
    made = []

    def __init__(self, env_kind, *, n_agents, **kw):
        self.N, self.kw, self.G = n_agents, kw, 0
        self.calls, self.selectors, self.targets = [], None, None
        StubEngine.made.append(self)

    def set_hparams(self, sets, group):
        self.sets, self.group = [dict(s) for s in sets], np.asarray(group)
        self.G = len(sets)
        self.calls.append(("set_hparams",))

    def set_selectors(self, kinds):
        self.selectors = [int(x) for x in kinds]
        self.calls.append(("set_selectors", self.selectors))

    def set_targets(self, kinds):
        self.targets = [int(x) for x in kinds]
        self.calls.append(("set_targets", self.targets))

    def set_planning_steps(self, steps):
        pass

    def set_active_sets(self, mask):
        pass

    def retune_hparams(self, sets):
        self.sets = [dict(s) for s in sets]
        self.calls.append(("retune",))

    def clone_agents(self, src, dst):
        self.calls.append(("clone", np.asarray(src).tolist(), np.asarray(dst).tolist()))

    def _sums(self, n):
        s = np.zeros((n, self.G, 4))
        for g in range(self.G):
            k = float((self.group == g).sum())
            sel = self.selectors[g] if self.selectors else self.kw["selector"]
            s[:, g, 0], s[:, g, 1] = k * 10.0, k * (100.0 * self.sets[g]["learning_rate"] + 10.0 * sel)
        return s

    def train(self, n, eval_at, ep_begin=0):
        return dict(sums=self._sums(n - ep_begin), train_steps=(n - ep_begin) * self.G)

    def evaluate(self, n, sums=True):
        return dict(sums=self._sums(n))

    def close(self):
        pass


def stubbed(monkeypatch):
    monkeypatch.setattr(driver.abi, "Engine", StubEngine)
    monkeypatch.setattr(driver.time, "perf_counter", lambda: 0.0)
    StubEngine.made = []


def test_single_selector_json_unchanged(monkeypatch):
    stubbed(monkeypatch)
    for name in ("eps", "ucb"):
        res = driver.run_sweep("taxi", {"learning_rate": [0.1, 0.2]}, selector=name, agents_per_point=2, n_episodes=20,
                               moving_average_window=20, verbose=False)
        eng = StubEngine.made[-1]
        assert [c[0] for c in eng.calls] == ["set_hparams"] and eng.kw["selector"] == driver.SELECTOR_NAMES[name]
        assert res["selector"] == name and "selector" not in res["points"][0]["params"]
    import test_targets_cpu as T                                               # the engine-wide JSON, byte for byte
    monkeypatch.setattr(driver.abi, "Engine", T.StubEngine)
    res = driver.run_sweep("taxi", {"learning_rate": [0.1, 0.2]}, selector="eps", target="qlearning", agents_per_point=2,
                           n_episodes=20, moving_average_window=20, verbose=False)
    assert json.dumps(res) == T.SINGLE_TARGET_JSON


def test_sweep_with_the_axis(monkeypatch, tmp_path):
    stubbed(monkeypatch)
    out = tmp_path / "sweep.json"
    res = driver.main_sweep(["taxi", "--selector", "eps,ucb", "--learning_rate", "0.1,0.2", "--confidence_level", "0.5,2",
                             "-n", "20", "--agents_per_point", "2", "--out", str(out)])
    eng = StubEngine.made[0]
    assert eng.kw["selector"] == abi.SEL_UCB                                   # created with UCB: the store fits both
    assert eng.calls == [("set_hparams",), ("set_selectors", [0, 0, 0, 0, 1, 1, 1, 1])]
    data = json.loads(out.read_text())
    assert data["selector"] is None and data["grid"]["selector"] == ["eps", "ucb"]
    assert [p["params"]["selector"] for p in data["points"]] == ["eps"] * 4 + ["ucb"] * 4
    assert data["ranking"] == res["ranking"] and data["ranking"][0] in (6, 7)
    driver.run_sweep("taxi", {"selector": ["eps"], "learning_rate": [0.1]}, agents_per_point=2, n_episodes=20, verbose=False)
    assert StubEngine.made[-1].kw["selector"] == abi.SEL_EPS_GREEDY            # an axis without UCB: created with eps


def test_pbt_explore_inherits_or_resamples():
    flags = dict(selector="eps", target="sarsa", learning_rate=0.1)
    axes = ["selector", "target", "learning_rate"]
    with pytest.raises(ValueError):
        driver.pbt_explore(flags, axes, np.random.default_rng(0), ["sarsa", "qlearning"])   # the selector values are needed
    sels = ["eps", "ucb"]
    outs = [driver.pbt_explore(flags, axes, np.random.default_rng(s), ["sarsa", "qlearning"], 0.25, sels) for s in range(400)]
    kept = sum(o["selector"] == "eps" for o in outs)
    assert 0.8 * 400 < kept < 0.95 * 400 and {o["selector"] for o in outs} == set(sels)   # 0.75 + 0.25 / 2 stay on eps
    assert all(driver.pbt_explore(flags, axes, np.random.default_rng(s), ["sarsa"], 0.0, sels)["selector"] == "eps" for s in range(50))
    # the draws in order: the selector's in its axis' place (first here), then the target's, then the numeric factor
    for s in range(20):
        a, b = np.random.default_rng(s), np.random.default_rng(s)
        got = driver.pbt_explore(flags, axes, a, ["sarsa", "qlearning"], 0.5, sels)
        want = dict(flags)
        if b.random() < 0.5:
            want["selector"] = sels[int(b.integers(2))]
        if b.random() < 0.5:
            want["target"] = ["sarsa", "qlearning"][int(b.integers(2))]
        want["learning_rate"] = float(min(max(0.1 * driver.PBT_FACTORS[int(b.integers(2))], driver.PBT_BOUNDS["learning_rate"][0]), 1.0))
        assert got == want
    # without the axis: the draws of the numeric axes alone, as before
    for s in range(20):
        a, b = np.random.default_rng(s), np.random.default_rng(s)
        got = driver.pbt_explore(dict(learning_rate=0.1, confidence_level=1.0), ["learning_rate", "confidence_level"], a)
        f1, f2 = driver.PBT_FACTORS[int(b.integers(2))], driver.PBT_FACTORS[int(b.integers(2))]
        assert got == dict(learning_rate=float(min(max(0.1 * f1, driver.PBT_BOUNDS["learning_rate"][0]), 1.0)), confidence_level=1.0 * f2)
        assert a.integers(1 << 30) == b.integers(1 << 30)
    assert list(inspect.signature(driver.pbt_explore).parameters)[:5] == ["flags", "axes", "rng", "targets", "resample_probability"]


def test_pbt_with_the_axis_calls_in_order(monkeypatch):
    stubbed(monkeypatch)
    grid = {"selector": ["eps", "ucb"], "learning_rate": [0.1, 0.2, 0.3, 0.4]}
    res = driver.run_pbt("taxi", grid, interval=10, fraction=0.25, pbt_seed=11, resample_probability=0.5, agents_per_point=2,
                         n_episodes=60, verbose=False)
    eng = StubEngine.made[0]
    calls = eng.calls
    assert calls[:2] == [("set_hparams",), ("set_selectors", [0, 0, 0, 0, 1, 1, 1, 1])]
    kinds = [0, 0, 0, 0, 1, 1, 1, 1]
    i, redrawn = 2, 0
    for step in res["lineage"]:
        assert step["pairs"]
        # the winners' selectors first, then the clone, then the retune, then a second call only where a redraw differs
        assert calls[i][0] == "set_selectors" and calls[i + 1][0] == "clone" and calls[i + 2][0] == "retune"
        inherited = list(kinds)
        for p in step["pairs"]:
            inherited[p["loser"]] = kinds[p["winner"]]
        assert calls[i][1] == inherited
        drawn = list(inherited)
        for p in step["pairs"]:
            drawn[p["loser"]] = driver.SELECTOR_NAMES[p["flags"]["selector"]]
        i += 3
        if drawn != inherited:
            assert calls[i] == ("set_selectors", drawn)
            i += 1
            redrawn += 1
        kinds = drawn
    assert i == len(calls) and redrawn > 0
    assert [driver.SELECTOR_NAMES[p["final_params"]["selector"]] for p in res["points"]] == kinds
    assert res["resample_probability"] == 0.5 and res["selector"] is None
    again = driver.run_pbt("taxi", grid, interval=10, fraction=0.25, pbt_seed=11, resample_probability=0.5, agents_per_point=2,
                           n_episodes=60, verbose=False)
    assert json.dumps(again) == json.dumps(res)


def test_pbt_without_the_axis_is_unchanged(monkeypatch):
    stubbed(monkeypatch)
    grid = {"learning_rate": [0.1, 0.2, 0.3, 0.4]}
    res = driver.run_pbt("taxi", grid, interval=10, fraction=0.25, pbt_seed=11, agents_per_point=2, n_episodes=40, verbose=False)
    assert all(c[0] != "set_selectors" for c in StubEngine.made[0].calls)
    assert "resample_probability" not in res and res["selector"] == "eps"
    # the lineage is the draws of the numeric axis alone: replay them
    rng = np.random.default_rng(11)
    cur = [dict(driver.DEFAULTS, learning_rate=v) for v in grid["learning_rate"]]
    stub = StubEngine(0, n_agents=8, selector=0)
    stub.set_hparams([driver.point_hparams(c, 40) for c in cur], np.repeat(np.arange(4), 2))
    for step in res["lineage"]:
        pairs = driver.pbt_exploit(stub._sums(10), 0.25, rng)
        assert [(p["loser"], p["winner"]) for p in step["pairs"]] == [tuple(x) for x in pairs]
        for loser, winner in pairs:
            cur[loser] = driver.pbt_explore(cur[winner], ["learning_rate"], rng)
            assert step["pairs"][0]["flags"]["learning_rate"] == cur[loser]["learning_rate"]
        stub.retune_hparams([driver.point_hparams(c, 40) for c in cur])


def test_halving_with_the_axis(monkeypatch):
    stubbed(monkeypatch)
    res = driver.run_halving("taxi", {"selector": ["eps", "ucb"], "learning_rate": [0.1, 0.2]}, min_episodes=10, eta=2,
                             agents_per_point=2, n_episodes=30, verbose=False)
    assert StubEngine.made[0].calls[:2] == [("set_hparams",), ("set_selectors", [0, 0, 1, 1])]
    assert res["ranking"][0] == 3 and res["selector"] is None


def test_snapshot_load_order():
    src = inspect.getsource(snapshot)
    assert '"hp_selector"' in src and "set_selectors" in src
    load = inspect.getsource(snapshot.load_snapshot)
    # after the sets (which put every set on the engine's selector), before the tables and states (a change resets them)
    assert load.index("set_hparams") < load.index("set_selectors") < load.index("upload_tables") < load.index("set_states")


def ptxas_record(frag, pattern):
    for f in glob.glob(os.path.join(ROOT, "rl-rust_b200", "build", pattern)):
        txt = open(f).read()
        i = txt.find("Function properties for _ZN3rlb" + frag)
        if i >= 0:
            rec = txt[i:i + 600]
            return (int(re.search(r"Used (\d+) registers", rec).group(1)), int(re.search(r"(\d+) bytes spill stores", rec).group(1)),
                    int(re.search(r"(\d+) bytes stack frame", rec).group(1)))
    raise AssertionError("no ptxas record for %s" % frag)


# the _hp twins whose code the position base and the agent list touch, with the figures ptxas gives them (registers,
# spill bytes, stack): the hybrid store's k_run_hp (the base) and the step kernels of the bench cells (the list)
HP_RECORDS = {
    "C2 k_run_hp<FROZEN_LAKE,f32,Basic,eps,traces,hybrid>": ("8k_run_hpILi1EfLi0ELi0ELb1ELi3ELb0E", (209, 0, 0)),
    "k_run_hp<FROZEN_LAKE,f32,Basic,UCB,traces,hybrid>": ("8k_run_hpILi1EfLi0ELi1ELb1ELi3ELb0E", (232, 0, 0)),
    "k_run_hp<CLIFF,f32,Basic,eps,traces,hybrid>": ("8k_run_hpILi2EfLi0ELi0ELb1ELi3ELb0E", (207, 0, 0)),
    "k_update_hp<TAXI,f32,Basic,eps,one-step>": ("11k_update_hpILi3EfLi0ELi0ELb0E", (72, 0, 0)),
    "k_get_action_hp<TAXI,f32,Basic,UCB,one-step>": ("15k_get_action_hpILi3EfLi0ELi1ELb0E", (56, 0, 0)),
}


@pytest.mark.parametrize("name", sorted(HP_RECORDS))
def test_ptxas_records_of_the_hp_twins(name):
    if not glob.glob(os.path.join(ROOT, "rl-rust_b200", "build", "*_hp.ptxas.log")):
        import __graft_entry__
        __graft_entry__.build()
    frag, (regs, spill, stack) = HP_RECORDS[name]
    got = ptxas_record(frag, "*_hp.ptxas.log")
    assert got[0] <= regs and got[1] <= spill and got[2] <= stack, (name, got)

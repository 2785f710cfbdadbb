"""The bootstrap target per hyper-parameter set without a GPU: the new entry point being declared, exported and bound,
the target grid axis against a single engine-wide name and what both reject, the calls a stubbed engine receives (none
without the axis) and the JSON, PBT's inherit-or-resample rule and its draws without the axis, and the snapshot field."""
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

ALL = ["sarsa", "qlearning", "expected_sarsa"]


def test_entry_point_is_declared_exported_and_bound():
    hdr = open(os.path.join(ROOT, "include", "rlb.h")).read()
    assert re.search(r"rlb_status rlb_engine_set_targets\(rlb_engine\* e, const int32_t\* targets, uint32_t n_sets\);", hdr)
    assert "#define RLB_ABI_VERSION 2" in hdr
    assert "rlb_engine_set_targets" in abi.EXPORTS and hasattr(abi.lib, "rlb_engine_set_targets")
    nm = subprocess.run(["nm", "-D", "--defined-only", abi.LIB_PATH], capture_output=True, text=True)
    if nm.returncode == 0:
        assert " rlb_engine_set_targets" in nm.stdout
    fake = abi.Engine.__new__(abi.Engine)       # no device: the checks run before the library is called
    fake.G = 3
    for bad in ([0, 1], [[0, 1, 2]], [0, 1, 3], [-1, 0, 1], [0.0, 1.0, 2.0], ["sarsa", "qlearning", "sarsa"]):
        with pytest.raises(ValueError):
            fake.set_targets(np.asarray(bad))


def test_grid_accepts_the_axis_and_rejects_unknown_names():
    pts = driver.expand_grid({"target": ["sarsa", "expected_sarsa"], "learning_rate": [0.1, 0.2]})
    assert pts == [dict(target="sarsa", learning_rate=0.1), dict(target="sarsa", learning_rate=0.2),
                   dict(target="expected_sarsa", learning_rate=0.1), dict(target="expected_sarsa", learning_rate=0.2)]
    for bad in (["sarsa", "q"], [0, 1], [None]):
        with pytest.raises(ValueError):
            driver.expand_grid({"target": bad})
    hp = driver.point_hparams(dict(driver.DEFAULTS, target="sarsa"), 100)
    assert "target" not in hp and set(hp) == set(abi.HPARAM_FIELDS)
    assert "target" not in driver.SWEEP_FLAGS and "target" not in driver.DEFAULTS


def test_cli_axis_against_a_single_engine_wide_name():
    ap = driver.sweep_parser("test")
    env, grid, _, kw = driver.parse_sweep_args(ap, ["taxi", "--target", "sarsa,qlearning,expected_sarsa", "--learning_rate", "0.1,0.2"])
    assert grid == {"target": ALL, "learning_rate": [0.1, 0.2]} and kw["target"] == "sarsa"
    _, grid, _, kw = driver.parse_sweep_args(driver.sweep_parser("test"), ["taxi", "--target", "expected_sarsa", "--learning_rate", "0.1,0.2"])
    assert grid == {"learning_rate": [0.1, 0.2]} and kw["target"] == "expected_sarsa"      # one name: engine-wide
    _, grid, _, _ = driver.parse_sweep_args(driver.sweep_parser("test"), ["taxi", "--grid", "target=qlearning,sarsa"])
    assert grid == {"target": ["qlearning", "sarsa"]}
    _, grid, _, kw = driver.parse_sweep_args(driver.sweep_parser("test"), ["taxi", "--learning_rate", "0.1"])
    assert kw["target"] == "qlearning" and "target" not in grid                            # the default
    for bad in (["--target", "sarsa,q"], ["--target", "Q"], ["--grid", "target=x"], ["--grid", "target="]):
        with pytest.raises(SystemExit):
            driver.parse_sweep_args(driver.sweep_parser("test"), ["taxi", "--learning_rate", "0.1"] + bad)


class StubEngine:
    """Stands in for abi.Engine: every agent of set g returns 100 * learning_rate + its set's target per episode.
    Records the targets it is given."""
    made = []

    def __init__(self, env_kind, *, n_agents, **kw):
        self.N, self.kw, self.G = n_agents, kw, 0
        self.target_calls, self.targets, self.planning = [], None, None
        StubEngine.made.append(self)

    def set_hparams(self, sets, group):
        self.sets, self.group = [dict(s) for s in sets], np.asarray(group)
        self.G = len(sets)

    def set_targets(self, kinds):
        self.targets = [int(x) for x in kinds]
        self.target_calls.append(self.targets)

    def set_planning_steps(self, steps):
        self.planning = [int(x) for x in steps]

    def set_active_sets(self, mask):
        pass

    def retune_hparams(self, sets):
        self.sets = [dict(s) for s in sets]

    def clone_agents(self, src, dst):
        pass

    def _sums(self, n):
        s = np.zeros((n, self.G, 4))
        for g in range(self.G):
            k = float((self.group == g).sum())
            t = self.targets[g] if self.targets else self.kw["target"]
            s[:, g, 0], s[:, g, 1] = k * 10.0, k * (100.0 * self.sets[g]["learning_rate"] + t)
        return s

    def train(self, n, eval_at, ep_begin=0):
        return dict(sums=self._sums(n - ep_begin), train_steps=(n - ep_begin) * self.G)

    def evaluate(self, n, sums=True):
        return dict(sums=self._sums(n))

    def close(self):
        pass


def stubbed(monkeypatch):
    monkeypatch.setattr(driver.abi, "Engine", StubEngine)
    monkeypatch.setattr(driver.time, "perf_counter", lambda: 0.0)   # "seconds" in the JSON: the same every run
    StubEngine.made = []


# run_sweep's JSON for `--target qlearning`, engine stubbed, as the engine-wide target has always written it
SINGLE_TARGET_JSON = (
    '{"env": "taxi", "agent": "onestep", "selector": "eps", "target": "qlearning", "policy": "basic", "real": "f64"'
    ', "n_episodes": 20, "agents_per_point": 2, "grid": {"learning_rate": [0.1, 0.2]}, "points": [{"params": {"lear'
    'ning_rate": 0.1}, "hparams": {"learning_rate": 0.1, "discount_factor": 0.95, "lambda_factor": 0.5, "initial_ep'
    'silon": 1.0, "epsilon_decay": 0.1, "final_epsilon": 0.0, "confidence_level": 0.5, "default_value": 0.0}, "trai'
    'n_rewards": [11.0, 11.0, 11.0, 11.0, 11.0, 11.0, 11.0, 11.0, 11.0, 11.0, 11.0, 11.0, 11.0, 11.0, 11.0, 11.0, 1'
    '1.0, 11.0, 11.0, 11.0], "train_episodes_length": [10.0, 10.0, 10.0, 10.0, 10.0, 10.0, 10.0, 10.0, 10.0, 10.0, '
    '10.0, 10.0, 10.0, 10.0, 10.0, 10.0, 10.0, 10.0, 10.0, 10.0], "test_rewards": [11.0, 11.0, 11.0, 11.0, 11.0, 11'
    '.0, 11.0, 11.0, 11.0, 11.0, 11.0, 11.0, 11.0, 11.0, 11.0, 11.0, 11.0, 11.0, 11.0, 11.0], "test_episodes_length'
    '": [10.0, 10.0, 10.0, 10.0, 10.0, 10.0, 10.0, 10.0, 10.0, 10.0, 10.0, 10.0, 10.0, 10.0, 10.0, 10.0, 10.0, 10.0'
    ', 10.0, 10.0], "eval_mean_return": 11.0}, {"params": {"learning_rate": 0.2}, "hparams": {"learning_rate": 0.2,'
    ' "discount_factor": 0.95, "lambda_factor": 0.5, "initial_epsilon": 1.0, "epsilon_decay": 0.1, "final_epsilon":'
    ' 0.0, "confidence_level": 0.5, "default_value": 0.0}, "train_rewards": [21.0, 21.0, 21.0, 21.0, 21.0, 21.0, 21'
    '.0, 21.0, 21.0, 21.0, 21.0, 21.0, 21.0, 21.0, 21.0, 21.0, 21.0, 21.0, 21.0, 21.0], "train_episodes_length": [1'
    '0.0, 10.0, 10.0, 10.0, 10.0, 10.0, 10.0, 10.0, 10.0, 10.0, 10.0, 10.0, 10.0, 10.0, 10.0, 10.0, 10.0, 10.0, 10.'
    '0, 10.0], "test_rewards": [21.0, 21.0, 21.0, 21.0, 21.0, 21.0, 21.0, 21.0, 21.0, 21.0, 21.0, 21.0, 21.0, 21.0,'
    ' 21.0, 21.0, 21.0, 21.0, 21.0, 21.0], "test_episodes_length": [10.0, 10.0, 10.0, 10.0, 10.0, 10.0, 10.0, 10.0,'
    ' 10.0, 10.0, 10.0, 10.0, 10.0, 10.0, 10.0, 10.0, 10.0, 10.0, 10.0, 10.0], "eval_mean_return": 21.0}], "ranking'
    '": [1, 0], "seconds": 0.0, "train_steps": 40}')


def test_single_target_json_unchanged(monkeypatch, tmp_path):
    stubbed(monkeypatch)
    out = tmp_path / "sweep.json"
    driver.main_sweep(["taxi", "--target", "qlearning", "--learning_rate", "0.1,0.2", "-n", "20", "--moving_average_window", "20",
                       "--agents_per_point", "2", "--out", str(out)])
    assert StubEngine.made[0].target_calls == [] and StubEngine.made[0].kw["target"] == abi.TARGET_QLEARNING
    assert out.read_text() == SINGLE_TARGET_JSON
    res = driver.run_sweep("taxi", {"learning_rate": [0.1, 0.2]}, target="qlearning", agents_per_point=2, n_episodes=20,
                           moving_average_window=20, verbose=False)
    assert json.dumps(res) == SINGLE_TARGET_JSON


def test_sweep_with_the_axis(monkeypatch, tmp_path):
    stubbed(monkeypatch)
    out = tmp_path / "sweep.json"
    res = driver.main_sweep(["taxi", "--target", "sarsa,expected_sarsa", "--learning_rate", "0.1,0.2", "--planning_steps", "0,3",
                             "-n", "20", "--agents_per_point", "2", "--out", str(out)])
    eng = StubEngine.made[0]
    assert eng.target_calls == [[0, 0, 0, 0, 2, 2, 2, 2]]                   # after set_hparams, one target per point
    assert eng.planning == [0, 3, 0, 3, 0, 3, 0, 3]
    data = json.loads(out.read_text())
    assert data["target"] is None and data["grid"]["target"] == ["sarsa", "expected_sarsa"]
    assert [p["params"]["target"] for p in data["points"]] == ["sarsa"] * 4 + ["expected_sarsa"] * 4
    assert all("target" not in p["hparams"] for p in data["points"])
    assert data["ranking"] == res["ranking"] and data["ranking"][0] in (6, 7)  # lr 0.2 with target 2 scores highest


def test_pbt_explore_inherits_or_resamples():
    flags = dict(target="sarsa", learning_rate=0.1)
    axes = ["target", "learning_rate"]
    with pytest.raises(ValueError):
        driver.pbt_explore(flags, axes, np.random.default_rng(0))          # the axis values are needed
    outs = [driver.pbt_explore(flags, axes, np.random.default_rng(s), ALL, 0.25) for s in range(400)]
    assert outs == [driver.pbt_explore(flags, axes, np.random.default_rng(s), ALL, 0.25) for s in range(400)]   # deterministic
    kept = sum(o["target"] == "sarsa" for o in outs)
    assert 0.75 * 400 < kept < 0.95 * 400 and {o["target"] for o in outs} == set(ALL)   # 0.75 + 0.25 / 3 stay on sarsa
    assert all(o["learning_rate"] in (pytest.approx(0.08), pytest.approx(0.12)) for o in outs)
    assert all(driver.pbt_explore(flags, axes, np.random.default_rng(s), ALL, 0.0)["target"] == "sarsa" for s in range(50))
    # the draws without a target axis are the ones made before: one factor per numeric axis, nothing else
    for s in range(20):
        a, b = np.random.default_rng(s), np.random.default_rng(s)
        got = driver.pbt_explore(dict(learning_rate=0.1, planning_steps=4), ["learning_rate", "planning_steps"], a)
        f1, f2 = driver.PBT_FACTORS[int(b.integers(2))], driver.PBT_FACTORS[int(b.integers(2))]
        assert got == dict(learning_rate=float(min(max(0.1 * f1, driver.PBT_BOUNDS["learning_rate"][0]), 1.0)),
                           planning_steps=driver.pbt_perturb_planning(4, f2))
        assert a.integers(1 << 30) == b.integers(1 << 30)
    assert list(inspect.signature(driver.pbt_explore).parameters)[:3] == ["flags", "axes", "rng"]


def test_pbt_with_the_axis(monkeypatch):
    stubbed(monkeypatch)
    grid = {"target": ALL, "learning_rate": [0.1, 0.2]}
    res = driver.run_pbt("taxi", grid, interval=10, fraction=0.34, pbt_seed=7, resample_probability=0.5, agents_per_point=2,
                         n_episodes=40, verbose=False)
    eng = StubEngine.made[0]
    assert len(eng.target_calls) == 1 + 3                                   # grid_engine, then one per chunk boundary
    for step, targets in zip(res["lineage"], eng.target_calls[1:]):
        for p in step["pairs"]:
            assert p["flags"]["target"] in ALL and targets[p["loser"]] == driver.TARGET_KINDS[p["flags"]["target"]]
    assert [driver.TARGET_KINDS[p["final_params"]["target"]] for p in res["points"]] == eng.target_calls[-1]
    assert res["resample_probability"] == 0.5
    again = driver.run_pbt("taxi", grid, interval=10, fraction=0.34, pbt_seed=7, resample_probability=0.5, agents_per_point=2,
                           n_episodes=40, verbose=False)
    assert json.dumps(again) == json.dumps(res)
    without = driver.run_pbt("taxi", {"learning_rate": [0.1, 0.2]}, interval=10, agents_per_point=2, n_episodes=40, verbose=False)
    assert "resample_probability" not in without and StubEngine.made[-1].target_calls == []
    with pytest.raises(ValueError):
        driver.run_pbt("taxi", grid, interval=10, resample_probability=1.5, agents_per_point=2, n_episodes=40, verbose=False)


def test_halving_with_the_axis(monkeypatch):
    stubbed(monkeypatch)
    res = driver.run_halving("taxi", {"target": ALL}, min_episodes=10, eta=3, agents_per_point=2, n_episodes=30, verbose=False)
    assert StubEngine.made[0].target_calls == [[0, 1, 2]]
    assert res["ranking"][0] == 2 and res["target"] is None


def test_snapshot_field():
    src = inspect.getsource(snapshot)
    assert '"hp_target"' in src and "set_targets" in src
    load = inspect.getsource(snapshot.load_snapshot)
    assert load.index("set_hparams") < load.index("set_targets") < load.index("set_active_sets")

"""Successive halving without a GPU: the rung schedule, the selection with its ties, the driver's rungs, masks and JSON
with the engine stubbed, the rl_halving CLI, and the new entry point being declared, exported and bound."""
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


def test_rung_schedule():
    assert driver.halving_rungs(1000, 100, 2) == [100, 200, 400, 800, 1000]
    assert driver.halving_rungs(1000, 100, 3) == [100, 300, 900, 1000]
    assert driver.halving_rungs(900, 100, 3) == [100, 300, 900]
    assert driver.halving_rungs(100, 100, 3) == [100]
    assert driver.halving_rungs(100, 500, 3) == [100]                      # min_episodes >= n: one rung, run_sweep's run
    assert driver.halving_rungs(10, 1, 10) == [1, 10]
    for bad in ((100, 0, 3), (100, 10, 1)):
        with pytest.raises(ValueError):
            driver.halving_rungs(*bad)


def test_selection_keeps_the_best_with_ties_by_set_index():
    sums = np.zeros((5, 6, 4))
    sums[:, :, 1] = [[3.0, 1.0, 3.0, 2.0, 5.0, 1.0]] * 5
    kept, dropped = driver.halving_select(sums, [0, 1, 2, 3, 4, 5], 2)
    assert kept == [0, 2, 4] and dropped == [3, 1, 5]                      # 4, then the tie 0 < 2; dropped strongest first
    kept, dropped = driver.halving_select(sums, [0, 1, 2, 3, 4, 5], 3)
    assert kept == [0, 4] and dropped == [2, 3, 1, 5]
    kept, dropped = driver.halving_select(sums, [1, 5], 3)                 # max(1, floor(2 / 3)) = 1
    assert kept == [1] and dropped == [5]
    kept, dropped = driver.halving_select(sums, [3], 2)
    assert kept == [3] and dropped == []


class StubEngine:
    """Stands in for abi.Engine.  Every agent of set g returns 100 * learning_rate of its set per episode and lasts 10
    steps; paused sets' rows of the sums are zero, as the library's are.  Records every train call and mask."""
    made = []

    def __init__(self, env_kind, *, n_agents, **kw):
        self.N, self.kw, self.G = n_agents, kw, 0
        self.chunks, self.masks, self.evals = [], [], []
        self.active_sets = None
        StubEngine.made.append(self)

    def set_hparams(self, sets, group):
        self.sets, self.group = [dict(s) for s in sets], np.asarray(group)
        self.G, self.active_sets = len(sets), None

    def set_active_sets(self, mask):
        assert mask is None or len(mask) == self.G
        self.active_sets = None if mask is None or np.all(mask) else np.asarray(mask, bool)
        self.masks.append(None if mask is None else np.asarray(mask, bool).copy())

    def _sums(self, n):
        s = np.zeros((n, self.G, 4))
        for g in range(self.G):
            if self.active_sets is not None and not self.active_sets[g]:
                continue
            k = float((self.group == g).sum())
            s[:, g, 0], s[:, g, 1] = k * 10.0, k * 100.0 * self.sets[g]["learning_rate"]
        return s

    def train(self, n, eval_at, ep_begin=0):
        self.chunks.append((ep_begin, n, eval_at))
        act = self.G if self.active_sets is None else int(self.active_sets.sum())
        return dict(sums=self._sums(n - ep_begin), train_steps=(n - ep_begin) * act)

    def evaluate(self, n, sums=True):
        self.evals.append(None if self.active_sets is None else self.active_sets.copy())
        return dict(sums=self._sums(n))

    def close(self):
        pass


LRS = [0.4, 0.1, 0.8, 0.3, 0.5, 0.7, 0.2, 0.6, 0.8]


def run_stubbed(monkeypatch, fn="run_halving", **kw):
    monkeypatch.setattr(driver.abi, "Engine", StubEngine)
    StubEngine.made = []
    args = dict(agents_per_point=4, n_episodes=200, verbose=False)
    args.update(kw)
    res = getattr(driver, fn)("taxi", {"learning_rate": LRS}, **args)
    return res, StubEngine.made[0]


def test_rungs_masks_and_json(monkeypatch):
    res, eng = run_stubbed(monkeypatch, min_episodes=20, eta=3)
    per, n = 4, 200
    assert eng.N == 9 * per and np.array_equal(eng.group, np.repeat(np.arange(9), per))   # run_sweep's layout
    assert eng.chunks == [(0, 20, 20), (20, 60, 20), (60, 180, 20), (180, 200, 20)]      # chunks of one train(n, n/10)
    # rung 0: 9 sets -> keep 3: lr 0.8 (sets 2 and 8, tie by index) and 0.7 (set 5)
    assert [r["active"] for r in res["rungs"]] == [list(range(9)), [2, 5, 8], [2], [2]]
    assert [r["dropped"] for r in res["rungs"]] == [[0, 1, 3, 4, 6, 7], [5, 8], [], []]
    assert [r["budget"] for r in res["rungs"]] == [20, 60, 180, 200]
    assert [list(np.flatnonzero(m)) for m in eng.masks] == [[2, 5, 8], [2]]
    assert len(eng.evals) == 1 and list(np.flatnonzero(eng.evals[0])) == [2]          # evaluate runs over the survivors
    assert res["min_episodes"] == 20 and res["eta"] == 3
    assert res["train_steps"] == 20 * 9 + 40 * 3 + 120 + 20
    pts = res["points"]
    assert [p["episodes_trained"] for p in pts] == [20, 20, 200, 20, 20, 60, 20, 20, 60]
    assert [p["rung"] for p in pts] == [0, 0, 3, 0, 0, 1, 0, 0, 1]
    window = n // driver.DEFAULTS["moving_average_window"]
    for g, p in enumerate(pts):
        e = p["episodes_trained"]
        assert p["train_rewards"] == driver.moving_average(window, np.full(e, 100.0 * LRS[g]))
        assert p["train_episodes_length"] == driver.moving_average(window, np.full(e, 10.0))
        assert p["last_rung_mean_return"] == pytest.approx(100.0 * LRS[g])
        if g == 2:
            assert p["eval_mean_return"] == pytest.approx(80.0)
            assert p["test_rewards"] == driver.moving_average(window, np.full(n, 80.0))
        else:
            assert p["eval_mean_return"] is None and p["test_rewards"] is None and p["test_episodes_length"] is None
    # survivors by evaluate return, then by episodes trained, then by the last rung's return
    assert res["ranking"] == [2, 8, 5, 7, 4, 0, 3, 6, 1]
    json.dumps(res)


def test_a_single_rung_is_run_sweep(monkeypatch):
    sweep, _ = run_stubbed(monkeypatch, fn="run_sweep")
    halving, eng = run_stubbed(monkeypatch, min_episodes=200, eta=2)
    assert eng.chunks == [(0, 200, 20)] and eng.masks == []
    for k in ("points", "ranking", "train_steps", "grid", "n_episodes", "agents_per_point"):
        if k == "points":
            for a, b in zip(sweep["points"], halving["points"]):
                b = dict(b)
                assert b.pop("episodes_trained") == 200 and b.pop("rung") == 0
                b.pop("last_rung_mean_return")
                assert a == b
        else:
            assert sweep[k] == halving[k], k


def test_halving_is_deterministic(monkeypatch):
    a, _ = run_stubbed(monkeypatch, min_episodes=10, eta=2)
    b, _ = run_stubbed(monkeypatch, min_episodes=10, eta=2)
    a.pop("seconds"), b.pop("seconds")
    assert json.dumps(a) == json.dumps(b)
    with pytest.raises(ValueError):
        run_stubbed(monkeypatch, min_episodes=10, eta=1)


def test_rl_halving_cli(monkeypatch, tmp_path):
    monkeypatch.setattr(driver.abi, "Engine", StubEngine)
    StubEngine.made = []
    out = tmp_path / "halving.json"
    res = driver.main_halving(["taxi", "--grid", "learning_rate=0.1,0.2,0.3,0.4", "--exploration_time", "0.25,0.5", "-n", "100",
                               "--agents_per_point", "2", "--min_episodes", "10", "--eta", "2", "--out", str(out)])
    data = json.loads(out.read_text())
    assert data["grid"] == {"exploration_time": [0.25, 0.5], "learning_rate": [0.1, 0.2, 0.3, 0.4]}
    assert data["min_episodes"] == 10 and data["eta"] == 2
    assert [r["budget"] for r in data["rungs"]] == [10, 20, 40, 80, 100]
    assert [len(r["active"]) for r in data["rungs"]] == [8, 4, 2, 1, 1]
    assert StubEngine.made[0].chunks[-1] == (80, 100, 10) and data["ranking"] == res["ranking"]
    with pytest.raises(SystemExit):
        driver.main_halving(["taxi", "--grid", "learning_rate=0.1,0.2"])                  # --min_episodes is required
    tool = open(os.path.join(ROOT, "tools", "rl_halving.py")).read()
    assert "main_halving" in tool


def test_set_active_sets_is_declared_exported_and_bound(tmp_path):
    hdr = open(os.path.join(ROOT, "include", "rlb.h")).read()
    assert re.search(r"rlb_status rlb_engine_set_active_sets\(rlb_engine\* e, const uint8_t\* active, uint32_t n_sets\);", hdr)
    assert "rlb_engine_set_active_sets" in abi.EXPORTS
    assert hasattr(abi.lib, "rlb_engine_set_active_sets")
    nm = subprocess.run(["nm", "-D", "--defined-only", abi.LIB_PATH], capture_output=True, text=True)
    if nm.returncode == 0:
        assert " rlb_engine_set_active_sets" in nm.stdout
    assert hasattr(abi.Engine, "set_active_sets")

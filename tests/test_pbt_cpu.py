"""Population-based training without a GPU: the driver's ranking, exploit pairs, perturbation, clamping, lineage and JSON
with the engine stubbed, the rl_pbt CLI, and the register budget of k_clone_agents."""
import glob
import importlib
import json
import os
import re

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
abi = importlib.import_module("rl-rust_b200._abi")
driver = importlib.import_module("rl-rust_b200.driver")


def test_clone_kernel_does_not_spill():
    logs = glob.glob(os.path.join(ROOT, "rl-rust_b200", "build", "rlb_clone.ptxas.log"))
    if not logs:
        import __graft_entry__
        __graft_entry__.build()
        logs = glob.glob(os.path.join(ROOT, "rl-rust_b200", "build", "rlb_clone.ptxas.log"))
    txt = open(logs[0]).read()
    i = txt.find("Function properties for ")
    while i >= 0 and "k_clone_agents" not in txt[i:txt.find("\n", i)]:
        i = txt.find("Function properties for ", i + 1)
    assert i >= 0, "no ptxas record for k_clone_agents"
    rec = txt[i:i + 400]
    assert int(re.search(r"(\d+) bytes spill stores", rec).group(1)) == 0
    assert int(re.search(r"(\d+) bytes spill loads", rec).group(1)) == 0
    assert int(re.search(r"(\d+) bytes stack frame", rec).group(1)) == 0


class StubEngine:
    """Stands in for abi.Engine.  Every agent of set g returns 100 * learning_rate of its set per episode, so the ranking
    follows the learning rates in force; records every clone and retune."""
    made = []

    def __init__(self, env_kind, *, n_agents, **kw):
        self.N, self.kw, self.G = n_agents, kw, 0
        self.clones, self.retunes, self.chunks = [], [], []
        StubEngine.made.append(self)

    def set_hparams(self, sets, group):
        self.sets, self.group = [dict(s) for s in sets], np.asarray(group)
        self.G = len(sets)

    def retune_hparams(self, sets):
        assert len(sets) == self.G
        self.sets = [dict(s) for s in sets]
        self.retunes.append([dict(s) for s in sets])

    def clone_agents(self, src, dst):
        self.clones.append((np.asarray(src).copy(), np.asarray(dst).copy()))

    def _sums(self, n):
        s = np.zeros((n, self.G, 4))
        for g in range(self.G):
            k = float((self.group == g).sum())
            s[:, g, 0], s[:, g, 1] = k * 10.0, k * 100.0 * self.sets[g]["learning_rate"]
        return s

    def train(self, n, eval_at, ep_begin=0):
        self.chunks.append((ep_begin, n, eval_at))
        return dict(sums=self._sums(n - ep_begin), train_steps=n - ep_begin)

    def evaluate(self, n, sums=True):
        return dict(sums=self._sums(n))

    def close(self):
        pass


LRS = [0.1, 0.2, 0.3, 0.4, 0.5, 0.6, 0.7, 0.8]


def run_stubbed(monkeypatch, **kw):
    monkeypatch.setattr(driver.abi, "Engine", StubEngine)
    StubEngine.made = []
    args = dict(interval=50, fraction=0.25, agents_per_point=4, n_episodes=200, verbose=False)
    args.update(kw)
    res = driver.run_pbt("taxi", {"learning_rate": LRS, "discount_factor": [0.9]}, **args)
    return res, StubEngine.made[0]


def test_exploit_pairs_bottom_with_top_and_clones_agent_j_to_agent_j(monkeypatch):
    res, eng = run_stubbed(monkeypatch)
    per = 4
    assert eng.N == 8 * per and np.array_equal(eng.group, np.repeat(np.arange(8), per))   # run_sweep's layout
    assert eng.chunks == [(0, 50, 20), (50, 100, 20), (100, 150, 20), (150, 200, 20)]    # one train(n, n/10) in chunks
    assert len(res["lineage"]) == 3 and len(eng.clones) == 3 and len(eng.retunes) == 3
    # first boundary: the learning rates rank the sets; bottom 2 = sets 0 and 1 (weakest first), top 2 = sets 7 and 6
    first = res["lineage"][0]
    assert first["episode"] == 50
    assert [p["loser"] for p in first["pairs"]] == [0, 1]
    assert all(p["winner"] in (6, 7) for p in first["pairs"])
    src, dst = eng.clones[0]
    want_src = np.concatenate([p["winner"] * per + np.arange(per) for p in first["pairs"]])
    want_dst = np.concatenate([p["loser"] * per + np.arange(per) for p in first["pairs"]])
    assert np.array_equal(src, want_src) and np.array_equal(dst, want_dst)
    # explore: the winner's flags, every grid axis times 0.8 or 1.2, through point_hparams to retune_hparams
    for p in first["pairs"]:
        w_lr = LRS[p["winner"]]
        assert p["flags"]["learning_rate"] in (0.8 * w_lr, 1.2 * w_lr)
        assert p["flags"]["discount_factor"] in (0.9 * 0.8, 1.0)                           # 1.08 clamped into [0, 1]
        got = eng.retunes[0][p["loser"]]
        assert got["learning_rate"] == p["flags"]["learning_rate"] and got["discount_factor"] == p["flags"]["discount_factor"]
        assert got["epsilon_decay"] == driver.point_hparams(dict(driver.DEFAULTS, **p["flags"]), 200)["epsilon_decay"]
    for g in range(2, 8):                                                                  # the others keep their values
        assert eng.retunes[0][g]["learning_rate"] == LRS[g]
    # final flags in the output follow the lineage
    last = {}
    for step in res["lineage"]:
        for p in step["pairs"]:
            last[p["loser"]] = p["flags"]
    for g, pt in enumerate(res["points"]):
        assert pt["params"] == {"learning_rate": LRS[g], "discount_factor": 0.9}
        assert pt["final_params"] == last.get(g, pt["params"])
        assert pt["hparams"]["learning_rate"] == pt["final_params"]["learning_rate"]


def test_pbt_is_deterministic_for_a_seed(monkeypatch):
    a, _ = run_stubbed(monkeypatch, pbt_seed=11)
    b, _ = run_stubbed(monkeypatch, pbt_seed=11)
    c, _ = run_stubbed(monkeypatch, pbt_seed=12)
    a.pop("seconds"), b.pop("seconds"), c.pop("seconds")
    assert json.dumps(a) == json.dumps(b)
    assert a["lineage"] != c["lineage"]


def test_fraction_zero_never_clones(monkeypatch):
    res, eng = run_stubbed(monkeypatch, fraction=0.0)
    assert eng.clones == [] and eng.retunes == []
    assert all(step["pairs"] == [] for step in res["lineage"])
    with pytest.raises(ValueError):
        run_stubbed(monkeypatch, fraction=0.6)                                             # top and bottom would overlap


def test_explore_clamps_each_flag_into_its_range():
    class Up:                                                                              # always draws the factor 1.2
        @staticmethod
        def integers(n):
            return 1
    f = dict(driver.DEFAULTS, learning_rate=0.9, discount_factor=0.95, lambda_factor=0.99, initial_epsilon=1.0, final_epsilon=0.9,
             exploration_time=0.5, confidence_level=3.0)
    out = driver.pbt_explore(f, list(driver.SWEEP_FLAGS), Up)
    assert out["learning_rate"] == 1.0 and out["discount_factor"] == 1.0 and out["lambda_factor"] == 1.0
    assert out["initial_epsilon"] == 1.0 and out["final_epsilon"] == 1.0
    assert out["exploration_time"] == 0.5 * 1.2 and out["confidence_level"] == 3.0 * 1.2
    zero = dict(f, learning_rate=0.0, exploration_time=0.0, confidence_level=-1.0, discount_factor=-0.5)
    out = driver.pbt_explore(zero, list(driver.SWEEP_FLAGS), Up)
    assert out["learning_rate"] > 0.0 and out["exploration_time"] > 0.0                    # (0, 1] and > 0
    assert out["confidence_level"] == 0.0 and out["discount_factor"] == 0.0                # >= 0 and [0, 1]
    assert out["max_steps"] == f["max_steps"]                                              # flags off the grid stay


def test_rl_pbt_cli(monkeypatch, tmp_path):
    monkeypatch.setattr(driver.abi, "Engine", StubEngine)
    StubEngine.made = []
    out = tmp_path / "pbt.json"
    res = driver.main_pbt(["taxi", "--grid", "learning_rate=0.1,0.2,0.3,0.4", "--exploration_time", "0.25,0.5", "-n", "100",
                           "--agents_per_point", "2", "--interval", "30", "--fraction", "0.25", "--pbt_seed", "0x10",
                           "--out", str(out)])
    data = json.loads(out.read_text())
    assert data["grid"] == {"exploration_time": [0.25, 0.5], "learning_rate": [0.1, 0.2, 0.3, 0.4]}
    assert data["interval"] == 30 and data["fraction"] == 0.25 and data["pbt_seed"] == 16
    assert len(data["points"]) == 8 and len(data["lineage"]) == 3                          # chunks 30, 30, 30, 10
    assert [len(s["pairs"]) for s in data["lineage"]] == [2, 2, 2]
    assert set(data["lineage"][0]["pairs"][0]["flags"]) == {"exploration_time", "learning_rate"}
    assert StubEngine.made[0].chunks[-1] == (90, 100, 10)
    assert len(data["points"][0]["train_rewards"]) == 100 and data["ranking"] == res["ranking"]
    with pytest.raises(SystemExit):
        driver.main_pbt(["taxi", "--grid", "learning_rate=0.1,0.2"])                       # --interval is required

"""Per-agent hyper-parameter sets without a GPU: the rlb_hparams layout on both sides of the ABI, the register budgets of
the k_run_hp twins of the bench kernels, and the sweep driver's grid, decay and JSON with the engine stubbed."""
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


def test_hparams_layout_matches_the_header(tmp_path):
    import ctypes as C
    src = tmp_path / "sz.c"
    src.write_text('#include <stddef.h>\n#include <stdio.h>\n#include "rlb.h"\nint main(void) { printf("%zu %zu %zu\\n", sizeof(rlb_hparams), '
                   'offsetof(rlb_hparams, confidence_level), offsetof(rlb_hparams, default_value)); return 0; }\n')
    exe = str(tmp_path / "sz")
    subprocess.check_call(["cc", "-I", os.path.join(ROOT, "include"), str(src), "-o", exe])
    size, off_c, off_d = map(int, subprocess.check_output([exe]).split())
    assert size == 64 == C.sizeof(abi.RlbHparams) == abi.HPARAMS_DTYPE.itemsize
    assert off_c == abi.RlbHparams.confidence_level.offset == abi.HPARAMS_DTYPE.fields["confidence_level"][1]
    assert off_d == abi.RlbHparams.default_value.offset == abi.HPARAMS_DTYPE.fields["default_value"][1]
    assert tuple(f for f, _ in abi.RlbHparams._fields_) == abi.HPARAM_FIELDS == abi.HPARAMS_DTYPE.names


# the k_run_hp twins of tests/test_build_cpu.py's bench kernels, with its budgets: (fragment, registers, spill bytes, stack)
HP_KERNELS = {
    "C4 k_run_hp<TAXI,f32,Basic,eps,one-step,HBM>": ("k_run_hpILi3EfLi0ELi0ELb0ELi1ELb0E", 64, 400, 200),
    "C3 k_run_hp<CLIFF,f32,Double,UCB,one-step,HBM>": ("k_run_hpILi2EfLi1ELi1ELb0ELi1ELb0E", 96, 300, 120),
    "C1 k_run_hp<BLACKJACK,f32,Basic,eps,one-step,HBM>": ("k_run_hpILi0EfLi0ELi0ELb0ELi1ELb0E", 64, 400, 200),
    "C2 k_run_hp<FROZEN_LAKE,f32,Basic,eps,traces,hybrid>": ("k_run_hpILi1EfLi0ELi0ELb1ELi3ELb0E", 255, 0, 0),
    "C5 k_run_hp<TAXI,f32,Basic,eps,traces,HBM-lazy>": ("k_run_hpILi3EfLi0ELi0ELb1ELi4ELb0E", 168, 0, 0),
    "C5 k_run_hp<TAXI,f32,Double,UCB,traces,HBM-lazy>": ("k_run_hpILi3EfLi1ELi1ELb1ELi4ELb0E", 128, 300, 128),
}


@pytest.mark.parametrize("name", sorted(HP_KERNELS))
def test_hp_kernels_stay_within_their_twins_budgets(name):
    frag, max_regs, max_spill, max_stack = HP_KERNELS[name]
    logs = glob.glob(os.path.join(ROOT, "rl-rust_b200", "build", "*_hp.ptxas.log"))
    if not logs:
        import __graft_entry__
        __graft_entry__.build()
        logs = glob.glob(os.path.join(ROOT, "rl-rust_b200", "build", "*_hp.ptxas.log"))
    found = None
    for f in logs:
        txt = open(f).read()
        i = txt.find("Function properties for _ZN3rlb8" + frag)
        if i >= 0:
            found = txt[i:i + 600]
            break
    assert found, "no ptxas record for %s" % name
    stack = int(re.search(r"(\d+) bytes stack frame", found).group(1))
    spill = int(re.search(r"(\d+) bytes spill stores", found).group(1))
    regs = int(re.search(r"Used (\d+) registers", found).group(1))
    assert regs <= max_regs and spill <= max_spill and stack <= max_stack, (name, regs, spill, stack)


def test_grid_expansion_and_decay():
    pts = driver.expand_grid({"learning_rate": [0.01, 0.1], "exploration_time": [0.25, 0.5, 0.75]})
    assert len(pts) == 6 and pts[0] == dict(learning_rate=0.01, exploration_time=0.25) and pts[-1] == dict(learning_rate=0.1, exploration_time=0.75)
    f = dict(driver.DEFAULTS, initial_epsilon=0.8, exploration_time=0.25)
    hp = driver.point_hparams(f, 1000)
    assert hp["epsilon_decay"] == 0.8 / (0.25 * 1000)             # run_experiment's derivation (bin/taxi.rs:78)
    assert set(hp) == set(abi.HPARAM_FIELDS)
    with pytest.raises(ValueError):
        driver.expand_grid({"max_steps": [10, 20]})                # an env parameter, not an agent constructor argument


class StubEngine:
    """Stands in for abi.Engine: records the sets and returns sums in which set g's agents all return g + 1 per episode
    and last 10 + g steps."""
    made = []

    def __init__(self, env_kind, *, n_agents, **kw):
        self.N, self.kw, self.G = n_agents, kw, 0
        StubEngine.made.append(self)

    def set_hparams(self, sets, group):
        self.sets, self.group = sets, np.asarray(group)
        self.G = len(sets)

    def _sums(self, n):
        s = np.zeros((n, self.G, 4))
        for g in range(self.G):
            k = float((self.group == g).sum())
            s[:, g, 0], s[:, g, 1] = k * (10 + g), k * (g + 1)
        return s

    def train(self, n, eval_at):
        return dict(sums=self._sums(n), train_steps=123)

    def evaluate(self, n, sums=True):
        return dict(sums=self._sums(n))

    def close(self):
        pass


def test_sweep_json_with_the_engine_stubbed(monkeypatch, tmp_path):
    monkeypatch.setattr(driver.abi, "Engine", StubEngine)
    StubEngine.made = []
    out = tmp_path / "sweep.json"
    res = driver.main_sweep(["taxi", "--grid", "learning_rate=0.01,0.05,0.1,0.2", "--grid", "exploration_time=0.25,0.5,0.75",
                             "--agent", "onestep", "--selector", "eps", "--target", "qlearning", "-n", "100",
                             "--agents_per_point", "8", "--out", str(out)])
    eng = StubEngine.made[0]
    assert eng.N == 12 * 8 and len(eng.sets) == 12
    assert np.array_equal(eng.group, np.repeat(np.arange(12), 8))   # contiguous groups
    assert eng.sets[1]["epsilon_decay"] == 1.0 / (0.5 * 100) and eng.sets[1]["learning_rate"] == 0.01
    data = json.loads(out.read_text())
    assert data["grid"] == {"learning_rate": [0.01, 0.05, 0.1, 0.2], "exploration_time": [0.25, 0.5, 0.75]}
    assert len(data["points"]) == 12 and data["ranking"][0] == 11 and data["ranking"][-1] == 0
    p = data["points"][3]
    assert p["params"] == dict(learning_rate=0.05, exploration_time=0.25)
    assert p["eval_mean_return"] == 4.0
    assert p["train_rewards"] == driver.moving_average(1, np.full(100, 4.0))
    assert p["test_episodes_length"] == driver.moving_average(1, np.full(100, 13.0))
    assert res["n_episodes"] == 100 and res["agents_per_point"] == 8

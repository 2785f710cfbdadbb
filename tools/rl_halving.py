#!/usr/bin/env python
"""Successive halving over one run of a reference bin, every grid point a set of agents of one engine:
python tools/rl_halving.py taxi --grid learning_rate=0.01,0.05,0.1,0.2 --grid exploration_time=0.25,0.5,0.75 \
    --agent onestep --selector eps --target qlearning -n 1000 --agents_per_point 16384 --min_episodes 100 --eta 2 --out halving.json
(see rl-rust_b200/driver.py: run_halving)."""
import importlib
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
if __name__ == "__main__":
    importlib.import_module("rl-rust_b200.driver").main_halving()

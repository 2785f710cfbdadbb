"""Build budgets of k_eval, the evaluate-only kernel of the on-chip stores' evaluate blocks, from the ptxas logs the
Makefile keeps: it is worth its launches only at the occupancy its launch bounds ask for (RLB_EVAL_MINBLOCKS = 8 CTAs of
128 threads per SM for eps-greedy: 64 registers, no spills; RLB_EVAL_UCB_MINBLOCKS = 6 for UCB: 85 registers, a few
spilled words), so a change that pushes it past them shows up here."""
import glob
import os
import re

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

# (mangled-name fragment, max registers, max spill-store bytes, max stack-frame bytes)
KERNELS = {
    "C2 k_eval<FROZEN_LAKE,f32,Basic,eps>": ("k_evalILi1EfLi0ELi0ELb0EE", 64, 0, 0),
    "C2 k_eval<FROZEN_LAKE,f64,Basic,eps>": ("k_evalILi1EdLi0ELi0ELb0EE", 64, 0, 0),
    "C2 k_eval_hp<FROZEN_LAKE,f32,Basic,eps>": ("k_evalILi1EfLi0ELi0ELb1EE", 64, 0, 0),
    "C2 k_eval_hp<FROZEN_LAKE,f64,Basic,eps>": ("k_evalILi1EdLi0ELi0ELb1EE", 64, 0, 0),
    # UCB: RLB_EVAL_UCB_MINBLOCKS = 6 CTAs (85 registers); the f64 bonus math leaves a few spilled words
    "C2-UCB k_eval<FROZEN_LAKE,f32,Basic,UCB>": ("k_evalILi1EfLi0ELi1ELb0EE", 85, 64, 48),
    "C2-UCB k_eval<FROZEN_LAKE,f64,Basic,UCB>": ("k_evalILi1EdLi0ELi1ELb0EE", 85, 64, 48),
    "C2-UCB k_eval_hp<FROZEN_LAKE,f32,Basic,UCB>": ("k_evalILi1EfLi0ELi1ELb1EE", 85, 80, 56),
}


def ptxas_record(frag):
    logs = glob.glob(os.path.join(ROOT, "rl-rust_b200", "build", "*.ptxas.log"))
    if not logs:
        import __graft_entry__
        __graft_entry__.build()
        logs = glob.glob(os.path.join(ROOT, "rl-rust_b200", "build", "*.ptxas.log"))
    for f in logs:
        txt = open(f).read()
        i = txt.find("Function properties for _ZN3rlb6" + frag)
        if i >= 0:
            return txt[i:i + 600]
    return None


@pytest.mark.parametrize("name", sorted(KERNELS))
def test_eval_kernels_stay_in_their_budget(name):
    frag, max_regs, max_spill, max_stack = KERNELS[name]
    found = ptxas_record(frag)
    assert found, "no ptxas record for %s" % name
    stack = int(re.search(r"(\d+) bytes stack frame", found).group(1))
    spill = int(re.search(r"(\d+) bytes spill stores", found).group(1))
    regs = int(re.search(r"Used (\d+) registers", found).group(1))
    assert regs <= max_regs and spill <= max_spill and stack <= max_stack, (name, regs, spill, stack)


@pytest.mark.parametrize("env", [1, 2])
def test_eval_kernel_exists_for_every_variant_of_the_on_chip_envs(env):
    """FrozenLake and CliffWalking: f32 and f64 x Basic and Double x eps-greedy and UCB, plain and with sets."""
    for real in "fd":
        for policy in (0, 1):
            for sel in (0, 1):
                for hp in (0, 1):
                    frag = "k_evalILi%dE%sLi%dELi%dELb%dEE" % (env, real, policy, sel, hp)
                    assert ptxas_record(frag), frag

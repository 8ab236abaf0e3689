"""One seeded step() on the 122- and 372-bus grids with whatever ``OPFG_*`` knobs the environment sets, written to
an .npz: tests/test_kernel_builds.py runs it in a process of its own for each setting of the knobs the library reads
once per process, and compares the file with its own default run."""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

GRIDS = ("1-MV-semiurb--1-sw", "1-HV-urban--0-sw")
OUTPUTS = ("vm", "va", "converged", "iterations", "reward", "objective", "penalty", "cost", "valids", "violations",
           "penalties", "obs", "state")
INFO = ("pf_kernel_used", "cta_envs_per_cta", "cta_tables_staged", "radial_lanes_per_env", "radial_envs_per_cta",
        "score_threads_per_env")


def run_all(n_env=1000):
    import torch
    from opfgym_b200.engine import Engine
    from tests import common
    out = {}
    for name in GRIDS:
        case = common.make_case(name, n_profile_steps=96)
        eng = Engine(case.program, n_env, obs_dtype="float64")
        common.randomize(case, eng, seed=81)
        eng.step()
        torch.cuda.synchronize()
        for k in OUTPUTS:
            out[f"{name}/{k}"] = getattr(eng, k).cpu().numpy()
        out[f"{name}/info"] = np.array([eng.info[k] for k in INFO], np.int64)
        eng.close()
    return out


if __name__ == "__main__":
    np.savez(sys.argv[1], **run_all())

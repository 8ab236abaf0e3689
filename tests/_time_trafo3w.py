"""Developer tool (needs a GPU): kernel 5 time and step time at 32 768 environments on the radial stand-in, with and
without a trafo3w at the substation (its loading as an observation and as Trafo3wOverloadConstraint)."""
import sys; sys.path.insert(0, '.')
import subprocess
import torch
from tests import common
from tests._time_quick import fill, timeit
from opfgym_b200 import net as pn
from opfgym_b200.engine import Engine


def add_trafo3w(net):
    mv, lv = pn.create_bus(net, 20.0), pn.create_bus(net, 10.0)
    net.bus.loc[[mv, lv], "min_vm_pu"], net.bus.loc[[mv, lv], "max_vm_pu"] = 0.9, 1.1
    pn.create_transformer3w_from_parameters(
        net, 0, mv, lv, 110.0, 20.0, 10.0, 40.0, 30.0, 15.0, 12.0, 8.0, 14.0, 0.3, 0.2, 0.25, 20.0, 0.05,
        shift_mv_degree=150.0, shift_lv_degree=150.0, tap_side="mv", tap_neutral=0.0, tap_step_percent=1.5,
        tap_pos=0.0, max_loading_percent=40.0)
    idx = pn.create_loads(net, [mv, lv], [9.0, 4.0], [2.0, 1.0])
    for c in ("p_mw", "q_mvar"):
        net.load.loc[idx, f"min_min_{c}"] = 0.3 * net.load.loc[idx, c]
        net.load.loc[idx, f"max_max_{c}"] = 1.5 * net.load.loc[idx, c]


def main():
    name = sys.argv[1] if len(sys.argv) > 1 else "1-MV-semiurb--1-sw"
    B = int(sys.argv[2]) if len(sys.argv) > 2 else 32768
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip()
    print(f"{name}, {B} environments, {q}")
    for label, prep in (("without trafo3w", None), ("with trafo3w   ", add_trafo3w)):
        case = common.make_case(name, prepare=prep)
        eng = Engine(case.program, B)
        fill(case, eng, B)
        eng.step()
        score = min(timeit(eng.score) for _ in range(3))
        step = min(timeit(eng.step) for _ in range(3))
        print(f"{label}: kernel {eng.info['pf_kernel_used']}, n_trafo3w {case.program.scoring['n_trafo3w']}, "
              f"kernel 5 {score * 1e3:8.1f} us, step {step * 1e3:8.1f} us")


if __name__ == "__main__":
    main()

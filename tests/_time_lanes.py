"""Developer tool: power-flow kernel time, CTA-per-env vs lane-per-env (and any other pf_kernel given)."""
import sys; sys.path.insert(0, '.')
from tests import common
from tests._time_quick import fill, timeit
from opfgym_b200.engine import Engine


def main():
    name = sys.argv[1] if len(sys.argv) > 1 else "1-MV-semiurb--1-sw"
    B = int(sys.argv[2]) if len(sys.argv) > 2 else 32768
    kernels = sys.argv[3].split(',') if len(sys.argv) > 3 else ["cta", "lanes"]
    case = common.make_case(name)
    for kernel in kernels:
        eng = Engine(case.program, B, pf_kernel=kernel)
        fill(case, eng, B)
        eng.assemble()
        ms = timeit(eng.pf_solve)
        i = eng.info
        print(f"{name} B={B} {kernel:8s} kernel={i['pf_kernel_used']} T={i['radial_lanes_per_env']} E={i['radial_envs_per_cta']} "
              f"env_smem={i['radial_smem_bytes_per_env']} W={i['lane_warps_per_cta']} staged={i['lane_tables_staged']} "
              f"max_row={i['lane_max_row']} blocks={i['n_blocks']} levels={i['n_levels']} scratch={i['lane_scratch_bytes']/1e6:.0f} MB "
              f"pf={ms:.3f} ms -> {B/ms*1e3:.3e} env/s iters={eng.iterations.float().mean().item():.2f} "
              f"conv={eng.converged.float().mean().item():.4f}", flush=True)
        eng.close(); del eng


if __name__ == "__main__":
    main()

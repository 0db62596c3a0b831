"""polOrder 2 on triangles at scale on one GPU: ESV2007 on grids.simplex(s), the ALU ladder with 8 s^2 triangles (default
s = 1408: 15.9 M triangles, 95 M DoFs, about 18 GB of matrix values - the size of BASELINE config 4 at scale), assembly,
then "cg.mg2.simplex" to 1e-10 (twice: the first solve allocates the hierarchy) and "cg.blockdiagonal" capped at 300
iterations for comparison.  JSON on stdout: iterations, seconds, seconds per iteration, the true residual recomputed on
the device, L2 / H1-semi errors against ESV2007_EXACT, and the device's name and power limit.
    python tools/quick_bench_p2_mg.py [s]
"""
import json
import subprocess
import sys
import time

sys.path.insert(0, '.')
import dune_hdd_b200 as hdd  # noqa: E402


def device():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=60).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = "unknown"
    return q


def log(*a):
    print("[%.1f s]" % (time.time() - T0), *a, file=sys.stderr, flush=True)


T0 = time.time()


def main(s):
    g = hdd.grids.simplex(s)
    log("grid")
    d = hdd.SWIPDG(g, hdd.problems.ESV2007(), polorder=2)
    t = time.time(); d.init(); t_init = time.time() - t
    ta = min(d.assemble() for _ in range(2))
    log("init + assembly")
    out = {"config": "ESV2007, P2 on grids.simplex(%d): %d triangles" % (s, g.n_cells), "device": device(),
           "dofs": d.num_dofs(), "init_s": t_init, "assemble_s": ta}
    for typ, maxit in (("cg.mg2.simplex", 500), ("cg.mg2.simplex", 500), ("cg.blockdiagonal", 300)):
        try:
            _, info = d.uncached_solve({"type": typ, "precision": 1e-10, "max_iter": maxit}, return_info=True,
                                       copy_to_host=False)
            res = {k: info[k] for k in ("iterations", "converged", "relative_residual", "seconds", "seconds_per_iteration")}
        except hdd.discretizations.linear_solver_failed as e:  # the capped block-Jacobi comparison
            res = {"not_converged": str(e)[-160:], "capped_at": maxit}
        if "iterations" in res:
            res["true_residual"] = d.residual()
            e = d.error_norms(*hdd.problems.ESV2007_EXACT, order=6)
            res["L2"], res["H1_semi"] = e["L2"], e["H1_semi"]
        log(typ, res)
        out.setdefault(typ, []).append(res)
    return out


if __name__ == "__main__":
    print(json.dumps(main(int(sys.argv[1]) if len(sys.argv) > 1 else 1408)))

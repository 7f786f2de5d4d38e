"""CPU baseline leg: the UNMODIFIED Python reference timed on this box's host cores (BASELINE.md 4.1-4.3).

TEST / MEASUREMENT INFRASTRUCTURE ONLY (bench.py's cpu_baseline and ``--impl reference``).  The reference is the pip
install under oracle/_ref (oracle/make_ref.py; git-ignored, shipped to the GPU box), imported through
oracle/ref_harness.py's stubs exactly as when the goldens were made: turbine + mooring stripped, zero mean offset,
C_moor = diag(7e4, 7e4, 0, 0, 0, 1.2e8).  Timed: wall clock around ``Model.solveDynamics`` only (model construction
excluded), one sea state of the workload's seeded table per call; single process (the reference is single-threaded)
and P worker processes over distinct sea states.
"""
import json
import os
import subprocess
import sys
import time

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
REF = os.path.join(HERE, "_ref")

# workload -> (design file under oracle/_ref/inputs, nw, max_freq [Hz], sea-state seed, potModMaster override)
CONFIGS = {
    "cfg1": ("designs/OC3spar.yaml", None, None, None, None),
    "cfg2": ("designs/VolturnUS-S.yaml", 1024, 0.512, 2, 1),
    "sweep": ("designs/VolturnUS-S.yaml", 512, 0.40, 4, 1),
    "cfg3": ("examples/OC4semi-WAMIT_Coefs.yaml", 2048, 0.256, 3, None),
}


def available():
    return os.path.isdir(os.path.join(REF, "raft")) and os.path.isdir(os.path.join(REF, "inputs"))


def _worker(name, first_case, n_cases, budget_s):
    """Runs inside a fresh interpreter: build the reference model, then time solveDynamics per sea state."""
    os.environ["RAFT_REFERENCE_ROOT"] = REF
    os.environ.setdefault("OMP_NUM_THREADS", "1")
    sys.path.insert(0, ROOT)
    import numpy as np
    from oracle import ref_harness as rh
    path, nw, max_freq, seed, master = CONFIGS[name]
    design = rh.load_design(os.path.join(REF, "inputs", path), nw=nw, max_freq=max_freq)
    if master is not None:
        design["platform"]["potModMaster"] = master
    t0 = time.perf_counter()
    model = rh.build_model(design)
    t_build = time.perf_counter() - t0
    if seed is None:
        cases = [rh.make_case(Hs=2.0, Tp=8.0, heading=0.0)]                  # configs[0]: the file's own first case
    else:
        rng = np.random.default_rng(seed)
        n_all = max(64, first_case + n_cases)
        Hs, Tp = rng.uniform(1, 10, n_all), rng.uniform(5, 18, n_all)
        beta = rng.uniform(-180, 180, n_all)
        cases = [rh.make_case(Hs=Hs[i], Tp=Tp[i], heading=beta[i]) for i in range(first_case, first_case + n_cases)]
    done, t_solve = 0, 0.0
    for case in cases:
        t1 = time.perf_counter()
        rh.solve_dynamics(model, case)
        t_solve += time.perf_counter() - t1
        done += model.nw
        if t_solve > budget_s:
            break
    return dict(solves=done, seconds=t_solve, build_s=t_build, nw=int(model.nw))


def _spawn(name, first_case, n_cases, budget_s):
    env = dict(os.environ, PYTHONDONTWRITEBYTECODE="1", OMP_NUM_THREADS="1", OPENBLAS_NUM_THREADS="1", MKL_NUM_THREADS="1")
    return subprocess.Popen([sys.executable, os.path.abspath(__file__), "--worker", name, str(first_case), str(n_cases), str(budget_s)],
                            stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, env=env, cwd=ROOT)


def _collect(procs, timeout):
    out = []
    for p in procs:
        try:
            so, se = p.communicate(timeout=timeout)
        except subprocess.TimeoutExpired:
            p.kill()
            so, se = p.communicate()
        line = [x for x in so.splitlines() if x.startswith("{")]
        if p.returncode == 0 and line:
            out.append(json.loads(line[-1]))
        else:
            out.append(dict(error=(se or so)[-300:]))
    return out


def measure(workload="cfg2", budget_s=20.0, processes=None):
    """-> dict for the JSON line: solves/s of the unmodified reference, 1 process and P processes, on a bounded sample."""
    if not available():
        return dict(unavailable="oracle/_ref not installed (build() where the reference source tree is present, or oracle/make_ref.py)")
    name = workload if workload in CONFIGS else "cfg2"
    res = dict(kind="reference", code="unmodified WISDEM/RAFT (pip-installed under oracle/_ref), moorpy/ccblade/pyhams/matplotlib import lines stubbed",
               timed="Model.solveDynamics wall clock, model construction excluded")
    one = _collect([_spawn("cfg1", 0, 1, budget_s)], timeout=120)[0]
    if "error" not in one:
        res["cfg1_full"] = dict(value=one["solves"] / one["seconds"], unit="solves/s", cores=1, sample="designs/OC3spar.yaml, %d bins x 1 case (whole config)" % one["nw"])
    single = _collect([_spawn(name, 0, 4, budget_s)], timeout=budget_s * 6 + 120)[0]
    if "error" in single:
        res["error"] = single["error"]
        return res
    res["single_process"] = dict(value=single["solves"] / single["seconds"], unit="solves/s", cores=1,
                                 sample="%s: %d RAO solves (%d bins per sea state), %.1f s" % (name, single["solves"], single["nw"], single["seconds"]))
    P = processes or max(1, min(os.cpu_count() or 1, 32))
    many = [r for r in _collect([_spawn(name, i, 1, budget_s) for i in range(P)], timeout=budget_s * 8 + 240) if "error" not in r]
    if many:
        wall = max(r["seconds"] for r in many)
        res["multi_process"] = dict(value=sum(r["solves"] for r in many) / wall, unit="solves/s", cores=len(many), host_cpus=os.cpu_count(),
                                    sample="%s: %d processes x 1 sea state x %d bins, slowest worker %.1f s" % (name, len(many), many[0]["nw"], wall))
    return res


if __name__ == "__main__":
    if len(sys.argv) >= 6 and sys.argv[1] == "--worker":
        print(json.dumps(_worker(sys.argv[2], int(sys.argv[3]), int(sys.argv[4]), float(sys.argv[5]))))
    else:
        print(json.dumps(measure(sys.argv[1] if len(sys.argv) > 1 else "cfg2", budget_s=float(sys.argv[2]) if len(sys.argv) > 2 else 20.0), indent=1))

#!/usr/bin/env python
"""bench.py -- RAO solves/s of the B200-native hot path (BASELINE.json metric), one JSON line on rank 0.

    python bench.py --gpus N --steps K --warmup W [--impl reference] [--workload cfg2|cfg3|cfg3q|sweep] [--dump-outputs DIR]

A "step" is one pass of the hot path (Model.solveDynamics for every (design, case) unit of the batch:
excitation tables, drag-linearisation fixed-point loop, 6x6 complex impedance solve per frequency).

workload cfg2 (default; BASELINE.json configs[1]): VolturnUS-S strip-theory platform, 1024 bins
    (max_freq 0.512 Hz), 64 JONSWAP sea states (seed 2: Hs~U[1,10], Tp~U[5,18], IEC gamma,
    heading~U[-180,180)), nIter 10, tol 0.01, fp64.  65536 RAO solves per step per GPU.
    N > 1: weak scaling -- every rank gets its own 64 sea states (slice r of the seed-2 stream of 64N)
    and the step ends with ONE all-gather of the RAO block over NCCL (the path's only collective).
workload sweep (BASELINE.json configs[3] shard): 1250 VolturnUS-S geometry variants x 16 sea states x
    512 bins per GPU (10000 designs at N = 8), all-gather of the RAOs at the end of the step.

value = units of all ranks / max-over-ranks device time (CUDA events, inputs resident in HBM).
e2e   = same metric through the host-buffer C-ABI call (pinned host inputs -> H2D -> kernels -> D2H).

--dump-outputs DIR writes what the last timed step returned (Xi, status, ... of every unit) as DIR/<name>.npy in float64,
complex arrays as <name>_real / <name>_imag; inputs are seeded, so two builds can be compared output for output.  One GPU:
every output of the session (Xi, status, B_drag, and F_2nd / F_2nd_mean for cfg3q); N > 1: Xi and status of all ranks'
units, whichever exchange ran.  It covers the solveDynamics path of workloads cfg2, cfg3, cfg3q and sweep; the farm and
flex workloads (bench_extra.py) and --impl reference (the CPU checker, not this project's code) refuse it.
bench.py writes nothing into the tree, which may be read-only.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True          # no __pycache__ in the tree

METRIC = "RAO solves/sec (freq-bins x cases x designs)"
UNIT = "solves/s"
DUMP_LIMIT = 60 << 20                   # bytes of --dump-outputs in all (< 64 MB)


def sea_states(seed, n):
    rng = np.random.default_rng(seed)
    return dict(Hs=rng.uniform(1, 10, n), Tp=rng.uniform(5, 18, n), gamma=np.zeros(n),
                beta_deg=rng.uniform(-180, 180, n), spec=np.zeros(n, dtype=np.int32))


def load_packed(name):
    z = np.load(os.path.join(ROOT, "tests", "golden", name + ".npz"))
    return {k[2:]: z[k] for k in z.files if k.startswith("P_")}


def build_workload(args, rank, world):
    """-> (list of packed designs, case dict, config dict) for this rank."""
    from raft_b200 import grid
    if args.workload == "cfg2":
        P = grid.regrid(load_packed("cfg2_VolturnUS-S_nw64"), args.nw or 1024, 0.512)
        nC = args.cases or 64
        # weak scaling by cases: rank r draws its own sea states with seed 2 + 1000 r, so rank 0 solves the N = 1 workload at every N
        cs = sea_states(2 + 1000 * rank, nC)
        cfg = dict(workload="cfg2: designs/VolturnUS-S.yaml (strip theory, turbine+mooring stripped, C_moor=diag(7e4,7e4,0,0,0,1.2e8)), "
                            "%d freq bins x %d sea states per GPU (rank r: seed 2 + 1000 r), fp64, nIter=10, tol=0.01" % (len(P["w"]), nC),
                   designs_per_gpu=1, cases_per_gpu=nC, nw=len(P["w"]), submerged_nodes=int(len(P["node_ls"])))
        return [P], cs, cfg
    elif args.workload in ("cfg3", "cfg3q"):
        # BASELINE.json configs[2]: OC4semi with WAMIT added-mass/damping/excitation tables, 2048 bins x 256 sea states
        from raft_b200 import bem, packer
        from raft_b200.fowt import FOWT
        nw, nC = args.nw or 2048, args.cases or 256
        D = json.load(open(os.path.join(ROOT, "tests", "golden", "designs.json")))["cfg3_OC4semi-WAMIT_nw128"]
        z = np.load(os.path.join(ROOT, "tests", "golden", "cfg3_OC4semi-WAMIT_nw128.npz"))
        t = np.load(os.path.join(ROOT, "tests", "golden", "wamit_marin_semi.npz"))
        w = grid.make_w(0.256 / nw, 0.256)
        H = bem.read_hydro(t["A"], t["B"], t["w1"], t["Re"], t["Im"], t["w3"], t["heads"], w, rho=float(z["P_rho"]), g=float(z["P_g"]))
        mats = dict(M_struc=z["P_M0"] - z["A_hydro_morison"], C_struc=z["P_C0"] - z["C_moor"], C_moor=z["C_moor"], **H)
        second = ""
        if args.workload == "cfg3q":
            # as shipped: potSecOrder 2 -- difference-frequency forces from marin_semi.12d (k_qtf_force before the solve)
            q = np.load(os.path.join(ROOT, "tests", "golden", "cfg3q_OC4semi-QTF_nw96.npz"))
            mats.update(qtf=q["P_qtf"], qtf_w=q["P_qtf_w"], qtf_heads=q["P_qtf_heads"])
            D = dict(D, platform=dict(D["platform"], potSecOrder=2))
            second = " + second-order forces from marin_semi.12d (potSecOrder 2)"
        f = FOWT(D, w, depth=float(z["P_depth"]), matrices=mats)
        f.calcHydroConstants()
        cs = sea_states(3 + 1000 * rank, nC)
        cfg = dict(workload="cfg3: examples/OC4semi-WAMIT_Coefs.yaml (potModMaster 3: BEM A/B/X tables via readHydro of marin_semi.1/.3, "
                            "drag-only strips)%s, %d freq bins x %d sea states per GPU, fp64" % (second, nw, nC),
                   designs_per_gpu=1, cases_per_gpu=nC, nw=nw)
        return [f.pack()], cs, cfg
    else:
        from raft_b200 import sweep
        nD = args.designs or 1250
        nC = args.cases or 16
        base = json.load(open(os.path.join(ROOT, "tests", "golden", "designs.json")))["cfg2_VolturnUS-S_nw64"]
        z = np.load(os.path.join(ROOT, "tests", "golden", "cfg2_VolturnUS-S_nw64.npz"))
        mats = dict(M_struc=z["P_M0"] - z["A_hydro_morison"], C_struc=z["P_C0"] - z["C_moor"], C_moor=z["C_moor"])
        fac = sweep.sample_factors(nD * world, seed=40)[rank * nD:(rank + 1) * nD]
        nw, depth = args.nw or 512, float(z["P_depth"])
        t0 = time.perf_counter()
        batch = sweep.build_variants_batched(base, mats, fac, nw=nw, max_freq=0.40, depth=depth)      # all designs in one pass
        t_build = time.perf_counter() - t0
        t0 = time.perf_counter()
        sweep.build_variants_batched(base, mats, fac, nw=nw, max_freq=0.40, depth=depth)              # a later shard of the same sweep:
        t_build_warm = time.perf_counter() - t0                                                        # the grid's wave numbers are cached
        designs = SweepDesigns(batch, lambda i: sweep.build_variants(base, mats, fac[i:i + 1], nw=nw, max_freq=0.40, depth=depth)[0])
        cs = sea_states(4, nC)
        cfg = dict(workload="sweep: %d synthetic VolturnUS-S geometry variants x %d sea states x %d bins per GPU, fp64" % (nD, nC, batch.nw),
                   designs_per_gpu=nD, cases_per_gpu=nC, nw=batch.nw, table_build_s=t_build, table_build_warm_s=t_build_warm,
                   table_builder=("raft_b200.batch_builder (vectorised NumPy over the design axis)" if os.environ.get("RAFTK_NO_NATIVE_BUILDER")
                                  else "raftk_build_family_host (native C++ builder, csrc/raftk_builder.h)"))
        return designs, cs, cfg


class SweepDesigns:
    """The sweep shard: ``batch`` is the DesignBatch the batched builder produced (what is solved and timed); indexing
    gives the packed dict of one design from the PER-DESIGN builder (what the CPU checker / baseline consume)."""

    def __init__(self, batch, packed_of, index=None):
        self.batch, self._of, self._cache = batch, packed_of, {}
        self.index = list(range(batch.n_designs)) if index is None else index

    def __len__(self):
        return len(self.index)

    def __getitem__(self, i):
        if isinstance(i, slice):
            return [self[j] for j in range(*i.indices(len(self)))]
        j = self.index[i]
        if j not in self._cache:
            self._cache[j] = self._of(j)
        return self._cache[j]

    def __iter__(self):
        return (self[i] for i in range(len(self)))


def as_batch(designs):
    from raft_b200 import solver
    return designs.batch if isinstance(designs, SweepDesigns) else solver.DesignBatch(designs)


class ClockSampler:
    """SM clock and throttle reasons sampled DURING the timed region.  NVML (nvidia_ml_py) in a thread at
    ~2 ms period -- nvidia-smi -lms is too slow to start for millisecond-scale regions; falls back to one
    nvidia-smi query if NVML is unavailable."""

    def __init__(self, gpu_index):
        self.idx, self.sm, self.reasons, self.max_mhz, self.run, self.th, self.ok = gpu_index, [], set(), None, False, None, False
        try:
            import pynvml
            self.nv = pynvml
            pynvml.nvmlInit()
            uuid = None
            try:
                import torch
                uuid = str(torch.cuda.get_device_properties(gpu_index).uuid)
            except Exception:
                pass
            self.h = None
            if uuid:
                for cand in ("GPU-" + uuid, uuid):
                    try:
                        self.h = pynvml.nvmlDeviceGetHandleByUUID(cand.encode() if isinstance(cand, str) else cand)
                        break
                    except Exception:
                        self.h = None
            if self.h is None:
                self.h = pynvml.nvmlDeviceGetHandleByIndex(gpu_index)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
            self.ok = True
        except Exception:
            self.ok = False

    def _loop(self):
        nv = self.nv
        names = (("hw_slowdown", "nvmlClocksEventReasonHwSlowdown", 0x8), ("hw_thermal_slowdown", "nvmlClocksEventReasonHwThermalSlowdown", 0x40),
                 ("sw_thermal_slowdown", "nvmlClocksEventReasonSwThermalSlowdown", 0x20), ("sw_power_cap", "nvmlClocksEventReasonSwPowerCap", 0x4))
        while self.run:
            try:
                self.sm.append(float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)))
                try:
                    r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for nm, _, bit in names:
                    if r & bit:
                        self.reasons.add(nm)
            except Exception:
                pass
            time.sleep(0.002)

    def start(self):
        if self.ok:
            self.run = True
            self.th = threading.Thread(target=self._loop, daemon=True)
            self.th.start()

    def stop(self):
        if self.ok:
            self.run = False
            self.th.join(timeout=1.0)
            return dict(sm_mhz=float(np.median(self.sm)) if self.sm else None, sm_max_mhz=self.max_mhz,
                        reasons=sorted(self.reasons), samples=len(self.sm), source="nvml")
        try:
            q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
            o = subprocess.check_output(["nvidia-smi", "-i", str(self.idx), "--query-gpu=" + q, "--format=csv,noheader,nounits"], text=True)
            f = [x.strip() for x in o.strip().split(",")]
            rs = [n for n, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[2:6]) if v.lower().startswith("active")]
            return dict(sm_mhz=float(f[0]), sm_max_mhz=float(f[1]), reasons=rs, samples=1, source="nvidia-smi (after the region)")
        except Exception:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=["clock query unavailable"], samples=0)


def algorithmic_bytes_per_solve(Ns, Nm, nC, nw, bem=False):
    """SURVEY.md 8(d): Xi out (96) + zeta in (8) + per-frequency tables / nC + per-design tables / (nC nw)."""
    T_f = 784 if bem else 16
    T_d = 208 * Ns + 72 * Nm + 864
    return 96 + 8 + T_f / nC + T_d / (nC * nw)


def algorithmic_flops_per_solve(Ns, passes):
    """SURVEY.md 8(d): (250 Ns + 1.7e3) per pass + 150 Ns for the excitation pass (fp64, real flops)."""
    return (250 * Ns + 1.7e3) * passes + 150 * Ns


def cpu_oracle_rate(designs, cs, min_seconds, nthreads=0):
    """Time the pinned C oracle (kind 'port') on all host threads over a bounded sample of the workload."""
    from oracle import oracle as orc
    orc.build()
    ods = [orc.OracleDesign(P) for P in designs]
    nw = ods[0].nw
    orc.solve_cases(ods[0], {k: v[:1] for k, v in cs.items()}, nIter=10)      # warm-up / page-in
    done, t0, used = 0, time.perf_counter(), 1
    while True:
        for od in ods:
            _, _, used = orc.solve_cases(od, cs, nIter=10, nthreads=nthreads)
            done += len(cs["Hs"]) * nw
            if time.perf_counter() - t0 > min_seconds:
                break
        if time.perf_counter() - t0 > min_seconds:
            break
    dt = time.perf_counter() - t0
    return done / dt, used, done, dt


def response_err(Xi, ref, floor=1e-100):
    """Parity metric for responses [..,6,nw] (DESIGN.md section 6): per frequency, translations and rotations are each
    compared against the largest reference amplitude in their 3-DOF group at that frequency (every frequency is an
    independent linear solve; the three DOFs of a group share units).  Returns the max over everything of
    |Xi-ref| / group_max.  Bins whose group_max is below ``floor`` x the unit's peak amplitude are compared against that
    floor instead: there the wave spectrum itself is a SUBNORMAL double (JONSWAP's exp(-1.25 (Tp f)^-4) at the first
    non-zero bins, S ~ 1e-320 with a handful of significant bits), so the last-bit differences between two libm exp()
    implementations are O(1) relative there while the amplitudes are ~1e-160 of the response peak."""
    Xi, ref = np.asarray(Xi), np.asarray(ref)
    err = 0.0
    peak = np.abs(ref).max(axis=(-2, -1), keepdims=True) if ref.ndim >= 2 else np.abs(ref).max()
    for g in (slice(0, 3), slice(3, 6)):
        d = np.abs(Xi[..., g, :] - ref[..., g, :])
        scale = np.maximum(np.abs(ref[..., g, :]).max(axis=-2, keepdims=True), floor * peak)
        ok = scale > 0
        if np.any(ok):
            err = max(err, float((d / np.where(ok, scale, 1.0))[np.broadcast_to(ok, d.shape)].max()))
    return err


def parity_block(designs, cs, Xi, status, max_designs=8):
    """Outside the timed region: this rank's benchmarked outputs against the pinned C oracle on the SAME inputs
    (BASELINE.md 4.5).  Whole shard when it holds <= max_designs designs, else an evenly spaced sample of designs
    (every case and bin of each).  -> dict for the JSON line."""
    from oracle import oracle as orc
    orc.build()
    nD = len(designs)
    pick = list(range(nD)) if nD <= max_designs else sorted(set(np.linspace(0, nD - 1, max_designs).round().astype(int).tolist()))
    worst, mism, units = 0.0, 0, 0
    for d in pick:
        Xi_o, st_o, _ = orc.solve_cases(orc.OracleDesign(designs[int(d)]), cs, nIter=10, nthreads=os.cpu_count() or 1)
        mism += int(np.sum((status[d, :, 0] != st_o[:, 0]) | (status[d, :, 1] != st_o[:, 1])))
        worst = max(worst, response_err(Xi[d], Xi_o))
        units += Xi_o.shape[0]
    return dict(max_rel_err=worst, pass_mismatch_units=mism, units_checked=units, bins_per_unit=int(Xi.shape[-1]),
                designs_checked=len(pick), designs_in_shard=nD, rtol=1e-10, ok=bool(worst < 1e-10 and mism == 0),
                metric="response_err: max over (unit, DOF, bin) of |Xi - Xi_oracle| / max|Xi_oracle| over the DOF's "
                       "translation/rotation group at that bin (bins whose group amplitude is < 1e-100 of the unit's peak -- subnormal "
                       "wave spectrum -- are measured against that floor); pass_mismatch_units = (design, case) units whose number of "
                       "drag-linearisation passes or converged flag differ",
                checker="oracle/raft_oracle.c (pinned to reference pickles and reference runs: tests/test_oracle_golden.py)")


def sample_outputs(outs, limit=DUMP_LIMIT):
    """Host float64 copies of one step's outputs for --dump-outputs: complex arrays split into <name>_real / <name>_imag,
    integer arrays converted.  Every array leads with the (design, case) unit axes.  Past ``limit`` bytes in all, a fixed
    seeded sample of units is kept, the same units in every array (flattened unit axis), listed in ``sample_units``."""
    import torch
    t0 = next(iter(outs.values()))
    n_units = t0.shape[0] * t0.shape[1]
    per_unit = sum(t[0, 0].numel() * (16 if t.is_complex() else 8) for t in outs.values()) + 8
    keep = None
    if per_unit * n_units > limit:
        keep = np.sort(np.random.default_rng(0).choice(n_units, limit // per_unit, replace=False))
    res = {}
    for k, t in outs.items():
        if keep is not None:
            t = t.flatten(0, 1)[torch.as_tensor(keep, device=t.device)]
        a = t.cpu().numpy()
        if np.iscomplexobj(a):
            res[k + "_real"], res[k + "_imag"] = a.real.astype(np.float64), a.imag.astype(np.float64)
        else:
            res[k] = a.astype(np.float64)
    if keep is not None:
        res["sample_units"] = keep.astype(np.float64)
    return res


def run_reference(args, rank, world):
    """--impl reference: the reference's CPU implementation of the path on the box's host cores.  Two numbers:
    the pinned C oracle port with all host threads (the STRONG CPU figure: value of the line) and, when
    oracle/_ref holds the unmodified Python reference (oracle/make_ref.py), that code itself under the stub
    harness on a bounded sample (cpu_baseline.reference_numpy).  This process never maps libraftk.so."""
    if rank != 0:
        return
    os.environ["RAFTK_NO_NATIVE_BUILDER"] = "1"          # this process must not map libraftk.so: NumPy table builder
    designs, cs, cfg = build_workload(args, 0, 1)
    if len(designs) > 8:
        designs = designs[:8]                        # bounded sample of the sweep
    from oracle import oracle as orc
    orc.build()
    ods = [orc.OracleDesign(P) for P in designs]
    nw = ods[0].nw
    units = len(designs) * len(cs["Hs"]) * nw
    used = 1
    ncpu = os.cpu_count() or 1              # torchrun exports OMP_NUM_THREADS=1; the baseline may use every host core
    for _ in range(args.warmup):
        orc.solve_cases(ods[0], cs, nIter=10, nthreads=ncpu)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        for od in ods:
            _, _, used = orc.solve_cases(od, cs, nIter=10, nthreads=ncpu)
    dt = time.perf_counter() - t0
    val = units * args.steps / dt
    sample = "%d design(s) x %d sea states x %d bins per step, %d steps" % (len(designs), len(cs["Hs"]), nw, args.steps)
    threads = int(min(used, len(cs["Hs"])))          # the port parallelises over cases: never more threads than cases
    cpu = dict(value=val, unit=UNIT, cores=threads, host_cpus=ncpu, kind="port", sample=sample)
    ref = reference_numpy_rate(args.workload, budget_s=20.0)
    if ref is not None:
        cpu["reference_numpy"] = ref
    import raft_b200._lib as _l
    line = dict(metric=METRIC, value=val, unit=UNIT, n_gpus=args.gpus, steps=args.steps, warmup=args.warmup,
                ms_per_step=1e3 * dt / args.steps, higher_is_better=True, scaling="weak", vs_baseline=None, dtype="f64",
                data="synthetic", config=cfg, impl="reference", cpu_baseline=cpu,
                e2e=dict(value=val, unit=UNIT, h2d_bytes_per_step=0, d2h_bytes_per_step=0), gpu_launches=0,
                cuda_library_mapped=bool(_l.loaded()))
    print(json.dumps(line))


def reference_numpy_rate(workload, budget_s=20.0):
    """The UNMODIFIED Python reference (copied by oracle/make_ref.py into oracle/_ref, git-ignored, shipped to the GPU
    box) timed under oracle/ref_harness.py on a bounded sample of the workload, single process (it is single-threaded)
    and P processes.  None when oracle/_ref is absent or the harness cannot run."""
    try:
        from oracle import ref_timing
        return ref_timing.measure(workload, budget_s=budget_s)
    except Exception as e:                                   # noqa: BLE001  (report, never fail the bench on the baseline)
        return dict(unavailable="%s: %s" % (type(e).__name__, str(e)[:200]))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="cfg2", choices=["cfg2", "cfg3", "cfg3q", "sweep", "farm", "flex"])
    ap.add_argument("--nw", type=int, default=0)
    ap.add_argument("--cases", type=int, default=0)
    ap.add_argument("--designs", type=int, default=0)
    ap.add_argument("--turbines", type=int, default=0, help="farm workload: number of FOWTs (default 2 as shipped)")
    ap.add_argument("--cluster", type=int, default=0)
    ap.add_argument("--exchange", default="fused", choices=["fused", "nccl"],
                    help="N>1: 'fused' = the solve kernel stores every finished unit into all ranks' gathered arrays over NVLink "
                         "(peer-mapped memory) + an arrival-flag barrier; 'nccl' = solve, then one all_gather_into_tensor")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-parity", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the sustained-load and sweep-shard extra keys")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the outputs of the last timed step as DIR/<name>.npy (float64; a seeded sample of units past 60 MiB)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl == "reference" or args.workload in ("farm", "flex")):
        ap.error("--dump-outputs covers the solveDynamics path of workloads cfg2, cfg3, cfg3q and sweep")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch
    import torch.distributed as dist
    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback)"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    if args.workload in ("farm", "flex"):
        import bench_extra
        bench_extra.bench_special(args, rank, world, dev)
        if world > 1:
            dist.destroy_process_group()
        return
    from raft_b200 import solver, sweep

    designs, cs, cfg = build_workload(args, rank, world)
    line = measure(args, designs, cs, cfg, rank, world, dev, full=True)
    if not args.no_extras and args.workload == "cfg2":
        # the north-star's multi-GPU configuration next to the default line: configs[3] shard (design sweep), same
        # exchange, fewer steps; carried as an extra key so the driver's per-N records hold it too
        a2 = argparse.Namespace(**vars(args))
        a2.workload, a2.nw, a2.cases, a2.designs, a2.steps, a2.warmup = "sweep", 0, 0, args.designs or 0, max(2, min(args.steps, 3)), 3
        d2, c2, g2 = build_workload(a2, rank, world)
        t_build = g2["table_build_s"]
        sw = measure(a2, d2, c2, g2, rank, world, dev, full=False)
        if rank == 0 and sw is not None:
            sw["e2e_including_table_build"] = dict(
                value=sw["config"]["units_per_step"] / (t_build + sw["e2e"]["ms_per_step"] * 1e-3) if sw.get("e2e") else None, unit=UNIT,
                value_later_shards=sw["config"]["units_per_step"] / (g2["table_build_warm_s"] + sw["e2e"]["ms_per_step"] * 1e-3) if sw.get("e2e") else None,
                note="one sweep step end to end: node-table build of this rank's designs on the host (first shard: including the grid's "
                     "wave numbers; value_later_shards: grid cached) + H2D + solve + exchange + D2H")
            line["sweep"] = sw
    if rank == 0:
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


_FP64_PEAK = 0.0


def measure(args, designs, cs, cfg, rank, world, dev, full):
    """Time one workload on this rank's GPU (all ranks call it together).  -> the JSON line (dict) on rank 0."""
    import torch
    import torch.distributed as dist
    from raft_b200 import solver, sweep
    local = dev.index
    sh, gathered, exch_note = None, None, "none"
    if world > 1 and args.exchange == "fused":
        ok = torch.ones(1, device=dev)
        try:
            sh = sweep.ShardedSolve(as_batch(designs), cs, device=dev)
        except Exception as e:                                # noqa: BLE001  (CUDA IPC unavailable on this box -> NCCL)
            ok.zero_()
            exch_note = "fused exchange unavailable (%s: %s)" % (type(e).__name__, str(e)[:120])
        dist.all_reduce(ok, op=dist.ReduceOp.MIN)
        if ok.item() < 1:
            if sh is not None:
                sh.close()
            sh = None
    if sh is not None:
        batch, cases, sess = sh.batch, sh.cases, sh.sess
    else:
        batch, cases = as_batch(designs), solver.CaseTable(cs)
        sess = solver.DeviceSession(batch, cases, device=dev)
    nD, nC, nw = batch.n_designs, cases.n_cases, batch.nw
    units = nD * nC * nw
    Xi = sess.out["Xi"]
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)      # > 126 MB L2
    if world > 1 and sh is None:
        gathered = torch.empty((world,) + tuple(Xi.shape), dtype=Xi.dtype, device=dev)
    last = {}

    def step():
        if sh is not None:
            last["g"], last["s"] = sh.step(n_iter=10, tol=0.01, xi_start=0.0, cluster_size=args.cluster)
        else:
            sess.solve(n_iter=10, tol=0.01, xi_start=0.0, cluster_size=args.cluster)
            if world > 1:
                dist.all_gather_into_tensor(gathered, Xi)      # fallback exchange: one NCCL collective per step

    # everything with a variable host cost (NVML initialisation of the clock sampler: several ms, different on every rank;
    # its first queries; event creation) happens BEFORE the warm-up steps and the barrier that aligns the ranks -- a rank that
    # enters the timed loop late makes every other rank wait for it in the first exchange, and that wait would be booked as
    # step time (round 1's N = 8 number).  The sampler thread already polls during the warm-up; its samples are reset below.
    sampler = ClockSampler(local)
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    if not os.environ.get("RAFTK_BENCH_NO_SAMPLER"):          # diagnostic switch (tools/r02_n2c.sh): is the NVML thread visible in the step time?
        sampler.start()
    # N > 1: at least 10 untimed steps, so that both alternating gathered buffers of every peer have been written through
    # their NVLink mappings several times before the clock starts (one N = 2 box needed more than 5: profiles/r02_scaling.md)
    n_warm = args.warmup if world == 1 else max(args.warmup, 10)
    for _ in range(n_warm):
        step()
    torch.cuda.synchronize()
    sampler.sm.clear()
    sampler.reasons.clear()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()

    # ---- timed region: K steps, CUDA events on the launching stream, L2 flushed between steps ----
    launches0 = solver.launch_count()
    t_wall0 = time.perf_counter()
    for a, b in ev:
        flush.fill_(1)                       # not timed: evicts the previous step's tables/outputs from L2
        a.record()
        step()
        b.record()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    t_wall = time.perf_counter() - t_wall0
    launches = solver.launch_count() - launches0
    dump = None
    if args.dump_outputs and full:
        # now: the roofline solves below write the same buffers again.  At N > 1 the caller receives every rank's units;
        # both exchanges give Xi and status of all of them (the NCCL one gathers status here, outside the timed steps)
        if sh is not None:
            outs = dict(Xi=last["g"].flatten(0, 1), status=last["s"].flatten(0, 1))
        elif world > 1:
            st_all = torch.empty((world,) + tuple(sess.out["status"].shape), dtype=torch.int32, device=dev)
            dist.all_gather_into_tensor(st_all, sess.out["status"])
            outs = dict(Xi=gathered.flatten(0, 1), status=st_all.flatten(0, 1))
        else:
            outs = sess.out
        if rank == 0:
            dump = sample_outputs(outs)
    clocks = sampler.stop() if sampler.run or not sampler.ok else dict(sm_mhz=None, sm_max_mhz=sampler.max_mhz, reasons=["sampler disabled (diagnostic run)"], samples=0)
    ms = sum(a.elapsed_time(b) for a, b in ev)
    t_ms = torch.tensor([ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t_ms, op=dist.ReduceOp.MAX)
    ms = float(t_ms.item())
    value = units * world * args.steps / (ms * 1e-3)
    if sh is not None:
        assert not sh.timed_out(), "peer arrival barrier timed out"
        nb = Xi.numel() * 16
        exch_note = ("fused into k_rao_fused: every finished unit's Xi (%d B per rank and step) is stored into all %d ranks' gathered "
                     "arrays through peer-mapped pointers (NVLink), then a flag barrier kernel; no NCCL on the data path" % (nb, world))
    elif world > 1:
        exch_note = "all_gather_into_tensor of Xi (%d B per rank) once per step; %s" % (Xi.numel() * 16, exch_note)

    # ---- what the exchange delivered: every rank's block must equal what that rank computed -----------------
    exchange_check = None
    if sh is not None:
        g, s = last["g"], last["s"]
        mine = g[sh.rank].contiguous()
        allb = [torch.empty_like(mine) for _ in range(world)]
        dist.all_gather(allb, mine)
        exchange_check = bool(all(torch.equal(g[r], allb[r]) for r in range(world)))
        assert exchange_check, "fused exchange delivered different data than NCCL all_gather of the same blocks"

    # ---- roofline of the dominant kernel (drag-linearise + solve), timed live with CUDA events ----
    solver.profile_enable(True)
    kms, kn = [0.0, 0.0, 0.0], [0, 0, 0]
    reps = max(3, min(args.steps, 10))
    for _ in range(reps):
        flush.fill_(1)
        sess.solve(n_iter=10, tol=0.01, xi_start=0.0, cluster_size=args.cluster)
        m, n = solver.profile_read()
        kms = [x + y for x, y in zip(kms, m)]
        kn = [x + y for x, y in zip(kn, n)]
    solver.profile_enable(False)
    torch.cuda.synchronize()
    status = sess.out["status"].cpu().numpy()
    Xi_host = sess.out["Xi"].cpu().numpy() if not args.no_parity and rank == 0 else None
    mean_passes = float(status[..., 0].mean())
    k2_ms = kms[2] / max(kn[2], 1)
    per_rank = None
    if world > 1:
        # the solve kernel alone on every rank's own units (no exchange): what the slowest rank costs, as opposed to the exchange
        mine = torch.tensor([k2_ms * kn[2] / reps, float(status[..., 0].max()), mean_passes], dtype=torch.float64, device=dev)
        allr = [torch.zeros_like(mine) for _ in range(world)]
        dist.all_gather(allr, mine)
        per_rank = dict(solve_ms=[round(float(v[0]), 5) for v in allr], max_passes=[int(v[1]) for v in allr], mean_passes=[round(float(v[2]), 3) for v in allr])
    launches_per_step = kn[2] / reps
    Ns, Nm = batch.n_nodes_total / batch.n_designs, batch.n_members_total / batch.n_designs      # mean per design
    b_alg = algorithmic_bytes_per_solve(Ns, Nm, nC, nw, bem=batch.n_bem_head > 0)
    units_per_launch = units / launches_per_step
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
    achieved = b_alg * units_per_launch / (k2_ms * 1e-3) / 1e9
    traffic = None
    try:
        traffic = json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic.json"))).get(args.workload)
    except Exception:
        pass
    roofline = dict(bound="hbm", achieved=achieved, peak=hbm_peak, unit="GB/s", frac=achieved / hbm_peak, traffic=traffic,
                    kernel="k_rao_fused (excitation + drag linearisation + 6x6 solves, on-chip)" if kn[1] == 0 else "k_drag_solve",
                    kernel_ms=k2_ms, share_of_step=kms[2] / max(sum(kms), 1e-30),
                    algorithmic_bytes_per_solve=b_alg, peak_source="MEASURED_PEAKS.json" if peaks else "fallback 6.65 TB/s",
                    other_kernels_ms=dict(depth_table=kms[0] / max(kn[0], 1), excitation=kms[1] / max(kn[1], 1)),
                    note="the contract's two bounds are hbm | tensor; this kernel is neither: ~80 kflop of dependent FP64 per 104 "
                         "algorithmic bytes, DRAM traffic below the algorithmic bytes (tables live on chip). Its binding resource is "
                         "the FP64 pipe: see roofline_fp64 (same kernel, same timing)")
    global _FP64_PEAK
    if rank == 0 and full:
        _FP64_PEAK = solver.fp64_peak_gflops(20000)
    fp64_peak = _FP64_PEAK if rank == 0 else 0.0          # extra keys (sweep shard) reuse the peak measured for the main line
    f_alg = algorithmic_flops_per_solve(Ns, mean_passes)
    fp64_ach = f_alg * units_per_launch / (k2_ms * 1e-3) / 1e9
    roofline_fp64 = dict(bound="fp64", achieved=fp64_ach / 1e3, peak=fp64_peak / 1e3, unit="TFLOP/s",
                         frac=(fp64_ach / fp64_peak) if fp64_peak > 0 else None, algorithmic_flops_per_solve=f_alg,
                         mean_passes=mean_passes, peak_source="DFMA micro-kernel measured in this run")

    # ---- e2e: host buffers in and out, H2D + D2H (and at N > 1 the exchange) inside the timed region ----
    e2e = None
    if not args.no_e2e:
        if sh is not None:
            for _ in range(args.warmup):
                sh.step_host(n_iter=10, cluster_size=args.cluster)
            dist.barrier()
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for _ in range(args.steps):
                xi_h, st_h, h2d, d2h = sh.step_host(n_iter=10, cluster_size=args.cluster)
            dt_e = time.perf_counter() - t0
            st_e = st_h.numpy()
        else:
            for k_, v in list(batch.arrays.items()):
                p = solver.pinned_empty(v.shape, v.dtype); p[...] = v; batch.arrays[k_] = p
            for k_, v in list(cases.arrays.items()):
                p = solver.pinned_empty(v.shape, v.dtype); p[...] = v; cases.arrays[k_] = p
            outs = dict(Xi=solver.pinned_empty([nD, nC, 6, nw], np.complex128), status=solver.pinned_empty([nD, nC, 4], np.int32),
                        B_drag=solver.pinned_empty([nD, nC, 6, 6], np.float64))
            h2d = batch.input_bytes() + cases.input_bytes()
            d2h = int(sum(v.nbytes for v in outs.values()))
            for _ in range(args.warmup):
                solver.solve_dynamics(batch, cases, n_iter=10, cluster_size=args.cluster, out=outs)
            torch.cuda.synchronize()
            if world > 1:
                dist.barrier()
            t0 = time.perf_counter()
            for _ in range(args.steps):
                solver.solve_dynamics(batch, cases, n_iter=10, cluster_size=args.cluster, out=outs)
                if world > 1:
                    dist.all_gather_into_tensor(gathered, Xi)
                    torch.cuda.synchronize()
            torch.cuda.synchronize()
            dt_e = time.perf_counter() - t0
            st_e = outs["status"]
        te = torch.tensor([dt_e], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(te, op=dist.ReduceOp.MAX)
        assert np.array_equal(st_e, status), "e2e and resident paths disagree"
        e2e = dict(value=units * world * args.steps / float(te.item()), unit=UNIT, h2d_bytes_per_step=int(h2d),
                   d2h_bytes_per_step=int(d2h), ms_per_step=1e3 * float(te.item()) / args.steps,
                   includes=("pinned host inputs -> H2D, solve%s, D2H of this rank's Xi + status; wall clock, max over ranks"
                             % (" + fused exchange + arrival barrier" if sh is not None else (" + all-gather" if world > 1 else ""))))

    # ---- sustained load: >= 2 s of back-to-back steps (no flush: inputs + outputs exceed nothing, tables are on chip) ----
    sustained = None
    if full and not args.no_extras:
        samp2 = ClockSampler(local)
        n_rep = max(10, int(2.2e3 / max(ms / args.steps, 1e-3)))
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        samp2.start()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        a.record()
        for _ in range(n_rep):
            step()
        b.record()
        torch.cuda.synchronize()
        ck = samp2.stop()
        t_s = torch.tensor([a.elapsed_time(b)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t_s, op=dist.ReduceOp.MAX)
        sustained = dict(value=units * world * n_rep / (float(t_s.item()) * 1e-3), unit=UNIT, steps=n_rep, seconds=float(t_s.item()) * 1e-3,
                         ms_per_step=float(t_s.item()) / n_rep, clocks=ck, l2="not flushed (back-to-back steps)")

    parity = None
    if rank == 0 and not args.no_parity:
        parity = parity_block(designs, cs, Xi_host, status)
        parity["scope"] = "rank 0's shard of the benchmarked step" if world > 1 else "the benchmarked step"

    cpu = None
    if rank == 0 and world == 1 and full and not args.no_cpu_baseline:
        ncpu = os.cpu_count() or 1
        rate, used, done, dt = cpu_oracle_rate(designs[:4], cs, min_seconds=8.0, nthreads=ncpu)
        cpu = dict(value=rate, unit=UNIT, cores=int(min(used, len(cs["Hs"]))), host_cpus=ncpu, kind="port",
                   sample="%d RAO solves of the same workload (%.1f s, OpenMP over cases, C oracle pinned to the reference)" % (done, dt))
        ref = reference_numpy_rate(args.workload, budget_s=15.0)
        if ref is not None:
            cpu["reference_numpy"] = ref

    line = None
    if rank == 0:
        cfg.update(l2="flushed between timed steps (256 MiB write)", cluster_size=args.cluster or "auto",
                   units_per_step=units * world, mean_passes=mean_passes, wall_s_timed_region=t_wall, collective=exch_note,
                   warmup_steps_run=n_warm)
        line = dict(metric=METRIC, value=value, unit=UNIT, n_gpus=world, steps=args.steps, warmup=args.warmup,
                    ms_per_step=ms / args.steps, higher_is_better=True, scaling="weak", vs_baseline=None, dtype="f64",
                    data="synthetic", config=cfg, clocks=clocks, e2e=e2e, gpu_launches=int(launches),
                    roofline=roofline, roofline_fp64=roofline_fp64, cpu_baseline=cpu, parity=parity)
        if exchange_check is not None:
            line["exchange_verified"] = exchange_check
        if per_rank is not None:
            per_rank["exchange_and_skew_ms"] = ms / args.steps - max(per_rank["solve_ms"])
            per_rank["note"] = ("solve_ms: this rank's solve kernel(s) alone on its own units; a step lasts as long as the slowest rank (a unit's time "
                                "follows its pass count) plus the exchange")
            line["per_rank"] = per_rank
        if sustained is not None:
            line["sustained"] = sustained
    if dump is not None:
        os.makedirs(args.dump_outputs, exist_ok=True)
        for k, a in dump.items():
            np.save(os.path.join(args.dump_outputs, k + ".npy"), a)
    if sh is not None:
        torch.cuda.synchronize()
        dist.barrier()
        sh.close()
    del flush
    torch.cuda.empty_cache()
    return line


if __name__ == "__main__":
    main()

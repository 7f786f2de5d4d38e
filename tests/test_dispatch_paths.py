"""Every kernel path the dispatcher can select, each selected on purpose and checked against the C oracle or the golden fixtures.

The default-path tests run whichever kernel the planner picks for their shapes (almost always k_rao_fused2).  Here each test
first proves which path ran -- from the per-kind launch counts of ``solver.profile_read`` (0 = depth table / fused plan,
1 = excitation / farm, 2 = solve), from the ``solver.launch_count`` delta, or, where no counter tells two paths apart, by
restating the planner's size rule of raftk.cu and asserting which side of the limit the shape is on -- and then compares the
result with the oracle.  A planner change that moves a shape to another kernel makes these tests fail instead of silently
testing the default kernel again.

Paths: the v1 solver (k_depth_table + k_excitation + k_drag_solve mode 0) reached by a 4097-bin grid and forced, incl. its
design-chunk loop; the one-bin fused kernel at both block sizes, with F0 spilled to the workspace, and at a shape the two-bin
kernel would take; the step-class overflow flag and the host's re-run; page-locked outputs written by the solve's epilogue;
the diagonal second-order kernel k_qtf_force<false/true>; the shared-memory farm kernel at 6N = 12; the generalised-DOF LU
at n_dof from 6 to 256, blocked and unblocked."""
import ctypes as C
import os

import numpy as np
import pytest

from conftest import GOLDEN, QTF_GOLDEN, load_golden, relerr, response_err

pytestmark = pytest.mark.gpu
RTOL = 1e-10

# ---- the planner's size rules (raftk_common.cuh, raftk_fused.cuh, raftk_fused2.cuh, raftk.cu) -------------------------------
MEM_STRIDE, CHUNK_NODES, IMEM_STRIDE, NCOEF, F2_T, F2_TRW = 24, 10, 6, 5, 128, 8
SIG_FUSED2, SIG_FUSED1 = [1, 0, 1], [0, 0, 1]


def _classes(b):
    maxW = b.max_w_classes if b.max_w_classes > 0 else b.max_nodes
    maxH = b.max_h_classes if b.max_h_classes > 0 else b.max_nodes
    maxZ = min(b.max_z_classes, b.max_members) if b.max_z_classes > 0 else b.max_members
    return maxW, maxH, maxZ


def fused_smem_bytes(Nm, NsP, nchunk, nwarps, nwl, maxW, maxH, maxZ, f0_smem):
    dbl = (Nm * MEM_STRIDE + 4 * NsP + 16 + NCOEF * NsP + Nm * 8 + 108 + nchunk * nwarps * 32 + 2 * (nchunk * 32 + 2) + nchunk * 32
           + nwarps * 16 * 33 + (12 + (12 if f0_smem else 0) + 4) * nwl + 2 * maxW + maxH + maxZ + 3 * NsP
           + 2 * (Nm + maxZ + (maxW + 1) + (maxH + 1)) * nwl)
    ints = Nm * IMEM_STRIDE + 4 * NsP + 40
    return dbl * 8 + ints * 4 + 32


def fused_try(b, cs):
    """raftk.cu fused_try with a workspace: (accepted, T, nwl, F0 in the workspace)."""
    nwl = -(-b.nw // cs)
    T = 256 if nwl > 128 else 128
    nchunk = -(-b.max_nodes // CHUNK_NODES)
    W, H, Z = _classes(b)
    limit = 112 * 1024 if T == 128 else 226 * 1024
    smem = fused_smem_bytes(b.max_members, b.max_nodes, nchunk, T // 32, nwl, W, H, Z, True)
    spill = smem > limit
    if spill:
        smem = fused_smem_bytes(b.max_members, b.max_nodes, nchunk, T // 32, nwl, W, H, Z, False)
    return smem <= limit and nwl <= 2 * T, T, nwl, spill


def fused2_fits(b, cs):
    """raftk.cu fused2_plan with an explicit cluster size: 192 < bins per CTA <= 256 and <= 113 KB of shared memory."""
    nwl = -(-b.nw // cs)
    if nwl > 2 * F2_T or nwl <= 3 * F2_T // 2:
        return False
    W, H, Z = _classes(b)
    Nm, Ns = b.max_members, b.max_nodes
    nchunk = -(-Ns // CHUNK_NODES)
    p = Nm * MEM_STRIDE + 8 * ((Ns + 1) & ~1) + 108 + 2 * W + H + Z
    p = (p + 1) & ~1
    q = (Nm * IMEM_STRIDE + 3 * (Ns + 12) + 4 + 2 * nchunk + 3) & ~3
    dbl = (p + q // 2) + NCOEF * Ns + Nm * 8 + 36 + nchunk * (F2_T // 32) * 32 + 2 * (nchunk * 32 + 2) + nchunk * 32 + (F2_T // 32) * F2_TRW * 33 + 2
    dbl += 2 * ((W + 1) + (H + 1)) * nwl + 12 * nwl
    return dbl * 8 + 64 <= 113 * 1024


def chunk_bytes(nDc, nC, max_nodes, nw):
    """raftk.cu chunk_bytes: the v1 solver's global tables for nDc designs."""
    al = lambda x: (x + 255) // 256 * 256
    return al(nDc * max_nodes * nw * 16) + al(nDc * nC * max_nodes * nw * 16) + al(nDc * nC * 6 * nw * 16) + al(nC * nw * 8)


def sea_states(seed, n):
    rng = np.random.default_rng(seed)
    return dict(Hs=rng.uniform(1, 10, n), Tp=rng.uniform(5, 18, n), gamma=np.zeros(n), beta_deg=rng.uniform(-180, 180, n),
                spec=np.zeros(n, dtype=np.int32))


@pytest.fixture(scope="module")
def solver():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    from raft_b200 import solver as s
    return s


@pytest.fixture
def prof(solver):
    """Per-kind launch counts of the last solve: prof() -> [plan/depth table, excitation/farm, solve]."""
    solver.profile_enable(True)
    yield lambda: solver.profile_read()[1]
    solver.profile_enable(False)


def _check_vs_oracle(out, Q, cs, oracle, n_iter=10, d=0):
    Xi_o, st_o, _ = oracle.solve_cases(oracle.OracleDesign(Q), cs, nIter=n_iter)
    assert np.array_equal(out["status"][d, :, 0], st_o[:, 0]), (out["status"][d], st_o)
    assert np.array_equal(out["status"][d, :, 1], st_o[:, 1])
    assert np.all(out["status"][d, :, 2] == 0)
    err = response_err(out["Xi"][d], Xi_o)
    assert err < RTOL, err
    return Xi_o


# ================================ v1 solver ========================================================================

def test_v1_solver_reached_by_a_fine_grid(solver, oracle, prof):
    """4097 bins: nwl = 513 > 2 T even at CS = 8, so neither fused planner accepts the slice and run() falls back to the v1
    kernels (full solve, k_drag_solve mode 0)."""
    from raft_b200 import grid
    _, P = load_golden("cfg2_VolturnUS-S_nw64")
    Q = grid.regrid(P, 4097, 0.5)
    b = solver.DesignBatch(Q)
    assert not fused_try(b, 8)[0] and not fused2_fits(b, 8)
    cs = sea_states(31, 3)
    out = solver.solve_dynamics(b, solver.CaseTable(cs), n_iter=10, want=("Xi", "status", "B_drag"))
    assert prof() == [1, 1, 1]
    _check_vs_oracle(out, Q, cs, oracle)


def _golden_cases(G):
    sc = G["ref_run_solve_cases"]
    return dict(Hs=sc[:, 0], Tp=sc[:, 1], gamma=np.zeros(len(sc)), beta_deg=sc[:, 2], spec=np.zeros(len(sc), dtype=np.int32))


@pytest.mark.parametrize("name", ["cfg1_OC3spar", "cfg2_VolturnUS-S_nw64", "test_VolturnUS-S"])
@pytest.mark.parametrize("cluster", [0, 2])
def test_v1_forced_vs_reference_run(name, cluster, solver, oracle, prof, monkeypatch):
    monkeypatch.setenv("RAFTK_FORCE_V1", "1")
    G, P = load_golden(name)
    cases = _golden_cases(G)
    out = solver.solve_dynamics(solver.DesignBatch(P), solver.CaseTable(cases), n_iter=int(G["n_iter"]), xi_start=float(G["xi_start"]),
                                cluster_size=cluster)
    assert prof() == [1, 1, 1]
    assert np.array_equal(out["status"][0, :, 0], G["ref_run_solve_passes"]) and np.all(out["status"][0, :, 2] == 0)
    _, st_o, _ = oracle.solve_cases(oracle.OracleDesign(P), cases, nIter=int(G["n_iter"]), XiStart=float(G["xi_start"]))
    assert np.array_equal(out["status"][0, :, 1], st_o[:, 1])
    assert response_err(out["Xi"][0], G["ref_run_solve_Xi"]) < RTOL


def _three_designs():
    from raft_b200 import grid
    _, Pa = load_golden("cfg2_VolturnUS-S_nw64")
    _, Pb = load_golden("cfg1_OC3spar")
    Qa, Qb = grid.regrid(Pa, 96, 0.384), grid.regrid(Pb, 96, 0.384)
    Qb["depth"] = Qa["depth"]; Qb["k"] = Qa["k"]
    Qc = dict(Qa); Qc["C0"] = Qa["C0"] * 1.3
    return [Qa, Qb, Qc]


def test_v1_forced_design_batch_and_chunk_loop(solver, oracle, prof, monkeypatch):
    """Three designs on the v1 solver; then through DeviceSession with a workspace that holds two designs' tables, so the C-side
    design loop runs two chunks (2 + 1 designs): bit-identical to the single-chunk run."""
    import torch
    monkeypatch.setenv("RAFTK_FORCE_V1", "1")
    Qs = _three_designs()
    batch = solver.DesignBatch(Qs)
    cs = sea_states(11, 5)
    host = solver.solve_dynamics(batch, solver.CaseTable(cs), n_iter=10)
    assert prof() == [1, 1, 1]
    for d, Q in enumerate(Qs):
        _check_vs_oracle(host, Q, cs, oracle, d=d)
    nC, mn, nw = 5, batch.max_nodes, batch.nw
    ws = chunk_bytes(2, nC, mn, nw)
    assert chunk_bytes(1, nC, mn, nw) < ws < chunk_bytes(3, nC, mn, nw)
    sess = solver.DeviceSession(batch, solver.CaseTable(cs), workspace_bytes=ws)
    dev = sess.solve(n_iter=10)
    torch.cuda.synchronize()
    assert prof() == [2, 2, 2]
    assert np.array_equal(dev["Xi"].cpu().numpy(), host["Xi"])
    assert np.array_equal(dev["status"].cpu().numpy(), host["status"])
    assert np.array_equal(dev["B_drag"].cpu().numpy(), host["B_drag"])


def test_v1_refuses_what_only_the_fused_solver_does(solver, monkeypatch):
    """Wave trains and Xi_init / Xi_last need the fused solver: the v1 fallback refuses them with RAFTK_EINVAL and a message."""
    from raft_b200 import _lib, packer
    monkeypatch.setenv("RAFTK_FORCE_V1", "1")
    _, P = load_golden("cfg2_VolturnUS-S_nw64")
    b = solver.DesignBatch(P)
    trains = dict(wave_spectrum=["JONSWAP"] * 2, wave_height=[3.0, 1.0], wave_period=[9.0, 14.0], wave_heading=[0.0, 60.0], wave_gamma=[0.0, 0.0])
    table, _, _ = packer.pack_case_trains([trains])
    with pytest.raises(_lib.RaftkError, match="wave-train cases"):
        solver.solve_dynamics(b, solver.CaseTable(table), n_iter=10)
    cs = sea_states(5, 2)
    with pytest.raises(_lib.RaftkError, match="Xi_last need the fused solver"):
        solver.solve_dynamics(b, solver.CaseTable(cs), n_iter=10, want=("Xi", "status", "Xi_last"))
    Xi0 = np.zeros([1, 2, 6, b.nw], dtype=complex)
    with pytest.raises(_lib.RaftkError, match="Xi_init"):
        solver.solve_dynamics(b, solver.CaseTable(cs, Xi_init=Xi0), n_iter=10)
    ok = solver.solve_dynamics(b, solver.CaseTable(cs), n_iter=10)           # the same batch solves without them
    assert np.all(ok["status"][0, :, 2] == 0) and np.all(ok["status"][0, :, 0] > 0)


# ================================ one-bin fused kernel k_rao_fused<T> ===================================================

@pytest.mark.parametrize("name,nw,cluster,T", [
    ("cfg2_VolturnUS-S_nw64", 64, 1, 128),          # nwl <= 128
    ("cfg2_VolturnUS-S_nw64", 160, 1, 256),         # 128 < nwl <= 192
    ("cfg2_VolturnUS-S_nw64", 300, 1, 256),         # 256 < nwl <= 512
    ("cfg1_OC3spar", 131, 2, 128),                  # ragged: the second CTA owns 65 of 66 bins
])
def test_one_bin_fused_kernel_vs_oracle(name, nw, cluster, T, solver, oracle, prof):
    from raft_b200 import grid
    _, P = load_golden(name)
    Q = grid.regrid(P, nw, 0.512)
    b = solver.DesignBatch(Q)
    ok, T_, nwl, spill = fused_try(b, cluster)
    assert ok and T_ == T and not spill and not fused2_fits(b, cluster)
    cs = sea_states(40 + nw, 3)
    out = solver.solve_dynamics(b, solver.CaseTable(cs), n_iter=10, cluster_size=cluster)
    assert prof() == SIG_FUSED1
    _check_vs_oracle(out, Q, cs, oracle)


def test_one_bin_fused_kernel_with_F0_in_the_workspace(solver, oracle, prof):
    """cfg1 on 4096 bins: the planner takes CS = 8 (512 bins per CTA, T = 256); with F0 in shared memory the slice needs more
    than 226 KB, without it it fits, so the linear excitation lives in the workspace (FPlan.f0_global)."""
    from raft_b200 import grid
    _, P = load_golden("cfg1_OC3spar")
    Q = grid.regrid(P, 4096, 0.5)
    b = solver.DesignBatch(Q)
    ok, T, nwl, spill = fused_try(b, 8)
    assert ok and T == 256 and nwl == 512 and spill and not fused2_fits(b, 8)
    cs = sea_states(43, 3)
    out = solver.solve_dynamics(b, solver.CaseTable(cs), n_iter=10)
    assert prof() == SIG_FUSED1
    _check_vs_oracle(out, Q, cs, oracle)


def test_first_generation_kernel_at_a_two_bin_shape(solver, oracle, prof, monkeypatch):
    """RAFTK_FUSED_GEN1=1 on cfg2 at 1024 bins (the planner's default is k_rao_fused2 at CS = 4): the oracle, and the default
    kernel to rounding (DESIGN.md section 6: the two kernels agree to rounding, not bit for bit)."""
    from raft_b200 import grid
    _, P = load_golden("cfg2_VolturnUS-S_nw64")
    Q = grid.regrid(P, 1024, 0.512)
    b = solver.DesignBatch(Q)
    cs = sea_states(44, 3)
    ref = solver.solve_dynamics(b, solver.CaseTable(cs), n_iter=10)
    assert prof() == SIG_FUSED2 and fused2_fits(b, 4)
    monkeypatch.setenv("RAFTK_FUSED_GEN1", "1")
    out = solver.solve_dynamics(b, solver.CaseTable(cs), n_iter=10)
    assert prof() == SIG_FUSED1
    _check_vs_oracle(out, Q, cs, oracle)
    assert np.array_equal(out["status"], ref["status"])
    assert response_err(out["Xi"][0], ref["Xi"][0]) < 1e-13


# ================================ step-class overflow ================================================================

def _raw_host_solve(solver, batch, cases, outs, n_iter=10):
    """raftk_solve_dynamics_host once, without solve_dynamics' re-run."""
    from raft_b200 import _lib
    d = batch.struct(solver._host_ptr(batch.arrays))
    c = cases.struct(solver._host_ptr(cases.arrays))
    o = _lib.RaftkSolveOpts(n_iter, 0, 0.01, 0.0, 0, 0)
    os_ = solver._out_struct(outs, lambda a: a.ctypes.data)
    _lib.check(_lib.lib.raftk_solve_dynamics_host(C.byref(d), C.byref(c), C.byref(o), C.byref(os_)))


@pytest.mark.parametrize("nw,sig", [(64, SIG_FUSED1), (256, SIG_FUSED2)])
def test_step_class_overflow_and_rerun(nw, sig, solver, oracle, prof):
    """Hints smaller than the device's deduplication: the unit runs no pass, holds zeros (even over a NaN-filled buffer) and
    carries RAFTK_FLAG_PLAN; solve_dynamics re-runs with the table sizes the device's class numbering needs, on the same kernel
    as the correctly hinted call, and returns its result bit for bit."""
    from raft_b200 import _lib, grid
    _, P = load_golden("cfg1_OC3spar")
    Q = grid.regrid(P, nw, 0.512)
    cs = sea_states(45, 3)
    good = solver.DesignBatch(Q)
    assert max(good.max_w_classes, good.max_h_classes, good.max_z_classes) > 1
    assert solver.device_step_classes(good) == (good.max_w_classes, good.max_h_classes, good.max_z_classes)
    ref = solver.solve_dynamics(good, solver.CaseTable(cs), n_iter=10)
    assert prof() == sig
    _check_vs_oracle(ref, Q, cs, oracle)

    low = solver.DesignBatch(Q)
    low.max_w_classes = low.max_h_classes = low.max_z_classes = 1          # before the first call (the struct is cached)
    outs = dict(Xi=np.full([1, 3, 6, nw], np.nan, dtype=complex), status=np.full([1, 3, 4], -1, dtype=np.int32))
    _raw_host_solve(solver, low, solver.CaseTable(cs), outs)
    assert prof() == sig
    assert np.all(outs["status"][0, :, 2] == solver.FLAG_PLAN) and np.all(outs["status"][0, :, 0] == 0)
    assert np.all(outs["Xi"] == 0)
    with pytest.raises(_lib.RaftkError, match="overflowed"):
        solver.raise_on_flags(outs["status"])
    rec = solver.solve_dynamics(low, solver.CaseTable(cs), n_iter=10)
    assert prof() == sig                                                     # the last launch is the re-run: same kernel
    for k in ("Xi", "status", "B_drag"):
        assert np.array_equal(rec[k], ref[k]), k
    solver.raise_on_flags(rec["status"])

    # worst-case tables (hint 0): on the same kernel only table offsets differ -> the same bits.  When they do not fit the
    # kernel the hints ran on, the planner moves the call to the next kernel that fits them, which agrees to rounding.
    worst = solver.DesignBatch(Q)
    worst.max_w_classes = worst.max_h_classes = worst.max_z_classes = 0
    if sig == SIG_FUSED2:
        same_kernel = fused2_fits(worst, 1)
        sig0 = sig if same_kernel else (SIG_FUSED1 if fused_try(worst, 1)[0] or fused_try(worst, 2)[0] else [1, 1, 1])
    else:
        same_kernel = fused_try(worst, 1)[0]
        sig0 = sig if same_kernel else [1, 1, 1]
    w0 = solver.solve_dynamics(worst, solver.CaseTable(cs), n_iter=10)
    assert prof() == sig0
    assert np.array_equal(w0["status"], ref["status"])
    if same_kernel:
        assert np.array_equal(w0["Xi"], ref["Xi"]) and np.array_equal(w0["B_drag"], ref["B_drag"])
    else:
        assert response_err(w0["Xi"][0], ref["Xi"][0]) < 1e-13


def test_step_class_overflow_rerun_keeps_what_only_the_fused_solver_does(solver, prof):
    """An overflowing call with wave trains and Xi_last on cfg2 at 256 bins: its worst-case tables fit no fused kernel (the v1
    solver would refuse the call), so the re-run must use the device's class counts -- and it reproduces the hinted call."""
    from raft_b200 import grid, packer
    _, P = load_golden("cfg2_VolturnUS-S_nw64")
    Q = grid.regrid(P, 256, 0.512)
    worst = solver.DesignBatch(Q)
    worst.max_w_classes = worst.max_h_classes = worst.max_z_classes = 0
    assert not any(fused2_fits(worst, cs) for cs in (1, 2)) and not any(fused_try(worst, cs)[0] for cs in (1, 2))
    trains = dict(wave_spectrum=["JONSWAP"] * 2, wave_height=[3.0, 1.0], wave_period=[9.0, 14.0], wave_heading=[0.0, 60.0], wave_gamma=[0.0, 0.0])
    table, _, _ = packer.pack_case_trains([dict(wave_spectrum="JONSWAP", wave_height=2.0, wave_period=9.0, wave_heading=10.0), trains])
    want = ("Xi", "status", "B_drag", "Xi_last")
    ref = solver.solve_dynamics(solver.DesignBatch(Q), solver.CaseTable(table), n_iter=10, want=want)
    assert prof() == [1, 0, 2] and np.all(ref["status"][0, :, 2] == 0)
    low = solver.DesignBatch(Q)
    low.max_w_classes = low.max_h_classes = low.max_z_classes = 1
    rec = solver.solve_dynamics(low, solver.CaseTable(table), n_iter=10, want=want)
    assert prof() == [1, 0, 2]
    for k in want:
        assert np.array_equal(rec[k], ref[k]), k


# ================================ direct device-to-host epilogue ======================================================

def _pinned_like(solver, ref, keys):
    out = {}
    for k in keys:
        a = solver.pinned_empty(ref[k].shape, ref[k].dtype)
        a[...] = np.nan if a.dtype.kind in "fc" else -7
        out[k] = a
    return out


def _pageable_like(ref, keys):
    return {k: np.full(ref[k].shape, np.nan, dtype=ref[k].dtype) if ref[k].dtype.kind in "fc" else np.full(ref[k].shape, -7, dtype=ref[k].dtype)
            for k in keys}


D2H_CASES = [
    # id, name, nw, cluster, pinned keys, want, signature
    ("fused2", "cfg2_VolturnUS-S_nw64", 256, 0, ("Xi", "status"), ("Xi", "status", "B_drag"), SIG_FUSED2),
    ("fused1", "cfg2_VolturnUS-S_nw64", 64, 1, ("Xi", "status"), ("Xi", "status", "B_drag"), SIG_FUSED1),
    ("fused2_ragged", "cfg2_VolturnUS-S_nw64", 777, 0, ("Xi", "status"), ("Xi", "status"), SIG_FUSED2),
    ("fused1_ragged", "cfg1_OC3spar", 131, 2, ("Xi", "status"), ("Xi", "status"), SIG_FUSED1),
    ("xi_last", "cfg2_VolturnUS-S_nw64", 256, 0, ("Xi", "status", "Xi_last"), ("Xi", "status", "Xi_last"), SIG_FUSED2),
    ("pageable_status", "cfg2_VolturnUS-S_nw64", 256, 0, ("Xi",), ("Xi", "status", "B_drag"), SIG_FUSED2),
    ("v1_shape", "cfg1_OC3spar", 4097, 0, ("Xi", "status"), ("Xi", "status"), [1, 1, 1]),
]


@pytest.mark.parametrize("case", D2H_CASES, ids=[c[0] for c in D2H_CASES])
@pytest.mark.parametrize("no_direct", [False, True], ids=["direct", "copy"])
def test_page_locked_outputs_equal_pageable(case, no_direct, solver, prof, monkeypatch):
    """solve_dynamics(out=...) into page-locked buffers (the solve's epilogue stores Xi / status straight into host memory on
    the fused paths, the copy serves the v1 shape and RAFTK_NO_DIRECT_D2H=1) equals the pageable run bit for bit.  Every
    buffer starts as NaN / -7: a bin the epilogue never stored stays visible.  Whether host_run takes the direct store is not
    observable from here (it follows from a fused plan and a page-locked Xi, both asserted); a missing store in the epilogue
    shows up as NaN, a direct store that no longer happens leaves the copy, which gives the same bits."""
    from raft_b200 import grid
    _, name, nw, cluster, pinned, want, sig = case
    if no_direct:
        monkeypatch.setenv("RAFTK_NO_DIRECT_D2H", "1")
    _, P = load_golden(name)
    b = solver.DesignBatch(grid.regrid(P, nw, 0.5 if nw == 4097 else 0.512))
    cs = solver.CaseTable(sea_states(46, 3))
    ref = solver.solve_dynamics(b, cs, n_iter=10, cluster_size=cluster, want=want)
    assert prof() == sig
    out = _pinned_like(solver, ref, pinned)
    out.update(_pageable_like(ref, [k for k in want if k not in pinned]))
    import torch
    assert torch.from_numpy(out["Xi"]).is_pinned()                       # what host_run's cudaPointerGetAttributes test sees
    assert not torch.from_numpy(out["status"]).is_pinned() or "status" in pinned
    res = solver.solve_dynamics(b, cs, n_iter=10, cluster_size=cluster, want=want, out=out)
    assert prof() == sig
    for k in want:
        assert res[k] is out[k]
        assert np.array_equal(out[k], ref[k]), k
    assert np.all(ref["status"][0, :, 2] == 0)


@pytest.mark.parametrize("nw,cluster,sig", [(256, 0, SIG_FUSED2), (64, 1, SIG_FUSED1)])
def test_page_locked_outputs_of_wave_trains(nw, cluster, sig, solver, oracle, prof):
    """Wave-train table: primaries are stored by the first launch, secondaries by the second; status column 3 of a secondary
    points at its primary (+1)."""
    from raft_b200 import grid, packer
    _, P = load_golden("cfg2_VolturnUS-S_nw64")
    Q = grid.regrid(P, nw, 0.512)
    b = solver.DesignBatch(Q)
    tr = np.array([[6.0, 12.0, 30.0], [2.5, 7.0, -100.0], [1.0, 16.0, 170.0]])
    trains = dict(wave_spectrum=["JONSWAP"] * 3, wave_height=list(tr[:, 0]), wave_period=list(tr[:, 1]), wave_heading=list(tr[:, 2]),
                  wave_gamma=[0.0] * 3)
    table, _, _ = packer.pack_case_trains([dict(wave_spectrum="JONSWAP", wave_height=2.0, wave_period=9.0, wave_heading=10.0), trains])
    cs = solver.CaseTable(table)
    ref = solver.solve_dynamics(b, cs, n_iter=10, cluster_size=cluster)
    assert prof() == [sig[0], 0, 2]
    out = _pinned_like(solver, ref, ("Xi", "status"))
    out.update(_pageable_like(ref, ("B_drag",)))
    solver.solve_dynamics(b, cs, n_iter=10, cluster_size=cluster, out=out)
    for k in ("Xi", "status", "B_drag"):
        assert np.array_equal(out[k], ref[k]), k
    assert list(out["status"][0, :, 3]) == [0, 0, 2, 2]
    Xo, _ = oracle.solve_dynamics_trains(oracle.OracleDesign(Q), np.zeros(3, dtype=np.int32), tr[:, 0], tr[:, 1], np.zeros(3), tr[:, 2], nIter=10)
    assert response_err(out["Xi"][0, 1:4], Xo) < RTOL


# ================================ diagonal second-order kernel k_qtf_force ===============================================

def _qtf_design(P, nw):
    w = np.arange(1, nw + 1) * (2 * np.pi * 0.256 / nw)
    Pb = dict(P, w=w, k=w ** 2 / 9.81, dw=w[1] - w[0])
    for key in ("A_w", "B_w", "X_BEM", "bem_headings"):
        Pb.pop(key, None)
    return Pb


def _tiles_fit(nw, n_qtf_w):
    """raftk.cu run_qtf: the tile kernel runs when its tables fit 226 KB and nw <= 4096."""
    return nw * 68 + (n_qtf_w - 1) * 8 + 16 <= 226 * 1024 and nw <= 4096


def test_diagonal_qtf_kernel_single_heading_vs_oracle(solver, oracle):
    G, P = load_golden(QTF_GOLDEN)
    nw = 3500
    Pb = _qtf_design(P, nw)
    assert len(Pb["qtf_heads"]) == 1 and not _tiles_fit(nw, len(Pb["qtf_w"]))
    cs = sea_states(47, 3)
    n0 = solver.launch_count()
    f = solver.second_order_force(solver.DesignBatch(Pb), solver.CaseTable(cs))
    assert solver.launch_count() - n0 == 1
    od = oracle.OracleDesign(Pb)
    for c in range(3):
        S = oracle.jonswap(Pb["w"], cs["Hs"][c], cs["Tp"][c], 0.0)
        fm, fo = oracle.hydro_force_2nd(od, cs["beta_deg"][c] * 0.017453292519943295, S)
        assert relerr(f["F_2nd"][0, c], fo) < RTOL and relerr(f["F_2nd_mean"][0, c], fm) < RTOL


def test_diagonal_qtf_kernel_heading_interpolation_vs_oracle(solver, oracle):
    """The synthetic 4-heading table of test_second_order_heading_interpolation_and_design_axis (k_qtf_force<true>) at
    headings inside the table, on its entries and outside it (clamped ends)."""
    G, P = load_golden(QTF_GOLDEN)
    Pm = dict(P)
    Pm["qtf"] = np.stack([P["qtf"][:, :, 0, :] * s for s in G["mh_scale"]], axis=2)
    Pm["qtf_heads"] = G["mh_heads"]
    nw = 3500
    Pb = _qtf_design(Pm, nw)
    h = np.rad2deg(np.asarray(G["mh_heads"], dtype=float))             # the table's headings are in radians, cases in degrees
    betas = np.asarray(G["mh_betas_deg"], dtype=float)
    on = np.isclose(betas[:, None], h[None, :], rtol=0, atol=1e-9).any(axis=1)
    outside = (betas < h[0]) | (betas > h[-1])
    assert on.any() and outside.any() and (~on & ~outside).any()
    n = len(betas)
    cs = dict(Hs=np.full(n, 4.0), Tp=np.full(n, 10.0), gamma=np.zeros(n), beta_deg=betas, spec=np.zeros(n, dtype=np.int32))
    n0 = solver.launch_count()
    f = solver.second_order_force(solver.DesignBatch(Pb), solver.CaseTable(cs))
    assert solver.launch_count() - n0 == 1 and not _tiles_fit(nw, len(Pb["qtf_w"]))
    od = oracle.OracleDesign(Pb)
    S = oracle.jonswap(Pb["w"], 4.0, 10.0, 0.0)
    for c in range(n):
        fm, fo = oracle.hydro_force_2nd(od, betas[c] * 0.017453292519943295, S)
        assert relerr(f["F_2nd"][0, c], fo) < RTOL and relerr(f["F_2nd_mean"][0, c], fm) < RTOL, c


def test_diagonal_qtf_kernel_forced_equals_tiles(solver, monkeypatch):
    """nw = 2048 (BASELINE config 3): the tile kernel by default, RAFTK_QTF_DIAG=1 forces the diagonal one; they agree to
    rounding (the tile kernel sums partial results with atomics)."""
    G, P = load_golden(QTF_GOLDEN)
    Pb = _qtf_design(P, 2048)
    b = solver.DesignBatch(Pb)
    cs = solver.CaseTable(sea_states(48, 3))
    assert _tiles_fit(2048, b.n_qtf_w)
    n0 = solver.launch_count()
    tiles = solver.second_order_force(b, cs)
    assert solver.launch_count() - n0 == 2
    monkeypatch.setenv("RAFTK_QTF_DIAG", "1")
    n0 = solver.launch_count()
    diag = solver.second_order_force(b, cs)
    assert solver.launch_count() - n0 == 1
    assert relerr(diag["F_2nd"], tiles["F_2nd"]) < 1e-13 and relerr(diag["F_2nd_mean"], tiles["F_2nd_mean"]) < 1e-13


# ================================ farm: shared-memory warp kernel at 6N = 12 ============================================

def test_farm_warp_kernel_at_12_dofs(solver, monkeypatch):
    """raftk.cu farm_launch: 6N = 12 runs k_farm_rows unless RAFTK_FARM_SMEM is set, then k_farm_response<warp> (6N <= 24).
    Both are one launch of profile kind 1, so no counter tells them apart: this test relies on the environment switch (and
    on the rule restated here) to select the warp kernel."""
    z = np.load(os.path.join(GOLDEN, "farm_VolturnUS-S_farm_nw48.npz"))
    N = int(z["n_fowt"])
    assert 6 * N == 12
    packs = [{k[len("P%d_" % i):]: z[k] for k in z.files if k.startswith("P%d_" % i)} for i in range(N)]
    rows = z["cases"]
    cs = dict(Hs=rows[:, 0], Tp=rows[:, 1], gamma=np.zeros(len(rows)), beta_deg=rows[:, 2], spec=np.zeros(len(rows), dtype=np.int32))
    kw = dict(C_arr=z["C_array"], n_iter=int(z["n_iter"]), xi_start=float(z["xi_start"]))
    by_rows = solver.solve_dynamics_farm(solver.DesignBatch(packs), solver.CaseTable(cs), **kw)
    monkeypatch.setenv("RAFTK_FARM_SMEM", "1")
    warp = solver.solve_dynamics_farm(solver.DesignBatch(packs), solver.CaseTable(cs), **kw)
    assert not np.any(warp["info"]) and np.all(warp["status"][..., 2] == 0)
    ref = z["ref_run_Xi"][:, 0]
    err = max(response_err(warp["Xi_sys"][:, 6 * i:6 * i + 6], ref[:, 6 * i:6 * i + 6]) for i in range(N))
    assert err < RTOL, err
    assert max(response_err(warp["Xi_sys"][:, 6 * i:6 * i + 6], by_rows["Xi_sys"][:, 6 * i:6 * i + 6]) for i in range(N)) < 1e-12
    assert np.array_equal(warp["Xi"], by_rows["Xi"])


# ================================ generalised DOFs: LU at other sizes ==================================================

GB = 8


def _flex():
    z = np.load(os.path.join(GOLDEN, "flex_VolturnUS-S-flexible.npz"))
    P = {k[2:]: z[k] for k in z.files if k.startswith("P_")}
    nw = 24                                                   # the first 24 bins of the fixture's grid
    for k in ("w", "k"):
        P[k] = P[k][:nw]
    for k in ("node_in_p1_w", "node_in_p2_w", "node_Imat_w"):
        P[k] = np.ascontiguousarray(P[k][..., :nw])
    return z, P


def _reduced(z, P, n, seed, cross_panel=False):
    """n < 150: Galerkin reduction on a seeded orthonormal basis R [150, n]; n > 150: decoupled extra DOFs (zero Tn columns,
    diagonal SPD mass / damping / stiffness)."""
    M, B, Cm, Tn = z["gen_M"], z["gen_B"], z["gen_C"], P["gen_Tn"]
    rng = np.random.default_rng(seed)
    if n <= 150:
        R = np.linalg.qr(rng.normal(size=(150, n)))[0] if n < 150 else np.eye(150)
        if cross_panel:
            R = R[:, _pivot_order(M, B, Cm, R, P["w"])]
        Mr, Br, Cr, Tr = R.T @ M @ R, R.T @ B @ R, R.T @ Cm @ R, Tn @ R
    else:
        e = n - 150
        s = np.abs(np.diag(M)).mean(), np.abs(np.diag(B)).mean() + 1.0, np.abs(np.diag(Cm)).mean()
        Mr, Br, Cr = (np.block([[X, np.zeros((150, e))], [np.zeros((e, 150)), np.diag(rng.uniform(0.5, 2.0, e) * sc)]]) for X, sc in zip((M, B, Cm), s))
        Tr = np.concatenate([Tn, np.zeros(Tn.shape[:2] + (e,))], axis=2)
    Q = dict(P, gen_nDOF=np.int32(n), gen_Tn=np.ascontiguousarray(Tr))
    return Q, np.ascontiguousarray(Mr), np.ascontiguousarray(Br), np.ascontiguousarray(Cr)


def _impedance(M, B, Cm, w):
    return -w * w * M + 1j * w * B + Cm


def _pivots(Z):
    """Pivot rows of partial pivoting on |re| + |im|, first maximum wins (the kernels' rule)."""
    A = Z.copy()
    n = len(A)
    piv = []
    for k in range(n):
        m = np.abs(A[k:, k].real) + np.abs(A[k:, k].imag)
        p = k + int(np.argmax(m))
        piv.append(p)
        A[[k, p]] = A[[p, k]]
        A[k + 1:, k] /= A[k, k]
        A[k + 1:, k + 1:] -= np.outer(A[k + 1:, k], A[k, k + 1:])
    return piv


def _pivot_order(M, B, Cm, R, w):
    """Column order of R that makes the first pivot of most bins come from below row GB: DOF 0 is the reduced DOF whose
    largest coupling is off its diagonal most often, the DOF it couples to is placed at row GB + 3."""
    n = R.shape[1]
    Zs = [_impedance(R.T @ M @ R, R.T @ B @ R, R.T @ Cm @ R, wi) for wi in w]
    best, pair = -1, (0, 1)
    for j in range(n):
        col = np.array([np.abs(Z[:, j].real) + np.abs(Z[:, j].imag) for Z in Zs])
        am = col.argmax(axis=1)
        for q in set(am.tolist()) - {j}:
            cnt = int(np.sum(am == q))
            if cnt > best:
                best, pair = cnt, (j, q)
    j, q = pair
    rest = [x for x in range(n) if x not in pair]
    order = [j] + rest[:GB + 2] + [q] + rest[GB + 2:]
    return np.array(order)


def _lu_smem(n):
    """raftk.cu: the blocked LU's panel + row block; it runs when <= 110 KB (always for n_dof <= 256)."""
    return (n * GB + GB * (n + 1)) * 16


def _general_vs_oracle(solver, oracle, z, Q, M, B, Cm, n_cases=2):
    cs = z["ref_run_solve_cases"][:n_cases]
    table = dict(Hs=cs[:, 0], Tp=cs[:, 1], gamma=np.zeros(n_cases), beta_deg=cs[:, 2], spec=np.zeros(n_cases, dtype=np.int32))
    n_iter, xi0 = int(z["n_iter"]), float(z["xi_start"])
    Xi, st = solver.general_solve_dynamics(Q, M, B, Cm, solver.CaseTable(table), n_iter=n_iter, xi_start=xi0)
    gd = oracle.GeneralDesign(Q)
    for c in range(n_cases):
        Xo, so = oracle.general_solve_dynamics(gd, M, B, Cm, 0, cs[c, 0], cs[c, 1], 0.0, cs[c, 2], nIter=n_iter, XiStart=xi0)
        assert st[c, 0] == so[0] and st[c, 1] == so[1] and st[c, 2] == 0, (c, st[c], so)
        err = relerr(Xi[c], Xo)
        assert err < RTOL, (c, err)
    return Xi, st


@pytest.mark.parametrize("n", [6, 7, 8, 9, 17, 150, 151, 256])
def test_general_lu_sizes_vs_oracle(n, solver, oracle):
    z, P = _flex()
    Q, M, B, Cm = _reduced(z, P, n, seed=n)
    assert _lu_smem(n) <= 110 * 1024
    if n in (7, 151):
        # a partial last panel whose pivoting swaps rows (checked on the drag-free impedance): its row swaps are exercised
        kb = n - n % GB
        assert any(p != k for wi in Q["w"] for k, p in enumerate(_pivots(_impedance(M, B, Cm, wi))) if k >= kb)
    _general_vs_oracle(solver, oracle, z, Q, M, B, Cm, n_cases=1 if n == 256 else 2)


def test_general_lu_pivot_across_a_panel_boundary(solver, oracle):
    z, P = _flex()
    Q, M, B, Cm = _reduced(z, P, 17, seed=5, cross_panel=True)
    first = [_pivots(_impedance(M, B, Cm, wi))[0] for wi in Q["w"]]
    assert sum(p >= GB for p in first) >= len(first) // 2, first
    _general_vs_oracle(solver, oracle, z, Q, M, B, Cm)


@pytest.mark.parametrize("n", [17, 151])
def test_general_lu_unblocked_kernel(n, solver, oracle, monkeypatch):
    """RAFTK_GEN_UNBLOCKED=1 keeps the column-at-a-time kernel k_gen_solve: same pivot rule and elimination order as the blocked
    kernel, so the same pass counts and the oracle within tolerance.  The two kernels launch alike and may round alike, so
    no counter or result tells them apart: this test relies on the environment switch to select k_gen_solve."""
    z, P = _flex()
    Q, M, B, Cm = _reduced(z, P, n, seed=n)
    blocked = _general_vs_oracle(solver, oracle, z, Q, M, B, Cm)
    monkeypatch.setenv("RAFTK_GEN_UNBLOCKED", "1")
    un = _general_vs_oracle(solver, oracle, z, Q, M, B, Cm)
    assert np.array_equal(un[1], blocked[1]) and relerr(un[0], blocked[0]) < 1e-12

"""GPU parity tests proper: the sm_100a kernels, called through the C ABI, against
(a) the golden fixtures (reference pickles + reference runs) and (b) the C oracle on larger seeded inputs.

Tolerance: BASELINE.json north_star states fp64 rtol 1e-10 on the RAOs; the metric is
conftest.response_err (per frequency, relative to the largest amplitude in the DOF's unit group).
Pass counts of the drag-linearisation loop must match exactly."""
import numpy as np
import pytest

from conftest import golden_names, load_golden, relerr, response_err

pytestmark = pytest.mark.gpu
NAMES = golden_names()
PICKLED = [n for n in NAMES if n.startswith("test_")]
RTOL = 1e-10


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


@pytest.mark.parametrize("name", PICKLED)
def test_excitation_vs_reference_pickle(name, solver):
    """FOWT.calcHydroExcitation vs the reference's 72-case golden pickle, all cases in one launch."""
    G, P = load_golden(name)
    n = len(G["ref_pickle_exc_F_hydro_iner"])
    cases = solver.CaseTable(dict(Hs=G["ref_pickle_exc_height"].reshape(n), Tp=G["ref_pickle_exc_period"].reshape(n),
                                  gamma=np.zeros(n), beta_deg=G["ref_pickle_exc_heading"].reshape(n), spec=np.zeros(n, dtype=np.int32)))
    out = solver.hydro_excitation(solver.DesignBatch(P), cases)
    ref = G["ref_pickle_exc_F_hydro_iner"]
    if np.abs(ref).max() > 0:
        assert relerr(out["F_iner"][0], ref) < RTOL
    else:
        assert np.abs(out["F_iner"]).max() == 0


@pytest.mark.parametrize("name", NAMES)
def test_excitation_and_linearization_vs_reference_run(name, solver):
    """calcHydroExcitation + calcHydroLinearization(Xi) + calcDragExcitation(0) vs the reference run (unit spectrum)."""
    G, P = load_golden(name)
    cases = solver.CaseTable(dict(Hs=[2.0], Tp=[10.0], gamma=[0.0], beta_deg=[0.0], spec=np.array([1], dtype=np.int32)))
    b = solver.DesignBatch(P)
    exc = solver.hydro_excitation(b, cases)
    assert relerr(exc["zeta"][0], G["ref_run_lin_zeta"]) < 1e-14
    for mine, key in ((exc["F_iner"][0, 0], "ref_run_lin_F_hydro_iner"), (exc["F_BEM"][0, 0], "ref_run_lin_F_BEM")):
        if np.abs(G[key]).max() > 0:
            assert relerr(mine, G[key]) < RTOL
        else:
            assert np.abs(mine).max() == 0
    lin = solver.hydro_linearization(b, cases, G["ref_run_lin_Xi"])
    assert relerr(lin["B_drag"][0, 0], G["ref_run_lin_B_hydro_drag"]) < RTOL
    assert relerr(lin["F_drag"][0, 0], G["ref_run_lin_F_hydro_drag"]) < RTOL
    if "ref_pickle_lin_B_hydro_drag" in G:
        assert relerr(lin["B_drag"][0, 0], G["ref_pickle_lin_B_hydro_drag"]) < RTOL
        assert relerr(lin["F_drag"][0, 0], G["ref_pickle_lin_F_hydro_drag"]) < RTOL


@pytest.mark.parametrize("name", NAMES)
@pytest.mark.parametrize("cluster", [0, 1, 2])
def test_solve_dynamics_vs_reference_run(name, cluster, solver, oracle):
    """Model.solveDynamics vs the unmodified reference: responses within 1e-10, identical pass counts."""
    G, P = load_golden(name)
    sc = G["ref_run_solve_cases"]
    cases = solver.CaseTable(dict(Hs=sc[:, 0], Tp=sc[:, 1], gamma=np.zeros(len(sc)), beta_deg=sc[:, 2],
                                  spec=np.zeros(len(sc), dtype=np.int32)))
    out = solver.solve_dynamics(solver.DesignBatch(P), cases, n_iter=int(G["n_iter"]), xi_start=float(G["xi_start"]),
                                cluster_size=cluster)
    assert np.array_equal(out["status"][0, :, 0], G["ref_run_solve_passes"])
    # converged flag: the reference only prints a warning when the loop runs out (raft_model.py:1138-1140);
    # the pinned oracle carries the flag
    _, st_o, _ = oracle.solve_cases(oracle.OracleDesign(P), cases.arrays, nIter=int(G["n_iter"]), XiStart=float(G["xi_start"]))
    assert np.array_equal(out["status"][0, :, 1], st_o[:, 1]) and np.all(out["status"][0, :, 2] == 0)
    assert response_err(out["Xi"][0], G["ref_run_solve_Xi"]) < RTOL


@pytest.mark.parametrize("name,nw,max_freq,nC", [("cfg2_VolturnUS-S_nw64", 256, 0.512, 12), ("cfg1_OC3spar", 333, 0.40, 5)])
@pytest.mark.parametrize("cluster", [1, 4, 8])
def test_solve_dynamics_vs_oracle_seeded(name, nw, max_freq, nC, cluster, solver, oracle):
    """Larger seeded sweeps against the C oracle (which is pinned to the reference), incl. ragged nw and clusters."""
    from raft_b200 import grid
    _, P = load_golden(name)
    Q = grid.regrid(P, nw, max_freq)
    cs = sea_states(7, nC)
    out = solver.solve_dynamics(solver.DesignBatch(Q), solver.CaseTable(cs), n_iter=10, cluster_size=cluster)
    Xi_o, st_o, _ = oracle.solve_cases(oracle.OracleDesign(Q), cs, nIter=10)
    assert np.array_equal(out["status"][0, :, 0], st_o[:, 0])
    assert np.array_equal(out["status"][0, :, 1], st_o[:, 1])
    assert response_err(out["Xi"][0], Xi_o) < RTOL


def test_bem_design_vs_oracle_seeded(solver, oracle):
    _, P = load_golden("cfg3_OC4semi-WAMIT_nw128")
    cs = sea_states(3, 9)
    cs["beta_deg"][:3] = [0.0, 360.0, -180.0]          # heading-bracket edge cases (raft_fowt.py:1810-1828)
    out = solver.solve_dynamics(solver.DesignBatch(P), solver.CaseTable(cs), n_iter=10, want=("Xi", "status", "F_BEM"))
    od = oracle.OracleDesign(P)
    Xi_o, st_o, _ = oracle.solve_cases(od, cs, nIter=10)
    assert np.array_equal(out["status"][0, :, 0], st_o[:, 0])
    assert response_err(out["Xi"][0], Xi_o) < RTOL
    for c in range(3):
        _, F_BEM, _, _ = oracle.calc_hydro_excitation(od, 0, cs["Hs"][c], cs["Tp"][c], 0.0, cs["beta_deg"][c])
        assert relerr(out["F_BEM"][0, c], F_BEM) < RTOL


def test_design_batch_and_device_session(solver, oracle):
    """Several designs x cases in one batch; device-resident path equals the host path bit for bit."""
    import torch
    from raft_b200 import grid
    _, Pa = load_golden("cfg2_VolturnUS-S_nw64")
    _, Pb = load_golden("cfg1_OC3spar")
    Qa, Qb = grid.regrid(Pa, 96, 0.384), grid.regrid(Pb, 96, 0.384)
    Qb["depth"] = Qa["depth"]; Qb["k"] = Qa["k"]            # one batch shares the site
    Qc = dict(Qa); Qc["C0"] = Qa["C0"] * 1.3
    batch = solver.DesignBatch([Qa, Qb, Qc])
    cs = sea_states(11, 5)
    host = solver.solve_dynamics(batch, solver.CaseTable(cs), n_iter=10)
    for d, Q in enumerate((Qa, Qb, Qc)):
        Xi_o, st_o, _ = oracle.solve_cases(oracle.OracleDesign(Q), cs, nIter=10)
        assert np.array_equal(host["status"][d, :, 0], st_o[:, 0])
        assert response_err(host["Xi"][d], Xi_o) < RTOL
    sess = solver.DeviceSession(batch, solver.CaseTable(cs))
    dev = sess.solve(n_iter=10)
    torch.cuda.synchronize()
    assert np.array_equal(dev["Xi"].cpu().numpy(), host["Xi"])
    assert np.array_equal(dev["status"].cpu().numpy(), host["status"])
    # a session with half the workspace: the fused solver has no design chunks (at 96 bins the smaller workspace only decides
    # whether F0 may live there) and must give the same answer; the v1 solver's design-chunk loop is pinned in
    # tests/test_dispatch_paths.py::test_v1_forced_design_batch_and_chunk_loop
    small = solver.DeviceSession(batch, solver.CaseTable(cs), workspace_bytes=sess.workspace_bytes // 2)
    dev2 = small.solve(n_iter=10)
    torch.cuda.synchronize()
    assert np.array_equal(dev2["Xi"].cpu().numpy(), host["Xi"])


def test_edge_cases(solver, oracle):
    """Still water, unit/constant spectra, non-converging loop (n_iter=0,1), XiStart != 0, explicit zeta."""
    _, P = load_golden("cfg1_OC3spar")
    b = solver.DesignBatch(P)
    od = oracle.OracleDesign(P)
    cs = dict(Hs=np.array([3.0, 3.0, 3.0, 3.0]), Tp=np.array([9.0] * 4), gamma=np.array([0.0, 3.3, 0.0, 0.0]),
              beta_deg=np.array([15.0, 15.0, 15.0, 15.0]), spec=np.array([3, 0, 1, 2], dtype=np.int32))
    for n_iter, xi0 in ((0, 0.0), (1, 0.0), (10, 0.1)):
        out = solver.solve_dynamics(b, solver.CaseTable(cs), n_iter=n_iter, xi_start=xi0)
        Xi_o, st_o, _ = oracle.solve_cases(od, cs, nIter=n_iter, XiStart=xi0)
        assert np.array_equal(out["status"][0, :, :2], st_o[:, :2])
        assert response_err(out["Xi"][0, 1:], Xi_o[1:]) < RTOL
        assert np.abs(out["Xi"][0, 0] - Xi_o[0]).max() <= 1e-10 * max(1e-300, np.abs(Xi_o[0]).max()) or np.abs(Xi_o[0]).max() == 0
    zeta = np.abs(np.sin(np.arange(b.nw) * 0.1))[None, :] * 0.3
    out = solver.solve_dynamics(b, solver.CaseTable({k: v[:1] for k, v in cs.items()}, zeta=zeta), n_iter=10, want=("Xi", "status", "zeta"))
    assert np.array_equal(out["zeta"], zeta)
    assert out["status"][0, 0, 1] == 1 and np.isfinite(out["Xi"]).all()
    with pytest.raises(ValueError):
        solver.CaseTable(dict(cs, spec=np.array([0, 1, 2, 7], dtype=np.int32)))


def test_system_solve_vs_oracle(solver, oracle):
    """Farm 6N x 6N system response (raft_model.py:1164-1216) vs the oracle's inverse-based response."""
    rng = np.random.default_rng(5)
    for n, nw, nrhs in ((12, 64, 1), (48, 33, 3), (96, 16, 2)):
        A = rng.normal(size=(nw, n, n)) + 1j * rng.normal(size=(nw, n, n)) + 4 * np.eye(n)[None]
        F = rng.normal(size=(nw, n, nrhs)) + 1j * rng.normal(size=(nw, n, nrhs))
        X, info = solver.system_solve(A, F)
        assert np.all(info == 0)
        for r in range(nrhs):
            Xo = oracle.system_response(A, F[:, :, r])
            assert relerr(X[:, :, r], Xo) < 1e-11


# ---- reference-facing API mirror (raft_b200.Model / FOWT) ------------------------------------------------------
def _model_from_golden(name):
    import json, os
    from conftest import GOLDEN
    from raft_b200.model import Model
    G, P = load_golden(name)
    D = json.load(open(os.path.join(GOLDEN, "designs.json")))[name]
    design = dict(D, site=dict(D["site"], water_depth=float(P["depth"])))
    mats = dict(M_struc=P["M0"] - G["A_hydro_morison"], C_struc=P["C0"] - G["C_moor"], C_moor=G["C_moor"])
    return Model(design, matrices=mats), G, P


@pytest.mark.parametrize("name", ["cfg2_VolturnUS-S_nw64", "cfg1_OC3spar", "test_VolturnUS-S"])
def test_model_api_vs_reference_run(name, solver):
    """Design dict -> own builder -> packer -> C ABI -> kernels, against the unmodified reference's responses."""
    model, G, P = _model_from_golden(name)
    for i, (Hs, Tp, beta) in enumerate(G["ref_run_solve_cases"]):
        case = dict(wave_spectrum="JONSWAP", wave_height=Hs, wave_period=Tp, wave_heading=beta, wave_gamma=0.0)
        Xi = model.solveDynamics(case)
        assert Xi.shape == (2, 6, model.nw) and np.all(Xi[1] == 0)
        assert response_err(Xi[0], G["ref_run_solve_Xi"][i]) < RTOL
    # all cases of the fixture in one batched analyzeCases call
    cases = [dict(wave_spectrum="JONSWAP", wave_height=h, wave_period=t, wave_heading=b) for h, t, b in G["ref_run_solve_cases"]]
    res = model.analyzeCases(cases=cases)
    assert np.array_equal(res["status"][:, 0, 0], G["ref_run_solve_passes"])
    assert response_err(res["Xi"], G["ref_run_solve_Xi"]) < RTOL
    # fowt.Z left behind = impedance of the last pass (raft_model.py:1155): Z Xi = F_BEM + F_iner + F_drag
    f = model.fowtList[0]
    lhs = np.einsum("abw,bw->aw", f.Z, res["Xi"][-1])
    rhs = f.F_BEM[0] + f.F_hydro_iner[0] + f.F_hydro_drag
    assert relerr(lhs, rhs) < 1e-9


def test_fowt_api_vs_reference_run(solver):
    """FOWT.calcHydroExcitation / calcHydroLinearization / calcDragExcitation mirror on the reference's own recipe."""
    model, G, P = _model_from_golden("test_VolturnUS-S")
    f = model.fowtList[0]
    f.calcHydroExcitation(dict(wave_spectrum="unit", wave_heading=0, wave_period=10, wave_height=2))
    assert f.nWaves == 1 and relerr(f.zeta[0], G["ref_run_lin_zeta"]) < 1e-14
    assert relerr(f.F_hydro_iner[0], G["ref_run_lin_F_hydro_iner"]) < RTOL
    B = f.calcHydroLinearization(G["ref_run_lin_Xi"])
    assert relerr(B, G["ref_pickle_lin_B_hydro_drag"]) < RTOL
    assert relerr(f.calcDragExcitation(0), G["ref_pickle_lin_F_hydro_drag"]) < RTOL
    with pytest.raises(ValueError):
        f.calcHydroExcitation(dict(wave_spectrum="bogus", wave_heading=0, wave_period=10, wave_height=2))


def test_fowt_drag_excitation_of_secondary_train(solver, oracle):
    """FOWT.calcDragExcitation(ih > 0) (raft_fowt.py:1940-1957, raft_member.py:2128-2152): the drag load of wave train ih with
    the Bmat that calcHydroLinearization(Xi) left behind for train 0, against the oracle's Bmat applied to train ih's kinematics."""
    model, G, P = _model_from_golden("cfg2_VolturnUS-S_nw64")
    f = model.fowtList[0]
    trains = [(6.0, 12.0, 30.0), (2.5, 7.0, -100.0), (1.0, 16.0, 170.0)]
    f.calcHydroExcitation(dict(wave_spectrum=["JONSWAP"] * 3, wave_height=[t[0] for t in trains], wave_period=[t[1] for t in trains],
                               wave_heading=[t[2] for t in trains], wave_gamma=[0.0] * 3))
    rng = np.random.default_rng(4)
    Xi = (rng.normal(size=(6, model.nw)) + 1j * rng.normal(size=(6, model.nw))) * np.array([1, 1, 1, 0.02, 0.02, 0.02])[:, None]
    B = f.calcHydroLinearization(Xi)
    od = oracle.OracleDesign(P)
    u = [oracle.calc_hydro_excitation(od, 0, Hs, Tp, 0.0, beta)[3] for Hs, Tp, beta in trains]
    Bmat, B_o, F0_o = oracle.calc_hydro_linearization(od, u[0], Xi)
    assert relerr(B, B_o) < RTOL and relerr(f.calcDragExcitation(0), F0_o) < RTOL
    for ih in (1, 2):
        F = np.zeros([6, model.nw], dtype=complex)
        for j in range(od.Ns):
            fj = np.einsum("ab,bw->aw", Bmat[j], u[ih][j])                       # translateForce3to6DOF: [f ; r x f]
            F[:3] += fj
            F[3:] += np.cross(P["node_r"][j] - P["prp"], fj.T).T
        assert relerr(f.calcDragExcitation(ih), F) < RTOL, ih


def test_sweep_single_gpu_vs_oracle(solver, oracle):
    """Synthetic geometry variants (ragged node counts) in one batch: every design against the oracle."""
    import json, os
    import torch
    from conftest import GOLDEN
    from raft_b200 import sweep
    G, P = load_golden("cfg2_VolturnUS-S_nw64")
    D = json.load(open(os.path.join(GOLDEN, "designs.json")))["cfg2_VolturnUS-S_nw64"]
    mats = dict(M_struc=P["M0"] - G["A_hydro_morison"], C_struc=P["C0"] - G["C_moor"], C_moor=G["C_moor"])
    V = sweep.build_variants(D, mats, sweep.sample_factors(12, seed=40), nw=160, max_freq=0.4, depth=float(P["depth"]))
    assert len(set(len(v["node_ls"]) for v in V)) > 1
    cs = sea_states(4, 3)
    Xi, st = sweep.solve_sweep(V, cs, n_iter=10)
    torch.cuda.synchronize()
    Xi, st = Xi.cpu().numpy(), st.cpu().numpy()
    assert np.all(st[..., 2] == 0)
    for d, Q in enumerate(V):
        Xi_o, st_o, _ = oracle.solve_cases(oracle.OracleDesign(Q), cs, nIter=10)
        assert np.array_equal(st[d, :, 0], st_o[:, 0]), d
        assert response_err(Xi[d], Xi_o) < RTOL, d


def test_farm_coupled_response_vs_oracle(solver, oracle):
    """Two-unit farm (raft_model.py:1164-1216): independent linearisation per FOWT, then the coupled 12x12 system
    with an injected array-mooring stiffness, against the oracle's Z / inverse-based system response."""
    import json, os
    from conftest import GOLDEN
    from raft_b200.model import Model
    G, P = load_golden("cfg2_VolturnUS-S_nw64")
    D = json.load(open(os.path.join(GOLDEN, "designs.json")))["cfg2_VolturnUS-S_nw64"]
    mats = dict(M_struc=P["M0"] - G["A_hydro_morison"], C_struc=P["C0"] - G["C_moor"], C_moor=G["C_moor"])
    design = dict(settings=D["settings"], site=dict(D["site"], water_depth=float(P["depth"])), platforms=[D["platform"]],
                  array=dict(keys=["ID", "turbineID", "platformID", "mooringID", "x_location", "y_location", "heading_adjust"],
                             data=[[1, 0, 1, 0, 0.0, 0.0, 0.0], [2, 0, 1, 0, 1600.0, 0.0, 0.0]]))
    rng = np.random.default_rng(1)
    A = rng.normal(size=(12, 12)) * 2e4
    C_arr = A @ A.T / 12 + np.diag([5e4] * 12)
    model = Model(design, matrices=mats, array_stiffness=C_arr)
    assert model.nDOF == 12
    case = dict(wave_spectrum="JONSWAP", wave_height=6.0, wave_period=12.0, wave_heading=20.0)
    Xi = model.solveDynamics(case)[0]                       # [12, nw]
    # oracle: per-FOWT loop (Z_i, F_i = Z_i Xi_i), then inv(Z_sys) F
    nw = model.nw
    Z = np.zeros([nw, 12, 12], dtype=complex)
    F = np.zeros([nw, 12], dtype=complex)
    for i, f in enumerate(model.fowtList):
        Xi_i, st, Z_i, _ = oracle.solve_dynamics(oracle.OracleDesign(f.pack()), 0, 6.0, 12.0, 0.0, 20.0, nIter=model.nIter,
                                                 XiStart=model.XiStart, want_Z=True)
        Z[:, 6 * i:6 * i + 6, 6 * i:6 * i + 6] = Z_i
        F[:, 6 * i:6 * i + 6] = np.einsum("wab,bw->wa", Z_i, Xi_i)
    Xo = oracle.system_response(Z + C_arr[None], F).T
    assert response_err(np.stack([Xi[:6], Xi[6:]]), np.stack([Xo[:6], Xo[6:]])) < 1e-9
    # the second unit sees the wave later: phase differs, amplitude spectrum of the uncoupled problem would not
    assert not np.allclose(Xi[:6], Xi[6:])


def test_cfg3_bem_tables_from_wamit_vs_oracle(solver, oracle):
    """configs[2] pipeline off the build box: raw WAMIT tables -> readHydro on a 512-bin grid -> fused solver, vs oracle."""
    import json, os
    from conftest import GOLDEN
    from raft_b200 import bem, grid
    from raft_b200.fowt import FOWT
    G, P = load_golden("cfg3_OC4semi-WAMIT_nw128")
    D = json.load(open(os.path.join(GOLDEN, "designs.json")))["cfg3_OC4semi-WAMIT_nw128"]
    t = np.load(os.path.join(GOLDEN, "wamit_marin_semi.npz"))
    w = grid.make_w(0.256 / 512, 0.256)
    H = bem.read_hydro(t["A"], t["B"], t["w1"], t["Re"], t["Im"], t["w3"], t["heads"], w, rho=float(P["rho"]), g=float(P["g"]))
    mats = dict(M_struc=P["M0"] - G["A_hydro_morison"], C_struc=P["C0"] - G["C_moor"], C_moor=G["C_moor"], **H)
    f = FOWT(D, w, depth=float(P["depth"]), matrices=mats)
    f.calcHydroConstants()
    Q = f.pack()
    assert Q["X_BEM"].shape == (37, 6, 512) and Q["A_w"].shape == (6, 6, 512)
    cs = sea_states(3, 6)
    out = solver.solve_dynamics(solver.DesignBatch(Q), solver.CaseTable(cs), n_iter=10)
    Xi_o, st_o, _ = oracle.solve_cases(oracle.OracleDesign(Q), cs, nIter=10)
    assert np.array_equal(out["status"][0, :, 0], st_o[:, 0])
    assert response_err(out["Xi"][0], Xi_o) < RTOL


def test_response_stats_vs_reference_formulas(solver):
    """std / PSD reductions of saveTurbineOutputs (helpers.getRMS :684, getPSD :694, rad2deg on rotations)."""
    rng = np.random.default_rng(9)
    Xi = (rng.normal(size=(3, 5, 6, 333)) + 1j * rng.normal(size=(3, 5, 6, 333))) * rng.uniform(0.01, 2, size=(3, 5, 6, 1))
    dw = 0.0123
    sd, psd = solver.response_stats(Xi, dw)
    Xd = Xi.copy(); Xd[..., 3:, :] = Xd[..., 3:, :] * (180.0 / np.pi)      # helpers.rad2deg (works on complex amplitudes)
    assert relerr(sd, np.sqrt(0.5 * np.sum(np.abs(Xd) ** 2, axis=-1))) < 1e-14
    assert relerr(psd, 0.5 * np.abs(Xd) ** 2 / dw) < 1e-14
    model, G, P = _model_from_golden("cfg1_OC3spar")
    res = model.analyzeCases(cases=[dict(wave_spectrum="JONSWAP", wave_height=2.0, wave_period=8.0, wave_heading=0.0)])
    m = res["case_metrics"][0][0]
    ref = G["ref_run_solve_Xi"][0]
    assert abs(m["surge_std"] - np.sqrt(0.5 * np.sum(np.abs(ref[0]) ** 2))) < 1e-10 * m["surge_std"]
    assert relerr(m["pitch_PSD"], 0.5 * np.abs(ref[4] * 180.0 / np.pi) ** 2 / (P["w"][1] - P["w"][0])) < 1e-9
    # a case with several wave trains: getRMS / getPSD sum the squares over the trains (helpers.py:678-700)
    tr = G["ref_run_trains"]
    case = dict(wave_spectrum=["JONSWAP"] * len(tr), wave_height=list(tr[:, 0]), wave_period=list(tr[:, 1]),
                wave_heading=list(tr[:, 2]), wave_gamma=[0.0] * len(tr))
    m = model.analyzeCases(0, None, False, cases=[case])["case_metrics"][0][0]
    ref = np.concatenate([G["ref_run_trains_Xi"], np.zeros_like(G["ref_run_trains_Xi"][:1])])      # [nWaves+1, 6, nw]
    dw = P["w"][1] - P["w"][0]
    assert abs(m["heave_std"] - np.sqrt(0.5 * np.sum(np.abs(ref[:, 2]) ** 2))) < 1e-10 * m["heave_std"]
    assert relerr(m["roll_PSD"], np.sum(0.5 * np.abs(ref[:, 3] * 57.29577951308232) ** 2 / dw, axis=0)) < 1e-9
    assert m["surge_RA"].shape == (len(tr) + 1, model.nw) and relerr(m["surge_RA"], ref[:, 0]) < 1e-9
    assert m["surge_max"] == 3 * m["surge_std"]


def test_error_paths_nan_and_singular(solver):
    """NaN in the response stops the unit and sets RAFTK_FLAG_NAN (the reference raises at raft_model.py:1098);
    a singular impedance sets RAFTK_FLAG_SINGULAR; the Model mirror turns the NaN flag into the reference's exception."""
    _, P = load_golden("cfg1_OC3spar")
    cs = solver.CaseTable(dict(Hs=[3.0], Tp=[9.0], gamma=[0.0], beta_deg=[10.0], spec=np.array([0], dtype=np.int32)))
    Q = dict(P); Q["M0"] = P["M0"].copy(); Q["M0"][2, 2] = np.nan
    out = solver.solve_dynamics(solver.DesignBatch(Q), cs, n_iter=10)
    assert out["status"][0, 0, 2] & 1 and out["status"][0, 0, 0] == 1 and out["status"][0, 0, 1] == 0
    Z = dict(P); Z["M0"] = np.zeros((6, 6)); Z["B0"] = np.zeros((6, 6)); Z["C0"] = np.zeros((6, 6))
    for k in ("node_cd_q", "node_cd_p1", "node_cd_p2"):
        Z[k] = np.zeros_like(P[k])
    out = solver.solve_dynamics(solver.DesignBatch(Z), cs, n_iter=2)
    assert out["status"][0, 0, 2] & 2
    model, G, _ = _model_from_golden("cfg1_OC3spar")
    model.fowtList[0].M_struc[0, 0] = np.nan
    with pytest.raises(Exception, match="Nan detected in response vector Xi."):
        model.solveDynamics(dict(wave_spectrum="JONSWAP", wave_height=2.0, wave_period=8.0, wave_heading=0.0))


def test_pipelined_solve_chunks_match_single_launch(solver):
    """PipelinedSolve (the N>1 step: chunked launches whose all-gathers overlap the next chunk) gives, chunk by
    chunk, the same bits as one launch over the whole batch -- split by cases and by designs."""
    import torch
    from raft_b200 import grid, sweep
    _, P = load_golden("cfg2_VolturnUS-S_nw64")
    Q = grid.regrid(P, 128, 0.512)
    cs = sea_states(2, 10)
    full = solver.solve_dynamics(solver.DesignBatch(Q), solver.CaseTable(cs), n_iter=10)
    pipe = sweep.PipelinedSolve(Q, cs, n_chunks=3, split="cases")
    pipe.step(n_iter=10)
    torch.cuda.synchronize()
    Xi = np.concatenate([s.out["Xi"].cpu().numpy() for s in pipe.sessions], axis=1)
    assert np.array_equal(Xi, full["Xi"]) and np.array_equal(pipe.status(), full["status"].reshape(-1, 4))
    assert pipe.units == 10 * 128
    Q2 = dict(Q); Q2["C0"] = Q["C0"] * 1.2
    both = solver.solve_dynamics(solver.DesignBatch([Q, Q2, Q]), solver.CaseTable(cs), n_iter=10)
    pipe = sweep.PipelinedSolve([Q, Q2, Q], cs, n_chunks=2, split="designs")
    pipe.step(n_iter=10)
    torch.cuda.synchronize()
    Xi = np.concatenate([s.out["Xi"].cpu().numpy() for s in pipe.sessions], axis=0)
    assert np.array_equal(Xi, both["Xi"])


@pytest.mark.parametrize("name", ["cfg1_OC3spar", "cfg2_VolturnUS-S_nw64"])
def test_wave_trains_vs_reference_run(name, solver, oracle):
    """A case with several wave trains (lists in the case dict): train 0 drives the linearisation, every train's
    response uses that impedance and drag coefficients (raft_model.py:1200-1236) -- against the unmodified reference."""
    model, G, P = _model_from_golden(name)
    tr = G["ref_run_trains"]
    case = dict(wave_spectrum=["JONSWAP"] * len(tr), wave_height=list(tr[:, 0]), wave_period=list(tr[:, 1]),
                wave_heading=list(tr[:, 2]), wave_gamma=[0.0] * len(tr))
    Xi = model.solveDynamics(case)
    assert Xi.shape == (len(tr) + 1, 6, model.nw) and np.all(Xi[-1] == 0)
    for ih in range(len(tr)):
        assert response_err(Xi[ih], G["ref_run_trains_Xi"][ih]) < RTOL, ih
    # low level: mixed table (two independent cases + the trains), secondary status rows point at their primary
    from raft_b200 import packer
    cases = [dict(wave_spectrum="JONSWAP", wave_height=2.0, wave_period=9.0, wave_heading=10.0), case,
             dict(wave_spectrum="JONSWAP", wave_height=4.0, wave_period=11.0, wave_heading=-60.0)]
    table, owner, first = packer.pack_case_trains(cases)
    out = solver.solve_dynamics(solver.DesignBatch(P), solver.CaseTable(table), n_iter=int(G["n_iter"]), xi_start=float(G["xi_start"]))
    assert list(first) == [0, 1, 1 + len(tr)] and list(table["primary"]) == [0] + [1] * len(tr) + [1 + len(tr)]
    assert np.array_equal(out["status"][0, 2:1 + len(tr), 3], np.full(len(tr) - 1, 2))
    Xo, _ = oracle.solve_dynamics_trains(oracle.OracleDesign(P), table["spec"][1:1 + len(tr)], tr[:, 0], tr[:, 1], np.zeros(len(tr)), tr[:, 2],
                                         nIter=int(G["n_iter"]), XiStart=float(G["xi_start"]))
    assert response_err(out["Xi"][0, 1:1 + len(tr)], Xo) < RTOL
    solo = solver.solve_dynamics(solver.DesignBatch(P), solver.CaseTable(packer.pack_cases([cases[0], cases[2]])), n_iter=int(G["n_iter"]),
                                 xi_start=float(G["xi_start"]))
    assert np.array_equal(solo["Xi"][0, 0], out["Xi"][0, 0]) and np.array_equal(solo["Xi"][0, 1], out["Xi"][0, -1])


def _random_design(rng, n_members):
    """Synthetic platform with inclined / tapered / rectangular / potMod members (exercises both step-class kinds on
    one member, ragged sections, surface-piercing strips)."""
    members = []
    for i in range(n_members):
        kind = rng.integers(0, 4)
        zA = -rng.uniform(8, 40)
        if kind == 0:      # vertical column, possibly surface piercing, tapered
            x, y = rng.uniform(-40, 40, 2)
            rA, rB = [x, y, zA], [x, y, zA + rng.uniform(5, 60)]
        elif kind == 1:    # horizontal pontoon
            rA = [rng.uniform(-40, 40), rng.uniform(-40, 40), zA]
            rB = [rA[0] + rng.uniform(5, 40), rA[1] + rng.uniform(-30, 30), zA]
        else:              # inclined brace
            rA = [rng.uniform(-40, 40), rng.uniform(-40, 40), zA]
            rB = [rA[0] + rng.uniform(-30, 30), rA[1] + rng.uniform(-30, 30), zA + rng.uniform(3, 45)]
        rect = rng.random() < 0.4
        nst = int(rng.integers(2, 5))
        st = np.sort(rng.uniform(0, 1, nst)); st[0], st[-1] = 0.0, 1.0
        if rect:
            d = [[float(rng.uniform(2, 9)), float(rng.uniform(2, 9))] for _ in range(nst)]
        else:
            d = [float(rng.uniform(2, 12)) for _ in range(nst)]
        members.append(dict(name="m%d" % i, type="rigid", rA=[float(v) for v in rA], rB=[float(v) for v in rB],
                            shape="rect" if rect else "circ", stations=[float(v) for v in st], d=d,
                            gamma=float(rng.uniform(0, 90)) if rect else 0.0, potMod=bool(rng.random() < 0.25),
                            Cd=float(rng.uniform(0.4, 1.2)), Ca=float(rng.uniform(0.5, 1.1)), CdEnd=0.6, CaEnd=0.6,
                            Cd_q=float(rng.uniform(0.0, 0.1)), dlsMax=float(rng.uniform(1.5, 6.0))))
    return dict(site=dict(water_depth=float(rng.uniform(60, 400)), rho_water=1025.0, g=9.81),
                platform=dict(potModMaster=0, dlsMax=5.0, members=members))


@pytest.mark.parametrize("seed", [1, 2, 3, 4])
def test_random_designs_vs_oracle(seed, solver, oracle):
    """Randomised geometry / grid / sea states / cluster size against the oracle (generic code paths that the
    BASELINE designs do not reach: inclined members, mixed step classes, tapered rectangular sections)."""
    from raft_b200 import grid
    from raft_b200.fowt import FOWT
    rng = np.random.default_rng(seed)
    design = _random_design(rng, int(rng.integers(2, 9)))
    nw = int(rng.integers(40, 300))
    w = grid.make_w(0.3 / nw, 0.3)
    m = rng.uniform(0.5, 3.0) * 1e7
    mats = dict(M_struc=np.diag([m, m, m, m * 900, m * 900, m * 1500]) + rng.normal(size=(6, 6)) * m * 0.01,
                C_struc=np.diag([0, 0, 0, -m * 5, -m * 5, 0.0]),
                C_hydro=np.diag([0, 0, rng.uniform(2, 6) * 1e6, rng.uniform(1, 4) * 1e9, rng.uniform(1, 4) * 1e9, 0.0]),
                C_moor=np.diag([7e4, 7e4, 0, 0, 0, 1.2e8]), B_struc=np.diag(rng.uniform(0, 1e5, 6)))
    f = FOWT(design, w, depth=design["site"]["water_depth"], matrices=mats)
    f.calcHydroConstants()
    Q = f.pack()
    assert len(Q["node_ls"]) > 0
    cs = sea_states(seed + 100, int(rng.integers(2, 7)))
    cs["spec"][-1] = 1                                            # one unit-spectrum case
    cluster = int(rng.choice([0, 1, 2, 4]))
    out = solver.solve_dynamics(solver.DesignBatch(Q), solver.CaseTable(cs), n_iter=12, cluster_size=cluster)
    Xi_o, st_o, _ = oracle.solve_cases(oracle.OracleDesign(Q), cs, nIter=12)
    assert np.array_equal(out["status"][0, :, :2], st_o[:, :2]), (out["status"][0], st_o)
    assert np.all(out["status"][0, :, 2] == 0)
    assert response_err(out["Xi"][0], Xi_o) < RTOL


# ---- second-order (difference-frequency) forces from an external QTF table: potSecOrder 2 -------------------------

def test_second_order_force_vs_reference_run(solver, oracle):
    """FOWT.calcHydroForce_2ndOrd for all cases in one launch + Model.solveDynamics with the force added
    (raft_model.py:1035-1048), vs the unmodified reference run with the shipped marin_semi.12d."""
    from conftest import QTF_GOLDEN
    G, P = load_golden(QTF_GOLDEN)
    cs = G["ref_run_solve_cases"]
    n = len(cs)
    table = dict(Hs=cs[:, 0], Tp=cs[:, 1], gamma=np.zeros(n), beta_deg=cs[:, 2], spec=np.zeros(n, dtype=np.int32))
    b = solver.DesignBatch(P)
    assert b.n_qtf_w == 56 and b.n_qtf_head == 1 and b.qtf_shared == 1
    f2 = solver.second_order_force(b, solver.CaseTable(table))
    assert relerr(f2["F_2nd"][0], G["ref_run_F2nd"]) < RTOL
    assert relerr(f2["F_2nd_mean"][0], G["ref_run_F2nd_mean"]) < RTOL
    assert np.all(f2["F_2nd"][0][:, :, -1] == 0.0)
    # explicit amplitudes instead of a spectrum id: S = zeta^2 / (2 dw)
    zeta = np.sqrt(2 * G["ref_run_S"] * float(P["dw"]))
    f2z = solver.second_order_force(b, solver.CaseTable(table, zeta=zeta))
    assert relerr(f2z["F_2nd"][0], G["ref_run_F2nd"]) < RTOL
    for cluster in (0, 1, 2):
        out = solver.solve_dynamics(b, solver.CaseTable(table), n_iter=int(G["n_iter"]), xi_start=float(G["xi_start"]),
                                    cluster_size=cluster, want=("Xi", "status", "F_2nd", "F_2nd_mean"))
        assert np.array_equal(out["status"][0, :, 0], G["ref_run_solve_passes"])
        assert response_err(out["Xi"][0], G["ref_run_solve_Xi"]) < RTOL
        assert relerr(out["F_2nd"][0], G["ref_run_F2nd"]) < RTOL
    # device-resident route: the solve computes the force into out['F_2nd'] on the same stream
    import torch
    ses = solver.DeviceSession(b, solver.CaseTable(table))
    o = ses.solve(n_iter=int(G["n_iter"]), xi_start=float(G["xi_start"]), cluster_size=2)
    torch.cuda.synchronize()
    # (the tile kernel combines partial sums with atomic adds: equal to rounding, not bit for bit)
    assert response_err(o["Xi"].cpu().numpy()[0], out["Xi"][0]) < 1e-13 and relerr(o["F_2nd"].cpu().numpy(), out["F_2nd"]) < 1e-13
    assert relerr(ses.second_order_force()["F_2nd_mean"].cpu().numpy(), out["F_2nd_mean"]) < 1e-13
    # precomputed force handed in through cases.F_2nd == computed inside the solve; without it the response differs
    P0 = {k: v for k, v in P.items() if not k.startswith("qtf")}
    pre = solver.solve_dynamics(solver.DesignBatch(P0), solver.CaseTable(table, F_2nd=f2["F_2nd"]), n_iter=int(G["n_iter"]),
                                xi_start=float(G["xi_start"]))
    assert response_err(pre["Xi"][0], out["Xi"][0]) < 1e-13
    none = solver.solve_dynamics(solver.DesignBatch(P0), solver.CaseTable(table), n_iter=int(G["n_iter"]), xi_start=float(G["xi_start"]))
    assert response_err(none["Xi"][0], G["ref_run_solve_Xi"]) > 1e-4


def test_second_order_heading_interpolation_and_design_axis(solver, oracle):
    """4-heading synthetic table (interp1d incl. the clamped ends) vs the reference run; two designs with DIFFERENT
    tables in one batch vs the oracle; a larger grid (odd nw) vs the oracle."""
    from conftest import QTF_GOLDEN
    G, P = load_golden(QTF_GOLDEN)
    Pm = dict(P)
    Pm["qtf"] = np.stack([P["qtf"][:, :, 0, :] * s for s in G["mh_scale"]], axis=2)
    Pm["qtf_heads"] = G["mh_heads"]
    betas = G["mh_betas_deg"]
    n = len(betas)
    zeta = np.repeat(np.sqrt(2 * G["ref_run_S"][:1] * float(P["dw"])), n, axis=0)
    table = dict(Hs=np.ones(n), Tp=np.ones(n), gamma=np.zeros(n), beta_deg=betas, spec=np.zeros(n, dtype=np.int32))
    f2 = solver.second_order_force(solver.DesignBatch(Pm), solver.CaseTable(table, zeta=zeta))
    assert relerr(f2["F_2nd"][0], G["ref_run_mh_F2nd"]) < RTOL
    assert relerr(f2["F_2nd_mean"][0], G["ref_run_mh_F2nd_mean"]) < RTOL
    # design axis: [single-heading, 4-heading padded to a common axis is not allowed] -> two 4-heading designs
    Pn = dict(Pm)
    Pn["qtf"] = Pm["qtf"][:, :, ::-1, :] * (0.5 - 0.25j)
    b2 = solver.DesignBatch([Pm, Pn])
    assert b2.qtf_shared == 0
    cs = sea_states(11, 5)
    out = solver.solve_dynamics(b2, solver.CaseTable(cs), n_iter=10, want=("Xi", "status", "F_2nd", "F_2nd_mean"))
    for d, Pd in enumerate((Pm, Pn)):
        od = oracle.OracleDesign(Pd)
        Xi_o, st_o, _ = oracle.solve_cases(od, cs, nIter=10)
        assert np.array_equal(out["status"][d, :, 0], st_o[:, 0])
        assert response_err(out["Xi"][d], Xi_o) < RTOL
        for c in range(5):
            S = oracle.jonswap(Pd["w"], cs["Hs"][c], cs["Tp"][c], 0.0)
            fm, f = oracle.hydro_force_2nd(od, cs["beta_deg"][c] * 0.017453292519943295, S)
            assert relerr(out["F_2nd"][d, c], f) < RTOL and relerr(out["F_2nd_mean"][d, c], fm) < RTOL
    # shared table broadcast over a design axis (same dict object twice)
    b3 = solver.DesignBatch([Pm, Pm])
    assert b3.qtf_shared == 1
    f3 = solver.second_order_force(b3, solver.CaseTable(cs))
    assert np.array_equal(f3["F_2nd"][0], f3["F_2nd"][1]) and relerr(f3["F_2nd"][0], out["F_2nd"][0]) < 1e-13


def test_second_order_model_api_from_files(solver, tmp_path):
    """configs[2] from its shipped files, potFirstOrder 1 + potSecOrder 2: .1/.3 -> readHydro, .12d -> FOWT.readQTF,
    Model.solveDynamics / analyzeCases incl. a multi-train case, vs the unmodified reference run."""
    import json, os
    from conftest import GOLDEN, QTF_GOLDEN
    from raft_b200 import bem, grid
    from raft_b200.model import Model
    G, P = load_golden(QTF_GOLDEN)
    D = json.load(open(os.path.join(GOLDEN, "designs.json")))["cfg3_OC4semi-WAMIT_nw128"]
    t = np.load(os.path.join(GOLDEN, "wamit_marin_semi.npz"))
    np.savetxt(str(tmp_path / "semi.12d"), t["qtf_rows"], fmt="%.5e")
    nw = len(P["w"])
    w = grid.make_w(0.256 / nw, 0.256)
    assert np.array_equal(w, P["w"])
    H = bem.read_hydro(t["A"], t["B"], t["w1"], t["Re"], t["Im"], t["w3"], t["heads"], w, rho=float(P["rho"]), g=float(P["g"]))
    plat = dict(D["platform"], potSecOrder=2, hydroPath=str(tmp_path / "semi"))
    design = dict(D, platform=plat, site=dict(D["site"], water_depth=float(P["depth"])),
                  settings=dict(D["settings"], min_freq=0.256 / nw, max_freq=0.256))
    mats = dict(M_struc=P["M0"] - G["A_hydro_morison"], C_struc=P["C0"] - G["C_moor"], C_moor=G["C_moor"], **H)
    model = Model(design, matrices=mats)
    f = model.fowtList[0]
    assert f.potSecOrder == 2 and np.array_equal(f.qtf, P["qtf"])
    cases = [dict(wave_spectrum="JONSWAP", wave_height=h, wave_period=tp, wave_heading=b) for h, tp, b in G["ref_run_solve_cases"]]
    res = model.analyzeCases(cases=cases)
    assert np.array_equal(res["status"][:, 0, 0], G["ref_run_solve_passes"])
    assert response_err(res["Xi"], G["ref_run_solve_Xi"]) < RTOL
    assert relerr(f.Fhydro_2nd[0].real, G["ref_run_F2nd"][-1]) < RTOL and relerr(f.Fhydro_2nd_mean[0], G["ref_run_F2nd_mean"][-1]) < RTOL
    tr = G["ref_run_trains"]
    case = dict(wave_spectrum=["JONSWAP"] * len(tr), wave_height=list(tr[:, 0]), wave_period=list(tr[:, 1]),
                wave_heading=list(tr[:, 2]), wave_gamma=[0.0] * len(tr))
    Xi = model.solveDynamics(case)
    for ih in range(len(tr)):
        assert response_err(Xi[ih], G["ref_run_trains_Xi"][ih]) < RTOL, ih
    assert relerr(f.Fhydro_2nd.real, G["ref_run_trains_F2nd"]) < RTOL
    # FOWT.calcHydroForce_2ndOrd mirror
    fm, f2 = f.calcHydroForce_2ndOrd(G["ref_run_solve_cases"][0, 2] * 0.017453292519943295, G["ref_run_S"][0])
    assert relerr(f2, G["ref_run_F2nd"][0]) < RTOL and relerr(fm, G["ref_run_F2nd_mean"][0]) < RTOL


def test_second_order_force_full_grid_properties(solver, oracle):
    """BASELINE config-3 size (nw = 2048): spot-check a case against the oracle and check size-independent
    properties -- scaling S by a makes f scale by a (f ~ sqrt(S S)), f_mean by a; zero outside the table's band."""
    from conftest import QTF_GOLDEN
    G, P = load_golden(QTF_GOLDEN)
    nw = 2048
    w = np.arange(1, nw + 1) * (2 * np.pi * 0.256 / nw)
    Pb = dict(P, w=w, k=w ** 2 / 9.81, dw=w[1] - w[0])
    for key in ("A_w", "B_w", "X_BEM", "bem_headings"):
        Pb.pop(key, None)
    b = solver.DesignBatch(Pb)
    cs = sea_states(3, 6)
    f = solver.second_order_force(b, solver.CaseTable(cs))
    od = oracle.OracleDesign(Pb)
    S = oracle.jonswap(w, cs["Hs"][2], cs["Tp"][2], 0.0)
    fm_o, f_o = oracle.hydro_force_2nd(od, cs["beta_deg"][2] * 0.017453292519943295, S)
    assert relerr(f["F_2nd"][0, 2], f_o) < RTOL and relerr(f["F_2nd_mean"][0, 2], fm_o) < RTOL
    zeta = np.sqrt(2 * S * (w[1] - w[0]))
    one = dict(Hs=[1.0, 1.0], Tp=[1.0, 1.0], gamma=[0.0, 0.0], beta_deg=[0.0, 0.0], spec=np.zeros(2, dtype=np.int32))
    fz = solver.second_order_force(b, solver.CaseTable(one, zeta=np.stack([zeta, 2.0 * zeta])))
    assert relerr(fz["F_2nd"][0, 1], 4.0 * fz["F_2nd"][0, 0]) < 1e-13
    assert relerr(fz["F_2nd_mean"][0, 1], 4.0 * fz["F_2nd_mean"][0, 0]) < 1e-13
    # difference frequencies beyond the table's span (w_max - w_min of the QTF axis) carry no force
    span = P["qtf_w"][-1] - P["qtf_w"][0]
    mu = np.arange(1, nw + 1) * (w[1] - w[0])              # bin m holds difference frequency (m+1) dw
    assert np.all(fz["F_2nd"][0, 0][:, mu > span * (1 + 1e-12)] == 0.0)


# ---- turbine output channels (nacelle accelerations, tower-base moment): raft_fowt.py:2401-2444, 2504-2538 --------

def test_channel_stats_vs_reference_saveTurbineOutputs(solver):
    """Design WITH its turbine (mass matrices incl. tower + RNA packed from the live reference): GPU solve of every
    train, then k_channel_stats, against the metrics the unmodified reference's saveTurbineOutputs produced."""
    import os
    from conftest import GOLDEN
    z = np.load(os.path.join(GOLDEN, "turb_VolturnUS-S.npz"))
    P = {k[2:]: z[k] for k in z.files if k.startswith("P_")}
    names = [n.split(":")[0] for n in z["ch_names"]]
    b = solver.DesignBatch(P)
    dw = float(P["dw"])
    from raft_b200 import packer
    for ic in range(3):
        tr = z["ref_run_case%d_trains" % ic]
        case = dict(wave_spectrum=["JONSWAP"] * len(tr), wave_height=list(tr[:, 0]), wave_period=list(tr[:, 1]),
                    wave_heading=list(tr[:, 2]), wave_gamma=[0.0] * len(tr))
        table, owner, first = packer.pack_case_trains([case])
        out = solver.solve_dynamics(b, solver.CaseTable(table), n_iter=int(z["n_iter"]), xi_start=float(z["xi_start"]))
        ref = z["ref_run_case%d_Xi" % ic]
        assert response_err(out["Xi"][0], ref[:-1]) < RTOL
        sd, psd, amp = solver.channel_stats(z["ch_coef"], out["Xi"][0], dw, amp=True)     # [nT,nch], [nT,nch,nw]
        sd_c, psd_c = np.sqrt((sd ** 2).sum(axis=0)), psd.sum(axis=0)
        for k, nm in enumerate(names):
            r = z["ref_run_case%d_%s_std" % (ic, nm)][0]
            assert abs(sd_c[k] - r) < 1e-9 * r, (ic, nm)
            assert relerr(psd_c[k], z["ref_run_case%d_%s_PSD" % (ic, nm)][:, 0]) < 1e-9, (ic, nm)
        assert relerr(amp, np.einsum("kaw,taw->tkw", z["ch_coef"], out["Xi"][0])) < 1e-14
    # design axis: two designs with different coefficient sets in one call
    rng = np.random.default_rng(4)
    coef = rng.normal(size=(2, 3, 6, 77)) + 1j * rng.normal(size=(2, 3, 6, 77))
    Xi = rng.normal(size=(2, 5, 6, 77)) + 1j * rng.normal(size=(2, 5, 6, 77))
    sd, psd, amp = solver.channel_stats(coef, Xi, 0.05, amp=True)
    Y = np.einsum("dkaw,dcaw->dckw", coef, Xi)
    assert relerr(amp, Y) < 1e-14 and relerr(sd, np.sqrt(0.5 * np.sum(np.abs(Y) ** 2, axis=-1))) < 1e-14
    assert relerr(psd, 0.5 * np.abs(Y) ** 2 / 0.05) < 1e-14


def test_model_api_turbine_channels(solver):
    """Model(..., channels=...) fills AxRNA/AyRNA/AzRNA/Mbase metrics like saveTurbineOutputs; platform built by the
    own builder, turbine mass/inertia injected through M_struc (statics are out of scope)."""
    import json, os
    from conftest import GOLDEN
    from raft_b200.model import Model
    z = np.load(os.path.join(GOLDEN, "turb_VolturnUS-S.npz"))
    P = {k[2:]: z[k] for k in z.files if k.startswith("P_")}
    G0, _ = load_golden("test_VolturnUS-S")
    D = json.load(open(os.path.join(GOLDEN, "designs.json")))["test_VolturnUS-S"]
    design = dict(D, site=dict(D["site"], water_depth=float(P["depth"])))
    mats = dict(M_struc=P["M0"] - G0["A_hydro_morison"], C_struc=P["C0"] - G0["C_moor"], C_moor=G0["C_moor"], B_struc=P["B0"])
    ch = dict(names=[(n.split(":")[0], int(n.split(":")[1])) for n in z["ch_names"]], coef=z["ch_coef"], avg=z["ch_avg"])
    model = Model(design, matrices=mats, channels=ch)
    cases = []
    for ic in range(3):
        tr = z["ref_run_case%d_trains" % ic]
        cases.append(dict(wave_spectrum=["JONSWAP"] * len(tr), wave_height=list(tr[:, 0]), wave_period=list(tr[:, 1]),
                          wave_heading=list(tr[:, 2]), wave_gamma=[0.0] * len(tr)))
    res = model.analyzeCases(cases=cases)
    for ic in range(3):
        m = res["case_metrics"][ic][0]
        for nm in ("surge", "pitch", "yaw", "AxRNA", "AyRNA", "AzRNA", "Mbase"):
            for suffix in ("_std", "_avg", "_max", "_min"):
                ref = np.ravel(z["ref_run_case%d_%s%s" % (ic, nm, suffix)])[0]
                mine = np.ravel(m[nm + suffix])[0]
                if nm in ("surge", "pitch", "yaw") and suffix != "_std":
                    continue                                 # platform means come from the statics solve (out of scope)
                assert abs(mine - ref) <= 1e-8 * max(abs(ref), 1e-12), (ic, nm, suffix)
            refp = z["ref_run_case%d_%s_PSD" % (ic, nm)]
            assert relerr(np.ravel(m[nm + "_PSD"]), np.ravel(refp)) < 1e-8, (ic, nm)


# ---- slender-body QTF (potSecOrder 1): raft_fowt.py:1988-2078, raft_member.py:1488-1792 ---------------------------

def _slender_golden():
    import os
    from conftest import GOLDEN
    z = np.load(os.path.join(GOLDEN, "slender_VolturnUS-S.npz"))
    return z, {k[2:]: z[k] for k in z.files if k.startswith("P_")}


def test_slender_qtf_vs_reference_pickle_and_run(solver, oracle):
    """k_slender_tables / k_slender_pairs: fixed body vs the reference's own golden pickle; moving body vs the QTFs the
    reference computed inside solveDynamics; random motions and headings vs the oracle (all pairs in one call)."""
    z, P = _slender_golden()
    n2 = len(P["qs_w"])
    deg = 0.017453292519943295
    q = solver.qtf_slender(P, [z["ref_pickle_case"][2] * deg], np.zeros([1, 6, n2], dtype=complex))
    for a in range(6):
        assert relerr(q[0][..., a], z["ref_pickle_qtf"][:, :, 0, a]) < RTOL, a
    cases = z["ref_run_solve_cases"]
    Xi2 = np.array([[np.interp(P["qs_w"], P["w"], z["ref_run_solve_Xi0"][i][a], left=0, right=0) for a in range(6)] for i in range(len(cases))])
    q = solver.qtf_slender(P, cases[:, 2] * deg, Xi2)
    for i in range(len(cases)):
        for a in range(6):
            assert relerr(q[i][..., a], z["ref_run_solve_qtf"][i][..., a]) < RTOL, (i, a)
    rng = np.random.default_rng(5)
    Xr = (rng.normal(size=(4, 6, n2)) + 1j * rng.normal(size=(4, 6, n2))) * np.array([1, 1, 1, 0.03, 0.03, 0.03])[None, :, None]
    betas = rng.uniform(-np.pi, np.pi, 4)
    q = solver.qtf_slender(P, betas, Xr)
    od = oracle.OracleDesign(P)
    for c in range(4):
        qo = oracle.qtf_slender(od, betas[c], Xr[c])
        for a in range(6):
            assert relerr(q[c][..., a], qo[..., a]) < RTOL, (c, a)
        off = ~np.eye(n2, dtype=bool)
        assert np.array_equal(q[c][off], np.conj(np.swapaxes(q[c], 0, 1))[off])          # Hermitian fill


def test_slender_solve_flow_vs_reference_run(solver, oracle):
    """Model.solveDynamics with potSecOrder 1: loop, QTF from the motions, second-order force, loop continued from the
    same iterate -- responses, pass counts, force and QTF against the unmodified reference; Xi_init / Xi_last plumbing."""
    z, P = _slender_golden()
    cs = z["ref_run_solve_cases"]
    n = len(cs)
    table = dict(Hs=cs[:, 0], Tp=cs[:, 1], gamma=np.zeros(n), beta_deg=cs[:, 2], spec=np.zeros(n, dtype=np.int32))
    out = solver.solve_dynamics_slender(P, solver.CaseTable(table), n_iter=int(z["n_iter"]), xi_start=float(z["xi_start"]))
    assert np.array_equal(out["status"][0, :, 0], z["ref_run_solve_passes"])
    assert response_err(out["Xi"][0], z["ref_run_solve_Xi"]) < RTOL
    assert relerr(out["F_2nd"][0], z["ref_run_solve_F2nd"]) < RTOL and relerr(out["F_2nd_mean"][0], z["ref_run_solve_F2nd_mean"]) < RTOL
    for i in range(n):
        assert relerr(out["qtf"][0, i], z["ref_run_solve_qtf"][i]) < RTOL
    # oracle agrees on the converged flag as well
    od = oracle.OracleDesign(P)
    for i in range(n):
        _, st = oracle.solve_dynamics(od, 0, cs[i, 0], cs[i, 1], 0.0, cs[i, 2], nIter=int(z["n_iter"]), XiStart=float(z["xi_start"]))
        assert out["status"][0, i, 1] == st[1]
    # Xi_last of a converged solve is the iterate of its last pass: restarting from it with no extra force reproduces Xi in one pass
    plain = solver.DesignBatch({k: v for k, v in P.items() if not k.startswith("qs_")})
    A = solver.solve_dynamics(plain, solver.CaseTable(table), n_iter=int(z["n_iter"]), xi_start=float(z["xi_start"]), cluster_size=2, want=("Xi", "status", "Xi_last"))
    Bq = solver.solve_dynamics(plain, solver.CaseTable(table, Xi_init=A["Xi_last"]), n_iter=int(z["n_iter"]), cluster_size=2)
    conv = A["status"][0, :, 1] == 1
    assert conv.any() and np.all(Bq["status"][0, conv, 0] == 1)
    assert np.array_equal(Bq["Xi"][0, conv], A["Xi"][0, conv])


def test_slender_model_api(solver):
    """raft_b200.Model / FOWT with potSecOrder 1 from the design dict: calcQTF_slenderBody mirror (fixed body, golden
    pickle) and solveDynamics / analyzeCases against the reference run."""
    import json, os
    from conftest import GOLDEN
    from raft_b200.model import Model
    z, P = _slender_golden()
    D = json.load(open(os.path.join(GOLDEN, "designs.json")))["test_VolturnUS-S"]
    design = dict(D, platform=dict(D["platform"], potSecOrder=1), site=dict(D["site"], water_depth=float(P["depth"])))
    mats = dict(M_struc=P["M0"] - z["A_hydro_morison"], C_struc=P["C0"] - z["C_moor"], C_moor=z["C_moor"])
    model = Model(design, matrices=mats)
    f = model.fowtList[0]
    assert f.potSecOrder == 1 and np.array_equal(f.w1_2nd, P["qs_w"]) and relerr(f.k1_2nd, P["qs_k"]) < 1e-15
    h, t, b = z["ref_pickle_case"]
    f.calcHydroExcitation(dict(wave_spectrum="JONSWAP", wave_height=h, wave_period=t, wave_heading=b, wave_gamma=0))
    q = f.calcQTF_slenderBody(0)
    assert q.shape == z["ref_pickle_qtf"].shape
    for a in range(6):
        assert relerr(q[..., a], z["ref_pickle_qtf"][..., a]) < 1e-9, a
    cases = [dict(wave_spectrum="JONSWAP", wave_height=h_, wave_period=t_, wave_heading=b_) for h_, t_, b_ in z["ref_run_solve_cases"]]
    res = model.analyzeCases(cases=cases)
    assert np.array_equal(res["status"][:, 0, 0], z["ref_run_solve_passes"])
    assert response_err(res["Xi"], z["ref_run_solve_Xi"]) < 1e-9
    assert relerr(f.Fhydro_2nd[0].real, z["ref_run_solve_F2nd"][-1]) < 1e-9
    with pytest.raises(NotImplementedError):
        model.solveDynamics(dict(wave_spectrum=["JONSWAP"] * 2, wave_height=[2.0, 1.0], wave_period=[8.0, 12.0], wave_heading=[0.0, 40.0], wave_gamma=[0.0, 0.0]))

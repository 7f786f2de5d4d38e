#!/usr/bin/env python
"""Generate the golden fixtures under tests/golden/ (run in the BUILD CONTAINER only).

Needs the read-only reference tree at /root/reference; nothing here travels to the GPU box except
the .npz files it writes.  Two sources of truth go into every fixture:

  ref_pickle_*  : arrays copied out of the reference's OWN golden pickles
                  (/root/reference/tests/test_data/<design>_true_hydroExcitation.pkl, ..._hydroLinearization.pkl;
                  produced by tests/test_fowt.py:111-175 of the reference with the full turbine+mooring design)
  ref_run_*     : outputs of the UNMODIFIED reference executed here under the stub harness
                  (oracle/ref_harness.py: moorpy/ccblade/matplotlib stubbed, turbine+mooring stripped,
                  synthetic C_moor) -- FOWT.calcHydroExcitation / calcHydroLinearization / Model.solveDynamics
  P_*           : the packed input tables (raft_b200.packer.pack_fowt on the live reference objects)

Usage:  python tests/golden/make_golden.py [--only NAME]
"""
import argparse
import os
import pickle
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from oracle import ref_harness as rh  # noqa: E402
from raft_b200 import packer  # noqa: E402

REF = rh.REF_ROOT
OUT = os.path.dirname(os.path.abspath(__file__))


def savez_lzma(path, **arrays):
    """np.savez with LZMA-compressed members (zip method 14; np.load reads it as is): the fixtures holding large
    float64 tables stay under 1 MB, where deflate would leave them at 2-3 MB."""
    import io
    import zipfile
    with zipfile.ZipFile(path, "w", compression=zipfile.ZIP_LZMA) as zf:
        for k, v in arrays.items():
            b = io.BytesIO()
            np.lib.format.write_array(b, np.asanyarray(v), allow_pickle=False)
            zf.writestr(k + ".npy", b.getvalue())


def seeded_cases(seed, n):
    """SURVEY.md 8d sea-state distribution: Hs~U[1,10], Tp~U[5,18], gamma=0 (IEC auto), beta~U[-180,180)."""
    rng = np.random.default_rng(seed)
    Hs = rng.uniform(1, 10, n)
    Tp = rng.uniform(5, 18, n)
    beta = rng.uniform(-180, 180, n)
    return Hs, Tp, beta


def count_passes(fowt):
    """Wrap calcHydroLinearization to count the passes of the drag loop (raft_model.py:1063)."""
    cnt = [0]
    orig = fowt.calcHydroLinearization

    def wrapped(Xi):
        cnt[0] += 1
        return orig(Xi)
    fowt.calcHydroLinearization = wrapped
    return cnt, orig


def run_solves(model, cases):
    fowt = model.fowtList[0]
    cnt, orig = count_passes(fowt)
    Xi, passes = [], []
    for (Hs, Tp, beta) in cases:
        cnt[0] = 0
        x = rh.solve_dynamics(model, rh.make_case(Hs, Tp, beta))
        Xi.append(np.array(x[0]))
        passes.append(cnt[0])
    fowt.calcHydroLinearization = orig
    return np.array(Xi), np.array(passes, dtype=np.int32)


DESIGNS = {}


def _plain(x):
    """YAML-loaded design section -> plain JSON types."""
    if isinstance(x, dict):
        return {str(k): _plain(v) for k, v in x.items()}
    if isinstance(x, (list, tuple)):
        return [_plain(v) for v in x]
    if isinstance(x, np.ndarray):
        return x.tolist()
    if isinstance(x, (np.floating, np.integer)):
        return x.item()
    return x


def fixture(name, yaml_path, nw=None, max_freq=None, solve_cases=(), pickles=None, lin_check=True, trains=None):
    t0 = time.time()
    design = rh.load_design(yaml_path, nw=nw, max_freq=max_freq)
    # the input side of the fixture: the design sections the hot path reads (platform members, site, settings)
    plat = {k: v for k, v in design["platform"].items() if k not in ("hydroPath",)}
    DESIGNS[name] = _plain(dict(settings=design.get("settings", {}), site=design["site"], platform=plat))
    model = rh.build_model(design)
    fowt = model.fowtList[0]
    P = packer.pack_fowt(fowt)
    out = {"P_" + k: np.asarray(v) for k, v in P.items()}
    out["n_iter"] = np.int32(int(model.nIter))
    out["xi_start"] = np.float64(model.XiStart)
    out["C_moor"] = np.array(fowt.C_moor)
    out["A_hydro_morison"] = np.array(fowt.A_hydro_morison)

    if pickles:
        with open(pickles + "_true_hydroExcitation.pkl", "rb") as f:
            tv = pickle.load(f)
        out["ref_pickle_exc_heading"] = np.array([t["case"]["wave_heading"] for t in tv], dtype=float)
        out["ref_pickle_exc_period"] = np.array([t["case"]["wave_period"] for t in tv], dtype=float)
        out["ref_pickle_exc_height"] = np.array([t["case"]["wave_height"] for t in tv], dtype=float)
        out["ref_pickle_exc_F_hydro_iner"] = np.array([t["F_hydro_iner"][0] for t in tv])
        assert np.allclose(tv[0]["w"], P["w"])
        with open(pickles + "_true_hydroLinearization.pkl", "rb") as f:
            tv = pickle.load(f)
        out["ref_pickle_lin_B_hydro_drag"] = np.array(tv["B_hydro_drag"])
        out["ref_pickle_lin_F_hydro_drag"] = np.array(tv["F_hydro_drag"])
        with open(pickles + "_true_hydroConstants.pkl", "rb") as f:
            tv = pickle.load(f)
        out["ref_pickle_A_hydro_morison"] = np.array(tv["A_hydro_morison"])

    if lin_check:
        # the reference's own linearisation test recipe (tests/test_fowt.py:150-175), run live
        case = dict(rh.make_case(2, 10, 0), wave_spectrum="unit")
        fowt.calcHydroExcitation(case, memberList=fowt.memberList)
        phase = np.linspace(0, 2 * np.pi, fowt.nw * fowt.nDOF).reshape(fowt.nDOF, fowt.nw)
        Xi = 0.1 * np.exp(1j * phase)
        out["ref_run_lin_Xi"] = Xi
        out["ref_run_lin_B_hydro_drag"] = np.array(fowt.calcHydroLinearization(Xi))
        out["ref_run_lin_F_hydro_drag"] = np.array(fowt.calcDragExcitation(0))
        out["ref_run_lin_F_hydro_iner"] = np.array(fowt.F_hydro_iner[0])
        out["ref_run_lin_F_BEM"] = np.array(fowt.F_BEM[0])
        out["ref_run_lin_zeta"] = np.array(fowt.zeta[0])

    if len(solve_cases):
        Xi, passes = run_solves(model, solve_cases)
        out["ref_run_solve_cases"] = np.array(solve_cases, dtype=float)      # rows (Hs, Tp, heading_deg)
        out["ref_run_solve_Xi"] = Xi
        out["ref_run_solve_passes"] = passes

    if trains is not None:
        # one case with several wave trains (lists in the case dict, raft_fowt.py:1742-1752): Model.Xi[ih]
        case = rh.make_case()
        case.update(wave_heading=[t[2] for t in trains], wave_period=[t[1] for t in trains], wave_height=[t[0] for t in trains],
                    wave_spectrum=["JONSWAP"] * len(trains), wave_gamma=[0.0] * len(trains))
        x = rh.solve_dynamics(model, case)
        out["ref_run_trains"] = np.array(trains, dtype=float)                # rows (Hs, Tp, heading_deg)
        out["ref_run_trains_Xi"] = np.array(x[:len(trains)])

    path = os.path.join(OUT, name + ".npz")
    np.savez_compressed(path, **out)
    print("%-28s nw=%4d Ns=%3d cases=%2d  %.1f s  %.0f KB" % (name, len(P["w"]), len(P["node_ls"]), len(solve_cases),
                                                             time.time() - t0, os.path.getsize(path) / 1024))


def fixture_qtf(name, yaml_path, nw, max_freq, solve_cases, trains):
    """potSecOrder 2 (external .12d QTF): readQTF state, calcHydroForce_2ndOrd per case, Model.solveDynamics with the
    second-order force added (raft_model.py:1035-1048, :1210-1212), a multi-train case, and a synthetic 4-heading table
    (the shipped file has one heading) to exercise the heading interpolation (raft_fowt.py:2178-2187)."""
    import contextlib
    import io
    t0 = time.time()
    design = rh.load_design(yaml_path, nw=nw, max_freq=max_freq, sec_order=True)
    assert int(design["platform"]["potSecOrder"]) == 2
    model = rh.build_model(design)
    fowt = model.fowtList[0]
    P = packer.pack_fowt(fowt)
    out = {"P_" + k: np.asarray(v) for k, v in P.items()}
    out["n_iter"] = np.int32(int(model.nIter))
    out["xi_start"] = np.float64(model.XiStart)
    out["C_moor"] = np.array(fowt.C_moor)
    out["A_hydro_morison"] = np.array(fowt.A_hydro_morison)
    cnt, orig = count_passes(fowt)
    Xi, passes, F2, F2m, S = [], [], [], [], []
    for (Hs, Tp, beta) in solve_cases:
        cnt[0] = 0
        x = rh.solve_dynamics(model, rh.make_case(Hs, Tp, beta))
        Xi.append(np.array(x[0])), passes.append(cnt[0])
        F2.append(np.array(fowt.Fhydro_2nd[0].real)), F2m.append(np.array(fowt.Fhydro_2nd_mean[0])), S.append(np.array(fowt.S[0]))
        assert np.abs(fowt.Fhydro_2nd[0].imag).max() == 0.0
    fowt.calcHydroLinearization = orig
    out["ref_run_solve_cases"] = np.array(solve_cases, dtype=float)
    out["ref_run_solve_Xi"], out["ref_run_solve_passes"] = np.array(Xi), np.array(passes, dtype=np.int32)
    out["ref_run_F2nd"], out["ref_run_F2nd_mean"], out["ref_run_S"] = np.array(F2), np.array(F2m), np.array(S)
    case = rh.make_case()
    case.update(wave_heading=[t[2] for t in trains], wave_period=[t[1] for t in trains], wave_height=[t[0] for t in trains],
                wave_spectrum=["JONSWAP"] * len(trains), wave_gamma=[0.0] * len(trains))
    x = rh.solve_dynamics(model, case)
    out["ref_run_trains"] = np.array(trains, dtype=float)
    out["ref_run_trains_Xi"] = np.array(x[:len(trains)])
    out["ref_run_trains_F2nd"] = np.array(fowt.Fhydro_2nd.real)
    # synthetic multi-heading table: scaled copies of the shipped one
    scale = np.array([1.0, 0.7 + 0.2j, 1.3, -0.4 + 1.0j])
    heads = np.deg2rad(np.array([-90.0, 0.0, 45.0, 180.0]))
    q1 = fowt.qtf[:, :, 0, :]
    fowt.qtf = np.stack([q1 * s for s in scale], axis=2)
    fowt.heads_2nd = heads
    betas = np.array([-120.0, -90.0, -30.0, 0.0, 20.0, 45.0, 100.0, 180.0, 200.0])
    S0 = out["ref_run_S"][0]
    f, fm = [], []
    for b in betas:
        with contextlib.redirect_stdout(io.StringIO()):
            a, bb = fowt.calcHydroForce_2ndOrd(b * 0.017453292519943295, S0)
        fm.append(np.array(a)), f.append(np.array(bb))
    out["mh_scale"], out["mh_heads"], out["mh_betas_deg"] = scale, heads, betas
    out["ref_run_mh_F2nd"], out["ref_run_mh_F2nd_mean"] = np.array(f), np.array(fm)
    path = os.path.join(OUT, name + ".npz")
    np.savez_compressed(path, **out)
    print("%-28s nw=%4d cases=%2d  %.1f s  %.0f KB" % (name, nw, len(solve_cases), time.time() - t0, os.path.getsize(path) / 1024))


def fixture_turbine(name, yaml_path):
    """A design WITH its turbine (rotor + rigid tower; CCBlade stubbed, turbine off, mooring stripped): the turbine
    channels of FOWT.saveTurbineOutputs -- nacelle accelerations and tower-base moment (raft_fowt.py:2401-2444,
    2504-2538) -- from the unmodified reference, for single- and multi-train cases."""
    import contextlib
    import io
    t0 = time.time()
    design = rh.load_design(yaml_path, strip=False)
    design.pop("mooring", None)
    design["platform"]["potSecOrder"] = 0
    model = rh.build_model(design)
    fowt = model.fowtList[0]
    fowt.Xi0 = np.array([0.0, 0.0, 0.0, 0.0, 0.02, 0.0])      # mean pitch of a statics solve (out of scope), for Mbase_avg
    P = packer.pack_fowt(fowt)
    ch = packer.pack_turbine_channels(fowt)
    out = {"P_" + k: np.asarray(v) for k, v in P.items()}
    out["n_iter"], out["xi_start"] = np.int32(int(model.nIter)), np.float64(model.XiStart)
    out["ch_names"] = np.array(["%s:%d" % nm for nm in ch["names"]])
    out["ch_coef"], out["ch_avg"] = ch["coef"], ch["avg"]
    cases = [rh.make_case(6.0, 12.0, 30.0), rh.make_case(2.0, 7.5, -75.0)]
    c3 = rh.make_case()
    c3.update(wave_heading=[0.0, 60.0], wave_period=[10.0, 14.0], wave_height=[4.0, 2.0], wave_spectrum=["JONSWAP"] * 2, wave_gamma=[0.0, 0.0])
    cases.append(c3)
    keys = [d + s for d in ("surge", "sway", "heave", "roll", "pitch", "yaw", "AxRNA", "AyRNA", "AzRNA", "Mbase")
            for s in ("_avg", "_std", "_max", "_min", "_PSD")]
    for ic, case in enumerate(cases):
        x = rh.solve_dynamics(model, case)
        res = {}
        with contextlib.redirect_stdout(io.StringIO()):
            fowt.saveTurbineOutputs(res, case)
        out["ref_run_case%d_Xi" % ic] = np.array(x)                      # [nWaves+1, 6, nw]
        out["ref_run_case%d_trains" % ic] = np.array([np.atleast_1d(case[k]) for k in ("wave_height", "wave_period", "wave_heading")], dtype=float).T
        for k in keys:
            out["ref_run_case%d_%s" % (ic, k)] = np.array(res[k])
    path = os.path.join(OUT, name + ".npz")
    np.savez_compressed(path, **out)
    print("%-28s nw=%4d cases=%2d  %.1f s  %.0f KB" % (name, len(P["w"]), len(cases), time.time() - t0, os.path.getsize(path) / 1024))


def fixture_slender(name, yaml_path, pickle_path, solve_cases):
    """potSecOrder 1 (slender-body QTF): the reference's OWN golden QTF (tests/test_data/*_true_calcQTF_slenderBody.pkl,
    fixed body, reference test test_fowt.py:192-216), plus reference runs of Model.solveDynamics with the QTF computed
    inside the loop (raft_model.py:1106-1131): recorded motion RAOs, QTF with motions, second-order force, response, passes."""
    t0 = time.time()
    design = rh.load_design(yaml_path, sec_order=True)
    assert int(design["platform"]["potSecOrder"]) == 1
    model = rh.build_model(design)
    fowt = model.fowtList[0]
    P = packer.pack_fowt(fowt)
    out = {"P_" + k: np.asarray(v) for k, v in P.items()}
    out["n_iter"], out["xi_start"] = np.int32(int(model.nIter)), np.float64(model.XiStart)
    out["C_moor"], out["A_hydro_morison"] = np.array(fowt.C_moor), np.array(fowt.A_hydro_morison)
    with open(pickle_path, "rb") as f:
        tv = pickle.load(f)
    out["ref_pickle_qtf"] = np.array(tv["qtf"])                                          # [nw2, nw2, 1, 6]
    out["ref_pickle_case"] = np.array([float(np.ravel(tv["case"][k])[0]) for k in ("wave_height", "wave_period", "wave_heading")])
    rec = {}
    orig = fowt.calcQTF_slenderBody

    def wrapped(waveHeadInd, Xi0=None, **kw):
        rec["Xi0"] = np.array(Xi0)
        kw.pop("verbose", None)
        r = orig(waveHeadInd, Xi0=Xi0, **kw)
        rec["qtf"] = np.array(fowt.qtf)
        return r
    fowt.calcQTF_slenderBody = wrapped
    cnt, orig_lin = count_passes(fowt)
    keys = ("Xi", "passes", "Xi0", "qtf", "F2nd", "F2nd_mean")
    acc = {k: [] for k in keys}
    for (Hs, Tp, beta) in solve_cases:
        cnt[0] = 0
        x = rh.solve_dynamics(model, rh.make_case(Hs, Tp, beta))
        acc["Xi"].append(np.array(x[0])), acc["passes"].append(cnt[0]), acc["Xi0"].append(rec["Xi0"]), acc["qtf"].append(rec["qtf"][:, :, 0, :])
        acc["F2nd"].append(np.array(fowt.Fhydro_2nd[0].real)), acc["F2nd_mean"].append(np.array(fowt.Fhydro_2nd_mean[0]))
    fowt.calcHydroLinearization = orig_lin
    out["ref_run_solve_cases"] = np.array(solve_cases, dtype=float)
    for k in keys:
        out["ref_run_solve_" + k] = np.array(acc[k])
    path = os.path.join(OUT, name + ".npz")
    np.savez_compressed(path, **out)
    print("%-28s nw=%4d nw2=%3d cases=%2d  %.1f s  %.0f KB" % (name, len(P["w"]), len(P["qs_w"]), len(solve_cases), time.time() - t0,
                                                             os.path.getsize(path) / 1024))


def fixture_flexible(name, yaml_path, pickles):
    """Generalised degrees of freedom (flexible members, nDOF = 150): the reference's golden excitation / linearisation
    pickles of VolturnUS-S-flexible with the tables packed by packer.pack_general_dofs (oracle groundwork for the next row).
    The design keeps its turbine (the tower is one of the flexible members); CCBlade is stubbed, mooring stripped."""
    import contextlib
    import copy
    import io
    t0 = time.time()
    raft = rh.load_reference()
    design = rh.load_design(yaml_path, strip=False)
    design.pop("mooring", None)
    design["platform"]["potSecOrder"] = 0
    with contextlib.redirect_stdout(io.StringIO()):
        model = raft.Model(copy.deepcopy(design))
        fowt = model.fowtList[0]
        fowt.setPosition(np.zeros(fowt.nDOF))
        fowt.calcStatics()
        fowt.calcTurbineConstants(rh.make_case(), ptfm_pitch=0)
        fowt.calcHydroConstants()
    P = packer.pack_general_dofs(fowt)
    out = {"P_" + k: np.asarray(v) for k, v in P.items()}
    with open(pickles + "_true_hydroExcitation.pkl", "rb") as f:
        tv = pickle.load(f)
    out["ref_pickle_exc_heading"] = np.array([t["case"]["wave_heading"] for t in tv], dtype=float)
    out["ref_pickle_exc_period"] = np.array([t["case"]["wave_period"] for t in tv], dtype=float)
    out["ref_pickle_exc_height"] = np.array([t["case"]["wave_height"] for t in tv], dtype=float)
    out["ref_pickle_exc_F_hydro_iner"] = np.array([t["F_hydro_iner"][0] for t in tv])
    with open(pickles + "_true_hydroLinearization.pkl", "rb") as f:
        tv = pickle.load(f)
    out["ref_pickle_lin_B_hydro_drag"], out["ref_pickle_lin_F_hydro_drag"] = np.array(tv["B_hydro_drag"]), np.array(tv["F_hydro_drag"])
    # full Model.solveDynamics of the 150-DOF system (synthetic mooring stiffness on the rigid-body DOFs 0..5)
    n = fowt.nDOF
    Cmoor = np.zeros([n, n])
    Cmoor[:6, :6] = rh.C_MOOR_DEFAULT
    fowt.C_moor = Cmoor
    out["gen_M"] = np.sum(fowt.A_aero, axis=3)[:, :, 0] + fowt.M_struc + fowt.A_hydro_morison      # raft_model.py:1045-1047 (turbine off: no w dependence)
    out["gen_B"] = np.sum(fowt.B_aero, axis=3)[:, :, 0] + fowt.B_struc + np.sum(fowt.B_gyro, axis=2)
    out["gen_C"] = fowt.C_struc + fowt.C_hydro + Cmoor + fowt.C_elast
    assert np.abs(fowt.A_aero).max() == 0 and np.abs(fowt.A_BEM).max() == 0
    cnt, orig = count_passes(fowt)
    cases = [(6.0, 12.0, 30.0), (2.0, 8.0, -60.0)]
    Xi, passes = [], []
    for (Hs, Tp, beta) in cases:
        cnt[0] = 0
        x = rh.solve_dynamics(model, rh.make_case(Hs, Tp, beta))
        Xi.append(np.array(x[0])), passes.append(cnt[0])
    fowt.calcHydroLinearization = orig
    out["n_iter"], out["xi_start"] = np.int32(int(model.nIter)), np.float64(model.XiStart)
    out["ref_run_solve_cases"], out["ref_run_solve_Xi"], out["ref_run_solve_passes"] = np.array(cases), np.array(Xi), np.array(passes, dtype=np.int32)
    path = os.path.join(OUT, name + ".npz")
    savez_lzma(path, **out)
    print("%-28s nDOF=%3d Ns=%3d  %.1f s  %.0f KB" % (name, int(P["gen_nDOF"]), len(P["node_ls"]), time.time() - t0, os.path.getsize(path) / 1024))


def fixture_farm(name, yaml_path, nw, max_freq, cases, seed=5):
    """Coupled 6N-DOF farm (raft_model.py:1164-1236) run by the UNMODIFIED reference: SURVEY.md 8c recipe -- array rows with
    turbineID = mooringID = 0, array_mooring dropped, ``model.ms`` replaced by an object whose getCoupledStiffnessA returns a
    seeded SPD array-mooring stiffness, moorMod 0.  Stores every FOWT's packed tables (P<i>_*), the coupling matrix and
    Model.Xi [nH+1, 6N, nw] per case."""
    import yaml
    t0 = time.time()
    with open(yaml_path) as f:
        design = yaml.load(f, Loader=yaml.FullLoader)
    for k in ("turbine", "turbines", "mooring", "array_mooring"):
        design.pop(k, None)
    design["platform"]["potSecOrder"] = 0
    ks = design["array"]["keys"]
    for row in design["array"]["data"]:
        row[ks.index("turbineID")] = 0
        row[ks.index("mooringID")] = 0
    design["settings"]["max_freq"] = float(max_freq)
    design["settings"]["min_freq"] = float(max_freq) / nw
    model = rh.build_model(design)
    n = model.nDOF
    rng = np.random.default_rng(seed)
    A = rng.normal(size=(n, n)) * 2e4
    C_arr = A @ A.T / n + np.diag([5e4] * n)

    class _MS:
        def getCoupledStiffnessA(self, lines_only=True):
            return C_arr
    model.ms, model.moorMod = _MS(), 0
    out = dict(C_array=C_arr, n_fowt=np.int32(model.nFOWT), n_iter=np.int32(int(model.nIter)), xi_start=np.float64(model.XiStart),
               cases=np.array(cases, dtype=float), array_xyh=np.array([[f.x_ref, f.y_ref, f.heading_adjust] for f in model.fowtList], dtype=float))
    plat = {k: v for k, v in design["platform"].items() if k not in ("hydroPath",)}
    DESIGNS[name] = _plain(dict(settings=design.get("settings", {}), site=design["site"], platform=plat, array=design["array"]))
    counters = [count_passes(f) for f in model.fowtList]
    Xi, passes = [], []
    for (Hs, Tp, beta) in cases:
        for c, _ in counters:
            c[0] = 0
        x = rh.solve_dynamics(model, rh.make_case(Hs, Tp, beta))
        Xi.append(np.array(x))
        passes.append([c[0] for c, _ in counters])
    for f, (_, orig) in zip(model.fowtList, counters):
        f.calcHydroLinearization = orig
    out["ref_run_Xi"] = np.array(Xi)                                   # [nCases, nH+1, 6N, nw]
    out["ref_run_passes"] = np.array(passes, dtype=np.int32)           # [nCases, nFOWT]
    for i, f in enumerate(model.fowtList):
        P = packer.pack_fowt(f)
        out.update({"P%d_%s" % (i, k): np.asarray(v) for k, v in P.items()})
        out["C_moor%d" % i] = np.array(f.C_moor)
        out["A_hydro_morison%d" % i] = np.array(f.A_hydro_morison)
    np.savez_compressed(os.path.join(OUT, name + ".npz"), **out)
    print("%s: %d FOWTs, nw %d, %d cases, passes %s (%.1f s)" % (name, model.nFOWT, model.nw, len(cases), passes, time.time() - t0))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--only", default=None)
    args = ap.parse_args()
    td = os.path.join(REF, "tests", "test_data")
    jobs = []
    # the reference's own test designs / grids (nw = 40) + its golden pickles
    for nm in ("OC3spar", "VolturnUS-S", "OC4semi-WAMIT_Coefs"):
        cases = [(2.0, 8.0, 0.0), (6.0, 12.0, 30.0), (9.5, 15.0, -135.0), (1.2, 5.5, 90.0)]
        jobs.append(dict(name="test_" + nm, yaml_path=os.path.join(td, nm + ".yaml"), solve_cases=cases,
                         pickles=os.path.join(td, nm)))
    # BASELINE.json configs at reduced size (same recipes as SURVEY.md 8d, fewer bins/cases)
    Hs, Tp, beta = seeded_cases(2, 6)
    jobs.append(dict(name="cfg1_OC3spar", yaml_path=os.path.join(REF, "designs", "OC3spar.yaml"),
                     solve_cases=[(2.0, 8.0, 0.0)], trains=[(2.0, 8.0, 0.0), (3.0, 12.0, 45.0)]))
    jobs.append(dict(name="cfg2_VolturnUS-S_nw64", yaml_path=os.path.join(REF, "designs", "VolturnUS-S.yaml"),
                     nw=64, max_freq=0.512, solve_cases=list(zip(Hs, Tp, beta)),
                     trains=[(6.0, 12.0, 30.0), (2.5, 7.0, -100.0), (1.0, 16.0, 170.0)]))
    Hs, Tp, beta = seeded_cases(3, 4)
    jobs.append(dict(name="cfg3_OC4semi-WAMIT_nw128", yaml_path=os.path.join(REF, "examples", "OC4semi-WAMIT_Coefs.yaml"),
                     nw=128, max_freq=0.256, solve_cases=list(zip(Hs, Tp, beta))))
    for j in jobs:
        if args.only and args.only not in j["name"]:
            continue
        fixture(**j)
    if not args.only or args.only in "cfg3q_OC4semi-QTF_nw96":
        Hs, Tp, beta = seeded_cases(5, 3)
        fixture_qtf("cfg3q_OC4semi-QTF_nw96", os.path.join(REF, "examples", "OC4semi-WAMIT_Coefs.yaml"), nw=96, max_freq=0.256,
                    solve_cases=list(zip(Hs, Tp, beta)) + [(6.0, 12.0, 30.0)], trains=[(6.0, 12.0, 30.0), (2.5, 7.0, -100.0)])
    if not args.only or args.only in "pin_VolturnUS-S-pointInertia":
        # fourth rigid design of the reference's test set (point inertias in the mass matrix): oracle-only fixture, the
        # kernels see the same member tables as test_VolturnUS-S with another M0
        fixture(name="pin_VolturnUS-S-pointInertia", yaml_path=os.path.join(td, "VolturnUS-S-pointInertia.yaml"),
                solve_cases=[(6.0, 12.0, 30.0), (2.0, 8.0, 0.0)], pickles=os.path.join(td, "VolturnUS-S-pointInertia"))
        DESIGNS.pop("pin_VolturnUS-S-pointInertia", None)
    if not args.only or args.only in "pinq_VolturnUS-S-pointInertia":
        # the reference's second slender-body QTF golden (oracle-only fixture: tables + its pickle, no solves)
        fixture_slender("pinq_VolturnUS-S-pointInertia", os.path.join(td, "VolturnUS-S-pointInertia.yaml"),
                        os.path.join(td, "VolturnUS-S-pointInertia_true_calcQTF_slenderBody.pkl"), solve_cases=[(6.0, 12.0, 30.0)])
    if not args.only or args.only in "flex_VolturnUS-S-flexible":
        fixture_flexible("flex_VolturnUS-S-flexible", os.path.join(td, "VolturnUS-S-flexible.yaml"), os.path.join(td, "VolturnUS-S-flexible"))
    if not args.only or args.only in "slender_VolturnUS-S":
        fixture_slender("slender_VolturnUS-S", os.path.join(td, "VolturnUS-S.yaml"), os.path.join(td, "VolturnUS-S_true_calcQTF_slenderBody.pkl"),
                        solve_cases=[(6.0, 12.0, 30.0), (2.0, 7.5, -75.0), (9.0, 15.0, 160.0)])
    if not args.only or args.only in "farm_VolturnUS-S_farm_nw48":
        fixture_farm("farm_VolturnUS-S_farm_nw48", os.path.join(REF, "designs", "VolturnUS-S_farm.yaml"), nw=48, max_freq=0.1024,
                     cases=[(6.0, 12.0, 0.0), (3.5, 9.0, 40.0), (8.0, 14.0, -120.0)])
    if not args.only or args.only in "turb_VolturnUS-S":
        fixture_turbine("turb_VolturnUS-S", os.path.join(td, "VolturnUS-S.yaml"))
    if not args.only:
        # raw WAMIT tables of the OC4 semi (reference data files examples/OC4semi-WAMIT_Coefs/marin_semi.1/.3),
        # read with the product reader, so that readHydro can be exercised at any grid size off the build box
        from raft_b200 import bem
        hp = os.path.join(REF, "examples", "OC4semi-WAMIT_Coefs", "marin_semi")
        A, B, w1 = bem.read_wamit1(hp + ".1")
        _, _, Re, Im, w3, heads = bem.read_wamit3(hp + ".3")
        qtf_rows = np.loadtxt(hp + ".12d")                  # raw .12d rows, for the QTF reader test off the build box
        savez_lzma(os.path.join(OUT, "wamit_marin_semi.npz"), A=A, B=B, w1=w1, Re=Re.astype(np.float64),
                   Im=Im.astype(np.float64), w3=w3, heads=heads, qtf_rows=qtf_rows.astype(np.float32))
        print("wamit_marin_semi.npz %.0f KB" % (os.path.getsize(os.path.join(OUT, "wamit_marin_semi.npz")) / 1024))
    import json
    dj = os.path.join(OUT, "designs.json")
    merged = json.load(open(dj)) if (args.only and os.path.exists(dj)) else {}
    merged.update(DESIGNS)                                   # --only: refresh that fixture's entry, keep the others
    with open(dj, "w") as f:
        json.dump(merged, f, indent=0, sort_keys=True)


if __name__ == "__main__":
    main()

"""ctypes front-end of the plain-C oracle (oracle/raft_oracle.c).

TEST INFRASTRUCTURE ONLY -- importable from tests/, __graft_entry__.smoke() and bench.py's
cpu_baseline / --impl reference legs.  The product package ``raft_b200`` never imports this.
"""
import atexit
import ctypes as C
import os
import shutil
import subprocess
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, "raft_oracle.c")
LIB = os.path.join(HERE, "_build", "libraft_oracle.so")

c_double_p = C.POINTER(C.c_double)
c_int_p = C.POINTER(C.c_int)


class RoDesign(C.Structure):
    _fields_ = [
        ("n_nodes", C.c_int), ("n_members", C.c_int), ("nw", C.c_int), ("n_bem_head", C.c_int),
        ("depth", C.c_double), ("rho", C.c_double), ("g", C.c_double), ("dw", C.c_double),
        ("x_ref", C.c_double), ("y_ref", C.c_double), ("heading_adjust", C.c_double),
        ("prp", c_double_p), ("w", c_double_p), ("k", c_double_p),
        ("mem_q", c_double_p), ("mem_p1", c_double_p), ("mem_p2", c_double_p), ("mem_rA", c_double_p),
        ("mem_circ", c_int_p),
        ("node_r", c_double_p), ("node_mem", c_int_p), ("node_Imat", c_double_p), ("node_a_i", c_double_p),
        ("a_q", c_double_p), ("a_p1", c_double_p), ("a_p2", c_double_p), ("a_End", c_double_p),
        ("Cd_q", c_double_p), ("Cd_p1", c_double_p), ("Cd_p2", c_double_p), ("Cd_End", c_double_p),
        ("M0", c_double_p), ("B0", c_double_p), ("C0", c_double_p),
        ("A_w", c_double_p), ("B_w", c_double_p),
        ("X_BEM", C.c_void_p), ("bem_headings", c_double_p), ("node_Imat_w", C.c_void_p),
        ("n_qtf_w", C.c_int), ("n_qtf_head", C.c_int),
        ("qtf_w", c_double_p), ("qtf_heads", c_double_p), ("qtf", C.c_void_p),
        ("qs", C.c_void_p), ("qs_nw", C.c_int), ("qs_w", c_double_p), ("qs_k", c_double_p),
    ]


_QS_ARRAYS = ("mem_q", "mem_p1", "mem_p2", "mem_mcf", "mem_wl", "mem_r_int", "mem_a_wl", "mem_rwl", "mem_R_wl", "node_mem", "node_r",
              "node_v_side", "node_Ca_p1", "node_Ca_p2", "node_Ca_End", "node_v_end", "node_a_i", "seg_mem", "seg_z1", "seg_z2", "seg_R",
              "seg_rmid", "M_struc")


class RoQtfDesign(C.Structure):
    """ro_qtf_design: member tables of the slender-body QTF (raft_b200.packer.pack_qtf_members, keys qs_*)."""
    _fields_ = [("n_nodes", C.c_int), ("n_members", C.c_int), ("n_seg", C.c_int),
                ("depth", C.c_double), ("rho", C.c_double), ("g", C.c_double)] + [(n, C.c_void_p) for n in _QS_ARRAYS]


def _qs_struct(P, keep):
    q = RoQtfDesign()
    q.n_nodes, q.n_members, q.n_seg = len(P["qs_node_mem"]), len(P["qs_mem_mcf"]), len(P["qs_seg_mem"])
    q.depth, q.rho, q.g = float(P["qs_depth"]), float(P["qs_rho"]), float(P["qs_g"])
    for n in _QS_ARRAYS:
        a = np.ascontiguousarray(P["qs_" + n])
        if a.dtype.kind == "i":
            a = np.ascontiguousarray(a, dtype=np.int32)
        else:
            a = np.ascontiguousarray(a, dtype=np.float64)
        keep["qs_" + n] = a
        setattr(q, n, a.ctypes.data)
    return q


_tmp_lib = None


def build(force=False):
    """Compile the C oracle with gcc (no -march flags: plain IEEE double, no FMA contraction) into oracle/_build, or
    into a fresh temporary directory when the tree is read-only (bench.py may run from one)."""
    global _tmp_lib
    lib = LIB
    if force or not os.path.exists(lib) or os.path.getmtime(lib) < os.path.getmtime(SRC):
        if _tmp_lib is not None and not force:
            return _tmp_lib
        try:
            os.makedirs(os.path.dirname(lib), exist_ok=True)
            writable = os.access(os.path.dirname(lib), os.W_OK)
        except OSError:
            writable = False
        if not writable:
            tmp = tempfile.mkdtemp(prefix="raft_oracle_")
            atexit.register(shutil.rmtree, tmp, True)          # the mapped library outlives its file
            lib = _tmp_lib = os.path.join(tmp, os.path.basename(LIB))
        subprocess.check_call(["gcc", "-O2", "-fPIC", "-shared", "-fopenmp", "-ffp-contract=off",
                               "-o", lib, SRC, "-lm"])
    return lib


_lib = None


def lib():
    global _lib
    if _lib is None:
        _lib = C.CDLL(build())
        _lib.ro_wave_number.restype = C.c_double
        _lib.ro_wave_number.argtypes = [C.c_double, C.c_double]
    return _lib


def _dp(a):
    return a.ctypes.data_as(c_double_p)


def _ip(a):
    return a.ctypes.data_as(c_int_p)


class OracleDesign:
    """Holds contiguous copies of a packed design (raft_b200.packer.pack_fowt output) + the C struct."""

    def __init__(self, P):
        f8 = lambda a: np.ascontiguousarray(a, dtype=np.float64)
        i4 = lambda a: np.ascontiguousarray(a, dtype=np.int32)
        self.keep = k = {}
        for name in ("prp", "w", "k", "mem_q", "mem_p1", "mem_p2", "mem_rA", "node_r", "node_Imat", "node_a_i",
                     "node_a_q", "node_a_p1", "node_a_p2", "node_a_End", "node_Cd_q", "node_Cd_p1", "node_Cd_p2",
                     "node_Cd_End", "M0", "B0", "C0"):
            k[name] = f8(P[name])
        k["mem_circ"] = i4(P["mem_circ"])
        k["node_mem"] = i4(P["node_mem"])
        self.nw = len(k["w"])
        self.Ns = len(k["node_mem"])
        d = RoDesign()
        d.n_nodes, d.n_members, d.nw = self.Ns, len(k["mem_circ"]), self.nw
        d.depth, d.rho, d.g, d.dw = float(P["depth"]), float(P["rho"]), float(P["g"]), float(P["dw"])
        d.x_ref, d.y_ref = float(P.get("x_ref", 0.0)), float(P.get("y_ref", 0.0))
        d.heading_adjust = float(P.get("heading_adjust", 0.0))
        d.prp, d.w, d.k = _dp(k["prp"]), _dp(k["w"]), _dp(k["k"])
        d.mem_q, d.mem_p1, d.mem_p2, d.mem_rA = _dp(k["mem_q"]), _dp(k["mem_p1"]), _dp(k["mem_p2"]), _dp(k["mem_rA"])
        d.mem_circ = _ip(k["mem_circ"])
        d.node_r, d.node_mem, d.node_Imat, d.node_a_i = _dp(k["node_r"]), _ip(k["node_mem"]), _dp(k["node_Imat"]), _dp(k["node_a_i"])
        d.a_q, d.a_p1, d.a_p2, d.a_End = _dp(k["node_a_q"]), _dp(k["node_a_p1"]), _dp(k["node_a_p2"]), _dp(k["node_a_End"])
        d.Cd_q, d.Cd_p1, d.Cd_p2, d.Cd_End = _dp(k["node_Cd_q"]), _dp(k["node_Cd_p1"]), _dp(k["node_Cd_p2"]), _dp(k["node_Cd_End"])
        d.M0, d.B0, d.C0 = _dp(k["M0"]), _dp(k["B0"]), _dp(k["C0"])
        if "A_w" in P and P["A_w"] is not None:
            k["A_w"], k["B_w"] = f8(P["A_w"]), f8(P["B_w"])
            d.A_w, d.B_w = _dp(k["A_w"]), _dp(k["B_w"])
        if "X_BEM" in P and P["X_BEM"] is not None:
            k["X_BEM"] = np.ascontiguousarray(P["X_BEM"], dtype=np.complex128)
            k["bem_headings"] = f8(P["bem_headings"])
            d.X_BEM = k["X_BEM"].ctypes.data_as(C.c_void_p)
            d.bem_headings = _dp(k["bem_headings"])
            d.n_bem_head = len(k["bem_headings"])
        if "node_Imat_w" in P and P["node_Imat_w"] is not None:
            k["node_Imat_w"] = np.ascontiguousarray(P["node_Imat_w"], dtype=np.complex128)
            d.node_Imat_w = k["node_Imat_w"].ctypes.data_as(C.c_void_p)
        if P.get("qtf") is not None:
            # fowt.qtf [nw1, nw2, nheads, 6], fowt.w1_2nd, fowt.heads_2nd (raft_fowt.py:2100-2128)
            k["qtf"] = np.ascontiguousarray(P["qtf"], dtype=np.complex128)
            k["qtf_w"], k["qtf_heads"] = f8(P["qtf_w"]), f8(P["qtf_heads"])
            d.n_qtf_w, d.n_qtf_head = len(k["qtf_w"]), len(k["qtf_heads"])
            assert k["qtf"].shape == (d.n_qtf_w, d.n_qtf_w, d.n_qtf_head, 6)
            d.qtf_w, d.qtf_heads = _dp(k["qtf_w"]), _dp(k["qtf_heads"])
            d.qtf = k["qtf"].ctypes.data_as(C.c_void_p)
        if P.get("qs_w") is not None:
            # slender-body QTF (potSecOrder 1): member tables + second-order grid
            self.qs = _qs_struct(P, k)
            k["qs_w"], k["qs_k"] = f8(P["qs_w"]), f8(P["qs_k"])
            d.qs = C.addressof(self.qs)
            d.qs_nw, d.qs_w, d.qs_k = len(k["qs_w"]), _dp(k["qs_w"]), _dp(k["qs_k"])
        self.c = d


def wave_number(omega, h):
    return lib().ro_wave_number(float(omega), float(h))


def wave_kin(zeta0, beta, w, k, h, r, rho=1025.0, g=9.81):
    """helpers.getWaveKin -> u[3,nw], ud[3,nw], pDyn[nw]."""
    zeta0, w, k, r = (np.ascontiguousarray(x, dtype=np.float64) for x in (zeta0, w, k, r))
    nw = len(w)
    u, ud, p = np.zeros([3, nw], complex), np.zeros([3, nw], complex), np.zeros(nw, complex)
    lib().ro_wave_kin(_dp(zeta0), C.c_double(beta), _dp(w), _dp(k), C.c_double(h), _dp(r), C.c_int(nw),
                      C.c_double(rho), C.c_double(g), u.ctypes.data_as(C.c_void_p), ud.ctypes.data_as(C.c_void_p),
                      p.ctypes.data_as(C.c_void_p))
    return u, ud, p


def get_kinematics(r, Xi, ws):
    r, ws = np.ascontiguousarray(r, dtype=np.float64), np.ascontiguousarray(ws, dtype=np.float64)
    Xi = np.ascontiguousarray(Xi, dtype=np.complex128)
    nw = len(ws)
    dr, v, a = (np.zeros([3, nw], complex) for _ in range(3))
    lib().ro_get_kinematics(_dp(r), Xi.ctypes.data_as(C.c_void_p), _dp(ws), C.c_int(nw), dr.ctypes.data_as(C.c_void_p),
                            v.ctypes.data_as(C.c_void_p), a.ctypes.data_as(C.c_void_p))
    return dr, v, a


def translate_force(f, r):
    f = np.ascontiguousarray(f, dtype=np.complex128)
    r = np.ascontiguousarray(r, dtype=np.float64)
    out = np.zeros(6, complex)
    lib().ro_translate_force(f.ctypes.data_as(C.c_void_p), _dp(r), out.ctypes.data_as(C.c_void_p))
    return out


def translate_matrix(M, r):
    M = np.ascontiguousarray(M, dtype=np.float64)
    r = np.ascontiguousarray(r, dtype=np.float64)
    out = np.zeros([6, 6])
    lib().ro_translate_matrix(_dp(M), _dp(r), _dp(out))
    return out


def jonswap(w, Hs, Tp, gamma=0.0):
    w = np.ascontiguousarray(w, dtype=np.float64)
    S = np.zeros_like(w)
    lib().ro_jonswap(_dp(w), C.c_int(len(w)), C.c_double(Hs), C.c_double(Tp), C.c_double(gamma), _dp(S))
    return S


def calc_hydro_excitation(od, spec, Hs, Tp, gamma, beta_deg):
    """-> zeta[nw], F_BEM[6,nw], F_iner[6,nw], u[Ns,3,nw]  (FOWT.calcHydroExcitation, one wave train)."""
    nw, Ns = od.nw, od.Ns
    zeta = np.zeros(nw)
    F_BEM = np.zeros([6, nw], dtype=np.complex128)
    F_iner = np.zeros([6, nw], dtype=np.complex128)
    u = np.zeros([max(Ns, 1), 3, nw], dtype=np.complex128)
    rc = lib().ro_calc_hydro_excitation(C.byref(od.c), C.c_int(spec), C.c_double(float(Hs)), C.c_double(float(Tp)), C.c_double(float(gamma)),
                                        C.c_double(float(beta_deg)), _dp(zeta), F_BEM.ctypes.data_as(C.c_void_p),
                                        F_iner.ctypes.data_as(C.c_void_p), u.ctypes.data_as(C.c_void_p))
    if rc:
        raise ValueError("Wave spectrum input not recognized.")
    return zeta, F_BEM, F_iner, u[:Ns]


def calc_hydro_linearization(od, u, Xi):
    """-> Bmat[Ns,3,3], B_drag[6,6], F_drag[6,nw]  (FOWT.calcHydroLinearization)."""
    nw, Ns = od.nw, od.Ns
    u = np.ascontiguousarray(u, dtype=np.complex128)
    Xi = np.ascontiguousarray(Xi, dtype=np.complex128)
    Bmat = np.zeros([max(Ns, 1), 3, 3])
    B = np.zeros([6, 6])
    F = np.zeros([6, nw], dtype=np.complex128)
    lib().ro_calc_hydro_linearization(C.byref(od.c), u.ctypes.data_as(C.c_void_p), Xi.ctypes.data_as(C.c_void_p),
                                      _dp(Bmat), _dp(B), F.ctypes.data_as(C.c_void_p))
    return Bmat[:Ns], B, F


def hydro_force_2nd(od, beta, S0):
    """FOWT.calcHydroForce_2ndOrd(beta [rad], S0[nw]) with the design's QTF table -> f_mean[6], f[6,nw]."""
    S0 = np.ascontiguousarray(S0, dtype=np.float64)
    fm, f = np.zeros(6), np.zeros([6, od.nw])
    lib().ro_hydro_force_2nd(C.byref(od.c), C.c_double(float(beta)), _dp(S0), _dp(fm), _dp(f))
    return fm, f


class RoGeneral(C.Structure):
    _fields_ = [("d", C.c_void_p), ("nDOF", C.c_int), ("Tn", c_double_p), ("rr", c_double_p)]


class GeneralDesign:
    """Generalised-DOF design (raft_b200.packer.pack_general_dofs): node tables + per-node T blocks."""

    def __init__(self, P):
        self.od = OracleDesign(P)
        self.n = int(P["gen_nDOF"])
        self.Tn = np.ascontiguousarray(P["gen_Tn"], dtype=np.float64)
        self.rr = np.ascontiguousarray(P["gen_rr"], dtype=np.float64)
        self.c = RoGeneral(C.addressof(self.od.c), self.n, _dp(self.Tn), _dp(self.rr))


def general_excitation(gd, spec, Hs, Tp, gamma, beta_deg):
    """FOWT.calcHydroExcitation with nDOF reduced degrees of freedom -> zeta [nw], F_hydro_iner [nDOF,nw], u [Ns,3,nw]."""
    nw, Ns = gd.od.nw, gd.od.Ns
    zeta = np.zeros(nw)
    F = np.zeros([gd.n, nw], dtype=np.complex128)
    u = np.zeros([max(Ns, 1), 3, nw], dtype=np.complex128)
    rc = lib().ro_general_excitation(C.byref(gd.c), C.c_int(spec), C.c_double(float(Hs)), C.c_double(float(Tp)), C.c_double(float(gamma)),
                                     C.c_double(float(beta_deg)), _dp(zeta), F.ctypes.data_as(C.c_void_p), u.ctypes.data_as(C.c_void_p))
    if rc:
        raise ValueError("Wave spectrum input not recognized.")
    return zeta, F, u


def general_linearization(gd, u, Xi):
    """FOWT.calcHydroLinearization(Xi [nDOF,nw]) + calcDragExcitation(0) -> B_hydro_drag [nDOF,nDOF], F_hydro_drag [nDOF,nw]."""
    nw, Ns = gd.od.nw, gd.od.Ns
    Xi = np.ascontiguousarray(Xi, dtype=np.complex128)
    u = np.ascontiguousarray(u, dtype=np.complex128)
    Bmat = np.zeros([max(Ns, 1), 3, 3])
    B = np.zeros([gd.n, gd.n])
    F = np.zeros([gd.n, nw], dtype=np.complex128)
    lib().ro_general_linearization(C.byref(gd.c), u.ctypes.data_as(C.c_void_p), Xi.ctypes.data_as(C.c_void_p), _dp(Bmat), _dp(B),
                                   F.ctypes.data_as(C.c_void_p))
    return B, F


def general_solve_dynamics(gd, M, B, Cm, spec, Hs, Tp, gamma, beta_deg, nIter=10, tol=0.01, XiStart=0.0):
    """Model.solveDynamics with nDOF reduced degrees of freedom -> Xi [nDOF,nw], status (passes, converged, nan)."""
    n, nw = gd.n, gd.od.nw
    M, B, Cm = (np.ascontiguousarray(x, dtype=np.float64).reshape(n, n) for x in (M, B, Cm))
    Xi = np.zeros([n, nw], dtype=np.complex128)
    st = np.zeros(3, dtype=np.int32)
    rc = lib().ro_general_solve_dynamics(C.byref(gd.c), _dp(M), _dp(B), _dp(Cm), C.c_int(spec), C.c_double(float(Hs)), C.c_double(float(Tp)),
                                         C.c_double(float(gamma)), C.c_double(float(beta_deg)), C.c_int(nIter), C.c_double(tol),
                                         C.c_double(XiStart), Xi.ctypes.data_as(C.c_void_p), _ip(st))
    if rc:
        raise ValueError("Wave spectrum input not recognized.")
    return Xi, st


def qtf_slender(od, beta, Xi):
    """FOWT.calcQTF_slenderBody: heading ``beta`` [rad], motion RAOs ``Xi`` [6, nw2] on the second-order grid
    -> qtf [nw2, nw2, 6] complex, Hermitian-filled (fowt.qtf[:, :, 0, :])."""
    n2 = od.c.qs_nw
    Xi = np.ascontiguousarray(Xi, dtype=np.complex128)
    assert Xi.shape == (6, n2)
    out = np.zeros([n2, n2, 6], dtype=np.complex128)
    lib().ro_qtf_slender(C.byref(od.qs), C.c_int(n2), od.c.qs_w, od.c.qs_k, C.c_double(float(beta)),
                         Xi.ctypes.data_as(C.c_void_p), out.ctypes.data_as(C.c_void_p))
    return out


def solve_dynamics(od, spec, Hs, Tp, gamma, beta_deg, nIter=10, tol=0.01, XiStart=0.0, want_Z=False):
    """-> Xi[6,nw], status(passes, converged, nan) [, Z[nw,6,6], B_drag[6,6]]  (Model.solveDynamics, 1 FOWT)."""
    nw = od.nw
    Xi = np.zeros([6, nw], dtype=np.complex128)
    st = np.zeros(3, dtype=np.int32)
    Z = np.zeros([nw, 6, 6], dtype=np.complex128) if want_Z else None
    Bd = np.zeros([6, 6]) if want_Z else None
    rc = lib().ro_solve_dynamics(C.byref(od.c), C.c_int(spec), C.c_double(float(Hs)), C.c_double(float(Tp)), C.c_double(float(gamma)),
                                 C.c_double(float(beta_deg)), C.c_int(nIter), C.c_double(tol), C.c_double(XiStart),
                                 Xi.ctypes.data_as(C.c_void_p), _ip(st),
                                 Z.ctypes.data_as(C.c_void_p) if want_Z else None, _dp(Bd) if want_Z else None)
    if rc:
        raise ValueError("Wave spectrum input not recognized.")
    return (Xi, st, Z, Bd) if want_Z else (Xi, st)


def solve_dynamics_trains(od, spec, Hs, Tp, gamma, beta_deg, nIter=10, tol=0.01, XiStart=0.0):
    """Model.solveDynamics for one case with several wave trains -> Xi[nH,6,nw], status (train 0 drives the linearisation)."""
    spec = np.ascontiguousarray(spec, dtype=np.int32)
    Hs, Tp, gamma, beta_deg = (np.ascontiguousarray(x, dtype=np.float64) for x in (Hs, Tp, gamma, beta_deg))
    nH = len(spec)
    Xi = np.zeros([nH, 6, od.nw], dtype=np.complex128)
    st = np.zeros(3, dtype=np.int32)
    rc = lib().ro_solve_dynamics_trains(C.byref(od.c), C.c_int(nH), _ip(spec), _dp(Hs), _dp(Tp), _dp(gamma), _dp(beta_deg),
                                        C.c_int(nIter), C.c_double(tol), C.c_double(XiStart), Xi.ctypes.data_as(C.c_void_p), _ip(st))
    if rc:
        raise ValueError("Wave spectrum input not recognized.")
    return Xi, st


def solve_cases(od, cases, nIter=10, tol=0.01, XiStart=0.0, nthreads=0):
    """Batched over a packed case table (raft_b200.packer.pack_cases) -> Xi[nC,6,nw], status[nC,3], threads."""
    nC = len(cases["Hs"])
    Xi = np.zeros([nC, 6, od.nw], dtype=np.complex128)
    st = np.zeros([nC, 3], dtype=np.int32)
    spec = np.ascontiguousarray(cases["spec"], dtype=np.int32)
    Hs, Tp, gam, beta = (np.ascontiguousarray(cases[k], dtype=np.float64) for k in ("Hs", "Tp", "gamma", "beta_deg"))
    used = lib().ro_solve_cases(C.byref(od.c), C.c_int(nC), _ip(spec), _dp(Hs), _dp(Tp), _dp(gam), _dp(beta),
                                C.c_int(nIter), C.c_double(tol), C.c_double(XiStart),
                                Xi.ctypes.data_as(C.c_void_p), _ip(st), C.c_int(nthreads))
    return Xi, st, used


def system_response(Z_sys, F):
    """Z_sys[nw,n,n], F[nw,n] -> Xi[nw,n] through the explicit inverse (raft_model.py:1189-1216)."""
    Z_sys = np.ascontiguousarray(Z_sys, dtype=np.complex128)
    F = np.ascontiguousarray(F, dtype=np.complex128)
    nw, n = F.shape
    Xi = np.zeros([nw, n], dtype=np.complex128)
    bad = lib().ro_system_response(C.c_int(n), C.c_int(nw), Z_sys.ctypes.data_as(C.c_void_p),
                                   F.ctypes.data_as(C.c_void_p), Xi.ctypes.data_as(C.c_void_p))
    if bad:
        raise np.linalg.LinAlgError("singular system matrix at %d frequencies" % bad)
    return Xi

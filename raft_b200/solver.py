"""Host-side driver of the C ABI: packed designs + case table -> libraftk.so -> NumPy / torch results.

Two routes, both straight through the C ABI (no CPU fallback anywhere):

* ``solve_dynamics`` / ``hydro_excitation`` / ``hydro_linearization``: HOST buffers in and out
  (``raftk_*_host``).  This is the reference-facing call: what ``Model.solveDynamics`` would invoke
  when ``raft_b200`` is dropped into RAFT (INTEGRATION.md), and what ``bench.py`` times as ``e2e``.
* ``DeviceSession``: tables, workspace and outputs resident in HBM as torch tensors
  (``raftk_*_dev`` on torch's current stream).  ``bench.py`` times this as ``value``; the sweep
  driver (``raft_b200.sweep``) all-gathers its output tensor over NCCL.
"""
import ctypes as C

import numpy as np

from . import _lib
from ._lib import RaftkCases, RaftkDesigns, RaftkFarm, RaftkGeneral, RaftkOutputs, RaftkSlender, RaftkSolveOpts, check, lib

_F8 = np.float64
_I4 = np.int32


class _Tables(dict):
    """The named host arrays of a DesignBatch / CaseTable.  Every mutation bumps ``version``, which keys the cached C struct
    of the host-buffer calls (building the ~30-pointer ctypes struct costs ~25 us of Python per call otherwise -- 6 % of a
    0.4 ms end-to-end solve).  In-place edits of an array keep its address, so they need no invalidation."""
    version = 0

    def _bump(self):
        self.version += 1

    def __setitem__(self, k, v):
        dict.__setitem__(self, k, v); self._bump()

    def __delitem__(self, k):
        dict.__delitem__(self, k); self._bump()

    def update(self, *a, **kw):
        dict.update(self, *a, **kw); self._bump()

    def pop(self, *a):
        r = dict.pop(self, *a); self._bump(); return r

    def popitem(self):
        r = dict.popitem(self); self._bump(); return r

    def setdefault(self, k, d=None):
        r = dict.setdefault(self, k, d); self._bump(); return r

    def clear(self):
        dict.clear(self); self._bump()


def _host_struct(obj):
    """``obj.struct`` over the host arrays, cached until ``obj.arrays`` is mutated (a COPY is returned when the caller edits it)."""
    ver = obj.arrays.version if isinstance(obj.arrays, _Tables) else None
    c = getattr(obj, "_host_struct_cache", None)
    if ver is None or c is None or c[0] != ver:
        c = (ver, obj.struct(_host_ptr(obj.arrays)))
        obj._host_struct_cache = c
    return c[1]


class DesignBatch:
    """CSR concatenation of packed designs (``packer.pack_fowt`` dicts) sharing one frequency grid."""

    NODE_COLS = ("ls", "cd_q", "cd_p1", "cd_p2", "in_q", "in_p1", "in_p2", "pa")

    def __init__(self, packed):
        if isinstance(packed, dict):
            packed = [packed]
        if len(packed) == 0:
            raise ValueError("DesignBatch needs at least one design")
        P0 = packed[0]
        self.n_designs = len(packed)
        self.w = np.ascontiguousarray(P0["w"], dtype=_F8)
        self.k = np.ascontiguousarray(P0["k"], dtype=_F8)
        self.nw = len(self.w)
        self.depth, self.rho, self.g = float(P0["depth"]), float(P0["rho"]), float(P0["g"])
        self.dw = float(P0["dw"]) if "dw" in P0 else float(self.w[1] - self.w[0])
        a = self.arrays = _Tables()
        member_offset, mem_node_start = [0], [0]
        frames, rAs, arms, circs = [], [], [], []
        cols = {c: [] for c in self.NODE_COLS}
        max_nodes = max_members = 0
        for P in packed:
            if len(P["w"]) != self.nw or float(P["depth"]) != self.depth:
                raise ValueError("all designs of a batch must share the frequency grid and water depth")
            if P is not P0 and (not np.array_equal(np.asarray(P["w"], dtype=_F8), self.w) or float(P["rho"]) != self.rho
                                or float(P["g"]) != self.g):
                raise ValueError("all designs of a batch must share the frequency values, water density and g")
            nm = len(P["mem_circ"])
            frames.append(np.concatenate([P["mem_q"], P["mem_p1"], P["mem_p2"]], axis=1).reshape(nm, 9))
            rAs.append(np.asarray(P["mem_rA"], dtype=_F8).reshape(nm, 3))
            arms.append(np.asarray(P["mem_rA"], dtype=_F8).reshape(nm, 3) - np.asarray(P["prp"], dtype=_F8)[None, :])
            circs.append(np.asarray(P["mem_circ"], dtype=_I4))
            base = mem_node_start[-1]
            ms = np.asarray(P["mem_start"], dtype=np.int64)
            mem_node_start.extend((base + ms[1:]).tolist())
            member_offset.append(member_offset[-1] + nm)
            for c in self.NODE_COLS:
                cols[c].append(np.asarray(P["node_" + c], dtype=_F8))
            max_nodes = max(max_nodes, int(ms[-1]))
            max_members = max(max_members, nm)
        a["member_offset"] = np.array(member_offset, dtype=_I4)
        a["mem_frame"] = np.ascontiguousarray(np.concatenate(frames, axis=0), dtype=_F8)
        a["mem_rA"] = np.ascontiguousarray(np.concatenate(rAs, axis=0), dtype=_F8)
        a["mem_arm"] = np.ascontiguousarray(np.concatenate(arms, axis=0), dtype=_F8)
        a["mem_node_start"] = np.array(mem_node_start, dtype=_I4)
        a["mem_circ"] = np.ascontiguousarray(np.concatenate(circs), dtype=_I4)
        for c in self.NODE_COLS:
            a["node_" + c] = np.ascontiguousarray(np.concatenate(cols[c]), dtype=_F8)
        have_mcf = ["node_in_p1_w" in P and P["node_in_p1_w"] is not None for P in packed]
        if any(have_mcf):
            for c in ("in_p1", "in_p2"):
                a["node_%s_w" % c] = np.ascontiguousarray(np.concatenate([
                    np.asarray(P["node_%s_w" % c], dtype=np.complex128) if h
                    else np.repeat(np.asarray(P["node_" + c], dtype=np.complex128)[:, None], self.nw, axis=1)
                    for P, h in zip(packed, have_mcf)], axis=0))
        for mname in ("M0", "B0", "C0"):
            a[mname] = np.ascontiguousarray(np.stack([np.asarray(P[mname], dtype=_F8).reshape(36) for P in packed]))
        have_w = ["A_w" in P and P["A_w"] is not None for P in packed]
        if any(have_w):
            z = np.zeros([36, self.nw])
            a["A_w"] = np.ascontiguousarray(np.stack([np.asarray(P["A_w"], dtype=_F8).reshape(36, self.nw) if h else z
                                                      for P, h in zip(packed, have_w)]))
            a["B_w"] = np.ascontiguousarray(np.stack([np.asarray(P["B_w"], dtype=_F8).reshape(36, self.nw) if h else z
                                                      for P, h in zip(packed, have_w)]))
        self.n_bem_head = 0
        have_x = [P.get("X_BEM") is not None for P in packed]
        if any(have_x):
            # designs without BEM excitation in a mixed batch (strip-theory platform next to potMod ones) get zero tables
            Px = packed[have_x.index(True)]
            heads = np.ascontiguousarray(Px["bem_headings"], dtype=_F8)
            self.n_bem_head = len(heads)
            for P, h in zip(packed, have_x):
                if h and not np.array_equal(np.asarray(P["bem_headings"], dtype=_F8), heads):
                    raise ValueError("all designs of a batch must share the BEM heading list")
            zx = np.zeros([self.n_bem_head, 6, self.nw], dtype=np.complex128)
            a["bem_headings"] = heads
            a["X_BEM"] = np.ascontiguousarray(np.stack([np.asarray(P["X_BEM"], dtype=np.complex128) if h else zx
                                                        for P, h in zip(packed, have_x)]))
            a["bem_xyh"] = np.ascontiguousarray(np.array(
                [[float(P.get("x_ref", 0.0)), float(P.get("y_ref", 0.0)), float(P.get("heading_adjust", 0.0))] for P in packed],
                dtype=_F8))
        # external QTF (potSecOrder 2): packed [nw1,nw2,nheads,6] per design; one shared table when all designs
        # carry the same one (a geometry-preserving sweep), else stacked on a design axis
        self.n_qtf_w = self.n_qtf_head = 0
        self.qtf_shared = 0
        have_q = [P.get("qtf") is not None for P in packed]
        if any(have_q):
            if not all(have_q):
                raise ValueError("either all or none of the designs of a batch carry a QTF table")
            qw, qh = np.ascontiguousarray(P0["qtf_w"], dtype=_F8), np.ascontiguousarray(P0["qtf_heads"], dtype=_F8)
            for P in packed:
                if not (np.array_equal(P["qtf_w"], qw) and np.array_equal(P["qtf_heads"], qh)):
                    raise ValueError("all designs of a batch must share the QTF frequency and heading axes")
            self.n_qtf_w, self.n_qtf_head = len(qw), len(qh)
            a["qtf_w"], a["qtf_heads"] = qw, qh
            if all(P["qtf"] is P0["qtf"] for P in packed):
                self.qtf_shared = 1
                a["qtf"] = np.ascontiguousarray(P0["qtf"], dtype=np.complex128)
            else:
                a["qtf"] = np.ascontiguousarray(np.stack([np.asarray(P["qtf"], dtype=np.complex128) for P in packed]))
            if a["qtf"].shape[-4:] != (self.n_qtf_w, self.n_qtf_w, self.n_qtf_head, 6):
                raise ValueError("qtf must be [nw1, nw2, nheads, 6] with nw1 == nw2 == len(qtf_w)")
        a["w"], a["k"] = self.w, self.k
        self.n_members_total = int(member_offset[-1])
        self.n_nodes_total = int(mem_node_start[-1])
        self.max_nodes = max(1, max_nodes)
        self.max_members = max(1, max_members)
        self.max_w_classes, self.max_h_classes, self.max_z_classes = self._step_classes(packed)

    @classmethod
    def from_tables(cls, arrays, n_designs, depth, rho, g, dw, max_nodes, max_members, classes):
        """DesignBatch straight from CSR tables (``raft_b200.batch_builder``): ``arrays`` holds the raftk_designs columns
        (member_offset, mem_*, node_*, M0/B0/C0, w, k); ``classes`` = (max_w, max_h, max_z) step-class hints."""
        self = cls.__new__(cls)
        self.arrays = a = _Tables(arrays)
        self.n_designs = int(n_designs)
        self.w, self.k = a["w"], a["k"]
        self.nw = len(self.w)
        self.depth, self.rho, self.g, self.dw = float(depth), float(rho), float(g), float(dw)
        self.n_bem_head = self.n_qtf_w = self.n_qtf_head = self.qtf_shared = 0
        self.n_members_total = int(a["member_offset"][-1])
        self.n_nodes_total = int(a["mem_node_start"][-1])
        self.max_nodes, self.max_members = int(max_nodes), int(max_members)
        self.max_w_classes, self.max_h_classes, self.max_z_classes = (int(c) for c in classes)
        return self

    @staticmethod
    def _step_classes(packed):
        """Upper bounds on the number of distinct node spacings per design, as the fused kernel
        deduplicates them (phase classes keyed by (q_x,q_y)*step, depth classes by q_z*step), + slack."""
        mw = mh = mz = 0
        for P in packed:
            wk, hk, zk = [], [], []
            ms = np.asarray(P["mem_start"], dtype=np.int64)
            for m in range(len(ms) - 1):
                q = np.asarray(P["mem_q"][m], dtype=float)
                ls = np.asarray(P["node_ls"][ms[m]:ms[m + 1]], dtype=float)
                if len(ls):
                    z0 = float(P["mem_rA"][m][2]) + ls[0] * q[2]
                    if not any(abs(a - z0) <= 1e-12 * max(1.0, abs(z0)) for a in zk):
                        zk.append(z0)
                for step in np.diff(ls):
                    kx, ky, kz = q[0] * step, q[1] * step, q[2] * step
                    if abs(kx) > 1e-14 or abs(ky) > 1e-14:
                        tol = 1e-11 * (abs(kx) + abs(ky))
                        if not any(abs(a - kx) <= tol and abs(b - ky) <= tol for a, b in wk):
                            wk.append((kx, ky))
                    if abs(kz) > 1e-14:
                        if not any(abs(a - kz) <= 1e-11 * abs(kz) for a in hk):
                            hk.append(kz)
            mw, mh, mz = max(mw, len(wk)), max(mh, len(hk)), max(mz, len(zk))
        return max(1, mw), max(1, mh), max(1, mz)

    def input_bytes(self):
        return int(sum(v.nbytes for v in self.arrays.values()))

    def struct(self, ptr):
        """Build the C struct; ``ptr(name)`` returns the address (host or device) of array ``name`` or None."""
        s = RaftkDesigns()
        s.n_designs, s.nw = self.n_designs, self.nw
        s.n_members_total, s.n_nodes_total = self.n_members_total, self.n_nodes_total
        s.max_nodes, s.max_members = self.max_nodes, self.max_members
        s.max_w_classes, s.max_h_classes, s.max_z_classes = self.max_w_classes, self.max_h_classes, self.max_z_classes
        s.depth, s.rho, s.g, s.dw = self.depth, self.rho, self.g, self.dw
        for name in ("w", "k", "member_offset", "mem_frame", "mem_rA", "mem_arm", "mem_node_start", "mem_circ",
                     "node_ls", "node_cd_q", "node_cd_p1", "node_cd_p2", "node_in_q", "node_in_p1", "node_in_p2",
                     "node_pa", "node_in_p1_w", "node_in_p2_w", "M0", "B0", "C0", "A_w", "B_w",
                     "bem_headings", "X_BEM", "bem_xyh", "qtf_w", "qtf_heads", "qtf"):
            setattr(s, name, ptr(name) if name in self.arrays else None)
        s.n_bem_head = self.n_bem_head
        s.n_qtf_w, s.n_qtf_head, s.qtf_shared = self.n_qtf_w, self.n_qtf_head, self.qtf_shared
        return s


class CaseTable:
    """SoA case table (``packer.pack_cases`` dict, or keyword arrays)."""

    def __init__(self, cases, zeta=None, F_2nd=None, Xi_init=None):
        """``F_2nd``: optional real [nD,nC,6,nw] second-order force amplitudes added to the linear excitation.
        ``Xi_init``: optional complex [nD,nC,6,nw] starting iterate of the fixed-point loop (instead of xi_start)."""
        self.arrays = a = _Tables()
        for kname in ("Hs", "Tp", "gamma", "beta_deg"):
            a[kname] = np.ascontiguousarray(cases[kname], dtype=_F8)
        a["spec"] = np.ascontiguousarray(cases["spec"], dtype=_I4)
        if np.any((a["spec"] < 0) | (a["spec"] > 3)):
            raise ValueError("Wave spectrum input not recognized.")       # raft_fowt.py:1774
        self.n_cases = len(a["Hs"])
        if zeta is not None:
            a["zeta"] = np.ascontiguousarray(zeta, dtype=_F8)
        if cases.get("primary") is not None:
            pr = np.ascontiguousarray(cases["primary"], dtype=_I4)
            if len(pr) != self.n_cases or np.any(pr < 0) or np.any(pr >= self.n_cases) or np.any(pr[pr] != pr):
                raise ValueError("primary must map every case to a primary case (primary[primary[c]] == primary[c])")
            a["primary"] = pr
        if F_2nd is not None:
            a["F_2nd"] = np.ascontiguousarray(F_2nd, dtype=_F8)
        if Xi_init is not None:
            a["Xi_init"] = np.ascontiguousarray(Xi_init, dtype=np.complex128)

    def input_bytes(self):
        return int(sum(v.nbytes for v in self.arrays.values()))

    def struct(self, ptr):
        s = RaftkCases()
        s.n_cases = self.n_cases
        for name in ("Hs", "Tp", "gamma", "beta_deg", "spec", "zeta", "primary", "F_2nd", "Xi_init"):
            setattr(s, name, ptr(name) if name in self.arrays else None)
        return s


def _host_ptr(arrays):
    return lambda name: arrays[name].ctypes.data


def _alloc_outputs(nD, nC, nw, want, alloc=np.zeros):
    shapes = dict(Xi=([nD, nC, 6, nw], np.complex128), status=([nD, nC, 4], _I4), B_drag=([nD, nC, 6, 6], _F8),
                  F_drag=([nD, nC, 6, nw], np.complex128), F_iner=([nD, nC, 6, nw], np.complex128),
                  F_BEM=([nD, nC, 6, nw], np.complex128), zeta=([nC, nw], _F8),
                  F_2nd=([nD, nC, 6, nw], _F8), F_2nd_mean=([nD, nC, 6], _F8), Xi_last=([nD, nC, 6, nw], np.complex128))
    return {k: alloc(shapes[k][0], dtype=shapes[k][1]) for k in want}


def _out_struct(outs, ptr):
    o = RaftkOutputs()
    for k in ("Xi", "status", "B_drag", "F_drag", "F_iner", "F_BEM", "zeta", "F_2nd", "F_2nd_mean", "Xi_last"):
        setattr(o, k, ptr(outs[k]) if k in outs else None)
    return o


def solve_dynamics(batch, cases, n_iter=10, tol=0.01, xi_start=0.0, cluster_size=0,
                   want=("Xi", "status", "B_drag"), out=None):
    """Model.solveDynamics for every (design, case), host buffers in/out (raft_model.py:966-1302).

    Returns a dict of NumPy arrays: Xi [nD,nC,6,nw] complex128, status [nD,nC,4] int32
    (passes, converged, flags, 0), B_drag [nD,nC,6,6], and optionally F_drag / F_iner / F_BEM / zeta.
    Designs that carry a QTF table (potSecOrder 2) get the difference-frequency force added to the linear
    excitation (raft_model.py:1035-1048); ask for it with ``want`` F_2nd [nD,nC,6,nw] / F_2nd_mean [nD,nC,6].
    """
    want = tuple(dict.fromkeys(tuple(want) + ("Xi", "status")))
    outs = out if out is not None else _alloc_outputs(batch.n_designs, cases.n_cases, batch.nw, want)
    d = _host_struct(batch)
    c = _host_struct(cases)
    o = RaftkSolveOpts(int(n_iter), int(cluster_size), float(tol), float(xi_start), 0, 0)
    os_ = _out_struct(outs, lambda a: a.ctypes.data)
    check(lib.raftk_solve_dynamics_host(C.byref(d), C.byref(c), C.byref(o), C.byref(os_)))
    if np.any(outs["status"][..., 2] & FLAG_PLAN):
        # the device deduplicated more distinct node spacings than the host-side hint allowed for (near-tolerance
        # chains): those units ran no pass and hold zeros.  Re-run with the table sizes the device's own class numbering
        # needs: the same kernel as a correctly hinted call (worst-case sizes, hint 0, rarely fit on chip, and the v1 solver
        # they would fall back to refuses wave trains and Xi_init / Xi_last).  Hint 0 stays as the last resort.
        d = batch.struct(_host_ptr(batch.arrays))                 # a private copy: the cached struct keeps the hints
        d.max_w_classes, d.max_h_classes, d.max_z_classes = device_step_classes(batch)
        check(lib.raftk_solve_dynamics_host(C.byref(d), C.byref(c), C.byref(o), C.byref(os_)))
        if np.any(outs["status"][..., 2] & FLAG_PLAN):
            d.max_w_classes = d.max_h_classes = d.max_z_classes = 0
            check(lib.raftk_solve_dynamics_host(C.byref(d), C.byref(c), C.byref(o), C.byref(os_)))
        if np.any(outs["status"][..., 2] & FLAG_PLAN):
            raise _lib.RaftkError("step-class tables overflowed even with worst-case sizes")
    return outs


def _first_match(close):
    """Row j of the boolean matrix ``close`` [n, n] -> index of its first True among columns x < j, else j."""
    n = len(close)
    c = close & np.tri(n, k=-1, dtype=bool)
    return np.where(c.any(axis=1), c.argmax(axis=1), np.arange(n))


def device_step_classes(batch):
    """Step-class table sizes (max_w, max_h, max_z) that the fused kernels' class numbering needs for every design of
    ``batch``, restating its rule (raftk_fused.cuh / raftk_fused2.cuh k_fused_plan): a node's representative is the FIRST
    earlier node whose spacing key lies within the tolerance, and its class is the number of representatives before that
    node -- along a near-tolerance chain that can exceed the number of distinct keys the host-side hint counts."""
    a = batch.arrays
    mo, ms, fr, rA, ls = a["member_offset"], a["mem_node_start"], a["mem_frame"], a["mem_rA"], a["node_ls"]
    need = [1, 1, 1]
    for dd in range(batch.n_designs):
        m0, m1 = int(mo[dd]), int(mo[dd + 1])
        if m1 == m0:
            continue
        nb, ne = int(ms[m0]), int(ms[m1])
        k = np.zeros([ne - nb, 3])
        z0 = np.zeros(m1 - m0)
        for m in range(m0, m1):
            j0, j1 = int(ms[m]) - nb, int(ms[m + 1]) - nb
            if j1 > j0:
                z0[m - m0] = rA[m, 2] + ls[nb + j0] * fr[m, 2]
                step = ls[nb + j0 + 1:nb + j1] - ls[nb + j0:nb + j1 - 1]
                k[j0 + 1:j1] = fr[m, :3][None, :] * step[:, None]
        for cols, tol in (((0, 1), 1e-11 * (np.abs(k[:, 0]) + np.abs(k[:, 1]))), ((2,), 1e-11 * np.abs(k[:, 2]))):
            valid = np.any(np.abs(k[:, cols]) > 1e-14, axis=1)
            if not valid.any():
                continue
            close = np.ones((len(k), len(k)), dtype=bool)
            for col in cols:
                close &= np.abs(k[None, :, col] - k[:, None, col]) <= tol[:, None]
            rep = _first_match(close)
            isrep = valid & (rep == np.arange(len(k)))
            before = np.concatenate([[0], np.cumsum(isrep)])            # representatives before index x
            slot = 0 if cols == (0, 1) else 1
            need[slot] = max(need[slot], int(before[rep[valid]].max()) + 1)
        close = np.abs(z0[None, :] - z0[:, None]) <= 1e-12 * np.maximum(1.0, np.abs(z0))[:, None]
        rep = _first_match(close)
        before = np.concatenate([[0], np.cumsum(rep == np.arange(len(z0)))])
        need[2] = max(need[2], int(before[rep].max()) + 1)
    return tuple(need)


def solve_dynamics_farm(batch, cases, C_arr=None, M_arr=None, B_arr=None, n_iter=10, tol=0.01, xi_start=0.0, cluster_size=0,
                        want=("Xi", "status", "B_drag"), out=None):
    """Coupled farm response (raft_model.py:1164-1236), host buffers in/out, ONE call: the designs of ``batch`` are the N
    FOWTs of the array; every FOWT's drag linearisation runs as in ``solve_dynamics``, then the 6N x 6N system
    blockdiag(Z_i) + (-w^2 M_arr + i w B_arr + C_arr) is assembled and solved per (case, frequency) on the device.
    -> the per-FOWT output dict plus ``Xi_sys`` complex [nC, 6N, nw] and ``info`` [nC, nw] (k+1 of a zero pivot).
    ``out``: caller-owned result arrays (e.g. page-locked ones from ``pinned_empty``: device-to-host copies then run at
    the link rate instead of through the driver's staging of pageable memory); missing ones are allocated."""
    N, nC, nw = batch.n_designs, cases.n_cases, batch.nw
    n = 6 * N
    want = tuple(dict.fromkeys(tuple(want) + ("Xi", "status")))
    outs = dict(out) if out is not None else {}
    for k_, v in _alloc_outputs(N, nC, nw, tuple(k for k in want if k not in outs)).items():
        outs[k_] = v
    mats = {}
    for nm, v in (("M_arr", M_arr), ("B_arr", B_arr), ("C_arr", C_arr)):
        if v is not None:
            a = np.ascontiguousarray(v, dtype=_F8)
            if a.shape != (n, n):
                raise ValueError("%s must be [%d, %d]" % (nm, n, n))
            mats[nm] = a
    if "Xi_sys" not in outs:
        outs["Xi_sys"] = np.zeros([nC, n, nw], dtype=np.complex128)
    if "info" not in outs:
        outs["info"] = np.zeros([nC, nw], dtype=_I4)
    if outs["Xi_sys"].shape != (nC, n, nw) or outs["Xi_sys"].dtype != np.complex128 or not outs["Xi_sys"].flags.c_contiguous:
        raise ValueError("out['Xi_sys'] must be a C-contiguous complex128 array [%d, %d, %d]" % (nC, n, nw))
    f = RaftkFarm()
    f.n_fowt = N
    for nm in ("M_arr", "B_arr", "C_arr"):
        setattr(f, nm, mats[nm].ctypes.data if nm in mats else None)
    f.Xi_sys, f.info = outs["Xi_sys"].ctypes.data, outs["info"].ctypes.data
    d = _host_struct(batch)
    c = _host_struct(cases)
    o = RaftkSolveOpts(int(n_iter), int(cluster_size), float(tol), float(xi_start), 0, 0)
    os_ = _out_struct(outs, lambda a: a.ctypes.data)
    check(lib.raftk_solve_dynamics_farm_host(C.byref(d), C.byref(c), C.byref(o), C.byref(os_), C.byref(f)))
    return outs


FLAG_NAN, FLAG_SINGULAR, FLAG_PLAN = 1, 2, 4        # include/raftk.h RAFTK_FLAG_*


def raise_on_flags(status):
    """Translate the status flags of solved units into the reference's exceptions: NaN in the response ->
    ``Exception("Nan detected in response vector Xi.")`` (raft_model.py:1098-1099); a singular impedance ->
    ``numpy.linalg.LinAlgError`` (what ``np.linalg.solve`` raises at raft_model.py:1089)."""
    fl = np.asarray(status)[..., 2]
    if np.any(fl & FLAG_PLAN):
        raise _lib.RaftkError("fused solver: step-class tables overflowed the hint; outputs of those units are zero")
    if np.any(fl & FLAG_SINGULAR) and not np.any(fl & FLAG_NAN):
        raise np.linalg.LinAlgError("Singular matrix")
    if np.any(fl & FLAG_NAN):
        raise Exception("Nan detected in response vector Xi.")


def hydro_excitation(batch, cases, want=("F_iner", "F_BEM", "zeta")):
    """FOWT.calcHydroExcitation for every (design, case) (raft_fowt.py:1732-1888), host buffers."""
    outs = _alloc_outputs(batch.n_designs, cases.n_cases, batch.nw, want)
    d = batch.struct(_host_ptr(batch.arrays))
    c = cases.struct(_host_ptr(cases.arrays))
    os_ = _out_struct(outs, lambda a: a.ctypes.data)
    check(lib.raftk_hydro_excitation_host(C.byref(d), C.byref(c), C.byref(os_)))
    return outs


def qtf_slender(P, beta_rad, Xi_rao):
    """FOWT.calcQTF_slenderBody on the GPU (raft_fowt.py:1988-2078) for one design and n (heading, motion RAO) pairs.
    ``P``: packed design with the ``qs_*`` tables (``packer.pack_qtf_members``); ``beta_rad`` [n]; ``Xi_rao`` complex
    [n,6,nw2] motion RAOs on the second-order grid (zeros = fixed body) -> qtf complex [n,nw2,nw2,6], Hermitian-filled."""
    beta = np.ascontiguousarray(np.atleast_1d(beta_rad), dtype=_F8)
    Xi = np.ascontiguousarray(Xi_rao, dtype=np.complex128)
    n, nw2 = len(beta), len(P["qs_w"])
    if Xi.shape != (n, 6, nw2):
        raise ValueError("Xi_rao must be [n,6,nw2] on the second-order grid")
    keep = {}
    s = RaftkSlender()
    nm = len(P["qs_mem_mcf"])
    s.n_nodes, s.n_members, s.n_seg, s.nw = len(P["qs_node_mem"]), nm, len(P["qs_seg_mem"]), nw2
    s.depth, s.rho, s.g = float(P["qs_depth"]), float(P["qs_rho"]), float(P["qs_g"])
    start = np.concatenate([[0], np.cumsum(np.bincount(np.asarray(P["qs_node_mem"], dtype=np.int64), minlength=nm))])
    for name in _lib.SLENDER_ARRAYS:
        a = start if name == "mem_node_start" else np.asarray(P["qs_" + name])
        a = np.ascontiguousarray(a, dtype=_I4 if name in ("mem_mcf", "mem_wl", "mem_node_start", "seg_mem") else _F8)
        keep[name] = a
        setattr(s, name, a.ctypes.data)
    out = np.zeros([n, nw2, nw2, 6], dtype=np.complex128)
    check(lib.raftk_qtf_slender_host(C.byref(s), n, beta.ctypes.data, Xi.ctypes.data, out.ctypes.data))
    return out


def get_rao(Xi, zeta):
    """helpers.getRAO (helpers.py:762-784): response per unit wave amplitude, zero where |zeta| <= 1e-6."""
    Xi, zeta = np.asarray(Xi), np.asarray(zeta)
    ok = np.abs(zeta) > 1e-6
    out = np.zeros_like(Xi, dtype=complex)
    out[..., ok] = Xi[..., ok] / zeta[ok]
    return out


def solve_dynamics_slender(packed, cases, n_iter=10, tol=0.01, xi_start=0.0, cluster_size=0, want=("Xi", "status", "B_drag")):
    """Model.solveDynamics with potSecOrder 1 (raft_model.py:1052-1142) for every (design, case): (A) the drag-linearisation
    loop without second-order forces; (B) where it converged: motion RAOs -> slender-body QTF on the second-order grid ->
    difference-frequency force -> the loop continues from the SAME iterate with the force added and its counter reset
    (the reference sets iiter = 0 and the loop header increments it to 1, raft_model.py:1106-1131, so loop (B) runs at
    most n_iter passes: it is launched with n_iter - 1, i.e. max_pass = n_iter).  Units whose loop (A) did not converge
    keep its result and get no QTF / second-order force (zeros), like the reference, which never computes them there.
    n_iter = 0 is rejected: the reference would still add F_2nd to the final system response (documented deviation).
    ``packed``: list of packed designs carrying ``qs_*`` tables on one second-order grid; ``cases``: CaseTable (single
    wave train per case).  Extra outputs: F_2nd, F_2nd_mean, qtf [nD,nC,nw2,nw2,6]."""
    if isinstance(packed, dict):
        packed = [packed]
    if "primary" in cases.arrays:
        raise NotImplementedError("potSecOrder 1 with several wave trains fails in the reference itself (raft_model.py:1229 rebinds Fhydro_2nd)")
    if n_iter < 1:
        raise ValueError("potSecOrder 1 needs nIter >= 1")
    plain = [{k: v for k, v in P.items() if not k.startswith(("qtf", "qs_"))} for P in packed]
    batch = DesignBatch(plain)
    nD, nC, nw = batch.n_designs, cases.n_cases, batch.nw
    base = {k: v for k, v in cases.arrays.items() if k not in ("F_2nd", "Xi_init")}
    wantA = tuple(dict.fromkeys(tuple(want) + ("Xi", "status", "zeta", "Xi_last")))
    A = solve_dynamics(batch, CaseTable(base, zeta=base.get("zeta")), n_iter=n_iter, tol=tol, xi_start=xi_start, cluster_size=cluster_size, want=wantA)
    qw = np.ascontiguousarray(packed[0]["qs_w"], dtype=_F8)
    beta_rad = cases.arrays["beta_deg"] * 0.017453292519943295
    qtf = np.zeros([nD, nC, len(qw), len(qw), 6], dtype=np.complex128)
    for d, P in enumerate(packed):
        if not np.array_equal(P["qs_w"], qw):
            raise ValueError("all designs of a batch must share the second-order frequency grid")
        Xi2 = np.zeros([nC, 6, len(qw)], dtype=np.complex128)
        for c in range(nC):
            r = get_rao(A["Xi"][d, c], A["zeta"][c])
            for a in range(6):
                Xi2[c, a] = np.interp(qw, batch.w, r[a], left=0, right=0)          # raft_fowt.py:2021-2023
        qtf[d] = qtf_slender(P, beta_rad, Xi2)
    qb = DesignBatch(plain)
    qb.arrays["qtf_w"], qb.arrays["qtf_heads"] = qw, np.zeros(1)
    qb.arrays["qtf"] = np.ascontiguousarray(qtf.reshape(nD, nC, len(qw), len(qw), 1, 6))
    qb.n_qtf_w, qb.n_qtf_head, qb.qtf_shared = len(qw), 1, 2
    F2 = second_order_force(qb, CaseTable(base, zeta=base.get("zeta")))
    B = solve_dynamics(batch, CaseTable(base, zeta=base.get("zeta"), F_2nd=F2["F_2nd"], Xi_init=A["Xi_last"]), n_iter=n_iter - 1, tol=tol,
                       xi_start=xi_start, cluster_size=cluster_size, want=wantA)
    ok = A["status"][:, :, 1] == 1                                                   # units whose first loop converged
    out = {}
    for k in wantA:
        if k == "zeta":
            out[k] = A[k]
            continue
        sel = ok.reshape(ok.shape + (1,) * (A[k].ndim - 2))
        out[k] = np.where(sel, B[k], A[k])
    out["status"][:, :, 0] = A["status"][:, :, 0] + np.where(ok, B["status"][:, :, 0], 0)
    out["status"][:, :, 2] = A["status"][:, :, 2] | np.where(ok, B["status"][:, :, 2], 0)
    okf = ok[:, :, None, None]
    out["F_2nd"] = np.where(okf, F2["F_2nd"], 0.0)
    out["F_2nd_mean"] = np.where(ok[:, :, None], F2["F_2nd_mean"], 0.0)
    out["qtf"] = np.where(ok[:, :, None, None, None], qtf, 0.0)
    return out


def _general_struct(P, M, B, Cm, ptr_of):
    """raftk_general for a packed flexible design; ``ptr_of(name, array)`` returns the address to store (host or device)."""
    n, nw, Ns = int(P["gen_nDOF"]), len(P["w"]), len(P["node_ls"])
    g = RaftkGeneral()
    g.n_dof, g.nw, g.n_nodes = n, nw, Ns
    g.depth, g.rho, g.dw = float(P["depth"]), float(P["rho"]), float(P["dw"])
    mem = np.asarray(P["node_mem"], dtype=np.int64)
    frame = np.concatenate([np.asarray(P["mem_q"])[mem], np.asarray(P["mem_p1"])[mem], np.asarray(P["mem_p2"])[mem]], axis=1) if Ns else np.zeros([0, 9])
    cd = np.stack([np.asarray(P["node_a_q"]) * np.asarray(P["node_Cd_q"]), np.asarray(P["node_a_p1"]) * np.asarray(P["node_Cd_p1"]),
                   np.asarray(P["node_a_p2"]) * np.asarray(P["node_Cd_p2"]), np.asarray(P["node_a_End"]) * np.asarray(P["node_Cd_End"])], axis=1) if Ns else np.zeros([0, 4])
    arrays = dict(w=P["w"], k=P["k"], node_r=P["node_r"], node_frame=frame, node_circ=np.asarray(P["mem_circ"], dtype=_I4)[mem] if Ns else np.zeros(0, dtype=_I4),
                  node_Imat=P["node_Imat"], node_a_i=P["node_a_i"], node_cd=cd, Tn=P["gen_Tn"], rr=P["gen_rr"], M=M, B=B, C=Cm)
    if P.get("node_Imat_w") is not None:
        arrays["node_Imat_w"] = np.ascontiguousarray(P["node_Imat_w"], dtype=np.complex128)
    for name in _lib.GENERAL_ARRAYS:
        if name not in arrays:
            setattr(g, name, None)
            continue
        a = np.ascontiguousarray(arrays[name], dtype=_I4 if name == "node_circ" else (np.complex128 if name == "node_Imat_w" else _F8))
        setattr(g, name, ptr_of(name, a))
    return g


class GeneralSession:
    """Generalised-DOF solve with tables, workspace and outputs resident in HBM (torch tensors), kernels on torch's current
    stream: ``solve()`` enqueues raftk_general_solve_dynamics_dev -> (Xi [nC,nDOF,nw] complex, status [nC,4])."""

    def __init__(self, P, M, B, Cm, cases, device=None):
        import torch
        self.torch = torch
        self.device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        self.keep = {}

        def to_dev(name, a):
            t = torch.from_numpy(a.view(np.float64) if a.dtype == np.complex128 else a).to(self.device)
            self.keep[name] = t
            return t.data_ptr()
        with torch.cuda.device(self.device):
            self.g = _general_struct(P, M, B, Cm, to_dev)
            self.ct = {k: torch.from_numpy(v).to(self.device) for k, v in cases.arrays.items()}
            self.c_struct = cases.struct(lambda name: self.ct[name].data_ptr())
            n, nw, nC = int(P["gen_nDOF"]), len(P["w"]), cases.n_cases
            self.workspace_bytes = int(lib.raftk_general_workspace_bytes(C.byref(self.g), nC))
            self.workspace = torch.empty(self.workspace_bytes, dtype=torch.uint8, device=self.device)
            self.Xi = torch.zeros([nC, n, nw], dtype=torch.complex128, device=self.device)
            self.status = torch.zeros([nC, 4], dtype=torch.int32, device=self.device)

    def solve(self, n_iter=10, tol=0.01, xi_start=0.0):
        o = RaftkSolveOpts(int(n_iter), 0, float(tol), float(xi_start), 0, 0)
        with self.torch.cuda.device(self.device):
            check(lib.raftk_general_solve_dynamics_dev(C.byref(self.g), C.byref(self.c_struct), C.byref(o), self.Xi.data_ptr(), self.status.data_ptr(),
                                                       self.workspace.data_ptr(), self.workspace_bytes, self.torch.cuda.current_stream(self.device).cuda_stream))
        return self.Xi, self.status


def general_solve_dynamics(P, M, B, Cm, cases, n_iter=10, tol=0.01, xi_start=0.0):
    """Model.solveDynamics for one FOWT with generalised degrees of freedom (flexible members), host buffers:
    ``P`` from ``packer.pack_general_dofs`` (node tables + ``gen_Tn``, ``gen_rr``), constant system
    matrices ``M, B, Cm`` [nDOF,nDOF], ``cases`` a CaseTable -> (Xi complex [nC,nDOF,nw], status [nC,4])."""
    n, nw, Ns = int(P["gen_nDOF"]), len(P["w"]), len(P["node_ls"])
    keep = {}
    g = RaftkGeneral()
    g.n_dof, g.nw, g.n_nodes = n, nw, Ns
    g.depth, g.rho, g.dw = float(P["depth"]), float(P["rho"]), float(P["dw"])
    mem = np.asarray(P["node_mem"], dtype=np.int64)
    frame = np.concatenate([np.asarray(P["mem_q"])[mem], np.asarray(P["mem_p1"])[mem], np.asarray(P["mem_p2"])[mem]], axis=1) if Ns else np.zeros([0, 9])
    cd = np.stack([np.asarray(P["node_a_q"]) * np.asarray(P["node_Cd_q"]), np.asarray(P["node_a_p1"]) * np.asarray(P["node_Cd_p1"]),
                   np.asarray(P["node_a_p2"]) * np.asarray(P["node_Cd_p2"]), np.asarray(P["node_a_End"]) * np.asarray(P["node_Cd_End"])], axis=1) if Ns else np.zeros([0, 4])
    arrays = dict(w=P["w"], k=P["k"], node_r=P["node_r"], node_frame=frame, node_circ=np.asarray(P["mem_circ"], dtype=_I4)[mem] if Ns else np.zeros(0, dtype=_I4),
                  node_Imat=P["node_Imat"], node_a_i=P["node_a_i"], node_cd=cd, Tn=P["gen_Tn"], rr=P["gen_rr"], M=M, B=B, C=Cm)
    if P.get("node_Imat_w") is not None:
        arrays["node_Imat_w"] = np.ascontiguousarray(P["node_Imat_w"], dtype=np.complex128)
    for name in _lib.GENERAL_ARRAYS:
        if name not in arrays:
            setattr(g, name, None)
            continue
        a = arrays[name]
        a = np.ascontiguousarray(a, dtype=_I4 if name == "node_circ" else (np.complex128 if name == "node_Imat_w" else _F8))
        keep[name] = a
        setattr(g, name, a.ctypes.data)
    nC = cases.n_cases
    Xi = np.zeros([nC, n, nw], dtype=np.complex128)
    st = np.zeros([nC, 4], dtype=_I4)
    c = cases.struct(_host_ptr(cases.arrays))
    o = RaftkSolveOpts(int(n_iter), 0, float(tol), float(xi_start), 0, 0)
    check(lib.raftk_general_solve_dynamics_host(C.byref(g), C.byref(c), C.byref(o), Xi.ctypes.data, st.ctypes.data))
    return Xi, st


def second_order_force(batch, cases):
    """FOWT.calcHydroForce_2ndOrd (raft_fowt.py:2158-2253) for every (design, case) from the designs' QTF table,
    host buffers -> dict(F_2nd [nD,nC,6,nw] real amplitudes, F_2nd_mean [nD,nC,6])."""
    if batch.n_qtf_w == 0:
        raise ValueError("the designs carry no QTF table (potSecOrder 2 / packer.pack_qtf)")
    outs = _alloc_outputs(batch.n_designs, cases.n_cases, batch.nw, ("F_2nd", "F_2nd_mean"))
    d = batch.struct(_host_ptr(batch.arrays))
    c = cases.struct(_host_ptr(cases.arrays))
    os_ = _out_struct(outs, lambda a: a.ctypes.data)
    check(lib.raftk_second_order_force_host(C.byref(d), C.byref(c), C.byref(os_)))
    return outs


def hydro_linearization(batch, cases, Xi, want=("B_drag", "F_drag")):
    """FOWT.calcHydroLinearization(Xi) + calcDragExcitation(0) (raft_fowt.py:1891-1957), host buffers.

    ``Xi`` complex [nD,nC,6,nw] (or [6,nw], broadcast to every unit)."""
    nD, nC, nw = batch.n_designs, cases.n_cases, batch.nw
    Xi = np.asarray(Xi, dtype=np.complex128)
    if Xi.shape == (6, nw):
        Xi = np.broadcast_to(Xi, (nD, nC, 6, nw))
    Xi = np.ascontiguousarray(Xi)
    if Xi.shape != (nD, nC, 6, nw):
        raise ValueError("Xi must have shape [nD,nC,6,nw] or [6,nw]")
    outs = _alloc_outputs(nD, nC, nw, want)
    d = batch.struct(_host_ptr(batch.arrays))
    c = cases.struct(_host_ptr(cases.arrays))
    os_ = _out_struct(outs, lambda a: a.ctypes.data)
    check(lib.raftk_hydro_linearization_host(C.byref(d), C.byref(c), Xi.ctypes.data, C.byref(os_)))
    return outs


def system_solve(Z, F):
    """Farm system response (raft_model.py:1164-1216): Z [nw,n,n], F [nw,n] or [nw,n,nrhs] -> Xi, info."""
    Z = np.array(Z, dtype=np.complex128, order="C")
    F = np.array(F, dtype=np.complex128, order="C")
    squeeze = F.ndim == 2
    if squeeze:
        F = np.ascontiguousarray(F[:, :, None])
    nw, n, nrhs = F.shape
    if Z.shape != (nw, n, n):
        raise ValueError("Z must be [nw,n,n] matching F")
    info = np.zeros(nw, dtype=_I4)
    check(lib.raftk_system_solve_host(n, nw, nrhs, Z.ctypes.data, F.ctypes.data, info.ctypes.data))
    return (F[:, :, 0] if squeeze else F), info


_PINNED = []


def response_stats(Xi, dw, psd=True, rot_deg=True):
    """std / PSD per DOF of responses Xi [...,6,nw] (FOWT.saveTurbineOutputs, raft_fowt.py:2299-2353):
    std = sqrt(1/2 sum |Xi|^2), PSD = 1/2 |Xi|^2 / dw, rotations in degrees.  -> (std [...,6], PSD [...,6,nw] or None)."""
    Xi = np.ascontiguousarray(Xi, dtype=np.complex128)
    lead, nw = Xi.shape[:-2], Xi.shape[-1]
    if Xi.shape[-2] != 6:
        raise ValueError("Xi must be [..., 6, nw]")
    n = int(np.prod(lead)) if lead else 1
    sd = np.zeros(lead + (6,))
    P = np.zeros(lead + (6, nw)) if psd else None
    check(lib.raftk_response_stats_host(n, nw, float(dw), 1 if rot_deg else 0, Xi.ctypes.data, sd.ctypes.data,
                                        P.ctypes.data if psd else None))
    return sd, P


def channel_stats(coef, Xi, dw, psd=True, amp=False):
    """Statistics of linear output channels Y = sum_dof coef * Xi (nacelle accelerations, tower-base moment;
    raft_fowt.py:2401-2444, 2504-2538; coefficients from ``packer.pack_turbine_channels``).
    ``coef`` complex [nD,nch,6,nw] (or [nch,6,nw]); ``Xi`` complex [nD,nC,6,nw] (or [nC,6,nw])
    -> (std [nD,nC,nch], PSD [nD,nC,nch,nw] or None, amplitudes complex [nD,nC,nch,nw] or None)."""
    coef = np.ascontiguousarray(coef, dtype=np.complex128)
    Xi = np.ascontiguousarray(Xi, dtype=np.complex128)
    squeeze = coef.ndim == 3
    if squeeze:
        coef, Xi = coef[None], Xi[None]
    nD, nch, _, nw = coef.shape
    if Xi.ndim != 4 or Xi.shape[0] != nD or Xi.shape[2:] != (6, nw) or coef.shape[2] != 6:
        raise ValueError("coef must be [nD,nch,6,nw] and Xi [nD,nC,6,nw]")
    nC = Xi.shape[1]
    sd = np.zeros([nD, nC, nch])
    P = np.zeros([nD, nC, nch, nw]) if psd else None
    A = np.zeros([nD, nC, nch, nw], dtype=np.complex128) if amp else None
    check(lib.raftk_channel_stats_host(nD, nC, nch, nw, float(dw), coef.ctypes.data, Xi.ctypes.data, sd.ctypes.data,
                                       P.ctypes.data if psd else None, A.ctypes.data if amp else None))
    if squeeze:
        sd, P, A = sd[0], (P[0] if psd else None), (A[0] if amp else None)
    return sd, P, A


def pinned_empty(shape, dtype):
    """NumPy array backed by page-locked host memory (cudaHostAlloc) for the e2e path."""
    dtype = np.dtype(dtype)
    n = int(np.prod(shape)) * dtype.itemsize
    p = lib.raftk_host_alloc(max(n, 1))
    if not p:
        raise MemoryError("cudaHostAlloc failed")
    buf = (C.c_char * max(n, 1)).from_address(p)
    arr = np.frombuffer(buf, dtype=dtype, count=int(np.prod(shape))).reshape(shape)
    _PINNED.append((buf, p))        # keep alive; page-locked blocks live until process exit
    return arr


class DeviceSession:
    """Tables, workspace and outputs resident in HBM (torch tensors); kernels on torch's current stream."""

    def __init__(self, batch, cases, device=None, want=("Xi", "status", "B_drag"), workspace_bytes=None, tables=False, out_tensors=None):
        """``tables=True`` sizes the workspace for ``excitation()`` / ``linearization()`` (global wave tables);
        the default covers ``solve()`` only (the fused solver keeps its tables on chip).  ``out_tensors``: outputs the
        caller already owns (name -> tensor of the documented shape), e.g. this rank's block of a peer-shared array."""
        import torch
        self.torch = torch
        self.device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        self.batch, self.cases = batch, cases
        with torch.cuda.device(self.device):
            # every input table (design + case columns) lives in ONE device block, 256-byte aligned slots: a caller that
            # refreshes the tables from the host (sweep.ShardedSolve.step_host) sends them with a single copy
            items, total = [], 0
            for grp, arrs in (("d", batch.arrays), ("c", cases.arrays)):
                for k, v in arrs.items():
                    v = np.ascontiguousarray(v)
                    v = v.view(np.float64) if v.dtype == np.complex128 else v
                    items.append((grp, k, v, total))
                    total += (v.nbytes + 255) // 256 * 256
            host_block = np.zeros(max(total, 256), dtype=np.uint8)
            for _, _, v, off in items:
                host_block[off:off + v.nbytes] = v.reshape(-1).view(np.uint8)
            self.tables = torch.from_numpy(host_block).to(self.device)
            self.table_bytes = int(total)
            self.dt, self.ct = {}, {}
            for grp, k, v, off in items:
                tdt = torch.from_numpy(np.empty(0, dtype=v.dtype)).dtype
                t = self.tables[off:off + v.nbytes].view(tdt).view(v.shape) if v.nbytes else torch.from_numpy(v).to(self.device)
                (self.dt if grp == "d" else self.ct)[k] = t
            self.d_struct = batch.struct(lambda name: self.dt[name].data_ptr())
            self.c_struct = cases.struct(lambda name: self.ct[name].data_ptr())
            need = (lib.raftk_workspace_bytes if tables else lib.raftk_solve_workspace_bytes)(C.byref(self.d_struct), cases.n_cases)
            self.workspace_bytes = int(need if workspace_bytes is None else workspace_bytes)
            self.workspace = torch.empty(self.workspace_bytes, dtype=torch.uint8, device=self.device)
            nD, nC, nw = batch.n_designs, cases.n_cases, batch.nw
            want = tuple(dict.fromkeys(tuple(want) + ("Xi", "status") + (("F_2nd", "F_2nd_mean") if batch.n_qtf_w else ())))
            shapes = dict(Xi=([nD, nC, 6, nw], torch.complex128), status=([nD, nC, 4], torch.int32),
                          F_2nd=([nD, nC, 6, nw], torch.float64), F_2nd_mean=([nD, nC, 6], torch.float64),
                          B_drag=([nD, nC, 6, 6], torch.float64), F_drag=([nD, nC, 6, nw], torch.complex128),
                          F_iner=([nD, nC, 6, nw], torch.complex128), F_BEM=([nD, nC, 6, nw], torch.complex128),
                          zeta=([nC, nw], torch.float64))
            given = dict(out_tensors or {})
            for k, t in given.items():
                if tuple(t.shape) != tuple(shapes[k][0]) or t.dtype != shapes[k][1] or not t.is_contiguous():
                    raise ValueError("out_tensors[%r] must be a contiguous %s tensor of shape %s" % (k, shapes[k][1], shapes[k][0]))
            self.out = {k: (given[k] if k in given else torch.zeros(shapes[k][0], dtype=shapes[k][1], device=self.device)) for k in want}
            self.o_struct = _out_struct(self.out, lambda t: t.data_ptr())

    def _stream(self):
        return self.torch.cuda.current_stream(self.device).cuda_stream

    def _opts(self, n_iter, tol, xi_start, cluster_size):
        """Solve options; from the second call with the same cluster size on, the per-design plan blobs that the first call
        left in the session's workspace are reused (the session owns tables and workspace, so they cannot have changed)."""
        key = int(cluster_size)
        o = RaftkSolveOpts(int(n_iter), key, float(tol), float(xi_start), 1 if getattr(self, "_plan_key", None) == key else 0, 0)
        self._plan_key = key
        return o

    def solve(self, n_iter=10, tol=0.01, xi_start=0.0, cluster_size=0):
        """Enqueue Model.solveDynamics for all units on the current stream; returns the output dict (async)."""
        o = self._opts(n_iter, tol, xi_start, cluster_size)
        with self.torch.cuda.device(self.device):
            check(lib.raftk_solve_dynamics_dev(C.byref(self.d_struct), C.byref(self.c_struct), C.byref(o),
                                               C.byref(self.o_struct), self.workspace.data_ptr(), self.workspace_bytes,
                                               self._stream()))
        return self.out

    def solve_gather(self, peers, o_struct=None, n_iter=10, tol=0.01, xi_start=0.0, cluster_size=0, timeout_flag=None):
        """``solve`` with the multi-GPU exchange fused into the kernel (``raft_b200.sweep.PeerExchange``): every finished
        unit is stored into all ranks' gathered arrays over NVLink, then the stream waits for the peers' arrival flags."""
        o = self._opts(n_iter, tol, xi_start, cluster_size)
        os_ = self.o_struct if o_struct is None else o_struct
        with self.torch.cuda.device(self.device):
            check(lib.raftk_solve_dynamics_gather_dev(C.byref(self.d_struct), C.byref(self.c_struct), C.byref(o), C.byref(os_),
                                                      C.byref(peers), self.workspace.data_ptr(), self.workspace_bytes, self._stream()))
            check(lib.raftk_peer_barrier_dev(C.byref(peers), timeout_flag, self._stream()))

    def farm_response(self, C_arr=None, M_arr=None, B_arr=None):
        """Enqueue the coupled 6N-DOF system response of the LAST ``solve`` (the session's designs are the FOWTs of the
        array; it must have been created with want including B_drag, F_drag, F_iner [+ F_BEM]).  -> (Xi_sys [nC,6N,nw], info)."""
        torch = self.torch
        N, nC, nw = self.batch.n_designs, self.cases.n_cases, self.batch.nw
        n = 6 * N
        if not hasattr(self, "_farm"):
            with torch.cuda.device(self.device):
                mats = {nm: (torch.from_numpy(np.ascontiguousarray(v, dtype=_F8)).to(self.device) if v is not None else None)
                        for nm, v in (("M_arr", M_arr), ("B_arr", B_arr), ("C_arr", C_arr))}
                xi = torch.zeros([nC, n, nw], dtype=torch.complex128, device=self.device)
                info = torch.zeros([nC, nw], dtype=torch.int32, device=self.device)
            f = RaftkFarm()
            f.n_fowt = N
            for nm, t in mats.items():
                setattr(f, nm, t.data_ptr() if t is not None else None)
            f.Xi_sys, f.info = xi.data_ptr(), info.data_ptr()
            self._farm = (f, mats, xi, info)
        f, _, xi, info = self._farm
        with torch.cuda.device(self.device):
            check(lib.raftk_farm_response_dev(C.byref(self.d_struct), C.byref(self.c_struct), C.byref(self.o_struct), C.byref(f), self._stream()))
        return xi, info

    def second_order_force(self):
        """Enqueue FOWT.calcHydroForce_2ndOrd for all units -> out['F_2nd'], out['F_2nd_mean'] (async)."""
        with self.torch.cuda.device(self.device):
            check(lib.raftk_second_order_force_dev(C.byref(self.d_struct), C.byref(self.c_struct), C.byref(self.o_struct),
                                                   self._stream()))
        return self.out

    def excitation(self):
        with self.torch.cuda.device(self.device):
            check(lib.raftk_hydro_excitation_dev(C.byref(self.d_struct), C.byref(self.c_struct), C.byref(self.o_struct),
                                                 self.workspace.data_ptr(), self.workspace_bytes, self._stream()))
        return self.out

    def linearization(self, Xi):
        """Xi: complex128 torch tensor [nD,nC,6,nw] on the session's device (after ``excitation``)."""
        with self.torch.cuda.device(self.device):
            check(lib.raftk_hydro_linearization_dev(C.byref(self.d_struct), C.byref(self.c_struct), Xi.data_ptr(),
                                                    C.byref(self.o_struct), self.workspace.data_ptr(),
                                                    self.workspace_bytes, self._stream()))
        return self.out


def launch_count():
    return int(lib.raftk_launch_count())


def fp64_peak_gflops(iters=20000):
    return float(lib.raftk_fp64_peak_gflops(int(iters)))


def profile_enable(on=True):
    lib.raftk_profile_enable(1 if on else 0)


def profile_read():
    """-> (ms[3], launches[3]) device time of the depth-table, excitation and drag-solve kernels of the last call."""
    ms = (C.c_double * 3)()
    n = (C.c_int * 3)()
    check(lib.raftk_profile_read(ms, n))
    return list(ms), list(n)

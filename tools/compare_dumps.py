#!/usr/bin/env python3
"""Compare two bench.py --dump-outputs directories of the same workload (A = reference build, B = candidate).

Prints: status identical?, Xi bit-identical?, max |Xi_B - Xi_A| / max |Xi_A| per unit (worst unit), every other array's
largest relative difference, and B's parity block against the oracle when B's bench JSON line is given.

usage: tools/compare_dumps.py DIR_A DIR_B [B.json]"""
import json, os, sys
import numpy as np

a_dir, b_dir = sys.argv[1], sys.argv[2]
names = sorted(f[:-4] for f in os.listdir(a_dir) if f.endswith(".npy"))
load = lambda d, n: np.load(os.path.join(d, n + ".npy"))
st_same = np.array_equal(load(a_dir, "status"), load(b_dir, "status"))
xa = load(a_dir, "Xi_real") + 1j * load(a_dir, "Xi_imag")
xb = load(b_dir, "Xi_real") + 1j * load(b_dir, "Xi_imag")
bits = np.array_equal(load(a_dir, "Xi_real"), load(b_dir, "Xi_real")) and np.array_equal(load(a_dir, "Xi_imag"), load(b_dir, "Xi_imag"))
lead = xa.shape[:-3] if xa.ndim >= 3 else xa.shape[:1]
ua, ub = xa.reshape(int(np.prod(lead)), -1), xb.reshape(int(np.prod(lead)), -1)
err = float((np.abs(ub - ua).max(axis=1) / np.maximum(np.abs(ua).max(axis=1), 1e-300)).max())
others = []
for n in names:
    if n in ("status", "Xi_real", "Xi_imag", "sample_units"):
        continue
    p, q = load(a_dir, n), load(b_dir, n)
    others.append("%s %.2e" % (n, float(np.abs(q - p).max() / max(np.abs(p).max(), 1e-300))))
par = ""
if len(sys.argv) > 3:
    line = json.loads(open(sys.argv[3]).read().strip().splitlines()[-1])
    pb = line.get("parity") or {}
    par = " | B parity vs oracle: ok %s max_rel_err %.2e pass_mismatch_units %s" % (pb.get("ok"), pb.get("max_rel_err", float("nan")), pb.get("pass_mismatch_units"))
print("status identical %s | Xi bit-identical %s | Xi max rel diff per unit %.2e | %s%s" % (st_same, bits, err, ", ".join(others), par))

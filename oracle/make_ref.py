"""Recipe: put the UNMODIFIED reference where bench.py can time it on the GPU box.

    python oracle/make_ref.py        (needs the WISDEM/RAFT source tree: oracle/ref_harness.py REF_ROOT,
                                      i.e. $RAFT_REFERENCE_ROOT or the reference's documented location)

1. ``pip install --no-index --no-build-isolation --no-deps --target oracle/_ref`` of a scratch copy of the reference
   source tree (that tree may be read-only and setuptools writes build/ next to setup.py).  ``--no-deps``:
   moorpy / pyhams / ccblade / wisdem / openmdao / matplotlib are not needed; none of them is on the per-frequency hot
   path, and oracle/ref_harness.py stubs their import lines (SURVEY.md 8c).
2. copy the design INPUTS the baseline configurations read (YAML files and the WAMIT coefficient tables of
   configs[2]; data, not code) to oracle/_ref/inputs/.

oracle/_ref/ is git-ignored (never part of the history) and travels with the built tree like the built .so files.
Nothing under raft_b200/ reads it; only bench.py's CPU baseline legs do (oracle/ref_timing.py).  Outcome of the install
is recorded in DESIGN.md section 7.
"""
import os
import shutil
import subprocess
import sys
import tempfile

HERE = os.path.dirname(os.path.abspath(__file__))
if os.path.dirname(HERE) not in sys.path:
    sys.path.insert(0, os.path.dirname(HERE))
from oracle.ref_harness import REF_ROOT as REF  # noqa: E402  (the one setting of where the reference source lives)

DST = os.path.join(HERE, "_ref")
INPUTS = ["designs/OC3spar.yaml", "designs/VolturnUS-S.yaml", "designs/VolturnUS-S_farm.yaml",
          "examples/OC4semi-WAMIT_Coefs.yaml", "examples/OC4semi-WAMIT_Coefs/marin_semi.1", "examples/OC4semi-WAMIT_Coefs/marin_semi.3"]


def available():
    return os.path.isdir(os.path.join(REF, "raft"))


def installed():
    return os.path.isdir(os.path.join(DST, "raft")) and os.path.isdir(os.path.join(DST, "inputs"))


def main():
    if not available():
        print("reference tree %s not present: nothing to install" % REF)
        return 1
    if installed():
        print("oracle/_ref already installed")
        return 0
    with tempfile.TemporaryDirectory() as tmp:
        src = os.path.join(tmp, "reference")
        shutil.copytree(REF, src, ignore=shutil.ignore_patterns("docs", ".git", "examples"))
        subprocess.check_call(["chmod", "-R", "u+w", src])
        subprocess.check_call([sys.executable, "-m", "pip", "install", "-q", "--no-index", "--no-build-isolation", "--no-deps",
                               "--target", DST, "--upgrade", src])
    for rel in INPUTS:
        s = os.path.join(REF, rel)
        if os.path.exists(s):
            d = os.path.join(DST, "inputs", rel)
            os.makedirs(os.path.dirname(d), exist_ok=True)
            shutil.copyfile(s, d)
    print("installed the unmodified reference into", DST)
    return 0


if __name__ == "__main__":
    sys.exit(main())

#!/bin/bash
# A/B of two builds of libraftk.so (same ABI) on the flagship workload, runs alternating in one process tree.
#
# usage: tools/fused2_diet_ab.sh A B OUTDIR [ROUNDS]
#   A, B: a source tree (a directory holding raft_b200/csrc/raftk.cu, compiled here for sm_100a into OUTDIR) or a
#         prebuilt libraftk.so.  bench.py is always the one of the current tree; RAFTK_LIB selects the library.
#   OUTDIR: receives ab_cfg2.txt (one line per run), the raw JSON lines, the cfg3 runs, and the comparison of both
#           builds' --dump-outputs on cfg2 / cfg3 / sweep by tools/compare_dumps.py (the dumps are deleted afterwards).
set -e
A=$1; B=$2; OUT=$3; ROUNDS=${4:-5}
mkdir -p "$OUT"
NVCC=${NVCC:-/usr/local/cuda/bin/nvcc}
lib_of() {   # $1 = tree or .so, $2 = label
  if [ -d "$1" ]; then
    mkdir -p "$OUT/$2"
    "$NVCC" -gencode arch=compute_100a,code=sm_100a -O3 -lineinfo -std=c++17 -shared -Xcompiler -fPIC \
      -o "$OUT/$2/libraftk.so" "$1/raft_b200/csrc/raftk.cu" >&2
    echo "$(cd "$OUT/$2" && pwd)/libraftk.so"
  else
    echo "$(cd "$(dirname "$1")" && pwd)/$(basename "$1")"
  fi
}
LA=$(lib_of "$A" A); LB=$(lib_of "$B" B)
nvidia-smi --query-gpu=name,power.limit,clocks.sm,clocks.max.sm --format=csv | tee "$OUT/gpu.txt"
summ() {   # one line from a bench JSON line
  python -c "
import sys, json
d = json.loads(sys.stdin.read().strip().splitlines()[-1])
sw = d.get('extra', {}).get('sweep', d.get('sweep'))
sw = sw.get('value', sw) if isinstance(sw, dict) else sw
print('$1', 'value %.4e' % d['value'], 'ms_per_step %.4f' % d['ms_per_step'], 'sweep', sw, 'parity_ok', (d.get('parity') or {}).get('ok'))"
}
for r in $(seq 1 "$ROUNDS"); do
  for lab in A B; do
    lib=$LA; [ $lab = B ] && lib=$LB
    RAFTK_LIB=$lib python bench.py --steps 20 --warmup 3 2>/dev/null | tail -1 | tee -a "$OUT/cfg2_$lab.jsonl" | summ "cfg2 $lab run $r" | tee -a "$OUT/ab_cfg2.txt"
  done
done
for lab in A B; do
  lib=$LA; [ $lab = B ] && lib=$LB
  RAFTK_LIB=$lib python bench.py --workload cfg3 --steps 20 --warmup 3 --no-cpu-baseline 2>/dev/null | tail -1 | tee -a "$OUT/cfg3_$lab.jsonl" | summ "cfg3 $lab" | tee -a "$OUT/ab_cfg3.txt"
done
for wl in cfg2 cfg3 sweep; do
  for lab in A B; do
    lib=$LA; [ $lab = B ] && lib=$LB
    RAFTK_LIB=$lib python bench.py --workload $wl --steps 2 --warmup 1 --no-cpu-baseline --no-e2e --no-extras \
      --dump-outputs "$OUT/dump_${wl}_$lab" 2>/dev/null | tail -1 > "$OUT/dump_${wl}_$lab.json"
  done
  python tools/compare_dumps.py "$OUT/dump_${wl}_A" "$OUT/dump_${wl}_B" "$OUT/dump_${wl}_B.json" | sed "s/^/$wl: /" | tee -a "$OUT/compare.txt"
  rm -rf "$OUT/dump_${wl}_A" "$OUT/dump_${wl}_B"        # the arrays are large; the comparison above is the record
done

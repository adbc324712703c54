#!/usr/bin/env bash
# jf_aligner end to end on the bench's yeast-shape input (bench.py WORKLOAD: 12 Mbp genome, 50x of 10 kbp reads at
# 12 % error, seed 43), with the production flags plus -l -k --coords: wall time per read base and the
# MR_SHOW_TIMING stage busy times, for one or more builds alternated run by run, and whether their coords files
# are identical.  Then the device time of the coords printer's kernels (torch.profiler) and of the host formatter
# on one 32-Mbase batch of the same reads.
#
#   jf_aligner_rate.sh OUT_DIR [REPO_ROOT ...]     (default: this repository; each root holds pacbio_b200/bin)
# Environment: RUNS (2), CORES (all: run under taskset on cores 0..CORES-1), MR_BENCH_DIR (where bench.py keeps
# its inputs; they are generated there when missing).
set -euo pipefail
HERE="$(cd "$(dirname "$0")" && pwd)"
REPO="$(cd "$HERE/../.." && pwd)"
OUT="${1:?usage: jf_aligner_rate.sh OUT_DIR [REPO_ROOT ...]}"; shift
ROOTS=("$@"); [ ${#ROOTS[@]} -eq 0 ] && ROOTS=("$REPO")
RUNS="${RUNS:-2}"
mkdir -p "$OUT"

# the bench's inputs (bench.py data_files: same generator, arguments and directory)
DIR="${MR_BENCH_DIR:-${TMPDIR:-/tmp}/pacbio_b200_bench}/g12000000_c50_s43_r0_l10000"
PREFIX="$DIR/synth"
if [ ! -e "$PREFIX.done" ]; then
  mkdir -p "$DIR"
  GEN="$REPO/pacbio_b200/tools/gen_synth"
  [ -x "$GEN" ] || g++ -O2 -std=c++17 -pthread "$GEN.cc" -o "$GEN"
  NT=$(nproc); [ "$NT" -gt 32 ] && NT=32
  "$GEN" --genome 12000000 --coverage 50 --read-len 10000 --error 0.12 --seed 43 --sr-cov 3 --repeat-frac 0 \
         --unitig-k 41 --threads "$NT" --shards 1 --first-shard 0 --prefix "$PREFIX" > "$PREFIX.done.tmp"
  mv "$PREFIX.done.tmp" "$PREFIX.done"
fi
BASES=$(python3 -c "import json; print(json.load(open('$PREFIX.done')).get('read_bases', 0))" 2>/dev/null || echo 0)
[ "$BASES" -gt 0 ] 2>/dev/null || BASES=$(grep -v '^>' "$PREFIX.reads.fa" | tr -d '\n' | wc -c)
PIN=()
[ -n "${CORES:-}" ] && PIN=(taskset -c "0-$((CORES - 1))")
nvidia-smi --query-gpu=name,power.limit --format=csv,noheader 2>/dev/null | sed 's/^/gpu: /' || true
echo "cores: ${CORES:-$(nproc)}  read bases: $BASES"

for run in $(seq 1 "$RUNS"); do
  for i in "${!ROOTS[@]}"; do
    root="${ROOTS[$i]}"
    t0=$(date +%s.%N)
    MR_SHOW_TIMING=1 MR_INDEX_CACHE="$OUT/index$i.bin" "${PIN[@]}" "$root/pacbio_b200/bin/jf_aligner" -s 1M -m 15 --psa-min 13 -B 17 \
      -l "$PREFIX.unitigs_len.txt" -k 41 -r "$PREFIX.superreads.fa" -p "$PREFIX.reads.fa" --coords "$OUT/coords$i.txt" \
      2> "$OUT/stderr$i.txt"
    t1=$(date +%s.%N)
    python3 - "$t0" "$t1" "$BASES" "$run" "$root" "$OUT/stderr$i.txt" <<'EOF'
import sys
t0, t1, bases, run, root, err = float(sys.argv[1]), float(sys.argv[2]), int(sys.argv[3]), sys.argv[4], sys.argv[5], sys.argv[6]
stages = [l.strip() for l in open(err) if l.startswith("stage busy")]
print("run %s %s: %.2f s, %.3f ns/base (%.3f Gbases/s); %s" % (run, root, t1 - t0, 1e9 * (t1 - t0) / bases, bases / (t1 - t0) / 1e9,
                                                                stages[-1] if stages else "no stage line"))
EOF
  done
done
for i in "${!ROOTS[@]}"; do
  [ "$i" -eq 0 ] && continue
  if cmp -s "$OUT/coords0.txt" "$OUT/coords$i.txt"; then echo "coords of ${ROOTS[$i]}: identical to ${ROOTS[0]}"
  else echo "coords of ${ROOTS[$i]}: DIFFER from ${ROOTS[0]}"; fi
done
ls -l "$OUT"/coords*.txt | awk '{print "size", $5, $9}'

# device time of the printer's kernels and host time of the formatter, on the first batch (this repository's build)
python3 - "$PREFIX" "$REPO" <<'EOF'
import ctypes as C, os, sys, time
import numpy as np
prefix, repo = sys.argv[1], sys.argv[2]
sys.path.insert(0, repo); sys.path.insert(0, os.path.join(repo, "tests"))
import pacbio_b200 as pb
import torch
from torch.profiler import ProfilerActivity, profile
from test_gpu_coords_records import host_coords, host_lib
sr = pb.SuperReads(prefix + ".superreads.fa")
ulen = np.loadtxt(prefix + ".unitigs_len.txt", dtype=np.int64)[:, 1]
reads = pb.Reads(prefix + ".reads.fa")
n = int(np.searchsorted(reads.starts, 32 << 20))
reads = reads.slice(0, n)
ctx = pb.Context(0)
idx = ctx.index(sr, 13, 15, unitig_len=ulen)
srn = ctx.sr_names(sr.names, sr.unitig_ids, sr.unitig_off)
res = ctx.align(idx, reads, pb.default_params(unitigs_k=41, matching_bases=0.17, matching_mers=0.0), keep=True)
text = ctx.coords_records(res, reads.names, sr_names=srn)
reps = 10
with profile(activities=[ProfilerActivity.CUDA]) as prof:
    for _ in range(reps):
        ctx.coords_records(res, reads.names, sr_names=srn)
    torch.cuda.synchronize()
tot = {}
for e in prof.key_averages():
    if "coords_" in e.key or "scan_" in e.key:
        tot[e.key] = (getattr(e, "device_time_total", 0) or getattr(e, "cuda_time_total", 0)) / reps
for k, v in sorted(tot.items()):
    print("kernel %-70s %8.1f us per call" % (k[:70], v))
t0 = time.perf_counter()
for _ in range(3):
    ctx.coords_records(res, reads.names, sr_names=srn)
t1 = time.perf_counter()
H = host_lib()
read_len = np.diff(reads.starts.astype(np.int64))
t2 = time.perf_counter()
want = host_coords(H, res, sr.names, sr.unitig_ids, sr.unitig_off, reads.names, read_len, True, False)
t3 = time.perf_counter()
print("batch: %d reads, %d rows, %.1f MB of text; mr_coords_records %.2f ms per call (wall), host format_coords %.2f ms; "
      "identical: %s" % (reads.nreads, res.ncoords, len(text) / 1e6, (t1 - t0) / 3 * 1e3, (t3 - t2) * 1e3, want == text))
EOF

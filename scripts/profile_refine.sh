#!/bin/bash
# ncu --set full captures of the refinement-side kernels (PAMR, bilateral lattice, consistency loss), one launch each.
# usage: scripts/profile_refine.sh TAG OUTDIR   (the timings, the ncu report and its log go to OUTDIR)
set -u
TAG=${1:?usage: scripts/profile_refine.sh TAG OUTDIR}
OUT=${2:?usage: scripts/profile_refine.sh TAG OUTDIR}
mkdir -p "$OUT"
timeout 300 python scripts/bench_refine.py > "$OUT/bench_refine_${TAG}.json" || exit 1
timeout 900 ncu --set full --clock-control none --import-source on \
  -k regex:"pamr_iter_tma2_kernel|pamr_affinity_reg_kernel|lattice_|consistency_rows_kernel" --launch-skip 0 -c 40 -f -o "$OUT/prof_refine_${TAG}" \
  python scripts/_refine_once.py > "$OUT/ncu_refine_${TAG}.log" 2>&1
echo "refine capture rc=$?"

#!/bin/bash
# Generates tests/golden/ref_c1.* by running the UNMODIFIED reference program
# (oracle/_ref/gaussianMPI_ref: the reference sources compiled for sm_100a by
# `make -C oracle ref REF=<reference checkout>`, with the cutil.h / single-rank mpi.h shims) on a B200.
# Run from the repository root on a machine with a B200:   bash tests/golden/make_ref_golden.sh OUTDIR
# then copy OUTDIR/ref_c1* into tests/golden/ and commit.
#   ref_c1.*                          100 iterations (tests/test_oracle.py)
#   ref_c1_it20.summary, .stdout      20 iterations (tests/test_gpu_parity.py), and
#   ref_c1_it20.memberships.npy       the responsibilities of its first 2000 events, float64 [2000][8] as parsed from the "%f" text
set -euo pipefail
OUT=${1:?usage: make_ref_golden.sh OUTDIR}
ITERS=${GMM_REF_ITERS:-100}
mkdir -p "$OUT"
python - "$OUT" <<'PY'
import sys, os
sys.path.insert(0, os.getcwd())
import __graft_entry__ as e
pkg = e.load_package()
cfg = pkg.synth.CONFIGS["c1"]
ev = pkg.synth.make_blobs(cfg["N"], cfg["D"], cfg["K"])
pkg.synth.write_bin(os.path.join(sys.argv[1], "c1.bin"), ev)
PY
export OMP_NUM_THREADS=1 CUDA_VISIBLE_DEVICES=0
GMM_REF_ITERS=$ITERS ./oracle/_ref/gaussianMPI_ref 8 "$OUT/c1.bin" "$OUT/ref_c1" 8 > "$OUT/ref_c1.stdout" 2>&1
head -n 512 "$OUT/ref_c1.results" > "$OUT/ref_c1.results.head"
rm -f "$OUT/ref_c1.results"
printf "N=10000\nD=4\nK=8\nseed=20260921\niters=%s\n" "$ITERS" > "$OUT/ref_c1.meta"
GMM_REF_ITERS=20 ./oracle/_ref/gaussianMPI_ref 8 "$OUT/c1.bin" "$OUT/ref_c1_it20" 8 > "$OUT/ref_c1_it20.stdout" 2>&1
python - "$OUT/ref_c1_it20" <<'PY'
import sys
import numpy as np
rows = [l.rstrip("\n").split("\t") for l in open(sys.argv[1] + ".results")][:2000]
np.save(sys.argv[1] + ".memberships.npy", np.array([[float(v) for v in r[1].split(",")] for r in rows]))
PY
rm -f "$OUT/ref_c1_it20.results" "$OUT/c1.bin"
ls -la "$OUT"

#!/bin/bash
# Same-box A/B of the hoisted conditioner projection (GEMM1 over the three conv taps, W_cond . cond once per sampler call)
# against the parent commit's tree.
#   tools/ab_cond_hoist.sh prepare [REV]   in a git checkout, before the GPU run: REV's tree (default HEAD~1), built,
#                                          in build/ab_parent (git-ignored, so it travels with the working tree)
#   tools/ab_cond_hoist.sh run             on the B200: card and power limit, the new GPU tests (AB_TESTS: more test files),
#                                          alternating parent / new sampler benches (3 each) with their mel dumps
#                                          compared; everything goes to $AB_OUT/ab_cond_hoist.log
#   tools/ab_cond_hoist.sh full            one full bench.py of the new tree ($AB_OUT/ab_cond_hoist_full.log)
# AB_OUT: directory for the logs (default build/ab_out, git-ignored).
OUT=$(mkdir -p "${AB_OUT:-build/ab_out}" && cd "${AB_OUT:-build/ab_out}" && pwd)
case "$1" in
prepare)
  set -e
  rev=${2:-HEAD~1}
  rm -rf build/ab_parent
  mkdir -p build/ab_parent
  git archive "$rev" | tar -x -C build/ab_parent
  (cd build/ab_parent && python -c "import __graft_entry__ as g; g.build()")
  ;;
run)
  [ -f build/ab_parent/fish_diffusion_b200/libfishdiff_b200.so ] || { echo "run '$0 prepare' first"; exit 2; }
  MEL=$(mktemp -d)            # the mel dumps are 64 MB each: kept out of the output directory
  L=$OUT/ab_cond_hoist.log
  : > "$L"
  log() { echo "=== $1" >> "$L"; shift; "$@" >> "$L" 2>&1 || echo "(exit $?)" >> "$L"; }
  log "card" nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv
  log "gpu tests (new tree)" timeout 300 python -m pytest -m gpu -q -s -rf tests/test_gpu_cond_hoist.py ${AB_TESTS:-}
  # headline only (--no-extras --no-e2e): six runs of the 100-evaluation sampler fit one 10-minute call
  S="bench.py --no-vocoder --no-train --no-voc-train --no-cpu-baseline --no-extras --no-e2e --steps 3 --warmup 3"
  for rep in 1 2 3; do
    log "bench parent rep$rep" bash -c "cd build/ab_parent && timeout 300 python $S --dump-outputs $MEL/parent"
    log "bench new rep$rep" timeout 300 python $S --dump-outputs "$MEL/new"
  done
  log "mel new vs parent" python -c "
import numpy as np
a, b = np.load('$MEL/new/mel.npy').astype(np.float64), np.load('$MEL/parent/mel.npy').astype(np.float64)
print(f'shape {a.shape}  rel-L2 {np.linalg.norm(a - b) / np.linalg.norm(b):.3e}  max-abs {np.abs(a - b).max():.3e}')"
  rm -rf "$MEL"
  log "card after the A/B" nvidia-smi --query-gpu=name,power.limit,clocks.sm,clocks.max.sm --format=csv
  grep -E "passed|failed|rel-L2|^\{" "$L" | cut -c1-400 | tail -30
  ;;
full)
  nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv > "$OUT/ab_cond_hoist_full.log" 2>&1
  timeout 1800 python bench.py --gpus 1 >> "$OUT/ab_cond_hoist_full.log" 2>&1
  tail -1 "$OUT/ab_cond_hoist_full.log" | cut -c1-400
  ;;
*)
  echo "usage: $0 prepare [REV] | run | full"; exit 2 ;;
esac

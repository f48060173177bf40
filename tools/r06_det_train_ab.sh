#!/bin/bash
# Deterministic training mode: the GPU suite (the new tests with their printed bounds and atomic-path evidence),
# smoke(), then the training benchmarks with XMM_DETERMINISTIC = 0 / 1 alternated (three runs each, DN and SR-2x at the
# bench's shapes), and the default headline with --dump-outputs.  With a second tree of the previous commit (PARENT,
# built), the headline and the DN training dumps of both trees are compared element by element.
# Usage: tools/r06_det_train_ab.sh OUTDIR [PARENT]  (logs OUTDIR/r06_*)
set -o pipefail
O=${1:?usage: tools/r06_det_train_ab.sh OUTDIR [PARENT]}
P=${2:-}
mkdir -p "$O"
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv | tee $O/r06_card.txt
python -c "import __graft_entry__ as g; g.build()" > $O/r06_build.log 2>&1 || { tail -30 $O/r06_build.log; exit 1; }
timeout 600 python -m pytest tests/test_gpu_deterministic.py -q -s -m gpu 2>&1 | tail -60 > $O/r06_pytest_det.log
tail -3 $O/r06_pytest_det.log
timeout 1800 python -m pytest tests -q -m gpu 2>&1 | tail -25 > $O/r06_pytest_gpu.log
tail -3 $O/r06_pytest_gpu.log
timeout 300 python -c "import __graft_entry__ as g; g.smoke()" > $O/r06_smoke.log 2>&1; echo "smoke rc=$?" | tee -a $O/r06_smoke.log
for wl in train_dn train_sr; do
  for i in 1 2 3; do
    for d in 0 1; do
      XMM_DETERMINISTIC=$d timeout 600 python bench.py --gpus 1 --workload $wl --steps 30 --warmup 5 --no-cpu-baseline \
        --no-parity 2>$O/r06_bench_${wl}_det${d}_$i.err | tail -1 > $O/r06_bench_${wl}_det${d}_$i.json
      echo "$wl det=$d run $i: $(head -c 260 $O/r06_bench_${wl}_det${d}_$i.json)"
    done
  done
done | tee $O/r06_bench_det_ab.log
D=$(mktemp -d)
timeout 900 python bench.py --gpus 1 --dump-outputs $D/new 2>$O/r06_bench_headline.err | tail -1 > $O/r06_bench_headline.json
head -c 400 $O/r06_bench_headline.json; echo
timeout 900 python bench.py --gpus 1 --workload train_dn --steps 5 --warmup 2 --no-cpu-baseline --no-parity \
  --dump-outputs $D/new_train 2>/dev/null | tail -1 > /dev/null
if [ -n "$P" ]; then
  (cd "$P" && timeout 900 python bench.py --gpus 1 --dump-outputs $D/old 2>/dev/null | tail -1 > $O/r06_bench_headline_parent.json
   timeout 900 python bench.py --gpus 1 --workload train_dn --steps 5 --warmup 2 --no-cpu-baseline --no-parity \
     --dump-outputs $D/old_train 2>/dev/null | tail -1 > /dev/null)
  head -c 400 $O/r06_bench_headline_parent.json; echo
  python - "$D" <<'PY' 2>&1 | tee $O/r06_bench_outputs_vs_parent.log
import os, sys
import numpy as np
d = sys.argv[1]
for new, old in (("new", "old"), ("new_train", "old_train")):
    a, b = os.path.join(d, new), os.path.join(d, old)
    for f in sorted(os.listdir(a)):
        x, y = np.load(os.path.join(a, f)), np.load(os.path.join(b, f))
        same = np.array_equal(x, y)
        rel = float(np.linalg.norm((x - y).ravel()) / max(np.linalg.norm(y.ravel()), 1e-30))
        print(new, f, x.shape, "array_equal" if same else f"DIFFERENT (rel-L2 {rel:.2e})")
PY
fi
rm -rf "$D"

#!/bin/bash
# Gradient clipping: the new GPU tests (printed figures with -s), the rest of the GPU suite, smoke, the
# clipping probe (tools/clip_probe.py), then the default benchmark A/B against a built tree of the previous commit
# (PARENT, optional), alternated, two runs each, outputs compared with --dump-outputs.
# Usage: tools/r09_clip_ab.sh OUTDIR [PARENT] [quick]  (logs OUTDIR/r09_*; quick: new tests, smoke and probe only)
set -o pipefail
O=${1:?usage: tools/r09_clip_ab.sh OUTDIR [PARENT] [quick]}
P=${2:-}
Q=${3:-}
mkdir -p "$O"
O=$(cd "$O" && pwd)
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv | tee $O/r09_card.txt
python -c "import __graft_entry__ as g; g.build()" > $O/r09_build.log 2>&1 || { tail -30 $O/r09_build.log; exit 1; }
if [ -n "$P" ]; then
  (cd $P && python -c "import __graft_entry__ as g; g.build()" > $O/r09_build_parent.log 2>&1) || { tail -30 $O/r09_build_parent.log; exit 1; }
fi
timeout 900 python -m pytest tests/test_gpu_grad_clip.py -q -s -m gpu 2>&1 | tail -150 > $O/r09_pytest_clip.log
tail -25 $O/r09_pytest_clip.log
timeout 300 python -c "import __graft_entry__ as g; g.smoke()" > $O/r09_smoke.log 2>&1; echo "smoke rc=$?" | tee -a $O/r09_smoke.log
timeout 900 python tools/clip_probe.py --out $O/r09_clip_probe.log 2>&1 | tail -8
[ "$Q" = quick ] && exit 0
timeout 2400 python -m pytest tests -q -m gpu --deselect tests/test_gpu_grad_clip.py 2>&1 | tail -25 > $O/r09_pytest_gpu.log
tail -5 $O/r09_pytest_gpu.log
[ -n "$P" ] || exit 0
D=$(mktemp -d)
for i in 1 2; do
  for arm in new parent; do
    dir=.; [ $arm = parent ] && dir=$P
    (cd $dir && timeout 900 python bench.py --gpus 1 --steps 10 --warmup 3 --dump-outputs $D/${arm}_$i \
      2>$O/r09_bench_${arm}_$i.err | tail -1 > $O/r09_bench_${arm}_$i.json)
    python - $O/r09_bench_${arm}_$i.json $arm $i <<'PY'
import json, sys
d = json.load(open(sys.argv[1]))
ex = d.get("extra", {})
tr = {k: round(v.get("value", 0), 1) for k, v in ex.items() if k.startswith("train_")}
print(sys.argv[2], sys.argv[3], d.get("metric"), round(d.get("value", 0), 1), tr)
PY
  done
done | tee $O/r09_bench_ab.log
python - "$D" <<'PY' 2>&1 | tee $O/r09_bench_outputs_vs_parent.log
import os, sys
import numpy as np
d = sys.argv[1]
for i in (1, 2):
    a, b = os.path.join(d, f"new_{i}"), os.path.join(d, f"parent_{i}")
    for f in sorted(os.listdir(a)):
        x, y = np.load(os.path.join(a, f)), np.load(os.path.join(b, f))
        print(i, f, x.shape, "array_equal" if np.array_equal(x, y) else "DIFFERENT")
PY
rm -rf "$D"

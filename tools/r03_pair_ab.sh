#!/bin/bash
# CTA pairs for conv4 + conv5 of the fused dense block (XMM_RDB_PAIR = 0: single CTAs, 2: conv4 + conv5 as pairs): the
# GPU suite, smoke(), the dense-block probe and the headline bench, the two arms alternated on one box; then the stall
# counters of an XMM_RDB_PROFILE build.  Usage: tools/r03_pair_ab.sh OUTDIR (logs OUTDIR/r03_*).  The last step rebuilds libxmm_b200.so with the
# counters compiled in: rebuild it (__graft_entry__.build(force=True)) before using the tree again.
set -o pipefail
O=${1:?usage: tools/r03_pair_ab.sh OUTDIR}
mkdir -p "$O"
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv | tee $O/r03_card.txt
python -c "import __graft_entry__ as g; g.build()" > $O/r03_build.log 2>&1 || { tail -30 $O/r03_build.log; exit 1; }
timeout 1500 python -m pytest tests -q -m gpu 2>&1 | tail -25 > $O/r03_pytest_gpu.log
tail -3 $O/r03_pytest_gpu.log
timeout 300 python -c "import __graft_entry__ as g; g.smoke()" > $O/r03_smoke.log 2>&1; echo "smoke rc=$?" | tee -a $O/r03_smoke.log
{
  for b in 64 16 1; do
    for i in 1 2 3; do
      for p in 0 2; do echo -n "pair=$p "; XMM_RDB_PAIR=$p timeout 120 python tools/rdb_probe.py 259 $b 10; done
    done
  done
} 2>&1 | tee $O/r03_rdb_probe_pair_ab.log
D=$(mktemp -d)
for i in 1 2 3; do
  for p in 0 2; do
    XMM_RDB_PAIR=$p timeout 900 python bench.py --gpus 1 --steps 20 --dump-outputs $D/p${p}_$i 2>$O/r03_bench_p${p}_$i.err \
      | tail -1 > $O/r03_bench_pair${p}_$i.json
    echo "pair=$p run $i: $(head -c 300 $O/r03_bench_pair${p}_$i.json)"
  done
done | tee $O/r03_bench_pair_ab.log
python - "$D" <<'PY' 2>&1 | tee $O/r03_bench_outputs_equal.log
import glob, os, sys
import numpy as np
d = sys.argv[1]
a, b = os.path.join(d, "p0_1"), os.path.join(d, "p2_1")
for f in sorted(os.listdir(a)):
    x, y = np.load(os.path.join(a, f)), np.load(os.path.join(b, f))
    print(f, x.shape, "array_equal" if np.array_equal(x, y) else "DIFFERENT")
PY
rm -rf "$D"
/usr/local/cuda/bin/nvcc -gencode arch=compute_100a,code=sm_100a -lineinfo -O3 -std=c++17 -Xcompiler -fPIC -shared \
  -DXMM_RDB_PROFILE=1 -o xmm_superres_denoise_b200/libxmm_b200.so xmm_superres_denoise_b200/csrc/xmm_b200.cu || exit 1
for p in 0 2; do
  echo "XMM_RDB_PAIR=$p"
  XMM_RDB_PAIR=$p XMM_RDB_PROF=1 timeout 120 python tools/rdb_probe.py 259 64 2 2>&1 | grep "conv3x3_rdb<" | tail -2
done 2>&1 | tee $O/r03_rdb_phase_counters.log

#!/bin/bash
# variants built beforehand: lib_base.so from the parent commit, then `python tools/ab.py build new: newall:LR_DIV_ZD_ALL`
# (new: zero guard in orthonormal_basis only; newall: in every vector quotient, the form that shipped and whose knob is gone)
set -u
O=${1:?usage: bash tools/runs/gpu_r03_a.sh OUTDIR}; mkdir -p "$O"
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm,driver_version --format=csv > $O/card.txt 2>&1
cat $O/card.txt
echo "== div_probe"; python tools/div_probe.py 2>&1 | tee $O/div_probe.txt
echo "== ab"; python tools/ab.py run base new newall --rounds 3 2>&1 | tee $O/ab.txt
for v in base new; do
  echo "== bench $v"
  LUMILLY_LIB=$PWD/lumillyrender_b200/variants/lib_$v.so python bench.py --gpus 1 --steps 5 --warmup 2 --no-cpu-baseline --dump-outputs $O/dump_$v > $O/bench_$v.json 2> $O/bench_$v.err; echo rc=$?
  tail -c 600 $O/bench_$v.json
done
python - "$O" <<'PY' 2>&1 | tee $O/compare.txt
import json, os, sys, numpy as np
O = sys.argv[1]
a = np.load(os.path.join(O, "dump_base/image.npy")); b = np.load(os.path.join(O, "dump_new/image.npy"))
print("image bit-identical:", a.shape == b.shape and np.array_equal(a.view(np.uint32), b.view(np.uint32)))
ja = json.loads(open(os.path.join(O, "bench_base.json")).read().strip().splitlines()[-1]); jb = json.loads(open(os.path.join(O, "bench_new.json")).read().strip().splitlines()[-1])
for k in ("value", "image_mean", "rays_per_sample"):
    print(k, ja.get(k), jb.get(k), ja.get(k) == jb.get(k))
PY
echo "== smoke + suite (default build = new)"
python -c "import __graft_entry__ as g; g.build(); g.smoke()" 2>&1 | tail -5 | tee $O/smoke.txt
python -m pytest tests -q -x -p no:cacheprovider 2>&1 | tail -15 | tee $O/pytest.txt

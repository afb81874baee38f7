#!/bin/bash
# the shipped form (every vector quotient through div_zero_dividend, x / pi and the checker's fmod without a division)
# against the parent build (lib_base.so built from the parent commit, lib_final.so by `python tools/ab.py build final:`):
# interleaved sweep, bench with dumped images, smoke and the whole suite on the default build
set -u
O=${1:?usage: bash tools/runs/gpu_r03_b.sh OUTDIR}; mkdir -p "$O"
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm,driver_version --format=csv > $O/card.txt 2>&1
echo "== ab"; python tools/ab.py run base final --rounds 3 2>&1 | tee $O/ab.txt
for v in base final base final; do
  echo "== bench $v"
  LUMILLY_LIB=$PWD/lumillyrender_b200/variants/lib_$v.so python bench.py --gpus 1 --steps 5 --warmup 2 --no-cpu-baseline --dump-outputs $O/dump_$v >> $O/bench_$v.json 2> $O/bench_$v.err; echo rc=$?
done
python - "$O" <<'PY' 2>&1 | tee $O/compare.txt
import json, os, sys, numpy as np
O = sys.argv[1]
a = np.load(os.path.join(O, "dump_base/image.npy")); b = np.load(os.path.join(O, "dump_final/image.npy"))
print("image bit-identical:", a.shape == b.shape and np.array_equal(a.view(np.uint32), b.view(np.uint32)))
ja = [json.loads(l) for l in open(os.path.join(O, "bench_base.json")) if l.startswith("{")]
jb = [json.loads(l) for l in open(os.path.join(O, "bench_final.json")) if l.startswith("{")]
for k in ("image_mean", "rays_per_sample"):
    print(k, [j.get(k) for j in ja], [j.get(k) for j in jb])
print("value base", [round(j["value"], 1) for j in ja], "final", [round(j["value"], 1) for j in jb])
for i, c in enumerate(ja[0].get("configs", [])):
    print(c.get("name") or c.get("config"), "base", [round(j["configs"][i]["msamples_per_s"], 1) for j in ja], "final", [round(j["configs"][i]["msamples_per_s"], 1) for j in jb])
PY
echo "== smoke + suite (default build)"
python -c "import __graft_entry__ as g; g.build(); g.smoke()" 2>&1 | tail -5 | tee $O/smoke.txt
python -m pytest tests -q -p no:cacheprovider 2>&1 | tail -15 | tee $O/pytest.txt

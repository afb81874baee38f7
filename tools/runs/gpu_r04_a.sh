#!/bin/bash
# pixel-sharded films on several GPUs (lr_multi_film_*) against the parent commit, whose tree (its own Python package and
# library: the new bindings need symbols the parent library lacks) is unpacked and built beforehand under .ab_parent/
# (`git archive <parent> | tar -x -C .ab_parent` + its build.py).  Interleaved sweep, bench with dumped images (the existing
# single-GPU path must keep its bits and its speed), the multi-film probe on every device count the box has, smoke and the
# whole suite of this tree
set -u
O=$(realpath -m "${1:?usage: bash tools/runs/gpu_r04_a.sh OUTDIR}"); mkdir -p "$O"
nvidia-smi --query-gpu=index,name,power.limit,clocks.max.sm,driver_version --format=csv > $O/card.txt 2>&1
cat $O/card.txt
echo "== ab"
for r in 1 2 3; do
  (cd .ab_parent && python tools/sweep.py base) 2>&1 | tee -a $O/ab.txt
  python tools/sweep.py final 2>&1 | tee -a $O/ab.txt
done
for v in base final base final; do
  echo "== bench $v"
  if [ $v = base ]; then D=.ab_parent; else D=.; fi
  (cd $D && python bench.py --gpus 1 --steps 5 --warmup 2 --no-cpu-baseline --dump-outputs $O/dump_$v >> $O/bench_$v.json 2> $O/bench_$v.err); echo rc=$?
done
python - "$O" <<'PY' 2>&1 | tee $O/bench_compare.txt
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
echo "== multi film probe"; python tools/multi_film_probe.py 2>&1 | tee $O/multi_film_probe.txt
echo "== smoke + suite"
python -c "import __graft_entry__ as g; g.build(); g.smoke()" 2>&1 | tail -5 | tee $O/smoke.txt
python -m pytest tests -q -p no:cacheprovider -rs 2>&1 | tail -25 | tee $O/pytest.txt

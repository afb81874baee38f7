#!/bin/bash
# adaptive sampling on films (lr_film_render_adaptive) against the parent commit, whose tree is unpacked and built beforehand
# under build/ab_parent/ (`git archive <parent> | tar -x -C build/ab_parent` + its build.py): interleaved bench with dumped
# images (image, image_mean and rays_per_sample must not move, Msamples/s within the noise), the adaptive probe on full-size
# films, smoke and the whole suite of this tree
set -u
O=$(realpath -m "${1:?usage: bash tools/runs/gpu_r07_a.sh OUTDIR}"); mkdir -p "$O"
nvidia-smi --query-gpu=index,name,power.limit,clocks.max.sm,driver_version --format=csv > $O/card.txt 2>&1
cat $O/card.txt
mkdir -p models && ln -sfn "$PWD/models" build/ab_parent/models     # one copy of the generated assets for both trees
for v in base final base final; do
  echo "== bench $v"
  if [ $v = base ]; then D=build/ab_parent; else D=.; fi
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
rm -rf $O/dump_base $O/dump_final
echo "== adaptive probe"; python tools/adaptive_probe.py 2> $O/adaptive_probe.err | tee $O/adaptive_probe.txt
echo "== smoke + suite"
python -c "import __graft_entry__ as g; g.build(); g.smoke()" 2>&1 | tail -5 | tee $O/smoke.txt
python -m pytest tests -v -p no:cacheprovider -rs > $O/pytest_full.txt 2>&1
grep -E "test_adaptive_film|test_multi_film" $O/pytest_full.txt | tee $O/pytest.txt
tail -12 $O/pytest_full.txt | tee -a $O/pytest.txt

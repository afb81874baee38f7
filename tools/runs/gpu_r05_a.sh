#!/bin/bash
# one film behind both film handles, one device discipline in api.cpp: against the parent commit, whose tree is unpacked and
# built beforehand under build/ab_parent/ (`git archive <parent> | tar -x -C build/ab_parent` + its build.py).  Interleaved bench
# with dumped images (image, image_mean and rays_per_sample must not move, nor the rate), the multi-film probe on both
# trees (render rate, gather + save time, image bits), smoke and the whole suite of this tree
set -u
O=$(realpath -m "${1:?usage: bash tools/runs/gpu_r05_a.sh OUTDIR}"); mkdir -p "$O"
nvidia-smi --query-gpu=index,name,power.limit,clocks.max.sm,driver_version --format=csv > $O/card.txt 2>&1
cat $O/card.txt
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
for v in base final; do
  echo "== multi film probe $v"
  if [ $v = base ]; then D=build/ab_parent; else D=.; fi
  (cd $D && python tools/multi_film_probe.py) 2>&1 | tee $O/multi_film_probe_$v.txt
  # the images of both handles on the probe's workload (64 spp in chunks of 16, a checkpoint resumed half way), to compare
  (cd $D && python - "$O/films_$v.npz" <<'PY'
import os, sys, tempfile, numpy as np
sys.path.insert(0, os.getcwd())
import lumillyrender_b200 as lr
lr.init(0)
lr.ensure_assets(os.getcwd(), bunny_tris=144046, need_ibl=False)
d = lr.Description(os.path.join("scenes", "sample.toml"), asset_root=os.getcwd(), resolution=(1920, 1370))
s, ms = d.scene(), d.multi_scene([0])
out = {}
for name, owner in (("film", s), ("multi_film", ms)):
    ck = os.path.join(tempfile.mkdtemp(), "film.ck")
    f = owner.film(sumsq=True, seed=0, splits=1)
    f.render(16); f.render(16); f.save(ck); f.close()
    f = owner.load_film(ck)
    f.render(16); f.render(16)
    out[name], out[name + "_sq"] = f.read(sumsq=True)
    f.save(ck); f.close()
    out[name + "_ck"] = np.frombuffer(open(ck, "rb").read(), dtype=np.uint8)
np.savez(sys.argv[1], **out)
PY
  ) 2>&1 | tail -3
done
python - "$O" <<'PY' 2>&1 | tee $O/films_compare.txt
import os, sys, numpy as np
O = sys.argv[1]
a, b = np.load(os.path.join(O, "films_base.npz")), np.load(os.path.join(O, "films_final.npz"))
for k in sorted(a.files):
    print(k, "bit-identical base / final:", a[k].shape == b[k].shape and np.array_equal(a[k].view(np.uint8), b[k].view(np.uint8)))
print("film == multi_film (final):", all(np.array_equal(b["film" + s].view(np.uint8), b["multi_film" + s].view(np.uint8)) for s in ("", "_sq", "_ck")))
PY
echo "== smoke + suite"
python -c "import __graft_entry__ as g; g.build(); g.smoke()" 2>&1 | tail -5 | tee $O/smoke.txt
python -m pytest tests -q -p no:cacheprovider -rs 2>&1 | tail -25 | tee $O/pytest.txt

#!/bin/bash
# bench line + per-kernel table + autotuner choices (stderr) into OUTDIR; optional env passed through
tag=${1:-cur}
out=${2:?usage: run_bench.sh TAG OUTDIR}
mkdir -p "$out"
A3D_AUTOTUNE_VERBOSE=1 timeout 400 python bench.py --steps 200 --warmup 3 --no-cpu-baseline --ops-json "$out/bench_ops_$tag.json" > "$out/bench_$tag.json" 2> "$out/bench_$tag.err"; echo "bench $tag rc=$?"
python - "$tag" "$out" <<'PY'
import json,sys
tag,out=sys.argv[1:3]
d=json.loads(open(f"{out}/bench_{tag}.json").read().strip().splitlines()[-1])
print(tag, "ms/step", round(d["ms_per_step"],4), "img/s", round(d["value"]), "e2e", round(d["e2e"]["value"]), "conv TF", round(d["roofline"]["conv_tensor_tflops"],1), "frac", round(d["roofline"]["conv_tensor_frac_of_burst"],3))
ops=json.load(open(f"{out}/bench_ops_{tag}.json"))["ops"]
for o in ops:
    if o["op"].startswith(("a3d_conv2d","a3d_dense")): print(f'{o["op"]:28s} {o["detail"]:40s} {o["ms"]*1e3:7.1f} us')
PY
grep -- "-> candidate" "$out/bench_$tag.err"

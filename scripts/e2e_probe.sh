#!/bin/bash
# e2e pipeline experiments on a reduced workload (400k reads vs 300 Mbp): per-part kernel times (MM_TRACE) under
# different host thread counts, wait modes and host-library switches.
W="--config 2 --reads 400000 --ref-bp 300000000 --contigs 32 --sketch 220 --no-cpu-baseline --steps 2 --warmup 2"
run() { # name, env...
  local name=$1; shift
  env MM_TRACE=1 "$@" python bench.py $W > gpurun_out/e2e_$name.json 2> gpurun_out/e2e_$name.log
  python - "$name" <<'PY'
import json, re, sys
name = sys.argv[1]
j = json.load(open(f"gpurun_out/e2e_{name}.json"))
k = j["kernel_ms_per_step"]
tr = [l for l in open(f"gpurun_out/e2e_{name}.log") if l.startswith("[trace] lane") and "segs 134218" in l][-10:]
pat = re.compile(r"h2d ([\d.]+)\).*k1 ([\d.]+) k2 ([\d.]+) k3 ([\d.]+): prep ([\d.]+) scan ([\d.]+)")
rows = [tuple(map(float, pat.search(l).groups())) for l in tr if pat.search(l)]
avg = [sum(c) / len(c) for c in zip(*rows)] if rows else []
print(name, "value ms", round(j["ms_per_step"], 1), "kernels", {a: round(b, 1) for a, b in k.items()}, "e2e ms", round(j["e2e"]["ms_per_step"], 1),
      "per-part [h2d k1 k2 k3 prep scan]", [round(x, 2) for x in avg], flush=True)
PY
}
for v in "$@"; do
  case $v in
    base) run base ;;
    few8) run few8 BENCH_HOST_THREADS=8 ;;
    few8block) run few8block BENCH_HOST_THREADS=8 MM_BLOCKING_WAIT=1 ;;
    few2) run few2 BENCH_HOST_THREADS=2 ;;
    few2spin) run few2spin BENCH_HOST_THREADS=2 MM_BLOCKING_WAIT=0 ;;
    few4) run few4 BENCH_HOST_THREADS=4 ;;
    noramp) run noramp MM_NO_RAMP=1 ;;
    serial) run serial MM_LANES=1 ;;
    tail1) run tail1 MM_TAIL_THREADS=1 ;;
    tail6) run tail6 MM_TAIL_THREADS=6 ;;
    nogate) run nogate MM_NO_GATE=1 ;;
    block) run block MM_BLOCKING_WAIT=1 ;;
  esac
done

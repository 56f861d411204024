#!/bin/bash
# Round-3 A/B on one box (profiles/r03_ab.md): the in-tree library (step() with the recomputed-midpoint kernel pair)
# against the parent build in scratch/libR02.so, interleaved twice: bench defaults (value, sustained, alt_arith), two
# small sizes, and the strong-scaling line (nx = 8192, which keeps the stored-midpoint kernels).
# Results go to $OUT (default ab_out/).
OUT=${OUT:-ab_out}
mkdir -p "$OUT"
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv
one() { # tag lib bench-args...
  local tag=$1 lib=$2; shift 2
  PIC1DP_B200_LIB=$lib python bench.py "$@" > $OUT/r03_$tag.json 2> $OUT/r03_$tag.err
  python - <<PY
import json
try:
    d = json.loads(open("$OUT/r03_$tag.json").read().strip().splitlines()[-1])
    s, a, rd = d.get("sustained") or {}, d.get("alt_arith") or {}, d["roofline_detail"]
    print("$tag", "value %.4e step %.4f irk1 %.4f irk2 %.4f" % (d["value"], d["ms_per_step"], rd["irk1"]["ms_per_launch"],
          d["roofline"]["ms_per_launch"]),
          "sustained %.4e (%.4f ms)" % (s["value"], s["ms_per_step"]) if s else "",
          "alt_arith %.4e (%.4f ms)" % (a["value"], a["ms_per_step"]) if a else "",
          "sm_mhz", d["clocks"].get("sm_mhz"), d["clocks"].get("reasons"), "dep", d["deposit_mode"])
except Exception as e:
    print("$tag", "ERR", e, open("$OUT/r03_$tag.err").read()[-600:])
PY
}
for rep in 1 2; do
  for L in tree R02; do
    lib=""
    [ $L = R02 ] && lib=$PWD/scratch/libR02.so
    one default_${L}_$rep "$lib"
    one c0_${L}_$rep "$lib" --steps 200 --markers 6.4e6 --nx 192 --no-cpu-baseline --no-e2e
    one c1_${L}_$rep "$lib" --steps 200 --markers 1e7 --nx 256 --no-cpu-baseline --no-e2e
    one strong_${L}_$rep "$lib" --scaling strong --no-alt-arith --no-cpu-baseline --no-e2e
  done
done

#!/bin/bash
# the bench lines of the committed state on one box: the reference arm, the default line and the --in-flight 1 line
mkdir -p gpurun_out
timeout -s KILL 900 python bench.py --impl reference --steps 3 --warmup 1 > gpurun_out/final_bench_reference.json 2> gpurun_out/final_bench_reference.err
timeout -s KILL 1200 python bench.py > gpurun_out/final_bench.json 2> gpurun_out/final_bench.err
timeout -s KILL 600 python bench.py --in-flight 1 --no-cpu-baseline --no-extras > gpurun_out/final_bench_if1.json 2> gpurun_out/final_bench_if1.err
python - <<P
import json
for f in ("final_bench","final_bench_if1"):
    d=json.loads([l for l in open("gpurun_out/%s.json"%f) if l.startswith("{")][-1])
    print(f, d["value"], d["ms_per_step"], d["e2e"]["value"], d["e2e"]["ms_per_step"], d.get("parity_checked"))
    r=d["roofline"]; print(" ", r["kernel"], r["frac"], r.get("alone"), r.get("step"))
P

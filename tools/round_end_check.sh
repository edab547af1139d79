#!/bin/bash
# Round-end validation on a B200: full GPU suite, smoke, the bench line, launch list.
# usage: bash tools/round_end_check.sh <tag>
tag=${1:-r01k}
mkdir -p gpurun_out
python -m pytest tests -m gpu -q > gpurun_out/${tag}_gputests.log 2>&1; echo "tests rc=$?"; tail -4 gpurun_out/${tag}_gputests.log
python -c "import __graft_entry__ as g; g.smoke()" > gpurun_out/${tag}_smoke.log 2>&1; echo "smoke rc=$?"; tail -1 gpurun_out/${tag}_smoke.log
python bench.py > gpurun_out/${tag}_bench_line.json 2> gpurun_out/${tag}_bench.err; echo "bench rc=$?"
python - <<P
import json
for f in ("${tag}_bench_line",):
    try:
        d=json.load(open("gpurun_out/%s.json"%f))
        print(f, round(d["value"],2), round(d["ms_per_step"],1), round(d["e2e"]["value"],2), {k:round(v,1) for k,v in d["per_layer_ms"].items()}, {k:round(v["ms_per_step"],1) for k,v in d["kernel_ms"].items() if "tcn" in k})
    except Exception as e: print(f,"ERR",e)
P
timeout 100 ncu --metrics gpu__time_duration.sum --clock-control none --profile-from-start off --csv --log-file gpurun_out/${tag}_launches.csv python tools/prof_step.py --batch 8 > gpurun_out/${tag}_launches.log 2>&1; echo "ncu rc=$?"

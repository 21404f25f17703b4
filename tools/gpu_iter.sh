#!/bin/bash
# One development iteration on a B200: selected GPU tests ($1 = pytest -k expression), then one default bench.py run.
mkdir -p gpurun_out
timeout 1200 python -m pytest tests -m gpu -q -x -k "${1:-top_view or render}" > gpurun_out/pytest_iter.log 2>&1; echo "pytest rc=$?"; tail -15 gpurun_out/pytest_iter.log
# the bench's JSON line (stdout) and the MWB_DEBUG occupancy line (stderr); anything else is printed only if no result came
MWB_DEBUG=1 timeout 600 python bench.py --steps 100 --warmup 10 --no-cpu 2>&1 | python -c '
import json, sys
lines = sys.stdin.read().splitlines()
res = [l for l in lines if l.startswith("{")]
print("\n".join(l for l in lines if "[mwb]" in l)[:400])
if res:
    d = json.loads(res[-1])
    print("value=%.0f k2_ms=%.3f k1_ms=%.3f" % (d["value"], d["roofline"]["kernel_avg_ms"], d["roofline"]["k1_avg_ms"]))
else:
    print("bench failed:", "\n".join(lines[-20:]))
'

#!/bin/bash
# round 3, GPU session B: compressible witness slots -- probe again (cheap full-entropy case), GPU suite, smoke(), memcheck over
# smoke(), the write-shape sweep on compressible slots, and bench.py against the plain-slot arm in alternated pairs.
TAG=${1:-r03b}; OUT=${2:?usage: $0 TAG OUTPUT_DIR}; mkdir -p $OUT
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm,driver_version --format=csv | tee $OUT/${TAG}_gpu.txt
echo "== probe"; timeout 300 tools/probes/compress_probe > $OUT/${TAG}_compress_probe.log 2>&1; grep -E "compressible/plain|probe" $OUT/${TAG}_compress_probe.log
echo "== pytest -m gpu"; timeout 2400 python -m pytest tests -m gpu -q 2>&1 | tail -15 | tee $OUT/${TAG}_pytest_gpu.log
echo "== smoke"; timeout 300 python __graft_entry__.py smoke 2>&1 | tail -2 | tee $OUT/${TAG}_smoke.log
echo "== memcheck smoke"; if command -v compute-sanitizer > /dev/null; then
    timeout 400 compute-sanitizer --tool memcheck --print-limit 5 python __graft_entry__.py smoke > $OUT/${TAG}_memcheck_smoke.log 2>&1; echo "rc=$?" >> $OUT/${TAG}_memcheck_smoke.log
    grep -E "ERROR SUMMARY|smoke ok|rc=|Invalid|misaligned" $OUT/${TAG}_memcheck_smoke.log | head -8
else echo "compute-sanitizer not on PATH" | tee $OUT/${TAG}_memcheck_smoke.log; fi
echo "== sweep"; timeout 900 python tools/compressed_expand_sweep.py 2>&1 | tee $OUT/${TAG}_compressed_expand_sweep.log
echo "== A/B"; timeout 2400 python tools/slots_ab.py --pairs 3 -- --no-cpu-baseline 2>&1 | tee $OUT/${TAG}_slots_ab.log | python -c "
import sys, json
for l in sys.stdin:
    r = json.loads(l)
    if 'summary' in r: print(json.dumps(r))
    else: print(r['arm'], round(r['value'], 1), 'consumed', round(r['handoff']['consumed_on_gpu']['value'], 1), 'exported', round(r['handoff']['exported_to_host']['value'], 2),
               'latency', round(r['latency']['single_witness_ms'], 3), 'reduced', round(r['reduced_witness']['value'], 1), 'parity', r['parity']['digest_match'], 'selfcheck', r['selfcheck']['n_failed'], 'slots', r['details']['resident_slots'])
"

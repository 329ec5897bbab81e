#!/bin/bash
# round 3, GPU session C: final build (compressible slots without the shared-memory cap of k_expand_round; the reduced witness
# keeps plain slots) -- GPU suite, smoke(), memcheck over smoke(), bench.py against the plain-slot arm, and one Spend(31) pair.
TAG=${1:-r03c}; OUT=${2:?usage: $0 TAG OUTPUT_DIR}; mkdir -p $OUT
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm,driver_version --format=csv | tee $OUT/${TAG}_gpu.txt
echo "== pytest -m gpu"; timeout 600 python -m pytest tests -m gpu -q 2>&1 | tail -15 | tee $OUT/${TAG}_pytest_gpu.log
echo "== smoke"; timeout 300 python __graft_entry__.py smoke 2>&1 | tail -2 | tee $OUT/${TAG}_smoke.log
echo "== memcheck smoke"; if command -v compute-sanitizer > /dev/null; then
    timeout 300 compute-sanitizer --tool memcheck --print-limit 5 python __graft_entry__.py smoke > $OUT/${TAG}_memcheck_smoke.log 2>&1; echo "rc=$?" >> $OUT/${TAG}_memcheck_smoke.log
    grep -E "ERROR SUMMARY|smoke ok|rc=|Invalid|misaligned" $OUT/${TAG}_memcheck_smoke.log | head -8
else echo "compute-sanitizer not on PATH" | tee $OUT/${TAG}_memcheck_smoke.log; fi
echo "== A/B"; timeout 900 python tools/slots_ab.py --pairs 3 -- --no-cpu-baseline 2>&1 | tee $OUT/${TAG}_slots_ab.log | python -c "
import sys, json
for l in sys.stdin:
    r = json.loads(l)
    if 'summary' in r: print(json.dumps(r))
    else: print(r['arm'], round(r['value'], 1), 'e2e', round(r['e2e']['value'], 1), 'consumed', round(r['handoff']['consumed_on_gpu']['value'], 1), 'exported', round(r['handoff']['exported_to_host']['value'], 2),
               'latency', round(r['latency']['single_witness_ms'], 3), 'reduced', round(r['reduced_witness']['value'], 1), 'parity', r['parity']['digest_match'], 'selfcheck', r['selfcheck']['n_failed'], 'slots', r['details']['resident_slots'])
"
echo "== Spend(31) pair"; timeout 300 python tools/slots_ab.py --pairs 1 -- --circuit spend --batch 4096 2>&1 | tee $OUT/${TAG}_slots_ab_spend.log | tail -1

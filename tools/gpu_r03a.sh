#!/bin/bash
# round 3, GPU session A: compute data compression probe (tools/probes/compress_probe.cu) -- is a compressible allocation granted on
# this part, and does it make the witness store stream cheaper?  Card name and power limit are logged with the numbers.
TAG=${1:-r03a}; OUT=${2:?usage: $0 TAG OUTPUT_DIR}; mkdir -p $OUT
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm,driver_version --format=csv | tee $OUT/${TAG}_compress_probe.log
timeout 600 tools/probes/compress_probe 2>&1 | tee -a $OUT/${TAG}_compress_probe.log

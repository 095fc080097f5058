#!/bin/bash
# GPU-box helper: GPU tests, then the default bench shape without the e2e / CPU legs (EA_SOLVE_DEBUG cycle counters on a second run).
# usage: gpu_quick.sh <tag> [pytest -k expression]
cd "$(dirname "$0")/.."
TAG=${1:-rX}; K=${2:-}
O=gpurun_out; mkdir -p $O
if [ -n "$K" ]; then timeout 900 python -m pytest tests -m gpu -x -q -k "$K" > $O/${TAG}_tests.log 2>&1; else timeout 900 python -m pytest tests -m gpu -x -q > $O/${TAG}_tests.log 2>&1; fi
echo "tests rc=$?"; tail -5 $O/${TAG}_tests.log
STEPS=${STEPS:-30} bash tools/sweep_env.sh "" > $O/${TAG}_sweep.log 2>&1
STEPS=20 bash tools/sweep_env.sh "EA_SOLVE_DEBUG=1" >> $O/${TAG}_sweep.log 2>&1
cat $O/${TAG}_sweep.log

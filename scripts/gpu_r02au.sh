#!/bin/bash
# pass au: mma.sync in-block kernel as the default of the blocked sequential direction: route tests, full-size
# C3 comparisons, sampler timing in both precision modes.  usage: <tag>
set -u
TAG=${1:-r02au}
mkdir -p gpurun_out
rm -f gpurun_out/parity_fallbacks.jsonl gpurun_out/parity_fullsize.jsonl
timeout 600 python -m pytest tests -q -m gpu -p no:cacheprovider --timeout=300 -k "blocked or c3 or sequential or autoregressive" > gpurun_out/pytest_${TAG}.log 2>&1; echo "pytest rc=$?"; tail -4 gpurun_out/pytest_${TAG}.log
for prec in fp32 bf16; do
  timeout 120 python scripts/sampler_target.py --precision $prec --reps 10 > gpurun_out/sampler_${TAG}_$prec.json 2> gpurun_out/sampler_${TAG}_$prec.err; echo "sampler $prec rc=$?"; cat gpurun_out/sampler_${TAG}_$prec.json
done

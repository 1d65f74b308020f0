#!/bin/bash
# One gpurun call that refreshes the LeRF evidence under gpurun_out/<tag>/ (summaries are copied into profiles/ by hand afterwards):
#   gpurun --timeout 420 -- 'bash scripts/gpu_lerf.sh lerfN'
# parity (kernels, pipeline, C++ drop-in vs the reference's LeRFRenderer), the bench leg, the A/B switches, one ncu capture of the head kernels.
TAG=${1:-lerf}
OUT=gpurun_out/$TAG
mkdir -p $OUT
timeout 200 python -m pytest tests/test_gpu_lerf.py tests/test_gpu_lerf_host.py -q -s > $OUT/pytest.log 2>&1; echo "pytest exit $?"; tail -3 $OUT/pytest.log
timeout 90 python scripts/debug/lerf_leg.py 20 > $OUT/lerf_leg.json 2> $OUT/lerf_leg.err; echo "leg exit $?"
NRF_LERF_SLAB=1 timeout 90 python scripts/debug/lerf_leg.py 20 > $OUT/lerf_leg_slab.json 2>> $OUT/lerf_leg.err; echo "leg (slab kernel) exit $?"
timeout 120 ncu --set full --clock-control none --import-source on -k regex:lerf_ -c 8 -f -o $OUT/prof_lerf python scripts/debug/lerf_leg.py 1 > $OUT/ncu.log 2>&1; echo "ncu exit $?"
ls -la $OUT

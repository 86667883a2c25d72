#!/bin/bash
# Dev: field parity tests + 800x800x80 rebuild timing of the default EDT kernels and of the divide and conquer.
mkdir -p gpurun_out
export PYTHONPATH=.
python -m pytest tests/test_gpu_parity.py tests/test_gpu_rog.py tests/test_gpu_headline.py -m gpu -x -q -k "field or rog or baseline or raster" > gpurun_out/field_tests.log 2>&1
tail -2 gpurun_out/field_tests.log
echo "default"; KEEP_SQ=0 python scripts/field_probe.py 2>&1 | tail -2
echo "D&C"; TOPAY_EDT_SCAN=0 KEEP_SQ=0 python scripts/field_probe.py 2>&1 | tail -2

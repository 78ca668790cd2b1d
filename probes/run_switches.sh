#!/bin/bash
echo "--- chunked staged encoder (G4_STAGED_CHUNK_MB=1)"; G4_STAGED_CHUNK_MB=1 timeout 600 python -m pytest tests/test_gpu_deflate_encode.py tests/test_gpu_deflate_float.py tests/test_gpu_baseline_sizes.py -x -q 2>&1 | tail -2

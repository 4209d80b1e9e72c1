#!/bin/bash
# atlas wire-format check: GPU tests of the upload paths, then the e2e step for every way the atlas can travel
mkdir -p gpurun_out
{
timeout 600 python -m pytest tests/test_gpu_api.py tests/test_golden.py -x -q -m gpu 2>&1 | tail -3
echo "== async, host interleave (16-byte texels on the wire)"; FSPT_ATLAS_INTERLEAVE=cpu timeout 300 python tools/e2e_jitter.py --async 2>&1 | tail -3 | head -1
echo "== async, GPU interleave, RGB24 wire"; FSPT_ATLAS_INTERLEAVE=gpu timeout 300 python tools/e2e_jitter.py --async 2>&1 | tail -3 | head -1
echo "== async, pinned, direct RGBA"; timeout 300 python tools/e2e_jitter.py --async --pinned 2>&1 | tail -3 | head -1
echo "== sync, GPU interleave, RGB24 wire"; FSPT_ATLAS_INTERLEAVE=gpu timeout 300 python tools/e2e_jitter.py 2>&1 | tail -3 | head -1
echo "== laps: async, GPU interleave, RGB24"; FSPT_ATLAS_INTERLEAVE=gpu FSPT_TIMING=1 timeout 300 python tools/upload_time.py --async 2>&1 | tail -12 | head -10
} > gpurun_out/r02b_wire.log 2>&1
cat gpurun_out/r02b_wire.log

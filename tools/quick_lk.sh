#!/bin/bash
# Quick check on the GPU box: per-stage times of the LK + warp path (256 frames per launch) and the kernel / pipeline parity tests.
# usage (from the repo root, on a machine with a B200): bash tools/quick_lk.sh
cd "$(dirname "$0")/.."
python bench.py --steps 6 --warmup 3 --frames-per-gpu 256 --batch 256 --no-cpu-baseline --no-e2e --no-mode-probes 2>/dev/null | python -c "
import json,sys
for l in sys.stdin:
    if l.startswith('{'):
        d=json.loads(l); s=d['stages']
        print('value %.0f ms/step %.3f' % (d['value'], d['ms_per_step']), ' '.join('%s %.3f' % (k, v['ms_per_step']) for k, v in s.items()))
"
timeout 600 python -m pytest tests/test_gpu_kernels.py tests/test_gpu_pipeline.py -q -m gpu -x 2>&1 | tail -3

#!/bin/bash
# scale-shape parity tests + the c5s bench line: compacted tensor-core k_update (default), FFMA (GNCA_NO_TC=1)
timeout 600 python -m pytest tests/test_gpu_scale.py tests/test_gpu_step.py -x -q -m gpu > gpurun_out/tc_scale_test.log 2>&1; tail -6 gpurun_out/tc_scale_test.log
for v in GNCA_NONE=1 GNCA_NO_TC=1; do
  env $v timeout 200 python bench.py --workload c5s --steps 5 --warmup 3 --no-cpu-baseline 2> gpurun_out/tc_c5s.err | python -c "
import json,sys
d=[json.loads(l) for l in sys.stdin if l.startswith('{')][-1]
print('$v', 'ms/rollout %.3f' % d['ms_per_step'], d['roofline']['kernels'])"
  tail -2 gpurun_out/tc_c5s.err
done

#!/bin/bash
# schedule experiments of the INT8-sliced factorisation (one bench line each)
mkdir -p gpurun_out
timeout 900 python -m pytest tests/test_headline_gpu.py -m gpu -q -x > gpurun_out/oz3_pytest.log 2>&1; echo "pytest rc=$?"; tail -3 gpurun_out/oz3_pytest.log
B="python bench.py --steps 4 --warmup 2 --no-extras --no-cpu-baseline --no-prior-sweep --no-dmma-arm"
run() {
  name=$1; shift
  env "$@" timeout 300 $B > gpurun_out/oz3_$name.log 2>&1
  grep '^{' gpurun_out/oz3_$name.log | python -c "
import json,sys
for l in sys.stdin:
    d=json.loads(l); s=d['roofline']['stages_ms']; print('$name: ms/step %.2f chol %.2f trtri %.2f lauum %.2f  nll %.2e grad %.2e' % (d['ms_per_step'], s['cholesky'], s['trtri'], s['lauum'], d['parity']['rel_nll'], d['parity']['rel_grad']))
" || tail -3 gpurun_out/oz3_$name.log
}
run lazy X=1
run lazy_noverlap GPP_OVERLAP_INV=0
run nolazy GPP_OZ_LAZY_MIN=100000

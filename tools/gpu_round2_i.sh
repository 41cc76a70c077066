run() { # tag
  timeout 600 python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29519 bench.py --gpus 2 --config c3 > gpurun_out/i_c3_$1.json 2> gpurun_out/i_c3_$1.err
  python - <<PY
import json
try:
    d=json.load(open('gpurun_out/i_c3_$1.json')); print('c3 N=2 $1', '%.4g' % d['value'], round(d['ms_per_step'],2), d['config'].get('phase_ms_per_step_rank0'))
except Exception as e:
    print('$1 FAILED', e); print(open('gpurun_out/i_c3_$1.err').read()[-800:])
PY
}
nproc; free -g | head -2
run prio; run prio2

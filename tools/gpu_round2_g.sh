# what costs the last 2-5 % at N > 1?  c2 / c2w at N = $1: as shipped (exchange stream at the least priority) and N independent
# replicas without any collective
N=${1:-4}
run() { # config tag
  timeout 400 python -m torch.distributed.run --nnodes=1 --nproc-per-node $N --master-addr 127.0.0.1 --master-port 29519 bench.py --gpus $N --config $1 > gpurun_out/g_$1_$2.json 2> gpurun_out/g_$1_$2.err
  python - <<PY
import json
try:
    d=json.load(open('gpurun_out/g_$1_$2.json')); print('$1 $2', round(d['ms_per_step'],4), d.get('ms_per_step_per_rank'), 'tail', round(d['exchange_tail_ms'],3), 'e2e %.4g' % d['e2e']['value'], 'k3 alone', round(d['roofline']['kernel_ms'],4))
except Exception as e:
    print('$1 $2 FAILED', e); print(open('gpurun_out/g_$1_$2.err').read()[-800:])
PY
}
run c2 prio; run c2w prio
PGP_BENCH_NO_COMM=1 run c2 nocomm; PGP_BENCH_NO_COMM=1 run c2w nocomm

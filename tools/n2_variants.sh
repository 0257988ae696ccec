# exchange-schedule variants of the data-parallel step at N GPUs (default 2): ms/step, e2e ms/step
N=${N:-2}
run() { python -m torch.distributed.run --nnodes=1 --nproc-per-node $N --master-addr 127.0.0.1 --master-port 29513 bench.py --gpus $N --steps 12 --warmup 4 --no-extras --no-cpu-baseline "$@" 2>gpurun_out/nvar.err | python -c "
import json,sys; d=json.loads(sys.stdin.read()); print(round(d['ms_per_step'],3), round(d['e2e']['ms_per_step'],3))"; }
for v in "X=1" "NCCL_NTHREADS=256" "NCCL_NTHREADS=128" "NCCL_MAX_NCHANNELS=8" "NCCL_MAX_NCHANNELS=4 NCCL_NTHREADS=256" "PS_NCCL_PRIO=0"; do echo -n "$v: "; env $v bash -c "$(declare -f run); N=$N run"; done

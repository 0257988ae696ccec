# exchange variants of the data-parallel step at N GPUs: ms/step, e2e ms/step, rays/s
N=${N:-8}
run() { python -m torch.distributed.run --nnodes=1 --nproc-per-node $N --master-addr 127.0.0.1 --master-port 29513 bench.py --gpus $N --steps 12 --warmup 4 --no-extras --no-cpu-baseline "$@" 2>gpurun_out/nvar.err | python -c "
import json,sys; d=json.loads(sys.stdin.read()); print(round(d['ms_per_step'],3), round(d['e2e']['ms_per_step'],3), round(d['value']))"; }
for v in "PS_EXCHANGE=peer" "PS_EXCHANGE=nccl" "PS_EXCHANGE=peer PS_AR_CUTS=4,8,12,14,15"; do echo -n "$v: "; env $v bash -c "$(declare -f run); N=$N run"; done

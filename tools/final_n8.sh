T="timeout 150 python -m torch.distributed.run --nnodes=1 --nproc-per-node 8 --master-addr 127.0.0.1"
$T --master-port 29601 bench.py --gpus 8 --steps 20 --warmup 5 > gpurun_out/r2_final_bench_n8.json 2> gpurun_out/r2_final_bench_n8.err; tail -c 400 gpurun_out/r2_final_bench_n8.json; echo
$T --master-port 29603 bench.py --gpus 8 --config c5 --steps 10 --warmup 3 > gpurun_out/r2_final_bench_c5_n8.json 2>/dev/null; python -c "
import json; d=json.load(open('gpurun_out/r2_final_bench_c5_n8.json')); print('c5', d['value'], d['ms_per_step'], d['e2e'])"
$T --master-port 29604 bench.py --gpus 8 --optimizer fused --steps 12 --warmup 4 --no-extras --no-cpu-baseline > gpurun_out/r2_final_bench_n8_fusedopt.json 2>/dev/null; python -c "
import json; d=json.load(open('gpurun_out/r2_final_bench_n8_fusedopt.json')); print('fusedopt', d['ms_per_step'], d['e2e']['ms_per_step'])"
$T --master-port 29605 tools/event_trace.py > gpurun_out/r2_final_evtrace_n8.txt 2>&1; grep "# step" gpurun_out/r2_final_evtrace_n8.txt

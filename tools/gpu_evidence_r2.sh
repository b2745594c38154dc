#!/bin/bash
# Round-2 evidence in one gpurun call on >= 2 GPUs:  gpurun --gpus 2 --timeout 1500 -- 'bash tools/gpu_evidence_r2.sh r2p'
# Every ncu pass runs only after the same command has exited 0 without ncu.
TAG=${1:-r2x}
O=gpurun_out/$TAG
mkdir -p $O
set -x
nvidia-smi --query-compute-apps=pid,used_memory --format=csv,noheader
# (1) pipe issue-rate micro-benchmark (the "three half-rate pipes" model of DESIGN.md section 4)
(cd tools/microbench && nvcc -gencode arch=compute_100a,code=sm_100a -O3 -o pipe_mix pipe_mix.cu && ./pipe_mix) > $O/pipe_mix.txt 2>&1
# (2) launch list + full capture of the SQ kernel, full capture of the queue kernel (cfg5)
BP="python bench.py --steps 2 --warmup 1 --rays 1e9 --no-e2e --no-cpu-baseline --no-extras"
B5="python bench.py --workload cfg5 --steps 2 --warmup 1 --no-e2e --no-cpu-baseline --no-smoothing --no-extras"
timeout 300 $BP > $O/plain3.json 2> $O/plain3.err && {
  timeout 600 ncu --metrics gpu__time_duration.sum --clock-control none -c 400 --csv --log-file $O/launches.csv $BP > $O/ncu_l.log 2>&1
  timeout 600 ncu --set full --clock-control none --import-source on -k regex:trace_exchange -s 2 -c 1 -f -o $O/prof_sq $BP > $O/ncu_sq.log 2>&1
}
timeout 300 $B5 > $O/plain5.json 2> $O/plain5.err && \
  timeout 600 ncu --set full --clock-control none --import-source on -k regex:trace_exchange -s 2 -c 1 -f -o $O/prof_queue $B5 > $O/ncu_q.log 2>&1
# (3) NVLink traffic of the fused row hand-over: one process, two GPUs, rows gathered on device 0 (rthx_trace_exchange_multi, counts_out = NULL)
timeout 200 python tools/gpu_gather_probe.py > $O/gather_plain.log 2>&1 && \
  timeout 600 ncu --metrics nvltx__bytes.sum,nvlrx__bytes.sum,gpu__time_duration.sum,lts__t_sectors_srcunit_tex_aperture_peer_op_write.sum,lts__t_sectors_srcunit_tex_aperture_peer_op_red.sum --clock-control none -k regex:trace_exchange --csv --log-file $O/nvlink.csv python tools/gpu_gather_probe.py > $O/ncu_nv.log 2>&1
ls -la $O

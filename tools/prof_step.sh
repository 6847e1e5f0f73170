#!/bin/bash
# one full ncu capture of the thread-per-env step kernel on the 1M-env workload (c2w); summary only (the report is too large to copy back)
mkdir -p gpurun_out
CS_BENCH_LPE=${CS_BENCH_LPE:-1} ncu --set full --clock-control none --import-source on -k regex:flight_tpe_kernel -s 12 -c 1 -f -o /tmp/prof_c2w_tpe python tools/profile_run.py c2w 16 > /dev/null 2>&1
python tools/ncu_summary.py /tmp/prof_c2w_tpe.ncu-rep > gpurun_out/prof_c2w_tpe.txt
python tools/ncu_lines.py /tmp/prof_c2w_tpe.ncu-rep 30 >> gpurun_out/prof_c2w_tpe.txt
ncu -i /tmp/prof_c2w_tpe.ncu-rep --page raw --csv 2>/dev/null | python -c "
import csv,sys
rows=list(csv.reader(sys.stdin)); d=dict(zip(rows[0],rows[2]))
for k in sorted(d):
    if any(t in k for t in ('l1tex__t_requests','l1tex__t_sectors_pipe_lsu','l1tex__data_pipe_lsu_wavefronts','lsu_mem_global_op','l1tex__lsu_writeback','l1tex__t_bytes','lts__t_bytes.sum','l1tex__throughput','lts__throughput','sm__inst_executed_pipe_lsu','l1tex__data_pipe')): print(k, d[k])
" >> gpurun_out/prof_c2w_tpe.txt
cat gpurun_out/prof_c2w_tpe.txt

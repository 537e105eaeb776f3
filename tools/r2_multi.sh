#!/bin/bash
# 8-GPU evidence of round 2 (run on an 8-GPU machine): concurrent-copy ceiling, bench lines at N = 8 / 4 / 2.
set -u
OUT=gpurun_out; mkdir -p $OUT
TR="python -m torch.distributed.run --nnodes=1 --master-addr 127.0.0.1"
nvidia-smi topo -m > $OUT/r2f_topo_n8.txt 2>&1; lscpu | head -30 >> $OUT/r2f_topo_n8.txt; numactl -H >> $OUT/r2f_topo_n8.txt 2>&1
timeout 200 $TR --nproc-per-node 8 --master-port 29611 tools/pcie_peak.py > $OUT/r2f_pcie_peak_n8.txt 2> $OUT/r2f_pcie_peak_n8.err; echo "pcie n8 rc=$?"; cat $OUT/r2f_pcie_peak_n8.txt
timeout 200 $TR --nproc-per-node 4 --master-port 29612 tools/pcie_peak.py > $OUT/r2f_pcie_peak_n4.txt 2>> $OUT/r2f_pcie_peak_n8.err; echo "pcie n4 rc=$?"
timeout 200 $TR --nproc-per-node 2 --master-port 29613 tools/pcie_peak.py > $OUT/r2f_pcie_peak_n2.txt 2>> $OUT/r2f_pcie_peak_n8.err; echo "pcie n2 rc=$?"
for n in 8 4 2; do
  timeout 300 $TR --nproc-per-node $n --master-port $((29620 + n)) bench.py --gpus $n --steps 50 --warmup 3 > $OUT/r2f_bench_n$n.json 2> $OUT/r2f_bench_n$n.err; echo "bench n$n rc=$?"
  python -c "
import json,sys
d=json.loads(open('$OUT/r2f_bench_n$n.json').read().strip().splitlines()[-1])
print('N=$n value %.2fM e2e %.2fM (%.2f of raw ceiling %.2fM) stream_1m %.2fM host_fed %.2fM sustained %.2fM' % (d['value']/1e6, d['e2e']['value']/1e6, d['e2e']['frac_of_raw_copy_ceiling'], d['e2e']['raw_copy_ceiling_images_per_s']/1e6, d['stream_1m']['images_per_s']/1e6, d['stream_1m']['host_fed']['images_per_s']/1e6, d['sustained']['images_per_s']/1e6), d['stream_1m']['oracle_spot_check'])
" 2>&1 | tail -2
done
timeout 120 python bench.py --steps 50 --warmup 3 > $OUT/r2f_bench_n1_on8box.json 2> $OUT/r2f_bench_n1_on8box.err; echo "bench n1 rc=$?"
ls -la $OUT | tail -12

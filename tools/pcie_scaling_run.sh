#!/bin/bash
# The measurement behind profiles/r02_pcie_ceiling_n*.txt and r02_e2e_multi.txt: run on an 8-GPU box
#   gpurun --gpus 8 -- bash tools/pcie_scaling_run.sh
O=gpurun_out
bash tools/box_probe.sh > $O/r02_box_probe_8gpu.txt 2>&1
P="timeout 60 build/pcie_ceiling --secs 0.4"
for n in 1 2 4 8; do
  g=$(seq -s, 0 $((n-1)))
  { $P --gpus $g; [ $n -gt 1 ] && $P --gpus $g --threads; } > $O/r02_pcie_ceiling_n$n.txt 2>&1
done
{ $P --gpus 0,1,2,3,4,5,6,7 --sync block; $P --gpus 0,1,2,3,4,5,6,7 --pin; $P --gpus 0,1,2,3,4,5,6,7 --alloc register;
  $P --gpus 0,1,2,3,4,5,6,7 --alloc portable --threads;
  $P --gpus 0 --patterns zc_two,zcr_dmaw,dmar_zcw,dma_pieces
  $P --gpus 0,1,2,3,4,5,6,7 --patterns zc_two,zcr_dmaw,dmar_zcw,dma_pieces
  for pair in 0,1 0,2 0,4 0,7 4,5 0,1,4,5; do $P --gpus $pair --patterns dma_both,zc_inplace; done; } > $O/r02_pcie_ceiling_variants.txt 2>&1
E="timeout 90 build/e2e_multi --secs 1.5"
{ for n in 1 2 4 8; do $E --gpus $(seq -s, 0 $((n-1))); done
  $E --gpus 0,1,2,3,4,5,6,7 --threads
  $E --gpus 0,1,2,3,4,5,6,7 --pin
  FLUC_TTMLBLEND_SYNC=block $E --gpus 0,1,2,3,4,5,6,7
  $E --gpus 0,1,2,3,4,5,6,7 --opaque
  $E --gpus 0 --opaque; } > $O/r02_e2e_multi.txt 2>&1
timeout 200 python -m torch.distributed.run --nnodes=1 --nproc-per-node 8 --master-addr 127.0.0.1 --master-port 29511 \
  bench.py --gpus 8 --steps 20 --warmup 5 --no-cpu-baseline > $O/r02_t0_bench_n8.json 2> $O/r02_t0_bench_n8.err
tail -n 3 $O/r02_e2e_multi.txt

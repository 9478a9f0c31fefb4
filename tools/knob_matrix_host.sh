#!/bin/bash
# The host-frame tests only (zero copy, staging, host DMA batches through fluc_ttmlblend_set_host_dma,
# wait semantics) under every knob: the short companion of knob_matrix.sh.
#   gpurun -- bash tools/knob_matrix_host.sh
K="host_dma or wait_for or two_overlays or host_path or host_forget or unaligned or registered_host_frames"
for v in NONE=1 FLUC_TTMLBLEND_GROUPS=0 FLUC_TTMLBLEND_MULTI=0 FLUC_TTMLBLEND_LAZY=1 FLUC_TTMLBLEND_LAZY=0 \
         FLUC_TTMLBLEND_AUTOCROP=0 FLUC_TTMLBLEND_BULK=0 FLUC_TTMLBLEND_LANES=7 \
         FLUC_TTMLBLEND_PDL=0 FLUC_TTMLBLEND_OPAQUE_SKIP=1 FLUC_TTMLBLEND_OPAQUE_SKIP=0 \
         FLUC_TTMLBLEND_STAGE_THREADS=1 FLUC_TTMLBLEND_COMPACT_PARAMS=0 \
         FLUC_TTMLBLEND_SYNC=block FLUC_TTMLBLEND_STAGE_NT=0 FLUC_TTMLBLEND_HOST_DMA=1 FLUC_TTMLBLEND_HOST_DMA=0 \
         FLUC_TTMLBLEND_DMA_PIECE=0; do
  echo "== $v"
  env $v timeout 200 python -m pytest tests/test_gpu_hazards.py tests/test_gpu_configs.py tests/test_gpu_parity.py \
      -q -x -k "$K" 2>&1 | tail -1
done

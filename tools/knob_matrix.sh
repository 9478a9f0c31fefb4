#!/bin/bash
# Runs the parity tests with every alternative code path forced through its environment knob:
# table kernel only, no multi-layout launches, in-place launches always / never lazy, no
# auto-crop, register-staged instead of TMA-staged overlay, interleaved chunk order, and the
# host-frame knobs; then the global-alpha, move, resize, geometry and operator-domain files under each knob. Every line
# must end in "passed".
#   gpurun -- bash tools/knob_matrix.sh
K="rectangles_match_oracle or golden or fuzz or alpha_sweep or scaled_rectangles or regions or unaligned or chain or ping_pong or dependency or two_overlays or update or sparse_cues or host_path or host_dma"
for v in FLUC_TTMLBLEND_GROUPS=0 FLUC_TTMLBLEND_MULTI=0 FLUC_TTMLBLEND_LAZY=1 FLUC_TTMLBLEND_LAZY=0 \
         FLUC_TTMLBLEND_AUTOCROP=0 FLUC_TTMLBLEND_BULK=0 FLUC_TTMLBLEND_LANES=7 \
         FLUC_TTMLBLEND_PDL=0 FLUC_TTMLBLEND_OPAQUE_SKIP=1 FLUC_TTMLBLEND_OPAQUE_SKIP=0 \
         FLUC_TTMLBLEND_STAGE_THREADS=1 FLUC_TTMLBLEND_COMPACT_PARAMS=0 \
         FLUC_TTMLBLEND_SYNC=block FLUC_TTMLBLEND_STAGE_NT=0 FLUC_TTMLBLEND_HOST_DMA=1 FLUC_TTMLBLEND_HOST_DMA=0 \
         FLUC_TTMLBLEND_DMA_PIECE=0; do
  echo "== $v"
  env $v timeout 300 python -m pytest tests/test_gpu_parity.py tests/test_gpu_scale.py tests/test_gpu_regions.py \
      tests/test_gpu_hazards.py tests/test_gpu_update.py tests/test_gpu_configs.py \
      -q -x -k "$K" 2>&1 | tail -1
  # every global-alpha (JF_GA) instantiation and the operator domains under the same knob
  env $v timeout 600 python -m pytest tests/test_gpu_global_alpha.py tests/test_gpu_domain.py -q -x 2>&1 | tail -1
  # overlay_set_positions (batch prepare, left / top clipping at prepare time) under the same knob
  env $v timeout 600 python -m pytest tests/test_gpu_move.py -q -x 2>&1 | tail -1
  # overlay_set_render_rectangles (scale-and-scan batch, crop and lazy figures of the resized rectangles)
  env $v timeout 600 python -m pytest tests/test_gpu_resize.py -q -x 2>&1 | tail -1
  # frames above 4K up to 32768 wide: row-split windows, table-kernel fallbacks, offsets past 4 GiB
  env $v timeout 600 python -m pytest tests/test_gpu_geometry.py -q -x 2>&1 | tail -1
done

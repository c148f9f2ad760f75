#!/usr/bin/env bash
set -x
mkdir -p gpurun_out
timeout 300 ncu -k regex:"proto_patch|mask_upsample_pack2|proto_bin_fused|scan_tiles_kernel|pm_rows|process_mask_kernel|pm_clear" \
  --metrics gpu__time_duration.sum,dram__bytes_read.sum,dram__bytes_write.sum,lts__t_sector_hit_rate.pct,smsp__inst_executed.sum,launch__grid_size \
  --clock-control none -s 60 -c 60 --csv --log-file gpurun_out/r2g_slide30k_ncu.csv \
  python bench.py --slide-size 30000 --steps 2 --warmup 2 --no-cpu-baseline --no-sub --no-torch-cuda --no-e2e --slide-streams 1 > gpurun_out/r2g.log 2>&1
tail -2 gpurun_out/r2g.log | cut -c1-300

#!/bin/bash
# One-GPU evidence run of round 2: bench lines for every config, reference arm, ncu launch list + full captures.
# usage (on the GPU box): tools/final_r02.sh   -> gpurun_out/r02_*
O=gpurun_out
python bench.py > $O/r02_bench_n1.json 2> $O/r02_bench_n1.err
python bench.py --impl reference --steps 20 --warmup 5 > $O/r02_bench_reference_n1.json 2>/dev/null
for c in 1 3 4 5; do python bench.py --config $c --steps 40 --warmup 5 > $O/r02_bench_c${c}_n1.json 2>/dev/null; done
ncu --metrics gpu__time_duration.sum --clock-control none --csv --log-file $O/r02_launches.csv python bench.py --steps 3 --warmup 3 --no-cpu-baseline --no-strong > /dev/null 2>&1
ncu --set full --clock-control none --import-source on -k regex:"cone_trace|vox_shade|raster_small|raster_tiles|mip_fused3|vox_clear_sparse|vox_resolve_sparse" -s 40 -c 12 -o $O/r02_frame_kernels python tools/run_config.py 2 6 > $O/r02_ncu_frame.log 2>&1
python tools/timeline.py 2 > $O/r02_timeline_c2.txt 2>&1
ls -la $O | grep r02_ | tail -20

#!/bin/sh
# Copy the outputs of tools/final_evidence.sh <prefix> from gpurun_out/ into profiles/ under the round-2 final names.
# usage (here, after the gpurun call): tools/publish_evidence.sh fin "v20: <what the final code is>"
set -e
P=${1:-fin}; WHAT=${2:-final code}
cp gpurun_out/${P}_launches.csv profiles/r2_final_launches.csv
{ echo "# ncu launch list, round-2 FINAL code ($WHAT)"; echo; echo 'command: `python bench.py --workload config2 --steps 1 --warmup 1 --no-cpu --no-side --no-microbench` (exit 0 without ncu first), then the same under `ncu --metrics gpu__time_duration.sum --clock-control none -c 700 --csv` (tools/final_evidence.sh); raw: r2_final_launches.csv.  `k_extend<0, 1, W>` = no counters (speculative traversal), 4-wide, W = widened slab test (camera rays); `k_shade<1, D>` = Philox, D = deferred queue append (three windows per reservation; 0 = immediate append).'; echo; python tools/profile_report.py launches profiles/r2_final_launches.csv; } > profiles/r2_final_launches_summary.md
{ echo "# ncu --set full, round-2 FINAL code ($WHAT), BASELINE config 2 (1920x1080, one 64-spp frame): k_extend / k_shade of bounces 0, 1, 2"; echo; echo 'command: `ncu --set full --clock-control none --import-source on -k regex:k_extend|k_shade --launch-count 6 python tools/traffic_run.py --workload config2 --frames 1` (tools/final_evidence.sh; the plain command exited 0 first).  Summary made by tools/profile_report.py.'; echo; python tools/profile_report.py full gpurun_out/${P}_c2_full.ncu-rep; } > profiles/r2_final_ncu_full_config2.md
{ echo "# ncu --set full, round-2 FINAL code ($WHAT), BASELINE config 4 (9 999 392 triangles, 3840x2160, one frame, RT_MAX_PATHS_MI=128): k_extend / k_shade of bounces 1, 2"; echo; echo 'command: `RT_MAX_PATHS_MI=128 ncu --set full --clock-control none --import-source on -k regex:k_extend|k_shade --launch-skip 2 --launch-count 4 python tools/traffic_run.py --workload config4 --frames 1`'; echo; python tools/profile_report.py full gpurun_out/${P}_c4_full.ncu-rep; } > profiles/r2_final_ncu_full_config4.md
cp gpurun_out/${P}_bench.json profiles/r2_final_bench_line.json
cp gpurun_out/${P}_ref.json profiles/r2_final_bench_reference_arm.json
cp gpurun_out/${P}_config1.json profiles/r2_final_bench_config1.json
cp gpurun_out/${P}_config3.json profiles/r2_final_bench_config3.json
for w in config2 4k config4; do cp gpurun_out/traffic_$w.csv profiles/r2_traffic_$w.csv; done
python tools/extend_traffic.py gpurun_out/traffic_config2 gpurun_out/traffic_4k gpurun_out/traffic_config4 | grep -E "dram_bytes_per_segment|^config|^4k"

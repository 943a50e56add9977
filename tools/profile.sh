#!/bin/bash
# The ncu passes behind profiles/, run on a B200: tools/profile.sh [output directory, default profile_out].
# Databases and index files first, in a directory every pass reuses: building the index under ncu crashes the profiler's child process.
set -e
R=${ROUND:-r2b}
W=$(mktemp -d)
trap 'rm -rf "$W"' EXIT
python -c "import sys, bench; bench.load_databases(sys.argv[1])" "$W" > /dev/null
K="regex:seed_kernel|lis_kernel|lis_reset_kernel|finalize_kernel|traceback_kernel|pack_reads_kernel|bin_kernel"
O=${1:-profile_out}
mkdir -p "$O"
# launch list: durations of every launch of our kernels in a short bench run (shares vs the CUDA-event split of bench.py)
ncu --metrics gpu__time_duration.sum --clock-control none -k "$K" -c 400 --csv --log-file "$O"/${R}_launches.csv \
    python bench.py --reads 1000000 --steps 2 --warmup 1 --no-cpu-baseline --work-dir "$W" > "$O"/ncu_list.log 2>&1
# one full capture of the dominant kernel and one of the HBM-side kernel (400 k reads keep the replay short)
ncu --set full --clock-control none --import-source on -k regex:lis_kernel -s 1 -c 1 -f -o "$O"/${R}_lis \
    python bench.py --reads 400000 --steps 1 --warmup 1 --no-cpu-baseline --work-dir "$W" > "$O"/ncu_lis.log 2>&1
ncu --set full --clock-control none --import-source on -k regex:seed_kernel -s 8 -c 1 -f -o "$O"/${R}_seed \
    python bench.py --reads 400000 --steps 1 --warmup 1 --no-cpu-baseline --work-dir "$W" > "$O"/ncu_seed.log 2>&1
for k in lis seed; do
  ncu -i "$O"/${R}_$k.ncu-rep --page details > "$O"/${R}_${k}_kernel_ncu_details.txt 2>&1
  ncu -i "$O"/${R}_$k.ncu-rep --page raw --csv --metrics dram__bytes_read.sum,dram__bytes_write.sum,gpu__time_duration.sum,sm__inst_executed_pipe_alu.avg.pct_of_peak_sustained_active,sm__inst_executed_pipe_fma.avg.pct_of_peak_sustained_active,sm__inst_executed_pipe_lsu.avg.pct_of_peak_sustained_active,lts__t_sector_hit_rate.pct,smsp__thread_inst_executed_per_inst_executed.ratio,smsp__issue_active.avg.pct_of_peak_sustained_active > "$O"/${R}_${k}_raw.csv 2>&1
done

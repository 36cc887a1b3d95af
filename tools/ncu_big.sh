# ncu --set full captures of the large-chain cluster-editing kernels (one launch each):
#   cfg4 sample (500 tetraploid chains of 200-330 reads): k_cluster_sparse<256>
#   cfg1 (one chain of 1,400 reads): k_cluster_sparse<1024>
# Raw metric pages land in gpurun_out/<tag>_*_raw.csv; tools/large_chain_summary.py turns them into profiles/<tag>_large_chain_kernels.md
set -x
T=${1:-r2c}
ncu --set full --clock-control none --import-source on --kernel-name regex:'k_cluster_sparse' -c 1 -f -o /tmp/${T}_cfg4s python bench.py --workload cfg4 --scale 0.05 --steps 1 --warmup 1 --no-cpu-baseline > /dev/null 2>&1
ncu -i /tmp/${T}_cfg4s.ncu-rep --page raw --csv > gpurun_out/${T}_cfg4_sparse_raw.csv 2>/dev/null
ncu --set full --clock-control none --import-source on --kernel-name regex:'k_cluster_sparse' -c 1 -f -o /tmp/${T}_cfg1 python bench.py --workload cfg1 --scale 1.0 --steps 1 --warmup 1 --no-cpu-baseline > /dev/null 2>&1
ncu -i /tmp/${T}_cfg1.ncu-rep --page raw --csv > gpurun_out/${T}_cfg1_sparse_raw.csv 2>/dev/null
ncu -i /tmp/${T}_cfg1.ncu-rep --page source --csv --kernel-name regex:k_cluster_sparse > gpurun_out/${T}_cfg1_sparse_src.csv 2>/dev/null

mkdir -p gpurun_out; rm -rf gpurun_out/*
echo "== ncu gemm"; timeout -s KILL 400 ncu --set full --clock-control none --import-source on -k regex:gemm_.._kernel -o gpurun_out/gemm_fwd1 python scripts/ncu_gemm.py fwd1 > gpurun_out/ncu_gemm.log 2>&1; echo "ncu exit $?"; ls -la gpurun_out/*.ncu-rep
timeout -s KILL 900 python bench.py --steps 10 --warmup 3 > gpurun_out/bench.log 2>&1; echo "bench exit $?"; tail -c 6000 gpurun_out/bench.log

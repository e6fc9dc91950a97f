mkdir -p gpurun_out; rm -rf gpurun_out/*
echo "== probe"; timeout -s KILL 120 ./scripts/probe_umma 2>&1 | tee gpurun_out/probe_umma.log | tail -20
echo "== cin_v2 tests"; CTR_TEST_CIN_V2=1 timeout -s KILL 300 python -m pytest tests/test_gpu_cin_v2.py -m gpu -q --timeout 200 -p no:cacheprovider --tb=short > gpurun_out/pytest_cinv2.log 2>&1; echo "exit $?"; grep -E "^(FAILED|ERROR)|passed|failed|^E  " gpurun_out/pytest_cinv2.log | tail -12 | cut -c1-250
for v in 0 1; do
  CTR_CIN_V2=$v timeout -s KILL 300 python bench.py --workload xdeepfm --steps 5 --warmup 3 --no-cpu-baseline --no-secondary > gpurun_out/bench_xdeepfm_v2_$v.log 2>&1; echo "bench xdeepfm CIN_V2=$v exit $?"
  grep '^{' gpurun_out/bench_xdeepfm_v2_$v.log | python -c "
import sys,json
for l in sys.stdin:
    d=json.loads(l); print('ms/step', round(d['ms_per_step'],3), {k:round(v['ms_per_step'],3) for k,v in d['per_entry_ms'].items() if 'cin' in k})"
done

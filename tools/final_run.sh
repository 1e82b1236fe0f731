# One N=1 pass for the record: parity tier, bench line, ncu launch list of the same command, full capture of K1.
# Every step is bounded.
set -x
timeout 900 python -m pytest tests -m gpu -x -q --timeout 240 --timeout-method thread 2>&1 | tail -6
timeout 600 python bench.py > gpurun_out/bench_n1.json 2> gpurun_out/bench_n1.err; tail -c 300 gpurun_out/bench_n1.err
timeout 300 python bench.py --impl reference --steps 5 --warmup 1 > gpurun_out/bench_ref_n1.json 2>/dev/null
timeout 600 ncu --metrics gpu__time_duration.sum --clock-control none -c 400 --csv --log-file gpurun_out/r02_bench_launches.csv python bench.py --steps 2 --warmup 1 --no-cpu --no-e2e > gpurun_out/bench_under_ncu.log 2>&1
timeout 400 ncu --set full --clock-control none --import-source on -k regex:sketch_fill_uniform -c 1 -f -o gpurun_out/r02_k1 python bench.py --steps 1 --warmup 1 --no-cpu --no-e2e --no-secondary > /dev/null 2>&1
python -c "import __graft_entry__ as g; g.smoke()" 2>&1 | tail -2

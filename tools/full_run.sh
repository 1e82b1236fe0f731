# One comprehensive GPU pass: parity tier, the bench line, the K2 timings.  Every step is bounded.
set -x
timeout 900 python -m pytest tests -m gpu -x -q --timeout 240 --timeout-method thread 2>&1 | tail -25
timeout 600 python bench.py > gpurun_out/bench_n1.json 2> gpurun_out/bench_n1.err; tail -c 400 gpurun_out/bench_n1.err
timeout 300 python tools/bench_secondary.py --only-k2 > gpurun_out/k2_thresh.jsonl 2>&1

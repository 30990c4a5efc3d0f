# large-frame configuration (10 views x 16 persons, 64 frames): parity tests, bench
set +e
mkdir -p gpurun_out
timeout 900 python -m pytest tests -m gpu -q -x -k "stress or cluster or gat or aggregat or end_to_end" --timeout 300 > gpurun_out/st_pytest.log 2>&1; echo "exit $?" >> gpurun_out/st_pytest.log
timeout 600 python bench.py --config ring10 --persons 16 --frames 64 --steps 5 --cpu-budget 3 --latency-frames 0 > gpurun_out/st_ring10.log 2>&1; echo "exit $?" >> gpurun_out/st_ring10.log
tail -15 gpurun_out/st_pytest.log; tail -6 gpurun_out/st_probe.log; tail -3 gpurun_out/st_ring10.log | cut -c1-1800

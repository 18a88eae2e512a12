# Scan tail (one B200): GPU suite first, then the per-phase stamps.
mkdir -p gpurun_out/tail
O=gpurun_out/tail
timeout 900 python -m pytest tests -m gpu -q -x > $O/test_gpu.log 2>&1
echo "gpu suite rc=$?" | tee $O/status.txt
tail -6 $O/test_gpu.log
timeout 300 python scripts/phase_times.py > $O/phase_times.jsonl 2> $O/phase_times.err
echo "phase_times rc=$?" | tee -a $O/status.txt
cat $O/phase_times.jsonl; tail -3 $O/phase_times.err

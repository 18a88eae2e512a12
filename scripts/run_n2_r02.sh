# Round-2 2-GPU check (gpurun --gpus 2): the multi-GPU tests (fused NVLink exchange in the scan tail, merge through the
# heads of the per-rank rows) and the batch-1 bench with its in-run parity check.
mkdir -p gpurun_out/n2
O=gpurun_out/n2
timeout 600 python -m pytest tests/test_multigpu_gpu.py -m gpu -q > $O/test_multigpu.log 2>&1
echo "multigpu tests rc=$?" | tee $O/status.txt
tail -4 $O/test_multigpu.log
T="python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29533"
timeout 300 $T bench.py --gpus 2 --steps 50 --warmup 5 --no-cpu-baseline --secondary none > $O/bench_n2.json 2> $O/bench_n2.err
echo "bench rc=$?" | tee -a $O/status.txt
python - <<P
import json
d=json.loads(open("$O/bench_n2.json").read().strip().splitlines()[-1])
print(d["value"], d["ms_per_step"], d["e2e"]["ms_per_step"], d["parity_check"]["ok"], d["roofline"]["launch_ms"])
P

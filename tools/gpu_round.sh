#!/bin/bash
# One GPU visit: parity tests, bench (both arms), ncu launch list + full captures of the top kernels.
# usage (from repo root, on the GPU box): bash tools/gpu_round.sh <tag>
TAG=${1:-r1}
O=gpurun_out
mkdir -p $O
nvidia-smi --query-gpu=name,clocks.max.sm,power.limit --format=csv > $O/${TAG}_gpu.txt 2>&1
timeout 600 python -m pytest tests -m gpu -x -q > $O/${TAG}_pytest_gpu.log 2>&1
MZ_TREE_THREAD=1 timeout 300 python -m pytest tests/test_mcts_gpu.py -m gpu -x -q 2>&1 | tail -2 | sed 's/^/thread-per-tree kernels forced for A <= 4 (MZ_TREE_THREAD=1): /' >> $O/${TAG}_pytest_gpu.log
timeout 120 python -c "import __graft_entry__ as g; g.smoke()" >> $O/${TAG}_pytest_gpu.log 2>&1
echo "pytest exit $?" >> $O/${TAG}_pytest_gpu.log
timeout 600 python bench.py --steps 5 --warmup 3 > $O/${TAG}_bench_gomoku.json 2> $O/${TAG}_bench_gomoku.err
echo "bench exit $?" >> $O/${TAG}_bench_gomoku.err
timeout 300 python bench.py --workload tictactoe --steps 10 --warmup 3 --no-train-step > $O/${TAG}_bench_tictactoe.json 2> $O/${TAG}_bench_tictactoe.err
timeout 300 python bench.py --workload atari --steps 5 --warmup 3 --no-train-step --no-cpu-baseline > $O/${TAG}_bench_atari.json 2> $O/${TAG}_bench_atari.err
timeout 300 python bench.py --workload cartpole --steps 10 --warmup 3 --no-train-step --no-cpu-baseline > $O/${TAG}_bench_cartpole.json 2> $O/${TAG}_bench_cartpole.err
timeout 300 python bench.py --impl reference --steps 2 --warmup 1 > $O/${TAG}_bench_reference.json 2> $O/${TAG}_bench_reference.err
# launch list of a short search at the bench's per-launch batch (1024 trees per sub-batch)
timeout 600 ncu --metrics gpu__time_duration.sum --clock-control none -c 400 --csv --log-file $O/${TAG}_launches_gomoku.csv \
    python tools/profile_target.py gomoku 3 1024 > $O/${TAG}_ncu_launch.log 2>&1
timeout 600 ncu --set full --clock-control none --import-source on -k regex:conv3x3 -s 2 -c 1 -f -o $O/${TAG}_conv_full \
    python tools/profile_target.py gomoku 2 1024 > $O/${TAG}_ncu_full.log 2>&1
timeout 600 ncu --set full --clock-control none --import-source on -k regex:backup_select_kernel -s 150 -c 1 -f -o $O/${TAG}_select_full \
    python tools/profile_target.py gomoku 200 1024 > $O/${TAG}_ncu_select.log 2>&1
tail -3 $O/${TAG}_pytest_gpu.log
cat $O/${TAG}_bench_gomoku.json
tail -3 $O/${TAG}_bench_gomoku.err

#!/bin/bash
# hot/cold tree layout + in-place conv buffers: parity, bench, ncu captures of the tree kernels and the conv kernel
TAG=${1:-r2c}
O=gpurun_out; mkdir -p $O
timeout 1200 python -m pytest tests -m gpu -x -q 2>&1 | tail -15 > $O/${TAG}_pytest_gpu.log
cat $O/${TAG}_pytest_gpu.log
timeout 900 python bench.py --steps 5 --warmup 3 --no-cpu-baseline > $O/${TAG}_bench.json 2> $O/${TAG}_bench.err
tail -2 $O/${TAG}_bench.err; python tools/show_bench.py $O/${TAG}_bench.json
timeout 600 ncu --set full --clock-control none --import-source on -k regex:backup_select_kernel -s 150 -c 1 -f -o $O/${TAG}_tree_gomoku \
    python tools/profile_target.py gomoku 200 1024 > $O/${TAG}_ncu_tree_gomoku.log 2>&1
timeout 600 ncu --set full --clock-control none --import-source on -k regex:backup_select_kernel -s 20 -c 1 -f -o $O/${TAG}_tree_ttt262144 \
    python tools/profile_target.py tictactoe 25 262144 > $O/${TAG}_ncu_tree_ttt.log 2>&1
timeout 600 ncu --set full --clock-control none --import-source on -k regex:conv3x3 -s 2 -c 1 -f -o $O/${TAG}_conv_full \
    python tools/profile_target.py gomoku 2 1024 > $O/${TAG}_ncu_conv.log 2>&1
timeout 300 python bench.py --workload tictactoe --trees 262144 --steps 5 --warmup 3 --no-cpu-baseline --no-train-step --no-self-play --no-configs > $O/${TAG}_bench_ttt262144.json 2>/dev/null
python tools/show_bench.py $O/${TAG}_bench_ttt262144.json
ls -la $O/${TAG}_*

#!/bin/bash
# full validation: GPU suite (+ kernel variants), smoke, default bench, reference arm, sanitizer, launch list
TAG=${1:-r2m}
O=gpurun_out; mkdir -p $O
L=$O/${TAG}_pytest_gpu.log
timeout 1500 python -m pytest tests -m gpu -x -q > $L 2>&1; echo "pytest exit $?" >> $L
MZ_TREE_THREAD=1 timeout 600 python -m pytest tests/test_mcts_gpu.py -m gpu -x -q 2>&1 | tail -2 | sed 's/^/thread-per-tree kernels forced for A <= 4 (MZ_TREE_THREAD=1): /' >> $L
MZ_FUSED_SEARCH=0 MZ_NO_PDL=1 MZ_NO_FUSED_ROOT=1 timeout 600 python -m pytest tests/test_network_gpu.py tests/test_mcts_gpu.py -m gpu -x -q 2>&1 | tail -2 | sed 's/^/launch chain, no PDL, separate root launches: /' >> $L
timeout 300 python -c "import __graft_entry__ as g; g.smoke()" >> $L 2>&1; echo "smoke exit $?" >> $L
tail -12 $L
timeout 900 python bench.py --steps 10 --warmup 3 > $O/${TAG}_bench.json 2> $O/${TAG}_bench.err; echo "bench exit $?" >> $O/${TAG}_bench.err
tail -2 $O/${TAG}_bench.err; python tools/show_bench.py $O/${TAG}_bench.json
timeout 600 python bench.py --impl reference --steps 2 --warmup 1 > $O/${TAG}_bench_reference.json 2> /dev/null; cut -c1-400 $O/${TAG}_bench_reference.json
bash tools/gpu_sanitize.sh $TAG > /dev/null 2>&1; grep -c "ERROR SUMMARY: 0 errors" $O/${TAG}_sanitizer.log; grep "RACECHECK SUMMARY" $O/${TAG}_sanitizer.log
timeout 600 ncu --metrics gpu__time_duration.sum --clock-control none -c 500 --csv --log-file $O/${TAG}_launches_gomoku.csv python tools/profile_target.py gomoku 3 1024 > /dev/null 2>&1
timeout 300 ncu --metrics gpu__time_duration.sum --clock-control none -c 200 --csv --log-file $O/${TAG}_launches_tictactoe.csv python tools/profile_target.py tictactoe 25 4096 > /dev/null 2>&1
python tools/launch_summary.py $O/${TAG}_launches_gomoku.csv $O/${TAG}_launches_gomoku.txt | head -12
python tools/launch_summary.py $O/${TAG}_launches_tictactoe.csv $O/${TAG}_launches_tictactoe.txt | head -8

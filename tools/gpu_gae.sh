#!/bin/bash
# The advantage pass's checks and measurements (DESIGN.md §4.11), on one GPU:
#   tools/gpu_gae.sh OUT_DIR
# -> OUT_DIR/r9_card.txt        the card's name, power limit and clock
#    OUT_DIR/r9_gae_tests.txt   tests/test_gpu_gae.py and tests/test_gae_cpu.py
#    OUT_DIR/r9_gae_time.jsonl  evg_gae against a same-size copy and the torch per-turn loop (tools/gae_time.py)
#    OUT_DIR/r9_gpu.txt         the whole test suite
out=$(realpath -m "${1:?usage: tools/gpu_gae.sh OUT_DIR}")
cd "$(dirname "$0")/.."
mkdir -p "$out"
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv > "$out"/r9_card.txt
python -c 'import __graft_entry__ as g; g.build()' 2>&1 | tail -1
python -m pytest tests/test_gpu_gae.py tests/test_gae_cpu.py -q -p no:cacheprovider > "$out"/r9_gae_tests.txt 2>&1
tail -1 "$out"/r9_gae_tests.txt
python tools/gae_time.py > "$out"/r9_gae_time.jsonl
python -m pytest tests -q -p no:cacheprovider > "$out"/r9_gpu.txt 2>&1
tail -1 "$out"/r9_gpu.txt

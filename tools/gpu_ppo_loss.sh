#!/bin/bash
# The fused PPO loss head's checks and measurements (DESIGN.md §4.12), on one GPU:
#   tools/gpu_ppo_loss.sh OUT_DIR [full]
# -> OUT_DIR/r10_card.txt            the card's name, power limit and clock
#    OUT_DIR/r10_ptxas.txt           -Xptxas -v of csrc/evg_ppo_loss.cu
#    OUT_DIR/r10_ppo_loss_tests.txt  tests/test_gpu_ppo_loss.py and tests/test_ppo_loss_cpu.py
#    OUT_DIR/r10_ppo_loss_time.jsonl the fused head against the torch statement (tools/ppo_loss_time.py)
#    OUT_DIR/r10_gpu.txt             with `full`: the whole test suite, then smoke() and bench.py (r10_smoke.txt, r10_bench.json)
out=$(realpath -m "${1:?usage: tools/gpu_ppo_loss.sh OUT_DIR [full]}")
cd "$(dirname "$0")/.."
mkdir -p "$out"
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv > "$out"/r10_card.txt
python -c 'import __graft_entry__ as g; g.build()' 2>&1 | tail -1
tmp=$(mktemp -d)
/usr/local/cuda/bin/nvcc -gencode arch=compute_100a,code=sm_100a -O3 -std=c++17 -Xptxas -v -c \
    everglades-ai-wargame_b200/csrc/evg_ppo_loss.cu -o "$tmp"/ppo_loss.o 2>&1 | grep -E "Compiling|Used|spill" > "$out"/r10_ptxas.txt
rm -rf "$tmp"
python -m pytest tests/test_gpu_ppo_loss.py tests/test_ppo_loss_cpu.py -q -p no:cacheprovider > "$out"/r10_ppo_loss_tests.txt 2>&1
tail -1 "$out"/r10_ppo_loss_tests.txt
python tools/ppo_loss_time.py > "$out"/r10_ppo_loss_time.jsonl 2>&1
tail -3 "$out"/r10_ppo_loss_time.jsonl
if [ "$2" = full ]; then
    python -m pytest tests -q -p no:cacheprovider > "$out"/r10_gpu.txt 2>&1
    tail -1 "$out"/r10_gpu.txt
    python -c 'import __graft_entry__ as g; g.smoke()' > "$out"/r10_smoke.txt 2>&1
    tail -2 "$out"/r10_smoke.txt
    python bench.py --gpus 1 --steps 450 --warmup 150 > "$out"/r10_bench.json 2> "$out"/r10_bench.log
    tail -c 600 "$out"/r10_bench.json
fi

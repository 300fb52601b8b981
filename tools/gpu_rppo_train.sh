#!/bin/bash
# The recurrent actor's update operation: checks and measurements (DESIGN.md §4.13), on one GPU:
#   tools/gpu_rppo_train.sh OUT_DIR [full]
# -> OUT_DIR/r11_card.txt              the card's name, power limit and clock
#    OUT_DIR/r11_ptxas.txt             -Xptxas -v of csrc/evg_rppo_train.cu and csrc/evg_policy_rppo.cu
#    OUT_DIR/r11_rppo_train_tests.txt  tests/test_gpu_rppo_train.py and tests/test_rppo_train_cpu.py
#    OUT_DIR/r11_rppo_update_time.jsonl, r11_rppo_profile.txt   tools/rppo_update_time.py (profile in its own pass)
#    OUT_DIR/r11_act_ab.jsonl          the acting kernel, this tree against the parent commit's package and library
#                                      staged under build/parent when present, alternated three times (tools/rppo_act_time.py)
#    with `full`: OUT_DIR/r11_gpu.txt (the whole suite), r11_smoke.txt, r11_bench_n1.json
out=$(realpath -m "${1:?usage: tools/gpu_rppo_train.sh OUT_DIR [full]}")
cd "$(dirname "$0")/.."
mkdir -p "$out"
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv > "$out"/r11_card.txt
python -c 'import __graft_entry__ as g; g.build()' 2>&1 | tail -1
tmp=$(mktemp -d)
for f in evg_rppo_train evg_policy_rppo; do
    /usr/local/cuda/bin/nvcc -gencode arch=compute_100a,code=sm_100a -O3 -std=c++17 -Xptxas -v -c \
        everglades-ai-wargame_b200/csrc/$f.cu -o "$tmp"/$f.o 2>&1 | grep -E "Compiling|Used|spill"
done > "$out"/r11_ptxas.txt
rm -rf "$tmp"
python -m pytest tests/test_gpu_rppo_train.py tests/test_rppo_train_cpu.py -q -p no:cacheprovider > "$out"/r11_rppo_train_tests.txt 2>&1
tail -1 "$out"/r11_rppo_train_tests.txt
python tools/rppo_update_time.py --out "$out"/r11_rppo_update_time.jsonl > /dev/null 2> "$out"/r11_rppo_update_time.log
cat "$out"/r11_rppo_update_time.jsonl; tail -2 "$out"/r11_rppo_update_time.log
python tools/rppo_update_time.py --reps 1 --profile "$out"/r11_rppo_profile.txt > /dev/null 2>&1
grep "^#" "$out"/r11_rppo_profile.txt
if [ -f build/parent/tools/rppo_act_time.py ]; then
    for i in 1 2 3; do
        python build/parent/tools/rppo_act_time.py
        python tools/rppo_act_time.py
    done > "$out"/r11_act_ab.jsonl 2>&1
    cat "$out"/r11_act_ab.jsonl
fi
if [ "$2" = full ]; then
    python -m pytest tests -q -p no:cacheprovider > "$out"/r11_gpu.txt 2>&1
    tail -1 "$out"/r11_gpu.txt
    python -c 'import __graft_entry__ as g; g.smoke()' > "$out"/r11_smoke.txt 2>&1
    tail -2 "$out"/r11_smoke.txt
    python bench.py --gpus 1 --steps 450 --warmup 150 > "$out"/r11_bench_n1.json 2> "$out"/r11_bench.log
    tail -c 600 "$out"/r11_bench_n1.json
fi

#!/bin/bash
# The feed-forward networks' update operation: checks and measurements (DESIGN.md §4.14), on one GPU:
#   tools/gpu_ppo_train.sh OUT_DIR [full]
# -> OUT_DIR/r13_card.txt              the card's name, power limit and clock
#    OUT_DIR/r13_ptxas.txt             -Xptxas -v of csrc/evg_ppo_train.cu and the acting kernels it mirrors
#    OUT_DIR/r13_ppo_train_tests.txt   tests/test_gpu_ppo_train.py and tests/test_ppo_train_cpu.py
#    OUT_DIR/r13_ppo_update_time.jsonl tools/ppo_update_time.py
#    with `full`: OUT_DIR/r13_gpu.txt (the whole suite), r13_smoke.txt, r13_bench_n1.json
out=$(realpath -m "${1:?usage: tools/gpu_ppo_train.sh OUT_DIR [full]}")
cd "$(dirname "$0")/.."
mkdir -p "$out"
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv > "$out"/r13_card.txt
python -c 'import __graft_entry__ as g; g.build()' 2>&1 | tail -1
tmp=$(mktemp -d)
for f in evg_ppo_train evg_policy_ppo evg_policy_value evg_policy_rppo; do
    /usr/local/cuda/bin/nvcc -gencode arch=compute_100a,code=sm_100a -O3 -std=c++17 -Xptxas -v -c \
        everglades-ai-wargame_b200/csrc/$f.cu -o "$tmp"/$f.o 2>&1 | grep -E "Compiling|Used|spill"
done > "$out"/r13_ptxas.txt
rm -rf "$tmp"
# stop at the first failure: nothing else runs after a failed check of the new kernels
python -m pytest tests/test_gpu_ppo_train.py tests/test_ppo_train_cpu.py -q -s -p no:cacheprovider -x 2>&1 | grep -v '^\[build\]' \
    > "$out"/r13_ppo_train_tests.txt
[ "${PIPESTATUS[0]}" = 0 ] || { tail -20 "$out"/r13_ppo_train_tests.txt; exit 1; }
tail -1 "$out"/r13_ppo_train_tests.txt
python tools/ppo_update_time.py --out "$out"/r13_ppo_update_time.jsonl > /dev/null 2> "$out"/r13_ppo_update_time.log \
    || { tail -20 "$out"/r13_ppo_update_time.log; exit 1; }
cat "$out"/r13_ppo_update_time.jsonl
# the fused step and kernels against the parent commit's (its package and library staged under build/parent), alternated
if [ -f build/parent/tools/ppo_update_time.py ]; then
    for i in 1 2; do
        python build/parent/tools/ppo_update_time.py --rows 1048576 65536 --out "$out"/r13_ab_parent_$i.jsonl > /dev/null 2>> "$out"/r13_ab.log
        python tools/ppo_update_time.py --rows 1048576 65536 --out "$out"/r13_ab_this_$i.jsonl > /dev/null 2>> "$out"/r13_ab.log
    done
    python - "$out" > "$out"/r13_ab.txt <<'PY'
import glob, json, sys
out, t = sys.argv[1], {}
for f in sorted(glob.glob(out + "/r13_ab_*_*.jsonl")):
    side = f.rsplit("/", 1)[1].split("_")[2]
    for line in open(f):
        d = json.loads(line)
        t.setdefault((d["rows"], d["latent"], d["case"]), {}).setdefault(side, []).append(d["ms"])
print("# ms per pass, parent | this tree, each of two alternated runs (the median of its passes)")
for (rows, L, case), v in sorted(t.items()):
    print("%8d %4d %-44s %s | %s" % (rows, L, case, v.get("parent"), v.get("this")))
PY
    cat "$out"/r13_ab.txt
fi
if [ "$2" = full ]; then
    python -m pytest tests -q -p no:cacheprovider > "$out"/r13_gpu.txt 2>&1 || { tail -5 "$out"/r13_gpu.txt; exit 1; }
    tail -1 "$out"/r13_gpu.txt
    python -c 'import __graft_entry__ as g; g.smoke()' > "$out"/r13_smoke.txt 2>&1
    tail -2 "$out"/r13_smoke.txt
    python bench.py --gpus 1 --steps 450 --warmup 150 > "$out"/r13_bench_n1.json 2> "$out"/r13_bench.log
    tail -c 600 "$out"/r13_bench_n1.json
fi

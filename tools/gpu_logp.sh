#!/bin/bash
# The measurements of the fused actors' log-probability and starting-state outputs (DESIGN.md §4.6, §4.7), on one GPU:
#   tools/gpu_logp.sh OUT_DIR [PARENT_TREE PARENT_LIB]
# -> OUT_DIR/r7_logp_time.jsonl         kernel times with none / logp / logp + hidden_in / probs (tools/logp_time.py)
#    OUT_DIR/r7_policy_rollout.jsonl    a CUDA-graph rollout turn at 32,768 matches, --want none / logp / probs
#    OUT_DIR/r7_ab_parent.jsonl         (with PARENT_TREE / PARENT_LIB) the call without the new outputs, the parent
#                                       commit's library against this one, alternating: PARENT_TREE's
#                                       tools/wire_policy_time.py run with EVGSIM_LIB set to each library in turn
# PARENT_TREE: a checkout of the parent commit; PARENT_LIB: its library (tools/build_variant.sh in that checkout).
out=$(realpath -m "${1:?usage: tools/gpu_logp.sh OUT_DIR [PARENT_TREE PARENT_LIB]}")
cd "$(dirname "$0")/.."
mkdir -p "$out"
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv > "$out"/r7_card.txt
python tools/logp_time.py --envs 32768 --reps 20 --rounds 3 > "$out"/r7_logp_time.jsonl
: > "$out"/r7_policy_rollout.jsonl
for policy in ppo rppo; do
    for want in none logp probs; do
        python tools/policy_rollout.py --fused --graph --policy $policy --want $want --envs-per-gpu 32768 >> "$out"/r7_policy_rollout.jsonl
    done
done
if [ -n "$3" ]; then
    : > "$out"/r7_ab_parent.jsonl
    for round in 1 2 3; do
        for lib in "$3" "$PWD/everglades-ai-wargame_b200/libevgsim.so"; do
            EVGSIM_LIB=$lib python "$2/tools/wire_policy_time.py" --envs 32768 --reps 20 \
                | python -c 'import json, sys; [print(json.dumps(dict(json.loads(l), lib=sys.argv[1], round=int(sys.argv[2])))) for l in sys.stdin if "evg_policy_" in l and "ppo" in l]' \
                "$(basename "$lib")" $round >> "$out"/r7_ab_parent.jsonl
        done
    done
fi

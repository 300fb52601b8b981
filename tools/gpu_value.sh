#!/bin/bash
# The fused critic's checks and measurements (DESIGN.md §4.10), on one GPU:
#   tools/gpu_value.sh OUT_DIR
# -> OUT_DIR/r8_card.txt                       the card's name, power limit and clock
#    OUT_DIR/r8_gpu.txt                        the GPU test suite (pytest -m gpu)
#    OUT_DIR/r8_value_time.jsonl               evg_policy_value against torch's fp32 / bf16 forward (tools/value_time.py)
#    OUT_DIR/r8_policy_rollout_value.jsonl     the PPO turn with a value per turn: no critic, torch bf16, fused; eager
#                                              and CUDA graph (tools/policy_rollout.py --critic)
out=$(realpath -m "${1:?usage: tools/gpu_value.sh OUT_DIR}")
cd "$(dirname "$0")/.."
mkdir -p "$out"
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv > "$out"/r8_card.txt
python -c 'import __graft_entry__ as g; g.build()' 2>&1 | tail -1
python -m pytest tests -q -m gpu -p no:cacheprovider > "$out"/r8_gpu.txt 2>&1
tail -1 "$out"/r8_gpu.txt
: > "$out"/r8_value_time.jsonl
for n in 32768 1048576; do
    for latent in 128 248; do
        python tools/value_time.py $n $latent >> "$out"/r8_value_time.jsonl
    done
done
: > "$out"/r8_policy_rollout_value.jsonl
for graph in "" --graph; do
    for critic in none torch fused; do
        python tools/policy_rollout.py --fused --policy ppo --want logp --critic $critic --envs-per-gpu 32768 $graph >> "$out"/r8_policy_rollout_value.jsonl
    done
done

#!/usr/bin/env python
"""BASELINE.json configs[3]: PyTorch policy-in-the-loop self-play rollout.

    python tools/policy_rollout.py [--envs-per-gpu 32768] [--turns 300] [--policy dqn|ppo|rppo] [--dtype fp32|bf16] [--graph]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node 8 --master-addr 127.0.0.1 tools/policy_rollout.py

Both players are driven by one network of the reference's shape — DQN: Linear(105, 528) - ReLU - Linear(528, 132)
(agents/DQN/QNetwork.py:37-42, random weights), decoded like DQNAgent.filter_actions (evg_decode_dqn); PPO: the
actor's Linear(105, 128) - Tanh - Linear(128, 128) - Tanh - Linear(128, 132) - Tanh - Softmax head
(agents/PPO/ActorCritic.py:33-50, without the GRU), 7 indices sampled without replacement and unravelled like
PPOAgent.get_action (evg_decode_indices); RPPO: the same head, its output repeated 7 times through the actor's
GRU(128, 128) (hidden state carried over the 7 steps and from turn to turn, zeroed when a match ends), one index
sampled per step (ActorCritic.act with use_recurrent, agents/PPO/ActorCritic.py:79-105).  --graph captures the whole
turn (forward, sampling, decode, step) in a CUDA graph.  The observation tensor the step kernel writes is consumed in place
(a [N*2, 105] view, no copy, no dtype conversion kernel for fp32); the decoded int8 rows go straight back into the
step.  --fused runs the network in libevgsim's tcgen05 kernels instead of torch: DQN's forward in evg_policy_mlp (then
evg_decode_dqn), PPO's forward, sampling and unravel in evg_policy_ppo, the recurrent actor's head, GRU steps, draws
and unravel in evg_policy_rppo, which also carries the hidden state and zeroes it when a match starts over (their draws
come from the simulator's tape, not from torch's generator).  --obs wire (with --fused) steps the simulator in the wire
format and the fused kernel reads those rows (128 B per match instead of 840); --opponent puts a scripted agent
(env.agent_actions) on player 1's side, the fused network plays player 0.  --critic adds PPO's critic
(Linear(105, 128) - Tanh - Linear(128, 128) - Tanh - Linear(128, 1), ActorCritic's value_layer) evaluated on every turn's
observations, the value a PPO rollout stores next to the draws: in torch (bf16 forward, float32 observations) or fused
(evg_policy_value, on the same rows the actor read).  Matches shard over the ranks with no collective on the path; rank 0 prints one JSON line.
"""
import argparse
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import evgsim


class RecurrentActor(torch.nn.Module):
    """ActorCritic's actor with use_recurrent=True (agents/PPO/ActorCritic.py:33-50,79-105), batched over (match, player)."""

    def __init__(self, n_latent=128):
        super().__init__()
        self.action_head = torch.nn.Sequential(torch.nn.Linear(105, n_latent), torch.nn.Tanh(), torch.nn.Linear(n_latent, n_latent), torch.nn.Tanh())
        self.action_gru = torch.nn.GRU(n_latent, n_latent, batch_first=False)
        self.action_layer = torch.nn.Sequential(torch.nn.Linear(n_latent, 132), torch.nn.Tanh(), torch.nn.Softmax(dim=-1))

    def forward(self, x, hidden):
        h = self.action_head(x)                                   # [B, 128]
        seq, hidden = self.action_gru(h.unsqueeze(0).expand(7, -1, -1).contiguous(), hidden)  # the observation repeated for the 7 actions
        return self.action_layer(seq), hidden                     # [7, B, 132], [1, B, 128]


def build_policy(kind, dtype, device, seed=0):
    torch.manual_seed(seed)
    if kind == "dqn":
        net = torch.nn.Sequential(torch.nn.Linear(105, 528), torch.nn.ReLU(), torch.nn.Linear(528, 132))
    elif kind == "rppo":
        net = RecurrentActor()
    else:
        net = torch.nn.Sequential(torch.nn.Linear(105, 128), torch.nn.Tanh(), torch.nn.Linear(128, 128), torch.nn.Tanh(),
                                  torch.nn.Linear(128, 132), torch.nn.Tanh(), torch.nn.Softmax(dim=-1))
    return net.to(device=device, dtype=dtype).eval()


@torch.no_grad()
def policy_actions(env, net, kind, dtype, hidden=None):
    x = env.obs.view(-1, env.obs_len)  # [N*2, 105], the step kernel's output buffer itself
    x = x if dtype == torch.float32 else x.to(dtype)
    if kind == "rppo":
        probs, h = net(x, hidden)
        hidden.copy_(h)
        idx = torch.multinomial(probs.float().view(-1, 132), 1).view(7, env.num_envs, 2).permute(1, 2, 0).contiguous()
        return env.decode_indices(idx, div=12, mod=11)
    out = net(x)
    if kind == "dqn":
        return env.decode_dqn(out.float().view(env.num_envs, 2, -1))
    idx = torch.multinomial(out.float(), 7, replacement=False)  # PPOAgent.get_action draws 7 distinct flat indices
    return env.decode_indices(idx.view(env.num_envs, 2, 7), div=12, mod=11)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs-per-gpu", type=int, default=32768)  # 262,144 over 8 GPUs
    ap.add_argument("--turns", type=int, default=300)
    ap.add_argument("--warmup", type=int, default=150)
    ap.add_argument("--policy", default="dqn", choices=["dqn", "ppo", "rppo"])
    ap.add_argument("--dtype", default="fp32", choices=["fp32", "bf16"])
    ap.add_argument("--graph", action="store_true", help="replay the turn (forward, decode, step) from a CUDA graph")
    ap.add_argument("--fused", action="store_true",
                    help="the policy runs in libevgsim's fused tcgen05 kernels (evg_policy_mlp / evg_policy_ppo / evg_policy_rppo, bf16 operands) instead of torch")
    ap.add_argument("--obs", default="f32", choices=["f32", "wire"], help="observation format of the step and the fused policy's input")
    ap.add_argument("--opponent", default="none", choices=["none", "random", "base_rush", "swarm"],
                    help="with --fused: a scripted agent plays player 1, the network player 0")
    ap.add_argument("--want", default="none", choices=["none", "logp", "probs"],
                    help="with --fused --policy ppo|rppo: what a PPO rollout keeps of each turn besides the draws: nothing, each "
                         "draw's log-probability (and for rppo the starting state, hidden_in), or the whole distribution")
    ap.add_argument("--critic", default="none", choices=["none", "torch", "fused"],
                    help="with --fused --policy ppo|rppo: the state value of every row each turn, from a torch bf16 critic or "
                         "evg_policy_value")
    args = ap.parse_args()
    if (args.obs == "wire" or args.opponent != "none") and not args.fused:
        ap.error("--obs wire and --opponent need --fused")
    if args.want != "none" and not (args.fused and args.policy in ("ppo", "rppo")):
        ap.error("--want needs --fused and --policy ppo or rppo")
    if args.critic != "none" and not (args.fused and args.policy in ("ppo", "rppo")):
        ap.error("--critic needs --fused and --policy ppo or rppo")
    if args.critic == "torch" and args.obs != "f32":
        ap.error("--critic torch reads the float32 observations (--obs f32)")
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if world > 1:
        torch.distributed.init_process_group("nccl", device_id=torch.device("cuda", local))
    dtype = torch.float32 if args.dtype == "fp32" else torch.bfloat16
    E = args.envs_per_gpu
    first, _ = evgsim.shard_range(E * world, rank, world)
    env = evgsim.BatchedEvergladesEnv(E, device=local, seed=0, auto_reset=evgsim._capi.AUTORESET_TERMINAL, env_id_offset=first)
    net = build_policy(args.policy, dtype, env.device)
    env.reset(obs_format=args.obs)
    hidden = torch.zeros((1, 2 * E, 128), dtype=dtype, device=env.device) if args.policy == "rppo" and not args.fused else None

    fused = None
    if args.fused:  # the recurrent actor's kernel keeps its own state (fused.hidden) and resets it at turn 0
        from evgsim import policy as evp
        cls = {"dqn": evp.FusedDQN, "ppo": evp.FusedPPO, "rppo": evp.FusedRPPO}[args.policy]
        fused = cls(env, net.float()) if args.policy == "dqn" or args.opponent == "none" else cls(env, net.float(), player=0)
    opponent = {"none": None, "random": evgsim._capi.AGENT_RANDOM, "base_rush": evgsim._capi.AGENT_BASE_RUSH,
                "swarm": evgsim._capi.AGENT_SWARM}[args.opponent]

    critic_net = value = critic = None
    if args.critic != "none":
        torch.manual_seed(1)
        critic_net = torch.nn.Sequential(torch.nn.Linear(105, 128), torch.nn.Tanh(), torch.nn.Linear(128, 128), torch.nn.Tanh(),
                                         torch.nn.Linear(128, 1)).to(env.device).eval()
        if args.critic == "fused":
            from evgsim import policy as evp
            critic = evp.FusedValue(env, critic_net)
        else:
            critic_net = critic_net.to(torch.bfloat16)
            value = torch.empty((E, 2), dtype=torch.float32, device=env.device)

    want = {"none": {}, "probs": {"want_probs": True},
            "logp": {"want_logp": True, **({"want_hidden_in": True} if args.policy == "rppo" else {})}}[args.want]

    def turn():
        if fused is None:
            env.step(policy_actions(env, net, args.policy, dtype, hidden))
        else:
            actions = fused(obs_format=args.obs, **want)
            if critic is not None:  # V of the rows the actor read, into critic.value
                critic(obs_format=args.obs)
            elif value is not None:
                with torch.no_grad():
                    value.copy_(critic_net(env.obs.view(-1, env.obs_len).to(torch.bfloat16)).float().view(E, 2))
            if opponent is not None:  # player 1's rows from the scripted agent, player 0's from the network
                env.agent_actions(evgsim._capi.AGENT_EXTERNAL, opponent)
            env.step(actions, obs_format=args.obs)
        if hidden is not None:  # a finished match starts over with a fresh hidden state
            hidden.mul_((1 - env.done).to(dtype).repeat_interleave(2).view(1, -1, 1))

    run = turn
    if args.graph:
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            for _ in range(3):
                turn()
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g, stream=side):
                turn()
        torch.cuda.current_stream().wait_stream(side)
        run = g.replay
    for _ in range(args.warmup):
        run()
    torch.cuda.synchronize()
    if world > 1:
        torch.distributed.barrier()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(args.turns):
        run()
    b.record()
    torch.cuda.synchronize()
    ms = torch.tensor([a.elapsed_time(b)], dtype=torch.float64, device=env.device)
    if world > 1:
        torch.distributed.all_reduce(ms, op=torch.distributed.ReduceOp.MAX)
    stats = evgsim.gather_episode_stats(env.episode_stats(), device=env.device) if world > 1 else env.episode_stats()
    if rank == 0:
        sec = float(ms.item()) / 1e3
        print(json.dumps({"workload": "policy-in-the-loop self-play (BASELINE.json configs[3])", "policy": args.policy, "dtype": "bf16 operands, fp32 accumulate (%s)" % {"dqn": "evg_policy_mlp", "ppo": "evg_policy_ppo", "rppo": "evg_policy_rppo"}[args.policy] if args.fused else args.dtype, "fused_forward": bool(args.fused), "obs_format": args.obs, "opponent": args.opponent,
                          "cuda_graph": bool(args.graph), "want": args.want, "critic": args.critic,
                          "n_gpus": world, "envs_per_gpu": E, "turns": args.turns, "env_turns_per_s": E * world * args.turns / sec,
                          "ms_per_turn": sec * 1e3 / args.turns, "episodes": stats["episodes"], "wins": stats["wins"], "ties": stats["ties"]}))
    if world > 1:
        torch.distributed.destroy_process_group()


if __name__ == "__main__":
    main()

#!/usr/bin/env python
"""Time of the advantage pass (evg_gae, BatchedEvergladesEnv.gae) on a stored rollout, against a same-size copy and the
torch per-turn loop a training script would otherwise run.  One JSON line per case:
M in {4,096, 32,768, 262,144} matches, T in {64, 128} turns, rewards and done flags from the wire rows or float tensors.

- Inputs: T+1 wire rows of a real rollout (random self-play under AUTORESET_TERMINAL, after 30 warm-up turns) and random
  float32 values [T+1, M, 2]; the float source is the rows' rewards and done flags as float32 [T, M, 2] / uint8 [T, M].
- Every timed pass is one CUDA event pair after a 256 MB buffer is overwritten, so no pass finds its inputs in the
  126 MB L2; the median of `reps` passes after 3 warm-up passes is reported.
- bytes: what the pass must move, from the shapes: per match-turn 64 B of row sectors (word 0 and the rewards: two
  32-byte sectors of a row), 8 B of values and 16 B of outputs from wire rows (88 B), or 8 + 8 + 1 + 16 = 33 B from
  float tensors, plus the bootstrap values (8 B per match).  GB/s = bytes over the kernel's time.
- copy_us: a device-to-device copy of bytes / 2 (so that it reads and writes the pass's bytes), timed the same way.
- torch_*_us: the textbook GAE as a loop over the T turns in torch (float32, 8 small kernels a turn), eager and replayed from a
  CUDA graph; for the wire source preceded by torch's extraction of rewards and done flags from the rows (a strided
  copy each).  expand_wire would also write the observations (840 B per match on DemoMap), so it is not the baseline.

    python tools/gae_time.py [reps=20]
"""
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import torch
import evgsim
from ppo_time import gpu_info

GAMMA, LAM = 0.99, 0.95


def timed_us(fn, flush, reps):
    for _ in range(3):
        fn()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(reps)]
    for a, b in ev:
        flush.add_(1)
        a.record()
        fn()
        b.record()
    torch.cuda.synchronize()
    return sorted(a.elapsed_time(b) for a, b in ev)[reps // 2] * 1e3


def torch_gae(values, reward, done, adv, ret):
    T = reward.shape[0]
    nd = (1 - done.float()).unsqueeze(-1)
    a = torch.zeros_like(values[0])
    for t in range(T - 1, -1, -1):
        a = reward[t] + GAMMA * values[t + 1] * nd[t] - values[t] + (GAMMA * LAM) * nd[t] * a
        adv[t] = a
    torch.add(adv, values[:-1], out=ret)


def graphed(fn):
    fn()
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        fn()
    return g.replay


def main():
    reps = int(sys.argv[1]) if len(sys.argv) > 1 else 20
    gpu = gpu_info()
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    for M in (4096, 32768, 262144):
        env = evgsim.BatchedEvergladesEnv(M, seed=0, auto_reset=evgsim._capi.AUTORESET_TERMINAL)
        env.reset(obs_format="wire")
        for _ in range(30):
            env.step(env.random_actions(), obs_format="wire")
        rb = int(env._lib.evg_obs_row_bytes(env._h, evgsim._capi.OBS_WIRE))
        roff = evgsim._capi.WIRE_NODE0 + 4 * env.num_nodes + 3 * 2 * evgsim._capi.NUM_GROUPS
        for T in (64, 128):
            rows = torch.empty((T + 1, M, rb), dtype=torch.uint8, device=env.device)
            rows[0].copy_(env.obs_rows("wire"))
            for t in range(T):
                env.step(env.random_actions(), obs_format="wire")
                rows[t + 1].copy_(env.obs_rows("wire"))
            gen = torch.Generator(device=env.device).manual_seed(T)
            values = torch.randn((T + 1, M, 2), device=env.device, generator=gen)
            reward = rows[1:, :, roff:roff + 8].contiguous().view(torch.float32)
            done = rows[1:, :, 2].contiguous()
            adv, ret = torch.empty((T, M, 2), device=env.device), torch.empty((T, M, 2), device=env.device)
            adv_t, ret_t = torch.empty_like(adv), torch.empty_like(adv)
            env.gae(values, rows=rows, gamma=GAMMA, lam=LAM, adv=adv, ret=ret)
            a_w = adv.clone()
            env.gae(values, reward=reward, done=done, gamma=GAMMA, lam=LAM, adv=adv, ret=ret)
            assert torch.equal(adv, a_w), "wire and float sources disagree"
            torch_gae(values, reward, done, adv_t, ret_t)
            diff = (adv_t - adv).abs().max().item()
            for src in ("wire", "float"):
                per = 88 if src == "wire" else 33
                nbytes = M * T * per + M * 8
                if src == "wire":
                    def kernel():
                        env.gae(values, rows=rows, gamma=GAMMA, lam=LAM, adv=adv, ret=ret)

                    def baseline():
                        r = rows[1:, :, roff:roff + 8].contiguous().view(torch.float32)
                        d = rows[1:, :, 2].contiguous()
                        torch_gae(values, r, d, adv_t, ret_t)
                else:
                    def kernel():
                        env.gae(values, reward=reward, done=done, gamma=GAMMA, lam=LAM, adv=adv, ret=ret)

                    def baseline():
                        torch_gae(values, reward, done, adv_t, ret_t)
                src_buf = torch.empty(nbytes // 2, dtype=torch.uint8, device=env.device)
                dst_buf = torch.empty_like(src_buf)
                us = timed_us(kernel, flush, reps)
                out = {"gpu": gpu, "matches": M, "turns": T, "source": src, "gae_us": round(us, 2), "bytes": nbytes,
                       "gae_GBps": round(nbytes / us / 1e3, 1), "copy_us": round(timed_us(lambda: dst_buf.copy_(src_buf), flush, reps), 2),
                       "torch_eager_us": round(timed_us(baseline, flush, max(5, reps // 4)), 1),
                       "torch_graph_us": round(timed_us(graphed(baseline), flush, reps), 1),
                       "max_abs_diff_vs_torch": diff}
                print(json.dumps(out), flush=True)
                del src_buf, dst_buf
            del rows, values, reward, done, adv, ret, adv_t, ret_t
            torch.cuda.empty_cache()
        env.close()


if __name__ == "__main__":
    main()

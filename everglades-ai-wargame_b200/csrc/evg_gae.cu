// evg_gae.cu — PPO's advantages and returns of a stored rollout, GAE(lambda), in one launch (include/evgsim.h, evg_gae).
//
// One thread per match walks t = T-1 ... 0 and carries A_{t+1} and V_{t+1} in registers; for player -1 it carries both
// columns, so values, advantages and returns move as float2 and the two rewards are read together.  Consecutive threads
// take consecutive matches, so every per-turn access of a warp is one contiguous span (256 B of values, 256 B of each
// output for player -1); the wire rows are the exception, where a warp reads word 0 (the done byte) and the reward words
// of 32 rows, two 32-byte sectors of each.
//
// The pass is a chain of T dependent steps per thread, and at the sizes a training loop runs there are few threads: at
// 32,768 matches about 7 warps per SM.  The loads do not depend on the recurrence, so each batch of kGaeBatch turns issues
// all its loads (values, rewards, done flags) before the batch's arithmetic: per thread that is 16 x 17 B of float
// tensors or 16 x 72 B of row sectors and values in flight, against the ~50 KB per SM that the HBM's bandwidth-latency
// product asks for (7 warps x 32 threads x 272 B = 61 KB).  The recurrence itself stays strictly sequential in t, each
// operation rounded on its own (no FMA contraction), so the result is bit for bit tests/ppo_gae.py's reference_gae.
#include <type_traits>

#include "evg_internal.h"

namespace evg {

namespace {

constexpr int kGaeBatch = 16;    // turns whose loads are issued together
constexpr int kGaeThreads = 32;  // one warp per CTA, see launch_gae

struct GaeArgs {
    const uint32_t* rows;  // wire rows [T+1][M][words], or null when reward and done are both given
    const float* reward;   // [T][M][2] or null
    const uint8_t* done;   // [T][M] or null
    const float* values;   // [T+1][M][cols]
    float* adv;            // [T][M][cols]
    float* ret;
    int64_t n_matches;
    int32_t n_turns, words, reward_word, player;
    float gamma, lam;
};

// one column's step of the recurrence, include/evgsim.h's definition operation by operation
__device__ __forceinline__ float gae_step(float r, bool d, float v, float& vn, float& an, float gamma, float gl, float& ret)
{
    const float nv = d ? 0.f : vn, na = d ? 0.f : an;
    const float delta = __fsub_rn(__fadd_rn(r, __fmul_rn(gamma, nv)), v);
    const float a = __fadd_rn(delta, __fmul_rn(gl, na));
    ret = __fadd_rn(a, v);
    vn = v;
    an = a;
    return a;
}

__device__ __forceinline__ float2 ld_col(const float2* p) { return __ldg(p); }
__device__ __forceinline__ float ld_col(const float* p) { return __ldg(p); }

// kBoth: both players' columns (player -1), values and outputs as float2; else the one column of args.player
template <bool kBoth>
__global__ void __launch_bounds__(kGaeThreads) evg_gae_kernel(const __grid_constant__ GaeArgs g)
{
    using Col = typename std::conditional<kBoth, float2, float>::type;
    const int64_t m = (int64_t)blockIdx.x * kGaeThreads + threadIdx.x, M = g.n_matches;
    if (m >= M) return;
    const Col* values = reinterpret_cast<const Col*>(g.values) + m;
    Col* adv = reinterpret_cast<Col*>(g.adv) + m;
    Col* ret = reinterpret_cast<Col*>(g.ret) + m;
    const int p = kBoth ? 0 : g.player;
    const float gl = __fmul_rn(g.gamma, g.lam);
    Col vn = ld_col(values + g.n_turns * M), an;  // V_T, the bootstrap state, and A_T = 0
    if constexpr (kBoth) an = make_float2(0.f, 0.f);
    else an = 0.f;
#pragma unroll 1
    for (int t0 = g.n_turns - 1; t0 >= 0; t0 -= kGaeBatch) {
        Col v[kGaeBatch];
        float r0[kGaeBatch], r1[kGaeBatch];
        uint32_t d[kGaeBatch];
#pragma unroll
        for (int j = 0; j < kGaeBatch; ++j) {
            const int t = t0 - j;
            if (t < 0) break;
            const int64_t i = t * M + m;  // (turn t, match m); row t + 1 holds turn t's reward and done
            v[j] = ld_col(values + t * M);
            const uint32_t* row = g.rows + (i + M) * g.words;
            if (g.reward) {
                if constexpr (kBoth) {
                    const float2 r = __ldg(reinterpret_cast<const float2*>(g.reward) + i);
                    r0[j] = r.x, r1[j] = r.y;
                } else {
                    r0[j] = __ldg(g.reward + 2 * i + p);
                }
            } else {  // the reward pair is 4-byte aligned only: two word loads from the same sector
                r0[j] = __uint_as_float(__ldg(row + g.reward_word + p));
                if constexpr (kBoth) r1[j] = __uint_as_float(__ldg(row + g.reward_word + 1));
            }
            d[j] = g.done ? (uint32_t)__ldg(g.done + i) : (__ldg(row) >> 16) & 0xFFu;
        }
#pragma unroll
        for (int j = 0; j < kGaeBatch; ++j) {
            const int t = t0 - j;
            if (t < 0) break;
            Col a, rt;
            if constexpr (kBoth) {
                a.x = gae_step(r0[j], d[j] != 0, v[j].x, vn.x, an.x, g.gamma, gl, rt.x);
                a.y = gae_step(r1[j], d[j] != 0, v[j].y, vn.y, an.y, g.gamma, gl, rt.y);
            } else {
                a = gae_step(r0[j], d[j] != 0, v[j], vn, an, g.gamma, gl, rt);
            }
            adv[t * M] = a;
            ret[t * M] = rt;
        }
    }
}

}  // namespace

// Blocks of one warp: a thread's batch of loads takes ~100 registers (kGaeBatch turns of values, rewards and done), so
// registers, not the 32-CTA limit of an SM, bound the resident warps (18 per SM at 110 registers for both players, 28 at
// 71 for one), and the smallest CTA spreads a small rollout over the most SMs (4,096 matches: 128 SMs instead of the 32
// that 128-thread CTAs would use).
cudaError_t launch_gae(int n_turns, int64_t n_matches, int player, const uint32_t* rows, int words, int reward_word, const float* reward,
                       const uint8_t* done, const float* values, float gamma, float lam, float* adv, float* ret, cudaStream_t stream)
{
    const GaeArgs g{rows, reward, done, values, adv, ret, n_matches, n_turns, words, reward_word, player, gamma, lam};
    const unsigned blocks = (unsigned)((n_matches + kGaeThreads - 1) / kGaeThreads);
    if (player < 0) evg_gae_kernel<true><<<blocks, kGaeThreads, 0, stream>>>(g);
    else evg_gae_kernel<false><<<blocks, kGaeThreads, 0, stream>>>(g);
    return cudaGetLastError();
}

}  // namespace evg

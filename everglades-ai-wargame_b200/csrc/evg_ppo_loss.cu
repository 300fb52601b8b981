// evg_ppo_loss.cu — PPO's policy loss from the actor's last Linear output z: each stored draw's log-probability, the
// entropy and the clipped surrogate, and their gradient with respect to z (include/evgsim.h, evg_ppo_loss /
// evg_ppo_loss_grad; DESIGN.md §4.12).
//
// A warp holds one distribution (a row's z for K = 1, one of its seven for K = 7): lane l owns elements l + 32 s,
// s = 0 .. 7 (n <= 256), loaded as coalesced 4-byte words, so every warp-wide load is one 128-byte line whatever n is
// (n = 7 .. 256 includes widths whose rows are not 16-byte aligned).  Every sum over the n elements is the lane's
// ascending sum over s followed by the xor butterfly 16, 8, 4, 2, 1, so all lanes hold the same value and
// tests/ppo_loss.py restates the order.  The backward recomputes y, p, S, T and H from z with the forward's code, and
// reads only the forward's ratio of the row: per row it reads z once and writes dz once.
#include "evg_internal.h"

namespace evg {

namespace {

constexpr int kDraws = 7;
constexpr int kSlots = 8;  // elements per lane: n <= 256
constexpr unsigned kFull = 0xffffffffu;
constexpr int kWarps = 8;  // warps per CTA, except the K = 7 forward (seven: one row per CTA and pass)

struct LossArgs {
    const float* z;         // [B][K][n]
    const int64_t* idx;     // [B][7]
    const float* old_logp;  // [B][7] (forward)
    const float* adv;       // [B]
    const float* ratio_in;  // [B] (backward)
    const float* g_surr;    // [B] or null (backward)
    const float* g_ent;     // [B] or null (backward)
    float* surr;            // [B] (forward)
    float* ent;
    float* logp;            // [B][7]
    float* ratio;           // [B]
    float* dz;              // [B][K][n] (backward)
    int64_t n_rows;
    int n;
    float lo, hi;           // fl(1 - clip), fl(1 + clip)
};

__device__ __forceinline__ float warp_sum(float v)
{
#pragma unroll
    for (int s = 16; s; s >>= 1) v += __shfl_xor_sync(kFull, v, s);
    return v;
}

// One distribution's values in the warp: y = tanh(z), p = e^y / S, lp = y - log S, H = -sum p lp.
struct Dist {
    float y[kSlots], p[kSlots];
    float L, H;
};

__device__ __forceinline__ void load_dist(const float* __restrict__ zr, int n, int lane, Dist& d)
{
    // slots past n are skipped whole (the test is warp-uniform); a lane's elements past n hold y = p = 0, which add
    // nothing to any sum
    float x[kSlots];
#pragma unroll
    for (int s = 0; s < kSlots; ++s) {  // all loads before any arithmetic
        const int m = lane + 32 * s;
        x[s] = 0.f;
        if (32 * s < n && m < n) x[s] = __ldg(zr + m);
    }
    float se = 0.f;
#pragma unroll
    for (int s = 0; s < kSlots; ++s) {
        d.y[s] = d.p[s] = 0.f;
        if (32 * s < n) {
            d.y[s] = tanhf(x[s]);
            d.p[s] = lane + 32 * s < n ? expf(d.y[s]) : 0.f;  // e until S is known
            se += d.p[s];
        }
    }
    const float S = warp_sum(se);
    d.L = logf(S);
    float sh = 0.f;
#pragma unroll
    for (int s = 0; s < kSlots; ++s) {
        if (32 * s < n) {
            d.p[s] = d.p[s] / S;
            sh += d.p[s] * (d.y[s] - d.L);  // p = 0 past n
        }
    }
    d.H = -warp_sum(sh);
}

// y of element j (warp-uniform, 0 <= j < n) from the lane that owns it
__device__ __forceinline__ float y_of(const Dist& d, int j, int lane)
{
    float v = 0.f;  // a select per slot, not d.y[j >> 5], which would put d.y in local memory
#pragma unroll
    for (int s = 0; s < kSlots; ++s) v = lane + 32 * s == j ? d.y[s] : v;
    return __shfl_sync(kFull, v, j & 31);
}

// the row's seven draws in every lane; true when one lies outside [0, n)
__device__ __forceinline__ bool load_draws(const int64_t* __restrict__ idx, int64_t b, int n, int lane, int (&j)[kDraws])
{
    const int64_t mine = lane < kDraws ? __ldg(idx + b * kDraws + lane) : 0;
    const bool bad = __any_sync(kFull, mine < 0 || mine >= n);
    const int c = mine < 0 || mine >= n ? 0 : (int)mine;  // a bad row reads nothing out of bounds
#pragma unroll
    for (int k = 0; k < kDraws; ++k) j[k] = __shfl_sync(kFull, c, k);
    return bad;
}

// K = 1: T_k = sum of p over the elements not drawn before k (first draw index of the element >= k), in the warp order
__device__ __forceinline__ void totals_wo_replacement(const Dist& d, const int (&j)[kDraws], int n, int lane, int (&first)[kSlots],
                                                      float (&T)[kDraws])
{
#pragma unroll
    for (int s = 0; s < kSlots; ++s) {
        const int m = lane + 32 * s;
        first[s] = kDraws;
#pragma unroll
        for (int k = kDraws - 1; k >= 0; --k)
            if (j[k] == m) first[s] = k;
    }
#pragma unroll
    for (int k = 0; k < kDraws; ++k) {
        float t = 0.f;
#pragma unroll
        for (int s = 0; s < kSlots; ++s)
            if (32 * s < n) t += first[s] >= k ? d.p[s] : 0.f;
        T[k] = warp_sum(t);
    }
}

__device__ __forceinline__ float total(const Dist& d, int n)
{
    float t = 0.f;
#pragma unroll
    for (int s = 0; s < kSlots; ++s)
        if (32 * s < n) t += d.p[s];
    return warp_sum(t);
}

// the surrogate and the ratio from the seven log-probabilities and the stored ones (every lane holds ell; lane k < 7
// holds old_logp[k] in `old`)
__device__ __forceinline__ void finish_row(const LossArgs& g, int64_t b, int lane, float ell, float old, float ent, bool bad)
{
    float ell_old = 0.f;
#pragma unroll
    for (int k = 0; k < kDraws; ++k) ell_old += __shfl_sync(kFull, old, k);
    if (lane == 0) {
        const float A = __ldg(g.adv + b);
        const float r = expf(ell - ell_old);
        const float c = fminf(fmaxf(r, g.lo), g.hi);
        const float s = -fminf(r * A, c * A);
        const float nan = __int_as_float(0x7fc00000);
        g.surr[b] = bad ? nan : s;
        g.ent[b] = bad ? nan : ent;
        g.ratio[b] = bad ? nan : r;
    }
}

// K = 1: a warp per row, rows strided over the grid's warps
__global__ void __launch_bounds__(kWarps * 32) evg_ppo_loss_fwd1_kernel(const __grid_constant__ LossArgs g)
{
    const int lane = threadIdx.x & 31;
    const int64_t stride = (int64_t)gridDim.x * kWarps;
    for (int64_t b = (int64_t)blockIdx.x * kWarps + (threadIdx.x >> 5); b < g.n_rows; b += stride) {
        int j[kDraws];
        const bool bad = load_draws(g.idx, b, g.n, lane, j);
        const float old = lane < kDraws ? __ldg(g.old_logp + b * kDraws + lane) : 0.f;
        Dist d;
        load_dist(g.z + b * g.n, g.n, lane, d);
        int first[kSlots];
        float T[kDraws];
        totals_wo_replacement(d, j, g.n, lane, first, T);
        float ell = 0.f, mine = 0.f;
#pragma unroll
        for (int k = 0; k < kDraws; ++k) {
            const float lk = (y_of(d, j[k], lane) - d.L) - logf(T[k]);
            ell += lk;
            if (lane == k) mine = lk;
        }
        if (lane < kDraws) g.logp[b * kDraws + lane] = bad ? __int_as_float(0x7fc00000) : mine;
        finish_row(g, b, lane, ell, old, d.H, bad);
    }
}

// K = 7: a CTA of seven warps per row, warp k on distribution k, rows strided over the grid; the row's seven logp_k and
// H_k meet in shared memory (double-buffered, so one barrier a row)
__global__ void __launch_bounds__(kDraws * 32, 4) evg_ppo_loss_fwd7_kernel(const __grid_constant__ LossArgs g)
{
    __shared__ float s_lp[2][kDraws], s_h[2][kDraws];
    const int lane = threadIdx.x & 31, k = threadIdx.x >> 5;
    int buf = 0;
    for (int64_t b = blockIdx.x; b < g.n_rows; b += gridDim.x, buf ^= 1) {
        int j[kDraws];
        const bool bad = load_draws(g.idx, b, g.n, lane, j);
        const float old = k == 0 && lane < kDraws ? __ldg(g.old_logp + b * kDraws + lane) : 0.f;
        Dist d;
        load_dist(g.z + (b * kDraws + k) * g.n, g.n, lane, d);
        const float T = total(d, g.n);
        const float lk = (y_of(d, j[k], lane) - d.L) - logf(T);
        if (lane == 0) {
            s_lp[buf][k] = lk;
            s_h[buf][k] = d.H;
            g.logp[b * kDraws + k] = bad ? __int_as_float(0x7fc00000) : lk;
        }
        __syncthreads();
        if (k == 0) {
            float ell = 0.f, hs = 0.f;
#pragma unroll
            for (int q = 0; q < kDraws; ++q) {
                ell += s_lp[buf][q];
                hs += s_h[buf][q];
            }
            finish_row(g, b, lane, ell, old, hs / (float)kDraws, bad);
        }
    }
}

// dz of one (row, distribution) per warp, tasks strided over the grid's warps
template <int K>
__global__ void __launch_bounds__(kWarps * 32) evg_ppo_loss_bwd_kernel(const __grid_constant__ LossArgs g)
{
    const int lane = threadIdx.x & 31;
    const int64_t tasks = g.n_rows * K, stride = (int64_t)gridDim.x * kWarps;
    for (int64_t w = (int64_t)blockIdx.x * kWarps + (threadIdx.x >> 5); w < tasks; w += stride) {
        const int64_t b = w / K;
        const int k = (int)(w - b * K);
        int j[kDraws];
        const bool bad = load_draws(g.idx, b, g.n, lane, j);
        const float A = __ldg(g.adv + b), r = __ldg(g.ratio_in + b);
        const float gs = g.g_surr ? __ldg(g.g_surr + b) : 0.f;
        const float ge = g.g_ent ? __ldg(g.g_ent + b) : 0.f;
        Dist d;
        load_dist(g.z + w * g.n, g.n, lane, d);
        // d surr / d ell = -A r, or 0 where the clipped branch is the minimum (ties take the unclipped branch)
        const bool clipped = (A > 0.f && r > g.hi) || (A < 0.f && r < g.lo);
        const float G = clipped ? 0.f : (-A * r) * gs;
        const float E = ge / (float)K;
        // d ell / d y_m = c_m - p_m Q_m: c_m the draws of m, Q_m the sum of 1 / T_k over the draws that counted m
        float Q[kDraws];
        int first[kSlots];
        if constexpr (K == 1) {
            float T[kDraws];
            totals_wo_replacement(d, j, g.n, lane, first, T);
            float q = 0.f;
#pragma unroll
            for (int i = 0; i < kDraws; ++i) Q[i] = q += 1.f / T[i];
        } else {
            Q[0] = 1.f / total(d, g.n);
        }
        float* dzr = g.dz + w * g.n;
#pragma unroll
        for (int s = 0; s < kSlots; ++s) {
            const int m = lane + 32 * s;
            if (32 * s >= g.n) continue;  // warp-uniform
            float c, qm;
            if constexpr (K == 1) {
                c = 0.f;
                qm = Q[0];
#pragma unroll
                for (int i = 0; i < kDraws; ++i) {
                    c += j[i] == m ? 1.f : 0.f;
                    if (first[s] >= i) qm = Q[i];
                }
            } else {
                c = j[k] == m ? 1.f : 0.f;
                qm = Q[0];
            }
            float v = 0.f;
            if (G != 0.f) v = G * (c - d.p[s] * qm);
            if (E != 0.f) v = v - E * (d.p[s] * ((d.y[s] - d.L) + d.H));
            const float out = (1.f - d.y[s] * d.y[s]) * v;
            if (m < g.n) dzr[m] = bad ? __int_as_float(0x7fc00000) : out;
        }
    }
}

// persistent grid: as many CTAs as stay resident, no more than the work needs; per_sm caches the kernel's residency
template <typename Kern>
unsigned grid_for(Kern kern, int threads, int64_t ctas_needed, int sm_count, int& per_sm)
{
    if (per_sm == 0) {
        int v = 0;
        if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&v, kern, threads, 0) != cudaSuccess || v < 1) v = 1;
        per_sm = v;
    }
    const int64_t cap = (int64_t)per_sm * sm_count;
    return (unsigned)(ctas_needed < cap ? ctas_needed : cap);
}

}  // namespace

cudaError_t launch_ppo_loss(int64_t n_rows, int n_dist, int n, const float* z, const int64_t* idx, const float* old_logp, const float* adv,
                            float lo, float hi, float* surr, float* ent, float* logp, float* ratio, int sm_count, cudaStream_t stream)
{
    LossArgs g{};
    g.z = z, g.idx = idx, g.old_logp = old_logp, g.adv = adv, g.surr = surr, g.ent = ent, g.logp = logp, g.ratio = ratio;
    g.n_rows = n_rows, g.n = n, g.lo = lo, g.hi = hi;
    if (n_dist == 1) {
        static int per_sm = 0;
        const unsigned grid = grid_for(evg_ppo_loss_fwd1_kernel, kWarps * 32, (n_rows + kWarps - 1) / kWarps, sm_count, per_sm);
        evg_ppo_loss_fwd1_kernel<<<grid, kWarps * 32, 0, stream>>>(g);
    } else {
        static int per_sm = 0;
        const unsigned grid = grid_for(evg_ppo_loss_fwd7_kernel, kDraws * 32, n_rows, sm_count, per_sm);
        evg_ppo_loss_fwd7_kernel<<<grid, kDraws * 32, 0, stream>>>(g);
    }
    return cudaGetLastError();
}

cudaError_t launch_ppo_loss_grad(int64_t n_rows, int n_dist, int n, const float* z, const int64_t* idx, const float* adv, const float* ratio,
                                 float lo, float hi, const float* g_surr, const float* g_ent, float* dz, int sm_count, cudaStream_t stream)
{
    LossArgs g{};
    g.z = z, g.idx = idx, g.adv = adv, g.ratio_in = ratio, g.g_surr = g_surr, g.g_ent = g_ent, g.dz = dz;
    g.n_rows = n_rows, g.n = n, g.lo = lo, g.hi = hi;
    const int64_t ctas = (n_rows * n_dist + kWarps - 1) / kWarps;
    if (n_dist == 1) {
        static int per_sm = 0;
        const unsigned grid = grid_for(evg_ppo_loss_bwd_kernel<1>, kWarps * 32, ctas, sm_count, per_sm);
        evg_ppo_loss_bwd_kernel<1><<<grid, kWarps * 32, 0, stream>>>(g);
    } else {
        static int per_sm = 0;
        const unsigned grid = grid_for(evg_ppo_loss_bwd_kernel<kDraws>, kWarps * 32, ctas, sm_count, per_sm);
        evg_ppo_loss_bwd_kernel<kDraws><<<grid, kWarps * 32, 0, stream>>>(g);
    }
    return cudaGetLastError();
}

}  // namespace evg

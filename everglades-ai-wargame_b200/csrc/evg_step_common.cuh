// evg_step_common.cuh — device helpers of the thread-per-match step kernel (evg_step_tpm.cu).
#pragma once
#include "evg_internal.h"

namespace evg {

// numpy's pairwise float64 sum (np.sum at server.py:481) over hv[0..size), size <= MAXSZ <= 16.
template <int MAXSZ>
__device__ __forceinline__ double np_sum_regs(const double (&hv)[MAXSZ], int size)
{
    if (MAXSZ < 8 || size < 8) {  // n < 8: left to right from 0.0
        double res = 0.0;
#pragma unroll
        for (int i = 0; i < (MAXSZ < 7 ? MAXSZ : 7); ++i)
            if (i < size) res = __dadd_rn(res, hv[i]);
        return res;
    }
    double r[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) {
        r[k] = hv[k];
        if (MAXSZ == 16 && size == 16) r[k] = __dadd_rn(hv[k], hv[8 + k]);  // one more block of 8
    }
    double res = __dadd_rn(__dadd_rn(__dadd_rn(r[0], r[1]), __dadd_rn(r[2], r[3])),
                           __dadd_rn(__dadd_rn(r[4], r[5]), __dadd_rn(r[6], r[7])));
#pragma unroll
    for (int i = 8; i < (MAXSZ < 15 ? MAXSZ : 15); ++i)
        if (i < size && size < 16) res = __dadd_rn(res, hv[i]);  // remainder, sequential
    return res;
}

// (int)(hsum / n) exactly as the reference computes it (int() of the correctly rounded fp64 quotient, server.py:491)
// for 0 <= hsum <= 100 n, 1 <= n <= 16, without the fp64 division subroutine: q approximates the quotient to 2e-5;
// if hsum is an exact multiple of n the quotient is that integer; else, unless q is within 1e-3 of an integer, q
// and the rounded quotient lie strictly between the same two integers.  The division itself remains for the rest.
__device__ __forceinline__ int int_quotient(double hsum, int n)
{
    const double nd = (double)n;
    const double q = hsum * (double)__frcp_rn((float)n);
    const int kr = __double2int_rn(q);
    const double kd = (double)kr;
    if (__dmul_rn(kd, nd) == hsum) return kr;
    if (fabs(q - kd) > 1e-3) return (int)q;
    return (int)__ddiv_rn(hsum, nd);
}

// 256-bit global accesses (LDG.E.256 / STG.E.256 on sm_100a): a 64-byte health row of 8 units is two requests
__device__ __forceinline__ void ldg256(const double* p, double& a, double& b, double& c, double& d)
{
    asm volatile("ld.global.cs.v4.f64 {%0,%1,%2,%3}, [%4];" : "=d"(a), "=d"(b), "=d"(c), "=d"(d) : "l"(p));
}
__device__ __forceinline__ void stg256(double* p, double a, double b, double c, double d)
{
    asm volatile("st.global.v4.f64 [%0], {%1,%2,%3,%4};" ::"l"(p), "d"(a), "d"(b), "d"(c), "d"(d) : "memory");
}

// Read a group's health row (issued early so that DRAM latency overlaps the draws).  Groups start on
// 32-byte sectors and are padded to 4 slots, so 32-byte quads never leave the row.
template <int MAXSZ>
__device__ __forceinline__ void load_group(const double* __restrict__ hp, int size, double (&hv)[MAXSZ])
{
    static_assert(MAXSZ % 4 == 0, "rows are read in quads of units");
#pragma unroll
    for (int u = 0; u < MAXSZ; u += 4) {
        hv[u] = hv[u + 1] = hv[u + 2] = hv[u + 3] = 0.0;
        if (u < size) ldg256(hp + u, hv[u], hv[u + 1], hv[u + 2], hv[u + 3]);
    }
}

// Unit slots [0, size) of one target group (the whole group, or one 8-slot segment of it): apply the damage histogram
// to the units, write the touched quads back.  Returns the new alive mask; hv holds the new health values
// (server.py:573-643).  hist[tb + r] is the damage aimed at the r-th unit of the range that was alive before combat.
template <int MAXSZ, typename HistT, bool FMA_ONLY = false>
__device__ __forceinline__ uint32_t apply_units(double* __restrict__ hp, double (&hv)[MAXSZ], int size, uint32_t alive0,
                                                const HistT* __restrict__ hist, int tb, const double* __restrict__ ltab, double divisor,
                                                double rcp = 0.0)
{
    // pass 1: damage aimed at every alive unit.  infliction[uid]: uid -> r-th unit alive before combat (SURVEY A.3)
    uint32_t dv[MAXSZ];
    int rank = 0;
    uint32_t dmax = 0;
#pragma unroll
    for (int u = 0; u < MAXSZ; ++u) {
        const bool on = u < size && ((alive0 >> u) & 1u);
        dv[u] = on ? (uint32_t)hist[tb + rank] : 0u;
        rank += on ? 1 : 0;
        dmax = max(dmax, dv[u]);
    }
    // pass 2: loss = (10.*dmg)/(armor + (tgt_cntrl + fort_bns)*StructureDefense), server.py:592-601
    double loss[MAXSZ];
    if (FMA_ONLY || ltab == nullptr) {
        // without a division or a lookup: a = 10.*dmg exactly (2^52 trick), q0 = a*rcp, then Markstein's correction
        // fma(fma(-q0, D, a), rcp, q0); the host has checked that this IS a/D for every reachable dmg (Tables::fast_div)
#pragma unroll
        for (int u = 0; u < MAXSZ; ++u) {
            const double a = __dsub_rn(__hiloint2double(0x43300000, (int)(10u * dv[u])), 4503599627370496.0);
            const double q0 = __dmul_rn(a, rcp);
            loss[u] = __fma_rn(__fma_rn(-q0, divisor, a), rcp, q0);
        }
    } else {
        // from the table of those same fp64 quotients; all lookups are independent and issued together (ltab[0] == 0.0)
#pragma unroll
        for (int u = 0; u < MAXSZ; ++u) loss[u] = dv[u] ? __ldg(ltab + min(dv[u], (uint32_t)(kLossD - 1))) : 0.0;  // no request for unhit units
        if (dmax >= (uint32_t)kLossD) {  // damage sums beyond the table: the division itself
#pragma unroll
            for (int u = 0; u < MAXSZ; ++u)
                if (dv[u] >= (uint32_t)kLossD) loss[u] = __ddiv_rn(__dmul_rn(10.0, (double)dv[u]), divisor);
        }
    }
    uint32_t alive = alive0;
#pragma unroll
    for (int u = 0; u < MAXSZ; ++u) {
        if (FMA_ONLY || dv[u]) {  // (an unhit unit loses 0.0; dead and padding slots hold 0.0 or stay positive: both no-ops)
            double h = __dsub_rn(hv[u], loss[u]);  // server.py:609
            if (h <= 0.0) {                        // server.py:615-618
                h = 0.0;
                alive &= ~(1u << u);
            }
            hv[u] = h;
        }
    }
#pragma unroll
    for (int u = 0; u < MAXSZ; u += 4)  // one 32-byte store per quad that was hit (padding slots keep what was read)
        if (dv[u] | dv[u + 1] | dv[u + 2] | dv[u + 3]) stg256(hp + u, hv[u], hv[u + 1], hv[u + 2], hv[u + 3]);
    return alive;
}

// One target group handled by one lane: the new alive mask and the observation's avg health (server.py:480-491)
template <int MAXSZ, typename HistT, bool FMA_ONLY = false>
__device__ __forceinline__ uint32_t apply_group(double* __restrict__ hp, double (&hv)[MAXSZ], int size, uint32_t alive0,
                                                const HistT* __restrict__ hist, int tb, const double* __restrict__ ltab, double divisor,
                                                int* avg_out, double rcp = 0.0)
{
    const uint32_t alive = apply_units<MAXSZ, HistT, FMA_ONLY>(hp, hv, size, alive0, hist, tb, ltab, divisor, rcp);
    const double hsum = np_sum_regs<MAXSZ>(hv, size);
    *avg_out = alive ? int_quotient(hsum, __popc(alive)) : 0;  // int((health*1.)/units_alive), :491
    return alive;
}

// numpy's pairwise sum of a group of more than 8 units whose slots [0, 8) are lo[] and [8, size) are hi[] (two lanes' segments)
template <int HI>
__device__ __forceinline__ double np_sum_split(const double (&lo)[8], const double (&hi)[HI], int size)
{
    double r[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) {
        r[k] = lo[k];
        if (HI == 8 && size == 16) r[k] = __dadd_rn(lo[k], hi[k]);
    }
    double res = __dadd_rn(__dadd_rn(__dadd_rn(r[0], r[1]), __dadd_rn(r[2], r[3])),
                           __dadd_rn(__dadd_rn(r[4], r[5]), __dadd_rn(r[6], r[7])));
#pragma unroll
    for (int i = 0; i < (HI < 7 ? HI : 7); ++i)
        if (8 + i < size && size < 16) res = __dadd_rn(res, hi[i]);  // remainder, sequential
    return res;
}

// k-th (0-based) set bit of a 24-bit mask
__device__ __forceinline__ int kth_set_bit(uint32_t mask, int k)
{
    int pos = 0;
    int t = __popc(mask & 0xFFFu);
    if (k >= t) { pos = 12; k -= t; mask >>= 12; }
    t = __popc(mask & 0x3Fu);
    if (k >= t) { pos += 6; k -= t; mask >>= 6; }
    t = __popc(mask & 0x7u);
    if (k >= t) { pos += 3; k -= t; mask >>= 3; }
    t = mask & 1u;
    if (k >= t) { pos += 1; k -= t; mask >>= 1; }
    t = mask & 1u;
    if (k >= t) pos += 1;
    return pos;
}

}  // namespace evg

// evg_kernels.cu — hand-written sm_100a kernels of the batched Everglades turn step.
//
// Mapping: ONE WARP PER MATCH.  Lanes change role with the phase of the turn:
//   lane L < 24  <->  group (side = L/12, gid = L%12)     action decode, movement, scoring
//   lane n-1     <->  node n                               capture, scoring, board observation
//   half-warp u  <->  unit slot u of one target group      combat damage + fp64 health update
//   lane p       <->  (attacking group, block of 4 units)  Philox draws
// Static tables (map adjacency, unit definitions, loadout) are staged in shared memory once per
// CTA; a CTA is persistent (grid-stride over matches).  The resident record of a match is one
// 256-byte line (DemoMap) read/written with one 8-byte access per lane; observations are staged
// in shared memory and streamed out as contiguous float2 rows.  No tensor cores: the path is
// byte/integer work plus a handful of IEEE fp64 operations that decide unit deaths.
//
// Reference semantics (file:line) are cited per phase; the reference is
//   server.py = everglades-server/everglades_server/server.py
//   env.py    = gym-everglades/gym_everglades/envs/everglades_env.py
// and the CPU oracle that checks this file is oracle/evg_oracle.c.
#include "evg_internal.h"

namespace evg {

#define FULL 0xFFFFFFFFu

struct WarpSmem {
    uint32_t* rec;   // resident record, rec_words8*2 words
    uint32_t* acc;   // [2][nn] per (side,node) accumulators
    uint32_t* hist;  // [2][hist_words] damage histogram, 2 x u16 per word
    float* obs;      // [2][obs_len] observation staging
    double* hs;      // [24] post-combat health sum of each fighting group
    uint32_t* res;   // [24] post-combat alive mask of each fighting group
    uint32_t* cmd;   // [24] accepted command per group (action phase) / combat info per group (combat)
    uint8_t* pair;   // [96] (lane | block << 5) draw work list
    uint8_t* seg;    // [48] (lane | segment << 5) apply work list
    double* hbig;    // [n_big][16] post-combat unit healths of groups with more than 8 units
};

__device__ __forceinline__ WarpSmem carve(unsigned char* base, const Tables& S)
{
    WarpSmem W;
    W.rec = reinterpret_cast<uint32_t*>(base);
    W.acc = reinterpret_cast<uint32_t*>(base + S.sm_acc);
    W.hist = reinterpret_cast<uint32_t*>(base + S.sm_hist);
    W.obs = reinterpret_cast<float*>(base + S.sm_obs);
    unsigned char* m = base + S.sm_misc;
    W.hs = reinterpret_cast<double*>(m);
    W.res = reinterpret_cast<uint32_t*>(m + 192);
    W.cmd = reinterpret_cast<uint32_t*>(m + 288);
    W.pair = m + 384;
    W.seg = m + 480;
    W.hbig = reinterpret_cast<double*>(m + 528);
    return W;
}

// Per-(side,node) sums over the groups LISTED at the node (node.groups[pid]: location == node and
// not destroyed).  One shared-memory atomic per group packs three reductions:
//   [0:10)  units of all listed groups, moving or not   (board_state opponent count, server.py:446-449)
//   [10:24) sum count*control of non-moving groups       (capture points, server.py:718-724)
//   [24:29) number of non-moving groups                  (controllers, server.py:725-726)
template <int NODES>
__device__ __forceinline__ void node_accumulate(const Tables& S, const WarpSmem& W, int lane, bool is_grp, int side,
                                                uint32_t w0, uint32_t w1)
{
    const Geo<NODES> D(S);
    const int nn = D.nn();
    for (int i = lane; i < 2 * nn; i += 32) W.acc[i] = 0;
    __syncwarp();
    const uint32_t alive = w1 & 0xFFFFu;
    if (is_grp && alive) {
        const uint32_t cnt = __popc(alive);
        uint32_t v = cnt;
        if (!(w0 & W0_MOVING)) v |= (cnt * S.g_control[lane]) << 10 | 1u << 24;
        atomicAdd(&W.acc[side * nn + (w0 & W0_LOC_MASK)], v);
    }
    __syncwarp();
}

// board_state (server.py:382-455) + player_state (server.py:457-501) + concat (env.py:158-171)
// for both players, staged in shared memory and streamed out as one contiguous row.
// fmt == EVG_OBS_WIRE: the packed row of include/evgsim.h instead (out = that match's row; done/status/rewards go into it).
template <int NODES>
__device__ __forceinline__ void pack_obs(const Tables& S, const WarpSmem& W, int lane, bool is_grp, int side, int gid,
                                         uint32_t w0, uint32_t w1, uint32_t nw, uint32_t turn, float* out, int fmt = EVG_OBS_F32,
                                         bool done = false, int status = 0, float r0 = 0.f, float r1 = 0.f)
{
    const Geo<NODES> D(S);
    const int L = D.obs_len(), nn = D.nn();
    if (fmt == EVG_OBS_WIRE) {
        uint32_t* sw = reinterpret_cast<uint32_t*>(W.obs);
        const int n_nodes = D.n_nodes(), ww = wire_bytes(n_nodes) / 4, gw = 1 + n_nodes + 3 * kGroupLanes / 4;
        if (lane == 0) {
            sw[0] = turn | (done ? 1u : 0u) << 16 | (uint32_t)status << 24;
            sw[gw] = __float_as_uint(r0);
            sw[gw + 1] = __float_as_uint(r1);
            for (int i = gw + 2; i < ww; ++i) sw[i] = 0u;
        }
        if (lane < n_nodes)  // node lane + 1: controlState, listed units of player 0, of player 1
            sw[1 + lane] = (nw & 0xFFFFu) | (W.acc[lane + 1] & 255u) << 16 | (W.acc[nn + lane + 1] & 255u) << 24;
        if (is_grp) {
            uint8_t* b = reinterpret_cast<uint8_t*>(sw) + EVG_WIRE_NODE0 + 4 * n_nodes + 3 * lane;
            b[0] = (uint8_t)((w0 & W0_LOC_MASK) | ((w0 >> 21) & 1u) << 6);
            b[1] = (uint8_t)((w0 >> W0_AVG_SHIFT) & 127u);
            b[2] = (uint8_t)__popc(w1 & 0xFFFFu);
        }
        __syncwarp();
        uint2* o2 = reinterpret_cast<uint2*>(out);
        const uint2* s2 = reinterpret_cast<const uint2*>(sw);
        for (int i = lane; i < ww / 2; i += 32) __stcs(o2 + i, s2[i]);
        __syncwarp();
        return;
    }
    if (lane == 0) {
        W.obs[0] = (float)turn;
        W.obs[L] = (float)turn;
    }
    if (lane < D.n_nodes()) {
        const int n = lane + 1;
        const uint32_t f = S.node_flags[n];
        const float fd = (float)(f & 1u), fo = (float)((f >> 1) & 1u);
        const float cs = (float)(int)(int16_t)(nw & 0xFFFFu);  // raw sign for both viewers
        float* o0 = W.obs + 1 + 4 * lane;                      // player 0: slot k shows node k+1
        o0[0] = fd; o0[1] = fo; o0[2] = cs; o0[3] = (float)(W.acc[nn + n] & 1023u);
        float* o1 = W.obs + L + 1 + 4 * ((int)S.p1_map[n] - 1);  // player 1: node n sits in slot p1_map[n] (involution)
        o1[0] = fd; o1[1] = fo; o1[2] = cs; o1[3] = (float)(W.acc[n] & 1023u);
    }
    if (is_grp) {
        float* o = W.obs + side * L + 1 + 4 * D.n_nodes() + 5 * gid;
        const uint32_t loc = w0 & W0_LOC_MASK;
        o[0] = (float)(side ? (uint32_t)S.p1_map[loc] : loc);
        o[1] = (float)S.g_type[lane];
        o[2] = (float)((w0 >> W0_AVG_SHIFT) & 127u);
        o[3] = (float)((w0 >> 21) & 1u);
        o[4] = (float)__popc(w1 & 0xFFFFu);
    }
    __syncwarp();
    float2* o2 = reinterpret_cast<float2*>(out);  // 2*obs_len floats per match: always 8-byte aligned
    const float2* s2 = reinterpret_cast<const float2*>(W.obs);
#pragma unroll 4
    for (int i = lane; i < L; i += 32) __stcs(o2 + i, s2[i]);
    __syncwarp();
}

// ---------------------------------------------------------------------------------------------
// One turn of one match by one warp: env.py:32-73 step -> server.py:211-279 game_turn.
// ---------------------------------------------------------------------------------------------
template <int NODES>
__device__ __forceinline__ void step_match(const Tables& S, const WarpSmem& W, const StepArgs& A, int64_t env, int lane,
                                           unsigned long long* cta_stats)
{
    const Geo<NODES> D(S);
    const int n_nodes = D.n_nodes(), nn = D.nn(), rec_words8 = D.rec_words8();
    const bool is_grp = lane < kGroupLanes;
    const int side = lane >= EVG_NUM_GROUPS ? 1 : 0;
    const int gid = lane - side * EVG_NUM_GROUPS;

    // ---- load the resident record (one coalesced 8-byte access per lane) and this turn's action rows
    uint2* grec = reinterpret_cast<uint2*>(A.records) + env * rec_words8;
    uint2* srec2 = reinterpret_cast<uint2*>(W.rec);
    uint2 own = make_uint2(0u, 0u);
    if (lane < rec_words8) own = grec[lane];
    uint32_t arow = 0;
    // (L1-bypassing load: in the multi-turn rollout kernel the rows were written a moment ago by two lanes of this warp)
    if (lane < 2 * EVG_MAX_ACTIONS) arow = __ldcg(reinterpret_cast<const uint16_t*>(A.actions) + env * (2 * EVG_MAX_ACTIONS) + lane);
    if (lane < rec_words8) srec2[lane] = own;
    for (int i = lane + 32; i < rec_words8; i += 32) srec2[i] = grec[i];
    if (is_grp) W.cmd[lane] = 0xFFFFFFFFu;
    __syncwarp();
    uint32_t w0 = is_grp ? own.x : 0u, w1 = is_grp ? own.y : 0u;  // uint2 L = words 2L, 2L+1 = group lane L
    uint32_t nw = lane < n_nodes ? W.rec[kRecNode0 + lane] : 0u;
    uint32_t turn = __shfl_sync(FULL, own.x, kRecTurn / 2) + 1u;  // server.py:214
    uint32_t episode = __shfl_sync(FULL, own.y, kRecTurn / 2);

    // ---- action decode + validation, server.py:218-271.  One lane per action row (player = lane/7):
    // a row is valid if (t2) the group is not moving and (t3) the destination is adjacent; of the valid
    // rows naming one group the FIRST wins (t1 only ever sees accepted rows) = shared-memory atomicMin
    // on (row index, destination, distance).
    if (lane < 2 * EVG_MAX_ACTIONS) {
        const int ag = (int)(int8_t)(arow & 0xFFu);
        int an = (int)(int8_t)(arow >> 8);
        const int pl = lane >= EVG_MAX_ACTIONS ? 1 : 0;
        if ((unsigned)ag < (unsigned)EVG_NUM_GROUPS) {
            an = (unsigned)an <= (unsigned)n_nodes ? an : 0;
            if (pl) an = S.p1_map[an];  // server.py:233-234
            const int L = pl * EVG_NUM_GROUPS + ag;
            const uint32_t gw0 = W.rec[2 * L];
            EVG_CHECK((gw0 & W0_LOC_MASK) >= 1 && (gw0 & W0_LOC_MASK) <= (uint32_t)n_nodes && an >= 0 && an <= n_nodes);
            const uint32_t d = S.edge[gw0 & W0_LOC_MASK][an];
            if (d && !(gw0 & W0_MOVING)) atomicMin(&W.cmd[L], (uint32_t)lane << 16 | (uint32_t)an << 8 | d);
        }
    }
    __syncwarp();
    if (is_grp) {
        const uint32_t c = W.cmd[lane];
        if (c != 0xFFFFFFFFu)  // server.py:267-270
            w0 = (w0 & ~((0x3Fu << W0_DEST_SHIFT) | (0xFFu << W0_DIST_SHIFT))) | ((c >> 8) & 0x3Fu) << W0_DEST_SHIFT |
                 (c & 0xFFu) << W0_DIST_SHIFT | W0_READY;
    }

    // ---- combat, server.py:503-654
    {
        const uint32_t alive = w1 & 0xFFFFu;
        const uint32_t cnt = __popc(alive);
        const uint32_t loc = w0 & W0_LOC_MASK;
        const bool present = is_grp && alive && !(w0 & W0_MOVING);  // listed and not in transit (:523-530)
        // a node is contested when both players have a present group there (:539)
        const uint32_t peers = __match_any_sync(FULL, present ? loc : 64u + (uint32_t)lane);
        const uint32_t opp_lanes = side ? 0x00000FFFu : 0x00FFF000u;
        const bool fighting = present && (peers & opp_lanes) != 0;
        const uint32_t fmask = __ballot_sync(FULL, fighting);
        if (fmask) {
            {   // unit slots whose health this turn's combat reads and may write (ST_FOUGHT)
                const unsigned slots = __reduce_add_sync(FULL, fighting ? (unsigned)S.g_size[lane] : 0u);
                if (lane == 0) atomicAdd(&cta_stats[ST_FOUGHT], (unsigned long long)slots);
            }
            // Histogram slot of a target = (units of its side's fighting groups at lower-numbered nodes)
            // + (units of its side's groups listed before it at its node) + alive rank inside the group.
            // Inside one node that is exactly the uid the reference draws (SURVEY.md A.3: uid -> (group,
            // r-th unit alive before combat) is fixed before any damage lands).
            //   acc[x]      = fighting units at node x, side 0 | side 1 << 16   (np.sum(counts[pid]), :552-553)
            //   acc[nn + x] = exclusive prefix of acc over nodes = histogram base of (side, x)
            for (int i = lane; i < nn; i += 32) W.acc[i] = 0;
            __syncwarp();
            EVG_CHECK(!fighting || (loc >= 1 && loc <= (uint32_t)n_nodes));
            if (fighting) atomicAdd(&W.acc[loc], cnt << (16 * side));
            __syncwarp();
            const uint32_t tot = lane < n_nodes ? W.acc[lane + 1] : 0u;
            uint32_t inc = tot;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                if (NODES && o >= 2 * NODES) break;
                const uint32_t t = __shfl_up_sync(FULL, inc, o);
                if (lane >= o) inc += t;
            }
            const uint32_t totals = __shfl_sync(FULL, inc, 31);
            if (lane < n_nodes) W.acc[nn + lane + 1] = inc - tot;
            const int hw0 = (int)((totals & 0xFFFFu) + 1) >> 1, hw1 = (int)((totals >> 16) + 1) >> 1;
            EVG_CHECK(hw0 <= S.hist_words && hw1 <= S.hist_words);
            for (int i = lane; i < hw0; i += 32) W.hist[i] = 0;
            for (int i = lane; i < hw1; i += 32) W.hist[S.hist_words + i] = 0;
            __syncwarp();
            const uint32_t node_tot = W.acc[loc], node_base = W.acc[nn + loc];
            const uint32_t n = (node_tot >> (16 * (1 - side))) & 0xFFFFu;    // opposing units at my node
            const uint32_t hb = (node_base >> (16 * (1 - side))) & 0xFFFFu;  // opposing histogram base
            uint32_t tb = (node_base >> (16 * side)) & 0xFFFFu;
            // order inside the node list (node.groups[pid] is in arrival order, then gid)
            const uint32_t okey = ((w1 >> 16) << 4 | (uint32_t)gid) << 5 | cnt;
            uint32_t m = fighting ? (peers & ~opp_lanes & ~(1u << lane)) : 0u;
            while (__any_sync(FULL, m != 0)) {
                const int src = m ? __ffs(m) - 1 : lane;
                const uint32_t ok = __shfl_sync(FULL, okey, src);
                if (m && ok < okey) tb += ok & 31u;
                m &= m - 1;
            }
            if (fighting) {
                W.cmd[lane] = tb | hb << 8 | n << 16;
                W.res[lane] = alive;
            }
            // work lists: (group, block of 8 attackers) for the draws, (group, 8-slot segment) for the apply
            const uint32_t big = __ballot_sync(FULL, fighting && S.g_size[lane] > 8);
            const uint32_t b2 = __ballot_sync(FULL, fighting && cnt > 8);
            const uint32_t lt = (1u << lane) - 1u;
            const int o1 = __popc(fmask), npairs = o1 + __popc(b2), nsegs = o1 + __popc(big);
            EVG_CHECK(npairs <= 96 && nsegs <= 48);
            if (fighting) {
                W.pair[__popc(fmask & lt)] = (uint8_t)lane;
                W.seg[__popc(fmask & lt)] = (uint8_t)lane;
            }
            if ((b2 >> lane) & 1u) W.pair[o1 + __popc(b2 & lt)] = (uint8_t)(lane | 1 << 5);
            if ((big >> lane) & 1u) W.seg[o1 + __popc(big & lt)] = (uint8_t)(lane | 1 << 5);
            __syncwarp();
            // draws: every alive unit of a fighting group targets uid = randint(opposing alive units
            // at the node) and adds its type's damage to infliction[uid], server.py:549-566.
            // Tape: 8 draws of 16 bits per Philox block (oracle/tape.py).
            for (int base = 0; base < npairs; base += 32) {
                const int p = base + lane;
                if (p < npairs) {
                    const uint32_t pr = W.pair[p];
                    const int L = pr & 31, k = pr >> 5;
                    const int gs = L >= EVG_NUM_GROUPS ? 1 : 0, gg = L - gs * EVG_NUM_GROUPS;
                    const uint32_t gl = W.rec[2 * L] & W0_LOC_MASK;  // loc/alive untouched since the load
                    const int gcnt = __popc(W.rec[2 * L + 1] & 0xFFFFu);
                    const uint32_t info = W.cmd[L];
                    const uint32_t gn = info >> 16, ghb = (info >> 8) & 0xFFu;
                    const uint32_t dmg = S.g_damage[L];
                    uint32_t r[4];
                    philox4x32_10(S.env_base + (uint32_t)env, turn, gl | (uint32_t)gs << 8 | (uint32_t)gg << 16 | (uint32_t)k << 24,
                                  episode << 8, S.seed_lo, S.seed_hi, r);
                    uint32_t* hist = W.hist + (1 - gs) * S.hist_words;
#pragma unroll
                    for (int q = 0; q < 8; ++q)
                        if (8 * k + q < gcnt) {
                            const uint32_t half = (q & 1) ? r[q >> 1] >> 16 : r[q >> 1] & 0xFFFFu;
                            const uint32_t idx = ghb + ((half * gn) >> 16);
                            EVG_CHECK(gn >= 1 && (int)(idx >> 1) < S.hist_words);
                            atomicAdd(&hist[idx >> 1], dmg << ((idx & 1u) * 16));
                        }
                }
            }
            __syncwarp();
            // apply, server.py:573-643: four 8-slot segments per pass, one unit slot per lane.  Groups of
            // more than 8 units span two segments; their healths go through shared memory so that the
            // group lane can redo numpy's pairwise sum in order afterwards.
            const int q8 = lane >> 3, u8 = lane & 7;
            double* henv = A.health + env * S.health_slots;
            for (int base = 0; base < nsegs; base += 4) {
                const bool act = base + q8 < nsegs;
                const uint32_t pr = act ? W.seg[base + q8] : 0u;
                const int L = pr & 31, sg = pr >> 5, slot = sg * 8 + u8;
                const int gs = L >= EVG_NUM_GROUPS ? 1 : 0;
                const uint32_t galive = act ? W.rec[2 * L + 1] & 0xFFFFu : 0u;
                const int gsize = S.g_size[L];
                const bool mine = (galive >> slot) & 1u;
                double* hp = henv + S.g_slot[L] + slot;
                double h = 0.0;
                uint32_t d = 0;
                if (mine) {
                    const uint32_t idx = (W.cmd[L] & 0xFFu) + __popc(galive & ((1u << slot) - 1u));
                    EVG_CHECK((int)(idx >> 1) < S.hist_words && (int)S.g_slot[L] + slot < S.health_slots);
                    d = (W.hist[gs * S.hist_words + (idx >> 1)] >> ((idx & 1u) * 16)) & 0xFFFFu;
                    h = *hp;
                }
                bool dead = false;
                if (d) {
                    // loss = (10.*dmg)/(armor + (tgt_cntrl + fort_bns)*StructureDefense), server.py:592-601
                    const uint32_t gl = W.rec[2 * L] & W0_LOC_MASK;
                    const uint32_t nwd = W.rec[kRecNode0 + gl - 1];
                    const int cb = (int)(int8_t)((nwd >> 16) & 0xFFu);
                    const int bonus = (cb == gs ? 1 : 0) + ((S.node_flags[gl] >> 2) & 1);
                    const double node_def = __dmul_rn((double)bonus, S.node_def[gl]);
                    const double loss = __ddiv_rn(__dmul_rn(10.0, (double)d), __dadd_rn(S.unit_armor[S.g_type[L]], node_def));
                    h = __dsub_rn(h, loss);  // server.py:609
                    if (h <= 0.0) {          // server.py:615-618
                        h = 0.0;
                        dead = true;
                    }
                    *hp = h;
                }
                const uint32_t deadbits = (__ballot_sync(FULL, dead) >> (8 * q8)) & 0xFFu;
                if (act && u8 == 0 && deadbits) atomicAnd(&W.res[L], ~(deadbits << (8 * sg)));
                // np.sum(unitHealth), server.py:481: n == 8 is the pure 8-leaf tree, done in registers
                double v = __dadd_rn(h, __shfl_xor_sync(FULL, h, 1, 8));
                v = __dadd_rn(v, __shfl_xor_sync(FULL, v, 2, 8));
                v = __dadd_rn(v, __shfl_xor_sync(FULL, v, 4, 8));
                if (S.has_small_groups) {  // n < 8: plain left-to-right loop from 0.0
                    double seq = 0.0;
                    for (int i = 0; i < 7; ++i) {
                        const double x = __shfl_sync(FULL, h, i, 8);
                        if (i < gsize) seq = __dadd_rn(seq, x);
                    }
                    if (gsize < 8) v = seq;
                }
                if (act) {
                    if (gsize > 8) W.hbig[S.g_big[L] * 16 + slot] = h;  // slots >= size hold 0.0
                    else if (u8 == 0) W.hs[L] = v;
                }
            }
            __syncwarp();
            if (fighting) {
                const uint32_t nalive = W.res[lane];
                double hsum;
                const int gsize = S.g_size[lane];
                if (gsize > 8) {  // 8 < n <= 16: numpy's blocked pairwise sum, restated sequentially
                    const double* a = W.hbig + S.g_big[lane] * 16;
                    double r[8];
#pragma unroll
                    for (int k = 0; k < 8; ++k) r[k] = gsize == 16 ? __dadd_rn(a[k], a[8 + k]) : a[k];
                    hsum = __dadd_rn(__dadd_rn(__dadd_rn(r[0], r[1]), __dadd_rn(r[2], r[3])),
                                     __dadd_rn(__dadd_rn(r[4], r[5]), __dadd_rn(r[6], r[7])));
                    if (gsize < 16)
                        for (int i = 8; i < gsize; ++i) hsum = __dadd_rn(hsum, a[i]);
                } else {
                    hsum = W.hs[lane];
                }
                // player_state's int((health*1.)/units_alive), server.py:491 — one division for all groups
                const int avg = nalive ? (int)__ddiv_rn(hsum, (double)__popc(nalive)) : 0;
                w1 = (w1 & 0xFFFF0000u) | nalive;  // alive == 0: destroyed, leaves the node list (:623-627)
                w0 = (w0 & ~(127u << W0_AVG_SHIFT)) | ((uint32_t)avg & 127u) << W0_AVG_SHIFT;
            }
        }
    }

    // ---- movement, server.py:656-706 (destroyed groups are skipped, :663)
    if (is_grp && (w1 & 0xFFFFu)) {
        if (w0 & W0_READY) {
            w0 = (w0 & ~W0_READY) | W0_MOVING;  // first turn only flips ready -> moving (:664-667)
        } else if (w0 & W0_MOVING) {
            int dist = (int)((w0 >> W0_DIST_SHIFT) & 0xFFu) - (int)S.g_speed[lane];  // :671
            if (dist <= 0) {  // arrived: appended to the destination's list (:678-695)
                const uint32_t dest = (w0 >> W0_DEST_SHIFT) & 0x3Fu;
                w0 = (w0 & (127u << W0_AVG_SHIFT)) | dest;
                w1 = (w1 & 0xFFFFu) | turn << 16;
            } else {
                w0 = (w0 & ~(0xFFu << W0_DIST_SHIFT)) | (uint32_t)dist << W0_DIST_SHIFT;
            }
        }
    }

    // ---- capture, server.py:708-767 (current_turn > 0 here; the turn-0 case is the reset kernel's)
    node_accumulate<NODES>(S, W, lane, is_grp, side, w0, w1);
    int s0 = 0, s1 = 0;
    bool basecap = false;
    if (lane < n_nodes) {
        const int n = lane + 1;
        int cs = (int)(int16_t)(nw & 0xFFFFu), cb = (int)(int8_t)((nw >> 16) & 0xFFu);
        const uint32_t a0 = W.acc[n], a1 = W.acc[nn + n];
        const bool c0 = (a0 >> 24) != 0, c1 = (a1 >> 24) != 0;
        const int cp = S.node_cp[n];
        if (c0 != c1) {  // exactly one controller (:729)
            const int pid = c1 ? 1 : 0;
            if (abs(cs) < cp || pid != cb) {  // :731-732
                const int pts = (int)(((pid ? a1 : a0) >> 10) & 0x3FFFu), pxer = pid ? -1 : 1;
                const bool old_sign = cs < 0;  // :747-750, zero counts as player 0's sign
                cs += pts * pxer;
                const bool neutralize = old_sign != (cs < 0);
                if (abs(cs) >= cp) {  // :763-765
                    cs = cp * pxer;
                    cb = pid;
                }
                if (cb != -1 && neutralize) cb = -1;  // :766-767
                nw = ((uint32_t)cs & 0xFFFFu) | ((uint32_t)cb & 0xFFu) << 16;
            }
        }
        // ---- game_end scoring, server.py:298-310
        const int ts = S.node_team_start[n];
        if (ts != -1 && cb != -1 && cb != ts) {
            basecap = true;
            if (cb) s1 += S.capture_bonus; else s0 += S.capture_bonus;
        }
        if (cs != 0) {
            const int pts = abs(cs) == cp ? 2 * cp : abs(cs);
            if (cs > 0) s0 += pts; else s1 += pts;
        }
    }
    const uint32_t galive_now = w1 & 0xFFFFu;
    if (is_grp && galive_now) {  // server.py:313-317
        const int v = __popc(galive_now) * (int)S.g_cost[lane];
        if (side) s1 += v; else s0 += v;
    }
    s0 = __reduce_add_sync(FULL, s0);
    s1 = __reduce_add_sync(FULL, s1);
    const bool any_alive = __ballot_sync(FULL, is_grp && galive_now) != 0;
    const bool any_basecap = __ballot_sync(FULL, basecap) != 0;
    int status = EVG_STATUS_IN_PROGRESS;  // server.py:321-328, in that priority
    if ((int)turn >= S.turn_limit) status = EVG_STATUS_TIME_EXPIRED;
    else if (!any_alive) status = EVG_STATUS_ANNIHILATION;
    else if (any_basecap) status = EVG_STATUS_BASE_CAPTURE;
    const bool done = status != 0;

    // ---- reward / done, env.py:37-60.  float32(float64(score)/MAX_SCORE) == float32 IEEE division for
    // every score < 2^24 (no double-rounding case exists; checked exhaustively in tests/test_tape.py).
    float rw0, rw1;
    {
        const int mine = lane ? s1 : s0, other = lane ? s0 : s1;
        float r;
        if (done) r = mine == other ? 0.f : (mine > other ? 1.f : (lane ? -1.f : 0.f));
        else r = __fdiv_rn((float)mine, S.max_score_f);
        rw1 = __shfl_sync(FULL, r, 1);
        rw0 = __shfl_sync(FULL, r, 0);
        if (lane == 0) {
            reinterpret_cast<float2*>(A.reward)[env] = make_float2(rw0, rw1);
            A.done[env] = done ? 1 : 0;
            if (A.status) A.status[env] = (uint8_t)status;
            if (A.scores) reinterpret_cast<int2*>(A.scores)[env] = make_int2(s0, s1);
        }
    }

    // ---- observations of the post-turn state
    const int fmt = A.obs_fmt;
    float* obs_out = fmt == EVG_OBS_WIRE ? reinterpret_cast<float*>(reinterpret_cast<char*>(A.obs) + env * wire_bytes(n_nodes))
                                         : A.obs + env * 2 * D.obs_len();
    pack_obs<NODES>(S, W, lane, is_grp, side, gid, w0, w1, nw, turn, obs_out, fmt, done, status, rw0, rw1);

    // ---- termination with in-place auto-reset
    if (done && S.auto_reset != EVG_AUTORESET_OFF) {
        if (lane == 0) {
            atomicAdd(&cta_stats[ST_EPISODES], 1ull);
            atomicAdd(&cta_stats[s0 == s1 ? ST_TIES : (s0 > s1 ? ST_WIN0 : ST_WIN1)], 1ull);
            atomicAdd(&cta_stats[ST_TURNS], (unsigned long long)turn);
            atomicAdd(&cta_stats[ST_SCORE0], (unsigned long long)s0);
            atomicAdd(&cta_stats[ST_SCORE1], (unsigned long long)s1);
            atomicAdd(&cta_stats[ST_STATUS0 + status], 1ull);
        }
        if (is_grp) { w0 = S.init_w0[lane]; w1 = S.init_w1[lane]; }
        if (lane < n_nodes) nw = S.init_node[lane + 1];
        turn = 0;
        episode += 1;
        double* hp = A.health + env * S.health_slots;
        for (int i = lane; i < S.health_slots; i += 32) hp[i] = 100.0;  // definitions.py:62
        if (S.auto_reset == EVG_AUTORESET_NEXT) {
            node_accumulate<NODES>(S, W, lane, is_grp, side, w0, w1);
            pack_obs<NODES>(S, W, lane, is_grp, side, gid, w0, w1, nw, turn, obs_out, fmt, done, status, rw0, rw1);
        }
    }

    // ---- store the record
    if (is_grp) srec2[lane] = make_uint2(w0, w1);
    if (lane < n_nodes) W.rec[kRecNode0 + lane] = nw;
    if (lane == 0) srec2[kRecTurn / 2] = make_uint2(turn, episode);
    __syncwarp();
    for (int i = lane; i < rec_words8; i += 32) grec[i] = srec2[i];
    __syncwarp();
}

__device__ __forceinline__ const Tables& stage_tables(const Tables& T, unsigned char* smem)
{
    const uint32_t* src = reinterpret_cast<const uint32_t*>(&T);
    uint32_t* dst = reinterpret_cast<uint32_t*>(smem);
    for (int i = threadIdx.x; i < (int)(sizeof(Tables) / 4); i += blockDim.x) dst[i] = src[i];
    return *reinterpret_cast<const Tables*>(smem);
}

template <int NODES>
__global__ void __launch_bounds__(kThreads, 4) evg_step_kernel(const __grid_constant__ Tables T, const __grid_constant__ StepArgs A)
{
    extern __shared__ __align__(16) unsigned char smem[];
    const Tables& S = stage_tables(T, smem);
    unsigned long long* cta_stats = reinterpret_cast<unsigned long long*>(smem + T.sm_tables_bytes);
    if (threadIdx.x < ST_COUNT) cta_stats[threadIdx.x] = 0ull;
    __syncthreads();
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const WarpSmem W = carve(smem + T.sm_tables_bytes + 128 + warp * T.sm_warp_stride, S);
    for (int64_t env = (int64_t)blockIdx.x * kWarpsPerBlock + warp; env < A.n_envs; env += (int64_t)gridDim.x * kWarpsPerBlock)
        step_match<NODES>(S, W, A, env, lane, cta_stats);
    __syncthreads();
    if (threadIdx.x < ST_COUNT && cta_stats[threadIdx.x]) atomicAdd(&A.stats[threadIdx.x], cta_stats[threadIdx.x]);
}

// ---------------------------------------------------------------------------------------------
// Multi-turn rollout for small batches: fully scripted self-play (both players' rows from the on-device agents),
// `n_turns` game turns per launch.  A warp keeps its match for all the turns — the record and the health rows it
// re-reads every turn are its own last writes, still in L1/L2 — so a turn costs no launch and no action-buffer pass:
// lanes 0 and 1 generate the two players' rows (agents/State_Machine/*.py, same functions as evg_agents_kernel) into
// the match's slot of the action buffer, the warp steps the match (step_match, unchanged), repeat.  The output
// arrays hold the last turn's observations / rewards / done flags; episode statistics accumulate as usual.
// ---------------------------------------------------------------------------------------------
template <int NODES>
__global__ void __launch_bounds__(kThreads, 4) evg_rollout_kernel(const __grid_constant__ Tables T, const __grid_constant__ StepArgs A, int n_turns)
{
    extern __shared__ __align__(16) unsigned char smem[];
    const Tables& S = stage_tables(T, smem);
    unsigned long long* cta_stats = reinterpret_cast<unsigned long long*>(smem + T.sm_tables_bytes);
    if (threadIdx.x < ST_COUNT) cta_stats[threadIdx.x] = 0ull;
    __syncthreads();
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const WarpSmem W = carve(smem + T.sm_tables_bytes + 128 + warp * T.sm_warp_stride, S);
    const int rec_words = S.rec_words8 * 2;
    for (int64_t env = (int64_t)blockIdx.x * kWarpsPerBlock + warp; env < A.n_envs; env += (int64_t)gridDim.x * kWarpsPerBlock) {
        const uint32_t* rec = A.records + env * rec_words;
        for (int k = 0; k < n_turns; ++k) {
            if (lane < 2) {
                const int p = lane, kind = A.agent[p];
                const uint32_t turn = __ldcg(rec + kRecTurn) + 1u, episode = __ldcg(rec + kRecEpisode);
                uint32_t rows[EVG_MAX_ACTIONS];
                if (kind == EVG_AGENT_RANDOM) {
                    agent_random_rows(S.env_base + (uint32_t)env, turn, episode, p, S.n_nodes, S.seed_lo, S.seed_hi, rows);
                } else {
                    auto w0_of = [&](int L) -> uint32_t { return __ldcg(rec + 2 * L); };
                    uint2 st = A.agent_state[env * 2 + p];
                    if (kind == EVG_AGENT_BASE_RUSH) agent_base_rush_rows(S, w0_of, st, p, rows);
                    else agent_swarm_rows(S, w0_of, st, S.env_base + (uint32_t)env, turn, episode, p, rows);
                    A.agent_state[env * 2 + p] = st;
                }
                uint16_t* out = reinterpret_cast<uint16_t*>(A.actions_out + (env * 2 + p) * (EVG_MAX_ACTIONS * 2));
#pragma unroll
                for (int r = 0; r < EVG_MAX_ACTIONS; ++r) out[r] = (uint16_t)rows[r];
            }
            __syncwarp();
            step_match<NODES>(S, W, A, env, lane, cta_stats);
        }
    }
    __syncthreads();
    if (threadIdx.x < ST_COUNT && cta_stats[threadIdx.x]) atomicAdd(&A.stats[threadIdx.x], cta_stats[threadIdx.x]);
}

// ---------------------------------------------------------------------------------------------
// reset: env.py:75-116 + server.py:133-209 (all groups at their base in gid order, health 100,
// capture() at turn 0 -> bases at +-controlPoints); writes the first observation.
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kThreads) evg_reset_kernel(const __grid_constant__ Tables T, uint32_t* records, double* health,
                                                             const uint8_t* mask, void* obs, int obs_fmt, int64_t n_envs)
{
    extern __shared__ __align__(16) unsigned char smem[];
    const Tables& S = stage_tables(T, smem);
    __syncthreads();
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const WarpSmem W = carve(smem + T.sm_tables_bytes + 128 + warp * T.sm_warp_stride, S);
    const bool is_grp = lane < kGroupLanes;
    const int side = lane >= EVG_NUM_GROUPS ? 1 : 0, gid = lane - side * EVG_NUM_GROUPS;
    for (int64_t env = (int64_t)blockIdx.x * kWarpsPerBlock + warp; env < n_envs; env += (int64_t)gridDim.x * kWarpsPerBlock) {
        if (mask && !mask[env]) continue;
        uint32_t* rec = records + env * S.rec_words8 * 2;
        const uint32_t episode = mask ? rec[kRecEpisode] + 1u : 0u;
        __syncwarp();
        const uint32_t w0 = is_grp ? S.init_w0[lane] : 0u, w1 = is_grp ? S.init_w1[lane] : 0u;
        const uint32_t nw = lane < S.n_nodes ? S.init_node[lane + 1] : 0u;
        for (int i = lane; i < S.rec_words8 * 2; i += 32) {
            uint32_t v = 0;
            if (i < kRecGroupWords) v = (i & 1) ? S.init_w1[i >> 1] : S.init_w0[i >> 1];
            else if (i == kRecEpisode) v = episode;
            else if (i >= kRecNode0 && i < kRecNode0 + S.n_nodes) v = S.init_node[i - kRecNode0 + 1];
            rec[i] = v;
        }
        double* hp = health + env * S.health_slots;
        for (int i = lane; i < S.health_slots; i += 32) hp[i] = 100.0;
        if (obs) {
            node_accumulate<0>(S, W, lane, is_grp, side, w0, w1);
            float* out = obs_fmt == EVG_OBS_WIRE ? reinterpret_cast<float*>(static_cast<char*>(obs) + env * wire_bytes(S.n_nodes))
                                                 : static_cast<float*>(obs) + env * 2 * S.obs_len;
            pack_obs<0>(S, W, lane, is_grp, side, gid, w0, w1, nw, 0u, out, obs_fmt);
        }
    }
}

// ---------------------------------------------------------------------------------------------
// export / import: resident layout <-> EvgEnvState (one thread per match; test and checkpoint path)
// ---------------------------------------------------------------------------------------------
__device__ double np_pairwise_sum(const double* a, int n)
{
    if (n < 8) {
        double res = 0.0;
        for (int i = 0; i < n; ++i) res = __dadd_rn(res, a[i]);
        return res;
    }
    double r[8];
    for (int k = 0; k < 8; ++k) r[k] = a[k];
    const int m = n - (n % 8);
    int i;
    for (i = 8; i < m; i += 8)
        for (int k = 0; k < 8; ++k) r[k] = __dadd_rn(r[k], a[i + k]);
    double res = __dadd_rn(__dadd_rn(__dadd_rn(r[0], r[1]), __dadd_rn(r[2], r[3])),
                           __dadd_rn(__dadd_rn(r[4], r[5]), __dadd_rn(r[6], r[7])));
    for (; i < n; ++i) res = __dadd_rn(res, a[i]);
    return res;
}

__global__ void evg_export_kernel(const __grid_constant__ Tables T, const uint32_t* records, const double* health, int64_t first,
                                  int64_t count, EvgEnvState* out)
{
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= count) return;
    const int64_t env = first + i;
    const uint32_t* rec = records + env * T.rec_words8 * 2;
    EvgEnvState* s = out + i;
    s->turn = (int32_t)rec[kRecTurn];
    s->episode = (int32_t)rec[kRecEpisode];
    for (int n = 0; n <= EVG_MAX_NODES; ++n) {
        s->control_state[n] = 0;
        s->controlled_by[n] = -1;
    }
    for (int n = 1; n <= T.n_nodes; ++n) {
        const uint32_t nw = rec[kRecNode0 + n - 1];
        s->control_state[n] = (int16_t)(nw & 0xFFFFu);
        s->controlled_by[n] = (int8_t)((nw >> 16) & 0xFFu);
    }
    for (int k = 0; k < 5; ++k) s->pad1[k] = 0;
    for (int L = 0; L < kGroupLanes; ++L) {
        const uint32_t w0 = rec[2 * L], w1 = rec[2 * L + 1];
        EvgGroupState* g = &s->groups[L / EVG_NUM_GROUPS][L % EVG_NUM_GROUPS];
        const uint32_t dest = (w0 >> W0_DEST_SHIFT) & 0x3Fu, alive = w1 & 0xFFFFu;
        g->location = (int16_t)(w0 & W0_LOC_MASK);
        g->travel_destination = dest ? (int16_t)dest : (int16_t)-1;
        g->distance_remaining = (int16_t)((w0 >> W0_DIST_SHIFT) & 0xFFu);
        g->ready = (w0 & W0_READY) ? 1 : 0;
        g->moving = (w0 & W0_MOVING) ? 1 : 0;
        g->destroyed = alive ? 0 : 1;
        g->count = (uint8_t)__popc(alive);
        g->arrival = (int32_t)((w1 >> 16) * 16u + (uint32_t)(L % EVG_NUM_GROUPS));
        g->avg_health = (int32_t)((w0 >> W0_AVG_SHIFT) & 127u);
        const double* hp = health + env * T.health_slots + T.g_slot[L];
        for (int u = 0; u < EVG_MAX_GROUP_UNITS; ++u)
            s->health[L / EVG_NUM_GROUPS][L % EVG_NUM_GROUPS][u] = u < T.g_size[L] ? hp[u] : 0.0;
    }
}

__global__ void evg_import_kernel(const __grid_constant__ Tables T, uint32_t* records, double* health, int64_t first, int64_t count,
                                  const EvgEnvState* in, unsigned* bad)
{
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= count) return;
    const int64_t env = first + i;
    uint32_t* rec = records + env * T.rec_words8 * 2;
    const EvgEnvState* s = in + i;
    for (int k = kRecGroupWords; k < T.rec_words8 * 2; ++k) rec[k] = 0;
    rec[kRecTurn] = (uint32_t)s->turn;
    rec[kRecEpisode] = (uint32_t)s->episode;
    for (int n = 1; n <= T.n_nodes; ++n) {
        int cs = s->control_state[n], cb = s->controlled_by[n];
        const int cp = T.node_cp[n];
        if (cs > cp || cs < -cp || cb < -1 || cb > 1) {  // |controlState| <= ControlPoints, controlledBy in {-1, 0, 1}
            cs = cs > cp ? cp : (cs < -cp ? -cp : cs);
            cb = cb < -1 || cb > 1 ? -1 : cb;
            atomicAdd(bad, 1u);
        }
        rec[kRecNode0 + n - 1] = ((uint32_t)cs & 0xFFFFu) | ((uint32_t)cb & 0xFFu) << 16;
    }
    // unit slots between the groups' sizes and their 4-slot padding are read by the step kernels as part of 32-byte
    // quads: they hold 0.0 like every dead unit
    for (int i = 0; i < T.health_slots; ++i) health[env * T.health_slots + i] = 0.0;
    for (int L = 0; L < kGroupLanes; ++L) {
        const EvgGroupState* g = &s->groups[L / EVG_NUM_GROUPS][L % EVG_NUM_GROUPS];
        double* hp = health + env * T.health_slots + T.g_slot[L];
        uint32_t alive = 0;
        double tmp[EVG_MAX_GROUP_UNITS];
        const int size = T.g_size[L];
        for (int u = 0; u < size; ++u) {
            const double h = s->health[L / EVG_NUM_GROUPS][L % EVG_NUM_GROUPS][u];
            hp[u] = h;
            tmp[u] = h;
            if (h > 0.0) alive |= 1u << u;
        }
        // the cached observation field is derived state: recompute it (server.py:480-491)
        const int avg = alive ? (int)__ddiv_rn(np_pairwise_sum(tmp, size), (double)__popc(alive)) : 0;
        // Out-of-range fields would become shared-memory indices in the step kernels: they are forced into range here
        // (location 1..n_nodes, destination 0..n_nodes) and the record is counted in `bad`, which evg_import_state
        // turns into EVG_E_ARG.  BatchedEvergladesEnv.set_state validates on the host before it gets this far.
        int loc = g->location, dst = g->travel_destination > 0 ? g->travel_destination : 0;
        if (loc < 1 || loc > T.n_nodes || dst > T.n_nodes || g->distance_remaining < 0 || g->distance_remaining > 255) {
            loc = loc < 1 ? 1 : (loc > T.n_nodes ? T.n_nodes : loc);
            dst = dst > T.n_nodes ? 0 : dst;
            atomicAdd(bad, 1u);
        }
        const uint32_t dest = (uint32_t)dst & 0x3Fu;
        rec[2 * L] = ((uint32_t)loc & W0_LOC_MASK) | dest << W0_DEST_SHIFT |
                     ((uint32_t)g->distance_remaining & 0xFFu) << W0_DIST_SHIFT | (g->ready ? W0_READY : 0u) |
                     (g->moving ? W0_MOVING : 0u) | ((uint32_t)avg & 127u) << W0_AVG_SHIFT;
        rec[2 * L + 1] = alive | (((uint32_t)g->arrival >> 4) & 0xFFFFu) << 16;
    }
}

// ---------------------------------------------------------------------------------------------
// random_actions agent (agents/State_Machine/random_actions.py:38-46): 7 distinct groups of 12 and
// 7 distinct nodes of the map, paired in draw order, as a partial Fisher-Yates over the tape
// (same function as evo_agent_random in oracle/evg_oracle.c).  One thread per (match, player).
// ---------------------------------------------------------------------------------------------
__global__ void evg_agent_random_kernel(const __grid_constant__ Tables T, const uint32_t* records, int8_t* actions, int player,
                                        int64_t n_envs)
{
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int nplayers = player < 0 ? 2 : 1;
    if (i >= n_envs * nplayers) return;
    const int64_t env = i / nplayers;
    const int p = player < 0 ? (int)(i % nplayers) : player;
    const uint32_t* rec = records + env * T.rec_words8 * 2;
    const uint32_t turn = rec[kRecTurn] + 1u, episode = rec[kRecEpisode];
    int8_t* out = actions + (env * 2 + p) * (EVG_MAX_ACTIONS * 2);
    if (T.n_nodes <= kAgentMaxNodes) {
        uint32_t rows[EVG_MAX_ACTIONS];
        agent_random_rows(T.env_base + (uint32_t)env, turn, episode, p, T.n_nodes, T.seed_lo, T.seed_hi, rows);
#pragma unroll
        for (int k = 0; k < EVG_MAX_ACTIONS; ++k) reinterpret_cast<uint16_t*>(out)[k] = (uint16_t)rows[k];
        return;
    }
    // larger maps: the same shuffles over byte arrays
    uint32_t w[8];
    philox4x32_10(T.env_base + (uint32_t)env, turn, (uint32_t)p, 1u | episode << 8, T.seed_lo, T.seed_hi, w);
    philox4x32_10(T.env_base + (uint32_t)env, turn, (uint32_t)p | 1u << 8, 1u | episode << 8, T.seed_lo, T.seed_hi, w + 4);
    uint8_t gp[EVG_NUM_GROUPS], np_[EVG_MAX_NODES];
    for (int k = 0; k < EVG_NUM_GROUPS; ++k) gp[k] = (uint8_t)k;
    for (int k = 0; k < T.n_nodes; ++k) np_[k] = (uint8_t)(k + 1);
    for (int k = 0; k < EVG_MAX_ACTIONS; ++k) {
        const uint32_t hg = (k & 1) ? w[k >> 1] >> 16 : w[k >> 1] & 0xFFFFu;
        const uint32_t hn = (k & 1) ? w[4 + (k >> 1)] >> 16 : w[4 + (k >> 1)] & 0xFFFFu;
        const int j = k + (int)((hg * (uint32_t)(EVG_NUM_GROUPS - k)) >> 16);
        const uint8_t t = gp[k]; gp[k] = gp[j]; gp[j] = t;
        const int q = k + (int)((hn * (uint32_t)(T.n_nodes - k)) >> 16);
        const uint8_t t2 = np_[k]; np_[k] = np_[q]; np_[q] = t2;
        out[2 * k] = (int8_t)gp[k];
        out[2 * k + 1] = (int8_t)np_[k];
    }
}

// ---------------------------------------------------------------------------------------------
// Observation-driven scripted agents, one thread per (match, player); the "observation" they read is
// the resident record (location / in-transit flag of the player's groups, in the player's own node
// numbering), which is what obs[45+5g], obs[45+5g+3] hold.  Agent state: uint2 per (match, player),
// .x base_rushV1 {bit0 started, group_num[4:8), node_num[8:16)}, .y SwarmAgent's attack list as nibbles;
// zero = a fresh agent.  Same functions as evo_agent_base_rush / evo_agent_swarm (oracle/evg_oracle.c),
// which are checked against the reference's own Python agents (tests/golden/agents_v1.npz).
// ---------------------------------------------------------------------------------------------
__global__ void evg_agents_kernel(const __grid_constant__ Tables T, const uint32_t* records, uint2* agent_state, int8_t* actions,
                                  int agent0, int agent1, int64_t n_envs)
{
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_envs * 2) return;
    const int64_t env = i >> 1;
    const int p = (int)(i & 1);
    const int kind = p ? agent1 : agent0;
    if (kind == EVG_AGENT_EXTERNAL) return;
    const uint32_t* rec = records + env * T.rec_words8 * 2;
    const uint32_t turn = rec[kRecTurn] + 1u, episode = rec[kRecEpisode];
    uint16_t* out = reinterpret_cast<uint16_t*>(actions + (env * 2 + p) * (EVG_MAX_ACTIONS * 2));
    uint32_t rows[EVG_MAX_ACTIONS];
    if (kind == EVG_AGENT_RANDOM) {  // maps of <= 15 nodes (checked by the host)
        agent_random_rows(T.env_base + (uint32_t)env, turn, episode, p, T.n_nodes, T.seed_lo, T.seed_hi, rows);
    } else {
        auto w0_of = [&](int L) -> uint32_t { return rec[2 * L]; };
        uint2 st = agent_state[env * 2 + p];
        if (kind == EVG_AGENT_BASE_RUSH) agent_base_rush_rows(T, w0_of, st, p, rows);
        else agent_swarm_rows(T, w0_of, st, T.env_base + (uint32_t)env, turn, episode, p, rows);
        agent_state[env * 2 + p] = st;
    }
#pragma unroll
    for (int k = 0; k < EVG_MAX_ACTIONS; ++k) out[k] = (uint16_t)rows[k];
}

// ---------------------------------------------------------------------------------------------
// Policy-in-the-loop glue (SURVEY.md §8 f-2): network outputs -> int8 action rows, on the device.
// evg_decode_dqn_kernel restates DQNAgent.filter_actions (agents/DQN/DQNAgent.py:161-197) exactly: a greedy
// insertion over (node, group) in node-major order into 7 slots whose best-Q start at 0 and whose group ids start
// at 0; a group already placed in another slot may only improve its own slot; the node written is the 0-based
// column (the reference's off-by-one).  One thread per (match, player); q is [rows][12 * num_cols] float32.
// ---------------------------------------------------------------------------------------------
// q[i * row_stride + c * col_stride] is entry c of row i: row-major network output (row_stride = 12 * num_cols, col_stride = 1)
// or the transposed layout evg_policy_mlp writes (row_stride = 1, col_stride = rows), which this thread-per-row scan reads
// coalesced.  Every slot's best-Q only ever grows, so a candidate that does not beat the smallest of them is skipped at once.
// Lanes are different rows, so a branch taken by one lane is paid by all 32: per node the twelve candidates are first
// tested against the smallest best-Q (uniform, cheap), then each lane walks only ITS OWN survivors in order (a slot's
// best-Q only ever grows, so a candidate rejected by the first test stays rejected; survivors are re-tested) — the warp
// runs max-over-lanes(survivors) insertions per node instead of one per candidate position that any lane accepts.
constexpr int kDecodeThreads = 128;
__global__ void __launch_bounds__(kDecodeThreads) evg_decode_dqn_kernel(const float* __restrict__ q, int num_cols, int player, int8_t* actions, int64_t n_envs,
                                                                        int64_t row_stride, int64_t col_stride)
{
    __shared__ float vs[EVG_NUM_GROUPS][kDecodeThreads];  // this node's candidates, [group][thread]: a thread's own column, any index conflict-free
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int np_ = player < 0 ? 2 : 1;
    if (i >= n_envs * np_) return;  // (no CTA barrier below: a thread only ever reads what it wrote itself)
    const int64_t env = i / np_;
    const int p = player < 0 ? (int)(i % np_) : player;
    const float* qi = q + i * row_stride;
    float bq[EVG_MAX_ACTIONS];
    int bu[EVG_MAX_ACTIONS], bn[EVG_MAX_ACTIONS];
#pragma unroll
    for (int s = 0; s < EVG_MAX_ACTIONS; ++s) { bq[s] = 0.f; bu[s] = 0; bn[s] = 0; }
    float bmin = 0.f;
    for (int n = 0; n < num_cols; ++n) {
        float v[EVG_NUM_GROUPS];  // the twelve candidates of this node: independent loads in flight together
#pragma unroll
        for (int g = 0; g < EVG_NUM_GROUPS; ++g) v[g] = __ldcs(qi + (int64_t)(g * num_cols + n) * col_stride);
        uint32_t pm = 0;
#pragma unroll
        for (int g = 0; g < EVG_NUM_GROUPS; ++g) {
            pm |= (v[g] > bmin ? 1u : 0u) << g;
            vs[g][threadIdx.x] = v[g];
        }
        for (; pm; pm &= pm - 1) {
            const int g = __ffs(pm) - 1;
            const float vg = vs[g][threadIdx.x];
            if (!(vg > bmin)) continue;
            uint32_t eqm = 0, gtm = 0;  // slots that hold group g (`group_index in best_action_units`) / that v beats
#pragma unroll
            for (int s = 0; s < EVG_MAX_ACTIONS; ++s) {
                eqm |= (bu[s] == g ? 1u : 0u) << s;
                gtm |= (vg > bq[s] ? 1u : 0u) << s;
            }
            const uint32_t ok = eqm ? (gtm & eqm) : gtm;  // a group already placed may only improve its own slot
            if (ok) {
                const int s0 = __ffs(ok) - 1;  // the first slot in order that takes it
#pragma unroll
                for (int s = 0; s < EVG_MAX_ACTIONS; ++s)
                    if (s == s0) { bq[s] = vg; bu[s] = g; bn[s] = n; }
                bmin = bq[0];
#pragma unroll
                for (int s = 1; s < EVG_MAX_ACTIONS; ++s) bmin = fminf(bmin, bq[s]);
            }
        }
    }
    uint16_t* out = reinterpret_cast<uint16_t*>(actions + (env * 2 + p) * (EVG_MAX_ACTIONS * 2));
#pragma unroll
    for (int s = 0; s < EVG_MAX_ACTIONS; ++s) out[s] = (uint16_t)((uint32_t)bu[s] | (uint32_t)bn[s] << 8);
}

// PPOAgent.get_action's unravel (agents/PPO/PPOAgent.py:122-127): units = idx // 12, nodes = idx % 11 (sic).
__global__ void evg_decode_indices_kernel(const int64_t* idx, int div, int mod, int player, int8_t* actions, int64_t n_envs)
{
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int np_ = player < 0 ? 2 : 1;
    if (i >= n_envs * np_ * EVG_MAX_ACTIONS) return;
    const int64_t row = i / EVG_MAX_ACTIONS;
    const int k = (int)(i % EVG_MAX_ACTIONS);
    const int64_t env = row / np_;
    const int p = player < 0 ? (int)(row % np_) : player;
    const int64_t v = idx[i];
    int8_t* out = actions + ((env * 2 + p) * EVG_MAX_ACTIONS + k) * 2;
    out[0] = (int8_t)(v / div);
    out[1] = (int8_t)(v % mod);
}

// Reward shaping of the training scripts (utils/reward_shaping.py:17-56), one thread per (match, player).
// turnNum there is the number of steps played BEFORE this one = current_turn - 1, read from the observation.
__global__ void evg_shape_reward_kernel(int mode, const float* reward, const uint8_t* done, const float* obs, int obs_len,
                                        float* out, int64_t n_envs)
{
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_envs * 2) return;
    const int64_t env = i >> 1;
    const int p = (int)(i & 1);
    const float mine = reward[env * 2 + p], other = reward[env * 2 + 1 - p];
    const bool d = done[env] != 0, win = mine > other;
    const float turn_num = obs[env * 2 * obs_len] - 1.f;
    float r;
    switch (mode) {
        case EVG_SHAPE_BASIC: r = (d && win) ? 1.f : 0.f; break;                                     // basic_reward, :29-37
        case EVG_SHAPE_PENALIZE_LONG: r = d ? (win ? 100.f : -0.1f) : -0.001f; break;                // penalize_long_games, :17-27
        case EVG_SHAPE_SHORT_GAMES: r = d ? (win ? (float)((150.0 - (double)turn_num) / 150.0) : -1.f) : 0.f; break;  // :39-50
        default: r = mine; break;                                                                    // normalized_score, :52-57
    }
    out[i] = r;
}

// ---------------------------------------------------------------------------------------------
// launchers
// ---------------------------------------------------------------------------------------------
// DemoMap's node count gets a compile-time instantiation; any other map runs the generic one.
constexpr int kFastNodes = 11;

cudaError_t launch_rollout(const Tables& t, const StepArgs& a, int n_turns, int grid, size_t smem, cudaStream_t stream)
{
    if (t.n_nodes == kFastNodes) evg_rollout_kernel<kFastNodes><<<grid, kThreads, smem, stream>>>(t, a, n_turns);
    else evg_rollout_kernel<0><<<grid, kThreads, smem, stream>>>(t, a, n_turns);
    return cudaGetLastError();
}

cudaError_t set_step_smem(size_t smem)
{
    int limit = 0;
    cudaError_t e = optin_smem_limit(smem, &limit);
    if (e != cudaSuccess) return e;
    if ((e = cudaFuncSetAttribute(evg_rollout_kernel<kFastNodes>, cudaFuncAttributeMaxDynamicSharedMemorySize, limit)) != cudaSuccess) return e;
    if ((e = cudaFuncSetAttribute(evg_rollout_kernel<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, limit)) != cudaSuccess) return e;
    e = cudaFuncSetAttribute(evg_step_kernel<kFastNodes>, cudaFuncAttributeMaxDynamicSharedMemorySize, limit);
    if (e != cudaSuccess) return e;
    if ((e = cudaFuncSetAttribute(evg_step_kernel<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, limit)) != cudaSuccess) return e;
    return cudaFuncSetAttribute(evg_reset_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, limit);
}

cudaError_t step_occupancy(const Tables& t, size_t smem, int* blocks_per_sm)
{
    if (t.n_nodes == kFastNodes) return cudaOccupancyMaxActiveBlocksPerMultiprocessor(blocks_per_sm, evg_step_kernel<kFastNodes>, kThreads, smem);
    return cudaOccupancyMaxActiveBlocksPerMultiprocessor(blocks_per_sm, evg_step_kernel<0>, kThreads, smem);
}

cudaError_t launch_step(const Tables& t, const StepArgs& a, int grid, size_t smem, cudaStream_t stream)
{
    if (t.n_nodes == kFastNodes) evg_step_kernel<kFastNodes><<<grid, kThreads, smem, stream>>>(t, a);
    else evg_step_kernel<0><<<grid, kThreads, smem, stream>>>(t, a);
    return cudaGetLastError();
}

cudaError_t launch_reset(const Tables& t, uint32_t* records, double* health, const uint8_t* mask, void* obs, int obs_fmt,
                         int64_t n_envs, int grid, size_t smem, cudaStream_t stream)
{
    evg_reset_kernel<<<grid, kThreads, smem, stream>>>(t, records, health, mask, obs, obs_fmt, n_envs);
    return cudaGetLastError();
}

// EVG_OBS_I16: the float32 observation vector narrowed to int16 (every entry is an integer that fits), 8 values per thread
// (obs1 / out1 are the same arrays as obs / out, typed for the scalar tail: no __restrict__ on pointers that alias)
__global__ void evg_obs_to_i16_kernel(const float4* obs, uint4* out, const float* obs1, int16_t* out1, int64_t n8, int64_t n)
{
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n8) {
        const float4 a = __ldcs(obs + 2 * i), b = __ldcs(obs + 2 * i + 1);
        auto pk = [](float lo, float hi) { return ((uint32_t)(int)lo & 0xFFFFu) | (uint32_t)(int)hi << 16; };
        __stcs(out + i, make_uint4(pk(a.x, a.y), pk(a.z, a.w), pk(b.x, b.y), pk(b.z, b.w)));
    } else if (i == n8) {
        for (int64_t k = 8 * n8; k < n; ++k) out1[k] = (int16_t)(int)obs1[k];  // the last 0..7 values
    }
}

cudaError_t launch_obs_to_i16(const float* obs, int16_t* out, int64_t n_values, cudaStream_t stream)
{
    if (n_values <= 0) return cudaSuccess;
    const int64_t n8 = n_values / 8;
    evg_obs_to_i16_kernel<<<(unsigned)((n8 + 1 + 255) / 256), 256, 0, stream>>>(reinterpret_cast<const float4*>(obs), reinterpret_cast<uint4*>(out),
                                                                               obs, out, n8, n_values);
    return cudaGetLastError();
}

cudaError_t launch_export(const Tables& t, const uint32_t* records, const double* health, int64_t first, int64_t count,
                          EvgEnvState* out, cudaStream_t stream)
{
    if (count <= 0) return cudaSuccess;
    evg_export_kernel<<<(unsigned)((count + 127) / 128), 128, 0, stream>>>(t, records, health, first, count, out);
    return cudaGetLastError();
}

cudaError_t launch_import(const Tables& t, uint32_t* records, double* health, int64_t first, int64_t count,
                          const EvgEnvState* in, unsigned* bad, cudaStream_t stream)
{
    if (count <= 0) return cudaSuccess;
    evg_import_kernel<<<(unsigned)((count + 127) / 128), 128, 0, stream>>>(t, records, health, first, count, in, bad);
    return cudaGetLastError();
}

cudaError_t launch_agent_random(const Tables& t, const uint32_t* records, int8_t* actions, int player, int64_t n_envs,
                                cudaStream_t stream)
{
    const int64_t n = n_envs * (player < 0 ? 2 : 1);
    if (n <= 0) return cudaSuccess;
    evg_agent_random_kernel<<<(unsigned)((n + 255) / 256), 256, 0, stream>>>(t, records, actions, player, n_envs);
    return cudaGetLastError();
}

cudaError_t launch_decode_dqn(const float* q, int num_cols, int player, int8_t* actions, int64_t n_envs, int transposed, cudaStream_t stream)
{
    const int64_t n = n_envs * (player < 0 ? 2 : 1);
    if (n <= 0) return cudaSuccess;
    evg_decode_dqn_kernel<<<(unsigned)((n + kDecodeThreads - 1) / kDecodeThreads), kDecodeThreads, 0, stream>>>(q, num_cols, player, actions, n_envs,
                                                                           transposed ? 1 : (int64_t)EVG_NUM_GROUPS * num_cols, transposed ? n : 1);
    return cudaGetLastError();
}

cudaError_t launch_decode_indices(const int64_t* idx, int div, int mod, int player, int8_t* actions, int64_t n_envs, cudaStream_t stream)
{
    const int64_t n = n_envs * (player < 0 ? 2 : 1) * EVG_MAX_ACTIONS;
    if (n <= 0) return cudaSuccess;
    evg_decode_indices_kernel<<<(unsigned)((n + 255) / 256), 256, 0, stream>>>(idx, div, mod, player, actions, n_envs);
    return cudaGetLastError();
}

cudaError_t launch_shape_reward(int mode, const float* reward, const uint8_t* done, const float* obs, int obs_len, float* out,
                                int64_t n_envs, cudaStream_t stream)
{
    if (n_envs <= 0) return cudaSuccess;
    evg_shape_reward_kernel<<<(unsigned)((n_envs * 2 + 255) / 256), 256, 0, stream>>>(mode, reward, done, obs, obs_len, out, n_envs);
    return cudaGetLastError();
}

cudaError_t launch_agents(const Tables& t, const uint32_t* records, uint2* agent_state, int8_t* actions, int agent0, int agent1,
                          int64_t n_envs, cudaStream_t stream)
{
    if (n_envs <= 0) return cudaSuccess;
    evg_agents_kernel<<<(unsigned)((n_envs * 2 + 255) / 256), 256, 0, stream>>>(t, records, agent_state, actions, agent0, agent1, n_envs);
    return cudaGetLastError();
}

}  // namespace evg

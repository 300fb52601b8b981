// evg_step_tpm.cu — the turn step with ONE THREAD PER MATCH (a CTA = a block slice of 128 matches).
//
// Why: ncu on the warp-per-match kernel (profiles/r1_*) showed it issue-bound at ~1000 warp
// instructions per match-turn with only ~18 of 32 lanes active: the per-turn work of one match is too
// small and too irregular to fill a warp.  Here every lane runs a whole match, so the regular phases
// (actions, movement, capture, scoring, observation packing) execute with all 32 lanes busy and no
// shuffles, ballots or atomics.  Combat is the irregular part (matches fight different amounts), so it
// is WARP-COOPERATIVE: the fighting groups of the warp's 32 matches form one work list and every
// lane takes one (match, group) item at a time — draws into that match's shared-memory histogram
// with atomics, then the whole group's fp64 health update — so lanes stay busy however unevenly the
// fights are spread over the matches.
//
// Memory behaviour stays that of the warp kernel — HBM sees the same bytes:
//   * the 256-byte records of a warp's 32 matches are loaded/stored COOPERATIVELY (coalesced 16-byte
//     accesses) into per-thread rows of shared memory; row pitch P has P/2 odd, so "every thread reads
//     word w of its own row" is bank-conflict free for 4- and 8-byte accesses.  The loads are a SOFTWARE
//     PIPELINE: the next batch's records are requested into registers while this batch is still being
//     processed, so no batch starts with an exposed DRAM round trip;
//   * observations are packed by each thread into a 128-byte staging window of its row and streamed
//     out by the warp as contiguous float2 runs (two matches per store instruction);
//   * unit health is read as whole 64/96-byte group rows (full 32-byte sectors), only for groups that
//     fight, and only hit units are written back.
// Per warp besides the rows: two words per node and match, stored word-major (bank = lane for any dynamic
// index: member masks and unit totals in combat, capture accumulators afterwards), and a pool for the damage
// histograms of one combat round (a round is <= 32 work items, so <= 32 x 12 entries).  IEEE fp64 health
// arithmetic as in the reference; the per-hit quotient is a reciprocal and two FMAs where the host has proved
// that exact (Tables::fast_div), else a table of the same fp64 quotients / the division itself.
//
// Instruction fetch matters as much as data here (profiles/README.md): three CTAs per SM walk a ~90 KB kernel
// independently, so (1) ONE CTA barrier per batch, before the observation phase, keeps a CTA's four warps on the
// same instructions through the longest straight-line code, (2) code that a launch never executes lives in
// another instantiation (AGENTS) or out of line (statistics, partial warps, resets), (3) loops stay rolled where
// unrolling buys little.  The unroll factors, the barrier site, the request point of the record pipeline and the
// occupancy targets were each chosen by measurement (DESIGN.md section 4.1, profiles/README.md); the unroll factors
// and the observation split quote their timings where they are set.
//
// Reference semantics are cited per phase (server.py / env.py as in evg_kernels.cu); the checker is
// oracle/evg_oracle.c.
#include "evg_step_common.cuh"

namespace evg {

namespace {

// game_init state (server.py:133-209) for one match: its record row in shared memory (the health refill is the warp's
// job: refill_health below)
__device__ __noinline__ void reset_row(const Tables& S, uint32_t* R, int n_nodes, uint32_t* X = nullptr)
{
    // (rolled loops on purpose: this runs for one lane at a time when matches end at different times, and every
    // instruction of it that is fetched evicts one of the hot loop's from the instruction cache)
#pragma unroll 1
    for (int L = 0; L < kGroupLanes; ++L) {
        R[2 * L] = S.init_w0[L];
        R[2 * L + 1] = S.init_w1[L];
    }
#pragma unroll 1
    for (int n = 1; n <= n_nodes; ++n) R[kRecNode0 + n - 1] = S.init_node[n];
    if (X) {  // EVG_AUTORESET_NEXT: the observation shows the new match, so its node sums are needed too
        const int nn = n_nodes + 1;
#pragma unroll 1
        for (int i = 0; i < 2 * nn; ++i) X[32 * i] = 0;
#pragma unroll 1
        for (int L = 0; L < kGroupLanes; ++L) {
            const uint32_t w0 = R[2 * L], cnt = __popc(R[2 * L + 1] & 0xFFFFu);
            X[32 * ((L >= EVG_NUM_GROUPS ? nn : 0) + (w0 & W0_LOC_MASK))] += cnt | (cnt * S.g_control[L]) << 10 | 1u << 24;
        }
    }
}

// health 100.0 for every unit of the matches in `mask` (definitions.py:62), written by the whole warp match after match
// with coalesced 16-byte stores: one finished match costs 4 store instructions, not 100 by a single lane
__device__ __noinline__ void refill_health(double* health_warp, int slots, uint32_t mask, int lane)
{
    for (; mask; mask &= mask - 1) {
        double2* hp = reinterpret_cast<double2*>(health_warp + (size_t)(__ffs(mask) - 1) * slots);
        for (int i = lane; i < slots / 2; i += 32) hp[i] = make_double2(100.0, 100.0);
    }
}

// finished matches of a warp -> the global counters (rare: kept out of the kernel's hot instruction stream)
__device__ __noinline__ void episode_stats(unsigned long long* stats, bool reset_now, int s0, int s1, uint32_t turn, int status, int lane)
{
    const unsigned e = reset_now ? 1u : 0u;
    const unsigned v[ST_COUNT] = {e, e && s0 > s1, e && s1 > s0, e && s0 == s1, e ? turn : 0u, e ? (unsigned)s0 : 0u,
                                  e ? (unsigned)s1 : 0u, e && status == 0, e && status == 1, e && status == 2, e && status == 3};
#pragma unroll
    for (int k = 0; k < ST_COUNT; ++k) {
        const unsigned sum = __reduce_add_sync(0xFFFFFFFFu, v[k]);
        if (lane == 0 && sum) atomicAdd(&stats[k], (unsigned long long)sum);
    }
}

// records and action rows of a warp's matches straight from global memory into its rows: the path of partial warps
// and of the run-time-sized maps (the compile-time map takes them from the registers of its software pipeline)
template <int NODES>
__device__ __noinline__ void load_rows_direct(const StepArgs& A, uint32_t* wrow, int P, int RW, int RWU, int64_t warp_env0, int nvalid,
                                              int lane, bool prefetch_next, int64_t next_env0)
{
    if (prefetch_next && next_env0 + 32 <= A.n_envs) {  // pull the NEXT batch's records and action rows towards L2
        const char* nr = reinterpret_cast<const char*>(A.records) + next_env0 * RW * 4;
        for (int b = lane * 128; b < 32 * RW * 4; b += 32 * 128) asm volatile("prefetch.global.L2 [%0];" ::"l"(nr + b));
        const char* na = reinterpret_cast<const char*>(A.actions) + next_env0 * 28;
        if (lane < 7) asm volatile("prefetch.global.L2 [%0];" ::"l"(na + lane * 128));
    }
    const int q4 = RW / 4;  // 16-byte chunks per record
    const uint4* g4 = reinterpret_cast<const uint4*>(A.records) + warp_env0 * q4;
    const int total = nvalid * q4;
#pragma unroll 1
    for (int f0 = 0; f0 < total; f0 += 32 * 4) {
        uint4 v[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) v[i] = f0 + 32 * i + lane < total ? __ldcs(g4 + f0 + 32 * i + lane) : make_uint4(0u, 0u, 0u, 0u);
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const int f = f0 + 32 * i + lane;
            if (f < total) {
                const int m = NODES ? f >> 4 : f / q4, q = NODES ? f & 15 : f % q4;
                uint2* d = reinterpret_cast<uint2*>(wrow + (size_t)m * P + 4 * q);
                if (NODES || 4 * q < RWU) d[0] = make_uint2(v[i].x, v[i].y);
                if (4 * q + 2 < RWU) d[1] = make_uint2(v[i].z, v[i].w);  // the record's padding words are not kept
            }
        }
    }
}

// AGENTS: the instantiation that can generate scripted players' rows itself (evg_step_agents); the plain step
// leaves that code out, the kernel's instruction footprint being what its instruction cache misses are made of
// THREADS: 128 (a CTA = 4 warps sharing tables, barrier and instruction stream), or 32 for small batches: one warp
// per CTA spreads a few thousand matches over all SMs instead of a fifth of them.
// ROLL (with AGENTS, both players scripted): the launch plays A.n_turns game turns per batch (evg_rollout); a separate
// instantiation because the loop around the turn costs the single-turn kernel 4 % (0.544 vs 0.569 ms per 1 Mi matches)
// WIRE: the observation output is the packed wire row of include/evgsim.h (EVG_OBS_WIRE: 128 bytes per match on DemoMap,
// both players' observations + rewards + done in one cache line) instead of float32[2][obs_len] (840 bytes)
template <int NODES, int MAXSZ, typename HistT, int PITCH, bool AGENTS, int THREADS, bool WIRE = false, bool ROLL = false>
__global__ void __launch_bounds__(THREADS, THREADS == kTpmThreads ? kTpmMinCtas : kTpmLiteMinCtas) evg_step_tpm_kernel(const __grid_constant__ Tables T, const __grid_constant__ StepArgs A)
{
    extern __shared__ __align__(16) unsigned char smem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    // chunk of a 512-byte pair of records a lane moves in the whole-warp copies: lane bits 3 and 4 swapped, so that a
    // half-warp covers chunks 0..7 (or 8..15) of BOTH records and its 8-byte row accesses fall into 16 different bank pairs
    const int pl = (lane & 7) | ((lane >> 4) & 1) << 3 | ((lane >> 3) & 1) << 4;
    const int64_t nbatches = (A.n_envs + THREADS - 1) / THREADS;
    const bool ext_rows = A.agent[0] == EVG_AGENT_EXTERNAL || A.agent[1] == EVG_AGENT_EXTERNAL;
    // Software pipeline (compile-time map only: 16 chunks of 16 bytes per record): the NEXT batch's records and
    // action rows are requested into registers before this batch's observation phase, so their DRAM latency is
    // hidden behind a fifth of a batch's work instead of being exposed at the top of every batch
    // LITE = the one-warp-per-CTA instantiation for mid-size batches (a few thousand warps: one or two waves).  There the
    // number of RESIDENT warps decides, so everything a CTA would hold once is left out of shared memory — the static
    // tables and the constant observation entries are read from device memory through L1 instead (15.4 KB per CTA instead
    // of 19.7: 14 CTAs per SM instead of 11, 65,536 matches in ONE wave) — and the next-batch register pipeline, which a
    // CTA that runs one or two batches has no use for, gives its 71 registers back.
    constexpr bool LITE = THREADS == kTpmSmallThreads;
    // SEG (compile-time map): combat applies damage in segments of 8 unit slots, a group of 9..MAXSZ slots on two lanes
    constexpr bool SEG = NODES != 0 && MAXSZ > 8;
    constexpr int HVN = SEG ? 8 : MAXSZ;
    constexpr bool PIPE = NODES != 0 && !LITE && !ROLL;  // (a rollout loads records once per K turns: the pipeline's 71 registers are worth more to its turns)
    uint4 nxt[16];
    uint32_t nxa[7];
    bool have = false;
    auto request = [&](int64_t b) -> bool {
        const int64_t e0 = b * THREADS + warp * 32;
        if (b >= nbatches || e0 + 32 > A.n_envs) return false;  // partial warps take the direct path
        const uint4* g4 = reinterpret_cast<const uint4*>(A.records) + e0 * 16;
#pragma unroll
        for (int i = 0; i < 16; ++i) nxt[i] = __ldcs(g4 + pl + 32 * i);
#pragma unroll
        for (int k = 0; k < 7; ++k) nxa[k] = ext_rows ? __ldcs(reinterpret_cast<const uint32_t*>(A.actions) + (e0 + lane) * 7 + k) : 0u;
        return true;
    };
    if (PIPE) have = request(blockIdx.x);  // the first batch's records travel while the tables are staged
    // Batches are handed out DYNAMICALLY after the first wave (a CTA's first batch is its block index): matches in
    // different phases of the game cost different amounts (no fight / fights / in-place reset), and a static round-robin
    // leaves the SMs with the cheap batches idle at the end.  Thread 0 draws the batch after next from a global counter
    // ahead of the one CTA barrier of a batch and publishes it in shared memory; the counter pair (handed out, CTAs
    // finished) resets itself when the last CTA leaves.
    // (the two hand-over slots live in the CTA's copy of the tables: static shared memory would come off the opt-in limit)
    uint32_t first_draw = 0;
    if (!LITE && threadIdx.x == 0) first_draw = gridDim.x + atomicAdd(&A.sched[0], 1u);
    // ---- stage the static tables once per CTA
    if (!LITE) {   // from device memory with coalesced 16-byte loads (per-lane addresses into the parameter bank would be serialised)
        static_assert(sizeof(Tables) % 16 == 0, "Tables is copied in 16-byte pieces");
        uint4* dst = reinterpret_cast<uint4*>(smem);
        for (int i = threadIdx.x; i < (int)(sizeof(Tables) / 16); i += blockDim.x) dst[i] = __ldg(A.tables_dev + i);
    }
    const Tables* tables_ptr;  // (if constexpr: a pointer that could be either would be dereferenced with generic loads)
    if constexpr (LITE) tables_ptr = reinterpret_cast<const Tables*>(A.tables_dev);
    else tables_ptr = reinterpret_cast<const Tables*>(smem);
    const Tables& S = *tables_ptr;
    if (!LITE) __syncthreads();  // the run-time-sized instantiations read their sizes from the staged tables
    const Geo<NODES> G(S);
    const int n_nodes = G.n_nodes(), nn = G.nn(), RW = G.rec_words8() * 2, OL = G.obs_len();
    // the observation entries that never change (a third of them: the nodes' DEFENSE/OBSERVE flags in each viewer's
    // numbering and the groups' unit types) were converted to float once, by evg_bind (A.oconst_dev: 2*OL floats, then per
    // [player][viewer slot] the node's two flags); a CTA keeps a copy in shared memory, LITE reads them in place
    const int oc_floats = (2 * OL + 3) & ~3;
    const int oc_bytes = oc_floats * 4 + ((2 * n_nodes * 8 + 15) & ~15);
    const float* oconst;
    if constexpr (LITE) oconst = A.oconst_dev;
    else oconst = reinterpret_cast<const float*>(smem + T.sm_tables_bytes);
    const float2* ocpair = reinterpret_cast<const float2*>(oconst + oc_floats);
    volatile uint32_t* sched = reinterpret_cast<Tables*>(smem)->cta_sched;
    if (!LITE) {
        uint4* dst = reinterpret_cast<uint4*>(smem + T.sm_tables_bytes);
        for (int i = threadIdx.x; i < oc_bytes / 16; i += blockDim.x) dst[i] = __ldg(reinterpret_cast<const uint4*>(A.oconst_dev) + i);
        if (threadIdx.x == 0) {
            sched[0] = first_draw;
            // a sub-range launch (evg_step_host's chunks) covers global match ids that start further on
            reinterpret_cast<Tables*>(smem)->env_base += (uint32_t)A.env_first;
        }
        __syncthreads();
    }
    int par = 1;
    // (re-read from the tables where it is used: one more register held across the batch loop costs the 128-thread kernel 2 %)
    auto env_base_of = [&]() -> uint32_t { return LITE ? S.env_base + (uint32_t)A.env_first : S.env_base; };
    // player 1's node numbering (server.py:89): two registers of nibbles on the compile-time map, the byte table otherwise
    const uint64_t p1n = S.p1_nib;
    auto p1map = [&](uint32_t i) -> uint32_t { return NODES ? (uint32_t)(p1n >> (4 * i)) & 15u : (uint32_t)S.p1_map[i]; };
    int64_t next_batch = LITE ? (int64_t)blockIdx.x + gridDim.x : (int64_t)sched[0];
    const int P = PITCH ? PITCH : T.tpm_pitch;
    const int RWU = (kRecNode0 + n_nodes + 1) & ~1;  // record words a row keeps (the padding stays in global memory)
    // per warp: 32 rows (record + observation staging window), the node words of its 32 matches stored
    // word-major ([word][lane]: a thread's own accesses always hit bank `lane`, whatever the index), the pool
    const int WS = 32 * P + 64 * nn + T.tpm_pool_words;
    uint32_t* wrow = reinterpret_cast<uint32_t*>(smem + (LITE ? 0 : T.sm_tables_bytes + oc_bytes)) + (size_t)warp * WS;  // the warp's 32 rows
    uint32_t* R = wrow + (size_t)lane * P;  // my record
    uint32_t* wx = wrow + 32 * P;           // node words of the warp's matches: word i of match m at wx[32 * i + m]
    uint32_t* X = wx + lane;                // mine: X[32 * i]
    uint32_t* pool = wx + 64 * nn;          // the warp's histogram pool
    // persistent CTA: batches of 128 consecutive matches, round-robin over the grid; a warp only ever
    // touches its own 32 rows, so batches need no CTA-wide barrier
    for (int64_t batch = blockIdx.x; batch < nbatches;) {
    const int64_t warp_env0 = batch * THREADS + warp * 32;
    const int64_t env = warp_env0 + lane;
    const int64_t left = A.n_envs - warp_env0;
    const int nvalid = left >= 32 ? 32 : (left > 0 ? (int)left : 0);
    const bool valid = lane < nvalid;
    uint32_t aw[7];  // this turn's action rows (7 words per match)
    if (PIPE && have) {
        // ---- rows from the registers filled during the previous batch
#pragma unroll
        for (int k = 0; k < 7; ++k) aw[k] = nxa[k];
#pragma unroll
        for (int i = 0; i < 16; ++i) {
            const int f = pl + 32 * i, m = f >> 4, q = f & 15;
            uint2* d = reinterpret_cast<uint2*>(wrow + (size_t)m * P + 4 * q);
            d[0] = make_uint2(nxt[i].x, nxt[i].y);
            if (4 * q + 2 < RWU) d[1] = make_uint2(nxt[i].z, nxt[i].w);  // the record's padding words are not kept
        }
    } else {
        // ---- cooperative, coalesced load of the warp's records into the per-thread rows
        // (action rows requested before the records so the latencies overlap)
#pragma unroll
        for (int k = 0; k < 7; ++k) aw[k] = (valid && ext_rows) ? __ldcs(reinterpret_cast<const uint32_t*>(A.actions) + env * 7 + k) : 0u;
        load_rows_direct<NODES>(A, wrow, P, RW, RWU, warp_env0, nvalid, lane, !PIPE, next_batch * THREADS + warp * 32);
    }
    __syncwarp();

    uint32_t turn = 0, episode = 0;
    int s0 = 0, s1 = 0, status = 0;
    bool done = false;
    float r0 = 0.f, r1 = 0.f;
    bool reset_now = false;
    // Fully scripted self-play (evg_rollout): the batch stays in its rows for A.n_turns game turns — only the last one
    // pays for the observations and the record write-back, none for a launch.  Every other call runs the body once.
    const int n_turns = ROLL ? A.n_turns : 1;
#pragma unroll 1
    for (int tt = 0; tt < n_turns; ++tt) {
    const bool last = !ROLL || tt + 1 == n_turns;
    if (ROLL) { s0 = 0; s1 = 0; status = 0; }
    if (valid) {
        turn = R[kRecTurn] + 1u;  // server.py:214
        episode = R[kRecEpisode];

        // ---- action decode + validation, server.py:218-271 (rows in order; first valid row per group wins)
        {
            // rows of scripted players are generated here (agents/State_Machine/random_actions.py:38-46, tape
            // domain 1) instead of being read: no action buffer traffic, no second kernel
            uint32_t rows[2 * EVG_MAX_ACTIONS];
#pragma unroll
            for (int r = 0; r < 2 * EVG_MAX_ACTIONS; ++r) rows[r] = (aw[r >> 1] >> (16 * (r & 1))) & 0xFFFFu;
            if (AGENTS && (A.agent[0] != EVG_AGENT_EXTERNAL || A.agent[1] != EVG_AGENT_EXTERNAL)) {
                // the observation-driven agents read what obs[45 + 5g], obs[45 + 5g + 3] hold from the row itself; their
                // per-(match, player) state lives in the bound agents array, like the reference's agent objects
                auto w0_of = [&](int L) -> uint32_t { return R[2 * L]; };
#pragma unroll
                for (int pl = 0; pl < 2; ++pl) {
                    uint32_t* pr = rows + pl * EVG_MAX_ACTIONS;
                    if (A.agent[pl] == EVG_AGENT_RANDOM) {
                        agent_random_rows(env_base_of() + (uint32_t)env, turn, episode, pl, n_nodes, S.seed_lo, S.seed_hi, pr);
                    } else if (A.agent[pl] != EVG_AGENT_EXTERNAL) {
                        uint2 st = A.agent_state[env * 2 + pl];
                        if (A.agent[pl] == EVG_AGENT_BASE_RUSH) agent_base_rush_rows(S, w0_of, st, pl, pr);
                        else agent_swarm_rows(S, w0_of, st, env_base_of() + (uint32_t)env, turn, episode, pl, pr);
                        A.agent_state[env * 2 + pl] = st;
                    }
                }
                if (A.actions_out) {
                    uint32_t* ao = reinterpret_cast<uint32_t*>(A.actions_out) + env * 7;
#pragma unroll
                    for (int k = 0; k < 7; ++k) ao[k] = rows[2 * k] | rows[2 * k + 1] << 16;
                }
            }
            // all 14 rows are decoded and looked up first (independent shared-memory reads in flight together:
            // accepting a row changes neither the group's location nor its moving flag), then resolved in order
            int Lr[2 * EVG_MAX_ACTIONS];
            uint32_t neww[2 * EVG_MAX_ACTIONS];
            uint32_t okrows = 0;
#pragma unroll
            for (int r = 0; r < 2 * EVG_MAX_ACTIONS; ++r) {
                const uint32_t a = rows[r];
                const int ag = (int)(int8_t)(a & 0xFFu);
                int an = (int)(int8_t)(a >> 8);
                const int pl = r >= EVG_MAX_ACTIONS ? 1 : 0;
                const bool okg = (unsigned)ag < (unsigned)EVG_NUM_GROUPS;
                an = (unsigned)an <= (unsigned)n_nodes ? an : 0;
                if (pl) an = (int)p1map((uint32_t)an);  // server.py:233-234
                const int L = pl * EVG_NUM_GROUPS + (okg ? ag : 0);
                const uint32_t gw0 = R[2 * L];
                EVG_CHECK(L >= 0 && L < kGroupLanes && (gw0 & W0_LOC_MASK) >= 1 && (gw0 & W0_LOC_MASK) <= (uint32_t)n_nodes && an >= 0 && an <= n_nodes);
                const uint32_t d = S.edge[gw0 & W0_LOC_MASK][an];
                Lr[r] = L;
                if (okg && !(gw0 & W0_MOVING) && d) okrows |= 1u << r;  // t2 (not moving) and t3 (adjacent), :243-250
                neww[r] = (gw0 & ~((0x3Fu << W0_DEST_SHIFT) | (0xFFu << W0_DIST_SHIFT))) | (uint32_t)an << W0_DEST_SHIFT |
                          d << W0_DIST_SHIFT | W0_READY;  // :267-270
            }
            uint32_t used = 0;
#pragma unroll
            for (int r = 0; r < 2 * EVG_MAX_ACTIONS; ++r) {
                const bool ok = ((okrows >> r) & 1u) && !((used >> Lr[r]) & 1u);  // t1: the group has no accepted command yet, :241
                if (ok) {
                    used |= 1u << Lr[r];
                    R[2 * Lr[r]] = neww[r];
                }
            }
        }

        // (combat runs warp-cooperatively below, outside this per-thread block)
    }

    // ---- combat, server.py:503-654
    {
        // per-thread preparation.  Node words (word-major, X[32 * i]): i = x for player 0 and nn + x for player 1 hold, per node,
        // member mask of the groups present [0:12) | their alive units [16:24) | histogram base of that side [24:32)
        uint32_t fm = 0;          // my match's fighting groups (bit L = side * 12 + gid)
        uint32_t xm = 0;          // those of them whose second draw block is a work item
        uint32_t b0 = 0, b1 = 0;  // histogram entries per side = alive units of the fighting groups
        uint32_t my_slots = 0;    // unit slots of my match's fighting groups (ST_FOUGHT)
        if (valid) {
            for (int i = 0; i < 2 * nn; ++i) X[32 * i] = 0;
            {
                uint32_t* __restrict__ acc0 = X;
                uint32_t* __restrict__ acc1 = X + 32 * nn;
#pragma unroll 4
                for (int g = 0; g < EVG_NUM_GROUPS; ++g) {  // listed and not in transit, :516-535; entry 0 takes the rest
                    const uint2 wa = *reinterpret_cast<const uint2*>(R + 2 * g);
                    const uint2 wb = *reinterpret_cast<const uint2*>(R + 2 * (EVG_NUM_GROUPS + g));
                    const uint32_t aa = wa.y & 0xFFFFu, ab = wb.y & 0xFFFFu;
                    const bool pa = aa && !(wa.x & W0_MOVING), pb = ab && !(wb.x & W0_MOVING);
                    const uint32_t la = pa ? wa.x & W0_LOC_MASK : 0u, lb = pb ? wb.x & W0_LOC_MASK : 0u;
                    EVG_CHECK(la <= (uint32_t)n_nodes && lb <= (uint32_t)n_nodes);
                    // shared-memory reductions (no value returned): one instruction per update and nothing to wait for
                    atomicAdd(&acc0[32 * la], 1u << g | (uint32_t)__popc(aa) << 16);
                    atomicAdd(&acc1[32 * lb], 1u << g | (uint32_t)__popc(ab) << 16);
                }
            }
            for (int x = 1; x <= n_nodes; ++x) {
                const uint32_t a = X[32 * x], b = X[32 * (nn + x)];
                if ((a & 0xFFFu) && (b & 0xFFFu)) {  // both players present: contested, :539
                    fm |= (a & 0xFFFu) | (b & 0xFFFu) << EVG_NUM_GROUPS;
                    X[32 * x] = a | b0 << 24;  // np.sum(counts[pid]) at [16:24) (:552-553), node-local uid -> histogram entry base
                    X[32 * (nn + x)] = b | b1 << 24;
                    b0 += a >> 16;
                    b1 += b >> 16;
                }
            }
            // a fighting group with more than 8 units alive draws from two Philox blocks: its second block becomes
            // a work item of its own (a lane running both blocks would hold up its whole round for a second pass)
            // (SEG, the compile-time map: EVERY fighting group of more than 8 unit slots has a second item, which also
            // applies the damage to slots 8.. — the round's apply then runs over 8 slots per lane instead of 12)
            if (SEG) xm = fm & S.big_mask;
            else if (S.n_big <= 8)
                for (uint32_t m = fm & S.big_mask; m; m &= m - 1) {
                    const int L = __ffs(m) - 1;
                    if (__popc(R[2 * L + 1] & 0xFFFFu) > 8) xm |= 1u << L;
                }
            // the health rows of the groups that will fight: start them towards L2 now
            if (fm) {
                const char* he = reinterpret_cast<const char*>(A.health + env * S.health_slots);
                uint32_t slots = 0;
                for (uint32_t m = fm; m; m &= m - 1) {
                    const int L = __ffs(m) - 1;
                    const char* hr = he + (size_t)S.g_slot[L] * 8;
                    const uint32_t size = S.g_size[L];
                    asm volatile("prefetch.global.L2 [%0];" ::"l"(hr));
                    if (size > 8) asm volatile("prefetch.global.L2 [%0];" ::"l"(hr + 64));
                    slots += size;
                }
                // ST_FOUGHT: unit slots whose health this turn's combat reads; gathered per CTA in a spare table word
                // (LITE has no shared-memory tables: summed over the warp below)
                if (LITE) my_slots = slots;
                else atomicAdd(&reinterpret_cast<Tables*>(smem)->cta_fought, slots);
            }
        }
        __syncwarp();  // rows (actions applied, node words) are read by other lanes from here on
        if (LITE) {
            const uint32_t tot = __reduce_add_sync(0xFFFFFFFFu, my_slots);
            if (lane == 0 && tot) atomicAdd(&A.stats[ST_FOUGHT], (unsigned long long)tot);
        }
        // the warp's work list = concatenation of the matches' fighting groups (then their second draw blocks); a
        // round takes whole matches (a match has <= 32 items), so draws and apply of one match stay in one round and the
        // round's histograms fit the warp's pool: match m owns entries [upre[m] - upre[m_begin], +b0+b1)
        const int nitems = __popc(fm) + __popc(xm);
        int incl = nitems;
        uint32_t uincl = b0 + b1;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int t = __shfl_up_sync(0xFFFFFFFFu, incl, o);
            const uint32_t u = __shfl_up_sync(0xFFFFFFFFu, uincl, o);
            if (lane >= o) { incl += t; uincl += u; }
        }
        const int pre = incl - nitems;
        const uint32_t ub = (uincl - (b0 + b1)) | b0 << 16;  // entries before my match [0:16) | my side-0 entries [16:24)
        const int total = __shfl_sync(0xFFFFFFFFu, incl, 31);
        int m_begin = 0;
        while (total && m_begin < 32) {
            const int base = __shfl_sync(0xFFFFFFFFu, pre, m_begin);
            const int m_end = __popc(__ballot_sync(0xFFFFFFFFu, incl - base <= 32));
            const int nround = __shfl_sync(0xFFFFFFFFu, incl, m_end - 1) - base;
            const uint32_t ubase = __shfl_sync(0xFFFFFFFFu, ub, m_begin) & 0xFFFFu;
            const uint32_t uround = __shfl_sync(0xFFFFFFFFu, uincl, m_end - 1) - ubase;
            {
                const uint32_t zw = (uround * (uint32_t)sizeof(HistT) + 3u) / 4u;
#pragma unroll
                for (int j = 0; j < (MAXSZ * (int)sizeof(HistT) * 32 / 4 + 31) / 32; ++j)
                    if ((uint32_t)(lane + 32 * j) < zw) pool[lane + 32 * j] = 0;
            }
            const int q = base + lane;
            int m = 0;  // largest m with pre[m] <= q
#pragma unroll
            for (int step = 16; step; step >>= 1) {
                const int cand = m + step;
                const int pc = __shfl_sync(0xFFFFFFFFu, pre, cand & 31);
                if (cand < 32 && pc <= q) m = cand;
            }
            EVG_CHECK(m >= 0 && m < 32 && nround >= 1 && nround <= 32 && m_end > m_begin && m_end <= 32);
            EVG_CHECK((uround * (uint32_t)sizeof(HistT) + 3u) / 4u <= (uint32_t)T.tpm_pool_words);
            const int pm = __shfl_sync(0xFFFFFFFFu, pre, m);
            const uint32_t fmm = __shfl_sync(0xFFFFFFFFu, fm, m), xmm = __shfl_sync(0xFFFFFFFFu, xm, m);
            const uint32_t ubm = __shfl_sync(0xFFFFFFFFu, ub, m);
            const bool act = lane < nround;
            // item state kept across the two phases
            uint32_t* Rm = wrow + (size_t)m * P;
            const uint32_t* Xm = wx + m;
            int L = 0, side = 0, x = 1, tb = 0;
            uint32_t alive_seg = 0;
            uint32_t w0 = 0, w1 = 0, gf = 0;
            double hv[HVN];
            double* hp = A.health;
            const int nf = __popc(fmm);
            const bool extra = act && q - pm >= nf;  // a second draw block (SEG: and the group's unit slots from 8 on)
            int seg_size = 0;
            const bool own_item = act && !extra;
            __syncwarp();  // pool zeroed
            if (act) {
                L = extra ? kth_set_bit(xmm, q - pm - nf) : kth_set_bit(fmm, q - pm);
                EVG_CHECK(L >= 0 && L < kGroupLanes && (!act || (m >= m_begin && m < m_end)));
                gf = S.g_fight[L];  // health slot | unit slots << 12 | damage << 17 | unit type << 25
                if (SEG) {
                    const int size = (int)((gf >> 12) & 31u);
                    seg_size = extra ? size - 8 : min(size, 8);
                    hp = A.health + (warp_env0 + m) * S.health_slots + (gf & 0xFFFu) + (extra ? 8 : 0);
                    EVG_CHECK(warp_env0 + m < A.n_envs && (!extra || size > 8) && (int)(gf & 0xFFFu) + (size + 3) / 4 * 4 <= S.health_slots);
                    load_group<HVN>(hp, seg_size, hv);  // consumed after the draws
                } else if (!extra) {
                    hp = A.health + (warp_env0 + m) * S.health_slots + (gf & 0xFFFu);
                    EVG_CHECK(warp_env0 + m < A.n_envs && (int)(gf & 0xFFFu) + ((int)((gf >> 12) & 31u) + 3) / 4 * 4 <= S.health_slots);
                    load_group<HVN>(hp, (int)((gf >> 12) & 31u), hv);  // consumed after the draws
                }
                side = L >= EVG_NUM_GROUPS ? 1 : 0;
                const int gg = L - side * EVG_NUM_GROUPS;
                {
                    const uint2 w = *reinterpret_cast<const uint2*>(Rm + 2 * L);
                    w0 = w.x;
                    w1 = w.y;
                }
                x = (int)(w0 & W0_LOC_MASK);
                EVG_CHECK(x >= 1 && x <= n_nodes);
                const uint32_t cnt = __popc(w1 & 0xFFFFu);
                const uint32_t own = Xm[32 * (side * nn + x)], opp = Xm[32 * ((1 - side) * nn + x)];
                const uint32_t n = (opp >> 16) & 0xFFu;                        // opposing units at the node
                const uint32_t mb = (ubm & 0xFFFFu) - ubase, mb0 = ubm >> 16;  // my match's pool entries; its side-0 count
                const uint32_t hb = mb + (side ? 0u : mb0) + (opp >> 24);      // opposing histogram base at this node
                if (SEG || !extra) {
                    tb = (int)(mb + (side ? mb0 : 0u) + (own >> 24));          // my side's base at this node
                    // my group's range starts after the groups listed before it (arrival order, then gid:
                    // node.groups[pid], :198,690-691); sibling counts are still pre-combat here
                    const uint32_t key = (w1 >> 16) << 4 | (uint32_t)gg;
                    for (uint32_t sm = (own & 0xFFFu) & ~(1u << gg); sm; sm &= sm - 1) {
                        const int g = __ffs(sm) - 1;
                        const uint32_t w1g = Rm[2 * (side * EVG_NUM_GROUPS + g) + 1];
                        if (((w1g >> 16) << 4 | (uint32_t)g) < key) tb += __popc(w1g & 0xFFFFu);
                    }
                }
                // draws, :549-566: unit j targets uid = tape(...) among the opposing units at the node and adds
                // its type's damage to infliction[uid]; 8 draws of 16 bits per Philox block (oracle/tape.py).
                // This item draws for units [8 * jb, 8 * jb + nd)
                const uint32_t jb = extra ? 1u : 0u;
                const uint32_t nd = SEG ? (extra ? (cnt > 8u ? cnt - 8u : 0u) : min(cnt, 8u)) : (extra ? cnt - 8u : (((xmm >> L) & 1u) ? 8u : cnt));
                const uint32_t dmg = (gf >> 17) & 0xFFu;
                const uint2 te = *reinterpret_cast<const uint2*>(Rm + kRecTurn);  // turn, episode
                const uint32_t turn_m = te.x + 1u, ep_m = te.y;
                for (uint32_t b = jb; 8u * (b - jb) < nd; ++b) {
                    uint32_t r[4];
                    philox4x32_10(env_base_of() + (uint32_t)(warp_env0 + m), turn_m,
                                  (uint32_t)x | (uint32_t)side << 8 | (uint32_t)gg << 16 | b << 24, ep_m << 8, S.seed_lo, S.seed_hi, r);
#pragma unroll
                    for (uint32_t k = 0; k < 8; ++k)
                        if (8u * (b - jb) + k < nd) {
                            const uint32_t half = (k & 1) ? r[k >> 1] >> 16 : r[k >> 1] & 0xFFFFu;
                            const uint32_t idx = hb + ((half * n) >> 16);
                            EVG_CHECK(n >= 1 && idx < uround);
                            if (sizeof(HistT) == 1) atomicAdd(&pool[idx >> 2], dmg << ((idx & 3u) * 8));
                            else atomicAdd(&pool[idx >> 1], dmg << ((idx & 1u) * 16));
                        }
                }
            }
            __syncwarp();
            // apply, :573-643: both sides drew on pre-combat counts (:572); one lane updates one whole group
            if (SEG ? act : own_item) {
                const int type = (int)(gf >> 25);
                constexpr bool FMA_ONLY = NODES != 0;  // the compile-time map's kernel is only picked when Tables::fast_div holds
                const uint32_t nwd = Rm[kRecNode0 + x - 1];
                const int cb = (int)(int8_t)((nwd >> 16) & 0xFFu);
                const int bonus = (cb == side ? 1 : 0) + ((S.node_flags[x] >> 2) & 1);
                const int ti = (type * nn + x) * 3 + bonus;
                const double divisor = __dadd_rn(S.unit_armor[type], __dmul_rn((double)bonus, S.node_def[x]));
                const double* ltab = FMA_ONLY || S.fast_div ? nullptr : S.loss_tab + (size_t)ti * kLossD;
                const double rcp = FMA_ONLY || S.fast_div ? __ldg(S.rcp_tab + ti) : 0.0;
                EVG_CHECK(tb >= 0 && (uint32_t)tb + (uint32_t)__popc(w1 & 0xFFFFu) <= uround && ti >= 0);
                if constexpr (SEG) {
                    // my segment: slots [0, 8) of the group, or [8, size) whose histogram entries follow the first segment's
                    alive_seg = apply_units<HVN, HistT, FMA_ONLY>(hp, hv, seg_size, extra ? (w1 >> 8) & 0xFFu : w1 & 0xFFu, reinterpret_cast<const HistT*>(pool),
                                                                  extra ? tb + __popc(w1 & 0xFFu) : tb, ltab, divisor, rcp);
                } else {
                    int avg;
                    const uint32_t alive = apply_group<HVN, HistT, FMA_ONLY>(hp, hv, (int)((gf >> 12) & 31u), w1 & 0xFFFFu, reinterpret_cast<const HistT*>(pool),
                                                                             tb, ltab, divisor, &avg, rcp);
                    // alive == 0: destroyed, leaves the node list (:623-627)
                    *reinterpret_cast<uint2*>(Rm + 2 * L) = make_uint2((w0 & ~(127u << W0_AVG_SHIFT)) | ((uint32_t)avg & 127u) << W0_AVG_SHIFT,
                                                                       (w1 & 0xFFFF0000u) | alive);
                }
            }
            if constexpr (SEG) {
                // a group of more than 8 slots: its first lane collects the second segment's outcome, then alive mask and
                // avg health (numpy's pairwise sum over all of its slots, :480-491) as for any other group
                const bool big = own_item && ((xmm >> L) & 1u);
                uint32_t alive_hi = 0;
                double hi[MAXSZ - 8];
#pragma unroll
                for (int k = 0; k < MAXSZ - 8; ++k) hi[k] = 0.0;
                if (__ballot_sync(0xFFFFFFFFu, extra)) {
                    const int src = big ? pm + nf + __popc(xmm & ((1u << L) - 1u)) - base : lane;
                    EVG_CHECK(src >= 0 && src < 32 && (!big || src < nround));
                    alive_hi = __shfl_sync(0xFFFFFFFFu, alive_seg, src);
#pragma unroll
                    for (int k = 0; k < MAXSZ - 8; ++k) hi[k] = __shfl_sync(0xFFFFFFFFu, hv[k], src);
                }
                if (own_item) {
                    const int size = (int)((gf >> 12) & 31u);
                    const uint32_t alive = alive_seg | (big ? alive_hi << 8 : 0u);
                    const double hsum = big ? np_sum_split<MAXSZ - 8>(hv, hi, size) : np_sum_regs<HVN>(hv, size);
                    const int avg = alive ? int_quotient(hsum, __popc(alive)) : 0;  // int((health*1.)/units_alive), :491
                    // alive == 0: destroyed, leaves the node list (:623-627)
                    *reinterpret_cast<uint2*>(Rm + 2 * L) = make_uint2((w0 & ~(127u << W0_AVG_SHIFT)) | ((uint32_t)avg & 127u) << W0_AVG_SHIFT,
                                                                       (w1 & 0xFFFF0000u) | alive);
                }
            }
            __syncwarp();
            m_begin = m_end;
        }
    }

    if (PIPE && last) have = request(next_batch);  // in flight through movement, capture and the observations
    if (valid) {
        // ---- movement (server.py:656-706) fused with the per-(side,node) sums capture and observations need:
        //   [0:10) units of all listed groups (:446-449), [10:24) count*control of non-moving groups (:718-724),
        //   [24:29) number of non-moving groups (:725-726); plus unit points for the score (:313-317)
        for (int i = 0; i < 2 * nn; ++i) X[32 * i] = 0;
        bool any_alive = false;
        {
            uint32_t* __restrict__ acc0 = X;
            uint32_t* __restrict__ acc1 = X + 32 * nn;
            // written with selects: the four cases (idle, ready, under way, arriving) differ per match, so branches
            // would run them one after the other
            auto move = [&](int L, uint32_t gm, uint32_t& v, uint32_t& loc, int& pts) {
                const uint2 w = *reinterpret_cast<const uint2*>(R + 2 * L);
                const uint32_t w0 = w.x, alive = w.y & 0xFFFFu;
                const bool live = alive != 0;  // destroyed groups are skipped, :663
                const bool rdy = (w0 & W0_READY) != 0, mov = (w0 & W0_MOVING) != 0;
                const int dist = (int)((w0 >> W0_DIST_SHIFT) & 0xFFu) - (int)(gm & 0xFFu);  // :671
                const bool arrive = live && !rdy && mov && dist <= 0;
                const uint32_t w_rdy = (w0 & ~W0_READY) | W0_MOVING;  // first turn only flips ready -> moving (:664-667)
                const uint32_t w_arr = (w0 & (127u << W0_AVG_SHIFT)) | ((w0 >> W0_DEST_SHIFT) & 0x3Fu);  // appended to the destination's list (:678-695)
                const uint32_t w_go = (w0 & ~(0xFFu << W0_DIST_SHIFT)) | ((uint32_t)dist & 0xFFu) << W0_DIST_SHIFT;
                uint32_t n0 = rdy ? w_rdy : (mov ? (dist <= 0 ? w_arr : w_go) : w0);
                n0 = live ? n0 : w0;
                R[2 * L] = n0;
                if (arrive) R[2 * L + 1] = alive | turn << 16;
                const uint32_t cnt = __popc(alive);
                const uint32_t hold = (n0 & W0_MOVING) ? 0u : ((cnt * ((gm >> 8) & 0xFFu)) << 10 | 1u << 24);
                v = live ? (cnt | hold) : 0u;
                loc = live ? (n0 & W0_LOC_MASK) : 0u;
                pts = (int)(cnt * (gm >> 16));
                any_alive |= live;
            };
            // rolled: the footprint costs more than the overlap buys (unrolled 1: 0.4965 ms, 2: 0.4983, 3: 0.5016,
            // 4: 0.5078 per 1 Mi match-turns)
#pragma unroll 1
            for (int g = 0; g < EVG_NUM_GROUPS; ++g) {
                uint32_t va, la, vb, lb;
                int pa, pb;
                const uint2 gm = *reinterpret_cast<const uint2*>(&S.g_move[2 * g]);  // {player 0's, player 1's}: speed | control << 8 | cost << 16
                move(g, gm.x, va, la, pa);
                move(EVG_NUM_GROUPS + g, gm.y, vb, lb, pb);
                EVG_CHECK(la <= (uint32_t)n_nodes && lb <= (uint32_t)n_nodes);
                atomicAdd(&acc0[32 * la], va);  // entry 0 collects the (zero) contributions of dead groups
                atomicAdd(&acc1[32 * lb], vb);
                s0 += pa;
                s1 += pb;
            }
        }

        // ---- capture (server.py:708-767; current_turn > 0 here) and node scoring (server.py:298-310)
        bool basecap = false;
        const int capture_bonus = S.capture_bonus;
#pragma unroll 1
        for (int n = 1; n <= n_nodes; ++n) {
            const uint32_t nw = R[kRecNode0 + n - 1];
            int cs = (int)(int16_t)(nw & 0xFFFFu), cb = (int)(int8_t)((nw >> 16) & 0xFFu);
            const uint32_t a0 = X[32 * n], a1 = X[32 * (nn + n)];
            const bool c0 = (a0 >> 24) != 0, c1 = (a1 >> 24) != 0;
            const uint32_t ncap = S.node_cap[n];  // control points | (TeamStart + 1) << 16
            const int cp = (int)(ncap & 0xFFFFu);
            const int pid = c1 ? 1 : 0;
            const bool upd = c0 != c1 && (abs(cs) < cp || pid != cb);  // exactly one controller (:729), :731-732
            {
                const int pts = (int)(((pid ? a1 : a0) >> 10) & 0x3FFFu), pxer = pid ? -1 : 1;
                int cs2 = cs + pts * pxer;
                const bool neutralize = (cs < 0) != (cs2 < 0);  // :747-750, zero counts as player 0's sign
                const bool full = abs(cs2) >= cp;                 // :763-765
                cs2 = full ? cp * pxer : cs2;
                int cb2 = full ? pid : cb;
                cb2 = neutralize ? -1 : cb2;  // :766-767
                cs = upd ? cs2 : cs;
                cb = upd ? cb2 : cb;
                if (upd) R[kRecNode0 + n - 1] = ((uint32_t)cs & 0xFFFFu) | ((uint32_t)cb & 0xFFu) << 16;
            }
            const int ts = (int)(ncap >> 16) - 1;
            const bool bc = ts != -1 && cb != -1 && cb != ts;
            basecap |= bc;
            const int bonus = bc ? capture_bonus : 0;
            const int npts = abs(cs) == cp ? 2 * cp : abs(cs);
            s0 += (cb ? 0 : bonus) + (cs > 0 ? npts : 0);
            s1 += (cb ? bonus : 0) + (cs < 0 ? npts : 0);
        }
        if ((int)turn >= S.turn_limit) status = EVG_STATUS_TIME_EXPIRED;  // server.py:321-328, in that priority
        else if (!any_alive) status = EVG_STATUS_ANNIHILATION;
        else if (basecap) status = EVG_STATUS_BASE_CAPTURE;
        done = status != 0;

        // ---- reward / done, env.py:37-60 (float32 division == float32(float64 quotient), tests/test_tape.py)
        if (done) {
            r0 = s0 > s1 ? 1.f : 0.f;
            r1 = s1 > s0 ? 1.f : (s1 < s0 ? -1.f : 0.f);
        } else {
            r0 = __fdiv_rn((float)s0, S.max_score_f);
            r1 = __fdiv_rn((float)s1, S.max_score_f);
        }
        if (last) {
            reinterpret_cast<float2*>(A.reward)[env] = make_float2(r0, r1);
            A.done[env] = done ? 1 : 0;
            if (A.status) A.status[env] = (uint8_t)status;
            if (A.scores) reinterpret_cast<int2*>(A.scores)[env] = make_int2(s0, s1);
        }
    }
    reset_now = valid && done && S.auto_reset != EVG_AUTORESET_OFF;
    // ---- episode end: statistics, aggregated over the warp before touching the global counters
    if (const uint32_t rmask = __ballot_sync(0xFFFFFFFFu, reset_now)) {
        episode_stats(A.stats, reset_now, s0, s1, turn, status, lane);
        refill_health(A.health + warp_env0 * S.health_slots, S.health_slots, rmask, lane);
    }
    if (reset_now && S.auto_reset == EVG_AUTORESET_NEXT) {
        reset_row(S, R, n_nodes, X);
        turn = 0;
        episode += 1;
    }
    if (ROLL && !last) {  // on to the next turn of the rollout (nobody sees this turn's terminal observation)
        if (reset_now && S.auto_reset == EVG_AUTORESET_TERMINAL) {
            reset_row(S, R, n_nodes);
            turn = 0;
            episode += 1;
        }
        if (valid) {
            R[kRecTurn] = turn;
            R[kRecEpisode] = episode;
        }
        __syncwarp();
    }
    }  // turns of a rollout

    if (!LITE && threadIdx.x == 0) sched[par] = gridDim.x + atomicAdd(&A.sched[0], 1u);  // the batch after next
    // the CTA's one barrier of a batch: it keeps the four warps on the same instructions through the observation code,
    // and the batch hand-over relies on it (sched[par], written above, is read below by every thread)
    __syncthreads();
    const int64_t after_next = LITE ? next_batch + gridDim.x : (int64_t)sched[par];
    par ^= 1;

    // ---- observations: board_state (server.py:382-455) + player_state (:457-501) + concat (env.py:158-171).
    // Each thread packs kTpmStage words at a time into the staging window of its row; the warp streams the
    // windows out as contiguous 8-byte runs (64 / kTpmStage matches x 4 * kTpmStage bytes per store instruction).
    // The output row of a match is either float32[2][obs_len] (the reference's vector) or, WIRE, the packed row of
    // include/evgsim.h (EVG_OBS_WIRE) that holds the same information once, with the step's rewards and done flag.
    {
        constexpr int SP = kTpmStage / 2;   // 8-byte pairs per window
        constexpr int MPI = 32 / SP;        // matches per store instruction
        uint2* stage = reinterpret_cast<uint2*>(R + RWU);  // P and RWU are even: 8-byte aligned
        const int stage_off = RWU;
        const int WW = (EVG_WIRE_NODE0 + 4 * n_nodes + 3 * kGroupLanes + 8 + 15) / 16 * 4;  // words of a wire row
        const int npairs = WIRE ? WW / 2 : OL;  // 8-byte pairs per match (2*OL floats = OL pairs)
        uint32_t* obs_base = reinterpret_cast<uint32_t*>(A.obs) + warp_env0 * 2 * npairs;
        auto value = [&](int f) -> uint32_t {  // float32 format: the bits of entry f of the match's 2*OL floats
            const int p = f >= OL ? 1 : 0, i = f - p * OL;
            if (i == 0) return __float_as_uint((float)turn);
            if (i < 1 + 4 * n_nodes) {
                const int k = (i - 1) >> 2, j = (i - 1) & 3;
                const int x = p ? (int)p1map((uint32_t)(k + 1)) : k + 1;  // server.py:437-439
                if (j < 2) {  // 'DEFENSE' / 'OBSERVE' in resource, :442-443: both flags of a node from one 8-byte load
                    const float2 c2 = ocpair[p * n_nodes + k];
                    return __float_as_uint(j ? c2.y : c2.x);
                }
                if (j == 2) return __float_as_uint((float)(int)(int16_t)(R[kRecNode0 + x - 1] & 0xFFFFu));  // raw sign for both viewers
                return __float_as_uint((float)(X[32 * ((p ? 0 : nn) + x)] & 1023u));                          // opposing listed units
            }
            const int q = i - 1 - 4 * n_nodes, g = q / 5, j = q - 5 * g;
            const int L = p * EVG_NUM_GROUPS + g;
            const uint2 w = *reinterpret_cast<const uint2*>(R + 2 * L);  // one 8-byte load serves a group's five entries
            const uint32_t w0 = w.x;
            if (j == 0) return __float_as_uint((float)(p ? p1map(w0 & W0_LOC_MASK) : (w0 & W0_LOC_MASK)));
            if (j == 1) return __float_as_uint(oconst[f]);  // unit type id
            if (j == 2) return __float_as_uint((float)((w0 >> W0_AVG_SHIFT) & 127u));
            if (j == 3) return __float_as_uint((float)((w0 >> 21) & 1u));
            return __float_as_uint((float)__popc(w.y & 0xFFFFu));
        };
        // wire format: a group's three bytes = location (real numbering) | moving << 6, avg health, units alive
        auto gwire = [&](int L) -> uint32_t {
            const uint2 w = *reinterpret_cast<const uint2*>(R + 2 * L);
            return (w.x & W0_LOC_MASK) | ((w.x >> 21) & 1u) << 6 | ((w.x >> W0_AVG_SHIFT) & 127u) << 8 | (uint32_t)__popc(w.y & 0xFFFFu) << 16;
        };
        auto wire = [&](int w) -> uint32_t {  // word w of the wire row
            if (w == 0) return turn | (done ? 1u : 0u) << 16 | (uint32_t)status << 24;
            if (w <= n_nodes)  // node w: controlState int16, listed units of player 0, of player 1 (:446-449)
                return (R[kRecNode0 + w - 1] & 0xFFFFu) | (X[32 * w] & 255u) << 16 | (X[32 * (nn + w)] & 255u) << 24;
            const int wi = w - 1 - n_nodes;
            if (wi < 18) {  // 24 groups x 3 bytes = 6 quads of 3 words
                const int q = wi / 3, r = wi - 3 * q;
                const uint32_t a = gwire(4 * q + r), b = gwire(4 * q + r + 1);
                return r == 0 ? (a | b << 24) : r == 1 ? (a >> 8 | b << 16) : (a >> 16 | b << 8);
            }
            if (wi == 18) return __float_as_uint(r0);
            if (wi == 19) return __float_as_uint(r1);
            return 0u;
        };
        const int sub = lane / SP, cp = lane % SP;
        const int nchunks = (npairs + SP - 1) / SP;
        constexpr int kFastChunks = WIRE ? ((EVG_WIRE_NODE0 + 4 * NODES + 3 * kGroupLanes + 8 + 15) / 16 * 2 + SP - 1) / SP
                                         : (1 + 4 * NODES + 60 + SP - 1) / SP;
#pragma unroll
        for (int c = 0; c < (NODES ? kFastChunks : nchunks); ++c) {
            if (valid) {
                // reads first (they can be merged and overlapped), then the staging stores — in kSplit groups per window:
                // fewer values alive at once next to the 71 registers of the record pipeline (2 groups: 0.5004 ms, 1: 0.5024,
                // 4: 0.5044)
                constexpr int kSplit = 2;
                constexpr int GP = SP / kSplit;  // pairs per group
#pragma unroll
                for (int h = 0; h < kSplit; ++h) {
                    uint32_t vals[2 * GP];
#pragma unroll
                    for (int k = 0; k < 2 * GP; ++k) {
                        const int f = 2 * SP * c + 2 * GP * h + k;
                        vals[k] = f < 2 * npairs ? (WIRE ? wire(f) : value(f)) : 0u;
                    }
#pragma unroll
                    for (int k = 0; k < GP; ++k)
                        if (SP * c + GP * h + k < npairs) stage[GP * h + k] = make_uint2(vals[2 * k], vals[2 * k + 1]);
                }
            }
            __syncwarp();
            const int pr = SP * c + cp;
            if (pr < npairs) {
                const uint32_t* srow = wrow + stage_off + 2 * cp;
                uint32_t* orow = obs_base + 2 * pr;
                if (nvalid == 32) {  // whole warp: no per-match predicates
                    // 16 iterations, unrolled by 4: 0.4924 ms (8: 0.4942, 16: 0.4965, 2: 0.4971)
#pragma unroll 4
                    for (int it = 0; it < 32 / MPI; ++it) {
                        const int m = MPI * it + sub;
                        const uint2 v = *reinterpret_cast<const uint2*>(srow + (size_t)m * P);
                        __stcs(reinterpret_cast<uint2*>(orow + (size_t)m * 2 * npairs), v);
                    }
                } else {
#pragma unroll 1
                    for (int m = sub; m < nvalid; m += MPI) {
                        const uint2 v = *reinterpret_cast<const uint2*>(srow + (size_t)m * P);
                        __stcs(reinterpret_cast<uint2*>(orow + (size_t)m * 2 * npairs), v);
                    }
                }
            }
            __syncwarp();
        }
    }
    if (reset_now && S.auto_reset == EVG_AUTORESET_TERMINAL) {
        reset_row(S, R, n_nodes);
        turn = 0;
        episode += 1;
    }
    if (valid) {
        R[kRecTurn] = turn;
        R[kRecEpisode] = episode;
    }
    __syncwarp();

    // ---- cooperative, coalesced store of the records (the padding words are written as zeros)
    {
        const int q4 = RW / 4;
        uint4* g4 = reinterpret_cast<uint4*>(A.records) + warp_env0 * q4;
        const int total = nvalid * q4;
        const int used = kRecNode0 + n_nodes;
        auto put = [&](int f) {
            const int m = NODES ? f >> 4 : f / q4, q = NODES ? f & 15 : f % q4;
            const uint32_t* sw = wrow + (size_t)m * P + 4 * q;
            uint2 a = make_uint2(0u, 0u), b = make_uint2(0u, 0u);
            if (NODES || 4 * q < RWU)  // (asm: one 8-byte load; the compiler would split it around the zeroing of a.y below)
                asm volatile("ld.shared.v2.u32 {%0,%1}, [%2];" : "=r"(a.x), "=r"(a.y) : "r"((uint32_t)__cvta_generic_to_shared(sw)));
            if (4 * q + 2 < RWU) b = *reinterpret_cast<const uint2*>(sw + 2);
            if (4 * q + 1 >= used) a.y = 0u;
            if (4 * q + 3 >= used) b.y = 0u;
            g4[f] = make_uint4(a.x, a.y, b.x, b.y);
        };
        if (NODES && nvalid == 32) {
            // 16 chunks per lane, unrolled by 8: 0.4882 ms (4: 0.4904, 2: 0.4922, 16: 0.4924)
#pragma unroll 8
            for (int i = 0; i < (NODES ? 16 : 1); ++i) put(pl + 32 * i);
        } else {
#pragma unroll 1
            for (int f = lane; f < total; f += 32) put(f);
        }
    }
    __syncwarp();
    batch = next_batch;
    next_batch = after_next;
    }  // batch loop
    if (LITE) return;
    __syncthreads();
    if (threadIdx.x == 0) {
        if (S.cta_fought) atomicAdd(&A.stats[ST_FOUGHT], (unsigned long long)S.cta_fought);
        __threadfence();
        if (atomicAdd(&A.sched[1], 1u) == gridDim.x - 1) {  // the last CTA out: every hand-out has happened
            A.sched[0] = 0u;
            A.sched[1] = 0u;
        }
    }
}

// DemoMap row: 62 record words + the staging window, pitch / 2 odd
constexpr int kFastPitch = (((62 + kTpmStage) / 2) & 1) ? 62 + kTpmStage : 62 + kTpmStage + 2;

// which family of instantiations serves this config
enum Variant { V_FAST = 0, V_GENERIC8, V_GENERIC16 };
using TpmKernel = void (*)(Tables, StepArgs);

Variant pick(const Tables& t)
{
    // (n_big <= 8: every group of more than 8 slots can have its second work item, a match's items still fit one round)
    if (t.n_nodes == 11 && t.max_group_size <= 12 && !t.tpm_hist16 && t.tpm_pitch == kFastPitch && t.fast_div && t.n_big <= 8) return V_FAST;
    return t.tpm_hist16 ? V_GENERIC16 : V_GENERIC8;
}

// The kernel that serves a launch of one variant's kernel family, nullptr for a combination that is not instantiated.
// The compile-time map leaves the agents' code out of a plain step (AGENTS = false) and has no wire-row instantiation
// with scripted agents: no C ABI entry point fuses the agents into a step that writes wire rows (evg_step_agents and
// evg_rollout write float32).  The run-time-sized kernels carry the agents' code in every instantiation.
template <int NODES, int MAXSZ, typename HistT, int PITCH, int THREADS>
TpmKernel family_kernel(bool agents, bool wire, bool roll)
{
    constexpr bool PLAIN_AGENTS = NODES == 0;
    if (wire) return roll || (agents && !PLAIN_AGENTS) ? nullptr : evg_step_tpm_kernel<NODES, MAXSZ, HistT, PITCH, PLAIN_AGENTS, THREADS, true>;
    if (roll) return evg_step_tpm_kernel<NODES, MAXSZ, HistT, PITCH, true, THREADS, false, true>;
    if (agents) return evg_step_tpm_kernel<NODES, MAXSZ, HistT, PITCH, true, THREADS>;
    return evg_step_tpm_kernel<NODES, MAXSZ, HistT, PITCH, PLAIN_AGENTS, THREADS>;
}

// The one table of thread-per-match instantiations: one-warp CTAs exist for the compile-time map only
TpmKernel tpm_kernel(Variant v, int threads, bool agents, bool wire, bool roll)
{
    if (threads == kTpmSmallThreads) return v == V_FAST ? family_kernel<11, 12, uint8_t, kFastPitch, kTpmSmallThreads>(agents, wire, roll) : nullptr;
    switch (v) {
        case V_FAST: return family_kernel<11, 12, uint8_t, kFastPitch, kTpmThreads>(agents, wire, roll);
        case V_GENERIC8: return family_kernel<0, 16, uint8_t, 0, kTpmThreads>(agents, wire, roll);
        default: return family_kernel<0, 16, uint16_t, 0, kTpmThreads>(agents, wire, roll);
    }
}

}  // namespace

bool tpm_has_small(const Tables& t) { return pick(t) == V_FAST; }

cudaError_t tpm_prepare(const Tables& t, int threads, size_t* smem_out, int* blocks_per_sm)
{
    // the one-warp CTAs keep neither the tables nor the constant observation entries in shared memory (LITE).
    // DemoMap, 128-thread CTAs: 65,696 B; three CTAs + the driver's 1 KiB each = 195.5 KiB, inside the SM's 196 KiB
    // shared-memory configuration.  One more KB per CTA selects the 228 KiB configuration, L1 drops from 60 to 28 KiB
    // and the step kernel loses 15 % (DESIGN.md section 4.4): do not grow this.
    const size_t smem = (threads == kTpmSmallThreads ? 0 : (size_t)t.sm_tables_bytes + (size_t)oconst_bytes(t.n_nodes)) +
                        (size_t)(threads / 32) * (32 * t.tpm_pitch + 64 * (t.n_nodes + 1) + t.tpm_pool_words) * 4;
    *smem_out = smem;
    const Variant v = pick(t);
    const TpmKernel plain = tpm_kernel(v, threads, false, false, false);
    if (!plain) return cudaErrorInvalidValue;
    cudaError_t e;
    int limit = 0;
    if ((e = optin_smem_limit(smem, &limit)) != cudaSuccess) return e;
    for (int c = 0; c < 8; ++c)  // every (agents, wire, roll) this simulator can launch with
        if (const TpmKernel k = tpm_kernel(v, threads, c & 1, c & 2, c & 4))
            if ((e = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, limit)) != cudaSuccess) return e;
    return cudaOccupancyMaxActiveBlocksPerMultiprocessor(blocks_per_sm, plain, threads, smem);
}

// The float32 observation vector is the default output; the wire row (EVG_OBS_WIRE) has its own instantiations.
cudaError_t launch_step_tpm(const Tables& t, const StepArgs& a, int threads, size_t smem, int max_grid, cudaStream_t stream)
{
    const bool roll = a.n_turns > 1;  // (evg_rollout: both players scripted, float32 observations)
    if (roll && (a.agent[0] == EVG_AGENT_EXTERNAL || a.agent[1] == EVG_AGENT_EXTERNAL)) return cudaErrorInvalidValue;
    const TpmKernel k = tpm_kernel(pick(t), threads, a.agent[0] != EVG_AGENT_EXTERNAL || a.agent[1] != EVG_AGENT_EXTERNAL,
                                   a.obs_fmt == EVG_OBS_WIRE, roll);
    if (!k) return cudaErrorInvalidValue;
    const int64_t nb = (a.n_envs + threads - 1) / threads;
    const unsigned grid = (unsigned)(nb < max_grid ? nb : max_grid);
    k<<<grid, threads, smem, stream>>>(t, a);
    return cudaGetLastError();
}

}  // namespace evg

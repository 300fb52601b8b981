// evg_capi.cu — host side of the C ABI declared in include/evgsim.h.
// Validates the config, derives the device tables and launch geometry, and forwards every call to
// the kernels of evg_kernels.cu.  Owns no device memory: all arrays are the caller's (evg_bind).
#include <cstdarg>
#include <cstddef>
#include <cstdio>
#include <cstring>
#include <cstdlib>
#include <new>
#include <cmath>
#include <string>
#include <vector>

#include "evg_internal.h"

namespace {

thread_local std::string g_last_error;

int fail(int code, const char* fmt, ...)
{
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    g_last_error = buf;
    return code;
}

int cuda_fail(cudaError_t e, const char* what)
{
    return fail(EVG_E_CUDA, "%s: %s (%s)", what, cudaGetErrorName(e), cudaGetErrorString(e));
}

inline int round_up(int v, int a) { return (v + a - 1) / a * a; }

}  // namespace

struct EvgSim {
    EvgConfig cfg;
    evg::Tables tables;
    int64_t n_envs;
    int device;
    int grid;
    size_t smem;
    void* bound[EVG_BIND_COUNT];
    bool is_bound;
    int64_t launches;
    int64_t steps;
    EvgLayout layout;
    bool use_tpm;     // the thread-per-match step kernel, or the warp-per-match one (small batches, EVG_STEP_KERNEL=warp)
    const uint4* tables_dev;  // Tables in device memory (inside bind slot EVG_BIND_TABLES)
    const float* oconst_dev;  // the constant observation entries behind it
    // evg_step_host's chunk pipeline: two streams of the library's own, created on first use
    cudaStream_t host_stream[2] = {nullptr, nullptr};
    cudaEvent_t host_start = nullptr, host_done[2] = {nullptr, nullptr};
    size_t tpm_smem;
    int tpm_grid;     // persistent CTAs: SMs x resident CTAs
    int tpm_threads;  // 128, or 32 (one warp per CTA) for small batches
    int sm_count;
};

namespace {

// EvgConfig -> Tables.  Returns 0 or EVG_E_CONFIG with the reason in g_last_error.
int build_tables(const EvgConfig& c, uint64_t seed, int64_t env_id_offset, evg::Tables* out)
{
    evg::Tables t;
    memset(&t, 0, sizeof(t));
    if (c.abi_version != EVG_ABI_VERSION) return fail(EVG_E_CONFIG, "EvgConfig.abi_version %d != %d", c.abi_version, EVG_ABI_VERSION);
    if (c.n_nodes < 2 || c.n_nodes > EVG_MAX_NODES) return fail(EVG_E_CONFIG, "n_nodes %d outside 2..%d", c.n_nodes, EVG_MAX_NODES);
    if (c.n_unit_types < 1 || c.n_unit_types > EVG_MAX_UNIT_TYPES) return fail(EVG_E_CONFIG, "n_unit_types %d outside 1..%d", c.n_unit_types, EVG_MAX_UNIT_TYPES);
    if (c.turn_limit < 1 || c.turn_limit > 65535) return fail(EVG_E_CONFIG, "turn_limit %d outside 1..65535", c.turn_limit);
    if (c.capture_bonus < 0 || c.capture_bonus > 1000000) return fail(EVG_E_CONFIG, "capture_bonus %d outside 0..1e6", c.capture_bonus);
    if (c.max_score < 1) return fail(EVG_E_CONFIG, "max_score %d must be positive", c.max_score);
    if (c.auto_reset < EVG_AUTORESET_OFF || c.auto_reset > EVG_AUTORESET_NEXT) return fail(EVG_E_CONFIG, "auto_reset %d unknown", c.auto_reset);
    t.n_nodes = c.n_nodes;
    t.obs_len = 1 + 4 * c.n_nodes + 5 * EVG_NUM_GROUPS;
    t.turn_limit = c.turn_limit;
    t.capture_bonus = c.capture_bonus;
    t.auto_reset = c.auto_reset;
    if (c.max_score >= (1 << 24)) return fail(EVG_E_CONFIG, "max_score %d must be below 2^24", c.max_score);
    t.max_score_f = (float)c.max_score;
    t.seed_lo = (uint32_t)seed;
    t.seed_hi = (uint32_t)(seed >> 32);
    t.env_base = (uint32_t)env_id_offset;

    int start[EVG_NUM_PLAYERS] = {-1, -1};
    if (c.p1_node_map[0] != 0) return fail(EVG_E_CONFIG, "p1_node_map[0] must be 0");
    for (int n = 1; n <= c.n_nodes; ++n) {
        if (c.node_control_points[n] < 1 || c.node_control_points[n] > 32767) return fail(EVG_E_CONFIG, "node %d ControlPoints %d outside 1..32767", n, c.node_control_points[n]);
        if (!(c.node_defense[n] >= 0.0) || c.node_defense[n] > 1e6) return fail(EVG_E_CONFIG, "node %d StructureDefense %g invalid", n, c.node_defense[n]);
        const int ts = c.node_team_start[n];
        if (ts < -1 || ts > 1) return fail(EVG_E_CONFIG, "node %d TeamStart %d outside -1..1", n, ts);
        if (ts >= 0) start[ts] = n;  // team_starts[teamStart] = ID, last one wins (server.py:67-68)
        const int m = c.p1_node_map[n];
        if (m < 1 || m > c.n_nodes || c.p1_node_map[m] != n) return fail(EVG_E_CONFIG, "p1_node_map is not an involution at node %d", n);
        t.node_cp[n] = (int16_t)c.node_control_points[n];
        t.node_def[n] = c.node_defense[n];
        t.node_team_start[n] = (int8_t)ts;
        t.node_flags[n] = (uint8_t)((c.node_has_defense[n] ? 1 : 0) | (c.node_has_observe[n] ? 2 : 0) | (c.node_has_defend[n] ? 4 : 0));
        t.p1_map[n] = (uint8_t)m;
        for (int b = 1; b <= c.n_nodes; ++b) t.edge[n][b] = c.edge_distance[n][b];
    }
    for (int p = 0; p < EVG_NUM_PLAYERS; ++p)
        if (start[p] < 0) return fail(EVG_E_CONFIG, "no node has TeamStart == %d", p);
    for (int k = 0; k < c.n_unit_types; ++k) {
        if (!(c.unit_armor[k] > 0.0) || c.unit_armor[k] > 1e6) return fail(EVG_E_CONFIG, "unit type %d Health %g must be in (0, 1e6]", k, c.unit_armor[k]);
        if (c.unit_damage[k] < 0 || c.unit_damage[k] > 255 || c.unit_speed[k] < 0 || c.unit_speed[k] > 255 || c.unit_control[k] < 0 ||
            c.unit_control[k] > 63 || c.unit_cost[k] < 0 || c.unit_cost[k] > 255)
            return fail(EVG_E_CONFIG, "unit type %d: Damage/Speed/Cost must be 0..255 and Control 0..63", k);
        t.unit_armor[k] = c.unit_armor[k];
        t.ut_damage[k] = (uint8_t)c.unit_damage[k];
        t.ut_speed[k] = (uint8_t)c.unit_speed[k];
        t.ut_control[k] = (uint8_t)c.unit_control[k];
        t.ut_cost[k] = (uint8_t)c.unit_cost[k];
    }
    int max_units = 0, max_size = 0, small = 0, per_player_slots = 0, n_big = 0, max_dmg_sum = 0;
    for (int p = 0; p < EVG_NUM_PLAYERS; ++p) {
        int slots = 0, units = 0, dmg_sum = 0;
        for (int g = 0; g < EVG_NUM_GROUPS; ++g) {
            const int L = p * EVG_NUM_GROUPS + g, size = c.group_size[p][g], type = c.group_type[p][g];
            if (size < 1 || size > EVG_MAX_GROUP_UNITS) return fail(EVG_E_CONFIG, "group %d of player %d has %d units; supported 1..%d", g, p, size, EVG_MAX_GROUP_UNITS);
            if (type >= c.n_unit_types) return fail(EVG_E_CONFIG, "group %d of player %d has unknown unit type %d", g, p, type);
            t.g_type[L] = (uint8_t)type;
            t.g_size[L] = (uint8_t)size;
            t.g_big[L] = size > 8 ? (uint8_t)n_big++ : (uint8_t)0;
            if (size > 8) t.big_mask |= 1u << L;
            t.g_damage[L] = t.ut_damage[type];
            t.g_speed[L] = t.ut_speed[type];
            t.g_control[L] = t.ut_control[type];
            t.g_cost[L] = t.ut_cost[type];
            t.g_slot[L] = (uint16_t)slots;  // per-player offset for now
            slots += round_up(size, 4);     // every group starts on a 32-byte sector
            units += size;
            dmg_sum += size * c.unit_damage[type];
            if (size > max_size) max_size = size;
            if (size < 8) small = 1;
            t.init_w0[L] = (uint32_t)start[p] | 100u << evg::W0_AVG_SHIFT;  // health 100.0 each (definitions.py:62)
            t.init_w1[L] = (1u << size) - 1u;                               // all alive, arrival turn 0 (listed in gid order)
        }
        if (slots > per_player_slots) per_player_slots = slots;
        if (units > max_units) max_units = units;
        if (dmg_sum > max_dmg_sum) max_dmg_sum = dmg_sum;
    }
    for (int g = 0; g < EVG_NUM_GROUPS; ++g) t.g_slot[EVG_NUM_GROUPS + g] = (uint16_t)(t.g_slot[EVG_NUM_GROUPS + g] + per_player_slots);
    for (int L = 0; L < evg::kGroupLanes; ++L) {
        t.g_move[2 * (L % EVG_NUM_GROUPS) + L / EVG_NUM_GROUPS] = (uint32_t)t.g_speed[L] | (uint32_t)t.g_control[L] << 8 | (uint32_t)t.g_cost[L] << 16;
        t.g_fight[L] = (uint32_t)t.g_slot[L] | (uint32_t)t.g_size[L] << 12 | (uint32_t)t.g_damage[L] << 17 | (uint32_t)t.g_type[L] << 25;
    }
    if (c.n_nodes <= 15)
        for (int n = 0; n <= c.n_nodes; ++n) t.p1_nib |= (uint64_t)(t.p1_map[n] & 15u) << (4 * n);
    for (int n = 1; n <= c.n_nodes; ++n) t.node_cap[n] = ((uint32_t)t.node_cp[n] & 0xFFFFu) | (uint32_t)(t.node_team_start[n] + 1) << 16;
    t.health_slots = 2 * per_player_slots;
    t.max_group_size = max_size;
    t.has_small_groups = small;
    t.n_big = n_big;
    t.hist_words = (max_units + 1) / 2 + 1;
    for (int p = 0; p < EVG_NUM_PLAYERS; ++p) {
        const int enemy = start[1 - p];
        t.base_own[p] = (uint8_t)(p ? c.p1_node_map[enemy] : enemy);
        for (int a = 1; a <= c.n_nodes; ++a) {  // a = own-numbered node
            const int real = p ? c.p1_node_map[a] : a;
            int best = 0;
            for (int b = 1; b <= c.n_nodes; ++b)
                if (c.edge_distance[real][b]) {
                    const int own = p ? c.p1_node_map[b] : b;
                    if (own > best) best = own;
                }
            t.maxnb_own[p][a] = (uint8_t)best;
        }
    }
    // node state after game_init's capture() at turn 0 (server.py:206,744-745,763-765)
    for (int n = 1; n <= c.n_nodes; ++n) {
        int cs = 0, cb = c.node_team_start[n];
        for (int p = 0; p < EVG_NUM_PLAYERS; ++p)
            if (start[p] == n) {
                cs = p == 0 ? c.node_control_points[n] : -c.node_control_points[n];
                cb = p;
            }
        t.init_node[n] = ((uint32_t)cs & 0xFFFFu) | ((uint32_t)cb & 0xFFu) << 16;
    }
    // resident record: 48 group words + turn + episode + n_nodes node words, padded to 32 bytes
    const int rec_bytes = round_up((evg::kRecNode0 + c.n_nodes) * 4, 32);
    t.rec_words8 = rec_bytes / 8;
    // per-warp shared-memory carve-up
    const int nn = c.n_nodes + 1;
    t.sm_acc = round_up(rec_bytes, 16);
    t.sm_hist = t.sm_acc + round_up(2 * nn * 4, 16);
    t.sm_obs = t.sm_hist + round_up(2 * t.hist_words * 4, 16);
    t.sm_misc = t.sm_obs + round_up(2 * t.obs_len * 4, 16);
    t.sm_warp_stride = t.sm_misc + 528 + n_big * 16 * 8;
    t.sm_tables_bytes = round_up((int)sizeof(evg::Tables), 16);
    // u8 damage histograms when no target can collect > 255 damage in a turn
    t.tpm_hist16 = max_dmg_sum > 255 ? 1 : 0;
    t.max_damage_sum = max_dmg_sum;
    {   // thread-per-match kernel: per-thread row = the record's used words + the observation staging window; two
        // words per node and match are kept word-major per warp; the damage histograms of one round (<= 32
        // fighting groups) live in a per-warp pool
        int pitch = round_up(evg::kRecNode0 + c.n_nodes, 2) + evg::kTpmStage;
        if (((pitch / 2) & 1) == 0) pitch += 2;
        t.tpm_pitch = pitch;
        t.tpm_pool_words = (32 * round_up(max_size, 4) * (t.tpm_hist16 ? 2 : 1) + 3) / 4;
    }
    // The step kernel forms (10.*d)/D without a division: q0 = a*r with r = 1/D, then q = fma(fma(-q0, D, a), r, q0)
    // (Markstein's correction).  It is used only if it reproduces a/D for EVERY reachable numerator a = 10*d of
    // every divisor D = armor + bonus*StructureDefense, which is checked here exhaustively.
    {
        bool fast = !getenv("EVG_NO_FAST_DIV");
        for (int k = 0; k < c.n_unit_types && fast; ++k)
            for (int x = 1; x <= c.n_nodes && fast; ++x)
                for (int b = 0; b < 3 && fast; ++b) {
                    volatile double node_def = (double)b * c.node_defense[x];
                    volatile double divisor = c.unit_armor[k] + node_def;
                    volatile double r = 1.0 / divisor;
                    for (int d = 1; d <= t.max_damage_sum && fast; ++d) {
                        volatile double a = 10.0 * (double)d;
                        volatile double q0 = a * r;
                        volatile double rem = fma(-q0, divisor, a);
                        volatile double q = fma(rem, r, q0);
                        volatile double ref = a / divisor;
                        if (!(q == ref)) fast = false;
                    }
                }
        t.fast_div = fast ? 1 : 0;
    }
    *out = t;
    return EVG_OK;
}

int check_sim(const EvgSim* s, bool need_bound)
{
    if (!s) return fail(EVG_E_ARG, "null EvgSim handle");
    if (need_bound && !s->is_bound) return fail(EVG_E_STATE, "evg_bind() must be called before this entry point");
    cudaError_t e = cudaSetDevice(s->device);
    if (e != cudaSuccess) return cuda_fail(e, "cudaSetDevice");
    return EVG_OK;
}

// where the wire-row expansion of a bound simulator finds the map's constant entries and player 1's node numbering
evg::WireSrc wire_src(const EvgSim* s)
{
    evg::WireSrc w;
    w.oconst = s->oconst_dev;
    w.p1_map = reinterpret_cast<const uint8_t*>(s->tables_dev) + offsetof(evg::Tables, p1_map);
    w.n_nodes = s->tables.n_nodes;
    w.obs_len = s->tables.obs_len;
    w.words = evg::wire_bytes(s->tables.n_nodes) / 4;
    return w;
}

}  // namespace

extern "C" {

int evg_abi_version(void) { return EVG_ABI_VERSION; }

const char* evg_last_error(void) { return g_last_error.c_str(); }

int evg_default_config(EvgConfig* cfg)
{
    if (!cfg) return fail(EVG_E_ARG, "null config");
    memset(cfg, 0, sizeof(*cfg));
    cfg->abi_version = EVG_ABI_VERSION;
    cfg->n_nodes = 11;
    cfg->n_unit_types = 3;
    cfg->turn_limit = 150;     // server.py:321
    cfg->capture_bonus = 1000; // server.py:304
    cfg->max_score = 3700;     // env.py:11
    cfg->auto_reset = EVG_AUTORESET_OFF;
    // DemoMap.json (SURVEY.md Appendix A.1): node -> (neighbour, distance)...
    static const int edges[18][3] = {{1, 2, 6}, {1, 4, 6}, {2, 3, 4}, {2, 5, 4}, {3, 4, 4}, {3, 5, 6}, {3, 6, 3}, {3, 7, 6}, {4, 7, 4},
                                     {5, 8, 4}, {5, 9, 6}, {6, 9, 3}, {7, 9, 6}, {7, 10, 4}, {8, 9, 4}, {8, 11, 6}, {9, 10, 4}, {10, 11, 6}};
    for (const auto& e : edges) {
        cfg->edge_distance[e[0]][e[1]] = (uint8_t)e[2];
        cfg->edge_distance[e[1]][e[0]] = (uint8_t)e[2];
    }
    static const double defense[12] = {0, 1, 1.5, 1.75, 1.5, 1.75, 1.75, 1.75, 1.5, 1.75, 1.5, 1};
    static const uint8_t p1map[12] = {0, 11, 8, 9, 10, 5, 6, 7, 2, 3, 4, 1};  // server.py:89
    for (int n = 0; n <= EVG_MAX_NODES; ++n) cfg->node_team_start[n] = -1;
    for (int n = 1; n <= 11; ++n) {
        cfg->node_control_points[n] = (n == 1 || n == 11) ? 500 : 100;
        cfg->node_defense[n] = defense[n];
        cfg->p1_node_map[n] = p1map[n];
    }
    cfg->node_team_start[1] = 0;
    cfg->node_team_start[11] = 1;
    cfg->node_has_observe[2] = cfg->node_has_observe[8] = 1;
    cfg->node_has_defense[4] = cfg->node_has_defense[10] = 1;
    // UnitDefinitions.json: tank, controller, striker
    static const double armor[3] = {3, 2, 1};
    static const int damage[3] = {1, 1, 2}, speed[3] = {1, 1, 2}, control[3] = {1, 2, 1};
    for (int k = 0; k < 3; ++k) {
        cfg->unit_armor[k] = armor[k];
        cfg->unit_damage[k] = damage[k];
        cfg->unit_speed[k] = speed[k];
        cfg->unit_control[k] = control[k];
        cfg->unit_cost[k] = 1;
    }
    // env.py:145-156: classes cycle controller, striker, tank; 8 units each, the last group 12
    static const uint8_t cycle[3] = {1, 2, 0};
    for (int p = 0; p < EVG_NUM_PLAYERS; ++p)
        for (int g = 0; g < EVG_NUM_GROUPS; ++g) {
            cfg->group_type[p][g] = cycle[g % 3];
            cfg->group_size[p][g] = g == EVG_NUM_GROUPS - 1 ? 12 : 8;
        }
    return EVG_OK;
}

int evg_create(const EvgConfig* cfg, int64_t n_envs, uint64_t seed, int64_t env_id_offset, int device, EvgSim** out)
{
    if (!cfg || !out) return fail(EVG_E_ARG, "null argument");
    *out = nullptr;
    if (n_envs < 1 || n_envs > (int64_t)1 << 31) return fail(EVG_E_ARG, "n_envs %lld outside 1..2^31", (long long)n_envs);
    if (env_id_offset < 0 || env_id_offset + n_envs > (int64_t)1 << 32) return fail(EVG_E_ARG, "global match ids must fit 32 bits");
    evg::Tables t;
    int rc = build_tables(*cfg, seed, env_id_offset, &t);
    if (rc) return rc;
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev < 1) return fail(EVG_E_CUDA, "no CUDA device available (%s); libevgsim has no CPU path", e == cudaSuccess ? "count 0" : cudaGetErrorString(e));
    if (device < 0 || device >= ndev) return fail(EVG_E_ARG, "device %d outside 0..%d", device, ndev - 1);
    if ((e = cudaSetDevice(device)) != cudaSuccess) return cuda_fail(e, "cudaSetDevice");
    cudaDeviceProp prop;
    if ((e = cudaGetDeviceProperties(&prop, device)) != cudaSuccess) return cuda_fail(e, "cudaGetDeviceProperties");
    EvgSim* s = new (std::nothrow) EvgSim();
    if (!s) return fail(EVG_E_ARG, "out of host memory");
    s->cfg = *cfg;
    s->tables = t;
    s->n_envs = n_envs;
    s->device = device;
    s->is_bound = false;
    s->launches = 0;
    s->steps = 0;
    s->smem = (size_t)t.sm_tables_bytes + 128 + (size_t)evg::kWarpsPerBlock * t.sm_warp_stride;
    const char* which = getenv("EVG_STEP_KERNEL");
    // default: a thread per match, except for small batches, where a warp per match spreads the few matches over all
    // SMs (measured: 4,096 matches 2.0e8 vs 1.2e8 env-turns/s; break-even near 16k, profiles/README.md)
    s->use_tpm = which ? strcmp(which, "warp") != 0 : n_envs >= 12288;
    // Thread-per-match kernel: 128-thread CTAs, except where a batch needs a second round of them although all of it fits
    // one wave of one-warp CTAs (the LITE instantiation keeps no tables in shared memory: 14 CTAs per SM, 66,304 matches
    // resident on 148 SMs).  Measured step times, lite / 128-thread (profiles/README.md): 32,768 matches 32 / 30 us,
    // 65,536 46 / 55 us, 98,304 70 / 65 us, 262,144 178 / 144 us.  EVG_TPM_SMALL_MAX=<matches> forces the one-warp CTAs up to
    // that batch size (0: never).
    {
        int per_sm128 = 0, per_sm32 = 0;
        size_t smem128 = 0, smem32 = 0;
        if ((e = evg::tpm_prepare(t, evg::kTpmThreads, &smem128, &per_sm128)) != cudaSuccess || per_sm128 < 1) { delete s; return cuda_fail(e, "thread-per-match kernel setup"); }
        s->tpm_threads = evg::kTpmThreads;
        s->tpm_smem = smem128;
        s->tpm_grid = prop.multiProcessorCount * per_sm128;
        if (evg::tpm_has_small(t)) {
            if ((e = evg::tpm_prepare(t, evg::kTpmSmallThreads, &smem32, &per_sm32)) != cudaSuccess || per_sm32 < 1) { delete s; return cuda_fail(e, "thread-per-match kernel setup (one-warp CTAs)"); }
            const int64_t nb128 = (n_envs + evg::kTpmThreads - 1) / evg::kTpmThreads;
            const int64_t lite_capacity = (int64_t)prop.multiProcessorCount * per_sm32 * evg::kTpmSmallThreads;
            bool lite = nb128 > s->tpm_grid && n_envs <= lite_capacity;
            if (const char* small = getenv("EVG_TPM_SMALL_MAX")) lite = n_envs <= atoll(small);
            if (lite) {
                s->tpm_threads = evg::kTpmSmallThreads;
                s->tpm_smem = smem32;
                s->tpm_grid = prop.multiProcessorCount * per_sm32;
            }
        }
    }
    s->sm_count = prop.multiProcessorCount;
    // the shared-memory opt-ins are per device: made on the simulator's, for the step and the policy kernels
    if ((e = evg::set_step_smem(s->smem)) != cudaSuccess || (e = evg::set_policy_mlp_smem()) != cudaSuccess || (e = evg::set_policy_ppo_smem()) != cudaSuccess ||
        (e = evg::set_policy_rppo_smem()) != cudaSuccess || (e = evg::set_policy_value_smem()) != cudaSuccess ||
        (e = evg::set_rppo_train_smem()) != cudaSuccess) { delete s; return cuda_fail(e, "cudaFuncSetAttribute(max dynamic smem)"); }
    int per_sm = 0;
    if ((e = evg::step_occupancy(t, s->smem, &per_sm)) != cudaSuccess || per_sm < 1) { delete s; return cuda_fail(e, "occupancy query"); }
    // persistent CTAs: a whole number of resident waves, never more CTAs than matches need
    const int64_t need = (n_envs + evg::kWarpsPerBlock - 1) / evg::kWarpsPerBlock;
    const int64_t resident = (int64_t)prop.multiProcessorCount * per_sm;
    s->grid = (int)(need < resident ? need : resident);
    EvgLayout& L = s->layout;
    L.n_envs = n_envs;
    L.obs_len = t.obs_len;
    L.record_bytes = t.rec_words8 * 8;
    L.health_slots = t.health_slots;
    L.action_bytes = 2 * EVG_MAX_ACTIONS * 2;
    L.records_bytes = n_envs * L.record_bytes;
    L.health_bytes = n_envs * (int64_t)L.health_slots * 8;
    L.stats_bytes = (evg::ST_COUNT + evg::kSchedSlots + 1) * 8;  // + the step kernel's batch hand-out counters + evg_import_state's error counter
    L.agents_bytes = n_envs * 16;
    // loss table, then reciprocals, then the Tables struct itself (the step kernel stages it from here)
    // ... and the constant observation entries as floats
    L.tables_bytes = round_up((int)((int64_t)cfg->n_unit_types * (cfg->n_nodes + 1) * 3 * (evg::kLossD + 1) * 8), 16) + round_up((int)sizeof(evg::Tables), 16) +
                     round_up(evg::oconst_bytes(cfg->n_nodes), 16);
    *out = s;
    return EVG_OK;
}

int evg_destroy(EvgSim* sim)
{
    if (!sim) return fail(EVG_E_ARG, "null EvgSim handle");
    if (sim->host_start) {
        cudaSetDevice(sim->device);
        for (int i = 0; i < 2; ++i) {
            cudaStreamSynchronize(sim->host_stream[i]);
            cudaStreamDestroy(sim->host_stream[i]);
            cudaEventDestroy(sim->host_done[i]);
        }
        cudaEventDestroy(sim->host_start);
    }
    delete sim;
    return EVG_OK;
}

int evg_layout(const EvgSim* sim, EvgLayout* out)
{
    if (!sim || !out) return fail(EVG_E_ARG, "null argument");
    *out = sim->layout;
    return EVG_OK;
}

int evg_bind(EvgSim* sim, void* const* device_ptrs, int32_t n_ptrs)
{
    if (!sim || !device_ptrs) return fail(EVG_E_ARG, "null argument");
    if (n_ptrs != EVG_BIND_COUNT) return fail(EVG_E_ARG, "evg_bind expects %d pointers, got %d", EVG_BIND_COUNT, n_ptrs);
    for (int i = 0; i < EVG_BIND_COUNT; ++i) {
        if (!device_ptrs[i]) return fail(EVG_E_ARG, "bind slot %d is null", i);
        if ((uintptr_t)device_ptrs[i] % 16) return fail(EVG_E_ARG, "bind slot %d is not 16-byte aligned", i);
        sim->bound[i] = device_ptrs[i];
    }
    // derived table: the fp64 quotient of server.py:601 for every (unit type, node, bonus, damage sum < 32),
    // computed on the host in IEEE double (same operation order as the kernel's fallback division)
    {
        const EvgConfig& c = sim->cfg;
        const int nn = c.n_nodes + 1;
        const size_t n_div = (size_t)c.n_unit_types * nn * 3;
        std::vector<double> tab(n_div * (evg::kLossD + 1), 0.0);
        // ... followed by the reciprocal of every divisor (Tables::fast_div, build_tables)
        for (int t = 0; t < c.n_unit_types; ++t)
            for (int x = 1; x <= c.n_nodes; ++x)
                for (int b = 0; b < 3; ++b) {
                    volatile double node_def = (double)b * c.node_defense[x];
                    volatile double divisor = c.unit_armor[t] + node_def;
                    const size_t ti = (size_t)(t * nn + x) * 3 + b;
                    for (int d = 0; d < evg::kLossD; ++d) {
                        volatile double num = 10.0 * (double)d;
                        tab[ti * evg::kLossD + d] = num / divisor;
                    }
                    volatile double r = 1.0 / divisor;
                    tab[n_div * evg::kLossD + ti] = r;
                }
        cudaError_t e = cudaSetDevice(sim->device);
        if (e == cudaSuccess) e = cudaMemcpy(device_ptrs[EVG_BIND_TABLES], tab.data(), tab.size() * sizeof(double), cudaMemcpyHostToDevice);
        if (e != cudaSuccess) return cuda_fail(e, "upload of the loss table");
        sim->tables.loss_tab = (const double*)device_ptrs[EVG_BIND_TABLES];
        sim->tables.rcp_tab = sim->tables.loss_tab + n_div * evg::kLossD;
        char* tdev = (char*)device_ptrs[EVG_BIND_TABLES] + round_up((int)(tab.size() * sizeof(double)), 16);
        e = cudaMemcpy(tdev, &sim->tables, sizeof(evg::Tables), cudaMemcpyHostToDevice);
        if (e != cudaSuccess) return cuda_fail(e, "upload of the static tables");
        sim->tables_dev = (const uint4*)tdev;
        // the observation entries that never change, as the floats the step kernels copy into every observation:
        // the nodes' 'DEFENSE' / 'OBSERVE' flags in each viewer's numbering (server.py:437-443) and the groups' unit
        // types (server.py:476); everything else 0
        {
            const evg::Tables& t = sim->tables;
            const int OL = t.obs_len, n = t.n_nodes, oc_floats = (2 * OL + 3) & ~3;
            std::vector<float> oc(evg::oconst_bytes(n) / 4, 0.f);
            for (int p = 0; p < 2; ++p) {
                for (int k = 0; k < n; ++k) {
                    const int x = p ? t.p1_map[k + 1] : k + 1;
                    const float fd = (float)(t.node_flags[x] & 1u), fo = (float)((t.node_flags[x] >> 1) & 1u);
                    oc[p * OL + 1 + 4 * k] = fd;
                    oc[p * OL + 1 + 4 * k + 1] = fo;
                    oc[oc_floats + 2 * (p * n + k)] = fd;
                    oc[oc_floats + 2 * (p * n + k) + 1] = fo;
                }
                for (int g = 0; g < EVG_NUM_GROUPS; ++g) oc[p * OL + 1 + 4 * n + 5 * g + 1] = (float)t.g_type[p * EVG_NUM_GROUPS + g];
            }
            char* odev = tdev + round_up((int)sizeof(evg::Tables), 16);
            e = cudaMemcpy(odev, oc.data(), oc.size() * sizeof(float), cudaMemcpyHostToDevice);
            if (e != cudaSuccess) return cuda_fail(e, "upload of the constant observation entries");
            sim->oconst_dev = (const float*)odev;
        }
    }
    sim->is_bound = true;
    return EVG_OK;
}

int evg_obs_row_bytes(const EvgSim* sim, int32_t format)
{
    if (!sim) return 0;
    switch (format) {
        case EVG_OBS_F32: return 2 * sim->layout.obs_len * 4;
        case EVG_OBS_I16: return 2 * sim->layout.obs_len * 2;
        case EVG_OBS_WIRE: return evg::wire_bytes(sim->cfg.n_nodes);
        default: return 0;
    }
}

namespace {

// format checks shared by the *_fmt entry points; `rows`/`f32` may be NULL where the caller allows it
int check_fmt(const EvgSim* sim, int32_t format, const void* rows, const float* f32, const char* who)
{
    if (format < EVG_OBS_F32 || format > EVG_OBS_WIRE) return fail(EVG_E_ARG, "%s: unknown observation format %d", who, format);
    if (format == EVG_OBS_I16) {
        if (rows && !f32) return fail(EVG_E_ARG, "%s: EVG_OBS_I16 needs the float32 scratch d_obs_f32", who);
        if (sim->cfg.turn_limit > 32767) return fail(EVG_E_ARG, "%s: EVG_OBS_I16 cannot carry a turn counter up to %d", who, sim->cfg.turn_limit);
    }
    if (rows && (uintptr_t)rows % 16) return fail(EVG_E_ARG, "%s: observation rows must be 16-byte aligned", who);
    return EVG_OK;
}

// evg_policy_mlp's and evg_pack_mlp's checks: the observations, the network's shape and the images fit the kernel
int check_mlp_shape(const char* fn, const EvgSim* sim, int32_t hidden, int32_t out_dim, const void* d_w1_img, const void* d_w2_img)
{
    if (sim->layout.obs_len >= EVG_MLP_IN_PAD) return fail(EVG_E_ARG, "%s: observations of %d values + the bias input exceed the %d the kernel is tiled for", fn, sim->layout.obs_len, EVG_MLP_IN_PAD);
    if (hidden < 1 || hidden > 64 * EVG_MLP_CHUNK || out_dim < 1 || out_dim > EVG_MLP_OUT_PAD)
        return fail(EVG_E_ARG, "%s: hidden %d / out_dim %d outside the kernel's tiling (hidden <= %d, out <= %d)", fn, hidden, out_dim, 64 * EVG_MLP_CHUNK, EVG_MLP_OUT_PAD);
    if (((uintptr_t)d_w1_img | (uintptr_t)d_w2_img) % 16) return fail(EVG_E_ARG, "%s: weight images must be 16-byte aligned", fn);
    return EVG_OK;
}

// the same checks for the PPO actors (evg_policy_ppo / _rppo, evg_pack_ppo / _rppo); `aligned`: what the call reads in 16 B
int check_actor_shape(const char* fn, const EvgSim* sim, int32_t latent, int32_t out_dim, std::initializer_list<const void*> aligned)
{
    if (latent < 1 || latent > EVG_PPO_MAX_LATENT) return fail(EVG_E_ARG, "%s: latent %d outside 1..%d", fn, latent, EVG_PPO_MAX_LATENT);
    if (out_dim < EVG_MAX_ACTIONS || out_dim > EVG_PPO_OUT_PAD) return fail(EVG_E_ARG, "%s: out_dim %d outside %d..%d", fn, out_dim, EVG_MAX_ACTIONS, EVG_PPO_OUT_PAD);
    for (const void* p : aligned)
        if ((uintptr_t)p % 16) return fail(EVG_E_ARG, "%s: weight images (and a packed bias vector) must be 16-byte aligned", fn);
    if (sim->layout.obs_len >= EVG_PPO_IN_PAD) return fail(EVG_E_ARG, "%s: observations of %d values exceed the %d the kernel is tiled for", fn, sim->layout.obs_len, EVG_PPO_IN_PAD - 1);
    return EVG_OK;
}

// evg_pack_ppo and evg_pack_rppo (w_ih != null): the weights of evg_policy_ppo / _rppo
int pack_ppo_family(const char* fn, EvgSim* sim, const float* d_w1, const float* d_b1, const float* d_w2, const float* d_b2, const float* d_w3,
                    const float* d_b3, const float* d_w_ih, const float* d_b_ih, const float* d_w_hh, const float* d_b_hh, int32_t latent,
                    int32_t out_dim, void* d_w1_img, void* d_w2_img, void* d_wi_img, void* d_wh_img, void* d_w3_img, float* d_bias, void* stream)
{
    int rc = check_sim(sim, false);
    if (rc) return rc;
    if (!d_w1 || !d_b1 || !d_w2 || !d_b2 || !d_w3 || !d_b3 || !d_w1_img || !d_w2_img || !d_w3_img || !d_bias)
        return fail(EVG_E_ARG, "%s: null argument", fn);
    if ((rc = check_actor_shape(fn, sim, latent, out_dim, {d_w1_img, d_w2_img, d_wi_img, d_wh_img, d_w3_img, d_bias}))) return rc;
    cudaError_t e = evg::launch_pack_ppo(sim->layout.obs_len, d_w1, d_b1, d_w2, d_b2, d_w3, d_b3, d_w_ih, d_b_ih, d_w_hh, d_b_hh, latent, out_dim,
                                         d_w1_img, d_w2_img, d_wi_img, d_wh_img, d_w3_img, d_bias, (cudaStream_t)stream);
    if (e != cudaSuccess) return cuda_fail(e, "evg_policy_pack_kernel launch");
    sim->launches += 1;
    return EVG_OK;
}

}  // namespace

int evg_reset_fmt(EvgSim* sim, int32_t format, const uint8_t* d_mask, void* d_rows, float* d_obs_f32, void* stream)
{
    int rc = check_sim(sim, true);
    if (rc) return rc;
    if ((rc = check_fmt(sim, format, d_rows, d_obs_f32, "evg_reset_fmt"))) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    cudaError_t e;
    if (!d_mask) {
        if ((e = cudaMemsetAsync(sim->bound[EVG_BIND_STATS], 0, (size_t)sim->layout.stats_bytes, st)) != cudaSuccess) return cuda_fail(e, "cudaMemsetAsync(stats)");
        if ((e = cudaMemsetAsync(sim->bound[EVG_BIND_AGENTS], 0, (size_t)sim->n_envs * 16, st)) != cudaSuccess) return cuda_fail(e, "cudaMemsetAsync(agent state)");
        sim->steps = 0;
    }
    const bool i16 = format == EVG_OBS_I16 && d_rows;
    e = evg::launch_reset(sim->tables, (uint32_t*)sim->bound[EVG_BIND_RECORDS], (double*)sim->bound[EVG_BIND_HEALTH], d_mask,
                          i16 ? (void*)d_obs_f32 : d_rows, format == EVG_OBS_WIRE ? EVG_OBS_WIRE : EVG_OBS_F32, sim->n_envs, sim->grid, sim->smem, st);
    if (e != cudaSuccess) return cuda_fail(e, "evg_reset_kernel launch");
    sim->launches += 1;
    if (i16) {  // (with a mask the unmasked matches' rows are rewritten from the scratch as well: it holds their last observation)
        if ((e = evg::launch_obs_to_i16(d_obs_f32, (int16_t*)d_rows, sim->n_envs * 2 * sim->layout.obs_len, st)) != cudaSuccess) return cuda_fail(e, "evg_obs_to_i16_kernel launch");
        sim->launches += 1;
    }
    return EVG_OK;
}

int evg_reset(EvgSim* sim, const uint8_t* d_mask, float* d_obs, void* stream) { return evg_reset_fmt(sim, EVG_OBS_F32, d_mask, d_obs, nullptr, stream); }

// the step kernels' arguments for the whole batch
static evg::StepArgs step_args(EvgSim* sim, int agent0, int agent1, const int8_t* d_actions, int8_t* d_actions_out, void* d_obs,
                               float* d_reward, uint8_t* d_done, uint8_t* d_status, int32_t* d_scores, int obs_fmt, int sched_slot,
                               int n_turns)
{
    evg::StepArgs a;
    a.n_turns = n_turns;
    a.agent[0] = agent0;
    a.agent[1] = agent1;
    a.actions_out = d_actions_out;
    a.records = (uint32_t*)sim->bound[EVG_BIND_RECORDS];
    a.health = (double*)sim->bound[EVG_BIND_HEALTH];
    a.stats = (unsigned long long*)sim->bound[EVG_BIND_STATS];
    a.agent_state = (uint2*)sim->bound[EVG_BIND_AGENTS];
    a.sched = (unsigned*)((unsigned long long*)sim->bound[EVG_BIND_STATS] + evg::ST_COUNT + sched_slot);
    a.actions = d_actions;
    a.obs = (float*)d_obs;
    a.obs_fmt = obs_fmt;
    a.reward = d_reward;
    a.done = d_done;
    a.status = d_status;
    a.scores = d_scores;
    a.n_envs = sim->n_envs;
    a.tables_dev = sim->tables_dev;
    a.oconst_dev = sim->oconst_dev;
    a.env_first = 0;
    return a;
}

// first/count: the whole batch (0, n_envs), or a 128-aligned sub-range for the thread-per-match kernel (evg_step_host's
// chunks; all the per-match arrays are offset here, the kernel adds `first` to the global match ids)
static int step_impl(EvgSim* sim, int agent0, int agent1, const int8_t* d_actions, int8_t* d_actions_out, void* d_obs,
                     float* d_reward, uint8_t* d_done, uint8_t* d_status, int32_t* d_scores, void* stream, int64_t first = 0,
                     int64_t count = -1, int obs_fmt = EVG_OBS_F32, int sched_slot = 0, int n_turns = 1)
{
    evg::StepArgs a = step_args(sim, agent0, agent1, d_actions, d_actions_out, d_obs, d_reward, d_done, d_status, d_scores, obs_fmt,
                                sched_slot, n_turns);
    if (count >= 0) {
        const evg::Tables& t = sim->tables;
        a.records += first * t.rec_words8 * 2;
        a.health += first * t.health_slots;
        if (a.actions) a.actions += first * 2 * EVG_MAX_ACTIONS * 2;
        if (a.actions_out) a.actions_out += first * 2 * EVG_MAX_ACTIONS * 2;
        a.agent_state += first * 2;
        a.obs = (float*)((char*)d_obs + first * (obs_fmt == EVG_OBS_WIRE ? evg::wire_bytes(t.n_nodes) : 2 * t.obs_len * 4));
        a.reward += first * 2;
        a.done += first;
        if (a.status) a.status += first;
        if (a.scores) a.scores += first * 2;
        a.n_envs = count;
        a.env_first = first;
    }
    cudaError_t e = !sim->use_tpm ? evg::launch_step(sim->tables, a, sim->grid, sim->smem, (cudaStream_t)stream)
                                  : evg::launch_step_tpm(sim->tables, a, sim->tpm_threads, sim->tpm_smem, sim->tpm_grid, (cudaStream_t)stream);
    if (e != cudaSuccess) return cuda_fail(e, "evg_step kernel launch");
    sim->launches += 1;
    if (count < 0 || first == 0) sim->steps += n_turns;
    return EVG_OK;
}

int evg_step(EvgSim* sim, const int8_t* d_actions, float* d_obs, float* d_reward, uint8_t* d_done, uint8_t* d_status,
             int32_t* d_scores, void* stream)
{
    int rc = check_sim(sim, true);
    if (rc) return rc;
    if (!d_actions || !d_obs || !d_reward || !d_done) return fail(EVG_E_ARG, "evg_step: actions/obs/reward/done must be non-null");
    return step_impl(sim, EVG_AGENT_EXTERNAL, EVG_AGENT_EXTERNAL, d_actions, nullptr, d_obs, d_reward, d_done, d_status, d_scores, stream);
}

int evg_step_agents(EvgSim* sim, int32_t agent_p0, int32_t agent_p1, int8_t* d_actions, float* d_obs, float* d_reward,
                    uint8_t* d_done, uint8_t* d_status, int32_t* d_scores, void* stream)
{
    int rc = check_sim(sim, true);
    if (rc) return rc;
    if (!d_obs || !d_reward || !d_done) return fail(EVG_E_ARG, "evg_step_agents: obs/reward/done must be non-null");
    const int ag[2] = {agent_p0, agent_p1};
    bool any_ext = false, any_scripted = false;
    bool fusable = true;
    for (int p = 0; p < 2; ++p) {
        if (ag[p] < EVG_AGENT_EXTERNAL || ag[p] > EVG_AGENT_SWARM) return fail(EVG_E_ARG, "unknown agent id %d for player %d", ag[p], p);
        any_ext |= ag[p] == EVG_AGENT_EXTERNAL;
        any_scripted |= ag[p] != EVG_AGENT_EXTERNAL;
        fusable &= ag[p] != EVG_AGENT_RANDOM || sim->cfg.n_nodes <= evg::kAgentMaxNodes;  // the register-only random agent
    }
    if (any_ext && !d_actions) return fail(EVG_E_ARG, "evg_step_agents: d_actions is required for EVG_AGENT_EXTERNAL players");
    const bool fused = fusable && sim->use_tpm;
    if (!any_scripted || fused)
        return step_impl(sim, agent_p0, agent_p1, d_actions, any_scripted ? d_actions : nullptr, d_obs, d_reward, d_done, d_status, d_scores, stream);
    // not fusable (warp-per-match kernel selected, or a map too large for the register-only random agent): agent
    // kernel(s) into d_actions, then the plain step
    if (!d_actions) return fail(EVG_E_ARG, "evg_step_agents: d_actions is required when the agents cannot be fused into the step kernel");
    if ((rc = evg_agents(sim, agent_p0, agent_p1, d_actions, stream))) return rc;
    return step_impl(sim, EVG_AGENT_EXTERNAL, EVG_AGENT_EXTERNAL, d_actions, nullptr, d_obs, d_reward, d_done, d_status, d_scores, stream);
}

int evg_rollout(EvgSim* sim, int32_t agent_p0, int32_t agent_p1, int32_t n_turns, int8_t* d_actions, float* d_obs, float* d_reward,
                uint8_t* d_done, uint8_t* d_status, int32_t* d_scores, void* stream)
{
    int rc = check_sim(sim, true);
    if (rc) return rc;
    if (!d_actions || !d_obs || !d_reward || !d_done) return fail(EVG_E_ARG, "evg_rollout: actions/obs/reward/done must be non-null");
    if (n_turns < 0) return fail(EVG_E_ARG, "evg_rollout: n_turns %d is negative", n_turns);
    const int ag[2] = {agent_p0, agent_p1};
    for (int p = 0; p < 2; ++p)
        if (ag[p] <= EVG_AGENT_EXTERNAL || ag[p] > EVG_AGENT_SWARM) return fail(EVG_E_ARG, "evg_rollout: player %d needs a scripted agent, got %d", p, ag[p]);
    const bool random_big_map = (agent_p0 == EVG_AGENT_RANDOM || agent_p1 == EVG_AGENT_RANDOM) && sim->cfg.n_nodes > evg::kAgentMaxNodes;
    if (n_turns == 0) return EVG_OK;
    if (random_big_map) {  // agent kernel + step per turn; a caller may capture this in a CUDA graph
        for (int k = 0; k < n_turns; ++k)
            if ((rc = evg_step_agents(sim, agent_p0, agent_p1, d_actions, d_obs, d_reward, d_done, d_status, d_scores, stream))) return rc;
        return EVG_OK;
    }
    if (sim->use_tpm)  // one launch: a CTA keeps each of its batches in shared memory for all n_turns
        return step_impl(sim, agent_p0, agent_p1, d_actions, d_actions, d_obs, d_reward, d_done, d_status, d_scores, stream, 0, -1, EVG_OBS_F32, 0, n_turns);
    const evg::StepArgs a = step_args(sim, agent_p0, agent_p1, d_actions, d_actions, d_obs, d_reward, d_done, d_status, d_scores, EVG_OBS_F32, 0, n_turns);
    cudaError_t e = evg::launch_rollout(sim->tables, a, n_turns, sim->grid, sim->smem, (cudaStream_t)stream);
    if (e != cudaSuccess) return cuda_fail(e, "evg_rollout_kernel launch");
    sim->launches += 1;
    sim->steps += n_turns;
    return EVG_OK;
}

int evg_step_fmt(EvgSim* sim, int32_t format, const int8_t* d_actions, void* d_rows, float* d_obs_f32, float* d_reward,
                 uint8_t* d_done, uint8_t* d_status, int32_t* d_scores, void* stream)
{
    int rc = check_sim(sim, true);
    if (rc) return rc;
    if (!d_actions || !d_rows || !d_reward || !d_done) return fail(EVG_E_ARG, "evg_step_fmt: actions/rows/reward/done must be non-null");
    if ((rc = check_fmt(sim, format, d_rows, d_obs_f32, "evg_step_fmt"))) return rc;
    if (format != EVG_OBS_I16)
        return step_impl(sim, EVG_AGENT_EXTERNAL, EVG_AGENT_EXTERNAL, d_actions, nullptr, d_rows, d_reward, d_done, d_status, d_scores, stream, 0, -1, format);
    if ((rc = step_impl(sim, EVG_AGENT_EXTERNAL, EVG_AGENT_EXTERNAL, d_actions, nullptr, d_obs_f32, d_reward, d_done, d_status, d_scores, stream))) return rc;
    cudaError_t e = evg::launch_obs_to_i16(d_obs_f32, (int16_t*)d_rows, sim->n_envs * 2 * sim->layout.obs_len, (cudaStream_t)stream);
    if (e != cudaSuccess) return cuda_fail(e, "evg_obs_to_i16_kernel launch");
    sim->launches += 1;
    return EVG_OK;
}

int evg_step_host_fmt(EvgSim* sim, int32_t format, const int8_t* h_actions, void* h_rows, float* h_reward, uint8_t* h_done,
                      int8_t* d_actions, void* d_rows, float* d_obs_f32, float* d_reward, uint8_t* d_done, void* stream)
{
    int rc = check_sim(sim, true);
    if (rc) return rc;
    const bool wire = format == EVG_OBS_WIRE, i16 = format == EVG_OBS_I16;
    if (!h_actions || !h_rows || !d_actions || !d_rows || !d_reward || !d_done) return fail(EVG_E_ARG, "evg_step_host: buffers must be non-null");
    if (!wire && (!h_reward || !h_done)) return fail(EVG_E_ARG, "evg_step_host: h_reward/h_done may only be NULL with EVG_OBS_WIRE");
    if ((rc = check_fmt(sim, format, d_rows, d_obs_f32, "evg_step_host_fmt"))) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    const int64_t n = sim->n_envs;
    const size_t ab = (size_t)sim->layout.action_bytes, rb = (size_t)evg_obs_row_bytes(sim, format), fb = (size_t)2 * sim->layout.obs_len * 4;
    cudaError_t e = cudaSuccess;
    const char* what = "";
#define EVG_TRY(call, name) do { if (e == cudaSuccess && (e = (call)) != cudaSuccess) what = name; } while (0)
    // one sub-range [first, first + cnt): H2D of its action rows, the step, (the narrowing,) D2H of its results, all on `cs`
    auto chunk = [&](cudaStream_t cs, int64_t first, int64_t cnt, bool sub, int slot) -> int {
        EVG_TRY(cudaMemcpyAsync(d_actions + first * ab, h_actions + first * ab, (size_t)cnt * ab, cudaMemcpyHostToDevice, cs), "H2D actions");
        if (e != cudaSuccess) return EVG_OK;
        int r = step_impl(sim, EVG_AGENT_EXTERNAL, EVG_AGENT_EXTERNAL, d_actions, nullptr, i16 ? (void*)d_obs_f32 : d_rows, d_reward, d_done, nullptr,
                          nullptr, cs, sub ? first : 0, sub ? cnt : -1, wire ? EVG_OBS_WIRE : EVG_OBS_F32, slot);
        if (r) return r;
        if (i16) {
            EVG_TRY(evg::launch_obs_to_i16((const float*)((const char*)d_obs_f32 + first * fb), (int16_t*)((char*)d_rows + first * rb),
                                           cnt * 2 * sim->layout.obs_len, cs), "evg_obs_to_i16_kernel launch");
            if (e == cudaSuccess) sim->launches += 1;
        }
        EVG_TRY(cudaMemcpyAsync((char*)h_rows + first * rb, (const char*)d_rows + first * rb, (size_t)cnt * rb, cudaMemcpyDeviceToHost, cs), "D2H observations");
        if (h_reward) EVG_TRY(cudaMemcpyAsync(h_reward + first * 2, d_reward + first * 2, (size_t)cnt * 2 * 4, cudaMemcpyDeviceToHost, cs), "D2H reward");
        if (h_done) EVG_TRY(cudaMemcpyAsync(h_done + first, d_done + first, (size_t)cnt, cudaMemcpyDeviceToHost, cs), "D2H done");
        return EVG_OK;
    };
    // Large batches on the thread-per-match kernel go through in chunks on two streams of the library's own, so that
    // the D2H of one chunk (the PCIe-bound part) overlaps the H2D and the kernel of the next; everything is ordered
    // after what `stream` holds now, and `stream` waits for all of it — on the error paths too: whatever was
    // enqueued before a failure is joined into `stream` before the error is returned.
    int chunks = 16;  // (wire rows 2.66 -> 2.60 ms per 1 Mi matches against 8 chunks, int16 8.54 -> 8.25, float32 unchanged; tools/e2e_chunks.py)
    if (const char* c = getenv("EVG_HOST_CHUNKS")) chunks = atoi(c);
    if (chunks > 1 && sim->use_tpm && n >= 65536) {
        if (!sim->host_start) {
            cudaEvent_t ev0 = nullptr, ev[2] = {nullptr, nullptr};
            cudaStream_t hs[2] = {nullptr, nullptr};
            EVG_TRY(cudaEventCreateWithFlags(&ev0, cudaEventDisableTiming), "cudaEventCreate");
            for (int i = 0; i < 2; ++i) {
                EVG_TRY(cudaStreamCreateWithFlags(&hs[i], cudaStreamNonBlocking), "cudaStreamCreate");
                EVG_TRY(cudaEventCreateWithFlags(&ev[i], cudaEventDisableTiming), "cudaEventCreate");
            }
            if (e != cudaSuccess) {  // nothing enqueued yet: release what was created and report
                for (int i = 0; i < 2; ++i) {
                    if (hs[i]) cudaStreamDestroy(hs[i]);
                    if (ev[i]) cudaEventDestroy(ev[i]);
                }
                if (ev0) cudaEventDestroy(ev0);
                return cuda_fail(e, what);
            }
            sim->host_start = ev0;
            for (int i = 0; i < 2; ++i) { sim->host_stream[i] = hs[i]; sim->host_done[i] = ev[i]; }
        }
        const int64_t per = ((n + chunks - 1) / chunks + 127) / 128 * 128;
        EVG_TRY(cudaEventRecord(sim->host_start, st), "cudaEventRecord");
        for (int i = 0; i < 2; ++i) EVG_TRY(cudaStreamWaitEvent(sim->host_stream[i], sim->host_start, 0), "cudaStreamWaitEvent");
        int c = 0;
        for (int64_t first = 0; first < n && e == cudaSuccess && rc == EVG_OK; first += per, ++c)
            rc = chunk(sim->host_stream[c & 1], first, n - first < per ? n - first : per, true, c & 1);  // a counter pair per stream
        // join: `stream` waits for both library streams whatever happened above
        for (int i = 0; i < 2; ++i) {
            cudaError_t j = cudaEventRecord(sim->host_done[i], sim->host_stream[i]);
            if (j == cudaSuccess) j = cudaStreamWaitEvent(st, sim->host_done[i], 0);
            if (j != cudaSuccess) {  // cannot even order the streams: drain them here so nothing outlives the call unordered
                cudaStreamSynchronize(sim->host_stream[i]);
                if (e == cudaSuccess) { e = j; what = "joining the chunk streams"; }
            }
        }
    } else {
        rc = chunk(st, 0, n, false, 0);
    }
#undef EVG_TRY
    if (rc) return rc;
    if (e != cudaSuccess) return cuda_fail(e, what);
    return EVG_OK;
}

int evg_step_host(EvgSim* sim, const int8_t* h_actions, float* h_obs, float* h_reward, uint8_t* h_done, int8_t* d_actions,
                  float* d_obs, float* d_reward, uint8_t* d_done, void* stream)
{
    if (!h_reward || !h_done) return fail(EVG_E_ARG, "evg_step_host: host buffers must be non-null");
    return evg_step_host_fmt(sim, EVG_OBS_F32, h_actions, h_obs, h_reward, h_done, d_actions, d_obs, nullptr, d_reward, d_done, stream);
}

int evg_export_state(EvgSim* sim, int64_t first, int64_t count, EvgEnvState* d_states, void* stream)
{
    int rc = check_sim(sim, true);
    if (rc) return rc;
    if (!d_states || first < 0 || count < 0 || first + count > sim->n_envs) return fail(EVG_E_ARG, "evg_export_state: bad range [%lld,+%lld)", (long long)first, (long long)count);
    cudaError_t e = evg::launch_export(sim->tables, (const uint32_t*)sim->bound[EVG_BIND_RECORDS], (const double*)sim->bound[EVG_BIND_HEALTH],
                                       first, count, d_states, (cudaStream_t)stream);
    if (e != cudaSuccess) return cuda_fail(e, "evg_export_kernel launch");
    sim->launches += count > 0;
    return EVG_OK;
}

int evg_import_state(EvgSim* sim, int64_t first, int64_t count, const EvgEnvState* d_states, void* stream)
{
    int rc = check_sim(sim, true);
    if (rc) return rc;
    if (!d_states || first < 0 || count < 0 || first + count > sim->n_envs) return fail(EVG_E_ARG, "evg_import_state: bad range [%lld,+%lld)", (long long)first, (long long)count);
    // The kernel forces out-of-range fields (a location outside 1..n_nodes, a control state beyond the node's
    // ControlPoints, ...) into range — they would index shared memory in the step kernels — and counts such records;
    // the count is read back here (this entry point is a test / checkpoint path: it synchronises `stream`).
    cudaStream_t st = (cudaStream_t)stream;
    unsigned* bad = (unsigned*)((unsigned long long*)sim->bound[EVG_BIND_STATS] + evg::kImportBadSlot);
    cudaError_t e = cudaMemsetAsync(bad, 0, sizeof(unsigned), st);
    if (e != cudaSuccess) return cuda_fail(e, "cudaMemsetAsync");
    e = evg::launch_import(sim->tables, (uint32_t*)sim->bound[EVG_BIND_RECORDS], (double*)sim->bound[EVG_BIND_HEALTH], first, count, d_states, bad, st);
    if (e != cudaSuccess) return cuda_fail(e, "evg_import_kernel launch");
    sim->launches += count > 0;
    unsigned h_bad = 0;
    if ((e = cudaMemcpyAsync(&h_bad, bad, sizeof(unsigned), cudaMemcpyDeviceToHost, st)) != cudaSuccess) return cuda_fail(e, "D2H import check");
    if ((e = cudaStreamSynchronize(st)) != cudaSuccess) return cuda_fail(e, "cudaStreamSynchronize");
    if (h_bad) return fail(EVG_E_ARG, "evg_import_state: %u field group(s) out of range (location 1..n_nodes, destination <= n_nodes, |controlState| <= ControlPoints, controlledBy -1..1); they were forced into range", h_bad);
    return EVG_OK;
}

int evg_episode_stats(EvgSim* sim, EvgEpisodeStats* host_out, void* stream)
{
    int rc = check_sim(sim, true);
    if (rc) return rc;
    if (!host_out) return fail(EVG_E_ARG, "null output");
    unsigned long long h[evg::ST_COUNT];
    cudaStream_t st = (cudaStream_t)stream;
    cudaError_t e = cudaMemcpyAsync(h, sim->bound[EVG_BIND_STATS], sizeof(h), cudaMemcpyDeviceToHost, st);
    if (e != cudaSuccess) return cuda_fail(e, "D2H stats");
    if ((e = cudaStreamSynchronize(st)) != cudaSuccess) return cuda_fail(e, "cudaStreamSynchronize");
    host_out->episodes = (int64_t)h[evg::ST_EPISODES];
    host_out->wins[0] = (int64_t)h[evg::ST_WIN0];
    host_out->wins[1] = (int64_t)h[evg::ST_WIN1];
    host_out->ties = (int64_t)h[evg::ST_TIES];
    host_out->total_turns = (int64_t)h[evg::ST_TURNS];
    host_out->total_score[0] = (int64_t)h[evg::ST_SCORE0];
    host_out->total_score[1] = (int64_t)h[evg::ST_SCORE1];
    for (int k = 0; k < 4; ++k) host_out->status_count[k] = (int64_t)h[evg::ST_STATUS0 + k];
    host_out->env_turns = sim->steps * sim->n_envs;
    host_out->fought_unit_slots = (int64_t)h[evg::ST_FOUGHT];
    return EVG_OK;
}

int evg_agent_random(EvgSim* sim, int8_t* d_actions, int32_t player, void* stream)
{
    int rc = check_sim(sim, true);
    if (rc) return rc;
    if (!d_actions || player < -1 || player > 1) return fail(EVG_E_ARG, "evg_agent_random: bad argument");
    cudaError_t e = evg::launch_agent_random(sim->tables, (const uint32_t*)sim->bound[EVG_BIND_RECORDS], d_actions, player, sim->n_envs,
                                             (cudaStream_t)stream);
    if (e != cudaSuccess) return cuda_fail(e, "evg_agent_random_kernel launch");
    sim->launches += 1;
    return EVG_OK;
}

int evg_agents(EvgSim* sim, int32_t agent_p0, int32_t agent_p1, int8_t* d_actions, void* stream)
{
    int rc = check_sim(sim, true);
    if (rc) return rc;
    if (!d_actions) return fail(EVG_E_ARG, "evg_agents: d_actions is null");
    const int ag[2] = {agent_p0, agent_p1};
    for (int p = 0; p < 2; ++p) {
        if (ag[p] < EVG_AGENT_EXTERNAL || ag[p] > EVG_AGENT_SWARM) return fail(EVG_E_ARG, "unknown agent id %d for player %d", ag[p], p);
        if (ag[p] == EVG_AGENT_RANDOM && sim->cfg.n_nodes > evg::kAgentMaxNodes) {  // byte-array variant lives in evg_agent_random
            if ((rc = evg_agent_random(sim, d_actions, p, stream))) return rc;
        }
    }
    const int a0 = (ag[0] == EVG_AGENT_RANDOM && sim->cfg.n_nodes > evg::kAgentMaxNodes) ? EVG_AGENT_EXTERNAL : ag[0];
    const int a1 = (ag[1] == EVG_AGENT_RANDOM && sim->cfg.n_nodes > evg::kAgentMaxNodes) ? EVG_AGENT_EXTERNAL : ag[1];
    if (a0 == EVG_AGENT_EXTERNAL && a1 == EVG_AGENT_EXTERNAL) return EVG_OK;
    cudaError_t e = evg::launch_agents(sim->tables, (const uint32_t*)sim->bound[EVG_BIND_RECORDS], (uint2*)sim->bound[EVG_BIND_AGENTS], d_actions,
                                       a0, a1, sim->n_envs, (cudaStream_t)stream);
    if (e != cudaSuccess) return cuda_fail(e, "evg_agents_kernel launch");
    sim->launches += 1;
    return EVG_OK;
}

int evg_decode_dqn(EvgSim* sim, const float* d_q, int32_t num_cols, int32_t player, int8_t* d_actions, void* stream)
{
    return evg_decode_dqn_layout(sim, d_q, num_cols, player, 0, d_actions, stream);
}

int evg_decode_dqn_layout(EvgSim* sim, const float* d_q, int32_t num_cols, int32_t player, int32_t q_transposed, int8_t* d_actions, void* stream)
{
    int rc = check_sim(sim, false);
    if (rc) return rc;
    if (!d_q || !d_actions || num_cols < 1 || num_cols > 127 || player < -1 || player > 1) return fail(EVG_E_ARG, "evg_decode_dqn: bad argument");
    cudaError_t e = evg::launch_decode_dqn(d_q, num_cols, player, d_actions, sim->n_envs, q_transposed, (cudaStream_t)stream);
    if (e != cudaSuccess) return cuda_fail(e, "evg_decode_dqn_kernel launch");
    sim->launches += 1;
    return EVG_OK;
}

int evg_decode_indices(EvgSim* sim, const int64_t* d_idx, int32_t div, int32_t mod, int32_t player, int8_t* d_actions, void* stream)
{
    int rc = check_sim(sim, false);
    if (rc) return rc;
    if (!d_idx || !d_actions || div < 1 || mod < 1 || player < -1 || player > 1) return fail(EVG_E_ARG, "evg_decode_indices: bad argument");
    cudaError_t e = evg::launch_decode_indices(d_idx, div, mod, player, d_actions, sim->n_envs, (cudaStream_t)stream);
    if (e != cudaSuccess) return cuda_fail(e, "evg_decode_indices_kernel launch");
    sim->launches += 1;
    return EVG_OK;
}

// the observations of a policy call: float32 (wire = null) or, EVG_OBS_WIRE, rows whose expansion reads the bound tables
static int policy_source(const char* fn, const EvgSim* sim, int32_t format, const void* d_obs, evg::WireSrc* wire, bool* use_wire)
{
    if (format != EVG_OBS_F32 && format != EVG_OBS_WIRE) return fail(EVG_E_ARG, "%s: observation format %d (EVG_OBS_F32 or EVG_OBS_WIRE)", fn, format);
    *use_wire = format == EVG_OBS_WIRE;
    if (!*use_wire) return EVG_OK;
    if (!sim->is_bound) return fail(EVG_E_STATE, "%s: evg_bind() must be called before reading wire rows", fn);
    if ((uintptr_t)d_obs % 16) return fail(EVG_E_ARG, "%s: wire rows must be 16-byte aligned", fn);
    *wire = wire_src(sim);
    return EVG_OK;
}

int evg_policy_mlp_fmt(EvgSim* sim, int32_t format, const void* d_obs, int64_t rows, const void* d_w1_img, const void* d_w2_img, int32_t hidden,
                       int32_t out_dim, float* d_q, int32_t q_transposed, void* stream)
{
    int rc = check_sim(sim, false);
    if (rc) return rc;
    if (!d_obs || !d_w1_img || !d_w2_img || !d_q || rows < 0) return fail(EVG_E_ARG, "evg_policy_mlp: null argument");
    evg::WireSrc ws;
    bool wire;
    if ((rc = policy_source("evg_policy_mlp", sim, format, d_obs, &ws, &wire))) return rc;
    if (wire && rows % 2) return fail(EVG_E_ARG, "evg_policy_mlp: %lld observation rows: wire rows hold both players, the count must be even", (long long)rows);
    if ((rc = check_mlp_shape("evg_policy_mlp", sim, hidden, out_dim, d_w1_img, d_w2_img))) return rc;
    const int n_chunks = (hidden + 1 + EVG_MLP_CHUNK - 1) / EVG_MLP_CHUNK;  // + the hidden unit that carries b2
    cudaError_t e = evg::launch_policy_mlp(d_obs, rows, sim->layout.obs_len, d_w1_img, d_w2_img, n_chunks, out_dim, d_q, q_transposed, sim->sm_count,
                                           (cudaStream_t)stream, wire ? &ws : nullptr);
    if (e != cudaSuccess) return cuda_fail(e, "evg_policy_mlp_kernel launch");
    sim->launches += 1;
    return EVG_OK;
}

int evg_policy_mlp(EvgSim* sim, const float* d_obs, int64_t rows, const void* d_w1_img, const void* d_w2_img, int32_t hidden, int32_t out_dim,
                   float* d_q, int32_t q_transposed, void* stream)
{
    return evg_policy_mlp_fmt(sim, EVG_OBS_F32, d_obs, rows, d_w1_img, d_w2_img, hidden, out_dim, d_q, q_transposed, stream);
}

int evg_policy_ppo_logp(EvgSim* sim, int32_t format, const void* d_obs, int32_t player, const void* d_w1_img, const void* d_w2_img,
                        const void* d_w3_img, const float* d_bias, int32_t latent, int32_t out_dim, int32_t div, int32_t mod, int8_t* d_actions,
                        int64_t* d_idx, float* d_probs, float* d_logp, void* stream)
{
    int rc = check_sim(sim, true);  // the draws read turn and episode from the bound records
    if (rc) return rc;
    if (!d_obs || !d_w1_img || !d_w2_img || !d_w3_img || !d_bias || !d_actions) return fail(EVG_E_ARG, "evg_policy_ppo: null argument");
    if (player < -1 || player > 1) return fail(EVG_E_ARG, "evg_policy_ppo: player %d outside -1..1", player);
    if (div < 1 || mod < 1) return fail(EVG_E_ARG, "evg_policy_ppo: div %d / mod %d must be positive", div, mod);
    evg::WireSrc ws;
    bool wire;
    if ((rc = policy_source("evg_policy_ppo", sim, format, d_obs, &ws, &wire))) return rc;
    if ((rc = check_actor_shape("evg_policy_ppo", sim, latent, out_dim, {d_w1_img, d_w2_img, d_w3_img}))) return rc;
    cudaError_t e = evg::launch_policy_ppo(sim->tables, (const uint32_t*)sim->bound[EVG_BIND_RECORDS], d_obs, sim->n_envs, player, d_w1_img, d_w2_img,
                                           d_w3_img, d_bias, latent, out_dim, div, mod, d_actions, d_idx, d_probs, d_logp, sim->sm_count,
                                           (cudaStream_t)stream, wire ? &ws : nullptr);
    if (e != cudaSuccess) return cuda_fail(e, "evg_policy_ppo_kernel launch");
    sim->launches += 1;
    return EVG_OK;
}

int evg_policy_ppo_fmt(EvgSim* sim, int32_t format, const void* d_obs, int32_t player, const void* d_w1_img, const void* d_w2_img,
                       const void* d_w3_img, const float* d_bias, int32_t latent, int32_t out_dim, int32_t div, int32_t mod, int8_t* d_actions,
                       int64_t* d_idx, float* d_probs, void* stream)
{
    return evg_policy_ppo_logp(sim, format, d_obs, player, d_w1_img, d_w2_img, d_w3_img, d_bias, latent, out_dim, div, mod, d_actions, d_idx,
                               d_probs, nullptr, stream);
}

int evg_policy_ppo(EvgSim* sim, const float* d_obs, int32_t player, const void* d_w1_img, const void* d_w2_img, const void* d_w3_img,
                   const float* d_bias, int32_t latent, int32_t out_dim, int32_t div, int32_t mod, int8_t* d_actions, int64_t* d_idx,
                   float* d_probs, void* stream)
{
    return evg_policy_ppo_logp(sim, EVG_OBS_F32, d_obs, player, d_w1_img, d_w2_img, d_w3_img, d_bias, latent, out_dim, div, mod, d_actions, d_idx,
                               d_probs, nullptr, stream);
}

int evg_policy_rppo_logp(EvgSim* sim, int32_t format, const void* d_obs, int32_t player, const void* d_w1_img, const void* d_w2_img,
                         const void* d_wi_img, const void* d_wh_img, const void* d_w3_img, const float* d_bias, int32_t latent,
                         int32_t out_dim, int32_t div, int32_t mod, float* d_hidden, float* d_hidden_in, int8_t* d_actions,
                         int64_t* d_idx, float* d_probs, float* d_logp, void* stream)
{
    int rc = check_sim(sim, true);  // the draws and the turn-0 reset of the state read the bound records
    if (rc) return rc;
    if (!d_obs || !d_w1_img || !d_w2_img || !d_wi_img || !d_wh_img || !d_w3_img || !d_bias || !d_actions)
        return fail(EVG_E_ARG, "evg_policy_rppo: null argument");
    if (!d_hidden) return fail(EVG_E_ARG, "evg_policy_rppo: d_hidden (the GRU state, in and out) is null");
    if (player < -1 || player > 1) return fail(EVG_E_ARG, "evg_policy_rppo: player %d outside -1..1", player);
    if (div < 1 || mod < 1) return fail(EVG_E_ARG, "evg_policy_rppo: div %d / mod %d must be positive", div, mod);
    if (d_hidden_in && latent > 0) {  // the kernel reads d_hidden after it has written d_hidden_in
        const uintptr_t bytes = (uintptr_t)(sim->n_envs * (player < 0 ? 2 : 1) * latent) * sizeof(float);
        const uintptr_t h = (uintptr_t)d_hidden, hi = (uintptr_t)d_hidden_in;
        if (hi < h + bytes && h < hi + bytes) return fail(EVG_E_ARG, "evg_policy_rppo: d_hidden_in overlaps d_hidden");
    }
    evg::WireSrc ws;
    bool wire;
    if ((rc = policy_source("evg_policy_rppo", sim, format, d_obs, &ws, &wire))) return rc;
    if ((rc = check_actor_shape("evg_policy_rppo", sim, latent, out_dim, {d_w1_img, d_w2_img, d_wi_img, d_wh_img, d_w3_img}))) return rc;
    cudaError_t e = evg::launch_policy_rppo(sim->tables, (const uint32_t*)sim->bound[EVG_BIND_RECORDS], d_obs, sim->n_envs, player, d_w1_img, d_w2_img,
                                            d_wi_img, d_wh_img, d_w3_img, d_bias, latent, out_dim, div, mod, d_hidden, d_hidden_in, d_actions,
                                            d_idx, d_probs, d_logp, sim->sm_count, (cudaStream_t)stream, wire ? &ws : nullptr);
    if (e != cudaSuccess) return cuda_fail(e, "evg_policy_rppo_kernel launch");
    sim->launches += 1;
    return EVG_OK;
}

int evg_policy_rppo_fmt(EvgSim* sim, int32_t format, const void* d_obs, int32_t player, const void* d_w1_img, const void* d_w2_img,
                        const void* d_wi_img, const void* d_wh_img, const void* d_w3_img, const float* d_bias, int32_t latent, int32_t out_dim,
                        int32_t div, int32_t mod, float* d_hidden, int8_t* d_actions, int64_t* d_idx, float* d_probs, void* stream)
{
    return evg_policy_rppo_logp(sim, format, d_obs, player, d_w1_img, d_w2_img, d_wi_img, d_wh_img, d_w3_img, d_bias, latent, out_dim, div, mod,
                                d_hidden, nullptr, d_actions, d_idx, d_probs, nullptr, stream);
}

int evg_policy_rppo(EvgSim* sim, const float* d_obs, int32_t player, const void* d_w1_img, const void* d_w2_img, const void* d_wi_img,
                    const void* d_wh_img, const void* d_w3_img, const float* d_bias, int32_t latent, int32_t out_dim, int32_t div, int32_t mod,
                    float* d_hidden, int8_t* d_actions, int64_t* d_idx, float* d_probs, void* stream)
{
    return evg_policy_rppo_logp(sim, EVG_OBS_F32, d_obs, player, d_w1_img, d_w2_img, d_wi_img, d_wh_img, d_w3_img, d_bias, latent, out_dim, div,
                                mod, d_hidden, nullptr, d_actions, d_idx, d_probs, nullptr, stream);
}

// the critic's checks (evg_policy_value, evg_pack_value); `aligned`: what the call reads or writes in 16 B
static int check_value_shape(const char* fn, const EvgSim* sim, int32_t latent, std::initializer_list<const void*> aligned)
{
    if (latent < 1 || latent > EVG_PPO_MAX_LATENT) return fail(EVG_E_ARG, "%s: latent %d outside 1..%d", fn, latent, EVG_PPO_MAX_LATENT);
    for (const void* p : aligned)
        if ((uintptr_t)p % 16) return fail(EVG_E_ARG, "%s: weight images and the packed bias vector must be 16-byte aligned", fn);
    if (sim->layout.obs_len >= EVG_PPO_IN_PAD) return fail(EVG_E_ARG, "%s: observations of %d values exceed the %d the kernel is tiled for", fn, sim->layout.obs_len, EVG_PPO_IN_PAD - 1);
    return EVG_OK;
}

int evg_policy_value(EvgSim* sim, int32_t format, const void* d_obs, int64_t n_matches, int32_t player, const void* d_w1_img,
                     const void* d_w2_img, const void* d_w3_img, const float* d_bias, int32_t latent, float* d_value, void* stream)
{
    int rc = check_sim(sim, false);
    if (rc) return rc;
    if (!d_obs || !d_w1_img || !d_w2_img || !d_w3_img || !d_bias || !d_value) return fail(EVG_E_ARG, "evg_policy_value: null argument");
    if (n_matches < 0) return fail(EVG_E_ARG, "evg_policy_value: negative match count %lld", (long long)n_matches);
    if (player < -1 || player > 1) return fail(EVG_E_ARG, "evg_policy_value: player %d outside -1..1", player);
    if ((uintptr_t)d_obs % 4 || (uintptr_t)d_value % 4) return fail(EVG_E_ARG, "evg_policy_value: observations and values must be 4-byte aligned");
    evg::WireSrc ws;
    bool wire;
    if ((rc = policy_source("evg_policy_value", sim, format, d_obs, &ws, &wire))) return rc;
    if ((rc = check_value_shape("evg_policy_value", sim, latent, {d_w1_img, d_w2_img, d_w3_img, d_bias}))) return rc;
    if (n_matches == 0) return EVG_OK;
    cudaError_t e = evg::launch_policy_value(d_obs, n_matches, player, sim->layout.obs_len, d_w1_img, d_w2_img, d_w3_img, d_bias, latent, d_value,
                                             sim->sm_count, (cudaStream_t)stream, wire ? &ws : nullptr);
    if (e != cudaSuccess) return cuda_fail(e, "evg_policy_value_kernel launch");
    sim->launches += 1;
    return EVG_OK;
}

int evg_wire_expand(EvgSim* sim, const void* d_rows, int64_t n_rows, const int64_t* d_index, int64_t n_out, int32_t player, float* d_obs,
                    float* d_reward, uint8_t* d_done, void* stream)
{
    int rc = check_sim(sim, true);  // the constant entries and p1_map are in the bound tables
    if (rc) return rc;
    if (!d_rows || !d_obs) return fail(EVG_E_ARG, "evg_wire_expand: null argument");
    if (n_rows < 0 || n_out < 0) return fail(EVG_E_ARG, "evg_wire_expand: negative row count");
    if (!d_index && n_out != n_rows) return fail(EVG_E_ARG, "evg_wire_expand: without an index n_out (%lld) must equal n_rows (%lld)", (long long)n_out, (long long)n_rows);
    if (player < -1 || player > 1) return fail(EVG_E_ARG, "evg_wire_expand: player %d outside -1..1", player);
    if (((uintptr_t)d_rows | (uintptr_t)d_obs) % 16 || (uintptr_t)d_index % 8 || (uintptr_t)d_reward % 4)
        return fail(EVG_E_ARG, "evg_wire_expand: rows and obs must be 16-byte aligned, index 8-byte, reward 4-byte");
    cudaError_t e = evg::launch_wire_expand(wire_src(sim), (const uint32_t*)d_rows, n_rows, d_index, n_out, player, d_obs, d_reward, d_done,
                                            (cudaStream_t)stream);
    if (e != cudaSuccess) return cuda_fail(e, "evg_wire_expand_kernel launch");
    sim->launches += 1;
    return EVG_OK;
}

int evg_gae(EvgSim* sim, int32_t n_turns, int64_t n_matches, int32_t player, const void* d_rows, const float* d_reward, const uint8_t* d_done,
            const float* d_values, float gamma, float lam, float* d_adv, float* d_ret, void* stream)
{
    int rc = check_sim(sim, false);
    if (rc) return rc;
    if (n_turns < 1) return fail(EVG_E_ARG, "evg_gae: n_turns %d must be at least 1", n_turns);
    if (n_matches < 1 || n_matches > INT32_MAX) return fail(EVG_E_ARG, "evg_gae: n_matches %lld outside 1..2^31-1", (long long)n_matches);
    if (player < -1 || player > 1) return fail(EVG_E_ARG, "evg_gae: player %d outside -1..1", player);
    if (!d_values || !d_adv || !d_ret) return fail(EVG_E_ARG, "evg_gae: null values, adv or ret");
    if (!d_rows && (!d_reward || !d_done)) return fail(EVG_E_ARG, "evg_gae: the wire rows are needed unless both reward and done are given");
    if ((uintptr_t)d_rows % 16) return fail(EVG_E_ARG, "evg_gae: wire rows must be 16-byte aligned");
    const uintptr_t col = player < 0 ? 8 : 4;  // float2 operands of player -1
    if (((uintptr_t)d_values | (uintptr_t)d_adv | (uintptr_t)d_ret) % col || (uintptr_t)d_reward % col)
        return fail(EVG_E_ARG, "evg_gae: values, adv, ret and reward must be %d-byte aligned", (int)col);
    if (!(gamma >= 0.f && gamma <= 1.f) || !(lam >= 0.f && lam <= 1.f))  // NaN fails both comparisons
        return fail(EVG_E_ARG, "evg_gae: gamma %g and lambda %g must lie in [0, 1]", (double)gamma, (double)lam);
    const int n = sim->tables.n_nodes;
    cudaError_t e = evg::launch_gae(n_turns, n_matches, player, (const uint32_t*)d_rows, evg::wire_bytes(n) / 4,
                                    (EVG_WIRE_NODE0 + 4 * n + 3 * evg::kGroupLanes) / 4, d_reward, d_done, d_values, gamma, lam, d_adv,
                                    d_ret, (cudaStream_t)stream);
    if (e != cudaSuccess) return cuda_fail(e, "evg_gae_kernel launch");
    sim->launches += 1;
    return EVG_OK;
}

namespace {

// evg_ppo_loss / _grad's shared argument checks, before the handle's, so they hold without a device
int check_ppo_loss(const char* fn, int64_t n_rows, int32_t n_dist, int32_t n_actions, float clip, const void* const* f32, int n_f32,
                   const int64_t* d_idx)
{
    if (n_rows < 1 || n_rows > INT32_MAX) return fail(EVG_E_ARG, "%s: n_rows %lld outside 1..2^31-1", fn, (long long)n_rows);
    if (n_dist != 1 && n_dist != EVG_MAX_ACTIONS) return fail(EVG_E_ARG, "%s: n_dist %d must be 1 or %d", fn, n_dist, EVG_MAX_ACTIONS);
    if (n_actions < EVG_MAX_ACTIONS || n_actions > 256) return fail(EVG_E_ARG, "%s: n_actions %d outside %d..256", fn, n_actions, EVG_MAX_ACTIONS);
    if (!(clip >= 0.f && clip < 1.f)) return fail(EVG_E_ARG, "%s: clip %g outside [0, 1)", fn, (double)clip);  // NaN fails too
    if (!d_idx) return fail(EVG_E_ARG, "%s: null idx", fn);
    if ((uintptr_t)d_idx % 8) return fail(EVG_E_ARG, "%s: idx must be 8-byte aligned", fn);
    for (int i = 0; i < n_f32; ++i) {
        if (!f32[i]) return fail(EVG_E_ARG, "%s: null float32 operand %d", fn, i);
        if ((uintptr_t)f32[i] % 4) return fail(EVG_E_ARG, "%s: float32 operand %d must be 4-byte aligned", fn, i);
    }
    return EVG_OK;
}

}  // namespace

int evg_ppo_loss(EvgSim* sim, int64_t n_rows, int32_t n_dist, int32_t n_actions, const float* d_z, const int64_t* d_idx, const float* d_old_logp,
                 const float* d_adv, float clip, float* d_surr, float* d_ent, float* d_logp, float* d_ratio, void* stream)
{
    const void* f32[] = {d_z, d_old_logp, d_adv, d_surr, d_ent, d_logp, d_ratio};
    int rc = check_ppo_loss("evg_ppo_loss", n_rows, n_dist, n_actions, clip, f32, 7, d_idx);
    if (rc || (rc = check_sim(sim, false))) return rc;
    cudaError_t e = evg::launch_ppo_loss(n_rows, n_dist, n_actions, d_z, d_idx, d_old_logp, d_adv, 1.f - clip, 1.f + clip, d_surr, d_ent, d_logp,
                                         d_ratio, sim->sm_count, (cudaStream_t)stream);
    if (e != cudaSuccess) return cuda_fail(e, "evg_ppo_loss kernel launch");
    sim->launches += 1;
    return EVG_OK;
}

int evg_ppo_loss_grad(EvgSim* sim, int64_t n_rows, int32_t n_dist, int32_t n_actions, const float* d_z, const int64_t* d_idx, const float* d_adv,
                      const float* d_ratio, float clip, const float* d_g_surr, const float* d_g_ent, float* d_dz, void* stream)
{
    const void* f32[] = {d_z, d_adv, d_ratio, d_dz};
    int rc = check_ppo_loss("evg_ppo_loss_grad", n_rows, n_dist, n_actions, clip, f32, 4, d_idx);
    if (rc) return rc;
    if ((uintptr_t)d_g_surr % 4 || (uintptr_t)d_g_ent % 4) return fail(EVG_E_ARG, "evg_ppo_loss_grad: g_surr and g_ent must be 4-byte aligned");
    if ((rc = check_sim(sim, false))) return rc;
    cudaError_t e = evg::launch_ppo_loss_grad(n_rows, n_dist, n_actions, d_z, d_idx, d_adv, d_ratio, 1.f - clip, 1.f + clip, d_g_surr, d_g_ent,
                                              d_dz, sim->sm_count, (cudaStream_t)stream);
    if (e != cudaSuccess) return cuda_fail(e, "evg_ppo_loss_grad kernel launch");
    sim->launches += 1;
    return EVG_OK;
}

namespace {

// evg_rppo_train_*'s shared argument checks, before the handle's, so they hold without a device: the sizes, then every
// pointer non-null, images and the bias vector 16-byte aligned, float32 arrays 4-byte aligned
int check_rppo_train(const char* fn, int64_t n_rows, int32_t latent, int32_t out_dim, std::initializer_list<const void*> img,
                     std::initializer_list<const void*> f32)
{
    if (n_rows < 1 || n_rows > INT32_MAX) return fail(EVG_E_ARG, "%s: n_rows %lld outside 1..2^31-1", fn, (long long)n_rows);
    if (latent < 1 || latent > EVG_PPO_MAX_LATENT) return fail(EVG_E_ARG, "%s: latent %d outside 1..%d", fn, latent, EVG_PPO_MAX_LATENT);
    if (out_dim < EVG_MAX_ACTIONS || out_dim > EVG_PPO_OUT_PAD) return fail(EVG_E_ARG, "%s: out_dim %d outside %d..%d", fn, out_dim, EVG_MAX_ACTIONS, EVG_PPO_OUT_PAD);
    for (const void* p : img) {
        if (!p) return fail(EVG_E_ARG, "%s: null image or bias vector", fn);
        if ((uintptr_t)p % 16) return fail(EVG_E_ARG, "%s: images and the bias vector must be 16-byte aligned", fn);
    }
    for (const void* p : f32) {
        if (!p) return fail(EVG_E_ARG, "%s: null float32 array", fn);
        if ((uintptr_t)p % 4) return fail(EVG_E_ARG, "%s: float32 arrays must be 4-byte aligned", fn);
    }
    return EVG_OK;
}

}  // namespace

int evg_rppo_train_pack(EvgSim* sim, const float* d_w3, const float* d_b3, const float* d_w_ih, const float* d_b_ih, const float* d_w_hh,
                        const float* d_b_hh, int32_t latent, int32_t out_dim, void* d_wi_img, void* d_wh_img, void* d_wht_img, void* d_w3_img,
                        float* d_bias, void* stream)
{
    int rc = check_rppo_train("evg_rppo_train_pack", 1, latent, out_dim, {d_wi_img, d_wh_img, d_wht_img, d_w3_img, d_bias},
                              {d_w3, d_b3, d_w_ih, d_b_ih, d_w_hh, d_b_hh});
    if (rc || (rc = check_sim(sim, false))) return rc;
    cudaError_t e = evg::launch_pack_rppo_train(d_w3, d_b3, d_w_ih, d_b_ih, d_w_hh, d_b_hh, latent, out_dim, d_wi_img, d_wh_img, d_wht_img, d_w3_img,
                                                d_bias, (cudaStream_t)stream);
    if (e != cudaSuccess) return cuda_fail(e, "evg_policy_pack_kernel launch");
    sim->launches += 1;
    return EVG_OK;
}

int evg_rppo_train_forward(EvgSim* sim, int64_t n_rows, int32_t latent, int32_t out_dim, const float* d_x, const float* d_h0, const void* d_wi_img,
                           const void* d_wh_img, const void* d_w3_img, const float* d_bias, float* d_z, float* d_h, void* stream)
{
    int rc = check_rppo_train("evg_rppo_train_forward", n_rows, latent, out_dim, {d_wi_img, d_wh_img, d_w3_img, d_bias}, {d_x, d_h0, d_z, d_h});
    if (rc || (rc = check_sim(sim, false))) return rc;
    cudaError_t e = evg::launch_rppo_train_forward(n_rows, latent, out_dim, d_x, d_h0, d_wi_img, d_wh_img, d_w3_img, d_bias, d_z, d_h, sim->sm_count,
                                                   (cudaStream_t)stream);
    if (e != cudaSuccess) return cuda_fail(e, "evg_rppo_train_kernel<forward> launch");
    sim->launches += 1;
    return EVG_OK;
}

int evg_rppo_train_backward(EvgSim* sim, int64_t n_rows, int32_t latent, int32_t out_dim, const float* d_x, const float* d_h0, const float* d_h,
                            const void* d_wi_img, const void* d_wh_img, const void* d_wht_img, const float* d_bias, float* d_g, float* d_dgh,
                            float* d_s, void* stream)
{
    int rc = check_rppo_train("evg_rppo_train_backward", n_rows, latent, out_dim, {d_wi_img, d_wh_img, d_wht_img, d_bias},
                              {d_x, d_h0, d_h, d_g, d_dgh, d_s});
    if (rc || (rc = check_sim(sim, false))) return rc;
    cudaError_t e = evg::launch_rppo_train_backward(n_rows, latent, out_dim, d_x, d_h0, d_h, d_wi_img, d_wh_img, d_wht_img, d_bias, d_g, d_dgh, d_s,
                                                    sim->sm_count, (cudaStream_t)stream);
    if (e != cudaSuccess) return cuda_fail(e, "evg_rppo_train_kernel<backward> launch");
    sim->launches += 1;
    return EVG_OK;
}

int evg_pack_mlp(EvgSim* sim, const float* d_w1, const float* d_b1, const float* d_w2, const float* d_b2, int32_t hidden, int32_t out_dim,
                 void* d_w1_img, void* d_w2_img, void* stream)
{
    int rc = check_sim(sim, false);
    if (rc) return rc;
    if (!d_w1 || !d_b1 || !d_w2 || !d_b2 || !d_w1_img || !d_w2_img) return fail(EVG_E_ARG, "evg_pack_mlp: null argument");
    if ((rc = check_mlp_shape("evg_pack_mlp", sim, hidden, out_dim, d_w1_img, d_w2_img))) return rc;
    cudaError_t e = evg::launch_pack_mlp(sim->layout.obs_len, d_w1, d_b1, d_w2, d_b2, hidden, out_dim, d_w1_img, d_w2_img, (cudaStream_t)stream);
    if (e != cudaSuccess) return cuda_fail(e, "evg_policy_pack_kernel launch");
    sim->launches += 1;
    return EVG_OK;
}

int evg_pack_ppo(EvgSim* sim, const float* d_w1, const float* d_b1, const float* d_w2, const float* d_b2, const float* d_w3, const float* d_b3,
                 int32_t latent, int32_t out_dim, void* d_w1_img, void* d_w2_img, void* d_w3_img, float* d_bias, void* stream)
{
    return pack_ppo_family("evg_pack_ppo", sim, d_w1, d_b1, d_w2, d_b2, d_w3, d_b3, nullptr, nullptr, nullptr, nullptr, latent, out_dim,
                           d_w1_img, d_w2_img, nullptr, nullptr, d_w3_img, d_bias, stream);
}

int evg_pack_rppo(EvgSim* sim, const float* d_w1, const float* d_b1, const float* d_w2, const float* d_b2, const float* d_w3, const float* d_b3,
                  const float* d_w_ih, const float* d_b_ih, const float* d_w_hh, const float* d_b_hh, int32_t latent, int32_t out_dim,
                  void* d_w1_img, void* d_w2_img, void* d_wi_img, void* d_wh_img, void* d_w3_img, float* d_bias, void* stream)
{
    if (!d_w_ih || !d_b_ih || !d_w_hh || !d_b_hh || !d_wi_img || !d_wh_img) return fail(EVG_E_ARG, "evg_pack_rppo: null argument");
    return pack_ppo_family("evg_pack_rppo", sim, d_w1, d_b1, d_w2, d_b2, d_w3, d_b3, d_w_ih, d_b_ih, d_w_hh, d_b_hh, latent, out_dim,
                           d_w1_img, d_w2_img, d_wi_img, d_wh_img, d_w3_img, d_bias, stream);
}

int evg_pack_value(EvgSim* sim, const float* d_w1, const float* d_b1, const float* d_w2, const float* d_b2, const float* d_w3,
                   const float* d_b3, int32_t latent, void* d_w1_img, void* d_w2_img, void* d_w3_img, float* d_bias, void* stream)
{
    int rc = check_sim(sim, false);
    if (rc) return rc;
    if (!d_w1 || !d_b1 || !d_w2 || !d_b2 || !d_w3 || !d_b3 || !d_w1_img || !d_w2_img || !d_w3_img || !d_bias)
        return fail(EVG_E_ARG, "evg_pack_value: null argument");
    if ((rc = check_value_shape("evg_pack_value", sim, latent, {d_w1_img, d_w2_img, d_w3_img, d_bias}))) return rc;
    cudaError_t e = evg::launch_pack_value(sim->layout.obs_len, d_w1, d_b1, d_w2, d_b2, d_w3, d_b3, latent, d_w1_img, d_w2_img, d_w3_img, d_bias,
                                           (cudaStream_t)stream);
    if (e != cudaSuccess) return cuda_fail(e, "evg_policy_pack_kernel launch");
    sim->launches += 1;
    return EVG_OK;
}

int evg_shape_reward(EvgSim* sim, int32_t mode, const float* d_reward, const uint8_t* d_done, const float* d_obs, float* d_out,
                     void* stream)
{
    int rc = check_sim(sim, false);
    if (rc) return rc;
    if (!d_reward || !d_done || !d_obs || !d_out || mode < EVG_SHAPE_NORMALIZED_SCORE || mode > EVG_SHAPE_SHORT_GAMES)
        return fail(EVG_E_ARG, "evg_shape_reward: bad argument");
    cudaError_t e = evg::launch_shape_reward(mode, d_reward, d_done, d_obs, sim->layout.obs_len, d_out, sim->n_envs, (cudaStream_t)stream);
    if (e != cudaSuccess) return cuda_fail(e, "evg_shape_reward_kernel launch");
    sim->launches += 1;
    return EVG_OK;
}

int evg_step_kernel_kind(const EvgSim* sim) { return !sim ? -1 : sim->use_tpm ? 1 : 0; }

int64_t evg_launch_count(const EvgSim* sim) { return sim ? sim->launches : -1; }

}  // extern "C"

// evg_internal.h — device tables, resident record layout, the tape's Philox and launcher prototypes, shared by every
// translation unit: the kernels (evg_kernels.cu, evg_step_tpm.cu, evg_policy_*.cu, through evg_tcgen05.cuh for the
// tensor-core ones) and evg_capi.cu (the C ABI of include/evgsim.h).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/evgsim.h"

namespace evg {

constexpr int kWarpsPerBlock = 8;
constexpr int kThreads = kWarpsPerBlock * 32;
constexpr int kGroupLanes = EVG_NUM_PLAYERS * EVG_NUM_GROUPS;  // 24: lane = side*12 + gid
constexpr int kNN = EVG_MAX_NODES + 1;

// ---------------------------------------------------------------------------------------------
// Resident per-match record (DESIGN.md §3), 32-bit words, little endian:
//   [0..47]   24 group records, 2 words each (lane L owns words 2L, 2L+1)
//       w0: loc[0:6) dest[6:12) dist[12:20) ready[20] moving[21] avg_health[24:31)
//       w1: alive unit mask[0:16) arrival turn[16:32)
//   [48]      turn            [49] episode
//   [50+i]    node i+1: controlState int16 | controlledBy int8 << 16
// padded to a multiple of 32 bytes (DemoMap: 61 words -> 256 B = one 8-byte load per lane).
// Unit health lives apart: double[health_slots] per match, group (side,g) at slot g_slot[L].
// ---------------------------------------------------------------------------------------------
constexpr int kRecGroupWords = 2 * kGroupLanes;  // 48
constexpr int kRecTurn = 48;
constexpr int kRecEpisode = 49;
constexpr int kRecNode0 = 50;

constexpr uint32_t W0_LOC_MASK = 0x3Fu;
constexpr int W0_DEST_SHIFT = 6;
constexpr int W0_DIST_SHIFT = 12;
constexpr uint32_t W0_READY = 1u << 20;
constexpr uint32_t W0_MOVING = 1u << 21;
constexpr int W0_AVG_SHIFT = 24;

// Static tables, passed to every kernel by value (__grid_constant__) and staged in shared memory.
struct alignas(16) Tables {
    int32_t n_nodes, obs_len, rec_words8, health_slots;
    int32_t turn_limit, capture_bonus, auto_reset, max_group_size;
    int32_t has_small_groups, hist_words, n_big, pad1;  // hist_words: u32 words per side of the damage histogram
    uint32_t seed_lo, seed_hi, env_base;
    uint32_t cta_fought;  // 0 here; in a CTA's shared-memory copy: unit slots its matches fought this launch (ST_FOUGHT)
    float max_score_f;
    float pad5;
    // per-warp shared-memory carve-up (bytes)
    int32_t sm_acc, sm_hist, sm_obs, sm_misc, sm_warp_stride, sm_tables_bytes;
    uint32_t cta_sched[2];  // 0 here; in a CTA's shared-memory copy: the batch indices thread 0 drew for the CTA (thread-per-match kernel)
    double node_def[kNN];
    double unit_armor[EVG_MAX_UNIT_TYPES];
    uint32_t init_w0[kGroupLanes], init_w1[kGroupLanes];
    uint32_t init_node[kNN];
    int16_t node_cp[kNN];
    uint16_t g_slot[kGroupLanes];
    int8_t node_team_start[kNN];
    uint8_t node_flags[kNN];  // bit0 'DEFENSE' (obs), bit1 'OBSERVE' (obs), bit2 'DEFEND' (combat bonus)
    uint8_t p1_map[kNN];
    uint8_t ut_damage[EVG_MAX_UNIT_TYPES], ut_speed[EVG_MAX_UNIT_TYPES], ut_control[EVG_MAX_UNIT_TYPES],
        ut_cost[EVG_MAX_UNIT_TYPES];
    uint8_t g_type[kGroupLanes], g_size[kGroupLanes];
    uint8_t g_big[kGroupLanes];  // ordinal among the groups with more than 8 units (index into the hbig scratch)
    uint8_t g_damage[kGroupLanes], g_speed[kGroupLanes], g_control[kGroupLanes], g_cost[kGroupLanes];  // per group lane
    uint8_t base_own[2];          // the opposing base in each player's own numbering (base_rushV1's target)
    uint8_t pad_own[2];
    uint8_t maxnb_own[2][kNN];    // highest-numbered neighbour of an own-numbered node (SwarmAgent's move)
    uint8_t edge[kNN][kNN];
    // thread-per-match kernel (evg_step_tpm.cu): per-thread shared-memory row = record + scratch (pitch, in 32-bit
    // words) and a per-warp damage-histogram pool sized for one round of 32 fighting groups
    int32_t tpm_pitch, tpm_pool_words, tpm_hist16;
    uint32_t big_mask;  // group lanes (bit L) with more than 8 unit slots
    // per group, one word instead of several byte tables.  g_move[2 * gid + player]: speed [0:8) | control [8:14) | cost [16:24);
    // g_fight[lane]: health slot [0:12) | unit slots [12:17) | damage [17:25) | unit type [25:28)
    alignas(8) uint32_t g_move[kGroupLanes];
    uint32_t g_fight[kGroupLanes];
    uint32_t node_cap[kNN];  // control points [0:16) | (TeamStart + 1) [16:18)
    uint32_t pad_t;
    uint64_t p1_nib;  // p1_map as nibbles (node i at bits [4i, 4i+4)) for maps of <= 15 nodes: a register lookup
    int32_t pad_p[2];
    const double* loss_tab;  // [type][node][bonus][32]: (10.*d)/(armor + bonus*StructureDefense), d < 32
    const double* rcp_tab;   // [type][node][bonus]: 1 / (armor + bonus*StructureDefense), correctly rounded
    int32_t fast_div;        // 1: (10.*d)/divisor == the two-FMA correction of (10.*d)*rcp for every reachable d (checked on the host)
    int32_t max_damage_sum;  // most damage one unit can collect in a turn
};

constexpr int kLossD = 32;
constexpr int kAgentMaxNodes = 15;  // nibble-packed node permutation of the on-device random agent
constexpr int kTpmThreads = 128;
constexpr int kTpmSmallThreads = 32;  // the one-warp-per-CTA instantiation for small batches (compile-time map only)
constexpr int kTpmMinCtas = 3;        // resident 128-thread CTAs per SM the thread-per-match kernel is compiled for
constexpr int kTpmLiteMinCtas = 14;   // resident one-warp CTAs per SM the LITE instantiation is compiled for (register cap 144)
constexpr int kTpmStage = 32;         // observation staging window per match, 32-bit words

// device statistics accumulators (uint64 each); matches EvgEpisodeStats minus env_turns
// ST_FOUGHT: unit slots of the groups that took part in combat (every match-turn, finished or not): the health term of
// the step's algorithmic bytes is 16 B per such slot (SURVEY.md §8d), so bench.py can state it for the turns it timed
enum { ST_EPISODES = 0, ST_WIN0, ST_WIN1, ST_TIES, ST_TURNS, ST_SCORE0, ST_SCORE1, ST_STATUS0, ST_FOUGHT = ST_STATUS0 + 4, ST_COUNT };
constexpr int kSchedSlots = 2;  // behind the statistics in the same bound array: one counter pair (8 bytes) per concurrent launch
constexpr int kImportBadSlot = ST_COUNT + kSchedSlots;  // then: records evg_import_state had to force into range (uint32)

struct StepArgs {
    uint32_t* records;
    double* health;
    unsigned long long* stats;
    const int8_t* actions;
    float* obs;
    float* reward;
    uint8_t* done;
    uint8_t* status;
    int32_t* scores;
    int64_t n_envs;
    int32_t agent[2];      // EVG_AGENT_*: where each player's action rows come from
    int8_t* actions_out;   // optional: rows generated by scripted agents are also written here
    const uint4* tables_dev;  // the Tables struct in device memory (bind slot EVG_BIND_TABLES): staged with coalesced loads
    const float* oconst_dev;  // behind it: the constant observation entries as floats (oconst_bytes(n_nodes), filled by evg_bind)
    int64_t env_first;        // thread-per-match kernel: this launch covers matches [env_first, env_first + n_envs) of the
                              // simulator (all pointers above are already offset); 0 for a whole-batch launch
    int32_t n_turns;          // thread-per-match kernel, both players scripted: game turns this launch plays (evg_rollout); else 1
    unsigned* sched;          // thread-per-match kernel: {batches handed out after the first wave, CTAs finished}, zero between launches
    uint2* agent_state;       // per (match, player) state of the observation-driven scripted agents (bind slot EVG_BIND_AGENTS)
    int32_t obs_fmt;          // EVG_OBS_F32: `obs` is float32[n][2][obs_len]; EVG_OBS_WIRE: packed rows of wire_bytes(n_nodes)
};

// bytes of the constant observation entries a step kernel keeps at hand: 2 * obs_len floats (padded to 16 bytes), then
// per [player][viewer slot] the node's two flags as a float2
__host__ __device__ inline int oconst_bytes(int n_nodes)
{
    const int ol = 1 + 4 * n_nodes + 5 * EVG_NUM_GROUPS;
    return ((2 * ol + 3) & ~3) * 4 + ((2 * n_nodes * 8 + 15) & ~15);
}

// bytes of one match's wire row (include/evgsim.h, EVG_OBS_WIRE)
__host__ __device__ inline int wire_bytes(int n_nodes) { return (EVG_WIRE_NODE0 + 4 * n_nodes + 3 * kGroupLanes + 8 + 15) / 16 * 16; }

// What expanding a wire row into the float32 observation vector needs besides the row (evg_wire_expand.cu and the policy
// kernels' wire stager): the simulator's constant entries (oconst_bytes layout, StepArgs::oconst_dev) and player 1's node
// numbering (Tables::p1_map), both in the simulator's bound tables on the device
struct WireSrc {
    const float* oconst;
    const uint8_t* p1_map;
    int32_t n_nodes, obs_len;
    int32_t words;  // 32-bit words of a row
};

// Kernels that need more than 48 KB of dynamic shared memory are opted in up to the DEVICE limit, not up to what one
// simulator needs: the attribute is per function, and simulators of different configurations share the functions.
inline cudaError_t optin_smem_limit(size_t needed, int* limit)
{
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e == cudaSuccess) e = cudaDeviceGetAttribute(limit, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev);
    if (e == cudaSuccess && needed > (size_t)*limit) e = cudaErrorInvalidValue;
    return e;
}

// launchers (evg_kernels.cu); all asynchronous on `stream`, return the launch error
cudaError_t launch_step(const Tables& t, const StepArgs& a, int grid, size_t smem, cudaStream_t stream);
cudaError_t launch_rollout(const Tables& t, const StepArgs& a, int n_turns, int grid, size_t smem, cudaStream_t stream);
cudaError_t launch_reset(const Tables& t, uint32_t* records, double* health, const uint8_t* mask, void* obs, int obs_fmt,
                         int64_t n_envs, int grid, size_t smem, cudaStream_t stream);
// the policy launchers read float32 observations from `obs`, or wire rows when `wire` is not null
cudaError_t launch_policy_mlp(const void* obs, int64_t rows, int in_dim, const void* w1_img, const void* w2_img, int n_chunks, int out_dim, float* q,
                              int transposed, int sm_count, cudaStream_t stream, const WireSrc* wire = nullptr);
cudaError_t launch_policy_ppo(const Tables& t, const uint32_t* records, const void* obs, int64_t n_envs, int player, const void* w1_img,
                              const void* w2_img, const void* w3_img, const float* bias, int latent, int out_dim, int div, int mod,
                              int8_t* actions, int64_t* idx, float* probs, float* logp, int sm_count, cudaStream_t stream,
                              const WireSrc* wire = nullptr);
cudaError_t launch_policy_rppo(const Tables& t, const uint32_t* records, const void* obs, int64_t n_envs, int player, const void* w1_img,
                               const void* w2_img, const void* wi_img, const void* wh_img, const void* w3_img, const float* bias, int latent,
                               int out_dim, int div, int mod, float* hidden, float* hidden_in, int8_t* actions, int64_t* idx, float* probs,
                               float* logp, int sm_count, cudaStream_t stream, const WireSrc* wire = nullptr);
cudaError_t launch_policy_value(const void* obs, int64_t n_matches, int player, int in_dim, const void* w1_img, const void* w2_img,
                                const void* w3_img, const float* bias, int latent, float* value, int sm_count, cudaStream_t stream,
                                const WireSrc* wire = nullptr);
// wire rows -> float32 observations, reward and done (evg_wire_expand.cu); index / reward / done may be null
cudaError_t launch_wire_expand(const WireSrc& w, const uint32_t* rows, int64_t n_rows, const int64_t* index, int64_t n_out, int player,
                               float* obs, float* reward, uint8_t* done, cudaStream_t stream);
// GAE(lambda) advantages and returns of a stored rollout (evg_gae.cu); rows (`words` 32-bit words each, the rewards at
// `reward_word`) are read only for what reward / done do not give
cudaError_t launch_gae(int n_turns, int64_t n_matches, int player, const uint32_t* rows, int words, int reward_word, const float* reward,
                       const uint8_t* done, const float* values, float gamma, float lam, float* adv, float* ret, cudaStream_t stream);
// PPO's policy loss from the actor's last Linear output, forward and gradient (evg_ppo_loss.cu); lo / hi are
// fl(1 - clip) and fl(1 + clip); g_surr / g_ent may be null; sm_count sizes the persistent grid
cudaError_t launch_ppo_loss(int64_t n_rows, int n_dist, int n, const float* z, const int64_t* idx, const float* old_logp, const float* adv,
                            float lo, float hi, float* surr, float* ent, float* logp, float* ratio, int sm_count, cudaStream_t stream);
cudaError_t launch_ppo_loss_grad(int64_t n_rows, int n_dist, int n, const float* z, const int64_t* idx, const float* adv, const float* ratio,
                                 float lo, float hi, const float* g_surr, const float* g_ent, float* dz, int sm_count, cudaStream_t stream);
// the recurrent actor's GRU and action layer for the update, forward and backward (evg_rppo_train.cu)
cudaError_t launch_rppo_train_forward(int64_t n_rows, int latent, int out_dim, const float* x, const float* h0, const void* wi_img,
                                      const void* wh_img, const void* w3_img, const float* bias, float* z, float* h, int sm_count,
                                      cudaStream_t stream);
cudaError_t launch_rppo_train_backward(int64_t n_rows, int latent, int out_dim, const float* x, const float* h0, const float* h,
                                       const void* wi_img, const void* wh_img, const void* wht_img, const float* bias, float* g,
                                       float* dgh, float* s, int sm_count, cudaStream_t stream);
// PPO's feed-forward networks for the update, forward and backward (evg_ppo_train.cu); net = EVG_PPO_TRAIN_*
cudaError_t launch_ppo_train_forward(int net, const void* obs, int64_t n_matches, int player, int in_dim, int latent, int out_dim,
                                     const void* w1_img, const void* w2_img, const void* w3_img, const float* bias, float* out, float* h1,
                                     float* h2, int sm_count, cudaStream_t stream, const WireSrc* wire);
cudaError_t launch_ppo_train_backward(int64_t n_rows, int latent, const void* w2t_img, const float* g2, const float* h1, const float* h2,
                                      float* dd2, float* dd1, int sm_count, cudaStream_t stream);
// the float32 length of a network's packed bias vector: b1 | b2, then the actor's or the critic's b3
inline int ppo_train_bias_floats(int net)
{
    return 2 * EVG_PPO_MAX_LATENT + (net == EVG_PPO_TRAIN_ACTOR ? EVG_PPO_OUT_PAD : net == EVG_PPO_TRAIN_CRITIC ? EVG_VALUE_OUT_PAD : 0);
}
// the policy kernels' opt-in to their dynamic shared memory, on the current device (the attribute is per device)
cudaError_t set_ppo_train_smem();
cudaError_t set_rppo_train_smem();
cudaError_t set_policy_mlp_smem();
cudaError_t set_policy_ppo_smem();
cudaError_t set_policy_rppo_smem();
cudaError_t set_policy_value_smem();
// weight images of the policy kernels and the critic from the float32 parameters (evg_policy_pack.cu); launch_pack_ppo
// packs the recurrent actor's GRU as well when w_ih is not null
cudaError_t launch_pack_mlp(int in_dim, const float* w1, const float* b1, const float* w2, const float* b2, int hidden, int out_dim,
                            void* w1_img, void* w2_img, cudaStream_t stream);
cudaError_t launch_pack_ppo(int in_dim, const float* w1, const float* b1, const float* w2, const float* b2, const float* w3,
                            const float* b3, const float* w_ih, const float* b_ih, const float* w_hh, const float* b_hh, int latent,
                            int out_dim, void* w1_img, void* w2_img, void* wi_img, void* wh_img, void* w3_img, float* bias,
                            cudaStream_t stream);
// the feed-forward networks' training images (evg_ppo_train_forward / _backward's); w3 null for the head
cudaError_t launch_pack_ppo_train(int net, int in_dim, const float* w1, const float* b1, const float* w2, const float* b2, const float* w3,
                                  const float* b3, int latent, int out_dim, void* w1_img, void* w2_img, void* w3_img, void* w2t_img,
                                  float* bias, cudaStream_t stream);
// the recurrent actor's training images (evg_rppo_train_forward / _backward's)
cudaError_t launch_pack_rppo_train(const float* w3, const float* b3, const float* w_ih, const float* b_ih, const float* w_hh,
                                   const float* b_hh, int latent, int out_dim, void* wi_img, void* wh_img, void* wht_img, void* w3_img,
                                   float* bias, cudaStream_t stream);
cudaError_t launch_pack_value(int in_dim, const float* w1, const float* b1, const float* w2, const float* b2, const float* w3,
                              const float* b3, int latent, void* w1_img, void* w2_img, void* w3_img, float* bias, cudaStream_t stream);
cudaError_t launch_obs_to_i16(const float* obs, int16_t* out, int64_t n_values, cudaStream_t stream);
cudaError_t launch_export(const Tables& t, const uint32_t* records, const double* health, int64_t first, int64_t count,
                          EvgEnvState* out, cudaStream_t stream);
cudaError_t launch_import(const Tables& t, uint32_t* records, double* health, int64_t first, int64_t count,
                          const EvgEnvState* in, unsigned* bad, cudaStream_t stream);
cudaError_t launch_agent_random(const Tables& t, const uint32_t* records, int8_t* actions, int player, int64_t n_envs,
                                cudaStream_t stream);
cudaError_t launch_decode_dqn(const float* q, int num_cols, int player, int8_t* actions, int64_t n_envs, int transposed, cudaStream_t stream);
cudaError_t launch_decode_indices(const int64_t* idx, int div, int mod, int player, int8_t* actions, int64_t n_envs, cudaStream_t stream);
cudaError_t launch_shape_reward(int mode, const float* reward, const uint8_t* done, const float* obs, int obs_len, float* out,
                                int64_t n_envs, cudaStream_t stream);
cudaError_t launch_agents(const Tables& t, const uint32_t* records, uint2* agent_state, int8_t* actions, int agent0, int agent1,
                          int64_t n_envs, cudaStream_t stream);
cudaError_t step_occupancy(const Tables& t, size_t smem, int* blocks_per_sm);
cudaError_t set_step_smem(size_t smem);
// thread-per-match step (evg_step_tpm.cu)
bool tpm_has_small(const Tables& t);
cudaError_t tpm_prepare(const Tables& t, int threads, size_t* smem_out, int* blocks_per_sm);
cudaError_t launch_step_tpm(const Tables& t, const StepArgs& a, int threads, size_t smem, int max_grid, cudaStream_t stream);

#ifdef __CUDACC__
// -DEVG_CHECKED (tools/build_variant.sh checked -DEVG_CHECKED): every data-dependent shared-memory index, health offset
// and match index of the step kernels is asserted in range — the project's own substitute for compute-sanitizer's
// memcheck on pools where the sanitizer is not available.  The GPU test-suite is run against that build
// (EVGSIM_LIB=build/libevgsim_checked.so; profiles/README.md).  Compiles to nothing in the product build.
#ifdef EVG_CHECKED
#include <cassert>
#define EVG_CHECK(cond) assert(cond)
#else
#define EVG_CHECK(cond) ((void)0)
#endif

// Map size of a step kernel: compile-time (NODES > 0, DemoMap's 11 for the instantiated fast paths) or read from the
// tables (0).  The record size is in 8-byte units, as in Tables::rec_words8.
template <int NODES>
struct Geo {
    const Tables& S;
    __device__ __forceinline__ explicit Geo(const Tables& s) : S(s) {}
    __device__ __forceinline__ int n_nodes() const { return NODES ? NODES : S.n_nodes; }
    __device__ __forceinline__ int nn() const { return n_nodes() + 1; }
    __device__ __forceinline__ int obs_len() const { return 1 + 4 * n_nodes() + 5 * EVG_NUM_GROUPS; }
    __device__ __forceinline__ int rec_words8() const { return NODES ? ((kRecNode0 + NODES) * 4 + 31) / 32 * 4 : S.rec_words8; }
};

// Entry f (< obs_len) of player p's observation vector from a wire row (evgsim.wire.expand): every dynamic entry is one
// field of one 32-bit word of the row — the turn and a node's control state are the low halves of words 0 and x (node id
// x in real numbering), a unit count or a group byte is one byte — and the rest is a constant of the map (oconst).
// wire_entry() says which word and how to read it; wire_value() reads it.  Only the group location of player 1 needs a
// table lookup on the row's data (p1_map, clamped into the table for rows the step did not write).
enum : uint32_t { kWireConst = 0, kWireU16, kWireS16, kWireByte, kWireLoc, kWireLocP1, kWireMoving };

__device__ __forceinline__ int wire_entry(const WireSrc& w, int p, int f, uint32_t& op, uint32_t& shift)
{
    const int n = w.n_nodes;
    shift = 0;
    if (f == 0) {
        op = kWireU16;
        return 0;
    }
    if (f <= 4 * n) {  // node slot k of the viewer: DEFENSE, OBSERVE, control state, the OTHER player's units
        const int k = (f - 1) >> 2, j = (f - 1) & 3;
        op = j < 2 ? kWireConst : j == 2 ? kWireS16 : kWireByte;
        shift = 8 * (3 - p);
        return p ? __ldg(w.p1_map + k + 1) : k + 1;
    }
    const int t = f - 1 - 4 * n, g = t / 5, j = t - 5 * g;  // group g: location, type, avg health, moving, units alive
    const int b = EVG_WIRE_NODE0 + 4 * n + 3 * (EVG_NUM_GROUPS * p + g) + (j == 2 ? 1 : j == 4 ? 2 : 0);
    op = j == 1 ? kWireConst : j == 0 ? (p ? kWireLocP1 : kWireLoc) : j == 3 ? kWireMoving : kWireByte;
    shift = 8 * (b & 3);
    return b >> 2;
}

__device__ __forceinline__ float wire_value(const WireSrc& w, int p, int f, uint32_t op, uint32_t shift, uint32_t word)
{
    const uint32_t byte = (word >> shift) & 0xFFu;
    switch (op) {
        case kWireU16: return (float)(word & 0xFFFFu);
        case kWireS16: return (float)(int16_t)(word & 0xFFFFu);
        case kWireByte: return (float)byte;
        case kWireLoc: return (float)(byte & 63u);
        case kWireLocP1: return (float)__ldg(w.p1_map + min(byte & 63u, (uint32_t)(kNN - 1)));
        case kWireMoving: return (float)(byte >> 6);
        default: return __ldg(w.oconst + p * w.obs_len + f);
    }
}

// Philox4x32-10 (Salmon et al., SC'11); same function as oracle/tape.py, oracle/evg_oracle.c.
__device__ __forceinline__ void philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0, uint32_t k1,
                                               uint32_t out[4])
{
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        if (r) { k0 += 0x9E3779B9u; k1 += 0xBB67AE85u; }
        const uint32_t h0 = __umulhi(0xD2511F53u, c0), l0 = 0xD2511F53u * c0;
        const uint32_t h1 = __umulhi(0xCD9E8D57u, c2), l1 = 0xCD9E8D57u * c2;
        c0 = h1 ^ c1 ^ k0; c1 = l1; c2 = h0 ^ c3 ^ k1; c3 = l0;
    }
    out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}

__device__ __forceinline__ void swap_nibbles(uint64_t& x, int i, int j)
{
    const uint64_t d = ((x >> (4 * i)) ^ (x >> (4 * j))) & 15ull;
    x ^= d << (4 * i) | d << (4 * j);
}

// random_actions agent (agents/State_Machine/random_actions.py:38-46) for maps of <= 15 nodes, all in
// registers: 7 distinct group ids of 12 and 7 distinct node ids, paired in draw order, as partial
// Fisher-Yates shuffles of nibble-packed permutations over 16 tape halves (2 Philox blocks, domain 1).
// rows[k] = gid | node << 8.  Same function as evo_agent_random in oracle/evg_oracle.c.
__device__ __forceinline__ void agent_random_rows(uint32_t env_global, uint32_t turn, uint32_t episode, int player, int n_nodes,
                                                  uint32_t seed_lo, uint32_t seed_hi, uint32_t rows[EVG_MAX_ACTIONS])
{
    uint32_t w[8];
    philox4x32_10(env_global, turn, (uint32_t)player, 1u | episode << 8, seed_lo, seed_hi, w);
    philox4x32_10(env_global, turn, (uint32_t)player | 1u << 8, 1u | episode << 8, seed_lo, seed_hi, w + 4);
    uint64_t gp = 0xBA9876543210ull;                 // nibble i = group i
    uint64_t np = 0xFEDCBA987654321ull;              // nibble i = node i + 1
#pragma unroll
    for (int k = 0; k < EVG_MAX_ACTIONS; ++k) {
        const uint32_t hg = (k & 1) ? w[k >> 1] >> 16 : w[k >> 1] & 0xFFFFu;             // half k
        const uint32_t hn = (k & 1) ? w[4 + (k >> 1)] >> 16 : w[4 + (k >> 1)] & 0xFFFFu;  // half 8 + k
        swap_nibbles(gp, k, k + (int)((hg * (uint32_t)(EVG_NUM_GROUPS - k)) >> 16));
        uint32_t node = 0;
        if (k < n_nodes) {
            swap_nibbles(np, k, k + (int)((hn * (uint32_t)(n_nodes - k)) >> 16));
            node = (uint32_t)(np >> (4 * k)) & 15u;
        }
        rows[k] = ((uint32_t)(gp >> (4 * k)) & 15u) | node << 8;
    }
}

// base_rushV1.get_action (agents/State_Machine/base_rush_v1.py:62-111) for player p.  w0_of(L) returns word 0 of group
// lane L's record (location [0:6), moving bit 21); st.x = {bit0 started, group_num [4:8), node_num [8:16)}, 0 = a fresh
// agent.  Same function as evo_agent_base_rush (oracle/evg_oracle.c), which is pinned to games of the reference's class.
template <typename W0>
__device__ __forceinline__ void agent_base_rush_rows(const Tables& T, W0 w0_of, uint2& st, int p, uint32_t rows[EVG_MAX_ACTIONS])
{
    const bool started = st.x & 1u;
    uint32_t gnum = started ? (st.x >> 4) & 15u : 1u, nnum = started ? (st.x >> 8) & 255u : 2u;
#pragma unroll
    for (int k = 0; k < EVG_MAX_ACTIONS; ++k) {
        rows[k] = 0;
        if (started) {  // the first call only blows the turn (:73-76)
            const uint32_t loc = w0_of(p * EVG_NUM_GROUPS + k) & W0_LOC_MASK;  // GROUP k's location (:86-88)
            const uint32_t own = p ? (uint32_t)T.p1_map[loc] : loc;
            if (own != T.base_own[p]) {
                rows[k] = gnum | nnum << 8;
                gnum = gnum + 1 == EVG_NUM_GROUPS ? 0u : gnum + 1;
                if (gnum == 0) nnum = nnum % (uint32_t)T.n_nodes + 1u;
            }
        }
    }
    st.x = 1u | gnum << 4 | nnum << 8;
}

// SwarmAgent.get_action (agents/State_Machine/swarm_agent.py:79-102) for player p; st.y = the agent's attack list as
// nibbles (0 = a fresh agent), shuffled in place every turn by numpy's Fisher-Yates on the tape (domain 2).
template <typename W0>
__device__ __forceinline__ void agent_swarm_rows(const Tables& T, W0 w0_of, uint2& st, uint32_t env_global, uint32_t turn, uint32_t episode,
                                                 int p, uint32_t rows[EVG_MAX_ACTIONS])
{
    uint32_t lst = st.y ? st.y : 0xBA875421u;  // ATTACK_LIST [1,2,4,5,7,8,10,11], :24
    uint32_t w[4];
    philox4x32_10(env_global, turn, (uint32_t)p, 2u | episode << 8, T.seed_lo, T.seed_hi, w);
#pragma unroll
    for (int k = 0; k < 7; ++k) {  // np.random.shuffle: i = 7..1, j uniform in [0, i]
        const int ii = 7 - k;
        const uint32_t h = (k & 1) ? w[k >> 1] >> 16 : w[k >> 1] & 0xFFFFu;
        const int j = (int)((h * (uint32_t)(ii + 1)) >> 16);
        const uint32_t d = ((lst >> (4 * ii)) ^ (lst >> (4 * j))) & 15u;
        lst ^= d << (4 * ii) | d << (4 * j);
    }
    st.y = lst;
#pragma unroll
    for (int k = 0; k < EVG_MAX_ACTIONS; ++k) rows[k] = 0u | 1u << 8;  // default rows [0, 1], :81-82
    int n = 0;
#pragma unroll
    for (int k = 0; k < 8; ++k) {
        const uint32_t x = (lst >> (4 * k)) & 15u;
        const uint32_t w0 = w0_of(p * EVG_NUM_GROUPS + (int)x);
        if (n < EVG_MAX_ACTIONS && !(w0 & W0_MOVING)) {
            const uint32_t loc = w0 & W0_LOC_MASK;
            const uint32_t own = p ? (uint32_t)T.p1_map[loc] : loc;
            const uint32_t row = x | (uint32_t)T.maxnb_own[p][own] << 8;
#pragma unroll
            for (int q = 0; q < EVG_MAX_ACTIONS; ++q)
                if (q == n) rows[q] = row;
            ++n;
        }
    }
}
#endif

}  // namespace evg

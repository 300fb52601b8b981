/*
 * evgsim.h — C ABI of libevgsim: the batched, GPU-resident Everglades turn step.
 *
 * This is the drop-in boundary for ONE path of jlehett/everglades-ai-wargame:
 *     EvergladesEnv.reset / EvergladesEnv.step
 *         gym-everglades/gym_everglades/envs/everglades_env.py:32-116   ("env.py")
 *     -> EvergladesGame.game_init / game_turn / board_state / player_state
 *         everglades-server/everglades_server/server.py:133-501          ("server.py")
 * for N matches in lockstep.  The reference has no FFI (it is pure Python); the binding a
 * maintainer would add is a ctypes stub — see INTEGRATION.md.
 *
 * Rules of the boundary
 *   - plain C types only; no torch / CUDA runtime types in any signature (`stream` is a
 *     cudaStream_t passed as void*, 0 = the legacy default stream);
 *   - the library NEVER allocates device memory: the caller asks evg_layout() for sizes,
 *     allocates (torch.empty / cudaMalloc) and binds raw device pointers with evg_bind();
 *   - every call is asynchronous on `stream`; nothing synchronises unless stated;
 *   - every entry point returns 0 on success or a negative EVG_E_* code; evg_last_error()
 *     returns a thread-local human-readable message for the last failure.
 *   - there is NO CPU fallback: without a CUDA device evg_create() fails with EVG_E_CUDA.
 */
#ifndef EVGSIM_H
#define EVGSIM_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define EVG_ABI_VERSION 1

/* compile-time maxima of the state layout */
#define EVG_MAX_NODES 32       /* node IDs are 1..n_nodes (DemoMap: 11) */
#define EVG_MAX_UNIT_TYPES 8   /* UnitDefinitions.json entries (reference: 3) */
#define EVG_NUM_GROUPS 12      /* groups per player, env.py:19 */
#define EVG_MAX_GROUP_UNITS 16 /* unit slots per group (reference loadout: 8, last group 12) */
#define EVG_MAX_ACTIONS 7      /* rows of an action array that count, server.py:227 */
#define EVG_NUM_PLAYERS 2

/* error codes */
#define EVG_OK 0
#define EVG_E_ARG -1    /* null pointer / out-of-range argument */
#define EVG_E_CONFIG -2 /* EvgConfig fails validation (see evg_last_error) */
#define EVG_E_CUDA -3   /* CUDA runtime error (no device, launch failure, ...) */
#define EVG_E_STATE -4  /* call sequence error, e.g. step before bind */

/* game status, server.py:284-289 */
#define EVG_STATUS_IN_PROGRESS 0
#define EVG_STATUS_TIME_EXPIRED 1
#define EVG_STATUS_BASE_CAPTURE 2
#define EVG_STATUS_ANNIHILATION 3

/* what evg_step does with a match whose status != 0 */
#define EVG_AUTORESET_OFF 0       /* keep stepping it, like the reference server does */
#define EVG_AUTORESET_TERMINAL 1  /* reset in place; obs of that step = terminal obs (reference-identical) */
#define EVG_AUTORESET_NEXT 2      /* reset in place; obs of that step = first obs of the new match */

/*
 * Static game description: DemoMap.json + UnitDefinitions.json + GameSetup.json semantics
 * (server.py:40-131 board_init/unitTypes_init; env.py:15-22,145-156 constants and loadout).
 * All per-node arrays are indexed by node ID (entry 0 unused).
 */
typedef struct EvgConfig {
    int32_t abi_version; /* = EVG_ABI_VERSION */
    int32_t n_nodes;
    int32_t n_unit_types;
    int32_t turn_limit;    /* GameSetup.json TurnLimit; hard-coded 150 at server.py:321 */
    int32_t capture_bonus; /* GameSetup.json CaptureBonus; hard-coded 1000 at server.py:304 */
    int32_t max_score;     /* reward normaliser MAX_SCORE = 3700, env.py:11 */
    int32_t auto_reset;    /* EVG_AUTORESET_* */
    int32_t reserved0;

    int32_t node_control_points[EVG_MAX_NODES + 1]; /* "ControlPoints" */
    double node_defense[EVG_MAX_NODES + 1];         /* "StructureDefense" */
    int8_t node_team_start[EVG_MAX_NODES + 1];      /* "TeamStart": -1, 0 or 1 */
    uint8_t node_has_defense[EVG_MAX_NODES + 1];    /* 'DEFENSE' in Resource: obs flag, server.py:442 */
    uint8_t node_has_observe[EVG_MAX_NODES + 1];    /* 'OBSERVE' in Resource: obs flag, server.py:443 */
    uint8_t node_has_defend[EVG_MAX_NODES + 1];     /* 'DEFEND' in Resource: combat bonus, server.py:595
                                                       (never true on DemoMap, whose maps say "DEFENSE") */
    /* edge_distance[a][b] = "Distance" of the FIRST connection of node a whose ConnectedID is b
       (server.py:246-250), 0 = not connected */
    uint8_t edge_distance[EVG_MAX_NODES + 1][EVG_MAX_NODES + 1];
    /* player 1's view of node ids (server.py:89); must be an involution with map[0] = 0 */
    uint8_t p1_node_map[EVG_MAX_NODES + 1];

    double unit_armor[EVG_MAX_UNIT_TYPES];    /* "Health" — used as armour, server.py:592 */
    int32_t unit_damage[EVG_MAX_UNIT_TYPES];  /* "Damage" */
    int32_t unit_speed[EVG_MAX_UNIT_TYPES];   /* "Speed" */
    int32_t unit_control[EVG_MAX_UNIT_TYPES]; /* "Control" */
    int32_t unit_cost[EVG_MAX_UNIT_TYPES];    /* "Cost" */

    /* loadout, env.py:145-156: type id = index in UnitDefinitions.json (server.py:128-129) */
    uint8_t group_type[EVG_NUM_PLAYERS][EVG_NUM_GROUPS];
    uint8_t group_size[EVG_NUM_PLAYERS][EVG_NUM_GROUPS]; /* 1..EVG_MAX_GROUP_UNITS */
} EvgConfig;

/* One group, as the reference keeps it (definitions.py:35-47 EvgGroup + :58-64 EvgUnit). */
typedef struct EvgGroupState {
    int16_t location;           /* node ID */
    int16_t travel_destination; /* node ID or -1 */
    int16_t distance_remaining;
    uint8_t ready;
    uint8_t moving;
    uint8_t destroyed;
    uint8_t count;       /* alive units */
    int32_t arrival;     /* list-order stamp: groups of one player at one node are listed by
                            ascending arrival (node.groups[pid], server.py:198,690-691);
                            canonical value: gid at reset, turn*16+gid on arrival */
    int32_t avg_health;  /* int(sum(health)/alive) as player_state reports it (server.py:491) */
} EvgGroupState;

/* One match, array-of-structs view used by evg_export_state / evg_import_state (parity tests,
 * checkpointing).  The resident device layout is different (see evg_layout, DESIGN.md §3). */
typedef struct EvgEnvState {
    int32_t turn;    /* current_turn, server.py:140,214 */
    int32_t episode; /* how many matches this slot has finished or been reset out of; keys the tape
                        so that successive matches of one slot differ (0 after evg_reset(NULL)) */
    int16_t control_state[EVG_MAX_NODES + 1]; /* node.controlState, definitions.py:17 */
    int8_t controlled_by[EVG_MAX_NODES + 1];  /* node.controlledBy, definitions.py:16 */
    int8_t pad1[5];
    EvgGroupState groups[EVG_NUM_PLAYERS][EVG_NUM_GROUPS];
    double health[EVG_NUM_PLAYERS][EVG_NUM_GROUPS][EVG_MAX_GROUP_UNITS]; /* unitHealth, definitions.py:62 */
} EvgEnvState;

/* Sizes of the device arrays the caller must allocate and bind (bytes, for n_envs matches). */
typedef struct EvgLayout {
    int64_t n_envs;
    int32_t obs_len;       /* per player: 1 + 4*n_nodes + 5*12 (105 on DemoMap), env.py:165-167 */
    int32_t record_bytes;  /* per match: packed group/node/turn record */
    int32_t health_slots;  /* per match: fp64 unit-health slots (both players, padded) */
    int32_t action_bytes;  /* per match: 2*7*2 int8 */
    int64_t records_bytes; /* = n_envs * record_bytes           (bind slot EVG_BIND_RECORDS) */
    int64_t health_bytes;  /* = n_envs * health_slots * 8       (bind slot EVG_BIND_HEALTH)  */
    int64_t stats_bytes;   /* episode statistics accumulators   (bind slot EVG_BIND_STATS)   */
    int64_t tables_bytes;  /* derived lookup tables, filled by evg_bind (bind slot EVG_BIND_TABLES) */
    int64_t agents_bytes;  /* scripted-agent state, 16 B per match (bind slot EVG_BIND_AGENTS)     */
} EvgLayout;

#define EVG_BIND_RECORDS 0
#define EVG_BIND_HEALTH 1
#define EVG_BIND_STATS 2
#define EVG_BIND_TABLES 3
#define EVG_BIND_AGENTS 4
#define EVG_BIND_COUNT 5

/* Episode statistics accumulated on the device by evg_step (matches that ended). */
typedef struct EvgEpisodeStats {
    int64_t episodes;
    int64_t wins[2]; /* by final score, the test callers use (evaluate.py:155-160) */
    int64_t ties;
    int64_t total_turns;     /* sum of episode lengths */
    int64_t total_score[2];  /* sum of final scores */
    int64_t status_count[4]; /* histogram of EVG_STATUS_* at episode end */
    int64_t env_turns;       /* all match-turns stepped since creation / last clear */
    int64_t fought_unit_slots; /* unit slots of the groups that took part in combat, summed over all match-turns
                                  stepped (finished matches or not): 16 B of fp64 health traffic each, the variable
                                  term of the step's algorithmic bytes (SURVEY.md 8d; server.py:516-566) */
} EvgEpisodeStats;

typedef struct EvgSim EvgSim; /* opaque */

/* Fill `cfg` with the reference's DemoMap.json / UnitDefinitions.json / GameSetup.json values
 * and the env.py:145-156 loadout (useful when no JSON parser is at hand). */
int evg_default_config(EvgConfig* cfg);

/* Validate `cfg` and create a simulator for `n_envs` matches on CUDA device `device`.
 * Match i has global id env_id_offset + i; the combat tape is keyed on (seed, global id,
 * turn, node, side, group, unit) so trajectories do not depend on how matches are sharded.
 * Replaces: EvergladesEnv.__init__ (env.py:15-30) + EvergladesGame.__init__ (server.py:14-38). */
int evg_create(const EvgConfig* cfg, int64_t n_envs, uint64_t seed, int64_t env_id_offset, int device,
               EvgSim** out);
int evg_destroy(EvgSim* sim);

int evg_layout(const EvgSim* sim, EvgLayout* out);
/* Bind caller-owned device arrays (index = EVG_BIND_*). Must precede reset/step.  Uploads the derived
 * tables into slot EVG_BIND_TABLES (synchronous copy). */
int evg_bind(EvgSim* sim, void* const* device_ptrs, int32_t n_ptrs);

/* Put matches into the post-game_init state (server.py:133-209, env.py:75-116) and write their
 * observations.  d_mask: n_envs bytes, non-zero = reset this match; NULL = all.
 * d_obs: float32 [n_envs][2][obs_len] or NULL.  Also zeroes the statistics when d_mask is NULL. */
int evg_reset(EvgSim* sim, const uint8_t* d_mask, float* d_obs, void* stream);

/* One game turn for every match (env.py:32-73 step -> server.py:211-279 game_turn, 281-348
 * game_end, 382-501 observations).
 *   d_actions: int8 [n_envs][2][7][2] = (group id, node id in the acting player's numbering);
 *              rows with group/node out of range are ignored (the reference raises IndexError).
 *   d_obs:     float32 [n_envs][2][obs_len]   (reference: float64 arrays of integers)
 *   d_reward:  float32 [n_envs][2]            (env.py:37-60)
 *   d_done:    uint8   [n_envs]               (status != 0)
 *   d_status / d_scores: optional (may be NULL): uint8 [n_envs], int32 [n_envs][2]. */
int evg_step(EvgSim* sim, const int8_t* d_actions, float* d_obs, float* d_reward, uint8_t* d_done,
             uint8_t* d_status, int32_t* d_scores, void* stream);

/*
 * Observation formats.  EVG_OBS_F32 is the reference's vector (env.py:158-171) as float32.  The other two carry the SAME
 * information losslessly in fewer bytes, for consumers behind a narrow link (the host over PCIe: evg_step_host_fmt):
 *
 *   EVG_OBS_I16   int16 [n_envs][2][obs_len], same layout as the float32 vector (every entry is an integer in
 *                 [-32768, 32767]: turn <= 65535 is checked at create time against this format on use).
 *   EVG_OBS_WIRE  one packed row per match, evg_obs_row_bytes() bytes = round_up(4 + 4*n_nodes + 72 + 8, 16)
 *                 (128 on DemoMap: one cache line), little endian:
 *        [0:2)  turn uint16 (obs[0], server.py:432)    [2] done uint8    [3] status uint8 (EVG_STATUS_*)
 *        [4 + 4*(x-1) ...) for node id x = 1..n_nodes: controlState int16 (raw sign, server.py:444), units of player 0's
 *                 groups listed at the node uint8, units of player 1's groups uint8 (server.py:446-449; a viewer's
 *                 "opponent units" entry is the other player's byte)
 *        [G = 4 + 4*n_nodes + 3*(12*p + g) ...) group g of player p: byte 0 = location in REAL node numbering [0:6) |
 *                 moving << 6 (server.py:477,489), byte 1 = avg health (server.py:491), byte 2 = units alive (:480)
 *        [G + 72 : G + 80)  the step's rewards, float32[2] (env.py:37-60)
 *        zero padding to the row size.
 *   What the float32 vector holds besides is static: the nodes' DEFENSE/OBSERVE flags, the groups' unit types, and
 *   player 1's node numbering (server.py:437-439, 476) — a function of EvgConfig alone.  evgsim.wire.expand() /
 *   INTEGRATION.md give the expansion; tests/test_gpu_wire.py checks expand(wire) == float32 observations bit for bit.
 */
#define EVG_OBS_F32 0
#define EVG_OBS_I16 1
#define EVG_OBS_WIRE 2
#define EVG_WIRE_NODE0 4 /* byte offset of node 1's entry in a wire row */

/* where a player's action rows come from in evg_step_agents */
#define EVG_AGENT_EXTERNAL 0 /* the caller's rows in d_actions */
#define EVG_AGENT_RANDOM 1   /* on-device random_actions agent (agents/State_Machine/random_actions.py:38-46) */
#define EVG_AGENT_BASE_RUSH 2 /* base_rushV1 (agents/State_Machine/base_rush_v1.py:62-111); keeps its counters per match */
#define EVG_AGENT_SWARM 3    /* SwarmAgent (agents/State_Machine/swarm_agent.py:79-102); keeps its attack list per match */

/* evg_step with scripted opponents fused into the step kernel: rows of players whose agent is not
 * EVG_AGENT_EXTERNAL are generated on the device (and written to d_actions if it is non-NULL); rows of
 * EXTERNAL players are read from d_actions (then it must be non-NULL).  With both players scripted a
 * whole self-play turn is ONE kernel launch and no action buffer is touched. */
int evg_step_agents(EvgSim* sim, int32_t agent_p0, int32_t agent_p1, int8_t* d_actions, float* d_obs, float* d_reward,
                    uint8_t* d_done, uint8_t* d_status, int32_t* d_scores, void* stream);

/* `n_turns` turns of fully scripted self-play (both agents != EVG_AGENT_EXTERNAL) with the results of evg_step_agents
 * called n_turns times: the output arrays hold the last turn's values, statistics accumulate, d_actions (required) is
 * scratch for the generated rows.  ALL the turns run in ONE launch: small batches (evg_step_kernel_kind() == 0) on the
 * multi-turn warp-per-match kernel (a warp keeps its match for the whole rollout), larger ones on the thread-per-match
 * kernel, whose CTAs keep each batch in shared memory for all n_turns — a turn costs neither a launch nor an action-buffer
 * pass, and only the last one writes observations and records.  (Only EVG_AGENT_RANDOM on maps of more than 15 nodes
 * runs turn by turn: agent kernel + step.) */
int evg_rollout(EvgSim* sim, int32_t agent_p0, int32_t agent_p1, int32_t n_turns, int8_t* d_actions, float* d_obs, float* d_reward,
                uint8_t* d_done, uint8_t* d_status, int32_t* d_scores, void* stream);

/* Same turn through HOST buffers: H2D of the actions, the step, D2H of obs/reward/done, ordered after
 * what `stream` holds and complete when `stream` is (pinned host memory makes them truly asynchronous).
 * The device staging arrays are the caller's (same shapes as evg_step).  From 65,536 matches on, the
 * thread-per-match kernel runs the batch as EVG_HOST_CHUNKS (environment, default 16) sub-range launches on
 * two streams the library creates for this, so that the PCIe-bound D2H of one chunk hides the H2D and
 * the kernel of the next; results are those of evg_step. */
int evg_step_host(EvgSim* sim, const int8_t* h_actions, float* h_obs, float* h_reward, uint8_t* h_done,
                  int8_t* d_actions, float* d_obs, float* d_reward, uint8_t* d_done, void* stream);

/* Bytes per match of an observation format (0 for an unknown format or NULL sim). */
int evg_obs_row_bytes(const EvgSim* sim, int32_t format);

/* evg_reset / evg_step / evg_step_host with the observation output in `format` (EVG_OBS_*); with EVG_OBS_F32 they ARE
 * those calls.  d_rows / h_rows: n_envs rows of evg_obs_row_bytes(sim, format).  EVG_OBS_WIRE rows are written by the
 * step kernel itself (no float32 observations are produced at all); EVG_OBS_I16 needs a caller-provided float32
 * scratch d_obs_f32 [n_envs][2][obs_len] that the step writes and a conversion kernel narrows.  In evg_step_host_fmt
 * h_reward / h_done may be NULL with EVG_OBS_WIRE (the row carries them). */
int evg_reset_fmt(EvgSim* sim, int32_t format, const uint8_t* d_mask, void* d_rows, float* d_obs_f32, void* stream);
int evg_step_fmt(EvgSim* sim, int32_t format, const int8_t* d_actions, void* d_rows, float* d_obs_f32, float* d_reward,
                 uint8_t* d_done, uint8_t* d_status, int32_t* d_scores, void* stream);
int evg_step_host_fmt(EvgSim* sim, int32_t format, const int8_t* h_actions, void* h_rows, float* h_reward, uint8_t* h_done,
                      int8_t* d_actions, void* d_rows, float* d_obs_f32, float* d_reward, uint8_t* d_done, void* stream);

/* Array-of-structs snapshot <-> resident layout, matches [first, first+count).  d_states is a
 * DEVICE array of EvgEnvState (the caller copies it to/from the host). */
int evg_export_state(EvgSim* sim, int64_t first, int64_t count, EvgEnvState* d_states, void* stream);
/* Import validates what it is given: a location outside 1..n_nodes, a travel_destination above n_nodes, a
 * distance_remaining outside 0..255, |control_state| above the node's ControlPoints or a controlled_by outside -1..1 is
 * forced into range (these fields index tables in the step kernels) and the call returns EVG_E_ARG after importing the
 * rest.  Synchronises `stream`. */
int evg_import_state(EvgSim* sim, int64_t first, int64_t count, const EvgEnvState* d_states, void* stream);

/* Copy the statistics accumulators to the host (synchronises `stream`). */
int evg_episode_stats(EvgSim* sim, EvgEpisodeStats* host_out, void* stream);

/* On-device scripted opponents (agents/State_Machine, Python files), writing int8 [n_envs][2][7][2]
 * action rows for `player` (0, 1, or -1 = both).  See DESIGN.md §7 for their tape. */
int evg_agent_random(EvgSim* sim, int8_t* d_actions, int32_t player, void* stream);

/* Action rows of the scripted agents for both players (EVG_AGENT_EXTERNAL players are left untouched) into
 * int8 [n_envs][2][7][2].  base_rushV1 / SwarmAgent carry per-match state across turns and matches (like the
 * reference's agent objects); evg_reset(sim, NULL, ...) makes all of them fresh agents again. */
int evg_agents(EvgSim* sim, int32_t agent_p0, int32_t agent_p1, int8_t* d_actions, void* stream);

/* Policy-in-the-loop glue: decode network outputs into action rows on the device (player: 0, 1, or -1 = both;
 * inputs are then [n_envs][2][...], else [n_envs][...]).
 *   evg_decode_dqn:     float32 Q-values [..][12 * num_cols] -> rows, exactly as DQNAgent.filter_actions does
 *                       (agents/DQN/DQNAgent.py:161-197; greedy insertion, node = 0-based column index).
 *   evg_decode_indices: int64 flat indices [..][7] -> rows (idx / div, idx % mod); PPOAgent.get_action uses
 *                       div 12, mod 11 (agents/PPO/PPOAgent.py:122-127), DQN's replay encoding div 11, mod 11. */
int evg_decode_dqn(EvgSim* sim, const float* d_q, int32_t num_cols, int32_t player, int8_t* d_actions, void* stream);
/* the same with d_q optionally transposed: [12 * num_cols][rows], rows = n_envs * (player < 0 ? 2 : 1) */
int evg_decode_dqn_layout(EvgSim* sim, const float* d_q, int32_t num_cols, int32_t player, int32_t q_transposed, int8_t* d_actions, void* stream);
int evg_decode_indices(EvgSim* sim, const int64_t* d_idx, int32_t div, int32_t mod, int32_t player, int8_t* d_actions,
                       void* stream);

/* Policy-in-the-loop forward, fused on the tensor cores (tcgen05 + TMEM; csrc/evg_policy_mlp.cu):
 *     d_q[rows][out_dim] = Linear(hidden, out_dim)(relu(Linear(obs_len, hidden)(d_obs[rows][obs_len])))
 * — the reference's DQN network, agents/DQN/QNetwork.py:37,42 (105 -> 528 -> 132) — for the observation rows the step
 * has just written (rows = n_envs * 2 for both players), bf16 operands with fp32 accumulation; the hidden activations stay
 * on the SM.  Weights are passed as IMAGES in the kernel's shared-memory operand layout (bf16, K-major, 128-byte swizzle),
 * cut into chunks of EVG_MLP_CHUNK hidden units, with the biases inside (homogeneous coordinates): input feature obs_len
 * is the constant 1, hidden unit `hidden` is wired to relu(1 * 1) = 1.  With W1' = [W1 | b1] plus that unit's row, and
 * W2' = [W2 | b2], for chunk c (ceil((hidden + 1) / CHUNK) chunks):
 *     d_w1_img + c * (EVG_MLP_IN_PAD / 64) * EVG_MLP_CHUNK * 128 bytes:  W1'[c*CHUNK + n][k], n < CHUNK, k < IN_PAD
 *     d_w2_img + c * (EVG_MLP_CHUNK / 64) * EVG_MLP_OUT_PAD * 128 bytes: W2'[o][c*CHUNK + k], o < OUT_PAD, k < CHUNK
 * element (row r, column k) of a [R x K] block at byte (k/64)*R*128 + r*128 + ((((k%64)/8) ^ (r%8)) * 16) + (k%8)*2, zero
 * padded.  evgsim.policy.pack_mlp builds them from a torch module.  q_transposed != 0 writes d_q as [out_dim][rows]
 * instead (each output's values for all rows contiguous): the layout evg_decode_dqn_layout reads coalesced. */
#define EVG_MLP_IN_PAD 128
#define EVG_MLP_CHUNK 192
#define EVG_MLP_OUT_PAD 144
int evg_policy_mlp(EvgSim* sim, const float* d_obs, int64_t rows, const void* d_w1_img, const void* d_w2_img, int32_t hidden, int32_t out_dim,
                   float* d_q, int32_t q_transposed, void* stream);

/* PPO's feed-forward actor with the action sampling fused behind it, on the tensor cores (csrc/evg_policy_ppo.cu):
 *     probs = Softmax(Tanh(Linear(latent, out_dim)(Tanh(Linear(latent, latent)(Tanh(Linear(obs_len, latent)(obs)))))))
 * — agents/PPO/ActorCritic.py:33-50 without the GRU — for the rows of `player` (0, 1, or -1 = both) of the observation
 * tensor d_obs float32 [n_envs][2][obs_len], then PPOAgent.get_action (agents/PPO/PPOAgent.py:122-127): 7 distinct flat
 * indices drawn without replacement, written as action rows (idx / div, idx % mod) into d_actions int8 [n_envs][2][7][2]
 * (only `player`'s rows; PPO's unravel is div 12, mod 11).  bf16 operands, fp32 accumulation, biases added in fp32.
 * The draws are keyed on the tape (DESIGN.md section 7, domain 3): (seed, global match id, turn and episode of the match's
 * current state, player) — independent of batch size, sharding and call order.
 *   d_idx (optional):   int64 [n_envs][2][7] (player -1) or [n_envs][7], the drawn indices in draw order.
 *   d_probs (optional): float32 [n_envs][2][out_dim] or [n_envs][out_dim], the probabilities the draws were made from.
 *   (evg_policy_ppo_logp adds d_logp, each draw's log-probability; below.)
 * Weights are IMAGES in the kernel's shared-memory operand layout (bf16, K-major, 128-byte swizzle, zero padded, 16-byte
 * aligned).  With Lp = latent rounded up to 16 and Ka = latent rounded up to 64:
 *     d_w1_img: W1[n][k] as an [Lp x EVG_PPO_IN_PAD] block,  (EVG_PPO_IN_PAD / 64) * Lp * 128 bytes
 *     d_w2_img: W2[n][k] as an [Lp x Ka] block,              (Ka / 64) * Lp * 128 bytes
 *     d_w3_img: W3[o][k] as an [EVG_PPO_OUT_PAD x Ka] block, (Ka / 64) * EVG_PPO_OUT_PAD * 128 bytes
 * element (row r, column k) of an [R x K] block at byte (k/64)*R*128 + r*128 + ((((k%64)/8) ^ (r%8)) * 16) + (k%8)*2.
 *     d_bias: float32 [2 * EVG_PPO_MAX_LATENT + EVG_PPO_OUT_PAD] = b1 at 0, b2 at EVG_PPO_MAX_LATENT, b3 at
 *             2 * EVG_PPO_MAX_LATENT, zero padded.
 * evgsim.policy.pack_ppo builds them from a torch module.  1 <= latent <= EVG_PPO_MAX_LATENT, 7 <= out_dim <= EVG_PPO_OUT_PAD,
 * obs_len < EVG_PPO_IN_PAD. */
#define EVG_PPO_IN_PAD 128
#define EVG_PPO_MAX_LATENT 256
#define EVG_PPO_OUT_PAD 144
int evg_policy_ppo(EvgSim* sim, const float* d_obs, int32_t player, const void* d_w1_img, const void* d_w2_img, const void* d_w3_img,
                   const float* d_bias, int32_t latent, int32_t out_dim, int32_t div, int32_t mod, int8_t* d_actions, int64_t* d_idx,
                   float* d_probs, void* stream);

/* PPO's recurrent actor with its draws fused behind it, on the tensor cores (csrc/evg_policy_rppo.cu): the actor of
 * agents/PPO/ActorCritic.py:33-60 with use_recurrent (act, :79-105), for the rows of `player` (0, 1, or -1 = both) of
 * d_obs float32 [n_envs][2][obs_len], with its GRU state carried in d_hidden float32 [rows][latent] (rows = n_envs * 2
 * for player -1, row 2 m + p; n_envs for one player), read and written back:
 *     h = 0 if the match's resident record is at turn 0 (a reset, or an automatic reset under EVG_AUTORESET_TERMINAL /
 *         _NEXT; under EVG_AUTORESET_OFF a finished match keeps its state until it is reset)
 *     x = tanh(W2 tanh(W1 obs + b1) + b2)
 *     for k = 0..6: one step of torch.nn.GRU(latent, latent) with input x (gates r, z, n in weight_ih_l0 / weight_hh_l0's
 *         order: r = sigmoid(W_ir x + b_ir + W_hr h + b_hr), z likewise, n = tanh(W_in x + b_in + r * (W_hn h + b_hn)),
 *         h = (1 - z) * n + z * h), probs_k = softmax(tanh(W3 h + b3)), idx_k = one draw from probs_k, action row k =
 *         (idx_k / div, idx_k % mod) into d_actions int8 [n_envs][2][7][2] (only `player`'s rows).
 * bf16 operands (observations, weights, x, and h as an MMA operand), fp32 accumulation; biases, gate arithmetic and the
 * state h stay fp32.  Draw k uses uniform u_k of evg_policy_ppo's tape block pair (domain 3), one draw with replacement:
 * the first j whose ascending fp32 prefix sum of probs_k exceeds u_k times their ascending sum (none: the last j).
 *   d_idx (optional):   int64 [rows][7], the drawn indices.
 *   d_probs (optional): float32 [rows][7][out_dim], the distributions the draws were made from.
 *   (evg_policy_rppo_logp adds d_logp, each draw's log-probability, and d_hidden_in, the starting state; below.)
 * Images as for evg_policy_ppo (Lp = latent rounded up to 16, Ka = latent rounded up to 64): d_w1_img, d_w2_img,
 * d_w3_img exactly as there, and
 *     d_wi_img: weight_ih_l0 as three [Lp x Ka] blocks, gate g (r, z, n) at g * (Ka / 64) * Lp * 128 bytes
 *     d_wh_img: weight_hh_l0 likewise
 *     d_bias: float32 [2 * EVG_PPO_MAX_LATENT + EVG_PPO_OUT_PAD + 6 * EVG_PPO_MAX_LATENT] = b1, b2, b3 as for
 *             evg_policy_ppo, then bias_ih_l0 gate g at 2 * EVG_PPO_MAX_LATENT + EVG_PPO_OUT_PAD + g * EVG_PPO_MAX_LATENT
 *             and bias_hh_l0 gate g 3 * EVG_PPO_MAX_LATENT further, zero padded.
 * evgsim.policy.pack_rppo builds them.  1 <= latent <= EVG_PPO_MAX_LATENT, 7 <= out_dim <= EVG_PPO_OUT_PAD. */
int evg_policy_rppo(EvgSim* sim, const float* d_obs, int32_t player, const void* d_w1_img, const void* d_w2_img, const void* d_wi_img,
                    const void* d_wh_img, const void* d_w3_img, const float* d_bias, int32_t latent, int32_t out_dim, int32_t div, int32_t mod,
                    float* d_hidden, int8_t* d_actions, int64_t* d_idx, float* d_probs, void* stream);

/* The three policy calls above with the observations in `format` (EVG_OBS_*); with EVG_OBS_F32 they ARE those calls.
 * EVG_OBS_WIRE: d_obs holds wire rows (evg_obs_row_bytes(sim, EVG_OBS_WIRE) bytes each, 16-byte aligned) — the rows
 * evg_step_fmt wrote, or any rows of the same map (a replay minibatch) — and the kernels stage from them exactly the
 * bf16 operands they stage from the float32 vector evg_wire_expand would write, so every output is bit for bit that of
 * the float32 call on the expanded rows.  The actors read n_envs rows (match m's row is row m); evg_policy_mlp_fmt reads
 * rows / 2 of them (observation row i = player i % 2 of wire row i / 2; rows must be even).  Needs evg_bind (the rows
 * expand through the bound tables).  EVG_OBS_I16 and unknown formats return EVG_E_ARG. */
int evg_policy_mlp_fmt(EvgSim* sim, int32_t format, const void* d_obs, int64_t rows, const void* d_w1_img, const void* d_w2_img, int32_t hidden,
                       int32_t out_dim, float* d_q, int32_t q_transposed, void* stream);
int evg_policy_ppo_fmt(EvgSim* sim, int32_t format, const void* d_obs, int32_t player, const void* d_w1_img, const void* d_w2_img,
                       const void* d_w3_img, const float* d_bias, int32_t latent, int32_t out_dim, int32_t div, int32_t mod, int8_t* d_actions,
                       int64_t* d_idx, float* d_probs, void* stream);
int evg_policy_rppo_fmt(EvgSim* sim, int32_t format, const void* d_obs, int32_t player, const void* d_w1_img, const void* d_w2_img,
                        const void* d_wi_img, const void* d_wh_img, const void* d_w3_img, const float* d_bias, int32_t latent, int32_t out_dim,
                        int32_t div, int32_t mod, float* d_hidden, int8_t* d_actions, int64_t* d_idx, float* d_probs, void* stream);

/* The two actors of evg_policy_ppo_fmt / evg_policy_rppo_fmt (which are these calls with the new pointers NULL) with what
 * a PPO update needs of the behaviour policy, written by the same launch.  Every other output is bit for bit the same
 * whether these are asked for or not.
 *   d_logp (optional): float32 [rows][7] like d_idx ([n_envs][2][7] for player -1, [n_envs][7] for one player): the
 *       log-probability of each draw, logf(p_j / T_k) in fp32 (accurate logf), in [-7, 0] (every probability is at least
 *       1 / (1 + 143 e^2)).  j is the drawn index, p_j its fp32 probability (the value d_probs holds).
 *       evg_policy_ppo_logp: T_k is the sampler's own fp32 sum, in ascending j, of the probabilities not chosen before
 *       draw k (T_0 sums all of them) — the normaliser the draw used, also when no j was found through rounding and the
 *       largest not-chosen j was taken.  Summed over k: the log-probability of the ordered 7-tuple under sequential
 *       sampling without replacement.
 *       evg_policy_rppo_logp: T_k is the fp32 ascending sum of probs_k; on the path where no j is found, j = out_dim - 1.
 *   d_hidden_in (evg_policy_rppo_logp, optional): float32 [rows][latent] like d_hidden: the state each row's GRU started
 *       from in this call, +0.0 for a row whose match record is at turn 0, otherwise what d_hidden held.  It must not
 *       overlap d_hidden (EVG_E_ARG). */
int evg_policy_ppo_logp(EvgSim* sim, int32_t format, const void* d_obs, int32_t player, const void* d_w1_img, const void* d_w2_img,
                        const void* d_w3_img, const float* d_bias, int32_t latent, int32_t out_dim, int32_t div, int32_t mod,
                        int8_t* d_actions, int64_t* d_idx, float* d_probs, float* d_logp, void* stream);
int evg_policy_rppo_logp(EvgSim* sim, int32_t format, const void* d_obs, int32_t player, const void* d_w1_img, const void* d_w2_img,
                         const void* d_wi_img, const void* d_wh_img, const void* d_w3_img, const float* d_bias, int32_t latent,
                         int32_t out_dim, int32_t div, int32_t mod, float* d_hidden, float* d_hidden_in, int8_t* d_actions,
                         int64_t* d_idx, float* d_probs, float* d_logp, void* stream);

/* PPO's critic on the tensor cores (csrc/evg_policy_value.cu): the state value
 *     v = Linear(latent, 1)(Tanh(Linear(latent, latent)(Tanh(Linear(obs_len, latent)(obs)))))
 * — the value_layer of agents/PPO/ActorCritic.py — of n_matches matches' observations, for the rows of `player`
 * (0, 1, or -1 = both).  n_matches is the caller's, not n_envs: the env's current observations, or a whole stored rollout
 * ([T * N] rows flattened) in one call; 0 is a no-op.  Row i is (match i / 2, player i % 2) for player -1, else
 * (match i, player).
 *   format EVG_OBS_F32: d_obs float32 [n_matches][2][obs_len] (4-byte aligned).
 *   format EVG_OBS_WIRE: d_obs wire rows [n_matches][evg_obs_row_bytes(sim, EVG_OBS_WIRE)] (16-byte aligned, needs
 *       evg_bind), values bit for bit those of the float32 call on the expanded rows, as for evg_policy_ppo_fmt.
 *   EVG_OBS_I16 and unknown formats return EVG_E_ARG.
 *   d_value: float32 [n_matches][2] (player -1) or [n_matches].
 * bf16 operands (observations, W1, W2, w3, both hidden activations), fp32 accumulation, b1, b2, b3 added in fp32, no tanh
 * after the last layer.  Images as for evg_policy_ppo (Lp = latent rounded up to 16, Ka = latent rounded up to 64):
 *     d_w1_img: W1[n][k] as an [Lp x EVG_PPO_IN_PAD] block, exactly as evg_policy_ppo's
 *     d_w2_img: W2[n][k] as an [Lp x Ka] block, exactly as evg_policy_ppo's
 *     d_w3_img: w3 as an [EVG_VALUE_OUT_PAD x Ka] block: row 0 = w3[k], the other rows zero,
 *               (Ka / 64) * EVG_VALUE_OUT_PAD * 128 bytes
 *     d_bias: float32 [2 * EVG_PPO_MAX_LATENT + EVG_VALUE_OUT_PAD] = b1 at 0, b2 at EVG_PPO_MAX_LATENT, b3 at
 *             2 * EVG_PPO_MAX_LATENT, zero padded.
 * Images and d_bias 16-byte aligned.  evgsim.policy.pack_value builds them on the host, evg_pack_value on the device.
 * EVG_E_ARG for latent outside 1..EVG_PPO_MAX_LATENT, obs_len >= EVG_PPO_IN_PAD, a negative n_matches, a player outside
 * -1..1 and NULL pointers. */
#define EVG_VALUE_OUT_PAD 16
int evg_policy_value(EvgSim* sim, int32_t format, const void* d_obs, int64_t n_matches, int32_t player, const void* d_w1_img,
                     const void* d_w2_img, const void* d_w3_img, const float* d_bias, int32_t latent, float* d_value, void* stream);

/* Wire rows -> the float32 observation vector on the device (csrc/evg_wire_expand.cu), bit for bit what the step writes
 * in EVG_OBS_F32 and what evgsim.wire.expand computes on the host; for training consumers that store the rows (a replay or
 * rollout memory: 128 bytes per match on DemoMap against 840) and expand a sampled minibatch.
 *   d_rows:   n_rows wire rows of this simulator's map (16-byte aligned).
 *   d_index:  int64 [n_out]: output row i expands source row d_index[i] (duplicates and any order allowed); NULL: output
 *             row i expands row i, and n_out must equal n_rows.  An index outside [0, n_rows) never faults: that output
 *             row is all zeros, its reward 0 and its done flag 0.
 *   player:   -1: d_obs float32 [n_out][2][obs_len]; 0 or 1: d_obs float32 [n_out][obs_len], that player's vector only.
 *   d_reward (optional): float32 [n_out][2];  d_done (optional): uint8 [n_out].
 * d_obs 16-byte aligned.  The constant entries (node flags, unit types) and player 1's node numbering come from the bound
 * tables (needs evg_bind).  A row the step did not write expands to unspecified values, without a fault. */
int evg_wire_expand(EvgSim* sim, const void* d_rows, int64_t n_rows, const int64_t* d_index, int64_t n_out, int32_t player, float* d_obs,
                    float* d_reward, uint8_t* d_done, void* stream);

/* PPO's advantages and returns, GAE(lambda), of a stored rollout of T = n_turns >= 1 turns of M = n_matches matches
 * (csrc/evg_gae.cu; agents/PPO/PPOAgent.py:190-218).  A column is a (match, player): both players for player -1, that
 * one for 0 or 1.
 *   d_values: float32 [T+1][M][2] (player -1) or [T+1][M]: V of the states the actor read at turns 0..T, i.e.
 *             evg_policy_value on the T+1 stored wire rows; row T is the bootstrap state.
 *   The reward and done flag of turn t < T come from
 *     d_reward float32 [T][M][2] (both players' rewards, whatever `player` is) and d_done uint8 [T][M] when given, and
 *     otherwise from d_rows, wire rows [T+1][M][evg_obs_row_bytes(sim, EVG_OBS_WIRE)] as the step wrote them: row t+1
 *     holds turn t's rewards and done flag (row 0's are not read).  d_rows is needed when either of the two is NULL;
 *     rows with the caller's own (e.g. shaped) rewards take d_reward and the rows' done flags.
 *   d_adv, d_ret: float32 [T][M][2] or [T][M].
 * In float32, each operation rounded on its own (no fused multiply-add), backward from A_T = 0, gl = fl(gamma * lam):
 *     nv = d_t ? 0 : V_{t+1},   na = d_t ? 0 : A_{t+1}
 *     delta_t = fl(fl(r_t + fl(gamma * nv)) - V_t),   A_t = fl(delta_t + fl(gl * na)),   R_t = fl(A_t + V_t)
 * (0 is selected rather than multiplied by 1 - d, so a non-finite value past a done flag does not leak in).
 * The done flag cuts both the bootstrap and the trace, whatever ended the match: reaching the turn limit
 * (EVG_STATUS_TIME_EXPIRED) is a terminal of the game, with its score and reward, not a truncation.  Under
 * EVG_AUTORESET_TERMINAL / _NEXT the values are those of the rows the actor read, the terminal observation that _TERMINAL
 * shows to the next match's first turn included.  Under EVG_AUTORESET_OFF the pass takes each row's done flag as the step
 * wrote it.  A finished match that keeps being stepped is still simulated and its end conditions are evaluated again every
 * turn: done is 1 on every turn from the turn limit on, and on a turn where a capture or annihilation holds.  Each such
 * turn is then a one-turn episode, A_t = fl(r_t - V_t); a turn between them (a base taken back) traces into the next one.
 * None of them is a turn of a real match: masking them is the caller's.
 * One launch on `stream`, no allocation, no synchronisation.  EVG_E_ARG for n_turns < 1, n_matches outside 1..2^31-1, a
 * player outside -1..1, NULL values / adv / ret, no rows while d_reward or d_done is NULL, rows not 16-byte aligned,
 * values / adv / ret / reward not 8-byte aligned for player -1 (4-byte otherwise), and gamma or lam outside [0, 1] or NaN. */
int evg_gae(EvgSim* sim, int32_t n_turns, int64_t n_matches, int32_t player, const void* d_rows, const float* d_reward, const uint8_t* d_done,
            const float* d_values, float gamma, float lam, float* d_adv, float* d_ret, void* stream);

/* PPO's policy loss for B = n_rows stored rows, from the output of the actor's last Linear (before its Tanh and Softmax),
 * and its gradient (csrc/evg_ppo_loss.cu; DESIGN.md §4.12).  K = n_dist, n = n_actions (7..256, 132 on DemoMap):
 *   d_z       float32 [B][K][n]. K = 1: the feed-forward actor, one distribution, 7 draws without replacement
 *             (evg_policy_ppo_logp).  K = 7: the recurrent actor, distribution k serves draw k, with replacement
 *             (evg_policy_rppo_logp).
 *   d_idx     int64 [B][7], the draws as d_idx of those calls stored them;  d_old_logp float32 [B][7], their d_logp;
 *   d_adv     float32 [B], the row's advantage A;  clip: epsilon in [0, 1).
 * Per row, in float32 (accurate tanhf / expf / logf, no fast math):
 *   y = tanh(z),  S_k = sum_i exp(y_k,i) (no max subtraction: y lies in [-1, 1]),  p_k,i = exp(y_k,i) / S_k,
 *   log p_k,i = y_k,i - log S_k,  H_k = -sum_i p_k,i log p_k,i
 *   K = 1:  T_k = sum of p_i over the i not in idx[0..k-1];   K = 7:  T_k = sum_i p_k,i (the sampler's normaliser)
 *   logp_k = log p_{k or 0, idx_k} - log T_k;   ell = sum_{k=0..6} logp_k and ell_old = sum_k old_logp_k, both in k order
 *   ratio = exp(ell - ell_old);  surr = -min(ratio A, clamp(ratio, lo, hi) A), lo = fl(1 - clip), hi = fl(1 + clip)
 *   ent = fl(sum_k H_k / K), summed in k order
 * Sums over i run in a fixed order (each lane of a warp adds elements lane + 32 s in ascending s, then an xor butterfly
 * 16, 8, 4, 2, 1; tests/ppo_loss.py states it), so a row's logp fed back as its old_logp gives ratio == 1 exactly and
 * surr == -A.  p >= 1 / (1 + (n-1) e^2) and, for K = 1, T_6 >= (n - 6) min p, so every log is finite.
 * evg_ppo_loss writes d_surr [B], d_ent [B], d_logp [B][7] and d_ratio [B].
 * evg_ppo_loss_grad writes d_dz [B][K][n] = g_surr d surr/dz + g_ent d ent/dz from d_ratio (evg_ppo_loss's) and the
 * upstream gradients d_g_surr, d_g_ent float32 [B], either NULL for zero, recomputing y, p, T and H from d_z:
 *   G = 0 where A > 0 and ratio > hi or A < 0 and ratio < lo (the clipped branch is the minimum), else fl(fl(-A ratio) g_surr)
 *   (at a tie, ratio exactly lo, hi or 1, the unclipped branch's, as torch's autograd of the expression above gives)
 *   d ell / d y_k,m = c_k,m - p_k,m Q_k,m: K = 1, c = the number of draws of m, Q = sum of 1 / T_j over the draws j
 *   whose T_j counted m (a prefix sum in j);  K = 7, c = [m = idx_k], Q = 1 / T_k
 *   dz = (1 - y^2) (G (c - p Q) - (g_ent / K) p (log p + H_k)), a term skipped when its factor G or g_ent is 0, so dz is
 *   exactly +0 where both are 0 and a clipped row's dz is its entropy part alone.
 * A row with an index outside [0, n) reads nothing out of bounds: its surr, ent, ratio and seven logp, and all of its dz,
 * are NaN.  One launch on `stream` each, no allocation, no synchronisation.  EVG_E_ARG, checked before the handle, for
 * n_rows outside 1..2^31-1, K not 1 or 7, n outside 7..256, clip outside [0, 1) or NaN, a NULL operand other than
 * g_surr / g_ent, d_idx not 8-byte aligned and a float32 operand not 4-byte aligned. */
int evg_ppo_loss(EvgSim* sim, int64_t n_rows, int32_t n_dist, int32_t n_actions, const float* d_z, const int64_t* d_idx, const float* d_old_logp,
                 const float* d_adv, float clip, float* d_surr, float* d_ent, float* d_logp, float* d_ratio, void* stream);
int evg_ppo_loss_grad(EvgSim* sim, int64_t n_rows, int32_t n_dist, int32_t n_actions, const float* d_z, const int64_t* d_idx, const float* d_adv,
                      const float* d_ratio, float clip, const float* d_g_surr, const float* d_g_ent, float* d_dz, void* stream);

/* The recurrent actor's GRU and action layer for a PPO update, forward and backward, on the tensor cores
 * (csrc/evg_rppo_train.cu; DESIGN.md §4.13).  Per row of B = n_rows, L = latent (1..EVG_PPO_MAX_LATENT), out = out_dim
 * (7..EVG_PPO_OUT_PAD): x float32 [L] is the head's output (d_x [B][L]) and h_0 float32 [L] the stored starting state
 * (d_h0 [B][L], evg_policy_rppo_logp's d_hidden_in).  For k = 1..7, gates r, z, n in torch.nn.GRU's order:
 *     r = sigmoid(W_ir x + W_hr h + (b_ir + b_hr)),   u = sigmoid(W_iz x + W_hz h + (b_iz + b_hz)),   c = W_hn h + b_hn
 *     n = tanh(W_in x + b_in + r c),   h_k = (1 - u) n + u h_{k-1},   z_k = W3 bf16(h_k) + b3
 * z_k is action_layer[0]'s output before its Tanh: evg_ppo_loss's z with K = 7.  The arithmetic is evg_policy_rppo's:
 * bf16 operands (x, h as the MMA operand, the weights), fp32 accumulation, X W_ir^T and H W_hr^T in one accumulator then
 * the pre-summed bias, the same sigmoid (1 / (1 + expf(-v)) correctly rounded) and tanhf, h kept in fp32.  So from the
 * head output and state of an acting call, h_7 is what that call leaves in d_hidden.
 *   evg_rppo_train_pack: the images both read, packed on the device from the float32 parameters in torch's layouts
 *       (d_w3 [out][L], d_b3 [out], d_w_ih / d_w_hh [3L][L], d_b_ih / d_b_hh [3L]), every byte written:
 *         d_wi_img, d_wh_img: weight_ih_l0 / weight_hh_l0 exactly as for evg_policy_rppo (three [Lp x Ka] blocks)
 *         d_wht_img: gate g's W_hg^T, three [Lp x Ka] blocks the same size: element (j, i) of block g = w_hh[g L + i][j]
 *         d_w3_img: exactly as for evg_policy_rppo
 *         d_bias: float32 [EVG_PPO_OUT_PAD + 6 * EVG_PPO_MAX_LATENT] = b3, then b_ih gate g at EVG_PPO_OUT_PAD + g * 256
 *                 and b_hh gate g at EVG_PPO_OUT_PAD + (3 + g) * 256, zero padded.
 *   evg_rppo_train_forward: d_z float32 [B][7][out] and d_h float32 [B][7][L] = h_1..h_7.
 *   evg_rppo_train_backward, from d_h (the forward's) and d_g float32 [B][7][L], which holds W3^T dz_k on entry
 *       (dz = dL/dz; the caller's fp32 product with bf16(W3)) and g_k on return, recomputing r, u, n, c bit for bit:
 *     g_k = W3^T dz_k + carry_{k+1} (carry_8 = 0);  dn = g (1 - u),  da_n = dn (1 - n^2),  da_u = g (h_{k-1} - n) u (1 - u),
 *     da_r = da_n c r (1 - r);  dgi_k = [da_r, da_u, da_n],  dgh_k = [da_r, da_u, da_n r]
 *     carry_k = fl(g u) + bf16(W_hh)^T bf16(dgh_k)  (tensor cores, bf16(dgh_k) the MMA operand), added as
 *     d_g[k-1] = fl(fl(W3^T dz_{k-1} + g_k u_k) + W_hh^T dgh_k)
 *     d_dgh float32 [B][7][3L] = dgh_1..dgh_7;  d_s float32 [B][3L] = sum_k dgi_k (k = 7 down to 1).
 *   The parameter gradients are the reductions dW_ih = S^T bf16(x), dW_hh = sum_{rows,k} dgh_k^T bf16(h_{k-1}),
 *   dW3 = sum dz_k^T bf16(h_k), the biases' the column sums, and dx = bf16(W_ih)^T S; no gradient flows to h_0.
 * Images and d_bias 16-byte aligned, float32 arrays 4-byte aligned.  One launch on `stream` each, no allocation, no
 * synchronisation.  EVG_E_ARG, checked before the handle, for n_rows outside 1..2^31-1 (the pack takes none), latent or
 * out_dim out of range, a NULL pointer and a misaligned one. */
int evg_rppo_train_pack(EvgSim* sim, const float* d_w3, const float* d_b3, const float* d_w_ih, const float* d_b_ih, const float* d_w_hh,
                        const float* d_b_hh, int32_t latent, int32_t out_dim, void* d_wi_img, void* d_wh_img, void* d_wht_img, void* d_w3_img,
                        float* d_bias, void* stream);
int evg_rppo_train_forward(EvgSim* sim, int64_t n_rows, int32_t latent, int32_t out_dim, const float* d_x, const float* d_h0, const void* d_wi_img,
                           const void* d_wh_img, const void* d_w3_img, const float* d_bias, float* d_z, float* d_h, void* stream);
int evg_rppo_train_backward(EvgSim* sim, int64_t n_rows, int32_t latent, int32_t out_dim, const float* d_x, const float* d_h0, const float* d_h,
                            const void* d_wi_img, const void* d_wh_img, const void* d_wht_img, const float* d_bias, float* d_g, float* d_dgh,
                            float* d_s, void* stream);

/* The images above packed ON THE DEVICE from the network's float32 parameters (csrc/evg_policy_pack.cu), byte for byte
 * what evgsim.policy.pack_mlp / pack_ppo / pack_rppo / pack_value build on the host: one launch on `stream`, no host synchronisation,
 * so a training loop refreshes the images in place after each optimiser step (and can capture that in a CUDA graph).
 * Sources are device arrays in torch's layouts (contiguous, row-major): d_w1 [hidden or latent][obs_len], d_w2 / d_w3
 * [out][in] as nn.Linear.weight, biases [out]; d_w_ih / d_w_hh [3 * latent][latent] and d_b_ih / d_b_hh [3 * latent] as
 * nn.GRU's weight_ih_l0 ... (gates r, z, n).  The input width is the simulator's obs_len, the one the forward kernels read.
 *   evg_pack_mlp:  d_w1_img / d_w2_img as evg_policy_mlp reads them (W1' = [W1 | b1] plus the unit of ones, W2' = [W2 | b2],
 *                  ceil((hidden + 1) / EVG_MLP_CHUNK) chunks each).
 *   evg_pack_ppo:  d_w1_img, d_w2_img, d_w3_img and d_bias as evg_policy_ppo reads them.
 *   evg_pack_rppo: the same, plus d_wi_img / d_wh_img and the GRU biases in d_bias as evg_policy_rppo reads them.
 *   evg_pack_value: d_w1_img, d_w2_img, d_w3_img and d_bias as evg_policy_value reads them (d_w3 [1][latent], d_b3 [1]).
 * Every byte of every image and of d_bias is written, zero padding included.  Weights round to bf16 to nearest even
 * (overflow to +-Inf, subnormals kept); a NaN packs to a bf16 NaN of unspecified payload.  Images and d_bias must be
 * 16-byte aligned; hidden, latent, out_dim and obs_len are checked as the matching evg_policy_* checks them. */
int evg_pack_mlp(EvgSim* sim, const float* d_w1, const float* d_b1, const float* d_w2, const float* d_b2, int32_t hidden, int32_t out_dim,
                 void* d_w1_img, void* d_w2_img, void* stream);
int evg_pack_ppo(EvgSim* sim, const float* d_w1, const float* d_b1, const float* d_w2, const float* d_b2, const float* d_w3, const float* d_b3,
                 int32_t latent, int32_t out_dim, void* d_w1_img, void* d_w2_img, void* d_w3_img, float* d_bias, void* stream);
int evg_pack_rppo(EvgSim* sim, const float* d_w1, const float* d_b1, const float* d_w2, const float* d_b2, const float* d_w3, const float* d_b3,
                  const float* d_w_ih, const float* d_b_ih, const float* d_w_hh, const float* d_b_hh, int32_t latent, int32_t out_dim,
                  void* d_w1_img, void* d_w2_img, void* d_wi_img, void* d_wh_img, void* d_w3_img, float* d_bias, void* stream);
int evg_pack_value(EvgSim* sim, const float* d_w1, const float* d_b1, const float* d_w2, const float* d_b2, const float* d_w3,
                   const float* d_b3, int32_t latent, void* d_w1_img, void* d_w2_img, void* d_w3_img, float* d_bias, void* stream);

/* Reward shaping of the reference's training scripts (utils/reward_shaping.py:17-56) on the step's outputs:
 * d_out float32 [n_envs][2].  turnNum (steps played before this one) is read from the observation's turn
 * field, so use it with EVG_AUTORESET_OFF or _TERMINAL (the observation of a finished match is the terminal one). */
#define EVG_SHAPE_NORMALIZED_SCORE 0
#define EVG_SHAPE_BASIC 1
#define EVG_SHAPE_PENALIZE_LONG 2
#define EVG_SHAPE_SHORT_GAMES 3
int evg_shape_reward(EvgSim* sim, int32_t mode, const float* d_reward, const uint8_t* d_done, const float* d_obs, float* d_out,
                     void* stream);

/* Which step kernel evg_create() selected: 0 = a warp per match (small batches), 1 = a thread per match
 * (DESIGN.md section 4).  Scripted agents are fused into kernel 1 only; with kernel 0 evg_step_agents() needs
 * a non-NULL d_actions to pass the generated rows through.  -1 if sim is NULL. */
int evg_step_kernel_kind(const EvgSim* sim);

/* Number of kernels this library has launched since creation (bench.py's gpu_launches). */
int64_t evg_launch_count(const EvgSim* sim);

const char* evg_last_error(void);
int evg_abi_version(void);

#ifdef __cplusplus
}
#endif
#endif /* EVGSIM_H */

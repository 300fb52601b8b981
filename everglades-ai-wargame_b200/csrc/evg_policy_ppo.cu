// evg_policy_ppo.cu — the PPO actor of the policy-in-the-loop path on the 5th-generation tensor cores (tcgen05 + TMEM),
// sm_100a, with the action sampling fused behind it.
//
// The network is PPO's feed-forward actor (agents/PPO/ActorCritic.py:33-50 without the GRU; tools/policy_rollout.py):
//     probs = Softmax(Tanh(Linear(L, out)(Tanh(Linear(L, L)(Tanh(Linear(obs_len, L)(obs)))))))      1 <= L <= 256
// followed by PPOAgent.get_action (agents/PPO/PPOAgent.py:122-127): 7 distinct flat indices drawn from probs without
// replacement, each unravelled into an action row (idx / div, idx % mod).  One launch reads the observation tensor the
// step kernel wrote and writes the action rows; nothing else leaves the SM unless asked for (indices, probabilities).
//
//   CTA = 512 threads, persistent over tiles of 128 rows (UMMA M = 128: TMEM lane i holds row i of the accumulators;
//   four threads per row, one per quarter of the 16-column groups).  Per tile:
//       A  <- the tile's float32 observations -> bf16, K-major, 128-byte swizzle (prefetched into registers under the
//             previous tile's epilogue and sampling)
//       D1 = A . W1^T      (N = Lp = L rounded up to 16)   H = bf16(tanh(D1 + b1))
//       D2 = H . W2^T      (K = Lp in chunks of 128)       H = bf16(tanh(D2 + b2))   (H reused: layer 2 has retired)
//       D3 = H . W3^T      (N = 144)                       e = exp(tanh(D3 + b3)) -> shared memory, over A and H
//       one thread per row: p = e / sum(e), then the 7 draws (below) -> action rows
//   The biases are added in fp32 by the epilogues (tanh(1) is no constant one, so DQN's homogeneous trick does not
//   carry over).  The weight images — up to 264 KB of bf16 at L = 256 — do not fit next to A (32 KB) and H (64 KB), so
//   they are streamed from L2 every tile in pieces of at most two swizzle atoms (W1; W2 and W3 per 128 K-columns) through
//   two 64 KB slots: a piece is requested (cp.async.bulk onto the slot's mbarrier) as soon as the MMAs that read the
//   slot's previous piece have retired, so W2 arrives under epilogue 1, W3 under epilogue 2, and the next tile's W1 / W2
//   under this tile's sampling.  One elected thread issues copies and MMAs and commits the MMAs to an mbarrier.
//
// Sampling (the tape's domain 3, DESIGN.md §2): row (match m, player p), g = env_base + m, turn t and episode e read from
// the match's resident record — the state the rows will be played in.  w[0..3] = philox(g, t, p, 3 | e << 8),
// w[4..7] = philox(g, t, p | 1 << 8, 3 | e << 8); u_k = (w[k] >> 8) * 2^-24.  Draw k: T = fp32 sum in ascending j of the
// probabilities not chosen yet, x = u_k * T, walk the not-chosen j in ascending order accumulating c += p_j, take the
// first j with x < c (none, through rounding: the largest not-chosen j).  tests/ppo_sampling.py restates it.
// Chosen entries are overwritten with -0.0, which adds nothing to an fp32 sum of non-negative terms, and T of the next
// draw is accumulated during this draw's walk (the prefix before the chosen j, then every later term) — the same sums in
// the same order as the definition, in one pass per draw.
#include "evg_internal.h"
#include "evg_tcgen05.cuh"

namespace evg {

namespace {

constexpr int kInPad = EVG_PPO_IN_PAD;      // input features, padded (obs_len < 128)
constexpr int kMaxL = EVG_PPO_MAX_LATENT;   // latent width bound: 4 swizzle atoms of H, N <= 256 per MMA
constexpr int kOutPad = EVG_PPO_OUT_PAD;    // outputs, padded to a multiple of 16 (132 -> 144)
constexpr int kBiasFloats = 2 * kMaxL + kOutPad;
constexpr int kSlotBytes = 2 * kMaxL * 128;  // one weight piece: two swizzle atoms of up to 256 rows

// shared-memory carve-up (bytes; every operand block starts on a 1024-byte boundary, as the 128-byte swizzle needs)
constexpr int kSmA = 0;                                          // 2 atoms x [128 rows x 128 B]
constexpr int kSmH = kSmA + (kInPad / kAtomK) * kTileM * 128;    // 4 atoms x [128 rows x 128 B]
constexpr int kSmW = kSmH + (kMaxL / kAtomK) * kTileM * 128;     // 2 slots of kSlotBytes
constexpr int kSmBias = kSmW + 2 * kSlotBytes;                   // b1 [256] | b2 [256] | b3 [144], float32
constexpr int kSmBar = kSmBias + kBiasFloats * 4;                // 3 mbarriers + the TMEM base address
constexpr int kSmBytes = kSmBar + 32;
constexpr int kSmP = kSmA;  // e, then p: float32 [out][128 rows], over A and H once layer 3 has read H
static_assert(kSmH % 1024 == 0 && kSmW % 1024 == 0 && kSlotBytes % 1024 == 0 && kSmBar % 8 == 0, "operand blocks must be 1024-byte aligned");
static_assert(kOutPad * kTileM * 4 <= kSmW, "the probabilities must fit over A and H");
static_assert(kSmBytes <= 227 * 1024, "shared memory");

constexpr int kTmemD1 = 0, kTmemD2 = 256;  // D3 reuses D1's columns (read out before layer 3 is issued)

// nk: chunks of 128 K-columns of layers 2 and 3
// kWire: the observations are wire rows (ws), else float32
// kLogp: a.logp may be written (the instantiation without it is the kernel as it was before d_logp existed: the extra
//        registers of the draw loop slowed the wire call that does not ask for it)
template <bool kWire, bool kLogp>
__global__ void __launch_bounds__(kCtaThreads, 1) evg_policy_ppo_kernel(const __grid_constant__ ActorArgs a, const int nk, const __grid_constant__ WireSrc ws)
{
    extern __shared__ __align__(1024) unsigned char smem[];
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    uint64_t* bar = reinterpret_cast<uint64_t*>(smem + kSmBar);  // [0] / [1] weight slot 0 / 1 landed, [2] a layer's MMAs done
    float* sb = reinterpret_cast<float*>(smem + kSmBias);
    float* ps = reinterpret_cast<float*>(smem + kSmP);
    for (int i = tid; i < kBiasFloats; i += kCtaThreads) sb[i] = a.bias[i];
    const uint32_t tmem = cta_setup<3>(tid, bar, reinterpret_cast<uint32_t*>(smem + kSmBar + 24));
    const int r = (warp & 3) * 32 + lane, quarter = warp >> 2;
    const uint32_t lane_base = tmem + ((uint32_t)((warp & 3) * 32) << 16);
    const int lp = a.lp, n_pieces = 1 + 2 * nk;
    const uint32_t idesc_l = make_idesc(kTileM, lp), idesc_o = make_idesc(kTileM, kOutPad);
    const uint32_t sA = smem_u32(smem + kSmA), sH = smem_u32(smem + kSmH), sW = smem_u32(smem + kSmW);
    const int64_t n_tiles = (a.rows + kTileM - 1) / kTileM;
    const int64_t my_tiles = blockIdx.x < n_tiles ? (n_tiles - blockIdx.x + gridDim.x - 1) / gridDim.x : 0;
    const int64_t total_pieces = my_tiles * n_pieces;

    // weight piece s of this CTA's sequence (n_pieces per tile: W1, W2 per 128 K-columns, W3 per 128 K-columns) into slot s & 1
    auto load_piece = [&](int64_t s) {
        if (s >= total_pieces) return;
        const int q = (int)(s % n_pieces);
        const int ka_atoms = (lp + kAtomK - 1) / kAtomK;
        const unsigned char* src;
        uint32_t bytes;
        if (q == 0) {
            src = a.w1;
            bytes = (kInPad / kAtomK) * lp * 128;
        } else {
            const bool l2 = q <= nk;
            const int c = l2 ? q - 1 : q - 1 - nk, rows = l2 ? lp : kOutPad;
            const int atoms = ka_atoms - 2 * c < 2 ? ka_atoms - 2 * c : 2;
            src = (l2 ? a.w2 : a.w3) + (size_t)2 * c * rows * 128;
            bytes = (uint32_t)(atoms * rows * 128);
        }
        bulk_load(smem + kSmW + (s & 1) * kSlotBytes, src, bytes, &bar[s & 1]);
    };
    auto wait_piece = [&](int64_t s) {
        mbar_wait(&bar[s & 1], (uint32_t)((s >> 1) & 1));
        tc_fence_after();
    };
    // one layer's MMAs into TMEM column `tcol`: A = the activations from shared memory (k0 = first K step of the piece),
    // B = the piece in slot s & 1 ([rows_b x 128 K-columns] at most)
    auto issue = [&](uint32_t tcol, uint32_t a_base, int64_t s, int k0, int k1, int rows_b, uint32_t idesc) {
        wait_piece(s);
        const uint32_t b_base = sW + (uint32_t)((s & 1) * kSlotBytes);
        for (int k = k0; k < k1; ++k) {
            const int kk = k - k0;
            const uint32_t offA = (k >> 2) * (kTileM * 128) + (k & 3) * 32, offB = (kk >> 2) * (rows_b * 128) + (kk & 3) * 32;
            umma(tmem + tcol, make_desc(a_base + offA), make_desc(b_base + offB), idesc, k > 0);
        }
    };
    uint32_t ph_m = 0;
    auto wait_layer = [&]() {
        mbar_wait(&bar[2], ph_m);
        ph_m ^= 1;
        tc_fence_after();
    };
    Stager<kWire, false> a_tile;  // A

    if (tid == 0) {
        load_piece(0);
        load_piece(1);
    }
    if (my_tiles > 0) {
        a_tile.load(tid, a.obs, (int64_t)blockIdx.x * kTileM, a.rows, a.in_dim, a.player, ws);
        a_tile.store(tid, smem + kSmA, a.in_dim, a.player, ws);
        fence_async_smem();
    }
    __syncthreads();
    int64_t s0 = 0;  // this tile's first weight piece
    for (int64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, s0 += n_pieces) {
        const int64_t row0 = tile * kTileM;
        const int nrows = a.rows - row0 < kTileM ? (int)(a.rows - row0) : kTileM;
        const int lk = lp / 16;  // K steps of layers 2 and 3
        // ---- layer 1
        if (tid == 0) {
            tc_fence_after();
            issue(kTmemD1, sA, s0, 0, kInPad / 16, lp, idesc_l);
            umma_commit(&bar[2]);
        }
        wait_layer();
        if (tid == 0) load_piece(s0 + 2);
        epilogue_tanh_bias(smem + kSmH, lane_base + kTmemD1, sb, r, quarter, lp);
        // ---- layer 2
        if (tid == 0) {
            tc_fence_after();
            for (int c = 0; c < nk; ++c) issue(kTmemD2, sH, s0 + 1 + c, 8 * c, lk < 8 * c + 8 ? lk : 8 * c + 8, lp, idesc_l);
            umma_commit(&bar[2]);
        }
        wait_layer();
        if (tid == 0)
            for (int c = 0; c < nk; ++c) load_piece(s0 + 3 + c);
        epilogue_tanh_bias(smem + kSmH, lane_base + kTmemD2, sb + kMaxL, r, quarter, lp);
        // ---- layer 3
        if (tid == 0) {
            tc_fence_after();
            for (int c = 0; c < nk; ++c) issue(kTmemD1, sH, s0 + 1 + nk + c, 8 * c, lk < 8 * c + 8 ? lk : 8 * c + 8, kOutPad, idesc_o);
            umma_commit(&bar[2]);
        }
        wait_layer();
        if (tid == 0)
            for (int c = 0; c < nk; ++c) load_piece(s0 + 3 + nk + c);
        const bool next = tile + gridDim.x < n_tiles;
        if (next) a_tile.load(tid, a.obs, (tile + gridDim.x) * kTileM, a.rows, a.in_dim, a.player, ws);  // in flight under the epilogue and the sampling
        // ---- e = exp(tanh(D3 + b3)) of my row, my 16-column groups, into ps[j][row] (A and H are free: layer 3 has retired)
        {
            constexpr int kG = (kOutPad / 16 + 3) / 4;
            uint32_t v[kG][16];
#pragma unroll
            for (int i = 0; i < kG; ++i)
                if (quarter + 4 * i < kOutPad / 16) tmem_ld16(lane_base + kTmemD1 + 16 * (quarter + 4 * i), v[i]);
            tmem_wait_ld();
#pragma unroll
            for (int i = 0; i < kG; ++i) {
                if (quarter + 4 * i >= kOutPad / 16) continue;
#pragma unroll
                for (int e = 0; e < 16; ++e) {
                    const int j = 16 * (quarter + 4 * i) + e;
                    if (j < a.out_dim) ps[j * kTileM + r] = expf(tanhf(__uint_as_float(v[i][e]) + sb[2 * kMaxL + j]));
                }
            }
        }
        tc_fence_before();
        __syncthreads();
        // ---- softmax and the 7 draws: one thread per row
        if (tid < kTileM && tid < nrows) {
            const int64_t i = row0 + tid;
            const ActorRow row = actor_row(a, i);
            const uint32_t* rec = a.records + row.env * a.rec_words;
            const uint32_t turn = rec[kRecTurn], episode = rec[kRecEpisode];
            uint32_t w[2][4];
            draw_block(a, row, turn, episode, 0, w[0]);
            draw_block(a, row, turn, episode, 1, w[1]);
            float* pr = ps + tid;
            const int out_dim = a.out_dim;
            float sum = 0.f;
#pragma unroll 4
            for (int j = 0; j < out_dim; ++j) sum += pr[j * kTileM];
            float total = 0.f;  // T of the first draw
            float* gp = a.probs ? a.probs + i * out_dim : nullptr;
#pragma unroll 4
            for (int j = 0; j < out_dim; ++j) {
                const float q = pr[j * kTileM] / sum;
                pr[j * kTileM] = q;
                total += q;
                if (gp) gp[j] = q;
            }
            int64_t* ip = a.idx ? a.idx + i * EVG_MAX_ACTIONS : nullptr;
            float* lq = kLogp && a.logp ? a.logp + i * EVG_MAX_ACTIONS : nullptr;
#pragma unroll
            for (int k = 0; k < EVG_MAX_ACTIONS; ++k) {
                const float x = draw_uniform(w[k >> 2][k & 3]) * total;
                float c = 0.f, t = 0.f, c_last = 0.f;
                int sel = -1, last = -1;
#pragma unroll 4
                for (int j = 0; j < out_dim; ++j) {
                    const float q = pr[j * kTileM];
                    const float cn = c + q;
                    const bool open = !(__float_as_uint(q) >> 31);  // not chosen yet (chosen = -0.0)
                    if (open) { last = j; c_last = c; }
                    if (sel >= 0) t += q;
                    else if (open && x < cn) { sel = j; t = c; }
                    c = cn;
                }
                if (sel < 0) { sel = last; t = c_last; }
                if (lq) lq[k] = logf(pr[sel * kTileM] / total);  // total: this draw's T
                pr[sel * kTileM] = -0.f;
                total = t;
                if (ip) ip[k] = sel;
                store_action(a, row, k, sel);
            }
        }
        __syncthreads();  // the probabilities are read: A may be overwritten
        if (next) {
            a_tile.store(tid, smem + kSmA, a.in_dim, a.player, ws);
            fence_async_smem();
        }
        tc_fence_before();
        __syncthreads();
    }
    cta_teardown(tid, tmem);
}

}  // namespace

cudaError_t launch_policy_ppo(const Tables& t, const uint32_t* records, const void* obs, int64_t n_envs, int player, const void* w1_img,
                              const void* w2_img, const void* w3_img, const float* bias, int latent, int out_dim, int div, int mod,
                              int8_t* actions, int64_t* idx, float* probs, float* logp, int sm_count, cudaStream_t stream, const WireSrc* wire)
{
    const ActorArgs a = actor_args(t, records, obs, n_envs, player, w1_img, w2_img, w3_img, bias, latent, out_dim, div, mod, actions, idx, probs, logp);
    auto* kernel = wire ? (logp ? evg_policy_ppo_kernel<true, true> : evg_policy_ppo_kernel<true, false>)
                        : (logp ? evg_policy_ppo_kernel<false, true> : evg_policy_ppo_kernel<false, false>);
    return launch_persistent(kernel, a.rows, sm_count, kSmBytes, stream, a, (a.lp + 127) / 128, wire ? *wire : WireSrc{});
}

cudaError_t set_policy_ppo_smem()
{
    cudaError_t e = cudaSuccess;
    for (auto* kernel : {evg_policy_ppo_kernel<false, false>, evg_policy_ppo_kernel<true, false>, evg_policy_ppo_kernel<false, true>,
                         evg_policy_ppo_kernel<true, true>})
        if (e == cudaSuccess) e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmBytes);
    return e;
}

}  // namespace evg

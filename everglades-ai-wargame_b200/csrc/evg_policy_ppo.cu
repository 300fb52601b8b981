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

constexpr int kPpoThreads = 512;
constexpr int kTileM = 128;                 // observation rows per tile
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

constexpr int kTmemCols = 512;
constexpr int kTmemD1 = 0, kTmemD2 = 256;  // D3 reuses D1's columns (read out before layer 3 is issued)

struct PpoArgs {
    const float* obs;
    const unsigned char* w1;
    const unsigned char* w2;
    const unsigned char* w3;
    const float* bias;
    const uint32_t* records;
    int8_t* actions;
    int64_t* idx;
    float* probs;
    int64_t rows;  // n_envs * (player < 0 ? 2 : 1)
    int player, in_dim, lp, nk, out_dim, div, mod, rec_words;
    uint32_t env_base, seed_lo, seed_hi;
};

__global__ void __launch_bounds__(kPpoThreads, 1) evg_policy_ppo_kernel(const __grid_constant__ PpoArgs a)
{
    extern __shared__ __align__(1024) unsigned char smem[];
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    uint64_t* bar = reinterpret_cast<uint64_t*>(smem + kSmBar);  // [0] / [1] weight slot 0 / 1 landed, [2] a layer's MMAs done
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + kSmBar + 24);
    float* sb = reinterpret_cast<float*>(smem + kSmBias);
    float* ps = reinterpret_cast<float*>(smem + kSmP);
    for (int i = tid; i < kBiasFloats; i += kPpoThreads) sb[i] = a.bias[i];
    if (tid == 0) {
#pragma unroll
        for (int i = 0; i < 3; ++i) asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(smem_u32(&bar[i])));
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(kTmemCols));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::);
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem = *tmem_slot;
    const int r = (warp & 3) * 32 + lane, quarter = warp >> 2;
    const uint32_t lane_base = tmem + ((uint32_t)((warp & 3) * 32) << 16);
    const int lp = a.lp, nk = a.nk, n_pieces = 1 + 2 * nk;
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
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
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
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    };
    // a hidden layer's epilogue: my row, my 16-column groups (quarter, quarter + 4, ...): H = bf16(tanh(D + b))
    auto epilogue_hidden = [&](uint32_t tcol, const float* b) {
#pragma unroll 1
        for (int j0 = 16 * quarter; j0 < lp; j0 += 64) {
            uint32_t v[16];
            tmem_ld16(lane_base + tcol + j0, v);
            asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
            for (int g = 0; g < 2; ++g) {
                uint32_t w[4];
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                    const int j = j0 + 8 * g + 2 * e;
                    w[e] = pack_bf16(tanhf(__uint_as_float(v[8 * g + 2 * e]) + b[j]), tanhf(__uint_as_float(v[8 * g + 2 * e + 1]) + b[j + 1]));
                }
                *reinterpret_cast<uint4*>(smem + kSmH + swz_offset(kTileM, r, j0 + 8 * g)) = make_uint4(w[0], w[1], w[2], w[3]);
            }
        }
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");  // generic-proxy writes -> visible to the tensor core
        asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
        __syncthreads();
    };
    // A: a tile's observations -> bf16, swizzled; every thread owns 4 of the tile's 2048 16-byte chunks (8 features each)
    float af[kTileM * (kInPad / 8) / kPpoThreads][8];
    auto load_a = [&](int64_t row0) {
#pragma unroll
        for (int it = 0; it < kTileM * (kInPad / 8) / kPpoThreads; ++it) {
            const int i = tid + it * kPpoThreads, ar = i >> 4, k0 = (i & 15) * 8;
            const int64_t row = row0 + ar;
            const float* src = a.obs + (a.player < 0 ? row : 2 * row + a.player) * a.in_dim + k0;
#pragma unroll
            for (int e = 0; e < 8; ++e) af[it][e] = (row < a.rows && k0 + e < a.in_dim) ? __ldcs(src + e) : 0.f;
        }
    };
    auto store_a = [&]() {
#pragma unroll
        for (int it = 0; it < kTileM * (kInPad / 8) / kPpoThreads; ++it) {
            const int i = tid + it * kPpoThreads, ar = i >> 4, k0 = (i & 15) * 8;
            *reinterpret_cast<uint4*>(smem + kSmA + swz_offset(kTileM, ar, k0)) =
                make_uint4(pack_bf16(af[it][0], af[it][1]), pack_bf16(af[it][2], af[it][3]), pack_bf16(af[it][4], af[it][5]), pack_bf16(af[it][6], af[it][7]));
        }
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    };

    if (tid == 0) {
        load_piece(0);
        load_piece(1);
    }
    if (my_tiles > 0) {
        load_a((int64_t)blockIdx.x * kTileM);
        store_a();
    }
    __syncthreads();
    int64_t s0 = 0;  // this tile's first weight piece
    for (int64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, s0 += n_pieces) {
        const int64_t row0 = tile * kTileM;
        const int nrows = a.rows - row0 < kTileM ? (int)(a.rows - row0) : kTileM;
        const int lk = lp / 16;  // K steps of layers 2 and 3
        // ---- layer 1
        if (tid == 0) {
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            issue(kTmemD1, sA, s0, 0, kInPad / 16, lp, idesc_l);
            umma_commit(&bar[2]);
        }
        wait_layer();
        if (tid == 0) load_piece(s0 + 2);
        epilogue_hidden(kTmemD1, sb);
        // ---- layer 2
        if (tid == 0) {
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            for (int c = 0; c < nk; ++c) issue(kTmemD2, sH, s0 + 1 + c, 8 * c, lk < 8 * c + 8 ? lk : 8 * c + 8, lp, idesc_l);
            umma_commit(&bar[2]);
        }
        wait_layer();
        if (tid == 0)
            for (int c = 0; c < nk; ++c) load_piece(s0 + 3 + c);
        epilogue_hidden(kTmemD2, sb + kMaxL);
        // ---- layer 3
        if (tid == 0) {
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            for (int c = 0; c < nk; ++c) issue(kTmemD1, sH, s0 + 1 + nk + c, 8 * c, lk < 8 * c + 8 ? lk : 8 * c + 8, kOutPad, idesc_o);
            umma_commit(&bar[2]);
        }
        wait_layer();
        if (tid == 0)
            for (int c = 0; c < nk; ++c) load_piece(s0 + 3 + nk + c);
        const bool next = tile + gridDim.x < n_tiles;
        if (next) load_a((tile + gridDim.x) * kTileM);  // in flight under the epilogue and the sampling
        // ---- e = exp(tanh(D3 + b3)) of my row, my 16-column groups, into ps[j][row] (A and H are free: layer 3 has retired)
        {
            constexpr int kG = (kOutPad / 16 + 3) / 4;
            uint32_t v[kG][16];
#pragma unroll
            for (int i = 0; i < kG; ++i)
                if (quarter + 4 * i < kOutPad / 16) tmem_ld16(lane_base + kTmemD1 + 16 * (quarter + 4 * i), v[i]);
            asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
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
        asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
        __syncthreads();
        // ---- softmax and the 7 draws: one thread per row
        if (tid < kTileM && tid < nrows) {
            const int64_t i = row0 + tid;
            const int64_t env = a.player < 0 ? i >> 1 : i;
            const int p = a.player < 0 ? (int)(i & 1) : a.player;
            const uint32_t* rec = a.records + env * a.rec_words;
            const uint32_t turn = rec[kRecTurn], episode = rec[kRecEpisode], g = a.env_base + (uint32_t)env;
            uint32_t w[8];
            philox4x32_10(g, turn, (uint32_t)p, 3u | episode << 8, a.seed_lo, a.seed_hi, w);
            philox4x32_10(g, turn, (uint32_t)p | 1u << 8, 3u | episode << 8, a.seed_lo, a.seed_hi, w + 4);
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
            uint16_t* out = reinterpret_cast<uint16_t*>(a.actions + (env * 2 + p) * (EVG_MAX_ACTIONS * 2));
            int64_t* ip = a.idx ? a.idx + i * EVG_MAX_ACTIONS : nullptr;
#pragma unroll
            for (int k = 0; k < EVG_MAX_ACTIONS; ++k) {
                const float x = (float)(w[k] >> 8) * 0x1p-24f * total;
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
                pr[sel * kTileM] = -0.f;
                total = t;
                if (ip) ip[k] = sel;
                out[k] = (uint16_t)(((uint32_t)(sel / a.div) & 0xFFu) | ((uint32_t)(sel % a.mod) & 0xFFu) << 8);
            }
        }
        __syncthreads();  // the probabilities are read: A may be overwritten
        if (next) store_a();
        asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
        __syncthreads();
    }
    if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(kTmemCols));
}

}  // namespace

cudaError_t launch_policy_ppo(const Tables& t, const uint32_t* records, const float* obs, int64_t n_envs, int player, const void* w1_img,
                              const void* w2_img, const void* w3_img, const float* bias, int latent, int out_dim, int div, int mod,
                              int8_t* actions, int64_t* idx, float* probs, int sm_count, cudaStream_t stream)
{
    PpoArgs a;
    a.obs = obs;
    a.w1 = reinterpret_cast<const unsigned char*>(w1_img);
    a.w2 = reinterpret_cast<const unsigned char*>(w2_img);
    a.w3 = reinterpret_cast<const unsigned char*>(w3_img);
    a.bias = bias;
    a.records = records;
    a.actions = actions;
    a.idx = idx;
    a.probs = probs;
    a.rows = n_envs * (player < 0 ? 2 : 1);
    a.player = player;
    a.in_dim = t.obs_len;
    a.lp = (latent + 15) / 16 * 16;
    a.nk = (a.lp + 127) / 128;
    a.out_dim = out_dim;
    a.div = div;
    a.mod = mod;
    a.rec_words = t.rec_words8 * 2;
    a.env_base = t.env_base;
    a.seed_lo = t.seed_lo;
    a.seed_hi = t.seed_hi;
    if (a.rows <= 0) return cudaSuccess;
    static bool attr_set = false;
    if (!attr_set) {
        cudaError_t e = cudaFuncSetAttribute(evg_policy_ppo_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmBytes);
        if (e != cudaSuccess) return e;
        attr_set = true;
    }
    const int64_t tiles = (a.rows + kTileM - 1) / kTileM;
    const unsigned grid = (unsigned)(tiles < sm_count ? tiles : sm_count);
    evg_policy_ppo_kernel<<<grid, kPpoThreads, kSmBytes, stream>>>(a);
    return cudaGetLastError();
}

}  // namespace evg

// evg_policy_value.cu — the PPO critic on the 5th-generation tensor cores (tcgen05 + TMEM), sm_100a.
//
// The network is the critic of PPO's ActorCritic (agents/PPO/ActorCritic.py, value_layer; no copy of the reference is in
// this tree, so the shape is the one evgsim.policy.FusedValue accepts):
//     v = Linear(L, 1)(Tanh(Linear(L, L)(Tanh(Linear(obs_len, L)(obs)))))      1 <= L <= 256
// for M matches of observations (float32 [M][2][obs_len] or wire rows [M][row_bytes]), with M given by the caller: the
// env's current observations, or a whole stored rollout in one call.  Numerics are the actors' (DESIGN.md §4.6): bf16
// operands (observations, W1, W2, w3, both hidden activations), fp32 accumulation, b1 / b2 / b3 added in fp32.
//
//   CTA = 512 threads, persistent over tiles of 128 rows (four threads per row, one per quarter of the 16-column groups).
//   Per tile:
//       A  <- the tile's observations -> bf16, K-major, 128-byte swizzle (prefetched into registers under the previous
//             tile's layer-2 epilogue)
//       D1 = A . W1^T      (N = Lp = L rounded up to 16)   H = bf16(tanh(D1 + b1))
//       D2 = H . W2^T      (K = Lp in chunks of 128)       each thread: s_q = sum over its columns j, ascending in each
//                                                          16-column group and the groups ascending, of
//                                                          bf16(tanh(D2_j + b2_j)) * w3_j (fp32 fma)
//       v = ((s_0 + s_1) + s_2) + s_3 + b3     (the four quarters' partials added in this order by one thread per row)
//   The last layer is a dot product in the layer-2 epilogue rather than an MMA with w3 padded to N = 16: it saves one
//   MMA round trip (issue, commit, wait) per tile, and the second hidden layer never goes back to shared memory.
//   Weights stream like evg_policy_ppo's (two 64 KB slots, W1 as one piece, W2 per 128 K-columns); when L <= 128 the
//   two pieces of a tile are always W1 in slot 0 and W2 in slot 1, so they are loaded once per CTA and stay resident.
#include <cuda_bf16.h>

#include "evg_internal.h"
#include "evg_tcgen05.cuh"

namespace evg {

namespace {

constexpr int kInPad = EVG_PPO_IN_PAD;      // input features, padded (obs_len < 128)
constexpr int kMaxL = EVG_PPO_MAX_LATENT;   // latent width bound: 4 swizzle atoms of H, N <= 256 per MMA
constexpr int kBiasFloats = 2 * kMaxL + EVG_VALUE_OUT_PAD;
constexpr int kSlotBytes = 2 * kMaxL * 128;  // one weight piece: two swizzle atoms of up to 256 rows

// shared-memory carve-up (bytes; every operand block starts on a 1024-byte boundary, as the 128-byte swizzle needs)
constexpr int kSmA = 0;                                          // 2 atoms x [128 rows x 128 B]
constexpr int kSmH = kSmA + (kInPad / kAtomK) * kTileM * 128;    // 4 atoms x [128 rows x 128 B]
constexpr int kSmW = kSmH + (kMaxL / kAtomK) * kTileM * 128;     // 2 slots of kSlotBytes
constexpr int kSmBias = kSmW + 2 * kSlotBytes;                   // b1 [256] | b2 [256] | b3 [16], float32
constexpr int kSmW3 = kSmBias + kBiasFloats * 4;                 // w3 [256], bf16 (row 0 of the w3 image)
constexpr int kSmBar = kSmW3 + kMaxL * 2;                        // 3 mbarriers + the TMEM base address
constexpr int kSmBytes = kSmBar + 32;
constexpr int kSmPart = kSmA;  // the quarters' partial sums, float32 [4][128 rows], over A once layer 1 has read it
static_assert(kSmH % 1024 == 0 && kSmW % 1024 == 0 && kSlotBytes % 1024 == 0 && kSmBar % 8 == 0, "operand blocks must be 1024-byte aligned");
static_assert(4 * kTileM * 4 <= kSmH - kSmA, "the partial sums must fit over A");
static_assert(kSmBytes <= 227 * 1024, "shared memory");

constexpr int kTmemD1 = 0, kTmemD2 = 256;

// what the critic reads and writes: no records, tape, actions or draws
struct ValueArgs {
    const void* obs;  // float32 observations or wire rows
    const unsigned char* w1;
    const unsigned char* w2;
    const unsigned char* w3;
    const float* bias;
    float* value;  // [rows]
    int64_t rows;  // n_matches * (player < 0 ? 2 : 1)
    int player, in_dim, lp;
};

// nk: chunks of 128 K-columns of layer 2
// kWire: the observations are wire rows (ws), else float32
template <bool kWire>
__global__ void __launch_bounds__(kCtaThreads, 1) evg_policy_value_kernel(const __grid_constant__ ValueArgs a, const int nk, const __grid_constant__ WireSrc ws)
{
    extern __shared__ __align__(1024) unsigned char smem[];
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    uint64_t* bar = reinterpret_cast<uint64_t*>(smem + kSmBar);  // [0] / [1] weight slot 0 / 1 landed, [2] a layer's MMAs done
    float* sb = reinterpret_cast<float*>(smem + kSmBias);
    __nv_bfloat16* sw3 = reinterpret_cast<__nv_bfloat16*>(smem + kSmW3);
    float* part = reinterpret_cast<float*>(smem + kSmPart);
    for (int i = tid; i < kBiasFloats; i += kCtaThreads) sb[i] = a.bias[i];
    // element (0, k) of the [EVG_VALUE_OUT_PAD x Ka] w3 block: atom k / 64, row 0 (no swizzle), column k % 64
    for (int k = tid; k < kMaxL; k += kCtaThreads)
        sw3[k] = k < a.lp ? reinterpret_cast<const __nv_bfloat16*>(a.w3)[(k / kAtomK) * EVG_VALUE_OUT_PAD * 64 + k % kAtomK] : __float2bfloat16_rn(0.f);
    const uint32_t tmem = cta_setup<3>(tid, bar, reinterpret_cast<uint32_t*>(smem + kSmBar + 24));
    const int r = (warp & 3) * 32 + lane, quarter = warp >> 2;
    const uint32_t lane_base = tmem + ((uint32_t)((warp & 3) * 32) << 16);
    const int lp = a.lp, n_pieces = 1 + nk;
    const bool resident = n_pieces == 2;  // W1 always in slot 0, W2 always in slot 1: loaded once
    const uint32_t idesc_l = make_idesc(kTileM, lp);
    const uint32_t sA = smem_u32(smem + kSmA), sH = smem_u32(smem + kSmH), sW = smem_u32(smem + kSmW);
    const int64_t n_tiles = (a.rows + kTileM - 1) / kTileM;
    const int64_t my_tiles = blockIdx.x < n_tiles ? (n_tiles - blockIdx.x + gridDim.x - 1) / gridDim.x : 0;
    const int64_t total_pieces = my_tiles * n_pieces;

    // weight piece s of this CTA's sequence (n_pieces per tile: W1, W2 per 128 K-columns) into slot s & 1
    auto load_piece = [&](int64_t s) {
        if (s >= total_pieces || (resident && s >= 2)) return;
        const int q = (int)(s % n_pieces);
        const unsigned char* src;
        uint32_t bytes;
        if (q == 0) {
            src = a.w1;
            bytes = (kInPad / kAtomK) * lp * 128;
        } else {
            const int c = q - 1, ka_atoms = (lp + kAtomK - 1) / kAtomK;
            const int atoms = ka_atoms - 2 * c < 2 ? ka_atoms - 2 * c : 2;
            src = a.w2 + (size_t)2 * c * lp * 128;
            bytes = (uint32_t)(atoms * lp * 128);
        }
        bulk_load(smem + kSmW + (s & 1) * kSlotBytes, src, bytes, &bar[s & 1]);
    };
    auto wait_piece = [&](int64_t s) {
        mbar_wait(&bar[s & 1], resident ? 0u : (uint32_t)((s >> 1) & 1));
        tc_fence_after();
    };
    // one layer's MMAs into TMEM column `tcol`: A = the activations from shared memory (k0 = first K step of the piece),
    // B = the piece in slot s & 1 ([lp x 128 K-columns] at most)
    auto issue = [&](uint32_t tcol, uint32_t a_base, int64_t s, int k0, int k1) {
        wait_piece(s);
        const uint32_t b_base = sW + (uint32_t)((s & 1) * kSlotBytes);
        for (int k = k0; k < k1; ++k) {
            const int kk = k - k0;
            const uint32_t offA = (k >> 2) * (kTileM * 128) + (k & 3) * 32, offB = (kk >> 2) * (lp * 128) + (kk & 3) * 32;
            umma(tmem + tcol, make_desc(a_base + offA), make_desc(b_base + offB), idesc_l, k > 0);
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
        const int lk = lp / 16;  // K steps of layer 2
        // ---- layer 1
        if (tid == 0) {
            tc_fence_after();
            issue(kTmemD1, sA, s0, 0, kInPad / 16);
            umma_commit(&bar[2]);
        }
        wait_layer();
        if (tid == 0) load_piece(s0 + 2);
        epilogue_tanh_bias(smem + kSmH, lane_base + kTmemD1, sb, r, quarter, lp);
        // ---- layer 2
        if (tid == 0) {
            tc_fence_after();
            for (int c = 0; c < nk; ++c) issue(kTmemD2, sH, s0 + 1 + c, 8 * c, lk < 8 * c + 8 ? lk : 8 * c + 8);
            umma_commit(&bar[2]);
        }
        wait_layer();
        if (tid == 0)
            for (int c = 0; c < nk; ++c) load_piece(s0 + 3 + c);
        const bool next = tile + gridDim.x < n_tiles;
        if (next) a_tile.load(tid, a.obs, (tile + gridDim.x) * kTileM, a.rows, a.in_dim, a.player, ws);  // in flight under the epilogue
        // ---- the last layer: my row's partial sum over my 16-column groups, into part[quarter][row] (A is free: layer 1 has retired)
        {
            const float* b2 = sb + kMaxL;
            float s = 0.f;
#pragma unroll 1
            for (int j0 = 16 * quarter; j0 < lp; j0 += 64) {
                uint32_t v[16];
                tmem_ld16(lane_base + kTmemD2 + j0, v);
                tmem_wait_ld();
#pragma unroll
                for (int e = 0; e < 16; ++e) {
                    const float h = __bfloat162float(__float2bfloat16_rn(tanhf(__uint_as_float(v[e]) + b2[j0 + e])));
                    s = fmaf(h, __bfloat162float(sw3[j0 + e]), s);
                }
            }
            part[quarter * kTileM + r] = s;
        }
        tc_fence_before();
        __syncthreads();
        if (tid < nrows)
            a.value[row0 + tid] = (((part[tid] + part[kTileM + tid]) + part[2 * kTileM + tid]) + part[3 * kTileM + tid]) + sb[2 * kMaxL];
        __syncthreads();  // the partial sums are read: A may be overwritten
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

cudaError_t launch_policy_value(const void* obs, int64_t n_matches, int player, int in_dim, const void* w1_img, const void* w2_img,
                                const void* w3_img, const float* bias, int latent, float* value, int sm_count, cudaStream_t stream,
                                const WireSrc* wire)
{
    ValueArgs a;
    a.obs = obs;
    a.w1 = static_cast<const unsigned char*>(w1_img);
    a.w2 = static_cast<const unsigned char*>(w2_img);
    a.w3 = static_cast<const unsigned char*>(w3_img);
    a.bias = bias;
    a.value = value;
    a.rows = n_matches * (player < 0 ? 2 : 1);
    a.player = player;
    a.in_dim = in_dim;
    a.lp = (latent + 15) / 16 * 16;
    auto* kernel = wire ? evg_policy_value_kernel<true> : evg_policy_value_kernel<false>;
    return launch_persistent(kernel, a.rows, sm_count, kSmBytes, stream, a, (a.lp + 127) / 128, wire ? *wire : WireSrc{});
}

cudaError_t set_policy_value_smem()
{
    cudaError_t e = cudaSuccess;
    for (auto* kernel : {evg_policy_value_kernel<false>, evg_policy_value_kernel<true>})
        if (e == cudaSuccess) e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmBytes);
    return e;
}

}  // namespace evg

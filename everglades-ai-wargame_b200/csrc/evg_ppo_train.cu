// evg_ppo_train.cu — PPO's feed-forward networks for the update, forward and backward, on the 5th-generation tensor cores
// (tcgen05 + TMEM), sm_100a: the feed-forward actor, the critic and the recurrent actor's action head.  Definitions in
// include/evgsim.h (evg_ppo_train_forward / _backward), layout and budget in DESIGN.md §4.14.
//
// All three share Linear(obs_len, L) - Tanh - Linear(L, L) - Tanh; the actor adds Linear(L, out), the critic
// Linear(L, 1).  The forward is its network's acting kernel without the sampling, and issues the same MMAs (instruction
// N, K order, accumulate flags) from the same bf16 operands, so its outputs are the acting kernel's:
//     actor  (evg_policy_ppo):   every layer one N = Lp (N = 144 for the last) MMA per 16 K-columns
//     critic (evg_policy_value): the same two layers, then the fp32 dot product of evg_policy_value's epilogue
//     head   (evg_policy_rppo):  N split into pieces of <= 128 rows (TMEM column 128 rb + j still holds unit j)
//   CTA = 512 threads, persistent over tiles of 128 rows (four threads per row, one per quarter of the 16-column groups).
//   Weights stream through two 64 KB slots as in evg_policy_ppo (W1; W2 and W3 per 128 K-columns), resident when a tile
//   needs only two pieces.  The epilogues write h1 and h2 (fp32) of each live row besides bf16(h) into shared memory.
//
// The backward, per tile: dD2 = g2 (1 - h2^2) (fp32, written), A = bf16(dD2) swizzled, D = A . W2 (one K = Lp GEMM
// against the resident W2^T image, N = Lp), dD1 = D (1 - h1^2); its fp32 rows are read and written a warp per row.
#include "evg_internal.h"
#include "evg_tcgen05.cuh"

namespace evg {

namespace {

constexpr int kInPad = EVG_PPO_IN_PAD;
constexpr int kMaxL = EVG_PPO_MAX_LATENT;
constexpr int kOutPad = EVG_PPO_OUT_PAD;
constexpr int kBiasFloats = 2 * kMaxL + kOutPad;  // b1 | b2 | b3 (actor: 144, critic: b3 then w3 as 256 bf16)
constexpr int kSlotBytes = 2 * kMaxL * 128;
constexpr int kAtomBytes = kTileM * 128;

constexpr int kSmA = 0;
constexpr int kSmH = kSmA + (kInPad / kAtomK) * kAtomBytes;
constexpr int kSmW = kSmH + (kMaxL / kAtomK) * kAtomBytes;
constexpr int kSmBias = kSmW + 2 * kSlotBytes;
constexpr int kSmBar = kSmBias + kBiasFloats * 4;  // 3 mbarriers + the TMEM base address
constexpr int kSmBytes = kSmBar + 32;
constexpr int kSmPart = kSmA;  // critic: the quarters' partial sums over A, as evg_policy_value
constexpr int kSw3 = 2 * kMaxL + EVG_VALUE_OUT_PAD;  // critic: w3 in bf16 at this float of the bias region
static_assert(kSw3 + kMaxL / 2 <= kBiasFloats, "the critic's w3 must fit behind its b3");
static_assert(kSmH % 1024 == 0 && kSmW % 1024 == 0 && kSmBar % 8 == 0, "operand blocks must be 1024-byte aligned");
static_assert(kSmBytes <= 227 * 1024, "shared memory");

constexpr int kTmemD1 = 0, kTmemD2 = 256;  // the actor's D3 reuses D1's columns

// the backward: A = bf16(dD2) [128 x Lp], the whole W2^T image [Lp x Ka], then the mbarriers
constexpr int kBwSmWt = (kMaxL / kAtomK) * kAtomBytes;
constexpr int kBwSmBar = kBwSmWt + (kMaxL / kAtomK) * kMaxL * 128;
constexpr int kBwSmBytes = kBwSmBar + 32;
static_assert(kBwSmBytes <= 227 * 1024, "shared memory");

struct FwdArgs {
    const void* obs;
    const unsigned char* w1;
    const unsigned char* w2;
    const unsigned char* w3;
    const float* bias;
    float* out;  // actor: z [rows][out_dim]; critic: v [rows]; head: unused
    float* h1;   // [rows][latent]
    float* h2;
    int64_t rows;
    int player, in_dim, latent, lp, out_dim, bias_floats;
};

// kWire: the observations are wire rows (ws), else float32
// kNet: EVG_PPO_TRAIN_ACTOR / _CRITIC / _HEAD
template <bool kWire, int kNet>
__global__ void __launch_bounds__(kCtaThreads, 1) evg_ppo_train_forward_kernel(const __grid_constant__ FwdArgs a, const int nk, const __grid_constant__ WireSrc ws)
{
    constexpr bool kActor = kNet == EVG_PPO_TRAIN_ACTOR, kCritic = kNet == EVG_PPO_TRAIN_CRITIC, kSplit = kNet == EVG_PPO_TRAIN_HEAD;
    extern __shared__ __align__(1024) unsigned char smem[];
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    uint64_t* bar = reinterpret_cast<uint64_t*>(smem + kSmBar);  // [0] / [1] weight slot 0 / 1 landed, [2] a layer's MMAs done
    float* sb = reinterpret_cast<float*>(smem + kSmBias);
    for (int i = tid; i < a.bias_floats; i += kCtaThreads) sb[i] = a.bias[i];
    if (kCritic) {  // element (0, k) of the [EVG_VALUE_OUT_PAD x Ka] w3 block, as evg_policy_value stages it
        __nv_bfloat16* sw3 = reinterpret_cast<__nv_bfloat16*>(sb + kSw3);
        for (int k = tid; k < kMaxL; k += kCtaThreads)
            sw3[k] = k < a.lp ? reinterpret_cast<const __nv_bfloat16*>(a.w3)[(k / kAtomK) * EVG_VALUE_OUT_PAD * 64 + k % kAtomK] : __float2bfloat16_rn(0.f);
    }
    const uint32_t tmem = cta_setup<3>(tid, bar, reinterpret_cast<uint32_t*>(smem + kSmBar + 24));
    const int r = (warp & 3) * 32 + lane, quarter = warp >> 2;
    const uint32_t lane_base = tmem + ((uint32_t)((warp & 3) * 32) << 16);
    const int lp = a.lp, latent = a.latent, n_pieces = 1 + (kActor ? 2 : 1) * nk;
    const bool resident = n_pieces == 2;  // W1 always in slot 0, W2 always in slot 1: loaded once
    const uint32_t sA = smem_u32(smem + kSmA), sH = smem_u32(smem + kSmH), sW = smem_u32(smem + kSmW);
    const int64_t n_tiles = (a.rows + kTileM - 1) / kTileM;
    const int64_t my_tiles = blockIdx.x < n_tiles ? (n_tiles - blockIdx.x + gridDim.x - 1) / gridDim.x : 0;
    const int64_t total_pieces = my_tiles * n_pieces;

    // weight piece s of this CTA's sequence (W1, W2 per 128 K-columns, actor: W3 per 128 K-columns) into slot s & 1
    auto load_piece = [&](int64_t s) {
        if (s >= total_pieces || (resident && s >= 2)) return;
        const int q = (int)(s % n_pieces), ka_atoms = (lp + kAtomK - 1) / kAtomK;
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
    // one layer's MMAs into TMEM column `tcol`: A = the activations (k_steps steps of 16 K-columns), B = pieces s.. of
    // [rows_b x 128 K-columns] at most; N = rows_b, or (kSplit) pieces of <= 128 rows in row order, each over all of K
    auto layer = [&](uint32_t tcol, uint32_t a_base, int64_t s, int k_steps, int rows_b) {
        for (int c = 0; c * 8 < k_steps; ++c) {
            mbar_wait(&bar[(s + c) & 1], resident ? 0u : (uint32_t)(((s + c) >> 1) & 1));
            tc_fence_after();
        }
        const int nrb = kSplit ? (rows_b + 127) / 128 : 1;
        for (int rb = 0; rb < nrb; ++rb) {
            const int nh = kSplit ? (rows_b - 128 * rb < 128 ? rows_b - 128 * rb : 128) : rows_b;
            const uint32_t idesc = make_idesc(kTileM, nh);
            for (int k = 0; k < k_steps; ++k) {
                const int kk = k & 7;
                const uint32_t b_base = sW + (uint32_t)(((s + (k >> 3)) & 1) * kSlotBytes);
                const uint32_t offA = (k >> 2) * kAtomBytes + (k & 3) * 32, offB = (kk >> 2) * (rows_b * 128) + rb * 128 * 128 + (kk & 3) * 32;
                umma(tmem + tcol + 128 * rb, make_desc(a_base + offA), make_desc(b_base + offB), idesc, k > 0);
            }
        }
    };
    uint32_t ph_m = 0;
    auto wait_layer = [&]() {
        mbar_wait(&bar[2], ph_m);
        ph_m ^= 1;
        tc_fence_after();
    };
    // a hidden layer's epilogue, epilogue_tanh_bias's arithmetic: h = tanh(D + b) of my row's 16-column groups, fp32 to
    // my row of `hg` (live rows, j < L), bf16 to the swizzled operand at dst; then dst is made visible to the tensor core
    auto epilogue = [&](unsigned char* dst, uint32_t taddr, const float* b, float* hg) {
#pragma unroll 1
        for (int j0 = 16 * quarter; j0 < lp; j0 += 64) {
            uint32_t v[16];
            tmem_ld16(taddr + j0, v);
            tmem_wait_ld();
            float h[16];
#pragma unroll
            for (int e = 0; e < 16; ++e) h[e] = tanhf(__uint_as_float(v[e]) + b[j0 + e]);
            if (hg)
#pragma unroll
                for (int e = 0; e < 16; ++e)
                    if (j0 + e < latent) hg[j0 + e] = h[e];
#pragma unroll
            for (int g = 0; g < 2; ++g)
                *reinterpret_cast<uint4*>(dst + swz_offset(kTileM, r, j0 + 8 * g)) =
                    make_uint4(pack_bf16(h[8 * g], h[8 * g + 1]), pack_bf16(h[8 * g + 2], h[8 * g + 3]), pack_bf16(h[8 * g + 4], h[8 * g + 5]),
                               pack_bf16(h[8 * g + 6], h[8 * g + 7]));
        }
        fence_async_smem();
        tc_fence_before();
        __syncthreads();
    };
    Stager<kWire, false> a_tile;

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
    int64_t s0 = 0;
    for (int64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, s0 += n_pieces) {
        const int64_t row0 = tile * kTileM, my_row = row0 + r;
        const int nrows = a.rows - row0 < kTileM ? (int)(a.rows - row0) : kTileM;
        const bool live = r < nrows;
        const int lk = lp / 16;
        // ---- layer 1
        if (tid == 0) {
            tc_fence_after();
            layer(kTmemD1, sA, s0, kInPad / 16, lp);
            umma_commit(&bar[2]);
        }
        wait_layer();
        if (tid == 0) load_piece(s0 + 2);
        epilogue(smem + kSmH, lane_base + kTmemD1, sb, live ? a.h1 + my_row * latent : nullptr);
        // ---- layer 2
        if (tid == 0) {
            tc_fence_after();
            layer(kTmemD2, sH, s0 + 1, lk, lp);
            umma_commit(&bar[2]);
        }
        wait_layer();
        if (tid == 0)
            for (int c = 0; c < nk; ++c) load_piece(s0 + 3 + c);
        const bool next = tile + gridDim.x < n_tiles;
        float* h2row = live ? a.h2 + my_row * latent : nullptr;
        if (kCritic) {
            if (next) a_tile.load(tid, a.obs, (tile + gridDim.x) * kTileM, a.rows, a.in_dim, a.player, ws);
            // evg_policy_value's last layer: my row's partial sum over my 16-column groups, the quarters added in order
            const float* b2 = sb + kMaxL;
            const __nv_bfloat16* sw3 = reinterpret_cast<const __nv_bfloat16*>(sb + kSw3);
            float* part = reinterpret_cast<float*>(smem + kSmPart);
            float s = 0.f;
#pragma unroll 1
            for (int j0 = 16 * quarter; j0 < lp; j0 += 64) {
                uint32_t v[16];
                tmem_ld16(lane_base + kTmemD2 + j0, v);
                tmem_wait_ld();
#pragma unroll
                for (int e = 0; e < 16; ++e) {
                    const float t = tanhf(__uint_as_float(v[e]) + b2[j0 + e]);
                    if (h2row && j0 + e < latent) h2row[j0 + e] = t;
                    s = fmaf(__bfloat162float(__float2bfloat16_rn(t)), __bfloat162float(sw3[j0 + e]), s);
                }
            }
            part[quarter * kTileM + r] = s;
            tc_fence_before();
            __syncthreads();
            if (tid < nrows)
                a.out[row0 + tid] = (((part[tid] + part[kTileM + tid]) + part[2 * kTileM + tid]) + part[3 * kTileM + tid]) + sb[2 * kMaxL];
            __syncthreads();
        } else {
            epilogue(smem + kSmH, lane_base + kTmemD2, sb + kMaxL, h2row);
            if (kActor) {
                // ---- layer 3: z = D3 + b3
                if (tid == 0) {
                    tc_fence_after();
                    layer(kTmemD1, sH, s0 + 1 + nk, lk, kOutPad);
                    umma_commit(&bar[2]);
                }
                wait_layer();
                if (tid == 0)
                    for (int c = 0; c < nk; ++c) load_piece(s0 + 3 + nk + c);
            }
            if (next) a_tile.load(tid, a.obs, (tile + gridDim.x) * kTileM, a.rows, a.in_dim, a.player, ws);
            if (kActor) {
                float* zrow = a.out + my_row * a.out_dim;
#pragma unroll 1
                for (int i = 0; i < 3; ++i) {
                    const int gi = quarter + 4 * i;
                    if (gi >= kOutPad / 16) continue;
                    uint32_t v[16];
                    tmem_ld16(lane_base + kTmemD1 + 16 * gi, v);
                    tmem_wait_ld();
#pragma unroll
                    for (int e = 0; e < 16; ++e) {
                        const int j = 16 * gi + e;
                        if (live && j < a.out_dim) zrow[j] = __uint_as_float(v[e]) + sb[2 * kMaxL + j];
                    }
                }
            }
        }
        if (next) {  // layer 1 has retired long ago: A is free
            a_tile.store(tid, smem + kSmA, a.in_dim, a.player, ws);
            fence_async_smem();
        }
        tc_fence_before();
        __syncthreads();
    }
    cta_teardown(tid, tmem);
}

struct BwdArgs {
    const unsigned char* w2t;  // [Lp x Ka]: element (j, i) = W2[i][j]
    const float* g2;
    const float* h1;
    const float* h2;
    float* dd2;
    float* dd1;
    int64_t rows;
    int latent, lp;
};

__global__ void __launch_bounds__(kCtaThreads, 1) evg_ppo_train_backward_kernel(const __grid_constant__ BwdArgs a)
{
    extern __shared__ __align__(1024) unsigned char smem[];
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    uint64_t* bar = reinterpret_cast<uint64_t*>(smem + kBwSmBar);  // [0] W2^T landed, [1] the GEMM's MMAs done
    const uint32_t tmem = cta_setup<2>(tid, bar, reinterpret_cast<uint32_t*>(smem + kBwSmBar + 16));
    const int r = (warp & 3) * 32 + lane, quarter = warp >> 2;
    const uint32_t lane_base = tmem + ((uint32_t)((warp & 3) * 32) << 16);
    const int lp = a.lp, latent = a.latent, ka_atoms = (lp + kAtomK - 1) / kAtomK;
    const uint32_t sA = smem_u32(smem), sWt = smem_u32(smem + kBwSmWt), idesc = make_idesc(kTileM, lp);
    const int64_t n_tiles = (a.rows + kTileM - 1) / kTileM;
    // the whole image in one copy: bar[0] counts one arrival (each bulk_load arrives once)
    if (tid == 0 && blockIdx.x < n_tiles) bulk_load(smem + kBwSmWt, a.w2t, (uint32_t)(ka_atoms * lp * 128), &bar[0]);
    // Global memory is read and written a warp per tile row, lane = column (mod 32): the 128 B a warp touches are
    // contiguous.  D leaves TMEM by lane = row, so it goes through shared memory: the A region (free once the GEMM has
    // retired), fp32 [128][128] per pass of 128 columns, column c of row r at c ^ (r & 31) (no bank conflict either way).
    float* stage = reinterpret_cast<float*>(smem);
    uint32_t ph = 0;
    for (int64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        const int64_t row0 = tile * kTileM;
        // ---- dD2 -> d_dd2 and bf16 into A: warp w builds tile rows w, w + 16, ..
#pragma unroll 1
        for (int ar = warp; ar < kTileM; ar += kCtaThreads / 32) {
            const bool live = row0 + ar < a.rows;
            const size_t off = (size_t)(row0 + ar) * latent;
#pragma unroll 2
            for (int j = lane; j < lp; j += 32) {
                const bool in = live && j < latent;
                const float h = in ? a.h2[off + j] : 0.f;
                const float d = in ? a.g2[off + j] * (1.f - h * h) : 0.f;
                if (in) a.dd2[off + j] = d;
                *reinterpret_cast<__nv_bfloat16*>(smem + swz_offset(kTileM, ar, j)) = __float2bfloat16_rn(d);
            }
        }
        fence_async_smem();
        tc_fence_before();
        __syncthreads();
        // ---- D = bf16(dD2) . W2 (K = Lp, N = Lp)
        if (tid == 0) {
            mbar_wait(&bar[0], 0);
            tc_fence_after();
            for (int k = 0; k < lp / 16; ++k)
                umma(tmem, make_desc(sA + (k >> 2) * kAtomBytes + (k & 3) * 32), make_desc(sWt + (k >> 2) * (lp * 128) + (k & 3) * 32), idesc, k > 0);
            umma_commit(&bar[1]);
        }
        mbar_wait(&bar[1], ph);
        ph ^= 1;
        tc_fence_after();
        // ---- dD1 = D (1 - h1^2), per pass of 128 columns: TMEM -> stage (row r's own lane), then a warp per row
#pragma unroll 1
        for (int c0 = 0; c0 < lp; c0 += 128) {
#pragma unroll 1
            for (int j0 = c0 + 16 * quarter; j0 < lp && j0 < c0 + 128; j0 += 64) {
                uint32_t v[16];
                tmem_ld16(lane_base + j0, v);
                tmem_wait_ld();
#pragma unroll
                for (int e = 0; e < 16; ++e) stage[r * 128 + ((j0 - c0 + e) ^ (r & 31))] = __uint_as_float(v[e]);
            }
            tc_fence_before();
            __syncthreads();
#pragma unroll 1
            for (int ar = warp; ar < kTileM; ar += kCtaThreads / 32) {
                if (row0 + ar >= a.rows) break;
                const size_t off = (size_t)(row0 + ar) * latent;
#pragma unroll 2
                for (int c = lane; c < 128 && c0 + c < latent; c += 32) {
                    const float h = a.h1[off + c0 + c];
                    a.dd1[off + c0 + c] = stage[ar * 128 + (c ^ (ar & 31))] * (1.f - h * h);
                }
            }
            tc_fence_before();
            __syncthreads();  // the stage is read (and, after the last pass, D): A and TMEM may be rewritten
        }
    }
    cta_teardown(tid, tmem);
}

using FwdKernel = void (*)(FwdArgs, int, WireSrc);

template <bool kWire>
FwdKernel forward_kernel(int net)
{
    return net == EVG_PPO_TRAIN_ACTOR    ? evg_ppo_train_forward_kernel<kWire, EVG_PPO_TRAIN_ACTOR>
           : net == EVG_PPO_TRAIN_CRITIC ? evg_ppo_train_forward_kernel<kWire, EVG_PPO_TRAIN_CRITIC>
                                         : evg_ppo_train_forward_kernel<kWire, EVG_PPO_TRAIN_HEAD>;
}

}  // namespace

cudaError_t launch_ppo_train_forward(int net, const void* obs, int64_t n_matches, int player, int in_dim, int latent, int out_dim,
                                     const void* w1_img, const void* w2_img, const void* w3_img, const float* bias, float* out, float* h1,
                                     float* h2, int sm_count, cudaStream_t stream, const WireSrc* wire)
{
    FwdArgs a;
    a.obs = obs;
    a.w1 = static_cast<const unsigned char*>(w1_img);
    a.w2 = static_cast<const unsigned char*>(w2_img);
    a.w3 = static_cast<const unsigned char*>(w3_img);
    a.bias = bias;
    a.out = out;
    a.h1 = h1;
    a.h2 = h2;
    a.rows = n_matches * (player < 0 ? 2 : 1);
    a.player = player;
    a.in_dim = in_dim;
    a.latent = latent;
    a.lp = (latent + 15) / 16 * 16;
    a.out_dim = out_dim;
    a.bias_floats = ppo_train_bias_floats(net);
    const FwdKernel kernel = wire ? forward_kernel<true>(net) : forward_kernel<false>(net);
    return launch_persistent(kernel, a.rows, sm_count, kSmBytes, stream, a, (a.lp + 127) / 128, wire ? *wire : WireSrc{});
}

cudaError_t launch_ppo_train_backward(int64_t n_rows, int latent, const void* w2t_img, const float* g2, const float* h1, const float* h2,
                                      float* dd2, float* dd1, int sm_count, cudaStream_t stream)
{
    BwdArgs a;
    a.w2t = static_cast<const unsigned char*>(w2t_img);
    a.g2 = g2;
    a.h1 = h1;
    a.h2 = h2;
    a.dd2 = dd2;
    a.dd1 = dd1;
    a.rows = n_rows;
    a.latent = latent;
    a.lp = (latent + 15) / 16 * 16;
    return launch_persistent(evg_ppo_train_backward_kernel, n_rows, sm_count, kBwSmBytes, stream, a);
}

cudaError_t set_ppo_train_smem()
{
    cudaError_t e = cudaFuncSetAttribute(evg_ppo_train_backward_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kBwSmBytes);
    for (int net = 0; net < 3; ++net)
        for (FwdKernel kernel : {forward_kernel<false>(net), forward_kernel<true>(net)})
            if (e == cudaSuccess) e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmBytes);
    return e;
}

}  // namespace evg

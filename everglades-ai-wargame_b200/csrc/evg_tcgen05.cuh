// evg_tcgen05.cuh — the skeleton shared by the three fused policy kernels (evg_policy_mlp.cu, evg_policy_ppo.cu,
// evg_policy_rppo.cu): the 5th-generation tensor-core plumbing (tcgen05 MMAs into TMEM, mbarriers, bulk copies, the
// 128-byte-swizzled K-major operand layout), the CTA's setup and teardown, the observation-tile stager, the hidden-layer
// epilogue of the PPO actors, their draw plumbing, and the persistent-grid launch.
#pragma once
#include <cuda_bf16.h>
#include <stdint.h>

#include <type_traits>

#include "evg_internal.h"

namespace evg {

constexpr int kAtomK = 64;       // bf16 elements in one 128-byte swizzle row
constexpr int kTileM = 128;      // observation rows per tile (UMMA M = 128: TMEM lane i holds row i of the accumulators)
constexpr int kCtaThreads = 512; // four threads per row, one per quarter of the columns
constexpr int kObsCols = 128;    // observation columns of the A tile (EVG_MLP_IN_PAD = EVG_PPO_IN_PAD)
constexpr int kTmemCols = 512;   // every policy kernel allocates the SM's whole tensor memory: one CTA per SM
static_assert(EVG_MLP_IN_PAD == kObsCols && EVG_PPO_IN_PAD == kObsCols, "the observation tile is 128 columns wide");

// K-major operand tile with 128-byte swizzle: element (row r, column k) of a [rows x K] bf16 matrix lives in atom k / 64
// (a block of rows x 128 bytes), at row r, 16-byte chunk ((k % 64) / 8) ^ (r % 8)
__host__ __device__ inline int swz_offset(int rows, int r, int k)
{
    return (k / kAtomK) * rows * 128 + r * 128 + ((((k % kAtomK) >> 3) ^ (r & 7)) << 4) + (k & 7) * 2;
}

// the fields evg_policy_ppo_kernel and evg_policy_rppo_kernel share (filled by actor_args)
struct ActorArgs {
    const void* obs;  // float32 observations or wire rows
    const unsigned char* w1;
    const unsigned char* w2;
    const unsigned char* w3;
    const float* bias;
    const uint32_t* records;
    int8_t* actions;
    int64_t* idx;
    float* probs;
    float* logp;   // [rows][7]: log(p_j / T) of each draw (null: not written)
    int64_t rows;  // n_envs * (player < 0 ? 2 : 1)
    int player, in_dim, lp, out_dim, div, mod, rec_words;
    uint32_t env_base, seed_lo, seed_hi;
};

inline ActorArgs actor_args(const Tables& t, const uint32_t* records, const void* obs, int64_t n_envs, int player, const void* w1_img,
                            const void* w2_img, const void* w3_img, const float* bias, int latent, int out_dim, int div, int mod,
                            int8_t* actions, int64_t* idx, float* probs, float* logp)
{
    ActorArgs a;
    a.obs = obs;
    a.w1 = reinterpret_cast<const unsigned char*>(w1_img);
    a.w2 = reinterpret_cast<const unsigned char*>(w2_img);
    a.w3 = reinterpret_cast<const unsigned char*>(w3_img);
    a.bias = bias;
    a.records = records;
    a.actions = actions;
    a.idx = idx;
    a.probs = probs;
    a.logp = logp;
    a.rows = n_envs * (player < 0 ? 2 : 1);
    a.player = player;
    a.in_dim = t.obs_len;
    a.lp = (latent + 15) / 16 * 16;
    a.out_dim = out_dim;
    a.div = div;
    a.mod = mod;
    a.rec_words = t.rec_words8 * 2;
    a.env_base = t.env_base;
    a.seed_lo = t.seed_lo;
    a.seed_hi = t.seed_hi;
    return a;
}

#ifdef __CUDACC__
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

// ordering of tensor-core work around thread synchronisation, and of generic-proxy shared-memory writes before the
// tensor core (async proxy) reads them
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void tmem_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tmem_wait_st() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// The CTA's start: thread 0 initialises kBars mbarriers (arrival count 1), warp 0 allocates the tensor memory into
// *tmem_slot and gives up the allocation permit; returns the TMEM base address, visible to every thread.  This and the
// helpers below take the kernel's own tid = threadIdx.x rather than reading it again: a second read hid tid < 512 from
// the compiler, and the recurrent actor's whole schedule changed with it (1.6 % slower on a B200 at 1000 W).
template <int kBars>
__device__ __forceinline__ uint32_t cta_setup(int tid, uint64_t* bar, uint32_t* tmem_slot)
{
    if (tid == 0) {
#pragma unroll
        for (int i = 0; i < kBars; ++i) asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(smem_u32(&bar[i])));
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (tid < 32) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(kTmemCols));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::);
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    return *tmem_slot;
}

// the CTA's end: warp 0 frees the tensor memory it allocated
__device__ __forceinline__ void cta_teardown(int tid, uint32_t tmem)
{
    if (tid < 32) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(kTmemCols));
}

// shared-memory matrix descriptor (cute::UMMA::SmemDescriptor): start address >> 4 [0:14), leading byte offset >> 4
// [16:30) (unused for a swizzled K-major operand), stride byte offset >> 4 [32:46) = 1024 B between 8-row groups,
// version 1 [46:48), layout SWIZZLE_128B = 2 [61:64)
__device__ __forceinline__ uint64_t make_desc(uint32_t saddr)
{
    return (uint64_t)((saddr & 0x3FFFFu) >> 4) | (uint64_t)1 << 16 | (uint64_t)(1024 >> 4) << 32 | (uint64_t)1 << 46 | (uint64_t)2 << 61;
}

// instruction descriptor (cute::UMMA::InstrDescriptor): D fp32 [4:6) = 1, A bf16 [7:10) = 1, B bf16 [10:13) = 1, both
// K-major, N >> 3 at [17:23), M >> 4 at [24:29)
__device__ __forceinline__ uint32_t make_idesc(int m, int n)
{
    return 1u << 4 | 1u << 7 | 1u << 10 | (uint32_t)(n >> 3) << 17 | (uint32_t)(m >> 4) << 24;
}

__device__ __forceinline__ void umma(uint32_t tmem_d, uint64_t da, uint64_t db, uint32_t idesc, uint32_t accumulate)
{
    asm volatile(
        "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}\n" ::"r"(tmem_d), "l"(da), "l"(db), "r"(idesc), "r"(accumulate)
        : "memory");
}

__device__ __forceinline__ void umma_commit(uint64_t* bar)
{
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}

// wait for phase `parity` of an mbarrier; a bounded spin that traps instead of hanging the GPU if the MMAs never arrive
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity)
{
    const uint32_t a = smem_u32(bar);
    for (uint32_t spin = 0;; ++spin) {
        uint32_t done;
        asm volatile(
            "{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}\n"
            : "=r"(done)
            : "r"(a), "r"(parity)
            : "memory");
        if (done) return;
        if (spin > (1u << 26)) __trap();
    }
}

// has phase `parity` of an mbarrier completed?  (no wait)
__device__ __forceinline__ bool mbar_test(uint64_t* bar, uint32_t parity)
{
    uint32_t done;
    asm volatile("{\n\t.reg .pred p;\n\tmbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}\n"
                 : "=r"(done)
                 : "r"(smem_u32(bar)), "r"(parity)
                 : "memory");
    return done != 0;
}

__device__ __forceinline__ void tmem_ld4(uint32_t taddr, uint32_t (&v)[4])
{
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x4.b32 {%0, %1, %2, %3}, [%4];\n" : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]) : "r"(taddr));
}

__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&v)[16])
{
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];\n"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]), "=r"(v[9]), "=r"(v[10]),
          "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
        : "r"(taddr));
}

__device__ __forceinline__ void tmem_st16(uint32_t taddr, const uint32_t (&v)[16])
{
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};\n" ::"r"(taddr),
        "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]), "r"(v[8]), "r"(v[9]), "r"(v[10]), "r"(v[11]),
        "r"(v[12]), "r"(v[13]), "r"(v[14]), "r"(v[15])
        : "memory");
}

__device__ __forceinline__ uint32_t pack_bf16(float lo, float hi)
{
    const __nv_bfloat162 p = __floats2bfloat162_rn(lo, hi);
    return *reinterpret_cast<const uint32_t*>(&p);
}

// one bulk copy global -> shared memory, completion counted in bytes on `bar`
__device__ __forceinline__ void bulk_load(void* dst, const void* src, uint32_t bytes, uint64_t* bar)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst)), "l"(src), "r"(bytes),
                 "r"(smem_u32(bar))
                 : "memory");
}

// A tile of 128 observation rows -> bf16, K-major, 128-byte swizzle, 128 columns.  Every thread owns 4 of the tile's
// 2048 16-byte chunks (8 features each): load() issues all 32 loads together into registers (one DRAM round trip), so
// that they can be in flight under other work; store() converts and writes them.  Tile row ar is batch row row0 + ar,
// which reads observation row (player < 0 ? row : 2 row + player).  Rows past `rows` and features past in_dim are 0,
// except feature in_dim, which is the constant 1 that carries the first layer's bias when kBiasColumn.
template <bool kBiasColumn>
struct ObsTile {
    static constexpr int kIt = kTileM * (kObsCols / 8) / kCtaThreads;
    float f[kIt][8];

    __device__ __forceinline__ void load(int tid, const void* src_obs, int64_t row0, int64_t rows, int in_dim, int player, const WireSrc&)
    {
        const float* obs = static_cast<const float*>(src_obs);
#pragma unroll
        for (int it = 0; it < kIt; ++it) {
            const int i = tid + it * kCtaThreads, ar = i >> 4, k0 = (i & 15) * 8;
            const int64_t row = row0 + ar;
            const float* src = obs + (player < 0 ? row : 2 * row + player) * in_dim + k0;
#pragma unroll
            for (int e = 0; e < 8; ++e) f[it][e] = (row < rows && k0 + e < in_dim) ? __ldcs(src + e) : (kBiasColumn && k0 + e == in_dim ? 1.f : 0.f);
        }
    }
    __device__ __forceinline__ void store(int tid, unsigned char* dst, int, int, const WireSrc&) const
    {
#pragma unroll
        for (int it = 0; it < kIt; ++it) {
            const int i = tid + it * kCtaThreads, ar = i >> 4, k0 = (i & 15) * 8;
            *reinterpret_cast<uint4*>(dst + swz_offset(kTileM, ar, k0)) =
                make_uint4(pack_bf16(f[it][0], f[it][1]), pack_bf16(f[it][2], f[it][3]), pack_bf16(f[it][4], f[it][5]), pack_bf16(f[it][6], f[it][7]));
        }
    }
};

// The same tile from wire rows (EVG_OBS_WIRE): tile row ar = batch row row0 + ar is (match, player) = (row / 2, row % 2)
// when player < 0, else (row, player), and its values are what evg_wire_expand writes (wire_entry / wire_value).  The
// 16 threads that build a tile row (a half-warp: 8 features each) load its match's row together, word j + 16 q into
// thread j (kWords = 3 covers the 160-byte rows of a 16-node map; words past the row are not read): 8 bytes in flight per
// thread and tile row on DemoMap, 12 at 16 nodes, against the 32 of the float32 stager.  store() takes each entry's word
// from the thread that holds it with a shuffle inside the half-warp, so the stager needs no shared memory of its own.
// A thread's 8 features and its player are the same for every tile row it builds, so each entry's source is worked out
// once per store() and used for all kIt rows.
template <bool kBiasColumn>
struct WireTile {
    static constexpr int kIt = ObsTile<kBiasColumn>::kIt;
    static constexpr int kWords = 3;
    uint32_t w[kIt][kWords];
    uint32_t live;  // bit it: the tile row of iteration it is a batch row

    __device__ __forceinline__ void load(int tid, const void* src_rows, int64_t row0, int64_t rows, int, int player, const WireSrc& ws)
    {
        const uint32_t* base = static_cast<const uint32_t*>(src_rows);
        const int j = tid & 15;
        live = 0;
#pragma unroll
        for (int it = 0; it < kIt; ++it) {
            const int64_t row = row0 + ((tid + it * kCtaThreads) >> 4);
            const uint32_t* src = base + (player < 0 ? row >> 1 : row) * ws.words + j;
            if (row < rows) live |= 1u << it;
#pragma unroll
            for (int q = 0; q < kWords; ++q) w[it][q] = (row < rows && j + 16 * q < ws.words) ? __ldcs(src + 16 * q) : 0u;
        }
    }
    __device__ __forceinline__ void store(int tid, unsigned char* dst, int in_dim, int player, const WireSrc& ws) const
    {
        const int k0 = (tid & 15) * 8, p = player < 0 ? (tid >> 4) & 1 : player;
        uint32_t packed[kIt][4];
#pragma unroll
        for (int e = 0; e < 8; ++e) {
            const int k = k0 + e;
            uint32_t op = kWireConst, shift = 0;
            const int wi = k < in_dim ? wire_entry(ws, p, k, op, shift) : 0;
            const float pad = kBiasColumn && k == in_dim ? 1.f : 0.f;
            const float cst = k < in_dim && op == kWireConst ? wire_value(ws, p, k, op, 0, 0u) : pad;
#pragma unroll
            for (int it = 0; it < kIt; ++it) {
                uint32_t word = 0;
#pragma unroll
                for (int q = 0; q < kWords; ++q) {
                    const uint32_t v = __shfl_sync(0xFFFFFFFFu, w[it][q], wi & 15, 16);
                    if ((wi >> 4) == q) word = v;
                }
                const float x = !(live >> it & 1u) ? pad : op == kWireConst ? cst : wire_value(ws, p, k, op, shift, word);
                const uint32_t b = pack_bf16(x, 0.f) & 0xFFFFu;
                packed[it][e >> 1] = (e & 1) ? packed[it][e >> 1] | b << 16 : b;
            }
        }
#pragma unroll
        for (int it = 0; it < kIt; ++it) {
            const int ar = (tid + it * kCtaThreads) >> 4;
            *reinterpret_cast<uint4*>(dst + swz_offset(kTileM, ar, k0)) = make_uint4(packed[it][0], packed[it][1], packed[it][2], packed[it][3]);
        }
    }
};

// the observation stager of a policy kernel: float32 observations, or wire rows (kWire)
template <bool kWire, bool kBiasColumn>
using Stager = std::conditional_t<kWire, WireTile<kBiasColumn>, ObsTile<kBiasColumn>>;

// a PPO actor's hidden-layer epilogue: row r, the 16-column groups 16 quarter, + 64, ... below lp of the accumulators at
// TMEM address `taddr` (the thread's lane base + the layer's column): dst = bf16(tanh(D + b)), swizzled; then dst is made
// visible to the tensor core and the CTA synchronises
__device__ __forceinline__ void epilogue_tanh_bias(unsigned char* dst, uint32_t taddr, const float* b, int r, int quarter, int lp)
{
#pragma unroll 1
    for (int j0 = 16 * quarter; j0 < lp; j0 += 64) {
        uint32_t v[16];
        tmem_ld16(taddr + j0, v);
        tmem_wait_ld();
#pragma unroll
        for (int g = 0; g < 2; ++g) {
            uint32_t w[4];
#pragma unroll
            for (int e = 0; e < 4; ++e) {
                const int j = j0 + 8 * g + 2 * e;
                w[e] = pack_bf16(tanhf(__uint_as_float(v[8 * g + 2 * e]) + b[j]), tanhf(__uint_as_float(v[8 * g + 2 * e + 1]) + b[j + 1]));
            }
            *reinterpret_cast<uint4*>(dst + swz_offset(kTileM, r, j0 + 8 * g)) = make_uint4(w[0], w[1], w[2], w[3]);
        }
    }
    fence_async_smem();
    tc_fence_before();
    __syncthreads();
}

// row i of an actor's batch: (match, player) = (i / 2, i % 2) when both players are played, else (i, player)
struct ActorRow {
    int64_t env;
    int player;
};
__device__ __forceinline__ ActorRow actor_row(const ActorArgs& a, int64_t i) { return {a.player < 0 ? i >> 1 : i, a.player < 0 ? (int)(i & 1) : a.player}; }

// the draws of a row (match env, player p) at the turn and episode of the match's record, on the tape's domain 3
// (DESIGN.md §2): the uniform of draw k comes from word k % 4 of Philox block k / 4
__device__ __forceinline__ void draw_block(const ActorArgs& a, ActorRow row, uint32_t turn, uint32_t episode, int block, uint32_t (&w)[4])
{
    philox4x32_10(a.env_base + (uint32_t)row.env, turn, (uint32_t)row.player | (uint32_t)block << 8, 3u | episode << 8, a.seed_lo, a.seed_hi, w);
}
__device__ __forceinline__ float draw_uniform(uint32_t word) { return (float)(word >> 8) * 0x1p-24f; }

// action row k of (match env, player p) for flat index sel: (sel / div, sel % mod)
__device__ __forceinline__ void store_action(const ActorArgs& a, ActorRow row, int k, int sel)
{
    uint16_t* out = reinterpret_cast<uint16_t*>(a.actions + (row.env * 2 + row.player) * (EVG_MAX_ACTIONS * 2));
    out[k] = (uint16_t)(((uint32_t)(sel / a.div) & 0xFFu) | ((uint32_t)(sel % a.mod) & 0xFFu) << 8);
}

// the fused policy kernels are persistent over 128-row tiles: at most one CTA per SM (each takes all of its tensor
// memory), never more CTAs than tiles
template <typename... Params, typename... Args>
cudaError_t launch_persistent(void (*kernel)(Params...), int64_t rows, int sm_count, int smem, cudaStream_t stream, Args... args)
{
    if (rows <= 0) return cudaSuccess;
    const int64_t tiles = (rows + kTileM - 1) / kTileM;
    kernel<<<(unsigned)(tiles < sm_count ? tiles : sm_count), kCtaThreads, smem, stream>>>(args...);
    return cudaGetLastError();
}
#endif

}  // namespace evg

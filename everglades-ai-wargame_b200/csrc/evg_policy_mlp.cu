// evg_policy_mlp.cu — the policy-in-the-loop forward on the 5th-generation tensor cores (tcgen05 + TMEM), sm_100a.
//
// The only contraction on any configuration's path (BASELINE.json configs[3]): DQN's
//     Q = Linear(105, 528) - ReLU - Linear(528, 132)          agents/DQN/QNetwork.py:37,42
// evaluated for every (match, player) row of the observation tensor the step kernel has just written.  One kernel does
// both layers; the hidden activations never leave the SM:
//
//   CTA = 512 threads = one tile of 128 observation rows at a time (UMMA M = 128: TMEM lane i holds row i of the
//   accumulators; four threads per row, one per quarter of the columns), persistent over the tiles.
//   per tile:  A  <- the tile's float32 observations, converted to bf16 into the K-major 128-byte-swizzled layout
//              for each chunk c of 192 hidden units (528 -> 3 chunks, zero padded):
//                 D1[128 x 192]  = A[128 x 128] . W1c^T          8 x tcgen05.mma  (K = 16 each), accumulators in TMEM
//                 H              = bf16(relu(D1))                tcgen05.ld -> registers -> swizzled shared memory
//                 D2[128 x 144] += H[128 x 192] . W2c^T          12 x tcgen05.mma, accumulating over the chunks in TMEM
//              Q <- D2                                             tcgen05.ld -> registers -> global (float32)
//   Both biases ride inside the GEMMs (homogeneous coordinates): A carries a column of ones behind the obs_len features
//   whose weights are b1, and one padding hidden unit is wired to be relu(1) = 1 with b2 as its outgoing weights
//   (evgsim.policy.pack_mlp builds the images that way), so the epilogues are a ReLU and a store.
//   The weight chunks W1c / W2c are bf16 IMAGES of the shared-memory operand layout, fetched by the bulk-copy engine
//   (cp.async.bulk, one instruction per 48 / 54 KB image, completion on an mbarrier) as soon as the MMAs that read the
//   buffer's previous content have retired: W1(c+1) arrives under the activation epilogue and layer 2 of chunk c,
//   W2(c+1) under layer 1 and the epilogue of chunk c+1.  One elected thread issues copies and MMAs and commits the
//   MMAs to mbarriers (tcgen05.commit); the CTA waits on those.
//
// bf16 operands, fp32 accumulation.  Q is written either row-major [rows][out] (torch's layout) or transposed
// [out][rows] — what the thread-per-row decode (evg_decode_dqn, pinned to the reference's DQNAgent.filter_actions)
// reads coalesced.  tests/test_gpu_policy.py checks Q against torch fp32 within the bf16 tolerance stated there.
// Weight images are built on the host by evgsim.policy.pack_mlp (same swizzle function as evg_tcgen05.cuh).
#include <cuda_bf16.h>

#include "evg_internal.h"
#include "evg_tcgen05.cuh"

namespace evg {

namespace {

constexpr int kInPad = kObsCols;  // input features, padded (obs_len < 128: the bias input behind them)
constexpr int kChunk = 192;   // hidden units per chunk: 3 swizzle atoms of 64
constexpr int kOutPad = 144;  // outputs, padded to a multiple of 16 (12 groups x 11 nodes = 132)

// shared-memory carve-up (bytes; every operand block starts on a 1024-byte boundary, as the 128-byte swizzle needs)
constexpr int kSmA = 0;                                            // 2 atoms x [128 rows x 128 B]
constexpr int kSmH = kSmA + (kInPad / kAtomK) * kTileM * 128;      // 3 atoms x [128 rows x 128 B]
constexpr int kSmW1 = kSmH + (kChunk / kAtomK) * kTileM * 128;     // 2 atoms x [192 rows x 128 B]
constexpr int kSmW2 = kSmW1 + (kInPad / kAtomK) * kChunk * 128;    // 3 atoms x [144 rows x 128 B]
constexpr int kSmBar = kSmW2 + (kChunk / kAtomK) * kOutPad * 128;  // 4 mbarriers + the TMEM base address
constexpr int kSmBytes = kSmBar + 48;
constexpr int kW1ChunkBytes = (kInPad / kAtomK) * kChunk * 128;    // 49152
constexpr int kW2ChunkBytes = (kChunk / kAtomK) * kOutPad * 128;   // 55296
static_assert(kSmH % 1024 == 0 && kSmW1 % 1024 == 0 && kSmW2 % 1024 == 0 && (kOutPad * 128) % 1024 == 0 && (kChunk * 128) % 1024 == 0, "swizzle atoms must be 1024-byte aligned");

constexpr int kTmemD1 = 0, kTmemD2 = 256;  // D1 (192 columns) and D2 (144) in the 512 of kTmemCols

// q_col_stride == 1: Q[row * q_row_stride + col] (row-major); q_row_stride == 1: Q[col * q_col_stride + row] (transposed)
// kWire: obs holds wire rows (ws), observation row i = (match i / 2, player i % 2); else float32 rows
template <bool kWire>
__global__ void __launch_bounds__(kCtaThreads, 1)
evg_policy_mlp_kernel(const void* __restrict__ obs, int64_t rows, int in_dim, const unsigned char* __restrict__ w1_img,
                      const unsigned char* __restrict__ w2_img, int n_chunks, int out_dim, float* __restrict__ q, int64_t q_row_stride,
                      int64_t q_col_stride, const __grid_constant__ WireSrc ws)
{
    extern __shared__ __align__(1024) unsigned char smem[];
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    uint64_t* bar = reinterpret_cast<uint64_t*>(smem + kSmBar);  // [0] layer-1 MMAs done, [1] layer-2 MMAs done, [2] W1 image landed, [3] W2 image landed
    const uint32_t tmem = cta_setup<4>(tid, bar, reinterpret_cast<uint32_t*>(smem + kSmBar + 32));
    // my row = TMEM lane 32 * (warp % 4) + lane (a warp reaches the lane quarter warp % 4); my quarter of the columns = warp / 4
    const int r = (warp & 3) * 32 + lane, quarter = warp >> 2;
    const uint32_t lane_base = tmem + ((uint32_t)((warp & 3) * 32) << 16);
    const uint32_t idesc1 = make_idesc(kTileM, kChunk), idesc2 = make_idesc(kTileM, kOutPad);
    const uint32_t sA = smem_u32(smem + kSmA), sH = smem_u32(smem + kSmH), sW1 = smem_u32(smem + kSmW1), sW2 = smem_u32(smem + kSmW2);
    const int64_t n_tiles = (rows + kTileM - 1) / kTileM;
    const int64_t my_tiles = blockIdx.x < n_tiles ? (n_tiles - blockIdx.x + gridDim.x - 1) / gridDim.x : 0;
    const int64_t n_steps = my_tiles * n_chunks;  // (tile, chunk) steps of this CTA: the weight images cycle through the chunks
    uint32_t ph_m1 = 0, ph_m2 = 0, ph_w1 = 0, ph_w2 = 0;
    if (tid == 0 && n_steps > 0) {
        bulk_load(smem + kSmW1, w1_img, kW1ChunkBytes, &bar[2]);
        bulk_load(smem + kSmW2, w2_img, kW2ChunkBytes, &bar[3]);
    }
    Stager<kWire, true> a_tile;  // A: feature in_dim is the constant 1 that carries b1
    int64_t step = 0;
    bool l1_queued = false;  // the coming tile's first layer-1 MMAs were issued at the end of the previous tile
    for (int64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        const int64_t row0 = tile * kTileM;
        const int nrows = rows - row0 < kTileM ? (int)(rows - row0) : kTileM;
        if (tile == (int64_t)blockIdx.x) {  // the first tile: later ones are fetched and converted under the previous tile's last chunk
            a_tile.load(tid, obs, row0, rows, in_dim, -1, ws);
            a_tile.store(tid, smem + kSmA, in_dim, -1, ws);
            fence_async_smem();
            __syncthreads();
        }
        for (int c = 0; c < n_chunks; ++c, ++step) {
            const int cn = c + 1 == n_chunks ? 0 : c + 1;  // the chunk of the next step
            // ---- layer 1: D1 = A . W1c^T, as soon as W1c has landed.  Only a tile's first chunk is issued here: the later
            // ones are queued right behind the previous chunk's layer 2 (below), so that their latency is not paid again
            auto issue_layer1 = [&](uint32_t parity) {
                mbar_wait(&bar[2], parity);
                tc_fence_after();
#pragma unroll
                for (int k = 0; k < kInPad / 16; ++k) {  // within a swizzle atom the start address advances by 32 bytes per K = 16
                    const uint32_t offA = (k >> 2) * (kTileM * 128) + (k & 3) * 32, offB = (k >> 2) * (kChunk * 128) + (k & 3) * 32;
                    umma(tmem + kTmemD1, make_desc(sA + offA), make_desc(sW1 + offB), idesc1, k > 0);
                }
                umma_commit(&bar[0]);
            };
            if (tid == 0 && c == 0 && !l1_queued) issue_layer1(ph_w1);
            l1_queued = false;
            ph_w1 ^= 1;
            mbar_wait(&bar[0], ph_m1);  // D1 complete (and, the tensor pipe being in order, the previous step's layer 2: H is free)
            ph_m1 ^= 1;
            tc_fence_after();
            if (tid == 0 && step + 1 < n_steps) bulk_load(smem + kSmW1, w1_img + (size_t)cn * kW1ChunkBytes, kW1ChunkBytes, &bar[2]);
            const bool fetch_next_a = c + 1 == n_chunks && tile + gridDim.x < n_tiles;  // this tile's last layer-1 MMAs have read A: it is free
            if (fetch_next_a) a_tile.load(tid, obs, (tile + gridDim.x) * kTileM, rows, in_dim, -1, ws);  // in flight under the epilogue below
            // ---- hidden activations of my row, my 48 of the chunk's 192 columns: TMEM -> registers -> ReLU, bf16 -> swizzled H
            {
                constexpr int kLd = kChunk / 4 / 16;  // tensor-memory loads of 16 columns per thread: all issued, then one wait
                uint32_t v[kLd][16];
                const int jq1 = quarter * (kChunk / 4);
#pragma unroll
                for (int t = 0; t < kLd; ++t) tmem_ld16(lane_base + kTmemD1 + jq1 + 16 * t, v[t]);
                tmem_wait_ld();
#pragma unroll
                for (int t = 0; t < kLd; ++t) {
#pragma unroll
                    for (int g = 0; g < 2; ++g) {  // 8 hidden units = one 16-byte chunk of the swizzled row
                        uint32_t w[4];
#pragma unroll
                        for (int e = 0; e < 4; ++e)
                            w[e] = pack_bf16(fmaxf(__uint_as_float(v[t][8 * g + 2 * e]), 0.f), fmaxf(__uint_as_float(v[t][8 * g + 2 * e + 1]), 0.f));
                        *reinterpret_cast<uint4*>(smem + kSmH + swz_offset(kTileM, r, jq1 + 16 * t + 8 * g)) = make_uint4(w[0], w[1], w[2], w[3]);
                    }
                }
            }
            fence_async_smem();
            tc_fence_before();
            __syncthreads();
            // ---- layer 2: D2 += H . W2c^T
            if (tid == 0) {
                mbar_wait(&bar[3], ph_w2);
                tc_fence_after();
#pragma unroll
                for (int k = 0; k < kChunk / 16; ++k) {
                    const uint32_t offA = (k >> 2) * (kTileM * 128) + (k & 3) * 32, offB = (k >> 2) * (kOutPad * 128) + (k & 3) * 32;
                    umma(tmem + kTmemD2, make_desc(sH + offA), make_desc(sW2 + offB), idesc2, (c > 0 || k > 0) ? 1u : 0u);
                }
                umma_commit(&bar[1]);
                // the next chunk's layer 1 behind it: every thread has finished reading D1 (barrier above), the tensor pipe
                // runs in order, and W1's next chunk was requested when this chunk's layer 1 completed
                if (c + 1 < n_chunks) issue_layer1(ph_w1);
            }
            ph_w2 ^= 1;
            if (fetch_next_a) {  // the next tile's A, converted while layer 2 runs
                a_tile.store(tid, smem + kSmA, in_dim, -1, ws);
                fence_async_smem();
                __syncthreads();
                // ... and its first layer-1 MMAs queued now: they only write D1, so they run under this tile's Q store
                if (tid == 0) issue_layer1(ph_w1);
                l1_queued = true;
            }
            mbar_wait(&bar[1], ph_m2);  // the W2 buffer is free again; after the last chunk D2 is complete
            ph_m2 ^= 1;
            tc_fence_after();
            if (tid == 0 && step + 1 < n_steps) bulk_load(smem + kSmW2, w2_img + (size_t)cn * kW2ChunkBytes, kW2ChunkBytes, &bar[3]);
        }
        // ---- Q = D2: my row, my quarter of the columns (36 = 16 + 16 + 4)
        {
            float* qp = q + (row0 + r) * q_row_stride + (int64_t)(quarter * (kOutPad / 4)) * q_col_stride;
            const int jq = quarter * (kOutPad / 4);
            const bool live = r < nrows;
            uint32_t v[2][16], v4[4];
            tmem_ld16(lane_base + kTmemD2 + jq, v[0]);
            tmem_ld16(lane_base + kTmemD2 + jq + 16, v[1]);
            tmem_ld4(lane_base + kTmemD2 + jq + 32, v4);
            tmem_wait_ld();
#pragma unroll
            for (int j0 = 0; j0 < 32; j0 += 16) {
#pragma unroll
                for (int e = 0; e < 16; ++e, qp += q_col_stride)
                    if (live && jq + j0 + e < out_dim) *qp = __uint_as_float(v[j0 >> 4][e]);
            }
#pragma unroll
            for (int e = 0; e < 4; ++e, qp += q_col_stride)
                if (live && jq + 32 + e < out_dim) *qp = __uint_as_float(v4[e]);
        }
        tc_fence_before();
        __syncthreads();  // the next tile's first MMAs overwrite D1 / D2, its conversion overwrites A
    }
    cta_teardown(tid, tmem);
}

}  // namespace

cudaError_t launch_policy_mlp(const void* obs, int64_t rows, int in_dim, const void* w1_img, const void* w2_img, int n_chunks, int out_dim, float* q,
                              int transposed, int sm_count, cudaStream_t stream, const WireSrc* wire)
{
    return launch_persistent(wire ? evg_policy_mlp_kernel<true> : evg_policy_mlp_kernel<false>, rows, sm_count, kSmBytes, stream, obs, rows, in_dim,
                             reinterpret_cast<const unsigned char*>(w1_img), reinterpret_cast<const unsigned char*>(w2_img), n_chunks, out_dim, q,
                             (int64_t)(transposed ? 1 : out_dim), (int64_t)(transposed ? rows : 1), wire ? *wire : WireSrc{});
}

cudaError_t set_policy_mlp_smem()
{
    cudaError_t e = cudaFuncSetAttribute(evg_policy_mlp_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmBytes);
    return e != cudaSuccess ? e : cudaFuncSetAttribute(evg_policy_mlp_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmBytes);
}

}  // namespace evg

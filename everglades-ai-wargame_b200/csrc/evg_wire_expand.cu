// evg_wire_expand.cu — wire rows (include/evgsim.h, EVG_OBS_WIRE) back into the float32 observation vector, reward and done
// flag, on the device: what evgsim.wire.expand does on the host, for rows a training consumer stored (a replay or rollout
// memory keeps 128 B per match on DemoMap instead of 840) or a minibatch of them picked by an index.
//
// Memory-bound.  The output is the bulk of the traffic (4 * obs_len bytes per player against one row read), so the grid
// walks the output: each thread writes 4 consecutive floats of the flat [n_out][players][obs_len] array with one 16-byte
// store (a warp: 512 contiguous bytes), and reads, per value, the one word of its row that holds it (wire_entry).  The
// threads that fill one output row read the same row, so it comes from DRAM once (one 128-byte line on DemoMap) and from
// L1 for the other ~50 of them; the constant entries and p1_map are a few hundred bytes that stay in L1.  Reward and done
// are written by a second walk over the output rows in the same launch.
#include "evg_internal.h"

namespace evg {

namespace {

constexpr int kExpandThreads = 256;

__global__ void __launch_bounds__(kExpandThreads) evg_wire_expand_kernel(const __grid_constant__ WireSrc w, const uint32_t* __restrict__ rows,
                                                                        int64_t n_rows, const int64_t* __restrict__ index, int64_t n_out,
                                                                        int player, float* __restrict__ obs, float* __restrict__ reward,
                                                                        uint8_t* __restrict__ done)
{
    const int players = player < 0 ? 2 : 1, row_len = players * w.obs_len;
    const int64_t total = n_out * row_len;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; 4 * t < total; t += stride) {
        const int64_t i0 = 4 * t;
        int64_t o = i0 / row_len;
        int rem = (int)(i0 - o * row_len);
        float v[4];
#pragma unroll
        for (int e = 0; e < 4; ++e) {
            v[e] = 0.f;
            if (i0 + e < total) {
                const int64_t src = index ? __ldg(index + o) : o;
                if (src >= 0 && src < n_rows) {
                    const int pp = rem >= w.obs_len, f = rem - pp * w.obs_len, p = player < 0 ? pp : player;
                    uint32_t op, shift;
                    const int wi = wire_entry(w, p, f, op, shift);
                    v[e] = wire_value(w, p, f, op, shift, op == kWireConst ? 0u : __ldg(rows + src * w.words + wi));
                }
            }
            if (++rem == row_len) rem = 0, ++o;
        }
        if (i0 + 4 <= total) *reinterpret_cast<float4*>(obs + i0) = make_float4(v[0], v[1], v[2], v[3]);
        else
#pragma unroll
            for (int e = 0; e < 4; ++e)
                if (i0 + e < total) obs[i0 + e] = v[e];
    }
    if (!reward && !done) return;
    const int rw = (EVG_WIRE_NODE0 + 4 * w.n_nodes + 3 * kGroupLanes) / 4;  // the word of reward[0]
    for (int64_t o = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; o < n_out; o += stride) {
        const int64_t src = index ? __ldg(index + o) : o;
        const bool ok = src >= 0 && src < n_rows;
        const uint32_t* r = rows + (ok ? src : 0) * w.words;
        if (reward) {
            reward[2 * o] = ok ? __uint_as_float(__ldg(r + rw)) : 0.f;
            reward[2 * o + 1] = ok ? __uint_as_float(__ldg(r + rw + 1)) : 0.f;
        }
        if (done) done[o] = ok ? (uint8_t)(__ldg(r) >> 16) : (uint8_t)0;
    }
}

}  // namespace

cudaError_t launch_wire_expand(const WireSrc& w, const uint32_t* rows, int64_t n_rows, const int64_t* index, int64_t n_out, int player,
                               float* obs, float* reward, uint8_t* done, cudaStream_t stream)
{
    if (n_out <= 0) return cudaSuccess;
    const int64_t quads = (n_out * (player < 0 ? 2 : 1) * w.obs_len + 3) / 4;
    const int64_t need = (quads > n_out ? quads : n_out) + kExpandThreads - 1;
    const int64_t blocks = need / kExpandThreads < (1 << 30) ? need / kExpandThreads : (1 << 30);
    evg_wire_expand_kernel<<<(unsigned)blocks, kExpandThreads, 0, stream>>>(w, rows, n_rows, index, n_out, player, obs, reward, done);
    return cudaGetLastError();
}

}  // namespace evg

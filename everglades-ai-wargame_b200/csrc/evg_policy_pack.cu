// evg_policy_pack.cu — the fused policies' weight images packed on the device, sm_100a.
//
// evg_policy_mlp / _ppo / _rppo / _value read their weights as bf16 IMAGES of the shared-memory operand layout (K-major,
// 128-byte swizzle; include/evgsim.h).  evgsim.policy.pack_mlp / pack_ppo / pack_rppo / pack_value build them in numpy on
// the host; this kernel writes the same bytes from the torch parameters where they sit (float32, contiguous, nn.Linear /
// nn.GRU layout), in ONE launch, with no host synchronisation and no allocation, so that a training loop can refresh the images in place
// after every optimiser step (and capture that in a CUDA graph).
//
//   One thread per 16-byte destination chunk: 8 bf16 of one image row, or 4 fp32 of a bias vector.  The chunks are
//   enumerated in destination order (stores coalesce), and found through a small table of blocks, one per torch
//   parameter, passed by value (__grid_constant__).  A block is `pieces` consecutive [rows x cols] images (DQN's chunks
//   of EVG_MLP_CHUNK hidden units, a GRU matrix's three gates) or fp32 segments of `rows` values; piece p starts at
//   source row p * row_step and column p * col_step.  EVERY byte is written, zero padding included, so nothing of an
//   earlier image survives a refresh.
//
// Rounding is __float2bfloat16_rn: round to nearest even, overflow to +-Inf, subnormals kept — bit for bit what
// evgsim.policy.to_bf16_bits does for every non-NaN value.  A NaN stays a NaN (its payload is not specified).
// No tensor cores: it writes well under 1.5 MB (recurrent actor at L = 256).
#include <cuda_bf16.h>

#include "evg_internal.h"

namespace evg {

namespace {

constexpr int kPackThreads = 256;
constexpr int kPackMaxBlocks = 10;  // the recurrent actor: 5 images and 5 bias vectors (its training images: 4 and 3; the
                                    // feed-forward networks' training images: up to 4 and 3)

// Element (r, k) of piece p is source element (gr, gk) = (p * row_step + r, p * col_step + k):
//     r >= valid_rows                          -> 0 (a GRU gate's rows past L, which belong to the next gate)
//     gr < src_rows and gk < src_cols          -> src[gr * src_cols + gk]
//     gk == bias_col and gr < src_rows         -> bias[gr]     (DQN: b1 as input column obs_len, b2 as hidden unit `hidden`)
//     gk == bias_col and gr == one_row         -> 1            (DQN: the hidden unit that is relu(1) = 1)
//     otherwise                                -> 0
// A transposed block (the recurrent actor's training images) holds element (k, r) of that rule at (r, k).
// An fp32 vector is a [rows x 1] column with src_cols = 1.
struct PackBlock {
    void* dst;
    const float* src;
    const float* bias;
    int32_t is_vec;  // 0: bf16 images of [rows x cols] (cols a multiple of 64), 1: fp32 segments of `rows` values
    int32_t transposed;
    int32_t rows, cols, pieces;
    int32_t row_step, col_step, valid_rows;
    int32_t src_rows, src_cols, bias_col, one_row;
    int32_t first;  // index of the block's first 16-byte chunk in the launch
};

struct PackArgs {
    PackBlock b[kPackMaxBlocks];
    int32_t n_blocks, n_chunks;
};

__device__ __forceinline__ float pack_src(const PackBlock& b, int p, int r, int k)
{
    if (b.transposed) {
        const int t = r;
        r = k;
        k = t;
    }
    if (r >= b.valid_rows) return 0.f;
    const int gr = p * b.row_step + r, gk = p * b.col_step + k;
    if (gr < b.src_rows && gk < b.src_cols) return b.src[gr * b.src_cols + gk];
    if (gk == b.bias_col && gr < b.src_rows) return b.bias[gr];
    if (gk == b.bias_col && gr == b.one_row) return 1.f;
    return 0.f;
}

__global__ void __launch_bounds__(kPackThreads) evg_policy_pack_kernel(const __grid_constant__ PackArgs a)
{
    const int c = blockIdx.x * kPackThreads + threadIdx.x;
    if (c >= a.n_chunks) return;
    int i = 0;
    while (i + 1 < a.n_blocks && c >= a.b[i + 1].first) ++i;
    const PackBlock& b = a.b[i];
    const int local = c - b.first;
    uint4 v;
    if (b.is_vec) {
        const int per = b.rows / 4, p = local / per, r = (local - p * per) * 4;
        v.x = __float_as_uint(pack_src(b, p, r, 0));
        v.y = __float_as_uint(pack_src(b, p, r + 1, 0));
        v.z = __float_as_uint(pack_src(b, p, r + 2, 0));
        v.w = __float_as_uint(pack_src(b, p, r + 3, 0));
    } else {
        // chunk -> (piece, 64-column atom, row, 16-byte slot); the slot holds columns 8 * (slot ^ (row % 8)) .. + 7 of
        // the atom (the swizzle of include/evgsim.h)
        const int per = b.rows * b.cols / 8, p = local / per;
        const int o = local - p * per, atom_chunks = b.rows * 8, atom = o / atom_chunks;
        const int r = (o - atom * atom_chunks) / 8, slot = o & 7;
        const int k0 = atom * 64 + ((slot ^ (r & 7)) << 3);
        uint32_t w[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const __nv_bfloat16 lo = __float2bfloat16_rn(pack_src(b, p, r, k0 + 2 * j));
            const __nv_bfloat16 hi = __float2bfloat16_rn(pack_src(b, p, r, k0 + 2 * j + 1));
            w[j] = (uint32_t)__bfloat16_as_ushort(lo) | (uint32_t)__bfloat16_as_ushort(hi) << 16;
        }
        v = make_uint4(w[0], w[1], w[2], w[3]);
    }
    reinterpret_cast<uint4*>(b.dst)[local] = v;
}

PackBlock image(void* dst, const float* src, int rows, int cols, int src_rows, int src_cols)
{
    PackBlock b{};
    b.dst = dst;
    b.src = src;
    b.rows = rows;
    b.cols = cols;
    b.pieces = 1;
    b.valid_rows = rows;
    b.src_rows = src_rows;
    b.src_cols = src_cols;
    b.bias_col = b.one_row = -1;
    return b;
}

PackBlock vec(float* dst, const float* src, int len, int n)
{
    PackBlock b = image(dst, src, len, 1, n, 1);
    b.is_vec = 1;
    return b;
}

// the three gates (r, z, n) of a GRU parameter (torch's [3L x L] / [3L]): pieces L source rows apart, each zero padded
// past its L rows
PackBlock gates(PackBlock b, int latent)
{
    b.pieces = 3;
    b.row_step = latent;
    b.valid_rows = latent;
    return b;
}

cudaError_t launch(PackArgs& a, cudaStream_t stream)
{
    int n = 0;
    for (int i = 0; i < a.n_blocks; ++i) {
        a.b[i].first = n;
        n += a.b[i].pieces * (a.b[i].is_vec ? a.b[i].rows / 4 : a.b[i].rows * a.b[i].cols / 8);
    }
    a.n_chunks = n;
    evg_policy_pack_kernel<<<(n + kPackThreads - 1) / kPackThreads, kPackThreads, 0, stream>>>(a);
    return cudaGetLastError();
}

}  // namespace

cudaError_t launch_pack_mlp(int in_dim, const float* w1, const float* b1, const float* w2, const float* b2, int hidden, int out_dim,
                            void* w1_img, void* w2_img, cudaStream_t stream)
{
    const int n_chunks = (hidden + 1 + EVG_MLP_CHUNK - 1) / EVG_MLP_CHUNK;  // + the hidden unit that carries b2
    PackArgs a{};
    a.n_blocks = 2;
    a.b[0] = image(w1_img, w1, EVG_MLP_CHUNK, EVG_MLP_IN_PAD, hidden, in_dim);  // W1' = [W1 | b1], plus the unit of ones
    a.b[0].pieces = n_chunks;
    a.b[0].row_step = EVG_MLP_CHUNK;
    a.b[0].bias = b1;
    a.b[0].bias_col = in_dim;
    a.b[0].one_row = hidden;
    a.b[1] = image(w2_img, w2, EVG_MLP_OUT_PAD, EVG_MLP_CHUNK, out_dim, hidden);  // W2' = [W2 | b2]
    a.b[1].pieces = n_chunks;
    a.b[1].col_step = EVG_MLP_CHUNK;
    a.b[1].bias = b2;
    a.b[1].bias_col = hidden;
    return launch(a, stream);
}

cudaError_t launch_pack_ppo(int in_dim, const float* w1, const float* b1, const float* w2, const float* b2, const float* w3,
                            const float* b3, const float* w_ih, const float* b_ih, const float* w_hh, const float* b_hh, int latent,
                            int out_dim, void* w1_img, void* w2_img, void* wi_img, void* wh_img, void* w3_img, float* bias,
                            cudaStream_t stream)
{
    const int lp = (latent + 15) / 16 * 16, ka = (latent + 63) / 64 * 64, L = EVG_PPO_MAX_LATENT;
    PackArgs a{};
    a.b[0] = image(w1_img, w1, lp, EVG_PPO_IN_PAD, latent, in_dim);
    a.b[1] = image(w2_img, w2, lp, ka, latent, latent);
    a.b[2] = image(w3_img, w3, EVG_PPO_OUT_PAD, ka, out_dim, latent);
    a.b[3] = vec(bias, b1, L, latent);
    a.b[4] = vec(bias + L, b2, L, latent);
    a.b[5] = vec(bias + 2 * L, b3, EVG_PPO_OUT_PAD, out_dim);
    a.n_blocks = 6;
    if (w_ih) {  // the recurrent actor: its GRU's gates, and their biases behind b3
        float* gb = bias + 2 * L + EVG_PPO_OUT_PAD;
        a.b[6] = gates(image(wi_img, w_ih, lp, ka, 3 * latent, latent), latent);
        a.b[7] = gates(image(wh_img, w_hh, lp, ka, 3 * latent, latent), latent);
        a.b[8] = gates(vec(gb, b_ih, L, 3 * latent), latent);
        a.b[9] = gates(vec(gb + 3 * L, b_hh, L, 3 * latent), latent);
        a.n_blocks = 10;
    }
    return launch(a, stream);
}

cudaError_t launch_pack_rppo_train(const float* w3, const float* b3, const float* w_ih, const float* b_ih, const float* w_hh,
                                   const float* b_hh, int latent, int out_dim, void* wi_img, void* wh_img, void* wht_img, void* w3_img,
                                   float* bias, cudaStream_t stream)
{
    const int lp = (latent + 15) / 16 * 16, ka = (latent + 63) / 64 * 64, L = EVG_PPO_MAX_LATENT;
    PackArgs a{};
    a.b[0] = gates(image(wi_img, w_ih, lp, ka, 3 * latent, latent), latent);
    a.b[1] = gates(image(wh_img, w_hh, lp, ka, 3 * latent, latent), latent);
    a.b[2] = gates(image(wht_img, w_hh, lp, ka, 3 * latent, latent), latent);  // gate g's W_hg^T: (j, i) = w_hh[g L + i][j]
    a.b[2].transposed = 1;
    a.b[3] = image(w3_img, w3, EVG_PPO_OUT_PAD, ka, out_dim, latent);
    a.b[4] = vec(bias, b3, EVG_PPO_OUT_PAD, out_dim);
    a.b[5] = gates(vec(bias + EVG_PPO_OUT_PAD, b_ih, L, 3 * latent), latent);
    a.b[6] = gates(vec(bias + EVG_PPO_OUT_PAD + 3 * L, b_hh, L, 3 * latent), latent);
    a.n_blocks = 7;
    return launch(a, stream);
}

cudaError_t launch_pack_ppo_train(int net, int in_dim, const float* w1, const float* b1, const float* w2, const float* b2, const float* w3,
                                  const float* b3, int latent, int out_dim, void* w1_img, void* w2_img, void* w3_img, void* w2t_img,
                                  float* bias, cudaStream_t stream)
{
    const int lp = (latent + 15) / 16 * 16, ka = (latent + 63) / 64 * 64, L = EVG_PPO_MAX_LATENT;
    PackArgs a{};
    a.b[0] = image(w1_img, w1, lp, EVG_PPO_IN_PAD, latent, in_dim);
    a.b[1] = image(w2_img, w2, lp, ka, latent, latent);
    a.b[2] = image(w2t_img, w2, lp, ka, latent, latent);  // W2^T: (j, i) = w2[i][j]
    a.b[2].transposed = 1;
    a.b[3] = vec(bias, b1, L, latent);
    a.b[4] = vec(bias + L, b2, L, latent);
    a.n_blocks = 5;
    if (net == EVG_PPO_TRAIN_ACTOR) {
        a.b[5] = image(w3_img, w3, EVG_PPO_OUT_PAD, ka, out_dim, latent);
        a.b[6] = vec(bias + 2 * L, b3, EVG_PPO_OUT_PAD, out_dim);
        a.n_blocks = 7;
    } else if (net == EVG_PPO_TRAIN_CRITIC) {
        a.b[5] = image(w3_img, w3, EVG_VALUE_OUT_PAD, ka, 1, latent);
        a.b[6] = vec(bias + 2 * L, b3, EVG_VALUE_OUT_PAD, 1);
        a.n_blocks = 7;
    }
    return launch(a, stream);
}

cudaError_t launch_pack_value(int in_dim, const float* w1, const float* b1, const float* w2, const float* b2, const float* w3,
                              const float* b3, int latent, void* w1_img, void* w2_img, void* w3_img, float* bias, cudaStream_t stream)
{
    const int lp = (latent + 15) / 16 * 16, ka = (latent + 63) / 64 * 64, L = EVG_PPO_MAX_LATENT;
    PackArgs a{};
    a.b[0] = image(w1_img, w1, lp, EVG_PPO_IN_PAD, latent, in_dim);
    a.b[1] = image(w2_img, w2, lp, ka, latent, latent);
    a.b[2] = image(w3_img, w3, EVG_VALUE_OUT_PAD, ka, 1, latent);
    a.b[3] = vec(bias, b1, L, latent);
    a.b[4] = vec(bias + L, b2, L, latent);
    a.b[5] = vec(bias + 2 * L, b3, EVG_VALUE_OUT_PAD, 1);
    a.n_blocks = 6;
    return launch(a, stream);
}

}  // namespace evg

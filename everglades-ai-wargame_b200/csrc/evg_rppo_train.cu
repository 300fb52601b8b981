// evg_rppo_train.cu — the recurrent PPO actor's GRU and action layer for the update, forward and backward, on the
// 5th-generation tensor cores (tcgen05 + TMEM), sm_100a.  Definitions in include/evgsim.h (evg_rppo_train_forward /
// _backward), layout and budget in DESIGN.md §4.13.
//
// Both kernels are the acting kernel's GRU (evg_policy_rppo.cu) without its head and draws: CTA = 512 threads, persistent
// over tiles of 128 rows (TMEM lane i = row i; four threads per row, one per quarter of the 16-column groups), X = bf16(x)
// and H = bf16(h) as K-major swizzled operands in shared memory, a ring of five 16 KB weight slots streamed from L2, and per
// GRU step, per pass over <= 128 hidden units, the same MMAs into the same TMEM columns in the same order:
//     [0, 128) X . W_ir^T + H . W_hr^T   [128, 256) X . W_iz^T + H . W_hz^T   [256, 384) X . W_in^T   [384, 512) H . W_hn^T
// and the gate arithmetic of evg_gru.cuh.  So the backward's recomputed r, u, n, c are the forward's bit for bit.
//
//   Forward, per tile and step k: the passes write h_k (fp32) to d_h; H = bf16(h_k); D3 = H . W3^T (N = 144) into TMEM
//   [0, 144); z_k = D3 + b3 to d_z.  The state is read back from d_h (the row's own thread wrote it), not held in registers.
//   Backward, per tile, k = 7..1: H = bf16(h_{k-1}); the passes recompute the gates and, with g_k from d_g, write
//   dgh_k (fp32, d_dgh), add dgi_k into d_s and g_k u_k into g_{k-1}; then (k > 1) D = bf16(dgh_k) . W_hh over 3L into
//   TMEM [0, Lp): dgh_k is staged into the H region (free: the gates' MMAs have retired) up to four 64-column atoms at a
//   time, against the transposed images W_hg^T, and added into g_{k-1}.  So d_g[k-1] = fl(fl(W3^T dz_{k-1} + g_k u_k) + D).
#include "evg_gru.cuh"
#include "evg_internal.h"
#include "evg_tcgen05.cuh"

namespace evg {

namespace {

constexpr int kMaxL = EVG_PPO_MAX_LATENT;
constexpr int kOutPad = EVG_PPO_OUT_PAD;
constexpr int kSteps = EVG_MAX_ACTIONS;
constexpr int kSlots = 5;
constexpr int kPieceRows = 128;
constexpr int kSlotBytes = kPieceRows * 128;
constexpr int kAtomBytes = kTileM * 128;

// shared-memory biases (float32): b3, then b_ir + b_hr | b_iz + b_hz | b_in | b_hn, as the acting kernel adds them
constexpr int kB3 = 0, kBr = kOutPad, kBz = kBr + kMaxL, kBin = kBz + kMaxL, kBhn = kBin + kMaxL;
constexpr int kBiasFloats = kBhn + kMaxL;
constexpr int kImgBih = kOutPad, kImgBhh = kOutPad + 3 * kMaxL;  // b_ih / b_hh gate g in d_bias at + g * 256

constexpr int kSmX = 0;
constexpr int kSmH = kSmX + (kMaxL / kAtomK) * kAtomBytes;  // bf16(h); in the backward also bf16(dgh), four atoms at a time
constexpr int kSmW = kSmH + (kMaxL / kAtomK) * kAtomBytes;
constexpr int kSmBias = kSmW + kSlots * kSlotBytes;
constexpr int kMaxPieces = kSteps * 2 * 6 * 4 + (kSteps - 1) * 2 * 3 * 4;  // the backward's pieces of a tile at L = 256
constexpr int kSmTab = kSmBias + kBiasFloats * 4;
constexpr int kSmBar = kSmTab + kMaxPieces * 12;
constexpr int kSmBytes = kSmBar + (2 * kSlots + 1) * 8 + 8;
static_assert(kSmH % 1024 == 0 && kSmW % 1024 == 0 && kSmBar % 8 == 0, "operand blocks must be 1024-byte aligned");
static_assert(kSmBytes <= 227 * 1024, "shared memory");
static_assert(kSteps * 2 * (6 * 4 + 2 * 4) <= kMaxPieces, "the forward's pieces of a tile");

constexpr int kTmemZ = 128, kTmemNi = 256, kTmemNh = 384;

struct TrainArgs {
    const float* x;    // [rows][L]
    const float* h0;   // [rows][L]
    const unsigned char* wi;
    const unsigned char* wh;
    const unsigned char* wht;  // backward: gate g's W_hg^T
    const unsigned char* w3;   // forward
    const float* bias;
    float* z;    // forward: [rows][7][out_dim]
    float* h;    // [rows][7][L]: h_1..h_7 (forward writes, backward reads)
    float* g;    // backward: [rows][7][L], W3^T dz_k in, g_k out
    float* dgh;  // backward: [rows][7][3L]
    float* s;    // backward: [rows][3L], sum over k of dgi_k
    int64_t rows;
    int latent, lp, ka, nrb, out_dim;
};

template <bool kBackward>
__global__ void __launch_bounds__(kCtaThreads, 1) evg_rppo_train_kernel(const __grid_constant__ TrainArgs a)
{
    extern __shared__ __align__(1024) unsigned char smem[];
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    uint64_t* full = reinterpret_cast<uint64_t*>(smem + kSmBar);
    uint64_t* empty = full + kSlots;
    uint64_t* done = empty + kSlots;
    float* sb = reinterpret_cast<float*>(smem + kSmBias);
    for (int i = tid; i < kMaxL; i += kCtaThreads) {
        sb[kBr + i] = a.bias[kImgBih + i] + a.bias[kImgBhh + i];
        sb[kBz + i] = a.bias[kImgBih + kMaxL + i] + a.bias[kImgBhh + kMaxL + i];
        sb[kBin + i] = a.bias[kImgBih + 2 * kMaxL + i];
        sb[kBhn + i] = a.bias[kImgBhh + 2 * kMaxL + i];
        if (i < kOutPad) sb[kB3 + i] = a.bias[kB3 + i];
    }
    const uint32_t tmem = cta_setup<2 * kSlots + 1>(tid, full, reinterpret_cast<uint32_t*>(done + 1));
    const int r = (warp & 3) * 32 + lane, quarter = warp >> 2;
    const uint32_t lane_base = tmem + ((uint32_t)((warp & 3) * 32) << 16);
    const int lp = a.lp, ka = a.ka, nrb = a.nrb, latent = a.latent;
    const uint32_t sX = smem_u32(smem + kSmX), sH = smem_u32(smem + kSmH), sW = smem_u32(smem + kSmW);
    const int n_tiles = (int)((a.rows + kTileM - 1) / kTileM);
    const int my_tiles = (int)blockIdx.x < n_tiles ? (n_tiles - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x : 0;
    const int n_atoms = 3 * ka;  // atoms of dgh (backward)
    auto rows_of = [&](int rb) { return lp - kPieceRows * rb < kPieceRows ? lp - kPieceRows * rb : kPieceRows; };

    // the weight pieces of a tile, in issue order: per step its passes (W_i r, z, n then W_h r, z, n, ka atoms each),
    // then W3 (forward: 2 row blocks x ka) or, for k > 1, the carry's W_hg^T (backward: per group of <= 4 dgh atoms, per
    // row block, per atom)
    int per_tile = 0;
    if (tid == 0) {
        auto add = [&](const unsigned char* m, int rows, int rb, int c, int nh) {
            reinterpret_cast<const unsigned char**>(smem + kSmTab)[per_tile] = m + (size_t)c * rows * 128 + (size_t)rb * kPieceRows * 128;
            reinterpret_cast<uint32_t*>(smem + kSmTab + kMaxPieces * 8)[per_tile++] = (uint32_t)(nh * 128);
        };
        for (int step = 0; step < kSteps; ++step) {
            for (int rb = 0; rb < nrb; ++rb)
                for (int q = 0; q < 6; ++q)
                    for (int c = 0; c < ka; ++c) add((q < 3 ? a.wi : a.wh) + (size_t)(q % 3) * ka * lp * 128, lp, rb, c, rows_of(rb));
            if (!kBackward) {
                for (int rb = 0; rb < 2; ++rb)
                    for (int c = 0; c < ka; ++c) add(a.w3, kOutPad, rb, c, rb ? kOutPad - kPieceRows : kPieceRows);
            } else if (step < kSteps - 1) {
                for (int g0 = 0; g0 < n_atoms; g0 += 4)
                    for (int rb = 0; rb < nrb; ++rb)
                        for (int q = g0; q < n_atoms && q < g0 + 4; ++q)
                            add(a.wht + (size_t)(q / ka) * ka * lp * 128, lp, rb, q % ka, rows_of(rb));
            }
        }
        reinterpret_cast<int*>(smem + kSmBar)[2 * (2 * kSlots + 1) + 1] = per_tile;  // the word after the TMEM slot
    }
    __syncthreads();
    per_tile = reinterpret_cast<const int*>(smem + kSmBar)[2 * (2 * kSlots + 1) + 1];
    const int total = my_tiles * per_tile;
    auto load_piece = [&](int s) {
        const int q = s % per_tile;
        bulk_load(smem + kSmW + (s % kSlots) * kSlotBytes, reinterpret_cast<const unsigned char* const*>(smem + kSmTab)[q],
                  reinterpret_cast<const uint32_t*>(smem + kSmTab + kMaxPieces * 8)[q], &full[s % kSlots]);
    };
    // the issuing thread's producer, as the acting kernel's: requests every piece whose slot has retired, up to kSlots
    // ahead of the issue, without blocking
    int s = 0, loaded = 0;
    auto refill = [&]() {
        while (loaded < total && loaded < s + kSlots) {
            const int prev = loaded - kSlots;
            if (prev >= 0 && !mbar_test(&empty[prev % kSlots], (uint32_t)((prev / kSlots) & 1))) break;
            load_piece(loaded++);
        }
    };
    // MMAs of piece s: D[tcol..] (+)= A[:, atom at a_atom, ks K-steps of 16] . piece^T, N = nh
    auto issue = [&](uint32_t tcol, uint32_t a_atom, int ks, int nh, bool accumulate) {
        const int slot = s % kSlots;
        if (loaded == s) {
            mbar_wait(&empty[slot], (uint32_t)(((s - kSlots) / kSlots) & 1));
            load_piece(loaded++);
        }
        mbar_wait(&full[slot], (uint32_t)((s / kSlots) & 1));
        tc_fence_after();
        const uint32_t b_base = sW + (uint32_t)(slot * kSlotBytes), idesc = make_idesc(kTileM, nh);
        for (int kk = 0; kk < ks; ++kk) umma(tmem + tcol, make_desc(a_atom + kk * 32), make_desc(b_base + kk * 32), idesc, accumulate || kk > 0);
        umma_commit(&empty[slot]);
        ++s;
        refill();
    };
    auto ks_of = [&](int c) { return lp / 16 - 4 * c < 4 ? lp / 16 - 4 * c : 4; };
    uint32_t ph = 0;
    auto wait_done = [&]() {
        mbar_wait(done, ph);
        ph ^= 1;
        tc_fence_after();
        if (tid == 0) refill();
    };
    // bf16 of my row's 16-column groups below lp of an fp32 row (zero past L and for a row past the batch) into an operand
    auto stage_row = [&](uint32_t dst_off, const float* src, bool live) {
#pragma unroll 1
        for (int j0 = 16 * quarter; j0 < lp; j0 += 64) {
            float v[16];
#pragma unroll
            for (int e = 0; e < 16; ++e) v[e] = (live && j0 + e < latent) ? src[j0 + e] : 0.f;
#pragma unroll
            for (int q = 0; q < 2; ++q)
                *reinterpret_cast<uint4*>(smem + dst_off + swz_offset(kTileM, r, j0 + 8 * q)) =
                    make_uint4(pack_bf16(v[8 * q], v[8 * q + 1]), pack_bf16(v[8 * q + 2], v[8 * q + 3]),
                               pack_bf16(v[8 * q + 4], v[8 * q + 5]), pack_bf16(v[8 * q + 6], v[8 * q + 7]));
        }
    };
    auto publish = [&]() {  // make the generic-proxy shared-memory writes visible to the tensor core
        fence_async_smem();
        tc_fence_before();
        __syncthreads();
    };
    auto issue_gates = [&](int rb) {
        if (tid == 0) {
            tc_fence_after();
            const int nh = rows_of(rb);
            for (int g = 0; g < 3; ++g)
                for (int c = 0; c < ka; ++c) issue(128 * g, sX + c * kAtomBytes, ks_of(c), nh, c > 0);
            for (int g = 0; g < 3; ++g)
                for (int c = 0; c < ka; ++c) issue(g == 2 ? kTmemNh : 128 * g, sH + c * kAtomBytes, ks_of(c), nh, g < 2 || c > 0);
            umma_commit(done);
        }
        wait_done();
    };

    if (tid == 0) refill();
    for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        const int64_t row0 = (int64_t)tile * kTileM, my_row = row0 + r;
        const bool live = my_row < a.rows;
        const size_t lat = (size_t)latent;
        const float* h0row = a.h0 + my_row * lat;
        float* hrow = a.h + my_row * kSteps * lat;  // h_k of my row at hrow + (k - 1) L
        stage_row(kSmX, a.x + my_row * lat, live);
        if (!kBackward) stage_row(kSmH, h0row, live);
        publish();
#pragma unroll 1
        for (int it = 0; it < kSteps; ++it) {
            const int k = kBackward ? kSteps - it : it + 1;  // the GRU step, 1..7
            const float* hprev = k == 1 ? h0row : hrow + (k - 2) * lat;
            if (kBackward) {
                stage_row(kSmH, hprev, live);
                publish();
            }
#pragma unroll 1
            for (int rb = 0; rb < nrb; ++rb) {
                issue_gates(rb);
#pragma unroll 1
                for (int i = 0; i < 4; ++i) {
                    const int j0 = 16 * (quarter + 4 * i);
                    if ((i >> 1) != rb || j0 >= lp) continue;
                    const uint32_t col = lane_base + (uint32_t)(j0 - kPieceRows * rb);
#pragma unroll
                    for (int g4 = 0; g4 < 4; ++g4) {
                        uint32_t vr[4], vz[4], vn[4], vh[4];
                        tmem_ld4(col + 4 * g4, vr);
                        tmem_ld4(col + kTmemZ + 4 * g4, vz);
                        tmem_ld4(col + kTmemNi + 4 * g4, vn);
                        tmem_ld4(col + kTmemNh + 4 * g4, vh);
                        tmem_wait_ld();
#pragma unroll
                        for (int e = 0; e < 4; ++e) {
                            const int j = j0 + 4 * g4 + e;
                            if (!live || j >= latent) continue;
                            const GruGates q = gru_gates(__uint_as_float(vr[e]), __uint_as_float(vz[e]), __uint_as_float(vn[e]),
                                                         __uint_as_float(vh[e]), sb[kBr + j], sb[kBz + j], sb[kBin + j], sb[kBhn + j]);
                            const float hp = hprev[j];
                            if (!kBackward) {
                                hrow[(k - 1) * lat + j] = gru_state(q, hp);
                            } else {
                                // g_k: W3^T dz_k plus the carry from step k + 1, added into d_g[k - 1] by step k + 1
                                float* grow = a.g + my_row * kSteps * lat;
                                const float gk = grow[(k - 1) * lat + j];
                                const float dn = gk * (1.f - q.u), dan = dn * (1.f - q.n * q.n);
                                const float dau = gk * (hp - q.n) * (q.u * (1.f - q.u));
                                const float dar = dan * q.c * (q.r * (1.f - q.r));
                                float* dg = a.dgh + (my_row * kSteps + (k - 1)) * 3 * lat;
                                dg[j] = dar;
                                dg[lat + j] = dau;
                                dg[2 * lat + j] = dan * q.r;
                                float* srow = a.s + my_row * 3 * lat;
                                srow[j] = k == kSteps ? dar : srow[j] + dar;
                                srow[lat + j] = k == kSteps ? dau : srow[lat + j] + dau;
                                srow[2 * lat + j] = k == kSteps ? dan : srow[2 * lat + j] + dan;
                                if (k > 1) grow[(k - 2) * lat + j] += gk * q.u;
                            }
                        }
                    }
                }
                tc_fence_before();
                __syncthreads();  // the gates are read (and, backward, this pass's dgh is in memory for the staging)
            }
            if (!kBackward) {
                // ---- H = bf16(h_k); z_k = H . W3^T + b3
                stage_row(kSmH, hrow + (k - 1) * lat, live);
                publish();
                if (tid == 0) {
                    tc_fence_after();
                    for (int rb = 0; rb < 2; ++rb)
                        for (int c = 0; c < ka; ++c) issue(kPieceRows * rb, sH + c * kAtomBytes, ks_of(c), rb ? kOutPad - kPieceRows : kPieceRows, c > 0);
                    umma_commit(done);
                }
                wait_done();
                float* zrow = a.z + (my_row * kSteps + (k - 1)) * a.out_dim;
#pragma unroll 1
                for (int i = 0; i < 3; ++i) {
                    const int gi = quarter + 4 * i;
                    if (gi >= kOutPad / 16) continue;
                    uint32_t v[16];
                    tmem_ld16(lane_base + 16 * gi, v);
                    tmem_wait_ld();
#pragma unroll
                    for (int e = 0; e < 16; ++e) {
                        const int j = 16 * gi + e;
                        if (live && j < a.out_dim) zrow[j] = __uint_as_float(v[e]) + sb[kB3 + j];
                    }
                }
                tc_fence_before();
                __syncthreads();  // D3 is read: the next step's gates may overwrite it
            } else if (k > 1) {
                // ---- the carry: D = bf16(dgh_k) . W_hh over 3L (atom q = gate q / ka, columns 64 (q % ka) ..) into [0, Lp)
                const float* dg = a.dgh + (my_row * kSteps + (k - 1)) * 3 * lat;
#pragma unroll 1
                for (int g0 = 0; g0 < n_atoms; g0 += 4) {
                    const int n_group = n_atoms - g0 < 4 ? n_atoms - g0 : 4;
#pragma unroll 1
                    for (int q = g0; q < g0 + n_group; ++q) {
                        const int gate = q / ka, c = q % ka;
#pragma unroll 1
                        for (int j0 = 16 * quarter; j0 < 64; j0 += 64) {  // my 16 columns of the atom
                            float v[16];
#pragma unroll
                            for (int e = 0; e < 16; ++e) {
                                const int j = 64 * c + j0 + e;
                                v[e] = (live && j < latent) ? dg[gate * lat + j] : 0.f;
                            }
#pragma unroll
                            for (int hq = 0; hq < 2; ++hq)
                                *reinterpret_cast<uint4*>(smem + kSmH + (q - g0) * kAtomBytes + swz_offset(kTileM, r, j0 + 8 * hq)) =
                                    make_uint4(pack_bf16(v[8 * hq], v[8 * hq + 1]), pack_bf16(v[8 * hq + 2], v[8 * hq + 3]),
                                               pack_bf16(v[8 * hq + 4], v[8 * hq + 5]), pack_bf16(v[8 * hq + 6], v[8 * hq + 7]));
                        }
                    }
                    publish();
                    if (tid == 0) {
                        tc_fence_after();
                        for (int rb = 0; rb < nrb; ++rb)
                            for (int q = g0; q < g0 + n_group; ++q)
                                issue(kPieceRows * rb, sH + (q - g0) * kAtomBytes, ks_of(q % ka), rows_of(rb), q > 0);
                        umma_commit(done);
                    }
                    wait_done();  // the group's MMAs have retired: the staging region may be rewritten
                }
                float* grow = a.g + (my_row * kSteps + (k - 2)) * lat;
#pragma unroll 1
                for (int j0 = 16 * quarter; j0 < lp; j0 += 64) {
                    uint32_t v[16];
                    tmem_ld16(lane_base + j0, v);
                    tmem_wait_ld();
#pragma unroll
                    for (int e = 0; e < 16; ++e)
                        if (live && j0 + e < latent) grow[j0 + e] += __uint_as_float(v[e]);
                }
                tc_fence_before();
                __syncthreads();  // the carry is read: the next step's gates may overwrite it
            }
        }
    }
    cta_teardown(tid, tmem);
}

TrainArgs train_args(int64_t n_rows, int latent, int out_dim, const float* x, const float* h0, const void* wi_img, const void* wh_img,
                     const float* bias, float* h)
{
    TrainArgs a{};
    a.x = x;
    a.h0 = h0;
    a.wi = reinterpret_cast<const unsigned char*>(wi_img);
    a.wh = reinterpret_cast<const unsigned char*>(wh_img);
    a.bias = bias;
    a.h = h;
    a.rows = n_rows;
    a.latent = latent;
    a.out_dim = out_dim;
    a.lp = (latent + 15) / 16 * 16;
    a.ka = (latent + kAtomK - 1) / kAtomK;
    a.nrb = (a.lp + kPieceRows - 1) / kPieceRows;
    return a;
}

}  // namespace

cudaError_t launch_rppo_train_forward(int64_t n_rows, int latent, int out_dim, const float* x, const float* h0, const void* wi_img,
                                      const void* wh_img, const void* w3_img, const float* bias, float* z, float* h, int sm_count,
                                      cudaStream_t stream)
{
    TrainArgs a = train_args(n_rows, latent, out_dim, x, h0, wi_img, wh_img, bias, h);
    a.w3 = reinterpret_cast<const unsigned char*>(w3_img);
    a.z = z;
    return launch_persistent(evg_rppo_train_kernel<false>, n_rows, sm_count, kSmBytes, stream, a);
}

cudaError_t launch_rppo_train_backward(int64_t n_rows, int latent, int out_dim, const float* x, const float* h0, const float* h,
                                       const void* wi_img, const void* wh_img, const void* wht_img, const float* bias, float* g,
                                       float* dgh, float* s, int sm_count, cudaStream_t stream)
{
    TrainArgs a = train_args(n_rows, latent, out_dim, x, h0, wi_img, wh_img, bias, const_cast<float*>(h));
    a.wht = reinterpret_cast<const unsigned char*>(wht_img);
    a.g = g;
    a.dgh = dgh;
    a.s = s;
    return launch_persistent(evg_rppo_train_kernel<true>, n_rows, sm_count, kSmBytes, stream, a);
}

cudaError_t set_rppo_train_smem()
{
    cudaError_t e = cudaSuccess;
    for (auto* kernel : {evg_rppo_train_kernel<false>, evg_rppo_train_kernel<true>})
        if (e == cudaSuccess) e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmBytes);
    return e;
}

}  // namespace evg

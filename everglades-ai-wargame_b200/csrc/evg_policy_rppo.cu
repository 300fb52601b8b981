// evg_policy_rppo.cu — PPO's recurrent actor of the policy-in-the-loop path on the 5th-generation tensor cores (tcgen05 +
// TMEM), sm_100a, with its 7 draws fused behind it and its GRU state carried across turns.
//
// The network is the reference's actor with use_recurrent (agents/PPO/ActorCritic.py:33-60, act :79-105;
// tools/policy_rollout.py: RecurrentActor), 1 <= L <= 256:
//     x = tanh(W2 tanh(W1 obs + b1) + b2)                                  the action head, once per turn
//     for k = 0..6:  h = GRUCell(x, h)   (gate order r, z, n as torch.nn.GRU's weight_ih_l0 / weight_hh_l0)
//                    probs_k = softmax(tanh(W3 h + b3)),  idx_k = one draw from probs_k (with replacement)
// h starts at 0 when the match's resident record is at turn 0 (a fresh reset or an automatic one) and is read from / written
// back to d_hidden (float32 [rows][L]) otherwise.  Action row k = (idx_k / div, idx_k % mod).
//
//   CTA = 512 threads, persistent over tiles of 128 rows (TMEM lane i = row i; four threads per row, one per quarter of
//   the 16-column groups).  Shared memory: X (bf16 [128 x Lp], the head's activations, then x for all 7 steps), H (bf16
//   [128 x Lp]: the observation tile during the head, then bf16(h), the MMA operand), a ring of five 16 KB weight slots
//   and the fp32 biases.  Every weight matrix is streamed from L2 in pieces of <= 128 rows x one 64-column swizzle atom
//   (a contiguous sub-block of the [R x K] images of include/evgsim.h); piece s of the CTA's sequence goes to slot s % 5,
//   requested (without the issuing thread waiting for it) as soon as the MMAs of the piece before it in that slot have
//   retired, so the next phase's first pieces land under an epilogue or the sampling.
//   Per tile:   D = A . W1^T -> X = bf16(tanh(D + b1));   D = X . W2^T -> X = bf16(tanh(D + b2));   H = bf16(h0)
//   Per step, per pass over <= 128 hidden units (one pass for Lp <= 128, two above), TMEM columns
//       [0, 128) r:  X . W_ir^T + H . W_hr^T      [128, 256) z:  X . W_iz^T + H . W_hz^T
//       [256, 384)   X . W_in^T                   [384, 512)     H . W_hn^T
//   then the gate epilogue updates the fp32 state h (the thread that reads a (row, 16-column group) of the gates owns that
//   part of h: units below 128 in registers for all 7 steps, units 128.. in the CTA's own rows of d_hidden).  H is
//   rewritten only after the last pass's MMAs have retired (the second pass still reads the old H).  D3 = H . W3^T (N = 144) in columns [0, 144); all 512 threads turn
//   it into e = exp(tanh(D3 + b3)) and p = e / sum e (the row's four threads add their partial sums in a fixed order)
//   in TMEM columns [256, 400); one thread per row then makes the draw, whose two ascending sums are sequential.  W_i x is recomputed every step: 3L fp32 of it per row do not fit in TMEM
//   beside the gate accumulators.
//
// Draw k of row (match m, player p), g = env_base + m, turn t and episode e read from the match's record: the tape's domain
// 3 (DESIGN.md §2), w[0..3] = philox(g, t, p, 3 | e << 8), w[4..7] = philox(g, t, p | 1 << 8, 3 | e << 8),
// u_k = (w[k] >> 8) * 2^-24 — the uniforms of evg_policy_ppo.  T = fp32 sum of p_k in ascending j, x = u_k * T, the draw
// is the first j whose ascending fp32 prefix exceeds x (none, through rounding: the last j): tests/ppo_sampling.py's
// ppo_sample(probs_k, [u_k]).
#include "evg_internal.h"
#include "evg_tcgen05.cuh"

namespace evg {

namespace {

constexpr int kInPad = EVG_PPO_IN_PAD;      // input features, padded (obs_len < 128)
constexpr int kMaxL = EVG_PPO_MAX_LATENT;   // latent width bound: 4 swizzle atoms of X / H
constexpr int kOutPad = EVG_PPO_OUT_PAD;    // outputs, padded to a multiple of 16 (132 -> 144)
constexpr int kSlots = 5;
constexpr int kPieceRows = 128;             // rows of a weight piece (and hidden units of a GRU pass)
constexpr int kSlotBytes = kPieceRows * 128;

// shared-memory biases (float32): b1 | b2 | b3 as in the image, then b_ir + b_hr | b_iz + b_hz | b_in | b_hn
constexpr int kB1 = 0, kB2 = kMaxL, kB3 = 2 * kMaxL, kBr = 2 * kMaxL + kOutPad, kBz = kBr + kMaxL, kBin = kBz + kMaxL, kBhn = kBin + kMaxL;
constexpr int kBiasFloats = kBhn + kMaxL;
constexpr int kImgBih = 2 * kMaxL + kOutPad, kImgBhh = kImgBih + 3 * kMaxL;  // b_ih / b_hh in d_bias, gate g at + g * 256

constexpr int kSmX = 0;                                         // 4 atoms x [128 rows x 128 B]
constexpr int kSmH = kSmX + (kMaxL / kAtomK) * kTileM * 128;    // 4 atoms; the observation tile (2 atoms) during the head
constexpr int kSmW = kSmH + (kMaxL / kAtomK) * kTileM * 128;    // kSlots slots of kSlotBytes
constexpr int kSmBias = kSmW + kSlots * kSlotBytes;
constexpr int kSmRed = kSmBias + kBiasFloats * 4;               // float32 [4][128]: the quarters' partial sums of e
constexpr int kMaxPieces = 2 * 2 + 2 * 4 + EVG_MAX_ACTIONS * (2 * 6 * 4 + 2 * 4);  // weight pieces of a tile at L = 256
constexpr int kSmTab = kSmRed + 4 * kTileM * 4;                 // the tile's pieces: source [kMaxPieces] (8 B), bytes (4 B)
constexpr int kSmBar = kSmTab + kMaxPieces * 12;                // full[kSlots], empty[kSlots], mma-done, TMEM base
constexpr int kSmBytes = kSmBar + (2 * kSlots + 1) * 8 + 8;
static_assert(kSmH % 1024 == 0 && kSmW % 1024 == 0 && kSlotBytes % 1024 == 0 && kSmBar % 8 == 0, "operand blocks must be 1024-byte aligned");
static_assert(kSmBytes <= 227 * 1024, "shared memory");

constexpr int kTmemZ = 128, kTmemNi = 256, kTmemNh = 384;  // r at 0; D1 / D2 / D3 at 0, e / p at kTmemE
constexpr int kTmemE = 256;

struct RppoArgs : ActorArgs {
    const unsigned char* wi;
    const unsigned char* wh;
    float* hidden;
    float* hidden_in;  // [rows][L]: the state each row started this call from (null: not written)
    int latent, ka, nrb;
};

__device__ __forceinline__ float sigmoid(float v) { return __frcp_rn(1.f + expf(-v)); }  // = 1 / (1 + e^-v), correctly rounded

// kWire: the observations are wire rows (ws), else float32
// kExtra: a.logp / a.hidden_in may be written (the instantiation without them is the kernel as it was before they
//         existed: the draw loop's stores of T and p_j slowed the call that does not ask for them by 4-10 %)
template <bool kWire, bool kExtra>
__global__ void __launch_bounds__(kCtaThreads, 1) evg_policy_rppo_kernel(const __grid_constant__ RppoArgs a, const __grid_constant__ WireSrc ws)
{
    extern __shared__ __align__(1024) unsigned char smem[];
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    uint64_t* full = reinterpret_cast<uint64_t*>(smem + kSmBar);  // [s]: slot s landed
    uint64_t* empty = full + kSlots;                              // [s]: the MMAs reading slot s retired
    uint64_t* done = empty + kSlots;                              // a phase's MMAs retired
    float* sb = reinterpret_cast<float*>(smem + kSmBias);
    float* red = reinterpret_cast<float*>(smem + kSmRed);
    for (int i = tid; i < kMaxL; i += kCtaThreads) {
        sb[kB1 + i] = a.bias[kB1 + i];
        sb[kB2 + i] = a.bias[kB2 + i];
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
    const int n_tiles = (int)((a.rows + kTileM - 1) / kTileM);  // < 2^31: a batch of 2^38 rows does not fit in memory
    const int my_tiles = (int)blockIdx.x < n_tiles ? (n_tiles - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x : 0;
    // the CTA's weight pieces: per tile W1 (nrb x 2 atoms), W2 (nrb x ka), then per step and pass W_i r, z, n and W_h r,
    // z, n (ka atoms each), then W3 (2 row blocks x ka)
    const int n1 = 2 * nrb, n2 = nrb * ka, n_pass = 6 * ka, n_step = nrb * n_pass + 2 * ka;
    const int per_tile = n1 + n2 + EVG_MAX_ACTIONS * n_step;
    const int total = my_tiles * per_tile;  // pieces of this CTA: < 2^31 for any batch that fits in memory

    // the source and size of every piece of a tile, decoded once per CTA: the producer only looks them up
    for (int q0 = tid; q0 < per_tile; q0 += kCtaThreads) {
        int q = q0, rows, rb, c;
        const unsigned char* m;
        if (q < n1) {
            m = a.w1, rows = lp, rb = q >> 1, c = q & 1;
        } else if ((q -= n1) < n2) {
            m = a.w2, rows = lp, rb = q / ka, c = q % ka;
        } else if ((q = (q - n2) % n_step) < nrb * n_pass) {
            rb = q / n_pass, q %= n_pass;
            const int gate = (q % (3 * ka)) / ka;
            m = (q < 3 * ka ? a.wi : a.wh) + (size_t)gate * ka * lp * 128, rows = lp, c = q % ka;
        } else {
            q -= nrb * n_pass;
            m = a.w3, rows = kOutPad, rb = q / ka, c = q % ka;
        }
        const int nh = rows - kPieceRows * rb < kPieceRows ? rows - kPieceRows * rb : kPieceRows;
        reinterpret_cast<const unsigned char**>(smem + kSmTab)[q0] = m + (size_t)c * rows * 128 + (size_t)rb * kPieceRows * 128;
        reinterpret_cast<uint32_t*>(smem + kSmTab + kMaxPieces * 8)[q0] = (uint32_t)(nh * 128);
    }
    __syncthreads();
    auto load_piece = [&](int s) {
        const int q = s % per_tile;
        bulk_load(smem + kSmW + (s % kSlots) * kSlotBytes, reinterpret_cast<const unsigned char* const*>(smem + kSmTab)[q],
                  reinterpret_cast<const uint32_t*>(smem + kSmTab + kMaxPieces * 8)[q], &full[s % kSlots]);
    };
    // the issuing thread's producer: `loaded` pieces requested so far, `s` issued.  refill() requests, without blocking,
    // every piece whose slot's previous piece has retired, up to kSlots ahead of the issue; it runs after each issue and
    // after each phase's MMAs have retired (all slots free), so the next phase's pieces land under the epilogue
    int s = 0, loaded = 0;
    auto refill = [&]() {
        while (loaded < total && loaded < s + kSlots) {
            const int prev = loaded - kSlots;  // the piece that used the slot last (issued: prev < s)
            if (prev >= 0 && !mbar_test(&empty[prev % kSlots], (uint32_t)((prev / kSlots) & 1))) break;
            load_piece(loaded++);
        }
    };
    // MMAs of piece s: D[tcol..] (+)= A[:, 64 c ..] . piece^T, N = nh
    auto issue = [&](uint32_t tcol, uint32_t a_base, int c, int nh, int k_cols, bool accumulate) {
        const int slot = s % kSlots;
        if (loaded == s) {  // not requested yet: its slot's previous piece must retire first
            mbar_wait(&empty[slot], (uint32_t)(((s - kSlots) / kSlots) & 1));
            load_piece(loaded++);
        }
        mbar_wait(&full[slot], (uint32_t)((s / kSlots) & 1));
        tc_fence_after();
        const uint32_t b_base = sW + (uint32_t)(slot * kSlotBytes), idesc = make_idesc(kTileM, nh);
        const int ks = k_cols / 16 - 4 * c < 4 ? k_cols / 16 - 4 * c : 4;
        for (int kk = 0; kk < ks; ++kk)
            umma(tmem + tcol, make_desc(a_base + c * (kTileM * 128) + kk * 32), make_desc(b_base + kk * 32), idesc, accumulate || kk > 0);
        umma_commit(&empty[slot]);
        ++s;
        refill();
    };
    uint32_t ph = 0;
    auto wait_done = [&]() {
        mbar_wait(done, ph);
        ph ^= 1;
        tc_fence_after();
        if (tid == 0) refill();
    };
    auto rows_of = [&](int rb) { return lp - kPieceRows * rb < kPieceRows ? lp - kPieceRows * rb : kPieceRows; };
    // the fp32 state h of my row, columns j = 16 (quarter + 4 i) + [0, 16): units below 128 (i = 0, 1) in registers for all 7
    // steps of a tile; units 128..255 (i = 2, 3, only when L > 128) in my row of d_hidden itself, which the CTA owns for the
    // whole call (64 registers of state would not fit beside the rest at 512 threads).  Padding units (L <= j < Lp) and the
    // rows past a partial tile read as 0.
    float hs[2][16] = {};
    float* hrow = nullptr;
    bool live = false;
    // group i's 16 values of h: every load issued before any is used (one round trip for the part in d_hidden)
    auto h_load = [&](int i, float (&v)[16]) {
#pragma unroll
        for (int e = 0; e < 16; ++e) {
            const int j = 16 * (quarter + 4 * i) + e;
            v[e] = i < 2 ? hs[i & 1][e] : (live && j < latent) ? hrow[j] : 0.f;
        }
    };
    auto h_keep = [&](int i, const float (&v)[16]) {
#pragma unroll
        for (int e = 0; e < 16; ++e) {
            const int j = 16 * (quarter + 4 * i) + e;
            if (i < 2) hs[i & 1][e] = v[e];
            else if (live && j < latent) hrow[j] = v[e];
        }
    };
    auto h_to_smem = [&](int i, const float (&v)[16]) {  // H = bf16(h) of group i
        const int j0 = 16 * (quarter + 4 * i);
#pragma unroll
        for (int g = 0; g < 2; ++g)
            *reinterpret_cast<uint4*>(smem + kSmH + swz_offset(kTileM, r, j0 + 8 * g)) =
                make_uint4(pack_bf16(v[8 * g], v[8 * g + 1]), pack_bf16(v[8 * g + 2], v[8 * g + 3]), pack_bf16(v[8 * g + 4], v[8 * g + 5]),
                           pack_bf16(v[8 * g + 6], v[8 * g + 7]));
    };
    // H = bf16(h) for groups i < i_end, then make H visible to the tensor core
    auto store_h = [&](int i_end) {
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            if (i >= i_end || 16 * (quarter + 4 * i) >= lp) continue;
            float v[16];
            h_load(i, v);
            h_to_smem(i, v);
        }
        fence_async_smem();
        tc_fence_before();
        __syncthreads();
    };

    if (tid == 0) refill();
    for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        const int64_t row0 = (int64_t)tile * kTileM;
        const int nrows = a.rows - row0 < kTileM ? (int)(a.rows - row0) : kTileM;
        // ---- the observation tile -> bf16 into H; h0 of my row into registers (0 at turn 0)
        {
            Stager<kWire, false> obs_tile;
            obs_tile.load(tid, a.obs, row0, a.rows, a.in_dim, a.player, ws);
            obs_tile.store(tid, smem + kSmH, a.in_dim, a.player, ws);
        }
        fence_async_smem();
        const int64_t my_row = row0 + r;
        const int64_t my_env = actor_row(a, my_row).env;
        live = r < nrows;
        hrow = a.hidden + my_row * latent;
        const bool fresh = !live || a.records[my_env * a.rec_words + kRecTurn] == 0;
        float* hin = (kExtra && a.hidden_in && live) ? a.hidden_in + my_row * latent : nullptr;  // h0 of my row, written before it is overwritten
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int e = 0; e < 16; ++e) {
                const int j = 16 * (quarter + 4 * i) + e;
                if (i < 2) {
                    hs[i][e] = (!fresh && j < latent) ? hrow[j] : 0.f;
                    if (hin && j < latent) hin[j] = hs[i][e];
                } else if (fresh && live && j < latent) {
                    hrow[j] = 0.f;
                }
            }
        if (hin)  // units 128.. (L > 128), zeroed above for a fresh row: groups 16 (quarter + 8) and 16 (quarter + 12)
#pragma unroll 1
            for (int j = 16 * (quarter + 8); j < latent; j += j % 16 == 15 ? 49 : 1) hin[j] = hrow[j];
        tc_fence_before();
        __syncthreads();
        // ---- the action head
        if (tid == 0) {
            tc_fence_after();
            for (int rb = 0; rb < nrb; ++rb)
                for (int c = 0; c < 2; ++c) issue(kPieceRows * rb, sH, c, rows_of(rb), kInPad, c > 0);
            umma_commit(done);
        }
        wait_done();
        epilogue_tanh_bias(smem + kSmX, lane_base, sb + kB1, r, quarter, lp);
        if (tid == 0) {
            tc_fence_after();
            for (int rb = 0; rb < nrb; ++rb)
                for (int c = 0; c < ka; ++c) issue(kPieceRows * rb, sX, c, rows_of(rb), lp, c > 0);
            umma_commit(done);
        }
        wait_done();
        epilogue_tanh_bias(smem + kSmX, lane_base, sb + kB2, r, quarter, lp);  // X = x for the 7 steps (layer 2 has retired)
        store_h(4);               // H = bf16(h0) (layer 1 has retired: the observations are read)
#pragma unroll 1
        for (int k = 0; k < EVG_MAX_ACTIONS; ++k) {
            // ---- one GRU step, in passes over <= 128 hidden units
#pragma unroll 1
            for (int rb = 0; rb < nrb; ++rb) {
                if (tid == 0) {
                    tc_fence_after();
                    const int nh = rows_of(rb);
                    for (int g = 0; g < 3; ++g)
                        for (int c = 0; c < ka; ++c) issue(128 * g, sX, c, nh, lp, c > 0);
                    for (int g = 0; g < 3; ++g)
                        for (int c = 0; c < ka; ++c) issue(g == 2 ? kTmemNh : 128 * g, sH, c, nh, lp, g < 2 || c > 0);
                    umma_commit(done);
                }
                wait_done();
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    const int j0 = 16 * (quarter + 4 * i);
                    if ((i >> 1) != rb || j0 >= lp) continue;
                    const uint32_t col = lane_base + (uint32_t)(j0 - kPieceRows * rb);
                    float hv[16];
                    h_load(i, hv);
#pragma unroll
                    for (int g = 0; g < 4; ++g) {
                        uint32_t vr[4], vz[4], vn[4], vh[4];
                        tmem_ld4(col + 4 * g, vr);
                        tmem_ld4(col + kTmemZ + 4 * g, vz);
                        tmem_ld4(col + kTmemNi + 4 * g, vn);
                        tmem_ld4(col + kTmemNh + 4 * g, vh);
                        tmem_wait_ld();
#pragma unroll
                        for (int e = 0; e < 4; ++e) {
                            const int j = j0 + 4 * g + e;
                            const float rr = sigmoid(__uint_as_float(vr[e]) + sb[kBr + j]);
                            const float zz = sigmoid(__uint_as_float(vz[e]) + sb[kBz + j]);
                            const float nn = tanhf((__uint_as_float(vn[e]) + sb[kBin + j]) + rr * (__uint_as_float(vh[e]) + sb[kBhn + j]));
                            hv[4 * g + e] = (1.f - zz) * nn + zz * hv[4 * g + e];
                        }
                    }
                    h_keep(i, hv);
                    if (rb == nrb - 1) h_to_smem(i, hv);  // every MMA reading H has retired
                }
                tc_fence_before();
                __syncthreads();  // the gates are read: the next pass may overwrite them
            }
            store_h(2 * (nrb - 1));  // the earlier pass's part of H (the last pass's epilogue wrote its own)
            // ---- D3 = H . W3^T, e = exp(tanh(D3 + b3)) back into TMEM
            if (tid == 0) {
                tc_fence_after();
                for (int rb = 0; rb < 2; ++rb)
                    for (int c = 0; c < ka; ++c) issue(kPieceRows * rb, sH, c, rb ? kOutPad - kPieceRows : kPieceRows, lp, c > 0);
                umma_commit(done);
            }
            wait_done();
            // all four threads of a row: e over my 16-column groups, the row's sum in a fixed order (my partial sums
            // through shared memory, quarters 0..3), then p = e / sum over e
            {
                float part = 0.f;
#pragma unroll
                for (int i = 0; i < 3; ++i) {
                    const int gi = quarter + 4 * i;
                    if (gi >= kOutPad / 16) continue;
                    uint32_t v[16];
                    tmem_ld16(lane_base + 16 * gi, v);
                    tmem_wait_ld();
#pragma unroll
                    for (int e = 0; e < 16; ++e) {
                        const int j = 16 * gi + e;
                        const float ev = j < a.out_dim ? expf(tanhf(__uint_as_float(v[e]) + sb[kB3 + j])) : 0.f;
                        part += ev;
                        v[e] = __float_as_uint(ev);
                    }
                    tmem_st16(lane_base + kTmemE + 16 * gi, v);
                }
                red[quarter * kTileM + r] = part;
                tmem_wait_st();
                __syncthreads();
                const float sum = ((red[r] + red[kTileM + r]) + red[2 * kTileM + r]) + red[3 * kTileM + r];
                float* gp = (a.probs && live) ? a.probs + (my_row * EVG_MAX_ACTIONS + k) * a.out_dim : nullptr;
#pragma unroll
                for (int i = 0; i < 3; ++i) {
                    const int gi = quarter + 4 * i;
                    if (gi >= kOutPad / 16) continue;
                    uint32_t v[16];
                    tmem_ld16(lane_base + kTmemE + 16 * gi, v);
                    tmem_wait_ld();
#pragma unroll
                    for (int e = 0; e < 16; ++e) {
                        const int j = 16 * gi + e;
                        const float pj = __uint_as_float(v[e]) / sum;
                        v[e] = __float_as_uint(pj);
                        if (gp && j < a.out_dim) gp[j] = pj;
                    }
                    tmem_st16(lane_base + kTmemE + 16 * gi, v);
                }
            }
            tmem_wait_st();
            tc_fence_before();
            __syncthreads();
            tc_fence_after();
            // ---- the draw: one thread per row (warps 0-3 = TMEM lanes 0-127, whole warps for tcgen05.ld): T and the
            // prefix walk are the sampler's sequential ascending sums
            if (warp < 4) {
                const int n_groups = (a.out_dim + 15) / 16;
                float total = 0.f;
#pragma unroll 1
                for (int gi = 0; gi < n_groups; ++gi) {
                    uint32_t v[16];
                    tmem_ld16(lane_base + kTmemE + 16 * gi, v);
                    tmem_wait_ld();
#pragma unroll
                    for (int e = 0; e < 16; ++e) total += __uint_as_float(v[e]);  // p = 0 past out_dim adds nothing
                }
                const uint32_t turn = live ? a.records[my_env * a.rec_words + kRecTurn] : 0u;
                const uint32_t episode = live ? a.records[my_env * a.rec_words + kRecEpisode] : 0u;
                const ActorRow me{my_env, actor_row(a, my_row).player};  // (my_env kept: 128 registers without spills)
                uint32_t w[4];
                draw_block(a, me, turn, episode, k >> 2, w);
                const uint32_t wk = (k & 3) == 0 ? w[0] : (k & 3) == 1 ? w[1] : (k & 3) == 2 ? w[2] : w[3];
                const float x = draw_uniform(wk) * total;
                // T and p of the drawn j wait for the log-probability in red[r] and red[kTileM + r] (free until the next
                // step's partial sums), not in registers: this loop runs at the kernel's register bound
                if (kExtra) red[r] = total;
                float c = 0.f;
                int sel = -1;
#pragma unroll 1
                for (int gi = 0; gi < n_groups; ++gi) {
                    uint32_t v[16];
                    tmem_ld16(lane_base + kTmemE + 16 * gi, v);
                    tmem_wait_ld();
#pragma unroll
                    for (int e = 0; e < 16; ++e) {
                        const int j = 16 * gi + e;
                        if (j < a.out_dim) {
                            c += __uint_as_float(v[e]);
                            if (kExtra && sel < 0 && (x < c || j == a.out_dim - 1)) red[kTileM + r] = __uint_as_float(v[e]);
                            if (sel < 0 && x < c) sel = j;
                        }
                    }
                    if (__all_sync(0xFFFFFFFFu, sel >= 0)) break;
                }
                if (sel < 0) sel = a.out_dim - 1;
                if (live) {
                    if (kExtra && a.logp) a.logp[my_row * EVG_MAX_ACTIONS + k] = logf(red[kTileM + r] / red[r]);
                    if (a.idx) a.idx[my_row * EVG_MAX_ACTIONS + k] = sel;
                    store_action(a, me, k, sel);
                }
            }
            tc_fence_before();
            __syncthreads();  // D3 and p are read: the next step's gates may overwrite them
        }
        // ---- the final h of my row (units 128.. are in place already)
        if (live) {
#pragma unroll
            for (int i = 0; i < 2; ++i)
#pragma unroll
                for (int e = 0; e < 16; ++e) {
                    const int j = 16 * (quarter + 4 * i) + e;
                    if (j < latent) hrow[j] = hs[i][e];
                }
        }
    }
    cta_teardown(tid, tmem);
}

}  // namespace

cudaError_t launch_policy_rppo(const Tables& t, const uint32_t* records, const void* obs, int64_t n_envs, int player, const void* w1_img,
                               const void* w2_img, const void* wi_img, const void* wh_img, const void* w3_img, const float* bias, int latent,
                               int out_dim, int div, int mod, float* hidden, float* hidden_in, int8_t* actions, int64_t* idx, float* probs,
                               float* logp, int sm_count, cudaStream_t stream, const WireSrc* wire)
{
    RppoArgs a;
    static_cast<ActorArgs&>(a) =
        actor_args(t, records, obs, n_envs, player, w1_img, w2_img, w3_img, bias, latent, out_dim, div, mod, actions, idx, probs, logp);
    a.wi = reinterpret_cast<const unsigned char*>(wi_img);
    a.wh = reinterpret_cast<const unsigned char*>(wh_img);
    a.hidden = hidden;
    a.hidden_in = hidden_in;
    a.latent = latent;
    a.ka = (latent + kAtomK - 1) / kAtomK;
    a.nrb = (a.lp + kPieceRows - 1) / kPieceRows;
    const bool extra = logp || hidden_in;
    auto* kernel = wire ? (extra ? evg_policy_rppo_kernel<true, true> : evg_policy_rppo_kernel<true, false>)
                        : (extra ? evg_policy_rppo_kernel<false, true> : evg_policy_rppo_kernel<false, false>);
    return launch_persistent(kernel, a.rows, sm_count, kSmBytes, stream, a, wire ? *wire : WireSrc{});
}

cudaError_t set_policy_rppo_smem()
{
    cudaError_t e = cudaSuccess;
    for (auto* kernel : {evg_policy_rppo_kernel<false, false>, evg_policy_rppo_kernel<true, false>, evg_policy_rppo_kernel<false, true>,
                         evg_policy_rppo_kernel<true, true>})
        if (e == cudaSuccess) e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmBytes);
    return e;
}

}  // namespace evg

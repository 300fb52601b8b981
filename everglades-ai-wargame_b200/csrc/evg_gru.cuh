// evg_gru.cuh — the GRU gate arithmetic of the recurrent actor, shared by the acting kernel (evg_policy_rppo.cu) and the
// update's forward and backward (evg_rppo_train.cu), so that the gates the backward recomputes are bit for bit the ones
// the forward used, and both are the acting kernel's.
//
// From the fp32 accumulators of one hidden unit (torch.nn.GRU's gate order r, z, n): ar = X W_ir^T + H W_hr^T (one
// accumulator), az likewise, an = X W_in^T, ah = H W_hn^T, and the fp32 biases br = b_ir + b_hr, bz = b_iz + b_hz, bin,
// bhn:
//     r = sigmoid(ar + br),  u = sigmoid(az + bz),  c = ah + bhn,  n = tanh((an + bin) + r c),  h' = (1 - u) n + u h
#pragma once

namespace evg {

__device__ __forceinline__ float sigmoid(float v) { return __frcp_rn(1.f + expf(-v)); }  // = 1 / (1 + e^-v), correctly rounded

struct GruGates {
    float r, u, n, c;
};

__device__ __forceinline__ GruGates gru_gates(float ar, float az, float an, float ah, float br, float bz, float bin, float bhn)
{
    GruGates g;
    g.r = sigmoid(ar + br);
    g.u = sigmoid(az + bz);
    g.n = tanhf((an + bin) + g.r * (ah + bhn));
    g.c = ah + bhn;
    return g;
}

__device__ __forceinline__ float gru_state(const GruGates& g, float h) { return (1.f - g.u) * g.n + g.u * h; }

}  // namespace evg

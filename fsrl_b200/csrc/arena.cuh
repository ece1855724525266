// The flat fp32 parameter arena every learner keeps its networks in.  One network in -> H -> H -> out
// occupies
//     w1t[D][H] | b1[H] | w2t[H][H] | b2[H] | w3t[H][out] | b3[out] | extra[n_extra]
// of theta (grad / adam_m / adam_v use the same layout; extra holds e.g. the actor's log-sigma), and
// the backward kernels read W2 from an out-major copy w2n[o][k] = w2t[k][o], the "W2 mirror".
#pragma once
#include "common.cuh"
#include "fsrl_b200.h"

namespace fsrl {

// offsets (floats) of the parts of one network, relative to its start
struct NetLayout {
    long long w1, b1, w2, b2, w3, b3, extra, size;
    __host__ __device__ __forceinline__ NetLayout(int D, int H, int out, int n_extra)
        : w1(0), b1((long long)D * H), w2(b1 + H), b2(w2 + (long long)H * H), w3(b2 + H),
          b3(w3 + (long long)H * out), extra(b3 + out), size(extra + n_extra) {}
    __host__ __device__ __forceinline__ explicit NetLayout(const fsrl_netref_t& r) : NetLayout(r.D, r.H, r.out, r.n_extra) {}
};

// torch.optim.Adam scalars of one optimiser step (python doubles -> f32 at the op):
// w1 = 1 - beta1, b2 = beta2, w2 = 1 - beta2, bc2s = sqrt(1 - beta2^t), neg_step = -lr / (1 - beta1^t)
struct AdamStep {
    float w1, b2, w2, bc2s, eps, neg_step;
};

// torch's single-tensor Adam update of one element, in torch's operation order
__device__ __forceinline__ float adam_one(float p, float g, float& m, float& v, const AdamStep& a) {
    m = m + a.w1 * (g - m);                 // exp_avg.lerp_(grad, 1 - beta1)
    v = v * a.b2 + (a.w2 * g) * g;          // exp_avg_sq.mul_(beta2).addcmul_(grad, grad, 1 - beta2)
    const float denom = sqrtf(v) / a.bc2s + a.eps;
    return p + (a.neg_step * m) / denom;    // param.addcdiv_(exp_avg, denom, value=-step_size)
}

// W2 work is done in 32 x 32 tiles by 256-thread blocks: tile t of an H x H block covers rows
// [k0, k0 + 32) and columns [o0, o0 + 32) of w2t; thread (lx = tid % 32, ly = tid / 32) handles
// column o0 + lx of rows k0 + ly + 8 q, q < 4.
__device__ __forceinline__ void w2_tile_origin(int t, int H, int& k0, int& o0) {
    k0 = (t / (H / 32)) * 32;
    o0 = (t % (H / 32)) * 32;
}

// Once every thread has put its values of the tile into tile[kk][oo] = w2t[k0 + kk][o0 + oo], writes
// the tile transposed into the mirror w2n (coalesced on both sides).
__device__ __forceinline__ void w2_tile_store_mirror(const float (&tile)[32][33], float* w2n, int H, int k0, int o0) {
    __syncthreads();
    const int lx = threadIdx.x % 32, ly = threadIdx.x / 32;
#pragma unroll
    for (int q = 0; q < 4; ++q) {
        const int oo = ly + 8 * q;
        w2n[(size_t)(o0 + oo) * H + k0 + lx] = tile[lx][oo];
    }
}

// w2n[i][o][k] = w2t[i][k][o] for n nets of hidden width H in one launch (engine.cu)
struct W2Mirrors {
    const float* w2t[FSRL_ENG_MAX_NETS];
    float* w2n[FSRL_ENG_MAX_NETS];
};
int w2_mirror(const W2Mirrors& m, int n, int H, cudaStream_t s);

}  // namespace fsrl

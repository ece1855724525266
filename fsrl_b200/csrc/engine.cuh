// Shared declarations of the generic MLP engine (engine.cu) for the kernels built on top of it
// (cpo.cu): scratch-slot views, input gathering, weight-gradient roles.
#pragma once
#include "arena.cuh"
#include "mlp.cuh"

#define ENG_DISPATCH_H(Hv, ...)                                   \
    switch (Hv) {                                                 \
        case 64: { constexpr int HH = 64; __VA_ARGS__; } break;   \
        case 128: { constexpr int HH = 128; __VA_ARGS__; } break; \
        case 256: { constexpr int HH = 256; __VA_ARGS__; } break; \
        default: { constexpr int HH = 512; __VA_ARGS__; } break;  \
    }


namespace fsrl {

constexpr int EDOUT_LD = 16;

struct EngView {
    Mlp3 m;
    const float* w2n;
    float *g_w1t, *g_b1, *g_w2t, *g_b2, *g_w3t, *g_b3, *g_extra;
    float *s_h1, *s_h2, *s_dz1, *s_dz2, *s_out, *s_dout, *s_dx;
};

__host__ __device__ inline size_t eng_slot_floats(int H, int bmax) {
    return (size_t)bmax * (4 * (size_t)H + 2 * EDOUT_LD + FSRL_ENG_DX_LD);
}

// gradient pointers of a net whose gradient (layout L) starts at g
__device__ __forceinline__ void eng_grad_view(EngView& v, float* g, const NetLayout& L) {
    v.g_w1t = g + L.w1; v.g_b1 = g + L.b1; v.g_w2t = g + L.w2; v.g_b2 = g + L.b2;
    v.g_w3t = g + L.w3; v.g_b3 = g + L.b3; v.g_extra = g + L.extra;
}

__device__ __forceinline__ EngView eng_view(const fsrl_engine_t& e, const fsrl_netref_t& n) {
    EngView v;
    const int H = n.H, D = n.D, out = n.out;
    const NetLayout L(n);
    const float* th = e.theta + n.off;
    v.m.w1t = th + L.w1; v.m.b1 = th + L.b1; v.m.w2t = th + L.w2;
    v.m.b2 = th + L.b2;  v.m.w3t = th + L.w3; v.m.b3 = th + L.b3;
    eng_grad_view(v, e.grad + n.off, L);
    v.m.in = D; v.m.H = H; v.m.out = out;
    v.w2n = e.w2n + n.w2n_off;
    float* sc = e.scratch + (size_t)n.slot * eng_slot_floats(H, e.bmax);
    const size_t bh = (size_t)e.bmax * H;
    v.s_h1 = sc; v.s_h2 = sc + bh; v.s_dz1 = sc + 2 * bh; v.s_dz2 = sc + 3 * bh;
    v.s_out = sc + 4 * bh; v.s_dout = v.s_out + (size_t)e.bmax * EDOUT_LD;
    v.s_dx = v.s_dout + (size_t)e.bmax * EDOUT_LD;
    return v;
}

// input row = concat(xa[ia ? ia[row] : row][0..Da), xb[ib ? ib[row] : row][0..Db))
__device__ __forceinline__ float eng_input(const fsrl_eng_input_t& in, long long row, int k) {
    if (k < in.Da) {
        const long long r = in.ia ? (long long)in.ia[row] : row;
        return in.xa[r * in.Da + k];
    }
    const long long r = in.ib ? (long long)in.ib[row] : row;
    return in.xb[r * in.Db + (k - in.Da)];
}

// Role pointers let the same kernel serve plain gradients (defaults: the net's own scratch) and
// the two halves of a Hessian-vector product (cpo.cu): dW2t = L2^T G2, db2 = colsum(G2),
// dW1t = X^T G1, db1 = colsum(G1), dW3t = L3^T G3, db3/extra = colsum(G3).  A null role skips
// that part.  gridDim.z > 1 splits the rows; partial tiles are then combined with atomics
// (the destination must have been zeroed or hold the value to accumulate onto).
struct WgradRoles {
    const float *L2, *G2, *G1, *L3, *G3;
    float* dst;           // gradient base of the net (same layout as theta); null = e.grad + off
    int bias2, bias3;     // emit db2 / (db3, dextra)
    int parts;            // bit 0: W2 block, bit 1: layer 1 (W1, b1), bit 2: layer 3 (W3)
};


int eng_wgrad_roles(const fsrl_engine_t* e, const fsrl_netlist_t* nl, const fsrl_eng_input_t* in, long long B,
                    int accumulate, float* norm_sq, const WgradRoles& roles, cudaStream_t s);

}  // namespace fsrl

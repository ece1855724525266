// Generic minibatch MLP engine: forward (optionally saving activations), backward from a
// caller-supplied head gradient (optionally producing the input gradient), weight gradients,
// Adam on a set of networks and Polyak averaging -- the building blocks from which the
// SAC-/DDPG-Lagrangian and CPO updates are assembled (sac.cu, cpo.cu).  PPO keeps its fully
// fused kernels (ppo.cu).
//
// Replaces the eager autograd calls of the reference's off-policy learners:
//   /root/reference/fsrl/policy/sac_lag.py:185-258, ddpg_lag.py:165-213 (critics_loss /
//   policy_loss forward+backward+optimizer.step), base_policy.py:220-224 (soft_update).
//
// Every kernel processes up to FSRL_ENG_MAX_NETS networks of equal hidden width in one launch
// (blockIdx.y selects the net), reading parameters from the flat arena and exchanging
// activations through an L2-resident scratch slot per network.
#include "engine.cuh"

namespace fsrl {

// ---------------------------------------------------------------------------------------------
// forward
// ---------------------------------------------------------------------------------------------
template <int H>
__global__ void __launch_bounds__(MLP_TPB)
eng_forward_kernel(const fsrl_engine_t e, const fsrl_netlist_t nl, const fsrl_eng_input_t in, int B, int save) {
    using TT = MlpTile<H>;
    extern __shared__ __align__(16) float smem[];
    const fsrl_netref_t nr = nl.nets[blockIdx.y];
    const EngView nv = eng_view(e, nr);
    const MlpSmem<H> sm(smem, nr.D, nr.out);
    const int tid = threadIdx.x;
    const int r0 = blockIdx.x * TT::R;
    const int inp = TT::in_pad(nr.D);
    for (int i = tid; i < TT::R * inp; i += MLP_TPB) {
        const int r = i / inp, k = i % inp;
        sm.x[i] = (r0 + r < B && k < nr.D) ? eng_input(in, r0 + r, k) : 0.f;
    }
    __syncthreads();
    mlp_hidden_forward<H>(nv.m, sm);
    float out[MLP_MAX_OUT];
    mlp_head_forward<H>(nv.m, sm, out);
    const int r = tid / TT::PARTS, part = tid % TT::PARTS;
    if (part == 0 && r0 + r < B) {
#pragma unroll
        for (int j = 0; j < EDOUT_LD; j += 4)
            *reinterpret_cast<float4*>(nv.s_out + (size_t)(r0 + r) * EDOUT_LD + j) =
                make_float4(j < nr.out ? out[j] : 0.f, j + 1 < nr.out ? out[j + 1] : 0.f,
                            j + 2 < nr.out ? out[j + 2] : 0.f, j + 3 < nr.out ? out[j + 3] : 0.f);
    }
    if (save) {
        for (int el = tid; el < TT::R * (H / 4); el += MLP_TPB) {
            const int row = el / (H / 4), k4 = (el % (H / 4)) * 4;
            if (r0 + row < B) {
                *reinterpret_cast<float4*>(nv.s_h1 + (size_t)(r0 + row) * H + k4) =
                    *reinterpret_cast<const float4*>(sm.h1 + (size_t)row * TT::LDA + k4);
                *reinterpret_cast<float4*>(nv.s_h2 + (size_t)(r0 + row) * H + k4) =
                    *reinterpret_cast<const float4*>(sm.h2 + (size_t)row * TT::LDA + k4);
            }
        }
    }
}

// ---------------------------------------------------------------------------------------------
// backward: dz2 = (dout . W3^T) * relu'(h2); dz1 = (dz2 . W2) * relu'(h1); dx = dz1 . W1^T
// ---------------------------------------------------------------------------------------------
template <int H>
__global__ void __launch_bounds__(MLP_TPB)
eng_backward_kernel(const fsrl_engine_t e, const fsrl_netlist_t nl, int B, int want_dx) {
    using TT = MlpTile<H>;
    extern __shared__ __align__(16) float smem[];
    const fsrl_netref_t nr = nl.nets[blockIdx.y];
    const EngView nv = eng_view(e, nr);
    const int tid = threadIdx.x;
    const int r0 = blockIdx.x * TT::R;
    // smem: h1[R][LDA] | dz[R][LDA] | wst | w3s[H][out] | sdout[R][16]
    float* h1 = smem;
    float* dz = h1 + (size_t)TT::R * TT::LDA;
    float* wst = dz + (size_t)TT::R * TT::LDA;
    float* w3s = wst + TT::stage_floats();
    float* sdout = w3s + (size_t)H * MLP_MAX_OUT;
    const int out = nr.out;
    for (int i = tid; i < H * out; i += MLP_TPB) w3s[i] = __ldg(nv.m.w3t + i);
    for (int i = tid; i < TT::R * EDOUT_LD; i += MLP_TPB) {
        const int r = i / EDOUT_LD;
        sdout[i] = (r0 + r < B) ? nv.s_dout[(size_t)(r0 + r) * EDOUT_LD + (i % EDOUT_LD)] : 0.f;
    }
    __syncthreads();
    for (int el = tid; el < TT::R * (H / 4); el += MLP_TPB) {
        const int row = el / (H / 4), k4 = (el % (H / 4)) * 4;
        const bool ok = r0 + row < B;
        float a4[4] = {0.f, 0.f, 0.f, 0.f};
        for (int j = 0; j < out; ++j) {
            const float g = sdout[row * EDOUT_LD + j];
#pragma unroll
            for (int q = 0; q < 4; ++q) a4[q] = fmaf(g, w3s[(size_t)(k4 + q) * out + j], a4[q]);
        }
        float4 hv = make_float4(0.f, 0.f, 0.f, 0.f), h1v = hv;
        if (ok) {
            hv = *reinterpret_cast<const float4*>(nv.s_h2 + (size_t)(r0 + row) * H + k4);
            h1v = *reinterpret_cast<const float4*>(nv.s_h1 + (size_t)(r0 + row) * H + k4);
        }
        const float4 g4 = make_float4(hv.x > 0.f ? a4[0] : 0.f, hv.y > 0.f ? a4[1] : 0.f,
                                      hv.z > 0.f ? a4[2] : 0.f, hv.w > 0.f ? a4[3] : 0.f);
        *reinterpret_cast<float4*>(dz + (size_t)row * TT::LDA + k4) = g4;
        *reinterpret_cast<float4*>(h1 + (size_t)row * TT::LDA + k4) = h1v;
        if (ok) *reinterpret_cast<float4*>(nv.s_dz2 + (size_t)(r0 + row) * H + k4) = g4;
    }
    float c[TT::MT][TT::NT][4];
    tc_init_bias<H>(c, nullptr);
    tc_gemm<H>(c, dz, TT::LDA, H, nv.w2n, wst, false);
    // dz1 -> global scratch, and into smem (reusing dz) for the optional input gradient
    tc_foreach<H>(c, [&](int row, int col, float v0, float v1) {
        const float2 hv = *reinterpret_cast<const float2*>(h1 + (size_t)row * TT::LDA + col);
        const float2 g = make_float2(hv.x > 0.f ? v0 : 0.f, hv.y > 0.f ? v1 : 0.f);
        *reinterpret_cast<float2*>(dz + (size_t)row * TT::LDA + col) = g;
        if (r0 + row < B) *reinterpret_cast<float2*>(nv.s_dz1 + (size_t)(r0 + row) * H + col) = g;
    });
    if (want_dx) {
        __syncthreads();
        // dx[r][d] = sum_o dz1[r][o] * w1t[d][o]: one warp per (row, d) pair, lanes over o
        const int lane = tid & 31, warp = tid >> 5;
        for (int p = warp; p < TT::R * nr.D; p += MLP_TPB / 32) {
            const int row = p / nr.D, d = p % nr.D;
            float s = 0.f;
            for (int o = lane; o < H; o += 32) s = fmaf(dz[(size_t)row * TT::LDA + o], __ldg(nv.m.w1t + (size_t)d * H + o), s);
            s = warp_sum(s);
            if (lane == 0 && r0 + row < B) nv.s_dx[(size_t)(r0 + row) * FSRL_ENG_DX_LD + d] = s;
        }
    }
}

// ---------------------------------------------------------------------------------------------
// weight gradients (same tiling as ppo_wgrad): grad (+)= ...
// ---------------------------------------------------------------------------------------------
constexpr int EWG_TPB = 128, EWG_TK = 32, EWG_TO = 64, EWG_RC = 32;

__device__ __forceinline__ float eng_block_sum_128(float v, float* red) {
    v = warp_sum(v);
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    __syncthreads();
    if (lane == 0) red[w] = v;
    __syncthreads();
    return red[0] + red[1] + red[2] + red[3];
}

template <int H>
__global__ void __launch_bounds__(EWG_TPB)
eng_wgrad_kernel(const fsrl_engine_t e, const fsrl_netlist_t nl, const fsrl_eng_input_t in, int Btot,
                 int accumulate, float* norm_sq, const WgradRoles roles) {
    constexpr int NTK = H / EWG_TK, NTO = H / EWG_TO, NT = NTK * NTO;
    __shared__ __align__(16) float sL[EWG_RC][EWG_TO];
    __shared__ __align__(16) float sG[EWG_RC][EWG_TO];
    __shared__ float s_red[4];
    const int tid = threadIdx.x;
    const fsrl_netref_t nr = nl.nets[blockIdx.y];
    EngView nv = eng_view(e, nr);
    const bool split = gridDim.z > 1;
    // row range of this split
    const long long rows_per = (((long long)Btot + gridDim.z - 1) / gridDim.z + EWG_RC - 1) / EWG_RC * EWG_RC;
    const long long row_lo = (long long)blockIdx.z * rows_per;
    const int B = (int)((row_lo >= Btot) ? 0 : ((Btot - row_lo < rows_per) ? (Btot - row_lo) : rows_per));
    if (B == 0) return;
    if (roles.dst) eng_grad_view(nv, roles.dst, NetLayout(nr.D, H, nr.out, nr.n_extra));
    nv.s_h1 = const_cast<float*>(roles.L2 ? roles.L2 : nv.s_h1) + (size_t)row_lo * H;
    nv.s_dz2 = const_cast<float*>(roles.G2 ? roles.G2 : nv.s_dz2) + (size_t)row_lo * H;
    nv.s_dz1 = const_cast<float*>(roles.G1 ? roles.G1 : nv.s_dz1) + (size_t)row_lo * H;
    nv.s_h2 = const_cast<float*>(roles.L3 ? roles.L3 : nv.s_h2) + (size_t)row_lo * H;
    nv.s_dout = const_cast<float*>(roles.G3 ? roles.G3 : nv.s_dout) + (size_t)row_lo * EDOUT_LD;
    const int bx = blockIdx.x;
    const int nchunk = (B + EWG_RC - 1) / EWG_RC;
    const float beta = (accumulate && !split) ? 1.f : 0.f;
    float sq = 0.f;
    auto emit = [&](float* gp, float v) {       // write / accumulate / atomically combine one value
        if (split) { atomicAdd(gp, v); return v; }
        v += beta * (*gp);
        *gp = v;
        return v;
    };
    if (bx < NT) {
        if (!(roles.parts & 1)) return;
        const int k0 = (bx / NTO) * EWG_TK, o0 = (bx % NTO) * EWG_TO;
        const int tk = tid / 16, to = tid % 16;
        const bool do_bias = (k0 == 0) && roles.bias2;
        float acc[4][4];
#pragma unroll
        for (int i = 0; i < 4; ++i) { acc[i][0] = acc[i][1] = acc[i][2] = acc[i][3] = 0.f; }
        float bsum = 0.f;
        float4 pl[2], pg[4];
        auto prefetch = [&](int rb) {
#pragma unroll
            for (int q = 0; q < 2; ++q) {
                const int f = tid + q * EWG_TPB, rr = f / 8, cc = (f % 8) * 4;
                pl[q] = (rb + rr < B) ? __ldcg(reinterpret_cast<const float4*>(nv.s_h1 + (size_t)(rb + rr) * H + k0 + cc))
                                      : make_float4(0.f, 0.f, 0.f, 0.f);
            }
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                const int f = tid + q * EWG_TPB, rr = f / 16, cc = (f % 16) * 4;
                pg[q] = (rb + rr < B) ? __ldcg(reinterpret_cast<const float4*>(nv.s_dz2 + (size_t)(rb + rr) * H + o0 + cc))
                                      : make_float4(0.f, 0.f, 0.f, 0.f);
            }
        };
        prefetch(0);
        for (int ch = 0; ch < nchunk; ++ch) {
#pragma unroll
            for (int q = 0; q < 2; ++q) {
                const int f = tid + q * EWG_TPB;
                *reinterpret_cast<float4*>(&sL[f / 8][(f % 8) * 4]) = pl[q];
            }
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                const int f = tid + q * EWG_TPB;
                *reinterpret_cast<float4*>(&sG[f / 16][(f % 16) * 4]) = pg[q];
            }
            __syncthreads();
            if (ch + 1 < nchunk) prefetch((ch + 1) * EWG_RC);
#pragma unroll 8
            for (int rr = 0; rr < EWG_RC; ++rr) {
                const float4 l = *reinterpret_cast<const float4*>(&sL[rr][4 * tk]);
                const float4 g = *reinterpret_cast<const float4*>(&sG[rr][4 * to]);
                acc[0][0] = fmaf(l.x, g.x, acc[0][0]); acc[0][1] = fmaf(l.x, g.y, acc[0][1]);
                acc[0][2] = fmaf(l.x, g.z, acc[0][2]); acc[0][3] = fmaf(l.x, g.w, acc[0][3]);
                acc[1][0] = fmaf(l.y, g.x, acc[1][0]); acc[1][1] = fmaf(l.y, g.y, acc[1][1]);
                acc[1][2] = fmaf(l.y, g.z, acc[1][2]); acc[1][3] = fmaf(l.y, g.w, acc[1][3]);
                acc[2][0] = fmaf(l.z, g.x, acc[2][0]); acc[2][1] = fmaf(l.z, g.y, acc[2][1]);
                acc[2][2] = fmaf(l.z, g.z, acc[2][2]); acc[2][3] = fmaf(l.z, g.w, acc[2][3]);
                acc[3][0] = fmaf(l.w, g.x, acc[3][0]); acc[3][1] = fmaf(l.w, g.y, acc[3][1]);
                acc[3][2] = fmaf(l.w, g.z, acc[3][2]); acc[3][3] = fmaf(l.w, g.w, acc[3][3]);
            }
            if (do_bias && tid < EWG_TO) {
#pragma unroll 8
                for (int rr = 0; rr < EWG_RC; ++rr) bsum += sG[rr][tid];
            }
            __syncthreads();
        }
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            float* gp = nv.g_w2t + (size_t)(k0 + 4 * tk + i) * H + o0 + 4 * to;
#pragma unroll
            for (int j = 0; j < 4; ++j) { const float v = emit(gp + j, acc[i][j]); sq += v * v; }
        }
        if (do_bias && tid < EWG_TO) { const float v = emit(nv.g_b2 + o0 + tid, bsum); sq += v * v; }
    } else if (bx < NT + NTO) {
        if (!(roles.parts & 2)) return;
        const int D = nr.D;
        const int o0 = (bx - NT) * EWG_TO;
        const int o = tid % EWG_TO, dg = tid / EWG_TO;
        for (int d0 = 0; d0 < D; d0 += 16) {
            float acc[8];
#pragma unroll
            for (int q = 0; q < 8; ++q) acc[q] = 0.f;
            float bsum = 0.f;
            float4 pg[4];
            float px[4];
            auto prefetch = [&](int rb) {
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    const int f = tid + q * EWG_TPB, rr = f / 16, cc = (f % 16) * 4;
                    pg[q] = (rb + rr < B) ? __ldcg(reinterpret_cast<const float4*>(nv.s_dz1 + (size_t)(rb + rr) * H + o0 + cc))
                                          : make_float4(0.f, 0.f, 0.f, 0.f);
                }
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    const int f = tid + q * EWG_TPB, rr = f / 16, dd = d0 + (f % 16);
                    px[q] = (rb + rr < B && dd < D) ? eng_input(in, row_lo + rb + rr, dd) : 0.f;
                }
            };
            prefetch(0);
            for (int ch = 0; ch < nchunk; ++ch) {
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    const int f = tid + q * EWG_TPB;
                    *reinterpret_cast<float4*>(&sG[f / 16][(f % 16) * 4]) = pg[q];
                    sL[f / 16][f % 16] = px[q];
                }
                __syncthreads();
                if (ch + 1 < nchunk) prefetch((ch + 1) * EWG_RC);
#pragma unroll 8
                for (int rr = 0; rr < EWG_RC; ++rr) {
                    const float g = sG[rr][o];
                    const float4 xa4 = *reinterpret_cast<const float4*>(&sL[rr][8 * dg]);
                    const float4 xb4 = *reinterpret_cast<const float4*>(&sL[rr][8 * dg + 4]);
                    acc[0] = fmaf(xa4.x, g, acc[0]); acc[1] = fmaf(xa4.y, g, acc[1]);
                    acc[2] = fmaf(xa4.z, g, acc[2]); acc[3] = fmaf(xa4.w, g, acc[3]);
                    acc[4] = fmaf(xb4.x, g, acc[4]); acc[5] = fmaf(xb4.y, g, acc[5]);
                    acc[6] = fmaf(xb4.z, g, acc[6]); acc[7] = fmaf(xb4.w, g, acc[7]);
                    bsum += g;
                }
                __syncthreads();
            }
#pragma unroll
            for (int q = 0; q < 8; ++q) {
                const int d = d0 + 8 * dg + q;
                if (d < D) { const float v = emit(nv.g_w1t + (size_t)d * H + o0 + o, acc[q]); sq += v * v; }
            }
            if (d0 == 0 && dg == 0) { const float v = emit(nv.g_b1 + o0 + o, bsum); sq += v * v; }
        }
    } else {
        if (!(roles.parts & 4)) return;
        const int out = nr.out;
        const int k0 = (bx - NT - NTO) * EWG_TO;
        const int k = tid % EWG_TO, jg = tid / EWG_TO;
        float acc[8];
#pragma unroll
        for (int q = 0; q < 8; ++q) acc[q] = 0.f;
        float csum = 0.f;
        float4 pg[4];
        float4 pd;
        auto prefetch = [&](int rb) {
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                const int f = tid + q * EWG_TPB, rr = f / 16, cc = (f % 16) * 4;
                pg[q] = (rb + rr < B) ? __ldcg(reinterpret_cast<const float4*>(nv.s_h2 + (size_t)(rb + rr) * H + k0 + cc))
                                      : make_float4(0.f, 0.f, 0.f, 0.f);
            }
            const int rr = tid / 4, cc = (tid % 4) * 4;
            pd = (rb + rr < B) ? __ldcg(reinterpret_cast<const float4*>(nv.s_dout + (size_t)(rb + rr) * EDOUT_LD + cc))
                               : make_float4(0.f, 0.f, 0.f, 0.f);
        };
        prefetch(0);
        for (int ch = 0; ch < nchunk; ++ch) {
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                const int f = tid + q * EWG_TPB;
                *reinterpret_cast<float4*>(&sG[f / 16][(f % 16) * 4]) = pg[q];
            }
            *reinterpret_cast<float4*>(&sL[tid / 4][(tid % 4) * 4]) = pd;
            __syncthreads();
            if (ch + 1 < nchunk) prefetch((ch + 1) * EWG_RC);
#pragma unroll 8
            for (int rr = 0; rr < EWG_RC; ++rr) {
                const float h = sG[rr][k];
                const float4 da = *reinterpret_cast<const float4*>(&sL[rr][8 * jg]);
                const float4 db = *reinterpret_cast<const float4*>(&sL[rr][8 * jg + 4]);
                acc[0] = fmaf(h, da.x, acc[0]); acc[1] = fmaf(h, da.y, acc[1]);
                acc[2] = fmaf(h, da.z, acc[2]); acc[3] = fmaf(h, da.w, acc[3]);
                acc[4] = fmaf(h, db.x, acc[4]); acc[5] = fmaf(h, db.y, acc[5]);
                acc[6] = fmaf(h, db.z, acc[6]); acc[7] = fmaf(h, db.w, acc[7]);
            }
            if (k0 == 0 && tid < EDOUT_LD) {
#pragma unroll 8
                for (int rr = 0; rr < EWG_RC; ++rr) csum += sL[rr][tid];
            }
            __syncthreads();
        }
#pragma unroll
        for (int q = 0; q < 8; ++q) {
            const int j = 8 * jg + q;
            if (j < out) { const float v = emit(nv.g_w3t + (size_t)(k0 + k) * out + j, acc[q]); sq += v * v; }
        }
        if (k0 == 0 && tid < EDOUT_LD && roles.bias3) {
            if (tid < out) { const float v = emit(nv.g_b3 + tid, csum); sq += v * v; }
            else if (nr.n_extra > 0 && tid >= out && tid < out + nr.n_extra) {
                // head-gradient columns [out, out + n_extra) carry d loss / d extra (log-sigma)
                const float v = emit(nv.g_extra + (tid - out), csum); sq += v * v;
            }
        }
    }
    if (norm_sq) {
        const float tot = eng_block_sum_128(sq, s_red);
        if (tid == 0 && tot != 0.f) atomicAdd(norm_sq, tot);
    }
}

// ---------------------------------------------------------------------------------------------
// Adam over a set of nets (torch.optim.Adam arithmetic), optional L2 term, W2 mirror upkeep
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
eng_adam_kernel(const fsrl_engine_t e, const fsrl_netlist_t nl, const AdamStep ad, float gscale, float l2x2,
                const float* norm_sq, float max_norm) {
    __shared__ float tile[32][33];
    const fsrl_netref_t nr = nl.nets[blockIdx.y];
    const int H = nr.H;
    float scale = gscale;
    if (norm_sq && max_norm > 0.f) scale *= fminf(max_norm / (sqrtf(*norm_sq) + 1e-6f), 1.0f);
    const NetLayout L(nr);
    const int n_plain_blocks = (int)((L.size + 255) / 256);
    if ((int)blockIdx.x < n_plain_blocks) {
        const long long j = (long long)blockIdx.x * 256 + threadIdx.x;
        if (j >= L.size || (j >= L.w2 && j < L.b2)) return;
        const long long i = nr.off + j;
        float m = e.adam_m[i], v = e.adam_v[i];
        const float p = e.theta[i];
        const float g = e.grad[i] * scale + l2x2 * p;
        e.theta[i] = adam_one(p, g, m, v, ad);
        e.adam_m[i] = m; e.adam_v[i] = v;
    } else {
        const int tt = blockIdx.x - n_plain_blocks;
        if (tt >= (H / 32) * (H / 32)) return;
        int k0, o0;
        w2_tile_origin(tt, H, k0, o0);
        const long long base = nr.off + L.w2;
        const int lx = threadIdx.x % 32, ly = threadIdx.x / 32;
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const int kk = ly + 8 * q;
            const long long i = base + (long long)(k0 + kk) * H + o0 + lx;
            float m = e.adam_m[i], v = e.adam_v[i];
            float p = e.theta[i];
            const float g = e.grad[i] * scale + l2x2 * p;
            p = adam_one(p, g, m, v, ad);
            e.theta[i] = p; e.adam_m[i] = m; e.adam_v[i] = v;
            tile[kk][lx] = p;
        }
        w2_tile_store_mirror(tile, e.w2n + nr.w2n_off, H, k0, o0);
    }
}

// dst <- tau * src + (1 - tau) * dst over whole nets (soft_update, base_policy.py:220-224);
// keeps the W2 mirror of dst in sync
__global__ void __launch_bounds__(256)
eng_polyak_kernel(const fsrl_engine_t e, const fsrl_netlist_t dst, const fsrl_netlist_t src, float tau) {
    __shared__ float tile[32][33];
    const fsrl_netref_t nd = dst.nets[blockIdx.y], ns = src.nets[blockIdx.y];
    const int H = nd.H;
    const NetLayout L(nd);
    const int n_plain_blocks = (int)((L.size + 255) / 256);
    if ((int)blockIdx.x < n_plain_blocks) {
        const long long j = (long long)blockIdx.x * 256 + threadIdx.x;
        if (j >= L.size || (j >= L.w2 && j < L.b2)) return;
        e.theta[nd.off + j] = tau * e.theta[ns.off + j] + (1.0f - tau) * e.theta[nd.off + j];
    } else {
        const int tt = blockIdx.x - n_plain_blocks;
        if (tt >= (H / 32) * (H / 32)) return;
        int k0, o0;
        w2_tile_origin(tt, H, k0, o0);
        const int lx = threadIdx.x % 32, ly = threadIdx.x / 32;
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const int kk = ly + 8 * q;
            const long long j = L.w2 + (long long)(k0 + kk) * H + o0 + lx;
            const float p = tau * e.theta[ns.off + j] + (1.0f - tau) * e.theta[nd.off + j];
            e.theta[nd.off + j] = p;
            tile[kk][lx] = p;
        }
        w2_tile_store_mirror(tile, e.w2n + nd.w2n_off, H, k0, o0);
    }
}

__global__ void __launch_bounds__(256) w2_mirror_kernel(const __grid_constant__ W2Mirrors mr, int H) {
    __shared__ float tile[32][33];
    int k0, o0;
    w2_tile_origin(blockIdx.x, H, k0, o0);
    const float* src = mr.w2t[blockIdx.y];
    const int lx = threadIdx.x % 32, ly = threadIdx.x / 32;
#pragma unroll
    for (int q = 0; q < 4; ++q) tile[ly + 8 * q][lx] = src[(size_t)(k0 + ly + 8 * q) * H + o0 + lx];
    w2_tile_store_mirror(tile, mr.w2n[blockIdx.y], H, k0, o0);
}

int w2_mirror(const W2Mirrors& m, int n, int H, cudaStream_t s) {
    w2_mirror_kernel<<<dim3((H / 32) * (H / 32), n), 256, 0, s>>>(m, H);
    FSRL_LAUNCH_CHECK();
    return FSRL_OK;
}

static int eng_check(const fsrl_engine_t* e, const fsrl_netlist_t* nl) {
    FSRL_REQUIRE(e && nl, "engine: null descriptor");
    FSRL_REQUIRE(e->theta && e->grad && e->w2n && e->scratch, "engine: null buffer");
    FSRL_REQUIRE(nl->n >= 1 && nl->n <= FSRL_ENG_MAX_NETS, "engine: %d nets in one launch (max %d)", nl->n, FSRL_ENG_MAX_NETS);
    const int H = nl->nets[0].H;
    FSRL_REQUIRE(H == 64 || H == 128 || H == 256 || H == 512, "engine: hidden width %d unsupported", H);
    for (int i = 0; i < nl->n; ++i) {
        FSRL_REQUIRE(nl->nets[i].H == H, "engine: nets of one launch must share the hidden width");
        FSRL_REQUIRE(nl->nets[i].out >= 1 && nl->nets[i].out + nl->nets[i].n_extra <= EDOUT_LD, "engine: head too wide");
        FSRL_REQUIRE(nl->nets[i].D >= 1 && nl->nets[i].D <= FSRL_ENG_DX_LD, "engine: input dim %d unsupported", nl->nets[i].D);
    }
    return FSRL_OK;
}

// largest parameter count of the listed nets (grid size of the per-net element kernels)
static long long max_net_size(const fsrl_netlist_t* nl) {
    long long maxn = 0;
    for (int i = 0; i < nl->n; ++i) {
        const fsrl_netref_t& n = nl->nets[i];
        const long long tot = NetLayout(n).size;
        if (tot > maxn) maxn = tot;
    }
    return maxn;
}

}  // namespace fsrl

using namespace fsrl;

extern "C" size_t fsrl_engine_slot_floats(int H, int bmax) { return eng_slot_floats(H, bmax); }

extern "C" int fsrl_engine_forward(const fsrl_engine_t* e, const fsrl_netlist_t* nl,
                                   const fsrl_eng_input_t* in, int B, int save, void* stream) {
    int rc = eng_check(e, nl);
    if (rc) return rc;
    FSRL_REQUIRE(in && in->xa && B >= 0 && B <= e->bmax, "engine_forward: bad input / B=%d exceeds bmax=%d", B, e->bmax);
    if (B == 0) return FSRL_OK;
    for (int i = 0; i < nl->n; ++i)
        FSRL_REQUIRE(nl->nets[i].D == in->Da + in->Db, "engine_forward: net input dim %d != %d + %d", nl->nets[i].D, in->Da, in->Db);
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    ENG_DISPATCH_H(nl->nets[0].H, {
        using TT = MlpTile<HH>;
        const size_t smem = TT::smem_bytes(in->Da + in->Db);
        FSRL_CUDA(cudaFuncSetAttribute(eng_forward_kernel<HH>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        eng_forward_kernel<HH><<<dim3((B + TT::R - 1) / TT::R, nl->n), MLP_TPB, smem, s>>>(*e, *nl, *in, B, save);
    });
    FSRL_LAUNCH_CHECK();
    return FSRL_OK;
}

extern "C" int fsrl_engine_backward(const fsrl_engine_t* e, const fsrl_netlist_t* nl, int B, int want_dx, void* stream) {
    int rc = eng_check(e, nl);
    if (rc) return rc;
    FSRL_REQUIRE(B >= 0 && B <= e->bmax, "engine_backward: B=%d exceeds bmax=%d", B, e->bmax);
    if (B == 0) return FSRL_OK;
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    ENG_DISPATCH_H(nl->nets[0].H, {
        using TT = MlpTile<HH>;
        const size_t smem = sizeof(float) * (2 * (size_t)TT::R * TT::LDA + TT::stage_floats() + (size_t)HH * MLP_MAX_OUT + (size_t)TT::R * EDOUT_LD);
        FSRL_CUDA(cudaFuncSetAttribute(eng_backward_kernel<HH>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        eng_backward_kernel<HH><<<dim3((B + TT::R - 1) / TT::R, nl->n), MLP_TPB, smem, s>>>(*e, *nl, B, want_dx);
    });
    FSRL_LAUNCH_CHECK();
    return FSRL_OK;
}

namespace fsrl {
// zero the gradient range of the listed nets (needed before a split-K wgrad that does not accumulate)
__global__ void eng_zero_grad_kernel(const fsrl_engine_t e, const fsrl_netlist_t nl, float* dst_override) {
    const fsrl_netref_t nr = nl.nets[blockIdx.y];
    const long long n = NetLayout(nr).size;
    float* g = dst_override ? dst_override : e.grad + nr.off;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) g[i] = 0.f;
}

int eng_wgrad_roles(const fsrl_engine_t* e, const fsrl_netlist_t* nl, const fsrl_eng_input_t* in, long long B,
                    int accumulate, float* norm_sq, const WgradRoles& roles, cudaStream_t s) {
    // split the rows so that every CTA streams <= 4096 rows (keeps all SMs busy on big batches)
    int nsplit = (int)((B + 4095) / 4096);
    if (nsplit < 1) nsplit = 1;
    if (nsplit > 65535) nsplit = 65535;
    if (nsplit > 1) FSRL_REQUIRE(norm_sq == nullptr, "engine_wgrad: norm_sq is not available with split rows");
    const bool partial = roles.parts != 7 || !roles.bias2 || !roles.bias3;
    if (!accumulate && (nsplit > 1 || partial)) {
        // start from zero and let every part accumulate (atomically when the rows are split)
        FSRL_REQUIRE(roles.dst == nullptr || nl->n == 1, "engine_wgrad: dst override needs a single net");
        eng_zero_grad_kernel<<<dim3(64, nl->n), 256, 0, s>>>(*e, *nl, roles.dst);
        ++g_launches;
        accumulate = 1;
    }
    ENG_DISPATCH_H(nl->nets[0].H, {
        const dim3 g((HH / EWG_TK) * (HH / EWG_TO) + 2 * (HH / EWG_TO), nl->n, nsplit);
        eng_wgrad_kernel<HH><<<g, EWG_TPB, 0, s>>>(*e, *nl, *in, (int)B, accumulate, norm_sq, roles);
    });
    FSRL_LAUNCH_CHECK();
    return FSRL_OK;
}
}  // namespace fsrl

extern "C" int fsrl_engine_wgrad(const fsrl_engine_t* e, const fsrl_netlist_t* nl, const fsrl_eng_input_t* in,
                                 int B, int accumulate, float* norm_sq, void* stream) {
    int rc = eng_check(e, nl);
    if (rc) return rc;
    FSRL_REQUIRE(in && in->xa && B >= 0 && B <= e->bmax, "engine_wgrad: bad input / B");
    if (B == 0) return FSRL_OK;
    WgradRoles roles = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, 1, 1, 7};
    return eng_wgrad_roles(e, nl, in, B, accumulate, norm_sq, roles, static_cast<cudaStream_t>(stream));
}

extern "C" int fsrl_engine_adam(const fsrl_engine_t* e, const fsrl_netlist_t* nl, double lr, double beta1,
                                double beta2, double eps, long long step, double grad_scale, double l2_reg,
                                const float* norm_sq, double max_grad_norm, void* stream) {
    int rc = eng_check(e, nl);
    if (rc) return rc;
    FSRL_REQUIRE(e->adam_m && e->adam_v && step >= 1, "engine_adam: missing moments or step < 1");
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    const double bc1 = 1.0 - pow(beta1, (double)step), bc2 = 1.0 - pow(beta2, (double)step);
    const int H = nl->nets[0].H;
    const int blocks = (int)((max_net_size(nl) + 255) / 256) + (H / 32) * (H / 32);
    const AdamStep ad = {(float)(1.0 - beta1), (float)beta2, (float)(1.0 - beta2), (float)sqrt(bc2), (float)eps,
                         (float)(-(lr / bc1))};
    eng_adam_kernel<<<dim3(blocks, nl->n), 256, 0, s>>>(*e, *nl, ad, (float)grad_scale, (float)(2.0 * l2_reg), norm_sq,
                                                        (float)max_grad_norm);
    FSRL_LAUNCH_CHECK();
    return FSRL_OK;
}

extern "C" int fsrl_engine_polyak(const fsrl_engine_t* e, const fsrl_netlist_t* dst, const fsrl_netlist_t* src,
                                  double tau, void* stream) {
    int rc = eng_check(e, dst);
    if (rc) return rc;
    rc = eng_check(e, src);
    if (rc) return rc;
    FSRL_REQUIRE(dst->n == src->n, "polyak: net lists differ in length");
    FSRL_REQUIRE(tau >= 0.0 && tau <= 1.0, "tau should be in [0, 1]");
    const int H = dst->nets[0].H;
    for (int i = 0; i < dst->n; ++i) {
        const fsrl_netref_t& n = dst->nets[i];
        FSRL_REQUIRE(n.D == src->nets[i].D && n.H == src->nets[i].H && n.out == src->nets[i].out, "polyak: shape mismatch");
    }
    const int blocks = (int)((max_net_size(dst) + 255) / 256) + (H / 32) * (H / 32);
    eng_polyak_kernel<<<dim3(blocks, dst->n), 256, 0, static_cast<cudaStream_t>(stream)>>>(*e, *dst, *src, (float)tau);
    FSRL_LAUNCH_CHECK();
    return FSRL_OK;
}

extern "C" int fsrl_engine_sync_mirror(const fsrl_engine_t* e, const fsrl_netlist_t* nl, void* stream) {
    int rc = eng_check(e, nl);
    if (rc) return rc;
    W2Mirrors m = {};
    for (int i = 0; i < nl->n; ++i) {
        const fsrl_netref_t& n = nl->nets[i];
        m.w2t[i] = e->theta + n.off + NetLayout(n).w2;
        m.w2n[i] = e->w2n + n.w2n_off;
    }
    return w2_mirror(m, nl->n, nl->nets[0].H, static_cast<cudaStream_t>(stream));
}

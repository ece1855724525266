// Constrained Policy Optimization on the device: surrogate / KL head gradients, exact
// Hessian-vector products of the mean KL (Pearlmutter R-op through the MLP, not a
// Gauss-Newton approximation), conjugate-gradient vector kernels and line-search evaluation.
//
// Replaces (reference, torch autograd incl. double backward on the CPU):
//   /root/reference/fsrl/policy/cpo.py:163-175  _get_objective / _get_cost_surrogate
//   /root/reference/fsrl/policy/cpo.py:177-182  _MVP  (grad(grad(kl) . v) + damping * v)
//   /root/reference/fsrl/policy/cpo.py:184-204  _conjugate_gradients
//   /root/reference/fsrl/policy/cpo.py:238-254  kl, objective, cost surrogate and their gradients
//   /root/reference/fsrl/policy/cpo.py:313-333  backtracking line search evaluation
//
// The batch stays resident: one forward pass caches h1, h2 and the head output of every row
// in the engine scratch (HBM is 180 GB; c3's 2 M rows x 128 hidden cost 4.9 GB), every later
// gradient / Hessian-vector product re-uses the cache.
//
// R-op (v = tangent direction in parameter space, masks m1 = h1 > 0, m2 = h2 > 0):
//   forward   Rh1 = m1 * (x V1 + c1);  Rh2 = m2 * (Rh1 W2 + h1 V2 + c2);  Rz = Rh2 W3 + h2 V3 + c3
//   head      e = dKL/dz;  Re = d2KL/dz2 Rz + (cross terms with log-sigma) + dKL/dmu * mu'' Rz
//   backward  Rda2 = m2 * (Re W3^T + e V3^T);  Rda1 = m1 * (Rda2 W2^T + da2 V2^T)
//   Hv        W3: Rh2^T e + h2^T Re;  W2: Rh1^T da2 + h1^T Rda2;  W1: x^T Rda1;  biases: column sums
#include "engine.cuh"

namespace fsrl {

constexpr float LOG_SQRT_2PI_C = 0.9189385332046727f;

// ---- per-row head kernel --------------------------------------------------------------------------
// mode: 0 = evaluate sums only, 1 = d objective, 2 = d(-cost_surrogate), 3 = d kl
// sums[0..3] += objective_sum, cost_ratio_sum, kl_sum, (unused); dout rows [N][16]:
// cols [0,A) = d/dz, cols [A,2A) = d/dlog_sigma contributions.
__global__ void cpo_head_kernel(const fsrl_cpo_t d, long long N, int mode, double* __restrict__ sums) {
    __shared__ double red[3][8];
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    double s_obj = 0.0, s_cost = 0.0, s_kl = 0.0;
    if (i < N) {
        const long long r = d.perm ? (long long)d.perm[i] : i;
        const int A = d.A;
        const float invN = 1.0f / (float)N;
        float logp = 0.f, kl = 0.f;
        float mu[8], mup[8], z_[8], sg[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            if (j < A) {
                const float z = d.out[(size_t)i * 16 + j];
                const float t = tanhf(z);
                mu[j] = d.bounded ? d.max_action * t : z;
                mup[j] = d.bounded ? d.max_action * (1.0f - t * t) : 1.0f;
                const float ls = d.log_sigma[j];
                sg[j] = expf(ls);
                z_[j] = (d.act[(size_t)r * A + j] - mu[j]) / sg[j];
                logp += -0.5f * z_[j] * z_[j] - ls - LOG_SQRT_2PI_C;
                // kl_divergence(Normal(mu_old, s_old), Normal(mu, s))  (torch formula)
                const float so = d.std_old[(size_t)r * A + j], mo = d.mean_old[(size_t)r * A + j];
                const float vr = (so / sg[j]) * (so / sg[j]);
                const float t1 = ((mo - mu[j]) / sg[j]) * ((mo - mu[j]) / sg[j]);
                kl += 0.5f * (vr + t1 - 1.0f - logf(vr));
            }
        }
        const float ratio = expf(logp - d.logp_old[r]);
        const float ar = d.adv[r], ac = d.adv[(size_t)d.ld + r];
        s_obj = (double)(ratio * ar);
        s_cost = (double)(ratio * ac);
        s_kl = (double)kl;
        if (mode != 0) {
            float dd[16];
#pragma unroll
            for (int j = 0; j < 16; ++j) dd[j] = 0.f;
            if (mode == 1 || mode == 2) {
                const float gl = (mode == 1 ? ratio * ar : -ratio * ac) * invN;    // d f / d logp
#pragma unroll
                for (int j = 0; j < 8; ++j)
                    if (j < A) { dd[j] = gl * (z_[j] / sg[j]) * mup[j]; dd[A + j] = gl * (z_[j] * z_[j] - 1.0f); }
            } else {
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                    if (j < A) {
                        const float so = d.std_old[(size_t)r * A + j], mo = d.mean_old[(size_t)r * A + j];
                        const float kmu = (mu[j] - mo) / (sg[j] * sg[j]) * invN;
                        const float q = so * so + (mo - mu[j]) * (mo - mu[j]);
                        dd[j] = kmu * mup[j];
                        dd[A + j] = (1.0f - q / (sg[j] * sg[j])) * invN;
                    }
                }
            }
#pragma unroll
            for (int j = 0; j < 16; j += 4)
                *reinterpret_cast<float4*>(d.dout + (size_t)i * 16 + j) = make_float4(dd[j], dd[j + 1], dd[j + 2], dd[j + 3]);
        }
    }
    double v[3] = {s_obj, s_cost, s_kl};
    for (int k = 0; k < 3; ++k) {
        const double t = warp_sum(v[k]);
        if ((threadIdx.x & 31) == 0) red[k][threadIdx.x >> 5] = t;
    }
    __syncthreads();
    if (threadIdx.x < 3) {
        double t = 0.0;
        for (int w = 0; w < (int)(blockDim.x >> 5); ++w) t += red[threadIdx.x][w];
        atomicAdd(sums + threadIdx.x, t);
    }
}

// FOCOPS actor head (reference fsrl/policy/focops.py:188-215):
//   L_i = (KL(new || old)_i - (1/lambda) ratio_i (A^r_i - nu A^c_i)) * 1[KL_i <= eta]   (indicator detached)
// loss = mean_i L_i.  sums[0] += L_i, sums[1] += KL_i, sums[2] += indicator;  dout = d loss / d(z, log sigma).
// d.adv holds the per-minibatch-normalised advantages of the rows in d.perm.
__global__ void focops_head_kernel(const fsrl_cpo_t d, long long N, float inv_lambda, float nu, float eta,
                                   double* __restrict__ sums) {
    __shared__ double red[3][8];
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    double s_loss = 0.0, s_kl = 0.0, s_cnt = 0.0;
    if (i < N) {
        const long long r = d.perm ? (long long)d.perm[i] : i;
        const int A = d.A;
        const float invN = 1.0f / (float)N;
        float logp = 0.f, kl = 0.f;
        float mup[8], z_[8], sg[8], dklmu[8], dklls[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            if (j < A) {
                const float z = d.out[(size_t)i * 16 + j];
                const float t = tanhf(z);
                const float mu = d.bounded ? d.max_action * t : z;
                mup[j] = d.bounded ? d.max_action * (1.0f - t * t) : 1.0f;
                const float ls = d.log_sigma[j];
                sg[j] = expf(ls);
                z_[j] = (d.act[(size_t)r * A + j] - mu) / sg[j];
                logp += -0.5f * z_[j] * z_[j] - ls - LOG_SQRT_2PI_C;
                // kl_divergence(Normal(mu, s), Normal(mu_old, s_old))  (torch formula, p = new, q = old)
                const float so = d.std_old[(size_t)r * A + j], mo = d.mean_old[(size_t)r * A + j];
                const float vr = (sg[j] / so) * (sg[j] / so);
                const float t1 = ((mu - mo) / so) * ((mu - mo) / so);
                kl += 0.5f * (vr + t1 - 1.0f - logf(vr));
                dklmu[j] = (mu - mo) / (so * so);
                dklls[j] = vr - 1.0f;
            }
        }
        const float ratio = expf(logp - d.logp_old[r]);
        const float adv = d.adv[r] - nu * d.adv[(size_t)d.ld + r];
        const float keep = (kl <= eta) ? 1.0f : 0.0f;
        s_loss = (double)((kl - inv_lambda * ratio * adv) * keep);
        s_kl = (double)kl;
        s_cnt = (double)keep;
        float dd[16];
#pragma unroll
        for (int j = 0; j < 16; ++j) dd[j] = 0.f;
        const float gr = -inv_lambda * adv * ratio;          // d L / d logp (before mask and 1/N)
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            if (j < A) {
                dd[j] = keep * invN * (dklmu[j] + gr * (z_[j] / sg[j])) * mup[j];
                dd[A + j] = keep * invN * (dklls[j] + gr * (z_[j] * z_[j] - 1.0f));
            }
        }
#pragma unroll
        for (int j = 0; j < 16; j += 4)
            *reinterpret_cast<float4*>(d.dout + (size_t)i * 16 + j) = make_float4(dd[j], dd[j + 1], dd[j + 2], dd[j + 3]);
    }
    double v[3] = {s_loss, s_kl, s_cnt};
    for (int k = 0; k < 3; ++k) {
        const double t = warp_sum(v[k]);
        if ((threadIdx.x & 31) == 0) red[k][threadIdx.x >> 5] = t;
    }
    __syncthreads();
    if (threadIdx.x < 3) {
        double t = 0.0;
        for (int w = 0; w < (int)(blockDim.x >> 5); ++w) t += red[threadIdx.x][w];
        atomicAdd(sums + threadIdx.x, t);
    }
}

// R-head: Re and the log-sigma Hessian contributions from z, Rz and the tangent of log-sigma
__global__ void cpo_rhead_kernel(const fsrl_cpo_t d, long long N, const float* __restrict__ rz,
                                 const float* __restrict__ vs, float* __restrict__ rdout) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= N) return;
    const long long r = d.perm ? (long long)d.perm[i] : i;
    const int A = d.A;
    const float invN = 1.0f / (float)N;
    float dd[16];
#pragma unroll
    for (int j = 0; j < 16; ++j) dd[j] = 0.f;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
        if (j < A) {
            const float z = d.out[(size_t)i * 16 + j], Rz = rz[(size_t)i * 16 + j];
            const float t = tanhf(z);
            const float mu = d.bounded ? d.max_action * t : z;
            const float mup = d.bounded ? d.max_action * (1.0f - t * t) : 1.0f;
            const float mupp = d.bounded ? -2.0f * d.max_action * t * (1.0f - t * t) : 0.0f;
            const float sg = expf(d.log_sigma[j]);
            const float is2 = 1.0f / (sg * sg);
            const float so = d.std_old[(size_t)r * A + j], mo = d.mean_old[(size_t)r * A + j];
            const float dm = mu - mo;
            const float kmu = dm * is2 * invN;                 // dKL/dmu
            const float Rmu = mup * Rz;
            const float Rkmu = Rmu * is2 * invN - 2.0f * kmu * vs[j];
            dd[j] = Rkmu * mup + kmu * mupp * Rz;              // R(dKL/dz)
            const float q = so * so + dm * dm;
            // R(dKL/ds) = -(Rq)/s^2 + 2 q / s^2 * vs,  Rq = 2 (mu - mu_old) Rmu
            dd[A + j] = (-(2.0f * dm * Rmu) * is2 + 2.0f * q * is2 * vs[j]) * invN;
        }
    }
#pragma unroll
    for (int j = 0; j < 16; j += 4)
        *reinterpret_cast<float4*>(rdout + (size_t)i * 16 + j) = make_float4(dd[j], dd[j + 1], dd[j + 2], dd[j + 3]);
}

// ---- R-forward -----------------------------------------------------------------------------------------
// pv: tangent parameters in the net's theta layout.  P = primal slot (cached h1, h2), R = tangent slot.
template <int H>
__global__ void __launch_bounds__(MLP_TPB)
cpo_rfwd_kernel(const fsrl_engine_t e, const fsrl_netref_t np_, const fsrl_netref_t nr_, const float* __restrict__ pv,
                const fsrl_eng_input_t in, int B) {
    using TT = MlpTile<H>;
    extern __shared__ __align__(16) float smem[];
    const EngView P = eng_view(e, np_), Rv = eng_view(e, nr_);
    const int D = np_.D, out = np_.out;
    const int tid = threadIdx.x;
    const int r0 = blockIdx.x * TT::R;
    const int inp = TT::in_pad(D);
    // tangent parameter views
    const NetLayout L(D, H, out, np_.n_extra);
    const float* v_w1t = pv + L.w1; const float* v_b1 = pv + L.b1; const float* v_w2t = pv + L.w2;
    const float* v_b2 = pv + L.b2; const float* v_w3t = pv + L.w3; const float* v_b3 = pv + L.b3;
    float* xs = smem;                                   // [R][inp]
    float* ta = xs + (size_t)TT::R * inp;               // tile A [R][LDA]  (Rh1, later h2 cache)
    float* tb = ta + (size_t)TT::R * TT::LDA;           // tile B           (h1 cache, later Rh2)
    float* wst = tb + (size_t)TT::R * TT::LDA;
    float* w3s = wst + TT::stage_floats();              // [H][out] W3t
    float* v3s = w3s + (size_t)H * out;                 // [H][out] V3t
    for (int i = tid; i < TT::R * inp; i += MLP_TPB) {
        const int r = i / inp, k = i % inp;
        xs[i] = (r0 + r < B && k < D) ? eng_input(in, r0 + r, k) : 0.f;
    }
    for (int i = tid; i < H * out; i += MLP_TPB) { w3s[i] = __ldg(P.m.w3t + i); v3s[i] = __ldg(v_w3t + i); }
    // h1 cache tile -> tb
    for (int el = tid; el < TT::R * (H / 4); el += MLP_TPB) {
        const int row = el / (H / 4), k4 = (el % (H / 4)) * 4;
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (r0 + row < B) v = *reinterpret_cast<const float4*>(P.s_h1 + (size_t)(r0 + row) * H + k4);
        *reinterpret_cast<float4*>(tb + (size_t)row * TT::LDA + k4) = v;
    }
    __syncthreads();
    float c[TT::MT][TT::NT][4];
    // Rh1 = m1 * (x V1 + c1)
    tc_init_bias<H>(c, v_b1);
    tc_gemm<H>(c, xs, inp, D, v_w1t, wst, false);
    tc_foreach<H>(c, [&](int row, int col, float v0, float v1) {
        const float2 hv = *reinterpret_cast<const float2*>(tb + (size_t)row * TT::LDA + col);
        const float2 g = make_float2(hv.x > 0.f ? v0 : 0.f, hv.y > 0.f ? v1 : 0.f);
        *reinterpret_cast<float2*>(ta + (size_t)row * TT::LDA + col) = g;
        if (r0 + row < B) *reinterpret_cast<float2*>(Rv.s_h1 + (size_t)(r0 + row) * H + col) = g;
    });
    // Ra2 = Rh1 W2 + h1 V2 + c2
    tc_init_bias<H>(c, v_b2);
    tc_gemm<H>(c, ta, TT::LDA, H, P.m.w2t, wst, false);
    tc_gemm<H>(c, tb, TT::LDA, H, v_w2t, wst, false);
    // after the last GEMM's trailing barrier both tiles are free: tb <- Rh2, ta <- h2 cache
    tc_foreach<H>(c, [&](int row, int col, float v0, float v1) {
        float2 hv = make_float2(0.f, 0.f);
        if (r0 + row < B) hv = *reinterpret_cast<const float2*>(P.s_h2 + (size_t)(r0 + row) * H + col);
        const float2 g = make_float2(hv.x > 0.f ? v0 : 0.f, hv.y > 0.f ? v1 : 0.f);
        *reinterpret_cast<float2*>(tb + (size_t)row * TT::LDA + col) = g;
        *reinterpret_cast<float2*>(ta + (size_t)row * TT::LDA + col) = hv;
        if (r0 + row < B) *reinterpret_cast<float2*>(Rv.s_h2 + (size_t)(r0 + row) * H + col) = g;
    });
    __syncthreads();
    // Rz = Rh2 W3 + h2 V3 + c3   (PARTS lanes per row)
    const int r = tid / TT::PARTS, part = tid % TT::PARTS;
    float acc[MLP_MAX_OUT];
#pragma unroll
    for (int j = 0; j < MLP_MAX_OUT; ++j) acc[j] = 0.f;
    for (int k = part; k < H; k += TT::PARTS) {
        const float rh = tb[(size_t)r * TT::LDA + k], hh = ta[(size_t)r * TT::LDA + k];
#pragma unroll
        for (int j = 0; j < MLP_MAX_OUT; ++j)
            if (j < out) acc[j] = fmaf(rh, w3s[(size_t)k * out + j], fmaf(hh, v3s[(size_t)k * out + j], acc[j]));
    }
#pragma unroll
    for (int j = 0; j < MLP_MAX_OUT; ++j) {
        if (j < out) {
            float v = acc[j];
#pragma unroll
            for (int o = TT::PARTS / 2; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o, TT::PARTS);
            acc[j] = v + __ldg(v_b3 + j);
        }
    }
    if (part == 0 && r0 + r < B) {
#pragma unroll
        for (int j = 0; j < 16; j += 4)
            *reinterpret_cast<float4*>(Rv.s_out + (size_t)(r0 + r) * 16 + j) =
                make_float4(j < out ? acc[j] : 0.f, j + 1 < out ? acc[j + 1] : 0.f, j + 2 < out ? acc[j + 2] : 0.f,
                            j + 3 < out ? acc[j + 3] : 0.f);
    }
}

// ---- R-backward ----------------------------------------------------------------------------------------
template <int H>
__global__ void __launch_bounds__(MLP_TPB)
cpo_rbwd_kernel(const fsrl_engine_t e, const fsrl_netref_t np_, const fsrl_netref_t nr_, const float* __restrict__ pv,
                const float* __restrict__ pv_w2n, int B, int nhead) {
    using TT = MlpTile<H>;
    extern __shared__ __align__(16) float smem[];
    const EngView P = eng_view(e, np_), Rv = eng_view(e, nr_);
    const int D = np_.D, out = np_.out;
    const int tid = threadIdx.x;
    const int r0 = blockIdx.x * TT::R;
    const float* v_w3t = pv + NetLayout(D, H, out, np_.n_extra).w3;
    float* ta = smem;                                   // Rda2 tile
    float* tb = ta + (size_t)TT::R * TT::LDA;           // da2 (primal) tile
    float* wst = tb + (size_t)TT::R * TT::LDA;
    float* w3s = wst + TT::stage_floats();
    float* v3s = w3s + (size_t)H * out;
    float* se = v3s + (size_t)H * out;                  // e   [R][16]
    float* sre = se + (size_t)TT::R * 16;               // Re  [R][16]
    for (int i = tid; i < H * out; i += MLP_TPB) { w3s[i] = __ldg(P.m.w3t + i); v3s[i] = __ldg(v_w3t + i); }
    for (int i = tid; i < TT::R * 16; i += MLP_TPB) {
        const int r = i / 16;
        const bool ok = r0 + r < B;
        se[i] = ok ? P.s_dout[(size_t)(r0 + r) * 16 + (i % 16)] : 0.f;
        sre[i] = ok ? Rv.s_dout[(size_t)(r0 + r) * 16 + (i % 16)] : 0.f;
    }
    __syncthreads();
    for (int el = tid; el < TT::R * (H / 4); el += MLP_TPB) {
        const int row = el / (H / 4), k4 = (el % (H / 4)) * 4;
        const bool ok = r0 + row < B;
        float a4[4] = {0.f, 0.f, 0.f, 0.f};
        for (int j = 0; j < nhead; ++j) {
            const float re = sre[row * 16 + j], ee = se[row * 16 + j];
#pragma unroll
            for (int q = 0; q < 4; ++q)
                a4[q] = fmaf(re, w3s[(size_t)(k4 + q) * out + j], fmaf(ee, v3s[(size_t)(k4 + q) * out + j], a4[q]));
        }
        float4 hv = make_float4(0.f, 0.f, 0.f, 0.f), da2 = hv;
        if (ok) {
            hv = *reinterpret_cast<const float4*>(P.s_h2 + (size_t)(r0 + row) * H + k4);
            da2 = *reinterpret_cast<const float4*>(P.s_dz2 + (size_t)(r0 + row) * H + k4);
        }
        const float4 g4 = make_float4(hv.x > 0.f ? a4[0] : 0.f, hv.y > 0.f ? a4[1] : 0.f,
                                      hv.z > 0.f ? a4[2] : 0.f, hv.w > 0.f ? a4[3] : 0.f);
        *reinterpret_cast<float4*>(ta + (size_t)row * TT::LDA + k4) = g4;
        *reinterpret_cast<float4*>(tb + (size_t)row * TT::LDA + k4) = da2;
        if (ok) *reinterpret_cast<float4*>(Rv.s_dz2 + (size_t)(r0 + row) * H + k4) = g4;
    }
    float c[TT::MT][TT::NT][4];
    tc_init_bias<H>(c, nullptr);
    tc_gemm<H>(c, ta, TT::LDA, H, P.w2n, wst, false);        // Rda2 . W2
    tc_gemm<H>(c, tb, TT::LDA, H, pv_w2n, wst, false);       // da2 . V2
    tc_foreach<H>(c, [&](int row, int col, float v0, float v1) {
        if (r0 + row < B) {
            const float2 hv = *reinterpret_cast<const float2*>(P.s_h1 + (size_t)(r0 + row) * H + col);
            *reinterpret_cast<float2*>(Rv.s_dz1 + (size_t)(r0 + row) * H + col) =
                make_float2(hv.x > 0.f ? v0 : 0.f, hv.y > 0.f ? v1 : 0.f);
        }
    });
}

// ---- small vector kernels (P up to a few 100 k: single CTA, deterministic order) -----------------------
__global__ void __launch_bounds__(1024) vec_dot_kernel(const float* a, const float* b, long long n, double* out) {
    __shared__ double red[32];
    double s = 0.0;
    for (long long i = threadIdx.x; i < n; i += 1024) s += (double)a[i] * (double)b[i];
    s = warp_sum(s);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
    __syncthreads();
    if (threadIdx.x == 0) { double t = 0.0; for (int w = 0; w < 32; ++w) t += red[w]; *out = t; }
}
// y = a*x + b*y
__global__ void vec_axpby_kernel(float a, const float* x, float b, float* y, long long n) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) y[i] = a * x[i] + b * y[i];
}
// out = a + s * b
__global__ void vec_add_scaled_kernel(const float* a, float s, const float* b, float* out, long long n) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = a[i] + s * b[i];
}

}  // namespace fsrl

using namespace fsrl;

static int cpo_check(const fsrl_cpo_t* d) {
    FSRL_REQUIRE(d != nullptr, "cpo: null descriptor");
    FSRL_REQUIRE(d->N >= 2 && d->N <= d->eng.bmax, "cpo: N=%lld out of range (bmax %d)", d->N, d->eng.bmax);
    FSRL_REQUIRE(d->A >= 1 && d->A <= 8, "cpo: action dim out of range");
    FSRL_REQUIRE(d->obs && d->act && d->logp_old && d->mean_old && d->std_old && d->adv && d->out && d->dout && d->log_sigma,
                 "cpo: null batch pointer");
    return FSRL_OK;
}

// sums[0..2] (device doubles, zeroed here) <- sum ratio*adv_r, sum ratio*adv_c, sum kl over the batch;
// mode != 0 additionally writes the head gradient of objective (1), -cost surrogate (2) or kl (3)
extern "C" int fsrl_cpo_head(const fsrl_cpo_t* d, int mode, double* sums, void* stream) {
    int rc = cpo_check(d);
    if (rc) return rc;
    FSRL_REQUIRE(mode >= 0 && mode <= 3 && sums, "cpo_head: bad mode / sums");
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    FSRL_CUDA(cudaMemsetAsync(sums, 0, 4 * sizeof(double), s));
    cpo_head_kernel<<<(unsigned)((d->N + 255) / 256), 256, 0, s>>>(*d, d->N, mode, sums);
    FSRL_LAUNCH_CHECK();
    return FSRL_OK;
}

extern "C" int fsrl_focops_head(const fsrl_cpo_t* d, double inv_lambda, double nu, double eta, double* sums_dev4,
                                void* stream) {
    int rc = cpo_check(d);
    if (rc) return rc;
    FSRL_REQUIRE(sums_dev4 != nullptr, "focops_head: null sums");
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    FSRL_CUDA(cudaMemsetAsync(sums_dev4, 0, 4 * sizeof(double), s));
    focops_head_kernel<<<(unsigned)((d->N + 255) / 256), 256, 0, s>>>(*d, d->N, (float)inv_lambda, (float)nu, (float)eta, sums_dev4);
    FSRL_LAUNCH_CHECK();
    return FSRL_OK;
}

// hv <- H v + damping * v with H = Hessian of the mean KL w.r.t. the actor parameters.  Needs the
// caches of a saved forward pass and of the kl backward pass (P-slot h1, h2, out, dout = dKL/dz,
// dz2); uses the tangent slot `actor_r` for the R-quantities.
extern "C" int fsrl_cpo_hvp(const fsrl_cpo_t* d, const float* v, float* v_w2n_scratch, float* hv,
                            double damping, void* stream) {
    int rc = cpo_check(d);
    if (rc) return rc;
    FSRL_REQUIRE(v && hv && v_w2n_scratch, "cpo_hvp: null vector");
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    const fsrl_netref_t& np_ = d->actor.nets[0];
    const fsrl_netref_t& nr_ = d->actor_r.nets[0];
    const int H = np_.H, D = np_.D, out = np_.out;
    const int B = (int)d->N;
    const NetLayout L(D, H, out, np_.n_extra);
    const long long P = L.size;
    fsrl_eng_input_t in;
    in.xa = d->obs; in.ia = d->perm; in.xb = nullptr; in.ib = nullptr; in.Da = D; in.Db = 0;
    W2Mirrors vm = {};   // mirror of the tangent vector's W2 block
    vm.w2t[0] = v + L.w2;
    vm.w2n[0] = v_w2n_scratch;
    rc = w2_mirror(vm, 1, H, s);
    if (rc) return rc;
    ENG_DISPATCH_H(H, {
        using TT = MlpTile<HH>;
        const size_t smf = sizeof(float) * ((size_t)TT::R * TT::in_pad(D) + 2 * (size_t)TT::R * TT::LDA + TT::stage_floats() + 2 * (size_t)HH * out);
        FSRL_CUDA(cudaFuncSetAttribute(cpo_rfwd_kernel<HH>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smf));
        cpo_rfwd_kernel<HH><<<(B + TT::R - 1) / TT::R, MLP_TPB, smf, s>>>(d->eng, np_, nr_, v, in, B);
    });
    FSRL_LAUNCH_CHECK();
    {
        EngView Rv;   // host-side pointer arithmetic for the tangent slot's out / dout
        const size_t slotf = eng_slot_floats(H, d->eng.bmax);
        float* sc = d->eng.scratch + (size_t)nr_.slot * slotf;
        float* r_out = sc + 4 * (size_t)d->eng.bmax * H;
        float* r_dout = r_out + (size_t)d->eng.bmax * 16;
        (void)Rv;
        cpo_rhead_kernel<<<(unsigned)((d->N + 255) / 256), 256, 0, s>>>(*d, d->N, r_out, v + L.extra, r_dout);
        FSRL_LAUNCH_CHECK();
    }
    ENG_DISPATCH_H(H, {
        using TT = MlpTile<HH>;
        const size_t smb = sizeof(float) * (2 * (size_t)TT::R * TT::LDA + TT::stage_floats() + 2 * (size_t)HH * out + 2 * (size_t)TT::R * 16);
        FSRL_CUDA(cudaFuncSetAttribute(cpo_rbwd_kernel<HH>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smb));
        cpo_rbwd_kernel<HH><<<(B + TT::R - 1) / TT::R, MLP_TPB, smb, s>>>(d->eng, np_, nr_, v, v_w2n_scratch, B, d->A);
    });
    FSRL_LAUNCH_CHECK();
    // Hv = [Rh1^T da2 | x^T Rda1, colsum Rda1 | Rh2^T e]  +  [h1^T Rda2, colsum Rda2 | h2^T Re, colsum Re(+extra)]
    const size_t slotf = eng_slot_floats(H, d->eng.bmax);
    const size_t bh = (size_t)d->eng.bmax * H;
    float* Ps = d->eng.scratch + (size_t)np_.slot * slotf;
    float* Rs = d->eng.scratch + (size_t)nr_.slot * slotf;
    WgradRoles ra = {Rs /*Rh1*/, Ps + 3 * bh /*da2*/, Rs + 2 * bh /*Rda1*/, Rs + bh /*Rh2*/, Ps + 4 * bh + (size_t)d->eng.bmax * 16 /*e*/,
                     hv, 0, 0, 7};
    rc = eng_wgrad_roles(&d->eng, &d->actor, &in, B, 0, nullptr, ra, s);
    if (rc) return rc;
    WgradRoles rb = {Ps /*h1*/, Rs + 3 * bh /*Rda2*/, nullptr, Ps + bh /*h2*/, Rs + 4 * bh + (size_t)d->eng.bmax * 16 /*Re*/,
                     hv, 1, 1, 5};
    rc = eng_wgrad_roles(&d->eng, &d->actor, &in, B, 1, nullptr, rb, s);
    if (rc) return rc;
    vec_axpby_kernel<<<(unsigned)((P + 255) / 256), 256, 0, s>>>((float)damping, v, 1.0f, hv, P);
    FSRL_LAUNCH_CHECK();
    return FSRL_OK;
}

extern "C" int fsrl_vec_dot(const float* a, const float* b, long long n, double* out_dev, void* stream) {
    FSRL_REQUIRE(a && b && out_dev && n >= 0, "vec_dot: bad arguments");
    vec_dot_kernel<<<1, 1024, 0, static_cast<cudaStream_t>(stream)>>>(a, b, n, out_dev);
    FSRL_LAUNCH_CHECK();
    return FSRL_OK;
}
extern "C" int fsrl_vec_axpby(double a, const float* x, double b, float* y, long long n, void* stream) {
    FSRL_REQUIRE(x && y && n >= 0, "vec_axpby: bad arguments");
    if (n == 0) return FSRL_OK;
    vec_axpby_kernel<<<(unsigned)((n + 255) / 256), 256, 0, static_cast<cudaStream_t>(stream)>>>((float)a, x, (float)b, y, n);
    FSRL_LAUNCH_CHECK();
    return FSRL_OK;
}
extern "C" int fsrl_vec_add_scaled(const float* a, double s, const float* b, float* out, long long n, void* stream) {
    FSRL_REQUIRE(a && b && out && n >= 0, "vec_add_scaled: bad arguments");
    if (n == 0) return FSRL_OK;
    vec_add_scaled_kernel<<<(unsigned)((n + 255) / 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(a, (float)s, b, out, n);
    FSRL_LAUNCH_CHECK();
    return FSRL_OK;
}

// ---- conjugate gradients with every scalar on the device (cpo.py:184-204, trpo_lag.py:261-283) -------------------
// state (doubles): [0] rs_old  [1] p.z / r.r scratch  [2] alpha  [3] beta  [4] done flag (0 / 1)
__global__ void cg_alpha_kernel(double* st) {          // after dot(p, z) -> st[1]
    if (st[4] == 0.0) st[2] = st[0] / st[1];
}
__global__ void cg_beta_kernel(double* st, double tol) {   // after dot(r, r) -> st[1]
    if (st[4] != 0.0) return;
    const double rs_new = st[1];
    if (rs_new < tol) { st[4] = 1.0; return; }              // the reference's `break`: x, r updated, p not
    st[3] = rs_new / st[0];
    st[0] = rs_new;
}
// x += alpha p ; r -= alpha z      (python: vec_axpby((float)alpha, p, 1, x), vec_axpby((float)-alpha, z, 1, r))
__global__ void cg_step_xr_kernel(const double* st, const float* __restrict__ p, const float* __restrict__ z,
                                  float* __restrict__ x, float* __restrict__ r, long long n) {
    if (st[4] != 0.0) return;
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float a = (float)st[2], ma = (float)(-st[2]);
    x[i] = a * p[i] + 1.0f * x[i];
    r[i] = ma * z[i] + 1.0f * r[i];
}
// p = r + beta p                   (python: vec_axpby(1, r, (float)beta, p))
__global__ void cg_step_p_kernel(const double* st, const float* __restrict__ r, float* __restrict__ p, long long n) {
    if (st[4] != 0.0) return;
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    p[i] = 1.0f * r[i] + (float)st[3] * p[i];
}

// x = CG(H, rhs) with H v = fsrl_cpo_hvp(v): `nsteps` iterations enqueued back to back, no host synchronisation -- the
// residual test of the reference's loop (`if rs_new < tol: break`) is a device flag that turns the remaining
// iterations into no-ops, so the result equals the host-driven loop's.  work = 4 vectors of P floats (x, r, p, z are
// carved from it; x_out may alias none of them), state_dev = 8 doubles.  Replaces the per-iteration .item() round
// trips of policy/trust_region.py::_cg (single-GPU runs; data-parallel runs all-reduce every product on the host side).
extern "C" int fsrl_cg_solve(const fsrl_cpo_t* d, const float* rhs, float* x_out, float* work, float* v_w2n_scratch,
                             double* state_dev, long long P, int nsteps, double tol, double damping, void* stream) {
    int rc = cpo_check(d);
    if (rc) return rc;
    FSRL_REQUIRE(rhs && x_out && work && v_w2n_scratch && state_dev && P > 0 && nsteps >= 0, "cg_solve: bad arguments");
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    float *x = work, *r = work + P, *p = work + 2 * P, *z = work + 3 * P;
    const unsigned nb = (unsigned)((P + 255) / 256);
    FSRL_CUDA(cudaMemsetAsync(x, 0, sizeof(float) * P, s));
    FSRL_CUDA(cudaMemcpyAsync(r, rhs, sizeof(float) * P, cudaMemcpyDeviceToDevice, s));
    FSRL_CUDA(cudaMemcpyAsync(p, rhs, sizeof(float) * P, cudaMemcpyDeviceToDevice, s));
    FSRL_CUDA(cudaMemsetAsync(state_dev, 0, sizeof(double) * 8, s));
    vec_dot_kernel<<<1, 1024, 0, s>>>(r, r, P, state_dev + 0);      // rs_old
    FSRL_LAUNCH_CHECK();
    for (int it = 0; it < nsteps; ++it) {
        rc = fsrl_cpo_hvp(d, p, v_w2n_scratch, z, damping, stream);
        if (rc) return rc;
        vec_dot_kernel<<<1, 1024, 0, s>>>(p, z, P, state_dev + 1);
        cg_alpha_kernel<<<1, 1, 0, s>>>(state_dev);
        cg_step_xr_kernel<<<nb, 256, 0, s>>>(state_dev, p, z, x, r, P);
        vec_dot_kernel<<<1, 1024, 0, s>>>(r, r, P, state_dev + 1);
        cg_beta_kernel<<<1, 1, 0, s>>>(state_dev, tol);
        cg_step_p_kernel<<<nb, 256, 0, s>>>(state_dev, r, p, P);
        FSRL_LAUNCH_CHECK();
    }
    FSRL_CUDA(cudaMemcpyAsync(x_out, x, sizeof(float) * P, cudaMemcpyDeviceToDevice, s));
    return FSRL_OK;
}

// wgrad of the listed nets into an arbitrary destination vector (theta layout of ONE net): used for
// g = grad objective and b = grad(-cost surrogate)
extern "C" int fsrl_engine_wgrad_to(const fsrl_engine_t* e, const fsrl_netlist_t* nl, const fsrl_eng_input_t* in,
                                    long long B, float* dst, void* stream) {
    FSRL_REQUIRE(e && nl && in && dst && nl->n == 1, "wgrad_to: needs exactly one net and a destination");
    FSRL_REQUIRE(B >= 0 && B <= e->bmax, "wgrad_to: B out of range");
    WgradRoles roles = {nullptr, nullptr, nullptr, nullptr, nullptr, dst, 1, 1, 7};
    return eng_wgrad_roles(e, nl, in, B, 0, nullptr, roles, static_cast<cudaStream_t>(stream));
}

// ---- critic regression head + whole-batch advantage standardisation ---------------------------------
namespace fsrl {
// dout[i][0] = 2 (V_i - ret_i) / N for one critic slot; sums[0] += sum td^2
__global__ void mse_head_kernel(const float* __restrict__ out, const float* __restrict__ ret, const int* __restrict__ perm,
                                long long N, float* __restrict__ dout, double* __restrict__ sums) {
    __shared__ double red[8];
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    double s = 0.0;
    if (i < N) {
        const long long r = perm ? (long long)perm[i] : i;
        const float td = out[(size_t)i * 16] - ret[r];
        float4 z = make_float4(2.0f * td / (float)N, 0.f, 0.f, 0.f);
        *reinterpret_cast<float4*>(dout + (size_t)i * 16) = z;
        z.x = 0.f;
        *reinterpret_cast<float4*>(dout + (size_t)i * 16 + 4) = z;
        *reinterpret_cast<float4*>(dout + (size_t)i * 16 + 8) = z;
        *reinterpret_cast<float4*>(dout + (size_t)i * 16 + 12) = z;
        s = (double)td * (double)td;
    }
    s = warp_sum(s);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
    __syncthreads();
    if (threadIdx.x == 0) { double t = 0.0; for (int w = 0; w < (int)(blockDim.x >> 5); ++w) t += red[w]; atomicAdd(sums, t); }
}

// x <- (x - mean) / std (unbiased, no eps) over n elements: cpo.py:127-131 / trpo_lag.py:129-133
__global__ void __launch_bounds__(1024) standardize_kernel(float* x, long long n) {
    __shared__ double red[32];
    __shared__ double s_mean, s_rstd;
    double s = 0.0;
    for (long long i = threadIdx.x; i < n; i += 1024) s += (double)x[i];
    s = warp_sum(s);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
    __syncthreads();
    if (threadIdx.x == 0) { double t = 0.0; for (int w = 0; w < 32; ++w) t += red[w]; s_mean = t / (double)n; }
    __syncthreads();
    const float mean = (float)s_mean;
    double q = 0.0;
    for (long long i = threadIdx.x; i < n; i += 1024) { const float d = x[i] - mean; q += (double)(d * d); }
    q = warp_sum(q);
    __syncthreads();
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = q;
    __syncthreads();
    if (threadIdx.x == 0) { double t = 0.0; for (int w = 0; w < 32; ++w) t += red[w]; s_rstd = 1.0 / sqrt(t / (double)(n - 1)); }
    __syncthreads();
    const float rstd = (float)s_rstd;
    for (long long i = threadIdx.x; i < n; i += 1024) x[i] = (x[i] - mean) * rstd;
}
}  // namespace fsrl

// head gradient of mean((ret - V)^2) for one critic (P-slot out/dout [bmax][16]); sums_dev[0] += sum td^2
extern "C" int fsrl_mse_head(const float* out, const float* ret, const int* perm, long long N, float* dout,
                             double* sums_dev, void* stream) {
    FSRL_REQUIRE(out && ret && dout && sums_dev && N >= 1, "mse_head: bad arguments");
    fsrl::mse_head_kernel<<<(unsigned)((N + 255) / 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(out, ret, perm, N, dout, sums_dev);
    FSRL_LAUNCH_CHECK();
    return FSRL_OK;
}

extern "C" int fsrl_standardize(float* x, long long n, void* stream) {
    FSRL_REQUIRE(x && n >= 2, "standardize: need at least two elements");
    fsrl::standardize_kernel<<<1, 1024, 0, static_cast<cudaStream_t>(stream)>>>(x, n);
    FSRL_LAUNCH_CHECK();
    return FSRL_OK;
}

// PPO-Lagrangian minibatch update on the device: clipped surrogate + lambda * cost-advantage
// actor loss, value losses for the reward and cost critics, backward pass, global-norm clip
// and Adam -- three launches per minibatch, no host round trip inside a repeat.
//
// Replaces (reference, eager PyTorch + ~10 .item() syncs per minibatch):
//   /root/reference/fsrl/policy/ppo_lag.py:173-212  policy_loss (per-minibatch adv norm
//        :178-182, clipped surrogate :185-193, unclipped cost term :196-198, rescaling
//        :200-201, approx_kl :204)
//   /root/reference/fsrl/policy/ppo_lag.py:152-171  critics_loss
//   /root/reference/fsrl/policy/ppo_lag.py:223-247  forward/backward/clip_grad_norm_/Adam
//   /root/reference/fsrl/policy/lagrangian_base.py:145-166  safety_loss
//
// Phase A (ppo_fwd + ppo_bwd): grid (row tiles, column slabs, nets).  The permuted batch is
//   gathered once per repeat into contiguous arrays; ppo_fwd runs layers 1-2 with the N
//   dimension split over H/64 CTAs, ppo_bwd evaluates the head, the loss gradient and
//   back-propagates to dZ2 / dZ1 (again one column slab per CTA); activations needed for the
//   weight gradients go to an L2-resident scratch.
// Phase B (ppo_wgrad): weight gradients as outer-product accumulations over the minibatch,
//   each CTA owning a 32x64 tile of dW2t (no cross-CTA reduction), plus three small CTAs per
//   net for layer 1 / layer 3 / biases; sum of squares for the global norm via one atomic per
//   CTA.
// Phase C (adam): clip scale + Adam over the flat parameter buffer; the W2 blocks are
//   processed in 32x32 tiles through shared memory so that both the canonical W2t and its
//   out-major mirror (needed by the backward GEMM) are written coalesced.
#include "arena.cuh"
#include "mlp.cuh"
#include "ppo_persist.cuh"

namespace fsrl {

constexpr int ST_ACTOR_REW = 0, ST_ACTOR_SAFETY = 1, ST_KL = 2, ST_VF0 = 3, ST_VF1 = 4,
              ST_ENTROPY = 5, ST_GRADNORM = 6, ST_CLIPFRAC = 7;
constexpr float LOG_SQRT_2PI_P = 0.9189385332046727f;
constexpr int DOUT_LD = 16;   // scratch row stride of dOut (cols [A, 2A) carry dlog_sigma)

// Programmatic dependent launch (sm_90+): a kernel launched with the programmatic-serialization
// attribute may start while its predecessor in the stream is still running; everything it reads
// that the predecessor writes must come after pdl_wait() (= predecessor complete + flushed).
// pdl_trigger() lets the NEXT kernel's CTAs be scheduled as soon as SM resources free up.  Every
// kernel of the minibatch chain triggers only AFTER its own wait, so "predecessor complete"
// is transitive along the chain.  Both are no-ops for ordinary launches.
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

__device__ __forceinline__ int slot_mb(const fsrl_ppo_update_t& u, int mb_off) { return mb_off / u.batch_size; }

struct NetView {   // resolved pointers of one network inside the flat buffers
    Mlp3 m;
    const float* w2n;      // mirror [out][in] of w2t
    const float* log_sigma;
    float *g_w1t, *g_b1, *g_w2t, *g_b2, *g_w3t, *g_b3, *g_log_sigma;
    float *s_h1, *s_h2, *s_dz1, *s_dz2, *s_dout;   // scratch [Bmax][H] / [Bmax][16]
};

// arena layout of net n: the actor (n = 0) heads actor_out columns and carries its log-sigma as extras
__host__ __device__ __forceinline__ NetLayout ppo_layout(const fsrl_ppo_update_t& u, int n, int H) {
    return NetLayout(u.D, H, (n == 0) ? u.actor_out : 1, (n == 0 && u.head_indep) ? u.A : 0);
}

__device__ __forceinline__ NetView net_view(const fsrl_ppo_update_t& u, int n) {
    NetView v;
    const int H = u.H, D = u.D;
    const int out = (n == 0) ? u.actor_out : 1;
    const NetLayout L = ppo_layout(u, n, H);
    const float* th = u.theta + u.net_off[n];
    float* g = u.grad + u.net_off[n];
    v.m.w1t = th + L.w1; v.g_w1t = g + L.w1;
    v.m.b1 = th + L.b1;  v.g_b1 = g + L.b1;
    v.m.w2t = th + L.w2; v.g_w2t = g + L.w2;
    v.m.b2 = th + L.b2;  v.g_b2 = g + L.b2;
    v.m.w3t = th + L.w3; v.g_w3t = g + L.w3;
    v.m.b3 = th + L.b3;  v.g_b3 = g + L.b3;
    v.log_sigma = th + L.extra; v.g_log_sigma = g + L.extra;
    v.m.in = D; v.m.H = H; v.m.out = out;
    v.w2n = u.w2n + (size_t)n * H * H;
    float* sc = u.scratch + (size_t)n * u.bmax * (4 * (size_t)H + DOUT_LD);
    v.s_h1 = sc; v.s_h2 = sc + (size_t)u.bmax * H; v.s_dz1 = sc + 2 * (size_t)u.bmax * H;
    v.s_dz2 = sc + 3 * (size_t)u.bmax * H; v.s_dout = sc + 4 * (size_t)u.bmax * H;
    return v;
}

__device__ __forceinline__ float block_sum_256(float v, float* red) {
    v = warp_sum(v);
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    __syncthreads();
    if (lane == 0) red[w] = v;
    __syncthreads();
    float t = 0.f;
#pragma unroll
    for (int i = 0; i < MLP_TPB / 32; ++i) t += red[i];
    return t;
}

// ------------------------------------------------------------------------------------------
// Phase A, split in two launches so that every layer's N dimension is spread over H/64 CTAs
// (grid = row tiles x column slabs x nets = 192 CTAs for B = 256, H = 256):
//   A1 ppo_fwd : x -> h1 (full, tiny K) -> h2[:, slab]           (scratch: h1, h2)
//   A2 ppo_bwd : h2 (full) -> head -> loss gradient -> dz2 (full) -> dz1[:, slab]
// Rows are addressed through row_of(): the epoch driver first gathers the permuted batch into
// contiguous arrays (u.perm == nullptr afterwards), so minibatch rows are coalesced.
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ long long row_of(const fsrl_ppo_update_t& u, int mb_off, int i) {
    return u.perm ? (long long)u.perm[mb_off + i] : (long long)(mb_off + i);
}

template <int H>
__global__ void __launch_bounds__(MLP_TPB)
ppo_fwd_kernel(const fsrl_ppo_update_t u, int mb_off, int B) {
    using TT = MlpTile<H>;
    extern __shared__ __align__(16) float smem[];
    const int tid = threadIdx.x;
    const int net = blockIdx.z, slab = blockIdx.y;
    const int r0 = blockIdx.x * TT::R;
    const int c0 = slab * SLAB_NS;
    const int D = u.D;
    const int inp = TT::in_pad(D);
    const NetView nv = net_view(u, net);
    float* xs = smem;                                   // [R][inp]
    float* h1 = xs + (size_t)TT::R * inp;               // [R][LDA]
    float* bs = h1 + (size_t)TT::R * TT::LDA;           // [H][SLAB_LDB]  (aliased by the reduce buffer)
    // observations are constant during a repeat: loaded while the previous optimiser step drains
    for (int i = tid; i < TT::R * inp; i += MLP_TPB) {
        const int r = i / inp, k = i % inp;
        xs[i] = (r0 + r < B && k < D) ? u.obs[(size_t)row_of(u, mb_off, r0 + r) * D + k] : 0.f;
    }
    pdl_wait();                                         // parameters of the previous step are final
    pdl_trigger();
    // bias of this thread's epilogue columns: requested now, consumed after the GEMM
    const float4 b2v = __ldg(reinterpret_cast<const float4*>(nv.m.b2 + c0 + (tid % (SLAB_NS / 4)) * 4));
    if (net == 0 && slab == 0 && blockIdx.x == 0 && tid == 0) *u.norm_sq = 0.f;   // consumed by the previous step's Adam
    slab_load<H>(nv.m.w2t, H, c0, bs);                  // in flight during layer 1
    __syncthreads();
    float c[TT::MT][TT::NT][4];
    tc_init_bias<H>(c, nv.m.b1);
    tc_gemm_direct<H>(c, xs, inp, D, nv.m.w1t);
    tc_foreach<H>(c, [&](int row, int col, float v0, float v1) {
        const float2 h = make_float2(fmaxf(v0, 0.f), fmaxf(v1, 0.f));
        *reinterpret_cast<float2*>(h1 + (size_t)row * TT::LDA + col) = h;
        if (slab == 0 && r0 + row < u.bmax) *reinterpret_cast<float2*>(nv.s_h1 + (size_t)(r0 + row) * H + col) = h;
    });
    __pipeline_wait_prior(0);
    __syncthreads();
    slab_gemm<H>(h1, TT::LDA, bs, bs, [&](int row, int c4, float4 v) {
        const float4 b = b2v;                           // c4 == (tid % 16) * 4 for every element this thread visits
        if (r0 + row < u.bmax)
            *reinterpret_cast<float4*>(nv.s_h2 + (size_t)(r0 + row) * H + c0 + c4) =
                make_float4(fmaxf(v.x + b.x, 0.f), fmaxf(v.y + b.y, 0.f), fmaxf(v.z + b.z, 0.f), fmaxf(v.w + b.w, 0.f));
    });
}

// per-row head dot product  out[j] = sum_k h2[k] * w3s[k][j]  over this lane's k subset, with the
// column loop bounded at compile time (OUTP = next power of two >= wout)
template <int OUTP>
__device__ __forceinline__ void head_dot(const float* __restrict__ hrow, const float* __restrict__ w3s, int wout,
                                         int part, int parts, int H, float* out) {
    float acc[OUTP];
#pragma unroll
    for (int j = 0; j < OUTP; ++j) acc[j] = 0.f;
    for (int k = part; k < H; k += parts) {
        const float x = hrow[k];
        const float* w = w3s + (size_t)k * wout;
#pragma unroll
        for (int j = 0; j < OUTP; ++j)
            if (j < wout) acc[j] = fmaf(x, w[j], acc[j]);
    }
#pragma unroll
    for (int j = 0; j < OUTP; ++j) out[j] = acc[j];
}

template <int H>
__global__ void __launch_bounds__(MLP_TPB)
ppo_bwd_kernel(const fsrl_ppo_update_t u, int mb_off, int B, int slot) {
    using TT = MlpTile<H>;
    extern __shared__ __align__(16) float smem[];
    const int tid = threadIdx.x;
    const int net = blockIdx.z, slab = blockIdx.y;
    const int r0 = blockIdx.x * TT::R;
    const int c0 = slab * SLAB_NS;
    const NetView nv = net_view(u, net);
    const int wout = nv.m.out;
    float* h2 = smem;                                   // [R][LDA]
    float* dz = h2 + (size_t)TT::R * TT::LDA;           // [R][LDA]
    float* bs = dz + (size_t)TT::R * TT::LDA;           // [H][SLAB_LDB]
    float* w3s = bs + slab_buf_floats<H>();             // [H][out]
    float* sdout = w3s + (size_t)H * wout;              // [R][DOUT_LD]
    __shared__ float s_mean[2], s_rstd[2], s_b3[MLP_MAX_OUT], s_ls[8];
    // everything that does not depend on the forward launch (weights, per-row loss inputs) is
    // requested before pdl_wait(): it overlaps the forward kernel's tail
    slab_load<H>(nv.w2n, H, c0, bs);                    // W2 in [out][in] layout: rows o, columns k-slab
    for (int i = tid; i < H * wout; i += MLP_TPB) w3s[i] = __ldg(nv.m.w3t + i);
    // per-row scalars of the loss: issued now, consumed after the head
    const int r = tid / TT::PARTS, part = tid % TT::PARTS;
    const bool row_ok = (part == 0) && (r0 + r < B);
    const long long id = row_ok ? row_of(u, mb_off, r0 + r) : 0;
    float p_act[8], p_lpo = 0.f, p_adv0 = 0.f, p_adv1 = 0.f, p_ret = 0.f, p_val = 0.f;
#pragma unroll
    for (int j = 0; j < 8; ++j) p_act[j] = 0.f;
    if (row_ok) {
        if (net == 0) {
#pragma unroll
            for (int j = 0; j < 8; ++j) if (j < u.A) p_act[j] = u.act[(size_t)id * u.A + j];
            p_lpo = u.logp_old[id];
            p_adv0 = u.adv[id];
            if (u.C > 1) p_adv1 = u.adv[(size_t)u.ld + id];
        } else {
            p_ret = u.ret[(size_t)(net - 1) * u.ld + id];
            if (u.value_clip) p_val = u.values[(size_t)(net - 1) * u.ld + id];
        }
    }
    // per-minibatch advantage normalisation (ppo_lag.py:178-182): mean / 1/std of this minibatch
    // were computed for every minibatch of the repeat by ppo_adv_stats_kernel
    if (net == 0 && tid < u.C) {
        const float* ms = u.mb_stats + ((size_t)slot_mb(u, mb_off) * 2 + tid) * 2;
        s_mean[tid] = ms[0];
        s_rstd[tid] = ms[1];
    }
    if (tid >= 32 && tid < 32 + wout) s_b3[tid - 32] = __ldg(nv.m.b3 + tid - 32);
    if (net == 0 && tid >= 64 && tid < 64 + u.A) s_ls[tid - 64] = nv.log_sigma[tid - 64];
    pdl_wait();                                          // h1 / h2 of this minibatch are complete
    pdl_trigger();
    for (int el = tid; el < TT::R * (H / 4); el += MLP_TPB) {
        const int row = el / (H / 4), k4 = (el % (H / 4)) * 4;
        float* dst = h2 + (size_t)row * TT::LDA + k4;
        if (r0 + row < B) __pipeline_memcpy_async(dst, nv.s_h2 + (size_t)(r0 + row) * H + k4, 16);
        else *reinterpret_cast<float4*>(dst) = make_float4(0.f, 0.f, 0.f, 0.f);
    }
    __pipeline_commit();
    __pipeline_wait_prior(0);                            // slab (requested long ago) and h2 tile landed
    __syncthreads();
    // ---- head forward (every slab CTA recomputes it: H x out MACs per row, negligible) -----------
    float out[MLP_MAX_OUT];
#pragma unroll
    for (int j = 0; j < MLP_MAX_OUT; ++j) out[j] = 0.f;
    {
        const float* hrow = h2 + (size_t)r * TT::LDA;
        if (wout <= 1) head_dot<1>(hrow, w3s, wout, part, TT::PARTS, H, out);
        else if (wout <= 2) head_dot<2>(hrow, w3s, wout, part, TT::PARTS, H, out);
        else if (wout <= 4) head_dot<4>(hrow, w3s, wout, part, TT::PARTS, H, out);
        else if (wout <= 8) head_dot<8>(hrow, w3s, wout, part, TT::PARTS, H, out);
        else head_dot<16>(hrow, w3s, wout, part, TT::PARTS, H, out);
    }
#pragma unroll
    for (int j = 0; j < MLP_MAX_OUT; ++j) {
        if (j < wout) {
            float v = out[j];
#pragma unroll
            for (int o = TT::PARTS / 2; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o, TT::PARTS);
            out[j] = v + s_b3[j];
        }
    }
    // ---- loss gradient at the head: one thread per row -----------------------------------------
    float st_a = 0.f, st_b = 0.f, st_c = 0.f, st_d = 0.f;     // per-thread stat partials
    if (part == 0) {
        float dd[DOUT_LD];
#pragma unroll
        for (int j = 0; j < DOUT_LD; ++j) dd[j] = 0.f;
        if (row_ok) {
            const float invB = 1.0f / (float)B;
            if (net == 0) {
                const int A = u.A;
                float logp = 0.f, zz[8], sg[8], dmu[8];
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                    if (j < A) {
                        const float t = tanhf(out[j]);
                        const float mu = u.bounded ? u.max_action * t : out[j];
                        dmu[j] = u.bounded ? u.max_action * (1.0f - t * t) : 1.0f;
                        sg[j] = expf(s_ls[j]);
                        zz[j] = (p_act[j] - mu) / sg[j];
                        logp += -0.5f * zz[j] * zz[j] - s_ls[j] - LOG_SQRT_2PI_P;
                    }
                }
                const float lpo = p_lpo;
                const float ratio = expf(logp - lpo);
                const float ar = (p_adv0 - s_mean[0]) * s_rstd[0];
                const float surr1 = ratio * ar;
                const float rc = fminf(fmaxf(ratio, 1.0f - u.eps_clip), 1.0f + u.eps_clip);
                const float surr2 = rc * ar;
                // d(-min(surr1, surr2))/d ratio ; ties split evenly like torch.min's backward
                const bool inside = (ratio >= 1.0f - u.eps_clip) && (ratio <= 1.0f + u.eps_clip);
                float g_ratio;   // d loss_rew_i / d ratio  (before the 1/B of the mean)
                float lrew;
                if (surr1 < surr2) { g_ratio = -ar; lrew = -surr1; }
                else if (surr1 > surr2) { g_ratio = inside ? -ar : 0.f; lrew = -surr2; }
                else { g_ratio = inside ? -ar : -0.5f * ar; lrew = -surr1; }
                if (u.dual_clip > 0.f && ar < 0.f) {
                    // clip2 = max(min(s1,s2), dual_clip*adv) for negative advantages (:188-191)
                    const float c1 = fminf(surr1, surr2), c2 = u.dual_clip * ar;
                    if (c2 > c1) { g_ratio = 0.f; lrew = -c2; }
                    else if (c2 == c1) { g_ratio *= 0.5f; }
                }
                float g_saf = 0.f, lsaf = 0.f;
                if (u.use_lagrangian && u.C > 1) {
                    const float ac = (p_adv1 - s_mean[1]) * s_rstd[1];
                    g_saf = ac * u.lagrangian;          // d mean(ratio*adv_c*lambda) / d ratio
                    lsaf = ratio * ac * u.lagrangian;
                }
                // d loss / d logp = rescaling * (g_ratio + g_saf) * ratio / B
                const float gl = u.rescaling * (g_ratio + g_saf) * ratio * invB;
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                    if (j < A) {
                        dd[j] = gl * (zz[j] / sg[j]) * dmu[j];        // via mu
                        dd[A + j] = gl * (zz[j] * zz[j] - 1.0f);       // via log_sigma
                    }
                }
                st_a = lrew * invB; st_b = lsaf * invB; st_c = (lpo - logp) * invB;
            } else {
                const float v = out[0];
                const float ret = p_ret;
                float lv, gv;
                if (u.value_clip) {
                    const float vt = p_val;
                    const float dv = fminf(fmaxf(v - vt, -u.eps_clip), u.eps_clip);
                    const float vc = vt + dv;
                    const float vf1 = (ret - v) * (ret - v), vf2 = (ret - vc) * (ret - vc);
                    const bool in_clip = (v - vt > -u.eps_clip) && (v - vt < u.eps_clip);
                    if (vf1 > vf2) { lv = vf1; gv = 2.0f * (v - ret); }
                    else if (vf1 < vf2) { lv = vf2; gv = in_clip ? 2.0f * (vc - ret) : 0.f; }
                    else { lv = vf1; gv = in_clip ? 2.0f * (v - ret) : (v - ret); }
                } else {
                    lv = (ret - v) * (ret - v);
                    gv = 2.0f * (v - ret);
                }
                dd[0] = u.vf_coef * gv * invB;
                st_d = lv * invB;
            }
        }
#pragma unroll
        for (int j = 0; j < DOUT_LD; ++j) sdout[r * DOUT_LD + j] = dd[j];
        if (slab == 0 && r0 + r < u.bmax) {
#pragma unroll
            for (int j = 0; j < DOUT_LD; j += 4)
                *reinterpret_cast<float4*>(nv.s_dout + (size_t)(r0 + r) * DOUT_LD + j) =
                    make_float4(dd[j], dd[j + 1], dd[j + 2], dd[j + 3]);
        }
    }
    // minibatch statistics (loss/actor_rew, actor_safety, kl, vf_i): warp-level partial sums and one
    // fire-and-forget reduction per warp -- no block barrier on the critical path
    if (slab == 0) {
        float* stat = u.stats + (size_t)slot * FSRL_PPO_STATS;
        const int lane = tid & 31;
        if (net == 0) {
            const float a = warp_sum(st_a), b = warp_sum(st_b), c = warp_sum(st_c);
            if (lane == 0) {
                atomicAdd(stat + ST_ACTOR_REW, a); atomicAdd(stat + ST_ACTOR_SAFETY, b); atomicAdd(stat + ST_KL, c);
            }
            if (blockIdx.x == 0 && tid == 0) {
                float ent = 0.f;
                for (int j = 0; j < u.A; ++j) ent += 0.5f + LOG_SQRT_2PI_P + s_ls[j];
                stat[ST_ENTROPY] = ent;
            }
        } else {
            const float d = warp_sum(st_d);
            if (lane == 0) atomicAdd(stat + ST_VF0 + (net - 1), d);
        }
    }
    __syncthreads();
    // ---- backward through layer 3 and ReLU 2 (full width, redundant per slab: H x out per row) ----
    const int nout = (net == 0) ? u.A : 1;       // head columns that feed w3t (mu only)
    for (int e = tid; e < TT::R * (H / 4); e += MLP_TPB) {
        const int row = e / (H / 4), k4 = (e % (H / 4)) * 4;
        float a4[4] = {0.f, 0.f, 0.f, 0.f};
        for (int j = 0; j < nout; ++j) {
            const float g = sdout[row * DOUT_LD + j];
#pragma unroll
            for (int q = 0; q < 4; ++q) a4[q] = fmaf(g, w3s[(size_t)(k4 + q) * wout + j], a4[q]);
        }
        const float4 hv = *reinterpret_cast<const float4*>(h2 + (size_t)row * TT::LDA + k4);
        const float4 g4 = make_float4(hv.x > 0.f ? a4[0] : 0.f, hv.y > 0.f ? a4[1] : 0.f,
                                      hv.z > 0.f ? a4[2] : 0.f, hv.w > 0.f ? a4[3] : 0.f);
        *reinterpret_cast<float4*>(dz + (size_t)row * TT::LDA + k4) = g4;
        if (slab == 0 && r0 + row < u.bmax) *reinterpret_cast<float4*>(nv.s_dz2 + (size_t)(r0 + row) * H + k4) = g4;
    }
    __pipeline_wait_prior(0);
    __syncthreads();
    // the h2 tile is dead now: its space receives this slab's h1 columns (ReLU-1 mask of the epilogue)
    // while the GEMM runs (slab_gemm waits for outstanding async copies before its first barrier)
    for (int el = tid; el < TT::R * (SLAB_NS / 4); el += MLP_TPB) {
        const int row = el / (SLAB_NS / 4), c4 = (el % (SLAB_NS / 4)) * 4;
        if (r0 + row < u.bmax)
            __pipeline_memcpy_async(h2 + (size_t)row * SLAB_NS + c4, nv.s_h1 + (size_t)(r0 + row) * H + c0 + c4, 16);
    }
    __pipeline_commit();
    // ---- backward through layer 2: dH1[:, slab] = dZ2 . W2[:, slab], then ReLU 1 -------------------
    slab_gemm<H>(dz, TT::LDA, bs, bs, [&](int row, int c4, float4 v) {
        if (r0 + row < u.bmax) {
            const float4 hv = *reinterpret_cast<const float4*>(h2 + (size_t)row * SLAB_NS + c4);
            *reinterpret_cast<float4*>(nv.s_dz1 + (size_t)(r0 + row) * H + c0 + c4) =
                make_float4(hv.x > 0.f ? v.x : 0.f, hv.y > 0.f ? v.y : 0.f, hv.z > 0.f ? v.z : 0.f, hv.w > 0.f ? v.w : 0.f);
        }
    });
}

// contiguous copy of the permuted batch (one launch per repeat): minibatch k is then rows
// [k*bs, (k+1)*bs) of g = obs[N][D] | act[N][A] | logp[N] | adv[C][N] | ret[C][N] | values[C][N]
__global__ void ppo_gather_kernel(const fsrl_ppo_update_t u, long long n) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const long long r = u.perm[i];
    const int D = u.D, A = u.A, C = u.C;
    float* g = u.gather;
    for (int k = 0; k < D; ++k) g[i * D + k] = u.obs[r * D + k];
    g += n * D;
    for (int k = 0; k < A; ++k) g[i * A + k] = u.act[r * A + k];
    g += n * A;
    g[i] = u.logp_old[r];
    g += n;
    for (int c = 0; c < C; ++c) g[(size_t)c * n + i] = u.adv[(size_t)c * u.ld + r];
    g += (size_t)C * n;
    for (int c = 0; c < C; ++c) g[(size_t)c * n + i] = u.ret[(size_t)c * u.ld + r];
    g += (size_t)C * n;
    if (u.values) for (int c = 0; c < C; ++c) g[(size_t)c * n + i] = u.values[(size_t)c * u.ld + r];
}

// ------------------------------------------------------------------------------------------
// Phase B: weight gradients
// ------------------------------------------------------------------------------------------
constexpr int WG_TPB = 256, WG_T = 64, WG_TKT = 32, WG_RC = 128, WG_NST = 2, WG_LD = WG_T + 8;   // LD = 8 mod 32: conflict-free fragments
// shared memory of a weight-gradient role: WG_NST stages x (L chunk + G chunk), each [WG_RC][WG_LD]
// (re-used as the cross-warp reduce buffer), then fin[80][WG_T] (layer-1 results) and 256 partials.
// (measured: 64-row chunks x 3 stages, 132 KB, which would let a forward CTA co-reside, is 4% slower)
constexpr size_t WG_SMEM_FLOATS = 2 * WG_NST * (size_t)WG_RC * WG_LD + 80 * WG_T + 256;
static_assert(2 * WG_NST * WG_RC * WG_LD >= 8 * 32 * (WG_T + 8), "reduce buffer must fit in the staging area");

// One staged chunk of the weight-gradient contraction  C[m][n] += sum_r L[r][m] * G[r][n]
// (m < 16 MT, n < 8 NT; r over the WG_RC rows of the chunk, 8 rows per k-step, k-steps dealt
// round-robin to the 8 warps) as split-TF32 MMAs.  A = L^T is read "column-major" straight from
// the row-major chunk: with LD = 8 (mod 32) both fragment loads are bank-conflict free.
template <int MT, int NT>
__device__ __forceinline__ void wg_mma_chunk(const float* __restrict__ L, const float* __restrict__ G,
                                             float (&c)[MT][NT][4]) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int g = lane >> 2, t = lane & 3;
#pragma unroll
    for (int ks = 0; ks < WG_RC / 64; ++ks) {
        const int r = (ks * 8 + warp) * 8;
        const float* g0 = G + (size_t)(r + t) * WG_LD + g;
        const float* l0 = L + (size_t)(r + t) * WG_LD + g;
        uint32_t bh[NT][2], bl[NT][2];
#pragma unroll
        for (int nt = 0; nt < NT; ++nt) {
            split_tf32(g0[8 * nt], bh[nt][0], bl[nt][0]);
            split_tf32(g0[(size_t)4 * WG_LD + 8 * nt], bh[nt][1], bl[nt][1]);
        }
#pragma unroll
        for (int mt = 0; mt < MT; ++mt) {
            uint32_t ah[4], al[4];
            split_tf32(l0[16 * mt], ah[0], al[0]);
            split_tf32(l0[16 * mt + 8], ah[1], al[1]);
            split_tf32(l0[(size_t)4 * WG_LD + 16 * mt], ah[2], al[2]);
            split_tf32(l0[(size_t)4 * WG_LD + 16 * mt + 8], ah[3], al[3]);
#pragma unroll
            for (int nt = 0; nt < NT; ++nt) mma_tf32(c[mt][nt], al, bh[nt]);
#pragma unroll
            for (int nt = 0; nt < NT; ++nt) mma_tf32(c[mt][nt], ah, bl[nt]);
#pragma unroll
            for (int nt = 0; nt < NT; ++nt) mma_tf32(c[mt][nt], ah, bh[nt]);
        }
    }
}

// this warp's partial C tile -> red[warp][16 MT][8 NT + 8]
template <int MT, int NT>
__device__ __forceinline__ void wg_store_partial(float* red, const float (&c)[MT][NT][4]) {
    constexpr int LDR = 8 * NT + 8;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int g = lane >> 2, t = lane & 3;
    float* mine = red + (size_t)warp * 16 * MT * LDR;
#pragma unroll
    for (int mt = 0; mt < MT; ++mt)
#pragma unroll
        for (int nt = 0; nt < NT; ++nt) {
            *reinterpret_cast<float2*>(mine + (size_t)(16 * mt + g) * LDR + 8 * nt + 2 * t) = make_float2(c[mt][nt][0], c[mt][nt][1]);
            *reinterpret_cast<float2*>(mine + (size_t)(16 * mt + g + 8) * LDR + 8 * nt + 2 * t) = make_float2(c[mt][nt][2], c[mt][nt][3]);
        }
}
// sum over the 8 warps of 4 consecutive columns of the reduced tile
template <int MT, int NT>
__device__ __forceinline__ float4 wg_reduced4(const float* red, int m, int n4) {
    constexpr int LDR = 8 * NT + 8;
    float4 s4 = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
    for (int w = 0; w < 8; ++w) {
        const float4 v = *reinterpret_cast<const float4*>(red + ((size_t)w * 16 * MT + m) * LDR + n4);
        s4.x += v.x; s4.y += v.y; s4.z += v.z; s4.w += v.w;
    }
    return s4;
}

// Device-wide barrier for co-resident grids (cooperative launch): monotonically increasing ticket
// counter, one arrival per CTA, spin on an acquire load.
__device__ __forceinline__ void grid_barrier(unsigned long long* counter, unsigned long long target) {
    __syncthreads();
    if (threadIdx.x == 0) {
        __threadfence();
        atomicAdd(counter, 1ULL);
        unsigned long long v;
        const long long t0 = clock64();
        do {
            asm volatile("ld.acquire.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(counter));
            // a grid that is not co-resident would spin forever: fail loudly instead of hanging the GPU
            if (v < target && clock64() - t0 > 20000000000LL) asm volatile("trap;");
        } while (v < target);
        __threadfence();
    }
    __syncthreads();
}

// Roles by `bx` (per net): [0, NT)            dW2t tiles 32(k) x 64(o); k-tile 0 also owns db2
//                          [NT, NT+NTO)       layer 1: dW1t[:, o-tile], db1[o-tile]
//                          [NT+NTO, NT+2NTO)  layer 3: dW3t[k-tile, :] (+ db3, dlog_sigma)
// Every role streams the minibatch through a cp.async double buffer of 64-row chunks.  With
// FUSED the role keeps its gradient tile in registers, joins a grid barrier (the global norm is
// then complete) and applies clip + Adam to the parameters it owns -- no gradient round trip.
template <int H, bool FUSED>
__device__ __forceinline__ void ppo_wgrad_role(const fsrl_ppo_update_t& u, int mb_off, int B, int bx, int net,
                                               float* smem, const AdamStep ad, unsigned long long* bar,
                                               unsigned long long bar_target, int slot) {
    constexpr int NTT = H / WG_T, NTKT = H / WG_TKT, NT = NTKT * NTT;
    __shared__ float s_red[WG_TPB / 32];
    const int tid = threadIdx.x;
    const NetView nv = net_view(u, net);
    constexpr size_t WG_CHUNK = (size_t)WG_RC * WG_LD;
    auto sLp = [&](int buf) { return smem + (size_t)(2 * buf) * WG_CHUNK; };
    auto sGp = [&](int buf) { return smem + (size_t)(2 * buf + 1) * WG_CHUNK; };
    const int nchunk = (B + WG_RC - 1) / WG_RC;
    float sq = 0.f;
    // generic chunk loader: `wl` / `wg` floats per row from row-major sources with strides sl / sg
    auto stage = [&](int ch, int buf, const float* srcL, int strideL, int offL, int wl,
                     const float* srcG, int strideG, int offG, int wg) {
        const int rb = ch * WG_RC;
        for (int i = tid; i < WG_RC * (wl / 4); i += WG_TPB) {
            const int rr = i / (wl / 4), c4 = (i % (wl / 4)) * 4;
            float* dst = sLp(buf) + (size_t)rr * WG_LD + c4;
            if (rb + rr < B) __pipeline_memcpy_async(dst, srcL + (size_t)(rb + rr) * strideL + offL + c4, 16);
            else *reinterpret_cast<float4*>(dst) = make_float4(0.f, 0.f, 0.f, 0.f);
        }
        for (int i = tid; i < WG_RC * (wg / 4); i += WG_TPB) {
            const int rr = i / (wg / 4), c4 = (i % (wg / 4)) * 4;
            float* dst = sGp(buf) + (size_t)rr * WG_LD + c4;
            if (rb + rr < B) __pipeline_memcpy_async(dst, srcG + (size_t)(rb + rr) * strideG + offG + c4, 16);
            else *reinterpret_cast<float4*>(dst) = make_float4(0.f, 0.f, 0.f, 0.f);
        }
        __pipeline_commit();
    };
    // WG_NST-deep cp.async pipeline over the row chunks: stg(chunk, buffer) issues one commit group,
    // body(buffer) consumes a landed chunk
    auto pipeline = [&](auto&& stg, auto&& body) {
        for (int p = 0; p < WG_NST - 1; ++p) { if (p < nchunk) stg(p, p); else __pipeline_commit(); }
        for (int ch = 0; ch < nchunk; ++ch) {
            const int nx = ch + WG_NST - 1;
            if (nx < nchunk) stg(nx, nx % WG_NST); else __pipeline_commit();
            __pipeline_wait_prior(WG_NST - 1);
            __syncthreads();
            body(ch % WG_NST);
            __syncthreads();
        }
    };
    pdl_wait();            // dz1 / dz2 / dout of this minibatch are complete
    pdl_trigger();
    float gscale = 1.0f;   // clip coefficient (FUSED)
    auto finish = [&]() {  // norm contribution (+ barrier and clip scale when fused)
        const float tot = block_sum_256(sq, s_red);
        if (tid == 0 && tot != 0.f && u.world <= 1) atomicAdd(u.norm_sq, tot);   // DP: the norm of the REDUCED gradient is taken later
        if (FUSED) {
            grid_barrier(bar, bar_target);
            const float nsq = __ldcg(u.norm_sq);
            if (u.max_grad_norm > 0.f) gscale = fminf(u.max_grad_norm / (sqrtf(nsq) + 1e-6f), 1.0f);
            if (bx == 0 && net == 0 && tid == 0 && u.stats && slot >= 0)
                u.stats[(size_t)slot * FSRL_PPO_STATS + ST_GRADNORM] = sqrtf(nsq);
        }
    };
    const long long pbase = u.net_off[net];
    const NetLayout L = ppo_layout(u, net, H);
    if (bx < NT) {
        // ---- dW2t[k][o] = sum_r h1[r][k] * dz2[r][o] : 32 x 64 tile, 2 x 4 per thread (FFMA issue is the
        // bound on this chip, so the tiles are sized to spread over ~all SMs) ---------------------------
        const int k0 = (bx / NTT) * WG_TKT, o0 = (bx % NTT) * WG_T;
        const int tk = tid / 16, to = tid % 16;
        const bool do_bias = (k0 == 0);
        float c[2][8][4];
#pragma unroll
        for (int mt = 0; mt < 2; ++mt)
#pragma unroll
            for (int nt = 0; nt < 8; ++nt) { c[mt][nt][0] = c[mt][nt][1] = c[mt][nt][2] = c[mt][nt][3] = 0.f; }
        float bpart = 0.f;                                  // db2: thread (o = tid % 64, row group tid / 64)
        pipeline([&](int ch, int buf) { stage(ch, buf, nv.s_h1, H, k0, WG_TKT, nv.s_dz2, H, o0, WG_T); },
                 [&](int buf) {
                     wg_mma_chunk<2, 8>(sLp(buf), sGp(buf), c);
                     if (do_bias) {
                         const float* G = sGp(buf) + (tid % WG_T);
#pragma unroll 8
                         for (int rr = tid / WG_T; rr < WG_RC; rr += WG_TPB / WG_T) bpart += G[(size_t)rr * WG_LD];
                     }
                 });
        float* red = smem;                                  // staging is dead: cross-warp reduction buffer
        float* bred = smem + 2 * WG_NST * WG_CHUNK + 80 * WG_T;      // [4][WG_T] bias partials
        wg_store_partial<2, 8>(red, c);
        if (do_bias) bred[tid] = bpart;
        __syncthreads();
        float acc[2][4];
#pragma unroll
        for (int i = 0; i < 2; ++i) {
            const float4 v = wg_reduced4<2, 8>(red, 2 * tk + i, 4 * to);
            acc[i][0] = v.x; acc[i][1] = v.y; acc[i][2] = v.z; acc[i][3] = v.w;
        }
        float bsum = 0.f;
        if (do_bias && tid < WG_T) bsum = bred[tid] + bred[WG_T + tid] + bred[2 * WG_T + tid] + bred[3 * WG_T + tid];
#pragma unroll
        for (int i = 0; i < 2; ++i) sq += acc[i][0] * acc[i][0] + acc[i][1] * acc[i][1] + acc[i][2] * acc[i][2] + acc[i][3] * acc[i][3];
        if (do_bias && tid < WG_T) sq += bsum * bsum;
        finish();
        if (!FUSED) {
#pragma unroll
            for (int i = 0; i < 2; ++i)
                *reinterpret_cast<float4*>(nv.g_w2t + (size_t)(k0 + 2 * tk + i) * H + o0 + 4 * to) =
                    make_float4(acc[i][0], acc[i][1], acc[i][2], acc[i][3]);
            if (do_bias && tid < WG_T) nv.g_b2[o0 + tid] = bsum;
        } else {
            const long long w2s = pbase + L.w2;
            float np[2][4];
#pragma unroll
            for (int i = 0; i < 2; ++i) {
                const long long idx = w2s + (long long)(k0 + 2 * tk + i) * H + o0 + 4 * to;
                float4 p = *reinterpret_cast<float4*>(u.theta + idx);
                float4 m = *reinterpret_cast<float4*>(u.adam_m + idx);
                float4 v = *reinterpret_cast<float4*>(u.adam_v + idx);
                p.x = adam_one(p.x, acc[i][0] * gscale, m.x, v.x, ad); p.y = adam_one(p.y, acc[i][1] * gscale, m.y, v.y, ad);
                p.z = adam_one(p.z, acc[i][2] * gscale, m.z, v.z, ad); p.w = adam_one(p.w, acc[i][3] * gscale, m.w, v.w, ad);
                *reinterpret_cast<float4*>(u.theta + idx) = p;
                *reinterpret_cast<float4*>(u.adam_m + idx) = m;
                *reinterpret_cast<float4*>(u.adam_v + idx) = v;
                np[i][0] = p.x; np[i][1] = p.y; np[i][2] = p.z; np[i][3] = p.w;
            }
            float* mir = u.w2n + (size_t)net * H * H;      // out-major mirror: [o][k]
#pragma unroll
            for (int j = 0; j < 4; ++j)
                *reinterpret_cast<float2*>(mir + (size_t)(o0 + 4 * to + j) * H + k0 + 2 * tk) = make_float2(np[0][j], np[1][j]);
            if (do_bias && tid < WG_T) {
                const long long idx = pbase + L.b2 + o0 + tid;
                float m = u.adam_m[idx], v = u.adam_v[idx];
                u.theta[idx] = adam_one(u.theta[idx], bsum * gscale, m, v, ad);
                u.adam_m[idx] = m; u.adam_v[idx] = v;
            }
        }
    } else if (bx < NT + NTT) {
        // ---- layer 1: dW1t[d][o] = sum_r x[r][d] * dz1[r][o];  db1[o] = sum_r dz1[r][o] ---------
        // Inputs go through the MMA in passes of 16 "virtual" columns v: v < D is observation column v,
        // v == D is a column of ones (its output row is the bias gradient), the rest is zero padding.
        // Results land in fin[v][o] (shared), which survives the grid barrier of the fused variant.
        const int D = u.D;
        const int o0 = (bx - NT) * WG_T;
        const int o = tid % WG_T;
        const int rg = tid / WG_T;
        float* fin = smem + 2 * WG_NST * WG_CHUNK;                   // [16 npass][WG_T]
        auto stage1 = [&](int ch, int buf, int v0) {
            const int rb = ch * WG_RC;
            float* xs_ = sLp(buf);
            float* gs_ = sGp(buf);
            if ((D & 3) == 0) {            // 16-byte segments: a segment is entirely data or entirely padding
                for (int i = tid; i < WG_RC * 4; i += WG_TPB) {
                    const int rr = i / 4, v = v0 + 4 * (i % 4);
                    float* dst = xs_ + (size_t)rr * WG_LD + 4 * (i % 4);
                    if (rb + rr < B && v < D) __pipeline_memcpy_async(dst, u.obs + (size_t)row_of(u, mb_off, rb + rr) * D + v, 16);
                    else *reinterpret_cast<float4*>(dst) = make_float4((rb + rr < B && v == D) ? 1.0f : 0.f, 0.f, 0.f, 0.f);
                }
            } else {
                for (int i = tid; i < WG_RC * 16; i += WG_TPB) {
                    const int rr = i / 16, v = v0 + (i % 16);
                    float* dst = xs_ + (size_t)rr * WG_LD + (i % 16);
                    if (rb + rr < B && v < D) __pipeline_memcpy_async(dst, u.obs + (size_t)row_of(u, mb_off, rb + rr) * D + v, 4);
                    else *dst = (rb + rr < B && v == D) ? 1.0f : 0.f;
                }
            }
            for (int i = tid; i < WG_RC * (WG_T / 4); i += WG_TPB) {
                const int rr = i / (WG_T / 4), c4 = (i % (WG_T / 4)) * 4;
                float* dst = gs_ + (size_t)rr * WG_LD + c4;
                if (rb + rr < B) __pipeline_memcpy_async(dst, nv.s_dz1 + (size_t)(rb + rr) * H + o0 + c4, 16);
                else *reinterpret_cast<float4*>(dst) = make_float4(0.f, 0.f, 0.f, 0.f);
            }
            __pipeline_commit();
        };
        const int npass = (D + 1 + 15) / 16;
        for (int ps = 0; ps < npass; ++ps) {
            float c[1][8][4];
#pragma unroll
            for (int nt = 0; nt < 8; ++nt) { c[0][nt][0] = c[0][nt][1] = c[0][nt][2] = c[0][nt][3] = 0.f; }
            pipeline([&](int ch, int buf) { stage1(ch, buf, 16 * ps); },
                     [&](int buf) { wg_mma_chunk<1, 8>(sLp(buf), sGp(buf), c); });
            float* red = smem;
            wg_store_partial<1, 8>(red, c);
            __syncthreads();
            {
                const int m = tid / 16, n4 = (tid % 16) * 4;        // 16 x 64 outputs, 4 per thread
                *reinterpret_cast<float4*>(fin + (size_t)(16 * ps + m) * WG_T + n4) = wg_reduced4<1, 8>(red, m, n4);
            }
            __syncthreads();
        }
        // every thread now owns the outputs (d, o) with d = rg, rg + 4, ... < D; bias: rg == 0
        for (int d = rg; d < D; d += 4) { const float g = fin[(size_t)d * WG_T + o]; sq += g * g; }
        if (rg == 0) { const float g = fin[(size_t)D * WG_T + o]; sq += g * g; }
        finish();
        for (int d = rg; d < D; d += 4) {
            const float g = fin[(size_t)d * WG_T + o];
            if (!FUSED) nv.g_w1t[(size_t)d * H + o0 + o] = g;
            else {
                const long long idx = pbase + L.w1 + (long long)d * H + o0 + o;
                float m = u.adam_m[idx], v = u.adam_v[idx];
                u.theta[idx] = adam_one(u.theta[idx], g * gscale, m, v, ad);
                u.adam_m[idx] = m; u.adam_v[idx] = v;
            }
        }
        if (rg == 0) {
            const float g = fin[(size_t)D * WG_T + o];
            if (!FUSED) nv.g_b1[o0 + o] = g;
            else {
                const long long idx = pbase + L.b1 + o0 + o;
                float m = u.adam_m[idx], v = u.adam_v[idx];
                u.theta[idx] = adam_one(u.theta[idx], g * gscale, m, v, ad);
                u.adam_m[idx] = m; u.adam_v[idx] = v;
            }
        }
    } else {
        // ---- layer 3: dW3t[k][j] = sum_r h2[r][k] * dout[r][j];  db3;  dlog_sigma ------------------
        const int out = nv.m.out;
        const int A = u.A;
        const int k0 = (bx - NT - NTT) * WG_T;
        const int k = tid % WG_T, jg = tid / WG_T;          // j = 4*jg + q
        float c[4][2][4];
#pragma unroll
        for (int mt = 0; mt < 4; ++mt)
#pragma unroll
            for (int nt = 0; nt < 2; ++nt) { c[mt][nt][0] = c[mt][nt][1] = c[mt][nt][2] = c[mt][nt][3] = 0.f; }
        float cpart = 0.f;                                  // column sums of dout: thread (j = tid % 16, row group tid / 16)
        pipeline([&](int ch, int buf) { stage(ch, buf, nv.s_h2, H, k0, WG_T, nv.s_dout, DOUT_LD, 0, DOUT_LD); },
                 [&](int buf) {
                     wg_mma_chunk<4, 2>(sLp(buf), sGp(buf), c);
                     if (k0 == 0) {
                         const float* Dd = sGp(buf) + (tid % DOUT_LD);
#pragma unroll
                         for (int rr = tid / DOUT_LD; rr < WG_RC; rr += WG_TPB / DOUT_LD) cpart += Dd[(size_t)rr * WG_LD];
                     }
                 });
        float* red = smem;
        float* cred = smem + 2 * WG_NST * WG_CHUNK + 80 * WG_T;      // [16][DOUT_LD] column-sum partials
        wg_store_partial<4, 2>(red, c);
        if (k0 == 0) cred[tid] = cpart;
        __syncthreads();
        float acc[4];
        {
            const float4 v = wg_reduced4<4, 2>(red, k, 4 * jg);
            acc[0] = v.x; acc[1] = v.y; acc[2] = v.z; acc[3] = v.w;
        }
        float csum = 0.f;
        if (k0 == 0 && tid < DOUT_LD) {
#pragma unroll
            for (int q = 0; q < WG_TPB / DOUT_LD; ++q) csum += cred[q * DOUT_LD + tid];
        }
        const bool own_b3 = (k0 == 0) && tid < out;
        const bool own_ls = (k0 == 0) && net == 0 && u.head_indep && tid >= A && tid < 2 * A && tid < DOUT_LD;
#pragma unroll
        for (int q = 0; q < 4; ++q) if (4 * jg + q < out) sq += acc[q] * acc[q];
        if (own_b3 || own_ls) sq += csum * csum;
        finish();
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const int j = 4 * jg + q;
            if (j < out) {
                if (!FUSED) nv.g_w3t[(size_t)(k0 + k) * out + j] = acc[q];
                else {
                    const long long idx = pbase + L.w3 + (long long)(k0 + k) * out + j;
                    float m = u.adam_m[idx], v = u.adam_v[idx];
                    u.theta[idx] = adam_one(u.theta[idx], acc[q] * gscale, m, v, ad);
                    u.adam_m[idx] = m; u.adam_v[idx] = v;
                }
            }
        }
        if (own_b3 || own_ls) {
            const long long idx = own_b3 ? pbase + L.b3 + tid : pbase + L.extra + (tid - A);
            if (!FUSED) { if (own_b3) nv.g_b3[tid] = csum; else nv.g_log_sigma[tid - A] = csum; }
            else {
                float m = u.adam_m[idx], v = u.adam_v[idx];
                u.theta[idx] = adam_one(u.theta[idx], csum * gscale, m, v, ad);
                u.adam_m[idx] = m; u.adam_v[idx] = v;
            }
        }
    }
}

template <int H>
__global__ void __launch_bounds__(WG_TPB)
ppo_wgrad_kernel(const fsrl_ppo_update_t u, int mb_off, int B) {
    extern __shared__ __align__(16) float smem[];
    ppo_wgrad_role<H, false>(u, mb_off, B, blockIdx.x, blockIdx.y, smem, AdamStep{}, nullptr, 0ULL, -1);
}

// weight gradients + clip_grad_norm_ + Adam in one launch with a grid barrier (single-GPU path)
template <int H>
__global__ void __launch_bounds__(WG_TPB)
ppo_wgrad_adam_kernel(const fsrl_ppo_update_t u, int mb_off, int B, AdamStep ad, unsigned long long* bar,
                      unsigned long long bar_target, int slot) {
    extern __shared__ __align__(16) float smem[];
    ppo_wgrad_role<H, true>(u, mb_off, B, blockIdx.x, blockIdx.y, smem, ad, bar, bar_target, slot);
}

// ------------------------------------------------------------------------------------------
// Phase C: clip_grad_norm_ + Adam (torch.optim.Adam single-tensor arithmetic order)
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
adam_kernel(const fsrl_ppo_update_t u, const AdamStep ad, int slot, int n_plain_blocks) {
    __shared__ float tile[32][33];
    __shared__ float nred[8];
    pdl_wait();                        // gradients / norm partials of this step are complete
    pdl_trigger();
    const float gs = (u.world > 1) ? 1.0f / (float)u.world : 1.0f;     // average the summed gradients
    float scale = gs;
    float nsq_raw;
    if (u.world > 1 && u.p2p_on) {       // deterministic (rank-identical) sum of the per-CTA partials
        const int nblk = (int)((u.n_params + 1023) / 1024);
        float sp = 0.f;
        for (int i = threadIdx.x; i < nblk; i += 256) sp += __ldcg(u.p2p_part + i);
        nsq_raw = block_sum_256(sp, nred);
    } else {
        nsq_raw = *u.norm_sq;
    }
    const float nsq = nsq_raw * gs * gs;
    if (u.max_grad_norm > 0.f) {
        const float coef = u.max_grad_norm / (sqrtf(nsq) + 1e-6f);
        scale = gs * fminf(coef, 1.0f);
    }
    if (blockIdx.x == 0 && threadIdx.x == 0 && u.stats && slot >= 0)
        u.stats[(size_t)slot * FSRL_PPO_STATS + ST_GRADNORM] = sqrtf(nsq);
    const int H = u.H;
    if ((int)blockIdx.x < n_plain_blocks) {
        // everything except the W2 matrices: compact enumeration (layer 1 + bias, then b2 / layer 3 / extras
        // of each net), so only ceil(plain / 256) blocks are launched for it
        long long cc = (long long)blockIdx.x * 256 + threadIdx.x;
        long long i = -1;
        for (int n = 0; n < u.n_nets; ++n) {
            const long long size = ((n + 1 < u.n_nets) ? u.net_off[n + 1] : u.n_params) - u.net_off[n];
            const NetLayout L = ppo_layout(u, n, H);
            const long long pre = L.w2, post = size - L.b2;
            if (cc < pre) { i = u.net_off[n] + cc; break; }
            cc -= pre;
            if (cc < post) { i = u.net_off[n] + L.b2 + cc; break; }
            cc -= post;
        }
        if (i < 0) return;
        float m = u.adam_m[i], v = u.adam_v[i];
        const float g = (u.mask && u.mask[i] == 0) ? 0.f : u.grad[i] * scale;
        if (u.mask && u.mask[i] == 0) return;
        u.theta[i] = adam_one(u.theta[i], g, m, v, ad);
        u.adam_m[i] = m; u.adam_v[i] = v;
    } else {
        // W2 tiles: 32 x 32, update canonical W2t[k][o] and its mirror W2n[o][k]
        const int tpn = (H / 32) * (H / 32);
        const int t = blockIdx.x - n_plain_blocks;
        const int n = t / tpn;
        int k0, o0;
        w2_tile_origin(t % tpn, H, k0, o0);
        const long long base = u.net_off[n] + ppo_layout(u, n, H).w2;
        const int lx = threadIdx.x % 32, ly = threadIdx.x / 32;
        const bool frozen = u.mask && u.mask[base] == 0;
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const int kk = ly + 8 * q;
            const long long i = base + (long long)(k0 + kk) * H + o0 + lx;
            float p = u.theta[i];
            if (!frozen) {
                float m = u.adam_m[i], v = u.adam_v[i];
                p = adam_one(p, u.grad[i] * scale, m, v, ad);
                u.theta[i] = p; u.adam_m[i] = m; u.adam_v[i] = v;
            }
            tile[kk][lx] = p;
        }
        w2_tile_store_mirror(tile, u.w2n + (size_t)n * H * H, H, k0, o0);
    }
}

// Data-parallel gradient exchange over peer memory (NVLink), fused with the norm of the reduced
// gradient: every rank's weight-gradient kernel wrote its local gradient into its own exchange
// buffer (parity id & 1); this kernel (1) tells every peer "my step `id` is complete" by a
// system-scope release store into the peer's flag array, (2) waits until all ranks' flags reached
// `id`, (3) sums the ranks' buffers in rank order -- one 16-byte load per rank and element group,
// all in flight together -- into u.grad and accumulates sum g^2.  Every rank computes the same
// sum in the same order: parameters stay bit-identical without a broadcast.  Two buffers suffice:
// a rank can only overwrite parity b again after the barrier of step id + 1, which every peer
// joins after it has finished reading step id.
constexpr long long P2P_TIMEOUT_CYCLES = 40000000000LL;     // ~20 s: a missing peer must not hang the GPU
__global__ void __launch_bounds__(256) ppo_dp_reduce_kernel(const fsrl_ppo_update_t u, unsigned long long id) {
    __shared__ float red[8];
    pdl_wait();                       // the local weight gradients are complete
    pdl_trigger();
    const int tid = threadIdx.x;
    if (blockIdx.x == 0 && tid < u.world) {
        __threadfence_system();
        unsigned long long* f = u.p2p_flags[tid] + u.p2p_rank;
        asm volatile("st.release.sys.global.u64 [%0], %1;" :: "l"(f), "l"(id) : "memory");
    }
    if (tid < u.world) {
        const unsigned long long* f = u.p2p_flags[u.p2p_rank] + tid;
        const long long t0 = clock64();
        unsigned long long v;
        do {
            asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(f) : "memory");
        } while (v < id && clock64() - t0 < P2P_TIMEOUT_CYCLES);
        if (v < id) *u.p2p_err = 1;
    }
    __syncthreads();
    const int par = (int)(id & 1ULL);
    const long long i4 = ((long long)blockIdx.x * 256 + tid) * 4;
    float sq = 0.f;
    if (i4 < u.n_params) {
        float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
        float4 v[FSRL_P2P_MAX_RANKS];
#pragma unroll
        for (int r = 0; r < FSRL_P2P_MAX_RANKS; ++r) {
            if (r < u.world) {
                const float* src = u.p2p_xg[par][r] + i4;      // buffers are padded: the float4 never leaves them
                asm volatile("ld.volatile.global.v4.f32 {%0,%1,%2,%3}, [%4];"
                             : "=f"(v[r].x), "=f"(v[r].y), "=f"(v[r].z), "=f"(v[r].w) : "l"(src));
            }
        }
#pragma unroll
        for (int r = 0; r < FSRL_P2P_MAX_RANKS; ++r) {
            if (r < u.world) { acc.x += v[r].x; acc.y += v[r].y; acc.z += v[r].z; acc.w += v[r].w; }
        }
        if (i4 + 3 < u.n_params) {
            *reinterpret_cast<float4*>(u.grad + i4) = acc;
            sq = acc.x * acc.x + acc.y * acc.y + acc.z * acc.z + acc.w * acc.w;
        } else {
            const float a[4] = {acc.x, acc.y, acc.z, acc.w};
            for (int q = 0; q < 4 && i4 + q < u.n_params; ++q) { u.grad[i4 + q] = a[q]; sq += a[q] * a[q]; }
        }
    }
    const float tot = block_sum_256(sq, red);
    if (tid == 0) u.p2p_part[blockIdx.x] = tot;     // no atomics: the Adam kernel sums these in a fixed order
}

// sum of squares of the (all-reduced) gradient buffer -> *u.norm_sq
__global__ void __launch_bounds__(1024) grad_norm_kernel(const fsrl_ppo_update_t u) {
    __shared__ float red[32];
    float s = 0.f;
    for (long long i = threadIdx.x; i < u.n_params; i += 1024) { const float g = u.grad[i]; s += g * g; }
    s = warp_sum(s);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
    __syncthreads();
    if (threadIdx.x == 0) { float t = 0.f; for (int w = 0; w < 32; ++w) t += red[w]; *u.norm_sq = t; }
}

// per-minibatch sum and sum of squares of the advantages (block b = minibatch b of the repeat)
__global__ void __launch_bounds__(256) ppo_adv_moments_kernel(const fsrl_ppo_update_t u, long long n_total, int n_mb) {
    __shared__ double red[2][8];
    const int mb = blockIdx.x;
    const long long off = (long long)mb * u.batch_size;
    long long B = u.batch_size;
    if (mb == n_mb - 1) B = n_total - off;
    for (int c = 0; c < u.C; ++c) {
        double s = 0.0, q = 0.0;
        for (long long i = threadIdx.x; i < B; i += 256) {
            const double a = (double)u.adv[(size_t)c * u.ld + (u.perm ? (long long)u.perm[off + i] : off + i)];
            s += a; q += a * a;
        }
        s = warp_sum(s); q = warp_sum(q);
        __syncthreads();
        if ((threadIdx.x & 31) == 0) { red[0][threadIdx.x >> 5] = s; red[1][threadIdx.x >> 5] = q; }
        __syncthreads();
        if (threadIdx.x == 0) {
            double ts = 0.0, tq = 0.0;
            for (int w = 0; w < 8; ++w) { ts += red[0][w]; tq += red[1][w]; }
            u.moments_w[((size_t)mb * 2 + c) * 2] = ts;
            u.moments_w[((size_t)mb * 2 + c) * 2 + 1] = tq;
        }
    }
}

// mean and 1/std (unbiased, no eps: ppo_lag.py:181-182) of the advantages of every minibatch of
// the repeat: block b = minibatch b.  In a data-parallel run the sums were all-reduced first.
__global__ void __launch_bounds__(256) ppo_adv_stats_kernel(const fsrl_ppo_update_t u, long long n_total, int n_mb) {
    __shared__ double red[8];
    __shared__ double s_m;
    const int mb = blockIdx.x;
    const long long off = (long long)mb * u.batch_size;
    long long B = u.batch_size;
    if (mb == n_mb - 1) B = n_total - off;
    for (int c = 0; c < u.C; ++c) {
        float* out = u.mb_stats + ((size_t)mb * 2 + c) * 2;
        if (!u.norm_adv) { if (threadIdx.x == 0) { out[0] = 0.f; out[1] = 1.f; } continue; }
        if (u.moments) {
            if (threadIdx.x == 0) {
                const double* mo = u.moments + ((size_t)mb * 2 + c) * 2;
                const double nn = (double)B * (double)u.world;
                const double mean = mo[0] / nn;
                const double var = (mo[1] - nn * mean * mean) / (nn - 1.0);
                out[0] = (float)mean; out[1] = (float)(1.0 / sqrt(var));
            }
            continue;
        }
        // two-pass like torch: mean in fp32 arithmetic would differ in the last bits only; use f64 sums
        double sacc = 0.0;
        for (long long i = threadIdx.x; i < B; i += 256)
            sacc += (double)u.adv[(size_t)c * u.ld + (u.perm ? (long long)u.perm[off + i] : off + i)];
        sacc = warp_sum(sacc);
        __syncthreads();
        if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = sacc;
        __syncthreads();
        if (threadIdx.x == 0) { double t = 0.0; for (int w = 0; w < 8; ++w) t += red[w]; s_m = t / (double)B; }
        __syncthreads();
        const float mean = (float)s_m;
        double q = 0.0;
        for (long long i = threadIdx.x; i < B; i += 256) {
            const float d = u.adv[(size_t)c * u.ld + (u.perm ? (long long)u.perm[off + i] : off + i)] - mean;
            q += (double)(d * d);
        }
        q = warp_sum(q);
        __syncthreads();
        if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = q;
        __syncthreads();
        if (threadIdx.x == 0) {
            double t = 0.0; for (int w = 0; w < 8; ++w) t += red[w];
            out[0] = mean; out[1] = 1.0f / sqrtf((float)(t / (double)(B - 1)));
        }
    }
}

extern "C" int fsrl_allreduce_fused(void* comm, float* buf, long long n, void* stream);
extern "C" int fsrl_allreduce_f64(void* comm, double* buf, long long n, void* stream);

// blocks of adam_kernel that cover the parameters outside the W2 matrices (compact enumeration)
static int adam_plain_blocks(const fsrl_ppo_update_t& u, int H) {
    const long long plain = u.n_params - (long long)u.n_nets * H * H;
    return (int)((plain + 255) / 256);
}

// One link of the per-minibatch kernel chain: programmatic dependent launch (see pdl_wait), plus
// the cooperative attribute for the kernel that contains the grid barrier.
template <class... KArgs, class... Args>
static cudaError_t launch_chain(void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t s,
                                bool cooperative, Args... args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = s;
    cudaLaunchAttribute at[2];
    int n = 0;
    at[n].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at[n].val.programmaticStreamSerializationAllowed = 1;
    ++n;
    if (cooperative) { at[n].id = cudaLaunchAttributeCooperative; at[n].val.cooperative = 1; ++n; }
    cfg.attrs = at; cfg.numAttrs = n;
    ++g_launches;
    return cudaLaunchKernelEx(&cfg, kern, static_cast<KArgs>(args)...);
}

template <int H>
static int ppo_launch_minibatch(const fsrl_ppo_update_t& u, int mb_off, int B, int slot,
                                long long adam_t, long long bar_count, cudaStream_t s) {
    using TT = MlpTile<H>;
    const size_t smemF = sizeof(float) * ((size_t)TT::R * TT::in_pad(u.D) + (size_t)TT::R * TT::LDA + slab_buf_floats<H>());
    const size_t smemB = sizeof(float) * (2 * (size_t)TT::R * TT::LDA + slab_buf_floats<H>() + (size_t)H * (u.actor_out > 1 ? u.actor_out : 1) + (size_t)TT::R * DOUT_LD);
    static size_t setF = 0, setB = 0;                   // largest opt-in so far (D / actor_out vary per policy)
    if (smemF > setF) {
        FSRL_CUDA(cudaFuncSetAttribute(ppo_fwd_kernel<H>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smemF));
        setF = smemF;
    }
    if (smemB > setB) {
        FSRL_CUDA(cudaFuncSetAttribute(ppo_bwd_kernel<H>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smemB));
        setB = smemB;
    }
    const dim3 gA((B + TT::R - 1) / TT::R, H / SLAB_NS, u.n_nets);
    FSRL_CUDA(launch_chain(ppo_fwd_kernel<H>, gA, dim3(MLP_TPB), smemF, s, false, u, mb_off, B));
    FSRL_CUDA(launch_chain(ppo_bwd_kernel<H>, gA, dim3(MLP_TPB), smemB, s, false, u, mb_off, B, slot));
    constexpr int NTT = H / WG_T;
    const dim3 gB((H / WG_TKT) * NTT + 2 * NTT, u.n_nets);
    const size_t smemW = sizeof(float) * WG_SMEM_FLOATS;
    static bool attr_w = false;
    static int fuse_ok = -1;
    if (!attr_w) {
        FSRL_CUDA(cudaFuncSetAttribute(ppo_wgrad_kernel<H>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smemW));
        FSRL_CUDA(cudaFuncSetAttribute(ppo_wgrad_adam_kernel<H>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smemW));
        int per_sm = 0;
        FSRL_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, ppo_wgrad_adam_kernel<H>, WG_TPB, smemW));
        fuse_ok = (per_sm * sm_count() >= (int)(gB.x * 3)) ? 1 : 0;     // whole grid co-resident?
        attr_w = true;
    }
    // torch.optim.Adam scalars (python doubles -> f32 at the op)
    const double b1 = u.beta1, b2 = u.beta2;
    const double bc1 = 1.0 - pow(b1, (double)adam_t), bc2 = 1.0 - pow(b2, (double)adam_t);
    const AdamStep ad = {(float)(1.0 - b1), (float)b2, (float)(1.0 - b2), (float)sqrt(bc2), (float)u.adam_eps,
                         (float)(-(u.lr / bc1))};
    if (u.world <= 1 && fuse_ok == 1 && u.barrier != nullptr && u.mask == nullptr) {
        // single GPU: gradients never leave the registers -- tiles -> norm -> barrier -> clip + Adam
        unsigned long long target = (unsigned long long)(bar_count + 1) * gB.x * gB.y;
        // Ordinary (not cooperative) launch: measured 4.6 % faster per cycle.  The grid barrier is still
        // safe: fuse_ok guarantees grid <= SMs x CTAs/SM, every CTA of the grid becomes resident without
        // waiting on anything but the barrier (the preceding bwd CTAs drain unconditionally, the next fwd
        // CTAs are only scheduled after ALL of these have triggered), and grid_barrier traps after 20 s
        // instead of spinning forever should that reasoning ever be violated.
        FSRL_CUDA(launch_chain(ppo_wgrad_adam_kernel<H>, gB, dim3(WG_TPB), smemW, s, false, u, mb_off, B, ad, u.barrier,
                               target, slot));
        return FSRL_OK;
    }
    if (u.world > 1 && u.p2p_on) {
        // data parallel over peer memory: wgrad -> own exchange buffer, then signal / wait / sum / norm
        const unsigned long long id = (unsigned long long)adam_t;
        fsrl_ppo_update_t ux = u;
        ux.grad = const_cast<float*>(u.p2p_xg[id & 1ULL][u.p2p_rank]);
        FSRL_CUDA(launch_chain(ppo_wgrad_kernel<H>, gB, dim3(WG_TPB), smemW, s, false, ux, mb_off, B));
        const unsigned nblk = (unsigned)((u.n_params + 1023) / 1024);
        FSRL_CUDA(launch_chain(ppo_dp_reduce_kernel, dim3(nblk), dim3(256), (size_t)0, s, false, u, id));
    } else {
    FSRL_CUDA(launch_chain(ppo_wgrad_kernel<H>, gB, dim3(WG_TPB), smemW, s, false, u, mb_off, B));
    }
    if (u.world > 1 && !u.p2p_on) {
        // data parallel: ONE all-reduce of the flat gradient buffer per optimiser step, then the
        // global norm of the reduced gradient (the local partial norms are meaningless now)
        int rc = fsrl_allreduce_fused(u.comm, u.grad, u.n_params, s);
        if (rc) return rc;
        grad_norm_kernel<<<1, 1024, 0, s>>>(u);
        FSRL_LAUNCH_CHECK();
    }
    const int n_plain = adam_plain_blocks(u, H);
    const int n_tiles = u.n_nets * (H / 32) * (H / 32);
    FSRL_CUDA(launch_chain(adam_kernel, dim3(n_plain + n_tiles), dim3(256), (size_t)0, s, false, u, ad, slot, n_plain));
    return FSRL_OK;
}

// w2n[n] <- transpose of every net's W2 block, one launch
static int sync_mirror(const fsrl_ppo_update_t& u, cudaStream_t s) {
    W2Mirrors m = {};
    for (int n = 0; n < u.n_nets; ++n) {
        m.w2t[n] = u.theta + u.net_off[n] + ppo_layout(u, n, u.H).w2;
        m.w2n[n] = u.w2n + (size_t)n * u.H * u.H;
    }
    return w2_mirror(m, u.n_nets, u.H, s);
}

}  // namespace fsrl

using namespace fsrl;

static int check_update(const fsrl_ppo_update_t* u) {
    FSRL_REQUIRE(u != nullptr, "ppo: null descriptor");
    FSRL_REQUIRE(u->H == 64 || u->H == 128 || u->H == 256 || u->H == 512, "ppo: hidden width %d unsupported", u->H);
    FSRL_REQUIRE(u->n_nets >= 1 && u->n_nets <= 3 && u->C == u->n_nets - 1, "ppo: n_nets/C inconsistent");
    FSRL_REQUIRE(u->A >= 1 && u->A <= 8, "ppo: action dim %d out of range", u->A);
    FSRL_REQUIRE(u->theta && u->grad && u->adam_m && u->adam_v && u->w2n && u->scratch && u->norm_sq, "ppo: null buffer");
    if (u->world > 1 && u->p2p_on) {
        FSRL_REQUIRE(u->world <= FSRL_P2P_MAX_RANKS && u->p2p_rank >= 0 && u->p2p_rank < u->world && u->p2p_err && u->p2p_part,
                     "ppo: peer exchange needs world <= %d, a valid rank, an error flag and the partials", FSRL_P2P_MAX_RANKS);
        FSRL_REQUIRE(u->n_params <= 1024LL * FSRL_P2P_PARTIALS, "ppo: %lld parameters exceed the peer-exchange limit", u->n_params);
        for (int r = 0; r < u->world; ++r)
            FSRL_REQUIRE(u->p2p_xg[0][r] && u->p2p_xg[1][r] && u->p2p_flags[r], "ppo: peer %d is not mapped", r);
    }
    return FSRL_OK;
}

extern "C" size_t fsrl_ppo_scratch_floats(int n_nets, int H, int bmax) {
    return (size_t)n_nets * (size_t)bmax * (4 * (size_t)H + DOUT_LD);
}

extern "C" size_t fsrl_ppo_persist_ws_floats(int n_nets, int D, int H) { return ppo_persist_ws_floats(n_nets, D, H); }
extern "C" size_t fsrl_ppo_persist_p2p_floats(int n_nets) { return ppo_persist_p2p_floats(n_nets); }

extern "C" int fsrl_ppo_persist_active(const fsrl_ppo_update_t* u, long long n_total, int batch_size) {
    if (!u || u->persist_off) return 0;
    return ppo_persist_supported(*u, n_total, batch_size) ? 1 : 0;
}

extern "C" int fsrl_ppo_sync_mirror(const fsrl_ppo_update_t* u, void* stream) {
    int rc = check_update(u);
    if (rc) return rc;
    return sync_mirror(*u, static_cast<cudaStream_t>(stream));
}

// One repeat of PPOLagrangian.learn's inner loop (ppo_lag.py:223-247): every minibatch of
// Batch.split(batch_size, merge_last=True) over the permutation already in u->perm.
extern "C" int fsrl_ppo_lag_epoch(const fsrl_ppo_update_t* u, long long n_total, int batch_size,
                                  int stats_slot0, long long adam_t0, int* n_minibatches,
                                  void* stream) {
    int rc = check_update(u);
    if (rc) return rc;
    FSRL_REQUIRE(u->obs && u->act && u->logp_old && u->adv && u->ret && u->perm && u->stats, "ppo: null batch pointer");
    FSRL_REQUIRE(n_total <= 2147483647LL, "ppo: batch too large for 32-bit row offsets");
    FSRL_REQUIRE(batch_size >= 2 && n_total >= 2, "ppo: batch too small");
    FSRL_REQUIRE(2 * batch_size - 1 <= u->bmax || n_total <= u->bmax, "ppo: scratch bmax %d too small for batch_size %d", u->bmax, batch_size);
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    int count = 0;
    const bool merge_last = (n_total % batch_size) > 0;       // tianshou Batch.split
    fsrl_ppo_update_t ug = *u;
    if (u->barrier) FSRL_CUDA(cudaMemsetAsync(u->barrier, 0, sizeof(unsigned long long), s));
    if (u->gather) {
        // one coalescing pass per repeat: the permuted batch becomes contiguous, minibatch k is
        // rows [k*bs, (k+1)*bs) and no kernel chases indices afterwards
        ppo_gather_kernel<<<(unsigned)((n_total + 255) / 256), 256, 0, s>>>(*u, n_total);
        FSRL_LAUNCH_CHECK();
        float* g = u->gather;
        ug.obs = g; g += n_total * u->D;
        ug.act = g; g += n_total * u->A;
        ug.logp_old = g; g += n_total;
        ug.adv = g; g += (long long)u->C * n_total;
        ug.ret = g; g += (long long)u->C * n_total;
        ug.values = u->values ? g : nullptr;
        ug.ld = n_total;
        ug.perm = nullptr;
    }
    ug.batch_size = batch_size;
    u = &ug;
    FSRL_REQUIRE(u->world <= 1 || (u->comm && u->moments_w && u->batch_size == batch_size),
                 "ppo: data-parallel run needs comm, moments buffer and batch_size in the descriptor");
    if (u->world > 1) {
        // every rank must run the same number of equally sized minibatches
        FSRL_REQUIRE(!merge_last, "ppo: data-parallel run needs n_total %% batch_size == 0");
        const int n_mb = (int)(n_total / batch_size);
        ppo_adv_moments_kernel<<<n_mb, 256, 0, s>>>(*u, n_total, n_mb);
        FSRL_LAUNCH_CHECK();
        int rc2 = fsrl_allreduce_f64(u->comm, u->moments_w, (long long)n_mb * 4, s);
        if (rc2) return rc2;
    }
    {
        const long long n_mb_all = merge_last ? (n_total / batch_size) : (n_total + batch_size - 1) / batch_size;
        const int n_mb = (int)(n_mb_all < 1 ? 1 : n_mb_all);
        FSRL_REQUIRE(u->mb_stats != nullptr, "ppo: mb_stats buffer missing");
        ppo_adv_stats_kernel<<<n_mb, 256, 0, s>>>(*u, n_total, n_mb);
        FSRL_LAUNCH_CHECK();
    }
    if (!u->persist_off && ppo_persist_supported(*u, n_total, batch_size)) {
        // one persistent launch runs every minibatch of the repeat (csrc/ppo_persist.cu); the out-major
        // mirror of W2 that the three-launch chain reads is refreshed afterwards
        const int n_mb = (int)(n_total / batch_size);
        int rcp = ppo_persist_run(*u, n_mb, stats_slot0, adam_t0, s);
        if (rcp) return rcp;
        rcp = sync_mirror(*u, s);
        if (rcp) return rcp;
        if (n_minibatches) *n_minibatches = n_mb;
        return FSRL_OK;
    }
    for (long long off = 0; off < n_total; off += batch_size) {
        long long B = batch_size;
        bool last = false;
        if (merge_last && off + 2LL * batch_size >= n_total) { B = n_total - off; last = true; }
        if (off + B > n_total) B = n_total - off;
        FSRL_REQUIRE(B <= u->bmax, "ppo: minibatch of %lld rows exceeds scratch (%d)", B, u->bmax);
        int r2;
        switch (u->H) {
            case 64: r2 = ppo_launch_minibatch<64>(*u, (int)off, (int)B, stats_slot0 + count, adam_t0 + count + 1, count, s); break;
            case 128: r2 = ppo_launch_minibatch<128>(*u, (int)off, (int)B, stats_slot0 + count, adam_t0 + count + 1, count, s); break;
            case 256: r2 = ppo_launch_minibatch<256>(*u, (int)off, (int)B, stats_slot0 + count, adam_t0 + count + 1, count, s); break;
            default: r2 = ppo_launch_minibatch<512>(*u, (int)off, (int)B, stats_slot0 + count, adam_t0 + count + 1, count, s); break;
        }
        if (r2) return r2;
        ++count;
        if (last) break;
    }
    if (n_minibatches) *n_minibatches = count;
    return FSRL_OK;
}

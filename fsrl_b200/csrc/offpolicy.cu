// SAC-Lagrangian and DDPG-Lagrangian gradient steps on the device, assembled from the generic
// MLP engine (engine.cu) plus the small algorithm-specific kernels below.
//
// Replaces (reference):
//   fsrl/policy/base_policy.py:453-512 compute_nstep_returns + :543-567 nstep_return (numba)
//   fsrl/policy/sac_lag.py:136-145 _target_q, :147-183 forward (tanh-squashed Gaussian,
//       log-prob correction), :185-210 critics_loss, :212-258 policy_loss (+ auto alpha),
//       :260-269 learn, :132-134 sync_weight
//   fsrl/policy/ddpg_lag.py:120-131, :165-223
//
// One call runs `n_steps` complete gradient steps back to back (the loop of
// OffpolicyTrainer.policy_update_fn, offpolicy.py:102-104) without returning to the host.
#include "arena.cuh"

namespace fsrl {

constexpr int OD_LD = 16;    // row stride of the engine's out / dout scratch
constexpr float LOG_SQRT_2PI_O = 0.9189385332046727f;

__device__ __forceinline__ void gauss_pair_o(uint32_t a, uint32_t b, float& n0, float& n1) {
    const double u1 = ((double)a + 1.0) * (1.0 / 4294967296.0);
    const double u2 = (double)b * (1.0 / 4294967296.0);
    const double r = sqrt(-2.0 * log(u1));
    const double ang = 2.0 * 3.141592653589793 * u2;
    n0 = (float)(r * cos(ang));
    n1 = (float)(r * sin(ang));
}
constexpr uint32_t KEY_UPD = 0x55504454u;   // 'UPDT': noise stream of the update's rsample()

// ---- n-step bookkeeping (base_policy.py:481-493, :552-566) --------------------------------------
// For each sampled transition: walk buffer.next() n_step-1 times, accumulate the discounted
// reward / cost sums with the cut at done | unfinished, emit the terminal index, gamma^k and
// the value mask ~terminated[terminal].
__global__ void nstep_prepare_kernel(const fsrl_offpolicy_t d, const int* __restrict__ idx, int B) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B) return;
    const long long cap = d.cap;
    int chain[FSRL_MAX_NSTEP];
    int cur = idx[b];
    chain[0] = cur;
    for (int k = 1; k < d.n_step; ++k) {
        const int env = (int)(cur / cap);
        const int newest = (int)(env * cap + ((d.b_ptr[env] - 1 + cap) % cap));
        const bool done = d.b_term[cur] | d.b_trunc[cur];
        if (!done && cur != newest) cur = (int)(env * cap + ((cur % cap) + 1) % cap);
        chain[k] = cur;
    }
    double ret_r = 0.0, ret_c = 0.0;
    int g = d.n_step;
    for (int k = d.n_step - 1; k >= 0; --k) {
        const int now = chain[k];
        const int env = (int)(now / cap);
        const int newest = (int)(env * cap + ((d.b_ptr[env] - 1 + cap) % cap));
        const bool done = d.b_term[now] | d.b_trunc[now];
        const bool end = done || (now == newest);            // end_flag = done | unfinished (:492-493)
        if (end) { g = k + 1; ret_r = 0.0; ret_c = 0.0; }
        ret_r = (double)d.b_rew[now] + d.gamma * ret_r;
        ret_c = (double)d.b_cost[now] + d.gamma * ret_c;
    }
    double gp = 1.0;
    for (int i = 0; i < g; ++i) gp *= d.gamma;
    const int term = chain[d.n_step - 1];
    d.w_term_idx[b] = term;
    d.w_partial[b] = ret_r;
    d.w_partial[B + b] = ret_c;
    d.w_gpow[b] = gp;
    d.w_vmask[b] = d.b_term[term] ? 0.f : 1.f;                // value_mask (:375,:491)
}

// ---- SAC: rsample + tanh squash + log-prob (sac_lag.py:159-176) ----------------------------------
// out: [B][OD_LD] actor head (mu raw | sigma raw); writes act [B][A], logp [B] and the
// intermediates needed by the backward pass (eps, sigma, u) when `keep` != 0.
__global__ void sac_sample_kernel(const fsrl_offpolicy_t d, const float* __restrict__ out, int B,
                                  unsigned int stream_id, unsigned long long step, float* __restrict__ act,
                                  float* __restrict__ logp, float* __restrict__ keep) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B) return;
    const int A = d.A;
    float lp = 0.f;
    float eps[8];
#pragma unroll
    for (int c = 0; c < 2; ++c) {
        if (4 * c < A) {
            uint32_t rr[4];
            Philox::gen((uint32_t)b, (uint32_t)step, (uint32_t)(step >> 32) * 8u + (uint32_t)c, stream_id, d.seed, KEY_UPD, rr);
            gauss_pair_o(rr[0], rr[1], eps[4 * c], eps[4 * c + 1]);
            gauss_pair_o(rr[2], rr[3], eps[4 * c + 2], eps[4 * c + 3]);
        }
    }
    for (int j = 0; j < A; ++j) {
        const float o = out[(size_t)b * OD_LD + j];
        const float mu = d.bounded ? d.max_action * tanhf(o) : o;
        const float sraw = out[(size_t)b * OD_LD + A + j];
        const float sig = expf(fminf(fmaxf(sraw, d.sigma_min), d.sigma_max));
        const float u = fmaf(sig, eps[j], mu);
        const float a = tanhf(u);
        lp += -0.5f * eps[j] * eps[j] - logf(sig) - LOG_SQRT_2PI_O - logf(1.0f - a * a + d.tanh_eps);
        act[(size_t)b * A + j] = a;
        if (keep) { keep[(size_t)b * 24 + j] = eps[j]; keep[(size_t)b * 24 + 8 + j] = sig; keep[(size_t)b * 24 + 16 + j] = a; }
    }
    logp[b] = lp;
}

// target_i = (min(Q'_{2i}, Q'_{2i+1}) - alpha*logp') * vmask * gamma^k + partial_i  (f64 like numba)
__global__ void sac_target_kernel(const fsrl_offpolicy_t d, int B) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B) return;
    const float alpha = d.use_alpha ? *d.alpha : 0.f;
    for (int i = 0; i < d.C; ++i) {
        float tq;
        if (d.twin) tq = fminf(d.q_old_out[2 * i][(size_t)b * OD_LD], d.q_old_out[2 * i + 1][(size_t)b * OD_LD]);
        else tq = d.q_old_out[i][(size_t)b * OD_LD];
        if (d.use_alpha) tq = tq - alpha * d.w_logp_next[b];                   // sac_lag.py:144
        const float masked = tq * d.w_vmask[b];                                 // base_policy.py:502
        d.w_target[(size_t)i * B + b] = (float)((double)masked * d.w_gpow[b] + d.w_partial[(size_t)i * B + b]);
    }
}

// critic head gradients: d/dq of sum_i sum_j mean((q_ij - target_i)^2) ; stats loss/q_i
__global__ void critic_grad_kernel(const fsrl_offpolicy_t d, int B, float* __restrict__ stat) {
    __shared__ float red[2][8];
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    float l[2] = {0.f, 0.f};
    if (b < B) {
        const int per = d.twin ? 2 : 1;
        for (int i = 0; i < d.C; ++i) {
            const float tgt = d.w_target[(size_t)i * B + b];
            for (int j = 0; j < per; ++j) {
                const int n = per * i + j;
                const float td = d.q_out[n][(size_t)b * OD_LD] - tgt;
                d.q_dout[n][(size_t)b * OD_LD] = 2.0f * td / (float)B;
                l[i] += td * td / (float)B;
            }
        }
    }
    for (int i = 0; i < 2; ++i) {
        const float v = warp_sum(l[i]);
        if ((threadIdx.x & 31) == 0) red[i][threadIdx.x >> 5] = v;
    }
    __syncthreads();
    if (threadIdx.x < 2) {
        float t = 0.f;
        for (int w = 0; w < (int)(blockDim.x >> 5); ++w) t += red[threadIdx.x][w];
        if (t != 0.f) atomicAdd(stat + FSRL_OFF_ST_Q0 + threadIdx.x, t);
    }
}

// actor loss through the critics (sac_lag.py:216-232 / ddpg_lag.py:191-201): head gradients of
// the Q networks w.r.t. their outputs; stats actor_rew / actor_safety
__global__ void actor_q_grad_kernel(const fsrl_offpolicy_t d, int B, float* __restrict__ stat) {
    __shared__ float red[3][8];
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    float s_rew = 0.f, s_saf = 0.f, s_lp = 0.f;
    if (b < B) {
        const float invB = 1.0f / (float)B;
        const float alpha = d.use_alpha ? *d.alpha : 0.f;
        const int per = d.twin ? 2 : 1;
        for (int i = 0; i < d.C; ++i) {
            // weight of critic i in the actor loss: reward -1, cost +lambda (when lagrangian on)
            float w = (i == 0) ? -1.0f : (d.use_lagrangian ? d.lagrangian : 0.f);
            w *= d.rescaling * invB;
            float q;
            if (d.twin) {
                const float q0 = d.q_out[2 * i][(size_t)b * OD_LD], q1 = d.q_out[2 * i + 1][(size_t)b * OD_LD];
                q = fminf(q0, q1);
                // torch.min(a, b) backward: all to the smaller, split evenly on ties
                const float g0 = q0 < q1 ? 1.f : (q0 > q1 ? 0.f : 0.5f);
                d.q_dout[2 * i][(size_t)b * OD_LD] = w * g0;
                d.q_dout[2 * i + 1][(size_t)b * OD_LD] = w * (1.f - g0);
            } else {
                q = d.q_out[i][(size_t)b * OD_LD];
                d.q_dout[i][(size_t)b * OD_LD] = w;
            }
            if (i == 0) s_rew = -q * invB;
            else if (d.use_lagrangian) s_saf += d.lagrangian * q * invB;
        }
        if (d.use_alpha) {
            const float lp = d.w_logp[b];
            s_rew += alpha * lp * invB;                       // mean(alpha*logp - q)   (sac_lag.py:218)
            s_lp = lp * invB;
        }
    }
    float v[3] = {s_rew, s_saf, s_lp};
    for (int i = 0; i < 3; ++i) {
        const float t = warp_sum(v[i]);
        if ((threadIdx.x & 31) == 0) red[i][threadIdx.x >> 5] = t;
    }
    __syncthreads();
    if (threadIdx.x < 3) {
        float t = 0.f;
        for (int w = 0; w < (int)(blockDim.x >> 5); ++w) t += red[threadIdx.x][w];
        const int slot = threadIdx.x == 0 ? FSRL_OFF_ST_ACTOR_REW : (threadIdx.x == 1 ? FSRL_OFF_ST_ACTOR_SAFETY : FSRL_OFF_ST_LOGP);
        if (t != 0.f) atomicAdd(stat + slot, t);
    }
}

// d loss / d actor head from d loss / d action (sum of the critics' input gradients) and, for
// SAC, the entropy term alpha*logp through the tanh-squashed reparameterised sample
__global__ void actor_head_grad_kernel(const fsrl_offpolicy_t d, int B) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B) return;
    const int A = d.A, D = d.D;
    const int nq = (d.twin ? 2 : 1) * d.C;
    const float invB = 1.0f / (float)B;
    const float alpha = d.use_alpha ? *d.alpha : 0.f;
    float dd[OD_LD];
#pragma unroll
    for (int j = 0; j < OD_LD; ++j) dd[j] = 0.f;
    for (int j = 0; j < A; ++j) {
        float da = 0.f;
        for (int n = 0; n < nq; ++n) da += d.q_dx[n][(size_t)b * FSRL_ENG_DX_LD + D + j];
        const float o = d.actor_out[(size_t)b * OD_LD + j];
        if (d.use_alpha) {
            const float eps = d.w_keep[(size_t)b * 24 + j], sig = d.w_keep[(size_t)b * 24 + 8 + j];
            const float a = d.w_keep[(size_t)b * 24 + 16 + j];
            const float one_m = 1.0f - a * a;
            const float k = d.rescaling * alpha * invB;                        // weight of logp in the loss
            const float dlp_du = 2.0f * a * one_m / (one_m + d.tanh_eps);      // d logp / d u
            const float du = da * one_m + k * dlp_du;                          // d loss / d u
            const float dmu = du;
            const float dsig = du * eps - k / sig;                             // u = mu + sig*eps ; -log(sig)
            const float t = tanhf(o);
            dd[j] = d.bounded ? dmu * d.max_action * (1.0f - t * t) : dmu;
            const float sraw = d.actor_out[(size_t)b * OD_LD + A + j];
            const bool in = (sraw >= d.sigma_min) && (sraw <= d.sigma_max);    // clamp passes gradient on the closed range
            dd[A + j] = in ? dsig * sig : 0.f;
        } else {
            const float t = tanhf(o);                                           // act = max_action*tanh(o)
            dd[j] = da * d.max_action * (1.0f - t * t);
        }
    }
#pragma unroll
    for (int j = 0; j < OD_LD; j += 4)
        *reinterpret_cast<float4*>(d.actor_dout + (size_t)b * OD_LD + j) = make_float4(dd[j], dd[j + 1], dd[j + 2], dd[j + 3]);
}

// deterministic actor output -> action (tianshou Actor): a = max_action * tanh(o)
__global__ void ddpg_action_kernel(const fsrl_offpolicy_t d, const float* __restrict__ out, int B, float* __restrict__ act) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= B * d.A) return;
    const int b = i / d.A, j = i % d.A;
    act[i] = d.max_action * tanhf(out[(size_t)b * OD_LD + j]);
}

// automatic entropy tuning (sac_lag.py:237-250): one Adam step on log_alpha, alpha = exp(.)
__global__ void alpha_step_kernel(const fsrl_offpolicy_t d, const float* __restrict__ stat, float* __restrict__ stat_out,
                                  float inv_world) {
    if (threadIdx.x != 0 || blockIdx.x != 0) return;
    float* st = d.alpha_state;     // [log_alpha, m, v, t]
    if (inv_world != 1.0f) {       // the row was summed over the ranks: back to the global-batch means
        for (int i = 0; i <= FSRL_OFF_ST_LOGP; ++i) stat_out[i] = stat[i] * inv_world;
    }
    const float mean_lp = stat_out[FSRL_OFF_ST_LOGP];
    const float g = -(mean_lp + d.target_entropy);             // d/d log_alpha of -(log_alpha*(logp+H)).mean()
    const float la = st[0];
    stat_out[FSRL_OFF_ST_ALPHA_LOSS] = -la * (mean_lp + d.target_entropy);
    float m = st[1], v = st[2];
    const float t = st[3] + 1.0f;
    m = m + 0.1f * (g - m);
    v = v * 0.999f + (0.001f * g) * g;
    const float bc1 = 1.0f - powf(0.9f, t), bc2 = 1.0f - powf(0.999f, t);
    const float denom = sqrtf(v) / sqrtf(bc2) + 1e-8f;
    const float nla = la + (-(d.alpha_lr / bc1) * m) / denom;
    st[0] = nla; st[1] = m; st[2] = v; st[3] = t;
    *d.alpha = expf(nla);
    stat_out[FSRL_OFF_ST_ALPHA] = expf(nla);
}

static inline fsrl_eng_input_t mk_in(const float* xa, const int* ia, int Da, const float* xb, const int* ib, int Db) {
    fsrl_eng_input_t in;
    in.xa = xa; in.ia = ia; in.xb = xb; in.ib = ib; in.Da = Da; in.Db = Db;
    return in;
}

}  // namespace fsrl

using namespace fsrl;

#define OFF_CHECK(call) do { int rc__ = (call); if (rc__) return rc__; } while (0)

extern "C" int fsrl_allreduce_ranges(void* comm, float* base, const long long* offs, const long long* counts,
                                     int n_ranges, void* stream);
extern "C" int fsrl_allreduce_fused(void* comm, float* buf, long long n, void* stream);

// data parallel: sum the gradient slices of a net list over the ranks (averaged by Adam's grad_scale)
static int allreduce_grads(const fsrl_offpolicy_t* d, const fsrl_netlist_t* nl, void* stream) {
    long long offs[FSRL_ENG_MAX_NETS], counts[FSRL_ENG_MAX_NETS];
    for (int i = 0; i < nl->n; ++i) { offs[i] = nl->nets[i].off; counts[i] = NetLayout(nl->nets[i]).size; }
    return fsrl_allreduce_ranges(d->comm, d->eng.grad, offs, counts, nl->n, stream);
}

extern "C" int fsrl_nstep_prepare(const fsrl_offpolicy_t* d, const int* idx, int B, void* stream) {
    FSRL_REQUIRE(d && idx, "nstep: null pointer");
    FSRL_REQUIRE(d->n_step >= 1 && d->n_step <= FSRL_MAX_NSTEP, "n_step %d out of range [1, %d]", d->n_step, FSRL_MAX_NSTEP);
    FSRL_REQUIRE(B >= 0 && B <= d->eng.bmax, "nstep: B out of range");
    if (B == 0) return FSRL_OK;
    nstep_prepare_kernel<<<(B + 127) / 128, 128, 0, static_cast<cudaStream_t>(stream)>>>(*d, idx, B);
    FSRL_LAUNCH_CHECK();
    return FSRL_OK;
}

// n_steps gradient steps of SACLagrangian.learn / DDPGLagrangian.learn.  idx_all: [n_steps][B]
// sampled flat buffer indices (device, int32).  stats: [n_steps][FSRL_OFF_STATS] (zeroed by caller).
extern "C" int fsrl_offpolicy_steps(const fsrl_offpolicy_t* d, const int* idx_all, int n_steps, int B,
                                    long long critic_t0, long long actor_t0, unsigned long long noise_t0,
                                    float* stats, void* stream) {
    FSRL_REQUIRE(d && idx_all && stats, "offpolicy: null pointer");
    FSRL_REQUIRE(d->algo == FSRL_ALGO_SAC || d->algo == FSRL_ALGO_DDPG, "offpolicy: unknown algo %d", d->algo);
    FSRL_REQUIRE(B >= 2 && B <= d->eng.bmax, "offpolicy: B=%d out of range (bmax %d)", B, d->eng.bmax);
    FSRL_REQUIRE(d->A >= 1 && d->A <= 8 && d->C >= 1 && d->C <= 2, "offpolicy: A/C out of range");
    FSRL_REQUIRE(d->world <= 1 || d->comm != nullptr, "offpolicy: world=%d needs a communicator", d->world);
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    const int T = 128, G = (B + T - 1) / T;
    const bool sac = d->algo == FSRL_ALGO_SAC;
    const bool dp = d->world > 1;
    const double gscale = dp ? 1.0 / d->world : 1.0;
    const int D = d->D, A = d->A;
    for (int it = 0; it < n_steps; ++it) {
        const int* idx = idx_all + (size_t)it * B;
        float* stat = stats + (size_t)it * FSRL_OFF_STATS;
        // ---- process_fn: n-step targets (:496-509) --------------------------------------------------
        OFF_CHECK(fsrl_nstep_prepare(d, idx, B, stream));
        {
            const fsrl_netlist_t* actor_t = sac ? &d->actor : &d->actor_old;
            fsrl_eng_input_t in = mk_in(d->b_obs_next, d->w_term_idx, D, nullptr, nullptr, 0);
            OFF_CHECK(fsrl_engine_forward(&d->eng, actor_t, &in, B, 0, stream));
            const float* aout = sac ? d->actor_out : d->actor_old_out;
            if (sac) sac_sample_kernel<<<G, T, 0, s>>>(*d, aout, B, 0u, noise_t0 + it, d->w_act_next, d->w_logp_next, nullptr);
            else ddpg_action_kernel<<<(B * A + T - 1) / T, T, 0, s>>>(*d, aout, B, d->w_act_next);
            FSRL_LAUNCH_CHECK();
            fsrl_eng_input_t inq = mk_in(d->b_obs_next, d->w_term_idx, D, d->w_act_next, nullptr, A);
            OFF_CHECK(fsrl_engine_forward(&d->eng, &d->critics_old, &inq, B, 0, stream));
            sac_target_kernel<<<G, T, 0, s>>>(*d, B);
            FSRL_LAUNCH_CHECK();
        }
        // ---- critics_loss (sac_lag.py:185-210 / ddpg_lag.py:165-189) ---------------------------------
        {
            fsrl_eng_input_t in = mk_in(d->b_obs, idx, D, d->b_act, idx, A);
            OFF_CHECK(fsrl_engine_forward(&d->eng, &d->critics, &in, B, 1, stream));
            critic_grad_kernel<<<G, T, 0, s>>>(*d, B, stat);
            FSRL_LAUNCH_CHECK();
            OFF_CHECK(fsrl_engine_backward(&d->eng, &d->critics, B, 0, stream));
            OFF_CHECK(fsrl_engine_wgrad(&d->eng, &d->critics, &in, B, 0, nullptr, stream));
            if (dp) OFF_CHECK(allreduce_grads(d, &d->critics, stream));
            OFF_CHECK(fsrl_engine_adam(&d->eng, &d->critics, d->critic_lr, 0.9, 0.999, 1e-8, critic_t0 + it + 1, gscale, 0.0, nullptr, 0.0, stream));
        }
        // ---- policy_loss (sac_lag.py:212-258 / ddpg_lag.py:191-213) ----------------------------------
        {
            fsrl_eng_input_t in = mk_in(d->b_obs, idx, D, nullptr, nullptr, 0);
            OFF_CHECK(fsrl_engine_forward(&d->eng, &d->actor, &in, B, 1, stream));
            if (sac) sac_sample_kernel<<<G, T, 0, s>>>(*d, d->actor_out, B, 1u, noise_t0 + it, d->w_act, d->w_logp, d->w_keep);
            else ddpg_action_kernel<<<(B * A + T - 1) / T, T, 0, s>>>(*d, d->actor_out, B, d->w_act);
            FSRL_LAUNCH_CHECK();
            fsrl_eng_input_t inq = mk_in(d->b_obs, idx, D, d->w_act, nullptr, A);
            OFF_CHECK(fsrl_engine_forward(&d->eng, &d->critics, &inq, B, 1, stream));
            actor_q_grad_kernel<<<G, T, 0, s>>>(*d, B, stat);
            FSRL_LAUNCH_CHECK();
            OFF_CHECK(fsrl_engine_backward(&d->eng, &d->critics, B, 1, stream));
            actor_head_grad_kernel<<<G, T, 0, s>>>(*d, B);
            FSRL_LAUNCH_CHECK();
            OFF_CHECK(fsrl_engine_backward(&d->eng, &d->actor, B, 0, stream));
            OFF_CHECK(fsrl_engine_wgrad(&d->eng, &d->actor, &in, B, 0, nullptr, stream));
            if (dp) OFF_CHECK(allreduce_grads(d, &d->actor, stream));
            OFF_CHECK(fsrl_engine_adam(&d->eng, &d->actor, d->actor_lr, 0.9, 0.999, 1e-8, actor_t0 + it + 1, gscale, 0.0, nullptr, 0.0, stream));
            if (sac && d->auto_alpha) {
                if (dp) OFF_CHECK(fsrl_allreduce_fused(d->comm, stat, FSRL_OFF_ST_LOGP + 1, stream));
                alpha_step_kernel<<<1, 32, 0, s>>>(*d, stat, stat, (float)gscale);
                FSRL_LAUNCH_CHECK();
            }
        }
        // ---- sync_weight (sac_lag.py:132-134 / ddpg_lag.py:120-123) ----------------------------------
        OFF_CHECK(fsrl_engine_polyak(&d->eng, &d->critics_old, &d->critics, d->tau, stream));
        if (!sac) OFF_CHECK(fsrl_engine_polyak(&d->eng, &d->actor_old, &d->actor, d->tau, stream));
    }
    return FSRL_OK;
}

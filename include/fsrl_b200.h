/* fsrl_b200 -- C-ABI of the B200-native FSRL hot path.
 *
 * The reference (liuzuxin/FSRL) is pure Python and has NO FFI layer of its own
 * (SURVEY.md F1, 8b): its boundary is the Python class API (fsrl.policy / fsrl.data).  This
 * header is the boundary the new engine adds underneath that API: every entry point names
 * the reference function it replaces (file:line under /root/reference).  INTEGRATION.md
 * shows the ctypes binding a maintainer of the reference would add at each call site.
 *
 * Conventions (all entry points):
 *   - plain pointers + sizes, no torch types; every pointer is DEVICE memory unless the
 *     parameter is documented "host";
 *   - the caller owns every buffer (functions never allocate or free) and passes scratch
 *     space explicitly; `*_workspace_bytes` reports the size;
 *   - asynchronous on `stream` (a cudaStream_t passed as void*); no device sync inside;
 *   - returns 0 on success, <0 on error (FSRL_EINVAL -1, FSRL_ECUDA -2,
 *     FSRL_EWORKSPACE -3); fsrl_last_error() returns the thread-local message.  The
 *     reference signals errors with Python assert/exceptions; the Python host layer
 *     (fsrl_b200/_lib.py) re-raises these codes as the same exception types/messages;
 *   - fp32 storage; the GAE / n-step scans accumulate in fp64 like the reference.
 *   - one host thread per GPU/rank; entry points are not re-entrant on the same workspace.
 */
#ifndef FSRL_B200_H
#define FSRL_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* ---- plumbing ------------------------------------------------------------------- */
const char* fsrl_last_error(void);
int fsrl_abi_version(void);
size_t fsrl_abi_sizeof(int which); /* sizeof() of the descriptor structs, for binding self-checks */
int fsrl_sm_count(void);
/* Number of kernels this library has launched so far in this process (host-side counter,
 * one per checked launch). bench.py reports the difference across its timed region. */
unsigned long long fsrl_launch_count(void);

/* ---- a6/a7: dual GAE(lambda) -------------------------------------------------------
 * Replaces fsrl/policy/base_policy.py:524-540 (gae_return, numba) together with the
 * value_mask / end_flag / ret=adv+v / f32 cast of compute_gae_returns (:409-411,:429,
 * :438-446) for the reward and cost critics in ONE pass.
 *   v, vnext : [C][ld] f32   V_i(obs), V_i(obs_next)   (critic i at offset i*ld)
 *   rew,cost : [N] f32       metrics of critic 0 / 1 (cost may be NULL when C == 1)
 *   end_flag : [N] u8        terminated | truncated | unfinished-tail  (:410-411)
 *   terminated: [N] u8 or NULL; when given, vnext is masked by ~terminated (:375,:429)
 *   adv, ret : [C][ld] f32   outputs (batch.advs / batch.rets columns)
 * Flat order is the reference's batch order: env-major, chronological inside an env. */
size_t fsrl_gae_dual_workspace_bytes(int64_t N);
int fsrl_gae_dual(const float* v, const float* vnext, const float* rew, const float* cost,
                  const uint8_t* end_flag, const uint8_t* terminated, double gamma,
                  double gae_lambda, float* adv, float* ret, int64_t N, int64_t ld, int C,
                  void* workspace, size_t workspace_bytes, void* stream);


/* ---- network descriptor ----------------------------------------------------------------
 * A 2-hidden-layer MLP in -> H -> H -> out (tianshou Net/MLP + head; the reference builds
 * these at fsrl/agent/ppo_lag_agent.py:136-145).  Canonical layout: every Linear is stored
 * TRANSPOSED, Wt[in][out] row-major (torch's .weight is the strided view Wt.t()).
 * H must be 64, 128, 256 or 512. */
typedef struct fsrl_mlp3 {
    const float* w1t; /* [in][H]  */
    const float* b1;  /* [H]      */
    const float* w2t; /* [H][H]   */
    const float* b2;  /* [H]      */
    const float* w3t; /* [H][out] */
    const float* b3;  /* [out]    */
    int in, H, out;
} fsrl_mlp3_t;

/* ---- a1-a5: rollout collection ---------------------------------------------------------
 * One fsrl_rollout_steps() step == one iteration of the while-loop of
 * FastCollector.collect (fsrl/data/fast_collector.py:252-368): policy forward
 * (base_policy.py:178-190), exploration noise (ddpg_lag.py:225-231), map_action
 * (base_policy.py:226-256), env.step, cost extraction, buffer.add and the episode
 * bookkeeping incl. the surplus-env rule (:357-363), for all ready envs, on the device. */
enum { FSRL_MODE_TRAIN = 0, FSRL_MODE_EVAL = 1, FSRL_MODE_RANDOM = 2 };
enum { FSRL_HEAD_GAUSS_INDEP = 0, FSRL_HEAD_GAUSS_COND = 1, FSRL_HEAD_DETERMINISTIC = 2 };
enum { FSRL_BOUND_NONE = 0, FSRL_BOUND_CLIP = 1, FSRL_BOUND_TANH = 2 };
enum { FSRL_ENV_CAR_CIRCLE = 0, FSRL_ENV_CAR_RUN = 1, FSRL_ENV_BALL_CIRCLE = 2,
       FSRL_ENV_BALL_RUN = 3, FSRL_ENV_ANT_CIRCLE = 4, FSRL_ENV_POINT_GOAL = 5 };

/* per-collect statistics, device resident; the keys of collect()'s result dict
 * (fast_collector.py:399-408) are derived from it on the host */
typedef struct fsrl_collect_stats {
    unsigned long long step_count;  /* n/st */
    unsigned long long sum_ep_len;  /* sum of finished episode lengths */
    double total_cost;              /* total_cost */
    double sum_ep_rew;              /* sum of finished episode returns */
    int episode_count;              /* n/ep */
    int n_episode;                  /* target */
    int n_ready;                    /* len(ready_env_ids) */
    int term_count, trunc_count;
    int finished, finished_next;
    int pad;
} fsrl_collect_stats_t;

typedef struct fsrl_rollout {
    /* environment (SoA, device) */
    int kind, E, max_steps, inline_done;
    unsigned int seed_env, seed_act;
    float* env_state;        /* [S][E] */
    float* obs_cur;          /* [E][D] */
    int* env_t;              /* [E] step inside the running episode */
    unsigned int* ep_idx;    /* [E] episodes started (reset RNG counter) */
    unsigned int* act_ctr;   /* [E] actions sampled (noise RNG counter) */
    unsigned char* active;   /* [E] ready_env_ids as a mask */
    unsigned char* done_now; /* [E] 0 / 1 terminated / 2 truncated this step */
    double* ep_rew;          /* [E] running episode return */
    int* ep_len;             /* [E] running episode length */
    /* policy */
    fsrl_mlp3_t actor;
    const float* log_sigma;  /* [A] state-independent log-sigma (HEAD_GAUSS_INDEP) */
    int head, mode, bounded, action_bound, action_scaling, pad0;
    float max_action, expl_sigma, sigma_min, sigma_max, tanh_eps, pad1;
    float act_low[8], act_high[8];
    /* transition buffer: env-major sub-buffers of `cap` slots (tianshou VectorReplayBuffer
     * order), any pointer group may be NULL to collect without storing (evaluate()) */
    float *b_obs, *b_obs_next, *b_act, *b_rew, *b_cost, *b_logp;
    unsigned char *b_term, *b_trunc;
    int* b_ptr;              /* [E] next write slot */
    int* b_len;              /* [E] valid transitions */
    long long cap;
    fsrl_collect_stats_t* stats;
} fsrl_rollout_t;

int fsrl_env_dims(int kind, int* D, int* A, int* S, int* T);
/* reset_env (fast_collector.py:131-152): start a fresh episode in every env */
int fsrl_env_reset_all(const fsrl_rollout_t* r, void* stream);
/* start of collect(n_episode): ready set = first min(E, n_episode) envs (:233-236) */
int fsrl_collect_begin(const fsrl_rollout_t* r, int n_episode, void* stream);
/* n_steps vector steps; steps after stats->finished are no-ops */
int fsrl_rollout_steps(const fsrl_rollout_t* r, int n_steps, void* stream);

/* ---- a9/a10: PPO-Lagrangian update --------------------------------------------------------
 * Replaces PPOLagrangian.policy_loss / critics_loss / learn
 * (fsrl/policy/ppo_lag.py:152-257) and LagrangianPolicy.safety_loss
 * (fsrl/policy/lagrangian_base.py:145-166): per-minibatch advantage normalisation, clipped
 * surrogate, unclipped lambda-weighted cost term, rescaling, value losses, backward,
 * clip_grad_norm_ and Adam, with per-minibatch statistics accumulated on the device.
 *
 * All networks of the policy live in ONE flat fp32 buffer `theta`; network n (0 = actor,
 * 1.. = critics) starts at net_off[n] with layout
 *     w1t[D][H] | b1[H] | w2t[H][H] | b2[H] | w3t[H][out] | b3[out] | (actor) log_sigma[A]
 * grad / adam_m / adam_v mirror that layout; w2n[n][H][H] is the out-major copy of w2t kept
 * in sync by the Adam kernel (fsrl_ppo_sync_mirror initialises it). */
#define FSRL_PPO_STATS 8 /* per-minibatch: actor_rew, actor_safety, kl, vf0, vf1, entropy, grad_norm, - */
typedef struct fsrl_ppo_update {
    float *theta, *grad, *adam_m, *adam_v, *w2n, *scratch, *norm_sq, *stats;
    const unsigned char* mask;     /* optional [n_params]: 0 = frozen parameter */
    long long net_off[3];
    long long n_params;
    int n_nets, D, H, A, C, actor_out, bmax, head_indep;
    /* the processed batch (flat env-major arrays) and the minibatch permutation */
    const float *obs, *act, *logp_old, *adv, *ret, *values; /* adv/ret/values: [C][ld] */
    long long ld;
    const int* perm;
    /* hyper-parameters (ppo_lag.py:86-99) */
    float eps_clip, dual_clip, vf_coef, max_grad_norm;
    float max_action, lagrangian, rescaling, pad0;
    int bounded, norm_adv, value_clip, use_lagrangian;
    double lr, beta1, beta2, adam_eps;
    /* data-parallel run (world > 1): NCCL communicator, per-minibatch advantage moments
     * [n_mb][2][2] (sum, sum of squares; reduced over ranks once per repeat); moments must
     * alias moments_w */
    void* comm;
    double* moments_w;
    const double* moments;
    int world, batch_size;
    /* optional [N*(D+A+1+3C)] floats: the epoch driver gathers the permuted batch into it once
     * per repeat so that every minibatch is a contiguous row range */
    float* gather;
    /* [n_minibatches][2][2] floats: (mean, 1/std) of the advantages of every minibatch of the
     * repeat, filled by the epoch driver */
    float* mb_stats;
    /* device u64 ticket counter of the in-kernel grid barrier (fused wgrad + Adam launch) */
    unsigned long long* barrier;
    /* peer-memory gradient exchange (world > 1, optional; NCCL all-reduce when p2p_on == 0):
     * rank r's exchange block (fsrl_p2p_alloc) mapped into this process -- p2p_xg[b][r] its
     * gradient buffer of step parity b, p2p_flags[r] its arrival flags [FSRL_P2P_MAX_RANKS] --
     * entries [.][p2p_rank] are this rank's own block.  The weight-gradient kernel writes into the
     * local buffer; ppo_dp_reduce_kernel signals the peers, waits for their flags and sums all
     * ranks' buffers over NVLink in rank order (bit-identical result everywhere). */
    const float* p2p_xg[2][8];
    unsigned long long* p2p_flags[8];
    int* p2p_err;                  /* local: set to 1 if a peer never arrived (wait timed out) */
    float* p2p_part;               /* local [FSRL_P2P_PARTIALS]: per-CTA sums of g^2 (summed in a fixed
                                    * order by the Adam kernel: atomics would break rank lock-step) */
    int p2p_rank, p2p_on;
    /* persistent tcgen05 path (csrc/ppo_persist.cu; H = 256, batch 256): workspace of
     * fsrl_ppo_persist_ws_floats() floats for the operand images / partials / flags; NULL or
     * persist_off != 0 selects the three-launch chain.  With world > 1 the launch exchanges gradients
     * itself: it treats every p2p_xg[b][r] as fsrl_ppo_persist_p2p_floats() floats of packet regions
     * (one per source rank + one for reduced tiles; ranks push, receivers poll their own buffer) and
     * needs p2p_on, p2p_rank and p2p_stride >= that size; p2p_flags / p2p_part stay with the chain */
    float* persist_ws;
    long long persist_ws_floats;
    int persist_off, pad1;
    long long p2p_stride;          /* floats available in every p2p_xg buffer (fsrl_p2p_stride of the allocation) */
} fsrl_ppo_update_t;

size_t fsrl_ppo_scratch_floats(int n_nets, int H, int bmax);
size_t fsrl_ppo_persist_ws_floats(int n_nets, int D, int H);
/* floats each peer-mapped exchange buffer must hold for the data-parallel persistent path */
size_t fsrl_ppo_persist_p2p_floats(int n_nets);
/* 1 if fsrl_ppo_lag_epoch would take the persistent path for this descriptor / batch */
int fsrl_ppo_persist_active(const fsrl_ppo_update_t* u, long long n_total, int batch_size);
int fsrl_ppo_sync_mirror(const fsrl_ppo_update_t* u, void* stream);
/* one repeat of learn()'s inner loop: all minibatches of Batch.split(batch_size,
 * merge_last=True) over u->perm[0..n_total); Adam step counter continues from adam_t0;
 * statistics go to stats[stats_slot0 + i]; *n_minibatches (host) receives the count */
int fsrl_ppo_lag_epoch(const fsrl_ppo_update_t* u, long long n_total, int batch_size,
                       int stats_slot0, long long adam_t0, int* n_minibatches, void* stream);

/* ---- a6: batched critic / actor forward ---------------------------------------------------
 * y[r][:] = net(x[idx ? idx[r] : r][:]) for r < n_rows.  Replaces the chunked no_grad
 * critic passes of compute_gae_returns (fsrl/policy/base_policy.py:416-422). */
int fsrl_mlp_forward(const fsrl_mlp3_t* net, const float* x, const int* idx, long long n_rows,
                     float* y, void* stream);

/* ---- generic minibatch MLP engine (SAC / DDPG / CPO updates are assembled from it) --------
 * Replaces the eager autograd forward/backward/optimizer.step of the reference's learners
 * (fsrl/policy/sac_lag.py:185-258, ddpg_lag.py:165-213, cpo.py:147-162) and soft_update
 * (fsrl/policy/base_policy.py:220-224).  Networks live in the flat arena (layout as for
 * fsrl_ppo_update_t); each has a scratch slot of fsrl_engine_slot_floats(H, bmax) floats:
 *   h1 | h2 | dz1 | dz2 : [bmax][H],  out | dout : [bmax][16],  dx : [bmax][64]
 * forward writes `out` (+ h1, h2 when save != 0); the caller fills `dout` (d loss / d head
 * output, columns [out, out+n_extra) = d loss / d extra parameters); backward produces dz1,
 * dz2 (+ dx = d loss / d input); wgrad reduces them into `grad`; adam applies them. */
#define FSRL_ENG_MAX_NETS 8
#define FSRL_ENG_DX_LD 64
typedef struct fsrl_netref {
    long long off;      /* start of the net inside theta / grad / adam_m / adam_v */
    long long w2n_off;  /* start of its W2 mirror inside w2n */
    int D, H, out, n_extra;
    int slot, pad;
} fsrl_netref_t;
typedef struct fsrl_netlist {
    int n, pad;
    fsrl_netref_t nets[FSRL_ENG_MAX_NETS];
} fsrl_netlist_t;
typedef struct fsrl_engine {
    float *theta, *grad, *adam_m, *adam_v, *w2n, *scratch;
    int bmax, pad;
} fsrl_engine_t;
/* input row r = concat(xa[ia ? ia[r] : r][0..Da), xb[ib ? ib[r] : r][0..Db)) */
typedef struct fsrl_eng_input {
    const float* xa;
    const int* ia;
    const float* xb;
    const int* ib;
    int Da, Db;
} fsrl_eng_input_t;

size_t fsrl_engine_slot_floats(int H, int bmax);
int fsrl_engine_forward(const fsrl_engine_t* e, const fsrl_netlist_t* nets, const fsrl_eng_input_t* in,
                        int B, int save, void* stream);
int fsrl_engine_backward(const fsrl_engine_t* e, const fsrl_netlist_t* nets, int B, int want_dx, void* stream);
int fsrl_engine_wgrad(const fsrl_engine_t* e, const fsrl_netlist_t* nets, const fsrl_eng_input_t* in, int B,
                      int accumulate, float* norm_sq, void* stream);
/* torch.optim.Adam step `step` (1-based) on the listed nets; grad <- grad*grad_scale + 2*l2_reg*p
 * and, when norm_sq != NULL && max_grad_norm > 0, clip_grad_norm_ by sqrt(*norm_sq) */
int fsrl_engine_adam(const fsrl_engine_t* e, const fsrl_netlist_t* nets, double lr, double beta1,
                     double beta2, double eps, long long step, double grad_scale, double l2_reg,
                     const float* norm_sq, double max_grad_norm, void* stream);
int fsrl_engine_polyak(const fsrl_engine_t* e, const fsrl_netlist_t* dst, const fsrl_netlist_t* src,
                       double tau, void* stream);
int fsrl_engine_sync_mirror(const fsrl_engine_t* e, const fsrl_netlist_t* nets, void* stream);

/* ---- a12-a14, a16: SAC- / DDPG-Lagrangian gradient steps -------------------------------------
 * fsrl_offpolicy_steps runs n_steps iterations of `policy.update(batch_size, buffer)`
 * (fsrl/trainer/offpolicy.py:102-104): process_fn = n-step targets for the reward and cost
 * critics (fsrl/policy/base_policy.py:453-512,543-567; sac_lag.py:136-145; ddpg_lag.py:
 * 125-131), critics_loss, policy_loss (lambda-weighted cost-Q term + rescaling,
 * lagrangian_base.py:145-166; SAC: tanh-squashed rsample, log-prob correction, auto-alpha),
 * sync_weight.  Networks are engine netlists: SAC critics = C x DoubleCritic = 2C nets
 * (twin = 1, order r1 r2 c1 c2), DDPG critics = C nets. */
#define FSRL_MAX_NSTEP 8
#define FSRL_OFF_STATS 8
enum { FSRL_OFF_ST_Q0 = 0, FSRL_OFF_ST_Q1 = 1, FSRL_OFF_ST_ACTOR_REW = 2, FSRL_OFF_ST_ACTOR_SAFETY = 3,
       FSRL_OFF_ST_LOGP = 4, FSRL_OFF_ST_ALPHA_LOSS = 5, FSRL_OFF_ST_ALPHA = 6 };
enum { FSRL_ALGO_SAC = 0, FSRL_ALGO_DDPG = 1 };
typedef struct fsrl_offpolicy {
    fsrl_engine_t eng;
    fsrl_netlist_t actor, actor_old, critics, critics_old;
    int algo, D, A, C, twin, n_step, bounded, use_alpha, auto_alpha, use_lagrangian;
    unsigned int seed, pad0;
    double gamma, tau, critic_lr, actor_lr;
    float alpha_lr, target_entropy, max_action, sigma_min, sigma_max, tanh_eps, lagrangian, rescaling;
    /* replay buffer (env-major sub-buffer rings, see fsrl_rollout_t) */
    const float *b_obs, *b_obs_next, *b_act, *b_rew, *b_cost;
    const unsigned char *b_term, *b_trunc;
    const int *b_ptr, *b_len;
    long long cap;
    /* per-step work arrays, all sized for eng.bmax rows */
    int* w_term_idx;
    double *w_partial, *w_gpow;      /* [2][B], [B] */
    float *w_vmask, *w_target;       /* [B], [2][B] */
    float *w_act_next, *w_logp_next, *w_act, *w_logp, *w_keep; /* [B][A], [B], [B][A], [B], [B][24] */
    /* engine scratch views (host-resolved): head outputs / gradients / input gradients */
    float *actor_out, *actor_old_out, *actor_dout;
    float *q_out[4], *q_dout[4], *q_dx[4], *q_old_out[4];
    float* alpha;        /* device scalar */
    float* alpha_state;  /* device [log_alpha, adam_m, adam_v, adam_t] */
    /* data parallel (world > 1): every rank samples its own replay shard; per gradient step the
     * critics' and the actor's gradients are all-reduced (one grouped NCCL call each) and averaged,
     * and the entropy-tuning statistic is all-reduced so that alpha stays identical on all ranks */
    void* comm;
    int world, pad1;
} fsrl_offpolicy_t;

int fsrl_nstep_prepare(const fsrl_offpolicy_t* d, const int* idx, int B, void* stream);
int fsrl_offpolicy_steps(const fsrl_offpolicy_t* d, const int* idx_all, int n_steps, int B,
                         long long critic_t0, long long actor_t0, unsigned long long noise_t0,
                         float* stats, void* stream);

/* ---- a11: CPO (and the CG / Fisher machinery TRPO-Lag shares) ------------------------------------
 * Replaces CPO._get_objective/_get_cost_surrogate/_MVP/_conjugate_gradients/policy_loss
 * (fsrl/policy/cpo.py:163-204,234-351).  The batch is resident: a saved engine forward of the
 * actor (P slot = actor.nets[0].slot) caches h1, h2 and the head output for all N rows;
 * actor_r is the SAME network with a second scratch slot for the R-op quantities.
 *   fsrl_cpo_head(mode)  per-row ratio / KL terms: sums[0..2] = sum ratio*adv_r, sum ratio*adv_c,
 *                        sum kl; mode 1/2/3 also writes the head gradient of the objective,
 *                        of -cost_surrogate, of the mean KL into the P slot's dout
 *   fsrl_cpo_hvp         hv = Hessian(mean KL) v + damping v, exact (R-op), needs the P slot's
 *                        dout / dz2 of the KL gradient pass
 *   fsrl_vec_*           the O(P) vector arithmetic of conjugate gradients / line search */
typedef struct fsrl_cpo {
    fsrl_engine_t eng;
    fsrl_netlist_t actor, actor_r;
    long long N, ld;
    int A, bounded;
    float max_action, pad0;
    const float *obs, *act, *logp_old, *mean_old, *std_old, *adv; /* adv: [2][ld] */
    const int* perm;       /* optional minibatch row indices (NULL = rows 0..N-1) */
    const float* out;      /* P slot head output  [bmax][16] */
    float* dout;           /* P slot head gradient [bmax][16] */
    const float* log_sigma;
} fsrl_cpo_t;

int fsrl_cpo_head(const fsrl_cpo_t* d, int mode, double* sums_dev4, void* stream);
/* FOCOPS actor head (fsrl/policy/focops.py:188-215): loss = mean((KL(new||old) - ratio (A_r - nu A_c) /
 * lambda) * 1[KL <= eta]); d->adv = per-minibatch-normalised advantages; writes d->dout, and
 * sums_dev4 = [sum loss_i, sum KL_i, #rows inside the trust region, 0] */
int fsrl_focops_head(const fsrl_cpo_t* d, double inv_lambda, double nu, double eta, double* sums_dev4,
                     void* stream);
int fsrl_cpo_hvp(const fsrl_cpo_t* d, const float* v, float* v_w2n_scratch, float* hv, double damping,
                 void* stream);
/* x_out = CG(H, rhs), H v = fsrl_cpo_hvp(v): CPO._conjugate_gradients (fsrl/policy/cpo.py:184-204) / TRPOLagrangian
 * (trpo_lag.py:261-283) with every scalar on the device -- `nsteps` iterations enqueued without host synchronisation,
 * the reference's residual break is a device flag.  work: 4 P floats, state_dev: 8 doubles. */
int fsrl_cg_solve(const fsrl_cpo_t* d, const float* rhs, float* x_out, float* work, float* v_w2n_scratch,
                  double* state_dev, long long P, int nsteps, double tol, double damping, void* stream);
int fsrl_vec_dot(const float* a, const float* b, long long n, double* out_dev, void* stream);
int fsrl_vec_axpby(double a, const float* x, double b, float* y, long long n, void* stream);
int fsrl_vec_add_scaled(const float* a, double s, const float* b, float* out, long long n, void* stream);
/* critic regression head (cpo.py:147-157, trpo_lag.py:135-146): dout[i][0] = 2 (V_i - ret_i) / N,
 * sums_dev[0] += sum td^2;  fsrl_standardize: x <- (x - mean) / std (unbiased), cpo.py:127-131 */
int fsrl_mse_head(const float* out, const float* ret, const int* perm, long long N, float* dout,
                  double* sums_dev, void* stream);
int fsrl_standardize(float* x, long long n, void* stream);
int fsrl_engine_wgrad_to(const fsrl_engine_t* e, const fsrl_netlist_t* net1, const fsrl_eng_input_t* in,
                         long long B, float* dst, void* stream);

/* ---- 8(e): multi-GPU plumbing (one process per GPU, NCCL over NVLink) -------------------------
 * The reference has no distributed code; ranks own env shards and replay shards, and per
 * optimiser step ONE all-reduce of the flat gradient buffer is issued from the C update loop.
 * The 128-byte unique id is created on rank 0 and broadcast by the host (torch.distributed). */
int fsrl_comm_unique_id(char* out128);
int fsrl_comm_init(const char* id128, int rank, int world, void** comm_out);
int fsrl_comm_destroy(void* comm);
int fsrl_allreduce_fused(void* comm, float* buf, long long n, void* stream);
int fsrl_allreduce_f64(void* comm, double* buf, long long n, void* stream);
/* Peer-memory exchange block of one rank: [xg0 | xg1 | flags | err | partials], each gradient buffer padded
 * to fsrl_p2p_stride(n) floats.  alloc: cudaMalloc + zero + IPC handle (64 bytes) for the other
 * processes; open / close: map / unmap a peer's block; free: release the own block. */
#define FSRL_P2P_MAX_RANKS 8
#define FSRL_P2P_PARTIALS 4096   /* one per 1024 parameters: peer exchange handles up to 4M parameters */
long long fsrl_p2p_stride(long long n_floats);
long long fsrl_p2p_block_bytes(long long n_floats);
int fsrl_p2p_alloc(long long n_floats, void** base_out, char* ipc64_out);
int fsrl_p2p_open(const char* ipc64, void** peer_base_out);
int fsrl_p2p_close(void* peer_base);
int fsrl_p2p_free(void* base);
int fsrl_p2p_poll_error(const int* err_dev, int* out_host); /* 1 = a peer never arrived */
/* in-place sum of `n_ranges` sub-ranges [base + offs[i], base + offs[i] + counts[i]) in ONE grouped
 * NCCL call (the gradient slices of a net list inside the flat gradient buffer) */
int fsrl_allreduce_ranges(void* comm, float* base, const long long* offs, const long long* counts,
                          int n_ranges, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* FSRL_B200_H */

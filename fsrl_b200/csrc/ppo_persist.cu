// Persistent PPO-Lagrangian update: ONE launch per repeat runs every minibatch step of
// /root/reference/fsrl/policy/ppo_lag.py:223-247 (forward, clipped-surrogate + lambda * cost-advantage
// loss and value losses :152-212, lagrangian_base.py:145-166, backward, clip_grad_norm_, Adam) on a
// co-resident grid of 32 CTAs per network.  Blackwell-native data path: the three 256^3 GEMMs of a
// network and step run on tcgen05 tensor cores (kind::tf32, fp32-faithful 3-term split, accumulators
// in tensor memory), operands arrive as bulk asynchronous copies (TMA unit) of pre-split "plane
// layout" images that the producing CTAs write straight from their epilogues, and the CTAs of a
// step are chained by device-scope release/acquire counters instead of kernel launches.
//
// Work decomposition of one network (H = 256, minibatch = 256 rows = 4 row blocks of 64):
//   CTA c = 8 a + b           a = row block (4), b = 32-wide column block (8)
//   S   h1 tile   [64 r x 32 k]   FFMA (K = D)            -> images H1A (MN = r, K = k), H1T (MN = k, K = r)
//   G1  h2 tile   [64 r x 32 o] = h1[r, :] W2t[:, o]      A = H1A block a, B = W2A block b      (tcgen05)
//       head partial over the tile's 32 columns -> 8 partials per row block -> loss gradient dOut
//       dz2 tile = (dOut W3^T) * relu'(h2)                -> images DZA (MN = r, K = o), DZT (MN = o, K = r)
//   G2  (CTAs 0-15: ka = c / 4, rb = c % 4)  dh1^T tile [64 k x 64 r] = W2t[k, :] dz2[r, :]^T
//       A = W2B block ka, B = DZA block rb;  * relu'(h1) -> partial dW1 / db1 over the 64 rows
//   G3  (CTAs 16-31: ka, ob = c % 4)         dW2^T tile [64 o x 64 k] = dz2[:, o]^T h1[:, k]
//       A = DZT block ob, B = H1T block ka;  the CTA owns this tile of W2: Adam state (p, m, v) lives in
//       tensor memory for the whole launch, the updated tile is re-published as images W2A / W2B
//   small parameters (W1, b1, b2, W3, b3, log sigma): every CTA keeps the slices it consumes (+ their
//       Adam moments) in shared memory and applies the identical update to them (deterministic
//       replicas); gradients are fixed-order sums of per-row-block partials.
//   global-norm clip: per-CTA sums of squares -> one device-wide counter hop -> every CTA adds the
//       96 partials in the same order.
// All operand images are K-major SWIZZLE_NONE plane images (umma.cuh); transposed copies are written
// by the producer (MN-major tf32 operands would need the 128B_BASE32B swizzle).
//
// CTA = 320 threads: warp 0 bulk-copy producer, warp 1 MMA issuer, warps 2-9 epilogue (two per tensor-memory
// subpartition).  The 8 CTAs of a row block form a thread-block cluster: their head partials travel over distributed
// shared memory (st.async + mbarrier complete_tx); all other hops are flag lines in L2.  The cross terms of the 3-term
// split accumulate in their own tensor-memory columns (TM_C).  With world > 1 the <DP = true> instantiation exchanges
// gradients itself over peer memory (dp_* functions below: tagged + hashed 16-byte packets pushed into the peers' buffers).
// DESIGN.md 3a / 6 hold the measurements behind these choices.
#include "ppo_persist.cuh"
#include "arena.cuh"
#include "umma.cuh"
#include <cstdlib>
#include <cmath>
#include <vector>

namespace fsrl {
namespace pp {

using namespace umma;

constexpr int WQ = 2;                    // epilogue warps per tensor-memory subpartition (1 or 2)
constexpr int NEPI = 128 * WQ;           // epilogue threads: warps 2 .. 2 + 4 WQ - 1
constexpr int TPB = 64 + NEPI;           // warp 0: copy producer, warp 1: MMA issuer, then the epilogue warps
constexpr int C1 = 16 / WQ;              // columns a thread owns of a 32-column tile (G1: h2 / dz2)
constexpr int C2 = 32 / WQ;              // columns a thread owns of a 64-column tile (G2 / G3 and the W2 tile)
constexpr int RB = 64;                   // rows per row block
constexpr int MB = 256;                  // rows per minibatch
constexpr int SLOT_BYTES = 65536, NSLOT = 3;
constexpr int OUTP = 8;                  // padded head width
constexpr int H_ = 256;
constexpr int IMG = 65536;               // floats per image (256 x 256)
enum { I_H1A_HI, I_H1A_LO, I_H1T_HI, I_H1T_LO, I_DZA_HI, I_DZA_LO, I_DZT_HI, I_DZT_LO, I_W2A_HI, I_W2A_LO, I_W2B_HI, I_W2B_LO, N_IMG };
// per-network partial buffers (floats)
constexpr int HEADP_OFF = N_IMG * IMG;                          // [4 a][8 b][64 r][OUTP]
constexpr int DB2P_OFF = HEADP_OFF + 4 * 8 * 64 * OUTP;         // [4 a][H]
constexpr int DW3P_OFF = DB2P_OFF + 4 * H_;                     // [4 a][H][OUTP]
constexpr int DB3P_OFF = DW3P_OFF + 4 * H_ * OUTP;              // [4 a][16]
constexpr int DW1P_OFF = DB3P_OFF + 4 * 16;                     // [4 rb][MAXD + 1][H]
constexpr int MAXD = 40;
constexpr int NET_WS = DW1P_OFF + 4 * WQ * (MAXD + 1) * H_;   // [row block 4][warp-in-subpartition WQ][MAXD + 1][H]
constexpr int SUMSQ_FLOATS = 128;                               // global tail: per-CTA sums of squares
// flag lines (32 unsigned each): per net A, C, D1, B[4]; global D2
constexpr int FLAG_LINE = 32;
constexpr int F_A = 0, F_C = 1, F_D1 = 2, F_B = 3, F_PER_NET = 7;
constexpr int TM_COLS = 512, TM_P = 64, TM_M = 96, TM_V = 128;  // tensor-memory columns: [0,64) accumulators, Adam state
// The two cross terms a_lo b_hi + a_hi b_lo accumulate in their OWN tensor-memory columns [TM_C, TM_C + 64) and meet the
// a_hi b_hi sum only in the epilogue: the tensor core's accumulator add drops the low bits of a small addend, and the
// cross terms are 2^-11 of the main ones (tools/micro/umma_probe.cu accuracy study, K = 256: rms error vs fp64 1.7e-6 with
// one accumulator, 5.7e-7 with the corrections apart; an fp32 FMA chain: 1.9e-7).  Same MMA count, one more tcgen05.ld.
constexpr int TM_C = 256;
constexpr int TM_G = 160;                                        // reduced gradient tile (data-parallel runs)
// peer-mapped exchange buffer of one step parity (floats): one region per SOURCE rank [8] plus one for the W2 means
// (written by the packets' owners), each holding per net 16 gradient tiles and the locally reduced small-parameter
// slices of the 8 column blocks.  Ranks PUSH their pieces into
// every peer's buffer as 16-byte packets {3 floats, tag}: the tag (launch sequence number | step) travels with the data,
// so the receiver polls its own memory until every packet carries the tag -- one NVLink one-way latency per exchange,
// no system-scope fence (measured: ~6 us each with posted peer writes outstanding), no flag round trip, no remote loads.
// The tag word is XORed with a hash of the three payload words: a 16-byte vector store does NOT become visible atomically
// to a concurrent 16-byte load on the receiving GPU (measured on 2 x B200: about one packet in 1e9 showed the new tag
// next to a stale payload word, i.e. one diverging parameter update per ~10k optimiser steps; tools/dp_identity_check.py),
// so the receiver accepts a packet only if tag AND payload agree and simply polls again otherwise.
constexpr int NSMAX = (MAXD + 1) * 32 + 32 + 32 * OUTP + 16;
constexpr int TILE_PK = (64 * 64 / NEPI + 2) / 3;                // packets per thread of a 64 x 64 tile (16 floats -> 6)
constexpr int TILE_FLOATS = TILE_PK * NEPI * 4;                  // [packet][thread][4]
constexpr int SLICE_PK = (NSMAX + 2) / 3;
constexpr int XG_PER_NET = 16 * TILE_FLOATS + 8 * SLICE_PK * 4;
constexpr int XG_FLAG_FLOATS = 8 * 128 * 2;                      // (reserved: flag lines of the fenced protocol)
constexpr int MAX_MB = 16384;                                    // minibatches per launch (Adam scalar table)
constexpr long long WAIT_CYCLES = 6000000000LL;                  // ~3 s: a lost partner must not hang the GPU

constexpr int ST_ACTOR_REW = 0, ST_ACTOR_SAFETY = 1, ST_KL = 2, ST_VF0 = 3, ST_ENTROPY = 5, ST_GRADNORM = 6;
constexpr float LOG_SQRT_2PI = 0.9189385332046727f;

struct Args {
    fsrl_ppo_update_t u;     // batch pointers already gathered (contiguous rows, u.perm == nullptr)
    int n_mb, slot0;
    long long adam_t0;
    float* ws;
    unsigned* flags;
    int* err;
    const float* adam_tab;   // [n_mb][2]: 1 / sqrt(1 - beta2^t), -(lr / (1 - beta1^t)) of every step (host doubles -> f32)
    long long* dbg;          // optional [n_cta][DBG_N] clock stamps of step dbg_step
    int dbg_step;
    int cluster;             // launched as clusters of 8 CTAs (one row block): hop B runs over distributed shared memory
    unsigned dp_seq;         // data-parallel runs: launch sequence number (same on every rank), upper half of the packet tags
    int dp_direct;           // W2 gradient tiles exchanged in one hop (2 ranks) instead of the two-hop owner scheme
};
constexpr int DBG_N = 48;
#define STAMP(i) do { if (P.dbg && t == P.dbg_step) P.dbg[(size_t)blockIdx.x * DBG_N + (i)] = clock64(); } while (0)

struct AdamS { float w1, b2, w2, rbc2s, eps, neg_step; };
// torch.optim.Adam's single-tensor update, approximate variant of arena.cuh's adam_one.  The moments are the exact
// fp32 expressions; the parameter step p += step * m / (sqrt(v) / sqrt(bc2) + eps) uses the SFU reciprocal square
// root / reciprocal (about 2 ulp each, i.e. ~1e-10 absolute on a step of <= lr) instead of IEEE sqrt and division,
// whose slow-path calls serialise the 32 elements a lane owns (measured: 19k cycles per step for the 64 x 64 tile
// with IEEE arithmetic).
__device__ __forceinline__ float adam_one_approx(float p, float g, float& m, float& v, const AdamS& a) {
    m = m + a.w1 * (g - m);                 // exp_avg.lerp_(grad, 1 - beta1)
    v = v * a.b2 + (a.w2 * g) * g;          // exp_avg_sq.mul_(beta2).addcmul_(grad, grad, 1 - beta2)
    const float sq = v > 0.f ? v * rsqrtf(v) : 0.f;
    const float denom = fmaf(sq, a.rbc2s, a.eps);
    return p + __fdividef(a.neg_step * m, denom);
}

__device__ __forceinline__ void fail(int* err, int code) {
    *reinterpret_cast<volatile int*>(err) = code;
    __threadfence_system();
    asm volatile("trap;");
}
// one 16-byte packet {x, y, z, tag ^ hash(x, y, z)}: a single vector store into peer memory / a single vector load from
// local memory.  The fourth word vouches for the other three: a packet is accepted only if it carries the expected tag
// AND its payload hashes to what the sender hashed, so a reader can never combine a fresh tag with stale payload words
// (whatever the granularity at which the fabric / L2 make a 16-byte write visible).
__device__ __forceinline__ uint32_t pk_hash(float x, float y, float z) {
    const uint32_t a = __float_as_uint(x), b = __float_as_uint(y), c = __float_as_uint(z);
    return a ^ __funnelshift_l(b, b, 11) ^ __funnelshift_l(c, c, 22);
}
__device__ __forceinline__ bool pk_ok(const float4& v, uint32_t tag) { return (__float_as_uint(v.w) ^ pk_hash(v.x, v.y, v.z)) == tag; }
__device__ __forceinline__ void st_packet(float* p, float x, float y, float z, uint32_t tag) {
    asm volatile("st.relaxed.sys.global.v4.f32 [%0], {%1,%2,%3,%4};" ::"l"(p), "f"(x), "f"(y), "f"(z), "f"(__uint_as_float(tag ^ pk_hash(x, y, z))) : "memory");
}
__device__ __forceinline__ float4 ld_packet(const float* p) {
    float4 v;
    asm volatile("ld.relaxed.sys.global.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p) : "memory");
    return v;
}

// Wait for the packets of all ranks but `me` at src + r * stride (local memory, pushed by the peers) and add them to the
// own piece (ox, oy, oz) in rank order.  Deliberately not inlined: the exchange code runs once per step and the kernel's
// instruction footprint matters (measured: the step slows down by ~10 % when the exchange is unrolled into the epilogue).
__device__ __noinline__ float3 dp_gather(const float* src, long long stride, int me, int world, uint32_t tag,
                                        float ox, float oy, float oz, int* err, int code) {
    const long long t0w = clock64();
    float ax = 0.f, ay = 0.f, az = 0.f;
    for (int r0 = 0; r0 < world; r0 += 4) {                // four ranks' packets in flight, rank order kept
        float4 v[4];
        bool ok;
        do {
            ok = true;
#pragma unroll
            for (int k = 0; k < 4; ++k)
                if (r0 + k < world && r0 + k != me) v[k] = ld_packet(src + (size_t)(r0 + k) * stride);
#pragma unroll
            for (int k = 0; k < 4; ++k)
                if (r0 + k < world && r0 + k != me) ok = ok && pk_ok(v[k], tag);
            if (!ok && clock64() - t0w > 4 * WAIT_CYCLES) fail(err, code);
        } while (!ok);
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            if (r0 + k >= world) continue;
            if (r0 + k == me) { ax += ox; ay += oy; az += oz; }
            else { ax += v[k].x; ay += v[k].y; az += v[k].z; }
        }
    }
    return make_float3(ax, ay, az);
}
// one packet to every rank but `me`: dst_r = xg[r] + off
__device__ __noinline__ void dp_push_all(const float* const* xg, size_t off, int me, int world, float x, float y, float z, uint32_t tag) {
    for (int r = 0; r < world; ++r)
        if (r != me) st_packet(const_cast<float*>(xg[r]) + off, x, y, z, tag);
}

// ---- thread-block cluster: distributed shared memory pushes + remote mbarrier arrivals (hop B) ------------------------
__device__ __forceinline__ uint32_t mapa_u32(uint32_t local_saddr, uint32_t rank) {
    uint32_t r;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(local_saddr), "r"(rank));
    return r;
}
__device__ __forceinline__ void st_cluster4(uint32_t raddr, float4 v) {
    asm volatile("st.shared::cluster.v4.f32 [%0], {%1,%2,%3,%4};" ::"r"(raddr), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}
// asynchronous remote store that completes 16 transaction bytes on the destination CTA's mbarrier: the data signals
// its own arrival, so no release fence / arrival round trip follows the push
__device__ __forceinline__ void st_async4(uint32_t raddr, float4 v, uint32_t rbar) {
    asm volatile("st.async.weak.shared::cluster.mbarrier::complete_tx::bytes.v4.f32 [%0], {%1,%2,%3,%4}, [%5];"
                 ::"r"(raddr), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w), "r"(rbar) : "memory");
}
__device__ __forceinline__ bool mbar_wait_cluster(uint64_t* bar, uint32_t parity, long long timeout_cycles) {
    const long long t0 = clock64();
    while (true) {
        uint32_t ok;
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.acquire.cluster.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(ok) : "r"(smem_u32(bar)), "r"(parity) : "memory");
        if (ok) return true;
        if (clock64() - t0 > timeout_cycles) return false;
    }
}
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}

// one thread of a converged warp (CUTLASS elect_one_sync): lets the compiler issue the uniform-datapath
// instructions (UTCHMMA, UBLKCP) of the region directly instead of wrapping each in a vote loop
__device__ __forceinline__ bool elect_one() {
    uint32_t pred = 0;
    asm volatile(
        "{\n\t.reg .b32 rx;\n\t.reg .pred px;\n\t"
        "elect.sync rx|px, 0xffffffff;\n\t"
        "selp.u32 %0, 1, 0, px;\n\t}"
        : "=r"(pred));
    return pred != 0;
}
__device__ __forceinline__ void epi_bar() { asm volatile("bar.sync 1, %0;" ::"n"(NEPI) : "memory"); }
__device__ __forceinline__ void prefetch_l2(const void* p) { asm volatile("prefetch.global.L2 [%0];" ::"l"(p)); }

__device__ __forceinline__ void tmem_st32(uint32_t taddr, const float (&v)[32]) {
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,"
        "%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31,%32};"
        ::"r"(taddr), "r"(__float_as_uint(v[0])), "r"(__float_as_uint(v[1])), "r"(__float_as_uint(v[2])), "r"(__float_as_uint(v[3])),
          "r"(__float_as_uint(v[4])), "r"(__float_as_uint(v[5])), "r"(__float_as_uint(v[6])), "r"(__float_as_uint(v[7])),
          "r"(__float_as_uint(v[8])), "r"(__float_as_uint(v[9])), "r"(__float_as_uint(v[10])), "r"(__float_as_uint(v[11])),
          "r"(__float_as_uint(v[12])), "r"(__float_as_uint(v[13])), "r"(__float_as_uint(v[14])), "r"(__float_as_uint(v[15])),
          "r"(__float_as_uint(v[16])), "r"(__float_as_uint(v[17])), "r"(__float_as_uint(v[18])), "r"(__float_as_uint(v[19])),
          "r"(__float_as_uint(v[20])), "r"(__float_as_uint(v[21])), "r"(__float_as_uint(v[22])), "r"(__float_as_uint(v[23])),
          "r"(__float_as_uint(v[24])), "r"(__float_as_uint(v[25])), "r"(__float_as_uint(v[26])), "r"(__float_as_uint(v[27])),
          "r"(__float_as_uint(v[28])), "r"(__float_as_uint(v[29])), "r"(__float_as_uint(v[30])), "r"(__float_as_uint(v[31]))
        : "memory");
    asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_st16(uint32_t taddr, const float (&v)[16]) {
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16};"
        ::"r"(taddr), "r"(__float_as_uint(v[0])), "r"(__float_as_uint(v[1])), "r"(__float_as_uint(v[2])), "r"(__float_as_uint(v[3])),
          "r"(__float_as_uint(v[4])), "r"(__float_as_uint(v[5])), "r"(__float_as_uint(v[6])), "r"(__float_as_uint(v[7])),
          "r"(__float_as_uint(v[8])), "r"(__float_as_uint(v[9])), "r"(__float_as_uint(v[10])), "r"(__float_as_uint(v[11])),
          "r"(__float_as_uint(v[12])), "r"(__float_as_uint(v[13])), "r"(__float_as_uint(v[14])), "r"(__float_as_uint(v[15]))
        : "memory");
    asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_ld8(uint32_t taddr, float (&v)[8]) {
    uint32_t r[8];
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]) : "r"(taddr));
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
    for (int i = 0; i < 8; ++i) v[i] = __uint_as_float(r[i]);
}
// two loads in flight, one wait (NC = 8 / 16): the accumulator columns and their correction columns
template <int NC> __device__ __forceinline__ void tmem_ld_pair(uint32_t ta, uint32_t tb, float (&x)[NC], float (&y)[NC]) {
    static_assert(NC == 8 || NC == 16, "pair loads in use");
    uint32_t r[NC], q[NC];
    if constexpr (NC == 8) {
        asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                     : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]) : "r"(ta));
        asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                     : "=r"(q[0]), "=r"(q[1]), "=r"(q[2]), "=r"(q[3]), "=r"(q[4]), "=r"(q[5]), "=r"(q[6]), "=r"(q[7]) : "r"(tb));
    } else {
        asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
                     : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
                       "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]) : "r"(ta));
        asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
                     : "=r"(q[0]), "=r"(q[1]), "=r"(q[2]), "=r"(q[3]), "=r"(q[4]), "=r"(q[5]), "=r"(q[6]), "=r"(q[7]), "=r"(q[8]),
                       "=r"(q[9]), "=r"(q[10]), "=r"(q[11]), "=r"(q[12]), "=r"(q[13]), "=r"(q[14]), "=r"(q[15]) : "r"(tb));
    }
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
    for (int i = 0; i < NC; ++i) { x[i] = __uint_as_float(r[i]); y[i] = __uint_as_float(q[i]); }
}
// NC = 8 / 16 / 32 consecutive columns of this thread's tensor-memory lane
template <int NC> __device__ __forceinline__ void tmem_ldn(uint32_t taddr, float (&v)[NC]) {
    if constexpr (NC == 8) tmem_ld8(taddr, v);
    else if constexpr (NC == 16) tmem_ld16(taddr, v);
    else tmem_ld32(taddr, v);
}
template <int NC> __device__ __forceinline__ void tmem_stn(uint32_t taddr, const float (&v)[NC]) {
    static_assert(NC == 16 || NC == 32, "tensor-memory store widths in use");
    if constexpr (NC == 16) tmem_st16(taddr, v);
    else tmem_st32(taddr, v);
}

// The M = 64 accumulators occupy the lower 16 lanes of every tensor-memory subpartition (one MMA per k-step keeps the
// shared-memory operand traffic down -- the A tile is re-read by every instruction).  All 32 lanes of the WQ warps that
// share a subpartition split the columns: lane l < 16 of warp-in-subpartition wq keeps columns [col_lo, col_lo + NC), lane
// l + 16 receives columns [col_hi, col_hi + NC) of lane l.
template <int NC>
__device__ __forceinline__ void acc_ld_split(uint32_t taddr, int lane, int col_lo, int col_hi, float (&v)[NC]) {
    float w[NC];
    {
        float c[NC];
        tmem_ld_pair<NC>(taddr + col_hi, taddr + TM_C + col_hi, w, c);
#pragma unroll
        for (int j = 0; j < NC; ++j) w[j] += c[j];
        tmem_ld_pair<NC>(taddr + col_lo, taddr + TM_C + col_lo, v, c);
#pragma unroll
        for (int j = 0; j < NC; ++j) v[j] += c[j];
    }
#pragma unroll
    for (int j = 0; j < NC; ++j) {
        const float x = __shfl_sync(0xffffffffu, w[j], lane & 15);
        v[j] = (lane & 16) ? x : v[j];
    }
}

// Transposed K-major image of a 64-row tile through shared memory.  Every epilogue thread holds NC consecutive
// columns [c0, c0 + NC) of tile row `row` (hi / lo parts); the tile is W columns wide.  The transposed image
// stores 4 consecutive ROWS of one column as 16 contiguous bytes: element (col, row) at
//     img[(row_base + row) / 4 * 256 + (col_base + col) * 4 + (row_base + row) % 4],     lo image at + IMG.
// (W = tile width in columns.)  Writing it straight from the registers costs NC scattered 4-byte stores per thread and image (16 sectors per warp
// instruction); staged through `scr` (an idle operand-ring slot, row stride 65: conflict-free) it becomes
// float4 stores, 512 contiguous bytes per warp instruction.
template <int NC, int W>
__device__ __forceinline__ void transposed_stage(float* scr, const float (&hi)[NC], const float (&lo)[NC], int row, int c0) {
    constexpr int LO = W * 65;
#pragma unroll
    for (int j = 0; j < NC; ++j) {
        scr[(c0 + j) * 65 + row] = hi[j];
        scr[LO + (c0 + j) * 65 + row] = lo[j];
    }
}
template <int W>
__device__ __forceinline__ void transposed_flush(const float* scr, int et, float* img_hi, int row_base, int col_base) {
    constexpr int LO = W * 65;
    const int col = et % W;
    constexpr int GPT = 16 / (NEPI / W);                       // row groups (of 4 rows) per thread
    const int g0 = (et / W) * GPT;
    float* dst = img_hi + (size_t)(row_base >> 2) * 256 + (size_t)(col_base + col) * 4;
#pragma unroll
    for (int q = 0; q < GPT; ++q) {
        const int g = g0 + q;
        const float* sh = scr + col * 65 + 4 * g;
        *reinterpret_cast<float4*>(dst + (size_t)g * 256) = make_float4(sh[0], sh[1], sh[2], sh[3]);
        *reinterpret_cast<float4*>(dst + IMG + (size_t)g * 256) = make_float4(sh[LO], sh[LO + 1], sh[LO + 2], sh[LO + 3]);
    }
}
template <int NC, int W>
__device__ __forceinline__ void store_transposed(float* scr, const float (&hi)[NC], const float (&lo)[NC], int row, int c0,
                                                 int et, float* img_hi, int row_base, int col_base) {
    transposed_stage<NC, W>(scr, hi, lo, row, c0);
    epi_bar();
    transposed_flush<W>(scr, et, img_hi, row_base, col_base);
    epi_bar();                                                 // scratch may be reused
}

// sum over the 16 lanes of a half-warp (lanes l and l ^ 16 hold different data)
__device__ __forceinline__ float half_sum(float v) {
#pragma unroll
    for (int o = 8; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// layout of the small-parameter slices a CTA keeps in shared memory (floats)
struct SliceMap {
    int w1, b2, w3, b3, n;     // w1: [(D+1)][32] (row D = b1), b2: [32], w3: [32][OUTP], b3: [16] (b3 | log sigma at 8)
    __device__ __host__ SliceMap(int D) { w1 = 0; b2 = (D + 1) * 32; w3 = b2 + 32; b3 = w3 + 32 * OUTP; n = b3 + 16; }
};

// ---- data-parallel exchange, out of line ---------------------------------------------------------------------------------
// All of it lives in functions the kernel CALLS: inlined into the epilogue, the mere presence of this code slowed every
// phase of the step down by ~9 % (measured with the exchange compiled in but world = 1) -- register allocation and the
// instruction footprint of the ~7k-instruction epilogue are that tight.
struct DpCtx {
    const float* const* xg;   // [rank] exchange buffers of this step's parity (shared-memory table)
    long long region;         // floats per source-rank region
    int me, world;
    uint32_t tag;
    int* err;
    int direct;               // W2 tiles in ONE hop (every rank sums all ranks' tiles itself): less latency, W - 1 tile
                              // volumes per rank -- the choice for 2 ranks; the two-hop owner scheme beyond
};
__device__ __forceinline__ int dp_owner(int et, int q, int world) { return (int)((unsigned)((et >> 5) * TILE_PK + q) % (unsigned)world); }

// hop 1 of a W2 gradient tile: every packet of the local tile (tensor-memory accumulators) to its owner
__device__ __noinline__ void dp_tile_send(DpCtx d, size_t off, uint32_t tm_lane, int lane, int wq, int et) {
    float g[C2];
    acc_ld_split<C2>(tm_lane, lane, C2 * wq, 32 + C2 * wq, g);
#pragma unroll
    for (int q = 0; q < TILE_PK; ++q) {
        const size_t o_q = (size_t)d.me * d.region + off + (size_t)q * NEPI * 4;
        const float x = g[3 * q], y = 3 * q + 1 < C2 ? g[3 * q + 1] : 0.f, z = 3 * q + 2 < C2 ? g[3 * q + 2] : 0.f;
        if (d.direct) {
            dp_push_all(d.xg, o_q, d.me, d.world, x, y, z, d.tag);
        } else {
            const int o = dp_owner(et, q, d.world);
            if (o != d.me) st_packet(const_cast<float*>(d.xg[o]) + o_q, x, y, z, d.tag);
        }
    }
}
// hop 2: owned packets -- rank-ordered mean of the ranks' contributions, pushed into everybody's result region; the tile
// (owned entries final, the others still local) goes to tensor-memory columns TM_G
__device__ __noinline__ void dp_tile_reduce(DpCtx d, size_t off, uint32_t tm_lane, int lane, int wq, int et) {
    float g[C2];
    acc_ld_split<C2>(tm_lane, lane, C2 * wq, 32 + C2 * wq, g);
    const float inv_world = 1.0f / (float)d.world;
    const float* loc = d.xg[d.me];
#pragma unroll
    for (int q = 0; q < TILE_PK; ++q) {
        if (dp_owner(et, q, d.world) != d.me) continue;
        const float3 s3 = dp_gather(loc + off + (size_t)q * NEPI * 4, d.region, d.me, d.world, d.tag, g[3 * q],
                                    3 * q + 1 < C2 ? g[3 * q + 1] : 0.f, 3 * q + 2 < C2 ? g[3 * q + 2] : 0.f, d.err, 41);
        const float ax = s3.x * inv_world, ay = s3.y * inv_world, az = s3.z * inv_world;
        dp_push_all(d.xg, (size_t)FSRL_P2P_MAX_RANKS * d.region + off + (size_t)q * NEPI * 4, d.me, d.world, ax, ay, az, d.tag);
        g[3 * q] = ax;
        if (3 * q + 1 < C2) g[3 * q + 1] = ay;
        if (3 * q + 2 < C2) g[3 * q + 2] = az;
    }
    __syncwarp();      // the lanes left their poll loops at different times: tcgen05.st is .sync.aligned
    tmem_stn<C2>(tm_lane + TM_G + C2 * wq, g);
}
// the other owners' means: wait for them in the local result region, complete the tile in TM_G, return its sum of squares
__device__ __noinline__ float dp_tile_finish(DpCtx d, size_t off, uint32_t tm_lane, int lane, int wq, int et) {
    float g[C2];
    const long long t0w = clock64();
    if (d.direct) {
        // one hop: all ranks' tiles are (or will be) in the local contribution regions -- rank-ordered mean, rank by rank
        float own[C2];
        acc_ld_split<C2>(tm_lane, lane, C2 * wq, 32 + C2 * wq, own);
#pragma unroll
        for (int jq = 0; jq < C2; ++jq) g[jq] = 0.f;
        for (int r = 0; r < d.world; ++r) {
            if (r == d.me) {
#pragma unroll
                for (int jq = 0; jq < C2; ++jq) g[jq] += own[jq];
                continue;
            }
            const float* src = d.xg[d.me] + (size_t)r * d.region + off;
            float4 v[TILE_PK];
            bool ok;
            do {
                ok = true;
#pragma unroll
                for (int q = 0; q < TILE_PK; ++q) v[q] = ld_packet(src + (size_t)q * NEPI * 4);
#pragma unroll
                for (int q = 0; q < TILE_PK; ++q) ok = ok && pk_ok(v[q], d.tag);
                if (!ok && clock64() - t0w > 4 * WAIT_CYCLES) fail(d.err, 42);
            } while (!ok);
#pragma unroll
            for (int q = 0; q < TILE_PK; ++q) {
                g[3 * q] += v[q].x;
                if (3 * q + 1 < C2) g[3 * q + 1] += v[q].y;
                if (3 * q + 2 < C2) g[3 * q + 2] += v[q].z;
            }
        }
        const float inv_world = 1.0f / (float)d.world;
        float sq = 0.f;
#pragma unroll
        for (int jq = 0; jq < C2; ++jq) { g[jq] *= inv_world; sq = fmaf(g[jq], g[jq], sq); }
        __syncwarp();  // the lanes left their poll loops at different times: tcgen05.st is .sync.aligned
        tmem_stn<C2>(tm_lane + TM_G + C2 * wq, g);
        return sq;
    }
    const float* res = d.xg[d.me] + (size_t)FSRL_P2P_MAX_RANKS * d.region + off;
    tmem_ldn<C2>(tm_lane + TM_G + C2 * wq, g);
    float4 v[TILE_PK];
    bool ok;
    do {
        ok = true;
#pragma unroll
        for (int q = 0; q < TILE_PK; ++q)
            if (dp_owner(et, q, d.world) != d.me) v[q] = ld_packet(res + (size_t)q * NEPI * 4);
#pragma unroll
        for (int q = 0; q < TILE_PK; ++q)
            if (dp_owner(et, q, d.world) != d.me) ok = ok && pk_ok(v[q], d.tag);
        if (!ok && clock64() - t0w > 4 * WAIT_CYCLES) fail(d.err, 42);
    } while (!ok);
    float sq = 0.f;
#pragma unroll
    for (int q = 0; q < TILE_PK; ++q) {
        if (dp_owner(et, q, d.world) == d.me) continue;
        g[3 * q] = v[q].x;
        if (3 * q + 1 < C2) g[3 * q + 1] = v[q].y;
        if (3 * q + 2 < C2) g[3 * q + 2] = v[q].z;
    }
#pragma unroll
    for (int jq = 0; jq < C2; ++jq) sq = fmaf(g[jq], g[jq], sq);
    __syncwarp();
    tmem_stn<C2>(tm_lane + TM_G + C2 * wq, g);
    return sq;
}
// small-parameter slices of one column block (n floats in shared memory): row block 0 pushes them to every rank, every
// CTA of the column block replaces them by the rank-ordered mean (one hop: this exchange is on the step's critical path)
__device__ __noinline__ void dp_slices(DpCtx d, size_t off_s, float* sp_g, int n, int et, bool push) {
    const int n3 = (n + 2) / 3;
    const float inv_world = 1.0f / (float)d.world;
    if (push)
        for (int i = et; i < n3; i += NEPI)
            dp_push_all(d.xg, (size_t)d.me * d.region + off_s + 4 * (size_t)i, d.me, d.world,
                        sp_g[3 * i], 3 * i + 1 < n ? sp_g[3 * i + 1] : 0.f, 3 * i + 2 < n ? sp_g[3 * i + 2] : 0.f, d.tag);
    const float* loc = d.xg[d.me];
    for (int i = et; i < n3; i += NEPI) {
        const float3 s3 = dp_gather(loc + off_s + 4 * (size_t)i, d.region, d.me, d.world, d.tag, sp_g[3 * i],
                                    3 * i + 1 < n ? sp_g[3 * i + 1] : 0.f, 3 * i + 2 < n ? sp_g[3 * i + 2] : 0.f, d.err, 40);
        sp_g[3 * i] = s3.x * inv_world;
        if (3 * i + 1 < n) sp_g[3 * i + 1] = s3.y * inv_world;
        if (3 * i + 2 < n) sp_g[3 * i + 2] = s3.z * inv_world;
    }
}

// DP = false: single-GPU instantiation without any of the exchange code (smaller instruction footprint)
template <bool DP>
__global__ void __launch_bounds__(TPB, 1) ppo_persist_kernel(const Args P) {
    extern __shared__ __align__(1024) unsigned char smem_raw[];
    __shared__ __align__(8) uint64_t bar_full[NSLOT], bar_empty[NSLOT], bar_acc, bar_b;
    __shared__ uint32_t s_tmem;
    __shared__ float s_red[4][320];          // cross-subpartition partial sums
    __shared__ float s_misc[32];
    __shared__ AdamS s_adam;
    __shared__ const float* s_xg[2][FSRL_P2P_MAX_RANKS];   // peers' exchange buffers (a table the exchange helpers can index)
    const fsrl_ppo_update_t& u = P.u;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int net = blockIdx.x >> 5, c = blockIdx.x & 31, a = c >> 3, b = c & 7;
    const bool is_g2 = c < 16;
    const int ka = (c & 15) >> 2, q4 = c & 3;      // G2: (k block, row block) ; G3: (k block, o block)
    const int D = u.D, A = u.A, C = u.C, H = H_;
    const int out = (net == 0) ? A : 1;
    const int n_cta = 32 * u.n_nets;
    float* wsn = P.ws + (size_t)net * NET_WS;
    float* sumsq_g = P.ws + (size_t)u.n_nets * NET_WS;
    unsigned* fl_net = P.flags + (size_t)net * F_PER_NET * FLAG_LINE;
    unsigned* fl_d2 = P.flags + (size_t)u.n_nets * F_PER_NET * FLAG_LINE;
    unsigned char* ring = smem_raw;
    float* small = reinterpret_cast<float*>(smem_raw + NSLOT * SLOT_BYTES);
    const SliceMap sm(D);
    float* sp_p = small;                 // parameters
    float* sp_m = small + sm.n;          // Adam first moment
    float* sp_v = small + 2 * sm.n;      // Adam second moment
    float* sp_g = small + 3 * sm.n;      // reduced gradient of the current step
    float* land = small + 4 * sm.n;      // cluster mode: head partials pushed by the 8 CTAs of this row block [b][64][OUTP]

    if (tid == 0) {
        for (int i = 0; i < NSLOT; ++i) { mbar_init(&bar_full[i], 1); mbar_init(&bar_empty[i], 1); }
        mbar_init(&bar_acc, 1);
        mbar_init(&bar_b, 1);                // per step: one local expect_tx arrival + 16 KB of remote st.async bytes
        fence_mbar_init();
    }
    if (warp == 1) tmem_alloc<TM_COLS>(&s_tmem);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = s_tmem;
    if (DP && threadIdx.x < 2 * FSRL_P2P_MAX_RANKS) s_xg[threadIdx.x / FSRL_P2P_MAX_RANKS][threadIdx.x % FSRL_P2P_MAX_RANKS] = P.u.p2p_xg[threadIdx.x / FSRL_P2P_MAX_RANKS][threadIdx.x % FSRL_P2P_MAX_RANKS];
    if (DP) __syncthreads();
    if (P.cluster) cluster_sync_all();       // every CTA's barriers exist before a peer may arrive on them

    // parameter offsets of this network inside the flat arena
    const long long pbase = u.net_off[net];
    const NetLayout L(D, H, out, (net == 0 && u.head_indep) ? A : 0);
    const long long o_w1 = pbase + L.w1, o_b1 = pbase + L.b1, o_w2 = pbase + L.w2, o_b2 = pbase + L.b2,
                    o_w3 = pbase + L.w3, o_b3 = pbase + L.b3, o_ls = pbase + L.extra;

    if (warp == 0) {
        // ============================ bulk-copy producer ==========================================
        if (elect_one()) {
            unsigned qq = 0;
            for (int t = 0; t < P.n_mb; ++t) {
                if (!flag_wait_ge<true>(fl_net + F_A * FLAG_LINE, 32u * (t + 1), WAIT_CYCLES)) fail(P.err, 10);
                STAMP(12);
                fence_proxy_async();
                for (int j = 0; j < 4; ++j, ++qq) {               // G1: K = k in chunks of 64
                    const int s = qq % NSLOT;
                    if (!mbar_wait(&bar_empty[s], ((qq / NSLOT) & 1) ^ 1, WAIT_CYCLES)) fail(P.err, 11);
                    unsigned char* dst = ring + (size_t)s * SLOT_BYTES;
                    mbar_expect_tx(&bar_full[s], 49152);
                    const size_t ao = (size_t)a * 16384 + (size_t)j * 4096, bo = (size_t)b * 8192 + (size_t)j * 2048;
                    bulk_g2s(dst, wsn + (size_t)I_H1A_HI * IMG + ao, 16384, &bar_full[s]);
                    bulk_g2s(dst + 16384, wsn + (size_t)I_H1A_LO * IMG + ao, 16384, &bar_full[s]);
                    bulk_g2s(dst + 32768, wsn + (size_t)I_W2A_HI * IMG + bo, 8192, &bar_full[s]);
                    bulk_g2s(dst + 40960, wsn + (size_t)I_W2A_LO * IMG + bo, 8192, &bar_full[s]);
                }
                STAMP(13);
                if (!flag_wait_ge<true>(fl_net + F_C * FLAG_LINE, 32u * (t + 1), WAIT_CYCLES)) fail(P.err, 12);
                STAMP(14);
                fence_proxy_async();
                const int ia = is_g2 ? I_W2B_HI : I_DZT_HI, ib = is_g2 ? I_DZA_HI : I_H1T_HI;
                const int blk_a = is_g2 ? ka : q4, blk_b = is_g2 ? q4 : ka;
                for (int j = 0; j < 4; ++j, ++qq) {               // G2: K = o ; G3: K = r ; chunks of 64
                    const int s = qq % NSLOT;
                    if (!mbar_wait(&bar_empty[s], ((qq / NSLOT) & 1) ^ 1, WAIT_CYCLES)) fail(P.err, 13);
                    unsigned char* dst = ring + (size_t)s * SLOT_BYTES;
                    mbar_expect_tx(&bar_full[s], 65536);
                    const size_t ao = (size_t)blk_a * 16384 + (size_t)j * 4096, bo = (size_t)blk_b * 16384 + (size_t)j * 4096;
                    bulk_g2s(dst, wsn + (size_t)ia * IMG + ao, 16384, &bar_full[s]);
                    bulk_g2s(dst + 16384, wsn + (size_t)(ia + 1) * IMG + ao, 16384, &bar_full[s]);
                    bulk_g2s(dst + 32768, wsn + (size_t)ib * IMG + bo, 16384, &bar_full[s]);
                    bulk_g2s(dst + 49152, wsn + (size_t)(ib + 1) * IMG + bo, 16384, &bar_full[s]);
                }
            }
        }
    } else if (warp == 1) {
        // ============================ MMA issuer ==================================================
        if (elect_one()) {
            unsigned qq = 0;
            const uint32_t ring_a = smem_u32(ring);
            const uint32_t id32 = idesc_tf32(64, 32, false, false), id64 = idesc_tf32(64, 64, false, false);
            for (int t = 0; t < P.n_mb; ++t) {
                for (int j = 0; j < 4; ++j, ++qq) {               // ---- G1: D[64 r][32 o], two 16-column halves
                    const int s = qq % NSLOT;
                    if (!mbar_wait(&bar_full[s], (qq / NSLOT) & 1, WAIT_CYCLES)) fail(P.err, 20);
                    tc_fence_after();
                    if (j == 0) STAMP(16);
                    if (j == 3) STAMP(17);
                    const uint32_t base = ring_a + (uint32_t)s * SLOT_BYTES;
#pragma unroll 4
                    for (int ks = 0; ks < 8; ++ks) {
                        const uint64_t ah = smem_desc(base + ks * 2048, 1024, 128);
                        const uint64_t al = smem_desc(base + 16384 + ks * 2048, 1024, 128);
                        const uint64_t bh = smem_desc(base + 32768 + ks * 1024, 512, 128);
                        const uint64_t bl = smem_desc(base + 40960 + ks * 1024, 512, 128);
                        mma_tf32_ss(tmem + TM_C, al, bh, id32, (j | ks) != 0);
                        mma_tf32_ss(tmem + TM_C, ah, bl, id32, true);
                        mma_tf32_ss(tmem, ah, bh, id32, (j | ks) != 0);
                    }
                    mma_commit(&bar_empty[s]);
                }
                mma_commit(&bar_acc);
                STAMP(18);
                for (int j = 0; j < 4; ++j, ++qq) {               // ---- G2 / G3: D[64][64], two 32-column halves
                    const int s = qq % NSLOT;
                    if (!mbar_wait(&bar_full[s], (qq / NSLOT) & 1, WAIT_CYCLES)) fail(P.err, 21);
                    tc_fence_after();
                    if (j == 0) STAMP(19);
                    if (j == 3) STAMP(20);
                    const uint32_t base = ring_a + (uint32_t)s * SLOT_BYTES;
#pragma unroll 4
                    for (int ks = 0; ks < 8; ++ks) {
                        const uint64_t ah = smem_desc(base + ks * 2048, 1024, 128);
                        const uint64_t al = smem_desc(base + 16384 + ks * 2048, 1024, 128);
                        const uint64_t bh = smem_desc(base + 32768 + ks * 2048, 1024, 128);
                        const uint64_t bl = smem_desc(base + 49152 + ks * 2048, 1024, 128);
                        mma_tf32_ss(tmem + TM_C, al, bh, id64, (j | ks) != 0);
                        mma_tf32_ss(tmem + TM_C, ah, bl, id64, true);
                        mma_tf32_ss(tmem, ah, bh, id64, (j | ks) != 0);
                    }
                    mma_commit(&bar_empty[s]);
                }
                mma_commit(&bar_acc);
                STAMP(21);
            }
        }
    } else {
        // ============================ epilogue warps ===============================================
        const int et = tid - 64;                    // 0 .. NEPI - 1
        const int sp = warp & 3;                    // tensor-memory subpartition of this warp
        const int wq = (warp - 2) >> 2;             // which of the WQ warps of that subpartition
        const int r16 = lane & 15, half = lane >> 4;
        const int trow = 16 * sp + r16;             // row of the 64-row tile held by this lane
        const int cb1 = 16 * half + C1 * wq;        // first of this thread's C1 columns of a 32-column tile
        const int cb2 = 32 * half + C2 * wq;        // first of this thread's C2 columns of a 64-column tile
        const uint32_t tm_lane = tmem + ((uint32_t)(32 * sp) << 16);
        float* stat_base = u.stats;
        // ---- data-parallel exchange over peer memory (NVLink): every CTA pushes its local gradient piece into its
        // rank's region of EVERY rank's exchange buffer, one thread fences and release-stores the step id into the same
        // slot of every rank's flag array; the receiver waits for the ranks' flags and sums their pieces from its own
        // memory in rank order -- point-to-point between equal CTAs, one NVLink one-way latency, no remote loads,
        // bit-identical sums on every rank.
        const int world = (DP && u.world > 1) ? u.world : 1;
        const float inv_world = 1.0f / (float)world;
        // W2 tiles travel in two hops (reduce-scatter + all-gather, 2 (W - 1) / W tile volumes per rank instead of W - 1):
        // packet q of epilogue warp w is OWNED by rank (6 w + q) mod W -- every rank sends it there, the owner sums the
        // ranks' packets in rank order and pushes the mean into everybody's result region (region 8).  Both hops are
        // hidden behind the dW1 hop / slice reduction of the same step; the result is bit-identical on every rank.
        auto dp_ctx = [&](int t_) {
            DpCtx d;
            const unsigned long long id = (unsigned long long)(P.adam_t0 + t_ + 1);
            d.xg = s_xg[(int)(id & 1ULL)];
            d.region = (long long)u.n_nets * XG_PER_NET;
            d.me = u.p2p_rank; d.world = world;
            d.tag = (P.dp_seq << 16) | (uint32_t)((t_ + 1) & 0xffff);
            d.err = P.err;
            d.direct = P.dp_direct;
            return d;
        };

        // ---- initial state: small slices from the arena, the W2 tile (p, m, v) into tensor memory ----
        for (int i = et; i < sm.n; i += NEPI) {
            long long src = -1;
            if (i < sm.b2) { const int d = i / 32, kk = i % 32; src = (d < D) ? o_w1 + (long long)d * H + 32 * b + kk : o_b1 + 32 * b + kk; }
            else if (i < sm.w3) src = o_b2 + 32 * b + (i - sm.b2);
            else if (i < sm.b3) { const int oo = (i - sm.w3) / OUTP, jj = (i - sm.w3) % OUTP; if (jj < out) src = o_w3 + (long long)(32 * b + oo) * out + jj; }
            else { const int jj = i - sm.b3; if (jj < out) src = o_b3 + jj; else if (net == 0 && u.head_indep && jj >= 8 && jj < 8 + A) src = o_ls + (jj - 8); }
            sp_p[i] = src >= 0 ? u.theta[src] : 0.f;
            sp_m[i] = src >= 0 ? u.adam_m[src] : 0.f;
            sp_v[i] = src >= 0 ? u.adam_v[src] : 0.f;
            sp_g[i] = 0.f;
        }
        if (!is_g2) {
            const int o = 64 * q4 + trow;
            float pv[C2], mv[C2], vv[C2];
#pragma unroll
            for (int j = 0; j < C2; ++j) {
                const long long idx = o_w2 + (long long)(64 * ka + cb2 + j) * H + o;
                pv[j] = u.theta[idx]; mv[j] = u.adam_m[idx]; vv[j] = u.adam_v[idx];
            }
            tmem_stn<C2>(tm_lane + TM_P + C2 * wq, pv); tmem_stn<C2>(tm_lane + TM_M + C2 * wq, mv); tmem_stn<C2>(tm_lane + TM_V + C2 * wq, vv);
        }
        epi_bar();

        unsigned acc_phase = 0;
        for (int t = 0; t < P.n_mb; ++t) {
            const long long row0 = (long long)t * MB;                 // first row of the minibatch in the gathered arrays
            const int slot = P.slot0 + t;
            if (et == 0) {   // Adam scalars of this step (torch.optim.Adam: python doubles -> f32 at the op; host table)
                s_adam.w1 = (float)(1.0 - u.beta1); s_adam.b2 = (float)u.beta2; s_adam.w2 = (float)(1.0 - u.beta2);
                s_adam.rbc2s = __ldg(P.adam_tab + 2 * t); s_adam.eps = (float)u.adam_eps; s_adam.neg_step = __ldg(P.adam_tab + 2 * t + 1);
                STAMP(0);
                if (P.dbg && t == P.dbg_step) { long long gt; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(gt)); P.dbg[(size_t)blockIdx.x * DBG_N + 30] = gt; }
                if (P.dbg && t == P.dbg_step + 64) {     // 64 steps later: average cycles and ns per step
                    long long gt; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(gt));
                    P.dbg[(size_t)blockIdx.x * DBG_N + 31] = gt;
                    P.dbg[(size_t)blockIdx.x * DBG_N + 29] = clock64();
                }
            }
            // rows of the NEXT minibatch towards L2 while this one is processed
            if (t + 1 < P.n_mb && et < 64) {
                const long long r = row0 + MB + 64 * a + et;
                prefetch_l2(u.obs + r * D);
                if (D > 32) prefetch_l2(u.obs + r * D + 32);
                if (is_g2) { prefetch_l2(u.obs + (r + 128) * D); if (D > 32) prefetch_l2(u.obs + (r + 128) * D + 32); }
                if (net == 0) { prefetch_l2(u.act + r * A); prefetch_l2(u.logp_old + r); prefetch_l2(u.adv + r); if (C > 1) prefetch_l2(u.adv + u.ld + r); }
                else { prefetch_l2(u.ret + (long long)(net - 1) * u.ld + r); if (u.value_clip) prefetch_l2(u.values + (long long)(net - 1) * u.ld + r); }
            }
            // ---- S(a): publish the images of the owned W2 tile (from tensor memory) ------------------
            float* scratch = reinterpret_cast<float*>(ring);       // the operand ring is idle outside the GEMM phases
            if (!is_g2) {
                float pv[C2], phi[C2], plo[C2];
                tmem_ldn<C2>(tm_lane + TM_P + C2 * wq, pv);
                const int o = 64 * q4 + trow;                   // output unit of this lane
                float* w2a_hi = wsn + (size_t)I_W2A_HI * IMG + (size_t)(o >> 5) * 8192 + (size_t)(o & 31) * 4;
                float* w2a_lo = w2a_hi + IMG;
#pragma unroll
                for (int q = 0; q < C2 / 4; ++q) {              // k = 64 ka + cb2 + 4 q + (0..3)
                    float4 hi, lo;
                    tf32_split(pv[4 * q], hi.x, lo.x); tf32_split(pv[4 * q + 1], hi.y, lo.y);
                    tf32_split(pv[4 * q + 2], hi.z, lo.z); tf32_split(pv[4 * q + 3], hi.w, lo.w);
                    const size_t plane = (size_t)(16 * ka + (cb2 >> 2) + q) * 128;
                    *reinterpret_cast<float4*>(w2a_hi + plane) = hi;
                    *reinterpret_cast<float4*>(w2a_lo + plane) = lo;
                    phi[4 * q] = hi.x; phi[4 * q + 1] = hi.y; phi[4 * q + 2] = hi.z; phi[4 * q + 3] = hi.w;
                    plo[4 * q] = lo.x; plo[4 * q + 1] = lo.y; plo[4 * q + 2] = lo.z; plo[4 * q + 3] = lo.w;
                }
                // W2B (MN = k, K = o): "rows" are the output units o, "columns" the 64 k of block ka
                store_transposed<C2, 64>(scratch, phi, plo, trow, cb2, et, wsn + (size_t)I_W2B_HI * IMG + (size_t)ka * 16384, 64 * q4, 0);
            }
            // ---- S(b): h1 tiles [64 rows][32 columns of block b].  The CTAs that own a W2 tile are busy with its Adam
            // step and images, so the other half of the grid (CTAs 0-15: a in {0, 1}) computes the tiles of row
            // blocks a and a + 2 -- same column block, hence the same W1 slice.
            if (is_g2) {
                const int r = et & 63, kc = C1 * (et >> 6);  // row, first of C1 columns
                // both row blocks' observation rows are in flight before anything is stored
                const float* x0 = u.obs + (row0 + 64 * a + r) * D;
                const float* x1 = u.obs + (row0 + 64 * (a + 2) + r) * D;
                float acc2[2][C1];
#pragma unroll
                for (int j = 0; j < C1; ++j) acc2[0][j] = acc2[1][j] = sp_p[sm.w1 + D * 32 + kc + j];      // b1
                for (int d = 0; d < D; ++d) {
                    const float xv0 = __ldg(x0 + d), xv1 = __ldg(x1 + d);
                    const float* w = sp_p + sm.w1 + d * 32 + kc;
#pragma unroll
                    for (int j = 0; j < C1; ++j) { acc2[0][j] = fmaf(xv0, w[j], acc2[0][j]); acc2[1][j] = fmaf(xv1, w[j], acc2[1][j]); }
                }
                constexpr int TSCR = 2 * 32 * 65;                  // staging floats of one [64 x 32] tile (hi + lo)
#pragma unroll
                for (int rep = 0; rep < 2; ++rep) {
                    const int aa = a + 2 * rep;
                    float hi[C1], lo[C1];
                    float* a_hi = wsn + (size_t)I_H1A_HI * IMG + (size_t)aa * 16384 + (size_t)r * 4;
#pragma unroll
                    for (int q = 0; q < C1 / 4; ++q) {
#pragma unroll
                        for (int e = 0; e < 4; ++e) tf32_split(fmaxf(acc2[rep][4 * q + e], 0.f), hi[4 * q + e], lo[4 * q + e]);
                        const size_t plane = (size_t)(8 * b + (kc >> 2) + q) * 256;
                        *reinterpret_cast<float4*>(a_hi + plane) = make_float4(hi[4 * q], hi[4 * q + 1], hi[4 * q + 2], hi[4 * q + 3]);
                        *reinterpret_cast<float4*>(a_hi + IMG + plane) = make_float4(lo[4 * q], lo[4 * q + 1], lo[4 * q + 2], lo[4 * q + 3]);
                    }
                    transposed_stage<C1, 32>(scratch + rep * TSCR, hi, lo, r, kc);
                }
                epi_bar();
                // H1T (MN = k, K = r): block b / 2, columns 32 (b & 1) .. -- both tiles behind ONE pair of barriers
#pragma unroll
                for (int rep = 0; rep < 2; ++rep)
                    transposed_flush<32>(scratch + rep * TSCR, et, wsn + (size_t)I_H1T_HI * IMG + (size_t)(b >> 1) * 16384, 64 * (a + 2 * rep), 32 * (b & 1));
            }
            epi_bar();
            if (et == 0) { STAMP(1); flag_add_release(fl_net + F_A * FLAG_LINE); }

            // per-row loss inputs (independent of the GEMM): issued now, consumed after the head
            const long long grow = row0 + 64 * a + trow;
            float p_act[8], p_lpo = 0.f, p_adv0 = 0.f, p_adv1 = 0.f, p_ret = 0.f, p_val = 0.f, mean0 = 0.f, rstd0 = 1.f, mean1 = 0.f, rstd1 = 1.f;
#pragma unroll
            for (int j = 0; j < 8; ++j) p_act[j] = 0.f;
            if (net == 0) {
#pragma unroll
                for (int j = 0; j < 8; ++j) if (j < A) p_act[j] = __ldg(u.act + grow * A + j);
                p_lpo = __ldg(u.logp_old + grow);
                p_adv0 = __ldg(u.adv + grow);
                if (C > 1) p_adv1 = __ldg(u.adv + u.ld + grow);
                const float* ms = u.mb_stats + (size_t)t * 4;
                mean0 = __ldg(ms); rstd0 = __ldg(ms + 1); mean1 = __ldg(ms + 2); rstd1 = __ldg(ms + 3);
            } else {
                p_ret = __ldg(u.ret + (long long)(net - 1) * u.ld + grow);
                if (u.value_clip) p_val = __ldg(u.values + (long long)(net - 1) * u.ld + grow);
            }
            // the Gaussian's scale does not depend on the head: sigma and 1 / sigma before the GEMM wait (the actor's loss
            // phase is the longest of the three networks and every network waits for it at the global-norm hop)
            float p_ls[8], p_rsg[8];
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                p_ls[j] = (net == 0 && j < A) ? sp_p[sm.b3 + 8 + j] : 0.f;
                p_rsg[j] = 1.0f / expf(p_ls[j]);
            }

            // ---- G1 epilogue: h2 = relu(acc + b2), head partial over this tile's 32 columns -------------
            if (!mbar_wait(&bar_acc, acc_phase & 1, WAIT_CYCLES)) fail(P.err, 30);
            __syncwarp();      // every thread polled on its own: reconverge before the .sync.aligned tensor-memory loads
            ++acc_phase;
            tc_fence_after();
            if (et == 0) STAMP(2);
            float h2[C1];
            acc_ld_split<C1>(tm_lane, lane, C1 * wq, 16 + C1 * wq, h2);
            float hp[OUTP];
#pragma unroll
            for (int j = 0; j < OUTP; ++j) hp[j] = 0.f;
#pragma unroll
            for (int j = 0; j < C1; ++j) {
                h2[j] = fmaxf(h2[j] + sp_p[sm.b2 + cb1 + j], 0.f);
                const float* w = sp_p + sm.w3 + (cb1 + j) * OUTP;
#pragma unroll
                for (int jj = 0; jj < OUTP; ++jj) hp[jj] = fmaf(h2[j], w[jj], hp[jj]);
            }
#pragma unroll
            for (int jj = 0; jj < OUTP; ++jj) hp[jj] += __shfl_xor_sync(0xffffffffu, hp[jj], 16);
            if (WQ > 1) {                                       // the WQ warps of a subpartition hold different columns of the same rows
                float* xh = &s_red[0][0];
                if (half == 0 && wq > 0) {
#pragma unroll
                    for (int jj = 0; jj < OUTP; ++jj) xh[((wq - 1) * 64 + trow) * OUTP + jj] = hp[jj];
                }
                epi_bar();
                if (half == 0 && wq == 0) {
#pragma unroll
                    for (int w2 = 1; w2 < WQ; ++w2)
#pragma unroll
                        for (int jj = 0; jj < OUTP; ++jj) hp[jj] += xh[((w2 - 1) * 64 + trow) * OUTP + jj];
                }
            }
            float outv[OUTP];
#pragma unroll
            for (int jj = 0; jj < OUTP; ++jj) outv[jj] = sp_p[sm.b3 + jj];
            if (P.cluster) {
                // hop B inside the cluster (8 CTAs = the column blocks of this row block): push the partial rows into every
                // peer's landing zone, one remote mbarrier arrival per peer, then wait for the 8 arrivals on the own barrier
                if (et == 0) {
                    STAMP(3);
                    mbar_expect_tx(&bar_b, 8u * 64u * OUTP * (uint32_t)sizeof(float));
                }
                if (half == 0 && wq == 0) {
                    const uint32_t mine = smem_u32(land + ((size_t)b * 64 + trow) * OUTP);
                    const uint32_t bb_ = smem_u32(&bar_b);
#pragma unroll
                    for (int r = 0; r < 8; ++r) {
                        const uint32_t ra = mapa_u32(mine, r), rb = mapa_u32(bb_, r);
                        st_async4(ra, make_float4(hp[0], hp[1], hp[2], hp[3]), rb);
                        st_async4(ra + 16, make_float4(hp[4], hp[5], hp[6], hp[7]), rb);
                    }
                }
                if (!mbar_wait_cluster(&bar_b, t & 1, WAIT_CYCLES)) fail(P.err, 31);
                __syncwarp();
                if (et == 0) STAMP(4);
#pragma unroll
                for (int bb = 0; bb < 8; ++bb) {
                    const float* src = land + ((size_t)bb * 64 + trow) * OUTP;
                    const float4 v0 = *reinterpret_cast<const float4*>(src);
                    const float4 v1 = *reinterpret_cast<const float4*>(src + 4);
                    outv[0] += v0.x; outv[1] += v0.y; outv[2] += v0.z; outv[3] += v0.w;
                    outv[4] += v1.x; outv[5] += v1.y; outv[6] += v1.z; outv[7] += v1.w;
                }
            } else {
                if (half == 0 && wq == 0) {
                    float* dst = wsn + HEADP_OFF + ((size_t)(a * 8 + b) * 64 + trow) * OUTP;
                    *reinterpret_cast<float4*>(dst) = make_float4(hp[0], hp[1], hp[2], hp[3]);
                    *reinterpret_cast<float4*>(dst + 4) = make_float4(hp[4], hp[5], hp[6], hp[7]);
                }
                tc_fence_before();
                epi_bar();
                if (et == 0) {
                    STAMP(3);
                    flag_add_release(fl_net + (F_B + a) * FLAG_LINE);
                    if (!flag_wait_ge(fl_net + (F_B + a) * FLAG_LINE, 8u * (t + 1), WAIT_CYCLES)) fail(P.err, 31);
                    STAMP(4);
                }
                epi_bar();
#pragma unroll
                for (int bb = 0; bb < 8; ++bb) {
                    const float* src = wsn + HEADP_OFF + ((size_t)(a * 8 + bb) * 64 + trow) * OUTP;
                    const float4 v0 = __ldcg(reinterpret_cast<const float4*>(src));
                    const float4 v1 = __ldcg(reinterpret_cast<const float4*>(src + 4));
                    outv[0] += v0.x; outv[1] += v0.y; outv[2] += v0.z; outv[3] += v0.w;
                    outv[4] += v1.x; outv[5] += v1.y; outv[6] += v1.z; outv[7] += v1.w;
                }
            }
            // ---- loss gradient at the head (ppo_lag.py:152-212): dd[j] = d loss / d head_j --------------
            float dd[16];
#pragma unroll
            for (int j = 0; j < 16; ++j) dd[j] = 0.f;
            float st_a = 0.f, st_b = 0.f, st_c = 0.f, st_d = 0.f;
            {
                const float invB = 1.0f / (float)MB;
                if (net == 0) {
                    float logp = 0.f, zz[8], dmu[8];
#pragma unroll
                    for (int j = 0; j < 8; ++j) {
                        zz[j] = dmu[j] = 0.f;
                        if (j < A) {
                            const float tnh = tanhf(outv[j]);
                            const float mu = u.bounded ? u.max_action * tnh : outv[j];
                            dmu[j] = u.bounded ? u.max_action * (1.0f - tnh * tnh) : 1.0f;
                            zz[j] = (p_act[j] - mu) * p_rsg[j];
                            logp += -0.5f * zz[j] * zz[j] - p_ls[j] - LOG_SQRT_2PI;
                        }
                    }
                    const float ratio = expf(logp - p_lpo);
                    const float ar = (p_adv0 - mean0) * rstd0;
                    const float surr1 = ratio * ar;
                    const float rc = fminf(fmaxf(ratio, 1.0f - u.eps_clip), 1.0f + u.eps_clip);
                    const float surr2 = rc * ar;
                    const bool inside = (ratio >= 1.0f - u.eps_clip) && (ratio <= 1.0f + u.eps_clip);
                    float g_ratio, lrew;
                    if (surr1 < surr2) { g_ratio = -ar; lrew = -surr1; }
                    else if (surr1 > surr2) { g_ratio = inside ? -ar : 0.f; lrew = -surr2; }
                    else { g_ratio = inside ? -ar : -0.5f * ar; lrew = -surr1; }
                    if (u.dual_clip > 0.f && ar < 0.f) {
                        const float c1 = fminf(surr1, surr2), c2 = u.dual_clip * ar;
                        if (c2 > c1) { g_ratio = 0.f; lrew = -c2; }
                        else if (c2 == c1) { g_ratio *= 0.5f; }
                    }
                    float g_saf = 0.f, lsaf = 0.f;
                    if (u.use_lagrangian && C > 1) {
                        const float ac = (p_adv1 - mean1) * rstd1;
                        g_saf = ac * u.lagrangian;
                        lsaf = ratio * ac * u.lagrangian;
                    }
                    const float gl = u.rescaling * (g_ratio + g_saf) * ratio * invB;
#pragma unroll
                    for (int j = 0; j < 8; ++j) {
                        if (j < A) {
                            dd[j] = gl * (zz[j] * p_rsg[j]) * dmu[j];
                            dd[8 + j] = gl * (zz[j] * zz[j] - 1.0f);
                        }
                    }
                    st_a = lrew * invB; st_b = lsaf * invB; st_c = (p_lpo - logp) * invB;
                } else {
                    const float v = outv[0], ret = p_ret;
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
            if (et == 0) STAMP(26);
            // ---- dz2 tile = (dOut W3^T) * relu'(h2): images DZA / DZT; partial db2, dW3, db3 ----------------
            const int nfeed = (net == 0) ? A : 1;              // head columns that feed W3 (mu only)
            float dz[C1];
#pragma unroll
            for (int j = 0; j < C1; ++j) {
                const float* w = sp_p + sm.w3 + (cb1 + j) * OUTP;
                float g = 0.f;
#pragma unroll
                for (int jj = 0; jj < OUTP; ++jj) if (jj < nfeed) g = fmaf(dd[jj], w[jj], g);
                dz[j] = h2[j] > 0.f ? g : 0.f;
            }
            {
                float hi[C1], lo[C1];
                float* a_hi = wsn + (size_t)I_DZA_HI * IMG + (size_t)a * 16384 + (size_t)trow * 4;
#pragma unroll
                for (int q = 0; q < C1 / 4; ++q) {
#pragma unroll
                    for (int e = 0; e < 4; ++e) tf32_split(dz[4 * q + e], hi[4 * q + e], lo[4 * q + e]);
                    const size_t plane = (size_t)(8 * b + (cb1 >> 2) + q) * 256;
                    *reinterpret_cast<float4*>(a_hi + plane) = make_float4(hi[4 * q], hi[4 * q + 1], hi[4 * q + 2], hi[4 * q + 3]);
                    *reinterpret_cast<float4*>(a_hi + IMG + plane) = make_float4(lo[4 * q], lo[4 * q + 1], lo[4 * q + 2], lo[4 * q + 3]);
                }
                // DZT (MN = o, K = r): block b / 2, columns 32 (b & 1) ..
                store_transposed<C1, 32>(scratch, hi, lo, trow, cb1, et, wsn + (size_t)I_DZT_HI * IMG + (size_t)(b >> 1) * 16384, 64 * a, 32 * (b & 1));
            }
            if (et == 0) STAMP(27);
            // partial sums over this tile's 64 rows: half-warp butterflies (16 rows of a subpartition), one shared
            // memory exchange, then 4-way sums.  s_red row: [0,32) db2 | [32,32+32 nfeed) dW3 | [288,304) db3, dlog sigma | [304,308) loss sums
            {
                float* row = &s_red[sp][0];
#pragma unroll
                for (int j = 0; j < C1; ++j) {
                    const float sdz = half_sum(dz[j]);
                    if (r16 == 0) row[cb1 + j] = sdz;
                }
#pragma unroll
                for (int jj = 0; jj < OUTP; ++jj) {
                    if (jj < nfeed) {
#pragma unroll
                        for (int j = 0; j < C1; ++j) {
                            const float sv = half_sum(h2[j] * dd[jj]);
                            if (r16 == 0) row[32 + 32 * jj + cb1 + j] = sv;
                        }
                    }
                }
                if (b == 0 && wq == 0) {                            // per-row quantities: one warp of each subpartition
#pragma unroll
                    for (int j = 0; j < 16; ++j) {
                        const float sv = half_sum(dd[j]);
                        if (lane == 0) row[288 + j] = sv;
                    }
                    const float sa = half_sum(st_a), sb = half_sum(st_b), sc = half_sum(st_c), sdv = half_sum(st_d);
                    if (lane == 0) { row[304] = sa; row[305] = sb; row[306] = sc; row[307] = sdv; }
                }
            }
            epi_bar();
            if (et == 0) STAMP(28);
            for (int i = et; i < 32 + 32 * nfeed; i += NEPI) {
                const float tot = ((s_red[0][i] + s_red[1][i]) + s_red[2][i]) + s_red[3][i];
                if (i < 32) wsn[DB2P_OFF + a * H + 32 * b + i] = tot;
                else wsn[DW3P_OFF + ((size_t)a * H + 32 * b + ((i - 32) & 31)) * OUTP + ((i - 32) >> 5)] = tot;
            }
            if (b == 0) {                                       // db3 | d log sigma partial, loss statistics
                if (et < 20) {
                    const int i = 288 + et;
                    const float tot = ((s_red[0][i] + s_red[1][i]) + s_red[2][i]) + s_red[3][i];
                    if (et < 16) wsn[DB3P_OFF + a * 16 + et] = tot;
                    else if (stat_base) {
                        float* stat = stat_base + (size_t)slot * FSRL_PPO_STATS;
                        if (net == 0) { if (et == 16) atomicAdd(stat + ST_ACTOR_REW, tot); if (et == 17) atomicAdd(stat + ST_ACTOR_SAFETY, tot); if (et == 18) atomicAdd(stat + ST_KL, tot); }
                        else if (et == 19) atomicAdd(stat + ST_VF0 + (net - 1), tot);
                    }
                }
                if (net == 0 && a == 0 && et == 20 && stat_base) {
                    float ent = 0.f;
                    for (int jq = 0; jq < A; ++jq) ent += 0.5f + LOG_SQRT_2PI + sp_p[sm.b3 + 8 + jq];
                    stat_base[(size_t)slot * FSRL_PPO_STATS + ST_ENTROPY] = ent;
                }
            }
            epi_bar();
            if (et == 0) { STAMP(5); flag_add_release(fl_net + F_C * FLAG_LINE); }

            // ---- G2 / G3 epilogue ---------------------------------------------------------------------------
            // G2: what does not depend on the accumulators is requested BEFORE waiting for them -- the ReLU mask of
            // this lane's h1 entries (image H1A, complete since flag A) and this thread's share of the 64 x D
            // observation block of row block q4
            float mreg[C2];
            float xr[(64 * MAXD + NEPI - 1) / NEPI];
            const int nx = (64 * D + NEPI - 1) / NEPI;
            if (is_g2) {
                const int k = 64 * ka + trow;
                const float* msk = wsn + (size_t)I_H1A_HI * IMG + (size_t)q4 * 16384 + (size_t)(k >> 2) * 256 + (k & 3);
#pragma unroll
                for (int jq = 0; jq < C2; ++jq) mreg[jq] = __ldcg(msk + (size_t)(cb2 + jq) * 4);
                const float* xb = u.obs + (row0 + 64 * q4) * D;
#pragma unroll
                for (int q = 0; q < (64 * MAXD + NEPI - 1) / NEPI; ++q)
                    xr[q] = (q < nx && et + q * NEPI < 64 * D) ? __ldg(xb + et + q * NEPI) : 0.f;
                // cluster launches: the hop-B landing zone is idle until the next step -- the observation block is staged
                // there NOW, while the GEMM still runs (row r at r * D + (r >> 5): the two half-warps read different banks)
                if (P.cluster) {
#pragma unroll
                    for (int q = 0; q < (64 * MAXD + NEPI - 1) / NEPI; ++q) {
                        const int e = et + q * NEPI;
                        if (q < nx && e < 64 * D) { const int r = e / D; land[e + (r >> 5)] = xr[q]; }
                    }
                }
            }
            if (!mbar_wait(&bar_acc, acc_phase & 1, WAIT_CYCLES)) fail(P.err, 32);
            __syncwarp();      // every thread polled on its own: reconverge before the .sync.aligned tensor-memory loads
            ++acc_phase;
            tc_fence_after();
            if (et == 0) STAMP(6);
            float sq = 0.f;
            if (is_g2) {
                // without clusters the observation block goes to slot 0 of the operand ring, idle from here until the
                // next step's flag A
                float* xs = P.cluster ? land : reinterpret_cast<float*>(ring);
                if (!P.cluster) {
#pragma unroll
                    for (int q = 0; q < (64 * MAXD + NEPI - 1) / NEPI; ++q) {
                        const int e = et + q * NEPI;
                        if (q < nx && e < 64 * D) { const int r = e / D; xs[e + (r >> 5)] = xr[q]; }
                    }
                }
                // lane: k = 64 ka + trow ; rows cb2 + j of row block q4; partial set 2 q4 + wq (WQ sets per row block)
                float v[C2];
                acc_ld_split<C2>(tm_lane, lane, C2 * wq, 32 + C2 * wq, v);
                const int k = 64 * ka + trow;
#pragma unroll
                for (int jq = 0; jq < C2; ++jq) v[jq] = (mreg[jq] > 0.f) ? v[jq] : 0.f;
                epi_bar();
                if (et == 0) STAMP(22);
                const float* xh = xs + (size_t)cb2 * D + half;
                float* dst = wsn + DW1P_OFF + (size_t)(WQ * q4 + wq) * (MAXD + 1) * H + k;
                for (int d = 0; d < D; ++d) {
                    float sacc = 0.f;
#pragma unroll
                    for (int jq = 0; jq < C2; ++jq) sacc = fmaf(xh[jq * D + d], v[jq], sacc);
                    sacc += __shfl_xor_sync(0xffffffffu, sacc, 16);
                    if (half == 0) dst[(size_t)d * H] = sacc;
                }
                float sb1 = 0.f;
#pragma unroll
                for (int jq = 0; jq < C2; ++jq) sb1 += v[jq];
                sb1 += __shfl_xor_sync(0xffffffffu, sb1, 16);
                if (half == 0) dst[(size_t)D * H] = sb1;          // db1
                if (et == 0) STAMP(23);
                tc_fence_before();
                epi_bar();
                if (et == 0) flag_add_release(fl_net + F_D1 * FLAG_LINE);
            } else {
                float g[C2];
                acc_ld_split<C2>(tm_lane, lane, C2 * wq, 32 + C2 * wq, g);
                if (DP && world > 1) {
                    dp_tile_send(dp_ctx(t), (size_t)(net * 16 + (c - 16)) * TILE_FLOATS + (size_t)et * 4, tm_lane, lane, wq, et);
                    if (et == 0) STAMP(32);
                } else {
#pragma unroll
                    for (int jq = 0; jq < C2; ++jq) sq = fmaf(g[jq], g[jq], sq);
                }
            }
            // ---- small-parameter gradients: fixed-order sums of the row-block partials.  The b2 / W3 / b3 partials
            // are complete since flag C: they are summed while flag D1 (the dW1 partials) is still on its way.
            auto reduce_slices = [&](int lo, int hi) {
                for (int i0 = lo + et; i0 < hi; i0 += 4 * NEPI) {    // 4 elements x 4 partials in flight per thread
                    float pv[4][4 * WQ];
                    bool real[4];
                    int np[4];
#pragma unroll
                    for (int e = 0; e < 4; ++e) {
                        const int i = i0 + e * NEPI;
                        const float* src = wsn;
                        size_t stride = 0;
                        real[e] = false;
                        np[e] = 4;
                        if (i < hi) {
                            if (i < sm.b2) { src = wsn + DW1P_OFF + (size_t)(i / 32) * H + 32 * b + (i % 32); stride = (size_t)(MAXD + 1) * H; real[e] = true; np[e] = 4 * WQ; }
                            else if (i < sm.w3) { src = wsn + DB2P_OFF + 32 * b + (i - sm.b2); stride = H; real[e] = true; }
                            else if (i < sm.b3) {
                                const int oo = (i - sm.w3) / OUTP, jj = (i - sm.w3) % OUTP;
                                real[e] = jj < out;
                                src = wsn + DW3P_OFF + ((size_t)32 * b + oo) * OUTP + jj; stride = (size_t)H * OUTP;
                            } else {
                                const int jj = i - sm.b3;
                                real[e] = (jj < out) || (net == 0 && u.head_indep && jj >= 8 && jj < 8 + A);
                                src = wsn + DB3P_OFF + jj; stride = 16;
                            }
                        }
#pragma unroll
                        for (int q = 0; q < 4 * WQ; ++q) pv[e][q] = (real[e] && q < np[e]) ? __ldcg(src + q * stride) : 0.f;
                    }
#pragma unroll
                    for (int e = 0; e < 4; ++e) {
                        const int i = i0 + e * NEPI;
                        if (i < hi) {
                            float gsum = 0.f;
#pragma unroll
                            for (int q = 0; q < 4 * WQ; ++q) gsum += pv[e][q];          // fixed order
                            sp_g[i] = gsum;
                        }
                    }
                }
            };
            reduce_slices(sm.b2, sm.n);
            if (et == 0) { STAMP(7); if (!flag_wait_ge(fl_net + F_D1 * FLAG_LINE, 16u * (t + 1), WAIT_CYCLES)) fail(P.err, 33); STAMP(8); }
            epi_bar();
            reduce_slices(0, sm.b2);
            if (DP && world > 1) {
                const DpCtx d = dp_ctx(t);
                const size_t off_t = (size_t)(net * 16 + (c - 16)) * TILE_FLOATS + (size_t)et * 4;
                epi_bar();                                    // sp_g complete
                if (!is_g2 && !d.direct) { dp_tile_reduce(d, off_t, tm_lane, lane, wq, et); if (et == 0) STAMP(33); }
                dp_slices(d, (size_t)u.n_nets * 16 * TILE_FLOATS + (size_t)(net * 8 + b) * SLICE_PK * 4, sp_g, sm.n, et, a == 0);
                __syncwarp();
                if (et == 0) STAMP(38);
                if (!is_g2) { sq += dp_tile_finish(d, off_t, tm_lane, lane, wq, et); if (et == 0) STAMP(41); }
                epi_bar();                                    // sp_g holds the global mean before the norm / Adam read it
            }
            // every small parameter is counted once in the norm: W1/b1/b2/W3 slices by row block 0, b3 / log sigma by CTA 0.
            // (each thread re-reads only elements it wrote itself: same i = et + k NEPI mapping)
            if (a == 0) {
                for (int i = et; i < sm.n; i += NEPI) {
                    bool real = true;
                    if (i >= sm.w3 && i < sm.b3) real = ((i - sm.w3) % OUTP) < out;
                    else if (i >= sm.b3) { const int jj = i - sm.b3; real = (jj < out) || (net == 0 && u.head_indep && jj >= 8 && jj < 8 + A); }
                    if (real && (i < sm.b3 || b == 0)) sq = fmaf(sp_g[i], sp_g[i], sq);
                }
            }
            // ---- global gradient norm: per-CTA partial -> device-wide hop -> same summation order everywhere --
            sq = warp_sum(sq);
            if (lane == 0) s_misc[warp - 2] = sq;
            epi_bar();
            if (et == 0) {
                float tot = 0.f;
#pragma unroll
                for (int w2 = 0; w2 < NEPI / 32; ++w2) tot += s_misc[w2];
                sumsq_g[blockIdx.x] = tot;
                STAMP(9);
                flag_add_release(fl_d2);
                if (!flag_wait_ge(fl_d2, (unsigned)n_cta * (t + 1), WAIT_CYCLES)) fail(P.err, 34);
                STAMP(10);
            }
            epi_bar();
            float nq[4];
#pragma unroll
            for (int q = 0; q < 4; ++q) nq[q] = (lane + 32 * q < n_cta) ? __ldcg(sumsq_g + lane + 32 * q) : 0.f;
            float nsq = ((nq[0] + nq[1]) + nq[2]) + nq[3];                          // identical order in every warp of the grid
            nsq = warp_sum(nsq);
            float gscale = 1.0f;
            if (u.max_grad_norm > 0.f) gscale = fminf(u.max_grad_norm / (sqrtf(nsq) + 1e-6f), 1.0f);
            if (blockIdx.x == 0 && et == 0 && stat_base) stat_base[(size_t)slot * FSRL_PPO_STATS + ST_GRADNORM] = sqrtf(nsq);
            const AdamS ad = s_adam;
            if (et == 0) STAMP(24);
            // ---- clip + Adam: replicated small slices, then the owned W2 tile (tensor memory) --------------------
            for (int i = et; i < sm.n; i += NEPI) {
                float m = sp_m[i], v = sp_v[i];
                sp_p[i] = adam_one_approx(sp_p[i], sp_g[i] * gscale, m, v, ad);
                sp_m[i] = m; sp_v[i] = v;
            }
            if (et == 0) STAMP(25);
            if (!is_g2) {
                float g[C2], pv[C2], mv[C2], vv[C2];
                if (DP && world > 1) tmem_ldn<C2>(tm_lane + TM_G + C2 * wq, g);
                else acc_ld_split<C2>(tm_lane, lane, C2 * wq, 32 + C2 * wq, g);
                tmem_ldn<C2>(tm_lane + TM_P + C2 * wq, pv); tmem_ldn<C2>(tm_lane + TM_M + C2 * wq, mv); tmem_ldn<C2>(tm_lane + TM_V + C2 * wq, vv);
#pragma unroll
                for (int j = 0; j < C2; ++j) pv[j] = adam_one_approx(pv[j], g[j] * gscale, mv[j], vv[j], ad);
                tmem_stn<C2>(tm_lane + TM_P + C2 * wq, pv); tmem_stn<C2>(tm_lane + TM_M + C2 * wq, mv); tmem_stn<C2>(tm_lane + TM_V + C2 * wq, vv);
            }
            tc_fence_before();
            epi_bar();     // slices final before the next h1 tile / head reads them; s_adam may be rewritten
            if (et == 0) STAMP(11);
        }

        // ---- write the parameters and Adam moments back to the arena ------------------------------------------
        if (a == 0) {
            for (int i = et; i < sm.n; i += NEPI) {
                long long dst = -1;
                if (i < sm.b2) { const int d = i / 32, kk = i % 32; dst = (d < D) ? o_w1 + (long long)d * H + 32 * b + kk : o_b1 + 32 * b + kk; }
                else if (i < sm.w3) dst = o_b2 + 32 * b + (i - sm.b2);
                else if (i < sm.b3) { const int oo = (i - sm.w3) / OUTP, jj = (i - sm.w3) % OUTP; if (jj < out) dst = o_w3 + (long long)(32 * b + oo) * out + jj; }
                else if (b == 0) { const int jj = i - sm.b3; if (jj < out) dst = o_b3 + jj; else if (net == 0 && u.head_indep && jj >= 8 && jj < 8 + A) dst = o_ls + (jj - 8); }
                if (dst >= 0) { u.theta[dst] = sp_p[i]; u.adam_m[dst] = sp_m[i]; u.adam_v[dst] = sp_v[i]; }
            }
        }
        if (!is_g2) {
            float pv[C2], mv[C2], vv[C2];
            tmem_ldn<C2>(tm_lane + TM_P + C2 * wq, pv); tmem_ldn<C2>(tm_lane + TM_M + C2 * wq, mv); tmem_ldn<C2>(tm_lane + TM_V + C2 * wq, vv);
            const int o = 64 * q4 + trow;
#pragma unroll
            for (int j = 0; j < C2; ++j) {
                const long long idx = o_w2 + (long long)(64 * ka + cb2 + j) * H + o;
                u.theta[idx] = pv[j]; u.adam_m[idx] = mv[j]; u.adam_v[idx] = vv[j];
            }
        }
        tc_fence_before();
    }
    __syncthreads();
    if (P.cluster) cluster_sync_all();
    if (warp == 1) { tc_fence_after(); tmem_dealloc<TM_COLS>(tmem); }
}

static size_t smem_bytes(int D, bool cluster = false) {
    return (size_t)NSLOT * SLOT_BYTES + 4 * sizeof(float) * SliceMap(D).n + (cluster ? sizeof(float) * 8 * 64 * OUTP : 0);
}

}  // namespace pp

size_t ppo_persist_ws_floats(int n_nets, int D, int H) {
    (void)D; (void)H;
    return (size_t)n_nets * pp::NET_WS + pp::SUMSQ_FLOATS + (size_t)(n_nets * pp::F_PER_NET + 1) * pp::FLAG_LINE + 32 +
           2 * (size_t)pp::MAX_MB + 2 * (size_t)32 * n_nets * pp::DBG_N;
}

size_t ppo_persist_p2p_floats(int n_nets) { return (size_t)(FSRL_P2P_MAX_RANKS + 1) * n_nets * pp::XG_PER_NET + pp::XG_FLAG_FLOATS + 64; }

bool ppo_persist_supported(const fsrl_ppo_update_t& u, long long n_total, int batch_size) {
    if (u.H != 256 || batch_size != pp::MB || n_total % pp::MB != 0 || n_total < pp::MB || n_total / pp::MB > pp::MAX_MB) return false;
    if (u.mask != nullptr || u.gather == nullptr) return false;
    if (u.world > 1 && !(u.p2p_on && u.world <= FSRL_P2P_MAX_RANKS && (size_t)u.p2p_stride >= ppo_persist_p2p_floats(u.n_nets))) return false;
    if (u.D < 1 || u.D > pp::MAXD || u.A > 8 || u.n_nets < 1 || u.n_nets > 3) return false;
    if (u.persist_ws == nullptr || (size_t)u.persist_ws_floats < ppo_persist_ws_floats(u.n_nets, u.D, u.H)) return false;
    if (32 * u.n_nets > sm_count()) return false;
    static int smem_optin = -1;
    if (smem_optin < 0) {
        int dev = 0;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&smem_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev);
    }
    return pp::smem_bytes(u.D) + 8192 <= (size_t)smem_optin;
}

// ug: descriptor whose batch pointers are the gathered (contiguous) arrays; mb_stats filled.
int ppo_persist_run(const fsrl_ppo_update_t& ug, int n_mb, int stats_slot0, long long adam_t0, cudaStream_t s) {
    pp::Args a;
    a.u = ug;
    a.n_mb = n_mb; a.slot0 = stats_slot0; a.adam_t0 = adam_t0;
    a.ws = ug.persist_ws;
    const size_t fl_off = (size_t)ug.n_nets * pp::NET_WS + pp::SUMSQ_FLOATS;
    a.flags = reinterpret_cast<unsigned*>(ug.persist_ws + fl_off);
    const size_t n_flag_words = (size_t)(ug.n_nets * pp::F_PER_NET + 1) * pp::FLAG_LINE;
    a.err = reinterpret_cast<int*>(a.flags + n_flag_words);
    FSRL_CUDA(cudaMemsetAsync(a.flags, 0, (n_flag_words + 32) * sizeof(unsigned), s));
    // Adam bias corrections of every step, computed like torch.optim.Adam does (python doubles)
    float* tab_dev = reinterpret_cast<float*>(a.err + 32);
    static std::vector<float> tab;
    tab.resize(2 * (size_t)n_mb);
    for (int t = 0; t < n_mb; ++t) {
        const double tt = (double)(adam_t0 + t + 1);
        const double bc1 = 1.0 - pow(ug.beta1, tt), bc2 = 1.0 - pow(ug.beta2, tt);
        tab[2 * t] = (float)(1.0 / sqrt(bc2));
        tab[2 * t + 1] = (float)(-(ug.lr / bc1));
    }
    FSRL_CUDA(cudaMemcpyAsync(tab_dev, tab.data(), tab.size() * sizeof(float), cudaMemcpyHostToDevice, s));
    a.adam_tab = tab_dev;
    // tag of the exchange packets: ranks run their persistent launches in lock step, so the count agrees everywhere
    static unsigned dp_seq = 0;
    if (ug.world > 1) dp_seq = (dp_seq % 65535u) + 1u;
    a.dp_seq = dp_seq;
    a.dp_direct = ug.world <= 2;
    if (const char* e = getenv("FSRL_PPO_DP_DIRECT")) a.dp_direct = atoi(e) != 0;      // (experiments; must agree on all ranks)
    a.dbg = nullptr; a.dbg_step = -1;
    if (const char* e = getenv("FSRL_PPO_PERSIST_DBG")) {
        a.dbg = reinterpret_cast<long long*>(tab_dev + 2 * (size_t)pp::MAX_MB);
        a.dbg_step = atoi(e);
    }
    // clusters of 8 CTAs (the column blocks of one row block) when the landing zone fits and all clusters can be
    // co-resident; otherwise hop B goes through global memory like the other hops
    static int smem_optin = -1;
    if (smem_optin < 0) {
        int dev = 0;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&smem_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev);
    }
    bool cluster = !getenv("FSRL_PPO_NO_CLUSTER") && pp::smem_bytes(ug.D, true) + 8192 <= (size_t)smem_optin;
    size_t smem = pp::smem_bytes(ug.D, cluster);
    const bool dp = ug.world > 1;
    void (*kern)(const pp::Args) = dp ? pp::ppo_persist_kernel<true> : pp::ppo_persist_kernel<false>;
    static size_t set[2] = {0, 0};
    if (smem > set[dp]) {
        FSRL_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        set[dp] = smem;
    }
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(32 * ug.n_nets); cfg.blockDim = dim3(pp::TPB); cfg.dynamicSmemBytes = smem; cfg.stream = s;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = 8; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
    if (cluster) {
        cfg.attrs = at; cfg.numAttrs = 1;
        int n_clusters = 0;
        if (cudaOccupancyMaxActiveClusters(&n_clusters, kern, &cfg) != cudaSuccess || n_clusters < 4 * ug.n_nets) {
            cudaGetLastError();
            cluster = false;
            smem = pp::smem_bytes(ug.D, false);
            cfg.dynamicSmemBytes = smem;
        }
    }
    if (!cluster) { cfg.attrs = nullptr; cfg.numAttrs = 0; }
    a.cluster = cluster ? 1 : 0;
    FSRL_CUDA(cudaLaunchKernelEx(&cfg, kern, a));
    ++g_launches;
    return FSRL_OK;
}

}  // namespace fsrl

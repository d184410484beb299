// policy_fused.cu — ONE kernel for a whole rollout step of the DHGN actor / critic (DHGN/mappo_parallel.py:116-545 as used by
// MAPPO.run_episode :758-801): message passing + mean aggregation of the three relations, AGG_vertex, semantic layer, FCRA
// blocks, 2-layer GRU cell and the heads (softmax / sample / log-prob, value) for a tile of 128 (env, agent) rows, with every
// activation staying on chip.  HBM traffic per row is only what the step really needs: the env state / packed adjacency in,
// the history embeddings in, the new embedding, hidden states and action / log-prob / value out.
//
// Tensor cores: every 128-wide dense layer is a chain of "units" (one unit = [128 rows x K=128] x [K=128 x n_out]) issued as
// tcgen05.mma.kind::f16 with fp32 accumulation in TMEM.  fp32-level accuracy comes from a two-term fp16 split of BOTH operands,
// a = hi + lo with hi = fp16(a), lo = fp16(a - hi) (22 significant bits; |a - (hi + lo)| <= 2^-23 |a|, or 2^-25 absolute once lo is
// an fp16 subnormal, i.e. |a| < 1/8 - tensor cores take subnormal inputs exactly), and three products per K step
// (A_hi*B_hi + A_lo*B_hi + A_hi*B_lo, the 2^-22 lo*lo term is dropped - the same error budget as 3xTF32, see gemm_tf32x3.cu) at
// twice the TF32 rate and half the operand bytes.  The weights are pre-split and pre-swizzled once per rollout
// (marl_policy_pack) into the exact shared-memory image of each k-block, so that the producer is a single elected thread
// issuing cp.async.bulk copies (32 KB per stage) that complete on an mbarrier.
//
// CTA = one (row tile, network) work item, WW + 2 warps (WW = 16 worker warps, or 8 for 16-agent envs - see Lay<WW>):
//   warps 0..WW-1  workers: SIMT phases (messages, FCRA neighbour mean, hidden-state load) that write the activation tile X
//              straight into the canonical K-major SWIZZLE_128B operand layout (hi and lo planes), and the epilogues
//              (tcgen05.ld -> bias / ReLU / GRU cell / heads -> X again, plus the few global stores).  These phases are
//              latency-bound (dependent FMA / MUFU chains, shared-memory round trips): 16 warps at 96 registers run them
//              ~1.4x faster than 8 warps at 168;
//   warp WW    weight loader (elected lane): streams the packed units through a 4-stage ring;
//   warp WW+1  MMA issuer (elected lane) + TMEM allocation (all 512 columns: the GRU needs four 128-column accumulators).
// Workers and the issuer follow the same static unit program and hand the tile back and forth with two mbarriers
// (a_ready: one arrival per worker thread, mma_done: tcgen05.commit).
// Shared memory: X 64 KB (2 k-blocks of K = 64 x (hi 16 KB + lo 16 KB)) + 4 x 32 KB weight stages.
#include "common.cuh"
#include <cuda_fp16.h>
#include <stdlib.h>
#include <type_traits>

namespace marl {
namespace pf {

constexpr int ROWS = 128, E = 128, NSTAGE = 4, MAXD = 3, MAX_UNITS = 48, NKB = 2 /* k-blocks of 64 halves per K = 128 */;
constexpr int BAR_A_READY = 2 * NSTAGE, BAR_MMA_DONE = 2 * NSTAGE + 1;
constexpr int TILE = ROWS * 128;          // 16 KB: 128 rows x 128 B (one k-block of 64 halves)
constexpr int XKB = 2 * TILE;             // one k-block of X: hi plane + lo plane
constexpr int X_BYTES = NKB * XKB;        // K = 128
constexpr int WSTAGE = 2 * TILE;          // one k-block of a 128-row weight unit: hi + lo
constexpr int MISC_BYTES = 3072;           // barriers, fp32 state of the tile
constexpr int OXY_CAP = 256;               // boundary cells of one map staged per worker warp (fast message path: O <= 256)
constexpr int OXY_BYTES = 16 * OXY_CAP * 8; // up to 16 worker warps x 256 float2
// shared memory of the one-chain kernel: X | weight ring | barriers + fp32 state | boundary-cell staging
constexpr int RING_OFF = X_BYTES, MISC_OFF = RING_OFF + NSTAGE * WSTAGE, OXY_OFF = MISC_OFF + MISC_BYTES;
constexpr int SMEM_BYTES = OXY_OFF + OXY_BYTES;   // 227 KB
// Worker-warp count WW is a template parameter of the kernel: 16 worker warps (8 rows each in the SIMT phases, 32 columns each in
// the epilogues) when an env fits in 8 rows - the SIMT phases are latency-bound, twice the warps hide twice the latency - and 8
// worker warps (16 rows / 64 columns each) for N = 16, whose env-grouped message path needs a whole env per warp.
template <int WW>
struct Lay {
    static_assert(WW == 8 || WW == 16, "8 or 16 worker warps");
    static constexpr int RPW = ROWS / WW;            // rows per warp in the SIMT phases
    static constexpr int CPT = 128 / (WW / 4);       // accumulator columns per thread in the epilogues
    static constexpr int WORKERS = WW * 32, THREADS = (WW + 2) * 32;
};

struct Unit {
    uint32_t off;        // byte offset of the packed unit
    uint16_t n_out;      // 128 or 16
    uint16_t acc_col;    // TMEM column of the accumulator
    uint8_t accumulate;  // add to what the accumulator holds
    uint8_t last;        // last unit of its group (the workers take over afterwards)
    uint16_t pad;
};

struct NetArgs {
    const unsigned char *packed;
    int n_units;
    Unit u[MAX_UNITS];
    const float *msg_w[3], *msg_b[3];
    const float *b_av, *sem_w, *b_sem;
    int sem_ld;
    const float *b_aggf[MAXD], *b_f[MAXD];
    const float *b_ih[2], *b_hh[2];
    const float *b_comb[2];    // per GRU layer [4][E]: b_ir + b_hr, b_iz + b_hz, b_in, b_hn (pair kernel: 4 bias loads per cell group instead of 6)
    const float *head_b;
    const float *head_w_eff;   // critic: effective [E] row (fp32); actor: unused
    const float *hist[MAXD];   // [B,N,E] history embeddings, k = 0 most recent; null = zeros
    float *emb_out;            // [B,N,E]
    const float *hidden_in;    // [2, R, E] previous hidden state
    float *hidden_out;         // [2, R, E] new hidden state (may alias hidden_in)
    int all_ones;              // critic
};

struct StepArgs {
    int B, N, O, NW, OW, depth, rows_per_tile, n_tiles, A;
    int64_t R;
    const void *p_state, *e_state;   // double, or float in the STATE_F32 instantiations
    const int32_t *oxy, *map_id, *o_count;
    const uint32_t *p_adj;
    const uint8_t *e_adj;
    const uint32_t *o_adj;
    int32_t *action;
    float *logp, *value;
    uint64_t seed;
    const uint64_t *d_seed;   // non-null: the sampling seed is read from this device word when the kernel runs (seed is ignored)
    int t, deterministic, force_action, net_first, net_count;
    int64_t row_offset;   // RNG key offset of row 0 (sub-batch launches)
    long long *dbg;   // optional [grid,16] per-CTA phase cycle counters (profiling aid)
    NetArgs net[2];   // 0 actor, 1 critic
};

// ------------------------------------------------------------------------------------------------ PTX helpers
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar)
{
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity)
{
    uint32_t done;
    do {
        asm volatile(
            "{\n"
            ".reg .pred p;\n"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
            "selp.u32 %0, 1, 0, p;\n"
            "}\n"
            : "=r"(done)
            : "r"(bar), "r"(parity)
            : "memory");
    } while (!done);
}
__device__ __forceinline__ void bulk_g2s(uint32_t dst, const void *src, uint32_t bytes, uint32_t bar)
{
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst), "l"(src),
                 "r"(bytes), "r"(bar)
                 : "memory");
}
// K-major SWIZZLE_128B canonical layout (rows of 128 B, 8-row groups 1024 B apart)
__device__ __forceinline__ uint64_t make_desc(uint32_t smem_addr)
{
    uint64_t d = 0;
    d |= (uint64_t)((smem_addr & 0x3FFFF) >> 4);
    d |= (uint64_t)1 << 16;
    d |= (uint64_t)(1024 >> 4) << 32;
    d |= (uint64_t)1 << 46;
    d |= (uint64_t)2 << 61;
    return d;
}
// kind::f16 instruction descriptor: D = f32 (bit 4), A = B = f16 (format 0), both K-major, N >> 3 at bit 17, M >> 4 at bit 24
__device__ __forceinline__ uint32_t idesc_f16(int n) { return (1u << 4) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(ROWS >> 4) << 24); }
__device__ __forceinline__ void umma_f16(uint32_t tmem_c, uint64_t da, uint64_t db, uint32_t idesc, uint32_t accumulate)
{
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "setp.ne.b32 p, %4, 0;\n"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n"
        "}\n" ::"r"(tmem_c), "l"(da), "l"(db), "r"(idesc), "r"(accumulate)
        : "memory");
}
__device__ __forceinline__ void umma_commit(uint32_t bar)
{
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ bool elect_one()
{
    uint32_t pred;
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "elect.sync _|p, 0xffffffff;\n"
        "selp.u32 %0, 1, 0, p;\n"
        "}\n"
        : "=r"(pred));
    return pred != 0;
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

#define PF_TMEM_LD32(dst, addr)                                                                                         \
    asm volatile(                                                                                                       \
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "                                                                       \
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "                                       \
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"                       \
        : "=r"(dst[0]), "=r"(dst[1]), "=r"(dst[2]), "=r"(dst[3]), "=r"(dst[4]), "=r"(dst[5]), "=r"(dst[6]), "=r"(dst[7]),   \
          "=r"(dst[8]), "=r"(dst[9]), "=r"(dst[10]), "=r"(dst[11]), "=r"(dst[12]), "=r"(dst[13]), "=r"(dst[14]),            \
          "=r"(dst[15]), "=r"(dst[16]), "=r"(dst[17]), "=r"(dst[18]), "=r"(dst[19]), "=r"(dst[20]), "=r"(dst[21]),          \
          "=r"(dst[22]), "=r"(dst[23]), "=r"(dst[24]), "=r"(dst[25]), "=r"(dst[26]), "=r"(dst[27]), "=r"(dst[28]),          \
          "=r"(dst[29]), "=r"(dst[30]), "=r"(dst[31])                                                                      \
        : "r"(addr))
#define PF_TMEM_LD16(dst, addr)                                                                                         \
    asm volatile(                                                                                                       \
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 "                                                                       \
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"                                \
        : "=r"(dst[0]), "=r"(dst[1]), "=r"(dst[2]), "=r"(dst[3]), "=r"(dst[4]), "=r"(dst[5]), "=r"(dst[6]), "=r"(dst[7]),   \
          "=r"(dst[8]), "=r"(dst[9]), "=r"(dst[10]), "=r"(dst[11]), "=r"(dst[12]), "=r"(dst[13]), "=r"(dst[14]),            \
          "=r"(dst[15])                                                                                                    \
        : "r"(addr))
__device__ __forceinline__ void tmem_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// two-term fp16 split of a pair: hi = fp16(a) (saturating: the network's activations are far below 65504), lo = fp16(a - hi);
// hi + lo reproduces a to one fp32 ulp (2^-25 absolute below 1/8), so activations are read back from X at fp32 level.
__device__ __forceinline__ void split_h2(float a, float b, uint32_t &hi, uint32_t &lo)
{
    asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(hi) : "f"(b), "f"(a));          // low half = a, high half = b
    const float2 hf = __half22float2(*reinterpret_cast<const __half2 *>(&hi));
    asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(lo) : "f"(b - hf.y), "f"(a - hf.x));
}
__device__ __forceinline__ float2 join_h2(uint32_t hi, uint32_t lo)
{
    const float2 h = __half22float2(*reinterpret_cast<const __half2 *>(&hi)), l = __half22float2(*reinterpret_cast<const __half2 *>(&lo));
    return make_float2(h.x + l.x, h.y + l.y);
}
// K-major SWIZZLE_128B: a row of a k-block is 128 B = 64 halves; 16-byte chunk index XOR (row & 7)
__device__ __forceinline__ int x_off(int row, int c4) { return (c4 >> 4) * XKB + row * 128 + ((((c4 & 15) >> 1) ^ (row & 7)) << 4) + (c4 & 1) * 8; }
// element group (row, channels 4*c4 .. 4*c4+3) of the activation tile, both planes (8-byte accesses: conflict-free when the 32
// lanes of a warp walk c4 of one row, which is how the SIMT phases use it)
__device__ __forceinline__ void x_store4(unsigned char *X, int row, int c4, float4 v)
{
    uint2 h, l;
    split_h2(v.x, v.y, h.x, l.x);
    split_h2(v.z, v.w, h.y, l.y);
    const int off = x_off(row, c4);
    *reinterpret_cast<uint2 *>(X + off) = h;
    *reinterpret_cast<uint2 *>(X + off + TILE) = l;
}
__device__ __forceinline__ float4 x_load4(const unsigned char *X, int row, int c4)
{
    const int off = x_off(row, c4);
    const uint2 h = *reinterpret_cast<const uint2 *>(X + off), l = *reinterpret_cast<const uint2 *>(X + off + TILE);
    const float2 a = join_h2(h.x, l.x), b = join_h2(h.y, l.y);
    return make_float4(a.x, a.y, b.x, b.y);
}
// channels 8*c8 .. 8*c8+7 of one row (16-byte accesses: conflict-free when the lanes of a warp are 32 consecutive rows, which is
// how the epilogues use it)
__device__ __forceinline__ int x_off8(int row, int c8) { return (c8 >> 3) * XKB + row * 128 + (((c8 & 7) ^ (row & 7)) << 4); }
__device__ __forceinline__ void x_store8(unsigned char *X, int row, int c8, const float (&v)[8])
{
    uint4 h, l;
    split_h2(v[0], v[1], h.x, l.x);
    split_h2(v[2], v[3], h.y, l.y);
    split_h2(v[4], v[5], h.z, l.z);
    split_h2(v[6], v[7], h.w, l.w);
    const int off = x_off8(row, c8);
    *reinterpret_cast<uint4 *>(X + off) = h;
    *reinterpret_cast<uint4 *>(X + off + TILE) = l;
}
__device__ __forceinline__ void x_load8(const unsigned char *X, int row, int c8, float (&v)[8])
{
    const int off = x_off8(row, c8);
    const uint4 h = *reinterpret_cast<const uint4 *>(X + off), l = *reinterpret_cast<const uint4 *>(X + off + TILE);
    const float2 a = join_h2(h.x, l.x), b = join_h2(h.y, l.y), c = join_h2(h.z, l.z), d = join_h2(h.w, l.w);
    v[0] = a.x; v[1] = a.y; v[2] = b.x; v[3] = b.y; v[4] = c.x; v[5] = c.y; v[6] = d.x; v[7] = d.y;
}

struct Ctx {
    const StepArgs *a;
    const NetArgs *na;
    unsigned char *X;
    int64_t row0;        // first global row of the tile
    int warp, lane;
    uint32_t tmem, bar_a_ready, bar_mma_done;
    int group;           // groups completed so far (parity of mma_done)
    float4 *s_p;         // [128] fp32 pursuer state of the tile's rows (converted once)
    float4 *s_e;         // [32] fp32 evader state of the tile's envs (when the tile has <= 32 envs)
    float *s_val;        // [WW/4][128] scratch for the critic value (aliases s_p, which is dead by then)
    float2 *s_oxy;       // [worker warps][OXY_CAP] boundary cells of the env a warp is working on (obstacle relation)
};

__device__ __forceinline__ bool row_info(const Ctx &c, int r, int64_t &gr, int &env, int &i)
{
    gr = c.row0 + r;
    const bool ok = r < c.a->rows_per_tile && gr < c.a->R;
    env = ok ? (int)(gr / c.a->N) : 0;
    i = ok ? (int)(gr - (int64_t)env * c.a->N) : 0;
    return ok;
}
// F32 (MARL_POLICY_STATE_F32): the states are already (float) of the fp64 state - the rollout arena's records - and are read as is
template <bool F32>
__device__ __forceinline__ float4 load_state4(const void *base, int64_t idx)
{
    if constexpr (F32) {
        return reinterpret_cast<const float4 *>(base)[idx];
    } else {
        const double2 *q = reinterpret_cast<const double2 *>(static_cast<const double *>(base) + idx * 4);
        const double2 u = q[0], v = q[1];
        return make_float4((float)u.x, (float)u.y, (float)v.x, (float)v.y);
    }
}
template <bool F32>
__device__ __forceinline__ float4 load_p(const StepArgs *a, int64_t gr) { return load_state4<F32>(a->p_state, gr); }
template <bool F32>
__device__ __forceinline__ float4 load_e(const StepArgs *a, int env) { return load_state4<F32>(a->e_state, env); }
template <bool F32>
__device__ __forceinline__ float4 e_of(const Ctx &c, int r, int env)
{
    return (ROWS / c.a->N <= 32) ? c.s_e[r / c.a->N] : load_e<F32>(c.a, env);
}
__device__ __forceinline__ float dot4w(const float (&w)[4], float a0, float a1, float a2, float a3, float b)
{
    return fmaf(w[3], a3, fmaf(w[2], a2, fmaf(w[1], a1, fmaf(w[0], a0, 0.f)))) + b;
}
template <int WW>
__device__ __forceinline__ void worker_sync() { asm volatile("bar.sync 1, %0;" ::"n"(WW * 32) : "memory"); }

// workers: hand X to the issuer (signal_ready), then wait until the group's MMAs have completed (wait_done).  Work that does not
// touch X or TMEM — global loads of the NEXT phase's operands — goes between the two, so that its latency hides behind the MMAs.
__device__ __forceinline__ void signal_ready(Ctx &c)
{
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    tc_fence_before();
    mbar_arrive(c.bar_a_ready);
}
__device__ __forceinline__ void wait_done(Ctx &c)
{
    mbar_wait(c.bar_mma_done, (uint32_t)(c.group & 1));
    tc_fence_after();
    ++c.group;
}
__device__ __forceinline__ void hand_over(Ctx &c)
{
    signal_ready(c);
    wait_done(c);
}

// per-lane slices (channels 4*lane .. 4*lane+3) of one MSG layer, vector loads
__device__ __forceinline__ void load_msg_weights(const NetArgs *na, int rel, int lane, float (&w)[4][8], float (&b)[4])
{
    const float *W = na->msg_w[rel];
    const float4 bb = __ldg(reinterpret_cast<const float4 *>(na->msg_b[rel]) + lane);
    b[0] = bb.x; b[1] = bb.y; b[2] = bb.z; b[3] = bb.w;
    if (rel == 0) {
        const float4 *Wv = reinterpret_cast<const float4 *>(W) + 8 * lane;
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const float4 lo = __ldg(Wv + 2 * q), hi = __ldg(Wv + 2 * q + 1);
            w[q][0] = lo.x; w[q][1] = lo.y; w[q][2] = lo.z; w[q][3] = lo.w;
            w[q][4] = hi.x; w[q][5] = hi.y; w[q][6] = hi.z; w[q][7] = hi.w;
        }
    } else {
        const float4 *Wv = reinterpret_cast<const float4 *>(W) + 4 * lane;
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const float4 lo = __ldg(Wv + q);
            w[q][0] = lo.x; w[q][1] = lo.y; w[q][2] = lo.z; w[q][3] = lo.w;
            w[q][4] = w[q][5] = w[q][6] = w[q][7] = 0.f;
        }
    }
}

// ---- DHGN.message + mean aggregation, generic per-row path (any N) -> X ----------------------------------------------------
// Same arithmetic as msg_agg_fwd_kernel (policy_kernels.cu).  lane l owns channels 4l..4l+3.
template <int WW, bool F32>
__device__ void phase_msg_generic(const Ctx &c, int rel)
{
    constexpr int RPW = Lay<WW>::RPW;
    const StepArgs *a = c.a;
    const NetArgs *na = c.na;
    const int lane = c.lane, N = a->N;
    float w[4][8], b[4];
    load_msg_weights(na, rel, lane, w, b);
#pragma unroll 1
    for (int rr = 0; rr < RPW; ++rr) {
        const int r = RPW * c.warp + rr;
        int64_t gr;
        int env, i;
        const bool ok = row_info(c, r, gr, env, i);
        float out[4] = {0.f, 0.f, 0.f, 0.f};
        if (ok) {
            const float4 pi = c.s_p[r], ev = e_of<F32>(c, r, env);
            const float dex = pi.x - ev.x, dey = pi.y - ev.y, dez = pi.z - ev.z, dew = pi.w - ev.w;
            if (rel == 0) {
                int cnt = 0;
                for (int j = 0; j < N; ++j) {
                    const bool on = na->all_ones || ((a->p_adj[gr * a->NW + (j >> 5)] >> (j & 31)) & 1u);
                    if (!on) continue;
                    ++cnt;
                    const float4 pj = c.s_p[r - i + j];
                    const float d0 = pi.x - pj.x, d1 = pi.y - pj.y, d2 = pi.z - pj.z, d3 = pi.w - pj.w;
#pragma unroll
                    for (int q = 0; q < 4; ++q) {
                        float v = fmaf(w[q][3], d3, fmaf(w[q][2], d2, fmaf(w[q][1], d1, fmaf(w[q][0], d0, 0.f))));
                        v = fmaf(w[q][7], dew, fmaf(w[q][6], dez, fmaf(w[q][5], dey, fmaf(w[q][4], dex, v)))) + b[q];
                        out[q] += fmaxf(v, 0.f);
                    }
                }
                const float nrm = cnt ? 1.f / fmaxf((float)cnt, 1e-12f) : 0.f;
#pragma unroll
                for (int q = 0; q < 4; ++q) out[q] *= nrm;
            } else if (rel == 1) {
                const float e_on = na->all_ones ? 1.f : (float)a->e_adj[gr];
#pragma unroll
                for (int q = 0; q < 4; ++q)
                    out[q] = e_on * fmaxf(dot4w(reinterpret_cast<const float(&)[4]>(w[q]), dex, dey, dez, dew, b[q]), 0.f);
            } else {
                const int m = a->map_id ? a->map_id[env] : env;
                const int2 *oxy = reinterpret_cast<const int2 *>(a->oxy) + (int64_t)m * a->O;
                int cnt = 0;
                if (na->all_ones) {
                    cnt = a->o_count[m];
                    for (int k = 0; k < cnt; ++k) {
                        const int2 o = __ldg(oxy + k);
                        const float d0 = pi.x - (float)o.x, d1 = pi.y - (float)o.y;
#pragma unroll
                        for (int q = 0; q < 4; ++q)
                            out[q] += fmaxf(dot4w(reinterpret_cast<const float(&)[4]>(w[q]), d0, d1, pi.z, pi.w, b[q]), 0.f);
                    }
                } else {
                    for (int wd = 0; wd < a->OW; ++wd) {
                        uint32_t bits = a->o_adj[gr * a->OW + wd];
                        cnt += __popc(bits);
                        while (bits) {
                            const int k = wd * 32 + __ffs(bits) - 1;
                            bits &= bits - 1;
                            const int2 o = __ldg(oxy + k);
                            const float d0 = pi.x - (float)o.x, d1 = pi.y - (float)o.y;
#pragma unroll
                            for (int q = 0; q < 4; ++q)
                                out[q] += fmaxf(dot4w(reinterpret_cast<const float(&)[4]>(w[q]), d0, d1, pi.z, pi.w, b[q]), 0.f);
                        }
                    }
                }
                const float nrm = cnt ? 1.f / fmaxf((float)cnt, 1e-12f) : 0.f;
#pragma unroll
                for (int q = 0; q < 4; ++q) out[q] *= nrm;
            }
        }
        x_store4(c.X, r, lane, make_float4(out[0], out[1], out[2], out[3]));
    }
}

// ---- DHGN.message + mean aggregation, env-grouped path for N = NA in {4, 8, 16} (16 % NA == 0, O <= 256) -> X ---------------
// A warp owns 16/NA whole envs.  Everything shared by the rows of an env is computed once per env and kept in registers:
//   relation 0: relu(W0[:, :4](p_i - p_j) + W0[:, 4:](p_i - e) + b0) = relu(a_i - q_j),  q_j = W0[:, :4] p_j,
//               a_i = q_i + W0[:, 4:](p_i - e) + b0                       (3 instructions per (i, j, channel));
//   relation 2, critic (all cells of the map): sum_k relu(cc_i - u_k) = ((n cc_i - sum_k u_k) + sum_k |cc_i - u_k|) / 2 with
//               cc_i = W2 p_i + b2, u_k = W2[:, :2] o_k                    (2 instructions per (i, k, channel));
//   the map's boundary cells live in registers (lane l holds cells l, l+32, ...) and are broadcast with shuffles.
template <int NA, int WW>
__device__ void phase_msg_fast(const Ctx &c, int rel, const float (&w)[4][8], const float (&b)[4])
{
    constexpr int RPW = Lay<WW>::RPW;
    static_assert(RPW % NA == 0, "whole envs per warp");
    const StepArgs *a = c.a;
    const NetArgs *na = c.na;
    const int lane = c.lane;
    constexpr int RC = NA < 8 ? NA : 8;      // rows per register chunk of the critic's obstacle relation
#pragma unroll 1
    for (int g = 0; g < RPW / NA; ++g) {
        const int r0 = RPW * c.warp + g * NA;
        int64_t gr0;
        int env, i0;
        const bool ok = row_info(c, r0, gr0, env, i0);     // rows of an env are valid together
        if (!ok) {
#pragma unroll
            for (int i = 0; i < NA; ++i) x_store4(c.X, r0 + i, lane, make_float4(0.f, 0.f, 0.f, 0.f));
            continue;
        }
        const float4 ev = c.s_e[r0 / NA];
        if (rel == 0) {
            float qj[NA][4];
#pragma unroll
            for (int j = 0; j < NA; ++j) {
                const float4 pj = c.s_p[r0 + j];
#pragma unroll
                for (int q = 0; q < 4; ++q) qj[j][q] = fmaf(w[q][3], pj.w, fmaf(w[q][2], pj.z, fmaf(w[q][1], pj.y, w[q][0] * pj.x)));
            }
#pragma unroll
            const uint32_t my_word = (!na->all_ones && lane < NA) ? a->p_adj[(gr0 + lane) * a->NW] : 0xffffffffu;
#pragma unroll
            for (int i = 0; i < NA; ++i) {
                const uint32_t word = __shfl_sync(0xffffffffu, my_word, i);
                const int cnt = __popc(word & ((NA == 32) ? 0xffffffffu : ((1u << NA) - 1u)));
                const float4 pi = c.s_p[r0 + i];               // (re-read: keeping all NA states live costs 4 NA registers in the hottest loop)
                const float dex = pi.x - ev.x, dey = pi.y - ev.y, dez = pi.z - ev.z, dew = pi.w - ev.w;
                float ai[4], acc[4];
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    ai[q] = (qj[i][q] + fmaf(w[q][7], dew, fmaf(w[q][6], dez, fmaf(w[q][5], dey, w[q][4] * dex)))) + b[q];
                    acc[q] = 0.f;
                }
#pragma unroll
                for (int j = 0; j < NA; ++j) {
                    const bool on = (word >> j) & 1u;
#pragma unroll
                    for (int q = 0; q < 4; ++q) {
                        const float t = fmaxf(ai[q] - qj[j][q], 0.f);
                        acc[q] += on ? t : 0.f;
                    }
                }
                const float nrm = cnt ? 1.f / fmaxf((float)cnt, 1e-12f) : 0.f;
                x_store4(c.X, r0 + i, lane, make_float4(acc[0] * nrm, acc[1] * nrm, acc[2] * nrm, acc[3] * nrm));
            }
        } else if (rel == 1) {
            const float my_on = (!na->all_ones && lane < NA) ? (float)a->e_adj[gr0 + lane] : 1.f;
#pragma unroll
            for (int i = 0; i < NA; ++i) {
                const float4 pi = c.s_p[r0 + i];
                const float e_on = __shfl_sync(0xffffffffu, my_on, i);
                float o[4];
#pragma unroll
                for (int q = 0; q < 4; ++q)
                    o[q] = e_on * fmaxf(dot4w(reinterpret_cast<const float(&)[4]>(w[q]), pi.x - ev.x, pi.y - ev.y, pi.z - ev.z, pi.w - ev.w, b[q]), 0.f);
                x_store4(c.X, r0 + i, lane, make_float4(o[0], o[1], o[2], o[3]));
            }
        } else {
            const int m = a->map_id ? a->map_id[env] : env;
            const int2 *oxy = reinterpret_cast<const int2 *>(a->oxy) + (int64_t)m * a->O;
            // the map's boundary cells -> this warp's shared-memory staging (one broadcast LDS.64 per cell in the loops below;
            // the loops are unrolled so that several cells are in flight)
            float2 *so = c.s_oxy + c.warp * OXY_CAP;
            __syncwarp();                                      // the previous env's readers are done
#pragma unroll
            for (int t = 0; t < 8; ++t) {
                const int k = lane + 32 * t;
                if (t < a->OW && k < a->O) { const int2 o = __ldg(oxy + k); so[k] = make_float2((float)o.x, (float)o.y); }
            }
            __syncwarp();
            if (na->all_ones) {
                const int n = a->o_count[m];
                float sx = 0.f, sy = 0.f;
#pragma unroll
                for (int t = 0; t < 8; ++t) if (lane + 32 * t < n) { const float2 o = so[lane + 32 * t]; sx += o.x; sy += o.y; }
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) { sx += __shfl_xor_sync(0xffffffffu, sx, o); sy += __shfl_xor_sync(0xffffffffu, sy, o); }
                const float nrm = n ? 1.f / fmaxf((float)n, 1e-12f) : 0.f;
#pragma unroll 1
                for (int ch = 0; ch < NA / RC; ++ch) {
                    float cc[RC][4], acc[RC][4];
#pragma unroll
                    for (int rr = 0; rr < RC; ++rr) {
                        const float4 p = c.s_p[r0 + ch * RC + rr];
#pragma unroll
                        for (int q = 0; q < 4; ++q) { cc[rr][q] = dot4w(reinterpret_cast<const float(&)[4]>(w[q]), p.x, p.y, p.z, p.w, b[q]); acc[rr][q] = 0.f; }
                    }
                    auto cell = [&](const float2 o) {
                        float u[4];
#pragma unroll
                        for (int q = 0; q < 4; ++q) u[q] = fmaf(w[q][1], o.y, w[q][0] * o.x);
#pragma unroll
                        for (int rr = 0; rr < RC; ++rr)
#pragma unroll
                            for (int q = 0; q < 4; ++q) acc[rr][q] += fabsf(cc[rr][q] - u[q]);
                    };
                    int kk = 0;
#pragma unroll 1
                    for (; kk + 4 <= n; kk += 4) {                  // same k order as a plain loop: identical sums
                        const float4 o01 = *reinterpret_cast<const float4 *>(so + kk), o23 = *reinterpret_cast<const float4 *>(so + kk + 2);
                        cell(make_float2(o01.x, o01.y));
                        cell(make_float2(o01.z, o01.w));
                        cell(make_float2(o23.x, o23.y));
                        cell(make_float2(o23.z, o23.w));
                    }
#pragma unroll 1
                    for (; kk < n; ++kk) cell(so[kk]);
#pragma unroll
                    for (int rr = 0; rr < RC; ++rr) {
                        float o[4];
#pragma unroll
                        for (int q = 0; q < 4; ++q) {
                            const float su = fmaf(w[q][1], sy, w[q][0] * sx);          // sum_k u_k
                            o[q] = fmaxf(0.5f * (((float)n * cc[rr][q] - su) + acc[rr][q]), 0.f) * nrm;
                        }
                        x_store4(c.X, r0 + ch * RC + rr, lane, make_float4(o[0], o[1], o[2], o[3]));
                    }
                }
            } else {
                // this group's NA rows x OW adjacency words: lane l holds words l, l + 32, ... of the flattened [NA][OW] block.  An
                // agent sees one or two boundary cells on average, so almost every word is zero: a ballot of the non-zero words
                // lets a row visit only those (same cells in the same ascending order as a plain scan of all OW words).
                uint32_t my_bits[4];
#pragma unroll
                for (int t = 0; t < 4; ++t) {
                    const int idx = lane + 32 * t;
                    my_bits[t] = idx < NA * a->OW ? a->o_adj[gr0 * a->OW + idx] : 0u;
                }
                uint32_t nz[4];
#pragma unroll
                for (int t = 0; t < 4; ++t) nz[t] = __ballot_sync(0xffffffffu, my_bits[t] != 0u);
#pragma unroll 1
                for (int i = 0; i < NA; ++i) {
                    float cc[4] = {0.f, 0.f, 0.f, 0.f}, acc[4] = {0.f, 0.f, 0.f, 0.f};
                    int cnt = 0;
                    bool have_cc = false;
#pragma unroll 1
                    for (int t = 0; t < a->OW; ++t) {
                        const int idx = i * a->OW + t;
                        const uint32_t nzw = (idx >> 5) == 0 ? nz[0] : ((idx >> 5) == 1 ? nz[1] : ((idx >> 5) == 2 ? nz[2] : nz[3]));
                        if (!((nzw >> (idx & 31)) & 1u)) continue;                     // warp-uniform
                        const uint32_t v0 = __shfl_sync(0xffffffffu, my_bits[0], idx & 31), v1 = __shfl_sync(0xffffffffu, my_bits[1], idx & 31);
                        const uint32_t v2 = __shfl_sync(0xffffffffu, my_bits[2], idx & 31), v3 = __shfl_sync(0xffffffffu, my_bits[3], idx & 31);
                        uint32_t bits = (idx >> 5) == 0 ? v0 : ((idx >> 5) == 1 ? v1 : ((idx >> 5) == 2 ? v2 : v3));
                        if (!have_cc) {
                            const float4 pi = c.s_p[r0 + i];
#pragma unroll
                            for (int q = 0; q < 4; ++q) cc[q] = dot4w(reinterpret_cast<const float(&)[4]>(w[q]), pi.x, pi.y, pi.z, pi.w, b[q]);
                            have_cc = true;
                        }
                        cnt += __popc(bits);
                        while (bits) {                                                    // warp-uniform, in bit order
                            const int k0 = __ffs(bits) - 1;
                            bits &= bits - 1;
                            const float2 o0 = so[32 * t + k0];
#pragma unroll
                            for (int q = 0; q < 4; ++q) acc[q] += fmaxf(cc[q] - fmaf(w[q][1], o0.y, w[q][0] * o0.x), 0.f);
                        }
                    }
                    const float nrm = cnt ? 1.f / fmaxf((float)cnt, 1e-12f) : 0.f;
                    x_store4(c.X, r0 + i, lane, make_float4(acc[0] * nrm, acc[1] * nrm, acc[2] * nrm, acc[3] * nrm));
                }
            }
        }
    }
}

template <int NA, int WW>
__device__ void phase_msg_fast(const Ctx &c, int rel)
{
    float w[4][8], b[4];
    load_msg_weights(c.na, rel, c.lane, w, b);
    phase_msg_fast<NA, WW>(c, rel, w, b);
}

template <int WW>
__device__ __forceinline__ bool fast_env_path(const Ctx &c)
{
    const StepArgs *a = c.a;
    return (a->N == 4 || a->N == 8 || a->N == 16) && a->N <= Lay<WW>::RPW && a->O <= OXY_CAP;
}

template <int WW, bool F32>
__device__ void phase_msg(const Ctx &c, int rel)
{
    if (!fast_env_path<WW>(c)) phase_msg_generic<WW, F32>(c, rel);
    else if (c.a->N == 8) phase_msg_fast<8, WW>(c, rel);
    else if (c.a->N == 4) phase_msg_fast<4, WW>(c, rel);
    else if constexpr (WW == 8) phase_msg_fast<16, WW>(c, rel);
}

// ---- DHGN.fcra neighbour mean of the k-th history embedding -> X --------------------------------------------------------
template <int WW>
__device__ void phase_fcra_generic(const Ctx &c, int k)
{
    constexpr int RPW = Lay<WW>::RPW;
    const StepArgs *a = c.a;
    const NetArgs *na = c.na;
    const float *hist = na->hist[k];
    const int N = a->N;
#pragma unroll 1
    for (int rr = 0; rr < RPW; ++rr) {
        const int r = RPW * c.warp + rr;
        int64_t gr;
        int env, i;
        const bool ok = row_info(c, r, gr, env, i);
        float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
        if (ok && hist) {
            int cnt = 0;
            for (int j = 0; j < N; ++j) {
                const bool on = na->all_ones || ((a->p_adj[gr * a->NW + (j >> 5)] >> (j & 31)) & 1u);
                if (!on) continue;
                ++cnt;
                const float4 h = __ldg(reinterpret_cast<const float4 *>(hist + ((int64_t)env * N + j) * E) + c.lane);
                acc.x += h.x; acc.y += h.y; acc.z += h.z; acc.w += h.w;
            }
            const float nrm = cnt ? 1.f / fmaxf((float)cnt, 1e-12f) : 0.f;
            acc.x *= nrm; acc.y *= nrm; acc.z *= nrm; acc.w *= nrm;
        }
        x_store4(c.X, r, c.lane, acc);
    }
}

// env-grouped path, split in two: the history rows of the warp's envs are fetched (16 independent 512-byte warp loads, issued
// while the previous MMA group runs) and then averaged per row from registers
template <int NA, int WW>
__device__ __forceinline__ void fcra_prefetch(const Ctx &c, int k, float4 (&h)[Lay<WW>::RPW], uint32_t (&words)[4])
{
    constexpr int RPW = Lay<WW>::RPW;
    const StepArgs *a = c.a;
    const NetArgs *na = c.na;
    const float *hist = na->hist[k];
#pragma unroll
    for (int g = 0; g < RPW / NA; ++g) {
        const int r0 = RPW * c.warp + g * NA;
        int64_t gr0;
        int env, i0;
        const bool ok = row_info(c, r0, gr0, env, i0);
        words[g] = !ok ? 0u : ((!na->all_ones && c.lane < NA) ? a->p_adj[(gr0 + c.lane) * a->NW] : ((1u << NA) - 1u));
#pragma unroll
        for (int j = 0; j < NA; ++j)
            h[g * NA + j] = (ok && hist) ? __ldg(reinterpret_cast<const float4 *>(hist + (gr0 + j) * E) + c.lane) : make_float4(0.f, 0.f, 0.f, 0.f);
    }
}
template <int NA, int WW>
__device__ __forceinline__ void fcra_finish(const Ctx &c, const float4 (&h)[Lay<WW>::RPW], const uint32_t (&words)[4])
{
    constexpr int RPW = Lay<WW>::RPW;
#pragma unroll
    for (int g = 0; g < RPW / NA; ++g) {
        const int r0 = RPW * c.warp + g * NA;
#pragma unroll
        for (int i = 0; i < NA; ++i) {
            const uint32_t word = __shfl_sync(0xffffffffu, words[g], i);
            const int cnt = __popc(word & ((1u << NA) - 1u));
            float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
            for (int j = 0; j < NA; ++j) {
                const bool on = (word >> j) & 1u;
                const float4 hj = h[g * NA + j];
                acc.x += on ? hj.x : 0.f; acc.y += on ? hj.y : 0.f; acc.z += on ? hj.z : 0.f; acc.w += on ? hj.w : 0.f;
            }
            const float nrm = cnt ? 1.f / fmaxf((float)cnt, 1e-12f) : 0.f;
            x_store4(c.X, r0 + i, c.lane, make_float4(acc.x * nrm, acc.y * nrm, acc.z * nrm, acc.w * nrm));
        }
    }
}
template <int WW>
__device__ __forceinline__ void phase_fcra_prefetch(const Ctx &c, int k, float4 (&h)[Lay<WW>::RPW], uint32_t (&words)[4])
{
    if (!fast_env_path<WW>(c)) return;
    if (c.a->N == 8) fcra_prefetch<8, WW>(c, k, h, words);
    else if (c.a->N == 4) fcra_prefetch<4, WW>(c, k, h, words);
    else if constexpr (WW == 8) fcra_prefetch<16, WW>(c, k, h, words);
}
template <int WW>
__device__ __forceinline__ void phase_fcra_finish(const Ctx &c, int k, const float4 (&h)[Lay<WW>::RPW], const uint32_t (&words)[4])
{
    if (!fast_env_path<WW>(c)) phase_fcra_generic<WW>(c, k);
    else if (c.a->N == 8) fcra_finish<8, WW>(c, h, words);
    else if (c.a->N == 4) fcra_finish<4, WW>(c, h, words);
    else if constexpr (WW == 8) fcra_finish<16, WW>(c, h, words);
}

// ---- previous hidden state of GRU layer l -> X (16 independent 512-byte warp loads in flight) ----------------------------
template <int WW>
__device__ __forceinline__ void hidden_prefetch(const Ctx &c, int l, float4 (&v)[Lay<WW>::RPW])
{
    constexpr int RPW = Lay<WW>::RPW;
    const float *h = c.na->hidden_in + (int64_t)l * c.a->R * E;
#pragma unroll
    for (int rr = 0; rr < RPW; ++rr) {
        int64_t gr;
        int env, i;
        const bool ok = row_info(c, RPW * c.warp + rr, gr, env, i);
        v[rr] = ok ? *(reinterpret_cast<const float4 *>(h + gr * E) + c.lane) : make_float4(0.f, 0.f, 0.f, 0.f);
    }
}
template <int WW>
__device__ __forceinline__ void hidden_store(const Ctx &c, const float4 (&v)[Lay<WW>::RPW])
{
    constexpr int RPW = Lay<WW>::RPW;
#pragma unroll
    for (int rr = 0; rr < RPW; ++rr) x_store4(c.X, RPW * c.warp + rr, c.lane, v[rr]);
}

// global rows [R,E] -> X in chunks of 8 rows per warp.  The pair kernel issues the loads of all its chunks before it waits for the
// running MMA group and stores them to X after the wait.
template <int WW>
__device__ __forceinline__ void rows_prefetch8(const Ctx &c, const float *src, int chunk, float4 (&v)[8])
{
    constexpr int RPW = Lay<WW>::RPW;
#pragma unroll
    for (int rr = 0; rr < 8; ++rr) {
        int64_t gr;
        int env, i;
        const bool ok = row_info(c, RPW * c.warp + 8 * chunk + rr, gr, env, i);
        v[rr] = ok ? *(reinterpret_cast<const float4 *>(src + gr * E) + c.lane) : make_float4(0.f, 0.f, 0.f, 0.f);
    }
}
template <int WW>
__device__ __forceinline__ void rows_store8(const Ctx &c, int chunk, const float4 (&v)[8])
{
    constexpr int RPW = Lay<WW>::RPW;
#pragma unroll
    for (int rr = 0; rr < 8; ++rr) x_store4(c.X, RPW * c.warp + 8 * chunk + rr, c.lane, v[rr]);
}
// X <- rows of a global [R,E] tensor (all of the warp's rows)
template <int WW>
__device__ void fill_x(const Ctx &c, const float *src)
{
    float4 v[8];
#pragma unroll 1
    for (int ch = 0; ch < Lay<WW>::RPW / 8; ++ch) {
        rows_prefetch8<WW>(c, src, ch, v);
        rows_store8<WW>(c, ch, v);
    }
}

// X (hi + lo: fp32 to one ulp) -> global rows, coalesced: warp w copies its RPW rows, 512 bytes per row
template <int WW>
__device__ void copy_out(const Ctx &c, float *g)
{
    constexpr int RPW = Lay<WW>::RPW;
#pragma unroll 4
    for (int rr = 0; rr < RPW; ++rr) {
        const int r = RPW * c.warp + rr;
        int64_t gr;
        int env, i;
        if (row_info(c, r, gr, env, i)) *(reinterpret_cast<float4 *>(g + gr * E) + c.lane) = x_load4(c.X, r, c.lane);
    }
}

// ---- epilogue: X <- act(acc + bias [+ W_p p_i]) ; optional global copy ---------------------------------------------------
// thread <-> row 32*(warp&3)+lane (its TMEM lane), columns [CPT*(warp>>2), +CPT)
template <int WW>
__device__ void epi_store(const Ctx &c, int acc_col, const float *bias, bool relu, const float *wp, int wp_ld, float *gout)
{
    constexpr int CPT = Lay<WW>::CPT;
    const int row = 32 * (c.warp & 3) + c.lane, hh = c.warp >> 2;
    float4 p = make_float4(0.f, 0.f, 0.f, 0.f);
    if (wp) p = c.s_p[row];
    const uint32_t taddr = c.tmem + ((uint32_t)(32 * (c.warp & 3)) << 16) + (uint32_t)acc_col;
#pragma unroll 1
    for (int c0 = CPT * hh; c0 < CPT * hh + CPT; c0 += 32) {
        uint32_t v[32];
        PF_TMEM_LD32(v, taddr + (uint32_t)c0);
        tmem_wait_ld();
#pragma unroll
        for (int j = 0; j < 32; j += 8) {
            const int col = c0 + j;
            const float4 b0 = __ldg(reinterpret_cast<const float4 *>(bias + col)), b1 = __ldg(reinterpret_cast<const float4 *>(bias + col + 4));
            float o[8] = {__uint_as_float(v[j]) + b0.x, __uint_as_float(v[j + 1]) + b0.y, __uint_as_float(v[j + 2]) + b0.z, __uint_as_float(v[j + 3]) + b0.w,
                          __uint_as_float(v[j + 4]) + b1.x, __uint_as_float(v[j + 5]) + b1.y, __uint_as_float(v[j + 6]) + b1.z, __uint_as_float(v[j + 7]) + b1.w};
            if (wp) {
#pragma unroll
                for (int q = 0; q < 8; ++q) {
                    const float4 wv = __ldg(reinterpret_cast<const float4 *>(wp + (int64_t)(col + q) * wp_ld));
                    o[q] += fmaf(wv.w, p.w, fmaf(wv.z, p.z, fmaf(wv.y, p.y, fmaf(wv.x, p.x, 0.f))));
                }
            }
            if (relu) {
#pragma unroll
                for (int q = 0; q < 8; ++q) o[q] = fmaxf(o[q], 0.f);
            }
            x_store8(c.X, row, col >> 3, o);
        }
    }
    if (gout) {
        worker_sync<WW>();
        copy_out<WW>(c, gout);
    }
}

// MUFU.EX2 / MUFU.RCP directly: the same two hardware approximations __expf / __fdividef are built on, without their range
// handling (scaling around denormal exp results and huge divisors: 11 / 13 instructions per sigmoid / tanh instead of 4 / 6).  Here
// the argument of the reciprocal is 1 + 2^y >= 1, and a flushed-to-zero or infinite 2^y gives the correct limits 1, 0, -1.
__device__ __forceinline__ float rcp_approx(float x) { float y; asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
__device__ __forceinline__ float ex2_approx(float x) { float y; asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
__device__ __forceinline__ float fast_sigmoid(float x) { return rcp_approx(1.f + ex2_approx(-1.4426950408889634f * x)); }
__device__ __forceinline__ float fast_tanh(float x) { return 1.f - 2.f * rcp_approx(1.f + ex2_approx(2.8853900817779268f * x)); }

// ---- epilogue: GRU cell of layer l (torch gate order r, z, n); h' -> X (then coalesced to global); critic layer 1: value ---
// h_prev is read back from X (it is the A operand of the W_hh group; hi + lo = fp32 to one ulp).  The gates use ex2-based exp and the fast
// division (abs error ~1e-7, inside the 1e-5 forward tolerance).
template <int WW>
__device__ void epi_cell(const Ctx &c, int l, bool want_value)
{
    constexpr int CPT = Lay<WW>::CPT;
    const NetArgs *na = c.na;
    const int row = 32 * (c.warp & 3) + c.lane, hh = c.warp >> 2;
    const float *bi = na->b_ih[l], *bh = na->b_hh[l];
    const uint32_t taddr = c.tmem + ((uint32_t)(32 * (c.warp & 3)) << 16);
    float vdot = 0.f;
#pragma unroll 1
    for (int c0 = CPT * hh; c0 < CPT * hh + CPT; c0 += 16) {
        uint32_t ar[16], az[16], an[16], ahn[16];
        PF_TMEM_LD16(ar, taddr + (uint32_t)c0);
        PF_TMEM_LD16(az, taddr + (uint32_t)(128 + c0));
        PF_TMEM_LD16(an, taddr + (uint32_t)(256 + c0));
        PF_TMEM_LD16(ahn, taddr + (uint32_t)(384 + c0));
        float hp_all[2][8];
#pragma unroll
        for (int j = 0; j < 16; j += 8) x_load8(c.X, row, (c0 + j) >> 3, hp_all[j >> 3]);   // before any store to X (no false dependence)
        tmem_wait_ld();
        float hn_all[2][8];
#pragma unroll
        for (int j = 0; j < 16; j += 4) {
            const int col = c0 + j;
            const float4 hp4 = make_float4(hp_all[j >> 3][j & 4], hp_all[j >> 3][(j & 4) + 1], hp_all[j >> 3][(j & 4) + 2], hp_all[j >> 3][(j & 4) + 3]);
            const float4 bir = __ldg(reinterpret_cast<const float4 *>(bi + col)), bhr = __ldg(reinterpret_cast<const float4 *>(bh + col));
            const float4 biz = __ldg(reinterpret_cast<const float4 *>(bi + E + col)), bhz = __ldg(reinterpret_cast<const float4 *>(bh + E + col));
            const float4 bin = __ldg(reinterpret_cast<const float4 *>(bi + 2 * E + col)), bhn = __ldg(reinterpret_cast<const float4 *>(bh + 2 * E + col));
            float4 wv = make_float4(0.f, 0.f, 0.f, 0.f);
            if (want_value) wv = __ldg(reinterpret_cast<const float4 *>(na->head_w_eff + col));
            const float hp[4] = {hp4.x, hp4.y, hp4.z, hp4.w};
            const float f_bir[4] = {bir.x, bir.y, bir.z, bir.w}, f_bhr[4] = {bhr.x, bhr.y, bhr.z, bhr.w};
            const float f_biz[4] = {biz.x, biz.y, biz.z, biz.w}, f_bhz[4] = {bhz.x, bhz.y, bhz.z, bhz.w};
            const float f_bin[4] = {bin.x, bin.y, bin.z, bin.w}, f_bhn[4] = {bhn.x, bhn.y, bhn.z, bhn.w};
            const float f_w[4] = {wv.x, wv.y, wv.z, wv.w};
            float hn[4];
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                const float r = fast_sigmoid((__uint_as_float(ar[j + q]) + f_bir[q]) + f_bhr[q]);
                const float z = fast_sigmoid((__uint_as_float(az[j + q]) + f_biz[q]) + f_bhz[q]);
                const float n = fast_tanh((__uint_as_float(an[j + q]) + f_bin[q]) + r * (__uint_as_float(ahn[j + q]) + f_bhn[q]));
                hn[q] = (1.f - z) * n + z * hp[q];
                vdot = fmaf(f_w[q], hn[q], vdot);
            }
#pragma unroll
            for (int q = 0; q < 4; ++q) hn_all[j >> 3][(j & 4) + q] = hn[q];
        }
#pragma unroll
        for (int j = 0; j < 16; j += 8) x_store8(c.X, row, (c0 + j) >> 3, hn_all[j >> 3]);
    }
    if (want_value) c.s_val[hh * ROWS + row] = vdot;
    worker_sync<WW>();
    copy_out<WW>(c, na->hidden_out + (int64_t)l * c.a->R * E);
    if (want_value && hh == 0 && c.a->value) {
        int64_t gr;
        int env, i;
        if (row_info(c, row, gr, env, i)) {
            float v = c.s_val[row] + c.s_val[ROWS + row];
            if (WW == 16) v = (v + c.s_val[2 * ROWS + row]) + c.s_val[3 * ROWS + row];
            c.a->value[gr] = v + __ldg(na->head_b);
        }
    }
}

// ---- epilogue: actor head (softmax -> sample / argmax -> log-prob), same arithmetic and RNG as act_head_kernel -----------
template <int A>
__device__ void epi_head(const Ctx &c)
{
    if (c.warp >= 4) return;
    const int row = 32 * c.warp + c.lane;
    int64_t gr;
    int env, i;
    const bool ok = row_info(c, row, gr, env, i);
    uint32_t v[16];
    PF_TMEM_LD16(v, c.tmem + ((uint32_t)(32 * c.warp) << 16));
    tmem_wait_ld();
    if (!ok) return;
    float z[A], mx = -INFINITY;
#pragma unroll
    for (int k = 0; k < A; ++k) { z[k] = __uint_as_float(v[k]) + __ldg(c.na->head_b + k); mx = fmaxf(mx, z[k]); }
    float sm[A], den = 0.f;
#pragma unroll
    for (int k = 0; k < A; ++k) { sm[k] = expf(z[k] - mx); den += sm[k]; }
    float psum = 0.f;
#pragma unroll
    for (int k = 0; k < A; ++k) { sm[k] /= den; psum += sm[k]; }
    int act = 0;
    if (c.a->force_action) {
        act = min(max(c.a->action[gr], 0), A - 1);          // teacher forcing: log-prob of a given action
    } else if (c.a->deterministic) {
        float best = -1.f;
#pragma unroll
        for (int k = 0; k < A; ++k) if (sm[k] > best) { best = sm[k]; act = k; }
    } else {
        const uint64_t seed = c.a->d_seed ? *c.a->d_seed : c.a->seed;
        const uint64_t hsh = splitmix64(seed ^ splitmix64((uint64_t)(gr + c.a->row_offset) * 0x100000001B3ull + (uint64_t)c.a->t));
        const float u = (float)(hsh >> 40) * (1.0f / 16777216.0f) * psum;
        float cs = 0.f;
        act = A - 1;
#pragma unroll
        for (int k = 0; k < A; ++k) { cs += sm[k]; if (u < cs) { act = k; break; } }
    }
    const float ceps = 1.1920928955078125e-07f;
    float lpa = 0.f;
#pragma unroll
    for (int k = 0; k < A; ++k) if (k == act) lpa = logf(fminf(fmaxf(sm[k] / psum, ceps), 1.f - ceps));
    if (c.a->action && !c.a->force_action) c.a->action[gr] = act;
    if (c.a->logp) c.a->logp[gr] = lpa;
}

// FL: marl_policy_step.flags (MARL_POLICY_STATE_F32 / MARL_POLICY_EMBED_ONLY), one instantiation per combination
template <int WW, int FL>
__global__ void __launch_bounds__(Lay<WW>::THREADS, 1)
policy_step_kernel(const __grid_constant__ StepArgs a)
{
    constexpr bool F32 = (FL & MARL_POLICY_STATE_F32) != 0, EMB = (FL & MARL_POLICY_EMBED_ONLY) != 0;
    constexpr int RPW = Lay<WW>::RPW;
    extern __shared__ __align__(1024) unsigned char smem[];
    if ((smem_u32(smem) & 1023u) != 0u) __trap();          // SWIZZLE_128B atoms need 1024-byte alignment
    unsigned char *X = smem;
    unsigned char *Wst = smem + RING_OFF;
    uint64_t *bars = reinterpret_cast<uint64_t *>(smem + MISC_OFF);   // full[NSTAGE], empty[NSTAGE], a_ready, mma_done
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(bars + 2 * NSTAGE + 2);
    static_assert(2 * NSTAGE + 3 <= 16, "barrier block");
    float4 *s_p = reinterpret_cast<float4 *>(bars + 16);                                  // 128 x float4 (later: s_val)
    float4 *s_e = s_p + ROWS;                                                               // 32 x float4
    float2 *s_oxy = reinterpret_cast<float2 *>(smem + OXY_OFF);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    int net, tile;
    if (a.net_count == 2) { net = (int)blockIdx.x < a.n_tiles ? 1 : 0; tile = (int)blockIdx.x % a.n_tiles; }   // critic items first
    else { net = a.net_first; tile = blockIdx.x; }
    const NetArgs *na = &a.net[net];

    if (threadIdx.x == 0) {
        for (int s = 0; s < NSTAGE; ++s) {
            mbar_init(smem_u32(&bars[s]), 1);            // full: one arrive.expect_tx + the bulk copy's bytes
            mbar_init(smem_u32(&bars[NSTAGE + s]), 1);      // empty: one tcgen05.commit
        }
        mbar_init(smem_u32(&bars[BAR_A_READY]), Lay<WW>::WORKERS);   // a_ready
        mbar_init(smem_u32(&bars[BAR_MMA_DONE]), 1);        // mma_done
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == WW + 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "n"(512) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp < WW) {
        // ================================================================================= workers
        Ctx c;
        c.a = &a; c.na = na; c.X = X; c.row0 = (int64_t)tile * a.rows_per_tile; c.warp = warp; c.lane = lane;
        c.tmem = tmem_base; c.bar_a_ready = smem_u32(&bars[BAR_A_READY]); c.bar_mma_done = smem_u32(&bars[BAR_MMA_DONE]); c.group = 0; c.s_p = s_p; c.s_e = s_e; c.s_val = reinterpret_cast<float *>(s_p); c.s_oxy = s_oxy;
        {   // fp32 copies of the tile's pursuer / evader states (converted once; every SIMT phase reads them from smem)
            const int t = threadIdx.x;
            if (t < ROWS) {
                int64_t gr;
                int env, i;
                s_p[t] = row_info(c, t, gr, env, i) ? load_p<F32>(&a, gr) : make_float4(0.f, 0.f, 0.f, 0.f);
            } else if (t < ROWS + 32) {
                const int64_t env = c.row0 / a.N + (t - ROWS);
                s_e[t - ROWS] = (ROWS / a.N <= 32 && t - ROWS < ROWS / a.N && env < a.B) ? load_e<F32>(&a, (int)env) : make_float4(0.f, 0.f, 0.f, 0.f);
            }
            worker_sync<WW>();
        }
        long long tk[16];
#pragma unroll
        for (int q = 0; q < 16; ++q) tk[q] = 0;
        long long t_prev = clock64();
        const long long t_begin = t_prev;
        if (a.dbg && threadIdx.x == 0) {                            // profiling aid: wall-clock start (ns) and SM id of this CTA
            unsigned long long gt;
            unsigned smid;
            asm volatile("mov.u64 %0, %globaltimer;" : "=l"(gt));
            asm volatile("mov.u32 %0, %smid;" : "=r"(smid));
            tk[13] = (long long)gt;
            tk[15] = (long long)smid;
        }
#define PF_TICK(slot) do { const long long now_ = clock64(); tk[slot] += now_ - t_prev; t_prev = now_; } while (0)
        for (int r = 0; r < 3; ++r) {
            phase_msg<WW, F32>(c, r);
            PF_TICK(0 + r);
            hand_over(c);                                              // AGG_vertex_0 -> acc @0
            PF_TICK(11);
            epi_store<WW>(c, 0, na->b_av, true, nullptr, 0, nullptr);
            PF_TICK(3);
            hand_over(c);                                              // semantic, K-slice r -> acc @128
            PF_TICK(11);
        }
        epi_store<WW>(c, 128, na->b_sem, false, na->sem_w, na->sem_ld, nullptr);    // h0 (no activation)
        PF_TICK(4);
        float4 pre[RPW];
        for (int k = 0; k < a.depth; ++k) {
            uint32_t words[4] = {0u, 0u, 0u, 0u};
            signal_ready(c);                                           // FCRA_k, h part -> acc @128
            phase_fcra_prefetch<WW>(c, k, pre, words);                     //   ... while it runs: the history rows of the tile
            wait_done(c);
            PF_TICK(11);
            phase_fcra_finish<WW>(c, k, pre, words);
            PF_TICK(5);
            hand_over(c);                                              // AGG_fcra_k -> acc @0
            PF_TICK(11);
            epi_store<WW>(c, 0, na->b_aggf[k], true, nullptr, 0, nullptr);
            PF_TICK(6);
            hand_over(c);                                              // FCRA_k, m part -> acc @128 (+=)
            PF_TICK(11);
            epi_store<WW>(c, 128, na->b_f[k], true, nullptr, 0, k == a.depth - 1 ? na->emb_out : nullptr);
            PF_TICK(7);
        }
        if constexpr (EMB) {
            // embeddings only: the unit program ends with the FCRA chain (fill_net), nothing is left to hand over
        } else {
            for (int l = 0; l < 2; ++l) {
                signal_ready(c);                                           // W_ih: r @0, z @128, n @256
                hidden_prefetch<WW>(c, l, pre);                                //   ... while it runs: h_prev of this layer
                wait_done(c);
                PF_TICK(11);
                hidden_store<WW>(c, pre);
                PF_TICK(8);
                hand_over(c);                                              // W_hh: r += , z +=, hn @384
                PF_TICK(11);
                epi_cell<WW>(c, l, l == 1 && na->head_w_eff != nullptr);
                PF_TICK(9);
            }
        }
        if (!EMB && net == 0) {
            hand_over(c);                                              // actor head, n_out = 16 -> acc @0
            PF_TICK(11);
            epi_head<MARL_NUM_ACTIONS>(c);
            PF_TICK(10);
        }
        if (a.dbg && threadIdx.x == 0) {
            tk[12] = clock64() - t_begin;
            unsigned long long gt;
            asm volatile("mov.u64 %0, %globaltimer;" : "=l"(gt));
            tk[14] = (long long)gt;
            for (int q = 0; q < 16; ++q) a.dbg[(size_t)blockIdx.x * 16 + q] = tk[q];
        }
    } else if (warp == WW) {
        // ================================================================================= weight loader
        if (lane == 0) {
            int it = 0;
            for (int u = 0; u < na->n_units; ++u) {
                const Unit un = na->u[u];
                // one stage = a k-block of both operand planes (32 KB); the packed unit is [kb0: hi plane, lo plane][kb1: hi plane,
                // lo plane], so the stages are consecutive slices of it
                const uint32_t bytes = 2u * un.n_out * 128u;
                for (int st = 0; st < NKB; ++st, ++it) {
                    const int s = it % NSTAGE, round = it / NSTAGE;
                    if (round > 0) mbar_wait(smem_u32(&bars[NSTAGE + s]), (uint32_t)((round - 1) & 1));
                    mbar_expect_tx(smem_u32(&bars[s]), bytes);
                    bulk_g2s(smem_u32(Wst + s * WSTAGE), na->packed + un.off + (size_t)st * bytes, bytes, smem_u32(&bars[s]));
                }
            }
        }
    } else {
        // ================================================================================= MMA issuer (whole warp walks the
        // unit program, one elected lane issues: see policy_pair_kernel)
        {
            int it = 0, group = 0;
            bool fresh_group = true;
            for (int u = 0; u < na->n_units; ++u) {
                const Unit un = na->u[u];
                if (fresh_group) {
                    mbar_wait(smem_u32(&bars[BAR_A_READY]), (uint32_t)(group & 1));
                    tc_fence_after();
                    fresh_group = false;
                }
                const uint32_t idesc = idesc_f16(un.n_out);
                const uint32_t acc = tmem_base + un.acc_col;
                const uint32_t lo_off = (uint32_t)un.n_out * 128u;
                for (int kb = 0; kb < NKB; ++kb, ++it) {
                    const int s = it % NSTAGE, round = it / NSTAGE;
                    mbar_wait(smem_u32(&bars[s]), (uint32_t)(round & 1));
                    tc_fence_after();
                    const uint32_t xa = smem_u32(X + kb * XKB), wb = smem_u32(Wst + s * WSTAGE);
                    // descriptors of the first K=16 slice; the next slices are +32 bytes = +2 in the (addr >> 4) field
                    const uint64_t a_hi0 = make_desc(xa), a_lo0 = make_desc(xa + TILE), b_hi0 = make_desc(wb), b_lo0 = make_desc(wb + lo_off);
                    if (elect_one()) {
#pragma unroll
                        for (int kk = 0; kk < 4; ++kk) {
                            const uint64_t a_hi = a_hi0 + 2 * kk, a_lo = a_lo0 + 2 * kk, b_hi = b_hi0 + 2 * kk, b_lo = b_lo0 + 2 * kk;
                            umma_f16(acc, a_hi, b_hi, idesc, (un.accumulate || kb || kk) ? 1u : 0u);
                            umma_f16(acc, a_lo, b_hi, idesc, 1u);
                            umma_f16(acc, a_hi, b_lo, idesc, 1u);
                        }
                        umma_commit(smem_u32(&bars[NSTAGE + s]));
                    }
                    __syncwarp();
                }
                if (un.last) {
                    if (elect_one()) umma_commit(smem_u32(&bars[BAR_MMA_DONE]));
                    __syncwarp();
                    ++group;
                    fresh_group = true;
                }
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == WW + 1) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(512) : "memory");
}


// =================================================================================================================================
// PAIR kernel: ONE CTA runs the actor chain AND the critic chain of the same 128-row tile, interleaved step by step.
//
// The unit chain of one network is a dependence chain: SIMT phase -> MMA group -> epilogue -> MMA group -> ...  With one chain per
// CTA the 16 worker warps idle while the tensor pipe runs (~30 % of an item, DESIGN 4a) and the tensor pipe idles while they work.
// Here the workers alternate between the two chains: they finish a step of the actor chain, hand its tile to the issuer, and do
// the same step of the critic chain while the actor's MMAs run, and vice versa - the same 16 warps at 8 rows each (the code
// that fits 96 registers), so unlike two co-resident CTAs nothing is paid in registers or shared memory per warp.  And because
// the two networks share ONE encoder (DHGN/mappo_parallel.py:582-616) and the CTA holds the same rows for both, everything the
// two chains have in common is computed once: the fp32 copy of the states, the staged boundary cells, relation 0's q_j / a_i and
// its pair terms relu(a_i - q_j) (reduced under the comm-adjacency mask for the actor and unmasked for the critic in the same
// loop), relation 1's message (times e_adj for the actor).
//   shared memory : X_actor 64 KB + X_critic 64 KB + weight ring 64 KB + boundary-cell staging 32 KB + 3 KB        (227 KB)
//   tensor memory : 256 columns per chain.  The encoder needs two 128-column accumulators; the GRU runs in two 64-column halves
//                   (r @0, z @64, n_i @128, n_h @192) in the order  W_ih(half 0) | X <- h_prev | W_hh(half 0) -> cell 0 |
//                   W_hh(half 1) | X <- x | W_ih(half 1) -> cell 1 | X <- h',  i.e. three X fills per layer whose global loads are
//                   issued BEFORE the wait for the running MMA group; the new state goes straight from registers to memory (in
//                   place: a half only overwrites columns nobody reads from memory afterwards).
//   weight ring   : a FIFO of 16 KB slots; a k-block of a 128-row unit takes two slots, of a 64-row GRU unit one, so the ring holds
//                   one whole encoder unit or two GRU units ahead of the issuer.
// The loader and the issuer walk the two unit programs group by group in the order the workers signal them: A.g0, C.g0, A.g1, ...
struct MemPair {
    static constexpr int SLOT = 16384, NSLOT = 4, NENT = 8;
    static constexpr int XC_OFF = X_BYTES, RING_OFF = 2 * X_BYTES, MISC_OFF = RING_OFF + NSLOT * SLOT, OXY_OFF = MISC_OFF + MISC_BYTES;
    static constexpr int BYTES = OXY_OFF + OXY_BYTES;
    static constexpr int BAR_FULL = 0, BAR_EMPTY = NENT, BAR_READY = 2 * NENT, BAR_DONE = 2 * NENT + 2, NBAR = 2 * NENT + 4;   // [chain]
};
static_assert(MemPair::BYTES <= 232448, "PAIR kernel shared memory");
static_assert((MemPair::NBAR + 2) * 8 % 16 == 0 && (MemPair::NBAR + 2) * 8 + (ROWS + 32) * 16 <= MISC_BYTES, "PAIR kernel misc block");

// ring bookkeeping shared by the loader and the issuer (both walk the same unit lists, so both compute the same slots)
struct RingCursor {
    int cur = 0, seq = 0;
    __device__ __forceinline__ void next(uint32_t bytes, int &slot, int &k, int &e)
    {
        k = bytes > (uint32_t)MemPair::SLOT ? 2 : 1;
        if (k == 2 && (cur & 1)) ++cur;                    // two-slot entries start on an even slot (never wrap)
        slot = cur & (MemPair::NSLOT - 1);
        cur += k;
        e = seq++;
    }
};

// ---- relations 0 and 1 for BOTH chains at once (env-grouped fast path, N = NA in {4, 8}): same arithmetic, term for term, as
// phase_msg_fast run once per network - the pair terms / the evader message are simply not computed twice
template <int NA, int WW>
__device__ void phase_msg_pair01(const Ctx &c, unsigned char *XA, unsigned char *XC, int rel, const float (&w)[4][8], const float (&b)[4])
{
    constexpr int RPW = Lay<WW>::RPW;
    static_assert(RPW % NA == 0, "whole envs per warp");
    const StepArgs *a = c.a;
    const int lane = c.lane;
#pragma unroll 1
    for (int g = 0; g < RPW / NA; ++g) {
        const int r0 = RPW * c.warp + g * NA;
        int64_t gr0;
        int env, i0;
        const bool ok = row_info(c, r0, gr0, env, i0);
        if (!ok) {
#pragma unroll
            for (int i = 0; i < NA; ++i) {
                x_store4(XA, r0 + i, lane, make_float4(0.f, 0.f, 0.f, 0.f));
                x_store4(XC, r0 + i, lane, make_float4(0.f, 0.f, 0.f, 0.f));
            }
            continue;
        }
        const float4 ev = c.s_e[r0 / NA];
        if (rel == 0) {
            float qj[NA][4];
#pragma unroll
            for (int j = 0; j < NA; ++j) {
                const float4 pj = c.s_p[r0 + j];
#pragma unroll
                for (int q = 0; q < 4; ++q) qj[j][q] = fmaf(w[q][3], pj.w, fmaf(w[q][2], pj.z, fmaf(w[q][1], pj.y, w[q][0] * pj.x)));
            }
            const uint32_t my_word = lane < NA ? a->p_adj[(gr0 + lane) * a->NW] : 0u;
            const float nrm_c = 1.f / fmaxf((float)NA, 1e-12f);
#pragma unroll
            for (int i = 0; i < NA; ++i) {
                const uint32_t word = __shfl_sync(0xffffffffu, my_word, i);
                const int cnt = __popc(word & ((1u << NA) - 1u));
                const float4 pi = c.s_p[r0 + i];               // (re-read: keeping all NA states live costs 32 registers in the hottest loop)
                const float dex = pi.x - ev.x, dey = pi.y - ev.y, dez = pi.z - ev.z, dew = pi.w - ev.w;
                float ai[4], acc_a[4], acc_c[4];
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    ai[q] = (qj[i][q] + fmaf(w[q][7], dew, fmaf(w[q][6], dez, fmaf(w[q][5], dey, w[q][4] * dex)))) + b[q];
                    acc_a[q] = acc_c[q] = 0.f;
                }
#pragma unroll
                for (int j = 0; j < NA; ++j) {
                    const bool on = (word >> j) & 1u;
#pragma unroll
                    for (int q = 0; q < 4; ++q) {
                        const float t = fmaxf(ai[q] - qj[j][q], 0.f);
                        acc_c[q] += t;
                        acc_a[q] += on ? t : 0.f;
                    }
                }
                const float nrm_a = cnt ? 1.f / fmaxf((float)cnt, 1e-12f) : 0.f;
                x_store4(XA, r0 + i, lane, make_float4(acc_a[0] * nrm_a, acc_a[1] * nrm_a, acc_a[2] * nrm_a, acc_a[3] * nrm_a));
                x_store4(XC, r0 + i, lane, make_float4(acc_c[0] * nrm_c, acc_c[1] * nrm_c, acc_c[2] * nrm_c, acc_c[3] * nrm_c));
            }
        } else {
            const float my_on = lane < NA ? (float)a->e_adj[gr0 + lane] : 1.f;
#pragma unroll
            for (int i = 0; i < NA; ++i) {
                const float4 pi = c.s_p[r0 + i];
                const float e_on = __shfl_sync(0xffffffffu, my_on, i);
                float o[4];
#pragma unroll
                for (int q = 0; q < 4; ++q)
                    o[q] = fmaxf(dot4w(reinterpret_cast<const float(&)[4]>(w[q]), pi.x - ev.x, pi.y - ev.y, pi.z - ev.z, pi.w - ev.w, b[q]), 0.f);
                x_store4(XA, r0 + i, lane, make_float4(e_on * o[0], e_on * o[1], e_on * o[2], e_on * o[3]));
                x_store4(XC, r0 + i, lane, make_float4(1.f * o[0], 1.f * o[1], 1.f * o[2], 1.f * o[3]));
            }
        }
    }
}

// one 64-column half of the GRU cell for WW worker warps: thread <-> row 32*(warp&3)+lane, columns [CPH*(warp>>2), +CPH) of the half.
// h_prev comes from X (HP_FROM_X: X holds h_prev) or from memory (X holds x by then); the new state goes from registers to memory.
template <int WW, bool HP_FROM_X>
__device__ void epi_cell_half_w(const Ctx &c, int l, int half, bool want_value, float *s_part)
{
    constexpr int CG = WW / 4, CPH = 64 / CG;
    const NetArgs *na = c.na;
    const int row = 32 * (c.warp & 3) + c.lane, hh = c.warp >> 2;
    const float *bc = na->b_comb[l];
    const uint32_t taddr = c.tmem + ((uint32_t)(32 * (c.warp & 3)) << 16);
    int64_t gr;
    int env, i;
    const bool ok = row_info(c, row, gr, env, i);
    float *dst = na->hidden_out + ((int64_t)l * c.a->R + gr) * E;
    const float *hsrc = na->hidden_in + ((int64_t)l * c.a->R + gr) * E;
    float vdot = 0.f;
#pragma unroll 1
    for (int j0 = CPH * hh; j0 < CPH * hh + CPH; j0 += 8) {
        uint32_t ar[8], az[8], an[8], ahn[8];
        asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
                     : "=r"(ar[0]), "=r"(ar[1]), "=r"(ar[2]), "=r"(ar[3]), "=r"(ar[4]), "=r"(ar[5]), "=r"(ar[6]), "=r"(ar[7]) : "r"(taddr + (uint32_t)j0));
        asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
                     : "=r"(az[0]), "=r"(az[1]), "=r"(az[2]), "=r"(az[3]), "=r"(az[4]), "=r"(az[5]), "=r"(az[6]), "=r"(az[7]) : "r"(taddr + (uint32_t)(64 + j0)));
        asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
                     : "=r"(an[0]), "=r"(an[1]), "=r"(an[2]), "=r"(an[3]), "=r"(an[4]), "=r"(an[5]), "=r"(an[6]), "=r"(an[7]) : "r"(taddr + (uint32_t)(128 + j0)));
        asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
                     : "=r"(ahn[0]), "=r"(ahn[1]), "=r"(ahn[2]), "=r"(ahn[3]), "=r"(ahn[4]), "=r"(ahn[5]), "=r"(ahn[6]), "=r"(ahn[7]) : "r"(taddr + (uint32_t)(192 + j0)));
        const int col = 64 * half + j0;
        float hp[8];
        if constexpr (HP_FROM_X) {
            x_load8(c.X, row, col >> 3, hp);
        } else {
            float4 u = make_float4(0.f, 0.f, 0.f, 0.f), v = u;
            if (ok) { u = *reinterpret_cast<const float4 *>(hsrc + col); v = *reinterpret_cast<const float4 *>(hsrc + col + 4); }
            hp[0] = u.x; hp[1] = u.y; hp[2] = u.z; hp[3] = u.w; hp[4] = v.x; hp[5] = v.y; hp[6] = v.z; hp[7] = v.w;
        }
        tmem_wait_ld();
        float hn[8];
#pragma unroll
        for (int q4 = 0; q4 < 8; q4 += 4) {
            const float4 br = __ldg(reinterpret_cast<const float4 *>(bc + col + q4)), bz = __ldg(reinterpret_cast<const float4 *>(bc + E + col + q4));
            const float4 bin = __ldg(reinterpret_cast<const float4 *>(bc + 2 * E + col + q4)), bhn = __ldg(reinterpret_cast<const float4 *>(bc + 3 * E + col + q4));
            float4 wv = make_float4(0.f, 0.f, 0.f, 0.f);
            if (want_value) wv = __ldg(reinterpret_cast<const float4 *>(na->head_w_eff + col + q4));
            const float f_br[4] = {br.x, br.y, br.z, br.w}, f_bz[4] = {bz.x, bz.y, bz.z, bz.w};
            const float f_bin[4] = {bin.x, bin.y, bin.z, bin.w}, f_bhn[4] = {bhn.x, bhn.y, bhn.z, bhn.w};
            const float f_w[4] = {wv.x, wv.y, wv.z, wv.w};
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                const float r = fast_sigmoid(__uint_as_float(ar[q4 + q]) + f_br[q]);
                const float z = fast_sigmoid(__uint_as_float(az[q4 + q]) + f_bz[q]);
                const float n = fast_tanh((__uint_as_float(an[q4 + q]) + f_bin[q]) + r * (__uint_as_float(ahn[q4 + q]) + f_bhn[q]));
                hn[q4 + q] = (1.f - z) * n + z * hp[q4 + q];
                vdot = fmaf(f_w[q], hn[q4 + q], vdot);
            }
        }
        if (ok) {
            *reinterpret_cast<float4 *>(dst + col) = make_float4(hn[0], hn[1], hn[2], hn[3]);
            *reinterpret_cast<float4 *>(dst + col + 4) = make_float4(hn[4], hn[5], hn[6], hn[7]);
        }
    }
    if (want_value) s_part[(half * CG + hh) * ROWS + row] = vdot;
}

// Launched with WW + 4 warps: the worker warps (whole warpgroups) take the registers that the loader / issuer warpgroup (two working
// lanes, two idle warps) gives back with setmaxnreg, so the SIMT phases get 112 registers per thread instead of 96.
constexpr int PAIR_WORKER_REGS = 112, PAIR_OTHER_REGS = 32;      // 16 worker warps: the CTA owns 640 x 96 registers
constexpr int PAIR8_WORKER_REGS = 232, PAIR8_OTHER_REGS = 40;     //  8 worker warps (16-agent envs): 384 x 168   // the CTA owns 640 x 96 registers: 512 x 104 + 128 x 56 fits; the issuer lane needs ~50
// PROF: per-phase cycle counters in registers (tools/fused_phase_profile.py, MARL_POLICY_PROFILE=1); the production instantiation
// only writes the CTA's start / end %globaltimer, SM id and total cycles when a debug buffer is given, and keeps nothing live for it.
#define PP_TICK(slot) do { if constexpr (PROF) { const long long now_ = clock64(); tk[slot] += now_ - t_prev; t_prev = now_; } } while (0)
template <int WW, bool PROF, int FL>
__global__ void __launch_bounds__((WW + 4) * 32, 1)
policy_pair_kernel(const __grid_constant__ StepArgs a)
{
    constexpr bool F32 = (FL & MARL_POLICY_STATE_F32) != 0, EMB = (FL & MARL_POLICY_EMBED_ONLY) != 0;
    using M = MemPair;
    extern __shared__ __align__(1024) unsigned char smem[];
    if ((smem_u32(smem) & 1023u) != 0u) __trap();
    unsigned char *Wst = smem + M::RING_OFF;
    uint64_t *bars = reinterpret_cast<uint64_t *>(smem + M::MISC_OFF);   // full[8], empty[8], a_ready[2 chains], mma_done[2 chains]
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(bars + M::NBAR);
    float4 *s_p = reinterpret_cast<float4 *>(bars + M::NBAR + 2);                 // 16-byte aligned
    float4 *s_e = s_p + ROWS;
    float2 *s_oxy = reinterpret_cast<float2 *>(smem + M::OXY_OFF);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int tile = blockIdx.x;

    if (threadIdx.x == 0) {
        for (int e = 0; e < M::NENT; ++e) {
            mbar_init(smem_u32(&bars[M::BAR_FULL + e]), 1);
            mbar_init(smem_u32(&bars[M::BAR_EMPTY + e]), 1);
        }
        for (int ch = 0; ch < 2; ++ch) {
            mbar_init(smem_u32(&bars[M::BAR_READY + ch]), WW);            // one arrival per worker warp
            mbar_init(smem_u32(&bars[M::BAR_DONE + ch]), 1);
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == WW + 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "n"(512) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    if (warp < WW) asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(WW == 16 ? PAIR_WORKER_REGS : PAIR8_WORKER_REGS));
    else asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(WW == 16 ? PAIR_OTHER_REGS : PAIR8_OTHER_REGS));

    if (warp < WW) {
        // ================================================================================= workers
        Ctx c;
        c.a = &a; c.row0 = (int64_t)tile * a.rows_per_tile; c.warp = warp; c.lane = lane; c.group = 0; c.s_p = s_p; c.s_e = s_e;
        c.s_val = reinterpret_cast<float *>(s_oxy);      // value partials: the boundary-cell staging is dead once the GRU starts
        c.s_oxy = s_oxy;
        c.na = &a.net[0]; c.X = smem; c.tmem = tmem_base; c.bar_a_ready = 0; c.bar_mma_done = 0;
        {
            const int t = threadIdx.x;
            if (t < ROWS) {
                int64_t gr;
                int env, i;
                s_p[t] = row_info(c, t, gr, env, i) ? load_p<F32>(&a, gr) : make_float4(0.f, 0.f, 0.f, 0.f);
            } else if (t < ROWS + 32) {
                const int64_t env = c.row0 / a.N + (t - ROWS);
                s_e[t - ROWS] = (ROWS / a.N <= 32 && t - ROWS < ROWS / a.N && env < a.B) ? load_e<F32>(&a, (int)env) : make_float4(0.f, 0.f, 0.f, 0.f);
            }
            worker_sync<WW>();
        }
        long long tk[PROF ? 12 : 1];
#pragma unroll
        for (int q = 0; q < (PROF ? 12 : 1); ++q) tk[q] = 0;
        long long t_prev = PROF ? clock64() : 0;
        (void)tk; (void)t_prev;
        if (a.dbg && threadIdx.x == 0) {
            unsigned long long gt;
            unsigned smid;
            asm volatile("mov.u64 %0, %globaltimer;" : "=l"(gt));
            asm volatile("mov.u32 %0, %smid;" : "=r"(smid));
            long long *d = a.dbg + (size_t)blockIdx.x * 16;
            d[12] = clock64();
            d[13] = (long long)gt;
            d[15] = (long long)smid;
        }
        // EMB: both chains stop after the FCRA chain's last epilogue (step G0 - 1, which stores the embedding)
        const int D = a.depth, G0 = 7 + 3 * D, S_ACTOR = EMB ? G0 : G0 + 9, S_CRITIC = EMB ? G0 : G0 + 8;
        constexpr int NA_BIG = Lay<WW>::RPW;                           // env size whose rows fill a warp: 8 (16 worker warps) or 16 (8)
        const bool pair01 = (a.N == NA_BIG || (WW == 16 && a.N == 4)) && a.NW == 1;      // relations 0 and 1 computed once for both chains
        const uint32_t bar_ready0 = smem_u32(&bars[M::BAR_READY]), bar_done0 = smem_u32(&bars[M::BAR_DONE]);
#pragma unroll 1
        for (int s = 0; s < S_ACTOR; ++s) {
#pragma unroll 1
            for (int ch = 0; ch < 2; ++ch) {
                if (s >= (ch == 0 ? S_ACTOR : S_CRITIC)) continue;
                const bool shared = pair01 && (s == 0 || s == 2);
                if (shared && ch == 1) continue;               // done together with the actor's
                PP_TICK(8);
                const NetArgs *na = &a.net[ch];
                c.na = na;
                c.X = smem + ch * M::XC_OFF;
                c.tmem = tmem_base + 256u * (uint32_t)ch;
                c.bar_a_ready = bar_ready0 + 8u * (uint32_t)ch;
                c.bar_mma_done = bar_done0 + 8u * (uint32_t)ch;
                // The chain's previous MMA group must have finished before this step touches its accumulators or X.  Steps that fill X
                // from memory issue their global loads first and wait afterwards (the load latency hides behind the wait); loads and
                // stores stay in one straight-line block so that the rows live in registers, not on the stack.
                auto wait_prev = [&]() {
                    PP_TICK(9);
                    if (s > 0) {
                        mbar_wait(c.bar_mma_done, (uint32_t)((s - 1) & 1));
                        if (shared) mbar_wait(bar_done0 + 8u, (uint32_t)((s - 1) & 1));
                        tc_fence_after();
                    }
                    PP_TICK(11);
                };
                bool signal = true;
                // every dense layer's epilogue is the same code with different operands: ONE call site, so that the (large, fully
                // unrolled) epilogue exists once in the instruction stream instead of once per layer
                const int fk = s >= 7 ? (s - 7) / 3 : 0, fsub = s >= 7 ? (s - 7) % 3 : -1;
                const bool is_msg = s < 6 && (s & 1) == 0, is_fcra_fill = s >= 7 && s < G0 && fsub == 0;
                if (s < G0 && !is_msg && !is_fcra_fill) {
                    int acc_col = 0;
                    const float *bias = na->b_av, *wp = nullptr;
                    float *gout = nullptr;
                    bool relu = true;
                    if (s == 6) { acc_col = 128; bias = na->b_sem; relu = false; wp = na->sem_w; }        // h0 (no activation)
                    else if (s > 6 && fsub == 1) { bias = na->b_aggf[fk]; }
                    else if (s > 6) { acc_col = 128; bias = na->b_f[fk]; gout = fk == D - 1 ? na->emb_out : nullptr; }
                    wait_prev();
                    epi_store<WW>(c, acc_col, bias, relu, wp, na->sem_ld, gout);
                    if (EMB && s == G0 - 1) signal = false;
                    PP_TICK(1);
                } else if (is_msg) {                           // messages of relation s/2 -> X
                    if (pair01 && a.O <= OXY_CAP) {
                        // the layer's weights are fetched before the wait for the running MMA group (their L2 latency, ~700 cycles at
                        // the head of every message phase, passes meanwhile); straight-line per env size, so they stay in registers
                        float w[4][8], b[4];
                        load_msg_weights(na, s >> 1, lane, w, b);
                        wait_prev();
                        if (a.N == NA_BIG) {
                            if (shared) phase_msg_pair01<NA_BIG, WW>(c, smem, smem + M::XC_OFF, s >> 1, w, b);
                            else phase_msg_fast<NA_BIG, WW>(c, s >> 1, w, b);
                        } else if constexpr (WW == 16) {
                            if (shared) phase_msg_pair01<4, WW>(c, smem, smem + M::XC_OFF, s >> 1, w, b);
                            else phase_msg_fast<4, WW>(c, s >> 1, w, b);
                        }
                    } else {
                        wait_prev();
                        phase_msg<WW, F32>(c, s >> 1);
                    }
                    PP_TICK(0);
                } else if (is_fcra_fill) {
                    // (one straight-line block per env size: through the size-dispatching wrappers the row array ended up on the
                    // stack - the loads were stored to local memory before the wait and read back after it)
                    if (pair01 && a.O <= OXY_CAP && a.N == NA_BIG) {
                        float4 pre[Lay<WW>::RPW];
                        uint32_t words[4] = {0u, 0u, 0u, 0u};
                        fcra_prefetch<NA_BIG, WW>(c, fk, pre, words);
                        wait_prev();
                        fcra_finish<NA_BIG, WW>(c, pre, words);
                    } else if (WW == 16 && pair01 && a.O <= OXY_CAP && a.N == 4) {
                        float4 pre[Lay<WW>::RPW];
                        uint32_t words[4] = {0u, 0u, 0u, 0u};
                        fcra_prefetch<4, WW>(c, fk, pre, words);
                        wait_prev();
                        fcra_finish<4, WW>(c, pre, words);
                    } else {
                        wait_prev();
                        phase_fcra_generic<WW>(c, fk);
                    }
                    PP_TICK(2);
                } else if (s < G0 + 8) {
                    const int l = (s - G0) >> 2, gsub = (s - G0) & 3;
                    const bool want_value = l == 1 && na->head_w_eff != nullptr;
                    if (gsub == 0 || gsub == 2) {              // X <- h_prev (for W_hh of both halves) / X <- x again (for W_ih, half 1)
                        const float *src = gsub == 0 ? na->hidden_in + (int64_t)l * a.R * E : (l == 0 ? na->emb_out : na->hidden_out);
                        float4 pre[Lay<WW>::RPW / 8][8];
#pragma unroll
                        for (int q = 0; q < Lay<WW>::RPW / 8; ++q) rows_prefetch8<WW>(c, src, q, pre[q]);
                        wait_prev();
#pragma unroll
                        for (int q = 0; q < Lay<WW>::RPW / 8; ++q) rows_store8<WW>(c, q, pre[q]);
                        PP_TICK(3);
                    } else if (gsub == 1) {                    // W_hh(half 0) done: cell of half 0, h_prev read back from X
                        wait_prev();
                        epi_cell_half_w<WW, true>(c, l, 0, want_value, c.s_val);
                        PP_TICK(4);
                    } else {                                   // W_ih(half 1) done: cell of half 1, h_prev from memory (X holds x)
                        wait_prev();
                        epi_cell_half_w<WW, false>(c, l, 1, want_value, c.s_val);
                        worker_sync<WW>();                     // both halves of the new state are in memory
                        PP_TICK(4);
                        if (l == 0 || ch == 0) {               // X <- the layer's new state: input of layer 1 / of the actor head
                            fill_x<WW>(c, na->hidden_out + (int64_t)l * a.R * E);
                            PP_TICK(3);
                        } else {                               // critic, last layer: the value
                            signal = false;
                            const int row = 32 * (warp & 3) + lane, hh = warp >> 2;
                            int64_t gr;
                            int env, i;
                            if (want_value && hh == 0 && a.value && row_info(c, row, gr, env, i)) {
                                float v = 0.f;
#pragma unroll
                                for (int q = 0; q < 2 * (WW / 4); ++q) v += c.s_val[q * ROWS + row];
                                a.value[gr] = v + __ldg(na->head_b);
                            }
                        }
                    }
                } else {
                    wait_prev();
                    epi_head<MARL_NUM_ACTIONS>(c);
                    PP_TICK(5);
                    signal = false;
                }
                if (signal) {
                    // every lane makes its X stores visible to the tensor core's proxy and orders its TMEM loads; one lane per warp
                    // arrives (512 arrivals on one mbarrier serialise: ~1.2 K cycles per hand-over, exposed here because the MMA
                    // latency itself is hidden behind the other chain's step)
                    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                    tc_fence_before();
                    __syncwarp();
                    if (lane == 0) {
                        mbar_arrive(c.bar_a_ready);
                        if (shared) mbar_arrive(bar_ready0 + 8u);
                    }
                    PP_TICK(10);
                }
            }
        }
        if (a.dbg && threadIdx.x == 0) {
            unsigned long long gt;
            asm volatile("mov.u64 %0, %globaltimer;" : "=l"(gt));
            long long *d = a.dbg + (size_t)blockIdx.x * 16;
            d[12] = clock64() - d[12];
            d[14] = (long long)gt;
            if constexpr (PROF) {
                for (int q = 0; q < 6; ++q) d[q] = tk[q];
                d[9] = tk[9]; d[10] = tk[10]; d[11] = tk[11];
                d[15] = tk[8];       // (PROF only: the SM id slot carries the loop-overhead counter)
            }
        }
    } else if (warp == WW) {
        // ================================================================================= weight loader
        if (lane == 0) {
            RingCursor rc;
            int owner[M::NSLOT] = {-1, -1, -1, -1}, iu[2] = {0, 0};
            while (iu[0] < a.net[0].n_units || iu[1] < a.net[1].n_units) {
                for (int ch = 0; ch < 2; ++ch) {
                    const NetArgs *na = &a.net[ch];
                    bool last = iu[ch] >= na->n_units;
                    while (!last) {
                        const Unit un = na->u[iu[ch]++];
                        last = un.last != 0;
                        const uint32_t bytes = 2u * un.n_out * 128u;
                        for (int kb = 0; kb < NKB; ++kb) {
                            int slot, k, e;
                            rc.next(bytes, slot, k, e);
                            int need = owner[slot];
                            if (k == 2 && owner[slot + 1] > need) need = owner[slot + 1];
                            if (need >= 0) mbar_wait(smem_u32(&bars[M::BAR_EMPTY + (need & (M::NENT - 1))]), (uint32_t)((need / M::NENT) & 1));
                            owner[slot] = e;
                            if (k == 2) owner[slot + 1] = e;
                            const uint32_t full = smem_u32(&bars[M::BAR_FULL + (e & (M::NENT - 1))]);
                            mbar_expect_tx(full, bytes);
                            bulk_g2s(smem_u32(Wst + slot * M::SLOT), na->packed + un.off + (size_t)kb * bytes, bytes, full);
                        }
                    }
                }
            }
        }
    } else if (warp == WW + 1) {
        // ================================================================================= MMA issuer
        // The whole warp walks the unit program (warp-uniform control flow, every lane polls the barriers); one elected lane issues.
        // Under `if (lane == 0)` the compiler has to wrap every tcgen05.mma in a lane-serialising loop to get its operands into
        // uniform registers (~20 instructions per MMA): too slow for the 64-row GRU units, whose MMAs take 32 cycles each.
        RingCursor rc;
        int iu[2] = {0, 0}, grp[2] = {0, 0};
        long long t_ready = 0, t_full = 0, t0 = PROF ? clock64() : 0, t_start = t0;
        (void)t_start;
        while (iu[0] < a.net[0].n_units || iu[1] < a.net[1].n_units) {
#pragma unroll 1
            for (int ch = 0; ch < 2; ++ch) {
                const NetArgs *na = &a.net[ch];
                if (iu[ch] >= na->n_units) continue;
                mbar_wait(smem_u32(&bars[M::BAR_READY + ch]), (uint32_t)(grp[ch] & 1));
                if constexpr (PROF) { const long long n_ = clock64(); t_ready += n_ - t0; t0 = n_; }
                tc_fence_after();
                const uint32_t xbase = smem_u32(smem + ch * M::XC_OFF);
                bool last = false;
#pragma unroll 1
                while (!last) {
                    const Unit un = na->u[iu[ch]++];
                    last = un.last != 0;
                    const uint32_t idesc = idesc_f16(un.n_out);
                    const uint32_t acc = tmem_base + 256u * (uint32_t)ch + un.acc_col;
                    const uint32_t bytes = 2u * un.n_out * 128u, lo_off = (uint32_t)un.n_out * 128u;
#pragma unroll 1
                    for (int kb = 0; kb < NKB; ++kb) {
                        int slot, k, e;
                        rc.next(bytes, slot, k, e);
                        if constexpr (PROF) t0 = clock64();
                        mbar_wait(smem_u32(&bars[M::BAR_FULL + (e & (M::NENT - 1))]), (uint32_t)((e / M::NENT) & 1));
                        if constexpr (PROF) { const long long n_ = clock64(); t_full += n_ - t0; t0 = n_; }
                        tc_fence_after();
                        const uint32_t xa = xbase + kb * XKB, wb = smem_u32(Wst + slot * M::SLOT);
                        const uint64_t a_hi0 = make_desc(xa), a_lo0 = make_desc(xa + TILE), b_hi0 = make_desc(wb), b_lo0 = make_desc(wb + lo_off);
                        if (elect_one()) {
#pragma unroll
                            for (int kk = 0; kk < 4; ++kk) {
                                const uint64_t a_hi = a_hi0 + 2 * kk, a_lo = a_lo0 + 2 * kk, b_hi = b_hi0 + 2 * kk, b_lo = b_lo0 + 2 * kk;
                                umma_f16(acc, a_hi, b_hi, idesc, (un.accumulate || kb || kk) ? 1u : 0u);
                                umma_f16(acc, a_lo, b_hi, idesc, 1u);
                                umma_f16(acc, a_hi, b_lo, idesc, 1u);
                            }
                            umma_commit(smem_u32(&bars[M::BAR_EMPTY + (e & (M::NENT - 1))]));
                        }
                        __syncwarp();
                    }
                }
                if (elect_one()) umma_commit(smem_u32(&bars[M::BAR_DONE + ch]));
                __syncwarp();
                ++grp[ch];
                if constexpr (PROF) t0 = clock64();
            }
        }
        if constexpr (PROF) {
            if (a.dbg && lane == 0) {
                long long *d = a.dbg + (size_t)blockIdx.x * 16;
                d[6] = t_ready; d[7] = t_full; d[8] = clock64() - t_start;
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == WW + 1) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(512) : "memory");
}

// ---- weight packing: one unit = W[rows, k0 : k0+128] -> 2 k-blocks (K = 64) x (hi plane, lo plane) in the smem image ------------
__global__ void __launch_bounds__(256)
pack_unit_kernel(const float *__restrict__ W, int64_t ld, int rows_valid, int n_out, int k0, int split, int jump,
                 unsigned char *__restrict__ out)
{
    const int idx = blockIdx.x * 256 + threadIdx.x;      // (n, k)
    if (idx >= n_out * 128) return;
    const int n = idx >> 7, k = idx & 127;
    // unit rows >= split come from `jump` source rows further down (two 64-row halves of different GRU gates in one 128-row unit)
    const int src = n + (n >= split ? jump : 0);
    const float v = n < rows_valid ? W[(int64_t)src * ld + k0 + k] : 0.f;
    uint32_t hi, lo;
    split_h2(v, 0.f, hi, lo);
    const int kb = k >> 6, kk = k & 63;
    const size_t plane = (size_t)n_out * 128;
    const size_t off = (size_t)kb * 2 * plane + (size_t)n * 128 + ((((kk >> 3) ^ (n & 7))) << 4) + (kk & 7) * 2;
    *reinterpret_cast<unsigned short *>(out + off) = (unsigned short)(hi & 0xffffu);
    *reinterpret_cast<unsigned short *>(out + off + plane) = (unsigned short)(lo & 0xffffu);
}

// b_ir + b_hr, b_iz + b_hz, b_in, b_hn of one GRU layer -> out [4][E]
__global__ void __launch_bounds__(128)
combine_gru_bias_kernel(const float *__restrict__ b_ih, const float *__restrict__ b_hh, float *__restrict__ out)
{
    const int c = threadIdx.x;
    out[c] = b_ih[c] + b_hh[c];
    out[E + c] = b_ih[E + c] + b_hh[E + c];
    out[2 * E + c] = b_ih[2 * E + c];
    out[3 * E + c] = b_hh[2 * E + c];
}

struct UnitSrc {
    const float *W;
    int64_t ld;
    int rows, n_out, k0, acc_col, accumulate, last;
    int split = 1 << 30, jump = 0;      // see pack_unit_kernel
};

static int build_units(const marl_dhgn_weights *w, int depth, int is_actor, int A, UnitSrc *us, bool pair /* else one chain per CTA */)
{
    int n = 0;
    auto add = [&](const float *W, int64_t ld, int rows, int n_out, int k0, int acc, int accu, int last) {
        us[n++] = UnitSrc{W, ld, rows, n_out, k0, acc, accu, last};
    };
    auto add_rz = [&](const float *W, int acc, int accu) {      // rows [0,64) of gate r and of gate z of one half: one 128-row unit
        UnitSrc u{W, E, E, E, 0, acc, accu, 0};
        u.split = 64;
        u.jump = E - 64;
        us[n++] = u;
    };
    for (int r = 0; r < 3; ++r) {
        add(w->agg_v_w, E, E, E, 0, 0, 0, 1);
        add(w->sem_w, 3 * E + 4, E, E, 4 + E * r, 128, r > 0, 1);
    }
    for (int k = 0; k < depth; ++k) {
        add(w->fcra_w[k], 2 * E, E, E, E, 128, 0, 1);
        add(w->agg_f_w[k], E, E, E, 0, 0, 0, 1);
        add(w->fcra_w[k], 2 * E, E, E, 0, 128, 1, 1);
    }
    for (int l = 0; l < 2; ++l) {
        if (pair) {
            // pair kernel: 64-column halves, accumulators r @0, z @64, n_i @128, n_h @192, in the order
            // W_ih(half 0) | W_hh(half 0) | W_hh(half 1) | W_ih(half 1): X holds x, h_prev, h_prev, x (one re-staging of each)
            const float *wi = w->gru_w_ih[l], *wh = w->gru_w_hh[l];
            const int64_t ro = (int64_t)64 * E, g2 = (int64_t)2 * E * E;
            // the r and z rows of a half form ONE 128-row unit (accumulator columns r @0, z @64 are adjacent): 8 units per layer instead
            // of 12, and the A tile is read from shared memory twice per group instead of three times
            add_rz(wi, 0, 0); add(wi + g2, E, 64, 64, 0, 128, 0, 1);
            add_rz(wh, 0, 1); add(wh + g2, E, 64, 64, 0, 192, 0, 1);
            add_rz(wh + ro, 0, 0); add(wh + g2 + ro, E, 64, 64, 0, 192, 0, 1);
            add_rz(wi + ro, 0, 1); add(wi + g2 + ro, E, 64, 64, 0, 128, 0, 1);
        } else {
            for (int g = 0; g < 3; ++g) add(w->gru_w_ih[l] + (int64_t)g * E * E, E, E, E, 0, 128 * g, 0, g == 2);
            add(w->gru_w_hh[l], E, E, E, 0, 0, 1, 0);
            add(w->gru_w_hh[l] + (int64_t)E * E, E, E, E, 0, 128, 1, 0);
            add(w->gru_w_hh[l] + (int64_t)2 * E * E, E, E, E, 0, 384, 0, 1);
        }
    }
    if (is_actor) add(w->head_w, E, A, 16, 0, 0, 0, 1);
    return n;
}

// Rows per work item: whole envs, at most 128 rows (one MMA M tile).  A caller that runs several launches concurrently (env-group
// pipelines) asks for full tiles: 148 items on 148 SMs leave no SM for the neighbours' kernels and every collision costs a whole
// extra wave (measured: 4 pipelines of 148 items 61.5 ms per episode, of 128 items 52.1 ms).  For a lone launch:
// one CTA is resident per SM, so the launch runs in
// ceil(items / SMs) waves; a slightly smaller tile that fills the last wave beats a full tile that leaves most SMs idle in it
// (32768 rows x 2 networks: 512 items of 128 rows = 3.46 -> 4 waves, 586 items of 112 rows = 3.96 waves).  Cost model of one item:
// SIMT phases proportional to the rows, MMA phases constant (M = 128 regardless) - measured ~3 : 1 at 128 rows.
static int choose_rows_per_tile(int64_t R, int N, int nets, int requested)
{
    static int sms = 0;
    if (sms == 0) {
        int dev = 0;
        if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || sms <= 0) sms = 148;
    }
    const int full = (ROWS / N) * N;
    if (requested > 0 && requested <= full && requested % N == 0) return requested;
    int best = full;
    double best_cost = 0.0;
    for (int rpt = full; rpt >= N && rpt * 4 >= full * 3; rpt -= N) {
        const int64_t items = ((R + rpt - 1) / rpt) * nets;
        const double waves = (double)((items + sms - 1) / sms);
        const double cost = waves * (0.75 * rpt / full + 0.25);
        if (best_cost == 0.0 || cost < best_cost - 1e-12) { best_cost = cost; best = rpt; }
    }
    return best;
}

static int64_t unit_bytes(int n_out) { return (int64_t)n_out * 128 * 2 * NKB; }
static int64_t layout_bytes(int depth, int is_actor) { return (int64_t)(6 + 3 * depth + 12) * unit_bytes(E) + (is_actor ? unit_bytes(16) : 0); }

static int check_weights(const marl_dhgn_weights *w, int depth, int is_actor)
{
    MARL_REQUIRE(w != nullptr, "marl_policy: weights struct is NULL");
    MARL_REQUIRE(depth >= 1 && depth <= MAXD, "marl_policy: depth=%d unsupported (1..%d)", depth, MAXD);
    bool ok = w->agg_v_w && w->agg_v_b && w->sem_w && w->sem_b && w->head_b;
    for (int r = 0; r < 3; ++r) ok = ok && w->msg_w[r] && w->msg_b[r];
    for (int k = 0; k < depth; ++k) ok = ok && w->agg_f_w[k] && w->agg_f_b[k] && w->fcra_w[k] && w->fcra_b[k];
    for (int l = 0; l < 2; ++l) ok = ok && w->gru_w_ih[l] && w->gru_w_hh[l] && w->gru_b_ih[l] && w->gru_b_hh[l];
    ok = ok && w->head_w;
    MARL_REQUIRE(ok, "marl_policy: null weight pointer (%s)", is_actor ? "actor" : "critic");
    return MARL_OK;
}

}  // namespace pf
}  // namespace marl

using namespace marl;

extern "C" int64_t marl_policy_pack_bytes(int32_t depth, int32_t is_actor)
{
    if (depth < 1 || depth > pf::MAXD) return -1;
    return 2 * pf::layout_bytes(depth, is_actor) + 2 * 4 * pf::E * (int64_t)sizeof(float);   // [one chain per CTA][pair][combined GRU biases]
}

extern "C" int marl_policy_pack(const marl_dhgn_weights *w, int32_t depth, int32_t is_actor, int32_t action_dim, void *d_packed,
                                void *stream)
{
    int rc = pf::check_weights(w, depth, is_actor);
    if (rc) return rc;
    MARL_REQUIRE(d_packed && ((uintptr_t)d_packed & 1023) == 0, "marl_policy_pack: workspace must be 1024-byte aligned");
    MARL_REQUIRE(!is_actor || (action_dim >= 1 && action_dim <= 16), "marl_policy_pack: action_dim=%d (1..16)", action_dim);
    unsigned char *out = static_cast<unsigned char *>(d_packed);
    for (const bool pair : {false, true}) {
        pf::UnitSrc us[pf::MAX_UNITS];
        const int n = pf::build_units(w, depth, is_actor, action_dim, us, pair);
        for (int u = 0; u < n; ++u) {
            const int total = us[u].n_out * 128;
            pf::pack_unit_kernel<<<(total + 255) / 256, 256, 0, (cudaStream_t)stream>>>(us[u].W, us[u].ld, us[u].rows, us[u].n_out, us[u].k0, us[u].split, us[u].jump, out);
            rc = check_launch("pack_unit_kernel");
            if (rc) return rc;
            out += pf::unit_bytes(us[u].n_out);
        }
    }
    for (int l = 0; l < 2; ++l) {
        pf::combine_gru_bias_kernel<<<1, pf::E, 0, (cudaStream_t)stream>>>(w->gru_b_ih[l], w->gru_b_hh[l], reinterpret_cast<float *>(out) + l * 4 * pf::E);
        rc = check_launch("combine_gru_bias_kernel");
        if (rc) return rc;
    }
    return MARL_OK;
}

static int fill_net(pf::NetArgs &na, const marl_dhgn_weights *w, const marl_policy_net_io *io, int depth, int is_actor, int A, bool pair,
                    bool embed_only)
{
    int rc = pf::check_weights(w, depth, is_actor);
    if (rc) return rc;
    MARL_REQUIRE(io->d_packed && (embed_only || io->d_hidden) && io->d_emb_out, "marl_policy_rollout_step: null packed / hidden / emb_out (%s)",
                 is_actor ? "actor" : "critic");
    pf::UnitSrc us[pf::MAX_UNITS];
    na.n_units = pf::build_units(w, depth, is_actor, A, us, pair);
    if (embed_only) na.n_units = 6 + 3 * depth;           // the encoder and FCRA units lead the program (build_units)
    uint32_t off = (uint32_t)(pair ? pf::layout_bytes(depth, is_actor) : 0);
    for (int u = 0; u < na.n_units; ++u) {
        na.u[u] = pf::Unit{off, (uint16_t)us[u].n_out, (uint16_t)us[u].acc_col, (uint8_t)us[u].accumulate, (uint8_t)us[u].last, 0};
        off += (uint32_t)pf::unit_bytes(us[u].n_out);
    }
    na.packed = static_cast<const unsigned char *>(io->d_packed);
    for (int r = 0; r < 3; ++r) { na.msg_w[r] = w->msg_w[r]; na.msg_b[r] = w->msg_b[r]; }
    na.b_av = w->agg_v_b; na.sem_w = w->sem_w; na.b_sem = w->sem_b; na.sem_ld = 3 * pf::E + 4;
    for (int k = 0; k < pf::MAXD; ++k) {
        na.b_aggf[k] = k < depth ? w->agg_f_b[k] : nullptr;
        na.b_f[k] = k < depth ? w->fcra_b[k] : nullptr;
        na.hist[k] = k < depth ? io->d_hist[k] : nullptr;
    }
    for (int l = 0; l < 2; ++l) {
        na.b_ih[l] = w->gru_b_ih[l]; na.b_hh[l] = w->gru_b_hh[l];
        na.b_comb[l] = reinterpret_cast<const float *>(static_cast<const unsigned char *>(io->d_packed) + 2 * pf::layout_bytes(depth, is_actor)) + l * 4 * pf::E;
    }
    na.head_b = w->head_b;
    na.head_w_eff = is_actor ? nullptr : w->head_w;
    na.emb_out = io->d_emb_out;
    na.hidden_in = io->d_hidden;
    na.hidden_out = io->d_hidden_out ? io->d_hidden_out : io->d_hidden;
    na.all_ones = is_actor ? 0 : 1;
    return MARL_OK;
}

static int policy_rollout_step(const marl_policy_step *s, const marl_dhgn_weights *actor_w, const marl_policy_net_io *actor_io,
                               const marl_dhgn_weights *critic_w, const marl_policy_net_io *critic_io, const uint64_t *d_seed, void *stream)
{
    MARL_REQUIRE(s != nullptr, "marl_policy_rollout_step: step struct is NULL");
    MARL_REQUIRE(s->E == pf::E, "marl_policy_rollout_step: embedding_dim=%d (the fused kernel is built for 128)", s->E);
    MARL_REQUIRE(s->B > 0 && s->N >= 1 && s->N <= 128 && s->O >= 1 && s->depth >= 1 && s->depth <= pf::MAXD,
                 "marl_policy_rollout_step: B=%d N=%d O=%d depth=%d", s->B, s->N, s->O, s->depth);
    MARL_REQUIRE(s->action_dim == MARL_NUM_ACTIONS, "marl_policy_rollout_step: action_dim=%d (9)", s->action_dim);
    MARL_REQUIRE(s->d_p_state && s->d_e_state && s->d_oxy && s->d_o_count && s->d_p_adj_bits && s->d_e_adj && s->d_o_adj_bits,
                 "marl_policy_rollout_step: null observation pointer");
    MARL_REQUIRE((actor_w && actor_io) || (critic_w && critic_io), "marl_policy_rollout_step: no network given");
    MARL_REQUIRE((s->flags & ~(MARL_POLICY_STATE_F32 | MARL_POLICY_EMBED_ONLY)) == 0, "marl_policy_rollout_step: unknown flags 0x%x",
                 (unsigned)s->flags);
    MARL_REQUIRE(s->variant != 2, "marl_policy_rollout_step: variant 2 (two CTAs per SM) was removed; use 0, 1 or 3");
    MARL_REQUIRE(s->variant == 0 || s->variant == 1 || s->variant == 3, "marl_policy_rollout_step: variant=%d (0, 1 or 3)", s->variant);
    const bool embed_only = (s->flags & MARL_POLICY_EMBED_ONLY) != 0;
    pf::StepArgs a{};
    a.B = s->B; a.N = s->N; a.O = s->O; a.NW = (s->N + 31) / 32; a.OW = (s->O + 31) / 32; a.depth = s->depth; a.A = s->action_dim;
    a.R = (int64_t)s->B * s->N;
    const bool has_a = actor_w && actor_io, has_c = critic_w && critic_io;
    const int nets = (has_a ? 1 : 0) + (has_c ? 1 : 0);
    MARL_REQUIRE(s->variant != 3 || (has_a && has_c), "marl_policy_rollout_step: variant 3 (actor + critic chains in one CTA) needs both networks");
    // variant 0: the pair kernel whenever both networks are stepped, one chain per CTA for a single network
    const bool pair = s->variant == 3 || (s->variant == 0 && has_a && has_c);
    a.rows_per_tile = pf::choose_rows_per_tile(a.R, s->N, pair ? 1 : nets, s->tile_rows);
    a.n_tiles = (int)((a.R + a.rows_per_tile - 1) / a.rows_per_tile);
    a.p_state = s->d_p_state; a.e_state = s->d_e_state; a.oxy = s->d_oxy; a.map_id = s->d_map_id; a.o_count = s->d_o_count;
    a.p_adj = s->d_p_adj_bits; a.e_adj = s->d_e_adj; a.o_adj = s->d_o_adj_bits;
    a.action = s->d_action; a.logp = s->d_logp; a.value = s->d_value; a.seed = s->seed; a.d_seed = d_seed; a.t = s->t; a.deterministic = s->deterministic; a.force_action = s->force_action;
    a.row_offset = s->row_offset;
    a.dbg = static_cast<long long *>(s->d_debug);
    int rc;
    if (has_a) { rc = fill_net(a.net[0], actor_w, actor_io, s->depth, 1, s->action_dim, pair, embed_only); if (rc) return rc; }
    if (has_c) { rc = fill_net(a.net[1], critic_w, critic_io, s->depth, 0, s->action_dim, pair, embed_only); if (rc) return rc; }
    a.net_count = nets;
    a.net_first = has_a ? 0 : 1;
    const unsigned grid = (unsigned)(a.n_tiles * (pair ? 1 : a.net_count));
    auto launch = [&](auto kernel, int threads, int smem_bytes) -> int {
        const cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_bytes);
        if (e != cudaSuccess) { set_error("policy_step_kernel: smem %d: %s", smem_bytes, cudaGetErrorString(e)); return MARL_ECUDA; }
        kernel<<<grid, threads, smem_bytes, (cudaStream_t)stream>>>(a);
        return MARL_OK;
    };
    // one CTA per SM: 16 worker warps unless the env-grouped message path needs a whole 16-agent env per warp
    const bool pair8 = pair && s->N == 16 && s->O <= pf::OXY_CAP;       // 16-agent envs: a whole env per warp needs 8 worker warps
    const bool step8 = s->N == 16 && s->O <= pf::OXY_CAP;
    // the flags select a kernel instantiation (no runtime branch in the phases); flags = 0 is the default kernels
    auto dispatch = [&](auto fl) -> int {
        constexpr int FL = decltype(fl)::value;
        if (pair8) return launch(pf::policy_pair_kernel<8, false, FL>, (8 + 4) * 32, pf::MemPair::BYTES);
        if constexpr (FL == 0) {
            if (pair && getenv("MARL_POLICY_PROFILE")) return launch(pf::policy_pair_kernel<16, true, 0>, (16 + 4) * 32, pf::MemPair::BYTES);
        }
        if (pair) return launch(pf::policy_pair_kernel<16, false, FL>, (16 + 4) * 32, pf::MemPair::BYTES);
        if (!step8) return launch(pf::policy_step_kernel<16, FL>, pf::Lay<16>::THREADS, pf::SMEM_BYTES);
        return launch(pf::policy_step_kernel<8, FL>, pf::Lay<8>::THREADS, pf::SMEM_BYTES);
    };
    switch (s->flags) {
    case 0: rc = dispatch(std::integral_constant<int, 0>{}); break;
    case MARL_POLICY_STATE_F32: rc = dispatch(std::integral_constant<int, MARL_POLICY_STATE_F32>{}); break;
    case MARL_POLICY_EMBED_ONLY: rc = dispatch(std::integral_constant<int, MARL_POLICY_EMBED_ONLY>{}); break;
    default: rc = dispatch(std::integral_constant<int, MARL_POLICY_STATE_F32 | MARL_POLICY_EMBED_ONLY>{}); break;
    }
    if (rc) return rc;
    return check_launch("policy_step_kernel");
}

extern "C" int marl_policy_rollout_step(const marl_policy_step *s, const marl_dhgn_weights *actor_w, const marl_policy_net_io *actor_io,
                                        const marl_dhgn_weights *critic_w, const marl_policy_net_io *critic_io, void *stream)
{
    return policy_rollout_step(s, actor_w, actor_io, critic_w, critic_io, nullptr, stream);
}

extern "C" int marl_policy_rollout_step_dseed(const marl_policy_step *s, const marl_dhgn_weights *actor_w, const marl_policy_net_io *actor_io,
                                              const marl_dhgn_weights *critic_w, const marl_policy_net_io *critic_io, const uint64_t *d_seed,
                                              void *stream)
{
    MARL_REQUIRE(d_seed != nullptr, "marl_policy_rollout_step_dseed: d_seed is NULL");
    return policy_rollout_step(s, actor_w, actor_io, critic_w, critic_io, d_seed, stream);
}

// policy_kernels.cu — kernel family 5: the non-GEMM parts of the DHGN actor/critic forward and backward
// (DHGN/mappo_parallel.py:116-545, 686-715), fp32.  The dense 128-wide layers are plain library GEMMs on the host
// side; everything that is pairwise / sparse / pointwise is fused here so that no [.,N,N,8], [.,N,O,4] or dense 0/1
// adjacency tensor is ever materialised:
//   * message + L1-normalised aggregation for the three relations straight from the bit-packed adjacency,
//   * FCRA neighbour averaging of the history embeddings,
//   * GRU cell pointwise forward / backward,
//   * actor softmax/Categorical + critic head + PPO-clip and clipped value loss, forward and backward in one pass,
//   * global-norm gradient clipping and Adam on flat arenas.
// One warp per (sample, agent) row; lane l owns channels l, l+32, ... (E = 32*CPL), so every [.,E] access is a
// coalesced 128-byte line per CPL.
#include "common.cuh"
#include "msg_args.cuh"
#include <type_traits>

namespace marl {

static constexpr int kPolThreads = 128;   // 4 warps

template <int CPL>
struct MsgWeights {   // per-lane slices of MSG_layers.{0,1,2} (weights [E,8], [E,4], [E,4] row-major) and biases
    float w0[CPL][8], w1[CPL][4], w2[CPL][4], b0[CPL], b1[CPL], b2[CPL];
    __device__ __forceinline__ void load(const float *W0, const float *b0p, const float *W1, const float *b1p,
                                         const float *W2, const float *b2p, int lane)
    {
#pragma unroll
        for (int q = 0; q < CPL; ++q) {
            const int c = lane + 32 * q;
#pragma unroll
            for (int k = 0; k < 8; ++k) w0[q][k] = W0[c * 8 + k];
#pragma unroll
            for (int k = 0; k < 4; ++k) { w1[q][k] = W1[c * 4 + k]; w2[q][k] = W2[c * 4 + k]; }
            b0[q] = b0p[c]; b1[q] = b1p[c]; b2[q] = b2p[c];
        }
    }
};



// torch's F.linear accumulates k = 0..K-1 in order; keep that order (fp32 sums are order sensitive)
__device__ __forceinline__ float dot4(const float (&w)[4], float a0, float a1, float a2, float a3, float b)
{
    return fmaf(w[3], a3, fmaf(w[2], a2, fmaf(w[1], a1, fmaf(w[0], a0, 0.f)))) + b;
}

// ---- DHGN.message + mean aggregation (mappo_parallel.py:256-281, 323-348), forward ---------------------------
// agg[s,i,r,:] = sum_j w_ij ReLU(W_r a_ij + b_r),  w = adj / max(sum|adj|, 1e-12)   (F.normalize p=1)
template <int CPL>
__global__ void __launch_bounds__(kPolThreads)
msg_agg_fwd_kernel(MsgArgs a, const float *__restrict__ W0, const float *__restrict__ b0, const float *__restrict__ W1,
                   const float *__restrict__ b1, const float *__restrict__ W2, const float *__restrict__ b2,
                   float *__restrict__ agg /* [S,N,3,E] */)
{
    const int lane = threadIdx.x & 31, E = 32 * CPL;
    const int64_t row = (int64_t)blockIdx.x * (kPolThreads / 32) + (threadIdx.x >> 5);
    if (row >= (int64_t)a.S * a.N) return;
    MsgWeights<CPL> w;
    w.load(W0, b0, W1, b1, W2, b2, lane);
    const int64_t s = row / a.N;
    const int i = (int)(row - s * a.N);
    const float4 pi = *reinterpret_cast<const float4 *>(a.p + row * 4);
    const float4 ev = *reinterpret_cast<const float4 *>(a.e + s * 4);
    const float dex = pi.x - ev.x, dey = pi.y - ev.y, dez = pi.z - ev.z, dew = pi.w - ev.w;
    float acc0[CPL], acc2[CPL], m1[CPL];
#pragma unroll
    for (int q = 0; q < CPL; ++q) { acc0[q] = 0.f; acc2[q] = 0.f; }
    // relation 0: pursuer-pursuer, attribute [p_i - p_j, p_i - e]
    int cnt0 = 0;
    for (int j = 0; j < a.N; ++j) {
        const bool on = a.all_ones || ((a.p_adj[row * a.NW + (j >> 5)] >> (j & 31)) & 1u);
        if (!on) continue;
        ++cnt0;
        const float4 pj = *reinterpret_cast<const float4 *>(a.p + (s * a.N + j) * 4);
        const float d0 = pi.x - pj.x, d1 = pi.y - pj.y, d2 = pi.z - pj.z, d3 = pi.w - pj.w;
#pragma unroll
        for (int q = 0; q < CPL; ++q) {
            float v = fmaf(w.w0[q][3], d3, fmaf(w.w0[q][2], d2, fmaf(w.w0[q][1], d1, fmaf(w.w0[q][0], d0, 0.f))));
            v = fmaf(w.w0[q][7], dew, fmaf(w.w0[q][6], dez, fmaf(w.w0[q][5], dey, fmaf(w.w0[q][4], dex, v)))) + w.b0[q];
            acc0[q] += fmaxf(v, 0.f);
        }
    }
    // relation 1: pursuer-evader
    const float e_on = a.all_ones ? 1.f : (float)a.e_adj[row];
#pragma unroll
    for (int q = 0; q < CPL; ++q) m1[q] = e_on * fmaxf(dot4(w.w1[q], dex, dey, dez, dew, w.b1[q]), 0.f);
    // relation 2: pursuer-obstacle, attribute p_i - (ox, oy, 0, 0)
    const int ob = a.o_index[s];
    const float *oxy = a.oxy + (int64_t)ob * a.O * 2;
    int cnt2 = 0;
    if (a.all_ones) {
        const int n = a.o_count[ob];
        cnt2 = n;
        for (int k = 0; k < n; ++k) {
            const float2 o = *reinterpret_cast<const float2 *>(oxy + 2 * k);
            const float d0 = pi.x - o.x, d1 = pi.y - o.y;
#pragma unroll
            for (int q = 0; q < CPL; ++q) acc2[q] += fmaxf(dot4(w.w2[q], d0, d1, pi.z, pi.w, w.b2[q]), 0.f);
        }
    } else {
        for (int wd = 0; wd < a.OW; ++wd) {
            uint32_t bits = a.o_adj[row * a.OW + wd];
            cnt2 += __popc(bits);
            while (bits) {
                const int k = wd * 32 + __ffs(bits) - 1;
                bits &= bits - 1;
                const float2 o = *reinterpret_cast<const float2 *>(oxy + 2 * k);
                const float d0 = pi.x - o.x, d1 = pi.y - o.y;
#pragma unroll
                for (int q = 0; q < CPL; ++q) acc2[q] += fmaxf(dot4(w.w2[q], d0, d1, pi.z, pi.w, w.b2[q]), 0.f);
            }
        }
    }
    const float n0 = 1.f / fmaxf((float)cnt0, 1e-12f), n2 = 1.f / fmaxf((float)cnt2, 1e-12f);
    float *out = agg + row * 3 * E;
#pragma unroll
    for (int q = 0; q < CPL; ++q) {
        const int c = lane + 32 * q;
        out[c] = cnt0 ? acc0[q] * n0 : 0.f;
        out[E + c] = m1[q];
        out[2 * E + c] = cnt2 ? acc2[q] * n2 : 0.f;
    }
}

// ---- backward w.r.t. the three message layers (inputs are data: no input gradient) ---------------------------
// Pre-activations are recomputed; each warp walks many rows and keeps its dW slices in registers, then the CTA
// reduces through shared memory and writes its 19 x E row of partial sums to ws[blockIdx.x], reduced in a fixed order by
// msg_partials_reduce_kernel.
template <int CPL>
__global__ void __launch_bounds__(kPolThreads)
msg_agg_bwd_kernel(MsgArgs a, const float *__restrict__ W0, const float *__restrict__ b0, const float *__restrict__ W1,
                   const float *__restrict__ b1, const float *__restrict__ W2, const float *__restrict__ b2,
                   const float *__restrict__ d_agg, float *__restrict__ ws)
{
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, E = 32 * CPL;
    MsgWeights<CPL> w;
    w.load(W0, b0, W1, b1, W2, b2, lane);
    float g0[CPL][9], g1[CPL][5], g2[CPL][5];
#pragma unroll
    for (int q = 0; q < CPL; ++q) {
#pragma unroll
        for (int k = 0; k < 9; ++k) g0[q][k] = 0.f;
#pragma unroll
        for (int k = 0; k < 5; ++k) { g1[q][k] = 0.f; g2[q][k] = 0.f; }
    }
    const int64_t rows = (int64_t)a.S * a.N, stride = (int64_t)gridDim.x * (kPolThreads / 32);
    for (int64_t row = (int64_t)blockIdx.x * (kPolThreads / 32) + warp; row < rows; row += stride) {
        const int64_t s = row / a.N;
        const float4 pi = *reinterpret_cast<const float4 *>(a.p + row * 4);
        const float4 ev = *reinterpret_cast<const float4 *>(a.e + s * 4);
        const float dex = pi.x - ev.x, dey = pi.y - ev.y, dez = pi.z - ev.z, dew = pi.w - ev.w;
        const float *dg = d_agg + row * 3 * E;
        float d0g[CPL], d1g[CPL], d2g[CPL];
        // normalisation weights need the neighbour counts first
        int cnt0 = 0, cnt2 = 0;
        if (a.all_ones) cnt0 = a.N;
        else for (int wd = 0; wd < a.NW; ++wd) cnt0 += __popc(a.p_adj[row * a.NW + wd]);
        const int ob = a.o_index[s];
        if (a.all_ones) cnt2 = a.o_count[ob];
        else for (int wd = 0; wd < a.OW; ++wd) cnt2 += __popc(a.o_adj[row * a.OW + wd]);
        const float n0 = cnt0 ? 1.f / fmaxf((float)cnt0, 1e-12f) : 0.f, n2 = cnt2 ? 1.f / fmaxf((float)cnt2, 1e-12f) : 0.f;
        const float e_on = a.all_ones ? 1.f : (float)a.e_adj[row];
#pragma unroll
        for (int q = 0; q < CPL; ++q) {
            const int c = lane + 32 * q;
            d0g[q] = dg[c] * n0;
            d1g[q] = dg[E + c] * e_on;
            d2g[q] = dg[2 * E + c] * n2;
        }
        for (int j = 0; j < a.N; ++j) {
            const bool on = a.all_ones || ((a.p_adj[row * a.NW + (j >> 5)] >> (j & 31)) & 1u);
            if (!on) continue;
            const float4 pj = *reinterpret_cast<const float4 *>(a.p + (s * a.N + j) * 4);
            const float d[8] = {pi.x - pj.x, pi.y - pj.y, pi.z - pj.z, pi.w - pj.w, dex, dey, dez, dew};
#pragma unroll
            for (int q = 0; q < CPL; ++q) {
                float v = fmaf(w.w0[q][3], d[3], fmaf(w.w0[q][2], d[2], fmaf(w.w0[q][1], d[1], fmaf(w.w0[q][0], d[0], 0.f))));
                v = fmaf(w.w0[q][7], d[7], fmaf(w.w0[q][6], d[6], fmaf(w.w0[q][5], d[5], fmaf(w.w0[q][4], d[4], v)))) + w.b0[q];
                const float g = v > 0.f ? d0g[q] : 0.f;
#pragma unroll
                for (int k = 0; k < 8; ++k) g0[q][k] = fmaf(g, d[k], g0[q][k]);
                g0[q][8] += g;
            }
        }
#pragma unroll
        for (int q = 0; q < CPL; ++q) {
            const float v = dot4(w.w1[q], dex, dey, dez, dew, w.b1[q]);
            const float g = v > 0.f ? d1g[q] : 0.f;
            g1[q][0] = fmaf(g, dex, g1[q][0]); g1[q][1] = fmaf(g, dey, g1[q][1]);
            g1[q][2] = fmaf(g, dez, g1[q][2]); g1[q][3] = fmaf(g, dew, g1[q][3]);
            g1[q][4] += g;
        }
        const float *oxy = a.oxy + (int64_t)ob * a.O * 2;
        auto obstacle = [&](int k) {
            const float2 o = *reinterpret_cast<const float2 *>(oxy + 2 * k);
            const float d0 = pi.x - o.x, d1 = pi.y - o.y;
#pragma unroll
            for (int q = 0; q < CPL; ++q) {
                const float v = dot4(w.w2[q], d0, d1, pi.z, pi.w, w.b2[q]);
                const float g = v > 0.f ? d2g[q] : 0.f;
                g2[q][0] = fmaf(g, d0, g2[q][0]); g2[q][1] = fmaf(g, d1, g2[q][1]);
                g2[q][2] = fmaf(g, pi.z, g2[q][2]); g2[q][3] = fmaf(g, pi.w, g2[q][3]);
                g2[q][4] += g;
            }
        };
        if (a.all_ones) {
            for (int k = 0; k < cnt2; ++k) obstacle(k);
        } else {
            for (int wd = 0; wd < a.OW; ++wd) {
                uint32_t bits = a.o_adj[row * a.OW + wd];
                while (bits) { obstacle(wd * 32 + __ffs(bits) - 1); bits &= bits - 1; }
            }
        }
    }
    // CTA reduction: [warps][19*E] in shared memory, then one partial per element
    extern __shared__ float s_red[];
    float *mine = s_red + warp * 19 * E;
#pragma unroll
    for (int q = 0; q < CPL; ++q) {
        const int c = lane + 32 * q;
#pragma unroll
        for (int k = 0; k < 9; ++k) mine[k * E + c] = g0[q][k];
#pragma unroll
        for (int k = 0; k < 5; ++k) { mine[(9 + k) * E + c] = g1[q][k]; mine[(14 + k) * E + c] = g2[q][k]; }
    }
    __syncthreads();
    for (int idx = threadIdx.x; idx < 19 * E; idx += kPolThreads) {
        float v = 0.f;
        for (int wv = 0; wv < kPolThreads / 32; ++wv) v += s_red[wv * 19 * E + idx];
        ws[(int64_t)blockIdx.x * 19 * E + idx] = v;
    }
}

// Fixed-order sum of the message backward's per-CTA partials (MsgPartials, msg_args.cuh).  A CTA owns 32 consecutive output
// elements of one row k (E is a multiple of 32): lane = element, so every load is one coalesced 128-byte line.  Warp w adds the
// partials of the CTAs in its contiguous range [w*blocks/W, (w+1)*blocks/W) in index order, then warp 0 adds the W warp sums in
// warp order.  The order depends only on `blocks`, never on timing.
constexpr int kReduceWarps = 16;
__global__ void __launch_bounds__(32 * kReduceWarps)
msg_partials_reduce_kernel(MsgPartials p, float *__restrict__ gW0, float *__restrict__ gb0, float *__restrict__ gW1,
                           float *__restrict__ gb1, float *__restrict__ gW2, float *__restrict__ gb2)
{
    __shared__ float s_sum[kReduceWarps][32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int idx = blockIdx.x * 32 + lane, k = idx / p.E, c = idx - k * p.E;
    const int r = k < 9 ? 0 : (k < 14 ? 1 : 2), kr = k - (r == 0 ? 0 : (r == 1 ? 9 : 14));
    const float *src = p.rel_base[r] + (int64_t)kr * p.E + c;
    const int64_t stride = p.rel_stride[r];
    const int b0 = (int)((int64_t)warp * p.blocks / kReduceWarps), b1 = (int)((int64_t)(warp + 1) * p.blocks / kReduceWarps);
    float acc = 0.f;
#pragma unroll 8
    for (int b = b0; b < b1; ++b) acc += __ldcg(src + b * stride);
    s_sum[warp][lane] = acc;
    __syncthreads();
    if (warp != 0) return;
    float v = 0.f;
#pragma unroll
    for (int w = 0; w < kReduceWarps; ++w) v += s_sum[w][lane];
    const int KW = r == 0 ? 8 : 4;
    float *gW = r == 0 ? gW0 : (r == 1 ? gW1 : gW2), *gb = r == 0 ? gb0 : (r == 1 ? gb1 : gb2);
    if (kr < KW) gW[c * KW + kr] += v;
    else gb[c] += v;
}

int launch_msg_partials_reduce(const MsgPartials &p, float *gW0, float *gb0, float *gW1, float *gb1, float *gW2, float *gb2,
                               cudaStream_t stream)
{
    msg_partials_reduce_kernel<<<19 * p.E / 32, 32 * kReduceWarps, 0, stream>>>(p, gW0, gb0, gW1, gb1, gW2, gb2);
    return check_launch("msg_partials_reduce_kernel");
}

// ---- FCRA neighbour averaging (mappo_parallel.py:204-233, the L1norm(adj) @ hist part) -------------------------
// out[s,i,:] = sum_j w_ij hist[s,j,:].  hist rows live at hist + (s*N+j)*hist_stride (floats), which lets the caller
// point straight into a [T+D,B,N,E] history arena.
template <int CPL>
__global__ void __launch_bounds__(kPolThreads)
fcra_agg_kernel(int S, int N, int NW, const float *__restrict__ hist, int64_t sample_stride, int64_t agent_stride,
                const uint32_t *__restrict__ p_adj, int all_ones, float *__restrict__ out)
{
    const int lane = threadIdx.x & 31, E = 32 * CPL;
    const int64_t row = (int64_t)blockIdx.x * (kPolThreads / 32) + (threadIdx.x >> 5);
    if (row >= (int64_t)S * N) return;
    const int64_t s = row / N;
    float acc[CPL];
#pragma unroll
    for (int q = 0; q < CPL; ++q) acc[q] = 0.f;
    int cnt = 0;
    for (int j = 0; j < N; ++j) {
        const bool on = all_ones || ((p_adj[row * NW + (j >> 5)] >> (j & 31)) & 1u);
        if (!on) continue;
        ++cnt;
        const float *h = hist + s * sample_stride + j * agent_stride;
#pragma unroll
        for (int q = 0; q < CPL; ++q) acc[q] += h[lane + 32 * q];
    }
    const float nrm = cnt ? 1.f / fmaxf((float)cnt, 1e-12f) : 0.f;
#pragma unroll
    for (int q = 0; q < CPL; ++q) out[row * E + lane + 32 * q] = acc[q] * nrm;
}

// ---- GRU cell pointwise (torch.nn.GRU gate order r, z, n) -----------------------------------------------------
__device__ __forceinline__ float sigmoidf_(float x) { return 1.f / (1.f + __expf(-x)); }

__global__ void __launch_bounds__(256)
gru_cell_fwd_kernel(int64_t R, int E, const float *__restrict__ gi, const float *__restrict__ gh,
                    const float *__restrict__ h_prev, float *__restrict__ h_new, float *__restrict__ save_r,
                    float *__restrict__ save_z, float *__restrict__ save_n, float *__restrict__ save_hn)
{
    const int64_t total = R * E;
    for (int64_t idx = (int64_t)blockIdx.x * 256 + threadIdx.x; idx < total; idx += (int64_t)gridDim.x * 256) {
        const int64_t r_ = idx / E;
        const int c = (int)(idx - r_ * E);
        const float *gir = gi + r_ * 3 * E, *ghr = gh + r_ * 3 * E;
        const float r = 1.f / (1.f + expf(-(gir[c] + ghr[c])));
        const float z = 1.f / (1.f + expf(-(gir[E + c] + ghr[E + c])));
        const float hn = ghr[2 * E + c];
        const float n = tanhf(gir[2 * E + c] + r * hn);
        const float hp = h_prev[idx];
        h_new[idx] = (1.f - z) * n + z * hp;
        if (save_r) { save_r[idx] = r; save_z[idx] = z; save_n[idx] = n; save_hn[idx] = hn; }
    }
}

__global__ void __launch_bounds__(256)
gru_cell_bwd_kernel(int64_t R, int E, const float *__restrict__ dh_new, const float *__restrict__ sr,
                    const float *__restrict__ sz, const float *__restrict__ sn, const float *__restrict__ shn,
                    const float *__restrict__ h_prev, float *__restrict__ d_gi, float *__restrict__ d_gh,
                    float *__restrict__ dh_prev /* = dh_new * z (the W_hh term is added by the caller's GEMM) */)
{
    const int64_t total = R * E;
    for (int64_t idx = (int64_t)blockIdx.x * 256 + threadIdx.x; idx < total; idx += (int64_t)gridDim.x * 256) {
        const int64_t r_ = idx / E;
        const int c = (int)(idx - r_ * E);
        const float dh = dh_new[idx], r = sr[idx], z = sz[idx], n = sn[idx], hn = shn[idx], hp = h_prev[idx];
        const float dn = dh * (1.f - z);
        const float dz = dh * (hp - n);
        const float dpn = dn * (1.f - n * n);
        const float dpz = dz * z * (1.f - z);
        const float dpr = dpn * hn * r * (1.f - r);
        float *gi = d_gi + r_ * 3 * E, *gh = d_gh + r_ * 3 * E;
        gi[c] = dpr; gi[E + c] = dpz; gi[2 * E + c] = dpn;
        gh[c] = dpr; gh[E + c] = dpz; gh[2 * E + c] = dpn * r;
        dh_prev[idx] = dh * z;
    }
}

// ---- heads + PPO losses, forward and backward in one pass (mappo_parallel.py:437,446-456,526,692-706) ---------
struct HeadArgs {
    int64_t R;
    int E, A;                    // A = action_dim (9)
    const float *feat_a, *feat_c;   // [R,E] GRU outputs
    const float *Wa, *ba;        // [A,E], [A]
    const float *wc_eff, *bc;    // [E] spectral-normalised critic row, [1]
    const float *action;         // [R] float32 action ids (buffer['a_n'])
    const float *old_logp, *adv, *v_old, *v_target, *active;   // [R]
    float eps, ent_coef;
    float *logp, *entropy, *value;            // [R] outputs (also what tests compare)
    float *d_logits;             // [R,A]  d(actor_loss_sum)/d logits   (divide by sum(active) afterwards)
    float *d_value;              // [R]    d(critic_loss_sum)/d value
    float *sums;                 // [3] += {sum actor_term*active, sum critic_term*active, sum active}
    float *partials;             // [gridDim.x][3] per-CTA sums, reduced into sums by ppo_sums_reduce_kernel
};

// Each CTA writes its three sums to h.partials[blockIdx.x].
template <int CPL, int A>
__global__ void __launch_bounds__(kPolThreads)
ppo_head_kernel(HeadArgs h)
{
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, E = 32 * CPL;
    __shared__ float s_part[kPolThreads / 32][3];
    float wa[A][CPL], wc[CPL];
#pragma unroll
    for (int q = 0; q < CPL; ++q) {
        wc[q] = h.wc_eff[lane + 32 * q];
#pragma unroll
        for (int k = 0; k < A; ++k) wa[k][q] = h.Wa[k * E + lane + 32 * q];
    }
    float part[3] = {0.f, 0.f, 0.f};
    const int64_t stride = (int64_t)gridDim.x * (kPolThreads / 32);
    for (int64_t r = (int64_t)blockIdx.x * (kPolThreads / 32) + warp; r < h.R; r += stride) {
        float fa[CPL], fc[CPL];
#pragma unroll
        for (int q = 0; q < CPL; ++q) { fa[q] = h.feat_a[r * E + lane + 32 * q]; fc[q] = h.feat_c[r * E + lane + 32 * q]; }
        float z[A], v = 0.f;
#pragma unroll
        for (int k = 0; k < A; ++k) {
            float acc = 0.f;
#pragma unroll
            for (int q = 0; q < CPL; ++q) acc = fmaf(wa[k][q], fa[q], acc);
            z[k] = acc;
        }
#pragma unroll
        for (int q = 0; q < CPL; ++q) v = fmaf(wc[q], fc[q], v);
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
#pragma unroll
            for (int k = 0; k < A; ++k) z[k] += __shfl_xor_sync(0xffffffffu, z[k], o);
            v += __shfl_xor_sync(0xffffffffu, v, o);
        }
        // every lane now holds the full logits / value of this row; the scalar tail is done redundantly
        float mx = -INFINITY;
#pragma unroll
        for (int k = 0; k < A; ++k) { z[k] += h.ba[k]; mx = fmaxf(mx, z[k]); }
        v += h.bc[0];
        float sm[A], den = 0.f;
#pragma unroll
        for (int k = 0; k < A; ++k) { sm[k] = expf(z[k] - mx); den += sm[k]; }
        float psum = 0.f;
#pragma unroll
        for (int k = 0; k < A; ++k) { sm[k] = sm[k] / den; psum += sm[k]; }
        // Categorical(probs=prob): probs renormalised, logits = log(clamp(probs, eps, 1-eps)) (torch.distributions)
        const float ceps = 1.1920928955078125e-07f;
        float lp[A], msk[A], H = 0.f, sml = 0.f;
#pragma unroll
        for (int k = 0; k < A; ++k) {
            const float q_ = sm[k] / psum;
            const float pc = fminf(fmaxf(q_, ceps), 1.f - ceps);
            msk[k] = (q_ >= ceps && q_ <= 1.f - ceps) ? 1.f : 0.f;
            lp[k] = logf(pc);
            H -= lp[k] * q_;
            sml += q_ * (lp[k] + msk[k]);
            sm[k] = q_;
        }
        const int act = (int)h.action[r];
        float lpa = 0.f, ma = 0.f;
#pragma unroll
        for (int k = 0; k < A; ++k) if (k == act) { lpa = lp[k]; ma = msk[k]; }
        const float adv = h.adv[r], on = h.active[r];
        const float ratio = expf(lpa - h.old_logp[r]);
        const float clamped = fminf(fmaxf(ratio, 1.f - h.eps), 1.f + h.eps);
        const float s1 = ratio * adv, s2 = clamped * adv;
        const float a_term = -fminf(s1, s2) - h.ent_coef * H;
        const bool inside = ratio >= 1.f - h.eps && ratio <= 1.f + h.eps;
        // d min(s1,s2)/d ratio: torch splits ties evenly; inside the clip range both branches carry adv
        float dmin = 0.f;
        if (inside) dmin = adv;
        else if (s1 < s2) dmin = adv;
        else if (s1 == s2) dmin = 0.5f * adv;
        const float dlogp = -dmin * ratio * on;           // d(actor term * active)/d logp(a)
        const float vt = h.v_target[r], eo = v - vt;
        float c_term = eo * eo, dval = 2.f * eo * on;     // use_value_clip = False (:703-704): (values_now - v_target)^2
        if (h.v_old) {                                    // Trick: value clip (:699-702)
            const float vo = h.v_old[r];
            const float dv = v - vo;
            const float ec = fminf(fmaxf(dv, -h.eps), h.eps) + vo - vt;
            const float c1 = ec * ec, c2 = eo * eo;
            c_term = fmaxf(c1, c2);
            const float gc = (dv >= -h.eps && dv <= h.eps) ? 2.f * ec : 0.f, go = 2.f * eo;
            dval = (c1 > c2 ? gc : (c1 < c2 ? go : 0.5f * (gc + go))) * on;
        }
        if (lane == 0) {
            h.logp[r] = lpa; h.entropy[r] = H; h.value[r] = v; h.d_value[r] = dval;
            part[0] += a_term * on; part[1] += c_term * on; part[2] += on;
        }
        if (lane < A) {
            // d logp(a)/dz_j = m_a (delta_aj - s_j);  dH/dz_j = -s_j[(lp_j + m_j) - sum_k s_k (lp_k + m_k)]
            float sj = 0.f, lj = 0.f, mj = 0.f;
#pragma unroll
            for (int k = 0; k < A; ++k) if (k == lane) { sj = sm[k]; lj = lp[k]; mj = msk[k]; }
            const float dlp = ma * ((lane == act ? 1.f : 0.f) - sj);
            const float dH = -sj * ((lj + mj) - sml);
            h.d_logits[r * A + lane] = dlogp * dlp - h.ent_coef * on * dH;
        }
    }
    if (lane == 0) { s_part[warp][0] = part[0]; s_part[warp][1] = part[1]; s_part[warp][2] = part[2]; }
    __syncthreads();
    if (threadIdx.x < 3) {
        float v = 0.f;
        for (int wv = 0; wv < kPolThreads / 32; ++wv) v += s_part[wv][threadIdx.x];
        h.partials[blockIdx.x * 3 + threadIdx.x] = v;
    }
}

// sums[j] += the ppo_head_kernel partials j of all CTAs: thread t adds CTAs t, t + 256, ... in order, then a fixed tree.
__global__ void __launch_bounds__(256)
ppo_sums_reduce_kernel(int blocks, const float *__restrict__ partials, float *__restrict__ sums)
{
    __shared__ float s[3][256];
    float acc[3] = {0.f, 0.f, 0.f};
    for (int b = threadIdx.x; b < blocks; b += 256)
#pragma unroll
        for (int j = 0; j < 3; ++j) acc[j] += partials[b * 3 + j];
#pragma unroll
    for (int j = 0; j < 3; ++j) s[j][threadIdx.x] = acc[j];
    __syncthreads();
    for (int o = 128; o > 0; o >>= 1) {
        if (threadIdx.x < o)
#pragma unroll
            for (int j = 0; j < 3; ++j) s[j][threadIdx.x] += s[j][threadIdx.x + o];
        __syncthreads();
    }
    if (threadIdx.x < 3) sums[threadIdx.x] += s[threadIdx.x][0];
}

// Rollout-time actor head: softmax -> Categorical sample (counter RNG) or argmax -> log-prob; critic value.
template <int CPL, int A>
__global__ void __launch_bounds__(kPolThreads)
act_head_kernel(int64_t R, const float *__restrict__ feat_a, const float *__restrict__ feat_c,
                const float *__restrict__ Wa, const float *__restrict__ ba, const float *__restrict__ wc_eff,
                const float *__restrict__ bc, uint64_t seed, int t, int deterministic, int32_t *__restrict__ action,
                float *__restrict__ action_f, float *__restrict__ logp, float *__restrict__ value)
{
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, E = 32 * CPL;
    const int64_t r = (int64_t)blockIdx.x * (kPolThreads / 32) + warp;
    if (r >= R) return;
    float z[A], v = 0.f;
#pragma unroll
    for (int k = 0; k < A; ++k) z[k] = 0.f;
#pragma unroll
    for (int q = 0; q < CPL; ++q) {
        const float fa = feat_a[r * E + lane + 32 * q];
        if (feat_c) v = fmaf(wc_eff[lane + 32 * q], feat_c[r * E + lane + 32 * q], v);
#pragma unroll
        for (int k = 0; k < A; ++k) z[k] = fmaf(Wa[k * E + lane + 32 * q], fa, z[k]);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
#pragma unroll
        for (int k = 0; k < A; ++k) z[k] += __shfl_xor_sync(0xffffffffu, z[k], o);
        v += __shfl_xor_sync(0xffffffffu, v, o);
    }
    if (lane != 0) return;
    float mx = -INFINITY;
#pragma unroll
    for (int k = 0; k < A; ++k) { z[k] += ba[k]; mx = fmaxf(mx, z[k]); }
    float sm[A], den = 0.f;
#pragma unroll
    for (int k = 0; k < A; ++k) { sm[k] = expf(z[k] - mx); den += sm[k]; }
    float psum = 0.f;
#pragma unroll
    for (int k = 0; k < A; ++k) { sm[k] /= den; psum += sm[k]; }
    int a = 0;
    if (deterministic) {
        float best = -1.f;
#pragma unroll
        for (int k = 0; k < A; ++k) if (sm[k] > best) { best = sm[k]; a = k; }   // first maximum, like argmax
    } else {
        // inverse-CDF sampling with a counter-based uniform in [0,1) (the reference uses torch's CPU generator)
        const uint64_t hsh = splitmix64(seed ^ splitmix64((uint64_t)r * 0x100000001B3ull + (uint64_t)t));
        const float u = (float)(hsh >> 40) * (1.0f / 16777216.0f) * psum;
        float c = 0.f;
        a = A - 1;
#pragma unroll
        for (int k = 0; k < A; ++k) { c += sm[k]; if (u < c) { a = k; break; } }
    }
    const float ceps = 1.1920928955078125e-07f;
    float lpa = 0.f;
#pragma unroll
    for (int k = 0; k < A; ++k) if (k == a) lpa = logf(fminf(fmaxf(sm[k] / psum, ceps), 1.f - ceps));
    action[r] = a;
    if (action_f) action_f[r] = (float)a;
    if (logp) logp[r] = lpa;
    if (value) value[r] = v + bc[0];
}

// ---- global-norm clip + Adam on flat fp32 arenas -----------------------------------------------------------------
__global__ void __launch_bounds__(256)
sumsq_kernel(int64_t n, const float *__restrict__ g, double *__restrict__ partial)
{
    double acc = 0.0;
    for (int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x; i < n; i += (int64_t)gridDim.x * 256) acc += (double)g[i] * (double)g[i];
    __shared__ double s[256];
    s[threadIdx.x] = acc;
    __syncthreads();
    for (int o = 128; o > 0; o >>= 1) {
        if (threadIdx.x < o) s[threadIdx.x] += s[threadIdx.x + o];
        __syncthreads();
    }
    if (threadIdx.x == 0) partial[blockIdx.x] = s[0];
}

// torch.nn.utils.clip_grad_norm_: coef = max_norm / (total_norm + 1e-6), clamped to 1; every block re-reduces the
// partials in the same order, so the scale is deterministic.
__global__ void __launch_bounds__(256)
clip_scale_kernel(int64_t n, float *__restrict__ g, const double *__restrict__ partial, int n_partial, float max_norm,
                  float *__restrict__ total_norm_out)
{
    __shared__ float s_coef;
    if (threadIdx.x == 0) {
        double t = 0.0;
        for (int i = 0; i < n_partial; ++i) t += partial[i];
        const float norm = (float)sqrt(t);
        float coef = max_norm / (norm + 1e-6f);
        s_coef = coef < 1.f ? coef : 1.f;
        if (blockIdx.x == 0 && total_norm_out) *total_norm_out = norm;
    }
    __syncthreads();
    const float coef = s_coef;
    if (coef >= 1.f) return;
    for (int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x; i < n; i += (int64_t)gridDim.x * 256) g[i] *= coef;
}

// torch.optim.Adam (no amsgrad, no weight decay): m,v EMA; step_size = lr / (1 - b1^t); denom = sqrt(v)/sqrt(1-b2^t) + eps
__global__ void __launch_bounds__(256)
adam_kernel(int64_t n, float *__restrict__ p, const float *__restrict__ g, float *__restrict__ m, float *__restrict__ v,
            float lr, float b1, float b2, float eps, float bc1, float bc2_sqrt)
{
    const float step_size = lr / bc1;
    for (int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x; i < n; i += (int64_t)gridDim.x * 256) {
        const float gi = g[i];
        const float mi = m[i] + (gi - m[i]) * (1.f - b1);          // exp_avg.lerp_(grad, 1 - beta1)
        const float vi = v[i] * b2 + (1.f - b2) * gi * gi;           // exp_avg_sq.mul_(beta2).addcmul_(grad, grad, 1-beta2)
        m[i] = mi;
        v[i] = vi;
        const float denom = sqrtf(vi) / bc2_sqrt + eps;
        p[i] = p[i] - step_size * (mi / denom);
    }
}

template <typename F>
static int dispatch_cpl(int E, F &&f)
{
    if (E == 32) return f(std::integral_constant<int, 1>{});
    if (E == 64) return f(std::integral_constant<int, 2>{});
    if (E == 128) return f(std::integral_constant<int, 4>{});
    set_error("embedding_dim=%d unsupported (32, 64 or 128)", E);
    return MARL_EUNSUPPORTED;
}

static inline int grid_for_rows(int64_t rows) { return (int)((rows + kPolThreads / 32 - 1) / (kPolThreads / 32)); }

}  // namespace marl

using namespace marl;

#define MSG_ARGS_DECL                                                                                              \
    int32_t S, int32_t N, int32_t O, int32_t E, const float *d_p, const float *d_e, const float *d_oxy,           \
        const int32_t *d_o_index, const int32_t *d_o_count, const uint32_t *d_p_adj_bits, const uint8_t *d_e_adj, \
        const uint32_t *d_o_adj_bits, int32_t all_ones

static int fill_msg_args(MsgArgs &a, MSG_ARGS_DECL)
{
    MARL_REQUIRE(S > 0 && N > 0 && N <= MARL_MAX_AGENTS && O > 0, "dhgn_message: S=%d N=%d O=%d", S, N, O);
    MARL_REQUIRE(d_p && d_e && d_oxy && d_o_index && d_o_count, "dhgn_message: null pointer");
    MARL_REQUIRE(all_ones || (d_p_adj_bits && d_e_adj && d_o_adj_bits), "dhgn_message: adjacency missing");
    a.S = S; a.N = N; a.O = O; a.NW = (N + 31) / 32; a.OW = (O + 31) / 32;
    a.p = d_p; a.e = d_e; a.oxy = d_oxy; a.o_index = d_o_index; a.o_count = d_o_count;
    a.p_adj = d_p_adj_bits; a.e_adj = d_e_adj; a.o_adj = d_o_adj_bits; a.all_ones = all_ones;
    (void)E;
    return MARL_OK;
}

extern "C" int marl_dhgn_message_fwd(MSG_ARGS_DECL, const float *d_W0, const float *d_b0, const float *d_W1,
                                     const float *d_b1, const float *d_W2, const float *d_b2, float *d_agg, void *stream)
{
    MsgArgs a;
    int rc = fill_msg_args(a, S, N, O, E, d_p, d_e, d_oxy, d_o_index, d_o_count, d_p_adj_bits, d_e_adj, d_o_adj_bits, all_ones);
    if (rc) return rc;
    MARL_REQUIRE(d_W0 && d_b0 && d_W1 && d_b1 && d_W2 && d_b2 && d_agg, "marl_dhgn_message_fwd: null pointer");
    if (msg_grouped_supported(a, E)) return launch_msg_fwd_grouped(a, d_W0, d_b0, d_W1, d_b1, d_W2, d_b2, d_agg, (cudaStream_t)stream);
    return dispatch_cpl(E, [&](auto C_) -> int {
        constexpr int CPL = decltype(C_)::value;
        msg_agg_fwd_kernel<CPL><<<grid_for_rows((int64_t)S * N), kPolThreads, 0, (cudaStream_t)stream>>>(
            a, d_W0, d_b0, d_W1, d_b1, d_W2, d_b2, d_agg);
        return check_launch("msg_agg_fwd_kernel");
    });
}

#define MSG_BWD_DECL                                                                                                            \
    MSG_ARGS_DECL, const float *d_W0, const float *d_b0, const float *d_W1, const float *d_b1, const float *d_W2, const float *d_b2, \
        const float *d_grad_agg, float *d_gW0, float *d_gb0, float *d_gW1, float *d_gb1, float *d_gW2, float *d_gb2

static bool supported_width(int E) { return E == 32 || E == 64 || E == 128; }

extern "C" int64_t marl_dhgn_message_bwd_workspace_bytes(int32_t N, int32_t O, int32_t E)
{
    if (N <= 0 || N > MARL_MAX_AGENTS || O <= 0 || !supported_width(E)) return -1;
    MsgArgs a{};
    a.N = N; a.O = O; a.NW = (N + 31) / 32; a.OW = (O + 31) / 32;
    const int64_t ctas = msg_grouped_supported(a, E) ? kMsgBwdGroupedMaxCTAs : kMsgBwdRowMaxCTAs;
    return ctas * 19 * E * (int64_t)sizeof(float);
}

extern "C" int marl_dhgn_message_bwd_det(MSG_BWD_DECL, void *d_workspace, void *stream)
{
    MARL_REQUIRE(supported_width(E), "marl_dhgn_message_bwd_det: E=%d (32, 64 or 128)", E);
    MARL_REQUIRE(d_workspace, "marl_dhgn_message_bwd_det: null workspace");
    MsgArgs a;
    int rc = fill_msg_args(a, S, N, O, E, d_p, d_e, d_oxy, d_o_index, d_o_count, d_p_adj_bits, d_e_adj, d_o_adj_bits, all_ones);
    if (rc) return rc;
    MARL_REQUIRE(d_W0 && d_b0 && d_W1 && d_b1 && d_W2 && d_b2 && d_grad_agg && d_gW0 && d_gb0 && d_gW1 && d_gb1 && d_gW2 && d_gb2,
                 "marl_dhgn_message_bwd_det: null pointer");
    float *d_ws = static_cast<float *>(d_workspace);
    if (msg_grouped_supported(a, E))
        return launch_msg_bwd_grouped(a, d_W0, d_b0, d_W1, d_b1, d_W2, d_b2, d_grad_agg, d_gW0, d_gb0, d_gW1, d_gb1, d_gW2, d_gb2, d_ws,
                                      (cudaStream_t)stream);
    return dispatch_cpl(E, [&](auto C_) -> int {
        constexpr int CPL = decltype(C_)::value;
        int blocks = grid_for_rows((int64_t)S * N);
        if (blocks > kMsgBwdRowMaxCTAs) blocks = kMsgBwdRowMaxCTAs;   // persistent: fewer, longer warps -> fewer partials
        const size_t smem = sizeof(float) * (kPolThreads / 32) * 19 * E;
        msg_agg_bwd_kernel<CPL><<<blocks, kPolThreads, smem, (cudaStream_t)stream>>>(a, d_W0, d_b0, d_W1, d_b1, d_W2, d_b2,
                                                                                     d_grad_agg, d_ws);
        int rc2 = check_launch("msg_agg_bwd_kernel");
        if (rc2) return rc2;
        MsgPartials p;
        for (int r = 0; r < 3; ++r) { p.rel_base[r] = d_ws + (r == 0 ? 0 : (r == 1 ? 9 : 14)) * E; p.rel_stride[r] = 19 * E; }
        p.blocks = blocks; p.E = E;
        return launch_msg_partials_reduce(p, d_gW0, d_gb0, d_gW1, d_gb1, d_gW2, d_gb2, (cudaStream_t)stream);
    });
}

extern "C" int marl_fcra_agg(int32_t S, int32_t N, int32_t E, const float *d_hist, int64_t sample_stride,
                             int64_t agent_stride, const uint32_t *d_p_adj_bits, int32_t all_ones, float *d_out,
                             void *stream)
{
    MARL_REQUIRE(S > 0 && N > 0 && d_hist && d_out && (all_ones || d_p_adj_bits), "marl_fcra_agg: bad argument");
    return dispatch_cpl(E, [&](auto C_) -> int {
        constexpr int CPL = decltype(C_)::value;
        fcra_agg_kernel<CPL><<<grid_for_rows((int64_t)S * N), kPolThreads, 0, (cudaStream_t)stream>>>(
            S, N, (N + 31) / 32, d_hist, sample_stride, agent_stride, d_p_adj_bits, all_ones, d_out);
        return check_launch("fcra_agg_kernel");
    });
}

static inline int blocks_1d(int64_t n)
{
    int64_t b = (n + 255) / 256;
    return (int)(b > 148 * 8 ? 148 * 8 : (b < 1 ? 1 : b));
}

extern "C" int marl_gru_cell_fwd(int64_t R, int32_t E, const float *d_gi, const float *d_gh, const float *d_h_prev,
                                 float *d_h_new, float *d_save_r, float *d_save_z, float *d_save_n, float *d_save_hn,
                                 void *stream)
{
    MARL_REQUIRE(R > 0 && E > 0 && d_gi && d_gh && d_h_prev && d_h_new, "marl_gru_cell_fwd: bad argument");
    MARL_REQUIRE(!d_save_r || (d_save_z && d_save_n && d_save_hn), "marl_gru_cell_fwd: partial save buffers");
    gru_cell_fwd_kernel<<<blocks_1d(R * E), 256, 0, (cudaStream_t)stream>>>(R, E, d_gi, d_gh, d_h_prev, d_h_new, d_save_r,
                                                                            d_save_z, d_save_n, d_save_hn);
    return check_launch("gru_cell_fwd_kernel");
}

extern "C" int marl_gru_cell_bwd(int64_t R, int32_t E, const float *d_dh_new, const float *d_save_r,
                                 const float *d_save_z, const float *d_save_n, const float *d_save_hn,
                                 const float *d_h_prev, float *d_dgi, float *d_dgh, float *d_dh_prev, void *stream)
{
    MARL_REQUIRE(R > 0 && E > 0 && d_dh_new && d_save_r && d_save_z && d_save_n && d_save_hn && d_h_prev && d_dgi && d_dgh && d_dh_prev,
                 "marl_gru_cell_bwd: bad argument");
    gru_cell_bwd_kernel<<<blocks_1d(R * E), 256, 0, (cudaStream_t)stream>>>(R, E, d_dh_new, d_save_r, d_save_z, d_save_n,
                                                                            d_save_hn, d_h_prev, d_dgi, d_dgh, d_dh_prev);
    return check_launch("gru_cell_bwd_kernel");
}

#define PPO_HEAD_DECL                                                                                                       \
    int64_t R, int32_t E, int32_t A, const float *d_feat_a, const float *d_feat_c, const float *d_Wa, const float *d_ba,     \
        const float *d_wc_eff, const float *d_bc, const float *d_action, const float *d_old_logp, const float *d_adv,       \
        const float *d_v_old, const float *d_v_target, const float *d_active, float eps, float ent_coef, float *d_logp,     \
        float *d_entropy, float *d_value, float *d_dlogits, float *d_dvalue, float *d_sums

static inline int ppo_head_blocks(int64_t R)
{
    const int64_t blocks = (R + kPolThreads / 32 - 1) / (kPolThreads / 32);
    return (int)(blocks > 148 * 8 ? 148 * 8 : blocks);
}

extern "C" int64_t marl_ppo_head_workspace_bytes(int64_t R)
{
    return R > 0 ? (int64_t)ppo_head_blocks(R) * 3 * (int64_t)sizeof(float) : -1;
}

extern "C" int marl_ppo_head_det(PPO_HEAD_DECL, void *d_workspace, void *stream)
{
    MARL_REQUIRE(supported_width(E), "marl_ppo_head_det: E=%d (32, 64 or 128)", E);
    MARL_REQUIRE(d_workspace, "marl_ppo_head_det: null workspace");
    MARL_REQUIRE(R > 0 && A == MARL_NUM_ACTIONS, "marl_ppo_head_det: R=%lld A=%d (action_dim must be %d)", (long long)R, A,
                 MARL_NUM_ACTIONS);
    MARL_REQUIRE(d_feat_a && d_feat_c && d_Wa && d_ba && d_wc_eff && d_bc && d_action && d_old_logp && d_adv &&
                     d_v_target && d_active && d_logp && d_entropy && d_value && d_dlogits && d_dvalue && d_sums,
                 "marl_ppo_head_det: null pointer");
    float *d_ws = static_cast<float *>(d_workspace);
    HeadArgs h;
    h.R = R; h.E = E; h.A = A; h.feat_a = d_feat_a; h.feat_c = d_feat_c; h.Wa = d_Wa; h.ba = d_ba; h.wc_eff = d_wc_eff;
    h.bc = d_bc; h.action = d_action; h.old_logp = d_old_logp; h.adv = d_adv; h.v_old = d_v_old; h.v_target = d_v_target;
    h.active = d_active; h.eps = eps; h.ent_coef = ent_coef; h.logp = d_logp; h.entropy = d_entropy; h.value = d_value;
    h.d_logits = d_dlogits; h.d_value = d_dvalue; h.sums = d_sums; h.partials = d_ws;
    return dispatch_cpl(E, [&](auto C_) -> int {
        constexpr int CPL = decltype(C_)::value;
        const int blocks = ppo_head_blocks(R);
        ppo_head_kernel<CPL, MARL_NUM_ACTIONS><<<blocks, kPolThreads, 0, (cudaStream_t)stream>>>(h);
        int rc = check_launch("ppo_head_kernel");
        if (rc) return rc;
        ppo_sums_reduce_kernel<<<1, 256, 0, (cudaStream_t)stream>>>(blocks, d_ws, d_sums);
        return check_launch("ppo_sums_reduce_kernel");
    });
}

extern "C" int marl_act_head(int64_t R, int32_t E, int32_t A, const float *d_feat_a, const float *d_feat_c,
                             const float *d_Wa, const float *d_ba, const float *d_wc_eff, const float *d_bc,
                             uint64_t seed, int32_t t, int32_t deterministic, int32_t *d_action, float *d_action_f32,
                             float *d_logp, float *d_value, void *stream)
{
    MARL_REQUIRE(R > 0 && A == MARL_NUM_ACTIONS, "marl_act_head: R=%lld A=%d", (long long)R, A);
    MARL_REQUIRE(d_feat_a && d_Wa && d_ba && d_action && (!d_feat_c || (d_wc_eff && d_bc)), "marl_act_head: null pointer");
    return dispatch_cpl(E, [&](auto C_) -> int {
        constexpr int CPL = decltype(C_)::value;
        act_head_kernel<CPL, MARL_NUM_ACTIONS><<<grid_for_rows(R), kPolThreads, 0, (cudaStream_t)stream>>>(
            R, d_feat_a, d_feat_c, d_Wa, d_ba, d_wc_eff, d_bc, seed, t, deterministic, d_action, d_action_f32, d_logp, d_value);
        return check_launch("act_head_kernel");
    });
}

extern "C" int64_t marl_clip_workspace_bytes(int64_t n) { return sizeof(double) * blocks_1d(n); }

// ---- training-side pointwise / skinny pieces ------------------------------------------------------------------------------------
namespace marl {

// dst = out > 0 ? dy : 0  (backward of a fused ReLU epilogue), one pass instead of a compare and a multiply
__global__ void __launch_bounds__(256)
relu_bwd_kernel(int64_t n4, const float4 *__restrict__ dy, const float4 *__restrict__ out, float4 *__restrict__ dst)
{
    for (int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x; i < n4; i += (int64_t)gridDim.x * 256) {
        const float4 g = dy[i], o = out[i];
        dst[i] = make_float4(o.x > 0.f ? g.x : 0.f, o.y > 0.f ? g.y : 0.f, o.z > 0.f ? g.z : 0.f, o.w > 0.f ? g.w : 0.f);
    }
}

// Weight gradient of a layer with a tiny input width (the 4-wide state part of the semantic layer): partial[s][n][k] =
// sum over the rows of slice s of dY[r][n] * P[r][k], k < K <= 8, plus k = K: sum of dY[r][n] (the bias gradient).
// One thread per output feature n (coalesced rows of dY), the row of P is a broadcast load.  Deterministic: fixed slices,
// reduced in order by skinny_wgrad_reduce_kernel.
template <int KMAX>
__global__ void __launch_bounds__(128)
skinny_wgrad_kernel(int64_t R, int N, int K, const float *__restrict__ dY, int64_t lddy, const float *__restrict__ P, int64_t ldp,
                    int64_t rows_per_slice, float *__restrict__ partial)
{
    const int n = blockIdx.y * 128 + threadIdx.x;
    const int64_t r0 = (int64_t)blockIdx.x * rows_per_slice;
    int64_t r1 = r0 + rows_per_slice;
    if (r1 > R) r1 = R;
    float acc[KMAX], sum = 0.f;
#pragma unroll
    for (int k = 0; k < KMAX; ++k) acc[k] = 0.f;
    if (n < N) {
#pragma unroll 4
        for (int64_t r = r0; r < r1; ++r) {
            const float g = dY[r * lddy + n];
#pragma unroll
            for (int k = 0; k < KMAX; ++k)
                if (k < K) acc[k] = fmaf(g, __ldg(P + r * ldp + k), acc[k]);
            sum += g;
        }
        float *o = partial + ((size_t)blockIdx.x * N + n) * (K + 1);
#pragma unroll
        for (int k = 0; k < KMAX; ++k)
            if (k < K) o[k] = acc[k];
        o[K] = sum;
    }
}
// one warp per output (n, k <= K): lanes stride over the slices, then a fixed shuffle tree (deterministic)
__global__ void __launch_bounds__(128)
skinny_wgrad_reduce_kernel(int slices, int N, int K, const float *__restrict__ partial, float *__restrict__ dW, int64_t lddw,
                           float *__restrict__ dbias)
{
    const int idx = blockIdx.x * 4 + (threadIdx.x >> 5), lane = threadIdx.x & 31;       // (n, k) with k <= K
    if (idx >= N * (K + 1)) return;
    const int n = idx / (K + 1), k = idx - n * (K + 1);
    float acc = 0.f;
    for (int s = lane; s < slices; s += 32) acc += partial[((size_t)s * N + n) * (K + 1) + k];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    if (lane == 0) {
        if (k < K) dW[(int64_t)n * lddw + k] = acc;
        else if (dbias) dbias[n] = acc;
    }
}

}  // namespace marl

extern "C" int marl_relu_bwd(int64_t n, const float *d_dy, const float *d_out, float *d_dst, void *stream)
{
    MARL_REQUIRE(n > 0 && (n % 4) == 0 && d_dy && d_out && d_dst, "marl_relu_bwd: n=%lld (multiple of 4) / null pointer", (long long)n);
    MARL_REQUIRE((((uintptr_t)d_dy | (uintptr_t)d_out | (uintptr_t)d_dst) & 15) == 0, "marl_relu_bwd: pointers must be 16-byte aligned");
    const int64_t n4 = n / 4;
    const unsigned grid = (unsigned)((n4 + 255) / 256 < 148 * 16 ? (n4 + 255) / 256 : 148 * 16);
    relu_bwd_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(n4, reinterpret_cast<const float4 *>(d_dy), reinterpret_cast<const float4 *>(d_out),
                                                           reinterpret_cast<float4 *>(d_dst));
    return check_launch("relu_bwd_kernel");
}

static int64_t skinny_slices(int64_t R)
{
    const int64_t cap = 148 * 16;                       // 16 four-warp CTAs per SM: the row loop is a latency chain, it needs the warps
    const int64_t s = (R + 63) / 64;
    return s < cap ? (s < 1 ? 1 : s) : cap;
}

extern "C" int64_t marl_skinny_wgrad_workspace_bytes(int64_t R, int32_t N_out, int32_t K_in)
{
    if (R <= 0 || N_out <= 0 || K_in <= 0 || K_in > 16) return -1;
    return skinny_slices(R) * N_out * (K_in + 1) * 4;
}

extern "C" int marl_skinny_wgrad(int64_t R, int32_t N_out, int32_t K_in, const float *d_dY, int64_t lddy, const float *d_P, int64_t ldp,
                                 float *d_dW, int64_t lddw, float *d_dbias, void *d_workspace, void *stream)
{
    MARL_REQUIRE(R > 0 && N_out > 0 && K_in >= 1 && K_in <= 16, "marl_skinny_wgrad: R=%lld N_out=%d K_in=%d (1..16)", (long long)R, N_out, K_in);
    MARL_REQUIRE(d_dY && d_P && d_dW && d_workspace && lddy >= N_out && ldp >= K_in && lddw >= K_in, "marl_skinny_wgrad: bad pointer / leading dimension");
    const int64_t slices = skinny_slices(R);
    const int64_t rps = (R + slices - 1) / slices;
    float *partial = static_cast<float *>(d_workspace);
    const dim3 grid((unsigned)slices, (unsigned)((N_out + 127) / 128));
    if (K_in <= 4) skinny_wgrad_kernel<4><<<grid, 128, 0, (cudaStream_t)stream>>>(R, N_out, K_in, d_dY, lddy, d_P, ldp, rps, partial);
    else if (K_in <= 8) skinny_wgrad_kernel<8><<<grid, 128, 0, (cudaStream_t)stream>>>(R, N_out, K_in, d_dY, lddy, d_P, ldp, rps, partial);
    else skinny_wgrad_kernel<16><<<grid, 128, 0, (cudaStream_t)stream>>>(R, N_out, K_in, d_dY, lddy, d_P, ldp, rps, partial);
    int rc = check_launch("skinny_wgrad_kernel");
    if (rc) return rc;
    const int total = N_out * (K_in + 1);
    skinny_wgrad_reduce_kernel<<<(total + 3) / 4, 128, 0, (cudaStream_t)stream>>>((int)slices, N_out, K_in, partial, d_dW, lddw, d_dbias);
    return check_launch("skinny_wgrad_reduce_kernel");
}

extern "C" int marl_clip_grad_norm(int64_t n, float *d_grad, float max_norm, void *d_workspace, float *d_total_norm,
                                   void *stream)
{
    MARL_REQUIRE(n > 0 && d_grad && d_workspace && max_norm > 0, "marl_clip_grad_norm: bad argument");
    const int nb = blocks_1d(n);
    sumsq_kernel<<<nb, 256, 0, (cudaStream_t)stream>>>(n, d_grad, (double *)d_workspace);
    int rc = check_launch("sumsq_kernel");
    if (rc) return rc;
    clip_scale_kernel<<<nb, 256, 0, (cudaStream_t)stream>>>(n, d_grad, (const double *)d_workspace, nb, max_norm, d_total_norm);
    return check_launch("clip_scale_kernel");
}

extern "C" int marl_adam_step(int64_t n, float *d_param, const float *d_grad, float *d_exp_avg, float *d_exp_avg_sq,
                              float lr, float beta1, float beta2, float eps, int64_t step, void *stream)
{
    MARL_REQUIRE(n > 0 && d_param && d_grad && d_exp_avg && d_exp_avg_sq && step >= 1, "marl_adam_step: bad argument");
    const double bc1 = 1.0 - pow((double)beta1, (double)step), bc2 = 1.0 - pow((double)beta2, (double)step);
    adam_kernel<<<blocks_1d(n), 256, 0, (cudaStream_t)stream>>>(n, d_param, d_grad, d_exp_avg, d_exp_avg_sq, lr, beta1, beta2,
                                                                eps, (float)bc1, (float)sqrt(bc2));
    return check_launch("adam_kernel");
}

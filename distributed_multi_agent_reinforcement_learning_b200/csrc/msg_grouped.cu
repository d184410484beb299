// msg_grouped.cu — DHGN.message + L1-normalised mean aggregation (DHGN/mappo_parallel.py:256-281,323-348) for TRAINING batches,
// forward and backward, with one warp per SAMPLE (all N agents of one env at one time step) instead of one warp per row, so that
// everything the rows of a sample share is computed once (E = 128, N <= 16, O <= 256; other shapes use policy_kernels.cu):
//   relation 0:  relu(W0[:, :4](p_i - p_j) + W0[:, 4:](p_i - e) + b0) = relu(a_i - q_j), q_j = W0[:, :4] p_j: 3 instructions per
//                (i, j, channel) instead of 10;
//   relation 2, critic ("all ones" over the n cells of the map): sum_k relu(cc_i - u_k), cc_i = W2 p_i + b2, u_k = W2[:, :2] o_k shared
//                by the rows: 3 instructions per (i, k, channel) instead of 7 (the 2-instruction |.|-form of the rollout kernel is
//                not used here: its error scales with sum |cc - u| instead of the result, ~1e-5 on near-zero outputs);
//                the map's cells sit in registers (lane l holds cells l, l+32, ...) and are broadcast with shuffles;
//   backward:    only the SIGN of each pre-activation is needed; per (i, k, channel) a compare and three predicated adds
//                (count, sum of dx, sum of dy), the products with the upstream gradient are taken once per (row, channel).
// Lane l owns channels l, l+32, l+64, l+96 (the layout of agg [S,N,3,E] and of the per-row kernels).  HBM traffic is the
// output (forward) / the upstream gradient (backward): the kernels are FP32-issue bound.
#include "msg_args.cuh"

namespace marl {
namespace mg {

constexpr int E = 128, CPL = 4;

__device__ __forceinline__ float4 ld4(const float *p) { return *reinterpret_cast<const float4 *>(p); }

template <int KW>
__device__ __forceinline__ void load_w(const float *__restrict__ W, const float *__restrict__ b, int lane, float (&w)[CPL][KW], float (&bb)[CPL])
{
#pragma unroll
    for (int q = 0; q < CPL; ++q) {
        const int c = lane + 32 * q;
        bb[q] = __ldg(b + c);
#pragma unroll
        for (int k = 0; k < KW; k += 4) {
            const float4 v = __ldg(reinterpret_cast<const float4 *>(W + c * KW + k));
            w[q][k] = v.x; w[q][k + 1] = v.y; w[q][k + 2] = v.z; w[q][k + 3] = v.w;
        }
    }
}

// the map's cells: lane l holds cells l + 32 t
__device__ __forceinline__ void load_cells(const MsgArgs &a, int ob, int lane, float2 (&my_o)[8])
{
    const float2 *oxy = reinterpret_cast<const float2 *>(a.oxy) + (int64_t)ob * a.O;
#pragma unroll
    for (int t = 0; t < 8; ++t) {
        const int k = lane + 32 * t;
        my_o[t] = k < a.O ? __ldg(oxy + k) : make_float2(0.f, 0.f);
    }
}

// ------------------------------------------------------------------------------------------------------------ forward
template <int NA>
__global__ void __launch_bounds__(128)
msg_fwd_grouped_kernel(MsgArgs a, const float *__restrict__ W0, const float *__restrict__ b0, const float *__restrict__ W1,
                       const float *__restrict__ b1, const float *__restrict__ W2, const float *__restrict__ b2, float *__restrict__ agg)
{
    constexpr int RC = NA < 8 ? NA : 8;
    const int lane = threadIdx.x & 31, N = a.N;
    const int64_t s = (int64_t)blockIdx.x * 4 + (threadIdx.x >> 5);
    if (s >= a.S) return;
    float4 p[NA];
#pragma unroll
    for (int j = 0; j < NA; ++j) p[j] = j < N ? ld4(a.p + (s * N + j) * 4) : make_float4(0.f, 0.f, 0.f, 0.f);
    const float4 ev = ld4(a.e + s * 4);
    float *out = agg + s * N * 3 * E;
    const unsigned nmask = N >= 32 ? 0xffffffffu : ((1u << N) - 1u);
    {   // ---- relation 0
        float w[CPL][8], b[CPL], qj[NA][CPL];
        load_w<8>(W0, b0, lane, w, b);
#pragma unroll
        for (int j = 0; j < NA; ++j)
#pragma unroll
            for (int q = 0; q < CPL; ++q) qj[j][q] = fmaf(w[q][3], p[j].w, fmaf(w[q][2], p[j].z, fmaf(w[q][1], p[j].y, w[q][0] * p[j].x)));
        const uint32_t my_word = (!a.all_ones && lane < N) ? a.p_adj[(s * N + lane) * a.NW] : 0xffffffffu;
#pragma unroll
        for (int i = 0; i < NA; ++i) {
            if (i < N) {
                const uint32_t word = __shfl_sync(0xffffffffu, my_word, i) & nmask;
                const int cnt = __popc(word);
                const float dex = p[i].x - ev.x, dey = p[i].y - ev.y, dez = p[i].z - ev.z, dew = p[i].w - ev.w;
                float ai[CPL], acc[CPL];
#pragma unroll
                for (int q = 0; q < CPL; ++q) {
                    ai[q] = (qj[i][q] + fmaf(w[q][7], dew, fmaf(w[q][6], dez, fmaf(w[q][5], dey, w[q][4] * dex)))) + b[q];
                    acc[q] = 0.f;
                }
#pragma unroll
                for (int j = 0; j < NA; ++j) {
                    const bool on = (word >> j) & 1u;
#pragma unroll
                    for (int q = 0; q < CPL; ++q) {
                        const float t = fmaxf(ai[q] - qj[j][q], 0.f);
                        acc[q] += on ? t : 0.f;
                    }
                }
                const float nrm = cnt ? 1.f / fmaxf((float)cnt, 1e-12f) : 0.f;
#pragma unroll
                for (int q = 0; q < CPL; ++q) out[i * 3 * E + lane + 32 * q] = acc[q] * nrm;
            }
        }
    }
    {   // ---- relation 1
        float w[CPL][4], b[CPL];
        load_w<4>(W1, b1, lane, w, b);
        const float my_on = (!a.all_ones && lane < N) ? (float)a.e_adj[s * N + lane] : 1.f;
#pragma unroll
        for (int i = 0; i < NA; ++i) {
            if (i < N) {
                const float e_on = __shfl_sync(0xffffffffu, my_on, i);
                const float dex = p[i].x - ev.x, dey = p[i].y - ev.y, dez = p[i].z - ev.z, dew = p[i].w - ev.w;
#pragma unroll
                for (int q = 0; q < CPL; ++q)
                    out[i * 3 * E + E + lane + 32 * q] =
                        e_on * fmaxf(fmaf(w[q][3], dew, fmaf(w[q][2], dez, fmaf(w[q][1], dey, fmaf(w[q][0], dex, 0.f)))) + b[q], 0.f);
            }
        }
    }
    {   // ---- relation 2
        float w[CPL][4], b[CPL];
        load_w<4>(W2, b2, lane, w, b);
        const int ob = a.o_index[s];
        float2 my_o[8];
        load_cells(a, ob, lane, my_o);
        if (a.all_ones) {
            const int n = a.o_count[ob];
            const float nrm = n ? 1.f / fmaxf((float)n, 1e-12f) : 0.f;
#pragma unroll
            for (int ch = 0; ch < NA / RC; ++ch) {
                if (ch * RC >= N) break;
                float cc[RC][CPL], acc[RC][CPL];
#pragma unroll
                for (int rr = 0; rr < RC; ++rr)
#pragma unroll
                    for (int q = 0; q < CPL; ++q) {
                        const float4 pi = p[ch * RC + rr];
                        cc[rr][q] = fmaf(w[q][3], pi.w, fmaf(w[q][2], pi.z, fmaf(w[q][1], pi.y, fmaf(w[q][0], pi.x, 0.f)))) + b[q];
                        acc[rr][q] = 0.f;
                    }
#pragma unroll
                for (int t = 0; t < 8; ++t) {
                    const int kn = min(32, n - 32 * t);
                    for (int kk = 0; kk < kn; ++kk) {
                        const float ox = __shfl_sync(0xffffffffu, my_o[t].x, kk), oy = __shfl_sync(0xffffffffu, my_o[t].y, kk);
                        float u[CPL];
#pragma unroll
                        for (int q = 0; q < CPL; ++q) u[q] = fmaf(w[q][1], oy, w[q][0] * ox);
#pragma unroll
                        for (int rr = 0; rr < RC; ++rr)
#pragma unroll
                            for (int q = 0; q < CPL; ++q) acc[rr][q] += fmaxf(cc[rr][q] - u[q], 0.f);
                    }
                }
#pragma unroll
                for (int rr = 0; rr < RC; ++rr) {
                    const int i = ch * RC + rr;
                    if (i < N) {
#pragma unroll
                        for (int q = 0; q < CPL; ++q) out[i * 3 * E + 2 * E + lane + 32 * q] = acc[rr][q] * nrm;
                    }
                }
            }
        } else {
#pragma unroll 1
            for (int i = 0; i < N; ++i) {
                const float4 pi = ld4(a.p + (s * N + i) * 4);
                float cc[CPL], acc[CPL];
#pragma unroll
                for (int q = 0; q < CPL; ++q) {
                    cc[q] = fmaf(w[q][3], pi.w, fmaf(w[q][2], pi.z, fmaf(w[q][1], pi.y, fmaf(w[q][0], pi.x, 0.f)))) + b[q];
                    acc[q] = 0.f;
                }
                int cnt = 0;
#pragma unroll
                for (int t = 0; t < 8; ++t) {
                    uint32_t bits = t < a.OW ? a.o_adj[(s * N + i) * a.OW + t] : 0u;
                    cnt += __popc(bits);
                    while (bits) {
                        const int kk = __ffs(bits) - 1;
                        bits &= bits - 1;
                        const float ox = __shfl_sync(0xffffffffu, my_o[t].x, kk), oy = __shfl_sync(0xffffffffu, my_o[t].y, kk);
#pragma unroll
                        for (int q = 0; q < CPL; ++q) acc[q] += fmaxf(cc[q] - fmaf(w[q][1], oy, w[q][0] * ox), 0.f);
                    }
                }
                const float nrm = cnt ? 1.f / fmaxf((float)cnt, 1e-12f) : 0.f;
#pragma unroll
                for (int q = 0; q < CPL; ++q) out[i * 3 * E + 2 * E + lane + 32 * q] = acc[q] * nrm;
            }
        }
    }
}

// ------------------------------------------------------------------------------------------------------------ backward
// One launch per relation (REL): keeps the per-lane weight slices and gradient accumulators of only that relation in registers.
// Persistent warps walk samples with a grid stride; CTA reduction through shared memory, then either one atomicAdd per element
// (DET false) or the CTA's row of partial sums to ws[blockIdx.x], reduced in a fixed order by launch_msg_partials_reduce (DET true).
template <int NA, int REL, bool DET>
__global__ void __launch_bounds__(128)
msg_bwd_grouped_kernel(MsgArgs a, const float *__restrict__ W, const float *__restrict__ b, const float *__restrict__ d_agg,
                       float *__restrict__ gW, float *__restrict__ gb, float *__restrict__ ws)
{
    constexpr int KW = REL == 0 ? 8 : 4;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, N = a.N;
    float w[CPL][KW], bb[CPL], g[CPL][KW + 1];
    load_w<KW>(W, b, lane, w, bb);
#pragma unroll
    for (int q = 0; q < CPL; ++q)
#pragma unroll
        for (int k = 0; k <= KW; ++k) g[q][k] = 0.f;
    const unsigned nmask = N >= 32 ? 0xffffffffu : ((1u << N) - 1u);
    const int64_t stride = (int64_t)gridDim.x * 4;
    for (int64_t s = (int64_t)blockIdx.x * 4 + warp; s < a.S; s += stride) {
        float4 p[NA];
#pragma unroll
        for (int j = 0; j < NA; ++j) p[j] = j < N ? ld4(a.p + (s * N + j) * 4) : make_float4(0.f, 0.f, 0.f, 0.f);
        const float4 ev = ld4(a.e + s * 4);
        const float *dg = d_agg + s * N * 3 * E + REL * E;
        if (REL == 0) {
            float qj[NA][CPL];
#pragma unroll
            for (int j = 0; j < NA; ++j)
#pragma unroll
                for (int q = 0; q < CPL; ++q) qj[j][q] = fmaf(w[q][3], p[j].w, fmaf(w[q][2], p[j].z, fmaf(w[q][1], p[j].y, w[q][0] * p[j].x)));
            const uint32_t my_word = (!a.all_ones && lane < N) ? a.p_adj[(s * N + lane) * a.NW] : 0xffffffffu;
#pragma unroll
            for (int i = 0; i < NA; ++i) {
                if (i < N) {
                    const uint32_t word = __shfl_sync(0xffffffffu, my_word, i) & nmask;
                    const int cnt = __popc(word);
                    const float n0 = cnt ? 1.f / fmaxf((float)cnt, 1e-12f) : 0.f;
                    const float de[4] = {p[i].x - ev.x, p[i].y - ev.y, p[i].z - ev.z, p[i].w - ev.w};
                    float ai[CPL], cp[CPL], sd[CPL][4];
#pragma unroll
                    for (int q = 0; q < CPL; ++q) {
                        ai[q] = (qj[i][q] + fmaf(w[q][7], de[3], fmaf(w[q][6], de[2], fmaf(w[q][5], de[1], w[q][4] * de[0])))) + bb[q];
                        cp[q] = 0.f;
                        sd[q][0] = sd[q][1] = sd[q][2] = sd[q][3] = 0.f;
                    }
#pragma unroll
                    for (int j = 0; j < NA; ++j) {
                        if ((word >> j) & 1u) {                                         // warp-uniform
                            const float d[4] = {p[i].x - p[j].x, p[i].y - p[j].y, p[i].z - p[j].z, p[i].w - p[j].w};
#pragma unroll
                            for (int q = 0; q < CPL; ++q) {
                                const bool pos = ai[q] - qj[j][q] > 0.f;
                                cp[q] += pos ? 1.f : 0.f;
#pragma unroll
                                for (int k = 0; k < 4; ++k) sd[q][k] += pos ? d[k] : 0.f;
                            }
                        }
                    }
#pragma unroll
                    for (int q = 0; q < CPL; ++q) {
                        const float gq = dg[i * 3 * E + lane + 32 * q] * n0;
#pragma unroll
                        for (int k = 0; k < 4; ++k) {
                            g[q][k] = fmaf(gq, sd[q][k], g[q][k]);
                            g[q][4 + k] = fmaf(gq * cp[q], de[k], g[q][4 + k]);
                        }
                        g[q][8] = fmaf(gq, cp[q], g[q][8]);
                    }
                }
            }
        } else if (REL == 1) {
            const float my_on = (!a.all_ones && lane < N) ? (float)a.e_adj[s * N + lane] : 1.f;
#pragma unroll
            for (int i = 0; i < NA; ++i) {
                if (i < N) {
                    const float e_on = __shfl_sync(0xffffffffu, my_on, i);
                    const float de[4] = {p[i].x - ev.x, p[i].y - ev.y, p[i].z - ev.z, p[i].w - ev.w};
#pragma unroll
                    for (int q = 0; q < CPL; ++q) {
                        const float v = fmaf(w[q][3], de[3], fmaf(w[q][2], de[2], fmaf(w[q][1], de[1], fmaf(w[q][0], de[0], 0.f)))) + bb[q];
                        const float gq = v > 0.f ? dg[i * 3 * E + lane + 32 * q] * e_on : 0.f;
#pragma unroll
                        for (int k = 0; k < 4; ++k) g[q][k] = fmaf(gq, de[k], g[q][k]);
                        g[q][4] += gq;
                    }
                }
            }
        } else {
            const int ob = a.o_index[s];
            float2 my_o[8];
            load_cells(a, ob, lane, my_o);
            const int n_all = a.all_ones ? a.o_count[ob] : 0;
#pragma unroll
            for (int i = 0; i < NA; ++i) {
                if (i < N) {
                    float cc[CPL], cp[CPL], s0[CPL], s1[CPL];
#pragma unroll
                    for (int q = 0; q < CPL; ++q) {
                        cc[q] = fmaf(w[q][3], p[i].w, fmaf(w[q][2], p[i].z, fmaf(w[q][1], p[i].y, fmaf(w[q][0], p[i].x, 0.f)))) + bb[q];
                        cp[q] = s0[q] = s1[q] = 0.f;
                    }
                    int cnt = n_all;
#pragma unroll
                    for (int t = 0; t < 8; ++t) {
                        uint32_t bits;
                        if (a.all_ones) {
                            const int kn = min(32, n_all - 32 * t);
                            bits = kn <= 0 ? 0u : (kn >= 32 ? 0xffffffffu : ((1u << kn) - 1u));
                        } else {
                            bits = t < a.OW ? a.o_adj[(s * N + i) * a.OW + t] : 0u;
                            cnt += __popc(bits);
                        }
                        while (bits) {                                                  // warp-uniform
                            const int kk = __ffs(bits) - 1;
                            bits &= bits - 1;
                            const float ox = __shfl_sync(0xffffffffu, my_o[t].x, kk), oy = __shfl_sync(0xffffffffu, my_o[t].y, kk);
                            const float d0 = p[i].x - ox, d1 = p[i].y - oy;
#pragma unroll
                            for (int q = 0; q < CPL; ++q) {
                                const bool pos = cc[q] - fmaf(w[q][1], oy, w[q][0] * ox) > 0.f;
                                cp[q] += pos ? 1.f : 0.f;
                                s0[q] += pos ? d0 : 0.f;
                                s1[q] += pos ? d1 : 0.f;
                            }
                        }
                    }
                    const float n2 = cnt ? 1.f / fmaxf((float)cnt, 1e-12f) : 0.f;
#pragma unroll
                    for (int q = 0; q < CPL; ++q) {
                        const float gq = dg[i * 3 * E + lane + 32 * q] * n2;
                        g[q][0] = fmaf(gq, s0[q], g[q][0]);
                        g[q][1] = fmaf(gq, s1[q], g[q][1]);
                        g[q][2] = fmaf(gq * cp[q], p[i].z, g[q][2]);
                        g[q][3] = fmaf(gq * cp[q], p[i].w, g[q][3]);
                        g[q][4] = fmaf(gq, cp[q], g[q][4]);
                    }
                }
            }
        }
    }
    __shared__ float s_red[4][(KW + 1) * E];
#pragma unroll
    for (int q = 0; q < CPL; ++q)
#pragma unroll
        for (int k = 0; k <= KW; ++k) s_red[warp][k * E + lane + 32 * q] = g[q][k];
    __syncthreads();
    for (int idx = threadIdx.x; idx < (KW + 1) * E; idx += 128) {
        const float v = (s_red[0][idx] + s_red[1][idx]) + (s_red[2][idx] + s_red[3][idx]);
        if (DET) {
            ws[(int64_t)blockIdx.x * (KW + 1) * E + idx] = v;
        } else {
            const int k = idx / E, c = idx - k * E;
            if (k < KW) atomicAdd(gW + c * KW + k, v);
            else atomicAdd(gb + c, v);
        }
    }
}

}  // namespace mg

bool msg_grouped_supported(const MsgArgs &a, int E) { return E == mg::E && a.N <= 16 && a.O <= 256 && a.NW == 1; }

int launch_msg_fwd_grouped(const MsgArgs &a, const float *W0, const float *b0, const float *W1, const float *b1, const float *W2,
                           const float *b2, float *agg, cudaStream_t stream)
{
    const unsigned grid = (unsigned)((a.S + 3) / 4);
    if (a.N <= 4) mg::msg_fwd_grouped_kernel<4><<<grid, 128, 0, stream>>>(a, W0, b0, W1, b1, W2, b2, agg);
    else if (a.N <= 8) mg::msg_fwd_grouped_kernel<8><<<grid, 128, 0, stream>>>(a, W0, b0, W1, b1, W2, b2, agg);
    else mg::msg_fwd_grouped_kernel<16><<<grid, 128, 0, stream>>>(a, W0, b0, W1, b1, W2, b2, agg);
    return check_launch("msg_fwd_grouped_kernel");
}

template <int NA, bool DET>
static int launch_bwd_na(const MsgArgs &a, const float *W0, const float *b0, const float *W1, const float *b1, const float *W2, const float *b2,
                         const float *d_agg, float *gW0, float *gb0, float *gW1, float *gb1, float *gW2, float *gb2, float *ws,
                         cudaStream_t stream)
{
    const int64_t blocks = msg_bwd_grouped_blocks(a), E = mg::E;
    float *ws1 = DET ? ws + blocks * 9 * E : nullptr, *ws2 = DET ? ws + blocks * 14 * E : nullptr;
    mg::msg_bwd_grouped_kernel<NA, 0, DET><<<(unsigned)blocks, 128, 0, stream>>>(a, W0, b0, d_agg, gW0, gb0, ws);
    mg::msg_bwd_grouped_kernel<NA, 1, DET><<<(unsigned)blocks, 128, 0, stream>>>(a, W1, b1, d_agg, gW1, gb1, ws1);
    mg::msg_bwd_grouped_kernel<NA, 2, DET><<<(unsigned)blocks, 128, 0, stream>>>(a, W2, b2, d_agg, gW2, gb2, ws2);
    int rc = check_launch("msg_bwd_grouped_kernel");
    if (rc || !DET) return rc;
    MsgPartials p;
    p.rel_base[0] = ws; p.rel_base[1] = ws1; p.rel_base[2] = ws2;
    p.rel_stride[0] = 9 * E; p.rel_stride[1] = 5 * E; p.rel_stride[2] = 5 * E;
    p.blocks = (int)blocks; p.E = (int)E;
    return launch_msg_partials_reduce(p, gW0, gb0, gW1, gb1, gW2, gb2, stream);
}

template <int NA>
static int launch_bwd_na(const MsgArgs &a, const float *W0, const float *b0, const float *W1, const float *b1, const float *W2, const float *b2,
                         const float *d_agg, float *gW0, float *gb0, float *gW1, float *gb1, float *gW2, float *gb2, float *ws,
                         cudaStream_t stream)
{
    if (ws) return launch_bwd_na<NA, true>(a, W0, b0, W1, b1, W2, b2, d_agg, gW0, gb0, gW1, gb1, gW2, gb2, ws, stream);
    return launch_bwd_na<NA, false>(a, W0, b0, W1, b1, W2, b2, d_agg, gW0, gb0, gW1, gb1, gW2, gb2, ws, stream);
}

int launch_msg_bwd_grouped(const MsgArgs &a, const float *W0, const float *b0, const float *W1, const float *b1, const float *W2,
                           const float *b2, const float *d_agg, float *gW0, float *gb0, float *gW1, float *gb1, float *gW2, float *gb2,
                           float *ws, cudaStream_t stream)
{
    if (a.N <= 4) return launch_bwd_na<4>(a, W0, b0, W1, b1, W2, b2, d_agg, gW0, gb0, gW1, gb1, gW2, gb2, ws, stream);
    if (a.N <= 8) return launch_bwd_na<8>(a, W0, b0, W1, b1, W2, b2, d_agg, gW0, gb0, gW1, gb1, gW2, gb2, ws, stream);
    return launch_bwd_na<16>(a, W0, b0, W1, b1, W2, b2, d_agg, gW0, gb0, gW1, gb1, gW2, gb2, ws, stream);
}

}  // namespace marl

// stats_kernels.cu — kernel 3 (Welford reward normalisation, GAE reverse scan + advantage normalisation) and
// kernel 4 (minibatch row gather).  All HBM-streaming; one thread per (env, agent) chain, coalesced across chains.
#include "common.cuh"

namespace marl {

// ---- 3a: Welford (DHGN/normalization.py:4-35), one running estimate per env -----------------------------
// Block = whole envs only, so the shared per-env counter n can be read by every agent thread before it is bumped.
template <typename X>
__global__ void __launch_bounds__(128)
welford_kernel(int B, int N, int epb, const X *__restrict__ reward, long long *__restrict__ n_arr,
               double *__restrict__ mean, double *__restrict__ S, double *__restrict__ sd, float *__restrict__ out,
               int update)
{
    const int le = threadIdx.x / N, i = threadIdx.x - le * N;
    const int64_t b = (int64_t)blockIdx.x * epb + le;
    const bool ok = le < epb && b < B;
    long long n = 0;
    if (ok) n = n_arr[b];
    __syncthreads();
    if (!ok) return;
    const int64_t idx = b * N + i;
    const double x = (double)reward[idx];
    double m = mean[idx], s = S[idx], d = sd[idx];
    if (update) {
        n += 1;
        if (n == 1) {
            m = x;
            d = x;   // `self.std = x` on the first sample
        } else {
            const double old = m;
            m = dadd(old, ddiv(dsub(x, old), (double)n));
            s = dadd(s, dmul(dsub(x, old), dsub(x, m)));
            d = sqrt(ddiv(s, (double)n));
        }
        mean[idx] = m;
        S[idx] = s;
        sd[idx] = d;
        if (i == 0) n_arr[b] = n;
    }
    out[idx] = (float)ddiv(dsub(x, m), dadd(d, 1e-8));
}

// ---- 3b: GAE (DHGN/mappo_parallel.py:643-658) ------------------------------------------------------------
// One thread per (b,n) chain walks t = T-1..0.  Element (b,t,n) lives at b*sb + t*st + n (v: b*vsb + t*st_v + n),
// which covers both the reference layout [B,T,N] and the time-major rollout arena [T,B,N].
// fp32 arithmetic in torch's order: delta = (r + gamma*v[t+1] - v[t]) * active;  gae = delta + (gamma*lamda)*gae.
// Per-block partial sums (double) of adv and adv^2 go to the workspace for the deterministic normalisation pass.
static constexpr int kGaeThreads = 128;

__global__ void __launch_bounds__(kGaeThreads)
gae_scan_kernel(int B, int T, int N, const float *__restrict__ r, const float *__restrict__ v,
                const float *__restrict__ active, int64_t sb, int64_t st, int64_t vsb, int64_t vst, float gamma,
                float gl, float *__restrict__ adv, float *__restrict__ v_target, double *__restrict__ partial)
{
    const int64_t chain = (int64_t)blockIdx.x * kGaeThreads + threadIdx.x;
    double sum = 0.0, sq = 0.0;
    if (chain < (int64_t)B * N) {
        const int64_t b = chain / N, n = chain - b * N;
        const int64_t base = b * sb + n, vbase = b * vsb + n;
        float gae = 0.0f;
        float v_next = v[vbase + (int64_t)T * vst];
        for (int t = T - 1; t >= 0; --t) {
            const int64_t i = base + (int64_t)t * st;
            const float v_t = v[vbase + (int64_t)t * vst];
            const float delta = __fmul_rn(__fsub_rn(__fadd_rn(r[i], __fmul_rn(gamma, v_next)), v_t), active[i]);
            gae = __fadd_rn(delta, __fmul_rn(gl, gae));
            adv[i] = gae;
            v_target[i] = __fadd_rn(gae, v_t);
            sum += (double)gae;
            sq += (double)gae * (double)gae;
            v_next = v_t;
        }
    }
    __shared__ double s_sum[kGaeThreads / 32], s_sq[kGaeThreads / 32];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        sum += __shfl_down_sync(0xffffffffu, sum, o);
        sq += __shfl_down_sync(0xffffffffu, sq, o);
    }
    if ((threadIdx.x & 31) == 0) {
        s_sum[threadIdx.x >> 5] = sum;
        s_sq[threadIdx.x >> 5] = sq;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        double a = 0, q = 0;
        for (int w = 0; w < kGaeThreads / 32; ++w) { a += s_sum[w]; q += s_sq[w]; }
        partial[2 * blockIdx.x] = a;
        partial[2 * blockIdx.x + 1] = q;
    }
}

// GAE of a time-major rollout segment [T,B,N] whose episode ends after step k-1 (0 < k < T): steps k..T-1 are the next episode's
// start and bootstrap from v[T]; steps 0..k-1 end the previous episode and bootstrap from v_boot [B,N] (its value after its last
// step) instead of v[k].  Each piece is exactly gae_scan_kernel's recursion on its own steps: the recursion does not cross k.
// Partials as in gae_scan_kernel, over all T steps, for adv_norm_kernel.  The block reduction below repeats gae_scan_kernel's (kept
// apart so that kernel's code stays as it is): the two must stay in step, adv_norm_kernel reads one (sum, sum of squares) per block.
__global__ void __launch_bounds__(kGaeThreads)
gae_scan_boundary_kernel(int B, int T, int N, int k, const float *__restrict__ r, const float *__restrict__ v,
                         const float *__restrict__ v_boot, const float *__restrict__ active, float gamma, float gl,
                         float *__restrict__ adv, float *__restrict__ v_target, double *__restrict__ partial)
{
    const int64_t chain = (int64_t)blockIdx.x * kGaeThreads + threadIdx.x;
    const int64_t st = (int64_t)B * N;
    double sum = 0.0, sq = 0.0;
    if (chain < st) {
        float gae = 0.0f;
        float v_next = v[chain + (int64_t)T * st];
        for (int t = T - 1; t >= 0; --t) {
            if (t == k - 1) {                       // the previous episode's last step: its own bootstrap, a fresh recursion
                gae = 0.0f;
                v_next = v_boot[chain];
            }
            const int64_t i = chain + (int64_t)t * st;
            const float v_t = v[i];
            const float delta = __fmul_rn(__fsub_rn(__fadd_rn(r[i], __fmul_rn(gamma, v_next)), v_t), active[i]);
            gae = __fadd_rn(delta, __fmul_rn(gl, gae));
            adv[i] = gae;
            v_target[i] = __fadd_rn(gae, v_t);
            sum += (double)gae;
            sq += (double)gae * (double)gae;
            v_next = v_t;
        }
    }
    __shared__ double s_sum[kGaeThreads / 32], s_sq[kGaeThreads / 32];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        sum += __shfl_down_sync(0xffffffffu, sum, o);
        sq += __shfl_down_sync(0xffffffffu, sq, o);
    }
    if ((threadIdx.x & 31) == 0) {
        s_sum[threadIdx.x >> 5] = sum;
        s_sq[threadIdx.x >> 5] = sq;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        double a = 0, q = 0;
        for (int w = 0; w < kGaeThreads / 32; ++w) { a += s_sum[w]; q += s_sq[w]; }
        partial[2 * blockIdx.x] = a;
        partial[2 * blockIdx.x + 1] = q;
    }
}

// adv = (adv - mean) / (std_unbiased + 1e-5) * active over the whole tensor (mappo_parallel.py:655-658).
// Every block re-reduces the (few thousand) partials in the same order -> deterministic mean/std.
__global__ void __launch_bounds__(256)
adv_norm_kernel(int64_t total, int n_partial, const double *__restrict__ partial, const float *__restrict__ active,
                float *__restrict__ adv)
{
    __shared__ double s_a[256], s_q[256];
    double a = 0, q = 0;
    for (int i = threadIdx.x; i < n_partial; i += 256) { a += partial[2 * i]; q += partial[2 * i + 1]; }
    s_a[threadIdx.x] = a;
    s_q[threadIdx.x] = q;
    __syncthreads();
    for (int o = 128; o > 0; o >>= 1) {
        if (threadIdx.x < o) { s_a[threadIdx.x] += s_a[threadIdx.x + o]; s_q[threadIdx.x] += s_q[threadIdx.x + o]; }
        __syncthreads();
    }
    const double mean = s_a[0] / (double)total;
    double var = (s_q[0] - s_a[0] * mean) / (double)(total - 1);
    if (var < 0) var = 0;
    const float fm = (float)mean, fs = __fadd_rn((float)sqrt(var), 1e-5f);
    // the advantage tensor is dense in both supported layouts, so a flat grid-stride pass is coalesced
    for (int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x; i < total; i += (int64_t)gridDim.x * 256)
        adv[i] = __fmul_rn(__fdiv_rn(__fsub_rn(adv[i], fm), fs), active[i]);
}

// ---- 4: row gather (`batch[key][index]`, mappo_parallel.py:665-679) ---------------------------------------
template <typename V>
__global__ void __launch_bounds__(256)
gather_rows_kernel(const V *__restrict__ src, V *__restrict__ dst, const int64_t *__restrict__ index, int n_index,
                   int64_t row_vecs)
{
    const int64_t total = (int64_t)n_index * row_vecs;
    for (int64_t e = (int64_t)blockIdx.x * 256 + threadIdx.x; e < total; e += (int64_t)gridDim.x * 256) {
        const int64_t i = e / row_vecs, k = e - i * row_vecs;
        dst[e] = src[index[i] * row_vecs + k];
    }
}

}  // namespace marl

using namespace marl;

extern "C" int marl_welford_update(int32_t B, int32_t N, const int32_t *d_reward, int64_t *d_n, double *d_mean,
                                   double *d_S, double *d_std, float *d_out, int32_t update, void *stream)
{
    MARL_REQUIRE(B > 0 && N > 0 && N <= 128, "marl_welford_update: B=%d N=%d", B, N);
    MARL_REQUIRE(d_reward && d_n && d_mean && d_S && d_std && d_out, "marl_welford_update: null pointer");
    const int epb = 128 / N;
    const int blocks = (B + epb - 1) / epb;
    welford_kernel<int32_t><<<blocks, 128, 0, (cudaStream_t)stream>>>(B, N, epb, d_reward, (long long *)d_n, d_mean, d_S, d_std,
                                                                      d_out, update);
    return check_launch("welford_kernel");
}

extern "C" int marl_welford_update_f64(int32_t B, int32_t N, const double *d_x, int64_t *d_n, double *d_mean,
                                       double *d_S, double *d_std, float *d_out, int32_t update, void *stream)
{
    MARL_REQUIRE(B > 0 && N > 0 && N <= 128, "marl_welford_update_f64: B=%d N=%d", B, N);
    MARL_REQUIRE(d_x && d_n && d_mean && d_S && d_std && d_out, "marl_welford_update_f64: null pointer");
    const int epb = 128 / N;
    const int blocks = (B + epb - 1) / epb;
    welford_kernel<double><<<blocks, 128, 0, (cudaStream_t)stream>>>(B, N, epb, d_x, (long long *)d_n, d_mean, d_S, d_std,
                                                                     d_out, update);
    return check_launch("welford_kernel<double>");
}

extern "C" int64_t marl_gae_workspace_bytes(int32_t B, int32_t T, int32_t N)
{
    (void)T;
    const int64_t chains = (int64_t)B * N;
    return 2 * sizeof(double) * ((chains + kGaeThreads - 1) / kGaeThreads);
}

extern "C" int marl_gae(int32_t B, int32_t T, int32_t N, const float *d_r, const float *d_v, const float *d_active,
                        int32_t time_major, float gamma, float gamma_lamda, int32_t use_adv_norm, float *d_adv,
                        float *d_v_target, void *d_workspace, void *stream)
{
    MARL_REQUIRE(B > 0 && T > 0 && N > 0, "marl_gae: B=%d T=%d N=%d", B, T, N);
    MARL_REQUIRE(d_r && d_v && d_active && d_adv && d_v_target && d_workspace, "marl_gae: null pointer");
    const int64_t chains = (int64_t)B * N;
    const int blocks = (int)((chains + kGaeThreads - 1) / kGaeThreads);
    int64_t sb, st, vsb, vst;
    if (time_major) { sb = N; st = (int64_t)B * N; vsb = N; vst = (int64_t)B * N; }
    else { sb = (int64_t)T * N; st = N; vsb = (int64_t)(T + 1) * N; vst = N; }
    cudaStream_t s = (cudaStream_t)stream;
    gae_scan_kernel<<<blocks, kGaeThreads, 0, s>>>(B, T, N, d_r, d_v, d_active, sb, st, vsb, vst, gamma, gamma_lamda,
                                                   d_adv, d_v_target, (double *)d_workspace);
    int rc = check_launch("gae_scan_kernel");
    if (rc) return rc;
    if (use_adv_norm) {
        const int64_t total = chains * T;
        MARL_REQUIRE(total > 1, "marl_gae: adv-norm needs more than one sample");
        int nb = (int)((total + 255) / 256);
        if (nb > 148 * 8) nb = 148 * 8;
        adv_norm_kernel<<<nb, 256, 0, s>>>(total, blocks, (const double *)d_workspace, d_active, d_adv);
        rc = check_launch("adv_norm_kernel");
    }
    return rc;
}

extern "C" int marl_gae_boundary(int32_t B, int32_t T, int32_t N, int32_t k, const float *d_r, const float *d_v, const float *d_v_boot,
                                 const float *d_active, float gamma, float gamma_lamda, int32_t use_adv_norm, float *d_adv,
                                 float *d_v_target, void *d_workspace, void *stream)
{
    MARL_REQUIRE(B > 0 && T > 1 && N > 0 && k > 0 && k < T, "marl_gae_boundary: B=%d T=%d N=%d k=%d", B, T, N, k);
    MARL_REQUIRE(d_r && d_v && d_v_boot && d_active && d_adv && d_v_target && d_workspace, "marl_gae_boundary: null pointer");
    const int64_t chains = (int64_t)B * N;
    const int blocks = (int)((chains + kGaeThreads - 1) / kGaeThreads);
    cudaStream_t s = (cudaStream_t)stream;
    gae_scan_boundary_kernel<<<blocks, kGaeThreads, 0, s>>>(B, T, N, k, d_r, d_v, d_v_boot, d_active, gamma, gamma_lamda, d_adv,
                                                            d_v_target, (double *)d_workspace);
    int rc = check_launch("gae_scan_boundary_kernel");
    if (rc) return rc;
    if (use_adv_norm) {
        const int64_t total = chains * T;
        int nb = (int)((total + 255) / 256);
        if (nb > 148 * 8) nb = 148 * 8;
        adv_norm_kernel<<<nb, 256, 0, s>>>(total, blocks, (const double *)d_workspace, d_active, d_adv);
        rc = check_launch("adv_norm_kernel");
    }
    return rc;
}

extern "C" int marl_gather_rows(const void *d_src, void *d_dst, const int64_t *d_index, int32_t n_index,
                                int64_t row_bytes, int64_t n_src_rows, void *stream)
{
    (void)n_src_rows;
    MARL_REQUIRE(d_src && d_dst && d_index && n_index > 0 && row_bytes > 0,
                 "marl_gather_rows: bad argument (row_bytes=%lld)", (long long)row_bytes);
    cudaStream_t s = (cudaStream_t)stream;
    // widest element that divides the row and both base addresses: 16 bytes, 4, or single bytes (e.g. the u8 e_adj rows of
    // an odd-sized team)
    const uintptr_t align = (uintptr_t)row_bytes | (uintptr_t)d_src | (uintptr_t)d_dst;
    const int64_t elem = (align & 15) == 0 ? 16 : ((align & 3) == 0 ? 4 : 1);
    const int64_t row_vecs = row_bytes / elem;
    const int64_t total = (int64_t)n_index * row_vecs;
    int nb = (int)((total + 255) / 256);
    if (nb > 148 * 16) nb = 148 * 16;
    if (elem == 16) gather_rows_kernel<uint4><<<nb, 256, 0, s>>>((const uint4 *)d_src, (uint4 *)d_dst, d_index, n_index, row_vecs);
    else if (elem == 4) gather_rows_kernel<uint32_t><<<nb, 256, 0, s>>>((const uint32_t *)d_src, (uint32_t *)d_dst, d_index, n_index, row_vecs);
    else gather_rows_kernel<uint8_t><<<nb, 256, 0, s>>>((const uint8_t *)d_src, (uint8_t *)d_dst, d_index, n_index, row_vecs);
    return check_launch("gather_rows_kernel");
}

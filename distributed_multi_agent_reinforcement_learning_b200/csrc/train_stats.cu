// train_stats.cu — PPO diagnostics of one update (entropy, KL estimates, clip fractions, explained variance, advantage
// scale, gradient norms), reduced on the device from the per-row values the training forward already computes.
// Everything is accumulated in f64 in a fixed order (grid size a function of R only, fixed shuffle tree, per-CTA partials
// reduced in index order): bit-identical results from call to call, graph-capturable, no atomics.  The slots are documented
// beside MARL_PPO_STATS_SUMS / MARL_PPO_STATS_OUT in include/marl_b200.h.
#include "common.cuh"

namespace marl {

static constexpr int kStatThreads = 256;
static constexpr int kStatMaxBlocks = 1024;     // a constant, not a multiple of the SM count: the order depends on R alone
static constexpr int kS = MARL_PPO_STATS_SUMS;
enum { kMaxLr = 5, kMinLr = 6 };

static inline int stats_blocks(int64_t R)
{
    const int64_t b = (R + kStatThreads - 1) / kStatThreads;
    return (int)(b < kStatMaxBlocks ? b : kStatMaxBlocks);
}

// Each thread strides over rows r = tid, tid + grid, ...; a fixed shuffle tree per warp, then thread j < kS adds the warps'
// slot j in warp order and writes partial[blockIdx.x][j].
__global__ void __launch_bounds__(kStatThreads)
ppo_stats_kernel(int64_t R, const float *__restrict__ logp, const float *__restrict__ old_logp,
                 const float *__restrict__ entropy, const float *__restrict__ value, const float *__restrict__ v_old,
                 const float *__restrict__ v_target, const float *__restrict__ active, double eps,
                 double *__restrict__ partial)
{
    double s[kS];
#pragma unroll
    for (int j = 0; j < kS; ++j) s[j] = 0.0;
    s[kMaxLr] = -INFINITY;
    s[kMinLr] = INFINITY;
    const int64_t stride = (int64_t)gridDim.x * kStatThreads;
    for (int64_t r = (int64_t)blockIdx.x * kStatThreads + threadIdx.x; r < R; r += stride) {
        const double a = (double)active[r];
        if (a == 0.0) continue;                        // inactive rows contribute nothing (and may hold any value)
        const double lr = dsub((double)logp[r], (double)old_logp[r]);
        const double ratio = exp(lr);
        const double vt = (double)v_target[r], e = dsub(vt, (double)value[r]);
        s[0] = dadd(s[0], a);
        s[1] = dadd(s[1], dmul(a, (double)entropy[r]));
        s[2] = dsub(s[2], dmul(a, lr));
        s[3] = dadd(s[3], dmul(a, dsub(dsub(ratio, 1.0), lr)));
        if (fabs(dsub(ratio, 1.0)) > eps) s[4] = dadd(s[4], a);
        s[kMaxLr] = fmax(s[kMaxLr], lr);
        s[kMinLr] = fmin(s[kMinLr], lr);
        s[8] = dadd(s[8], dmul(a, vt));
        s[9] = dadd(s[9], dmul(a, dmul(vt, vt)));
        s[10] = dadd(s[10], dmul(a, e));
        s[11] = dadd(s[11], dmul(a, dmul(e, e)));
        if (v_old) {
            const double vo = (double)v_old[r], x = dsub(vt, vo);
            if (fabs(dsub((double)value[r], vo)) > eps) s[7] = dadd(s[7], a);
            s[12] = dadd(s[12], dmul(a, x));
            s[13] = dadd(s[13], dmul(a, dmul(x, x)));
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
#pragma unroll
        for (int j = 0; j < kS; ++j) {
            const double t = __shfl_down_sync(0xffffffffu, s[j], o);
            s[j] = j == kMaxLr ? fmax(s[j], t) : (j == kMinLr ? fmin(s[j], t) : dadd(s[j], t));
        }
    }
    __shared__ double s_w[kStatThreads / 32][kS];
    if ((threadIdx.x & 31) == 0) {
#pragma unroll
        for (int j = 0; j < kS; ++j) s_w[threadIdx.x >> 5][j] = s[j];
    }
    __syncthreads();
    if (threadIdx.x < kS) {
        const int j = threadIdx.x;
        double acc = s_w[0][j];
        for (int w = 1; w < kStatThreads / 32; ++w)
            acc = j == kMaxLr ? fmax(acc, s_w[w][j]) : (j == kMinLr ? fmin(acc, s_w[w][j]) : dadd(acc, s_w[w][j]));
        partial[(int64_t)blockIdx.x * kS + j] = acc;
    }
}

// One block: thread (g, j) = (t / kS, t % kS) folds the partials g, g + G, ... of slot j in order, then thread j folds the G
// group results in group order.  Slots 14 and 15 are set from the call's arguments.
__global__ void __launch_bounds__(kStatThreads)
ppo_stats_reduce_kernel(int blocks, const double *__restrict__ partial, int64_t R, int has_v_old, double *__restrict__ sums)
{
    constexpr int G = kStatThreads / kS;
    __shared__ double s_g[G][kS];
    const int j = threadIdx.x % kS, g = threadIdx.x / kS;
    double acc = j == kMaxLr ? -INFINITY : (j == kMinLr ? INFINITY : 0.0);
    for (int b = g; b < blocks; b += G) {
        const double v = partial[(int64_t)b * kS + j];
        acc = j == kMaxLr ? fmax(acc, v) : (j == kMinLr ? fmin(acc, v) : dadd(acc, v));
    }
    s_g[g][j] = acc;
    __syncthreads();
    if (threadIdx.x < kS) {
        double v = s_g[0][j];
        for (int q = 1; q < G; ++q) v = j == kMaxLr ? fmax(v, s_g[q][j]) : (j == kMinLr ? fmin(v, s_g[q][j]) : dadd(v, s_g[q][j]));
        if (j == 14) v = has_v_old ? 1.0 : 0.0;
        if (j == 15) v = (double)R;
        sums[j] = v;
    }
}

// One block: thread j < kS folds slot j of the n_mb minibatch rows in index order; thread kS handles the gradient norms.
__global__ void __launch_bounds__(32)
ppo_stats_combine_kernel(int n_mb, const double *__restrict__ mb_sums, const float *__restrict__ grad_norms, float max_norm,
                         double *__restrict__ out)
{
    const int j = threadIdx.x;
    if (j < kS) {
        double acc = mb_sums[j];
        for (int m = 1; m < n_mb; ++m) {
            const double v = mb_sums[(int64_t)m * kS + j];
            acc = j == kMaxLr ? fmax(acc, v) : (j == kMinLr ? fmin(acc, v) : dadd(acc, v));
        }
        out[j] = acc;
    } else if (j == kS) {
        double gmax = 0.0, last = 0.0, clipped = 0.0;
        if (grad_norms) {
            for (int m = 0; m < n_mb; ++m) {
                const double g = (double)grad_norms[m];
                gmax = m == 0 ? g : fmax(gmax, g);
                if (g > (double)max_norm) clipped = dadd(clipped, 1.0);
            }
            last = (double)grad_norms[n_mb - 1];
        }
        out[kS + 0] = (double)n_mb;
        out[kS + 1] = grad_norms ? (double)n_mb : 0.0;
        out[kS + 2] = gmax;
        out[kS + 3] = last;
        out[kS + 4] = clipped;
        for (int k = kS + 5; k < MARL_PPO_STATS_OUT; ++k) out[k] = 0.0;
    }
}

}  // namespace marl

using namespace marl;

static_assert(MARL_PPO_STATS_OUT >= MARL_PPO_STATS_SUMS + 5, "combine writes 5 slots after the minibatch sums");

extern "C" int64_t marl_ppo_stats_workspace_bytes(int64_t R)
{
    return R > 0 ? (int64_t)stats_blocks(R) * kS * (int64_t)sizeof(double) : -1;
}

extern "C" int marl_ppo_stats(int64_t R, const float *d_logp, const float *d_old_logp, const float *d_entropy, const float *d_value,
                              const float *d_v_old, const float *d_v_target, const float *d_active, float eps, double *d_sums,
                              void *d_workspace, void *stream)
{
    MARL_REQUIRE(R > 0, "marl_ppo_stats: R=%lld (must be > 0)", (long long)R);
    MARL_REQUIRE(d_logp && d_old_logp && d_entropy && d_value && d_v_target && d_active && d_sums && d_workspace,
                 "marl_ppo_stats: null pointer (only d_v_old may be NULL)");
    MARL_REQUIRE(isfinite(eps) && eps >= 0.f, "marl_ppo_stats: eps=%g (must be finite and >= 0)", (double)eps);
    const int blocks = stats_blocks(R);
    cudaStream_t s = (cudaStream_t)stream;
    double *ws = static_cast<double *>(d_workspace);
    ppo_stats_kernel<<<blocks, kStatThreads, 0, s>>>(R, d_logp, d_old_logp, d_entropy, d_value, d_v_old, d_v_target, d_active,
                                                     (double)eps, ws);
    int rc = check_launch("ppo_stats_kernel");
    if (rc) return rc;
    ppo_stats_reduce_kernel<<<1, kStatThreads, 0, s>>>(blocks, ws, R, d_v_old ? 1 : 0, d_sums);
    return check_launch("ppo_stats_reduce_kernel");
}

extern "C" int marl_ppo_stats_combine(int32_t n_mb, const double *d_mb_sums, const float *d_grad_norms, float max_norm, double *d_out,
                                      void *stream)
{
    MARL_REQUIRE(n_mb >= 1, "marl_ppo_stats_combine: n_mb=%d (must be >= 1)", n_mb);
    MARL_REQUIRE(d_mb_sums && d_out, "marl_ppo_stats_combine: null pointer (only d_grad_norms may be NULL)");
    MARL_REQUIRE(!d_grad_norms || (isfinite(max_norm) && max_norm > 0.f),
                 "marl_ppo_stats_combine: max_norm=%g (must be finite and > 0 with gradient norms)", (double)max_norm);
    ppo_stats_combine_kernel<<<1, 32, 0, (cudaStream_t)stream>>>(n_mb, d_mb_sums, d_grad_norms, max_norm, d_out);
    return check_launch("ppo_stats_combine_kernel");
}

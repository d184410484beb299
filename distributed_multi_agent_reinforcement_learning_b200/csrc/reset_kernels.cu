// reset_kernels.cu — episode initialisation on the device (Pursuit_Env.reset, pursuit_env.py:60-73 -> base_env.py:37-162,
// Occupied_Grid_Map.py:46-62) for thousands of envs: obstacle maps, target, pursuer placement with the chain-connectivity rule,
// evader placement.  In the reference this is ~70 % of the rollout wall time; as host code (maps.py, which reproduces the
// reference's global-RNG draw order bit for bit for the single-env facade) it is ~0.4 ms per env.  Here every env draws from its
// own counter-based stream (splitmix64 of (seed, env, draw index)), so results are rule-equivalent and distribution-equivalent to
// the reference, not stream-equivalent (the reference's interpreter-global Mersenne-Twister streams are inherently serial).
// Rejection sampling is sequential per env and cheap: one thread per env / per map; the work bitmap lives in a global scratch
// row.  The per-map sensor tables are then built by marl_raser_map_build.  The *_dseed entry points and the target-tape draw read the
// seed from a device word when the kernel runs, so a CUDA graph that captures a reset follows that word.  A reset that keeps the maps
// (an installed pool) skips the map and table build and may draw each env's map from the M installed ones (marl_map_draw).
#include "common.cuh"

namespace marl {

struct Stream64 {
    uint64_t key, ctr;
    __device__ __forceinline__ uint64_t next() { return splitmix64(key ^ splitmix64(ctr++)); }
    __device__ __forceinline__ double uniform() { return (double)(next() >> 11) * (1.0 / 9007199254740992.0); }      // [0,1)
    __device__ __forceinline__ int randint(int lo, int hi) { return lo + (int)(uniform() * (double)(hi - lo + 1)); }  // inclusive
    __device__ __forceinline__ void normal2(double mu0, double mu1, double sigma, double &a, double &b)
    {   // Box-Muller
        double u1 = uniform(), u2 = uniform();
        if (u1 < 1e-300) u1 = 1e-300;
        const double r = sqrt(-2.0 * log(u1)), th = 6.283185307179586 * u2;
        a = mu0 + sigma * r * cos(th);
        b = mu1 + sigma * r * sin(th);
    }
};

__device__ __forceinline__ bool bit_get(const uint32_t *bits, int HW, int x, int y) { return (bits[x * HW + (y >> 5)] >> (y & 31)) & 1u; }
__device__ __forceinline__ void bit_set(uint32_t *bits, int HW, int x, int y) { bits[x * HW + (y >> 5)] |= 1u << (y & 31); }

// base_env.py:37-50 + Occupied_Grid_Map.py:46-62: blocks of x,y in [-3,3) around N(center, variance); then the 2-cell inflation
__global__ void __launch_bounds__(64)
map_generate_kernel(EnvDev c, int M, int num_blocks, double cx, double cy, double sigma, uint64_t seed, const uint64_t *__restrict__ d_seed,
                    uint32_t *__restrict__ grid_bits, uint32_t *__restrict__ inflated_bits)
{
    const int m = blockIdx.x * 64 + threadIdx.x;
    if (m >= M) return;
    if (d_seed) seed = *d_seed;      // device-seeded launch (graph-capturable: the seed is read when the kernel runs)
    uint32_t *g = grid_bits + (size_t)m * c.W * c.HW, *inf = inflated_bits + (size_t)m * c.W * c.HW;
    for (int i = 0; i < c.W * c.HW; ++i) { g[i] = 0u; inf[i] = 0u; }
    Stream64 rng{splitmix64(seed ^ 0x6d61707300000000ull) ^ splitmix64((uint64_t)m), 0};
    for (int b = 0; b < num_blocks; ++b) {
        double a0, a1;
        rng.normal2(cx, cy, sigma, a0, a1);
        for (int ox = -3; ox < 3; ++ox)
            for (int oy = -3; oy < 3; ++oy) {
                const int x = pyround((double)ox + a0), y = pyround((double)oy + a1);
                if (x >= 0 && x < c.W && y >= 0 && y < c.H) {
                    bit_set(g, c.HW, x, y);
                    for (int dx = -2; dx <= 2; ++dx)
                        for (int dy = -2; dy <= 2; ++dy) {
                            const int xx = x + dx, yy = y + dy;
                            if (xx >= 0 && xx < c.W && yy >= 0 && yy < c.H) bit_set(inf, c.HW, xx, yy);
                        }
                }
            }
    }
}

// base_env.py:52-152 for one env per thread
__global__ void __launch_bounds__(64)
reset_place_kernel(EnvDev c, int B, const uint32_t *__restrict__ inflated_bits, const int32_t *__restrict__ map_id, uint64_t seed,
                   const uint64_t *__restrict__ d_seed, double min_dist, int extend, double comm_range, double sen_range, int max_draws, double *__restrict__ p_state,
                   double *__restrict__ e_state, int32_t *__restrict__ target, uint32_t *__restrict__ scratch, int32_t *__restrict__ fail)
{
    const int b = blockIdx.x * 64 + threadIdx.x;
    if (b >= B) return;
    if (d_seed) seed = *d_seed;
    const int m = map_id ? map_id[b] : b;
    const uint32_t *inf = inflated_bits + (size_t)m * c.W * c.HW;
    uint32_t *work = scratch + (size_t)b * c.W * c.HW;
    for (int i = 0; i < c.W * c.HW; ++i) work[i] = inf[i];
    Stream64 rng{splitmix64(seed ^ 0x706c616365000000ull) ^ splitmix64((uint64_t)b), 0};
    int draws = 0, failed = 0;
    // target: uniform integer cell, rejected while occupied in the inflated map (base_env.py:52-70)
    int tx = 0, ty = 0;
    for (;;) {
        tx = rng.randint(0, c.W - 1); ty = rng.randint(0, c.H - 1);
        if (!bit_get(inf, c.HW, tx, ty)) break;
        if (++draws > max_draws) { failed = 1; break; }
    }
    target[2 * b] = tx; target[2 * b + 1] = ty;
    // pursuers (base_env.py:72-120): free cell; no earlier pursuer closer than min_dist; 1..2 earlier pursuers within comm range
    const int N = c.N;
    double *ps = p_state + (size_t)b * N * 4;
    int placed = 0;
    while (placed < N && !failed) {
        const double x = rng.uniform() * (double)(c.W - 1), y = rng.uniform() * (double)(c.H - 1);
        if (++draws > max_draws) { failed = 1; break; }
        const int xc = pyround(x), yc = pyround(y);
        if (bit_get(work, c.HW, xc, yc)) continue;
        bool ok = placed == 0;
        if (placed > 0) {
            int close = 0, linked = 0;
            for (int q = 0; q < placed; ++q) {
                const double d = sqrt(sqnorm2(x - ps[4 * q], y - ps[4 * q + 1]));
                close += d < min_dist;
                linked += d < comm_range;
            }
            ok = close == 0 && linked > 0 && linked <= 2;
        }
        if (!ok) continue;
        ps[4 * placed] = x; ps[4 * placed + 1] = y; ps[4 * placed + 2] = 0.0; ps[4 * placed + 3] = 0.0;
        ++placed;
        for (int xx = max(0, xc - extend); xx <= min(c.W - 1, xc + extend); ++xx)
            for (int yy = max(0, yc - extend); yy <= min(c.H - 1, yc + extend); ++yy) bit_set(work, c.HW, xx, yy);
    }
    for (int q = placed; q < N; ++q) { ps[4 * q] = ps[4 * q + 1] = ps[4 * q + 2] = ps[4 * q + 3] = 0.0; }
    // evader (base_env.py:122-152, is_percepted): free point (pursuer footprints count as occupied) within sen_range of a pursuer CELL
    double ex = 0.0, ey = 0.0;
    while (!failed) {
        ex = rng.uniform() * (double)(c.W - 1); ey = rng.uniform() * (double)(c.H - 1);
        if (++draws > max_draws) { failed = 1; break; }
        if (bit_get(work, c.HW, pyround(ex), pyround(ey))) continue;
        bool seen = false;
        for (int q = 0; q < N; ++q) seen |= sqrt(sqnorm2((double)pyround(ps[4 * q]) - ex, (double)pyround(ps[4 * q + 1]) - ey)) < sen_range;
        if (seen) break;
    }
    e_state[4 * b] = ex; e_state[4 * b + 1] = ey; e_state[4 * b + 2] = 0.0; e_state[4 * b + 3] = 0.0;
    if (fail) fail[b] = failed;
}

// candidate-target tape of the mid-episode init_target (base_env.py:52-70): tape[b, l] = (randint(0, W-1), randint(0, H-1)), the
// distribution of the torch draw in BatchedPursuitEnv.reset_device, from env b's own stream of (seed, b)
__global__ void __launch_bounds__(64)
target_tape_kernel(int B, int L, int W, int H, const uint64_t *__restrict__ d_seed, int32_t *__restrict__ tape)
{
    const int b = blockIdx.x * 64 + threadIdx.x;
    if (b >= B) return;
    Stream64 rng{splitmix64(*d_seed ^ 0x7461706500000000ull) ^ splitmix64((uint64_t)b), 0};
    int32_t *row = tape + (size_t)b * L * 2;
    for (int l = 0; l < L; ++l) {
        row[2 * l] = rng.randint(0, W - 1);
        row[2 * l + 1] = rng.randint(0, H - 1);
    }
}

// per-env map draw of a reset that keeps the installed maps: map_id[b] = randint(0, M-1) from env b's own stream of (seed, b)
__global__ void __launch_bounds__(64)
map_draw_kernel(int B, int M, uint64_t seed, const uint64_t *__restrict__ d_seed, int32_t *__restrict__ map_id)
{
    const int b = blockIdx.x * 64 + threadIdx.x;
    if (b >= B) return;
    if (d_seed) seed = *d_seed;
    Stream64 rng{splitmix64(seed ^ 0x6472617700000000ull) ^ splitmix64((uint64_t)b), 0};
    map_id[b] = rng.randint(0, M - 1);
}

}  // namespace marl

using namespace marl;

static int map_generate(const marl_env_params *p, int32_t M, int32_t num_blocks, double center_x, double center_y, double variance,
                        uint64_t seed, const uint64_t *d_seed, uint32_t *d_grid_bits, uint32_t *d_inflated_bits, void *stream)
{
    EnvDev c;
    int rc = make_env_dev(p, &c);
    if (rc) return rc;
    MARL_REQUIRE(M > 0 && num_blocks >= 0 && variance >= 0 && d_grid_bits && d_inflated_bits, "marl_map_generate: bad arguments");
    map_generate_kernel<<<(M + 63) / 64, 64, 0, (cudaStream_t)stream>>>(c, M, num_blocks, center_x, center_y, variance, seed, d_seed, d_grid_bits,
                                                                      d_inflated_bits);
    return check_launch("map_generate_kernel");
}

static int env_reset_place(const marl_env_params *p, int32_t B, int32_t M, const uint32_t *d_inflated_bits, const int32_t *d_map_id,
                           uint64_t seed, const uint64_t *d_seed, double min_dist, int32_t extend, int32_t max_draws, double *d_p_state,
                           double *d_e_state, int32_t *d_target, uint32_t *d_scratch, int32_t *d_fail, void *stream)
{
    EnvDev c;
    int rc = make_env_dev(p, &c);
    if (rc) return rc;
    MARL_REQUIRE(B > 0 && M > 0 && d_inflated_bits && d_p_state && d_e_state && d_target && d_scratch && max_draws > 0 && extend >= 0 && min_dist >= 0,
                 "marl_env_reset_place: bad arguments");
    reset_place_kernel<<<(B + 63) / 64, 64, 0, (cudaStream_t)stream>>>(c, B, d_inflated_bits, d_map_id, seed, d_seed, min_dist, extend,
                                                                      p->d_comm_range, p->d_sen_range, max_draws, d_p_state, d_e_state, d_target,
                                                                      d_scratch, d_fail);
    return check_launch("reset_place_kernel");
}

extern "C" int marl_map_generate(const marl_env_params *p, int32_t M, int32_t num_blocks, double center_x, double center_y, double variance,
                                 uint64_t seed, uint32_t *d_grid_bits, uint32_t *d_inflated_bits, void *stream)
{
    return map_generate(p, M, num_blocks, center_x, center_y, variance, seed, nullptr, d_grid_bits, d_inflated_bits, stream);
}

extern "C" int marl_map_generate_dseed(const marl_env_params *p, int32_t M, int32_t num_blocks, double center_x, double center_y,
                                       double variance, const uint64_t *d_seed, uint32_t *d_grid_bits, uint32_t *d_inflated_bits, void *stream)
{
    MARL_REQUIRE(d_seed != nullptr, "marl_map_generate_dseed: d_seed is NULL");
    return map_generate(p, M, num_blocks, center_x, center_y, variance, 0, d_seed, d_grid_bits, d_inflated_bits, stream);
}

extern "C" int marl_env_reset_place(const marl_env_params *p, int32_t B, int32_t M, const uint32_t *d_inflated_bits, const int32_t *d_map_id,
                                    uint64_t seed, double min_dist, int32_t extend, int32_t max_draws, double *d_p_state, double *d_e_state,
                                    int32_t *d_target, uint32_t *d_scratch, int32_t *d_fail, void *stream)
{
    return env_reset_place(p, B, M, d_inflated_bits, d_map_id, seed, nullptr, min_dist, extend, max_draws, d_p_state, d_e_state, d_target,
                           d_scratch, d_fail, stream);
}

extern "C" int marl_env_reset_place_dseed(const marl_env_params *p, int32_t B, int32_t M, const uint32_t *d_inflated_bits,
                                          const int32_t *d_map_id, const uint64_t *d_seed, double min_dist, int32_t extend, int32_t max_draws,
                                          double *d_p_state, double *d_e_state, int32_t *d_target, uint32_t *d_scratch, int32_t *d_fail,
                                          void *stream)
{
    MARL_REQUIRE(d_seed != nullptr, "marl_env_reset_place_dseed: d_seed is NULL");
    return env_reset_place(p, B, M, d_inflated_bits, d_map_id, 0, d_seed, min_dist, extend, max_draws, d_p_state, d_e_state, d_target,
                           d_scratch, d_fail, stream);
}

extern "C" int marl_target_tape_generate(const marl_env_params *p, int32_t B, int32_t L, const uint64_t *d_seed, int32_t *d_tape, void *stream)
{
    EnvDev c;
    int rc = make_env_dev(p, &c);
    if (rc) return rc;
    MARL_REQUIRE(B > 0 && L > 0 && d_seed && d_tape, "marl_target_tape_generate: bad arguments (B=%d L=%d)", B, L);
    target_tape_kernel<<<(B + 63) / 64, 64, 0, (cudaStream_t)stream>>>(B, L, c.W, c.H, d_seed, d_tape);
    return check_launch("target_tape_kernel");
}

static int map_draw(const marl_env_params *p, int32_t B, int32_t M, uint64_t seed, const uint64_t *d_seed, int32_t *d_map_id, void *stream)
{
    EnvDev c;
    int rc = make_env_dev(p, &c);
    if (rc) return rc;
    MARL_REQUIRE(B > 0 && M > 0 && d_map_id, "marl_map_draw: bad arguments (B=%d M=%d d_map_id=%p)", B, M, (void *)d_map_id);
    map_draw_kernel<<<(B + 63) / 64, 64, 0, (cudaStream_t)stream>>>(B, M, seed, d_seed, d_map_id);
    return check_launch("map_draw_kernel");
}

extern "C" int marl_map_draw(const marl_env_params *p, int32_t B, int32_t M, uint64_t seed, int32_t *d_map_id, void *stream)
{
    return map_draw(p, B, M, seed, nullptr, d_map_id, stream);
}

extern "C" int marl_map_draw_dseed(const marl_env_params *p, int32_t B, int32_t M, const uint64_t *d_seed, int32_t *d_map_id, void *stream)
{
    MARL_REQUIRE(d_seed != nullptr, "marl_map_draw_dseed: d_seed is NULL");
    return map_draw(p, B, M, 0, d_seed, d_map_id, stream);
}

// sensor_maps.cu — kernel 2b: per-map boundary list + "raser" visibility table (pursuit_env.py:18-53).
// One CTA per map; the whole W*H boundary bitmap and the cell->list-index table live in shared memory.
#include "common.cuh"

namespace marl {

static constexpr int kMapThreads = 256;

__global__ void __launch_bounds__(kMapThreads)
raser_map_kernel(EnvDev c, const uint32_t *__restrict__ grid_bits, const double *__restrict__ beam_dir,
                 uint32_t *__restrict__ boundary_bits, int32_t *__restrict__ boundary_count,
                 int32_t *__restrict__ boundary_xy, uint32_t *__restrict__ raser_bits)
{
    extern __shared__ __align__(16) unsigned char smem[];
    const int W = c.W, H = c.H, HW = c.HW, WH = W * H, O = c.O, OW = c.OW;
    int16_t *s_index = reinterpret_cast<int16_t *>(smem);                 // [WH] list index of a boundary cell, -1 else
    uint32_t *s_grid = reinterpret_cast<uint32_t *>(s_index + ((WH + 3) & ~3));   // [W*HW] (both paddings keep s_beam 8-byte aligned)
    double *s_beam = reinterpret_cast<double *>(s_grid + ((W * HW + 1) & ~1));    // [beams*2]
    __shared__ int s_scan[kMapThreads];
    const int m = blockIdx.x, tid = threadIdx.x;
    const uint32_t *grid = grid_bits + (size_t)m * W * HW;
    for (int w = tid; w < W * HW; w += kMapThreads) s_grid[w] = grid[w];
    for (int k = tid; k < 2 * c.sensor_beams; k += kMapThreads) s_beam[k] = beam_dir[k];
    __syncthreads();
    // find_boundaries(mode='inner'), scikit-image 0.19.3 restated: foreground cell whose edge-replicated
    // 4-neighbourhood is not constant.  Cells are enumerated row-major (x*H+y) == np.argwhere order; each thread
    // owns a contiguous chunk so that a block scan of chunk counts yields the argwhere index.
    const int chunk = (WH + kMapThreads - 1) / kMapThreads;
    const int c0 = tid * chunk, c1 = min(WH, c0 + chunk);
    auto is_boundary = [&](int cell) {
        const int x = cell / H, y = cell - x * H;
        if (!grid_bit(s_grid, HW, x, y)) return false;
        const int xm = x > 0 ? x - 1 : 0, xp = x < W - 1 ? x + 1 : W - 1;
        const int ym = y > 0 ? y - 1 : 0, yp = y < H - 1 ? y + 1 : H - 1;
        return !(grid_bit(s_grid, HW, xm, y) && grid_bit(s_grid, HW, xp, y) && grid_bit(s_grid, HW, x, ym) &&
                 grid_bit(s_grid, HW, x, yp));
    };
    int cnt = 0;
    for (int cell = c0; cell < c1; ++cell) cnt += is_boundary(cell) ? 1 : 0;
    s_scan[tid] = cnt;
    __syncthreads();
    for (int o = 1; o < kMapThreads; o <<= 1) {   // Hillis-Steele inclusive scan
        const int v = tid >= o ? s_scan[tid - o] : 0;
        __syncthreads();
        s_scan[tid] += v;
        __syncthreads();
    }
    int idx = s_scan[tid] - cnt;
    const int total = s_scan[kMapThreads - 1];
    for (int cell = c0; cell < c1; ++cell) {
        int16_t v = -1;
        if (is_boundary(cell)) {
            v = (int16_t)idx;
            if (idx < O) {
                boundary_xy[((size_t)m * O + idx) * 2] = cell / H;
                boundary_xy[((size_t)m * O + idx) * 2 + 1] = cell % H;
            }
            ++idx;
        }
        s_index[cell] = v;
    }
    for (int k = total + tid; k < O; k += kMapThreads) {
        boundary_xy[((size_t)m * O + k) * 2] = 0;
        boundary_xy[((size_t)m * O + k) * 2 + 1] = 0;
    }
    if (tid == 0) boundary_count[m] = total;
    __syncthreads();
    // boundary bitmap in the grid layout
    for (int w = tid; w < W * HW; w += kMapThreads) {
        const int x = w / HW, y0 = (w - x * HW) * 32;
        uint32_t bits = 0;
        for (int b = 0; b < 32 && y0 + b < H; ++b) bits |= (s_index[x * H + y0 + b] >= 0 ? 1u : 0u) << b;
        boundary_bits[(size_t)m * W * HW + w] = bits;
    }
    // get_raser_map (pursuit_env.py:29-53): one thread per cell, 36 beams x radius ranges, fp64 address arithmetic
    // `int(x + r*cos)` exactly as Python evaluates it; beams stop at the map edge or at the first boundary cell.
    for (int cell = tid; cell < WH; cell += kMapThreads) {
        const int x = cell / H, y = cell - x * H;
        uint32_t row[32];   // OW <= 32
        for (int w = 0; w < OW; ++w) row[w] = 0;
        for (int beam = 0; beam < c.sensor_beams; ++beam) {
            const double dx = s_beam[2 * beam], dy = s_beam[2 * beam + 1];
            for (int r = 0; r < c.sensor_radius; ++r) {
                const double cx = dadd((double)x, dmul((double)r, dx)), cy = dadd((double)y, dmul((double)r, dy));
                if (cx < 0.0 || cx >= (double)W || cy < 0.0 || cy >= (double)H) break;
                const int hit = s_index[__double2int_rz(cx) * H + __double2int_rz(cy)];
                if (hit >= 0) {
                    if (hit < O) row[hit >> 5] |= 1u << (hit & 31);
                    break;
                }
            }
        }
        uint32_t *dst = raser_bits + ((size_t)m * WH + cell) * OW;
        for (int w = 0; w < OW; ++w) dst[w] = row[w];
    }
}

}  // namespace marl

using namespace marl;

extern "C" int marl_raser_map_build(const marl_env_params *p, int32_t M, const uint32_t *d_grid_bits,
                                    const double *d_beam_dir, uint32_t *d_boundary_bits, int32_t *d_boundary_count,
                                    int32_t *d_boundary_xy, uint32_t *d_raser_bits, void *stream)
{
    EnvDev c;
    int rc = make_env_dev(p, &c);
    if (rc) return rc;
    MARL_REQUIRE(M > 0, "marl_raser_map_build: M=%d", M);
    MARL_REQUIRE(d_grid_bits && d_beam_dir && d_boundary_bits && d_boundary_count && d_boundary_xy && d_raser_bits,
                 "marl_raser_map_build: null pointer");
    const int WH = c.W * c.H;
    const size_t smem = sizeof(int16_t) * ((WH + 3) & ~3) + sizeof(uint32_t) * ((c.W * c.HW + 1) & ~1) +
                        sizeof(double) * 2 * c.sensor_beams;
    if (smem > 48 * 1024) {
        cudaError_t e = cudaFuncSetAttribute(raser_map_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) { set_error("raser_map: smem %zu: %s", smem, cudaGetErrorString(e)); return MARL_ECUDA; }
    }
    raser_map_kernel<<<M, kMapThreads, smem, (cudaStream_t)stream>>>(c, d_grid_bits, d_beam_dir, d_boundary_bits,
                                                                     d_boundary_count, d_boundary_xy, d_raser_bits);
    return check_launch("raser_map_kernel");
}

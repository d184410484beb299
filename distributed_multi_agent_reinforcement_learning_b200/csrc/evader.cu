// evader.cu — kernel 1c: the A*-driven evader (pursuit_env.py:75-102 attacker_step, agent.py:197-271,
// astar.py:26-161, Occupied_Grid_Map.py:119-191).
//
// Replanning: one warp (= one CTA) per environment, whole search state in shared memory: the blocked-node bitmap
// as CW 64-bit words per x, g (fp64 — exact tie-breaking needs the reference's summation order), parent (u16)
// and the OPEN set.  The search lattice is [0, W] x [0, H], H + 1 rows: CW = 1 for H <= 63, CW = 2 for 64 <= H <= 127 (so
// H = 64 already takes the second word); node ids are x * 64 CW + y.  Shifts along y carry across the words.  heapq's pop order is the total order of (f, (x, y)) tuples (ties only between identical
// items), so ANY correct priority queue pops the same sequence.  The search is one warp walking a dependent chain (about six
// cycles per instruction), so a pop is built to be SHORT and independent of |OPEN|: OPEN is an unsorted shared-memory array cut
// into 32 stripes (slot i belongs to stripe i % 32, stored stripe-major); lane l keeps the minimum of stripe l in registers, so
// a pop is three REDUX steps over those 32 cached minima (order-preserving integer image of f, then node id and slot packed in
// one word) - no scan.  The popped slot is refilled by the first neighbour pushed in the same pop (by the last slot's entry
// when nothing is pushed), further pushes are appended round-robin over the stripes; afterwards only the popped stripe's minimum has to be recomputed, by all
// 32 lanes together (its <= 49 entries are contiguous), and the lanes that own an appended slot fold it into their minimum.
// The 8 neighbours are relaxed by 8 lanes in parallel; blocked nodes carry g = -1 from the start, so `new_cost < g` rejects
// them without a bitmap test.  Obstacle inflation / pursuer inflation / the half-open view window of Evader.rescan are
// separable bit operations on the columns.
#include "evader_move.cuh"

namespace marl {

static constexpr int kStripeCap = 49;               // OPEN entries per stripe; odd, so consecutive slots (different stripes) fall into different banks
static constexpr int kOpenCap = 32 * kStripeCap;    // 1568 entries
static constexpr int kPopBudget = 192;   // pops before the reachability check (p99 of successful searches is ~200; 32 .. 192 time the same)

struct EvaderArgs {
    int B, path_cap, tape_len;
    double *e_state;
    const double *p_state;
    int32_t *target;
    int16_t *path;
    int32_t *path_len;
    const int32_t *time_step;
    const uint32_t *grid_bits, *inflated_bits;
    const int32_t *map_id;
    const int32_t *target_tape;
    int32_t *tape_pos;
    int32_t *status;
    double *e_tape2;   // optional [2,B,4]: evader state before / after this attacker_step
};

// Column x of a bit-packed [W,HW] map as CW 64-bit words (words past HW read as zero)
template <int CW>
__device__ __forceinline__ void col_of(uint64_t (&v)[CW], const uint32_t *bits, int HW, int x)
{
#pragma unroll
    for (int k = 0; k < CW; ++k) {
        v[k] = (k == 0 || 2 * k < HW) ? (uint64_t)bits[x * HW + 2 * k] : 0ull;
        if (2 * k + 1 < HW) v[k] |= (uint64_t)bits[x * HW + 2 * k + 1] << 32;
    }
}

// Mask of the rows [0, n) of word k (n - 64 k >= 0)
__device__ __forceinline__ uint64_t low_rows(int n) { return n >= 64 ? ~0ull : ((1ull << n) - 1ull); }

// Word k of the column shifted by -e..e (Chebyshev inflation along y; bits carry across the words), clipped to H bits.  e <= 8.
template <int CW>
__device__ __forceinline__ uint64_t dilate_y(const uint64_t *c, int k, int e, uint64_t hmask)
{
    uint64_t r = c[k];
    for (int d = 1; d <= e; ++d) {
        r |= (c[k] << d) | (c[k] >> d);
        if (k > 0) r |= c[k - 1] >> (64 - d);
        if (k + 1 < CW) r |= c[k + 1] << (64 - d);
    }
    return r & hmask;
}

// Word and bit of row y in a column of CW words
template <int CW> __device__ __forceinline__ int row_word(int y) { return CW == 1 ? 0 : y >> 6; }
template <int CW> __device__ __forceinline__ int row_bit(int y) { return CW == 1 ? y : y & 63; }

struct SearchSmem {
    double *g;        // [NODES]
    double *of;       // [kOpenCap] f of OPEN entries, stripe-major: slot i at (i % 32) * kStripeCap + i / 32
    uint64_t *mov;    // [W1 * CW]
    uint64_t *blk;    // [W1 * CW], followed by the flood fill's reach [W1 * CW]
    uint16_t *par;    // [NODES]
    uint16_t *on;     // [kOpenCap] node of OPEN entries
};

__device__ __forceinline__ SearchSmem carve(unsigned char *smem, int CWW1, int NODES)
{
    SearchSmem s;
    s.g = reinterpret_cast<double *>(smem);
    s.of = s.g + NODES;
    s.mov = reinterpret_cast<uint64_t *>(s.of + kOpenCap);
    s.blk = s.mov + CWW1;
    s.par = reinterpret_cast<uint16_t *>(s.blk + 2 * CWW1);   // [blk][reach]
    s.on = s.par + ((NODES + 3) & ~3);
    return s;
}

// Node id = x * 64 CW + y: decoding a popped node is a shift and a mask instead of an integer division on the search's
// critical path, and the ids keep heapq's (x, y) tuple order.  Ids stay below (W + 1) * 64 CW <= 65535 (u16 `par` / `on`),
// and node << 11 | slot fits 32 bits (kOpenCap <= 2048).
template <int CW> struct NodeId {
    static constexpr int kShift = 5 + CW, kStride = 1 << kShift;
};
static constexpr size_t search_smem_bytes(int CW, int W)
{
    const size_t W1 = (size_t)W + 1, NODES = W1 * 64 * CW;
    return sizeof(double) * (NODES + kOpenCap) + sizeof(uint64_t) * 3 * CW * W1 + sizeof(uint16_t) * (((NODES + 3) & ~(size_t)3) + kOpenCap);
}
static constexpr size_t kSearchSmemCap = 227 * 1024;   // opt-in shared memory of one block on sm_100
// Map limits of the search: H <= 63 with one word per column, 64 <= H <= 127 with two, whose search state must fit one block's
// shared memory (about 1.3 KB per column plus OPEN: one search per SM at 128 x 128).
static constexpr int kMaxH1 = 63, kMaxW1 = 254, kMaxH2 = 127;
static constexpr int max_search_width(int CW)
{
    int W = 2;
    while (search_smem_bytes(CW, W + 1) <= kSearchSmemCap) ++W;
    return W;
}
static constexpr int kMaxW2 = max_search_width(2);
static_assert(kStripeCap <= 64 && kOpenCap <= 2048, "slot ids are 11 bits and a stripe is read by 2 x 32 lanes");
static_assert(search_smem_bytes(1, kMaxW1) <= kSearchSmemCap, "one-word search must fit at W = kMaxW1");
static_assert((kMaxW1 + 1) * NodeId<1>::kStride <= 65536 && (kMaxW2 + 1) * NodeId<2>::kStride <= 65536, "node ids are u16");

// Is `goal` reachable from `start` through unblocked nodes of the [0,W]x[0,H] lattice with 8-connected moves?
// Bit-parallel flood fill on the columns (one lane per column, in-place monotone OR until the fixed point).
// Used to cut the search short: when the goal is unreachable the reference's A* exhausts the whole component and
// returns [s_start] (astar.py:67-71) — the same answer this gives after a few thousand cycles.
template <int CW>
__device__ bool goal_reachable(const SearchSmem &sm, uint64_t *reach, int W1, int H1, int sx, int sy, int gx, int gy)
{
    const int lane = threadIdx.x & 31;
    uint64_t dom[CW];
#pragma unroll
    for (int k = 0; k < CW; ++k) dom[k] = low_rows(H1 - 64 * k);
    for (int i = lane; i < W1 * CW; i += 32) reach[i] = 0ull;
    __syncwarp();
    if (lane == 0) {
        const int i = sx * CW + row_word<CW>(sy);
        reach[i] = (1ull << row_bit<CW>(sy)) & ~sm.blk[i];
    }
    __syncwarp();
    for (;;) {
        bool changed = false;
        for (int x = lane; x < W1; x += 32) {
            uint64_t c[CW], nb[CW];
#pragma unroll
            for (int k = 0; k < CW; ++k) {
                c[k] = reach[x * CW + k];
                nb[k] = c[k];
                if (x > 0) nb[k] |= reach[(x - 1) * CW + k];
                if (x + 1 < W1) nb[k] |= reach[(x + 1) * CW + k];
            }
#pragma unroll
            for (int k = 0; k < CW; ++k) {
                uint64_t sh = (nb[k] << 1) | (nb[k] >> 1);
                if (k > 0) sh |= nb[k - 1] >> 63;
                if (k + 1 < CW) sh |= nb[k + 1] << 63;
                const uint64_t nw = (c[k] | nb[k] | sh) & ~sm.blk[x * CW + k] & dom[k];
                if (nw != c[k]) { reach[x * CW + k] = nw; changed = true; }
            }
        }
        __syncwarp();
        if ((reach[gx * CW + row_word<CW>(gy)] >> row_bit<CW>(gy)) & 1ull) return true;
        if (!__any_sync(0xffffffffu, changed)) return false;
    }
}

// Evader.replan (agent.py:232-259) for one env by one warp.  Returns the new path length (uniform across lanes);
// path receives [goal, ..., start].
template <int CW>
__device__ int replan_warp(const EnvDev &c, const SearchSmem &sm, const uint32_t *__restrict__ grid,
                           const double *__restrict__ p_state, int N, double ex, double ey, int tx, int ty,
                           int16_t *__restrict__ path, int path_cap, int &status)
{
    const int lane = threadIdx.x & 31;
    constexpr int kNodeShift = NodeId<CW>::kShift, kNodeStride = NodeId<CW>::kStride;
    const int W = c.W, H = c.H, W1 = W + 1, H1 = H + 1;
    uint64_t hmask[CW];
#pragma unroll
    for (int k = 0; k < CW; ++k) hmask[k] = low_rows(H - 64 * k);
    const int cx = pyround(ex), cy = pyround(ey);
    for (int i = lane; i < W1 * CW; i += 32) sm.mov[i] = 0ull;
    __syncwarp();
    for (int i = lane; i < N; i += 32) {   // set_moving_obstacle (Occupied_Grid_Map.py:119-124)
        const int mx = pyround(p_state[i * 4]), my = pyround(p_state[i * 4 + 1]);
        atomicOr((unsigned long long *)&sm.mov[mx * CW + row_word<CW>(my)], 1ull << row_bit<CW>(my));
    }
    __syncwarp();
    const int ux = (lane == 0 || lane == 1 || lane == 7) ? -1 : ((lane >= 3 && lane <= 5) ? 1 : 0);   // astar.py:11-12
    const int uy = (lane >= 1 && lane <= 3) ? 1 : ((lane >= 5 && lane <= 7) ? -1 : 0);
    const double step_cost = (ux != 0 && uy != 0) ? sqrt(2.0) : 1.0;   // math.hypot(1, 1)
    const int dn = ux * kNodeStride + uy;
    const int start = (cx << kNodeShift) | cy, goal = (tx << kNodeShift) | ty;
    int n_path = 1;
    for (int e = c.e_extend_dis; e >= 0; --e) {
        // ---- Evader.rescan (agent.py:202-230) as column algebra ----
        for (int x = lane; x < W1; x += 32) {
            uint64_t st[CW], pr[CW], view[CW];
#pragma unroll
            for (int k = 0; k < CW; ++k) st[k] = pr[k] = view[k] = 0ull;
            for (int xx = max(0, x - e); xx <= min(W - 1, x + e); ++xx) {
                uint64_t gc[CW];
                col_of<CW>(gc, grid, c.HW, xx);
#pragma unroll
                for (int k = 0; k < CW; ++k) {
                    st[k] |= dilate_y<CW>(gc, k, e, hmask[k]);
                    pr[k] |= dilate_y<CW>(sm.mov + xx * CW, k, e, hmask[k]);
                }
            }
            if (x >= W) {
#pragma unroll
                for (int k = 0; k < CW; ++k) st[k] = pr[k] = 0ull;
            }
            // local_observation: half-open window [p-R, p+R) intersected with the disc d2 <= R^2 (at most 2R <= 64 rows)
            const int R = c.e_sen_range, dx = cx - x;
            if (x < W && x >= cx - R && x < cx + R) {
                const int rem = c.e_view2_floor - dx * dx;
                if (rem >= 0) {
                    int k = 0;
                    while ((k + 1) * (k + 1) <= rem) ++k;
                    const int y0 = max(max(cy - k, cy - R), 0), y1 = min(min(cy + k, cy + R - 1), H - 1);
#pragma unroll
                    for (int w = 0; w < CW; ++w) {   // rows [y0, y1] of word w
                        const int a = CW == 1 ? y0 : max(y0 - 64 * w, 0), b = CW == 1 ? y1 : min(y1 - 64 * w, 63);
                        if (b >= a) view[w] = low_rows(b - a + 1) << a;
                    }
                }
            }
#pragma unroll
            for (int k = 0; k < CW; ++k) sm.blk[x * CW + k] = st[k] | (view[k] & pr[k]);
        }
        __syncwarp();
        // g: +inf on free nodes, -1 on blocked ones (column-wise: lane l writes rows l + 32 j of every column)
        for (int x = 0; x < W1; ++x) {
#pragma unroll
            for (int k = 0; k < CW; ++k) {
                const uint64_t col = sm.blk[x * CW + k];
                const unsigned lo = (unsigned)col, hi = (unsigned)(col >> 32);
                sm.g[(x << kNodeShift) + 64 * k + lane] = ((lo >> lane) & 1u) ? -1.0 : (double)INFINITY;
                sm.g[(x << kNodeShift) + 64 * k + 32 + lane] = ((hi >> lane) & 1u) ? -1.0 : (double)INFINITY;
            }
        }
        __syncwarp();
        // ---- AStar_2D.searching (astar.py:26-73) ----
        n_path = 1;
        const bool goal_blocked = (sm.blk[tx * CW + row_word<CW>(ty)] >> row_bit<CW>(ty)) & 1ull;
        // a blocked start expands nothing (astar.py:56-60 tests both ends of every move): OPEN runs empty after the first pop
        const bool start_blocked = (sm.blk[cx * CW + row_word<CW>(cy)] >> row_bit<CW>(cy)) & 1ull;
        if (!goal_blocked && !start_blocked) {
            unsigned long long *const ofb = reinterpret_cast<unsigned long long *>(sm.of);
            unsigned c_hi = 0xffffffffu, c_lo = 0xffffffffu, c_tag = 0xffffffffu;   // minimum of this lane's stripe: f bits, node << 11 | slot
            if (lane == 0) {
                const double f0 = 0.0 + 2.5 * (double)(abs(tx - cx) + abs(ty - cy));
                sm.g[start] = 0.0;
                sm.par[start] = (uint16_t)start;
                sm.of[0] = f0;
                sm.on[0] = (uint16_t)start;
                const unsigned long long k0 = (unsigned long long)__double_as_longlong(f0);     // f >= 0: order-preserving
                c_hi = (unsigned)(k0 >> 32); c_lo = (unsigned)k0; c_tag = (unsigned)start << 11;
            }
            int extent = 1, pops = 0;   // slots [0, extent) are in use
            __syncwarp();
            bool reached = false;
            for (;;) {
                if (++pops == kPopBudget) {   // long search: make sure it can succeed before spending more on it
                    if (!goal_reachable<CW>(sm, sm.blk + W1 * CW, W1, H1, cx, cy, tx, ty)) break;
                }
                // ---- pop: arg-min of (f, node) over the 32 cached stripe minima ----
                const unsigned mhi = __reduce_min_sync(0xffffffffu, c_hi);
                if (mhi == 0xffffffffu) break;                       // OPEN is empty
                const bool c1 = c_hi == mhi;
                const unsigned mlo = __reduce_min_sync(0xffffffffu, c1 ? c_lo : 0xffffffffu);
                const unsigned tag = __reduce_min_sync(0xffffffffu, (c1 && c_lo == mlo) ? c_tag : 0xffffffffu);
                const int s = (int)(tag >> 11), slot = (int)(tag & 2047u);
                if (s == goal) { reached = true; break; }
                const int o = slot & 31, jpop = slot >> 5;           // the popped entry: stripe o, position jpop
                // ---- (R) the minimum of stripe o WITHOUT the popped entry: all lanes read its (contiguous) entries.  Independent of
                // the relaxation (B) below - the two dependent chains are written interleaved so that they overlap ----
                const int len_o = (extent - o + 31) >> 5;            // slots o, o + 32, ... below extent (<= kStripeCap <= 64)
                unsigned b_hi = 0xffffffffu, b_lo = 0xffffffffu, b_tag = 0xffffffffu;
                {
                    const int j0 = lane, j1 = lane + 32;
                    const bool v0 = j0 < len_o && j0 != jpop, v1 = j1 < len_o && j1 != jpop;
                    unsigned long long k0 = ~0ull, k1 = ~0ull;
                    unsigned t0 = 0xffffffffu, t1 = 0xffffffffu;
                    if (v0) { const int p = o * kStripeCap + j0; k0 = ofb[p]; t0 = ((unsigned)sm.on[p] << 11) | (unsigned)((j0 << 5) | o); }
                    if (v1) { const int p = o * kStripeCap + j1; k1 = ofb[p]; t1 = ((unsigned)sm.on[p] << 11) | (unsigned)((j1 << 5) | o); }
                    const bool second = k1 < k0 || (k1 == k0 && t1 < t0);
                    const unsigned long long kb = second ? k1 : k0;
                    b_hi = (unsigned)(kb >> 32); b_lo = (unsigned)kb; b_tag = second ? t1 : t0;
                }
                // ---- (B) relax the 8 neighbours (astar.py:56-65) on lanes 0..7 ----
                const int sx = s >> kNodeShift, sy = s & (kNodeStride - 1);
                const int nx = sx + ux, ny = sy + uy;
                const bool inside = lane < 8 && (unsigned)nx <= (unsigned)W && (unsigned)ny <= (unsigned)H;
                const int nn = inside ? s + dn : s;                  // (outside: re-reads g[s], which new_cost never beats)
                const double g_s = sm.g[s], g_n = sm.g[nn];
                const unsigned rhi = __reduce_min_sync(0xffffffffu, b_hi);                                   // (R)
                const double nc = dadd(g_s, step_cost);                                                      // (B)
                const bool r1 = b_hi == rhi;
                const unsigned rlo = __reduce_min_sync(0xffffffffu, r1 ? b_lo : 0xffffffffu);                // (R)
                const bool push = inside && nc < g_n;                                                        // (B)
                const double nf = __fma_rn(2.5, (double)(abs(tx - nx) + abs(ty - ny)), nc);                  // 2.5 h is exact: same bits as nc + 2.5 * h
                const unsigned rtag = __reduce_min_sync(0xffffffffu, (r1 && b_lo == rlo) ? b_tag : 0xffffffffu);   // (R)
                if (push) {
                    sm.g[nn] = nc;
                    sm.par[nn] = (uint16_t)s;
                }
                const unsigned pm = __ballot_sync(0xffffffffu, push);
                const int n_push = __popc(pm);
                const int n_app = max(n_push - 1, 0);
                if (extent + n_app > kOpenCap) { status |= EV_HEAP_OVERFLOW; break; }
                if (n_push == 0) {
                    // ---- dead end (one pop in ten): the last slot's entry moves into the hole; the two stripes involved are re-read ----
                    const int last = extent - 1;
                    if (slot != last && lane == 0) {
                        const int ps = o * kStripeCap + jpop, pl = (last & 31) * kStripeCap + (last >> 5);
                        ofb[ps] = ofb[pl];
                        sm.on[ps] = sm.on[pl];
                    }
                    extent = last;
                    const int o2 = last & 31;
                    __syncwarp();
                    for (int st = o;;) {
                        const int len = (extent - st + 31) >> 5;
                        unsigned q_hi = 0xffffffffu, q_lo = 0xffffffffu, q_tag = 0xffffffffu;
                        for (int j = lane; j < len; j += 32) {
                            const int p = st * kStripeCap + j;
                            const unsigned long long k = ofb[p];
                            const unsigned t = ((unsigned)sm.on[p] << 11) | (unsigned)((j << 5) | st);
                            const unsigned khi = (unsigned)(k >> 32), klo = (unsigned)k;
                            if (khi < q_hi || (khi == q_hi && (klo < q_lo || (klo == q_lo && t < q_tag)))) { q_hi = khi; q_lo = klo; q_tag = t; }
                        }
                        const unsigned uhi = __reduce_min_sync(0xffffffffu, q_hi);
                        const bool u1 = q_hi == uhi;
                        const unsigned ulo = __reduce_min_sync(0xffffffffu, u1 ? q_lo : 0xffffffffu);
                        const unsigned utag = __reduce_min_sync(0xffffffffu, (u1 && q_lo == ulo) ? q_tag : 0xffffffffu);
                        if (lane == st) { c_hi = uhi; c_lo = ulo; c_tag = utag; }
                        if (o2 == st) break;
                        st = o2;                                     // the stripe that lost its last slot
                    }
                    continue;
                }
                if (lane == o) { c_hi = rhi; c_lo = rlo; c_tag = rtag; }
                if (push) {   // the first pusher refills the popped slot, the others append
                    const int rank = __popc(pm & ((1u << lane) - 1u));
                    const int i = rank == 0 ? slot : extent + rank - 1;
                    const int p = (i & 31) * kStripeCap + (i >> 5);
                    sm.of[p] = nf;
                    sm.on[p] = (uint16_t)nn;
                }
                __syncwarp();
                {   // the new entries are folded into their stripes' minima: lane o takes the refilled slot, the owner of an appended slot that one
                    const int d = (lane - extent) & 31;
                    const bool app = d < n_app;
                    const int ia = extent + d;
                    if (app) {
                        const int p = lane * kStripeCap + (ia >> 5);
                        const unsigned long long k = ofb[p];
                        const unsigned t = ((unsigned)sm.on[p] << 11) | (unsigned)ia;
                        const unsigned khi = (unsigned)(k >> 32), klo = (unsigned)k;
                        if (khi < c_hi || (khi == c_hi && (klo < c_lo || (klo == c_lo && t < c_tag)))) { c_hi = khi; c_lo = klo; c_tag = t; }
                    }
                    if (lane == o) {
                        const int p = o * kStripeCap + jpop;
                        const unsigned long long k = ofb[p];
                        const unsigned t = ((unsigned)sm.on[p] << 11) | (unsigned)slot;
                        const unsigned khi = (unsigned)(k >> 32), klo = (unsigned)k;
                        if (khi < c_hi || (khi == c_hi && (klo < c_lo || (klo == c_lo && t < c_tag)))) { c_hi = khi; c_lo = klo; c_tag = t; }
                    }
                }
                extent += n_app;
            }
            if (reached) {   // extract_path (astar.py:130-146): [goal, ..., start]
                if (lane == 0) {
                    int cur = goal, n = 1;
                    path[0] = (int16_t)tx;
                    path[1] = (int16_t)ty;
                    for (;;) {
                        const int par = sm.par[cur];
                        if (n < path_cap) {
                            path[2 * n] = (int16_t)(par >> kNodeShift);
                            path[2 * n + 1] = (int16_t)(par & (kNodeStride - 1));
                        }
                        ++n;
                        cur = par;
                        if (cur == start) break;
                    }
                    if (n > path_cap) { status |= EV_PATH_OVERFLOW; n = path_cap; }
                    n_path = n;
                }
                n_path = __shfl_sync(0xffffffffu, n_path, 0);
            }
        }
        if (n_path < 2 && lane == 0) {
            path[0] = (int16_t)cx;
            path[1] = (int16_t)cy;
        }
        __syncwarp();
        if (n_path >= 2) break;
    }
    status = __shfl_sync(0xffffffffu, status, 0) | status;
    return n_path;
}

// One attacker_step per env: replan when due, then move.  (Per-step API; the closed-loop rollout uses
// evader_replan_kernel + the move fused into rollout_kernel instead.)
template <int CW>
__global__ void __launch_bounds__(32)
evader_kernel(EnvDev c, EvaderArgs r, int replan_only)
{
    extern __shared__ __align__(16) unsigned char smem[];
    const int b = blockIdx.x, lane = threadIdx.x;
    if (b >= r.B) return;
    const int ts = r.time_step[b];
    const bool due = (ts % c.difficulty) == 0;
    if (replan_only && !due) return;
    const int m = r.map_id ? r.map_id[b] : b;
    const uint32_t *grid = r.grid_bits + (size_t)m * c.W * c.HW;
    EvaderRegs s;
    s.x = r.e_state[4 * b]; s.y = r.e_state[4 * b + 1]; s.vx = r.e_state[4 * b + 2]; s.vy = r.e_state[4 * b + 3];
    s.tx = r.target[2 * b]; s.ty = r.target[2 * b + 1];
    s.plen = r.path_len[b];
    s.status = 0;
    int16_t *path = r.path + (size_t)b * r.path_cap * 2;
    if (due) {
        const SearchSmem sm = carve(smem, (c.W + 1) * CW, (c.W + 1) * NodeId<CW>::kStride);
        s.plen = replan_warp<CW>(c, sm, grid, r.p_state + (size_t)b * c.N * 4, c.N, s.x, s.y, s.tx, s.ty, path, r.path_cap, s.status);
    }
    if (lane == 0) {
        if (!replan_only) {
            const double ox = s.x, oy = s.y, ovx = s.vx, ovy = s.vy;
            s.tape_pos = r.tape_pos[b];
            evader_move(c, grid, r.inflated_bits + (size_t)m * c.W * c.HW, path, r.target_tape + (size_t)b * r.tape_len * 2,
                        r.tape_len, s);
            r.e_state[4 * b] = s.x; r.e_state[4 * b + 1] = s.y; r.e_state[4 * b + 2] = s.vx; r.e_state[4 * b + 3] = s.vy;
            r.target[2 * b] = s.tx; r.target[2 * b + 1] = s.ty;
            r.tape_pos[b] = s.tape_pos;
            if (r.e_tape2) {   // 2-slot tape for marl_rollout_steps(K=1): [0]=before, [1]=after attacker_step
                double *t0 = r.e_tape2 + 4 * (size_t)b, *t1 = r.e_tape2 + 4 * ((size_t)r.B + b);
                t0[0] = ox; t0[1] = oy; t0[2] = ovx; t0[3] = ovy;
                t1[0] = s.x; t1[1] = s.y; t1[2] = s.vx; t1[3] = s.vy;
            }
        }
        r.path_len[b] = s.plen;
        if (r.status && s.status) r.status[b] |= s.status;
    }
}

static int launch_evader(const marl_env_params *p, int32_t B, int32_t M, EvaderArgs &r, int replan_only, void *stream)
{
    EnvDev c;
    int rc = make_env_dev(p, &c);
    if (rc) return rc;
    MARL_REQUIRE(B > 0 && M > 0 && r.path_cap >= 2 && r.tape_len >= 0, "marl_evader: B=%d M=%d path_cap=%d", B, M, r.path_cap);
    MARL_REQUIRE(r.map_id || M >= B, "marl_evader: map_id is NULL but M < B");
    const int CW = c.H <= kMaxH1 ? 1 : 2;   // the lattice has H + 1 rows: H = 64 already needs a second word
    if (c.H > kMaxH2 || c.W > (CW == 1 ? kMaxW1 : kMaxW2)) {
        set_error("marl_evader: map %dx%d unsupported by the column-bitmap search (H <= %d needs W <= %d, H <= %d needs W <= %d)",
                  c.W, c.H, kMaxH1, kMaxW1, kMaxH2, kMaxW2);
        return MARL_EUNSUPPORTED;
    }
    const size_t smem = search_smem_bytes(CW, c.W);
    MARL_REQUIRE(smem <= kSearchSmemCap, "marl_evader: %zu B shared memory needed", smem);
    const void *kern = CW == 1 ? (const void *)evader_kernel<1> : (const void *)evader_kernel<2>;
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) { set_error("evader: smem %zu: %s", smem, cudaGetErrorString(e)); return MARL_ECUDA; }
    r.B = B;
    if (CW == 1)
        evader_kernel<1><<<B, 32, smem, (cudaStream_t)stream>>>(c, r, replan_only);
    else
        evader_kernel<2><<<B, 32, smem, (cudaStream_t)stream>>>(c, r, replan_only);
    return check_launch("evader_kernel");
}

}  // namespace marl

using namespace marl;

extern "C" int marl_evader_step(const marl_env_params *p, int32_t B, int32_t M, double *d_e_state,
                                const double *d_p_state, int32_t *d_target, int16_t *d_path, int32_t *d_path_len,
                                int32_t path_cap, const int32_t *d_time_step, const uint32_t *d_grid_bits,
                                const uint32_t *d_inflated_bits, const int32_t *d_map_id, const int32_t *d_target_tape,
                                int32_t tape_len, int32_t *d_tape_pos, int32_t *d_status, double *d_e_tape2, void *stream)
{
    if (!(d_e_state && d_p_state && d_target && d_path && d_path_len && d_time_step && d_grid_bits && d_inflated_bits &&
          d_tape_pos && (d_target_tape || tape_len == 0))) {
        set_error("marl_evader_step: null pointer");
        return MARL_EINVAL;
    }
    EvaderArgs r;
    r.path_cap = path_cap; r.tape_len = tape_len;
    r.e_state = d_e_state; r.p_state = d_p_state; r.target = d_target; r.path = d_path; r.path_len = d_path_len;
    r.time_step = d_time_step; r.grid_bits = d_grid_bits; r.inflated_bits = d_inflated_bits; r.map_id = d_map_id;
    r.target_tape = d_target_tape; r.tape_pos = d_tape_pos; r.status = d_status; r.e_tape2 = d_e_tape2;
    return launch_evader(p, B, M, r, 0, stream);
}

extern "C" int marl_evader_replan(const marl_env_params *p, int32_t B, int32_t M, const double *d_e_state,
                                  const double *d_p_state, const int32_t *d_target, int16_t *d_path,
                                  int32_t *d_path_len, int32_t path_cap, const int32_t *d_time_step,
                                  const uint32_t *d_grid_bits, const int32_t *d_map_id, int32_t *d_status, void *stream)
{
    if (!(d_e_state && d_p_state && d_target && d_path && d_path_len && d_time_step && d_grid_bits)) {
        set_error("marl_evader_replan: null pointer");
        return MARL_EINVAL;
    }
    EvaderArgs r;
    r.path_cap = path_cap; r.tape_len = 0;
    r.e_state = const_cast<double *>(d_e_state); r.p_state = d_p_state; r.target = const_cast<int32_t *>(d_target);
    r.path = d_path; r.path_len = d_path_len; r.time_step = d_time_step; r.grid_bits = d_grid_bits;
    r.inflated_bits = nullptr; r.map_id = d_map_id; r.target_tape = nullptr; r.tape_pos = nullptr; r.status = d_status;
    r.e_tape2 = nullptr;
    return launch_evader(p, B, M, r, 1, stream);
}

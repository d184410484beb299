// msg_args.cuh — argument block shared by the DHGN message kernels (policy_kernels.cu, msg_grouped.cu).
#pragma once
#include "common.cuh"

namespace marl {

struct MsgArgs {
    int S, N, O, NW, OW;
    const float *p;            // [S,N,4]
    const float *e;            // [S,4]
    const float *oxy;          // [Bo,O,2] obstacle-cell coordinates (vx=vy=0 implied, pursuit_env.py:22-26)
    const int32_t *o_index;    // [S] row of oxy for this sample
    const int32_t *o_count;    // [Bo] slots that exist for all-ones adjacency (critic): O_b in rollout, O in training
    const uint32_t *p_adj;     // [S,N,NW] or null when all_ones
    const uint8_t *e_adj;      // [S,N]
    const uint32_t *o_adj;     // [S,N,OW]
    int all_ones;              // critic: AttributeDataset(is_critic=True) (mappo_parallel.py:64-65)
};

// sample-grouped kernels (msg_grouped.cu): E = 128, N <= 16, O <= 256; return MARL_EUNSUPPORTED otherwise
int launch_msg_fwd_grouped(const MsgArgs &a, const float *W0, const float *b0, const float *W1, const float *b1, const float *W2,
                           const float *b2, float *agg, cudaStream_t stream);
// ws == nullptr: every CTA adds its sums into gW / gb with atomics.  Otherwise CTA b of the launch of relation r writes its
// (KW_r + 1) x E sums (KW = 8, 4, 4) to ws + blocks * E * {0, 9, 14}[r] + b * (KW_r + 1) * E and nothing else;
// launch_msg_partials_reduce adds them.
int launch_msg_bwd_grouped(const MsgArgs &a, const float *W0, const float *b0, const float *W1, const float *b1, const float *W2,
                           const float *b2, const float *d_agg, float *gW0, float *gb0, float *gW1, float *gb1, float *gW2, float *gb2,
                           float *ws, cudaStream_t stream);
bool msg_grouped_supported(const MsgArgs &a, int E);

// Persistent grids of the message backward: the grouped kernels run at most 8 CTAs per SM, the per-row kernel at most 4.
constexpr int kMsgBwdGroupedMaxCTAs = 148 * 8, kMsgBwdRowMaxCTAs = 148 * 4;
inline int64_t msg_bwd_grouped_blocks(const MsgArgs &a)
{
    const int64_t b = ((int64_t)a.S + 3) / 4;
    return b < kMsgBwdGroupedMaxCTAs ? b : kMsgBwdGroupedMaxCTAs;
}

// Deterministic epilogue of the message backward.  A CTA's partial sums are 19 rows of E floats: rows 0-7 / 8 the weight
// columns / bias of relation 0, rows 9-12 / 13 relation 1, rows 14-17 / 18 relation 2.  Row k of CTA b lives at
// rel_base[r] + b * rel_stride[r] + (k - first row of r) * E.  The reduction adds every output element's partials in a fixed
// order and adds (+=) the result into gW / gb.
struct MsgPartials {
    const float *rel_base[3];
    int64_t rel_stride[3];
    int blocks, E;
};
int launch_msg_partials_reduce(const MsgPartials &p, float *gW0, float *gb0, float *gW1, float *gb1, float *gW2, float *gb2,
                               cudaStream_t stream);

}  // namespace marl

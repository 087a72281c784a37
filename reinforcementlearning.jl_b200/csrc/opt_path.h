// opt_path.h — which kernels run one optimiser step (sum the per-CTA gradient partials -> [exchange between ranks] -> global-norm
// clip -> Adam).  Plain C++ (also compiled for the host by the CPU test suite).
#pragma once
#include <cstdint>

enum OptPath {
    OPT_FUSED_TAIL,        // in the tail of the tensor-core loss + backward launch (nn_ac_loss_grad_step)
    OPT_ONE_KERNEL,        // reduce_clip_adam_kernel<false>
    OPT_ONE_KERNEL_XCHG,   // reduce_clip_adam_kernel<true>: the NVLink peer exchange inside the kernel (refused when the gradient
                           // does not fit the exchange inbox)
    OPT_NCCL_CHAIN,        // reduce_partials -> [NCCL all-reduce of gradient and loss sums when sharded] -> clip_adam
                           // (-> stats row when one is wanted)
};

// The fused tail stages every CTA's slice of the `rows` gradient-partial rows through shared memory (<= 512 parameters per CTA, at
// most 10 x 512 staged floats) and meets at grid barriers, so all `grid` CTAs must be co-resident (grid <= SMs, and <= 256 for the
// staged loss rows).
static inline bool opt_fused_tail_fits(int64_t np, int grid, int rows, int sm_count) {
    const int64_t per = (np + grid - 1) / grid;
    return per <= 512 && per * rows <= 10 * 512 && grid <= 256 && grid <= sm_count;
}

struct OptPathIn {
    int world;          // ranks of the communicator (1 without one)
    bool p2p;           // NVLink peer exchange attached
    bool exclusive;     // every rank owns its device (a launch that fills the device may wait for peers inside itself)
    bool fused_step;    // the caller can fuse the step into its loss + backward launch, and B200RL_FUSED_STEP allows it
    bool tc_bwd;        // the tensor-core loss + backward kernel runs the minibatch
    bool tail_fits;     // opt_fused_tail_fits
    bool fits_inbox;    // np + 4 <= kP2PXCap (gradient + 4 loss sums in one exchange)
    bool coresident;    // ceil(np / 256) <= SMs: reduce_clip_adam_kernel's grid barrier can complete
};

// Without a co-resident grid the step falls back to the kernel chain, on one GPU as well.  With the networks make_descs accepts that
// cannot happen on a B200: the largest (actor-critic, H = 128, 4 inputs, 4 outputs) has 34 949 parameters -> 137 CTAs of 148 SMs.
static inline OptPath opt_path(const OptPathIn& in) {
    const bool sharded = in.world > 1;
    if (in.fused_step && in.tc_bwd && in.tail_fits && (!sharded || (in.p2p && in.exclusive && in.fits_inbox))) return OPT_FUSED_TAIL;
    if ((sharded && !in.p2p) || !in.coresident) return OPT_NCCL_CHAIN;
    return in.p2p ? OPT_ONE_KERNEL_XCHG : OPT_ONE_KERNEL;
}

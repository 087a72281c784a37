// optim.cuh — device arithmetic of the optimiser step, shared by clip_adam_kernel, reduce_clip_adam_kernel (nn.cu) and the fused
// tail of ac_loss_grad_tc_kernel (nn_tc.cu): clip_by_global_norm! + Optimisers Adam, the grid barrier, the rank-order peer sum.
#pragma once
#include "nn.cuh"

// clip_by_global_norm!: the factor every gradient element is multiplied by, given the global norm gn
__device__ __forceinline__ float clip_scale(float gn, float max_norm) {
    float sc = 1.0f;
    if (max_norm > 0.f && max_norm <= gn) sc = max_norm / fmaxf(max_norm, gn);
    return sc;
}

// Optimisers Adam on one parameter with the bias corrections of beta^t = (bt1, bt2): updates m and v (both read before either is
// written), returns the parameter step
__device__ __forceinline__ float adam_apply(float g, float& m, float& v, float b1, float b2, float eps, float lr, float bt1, float bt2) {
    const float mk = b1 * m + (1.0f - b1) * g;
    const float vk = b2 * v + (1.0f - b2) * (g * g);
    m = mk; v = vk;
    return mk / (1.0f - bt1) / (sqrtf(vk / (1.0f - bt2)) + eps) * lr;
}

// Grid barrier (one thread per CTA): the CTA's writes ordered before the call become visible device-wide (fence cumulativity, as in
// cooperative groups), then wait until all G CTAs have arrived.  Needs all G CTAs co-resident; a barrier that never completes traps
// instead of hanging the GPU.
__device__ __forceinline__ void grid_arrive_wait(unsigned int* counter, unsigned int G) {
    __threadfence();
    atomicAdd(counter, 1u);
    unsigned int spins = 0;
    while (*reinterpret_cast<volatile unsigned int*>(counter) < G)
        if (++spins > (1u << 26)) __trap();
    __threadfence();
}

// Sum of word `idx` over the ranks in rank order (the own value for the own rank, the peers' packets of exchange `seq` from the
// own inbox): every rank computes the identical sum, so the replicas stay bit-identical without a broadcast.
__device__ __forceinline__ float p2p_sum_rank_order(const P2PTable& tab, unsigned slot, size_t idx, float local, unsigned seq) {
    float acc = 0.f;
    for (int r = 0; r < tab.nranks; ++r) acc += r == tab.rank ? local : __uint_as_float(p2p_recv(tab, 0, slot, r, idx, seq));
    return acc;
}

// One thread per CTA, after every thread of its CTA has read beta^t and the exchange sequence number: the last of the G CTAs to
// arrive at `arrivals` advances beta^t, zeroes the first n_counters barrier counters (so the launch can be replayed from a CUDA
// graph), stores the sequence number of a sharded step and ticks the update counter.
__device__ __forceinline__ void last_cta_epilogue(const OptStep& st, unsigned int* arrivals, int n_counters, unsigned int G, float bt1,
                                                  float bt2, bool xchg, unsigned int seq) {
    if (atomicAdd(arrivals, 1u) + 1u == G) {
        st.beta_t[0] = bt1 * st.b1; st.beta_t[1] = bt2 * st.b2;
        for (int i = 0; i < n_counters; ++i) st.counter[i] = 0u;
        if (xchg) *st.seq_ptr = seq;
        if (st.tick) *st.tick += 1u;
    }
}

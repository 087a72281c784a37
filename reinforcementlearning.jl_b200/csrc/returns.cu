// returns.cu — K5: generalized_advantage_estimation / discount_rewards(_reduced) as batched
// backward scans (RLCore/src/utils/basic.jl:138-235, :237-319, :334-417).
//
// One thread per series walks time backwards with the reference's exact operation order
//   gain  = r[i] + (gamma * gain) * c
//   delta = (r[i] + (gamma * v[i+1]) * c) - v[i];   gae = delta + ((gamma*lambda) * c) * gae
// (c::Bool multiply = strong zero), compiled with -fmad=false -> bit-identical to the serial
// CPU loop.  Loads are issued a chunk of time steps ahead of the dependent chain.
// (Few long series take a warp-segmented scan instead: scan_few_series below.)
//   dims = 2 ((N, T) PPO layout, series-fastest): a warp's 32 series are contiguous -> fully
//            coalesced 128-byte transactions at every time step.
//   dims = 1 (time-fastest): a CTA stages a [time-chunk x 32 series] tile through shared
//            memory with coalesced loads along time, then scans from shared memory.
// The fused variant also emits returns = adv + v and per-CTA partial sums for the advantage
// normalisation used by the PPO update (no second pass over the advantages).
#include "internal.h"
#include "jl_device.cuh"

namespace {

constexpr int kBlock = 128;
constexpr int kChunk = 8;

template <class T, int MODE>  // MODE 0: discount, 1: discount_reduced, 2: gae
__global__ void __launch_bounds__(kBlock) scan_series_fastest(T* __restrict__ out, const T* __restrict__ r, const T* __restrict__ v,
                                                             const uint8_t* __restrict__ term, const T* __restrict__ init, T gamma,
                                                             T lambda, int64_t S, int64_t n_time, T* __restrict__ ret_out,
                                                             double* __restrict__ partials) {
    int64_t s = (int64_t)blockIdx.x * kBlock + threadIdx.x;
    double sum = 0.0, sumsq = 0.0;
    if (s < S) {
        T acc = (MODE == 2) ? (T)0 : (init ? init[s] : (T)0);
        T vnext = (MODE == 2) ? v[s + S * n_time] : (T)0;
        T gl = gamma * lambda;
        for (int64_t hi = n_time; hi > 0; hi -= kChunk) {
            int n = hi < kChunk ? (int)hi : kChunk;
            T rr[kChunk], vv[kChunk];
            uint8_t tt[kChunk];
#pragma unroll
            for (int k = 0; k < kChunk; ++k) {
                if (k < n) {
                    int64_t i = hi - 1 - k;
                    rr[k] = r[s + S * i];
                    tt[k] = term ? term[s + S * i] : 0;
                    if (MODE == 2) vv[k] = v[s + S * i];
                }
            }
#pragma unroll
            for (int k = 0; k < kChunk; ++k) {
                if (k < n) {
                    int64_t i = hi - 1 - k;
                    bool c = !tt[k];
                    if (MODE == 2) {
                        T delta = (rr[k] + jld::mul_bool(gamma * vnext, c)) - vv[k];
                        acc = delta + jld::mul_bool(gl, c) * acc;
                        vnext = vv[k];
                        out[s + S * i] = acc;
                        if (ret_out) ret_out[s + S * i] = acc + vv[k];
                        if (partials) { sum += (double)acc; sumsq += (double)acc * (double)acc; }
                    } else {
                        acc = rr[k] + jld::mul_bool(gamma * acc, c);
                        if (MODE == 0) out[s + S * i] = acc;
                    }
                }
            }
        }
        if (MODE == 1) out[s] = acc;
    }
    if (MODE == 2 && partials) {  // deterministic per-CTA partial (fixed tree), reduced later in CTA order
        __shared__ double sh[2][kBlock / 32];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            sum += __shfl_xor_sync(0xffffffffu, sum, o);
            sumsq += __shfl_xor_sync(0xffffffffu, sumsq, o);
        }
        if ((threadIdx.x & 31) == 0) { sh[0][threadIdx.x >> 5] = sum; sh[1][threadIdx.x >> 5] = sumsq; }
        __syncthreads();
        if (threadIdx.x == 0) {
            double a = 0, b = 0;
            for (int k = 0; k < kBlock / 32; ++k) { a += sh[0][k]; b += sh[1][k]; }
            partials[2 * blockIdx.x] = a;
            partials[2 * blockIdx.x + 1] = b;
        }
    }
}

// dims = 1: time-fastest.  Warp w of the CTA owns series blockIdx*WARPS + w ... no: each CTA
// owns kTileS series; all threads cooperatively stage [kTileT time steps x kTileS series]
// through smem with loads coalesced along time; then thread s (< kTileS) scans its series.
constexpr int kTileS = 32;
template <class T> struct TileT { static constexpr int v = sizeof(T) == 8 ? 32 : 64; };
template <class T, int MODE>
__global__ void __launch_bounds__(kBlock) scan_time_fastest(T* __restrict__ out, const T* __restrict__ r, const T* __restrict__ v,
                                                           const uint8_t* __restrict__ term, const T* __restrict__ init, T gamma,
                                                           T lambda, int64_t S, int64_t n_time) {
    constexpr int kTileT = TileT<T>::v;
    __shared__ T sr[kTileS][kTileT + 1];
    __shared__ T sv[kTileS][kTileT + 1];
    __shared__ T so[kTileS][kTileT + 1];
    __shared__ uint8_t stt[kTileS][kTileT + 4];
    int64_t s0 = (int64_t)blockIdx.x * kTileS;
    int ls = threadIdx.x;  // scanning thread's local series (valid when < kTileS)
    int64_t s = s0 + ls;
    bool scanner = ls < kTileS && s < S;
    int64_t vstride = (MODE == 2) ? n_time + 1 : n_time;
    T acc = (T)0, vnext = (T)0, gl = gamma * lambda;
    if (scanner) {
        acc = (MODE == 2) ? (T)0 : (init ? init[s] : (T)0);
        if (MODE == 2) vnext = v[s * vstride + n_time];
    }
    for (int64_t hi = n_time; hi > 0; hi -= kTileT) {
        int64_t lo = hi > kTileT ? hi - kTileT : 0;
        int nt = (int)(hi - lo);
        for (int idx = threadIdx.x; idx < kTileS * kTileT; idx += kBlock) {
            int js = idx / kTileT, jt = idx % kTileT;
            if (jt < nt && s0 + js < S) {
                int64_t i = lo + jt;
                sr[js][jt] = r[(s0 + js) * n_time + i];
                stt[js][jt] = term ? term[(s0 + js) * n_time + i] : 0;
                if (MODE == 2) sv[js][jt] = v[(s0 + js) * vstride + i];
            }
        }
        __syncthreads();
        if (scanner) {
            for (int jt = nt - 1; jt >= 0; --jt) {
                bool c = !stt[ls][jt];
                if (MODE == 2) {
                    T vi = sv[ls][jt];
                    T delta = (sr[ls][jt] + jld::mul_bool(gamma * vnext, c)) - vi;
                    acc = delta + jld::mul_bool(gl, c) * acc;
                    vnext = vi;
                } else {
                    acc = sr[ls][jt] + jld::mul_bool(gamma * acc, c);
                }
                so[ls][jt] = acc;
            }
        }
        __syncthreads();
        if (MODE != 1) {
            for (int idx = threadIdx.x; idx < kTileS * kTileT; idx += kBlock) {
                int js = idx / kTileT, jt = idx % kTileT;
                if (jt < nt && s0 + js < S) out[(s0 + js) * n_time + lo + jt] = so[js][jt];
            }
        }
        __syncthreads();
    }
    if (MODE == 1 && scanner) out[s] = acc;
}

// Few series, long time axis (e.g. one episode of 300+ steps; north-star item (iii)): one WARP per series runs the backward linear
// recurrence x_i = b_i + a_i x_{i+1} as a warp-segmented scan — 32 time steps per round, Kogge-Stone composition of the affine
// maps (a, b) with shuffles, the round's last value carried into the next round.  The composition re-associates the float
// recurrence, so this variant is within ~1e-6 of the serial loop instead of bit-identical: it is only dispatched where the
// thread-per-series kernel would leave the machine idle (S < 1024 and >= 64 time steps; the reference's golden vectors and the
// PPO rollout path never take it).
template <class T, int MODE>
__global__ void __launch_bounds__(kBlock) scan_few_series(T* __restrict__ out, const T* __restrict__ r, const T* __restrict__ v,
                                                         const uint8_t* __restrict__ term, const T* __restrict__ init, T gamma, T lambda,
                                                         int64_t S, int64_t n_time, int64_t ss, int64_t ts, int64_t vss) {
    const int lane = threadIdx.x & 31;
    const int64_t s = (int64_t)blockIdx.x * (kBlock / 32) + (threadIdx.x >> 5);
    if (s >= S) return;                                    // whole warps leave together
    const T k = (MODE == 2) ? gamma * lambda : gamma;
    T carry = (MODE == 2) ? (T)0 : (init ? init[s] : (T)0);
    for (int64_t hi = n_time; hi > 0; hi -= 32) {
        const int64_t i = hi - 1 - lane;                   // lane 0 = the latest time step of this round
        T a = (T)1, b = (T)0;                              // identity map for lanes past the start of the series
        if (i >= 0) {
            const bool c = !(term && term[s * ss + i * ts]);
            a = c ? k : (T)0;
            if (MODE == 2) {
                const T vn = v[s * vss + (i + 1) * ts], vi = v[s * vss + i * ts];
                b = (r[s * ss + i * ts] + (c ? gamma * vn : (T)0)) - vi;
            } else {
                b = r[s * ss + i * ts];
            }
        }
        // inclusive scan of the maps in lane order: after it, x_lane = a * carry + b
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const T a2 = __shfl_up_sync(0xffffffffu, a, d), b2 = __shfl_up_sync(0xffffffffu, b, d);
            if (lane >= d) { b = a * b2 + b; a = a * a2; }
        }
        const T x = a * carry + b;
        if (i >= 0 && MODE != 1) out[s * ss + i * ts] = x;
        carry = __shfl_sync(0xffffffffu, x, 31);           // (lanes with i < 0 hold the identity map: x passes through)
    }
    if (MODE == 1 && lane == 0) out[s] = carry;
}

// Final reduce of the per-CTA partials in CTA order -> {mean, 1/clamp(std,1e-8,1000)} as float2.
__global__ void finalize_norm_kernel(const double* __restrict__ partials, int n_partials, double count, float* __restrict__ out2) {
    if (threadIdx.x != 0 || blockIdx.x != 0) return;
    double a = 0, b = 0;
    for (int k = 0; k < n_partials; ++k) { a += partials[2 * k]; b += partials[2 * k + 1]; }
    double mean = a / count;
    double var = (b - count * mean * mean) / (count - 1.0);
    if (var < 0) var = 0;
    float sd = (float)sqrt(var);
    sd = sd < 1e-8f ? 1e-8f : (sd > 1000.0f ? 1000.0f : sd);
    out2[0] = (float)mean;
    out2[1] = 1.0f / sd;
}

template <class T, int MODE>
int run_scan(b200rl_ctx* ctx, T* out, const T* r, const T* v, const uint8_t* term, const T* init, T gamma, T lambda, int64_t R,
             int64_t C, int dims, int on_device) {
    TRY(ctx_bind(ctx));
    REQUIRE(out && r && (MODE != 2 || v), B200RL_ERR_INVALID, "null array");
    REQUIRE(dims == 1 || dims == 2, B200RL_ERR_INVALID, "dims must be 1 or 2 (the reference throws a MethodError otherwise)");
    REQUIRE(R > 0 && C > 0, B200RL_ERR_INVALID, "empty matrix");
    int64_t S = dims == 1 ? C : R, n_time = dims == 1 ? R : C;
    size_t n = (size_t)R * C, nv = (MODE == 2) ? (size_t)S * (n_time + 1) : 0;
    size_t n_out = (MODE == 1) ? (size_t)S : n;
    T *d_out = out;
    const T *d_r = r, *d_v = v, *d_init = init;
    const uint8_t* d_term = term;
    char* base = nullptr;
    if (!on_device) {
        size_t bytes = (n_out + n + nv + (init ? S : 0)) * sizeof(T) + (term ? n : 0) + 64;
        void* p;
        TRY(ctx_scratch(ctx, bytes, &p));
        base = (char*)p;
        T* po = (T*)base; T* pr = po + n_out; T* pv = pr + n; T* pi = pv + nv; uint8_t* pt = (uint8_t*)(pi + (init ? S : 0));
        CUDA_TRY(cudaMemcpyAsync(pr, r, n * sizeof(T), cudaMemcpyHostToDevice, ctx->stream));
        if (MODE == 2) CUDA_TRY(cudaMemcpyAsync(pv, v, nv * sizeof(T), cudaMemcpyHostToDevice, ctx->stream));
        if (init) CUDA_TRY(cudaMemcpyAsync(pi, init, S * sizeof(T), cudaMemcpyHostToDevice, ctx->stream));
        if (term) CUDA_TRY(cudaMemcpyAsync(pt, term, n, cudaMemcpyHostToDevice, ctx->stream));
        d_out = po; d_r = pr; d_v = pv; d_init = init ? pi : nullptr; d_term = term ? pt : nullptr;
    }
    if (S < 1024 && n_time >= 64) {   // few long series: warp-segmented scan (see scan_few_series), either layout
        const int64_t ss = dims == 2 ? 1 : n_time, ts = dims == 2 ? S : 1, vss = dims == 2 ? 1 : n_time + 1;
        scan_few_series<T, MODE><<<grid_for(S, kBlock / 32), kBlock, 0, ctx->stream>>>(d_out, d_r, d_v, d_term, d_init, gamma, lambda, S, n_time,
                                                                                       ss, ts, vss);
    } else if (dims == 2)
        scan_series_fastest<T, MODE><<<grid_for(S, kBlock), kBlock, 0, ctx->stream>>>(d_out, d_r, d_v, d_term, d_init, gamma, lambda, S,
                                                                                     n_time, nullptr, nullptr);
    else
        scan_time_fastest<T, MODE><<<grid_for(S, kTileS), kBlock, 0, ctx->stream>>>(d_out, d_r, d_v, d_term, d_init, gamma, lambda, S,
                                                                                   n_time);
    LAUNCH_CHECK(ctx);
    if (!on_device) {
        CUDA_TRY(cudaMemcpyAsync(out, d_out, n_out * sizeof(T), cudaMemcpyDeviceToHost, ctx->stream));
        CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    }
    return B200RL_OK;
}

}  // namespace

// internal: fused GAE for the (N, T) rollout layout — advantages, returns and the
// normalisation constants {mean, inv_std} in `norm2` (device float[2]).  `partials` must
// hold 2 * ceil(S / 128) doubles.
int b200rl_gae_fused_internal(b200rl_ctx* ctx, float* adv, float* ret, const float* r, const float* v, const uint8_t* term,
                              float gamma, float lambda, int64_t S, int64_t n_time, double* partials, float* norm2) {
    unsigned grid = grid_for(S, kBlock);
    scan_series_fastest<float, 2><<<grid, kBlock, 0, ctx->stream>>>(adv, r, v, term, nullptr, gamma, lambda, S, n_time, ret,
                                                                  partials);
    LAUNCH_CHECK(ctx);
    if (norm2) {
        finalize_norm_kernel<<<1, 32, 0, ctx->stream>>>(partials, (int)grid, (double)S * (double)n_time, norm2);
        LAUNCH_CHECK(ctx);
    }
    return B200RL_OK;
}
int b200rl_gae_fused_partials_count(int64_t S) { return 2 * (int)grid_for(S, kBlock); }

extern "C" {
int b200rl_gae_f32(b200rl_ctx* ctx, float* adv, const float* r, const float* v, const uint8_t* term, float gamma, float lambda,
                   int64_t R, int64_t C, int dims, int on_device) {
    return run_scan<float, 2>(ctx, adv, r, v, term, nullptr, gamma, lambda, R, C, dims, on_device);
}
int b200rl_gae_f64(b200rl_ctx* ctx, double* adv, const double* r, const double* v, const uint8_t* term, double gamma, double lambda,
                   int64_t R, int64_t C, int dims, int on_device) {
    return run_scan<double, 2>(ctx, adv, r, v, term, nullptr, gamma, lambda, R, C, dims, on_device);
}
int b200rl_discount_rewards_f32(b200rl_ctx* ctx, float* out, const float* r, const uint8_t* term, const float* init, float gamma,
                                int64_t R, int64_t C, int dims, int on_device) {
    return run_scan<float, 0>(ctx, out, r, nullptr, term, init, gamma, 0.f, R, C, dims, on_device);
}
int b200rl_discount_rewards_f64(b200rl_ctx* ctx, double* out, const double* r, const uint8_t* term, const double* init, double gamma,
                                int64_t R, int64_t C, int dims, int on_device) {
    return run_scan<double, 0>(ctx, out, r, nullptr, term, init, gamma, 0.0, R, C, dims, on_device);
}
int b200rl_discount_rewards_reduced_f32(b200rl_ctx* ctx, float* out, const float* r, const uint8_t* term, const float* init,
                                        float gamma, int64_t R, int64_t C, int dims, int on_device) {
    return run_scan<float, 1>(ctx, out, r, nullptr, term, init, gamma, 0.f, R, C, dims, on_device);
}
int b200rl_discount_rewards_reduced_f64(b200rl_ctx* ctx, double* out, const double* r, const uint8_t* term, const double* init,
                                        double gamma, int64_t R, int64_t C, int dims, int on_device) {
    return run_scan<double, 1>(ctx, out, r, nullptr, term, init, gamma, 0.0, R, C, dims, on_device);
}
}

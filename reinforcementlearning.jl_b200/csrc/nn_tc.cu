// nn_tc.cu — K7 on tensor cores (tcgen05 / TMEM): PPO / A2C loss + backward for H = 64.
//
// The 64 x 64 layers are [128 samples x 64] x [64 x 64] GEMMs per tile: one warp issues tcgen05.mma (SWIZZLE_NONE canonical
// layout, see umma.cuh) with the FP32 accumulators in TMEM; the worker warps pull them back with tcgen05.ld.  Parity needs
// ~FP32 accuracy (1e-5 relative on losses), which no single tensor-core input format gives, so every product is a 3-term split
//     A*B ~= A_hi*B_hi + A_hi*B_lo + A_lo*B_hi,   x_hi = fp16(x * S), x_lo = fp16(x * S - x_hi)      (22 mantissa bits)
// with a power-of-two scale S per operand (exact; undone on the FP32 accumulator), accumulated in FP32.  Round 1 used the same
// split on kind::tf32 (K = 8 per instruction); kind::f16 covers K = 16 per instruction at the same 2^-22 product accuracy.
// A tcgen05.mma (M = 128, K = 16) occupies the pipe for 10 + N/2 cycles with A in TMEM and 43 + N/2 with A in shared memory
// (profiles/umma_pacing.py) PROVIDED it is issued under an elect.sync predicate (umma::elect_one): under `lane == 0` ptxas wraps
// every MMA in an ELECT / BRA.U.ANY loop that costs ~100 cycles of issue time.  fp16 has 5 exponent bits: activations
// must stay below 65504 in magnitude (scale 1), weights below 1023 (scale 64); gradients are scaled by ~1/(4 inv_B) at launch.
// Below 6e-5 the lo part is subnormal: absolute error <= 2^-25 per element, far inside the 1e-5 bar.  Layer 1 (K <= 4) and the
// heads (N <= 2) stay on FFMA.  The forward-only kernels (policy inference, fused rollout) live in fwd_tc.cu (same split).
#include "opt_path.h"
#include "optim.cuh"
#include "perm.cuh"
#include "tc_split.h"
#include "umma.cuh"

namespace {

constexpr int NT = 256;
constexpr int TM = 128;              // samples per tile = UMMA M
constexpr int H = 64;
constexpr int G_F = 128;             // weight image (fp16, K-major): byte stride between 8-element K chunks = one 8 x 16 B core matrix
constexpr int GW_S = 8 * G_F;        // stride between 8-row groups (64 K elements = 8 chunks)
constexpr int WIMG_BYTES = 16 * GW_S; // one [hi (64 rows) ; lo (64 rows)] x [K = 64] fp16 weight image = 16 KB
constexpr float kScaleW = 64.0f;     // power-of-two operand scales (see the header comment)
constexpr float kLog2Pi = 1.8378770664093453f;

__device__ __forceinline__ float act_f(int act, float z) { return act == B200RL_ACT_RELU ? fmaxf(z, 0.f) : tanhf(z); }
// two fp32 values -> packed fp16 pair {lo half = a, hi half = b}: the hi parts, and the fp16 of what they miss (the lo parts)
__device__ __forceinline__ void split2(float a, float b, uint32_t& hi, uint32_t& lo) {
    const __half2 h = __floats2half2_rn(a, b);
    const float2 back = __half22float2(h);
    const __half2 l = __floats2half2_rn(a - back.x, b - back.y);
    hi = *reinterpret_cast<const uint32_t*>(&h);
    lo = *reinterpret_cast<const uint32_t*>(&l);
}
__device__ __forceinline__ float half_bits_to_float(uint32_t bits16) { return __half2float(__ushort_as_half((unsigned short)bits16)); }
__device__ __forceinline__ float softplus_f(float x) { return x > 0.f ? x + log1pf(expf(-x)) : log1pf(expf(x)); }
__device__ __forceinline__ float normlogpdf1(float mu, float sigma, float x) {
    float s = sigma + 1e-8f, v = s * s, dd = x - mu;
    return -0.5f * ((logf(v) + (dd * dd) / v) + kLog2Pi);
}
__device__ __forceinline__ int64_t head_base(const MlpDesc& d) { return (int64_t)d.H * d.in + d.H + (int64_t)d.H * d.H + d.H; }
__device__ __forceinline__ int64_t head_w(const MlpDesc& d, int o, int j) {
    return head_base(d) + (d.heads2 ? (int64_t)o * (d.H + 1) + j : (int64_t)o + (int64_t)d.nout * j);
}
__device__ __forceinline__ int64_t head_b(const MlpDesc& d, int o) {
    return head_base(d) + (d.heads2 ? (int64_t)o * (d.H + 1) + d.H : (int64_t)d.nout * d.H + o);
}
__device__ __forceinline__ uint32_t wimg_off(int n, int k) { return (uint32_t)((n >> 3) * GW_S + (k >> 3) * G_F + (n & 7) * 16 + (k & 7) * 2); }

// =====================================================================================================
// K7 on tensor cores: PPO / A2C loss + backward for one minibatch, all three 64x64 GEMMs on tcgen05.
//   GEMM1  H2pre[s][o] = sum_i H1[s][i]  W2[o][i]     A = H1 (TMEM, written by tcgen05.st), B = W2 image (smem)
//   GEMM2  dH1[s][i]   = sum_j dP2[s][j] W2[j][i]     A = dP2 (TMEM),                        B = W2^T image (smem)
//   GEMM3  dW2[j][i]  += sum_s dP2[s][j] H1[s][i]     A = dP2^T, B = H1^T: feature-major K-major images (smem),
//                                                     accumulated in TMEM across ALL tiles of the CTA, read once.
// every product the 3-term fp16 split (hi*hi + hi*lo + lo*hi), FP32 accumulate.
// One CTA per SM (512 threads, role = blockIdx & 1), persistent, software-pipelined across tiles (see the loop).
// Thread <-> data: warp w: TMEM lane quadrant q = w % 4, feature block c = w / 4; thread = sample s = 32q + lane.
constexpr int NT7 = 512;
// Operands of the two GEMMs that reduce over the SAMPLES (GEMM3, GEMM4: K = sample) are MN-major (SWIZZLE_NONE) images: a core
// matrix is 8 k-rows (samples) x 16 B (8 consecutive features), element (feature f, sample s) at
//     (f / 8) * GS_T + (s / 8) * GF_T + (s % 8) * 16 + (f % 8) * 2        (descriptor: LBO = GF_T, SBO = GS_T; profiles/umma_probe_mn.py)
// With GF_T = 128 that is simply [feature block of 8][sample][8 features]: thread = sample writes 8 features as ONE 16-byte
// vector, and the 32 lanes of a warp cover 512 contiguous bytes (no bank conflicts).  Until round 2 these images were K-major
// (8 samples x one feature per 16 B): 32 two-byte transposed stores per thread and image, 4.5 M bank conflicts per launch.
constexpr int GF_T = 128;                 // stride between 8-sample k-blocks
constexpr int GS_T = 16 * GF_T;           // stride between 8-feature blocks (128 samples)
constexpr int FIMG = 8 * GS_T;            // [64 features x 128 samples] fp16 = 16 KB
// TMEM columns: R1 = D1 of GEMM1 (64 columns: hi*hi + hi*lo + lo*hi accumulated in place), then (after P3 consumed it) the dP2 A
// operand of GEMM2 in the same 64 columns (hi: 32 columns of fp16 pairs | lo: 32); D2 = GEMM2 accumulator (64 columns); D3 = GEMM3
// accumulator (all tiles; hi|lo operands stacked along M and N, one MMA per K step); AH = H1 A operand of GEMM1 (hi 32 | lo 32).
// D3 has 144 columns: the B operand of GEMM3 carries a constant "ones" row behind H1^T, so column 128 is sum_s dP2 = db2.
// D4 = GEMM4 accumulator (16 columns): dW1 | db1 = dP1^T x [x | 1], accumulated over all tiles like D3.
constexpr uint32_t COL_R1 = 0, COL_D2 = 128, COL_D3 = 256, COL_D4 = 400, COL_AH = 448;
constexpr float kScaleH = 64.0f, kScaleX = 64.0f;   // power-of-two scales of the H1 / observation operands (weights: kScaleW)
constexpr int kNo = 2;   // head outputs this kernel handles (nn_tc_bwd_supported: actor n_out <= 2, critic n_out = 1)

struct SmemBwd {
    static_assert(FIMG % 128 == 0 && WIMG_BYTES % 128 == 0 && (2 * GS_T) % 16 == 0, "hi/lo(/ones) images must be adjacent to form one operand");
    alignas(128) uint8_t FP_full[FIMG];    // dP2^T hi (rows = feature j, K = sample), fp16
    alignas(128) uint8_t FP_lo[FIMG];      // ... lo: directly behind, so [hi; lo] is one 128-row operand
    alignas(128) uint8_t FH_full[FIMG];    // H1^T hi
    alignas(128) uint8_t FH_lo[FIMG];
    alignas(16) uint8_t FH_ones[2 * GS_T]; // 16 more B rows (features 128..143) of GEMM3: feature 128 = 1.0 for every sample (-> db2), the rest 0; written once
    alignas(128) uint8_t FQ_full[FIMG];    // dP1^T hi | lo: A operand of GEMM4
    alignas(128) uint8_t FQ_lo[FIMG];
    alignas(128) uint8_t B1[WIMG_BYTES];   // rows 0..63: hi, 64..127: lo of (n = out o, k = in i)  = 64 W2[o + 64 i]
    alignas(128) uint8_t B2[WIMG_BYTES];   // (n = in i,  k = out j) = 64 W2[j + 64 i]
    // B operand of GEMM4, double-buffered by tile parity (written at publish time, read by the GEMM4 of the same tile one
    // phase later): rows 0..3 = x_i hi, row 4 = 1.0 (-> db1), rows 8..11 = x_i lo, the rest 0;  K = sample
    alignas(128) uint8_t XT[2][2 * GS_T];
    float W1[kInMax * H];
    float b1[H], b2[H];
    float W3[H * kNo];                     // [feature][head output]
    float b3[kNo];
    float Zp[4 * kNo * TM];                // head partials [c][o][s]
    float Red[32];
    double RedD[16];
    float step_scale;
    alignas(8) uint64_t bar1;
    alignas(8) uint64_t bar2;
    alignas(8) uint64_t bar3;
    alignas(8) uint64_t bar4;
    float AccW2[64 * 65 + 64];             // FP32 accumulators the flushes add D3 into: dW2[j][i] at j * 65 + i, then db2[j] (all still operand-scaled)
    float AccD4[64 * 9];                   // ... D4: dW1[f][i] at f * 9 + i, db1[f] at f * 9 + 4
    uint32_t tmem;
};
__device__ __forceinline__ uint32_t fimg_off(int f, int s) { return (uint32_t)((f >> 3) * GS_T + (s >> 3) * GF_T + (s & 7) * 16 + (f & 7) * 2); }
// 16 features (8 packed fp16 pairs) of sample s, starting at feature f0 (a multiple of 16): two 16-byte vectors
__device__ __forceinline__ void store16_feat(uint8_t* img, int f0, int s, const uint32_t (&v)[8]) {
    uint8_t* p = img + fimg_off(f0, s);
    *reinterpret_cast<uint4*>(p) = make_uint4(v[0], v[1], v[2], v[3]);
    *reinterpret_cast<uint4*>(p + GS_T) = make_uint4(v[4], v[5], v[6], v[7]);
}
__device__ __forceinline__ float dact_f(int act, float h) { return act == B200RL_ACT_RELU ? (h > 0.f ? 1.f : 0.f) : 1.f - h * h; }

__device__ __forceinline__ uint32_t mix32(uint32_t h) {
    h ^= h >> 16; h *= 0x85EBCA6Bu; h ^= h >> 13; h *= 0xC2B2AE35u; h ^= h >> 16;
    return h;
}
using b200perm::perm_index;
using b200perm::perm_index_bits;
__device__ __forceinline__ float block_sum512(float v, float* red) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    __syncthreads();
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
    __syncthreads();
    float t = 0.f;
    if (threadIdx.x == 0)
        for (int k = 0; k < NT7 / 32; ++k) t += red[k];
    return t;
}
__device__ __forceinline__ float sigmoid_f(float x) { return 1.f / (1.f + expf(-x)); }

// sum over the 32 lanes of NV values each (NV a power of two <= 32... here 32): lane L ends with the totals of
// values 2L*(NV/64).. — for NV = 32: lane L holds the total of value index L in v[0].
__device__ __forceinline__ float lane_transpose_reduce32(float (&v)[32], int lane) {
#pragma unroll
    for (int st = 0; st < 5; ++st) {
        const int half = 16 >> st, off = 16 >> st;
        const bool upper = (lane & off) != 0;
#pragma unroll
        for (int n = 0; n < half; ++n) {
            float send = upper ? v[n] : v[n + half];
            float keep = upper ? v[n + half] : v[n];
            v[n] = keep + __shfl_xor_sync(0xffffffffu, send, off);
        }
    }
    return v[0];   // value index = lane
}

// worker-only barrier (the MMA warp never joins it)
__device__ __forceinline__ void worker_sync() { asm volatile("bar.sync 1, 512;" ::: "memory"); }
// barrier of the four warps that share one TMEM lane quadrant q (= one 32-sample slice of the tile, feature blocks c = 0..3).
// Everything the workers exchange per tile (X, Aux, Zp, the TMEM columns of a lane) is exchanged between the four threads of ONE
// sample, i.e. inside such a group, so the per-tile barriers are group-local (ids 5..8, 128 threads) and the four groups — one
// per warp scheduler — drift freely within a tile; the tensor-core hand-overs (bar.arrive) and the mbarrier waits bound the drift.
__device__ __forceinline__ void group_sync(int q) { asm volatile("bar.sync %0, 128;" ::"r"(5 + q) : "memory"); }
// operand hand-over to the issuer warp: 512 worker threads arrive without waiting, the 32 issuer threads wait
__device__ __forceinline__ void ready_arrive(int id) { asm volatile("bar.arrive %0, 544;" ::"r"(id) : "memory"); }
__device__ __forceinline__ void ready_wait(int id) { asm volatile("bar.sync %0, 544;" ::"r"(id) : "memory"); }
// per-sample loss and d(loss)/d(head outputs); identical arithmetic on every thread that evaluates a sample
struct LossOut { float dz[kNo]; float l0, l1; };
__device__ __forceinline__ LossOut sample_loss(const MlpDesc& actor, int role, const AcHyper& hp, float inv_B, const float (&z)[kNo],
                                               float a_bits, float lp_old, float A, float ret) {
    LossOut r;
#pragma unroll
    for (int o = 0; o < kNo; ++o) r.dz[o] = 0.f;
    r.l0 = 0.f; r.l1 = 0.f;
    if (role == 1) {
        float err = ret - z[0];
        r.l0 = err * err;
        r.dz[0] = -2.0f * hp.w_critic * inv_B * err;
        return r;
    }
    float logp_a, gsel;
    if (!actor.heads2) {
        int na = actor.nout;
        float lp[kNo], pr[kNo];
        float m = -3.4e38f;
#pragma unroll
        for (int o = 0; o < kNo; ++o) if (o < na) m = fmaxf(m, z[o]);
        float se = 0.f;
#pragma unroll
        for (int o = 0; o < kNo; ++o) if (o < na) se += expf(z[o] - m);
        float ls = logf(se);
        float Hent = 0.f;
#pragma unroll
        for (int o = 0; o < kNo; ++o) {
            lp[o] = (z[o] - m) - ls;
            pr[o] = o < na ? expf(lp[o]) : 0.f;
            if (o < na) Hent -= pr[o] * lp[o];
        }
        int a = __float_as_int(a_bits) - 1;
        logp_a = 0.f;
#pragma unroll
        for (int o = 0; o < kNo; ++o) if (o == a) logp_a = lp[o];
        r.l1 = Hent;
        if (hp.algo == 0) {
            float ratio = expf(logp_a - lp_old);
            float u = ratio * A;
            float rc = fminf(fmaxf(ratio, 1.0f - hp.clip_range), 1.0f + hp.clip_range);
            float cc = rc * A;
            r.l0 = -fminf(u, cc);
            bool inside = ratio >= 1.0f - hp.clip_range && ratio <= 1.0f + hp.clip_range;
            gsel = (u < cc || inside) ? u : 0.f;
        } else {
            r.l0 = -(logp_a * A);
            gsel = A;
        }
        float dlogp = -hp.w_actor * inv_B * gsel;
#pragma unroll
        for (int o = 0; o < kNo; ++o)
            if (o < na) r.dz[o] = dlogp * ((o == a ? 1.f : 0.f) - pr[o]) + hp.w_entropy * inv_B * pr[o] * (lp[o] + Hent);
    } else {
        float mu = z[0], raw = z[1];
        float sp = softplus_f(raw);
        float sigma = fminf(fmaxf(sp, hp.min_sigma), hp.max_sigma);
        bool clamped = sp < hp.min_sigma || sp > hp.max_sigma;
        float a = a_bits;
        logp_a = normlogpdf1(mu, sigma, a);
        float Hent = logf(sigma) + 0.5f * (kLog2Pi + 1.0f);
        r.l1 = Hent;
        if (hp.algo == 0) {
            float ratio = expf(logp_a - lp_old);
            float u = ratio * A;
            float rc = fminf(fmaxf(ratio, 1.0f - hp.clip_range), 1.0f + hp.clip_range);
            float cc = rc * A;
            r.l0 = -fminf(u, cc);
            bool inside = ratio >= 1.0f - hp.clip_range && ratio <= 1.0f + hp.clip_range;
            gsel = (u < cc || inside) ? u : 0.f;
        } else {
            r.l0 = -(logp_a * A);
            gsel = A;
        }
        float dlogp = -hp.w_actor * inv_B * gsel;
        float sgm = sigma + 1e-8f, dd = a - mu;
        r.dz[0] = dlogp * (dd / (sgm * sgm));
        float dsig = dlogp * (-1.0f / sgm + (dd * dd) / (sgm * sgm * sgm)) - hp.w_entropy * inv_B * (1.0f / sigma);
        r.dz[1] = clamped ? 0.f : dsig * sigmoid_f(raw);
    }
    return r;
}

#ifdef B200RL_K7_TIMING   // debug build only (profiles/k7_phase_timing.py): per-phase cycle sums seen by CTA 0 / one watched thread
__device__ unsigned long long g_k7_phase[40];
__device__ int g_k7_watch = 0;   // watched worker thread (low 16 bits) of CTA (high bits; even = actor, odd = critic) whose timeline is recorded
#define K7_T(i) do { if (tid == (g_k7_watch & 0xFFFF) && (int)blockIdx.x == (g_k7_watch >> 16)) { long long now_ = clock64(); g_k7_phase[i] += (unsigned long long)(now_ - tprev_); tprev_ = now_; } } while (0)
// issuer warp of CTA 0 (lane 0): phases 18..23 = wait RdyA | issue G2 | wait RdyB | issue G1 + G3 | wait RdyC | issue G4
#define K7_TI(i) do { if (lane == 0 && (int)blockIdx.x == (g_k7_watch >> 16)) { long long now_ = clock64(); g_k7_phase[i] += (unsigned long long)(now_ - tprevi_); tprevi_ = now_; } } while (0)
#else
#define K7_T(i) do { } while (0)
#define K7_TI(i) do { } while (0)
#endif
// 16 worker warps + one warpgroup (warps 16..19) whose first warp feeds the tensor core.  The issuing thread blocks once the MMA
// queue is full (the issue side of a GEMM takes as long as its execution), which used to stall a worker warp — and with it
// everybody at the next barrier.  The register file is per scheduler (16 K registers, 5 warps
// each now), so the issuer warpgroup gives its registers back (setmaxnreg.dec 24) and the workers take 120 (setmaxnreg.inc).
constexpr int NT7_ALL = NT7 + 128;
// The tensor core adds into an FP32 accumulator with truncation: a chain of n accumulating MMAs biases a same-signed sum by
// ~n * 2^-25 relative (measured: 1e-4 on b1 / W2 gradients after 1 770 adds, profiles/k7_grad_error.py).  The accumulators that live
// across tiles (D3, D4) are therefore flushed into FP32 shared-memory accumulators (round-to-nearest adds) every kFlushTiles
// tiles and restarted: chains of 64 adds, bias ~2e-6.
constexpr int kFlushTiles = 8;
constexpr int kBarRdyA = 2, kBarRdyB = 3, kBarRdyC = 4;   // named barriers: workers arrive (bar.arrive), the issuer warp waits (bar.sync)

// ACT: the trunks' activation as a compile-time constant (B200RL_ACT_RELU / B200RL_ACT_TANH; -1 = read it from the descriptors, for
// an actor and a critic with different activations).  With the activation known the relu build carries no tanhf expansions at
// all (the runtime-act kernel was 107 KB of SASS, most of it 64 inlined tanhf bodies that a relu run branches around).
template <int ACT>
__global__ void __launch_bounds__(NT7_ALL, 1)
ac_loss_grad_tc_kernel(MlpDesc actor, MlpDesc critic, const float* params /* no __restrict__: the fused optimiser step rewrites them in the tail */, AcHyper hp, AcBatch b, float* partial,
                       float* __restrict__ loss_partial, int64_t np_total, float scale_base /* power of two ~ 1 / inv_B */,
                       OptStep st /* st.params != null: the optimiser step runs in the tail of this launch */,
                       int n_actor /* CTAs [0, n_actor) work on the actor, the rest on the critic */) {
    extern __shared__ __align__(1024) unsigned char smem_raw[];
    SmemBwd& sm = *reinterpret_cast<SmemBwd*>(smem_raw);
    // The actor's loss (softmax / Gaussian log-density, entropy, PPO ratio) makes its tiles ~4 % longer than the critic's, so the CTAs
    // are split unevenly (76 : 72 of 148 for the categorical PPO loss) and both roles finish together.  Gradient partials: row
    // `cta` holds the actor half written by actor CTA `cta` and the critic half written by critic CTA `cta`; the role with more
    // CTAs zero-fills the other half of its surplus rows.
    const int role = (int)blockIdx.x < n_actor ? 0 : 1;
    const int cta = role ? (int)blockIdx.x - n_actor : (int)blockIdx.x;
    const int nctas = role ? (int)gridDim.x - n_actor : n_actor;
    const int nrows = max(n_actor, (int)gridDim.x - n_actor);
    // Scale of the dP2 / dP1 operands (a power of two): dz / inv_B is O(ratio * A_hat) <= ~10 for the actor and 2 w_critic (R - V) for
    // the critic (as large as the returns).  x 64 / x 4 keeps the lo parts of typical entries in fp16's normal range and leaves
    // room up to |dz| / inv_B ~ 1e3 (actor) / 1.6e4 (critic) before a hi part would overflow fp16 (-> inf -> NaN loss: loud, not silent).
    const float scale_p = scale_base * (role ? 4.0f : 64.0f);
    const MlpDesc d = role ? critic : actor;
    const int act = ACT >= 0 ? ACT : d.act;
    const bool relu = act == B200RL_ACT_RELU;
    const int64_t poff = role ? actor.nparams() : 0;
    const float* __restrict__ p = params + poff;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int q = warp & 3, c = (warp >> 2) & 3;
    const int s = 32 * q + lane;
    {   // weights: small ones plain, W2 as two operand images
        const float* b1 = p + (int64_t)H * d.in;
        const float* W2 = b1 + H;
        const float* b2 = W2 + (int64_t)H * H;
        // relu(S z) = S relu(z) for a power-of-two S: the H1 operand scale is folded into W1 / b1 (bit-identical, one multiply less per feature)
        const float s1 = relu ? kScaleH : 1.0f;
        for (int k = tid; k < kInMax * H; k += NT7_ALL) sm.W1[k] = (k / H) < d.in ? p[k] * s1 : 0.f;
        for (int k = tid; k < H; k += NT7_ALL) { sm.b1[k] = b1[k] * s1; sm.b2[k] = b2[k]; }
        for (int k = tid; k < H * kNo; k += NT7_ALL) {
            int j = k / kNo, o = k % kNo;
            sm.W3[k] = o < d.nout ? p[head_w(d, o, j)] : 0.f;
        }
        if (tid < kNo) sm.b3[tid] = tid < d.nout ? p[head_b(d, tid)] : 0.f;
        for (int k = tid; k < H * H; k += NT7_ALL) {
            int o = k % H, i = k / H;
            const float w = W2[k] * kScaleW;
            const __half wh = __float2half_rn(w), wl = __float2half_rn(w - __half2float(wh));
            *reinterpret_cast<__half*>(sm.B1 + wimg_off(o, i)) = wh;
            *reinterpret_cast<__half*>(sm.B1 + wimg_off(H + o, i)) = wl;
            *reinterpret_cast<__half*>(sm.B2 + wimg_off(i, o)) = wh;
            *reinterpret_cast<__half*>(sm.B2 + wimg_off(H + i, o)) = wl;
        }
    }
    // constant operand rows of GEMM3's B: feature 128 = 1.0 (fp16 0x3C00) for every sample, 129..143 = 0 (the XT buffers are written whole by publish())
    for (int k = tid; k < 2 * TM; k += NT7_ALL)
        *reinterpret_cast<uint4*>(sm.FH_ones + 16 * k) = make_uint4(k < TM ? 0x3C00u : 0u, 0u, 0u, 0u);
    if (warp == 0) umma::tmem_alloc(&sm.tmem, 512);
    if (tid == 32) {
        umma::mbar_init(&sm.bar1, 1); umma::mbar_init(&sm.bar2, 1); umma::mbar_init(&sm.bar3, 1); umma::mbar_init(&sm.bar4, 1);
    }
    umma::fence_proxy_async();
    umma::fence_before_sync();
    __syncthreads();
    umma::fence_after_sync();
    const uint32_t tmem = sm.tmem;
    const uint32_t idesc = umma::make_idesc_f16(128, 64, 0, 0), idesc128 = umma::make_idesc_f16(128, 128, 0, 0);
    const uint32_t idesc144 = umma::make_idesc_f16(128, 144, 1, 1), idesc16 = umma::make_idesc_f16(128, 16, 1, 1);   // GEMM3 / GEMM4: MN-major A and B
    // undo the operand scales (exact powers of two): D1 = H1 W2, D2 = dP2 W2, D3 = dP2^T [H1 | 1], D4 = dP1^T [x | 1]
    const float inv_s1 = 1.0f / (kScaleH * kScaleW), inv_s2 = 1.0f / (scale_p * kScaleW), inv_s3 = 1.0f / (scale_p * kScaleH), inv_sp = 1.0f / scale_p,
                inv_s4 = 1.0f / (scale_p * kScaleX);
    const int64_t ntiles = (b.B + TM - 1) / TM;

    const uint64_t dB1f = umma::make_desc(umma::smem_u32(sm.B1), G_F, GW_S);
    const uint64_t dB2f = umma::make_desc(umma::smem_u32(sm.B2), G_F, GW_S);
    const uint64_t dFPf = umma::make_desc(umma::smem_u32(sm.FP_full), GF_T, GS_T);
    const uint64_t dFHf = umma::make_desc(umma::smem_u32(sm.FH_full), GF_T, GS_T);
    const uint64_t dFQf = umma::make_desc(umma::smem_u32(sm.FQ_full), GF_T, GS_T);
    if (warp >= NT7 / 32) {
        // ================= issuer warpgroup: warp 16 feeds the tensor core, warps 17..19 only return their registers ====
        asm volatile("setmaxnreg.dec.sync.aligned.u32 24;");
        if (warp == NT7 / 32) {
            // 3-term product of a TMEM A operand (hi fp16 pairs at a_col, lo at a_col + 32; 8 columns per K = 16 step) with a
            // [B_hi ; B_lo] weight image, all three terms accumulated into the SAME 64 columns: hi*hi, hi*lo, lo*hi (three N = 64
            // MMAs per K step, ~42 cycles each, instead of one N = 128 + one N = 64: the same pipe time, but the workers read back
            // 64 accumulator columns instead of 128 and add nothing)
            auto issue_ts3 = [&](uint32_t d_col, uint32_t a_col, uint64_t dB) {
                const uint64_t dBlo = dB + (uint64_t)((8 * GW_S) >> 4);   // rows 64..127 of the image
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    const uint64_t adv = (uint64_t)(k * (2 * G_F / 16));
                    umma::mma_f16_ts(tmem + d_col, tmem + a_col + 8 * k, dB + adv, idesc, k ? 1u : 0u);
                    umma::mma_f16_ts(tmem + d_col, tmem + a_col + 8 * k, dBlo + adv, idesc, 1u);
                    umma::mma_f16_ts(tmem + d_col, tmem + a_col + 32 + 8 * k, dB + adv, idesc, 1u);
                }
            };
            // GEMM3 (dW2 += dP2^T x H1, K = 128 samples), ONE M = 128 x N = 128 MMA per K = 16 step: FP_full|FP_lo are adjacent row
            // groups (A rows 0..63 = hi, 64..127 = lo) and FH_full|FH_lo adjacent column groups, so D3[0:64][0:64] = hi*hi,
            // D3[0:64][64:128] = hi*lo, D3[64:128][0:64] = lo*hi (and lo*lo, unused).
            uint32_t d3_acc = 0u;
            auto issue_g3 = [&]() {
#pragma unroll
                for (int k = 0; k < 8; ++k) {
                    const uint64_t adt = (uint64_t)(k * (2 * GF_T / 16));
                    umma::mma_f16(tmem + COL_D3, dFPf + adt, dFHf + adt, idesc144, k ? 1u : d3_acc);   // N = 144: [H1^T hi | H1^T lo | ones]
                }
            };
            // GEMM4 (dW1 | db1 += dP1^T x [x | 1], K = 128 samples): A rows 0..63 = hi, 64..127 = lo; B columns 0..7 = [x hi, 1], 8..15 = x lo
            uint32_t d4_acc = 0u;
            auto issue_g4 = [&](int buf) {
                const uint64_t dXT = umma::make_desc(umma::smem_u32(sm.XT[buf]), GF_T, GS_T);
#pragma unroll
                for (int k = 0; k < 8; ++k) {
                    const uint64_t adt = (uint64_t)(k * (2 * GF_T / 16));
                    umma::mma_f16(tmem + COL_D4, dFQf + adt, dXT + adt, idesc16, k ? 1u : d4_acc);
                }
            };
            // One warp issues every MMA (its elected lane: umma::elect_one), so the tensor pipe executes them in program order: G2(t)
            // reads R1 before G1(t+1) overwrites it without any cross-thread fence.  Per tile: G2(t) | G1(t+1) | G3(t) | G4(t).
            // d3_acc / d4_acc are warp-uniform (every lane tracks them).
            if (cta < ntiles) {
                ready_wait(kBarRdyB);                      // H1 operand of the first tile is in TMEM
                umma::fence_after_sync();
                if (umma::elect_one()) { issue_ts3(COL_R1, COL_AH, dB1f); umma::commit(&sm.bar1); }
                __syncwarp();
            }
            int buf = 0, ord = 0;     // ord = ordinal of the tile within this CTA (the workers count the same way)
#ifdef B200RL_K7_TIMING
            long long tprevi_ = clock64();
#endif
            for (int64_t tile = cta; tile < ntiles; tile += nctas, buf ^= 1, ++ord) {
                if (ord % kFlushTiles == 0) { d3_acc = 0u; d4_acc = 0u; }   // the workers have flushed D3 / D4 before handing this tile's operands over
                ready_wait(kBarRdyA);                      // dP2 operand (TMEM) and the dP2^T / H1^T images (smem) of this tile
                umma::fence_after_sync();
                K7_TI(18);
                if (umma::elect_one()) { issue_ts3(COL_D2, COL_R1, dB2f); umma::commit(&sm.bar2); }      // GEMM2: dH1 = dP2 x W2
                __syncwarp();
                K7_TI(19);
                if (tile + nctas < ntiles) {
                    ready_wait(kBarRdyB);                  // H1 operand of the next tile
                    umma::fence_after_sync();
                    K7_TI(20);
                    if (umma::elect_one()) { issue_ts3(COL_R1, COL_AH, dB1f); umma::commit(&sm.bar1); }  // GEMM1 of the next tile
                    __syncwarp();
                }
                if (umma::elect_one()) { issue_g3(); umma::commit(&sm.bar3); }                   // GEMM3 of this tile
                d3_acc = 1u;
                __syncwarp();
                K7_TI(21);
                ready_wait(kBarRdyC);                      // dP1^T image of this tile (its x^T | 1 operand was written at publish time)
                umma::fence_after_sync();
                K7_TI(22);
                if (umma::elect_one()) { issue_g4(buf); umma::commit(&sm.bar4); }                // GEMM4 of this tile
                d4_acc = 1u;
                __syncwarp();
                K7_TI(23);
            }
        }
    } else {
    // ================= 16 worker warps =======================================================================
    asm volatile("setmaxnreg.inc.sync.aligned.u32 112;");
    const uint32_t lane_base = (uint32_t)(32 * q) << 16;
    // persistent per-thread gradient partials (over this thread's sample slot), reduced once at the end
    float g3[2][16];                  // dW3[o][16c + k]   (db2, dW1, db1 and dW2 are reduced over the samples by the tensor core)
    float gb3a0 = 0.f, gb3a1 = 0.f;   // (c == 0 threads) sum_s dz[o]
#pragma unroll
    for (int k = 0; k < 16; ++k) { g3[0][k] = 0.f; g3[1][k] = 0.f; }
    float l0 = 0.f, l1 = 0.f;
    float mean = 0.f, inv_std = 1.f;
    if (hp.normalize_adv && b.norm2) { mean = b.norm2[0]; inv_std = b.norm2[1]; }
    uint32_t ph1 = 0, ph2 = 0, ph3 = 0, ph4 = 0;
    bool gemm4_pending = false;
    int xbuf = 0;                     // XT buffer of the tile being published (tile parity within this CTA)
    // Random gather, per THREAD: each of the four feature-block threads of a sample loads the sample's whole 32-byte record
    // {state | action bits, logp_old, advantage, return} itself (two 16-byte loads from one sector; the three repeats hit L1), so
    // nothing is exchanged through shared memory and no barrier separates the gather from layer 1 or from the loss.  Software
    // pipeline: the records are requested one tile ahead and the permuted index two tiles ahead (an index array adds a dependent
    // load; the Feistel permutation is ALU work), so neither latency is ever waited for.  No arithmetic on loaded values here.
#ifdef B200RL_K7_TIMING
    long long tprev_ = clock64();
#endif
    const int pbits = b200perm::perm_bits(b.perm_n);
    const uint32_t pkey = ac_perm_key(b);
    auto index_of = [&](int64_t t) -> int32_t {      // rollout index of this thread's sample in tile t, -1 = padding
        const int64_t j = t * TM + s;
        if (t >= ntiles || j >= b.B) return -1;
        return b.idx ? b.idx[j] : (int32_t)perm_index_bits((uint32_t)(b.perm_offset + j), b.perm_n, pkey, pbits);
    };
    auto request = [&](int32_t g, float (&x)[kInMax], float (&a)[4]) {
#pragma unroll
        for (int k = 0; k < kInMax; ++k) { x[k] = 0.f; a[k] = 0.f; }
        if (g < 0) return;
        if (b.rec) {
            const float4 v0 = b.rec[2 * (int64_t)g], v1 = b.rec[2 * (int64_t)g + 1];
            x[0] = v0.x; x[1] = v0.y; x[2] = v0.z; x[3] = v0.w;
            a[0] = v1.x; a[1] = v1.y; a[2] = v1.z; a[3] = v1.w;
        } else {                                     // separate rollout columns (direct API calls)
#pragma unroll
            for (int i = 0; i < kInMax; ++i)         // static indices only: a runtime-indexed array would live in local memory
                if (i < b.ns) x[i] = b.states[(int64_t)b.ns * g + i];
            a[0] = reinterpret_cast<const float*>(b.actions)[g];
            a[1] = b.logp_old ? b.logp_old[g] : 0.f;
            a[2] = b.adv[g];
            a[3] = b.ret[g];
        }
    };
    float pfx[kInMax] = {0.f, 0.f, 0.f, 0.f}, pfa[4] = {0.f, 0.f, 0.f, 0.f};   // records of the NEXT tile (in flight)
    float aux[4] = {0.f, 0.f, 0.f, 0.f};   // {action bits, logp_old, (normalised) advantage, return} of the tile whose loss is evaluated next
    int32_t gi_next = -1;             // index of this thread's sample two tiles ahead
    bool gemm3_pending = false;
    float* const out = partial + (int64_t)cta * np_total + poff;
    float* const gW1 = out;
    float* const gb1 = out + (int64_t)H * d.in;
    float* const gW2 = gb1 + H;
    float* const gb2 = gW2 + (int64_t)H * H;
    for (int k = tid; k < 64 * 65 + 64; k += NT7) sm.AccW2[k] = 0.f;
    for (int k = tid; k < 64 * 9; k += NT7) sm.AccD4[k] = 0.f;
    // flush D3 (dW2 | db2) / D4 (dW1 | db1) into the shared-memory accumulators and let the issuer restart them (see kFlushTiles).
    // Rows 0..63 of an accumulator (hi rows of the A operand) go first, rows 64..127 (lo rows) after a barrier: two threads per
    // entry, in a fixed order => deterministic.  (Stride 65 / 9: the 32 lanes of a warp hit 32 different banks.)
    auto flush_d3 = [&]() {
        if (q < 2) {
            float v[16], v2[16];
            umma::tmem_ld16x2(tmem + lane_base + COL_D3 + 16 * c, tmem + lane_base + COL_D3 + 64 + 16 * c, v, v2);
#pragma unroll
            for (int k = 0; k < 16; ++k) sm.AccW2[s * 65 + 16 * c + k] += v[k] + v2[k];
            if (c == 0) {
                umma::tmem_ld16(tmem + lane_base + COL_D3 + 128, v);
                sm.AccW2[64 * 65 + s] += v[0];
            }
        }
        worker_sync();
        if (q >= 2) {
            float v[16];
            umma::tmem_ld16(tmem + lane_base + COL_D3 + 16 * c, v);
#pragma unroll
            for (int k = 0; k < 16; ++k) sm.AccW2[(s - 64) * 65 + 16 * c + k] += v[k];
            if (c == 0) {
                umma::tmem_ld16(tmem + lane_base + COL_D3 + 128, v);
                sm.AccW2[64 * 65 + (s - 64)] += v[0];
            }
        }
        umma::fence_before_sync();
    };
    auto flush_d4 = [&]() {
        if (c == 0 && q < 2) {
            float d4[16];
            umma::tmem_ld16(tmem + lane_base + COL_D4, d4);
#pragma unroll
            for (int i = 0; i < kInMax; ++i) sm.AccD4[s * 9 + i] += d4[i] + d4[8 + i];
            sm.AccD4[s * 9 + 4] += d4[4];
        }
        worker_sync();
        if (c == 0 && q >= 2) {
            float d4[16];
            umma::tmem_ld16(tmem + lane_base + COL_D4, d4);
#pragma unroll
            for (int i = 0; i < 5; ++i) sm.AccD4[(s - 64) * 9 + i] += d4[i];
        }
        umma::fence_before_sync();
    };
    int ord = 0;   // ordinal of the current tile within this CTA
    // ---- software pipeline (one tile = 128 samples; tensor core and CUDA cores work on different tiles / phases) ----
    //   CUDA cores : ... P3(t) P45(t) | P0(t+1) P1(t+1) | P7(t) | P3(t+1) ...
    //   tensor core:              G2(t) ......... G1(t+1) .... G3(t) .....
    // G2(t) runs under P0/P1(t+1), G1(t+1) under P7(t), G3(t) under P3/P45(t+1); the issuer warp queues each GEMM as soon
    // as the workers have handed its operands over (ready_arrive), so no worker ever blocks on the MMA queue.
    // P0: the next tile's records leave the prefetch registers (x -> layer 1 and the x^T operand of GEMM4, scalars -> aux),
    // the records of the tile after it are requested, the index of the one after that computed / requested
    float xo[kInMax];
    auto publish = [&](int64_t t) {
#pragma unroll
        for (int i = 0; i < kInMax; ++i) xo[i] = pfx[i];
        aux[0] = pfa[0];
        aux[1] = role == 0 ? pfa[1] : 0.f;
        aux[2] = role == 0 ? (hp.normalize_adv ? (pfa[2] - mean) * inv_std : pfa[2]) : 0.f;
        aux[3] = role == 0 ? 0.f : pfa[3];
        if (c == 0) {
            uint32_t h01, l01, h23, l23;   // x^T operand of GEMM4 (features 0..3 hi, 8..11 lo)
            split2(xo[0] * kScaleX, xo[1] * kScaleX, h01, l01);
            split2(xo[2] * kScaleX, xo[3] * kScaleX, h23, l23);
            uint8_t* xt = sm.XT[xbuf] + fimg_off(0, s);
            *reinterpret_cast<uint4*>(xt) = make_uint4(h01, h23, 0x3C00u, 0u);          // features 0..3 = x hi, 4 = 1.0 (-> db1), 5..7 = 0
            *reinterpret_cast<uint4*>(xt + GS_T) = make_uint4(l01, l23, 0u, 0u);       // features 8..11 = x lo
        }
        K7_T(16);
        xbuf ^= 1;
        request(gi_next, pfx, pfa);                  // tile t + nctas
        gi_next = index_of(t + 2 * nctas);
        K7_T(17);
    };
    uint32_t h1pos = 0, h1pos_tile = 0;   // relu: bit k = (H1[16c + k] > 0) of the tile layer1() ran on last / of the tile P7 works on
    auto layer1 = [&]() {   // P1: H1 = act(W1 x + b1) -> TMEM A operand (hi | lo fp16 pairs)
        uint32_t pos = 0;
        uint32_t hi8[8], lo8[8];
#pragma unroll
        for (int ch = 0; ch < 4; ++ch) {
            const int f0 = 16 * c + 4 * ch;
            float4 bb = *reinterpret_cast<const float4*>(sm.b1 + f0);
            float h[4] = {bb.x, bb.y, bb.z, bb.w};
#pragma unroll
            for (int k = 0; k < kInMax; ++k) {
                float4 w = *reinterpret_cast<const float4*>(sm.W1 + k * H + f0);
                h[0] = fmaf(w.x, xo[k], h[0]); h[1] = fmaf(w.y, xo[k], h[1]); h[2] = fmaf(w.z, xo[k], h[2]); h[3] = fmaf(w.w, xo[k], h[3]);
            }
            if (relu) {   // W1 / b1 carry the operand scale already
#pragma unroll
                for (int e = 0; e < 4; ++e) { pos |= (h[e] > 0.f ? 1u : 0u) << (4 * ch + e); h[e] = fmaxf(h[e], 0.f); }
            } else {
#pragma unroll
                for (int e = 0; e < 4; ++e) h[e] = act_f(act, h[e]) * kScaleH;
            }
            split2(h[0], h[1], hi8[2 * ch], lo8[2 * ch]);
            split2(h[2], h[3], hi8[2 * ch + 1], lo8[2 * ch + 1]);
        }
        h1pos = pos;
        umma::tmem_st8(tmem + lane_base + COL_AH + 8 * c, hi8);
        umma::tmem_st8(tmem + lane_base + COL_AH + 32 + 8 * c, lo8);
        umma::tmem_st_wait();
    };
    if (cta < ntiles) {   // prologue: P0 / P1 of the first tile (the issuer queues its G1)
        request(index_of(cta), pfx, pfa);
        gi_next = index_of(cta + nctas);
        publish(cta);
        layer1();
        umma::fence_before_sync();
        ready_arrive(kBarRdyB);
    }
#ifdef B200RL_K7_TIMING
    tprev_ = clock64();
#endif
    for (int64_t tile = cta; tile < ntiles; tile += nctas) {
        const bool has_next = tile + nctas < ntiles;
        // ---- P3: H2 = act(D1 + b2) (registers) + head partials ---------------------------------------
        umma::mbar_wait(&sm.bar1, ph1);
        ph1 ^= 1u;
        umma::fence_after_sync();
        K7_T(0);
        float h2[16];
        {
            float v[16];
            umma::tmem_ld16(tmem + lane_base + COL_R1 + 16 * c, v);
            float zp[kNo] = {0.f, 0.f};
#pragma unroll
            for (int k = 0; k < 16; ++k) {
                const int f = 16 * c + k;
                h2[k] = act_f(act, fmaf(v[k], inv_s1, sm.b2[f]));   // operand scales undone (exact)
                float2 w = *reinterpret_cast<const float2*>(sm.W3 + f * kNo);
                zp[0] = fmaf(w.x, h2[k], zp[0]); zp[1] = fmaf(w.y, h2[k], zp[1]);
            }
#pragma unroll
            for (int o = 0; o < kNo; ++o) sm.Zp[(c * kNo + o) * TM + s] = zp[o];
        }
        K7_T(1);
        group_sync(q);
        K7_T(2);
        // ---- P4+P5: loss (evaluated by all four feature-block threads of a sample: no exchange, no idle warps),
        //            dW3 / db2 partials, dP2 = (W3^T dz) .* act'(H2) -> TMEM A operand (over D1, which this thread
        //            has just consumed) + dP2^T / H1^T images for GEMM3 ----------------------------------------------
        {
            float z[kNo];
#pragma unroll
            for (int o = 0; o < kNo; ++o)
                z[o] = sm.b3[o] + ((sm.Zp[o * TM + s] + sm.Zp[(kNo + o) * TM + s]) + (sm.Zp[(2 * kNo + o) * TM + s] + sm.Zp[(3 * kNo + o) * TM + s]));
            const bool valid = (tile * TM + s) < b.B;
            LossOut lo_ = sample_loss(actor, role, hp, b.inv_B, z, aux[0], aux[1], aux[2], aux[3]);
            float dz[kNo];
#pragma unroll
            for (int o = 0; o < kNo; ++o) dz[o] = valid ? lo_.dz[o] : 0.f;
            if (c == 0 && valid) { l0 += lo_.l0; l1 += lo_.l1; gb3a0 += dz[0]; gb3a1 += dz[1]; }
            // dP2 operand = scale_p * (W3^T dz) .* act'(H2): the power-of-two operand scale rides on dz (exact, bit-identical to scaling dP2)
            const float dzs0 = dz[0] * scale_p, dzs1 = dz[1] * scale_p;
            float dp[16];
#pragma unroll
            for (int k = 0; k < 16; ++k) {
                const int f = 16 * c + k;
                float2 w = *reinterpret_cast<const float2*>(sm.W3 + f * kNo);
                const float dh = fmaf(w.x, dzs0, w.y * dzs1);
                dp[k] = relu ? (h2[k] > 0.f ? dh : 0.f) : dh * (1.f - h2[k] * h2[k]);
                g3[0][k] = fmaf(dz[0], h2[k], g3[0][k]);
                g3[1][k] = fmaf(dz[1], h2[k], g3[1][k]);
            }
            uint32_t hi8[8], lo8[8];
#pragma unroll
            for (int m = 0; m < 8; ++m) split2(dp[2 * m], dp[2 * m + 1], hi8[m], lo8[m]);
            umma::tmem_st8(tmem + lane_base + COL_R1 + 8 * c, hi8);
            umma::tmem_st8(tmem + lane_base + COL_R1 + 32 + 8 * c, lo8);
            K7_T(3);
            if (gemm3_pending) {   // the previous tile's GEMM3 must have consumed the images before they are overwritten
                umma::mbar_wait(&sm.bar3, ph3);
                ph3 ^= 1u;
                umma::fence_after_sync();
                gemm3_pending = false;
            }
            if (ord > 0 && ord % kFlushTiles == 0) flush_d3();   // every GEMM3 so far has completed; the next one restarts the accumulator
            K7_T(4);
            store16_feat(sm.FP_full, 16 * c, s, hi8);
            store16_feat(sm.FP_lo, 16 * c, s, lo8);
            // H1 of this tile (hi | lo fp16 pairs) back from its TMEM operand -> H1^T image
            umma::tmem_ld8x2(tmem + lane_base + COL_AH + 8 * c, tmem + lane_base + COL_AH + 32 + 8 * c, hi8, lo8);
            store16_feat(sm.FH_full, 16 * c, s, hi8);
            store16_feat(sm.FH_lo, 16 * c, s, lo8);
            umma::tmem_st_wait();
        }
        K7_T(5);
        umma::fence_proxy_async();
        umma::fence_before_sync();
        ready_arrive(kBarRdyA);     // this thread's share of the GEMM2 / GEMM3 operands is in place
        gemm3_pending = true;       // (Zp is rewritten in P3 of the next tile, behind its wait for GEMM1, i.e. after every thread has passed
                                    //  this point: no barrier needed here)
        K7_T(6);
        K7_T(7);
        h1pos_tile = h1pos;         // this tile's H1 signs, before layer1() of the next tile replaces them
        if (has_next) {
            if (gemm4_pending) {   // the previous tile's GEMM4 must have consumed its XT buffer (same parity as the next tile's) and the
                umma::mbar_wait(&sm.bar4, ph4);   // dP1^T image before either is overwritten
                ph4 ^= 1u;
                umma::fence_after_sync();
                gemm4_pending = false;
            }
            publish(tile + nctas);
            K7_T(8);
            K7_T(9);
            layer1();
            umma::fence_before_sync();
            K7_T(10);
            ready_arrive(kBarRdyB);
            K7_T(11);
        }
        K7_T(12);
        // ---- P7: dP1 = D2 .* act'(H1) -> dP1^T image (GEMM4 reduces it against [x | 1] into dW1 | db1) ----------
        umma::mbar_wait(&sm.bar2, ph2);
        ph2 ^= 1u;
        umma::fence_after_sync();
        K7_T(13);
        {
            float v[16];
            umma::tmem_ld16(tmem + lane_base + COL_D2 + 16 * c, v);
#pragma unroll
            // D2 carries scale_p * kScaleW; the dP1 operand wants scale_p: one exact power-of-two factor (bit-identical to unscaling
            // to dH1 and rescaling)
            for (int k = 0; k < 16; ++k) v[k] *= 1.0f / kScaleW;
            if (relu) {   // act'(H1) = (H1 > 0): the signs layer1() kept in a register
#pragma unroll
                for (int k = 0; k < 16; ++k) v[k] = ((h1pos_tile >> k) & 1u) ? v[k] : 0.f;
            } else {
                const float inv_h = 1.0f / kScaleH;
#pragma unroll
                for (int g8 = 0; g8 < 2; ++g8) {                               // this tile's H1 = (hi + lo) / scale (image still intact)
                    const uint32_t off = fimg_off(16 * c + 8 * g8, s);
                    const uint4 hv = *reinterpret_cast<const uint4*>(sm.FH_full + off), lv = *reinterpret_cast<const uint4*>(sm.FH_lo + off);
                    const uint32_t hw[4] = {hv.x, hv.y, hv.z, hv.w}, lw[4] = {lv.x, lv.y, lv.z, lv.w};
#pragma unroll
                    for (int m = 0; m < 4; ++m) {
                        const float2 hf = __half22float2(*reinterpret_cast<const __half2*>(&hw[m])), lf = __half22float2(*reinterpret_cast<const __half2*>(&lw[m]));
                        v[8 * g8 + 2 * m] *= dact_f(act, (hf.x + lf.x) * inv_h);
                        v[8 * g8 + 2 * m + 1] *= dact_f(act, (hf.y + lf.y) * inv_h);
                    }
                }
            }
            if (gemm4_pending) {   // (last tile: no publish() waited for it)
                umma::mbar_wait(&sm.bar4, ph4);
                ph4 ^= 1u;
                umma::fence_after_sync();
                gemm4_pending = false;
            }
            if (ord > 0 && ord % kFlushTiles == 0) flush_d4();
            {
                uint32_t hi8[8], lo8[8];
#pragma unroll
                for (int m = 0; m < 8; ++m) split2(v[2 * m], v[2 * m + 1], hi8[m], lo8[m]);
                store16_feat(sm.FQ_full, 16 * c, s, hi8);
                store16_feat(sm.FQ_lo, 16 * c, s, lo8);
            }
            gemm4_pending = true;
        }
        K7_T(14);
#ifdef B200RL_K7_TIMING
        if (tid == (g_k7_watch & 0xFFFF) && (int)blockIdx.x == (g_k7_watch >> 16)) g_k7_phase[15] += 1;
#endif
        umma::fence_proxy_async();
        umma::fence_before_sync();
        ready_arrive(kBarRdyC);
        ++ord;
    }
    // ---- drain: last GEMM3 / GEMM4, final flush, then the head gradients (fixed-order reductions) ---------------
    if (gemm3_pending) umma::mbar_wait(&sm.bar3, ph3);
    if (gemm4_pending) umma::mbar_wait(&sm.bar4, ph4);
    umma::fence_after_sync();
    worker_sync();
    if (cta < ntiles) { flush_d3(); flush_d4(); }        // (a CTA without tiles writes the zeros the accumulators were initialised with)
    worker_sync();
    for (int k = tid; k < H * H; k += NT7) gW2[k] = sm.AccW2[(k & 63) * 65 + (k >> 6)] * inv_s3;     // gW2[j + 64 i]
    if (tid < H) {
        gb2[tid] = sm.AccW2[64 * 65 + tid] * inv_sp;
        gb1[tid] = sm.AccD4[tid * 9 + 4] * inv_sp;
        for (int i = 0; i < d.in; ++i) gW1[tid + H * i] = sm.AccD4[tid * 9 + i] * inv_s4;
    }
    if (cta >= (int)gridDim.x - nctas) {   // surplus row: the other role has no CTA `cta`, its half of the row is zero
        const int64_t ooff = role ? 0 : actor.nparams(), on = role ? actor.nparams() : critic.nparams();
        float* orow = partial + (int64_t)cta * np_total + ooff;
        for (int64_t kk = tid; kk < on; kk += NT7) orow[kk] = 0.f;
    }
    float* red = reinterpret_cast<float*>(sm.FP_full);   // images + weight images: contiguous, all MMAs are done
    static_assert(offsetof(SmemBwd, XT) - offsetof(SmemBwd, FP_full) >= (2 * TM * 65 + 2 * 8 * 64) * 4, "drain scratch");
    // per-sample-slot partials of dW3[0], dW3[1] -> two [128 slots][64] matrices in shared memory -> column sums in
    // a fixed order: 8 segment sums of 16 slots each (all 512 threads), then the 8 segments in order (64 threads per matrix)
    {
        constexpr int RS = 65;                // row stride 65: the 32 lanes (= 32 sample slots) of a store hit 32 different banks
        float* seg = red + 2 * TM * RS;       // [2][8][64]
#pragma unroll
        for (int k = 0; k < 16; ++k) {
            red[0 * TM * RS + s * RS + 16 * c + k] = g3[0][k];
            red[1 * TM * RS + s * RS + 16 * c + k] = g3[1][k];
        }
        worker_sync();
        {
            const int col = tid & 63, g = tid >> 6;   // 8 segments x 64 columns
#pragma unroll
            for (int m = 0; m < 2; ++m) {
                float a = 0.f;
#pragma unroll
                for (int ss = 0; ss < 16; ++ss) a += red[m * TM * RS + (16 * g + ss) * RS + col];
                seg[(m * 8 + g) * 64 + col] = a;
            }
        }
        worker_sync();
        if (tid < 2 * H) {
            const int m = tid >> 6, col = tid & 63;
            float a = 0.f;
#pragma unroll
            for (int g = 0; g < 8; ++g) a += seg[(m * 8 + g) * 64 + col];
            if (m < d.nout) out[head_w(d, m, col)] = a;
        }
        worker_sync();
    }
    if (c == 0) { red[s] = gb3a0; red[TM + s] = gb3a1; }
    worker_sync();
    if (warp < d.nout) {   // one warp per head output: 4 slots per lane in order, then a fixed butterfly (a 128-step dependent chain on one thread was ~2 us)
        float a = (red[warp * TM + lane] + red[warp * TM + 32 + lane]) + (red[warp * TM + 64 + lane] + red[warp * TM + 96 + lane]);
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) a += __shfl_xor_sync(0xffffffffu, a, o);
        if (lane == 0) out[head_b(d, warp)] = a;
    }
    // loss sums (worker-only block reduction)
    float t0 = l0, t1 = l1;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) { t0 += __shfl_xor_sync(0xffffffffu, t0, o); t1 += __shfl_xor_sync(0xffffffffu, t1, o); }
    worker_sync();
    if (lane == 0) { sm.Red[warp] = t0; sm.Red[16 + warp] = t1; }
    worker_sync();
    if (tid == 0) {
        float a0 = 0.f, a1 = 0.f;
        for (int k = 0; k < 16; ++k) { a0 += sm.Red[k]; a1 += sm.Red[16 + k]; }
        float* lp = loss_partial + (int64_t)blockIdx.x * 4;
        lp[0] = role ? 0.f : a0; lp[1] = role ? 0.f : a1; lp[2] = role ? a0 : 0.f; lp[3] = 0.f;
    }
    // ---- fused optimiser step (K8 inside K7's tail): same arithmetic and summation orders as reduce_clip_adam_kernel ----------
    if (st.params) {
        const unsigned int G = gridDim.x;
        K7_T(24);                                // (everything since the last tile: drain, head-gradient reductions, partial rows)
        worker_sync();                           // every worker's partial / loss rows are written (CTA scope) ...
        K7_T(25);
        if (tid == 0) grid_arrive_wait(st.counter, G);   // grid barrier A: every CTA's rows are written and ordered device-wide
        worker_sync();
        K7_T(26);
        const int per = (int)((np_total + G - 1) / G);           // parameters per CTA (<= 512: checked by the launcher)
        const int64_t k = (int64_t)blockIdx.x * per + tid;
        const bool mine = tid < per && k < np_total;
        const unsigned int seq = st.tab.nranks > 1 ? *st.seq_ptr + 1u : 0u;
        // The CTA's slice of every partial row is staged through shared memory by ALL worker threads (every L2 read in flight at
        // once: one round trip instead of one per 16 rows), then one thread per parameter adds its column in CTA order.
        float* stage = reinterpret_cast<float*>(sm.FP_full);            // images are dead: all MMAs have completed
        const int nstage = per * nrows;                                  // <= 64 * 76 floats with the BASELINE network
        const int64_t k0 = (int64_t)blockIdx.x * per;
        {   // (fixed trip count, loads first: a rolled loop would wait for each L2 round trip before issuing the next)
            constexpr int kMaxStage = 10;                                // 10 * 512 >= 64 * 74 (checked by the launcher)
            float t[kMaxStage];
#pragma unroll
            for (int j = 0; j < kMaxStage; ++j) {
                const int e = tid + j * NT7;
                const int row = e / per, col = e - row * per;
                t[j] = (e < nstage && k0 + col < np_total) ? __ldcg(partial + (int64_t)row * np_total + k0 + col) : 0.f;
            }
#pragma unroll
            for (int j = 0; j < kMaxStage; ++j) {
                const int e = tid + j * NT7;
                if (e < nstage) stage[e] = t[j];
            }
        }
        float* lstage = stage + nstage;
        if (blockIdx.x == 0) {
            float t[2];
#pragma unroll
            for (int j = 0; j < 2; ++j) t[j] = tid + j * NT7 < 4 * (int)G ? __ldcg(loss_partial + tid + j * NT7) : 0.f;
#pragma unroll
            for (int j = 0; j < 2; ++j) if (tid + j * NT7 < 4 * (int)G) lstage[tid + j * NT7] = t[j];
        }
        // Adam operands of this thread's parameter: requested now, consumed behind grid barrier B
        float m_k = 0.f, v_k = 0.f, p_k = 0.f;
        if (mine) { m_k = st.m[k]; v_k = st.v[k]; p_k = st.params[k]; }
        worker_sync();
        K7_T(27);
        float gk = 0.f;
        if (mine) {   // rows in CTA order; 8 shared-memory reads in flight
            for (int c0 = 0; c0 < nrows; c0 += 8) {
                float t[8];
#pragma unroll
                for (int j = 0; j < 8; ++j) t[j] = c0 + j < nrows ? stage[(c0 + j) * per + tid] : 0.f;
#pragma unroll
                for (int j = 0; j < 8; ++j) if (c0 + j < nrows) gk += t[j];
            }
        }
        float lsum = 0.f;
        const bool loss_thread = blockIdx.x == 0 && tid < 4;
        if (loss_thread) {
            for (unsigned int c0 = 0; c0 < G; c0 += 8) {
                float t[8];
#pragma unroll
                for (int j = 0; j < 8; ++j) t[j] = c0 + j < G ? lstage[(c0 + j) * 4 + tid] : 0.f;
#pragma unroll
                for (int j = 0; j < 8; ++j) if (c0 + j < G) lsum += t[j];
            }
        }
        if (st.tab.nranks > 1) {   // push the local sums into every peer's inbox, collect the peers' from the own inbox, sum in rank order
            const unsigned slot = seq & 1u;
            if (mine) p2p_push(st.tab, 0, slot, (size_t)k, __float_as_uint(gk), seq);
            if (loss_thread) p2p_push(st.tab, 0, slot, (size_t)np_total + tid, __float_as_uint(lsum), seq);
            // (rank-order sums as p2p_sum_rank_order, gradient and loss words in one loop: kept as it was, like the Adam step below)
            float acc = 0.f, lacc = 0.f;
            for (int r = 0; r < st.tab.nranks; ++r) {
                if (mine) acc += r == st.tab.rank ? gk : __uint_as_float(p2p_recv(st.tab, 0, slot, r, (size_t)k, seq));
                if (loss_thread) lacc += r == st.tab.rank ? lsum : __uint_as_float(p2p_recv(st.tab, 0, slot, r, (size_t)np_total + tid, seq));
            }
            gk = acc; lsum = lacc;
        }
        if (loss_thread) {
            if (st.loss_out4) st.loss_out4[tid] = lsum;
            if (st.stats_row) st.stats_row[tid] = lsum;
        }
        double sq = (double)gk * (double)gk;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) sq += __shfl_xor_sync(0xffffffffu, sq, o);
        if (lane == 0) sm.RedD[warp] = sq;
        worker_sync();
        K7_T(28);
        if (warp == 0) {
            if (lane == 0) {                     // grid barrier B: every CTA's sum of squares is published
                double t = 0.0;
                for (int w = 0; w < NT7 / 32; ++w) t += sm.RedD[w];
                st.cta_sumsq[blockIdx.x] = t;
                grid_arrive_wait(st.counter + 1, G);
            }
            __syncwarp();
            K7_T(29);
            // every lane fetches its share of the per-CTA sums (all reads in flight), adds them in CTA order, then a fixed
            // butterfly over the lanes: deterministic, and every CTA computes the identical total
            double part[8];
#pragma unroll
            for (int j = 0; j < 8; ++j) part[j] = (unsigned)(lane + 32 * j) < G ? __ldcg(st.cta_sumsq + lane + 32 * j) : 0.0;
            double tot = 0.0;
#pragma unroll
            for (int j = 0; j < 8; ++j) tot += part[j];
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) tot += __shfl_xor_sync(0xffffffffu, tot, o);
            if (lane == 0) {
                const float gn = (float)sqrt(tot);
                sm.step_scale = clip_scale(gn, st.max_norm);
                if (blockIdx.x == 0) {
                    if (st.gnorm_out) *st.gnorm_out = gn;
                    if (st.stats_row) st.stats_row[4] = gn;
                }
            }
        }
        worker_sync();
        K7_T(30);
        const float bt1 = st.beta_t[0], bt2 = st.beta_t[1];
        if (mine) {
            gk *= sm.step_scale;
            st.grad[k] = gk;
            // (adam_apply's arithmetic written out: through the helper, register allocation in K7's main loop changes and K7 runs ~0.7 % slower)
            const float mk = st.b1 * m_k + (1.0f - st.b1) * gk;
            const float vk = st.b2 * v_k + (1.0f - st.b2) * (gk * gk);
            st.m[k] = mk; st.v[k] = vk;
            st.params[k] = p_k - mk / (1.0f - bt1) / (sqrtf(vk / (1.0f - bt2)) + st.eps) * st.lr;
        }
        worker_sync();
        if (tid == 0) last_cta_epilogue(st, st.counter + 2, 3, G, bt1, bt2, st.tab.nranks > 1, seq);   // (every thread of every CTA
                                                                                                        //  has read beta^t / seq)
        K7_T(31);
    }
    }  // worker warps
    umma::fence_before_sync();
    __syncthreads();
    if (warp == 0) umma::tmem_dealloc(tmem, 512);
}

}  // namespace

// actor : critic CTA split (tc_split.h); B200RL_K7_ACTOR_CTAS overrides it for tuning runs
int nn_tc_actor_ctas(int grid, const MlpDesc& actor, const AcHyper& hp, int64_t ntiles) {
    static int forced = -2;
    if (forced == -2) { const char* e = getenv("B200RL_K7_ACTOR_CTAS"); forced = e ? atoi(e) : -1; }
    if (forced > 0 && forced < grid) return forced;
    (void)hp;
    return b200rl_tc_actor_ctas(grid, actor.heads2 != 0, ntiles);
}
int nn_tc_partial_rows(int grid, const MlpDesc& actor, const AcHyper& hp, int64_t B) {
    const int na = nn_tc_actor_ctas(grid, actor, hp, (B + TM - 1) / TM);
    return na > grid - na ? na : grid - na;
}
bool nn_tc_bwd_supported(const MlpDesc& actor, const MlpDesc& critic) {
    return actor.H == 64 && critic.H == 64 && actor.in <= kInMax && actor.nout <= 2 && critic.nout == 1;
}
int nn_tc_ac_loss_grad(b200rl_ctx* ctx, int grid, const MlpDesc& actor, const MlpDesc& critic, const float* params, const AcHyper& hp,
                       const AcBatch& b, float* partial, float* loss_partial, int64_t np, const OptStep* step) {
    OptStep st = {};
    const int n_actor = nn_tc_actor_ctas(grid, actor, hp, (b.B + TM - 1) / TM);
    if (step) {   // (opt_path chose OPT_FUSED_TAIL for these sizes)
        st = *step;
        REQUIRE(st.params == params && opt_fused_tail_fits(np, grid, max(n_actor, grid - n_actor), ctx->sm_count), B200RL_ERR_UNSUPPORTED,
                "fused optimiser step: bad configuration");
    }
    size_t smem = sizeof(SmemBwd) + 128;
    static unsigned long long attr_devices = 0;   // once per device
    if (first_use_on_device(attr_devices, ctx->device)) {
        CUDA_TRY(cudaFuncSetAttribute(ac_loss_grad_tc_kernel<B200RL_ACT_RELU>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        CUDA_TRY(cudaFuncSetAttribute(ac_loss_grad_tc_kernel<B200RL_ACT_TANH>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        CUDA_TRY(cudaFuncSetAttribute(ac_loss_grad_tc_kernel<-1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    }
    // dP2 ~ inv_B x O(1..100): scale it into fp16's normal range with a power of two (exact, undone on the accumulators)
    const float scale_base = exp2f(floorf(log2f(1.0f / b.inv_B)));
    if (actor.act == critic.act && actor.act == B200RL_ACT_RELU)
        ac_loss_grad_tc_kernel<B200RL_ACT_RELU><<<grid, NT7_ALL, smem, ctx->stream>>>(actor, critic, params, hp, b, partial, loss_partial, np, scale_base, st, n_actor);
    else if (actor.act == critic.act && actor.act == B200RL_ACT_TANH)
        ac_loss_grad_tc_kernel<B200RL_ACT_TANH><<<grid, NT7_ALL, smem, ctx->stream>>>(actor, critic, params, hp, b, partial, loss_partial, np, scale_base, st, n_actor);
    else
        ac_loss_grad_tc_kernel<-1><<<grid, NT7_ALL, smem, ctx->stream>>>(actor, critic, params, hp, b, partial, loss_partial, np, scale_base, st, n_actor);
    LAUNCH_CHECK(ctx);
    return B200RL_OK;
}

#ifdef B200RL_K7_TIMING
extern "C" int b200rl_debug_k7_watch(int tid) {
    cudaDeviceSynchronize();
    return cudaMemcpyToSymbol(g_k7_watch, &tid, sizeof tid) == cudaSuccess ? 0 : -1;
}
extern "C" int b200rl_debug_k7_phases(unsigned long long* out16, int reset) {
    cudaDeviceSynchronize();
    if (cudaMemcpyFromSymbol(out16, g_k7_phase, sizeof(unsigned long long) * 40) != cudaSuccess) return -1;
    if (reset) { unsigned long long z[24] = {0}; cudaMemcpyToSymbol(g_k7_phase, z, sizeof z); }
    return 0;
}
#endif

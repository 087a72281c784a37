// nn.cu — K6/K7/K8: fused actor-critic / Q-network kernels.
//
// Everything a minibatch needs stays on-chip: a CTA stages the layer weights and a tile of TM
// samples in shared memory and runs layer 1 -> layer 2 -> head -> loss -> backward through
// all layers without touching HBM in between; weight gradients are accumulated in registers
// across the CTA's tiles (persistent CTAs) and written once as a per-CTA partial, which a
// second kernel sums in CTA order (deterministic: same result run to run and for 1 vs G GPUs
// given the same shards).  The dense (H x H) layers are register-tiled FP32 GEMMs
// (8 samples x 4 outputs per thread, operands via LDS.128); see DESIGN.md §K6-K8 for the
// FLOP/byte budget and why the 1e-5 parity bar rules out plain TF32.
//
// Formulas (SURVEY Appendix B; in-tree anchors): logsoftmax + Gumbel-max sampling
// (RLCore/src/utils/networks.jl:405-432), Gaussian head + diagnormlogpdf (networks.jl:44-116,
// distributions.jl:9-34), clip_by_global_norm! (basic.jl:19-29), TargetNetwork sync
// (policies/learners/target_network.jl:70-88).
#include "opt_path.h"
#include "optim.cuh"
#include "perm.cuh"

namespace {

constexpr int NT = 256;
constexpr float kLog2Pi = 1.8378770664093453f;

template <int H> struct Cfg {
    static constexpr int TM = (H == 64) ? 128 : 64;   // samples per tile
    static constexpr int LDA = TM + 4;                // row stride of [feature][sample] tiles
    static constexpr int SG = TM / 8;                 // thread groups along samples
    static constexpr int OG = H / 4;                  // thread groups along outputs
    static constexpr int R = H / 16;                  // dW2 micro-tile edge
    static_assert(SG * OG == NT, "tile/threads mismatch");
};

template <int H, bool BWD> struct Smem {
    using C = Cfg<H>;
    float W1[kInMax * H];      // [i][o]
    float b1[H];
    float W2[H * H];           // [i][o]  (Flux native: W2[o + H*i])
    float b2[H];
    float W2T[BWD ? H * H : 4];  // [o][i]
    float W3[H * kOutMax];     // [j][o] canonical, zero padded
    float b3[kOutMax];
    float X[kInMax * C::LDA];
    float H1[H * C::LDA];
    float H2[H * C::LDA];
    float Out[kOutMax * C::LDA];
    float Dz[BWD ? kOutMax * C::LDA : 4];
    float Aux[4 * C::TM];      // per-sample scalars of the loss stage
    float Red[64];
};

__device__ __forceinline__ float act_f(int act, float z) { return act == B200RL_ACT_RELU ? fmaxf(z, 0.f) : tanhf(z); }
__device__ __forceinline__ float dact_f(int act, float h) { return act == B200RL_ACT_RELU ? (h > 0.f ? 1.f : 0.f) : 1.f - h * h; }

__device__ __forceinline__ uint32_t mix32(uint32_t h) {
    h ^= h >> 16; h *= 0x85EBCA6Bu; h ^= h >> 13; h *= 0xC2B2AE35u; h ^= h >> 16;
    return h;
}
// minibatch permutation: perm.cuh
using b200perm::perm_index;
using b200perm::perm_index_bits;

// head parameter addressing inside the flat parameter vector
__device__ __forceinline__ int64_t head_base(const MlpDesc& d) { return (int64_t)d.H * d.in + d.H + (int64_t)d.H * d.H + d.H; }
__device__ __forceinline__ int64_t head_w(const MlpDesc& d, int o, int j) {
    return head_base(d) + (d.heads2 ? (int64_t)o * (d.H + 1) + j : (int64_t)o + (int64_t)d.nout * j);
}
__device__ __forceinline__ int64_t head_b(const MlpDesc& d, int o) {
    return head_base(d) + (d.heads2 ? (int64_t)o * (d.H + 1) + d.H : (int64_t)d.nout * d.H + o);
}

template <int H, bool BWD> __device__ void load_weights(Smem<H, BWD>& sm, const MlpDesc& d, const float* __restrict__ p) {
    const int tid = threadIdx.x;
    const float* W1 = p;
    const float* b1 = p + (int64_t)H * d.in;
    const float* W2 = b1 + H;
    const float* b2 = W2 + (int64_t)H * H;
    for (int k = tid; k < kInMax * H; k += NT) sm.W1[k] = (k / H) < d.in ? W1[k] : 0.f;
    for (int k = tid; k < H; k += NT) { sm.b1[k] = b1[k]; sm.b2[k] = b2[k]; }
    for (int k = tid; k < H * H; k += NT) {
        float w = W2[k];
        sm.W2[k] = w;
        if (BWD) sm.W2T[(k % H) * H + (k / H)] = w;
    }
    for (int k = tid; k < H * kOutMax; k += NT) {
        int j = k / kOutMax, o = k % kOutMax;
        sm.W3[k] = o < d.nout ? p[head_w(d, o, j)] : 0.f;
    }
    if (tid < kOutMax) sm.b3[tid] = tid < d.nout ? p[head_b(d, tid)] : 0.f;
}

// ---- forward pieces -----------------------------------------------------------------------
// thread tile: samples {4tx..4tx+3} U {TM/2+4tx..+3}, outputs {4ty..4ty+3}
template <int H> __device__ __forceinline__ void tile_coords(int& tx, int& ty) {
    tx = threadIdx.x % Cfg<H>::SG;
    ty = threadIdx.x / Cfg<H>::SG;
}

// acc[c][q] += sum_k A[k][s_q] * Bm[k][4ty + c]
template <int H> __device__ __forceinline__ void gemm_tile(const float* __restrict__ A, const float* __restrict__ Bm, float (&acc)[4][8],
                                                            int tx, int ty) {
    using C = Cfg<H>;
    const float* a0p = A + 4 * tx;
    const float* a1p = A + C::TM / 2 + 4 * tx;
    const float* bp = Bm + 4 * ty;
#pragma unroll 4
    for (int k = 0; k < H; ++k) {
        float4 a0 = *reinterpret_cast<const float4*>(a0p + k * C::LDA);
        float4 a1 = *reinterpret_cast<const float4*>(a1p + k * C::LDA);
        float4 b = *reinterpret_cast<const float4*>(bp + k * H);
        const float av[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
        const float bv[4] = {b.x, b.y, b.z, b.w};
#pragma unroll
        for (int c = 0; c < 4; ++c)
#pragma unroll
            for (int q = 0; q < 8; ++q) acc[c][q] = fmaf(bv[c], av[q], acc[c][q]);
    }
}
template <int H> __device__ __forceinline__ void store_tile(float* __restrict__ D, const float (&v)[4][8], int tx, int ty) {
    using C = Cfg<H>;
#pragma unroll
    for (int c = 0; c < 4; ++c) {
        float* row = D + (4 * ty + c) * C::LDA;
        *reinterpret_cast<float4*>(row + 4 * tx) = make_float4(v[c][0], v[c][1], v[c][2], v[c][3]);
        *reinterpret_cast<float4*>(row + C::TM / 2 + 4 * tx) = make_float4(v[c][4], v[c][5], v[c][6], v[c][7]);
    }
}
template <int H> __device__ __forceinline__ void load_tile(const float* __restrict__ D, float (&v)[4][8], int tx, int ty) {
    using C = Cfg<H>;
#pragma unroll
    for (int c = 0; c < 4; ++c) {
        const float* row = D + (4 * ty + c) * C::LDA;
        float4 a = *reinterpret_cast<const float4*>(row + 4 * tx);
        float4 b = *reinterpret_cast<const float4*>(row + C::TM / 2 + 4 * tx);
        v[c][0] = a.x; v[c][1] = a.y; v[c][2] = a.z; v[c][3] = a.w;
        v[c][4] = b.x; v[c][5] = b.y; v[c][6] = b.z; v[c][7] = b.w;
    }
}

// X -> H1 -> H2 -> Out  (caller syncs before: X ready; after return Out is ready & synced)
template <int H, bool BWD> __device__ void forward_tile(Smem<H, BWD>& sm, const MlpDesc& d) {
    using C = Cfg<H>;
    int tx, ty;
    tile_coords<H>(tx, ty);
    float acc[4][8];
    {   // layer 1 (K = in <= 4)
        float xv[kInMax][8];
#pragma unroll
        for (int i = 0; i < kInMax; ++i) {
            float4 a = *reinterpret_cast<const float4*>(sm.X + i * C::LDA + 4 * tx);
            float4 b = *reinterpret_cast<const float4*>(sm.X + i * C::LDA + C::TM / 2 + 4 * tx);
            xv[i][0] = a.x; xv[i][1] = a.y; xv[i][2] = a.z; xv[i][3] = a.w;
            xv[i][4] = b.x; xv[i][5] = b.y; xv[i][6] = b.z; xv[i][7] = b.w;
        }
#pragma unroll
        for (int c = 0; c < 4; ++c) {
            float bias = sm.b1[4 * ty + c];
#pragma unroll
            for (int q = 0; q < 8; ++q) acc[c][q] = bias;
#pragma unroll
            for (int i = 0; i < kInMax; ++i) {
                float w = sm.W1[i * H + 4 * ty + c];
#pragma unroll
                for (int q = 0; q < 8; ++q) acc[c][q] = fmaf(w, xv[i][q], acc[c][q]);
            }
#pragma unroll
            for (int q = 0; q < 8; ++q) acc[c][q] = act_f(d.act, acc[c][q]);
        }
        store_tile<H>(sm.H1, acc, tx, ty);
    }
    __syncthreads();
#pragma unroll
    for (int c = 0; c < 4; ++c) {
        float bias = sm.b2[4 * ty + c];
#pragma unroll
        for (int q = 0; q < 8; ++q) acc[c][q] = bias;
    }
    gemm_tile<H>(sm.H1, sm.W2, acc, tx, ty);
#pragma unroll
    for (int c = 0; c < 4; ++c)
#pragma unroll
        for (int q = 0; q < 8; ++q) acc[c][q] = act_f(d.act, acc[c][q]);
    store_tile<H>(sm.H2, acc, tx, ty);
    __syncthreads();
    // head: one (output, sample) pair per thread
    for (int pidx = threadIdx.x; pidx < d.nout * C::TM; pidx += NT) {
        int o = pidx / C::TM, s = pidx % C::TM;
        float z = sm.b3[o];
#pragma unroll 8
        for (int k = 0; k < H; ++k) z = fmaf(sm.W3[k * kOutMax + o], sm.H2[k * C::LDA + s], z);
        sm.Out[o * C::LDA + s] = z;
    }
    __syncthreads();
}

// ---- backward pieces ------------------------------------------------------------------------
template <int H> struct GradAcc {
    float w2[Cfg<H>::R][Cfg<H>::R];  // dW2[jt + 16a][it + 16b]
    float w1[(kInMax * H) / NT];     // dW1 flat index tid + NT*r  -> (i = idx / H, j = idx % H)
    float w3[(kOutMax * H + NT - 1) / NT];  // dW3 flat index tid + NT*r -> (o = idx / H, j = idx % H)
    float b1[4], b2[4];              // owned by lanes with tx == 0: outputs 4ty + c
    float b3;                        // thread o < nout
};

// Dz ready (synced).  Accumulates all weight gradients of this tile.
template <int H> __device__ void backward_tile(Smem<H, true>& sm, const MlpDesc& d, GradAcc<H>& g) {
    using C = Cfg<H>;
    int tx, ty;
    tile_coords<H>(tx, ty);
    const int tid = threadIdx.x;
    // dW3 / db3 (needs H2 before it is overwritten)
#pragma unroll
    for (int r = 0; r < (kOutMax * H + NT - 1) / NT; ++r) {
        int idx = tid + NT * r;
        int o = idx / H, j = idx % H;
        if (o < d.nout) {
            float a = 0.f;
            const float* dz = sm.Dz + o * C::LDA;
            const float* h = sm.H2 + j * C::LDA;
#pragma unroll 4
            for (int s = 0; s < C::TM; s += 4) {
                float4 x = *reinterpret_cast<const float4*>(dz + s);
                float4 y = *reinterpret_cast<const float4*>(h + s);
                a = fmaf(x.x, y.x, a); a = fmaf(x.y, y.y, a); a = fmaf(x.z, y.z, a); a = fmaf(x.w, y.w, a);
            }
            g.w3[r] += a;
        }
    }
    if (tid < d.nout) {
        float a = 0.f;
        for (int s = 0; s < C::TM; ++s) a += sm.Dz[tid * C::LDA + s];
        g.b3 += a;
    }
    __syncthreads();
    float v[4][8];
    {   // dP2 = (W3^T dz) .* act'(H2), in place; db2
        load_tile<H>(sm.H2, v, tx, ty);
        float dzv[kOutMax][8];
#pragma unroll
        for (int o = 0; o < kOutMax; ++o) {
            float4 a = *reinterpret_cast<const float4*>(sm.Dz + o * C::LDA + 4 * tx);
            float4 b = *reinterpret_cast<const float4*>(sm.Dz + o * C::LDA + C::TM / 2 + 4 * tx);
            dzv[o][0] = a.x; dzv[o][1] = a.y; dzv[o][2] = a.z; dzv[o][3] = a.w;
            dzv[o][4] = b.x; dzv[o][5] = b.y; dzv[o][6] = b.z; dzv[o][7] = b.w;
        }
#pragma unroll
        for (int c = 0; c < 4; ++c) {
            float4 w = *reinterpret_cast<const float4*>(sm.W3 + (4 * ty + c) * kOutMax);
            const float wv[4] = {w.x, w.y, w.z, w.w};
            float bsum = 0.f;
#pragma unroll
            for (int q = 0; q < 8; ++q) {
                float dh = 0.f;
#pragma unroll
                for (int o = 0; o < kOutMax; ++o) dh = fmaf(wv[o], dzv[o][q], dh);
                float dp = dh * dact_f(d.act, v[c][q]);
                v[c][q] = dp;
                bsum += dp;
            }
#pragma unroll
            for (int off = C::SG / 2; off > 0; off >>= 1) bsum += __shfl_xor_sync(0xffffffffu, bsum, off);
            if (tx == 0) g.b2[c] += bsum;
        }
        store_tile<H>(sm.H2, v, tx, ty);
    }
    __syncthreads();
    {   // dW2[j][i] += sum_s dP2[j][s] * H1[i][s]
        const int jt = tid / 16, it = tid % 16;
#pragma unroll 2
        for (int s = 0; s < C::TM; s += 4) {
            float4 dj[C::R], hi[C::R];
#pragma unroll
            for (int a = 0; a < C::R; ++a) {
                dj[a] = *reinterpret_cast<const float4*>(sm.H2 + (jt + 16 * a) * C::LDA + s);
                hi[a] = *reinterpret_cast<const float4*>(sm.H1 + (it + 16 * a) * C::LDA + s);
            }
#pragma unroll
            for (int a = 0; a < C::R; ++a)
#pragma unroll
                for (int b = 0; b < C::R; ++b) {
                    float t = g.w2[a][b];
                    t = fmaf(dj[a].x, hi[b].x, t); t = fmaf(dj[a].y, hi[b].y, t);
                    t = fmaf(dj[a].z, hi[b].z, t); t = fmaf(dj[a].w, hi[b].w, t);
                    g.w2[a][b] = t;
                }
        }
    }
    __syncthreads();
    {   // dP1 = (W2^T dP2) .* act'(H1), in place; db1
        float acc[4][8];
#pragma unroll
        for (int c = 0; c < 4; ++c)
#pragma unroll
            for (int q = 0; q < 8; ++q) acc[c][q] = 0.f;
        gemm_tile<H>(sm.H2, sm.W2T, acc, tx, ty);
        load_tile<H>(sm.H1, v, tx, ty);
#pragma unroll
        for (int c = 0; c < 4; ++c) {
            float bsum = 0.f;
#pragma unroll
            for (int q = 0; q < 8; ++q) {
                float dp = acc[c][q] * dact_f(d.act, v[c][q]);
                v[c][q] = dp;
                bsum += dp;
            }
#pragma unroll
            for (int off = C::SG / 2; off > 0; off >>= 1) bsum += __shfl_xor_sync(0xffffffffu, bsum, off);
            if (tx == 0) g.b1[c] += bsum;
        }
        store_tile<H>(sm.H1, v, tx, ty);
    }
    __syncthreads();
    // dW1[j][i] += sum_s dP1[j][s] * X[i][s]
#pragma unroll
    for (int r = 0; r < (kInMax * H) / NT; ++r) {
        int idx = tid + NT * r;
        int i = idx / H, j = idx % H;
        float a = 0.f;
        const float* dp = sm.H1 + j * C::LDA;
        const float* x = sm.X + i * C::LDA;
#pragma unroll 4
        for (int s = 0; s < C::TM; s += 4) {
            float4 p4 = *reinterpret_cast<const float4*>(dp + s);
            float4 x4 = *reinterpret_cast<const float4*>(x + s);
            a = fmaf(p4.x, x4.x, a); a = fmaf(p4.y, x4.y, a); a = fmaf(p4.z, x4.z, a); a = fmaf(p4.w, x4.w, a);
        }
        g.w1[r] += a;
    }
    __syncthreads();
}

template <int H> __device__ void zero_grad(GradAcc<H>& g) {
#pragma unroll
    for (int a = 0; a < Cfg<H>::R; ++a)
#pragma unroll
        for (int b = 0; b < Cfg<H>::R; ++b) g.w2[a][b] = 0.f;
#pragma unroll
    for (int r = 0; r < (kInMax * H) / NT; ++r) g.w1[r] = 0.f;
#pragma unroll
    for (int r = 0; r < (kOutMax * H + NT - 1) / NT; ++r) g.w3[r] = 0.f;
#pragma unroll
    for (int c = 0; c < 4; ++c) { g.b1[c] = 0.f; g.b2[c] = 0.f; }
    g.b3 = 0.f;
}

// write this CTA's gradient partial in flat Flux order (out points at this network's slice)
template <int H> __device__ void write_grad(const GradAcc<H>& g, const MlpDesc& d, float* __restrict__ out) {
    using C = Cfg<H>;
    int tx, ty;
    tile_coords<H>(tx, ty);
    const int tid = threadIdx.x;
    float* gW1 = out;
    float* gb1 = out + (int64_t)H * d.in;
    float* gW2 = gb1 + H;
    float* gb2 = gW2 + (int64_t)H * H;
#pragma unroll
    for (int r = 0; r < (kInMax * H) / NT; ++r) {
        int idx = tid + NT * r;
        int i = idx / H, j = idx % H;
        if (i < d.in) gW1[j + H * i] = g.w1[r];
    }
    const int jt = tid / 16, it = tid % 16;
#pragma unroll
    for (int a = 0; a < C::R; ++a)
#pragma unroll
        for (int b = 0; b < C::R; ++b) gW2[(jt + 16 * a) + H * (it + 16 * b)] = g.w2[a][b];
    if (tx == 0) {
#pragma unroll
        for (int c = 0; c < 4; ++c) { gb1[4 * ty + c] = g.b1[c]; gb2[4 * ty + c] = g.b2[c]; }
    }
#pragma unroll
    for (int r = 0; r < (kOutMax * H + NT - 1) / NT; ++r) {
        int idx = tid + NT * r;
        int o = idx / H, j = idx % H;
        if (o < d.nout) out[head_w(d, o, j)] = g.w3[r];
    }
    if (tid < d.nout) out[head_b(d, tid)] = g.b3;
}

__device__ __forceinline__ float block_sum(float v, float* red) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    __syncthreads();
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
    __syncthreads();
    float t = 0.f;
    if (threadIdx.x == 0)
        for (int k = 0; k < NT / 32; ++k) t += red[k];
    return t;  // valid on thread 0
}

__device__ __forceinline__ float softplus_f(float x) { return x > 0.f ? x + log1pf(expf(-x)) : log1pf(expf(x)); }
__device__ __forceinline__ float sigmoid_f(float x) { return 1.f / (1.f + expf(-x)); }
__device__ __forceinline__ float normlogpdf1(float mu, float sigma, float x) {  // diagnormlogpdf, d = 1
    float s = sigma + 1e-8f;
    float v = s * s;
    float dd = x - mu;
    return -0.5f * ((logf(v) + (dd * dd) / v) + kLog2Pi);
}

// ------------------------------------------------------------- actor-critic loss + grad -----
template <int H>
__global__ void __launch_bounds__(NT, (H == 64) ? 2 : 1)
ac_loss_grad_kernel(MlpDesc actor, MlpDesc critic, const float* __restrict__ params, AcHyper hp, AcBatch b, float* __restrict__ partial,
                    float* __restrict__ loss_partial, int64_t np_total) {
    using C = Cfg<H>;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    Smem<H, true>& sm = *reinterpret_cast<Smem<H, true>*>(smem_raw);
    const int role = blockIdx.x & 1;
    const int cta = blockIdx.x >> 1, nctas = gridDim.x >> 1;
    const MlpDesc d = role ? critic : actor;
    const int64_t poff = role ? actor.nparams() : 0;
    load_weights<H, true>(sm, d, params + poff);
    GradAcc<H> g;
    zero_grad<H>(g);
    float l0 = 0.f, l1 = 0.f;  // actor: surrogate sum, entropy sum; critic: squared-error sum
    const int tid = threadIdx.x;
    float mean = 0.f, inv_std = 1.f;
    if (hp.normalize_adv && b.norm2) { mean = b.norm2[0]; inv_std = b.norm2[1]; }
    const int64_t ntiles = (b.B + C::TM - 1) / C::TM;
    __syncthreads();
    for (int64_t tile = cta; tile < ntiles; tile += nctas) {
        if (tid < C::TM) {  // gather
            int64_t j = tile * C::TM + tid;
            bool valid = j < b.B;
            int64_t gidx = 0;
            if (valid) gidx = b.idx ? (int64_t)b.idx[j] : (int64_t)perm_index((uint32_t)(b.perm_offset + j), b.perm_n, ac_perm_key(b));
            float x[kInMax] = {0.f, 0.f, 0.f, 0.f};
            float4 sc4 = make_float4(0.f, 0.f, 0.f, 0.f);
            if (valid) {
                if (b.rec) {   // packed records: the sample's state and scalars share one 32-byte sector
                    float4 v4 = b.rec[2 * gidx];
                    sc4 = b.rec[2 * gidx + 1];
                    x[0] = v4.x; x[1] = v4.y; x[2] = v4.z; x[3] = v4.w;
                } else if (b.ns == 4) {
                    float4 v4 = reinterpret_cast<const float4*>(b.states)[gidx];
                    x[0] = v4.x; x[1] = v4.y; x[2] = v4.z; x[3] = v4.w;
                } else {
                    for (int i = 0; i < b.ns; ++i) x[i] = b.states[(int64_t)b.ns * gidx + i];
                }
            }
#pragma unroll
            for (int i = 0; i < kInMax; ++i) sm.X[i * C::LDA + tid] = x[i];
            float a_bits = 0.f, lp = 0.f, adv = 0.f, ret = 0.f;
            if (valid && b.rec) {
                if (role == 0) {
                    a_bits = sc4.x;
                    lp = sc4.y;
                    adv = (sc4.z - mean) * inv_std;
                    if (!hp.normalize_adv) adv = sc4.z;
                } else {
                    ret = sc4.w;
                }
            } else if (valid) {
                if (role == 0) {
                    a_bits = reinterpret_cast<const float*>(b.actions)[gidx];  // raw 32-bit payload (int32 or float)
                    lp = b.logp_old ? b.logp_old[gidx] : 0.f;
                    adv = (b.adv[gidx] - mean) * inv_std;
                    if (!hp.normalize_adv) adv = b.adv[gidx];
                } else {
                    ret = b.ret[gidx];
                }
            }
            sm.Aux[tid] = a_bits;
            sm.Aux[C::TM + tid] = lp;
            sm.Aux[2 * C::TM + tid] = adv;
            sm.Aux[3 * C::TM + tid] = valid ? ret : __int_as_float(0x7fc00000);  // NaN marks an invalid slot
        }
        __syncthreads();
        forward_tile<H, true>(sm, d);
        if (tid < C::TM) {  // loss stage -> Dz
            const int s = tid;
            bool valid = (tile * C::TM + s) < b.B;
            float dz[kOutMax] = {0.f, 0.f, 0.f, 0.f};
            if (valid) {
                if (role == 1) {
                    float v = sm.Out[s];
                    float err = sm.Aux[3 * C::TM + s] - v;
                    l0 += err * err;
                    dz[0] = -2.0f * hp.w_critic * b.inv_B * err;
                } else {
                    float A = sm.Aux[2 * C::TM + s];
                    float lp_old = sm.Aux[C::TM + s];
                    float logp_a, gsel_scale;  // gsel_scale = d(surrogate)/d(logp_a)
                    if (!actor.heads2) {
                        int na = actor.nout;
                        float z[kOutMax], lp[kOutMax], pr[kOutMax];
                        float m = -3.4e38f;
#pragma unroll
                        for (int o = 0; o < kOutMax; ++o) { z[o] = sm.Out[o * C::LDA + s]; if (o < na) m = fmaxf(m, z[o]); }
                        float se = 0.f;
#pragma unroll
                        for (int o = 0; o < kOutMax; ++o) if (o < na) se += expf(z[o] - m);
                        float ls = logf(se);
                        float Hent = 0.f;
#pragma unroll
                        for (int o = 0; o < kOutMax; ++o) {
                            lp[o] = (z[o] - m) - ls;
                            pr[o] = o < na ? expf(lp[o]) : 0.f;
                            if (o < na) Hent -= pr[o] * lp[o];
                        }
                        int a = __float_as_int(sm.Aux[s]) - 1;
                        logp_a = 0.f;
#pragma unroll
                        for (int o = 0; o < kOutMax; ++o) if (o == a) logp_a = lp[o];
                        l1 += Hent;
                        if (hp.algo == 0) {
                            float ratio = expf(logp_a - lp_old);
                            float u = ratio * A;
                            float rc = fminf(fmaxf(ratio, 1.0f - hp.clip_range), 1.0f + hp.clip_range);
                            float c = rc * A;
                            l0 += -fminf(u, c);
                            bool inside = ratio >= 1.0f - hp.clip_range && ratio <= 1.0f + hp.clip_range;
                            gsel_scale = (u < c || inside) ? u : 0.f;
                        } else {
                            l0 += -(logp_a * A);
                            gsel_scale = A;
                        }
                        float dlogp = -hp.w_actor * b.inv_B * gsel_scale;
#pragma unroll
                        for (int o = 0; o < kOutMax; ++o)
                            if (o < na) dz[o] = dlogp * ((o == a ? 1.f : 0.f) - pr[o]) + hp.w_entropy * b.inv_B * pr[o] * (lp[o] + Hent);
                    } else {
                        float mu = sm.Out[s], raw = sm.Out[C::LDA + s];
                        float sp = softplus_f(raw);
                        float sigma = fminf(fmaxf(sp, hp.min_sigma), hp.max_sigma);
                        bool clamped = sp < hp.min_sigma || sp > hp.max_sigma;
                        float a = sm.Aux[s];
                        logp_a = normlogpdf1(mu, sigma, a);
                        float Hent = logf(sigma) + 0.5f * (kLog2Pi + 1.0f);
                        l1 += Hent;
                        if (hp.algo == 0) {
                            float ratio = expf(logp_a - lp_old);
                            float u = ratio * A;
                            float rc = fminf(fmaxf(ratio, 1.0f - hp.clip_range), 1.0f + hp.clip_range);
                            float c = rc * A;
                            l0 += -fminf(u, c);
                            bool inside = ratio >= 1.0f - hp.clip_range && ratio <= 1.0f + hp.clip_range;
                            gsel_scale = (u < c || inside) ? u : 0.f;
                        } else {
                            l0 += -(logp_a * A);
                            gsel_scale = A;
                        }
                        float dlogp = -hp.w_actor * b.inv_B * gsel_scale;
                        float sg = sigma + 1e-8f, dd = a - mu;
                        dz[0] = dlogp * (dd / (sg * sg));
                        float dsig = dlogp * (-1.0f / sg + (dd * dd) / (sg * sg * sg)) - hp.w_entropy * b.inv_B * (1.0f / sigma);
                        dz[1] = clamped ? 0.f : dsig * sigmoid_f(raw);
                    }
                }
            }
#pragma unroll
            for (int o = 0; o < kOutMax; ++o) sm.Dz[o * C::LDA + s] = dz[o];
        }
        __syncthreads();
        backward_tile<H>(sm, d, g);
    }
    write_grad<H>(g, d, partial + (int64_t)cta * np_total + poff);
    float t0 = block_sum(l0, sm.Red);
    float t1 = block_sum(l1, sm.Red);
    if (tid == 0) {
        float* lp = loss_partial + (int64_t)blockIdx.x * 4;  // actor rows: {surrogate, entropy, 0, 0}; critic rows: {0, 0, sq.err, 0}
        lp[0] = role ? 0.f : t0; lp[1] = role ? 0.f : t1; lp[2] = role ? t0 : 0.f; lp[3] = 0.f;
    }
}

// ------------------------------------------------------------- rollout inference ------------
__device__ __forceinline__ void load_rng32(const unsigned long long* rng, int64_t i, unsigned long long (&s)[4]) {
    const ulonglong2* p = reinterpret_cast<const ulonglong2*>(rng + 4 * i);
    ulonglong2 a = p[0], b = p[1];
    s[0] = a.x; s[1] = a.y; s[2] = b.x; s[3] = b.y;
}
__device__ __forceinline__ void store_rng32(unsigned long long* rng, int64_t i, const unsigned long long (&s)[4]) {
    ulonglong2* p = reinterpret_cast<ulonglong2*>(rng + 4 * i);
    p[0] = make_ulonglong2(s[0], s[1]);
    p[1] = make_ulonglong2(s[2], s[3]);
}
__device__ __forceinline__ unsigned long long xo_next(unsigned long long (&s)[4]) {
    unsigned long long tmp = s[0] + s[3];
    unsigned long long res = ((tmp << 23) | (tmp >> 41)) + s[0];
    unsigned long long t = s[1] << 17;
    s[2] ^= s[0]; s[3] ^= s[1]; s[1] ^= s[2]; s[0] ^= s[3]; s[2] ^= t;
    s[3] = (s[3] << 45) | (s[3] >> 19);
    return res;
}
__device__ __forceinline__ double xo_f64(unsigned long long (&s)[4]) { return (double)(xo_next(s) >> 11) * 0x1p-53; }
__device__ __forceinline__ float xo_f32(unsigned long long (&s)[4]) { return (float)((unsigned)(xo_next(s) >> 32) >> 8) * 0x1p-24f; }

// mode 0: actor-critic rollout (roles), 1: plain forward of `actor` desc (single role) -> head_out
template <int H>
__global__ void __launch_bounds__(NT, (H == 64) ? 2 : 1)
forward_kernel(MlpDesc actor, MlpDesc critic, const float* __restrict__ params, AcHyper hp, int mode, const float* __restrict__ obs,
               int64_t N, unsigned long long* __restrict__ rng, void* __restrict__ action_out, float* __restrict__ logp_out,
               float* __restrict__ value_out, float* __restrict__ head_out, float* __restrict__ state_copy) {
    using C = Cfg<H>;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    Smem<H, false>& sm = *reinterpret_cast<Smem<H, false>*>(smem_raw);
    const int nroles = mode == 0 ? 2 : 1;
    const int role = mode == 0 ? (blockIdx.x & 1) : 0;
    const int cta = blockIdx.x / nroles, nctas = gridDim.x / nroles;
    const MlpDesc d = role ? critic : actor;
    const int64_t poff = role ? actor.nparams() : 0;
    load_weights<H, false>(sm, d, params + poff);
    const int tid = threadIdx.x;
    const int64_t ntiles = (N + C::TM - 1) / C::TM;
    __syncthreads();
    for (int64_t tile = cta; tile < ntiles; tile += nctas) {
        if (tid < C::TM) {
            int64_t i = tile * C::TM + tid;
            float x[kInMax] = {0.f, 0.f, 0.f, 0.f};
            if (i < N) {
                if (d.in == 4) {
                    float4 v4 = reinterpret_cast<const float4*>(obs)[i];
                    x[0] = v4.x; x[1] = v4.y; x[2] = v4.z; x[3] = v4.w;
                    if (state_copy && role == 0) reinterpret_cast<float4*>(state_copy)[i] = v4;
                } else {
                    for (int k = 0; k < d.in; ++k) {
                        x[k] = obs[(int64_t)d.in * i + k];
                        if (state_copy && role == 0) state_copy[(int64_t)d.in * i + k] = x[k];
                    }
                }
            }
#pragma unroll
            for (int k = 0; k < kInMax; ++k) sm.X[k * C::LDA + tid] = x[k];
        }
        __syncthreads();
        forward_tile<H, false>(sm, d);
        if (tid < C::TM) {
            int64_t i = tile * C::TM + tid;
            if (i < N) {
                if (head_out && (mode == 1 || role == 0))
                    for (int o = 0; o < d.nout; ++o) head_out[(int64_t)d.nout * i + o] = sm.Out[o * C::LDA + tid];
                if (mode == 0 && role == 1) {
                    if (value_out) value_out[i] = sm.Out[tid];
                } else if (mode == 0) {
                    unsigned long long st[4];
                    load_rng32(rng, i, st);
                    if (!actor.heads2) {  // sample_categorical: argmax(-log(-log(u)) + logp), u Float64
                        int na = actor.nout;
                        float z[kOutMax], lp[kOutMax];
                        float m = -3.4e38f;
#pragma unroll
                        for (int o = 0; o < kOutMax; ++o) { z[o] = sm.Out[o * C::LDA + tid]; if (o < na) m = fmaxf(m, z[o]); }
                        float se = 0.f;
#pragma unroll
                        for (int o = 0; o < kOutMax; ++o) if (o < na) se += expf(z[o] - m);
                        float ls = logf(se);
                        int best = 0;
                        double bv = 0.0;
                        float blp = 0.f;
#pragma unroll
                        for (int o = 0; o < kOutMax; ++o) {
                            if (o < na) {
                                lp[o] = (z[o] - m) - ls;
                                double u = xo_f64(st);
                                double gv = -log(-log(u)) + (double)lp[o];
                                if (o == 0 || gv > bv) { bv = gv; best = o; blp = lp[o]; }
                            }
                        }
                        if (action_out) reinterpret_cast<int32_t*>(action_out)[i] = best + 1;
                        if (logp_out) logp_out[i] = blp;
                    } else {  // GaussianNetwork: a = mu + sigma * n
                        float mu = sm.Out[tid], raw = sm.Out[C::LDA + tid];
                        float sigma = fminf(fmaxf(softplus_f(raw), hp.min_sigma), hp.max_sigma);
                        float u1 = xo_f32(st), u2 = xo_f32(st);
                        float n = sqrtf(-2.0f * logf(1.0f - u1)) * cosf(6.2831855f * u2);
                        float a = mu + sigma * n;
                        if (action_out) reinterpret_cast<float*>(action_out)[i] = a;
                        if (logp_out) logp_out[i] = normlogpdf1(mu, sigma, a);
                    }
                    store_rng32(rng, i, st);
                }
            }
        }
        __syncthreads();
    }
}

// ------------------------------------------------------------- reduce / clip / Adam ---------
__global__ void reduce_partials_kernel(const float* __restrict__ partial, int n_partials, int64_t np, float* __restrict__ grad,
                                       const float* __restrict__ loss_partial, int n_loss, float* __restrict__ loss_out4) {
    int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (k < np) {
        float a = 0.f;
        for (int c = 0; c < n_partials; ++c) a += partial[(int64_t)c * np + k];
        grad[k] = a;
    }
    if (blockIdx.x == 0 && threadIdx.x < 4 && loss_out4) {
        float a = 0.f;
        for (int c = 0; c < n_loss; ++c) a += loss_partial[c * 4 + threadIdx.x];
        loss_out4[threadIdx.x] = a;
    }
}

// single CTA: gn = sqrt(sum g^2) (fixed tree, double), clip_by_global_norm!, Optimisers Adam
__global__ void __launch_bounds__(1024) clip_adam_kernel(float* __restrict__ p, float* __restrict__ g, float* __restrict__ m,
                                                         float* __restrict__ v, float* __restrict__ beta_t, int64_t np, float max_norm,
                                                         float lr, float b1, float b2, float eps, float grad_scale,
                                                         float* __restrict__ gnorm_out) {
    __shared__ double red[32];
    __shared__ float s_scale;
    double acc = 0.0;
    for (int64_t k = threadIdx.x; k < np; k += blockDim.x) {
        float x = g[k] * grad_scale;
        acc += (double)x * (double)x;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
    __syncthreads();
    if (threadIdx.x == 0) {
        double t = 0.0;
        for (int k = 0; k < (int)(blockDim.x >> 5); ++k) t += red[k];
        float gn = (float)sqrt(t);
        s_scale = clip_scale(gn, max_norm);
        if (gnorm_out) *gnorm_out = gn;
    }
    __syncthreads();
    const float sc = s_scale * grad_scale;
    const float bt1 = beta_t[0], bt2 = beta_t[1];
    for (int64_t k = threadIdx.x; k < np; k += blockDim.x) {
        float gk = g[k] * sc;
        g[k] = gk;
        p[k] -= adam_apply(gk, m[k], v[k], b1, b2, eps, lr, bt1, bt2);
    }
    __syncthreads();
    if (threadIdx.x == 0) { beta_t[0] = bt1 * b1; beta_t[1] = bt2 * b2; }
}

// Fused K8: partial reduce -> [peer exchange over NVLink] -> global norm -> clip -> Adam in ONE launch.  The CTAs meet at a
// device-wide counter (all ceil(np/256) <= 148 CTAs are co-resident), every CTA then sums the per-CTA sum-of-squares in
// CTA order, so the result is bit-identical to the two-kernel path and run-to-run deterministic.
// XCHG (sharded run, SURVEY §8e): every thread pushes its element of the local gradient into the peers' inboxes as a
// self-validating {value, sequence} packet (remote NVLink store), then reads the peers' packets from the own inbox and sums
// in rank order — every rank computes the identical global gradient, so the replicas stay bit-identical without a broadcast.
template <bool XCHG>
__global__ void __launch_bounds__(256) reduce_clip_adam_kernel(const float* __restrict__ partial, int n_partials, int64_t np,
                                                              const float* __restrict__ loss_partial, int n_loss, OptStep st) {
    __shared__ double red[8];
    __shared__ float s_scale;
    // The grid barrier counters reset themselves (the last CTA through the second counter zeroes both), the exchange sequence
    // number and the update tick live in device memory: nothing here depends on host-side launch counts, so the launch can be
    // captured in a CUDA graph and replayed, and no counter ever wraps.
    float* __restrict__ p = st.params; float* __restrict__ g = st.grad; float* __restrict__ m = st.m; float* __restrict__ v = st.v;
    const P2PTable& tab = st.tab;
    const unsigned int target = gridDim.x;
    const unsigned int seq = XCHG ? *st.seq_ptr + 1u : 0u;
    const int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    float gk = 0.f;
    if (k < np) {
        for (int c = 0; c < n_partials; ++c) gk += partial[(int64_t)c * np + k];
    }
    float lsum = 0.f;
    const bool loss_thread = blockIdx.x == 0 && threadIdx.x < 4;
    if (loss_thread)
        for (int c = 0; c < n_loss; ++c) lsum += loss_partial[c * 4 + threadIdx.x];
    if (XCHG) {   // push the local chunk into every peer's inbox, then collect the peers' chunks from the own inbox
        const unsigned slot = seq & 1u;
        if (k < np) p2p_push(tab, 0, slot, (size_t)k, __float_as_uint(gk), seq);
        if (loss_thread) p2p_push(tab, 0, slot, (size_t)np + threadIdx.x, __float_as_uint(lsum), seq);   // the 4 loss sums ride along
        if (k < np) gk = p2p_sum_rank_order(tab, slot, (size_t)k, gk, seq);
        if (loss_thread) lsum = p2p_sum_rank_order(tab, slot, (size_t)np + threadIdx.x, lsum, seq);
    }
    if (loss_thread) {
        if (st.loss_out4) st.loss_out4[threadIdx.x] = lsum;
        if (st.stats_row) st.stats_row[threadIdx.x] = lsum;
    }
    double acc = (double)gk * (double)gk;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
    __syncthreads();
    if (threadIdx.x < 32) {   // warp 0: lane 0 publishes and waits at the grid barrier, then all lanes fetch the per-CTA sums in parallel
        if (threadIdx.x == 0) {
            double t = 0.0;
            for (int w = 0; w < 8; ++w) t += red[w];
            st.cta_sumsq[blockIdx.x] = t;
            grid_arrive_wait(st.counter, target);
        }
        __syncwarp();
        // (one dependent L2 read per CTA was ~5 us of this ~14 us kernel; the loads now go out together, the adds keep the CTA order)
        double tot = 0.0;
        for (unsigned int c0 = 0; c0 < gridDim.x; c0 += 32) {
            const unsigned int c = c0 + threadIdx.x;
            const double mine = c < gridDim.x ? *reinterpret_cast<volatile double*>(st.cta_sumsq + c) : 0.0;
            const unsigned int n = min(32u, gridDim.x - c0);
            for (unsigned int l = 0; l < n; ++l) tot += __shfl_sync(0xffffffffu, mine, l);
        }
    if (threadIdx.x == 0) {
        float gn = (float)sqrt(tot);
        s_scale = clip_scale(gn, st.max_norm);
        if (blockIdx.x == 0) {
            if (st.gnorm_out) *st.gnorm_out = gn;
            if (st.stats_row) st.stats_row[4] = gn;
        }
    }
    }
    __syncthreads();
    const float bt1 = st.beta_t[0], bt2 = st.beta_t[1];
    if (k < np) {
        gk *= s_scale;
        g[k] = gk;
        p[k] -= adam_apply(gk, m[k], v[k], st.b1, st.b2, st.eps, st.lr, bt1, bt2);
    }
    // beta^t advances once every CTA has read it: the last CTA to pass a second counter does it
    __syncthreads();
    if (threadIdx.x == 0) {
        __threadfence();
        last_cta_epilogue(st, st.counter + 1, 2, target, bt1, bt2, XCHG, seq);
    }
}

__global__ void target_sync_kernel(float* __restrict__ target, const float* __restrict__ model, int64_t np, float rho) {
    int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (k < np) target[k] = rho * target[k] + (1.0f - rho) * model[k];
}

// ------------------------------------------------------------- DQN --------------------------
// phase A (forward_kernel mode 1 on the target / online nets) gives Q(s') tables; this kernel
// does the online forward on s, the TD loss and the backward.
template <int H>
__global__ void __launch_bounds__(NT, (H == 64) ? 2 : 1)
dqn_loss_grad_kernel(MlpDesc q, const float* __restrict__ params, const float* __restrict__ s, const int32_t* __restrict__ a,
                     const float* __restrict__ r, const uint8_t* __restrict__ t, const float* __restrict__ qnext_t,
                     const float* __restrict__ qnext_o, const float* __restrict__ w, int64_t B, float inv_B, float gamma, int huber,
                     float* __restrict__ partial, float* __restrict__ loss_partial, float* __restrict__ td_out) {
    using C = Cfg<H>;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    Smem<H, true>& sm = *reinterpret_cast<Smem<H, true>*>(smem_raw);
    const int cta = blockIdx.x, nctas = gridDim.x;
    load_weights<H, true>(sm, q, params);
    GradAcc<H> g;
    zero_grad<H>(g);
    float l0 = 0.f;
    const int tid = threadIdx.x;
    const int64_t ntiles = (B + C::TM - 1) / C::TM;
    const int64_t np = q.nparams();
    __syncthreads();
    for (int64_t tile = cta; tile < ntiles; tile += nctas) {
        if (tid < C::TM) {
            int64_t j = tile * C::TM + tid;
            float x[kInMax] = {0.f, 0.f, 0.f, 0.f};
            if (j < B)
                for (int i = 0; i < q.in; ++i) x[i] = s[(int64_t)q.in * j + i];
#pragma unroll
            for (int i = 0; i < kInMax; ++i) sm.X[i * C::LDA + tid] = x[i];
        }
        __syncthreads();
        forward_tile<H, true>(sm, q);
        if (tid < C::TM) {
            int64_t j = tile * C::TM + tid;
            float dz[kOutMax] = {0.f, 0.f, 0.f, 0.f};
            if (j < B) {
                int na = q.nout;
                float qn;
                if (qnext_o) {  // double DQN: argmax from the online net, value from the target net
                    int best = 0;
                    for (int o = 1; o < na; ++o) if (qnext_o[(int64_t)na * j + o] > qnext_o[(int64_t)na * j + best]) best = o;
                    qn = qnext_t[(int64_t)na * j + best];
                } else {
                    qn = qnext_t[(int64_t)na * j];
                    for (int o = 1; o < na; ++o) qn = fmaxf(qn, qnext_t[(int64_t)na * j + o]);
                }
                float R = r[j] + gamma * (t[j] ? 0.f : 1.f) * qn;
                int ai = a[j] - 1;
                float qv = 0.f;
#pragma unroll
                for (int o = 0; o < kOutMax; ++o) if (o == ai) qv = sm.Out[o * C::LDA + tid];
                float e = R - qv;
                td_out[j] = e;
                float wi = w ? w[j] : 1.f;
                float ae = fabsf(e), l, dl;
                if (huber) {
                    if (ae < 1.0f) { l = 0.5f * e * e; dl = -e; }
                    else { l = ae - 0.5f; dl = e > 0.f ? -1.f : 1.f; }
                } else { l = e * e; dl = -2.0f * e; }
                l0 += wi * l;
#pragma unroll
                for (int o = 0; o < kOutMax; ++o) if (o == ai) dz[o] = wi * inv_B * dl;
            }
#pragma unroll
            for (int o = 0; o < kOutMax; ++o) sm.Dz[o * C::LDA + tid] = dz[o];
        }
        __syncthreads();
        backward_tile<H>(sm, q, g);
    }
    write_grad<H>(g, q, partial + (int64_t)cta * np);
    float t0 = block_sum(l0, sm.Red);
    if (tid == 0) {
        float* lp = loss_partial + (int64_t)blockIdx.x * 4;
        lp[0] = t0; lp[1] = 0.f; lp[2] = 0.f; lp[3] = 0.f;
    }
}

// epsilon-greedy over a (na, N) Q table (EpsilonGreedyExplorer, explorers/epsilon_greedy_explorer.jl:69-131):
// with prob epsilon a uniform random action, else the arg-max (first max wins).
__global__ void q_act_kernel(const float* __restrict__ qv, int na, int64_t N, unsigned long long* __restrict__ rng, float epsilon,
                             int32_t* __restrict__ action_out) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= N) return;
    int best = 0;
    for (int o = 1; o < na; ++o) if (qv[(int64_t)na * i + o] > qv[(int64_t)na * i + best]) best = o;
    if (epsilon > 0.f) {
        unsigned long long st[4];
        load_rng32(rng, i, st);
        double u = xo_f64(st);
        if (u < (double)epsilon) {
            unsigned long long x = xo_next(st);
            best = (int)__umul64hi(x, (unsigned long long)na);
        }
        store_rng32(rng, i, st);
    }
    action_out[i] = best + 1;
}

// rand(rng, Base.OneTo(n)) — Lemire nearly-divisionless on UInt64 (Julia 1.10 SamplerRangeNDL), 1-based
__device__ __forceinline__ int xo_oneto(unsigned long long (&s)[4], unsigned long long n) {
    unsigned long long x = xo_next(s);
    unsigned long long hi = __umul64hi(x, n), lo = x * n;
    if (lo < n) {
        unsigned long long t = (0ull - n) % n;
        while (lo < t) {
            x = xo_next(s);
            hi = __umul64hi(x, n);
            lo = x * n;
        }
    }
    return (int)hi + 1;
}
// get_ϵ(s::EpsilonGreedyExplorer{:linear | :exp}, step) (epsilon_greedy_explorer.jl:69-91): Float64, evaluated left to
// right with explicitly rounded operations (no FMA contraction, like the reference's Julia code)
__device__ __forceinline__ double explorer_eps(const b200rl_explorer& e, long long step) {
    if (step <= e.warmup_steps) return e.eps_init;
    if (e.kind == 0) {
        if (step >= e.warmup_steps + e.decay_steps) return e.eps_stable;
        long long steps_left = e.warmup_steps + e.decay_steps - step;
        return __dadd_rn(e.eps_stable, __dmul_rn(__ddiv_rn((double)steps_left, (double)e.decay_steps), __dsub_rn(e.eps_init, e.eps_stable)));
    }
    long long n = step - e.warmup_steps;
    double scale = __dsub_rn(e.eps_init, e.eps_stable);
    return __dadd_rn(e.eps_stable, __dmul_rn(scale, exp(__ddiv_rn(__dmul_rn(-1.0, (double)n), (double)e.decay_steps))));
}
// BatchExplorer(EpsilonGreedyExplorer) over the columns of a (na, N) Q table (explorers/batch_explorer.jl:15-21,
// epsilon_greedy_explorer.jl:102-112): column i is planned with get_ϵ(step + i) — the inner explorer's step advances once
// per column — drawing from its own stream: rand(rng) >= ϵ ? (findmax | rand(rng, find_all_max)) : rand(rng, 1:na).
// The uniform draw happens even when ϵ = 0, exactly like the reference.
__global__ void q_explore_kernel(const float* __restrict__ qv, int na, int64_t N, unsigned long long* __restrict__ rng, b200rl_explorer ex,
                                 int32_t* __restrict__ action_out) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= N) return;
    const float* v = qv + (int64_t)na * i;
    const double eps = explorer_eps(ex, ex.step + i);
    unsigned long long st[4];
    load_rng32(rng, i, st);
    const double u = xo_f64(st);
    int action;
    if (u >= eps) {
        int best = 0;
        for (int o = 1; o < na; ++o) {
            const float a = v[o], b = v[best];
            if ((a != a && b == b) || a > b) best = o;     // findmax: first maximum, NaN ranks highest
        }
        action = best + 1;
        if (ex.is_break_tie) {
            float mx = v[0];
            for (int o = 1; o < na; ++o) mx = v[o] > mx ? v[o] : mx;
            int cnt = 0;
            for (int o = 0; o < na; ++o) cnt += v[o] == mx;
            int pick = xo_oneto(st, (unsigned long long)(cnt > 0 ? cnt : 1));
            for (int o = 0; o < na; ++o) {
                if (v[o] == mx && --pick == 0) { action = o + 1; break; }
            }
        }
    } else {
        action = xo_oneto(st, (unsigned long long)na);
    }
    store_rng32(rng, i, st);
    action_out[i] = action;
}

template <int H, bool BWD> constexpr size_t smem_bytes() { return sizeof(Smem<H, BWD>); }

template <class K> int set_smem(K kernel, size_t bytes) {
    CUDA_TRY(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes));
    return B200RL_OK;
}

}  // namespace

static int g_tc = -1;
bool nn_tc_enabled() {
    if (g_tc < 0) {
        const char* e = getenv("B200RL_TC");
        g_tc = (e && e[0] == '0') ? 0 : 1;
    }
    return g_tc != 0;
}
extern "C" int b200rl_set_tensor_cores(int enable) { g_tc = enable ? 1 : 0; return B200RL_OK; }
static int g_fused_step = -1;   // -1: not decided yet (environment), see nn_ac_loss_grad_step
extern "C" int b200rl_set_fused_step(int enable) { g_fused_step = enable ? 1 : 0; return B200RL_OK; }
bool nn_fused_step_enabled() {
    if (g_fused_step < 0) { const char* e = getenv("B200RL_FUSED_STEP"); g_fused_step = (e && e[0] == '0') ? 0 : 1; }
    return g_fused_step != 0;
}
static int tc_grid(b200rl_ctx* ctx) { return 2 * (ctx->sm_count / 2); }   // one 512-thread CTA per SM, split between the roles (nn_tc_actor_ctas)

int nn_grid_ctas(b200rl_ctx* ctx, int H) { return H == 64 ? ctx->sm_count : ctx->sm_count / 2; }

template <int H>
static int launch_forward(b200rl_ctx* ctx, int grid, const MlpDesc& actor, const MlpDesc& critic, const float* params, const AcHyper& hp,
                          int mode, const float* obs, int64_t N, unsigned long long* rng, void* action_out, float* logp_out,
                          float* value_out, float* head_out, float* state_copy) {
    TRY(set_smem(forward_kernel<H>, smem_bytes<H, false>()));
    forward_kernel<H><<<grid, NT, smem_bytes<H, false>(), ctx->stream>>>(actor, critic, params, hp, mode, obs, N, rng, action_out, logp_out,
                                                                         value_out, head_out, state_copy);
    LAUNCH_CHECK(ctx);
    return B200RL_OK;
}
template <int H>
static int launch_ac(b200rl_ctx* ctx, int grid, const MlpDesc& actor, const MlpDesc& critic, const float* params, const AcHyper& hp,
                     const AcBatch& b, float* partial, float* loss_partial, int64_t np) {
    TRY(set_smem(ac_loss_grad_kernel<H>, smem_bytes<H, true>()));
    ac_loss_grad_kernel<H><<<grid, NT, smem_bytes<H, true>(), ctx->stream>>>(actor, critic, params, hp, b, partial, loss_partial, np);
    LAUNCH_CHECK(ctx);
    return B200RL_OK;
}
template <int H>
static int launch_dqn(b200rl_ctx* ctx, int grid, const MlpDesc& q, const float* params, const float* s, const int32_t* a, const float* r,
                      const uint8_t* t, const float* qt, const float* qo, const float* w, int64_t B, float inv_B, float gamma, int huber,
                      float* partial, float* loss_partial, float* td_out) {
    TRY(set_smem(dqn_loss_grad_kernel<H>, smem_bytes<H, true>()));
    dqn_loss_grad_kernel<H><<<grid, NT, smem_bytes<H, true>(), ctx->stream>>>(q, params, s, a, r, t, qt, qo, w, B, inv_B, gamma, huber, partial,
                                                                             loss_partial, td_out);
    LAUNCH_CHECK(ctx);
    return B200RL_OK;
}

static int check_desc(const MlpDesc& d) {
    REQUIRE(d.in >= 1 && d.in <= kInMax, B200RL_ERR_UNSUPPORTED, "observation width must be 1..4");
    REQUIRE(d.nout >= 1 && d.nout <= kOutMax, B200RL_ERR_UNSUPPORTED, "head width must be 1..4");
    REQUIRE(d.H == 64 || d.H == 128, B200RL_ERR_UNSUPPORTED, "hidden width must be 64 or 128");
    REQUIRE(!d.heads2 || d.nout == 2, B200RL_ERR_UNSUPPORTED, "gaussian head supports 1-d actions");
    return B200RL_OK;
}
static int tiles_for(int H, int64_t n) {
    int64_t tm = H == 64 ? Cfg<64>::TM : Cfg<128>::TM;
    int64_t t = (n + tm - 1) / tm;
    return t > (1 << 30) ? (1 << 30) : (int)t;
}

int nn_policy_act(b200rl_ctx* ctx, const MlpDesc& actor, const MlpDesc& critic, const float* params, const AcHyper& hp, const float* obs,
                  int64_t N, unsigned long long* rng, void* action_out, float* logp_out, float* value_out, float* head_out,
                  float* state_copy) {
    TRY(check_desc(actor)); TRY(check_desc(critic));
    REQUIRE(actor.H == critic.H && actor.in == critic.in, B200RL_ERR_UNSUPPORTED, "actor and critic must share widths");
    int ctas = nn_grid_ctas(ctx, actor.H);
    int nt = tiles_for(actor.H, N);
    if (ctas > nt) ctas = nt;
    if (nn_tc_enabled() && nn_tc_supported(actor) && nn_tc_supported(critic))
        return nn_tc_forward(ctx, 2 * ctas, actor, critic, params, hp, 0, obs, N, rng, action_out, logp_out, value_out, head_out, state_copy);
    if (actor.H == 64) return launch_forward<64>(ctx, 2 * ctas, actor, critic, params, hp, 0, obs, N, rng, action_out, logp_out, value_out, head_out, state_copy);
    return launch_forward<128>(ctx, 2 * ctas, actor, critic, params, hp, 0, obs, N, rng, action_out, logp_out, value_out, head_out, state_copy);
}

int nn_mlp_forward(b200rl_ctx* ctx, const MlpDesc& net, const float* params, const float* obs, int64_t N, float* out) {
    TRY(check_desc(net));
    int ctas = net.H == 64 ? 2 * ctx->sm_count : ctx->sm_count;
    int nt = tiles_for(net.H, N);
    if (ctas > nt) ctas = nt;
    AcHyper hp{};
    if (nn_tc_enabled() && nn_tc_supported(net))
        return nn_tc_forward(ctx, ctas, net, net, params, hp, 1, obs, N, nullptr, nullptr, nullptr, nullptr, out, nullptr);
    if (net.H == 64) return launch_forward<64>(ctx, ctas, net, net, params, hp, 1, obs, N, nullptr, nullptr, nullptr, nullptr, out, nullptr);
    return launch_forward<128>(ctx, ctas, net, net, params, hp, 1, obs, N, nullptr, nullptr, nullptr, nullptr, out, nullptr);
}

int nn_ac_loss_grad(b200rl_ctx* ctx, const MlpDesc& actor, const MlpDesc& critic, const float* params, const AcHyper& hp, const AcBatch& b,
                    float* partial, float* loss_partial) {
    TRY(check_desc(actor)); TRY(check_desc(critic));
    REQUIRE(actor.H == critic.H && actor.in == critic.in, B200RL_ERR_UNSUPPORTED, "actor and critic must share widths");
    int64_t np = actor.nparams() + critic.nparams();
    int st;
    if (nn_tc_enabled() && nn_tc_bwd_supported(actor, critic))
        st = nn_tc_ac_loss_grad(ctx, tc_grid(ctx), actor, critic, params, hp, b, partial, loss_partial, np, nullptr);
    else if (actor.H == 64)
        st = launch_ac<64>(ctx, 2 * nn_grid_ctas(ctx, 64), actor, critic, params, hp, b, partial, loss_partial, np);
    else
        st = launch_ac<128>(ctx, 2 * nn_grid_ctas(ctx, 128), actor, critic, params, hp, b, partial, loss_partial, np);
    return st != B200RL_OK ? st : nn_ac_partial_rows(ctx, actor, critic, hp, b.B);  // number of gradient partials written (loss rows = 2x)
}
int nn_ac_partial_rows(b200rl_ctx* ctx, const MlpDesc& actor, const MlpDesc& critic, const AcHyper& hp, int64_t B) {
    if (nn_tc_enabled() && nn_tc_bwd_supported(actor, critic)) return nn_tc_partial_rows(tc_grid(ctx), actor, hp, B);
    return nn_grid_ctas(ctx, actor.H);
}
bool nn_tc_fused_tail_fits(b200rl_ctx* ctx, const MlpDesc& actor, const AcHyper& hp, int64_t B, int64_t np) {
    return opt_fused_tail_fits(np, tc_grid(ctx), nn_tc_partial_rows(tc_grid(ctx), actor, hp, B), ctx->sm_count);
}

// K7 + optimiser step in ONE launch.  A sharded run takes it only when every rank owns its device (P2PTable::exclusive): the launch
// occupies all SMs and waits for the peers' packets inside itself.
int nn_ac_loss_grad_step(b200rl_ctx* ctx, const MlpDesc& actor, const MlpDesc& critic, const AcHyper& hp, const AcBatch& b, float* partial,
                         float* loss_partial, const OptStep& st) {
    TRY(check_desc(actor)); TRY(check_desc(critic));
    const int64_t np = actor.nparams() + critic.nparams();
    TRY(nn_tc_ac_loss_grad(ctx, tc_grid(ctx), actor, critic, st.params, hp, b, partial, loss_partial, np, &st));
    return nn_tc_partial_rows(tc_grid(ctx), actor, hp, b.B);
}

int nn_reduce_partials(b200rl_ctx* ctx, const float* partial, int n_partials, int64_t np, float* grad, const float* loss_partial,
                       int n_loss_partials, float* loss_out4) {
    reduce_partials_kernel<<<grid_for(np, 256), 256, 0, ctx->stream>>>(partial, n_partials, np, grad, loss_partial, n_loss_partials, loss_out4);
    LAUNCH_CHECK(ctx);
    return B200RL_OK;
}

int nn_clip_adam(b200rl_ctx* ctx, float* params, float* grad, float* m, float* v, float* beta_t, int64_t np, float max_grad_norm, float lr,
                 float b1, float b2, float eps, float grad_scale, float* gnorm_out) {
    clip_adam_kernel<<<1, 1024, 0, ctx->stream>>>(params, grad, m, v, beta_t, np, max_grad_norm, lr, b1, b2, eps, grad_scale, gnorm_out);
    LAUNCH_CHECK(ctx);
    return B200RL_OK;
}

int nn_reduce_clip_adam(b200rl_ctx* ctx, const float* partial, int n_partials, int64_t np, const float* loss_partial, int n_loss, const OptStep& st) {
    unsigned grid = grid_for(np, 256);
    REQUIRE((int)grid <= ctx->sm_count, B200RL_ERR_UNSUPPORTED, "fused reduce+Adam needs all CTAs co-resident");
    if (st.tab.nranks > 1) {
        REQUIRE((size_t)np + 4 <= kP2PXCap, B200RL_ERR_UNSUPPORTED, "gradient larger than the peer exchange inbox");
        reduce_clip_adam_kernel<true><<<grid, 256, 0, ctx->stream>>>(partial, n_partials, np, loss_partial, n_loss, st);
    } else {
        reduce_clip_adam_kernel<false><<<grid, 256, 0, ctx->stream>>>(partial, n_partials, np, loss_partial, n_loss, st);
    }
    LAUNCH_CHECK(ctx);
    return B200RL_OK;
}

int nn_target_sync(b200rl_ctx* ctx, float* target, const float* model, int64_t np, float rho) {
    target_sync_kernel<<<grid_for(np, 256), 256, 0, ctx->stream>>>(target, model, np, rho);
    LAUNCH_CHECK(ctx);
    return B200RL_OK;
}

// returns the number of gradient partials written (> 0) or a negative status
int nn_dqn_loss_grad(b200rl_ctx* ctx, const MlpDesc& q, const float* params, const float* target, const float* s, const int32_t* a,
                     const float* r, const uint8_t* t, const float* s2, const float* w, int64_t B, float inv_B, float gamma, int huber,
                     int double_dqn, float* partial, float* loss_partial, float* td_out) {
    TRY(check_desc(q));
    // Q(s') tables in ctx scratch: target net always, online net for double DQN
    void* scratch;
    TRY(ctx_scratch(ctx, (size_t)B * q.nout * sizeof(float) * 2 + 256, &scratch));
    float* qt = (float*)scratch;
    float* qo = qt + (size_t)B * q.nout;
    TRY(nn_mlp_forward(ctx, q, target, s2, B, qt));
    if (double_dqn) TRY(nn_mlp_forward(ctx, q, params, s2, B, qo));
    int ctas = nn_dqn_max_partials(ctx, q.H);
    int nt = tiles_for(q.H, B);
    if (ctas > nt) ctas = nt;
    int st = q.H == 64 ? launch_dqn<64>(ctx, ctas, q, params, s, a, r, t, qt, double_dqn ? qo : nullptr, w, B, inv_B, gamma, huber, partial, loss_partial, td_out)
                       : launch_dqn<128>(ctx, ctas, q, params, s, a, r, t, qt, double_dqn ? qo : nullptr, w, B, inv_B, gamma, huber, partial, loss_partial, td_out);
    if (st != B200RL_OK) return st;
    return ctas;
}
int nn_dqn_max_partials(b200rl_ctx* ctx, int H) { return H == 64 ? 2 * ctx->sm_count : ctx->sm_count; }

int nn_q_explore(b200rl_ctx* ctx, const MlpDesc& q, const float* params, const float* obs, int64_t N, unsigned long long* rng,
                 const b200rl_explorer& ex, int32_t* action_out, float* q_out) {
    TRY(nn_mlp_forward(ctx, q, params, obs, N, q_out));
    q_explore_kernel<<<grid_for(N, 256), 256, 0, ctx->stream>>>(q_out, q.nout, N, rng, ex, action_out);
    LAUNCH_CHECK(ctx);
    return B200RL_OK;
}
int nn_q_act(b200rl_ctx* ctx, const MlpDesc& q, const float* params, const float* obs, int64_t N, unsigned long long* rng, float epsilon,
             int32_t* action_out, float* q_out) {
    TRY(nn_mlp_forward(ctx, q, params, obs, N, q_out));
    q_act_kernel<<<grid_for(N, 256), 256, 0, ctx->stream>>>(q_out, q.nout, N, rng, epsilon, action_out);
    LAUNCH_CHECK(ctx);
    return B200RL_OK;
}

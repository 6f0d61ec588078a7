// lfa.cu -- RandLA-Net local feature aggregation hot loop, fused:
//   neighbour gather -> LocSE 10-channel encoding -> shared MLP(s) -> attention scores
//   (Linear d->d) -> softmax over the K neighbours -> weighted sum        ==> agg [N, d]
// One kernel per attentive-pooling stage; nothing of shape [N, K, *] ever reaches HBM.
//
// Replaces (reference /root/reference/ml3d/torch/models/randlanet.py):
//   LocalSpatialEncoding.forward   :521-605   (gather_neighbor :533-553)
//   AttentivePooling.forward       :608-639   (score_fn + softmax(dim=-2) + sum)
//   the lse1/pool1/lse2/pool2 part of LocalFeatureAggregation.forward :667-692
// Stage 1: X = [f1[nbr] | r1],  r1 = lrelu(BN(W10 . enc10))
// Stage 2: X = [p1[nbr] | r2],  r2 = lrelu(BN(Wl2 . r1)),  r1 recomputed (cheaper than 4*K*d/2 B/pt)
// The pooled d-vector then goes through the generic gathered GEMM (gemm.cu) for
// the pool MLP / mlp2+shortcut.
//
// Layout per CTA (256 threads, P = 1024/D points, R = 16 P neighbour rows):
//   Xt [D][R+4]    feature-major tile of X      (64 KB)   A operand, LDS.128 along rows
//   R1t[D/2][R+4]  stage 2 only                 (32 KB)
//   Wsl[BK][D]     streamed weight k-slices
// Thread (p, cg) owns the 16 neighbour rows of point p x 4 score channels, so the
// softmax over K and the weighted sum stay in registers.
// FP32 SIMT version (bit-level close to the reference); the tcgen05 3xTF32
// variant plugs into the same tiles.
#include "../../include/o3dml_b200.h"
#include "common.cuh"
#include <string.h>

namespace o3dml {

constexpr int LFA_K = 16;
constexpr int LFA_THREADS = 256;
constexpr int LFA_BK = 16;

struct LfaParams {
    const float* coords;   // [B*N, 3]
    const void* nidx;      // [B, N, 16] batch-relative
    int nidx_is64;
    const float* feat;     // [B*N, D/2]  (f1 for stage 1, p1 for stage 2)
    int64_t total;         // B*N
    int64_t n_per_batch;   // N
    const float* w10t;     // [10][D/2]
    const float* s10;      // [D/2] folded BN scale
    const float* t10;      // [D/2] folded BN shift (+bias)
    const float* wl2t;     // [D/2][D/2]   stage 2
    const float* s2;
    const float* t2;
    const float* wst;      // [D][D] score weight, [in][out]
    const float* bs;       // [D]
    float* agg;            // [B*N, D]
};

template <int D>
struct LfaCfg {
    static constexpr int H = D / 2;
    static constexpr int P = 1024 / D;        // points per CTA
    static constexpr int R = LFA_K * P;       // neighbour rows per CTA
    static constexpr int RS = R + 4;          // padded row stride of the transposed tiles
    static constexpr int CG = D / 4;          // column groups (threads) per point
    static constexpr int XT_FLOATS = D * RS;
    static constexpr int R1_FLOATS = H * RS;
    static constexpr int ENC_FLOATS = 10 * R;
    static constexpr int WSL_FLOATS = LFA_BK * D;
    static constexpr int SCRATCH_FLOATS = ENC_FLOATS > WSL_FLOATS ? ENC_FLOATS : WSL_FLOATS;
    static constexpr int W10_FLOATS = 12 * H;  // 10 rows + scale + shift
    static size_t smem_bytes(int stage) {
        return sizeof(float) * (size_t)(XT_FLOATS + (stage == 2 ? R1_FLOATS : 0) + SCRATCH_FLOATS +
                                        W10_FLOATS) + R * sizeof(int);
    }
};

template <int D, int STAGE>
__global__ void __launch_bounds__(LFA_THREADS)
lfa_pool_kernel(const __grid_constant__ LfaParams p) {
    using C = LfaCfg<D>;
    constexpr int H = C::H, P = C::P, R = C::R, RS = C::RS, CG = C::CG;
    extern __shared__ __align__(16) float smem[];
    float* Xt = smem;                                   // [D][RS]
    float* R1t = Xt + C::XT_FLOATS;                     // [H][RS] (stage 2)
    float* scratch = R1t + (STAGE == 2 ? C::R1_FLOATS : 0);  // Enc[10][R]  /  Wsl[BK][D]
    float* W10 = scratch + C::SCRATCH_FLOATS;           // [12][H]
    int* nbr = reinterpret_cast<int*>(W10 + C::W10_FLOATS);  // [R] global neighbour row or -1

    const int tid = threadIdx.x;
    const int64_t pt0 = (int64_t)blockIdx.x * P;

    // ---- stage constants
    for (int i = tid; i < 10 * H; i += LFA_THREADS) W10[i] = p.w10t[i];
    for (int i = tid; i < H; i += LFA_THREADS) {
        W10[10 * H + i] = p.s10[i];
        W10[11 * H + i] = p.t10[i];
    }
    // ---- step 1a: neighbour ids + 10-channel encoding  -> Enc[10][R]
    float* Enc = scratch;
    for (int r = tid; r < R; r += LFA_THREADS) {
        const int pl = r / LFA_K;
        const int64_t g = pt0 + pl;
        int nb = -1;
        float e[10];
#pragma unroll
        for (int q = 0; q < 10; ++q) e[q] = 0.f;
        if (g < p.total) {
            const int64_t b = g / p.n_per_batch;
            const int64_t li = load_index(p.nidx, g * LFA_K + (r % LFA_K), p.nidx_is64);
            const int64_t gn = b * p.n_per_batch + li;
            nb = (int)gn;
            const float qx = p.coords[3 * g], qy = p.coords[3 * g + 1], qz = p.coords[3 * g + 2];
            const float cx = p.coords[3 * gn], cy = p.coords[3 * gn + 1], cz = p.coords[3 * gn + 2];
            const float dx = qx - cx, dy = qy - cy, dz = qz - cz;
            e[0] = sqrtf(__fadd_rn(__fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy)), __fmul_rn(dz, dz)));
            e[1] = dx; e[2] = dy; e[3] = dz;
            e[4] = qx; e[5] = qy; e[6] = qz;
            e[7] = cx; e[8] = cy; e[9] = cz;
        }
        nbr[r] = nb;
#pragma unroll
        for (int q = 0; q < 10; ++q) Enc[q * R + r] = e[q];
    }
    __syncthreads();

    // ---- step 1b: r1 = lrelu(BN(W10 . enc))  -> Xt[H + o][r] (stage 1) or R1t[o][r] (stage 2)
    {
        float* dst = (STAGE == 1) ? (Xt + (size_t)H * RS) : R1t;
        constexpr int OG = H / 8;  // groups of 8 outputs
        for (int w = tid; w < R * OG; w += LFA_THREADS) {
            const int r = w % R, og = w / R;
            float e[10];
#pragma unroll
            for (int q = 0; q < 10; ++q) e[q] = Enc[q * R + r];
#pragma unroll
            for (int o8 = 0; o8 < 8; ++o8) {
                const int o = og * 8 + o8;
                float a = 0.f;
#pragma unroll
                for (int q = 0; q < 10; ++q) a = fmaf(e[q], W10[q * H + o], a);
                a = fmaf(a, W10[10 * H + o], W10[11 * H + o]);
                dst[(size_t)o * RS + r] = a >= 0.f ? a : 0.2f * a;
            }
        }
    }
    // ---- step 1c: gather neighbour features -> Xt[c][r], c < H
    {
        constexpr int CH4 = H / 4;
        for (int w = tid; w < R * CH4; w += LFA_THREADS) {
            const int r = w % R, c4 = (w / R) * 4;
            const int nb = nbr[r];
            float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
            if (nb >= 0) v = *reinterpret_cast<const float4*>(p.feat + (size_t)nb * H + c4);
            Xt[(size_t)(c4 + 0) * RS + r] = v.x;
            Xt[(size_t)(c4 + 1) * RS + r] = v.y;
            Xt[(size_t)(c4 + 2) * RS + r] = v.z;
            Xt[(size_t)(c4 + 3) * RS + r] = v.w;
        }
    }
    __syncthreads();  // Enc dead from here on: scratch becomes the weight-slice buffer
    float* Wsl = scratch;
    const int pl = tid / CG, cg = tid % CG;  // point within CTA, column group
    const int rbase = pl * LFA_K;

    // ---- step 2 (stage 2): r2 = lrelu(BN(Wl2 . r1)) -> Xt[H + o][r]; thread = 16 rows x 2 cols
    if (STAGE == 2) {
        float acc[LFA_K][2];
#pragma unroll
        for (int j = 0; j < LFA_K; ++j) acc[j][0] = acc[j][1] = 0.f;
        constexpr int BK2 = H < LFA_BK ? H : LFA_BK;  // d_out = 16 has only 8 input channels
        for (int k0 = 0; k0 < H; k0 += BK2) {
            for (int i = tid; i < BK2 * H / 4; i += LFA_THREADS) {
                const int kk = i / (H / 4), c = (i % (H / 4)) * 4;
                *reinterpret_cast<float4*>(&Wsl[kk * H + c]) =
                    *reinterpret_cast<const float4*>(p.wl2t + (size_t)(k0 + kk) * H + c);
            }
            __syncthreads();
#pragma unroll
            for (int kk = 0; kk < BK2; ++kk) {
                const float* arow = R1t + (size_t)(k0 + kk) * RS + rbase;
                float a[LFA_K];
#pragma unroll
                for (int j4 = 0; j4 < LFA_K / 4; ++j4) {
                    const float4 t = *reinterpret_cast<const float4*>(arow + 4 * j4);
                    a[4 * j4] = t.x; a[4 * j4 + 1] = t.y; a[4 * j4 + 2] = t.z; a[4 * j4 + 3] = t.w;
                }
                const float2 b = *reinterpret_cast<const float2*>(&Wsl[kk * H + cg * 2]);
#pragma unroll
                for (int j = 0; j < LFA_K; ++j) {
                    acc[j][0] = fmaf(a[j], b.x, acc[j][0]);
                    acc[j][1] = fmaf(a[j], b.y, acc[j][1]);
                }
            }
            __syncthreads();
        }
#pragma unroll
        for (int e = 0; e < 2; ++e) {
            const int o = cg * 2 + e;
            const float s = p.s2[o], t = p.t2[o];
#pragma unroll
            for (int j = 0; j < LFA_K; ++j) {
                float v = fmaf(acc[j][e], s, t);
                Xt[(size_t)(H + o) * RS + rbase + j] = v >= 0.f ? v : 0.2f * v;
            }
        }
        __syncthreads();
    }

    // ---- step 3: scores = X . Ws + b ; softmax over the 16 rows ; agg = sum_j softmax * X
    float acc[LFA_K][4];
    {
        const float4 b4 = *reinterpret_cast<const float4*>(p.bs + cg * 4);
#pragma unroll
        for (int j = 0; j < LFA_K; ++j) {
            acc[j][0] = b4.x; acc[j][1] = b4.y; acc[j][2] = b4.z; acc[j][3] = b4.w;
        }
    }
    for (int k0 = 0; k0 < D; k0 += LFA_BK) {
        for (int i = tid; i < LFA_BK * D / 4; i += LFA_THREADS) {
            const int kk = i / (D / 4), c = (i % (D / 4)) * 4;
            *reinterpret_cast<float4*>(&Wsl[kk * D + c]) =
                *reinterpret_cast<const float4*>(p.wst + (size_t)(k0 + kk) * D + c);
        }
        __syncthreads();
#pragma unroll
        for (int kk = 0; kk < LFA_BK; ++kk) {
            const float* arow = Xt + (size_t)(k0 + kk) * RS + rbase;
            float a[LFA_K];
#pragma unroll
            for (int j4 = 0; j4 < LFA_K / 4; ++j4) {
                const float4 t = *reinterpret_cast<const float4*>(arow + 4 * j4);
                a[4 * j4] = t.x; a[4 * j4 + 1] = t.y; a[4 * j4 + 2] = t.z; a[4 * j4 + 3] = t.w;
            }
            const float4 b = *reinterpret_cast<const float4*>(&Wsl[kk * D + cg * 4]);
#pragma unroll
            for (int j = 0; j < LFA_K; ++j) {
                acc[j][0] = fmaf(a[j], b.x, acc[j][0]);
                acc[j][1] = fmaf(a[j], b.y, acc[j][1]);
                acc[j][2] = fmaf(a[j], b.z, acc[j][2]);
                acc[j][3] = fmaf(a[j], b.w, acc[j][3]);
            }
        }
        __syncthreads();
    }
    const int64_t g = pt0 + pl;
    float out[4];
#pragma unroll
    for (int e = 0; e < 4; ++e) {
        float m = acc[0][e];
#pragma unroll
        for (int j = 1; j < LFA_K; ++j) m = fmaxf(m, acc[j][e]);
        const float* xrow = Xt + (size_t)(cg * 4 + e) * RS + rbase;
        float num = 0.f, den = 0.f;
#pragma unroll
        for (int j4 = 0; j4 < LFA_K / 4; ++j4) {
            const float4 x = *reinterpret_cast<const float4*>(xrow + 4 * j4);
            const float e0 = expf(acc[4 * j4 + 0][e] - m), e1 = expf(acc[4 * j4 + 1][e] - m);
            const float e2 = expf(acc[4 * j4 + 2][e] - m), e3 = expf(acc[4 * j4 + 3][e] - m);
            den += (e0 + e1) + (e2 + e3);
            num = fmaf(e0, x.x, num);
            num = fmaf(e1, x.y, num);
            num = fmaf(e2, x.z, num);
            num = fmaf(e3, x.w, num);
        }
        out[e] = num / den;
    }
    if (g < p.total)
        *reinterpret_cast<float4*>(p.agg + (size_t)g * D + cg * 4) =
            make_float4(out[0], out[1], out[2], out[3]);
}

template <int D, int STAGE>
static int lfa_launch(const LfaParams& p, cudaStream_t st) {
    using C = LfaCfg<D>;
    const size_t smem = C::smem_bytes(STAGE);
    static PerDeviceOnce once;
    const int dev = current_device();
    if (once.need(dev)) {
        O3DML_CUDA(cudaFuncSetAttribute(lfa_pool_kernel<D, STAGE>,
                                        cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        once.done(dev);
    }
    const unsigned blocks = (unsigned)ceil_div<int64_t>(p.total, C::P);
    lfa_pool_kernel<D, STAGE><<<blocks, LFA_THREADS, smem, st>>>(p);
    O3DML_LAUNCH_CHECK();
    o3dml_count_launches(1);
    return O3DML_OK;
}


// ---------------------------------------------------------------------------------------------
// d_out = 16 (the first, largest level: N points x 16 neighbours, 8 + 8 channels) in the model.  The tiled
// kernel above keeps ~2.2 KB of shared memory per point, i.e. <= 12 warps per SM, and at this width the
// gathers (not the FMAs) are what has to be hidden.  Here one THREAD owns one neighbour row end to end in
// registers (encoding -> lse1 [-> lse2] -> 16 scores), and only the [16 rows x 16 channels] scores /
// features of a point cross shared memory once, channel-major, for the softmax over the neighbours.
// 256 threads = 16 points, 34 KB of shared memory.
//
// The layer's weights travel in the KERNEL PARAMETER block (constant bank 0): every FFMA takes its weight as
// a c[0][imm] operand, so no instruction and no register-file write is spent on loading weights.  (Read from
// shared memory as warp-uniform LDS.128, they cost 440 cycles of shared-memory return path per warp against
// 206 issue cycles: such a kernel is bound by the broadcast writes, not by the FMAs.)  The host passes the
// packed weights from HOST memory.
constexpr int L16_PTS = 16;                 // points per CTA pass
constexpr int L16_ROWS = L16_PTS * LFA_K;   // 256 rows = threads
constexpr int L16_RS = L16_ROWS + 4;        // channel-major row stride (conflict-free LDS.128)
constexpr int L16C_CTAS = 5;                // resident CTAs per SM the register allocation is held to (42 registers)

struct alignas(16) Lfa16W {
    float v[O3DML_LFA16_WEIGHT_FLOATS];
};
constexpr int W16_W10 = 0, W16_S10 = 80, W16_T10 = 88, W16_WL2 = 96, W16_S2 = 160, W16_T2 = 168,
              W16_WS = 176, W16_BS = 432;

// Each CTA walks groups of 16 points with a grid stride, and the neighbour index of its next group is
// requested one group ahead, kept as a raw loaded word until that group comes up (common.cuh): the two
// dependent round trips index -> coordinates / feature row were 23 % of the stall samples without it
// (profiles/r02_lfa_stalls.md).
template <int STAGE>
__global__ void __launch_bounds__(L16_ROWS, L16C_CTAS)
lfa16c_kernel(const __grid_constant__ LfaParams p, const __grid_constant__ Lfa16W w, int64_t num_groups) {
    constexpr int D = 16, H = 8;
    __shared__ __align__(16) float St[D * L16_RS];      // scores, channel-major
    __shared__ __align__(16) float Xs[D * L16_RS];      // X, channel-major
    const int tid = threadIdx.x;
    const int pl = tid >> 4, j = tid & 15;
    // 32-bit index arithmetic throughout (the launcher checks total < 2^31; a third of this issue-bound kernel's
    // instructions were 64-bit address / division sequences); a neighbour index is < n_per_batch, so the low word
    // of an int64 entry is the whole value
    const unsigned total = (unsigned)p.total, npb = (unsigned)p.n_per_batch;
    const unsigned ngrp = (unsigned)num_groups, gstride = gridDim.x;
    const int* nidx32 = reinterpret_cast<const int*>(p.nidx);
    const int ishift = p.nidx_is64 ? 1 : 0;
    // (base, raw) of the group whose neighbour index is in flight
    int raw_a = 0;
    unsigned base_a = 0;
    bool ok_a = false;
    auto request_index = [&](unsigned grp_) {
        const unsigned g_ = grp_ * L16_PTS + pl;
        ok_a = grp_ < ngrp && g_ < total;
        if (ok_a) {
            base_a = g_ - g_ % npb;
            raw_a = nidx32[((size_t)g_ * LFA_K + j) << ishift];   // stays a raw loaded word until its group comes up
        }
    };
    request_index(blockIdx.x);
    for (unsigned grp = blockIdx.x; grp < ngrp; grp += gstride) {
        const unsigned g = grp * L16_PTS + pl;
        float x[D];
#pragma unroll
        for (int c = 0; c < D; ++c) x[c] = 0.f;
        int gn = -1;
        float4 f0 = make_float4(0.f, 0.f, 0.f, 0.f), f1 = f0;
        float qx = 0.f, qy = 0.f, qz = 0.f, cx = 0.f, cy = 0.f, cz = 0.f;
        if (g < total) {
            gn = (int)(base_a + (unsigned)raw_a);
            const float* fr = p.feat + (size_t)(unsigned)gn * H;
            f0 = *reinterpret_cast<const float4*>(fr);
            f1 = *reinterpret_cast<const float4*>(fr + 4);
            const float* cq = p.coords + (size_t)g * 3;
            const float* cn = p.coords + (size_t)(unsigned)gn * 3;
            qx = cq[0]; qy = cq[1]; qz = cq[2];
            cx = cn[0]; cy = cn[1]; cz = cn[2];
        }
        request_index(grp + gstride);
        if (gn >= 0) {
            const float dx = qx - cx, dy = qy - cy, dz = qz - cz;
            float e[10];
            e[0] = sqrtf(__fadd_rn(__fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy)), __fmul_rn(dz, dz)));
            e[1] = dx; e[2] = dy; e[3] = dz;
            e[4] = qx; e[5] = qy; e[6] = qz;
            e[7] = cx; e[8] = cy; e[9] = cz;
            x[0] = f0.x; x[1] = f0.y; x[2] = f0.z; x[3] = f0.w;
            x[4] = f1.x; x[5] = f1.y; x[6] = f1.z; x[7] = f1.w;
            float r1[H];
#pragma unroll
            for (int o = 0; o < H; ++o) r1[o] = 0.f;
#pragma unroll
            for (int q = 0; q < 10; ++q)      // weight rows are consumed contiguously -> LDCU.128
#pragma unroll
                for (int o = 0; o < H; o += 2)
                    ffma2(r1[o], r1[o + 1], e[q], w.v[W16_W10 + q * H + o], w.v[W16_W10 + q * H + o + 1]);
#pragma unroll
            for (int o = 0; o < H; ++o) {
                const float a = fmaf(r1[o], w.v[W16_S10 + o], w.v[W16_T10 + o]);
                r1[o] = a >= 0.f ? a : 0.2f * a;
            }
            if (STAGE == 1) {
#pragma unroll
                for (int o = 0; o < H; ++o) x[H + o] = r1[o];
            } else {
                float r2[H];
#pragma unroll
                for (int o = 0; o < H; ++o) r2[o] = 0.f;
#pragma unroll
                for (int k = 0; k < H; ++k)
#pragma unroll
                    for (int o = 0; o < H; o += 2)
                        ffma2(r2[o], r2[o + 1], r1[k], w.v[W16_WL2 + k * H + o], w.v[W16_WL2 + k * H + o + 1]);
#pragma unroll
                for (int o = 0; o < H; ++o) {
                    const float a = fmaf(r2[o], w.v[W16_S2 + o], w.v[W16_T2 + o]);
                    x[H + o] = a >= 0.f ? a : 0.2f * a;
                }
            }
        }
        float sc[D];
#pragma unroll
        for (int c = 0; c < D; ++c) sc[c] = w.v[W16_BS + c];
#pragma unroll
        for (int k = 0; k < D; ++k)
#pragma unroll
            for (int c = 0; c < D; c += 2)
                ffma2(sc[c], sc[c + 1], x[k], w.v[W16_WS + k * D + c], w.v[W16_WS + k * D + c + 1]);
#pragma unroll
        for (int c = 0; c < D; ++c) {
            St[c * L16_RS + tid] = sc[c];
            Xs[c * L16_RS + tid] = x[c];
        }
        __syncthreads();
        {
            const float* srow = St + j * L16_RS + pl * LFA_K;
            const float* xrow = Xs + j * L16_RS + pl * LFA_K;
            float4 s4[4];
#pragma unroll
            for (int q = 0; q < 4; ++q) s4[q] = *reinterpret_cast<const float4*>(srow + 4 * q);
            float m = s4[0].x;
#pragma unroll
            for (int q = 0; q < 4; ++q) m = fmaxf(fmaxf(fmaxf(m, s4[q].x), s4[q].y), fmaxf(s4[q].z, s4[q].w));
            float num = 0.f, den = 0.f;
            const float ml = -m * kLog2e;
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                const float4 xv = *reinterpret_cast<const float4*>(xrow + 4 * q);
                // exp(s - m) = 2^(s * log2e - m * log2e): FFMA + MUFU per weight instead of the ~8 instructions of
                // expf (the weights are normalised right below; the tensor-core kernels do the same)
                const float e0 = ex2_ftz(fmaf(s4[q].x, kLog2e, ml)), e1 = ex2_ftz(fmaf(s4[q].y, kLog2e, ml));
                const float e2 = ex2_ftz(fmaf(s4[q].z, kLog2e, ml)), e3 = ex2_ftz(fmaf(s4[q].w, kLog2e, ml));
                den += (e0 + e1) + (e2 + e3);
                num = fmaf(e0, xv.x, num);
                num = fmaf(e1, xv.y, num);
                num = fmaf(e2, xv.z, num);
                num = fmaf(e3, xv.w, num);
            }
            if (g < total) p.agg[(size_t)g * D + j] = num / den;
        }
        __syncthreads();
    }
}

template <int STAGE>
static int lfa16c_launch(const LfaParams& p, const Lfa16W& w, cudaStream_t st) {
    const int64_t groups = ceil_div<int64_t>(p.total, L16_PTS);
    const int64_t cap = (int64_t)device_sm_count() * L16C_CTAS;
    const unsigned blocks = (unsigned)(groups < cap ? groups : cap);
    lfa16c_kernel<STAGE><<<blocks, L16_ROWS, 0, st>>>(p, w, groups);
    O3DML_LAUNCH_CHECK();
    o3dml_count_launches(1);
    return O3DML_OK;
}

}  // namespace o3dml

using namespace o3dml;

extern "C" int o3dml_randla_lfa_pool(int stage, int d, const float* coords, const void* neighbor_idx,
                                     int idx_is64, int num_neighbors, const float* feat,
                                     int64_t batch, int64_t n_per_batch, const float* w10_t,
                                     const float* s10, const float* t10, const float* wl2_t,
                                     const float* s2, const float* t2, const float* wscore_t,
                                     const float* bscore, float* agg, void* stream) {
    O3DML_CHECK(stage == 1 || stage == 2, "lfa: stage must be 1 or 2");
    O3DML_CHECK(num_neighbors == LFA_K, "lfa: the fused kernel is built for 16 neighbours");
    O3DML_CHECK(batch * n_per_batch < ((int64_t)1 << 31), "lfa: too many points");
    LfaParams p;
    p.coords = coords;
    p.nidx = neighbor_idx;
    p.nidx_is64 = idx_is64;
    p.feat = feat;
    p.total = batch * n_per_batch;
    p.n_per_batch = n_per_batch;
    p.w10t = w10_t; p.s10 = s10; p.t10 = t10;
    p.wl2t = wl2_t; p.s2 = s2; p.t2 = t2;
    p.wst = wscore_t; p.bs = bscore;
    p.agg = agg;
    if (p.total == 0) return O3DML_OK;
    O3DML_CHECK(stage == 1 || (wl2_t && s2 && t2), "lfa: stage 2 needs the lse2 weights");
    cudaStream_t st = (cudaStream_t)stream;
#define LFA_CASE(DD)                                                              \
    case DD:                                                                      \
        return stage == 1 ? lfa_launch<DD, 1>(p, st) : lfa_launch<DD, 2>(p, st);
    switch (d) {
        LFA_CASE(16)
        LFA_CASE(32)
        LFA_CASE(64)
        LFA_CASE(128)
        LFA_CASE(256)
        LFA_CASE(512)   // the 5-level configs (s3dis / semantic3d / toronto3d / parislille3d: dim_output [16,64,128,256,512])
        default:
            O3DML_FAIL(O3DML_ERR_UNSUPPORTED, "lfa: d_out %d not in {16,32,64,128,256,512}", d);
    }
#undef LFA_CASE
}

extern "C" int o3dml_randla_lfa16_pool(int stage, const float* coords, const void* neighbor_idx, int idx_is64,
                                       int num_neighbors, const float* feat, int64_t batch,
                                       int64_t n_per_batch, const float* h_weights, float* agg,
                                       void* stream) {
    O3DML_CHECK(stage == 1 || stage == 2, "lfa16: stage must be 1 or 2");
    O3DML_CHECK(num_neighbors == LFA_K, "lfa16: the fused kernel is built for 16 neighbours");
    O3DML_CHECK(batch * n_per_batch < ((int64_t)1 << 31), "lfa16: too many points");
    O3DML_CHECK(h_weights != nullptr, "lfa16: h_weights is null");
    cudaPointerAttributes attr;
    if (cudaPointerGetAttributes(&attr, h_weights) == cudaSuccess)
        O3DML_CHECK(attr.type != cudaMemoryTypeDevice, "lfa16: h_weights must point to HOST memory");
    else
        cudaGetLastError();
    LfaParams p;
    p.coords = coords; p.nidx = neighbor_idx; p.nidx_is64 = idx_is64; p.feat = feat;
    p.total = batch * n_per_batch; p.n_per_batch = n_per_batch;
    p.w10t = p.s10 = p.t10 = p.wl2t = p.s2 = p.t2 = p.wst = p.bs = nullptr;
    p.agg = agg;
    if (p.total == 0) return O3DML_OK;
    Lfa16W w;
    memcpy(w.v, h_weights, sizeof(w.v));
    cudaStream_t st = (cudaStream_t)stream;
    return stage == 1 ? lfa16c_launch<1>(p, w, st) : lfa16c_launch<2>(p, w, st);
}

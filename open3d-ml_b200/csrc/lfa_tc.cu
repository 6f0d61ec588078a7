// lfa_tc.cu -- RandLA-Net attentive-pooling stage on the 5th-gen tensor cores (tcgen05):
//   neighbour gather -> LocSE encoding (+ shared MLPs) -> score GEMM on tcgen05 with the
//   3xFP16 split (tc.cuh) -> softmax over the 16 neighbours -> weighted sum  ==> agg [N, d]
// Same contract as lfa_pool_kernel (lfa.cu); replaces randlanet.py:521-639 as used at :667-692.
//
// One MMA tile = 128 neighbour rows = 8 points x 16 neighbours:
//   A  [128 x d]  : X = [feat[nbr] | r1 or r2], built by the CTA in shared memory directly in the
//                   UMMA chunk-major layout (one conflict-free 16-byte store per (row, 8 channels)),
//                   as fp16 hi/lo pairs.  In stage 2 the first half of A first holds r1 (the A
//                   operand of the lse2 GEMM) and is then overwritten by the gathered features.
//   B  [d x d]    : score weight, host-packed hi/lo operand image; resident in shared memory for
//                   d <= 128, streamed through a 2-slot ring of 32-channel slices for d = 256
//   D  [128 x d]  : fp32 in TMEM, lane = neighbour row, column = score channel
// Epilogue: thread = one neighbour row (TMEM lane); softmax over the 16 rows of a point is a
// half-warp reduction (redux.sync max on order-preserving ints, reduce-scatter shuffles for the
// two sums), after which lane j of the half-warp owns output channel c0+j -> coalesced stores.
// Stage 2 chains a second MMA (r2 = lrelu(BN(Wl2 . r1)), N = d/2) through TMEM back into A
// (d = 16: that 8x8 product stays in registers).  The score bias is not applied: it is constant
// over the neighbours of a point and cancels in the softmax.  CTAs are persistent over tiles.
#include "../../include/o3dml_b200.h"
#include "common.cuh"
#include "tc.cuh"
#include <limits.h>

namespace o3dml {

constexpr int LTC_ROWS = 128;  // MMA M
constexpr int LTC_K = 16;      // neighbours
constexpr int LTC_SLICE = 32;  // channels per streamed weight slice

struct LfaTcParams {
    const float* coords;
    const void* nidx;
    int nidx_is64;
    const float* feat;     // [B*N, D/2]
    int64_t total, n_per_batch;
    const float* w10t;     // [10][D/2]
    const float* s10;
    const float* t10;
    const uint4* wl2_img;  // stage 2, d >= 32: [hi | lo] operand images of Wl2 [N=D/2][K=D/2]
    const float* wl2t;     // stage 2, d == 16: fp32 [in][out]
    const float* s2;
    const float* t2;
    const uint4* ws_img;   // [hi | lo] operand images of the score weight [N=D][K=D]
    float* agg;            // [B*N, D]
    int64_t num_tiles;
};

template <int D, int STAGE>
struct LtcCfg {
    static constexpr int H = D / 2;
    static constexpr bool STREAM = D > 128;          // weights do not fit next to the A tile
    static constexpr bool MMA2 = STAGE == 2 && H >= 16;  // lse2 on the tensor core
    // TRANS: the score GEMM runs transposed (M = score channel, N = neighbour row) and a second,
    // identity-weight GEMM delivers X^T the same way, so that one thread sees the 16 neighbours
    // of a (point, channel) in its own TMEM lane: the softmax needs no cross-lane traffic.
    static constexpr bool TRANS = !STREAM && D >= 64;
    static constexpr int NTH = (TRANS && D == 128) ? 512 : 256;   // threads per CTA
    static constexpr int NPART = NTH / LTC_ROWS;                  // threads sharing one row
    static constexpr int MINB = (TRANS && D == 64) ? 2 : 1;       // two CTAs per SM must fit the register file
    static constexpr int A_BYTES = D / 8 * LTC_ROWS * 16;  // one of hi / lo
    static constexpr int B_BYTES = STREAM ? 0 : TRANS ? D / 8 * LTC_ROWS * 16 : D / 8 * D * 16;
    static constexpr int I_BYTES = TRANS ? D / 8 * LTC_ROWS * 16 : 0;   // identity operand (hi only)
    static constexpr int B2_BYTES = (MMA2 && !STREAM) ? H / 8 * H * 16 : 0;
    static constexpr int RING_SLOT = STREAM ? 2 * (LTC_SLICE / 8) * D * 16 : 0;  // hi + lo of one slice
    static constexpr int W10_BYTES = 12 * H * 4;
    static constexpr int ST2_BYTES = STAGE == 2 ? (2 * H + (H < 16 ? H * H : 0)) * 4 : 0;
    static constexpr int TMEM_NEED = TRANS ? 256 : D + (MMA2 ? H : 0);
    static constexpr int TMEM_COLS = TMEM_NEED <= 32 ? 32 : TMEM_NEED <= 64 ? 64 : TMEM_NEED <= 128 ? 128
                                     : TMEM_NEED <= 256 ? 256 : 512;
    static constexpr size_t SMEM = 2 * A_BYTES + 2 * B_BYTES + I_BYTES + 2 * B2_BYTES + 2 * RING_SLOT +
                                   W10_BYTES + ST2_BYTES + 128;
};

// D[tmem_d] = A[128 x K] * B[N x K]^T, all operands resident in shared memory; one thread.
template <int N, int K>
__device__ __forceinline__ void issue_resident(uint32_t tmem_d, const uint8_t* a_hi, const uint8_t* a_lo,
                                               const uint8_t* b_hi, const uint8_t* b_lo) {
    constexpr uint32_t idesc = tc::idesc_f16(LTC_ROWS, N);
    constexpr uint32_t A_LBO = LTC_ROWS * 16, B_LBO = N * 16;
#pragma unroll
    for (int ks = 0; ks < K / 16; ++ks) {
        const uint64_t ah = tc::smem_desc(tc::smem_u32(a_hi) + ks * 2 * A_LBO, A_LBO, 128);
        const uint64_t al = tc::smem_desc(tc::smem_u32(a_lo) + ks * 2 * A_LBO, A_LBO, 128);
        const uint64_t bh = tc::smem_desc(tc::smem_u32(b_hi) + ks * 2 * B_LBO, B_LBO, 128);
        const uint64_t bl = tc::smem_desc(tc::smem_u32(b_lo) + ks * 2 * B_LBO, B_LBO, 128);
        tc::umma_f16(tmem_d, ah, bh, idesc, ks > 0);
        tc::umma_f16(tmem_d, ah, bl, idesc, 1);
        tc::umma_f16(tmem_d, al, bh, idesc, 1);
    }
}

// D[tmem_d][c][row] = X[row][c]: A = identity (128 x K, exact in fp16), B = the X tile (hi + lo).
template <int K>
__device__ __forceinline__ void issue_identity(uint32_t tmem_d, const uint8_t* i_hi, const uint8_t* x_hi,
                                               const uint8_t* x_lo) {
    constexpr uint32_t idesc = tc::idesc_f16(LTC_ROWS, LTC_ROWS);
    constexpr uint32_t LBO = LTC_ROWS * 16;
#pragma unroll
    for (int ks = 0; ks < K / 16; ++ks) {
        const uint64_t ih = tc::smem_desc(tc::smem_u32(i_hi) + ks * 2 * LBO, LBO, 128);
        const uint64_t xh = tc::smem_desc(tc::smem_u32(x_hi) + ks * 2 * LBO, LBO, 128);
        const uint64_t xl = tc::smem_desc(tc::smem_u32(x_lo) + ks * 2 * LBO, LBO, 128);
        tc::umma_f16(tmem_d, ih, xh, idesc, ks > 0);
        tc::umma_f16(tmem_d, ih, xl, idesc, 1);
    }
}

// Same product with B streamed from global memory (host-packed images) through a 2-slot ring of 32-channel
// slices.  ONE thread runs the whole stream: it hands each slice (hi + lo: two contiguous blocks of the image)
// to the bulk-copy engine (cp.async.bulk, bytes counted on full[slot]), waits for it, issues the slice's MMAs and
// commits them to free[slot] (ring reuse) -- the copy of slice s+1 overlaps the MMAs of slice s.  Everybody else
// only waits for `done` (the commit after the last slice).  Round 1 copied every slice with all 256 threads
// through registers (LDG -> STS, 256 KB per tile at d = 256) with a __syncthreads per slice: 14 % tensor-pipe
// activity, long-scoreboard stalls (profiles/r02_lfa_ncu_full.md).
// mb[0..1] = full, mb[2..3] = free, mb[4] = done; ph[] = this thread's wait parities of the five barriers.
template <int N, int K>
__device__ __forceinline__ void gemm_streamed(uint32_t tmem_d, const uint8_t* a_hi, const uint8_t* a_lo,
                                              const uint4* __restrict__ img, uint8_t* ring, int slot_bytes,
                                              uint64_t* mb, uint32_t* ph, int tid) {
    constexpr uint32_t idesc = tc::idesc_f16(LTC_ROWS, N);
    constexpr uint32_t A_LBO = LTC_ROWS * 16, B_LBO = N * 16;
    constexpr int CH = LTC_SLICE / 8;                 // 16-byte k-chunks per slice
    constexpr int SL_U4 = CH * N;                     // uint4 per slice per image
    constexpr int IMG_U4 = K / 8 * N;                 // uint4 per image (hi, then lo)
    constexpr int NSL = K / LTC_SLICE;
    constexpr uint32_t SL_BYTES = SL_U4 * 16;
    if (tid == 0) {
        auto copy_slice = [&](int s) {
            const int slot = s & 1;
            uint8_t* dst = ring + (size_t)slot * slot_bytes;
            tc::mbar_arrive_expect_tx(&mb[slot], 2 * SL_BYTES);
            tc::bulk_copy_g2s(dst, img + (size_t)s * SL_U4, SL_BYTES, &mb[slot]);
            tc::bulk_copy_g2s(dst + SL_BYTES, img + IMG_U4 + (size_t)s * SL_U4, SL_BYTES, &mb[slot]);
        };
        copy_slice(0);
        for (int s = 0; s < NSL; ++s) {
            const int slot = s & 1;
            if (s + 1 < NSL) {
                if (s >= 1) {     // slot (s+1)&1 was read by slice s-1: wait until those MMAs are done
                    tc::mbar_wait(&mb[2 + ((s + 1) & 1)], ph[2 + ((s + 1) & 1)]);
                    ph[2 + ((s + 1) & 1)] ^= 1;
                }
                copy_slice(s + 1);
            }
            tc::mbar_wait(&mb[slot], ph[slot]);
            ph[slot] ^= 1;
            const uint8_t* b_hi = ring + (size_t)slot * slot_bytes;
            const uint8_t* b_lo = b_hi + SL_BYTES;
#pragma unroll
            for (int ks = 0; ks < LTC_SLICE / 16; ++ks) {
                const int kc = s * CH + ks * 2;  // first k-chunk of this k-step in A
                const uint64_t ah = tc::smem_desc(tc::smem_u32(a_hi) + kc * A_LBO, A_LBO, 128);
                const uint64_t al = tc::smem_desc(tc::smem_u32(a_lo) + kc * A_LBO, A_LBO, 128);
                const uint64_t bh = tc::smem_desc(tc::smem_u32(b_hi) + ks * 2 * B_LBO, B_LBO, 128);
                const uint64_t bl = tc::smem_desc(tc::smem_u32(b_lo) + ks * 2 * B_LBO, B_LBO, 128);
                tc::umma_f16(tmem_d, ah, bh, idesc, (s | ks) > 0);
                tc::umma_f16(tmem_d, ah, bl, idesc, 1);
                tc::umma_f16(tmem_d, al, bh, idesc, 1);
            }
            tc::umma_commit(&mb[2 + slot]);
        }
        tc::umma_commit(&mb[4]);
        // the free[] commits of the last two slices are not waited for inside the loop: consume them here so
        // that the parities are in step for the next call (they complete no later than `done`)
        if (NSL >= 2) {
            tc::mbar_wait(&mb[2 + ((NSL - 2) & 1)], ph[2 + ((NSL - 2) & 1)]);
            ph[2 + ((NSL - 2) & 1)] ^= 1;
        }
        tc::mbar_wait(&mb[2 + ((NSL - 1) & 1)], ph[2 + ((NSL - 1) & 1)]);
        ph[2 + ((NSL - 1) & 1)] ^= 1;
    }
    tc::mbar_wait(&mb[4], ph[4]);
    ph[4] ^= 1;
    tc::tc_fence_after();
}

template <int D, int STAGE>
__global__ void __launch_bounds__((LtcCfg<D, STAGE>::NTH), (LtcCfg<D, STAGE>::MINB))
lfa_pool_tc_kernel(const __grid_constant__ LfaTcParams p) {
    using C = LtcCfg<D, STAGE>;
    constexpr int H = C::H, NTH = C::NTH, NPART = C::NPART;
    extern __shared__ __align__(128) uint8_t smem[];
    uint8_t* a_hi = smem;
    uint8_t* a_lo = a_hi + C::A_BYTES;
    uint8_t* b_hi = a_lo + C::A_BYTES;
    uint8_t* b_lo = b_hi + C::B_BYTES;
    uint8_t* i_hi = b_lo + C::B_BYTES;
    uint8_t* b2_hi = i_hi + C::I_BYTES;
    uint8_t* b2_lo = b2_hi + C::B2_BYTES;
    uint8_t* ring = b2_lo + C::B2_BYTES;
    float* W10 = reinterpret_cast<float*>(ring + 2 * C::RING_SLOT);  // [12][H]
    float* ST2 = W10 + 12 * H;                                       // [2][H] (+ Wl2^T [H][H] for H < 16)
    uint64_t* mbar = reinterpret_cast<uint64_t*>(reinterpret_cast<uint8_t*>(ST2) + C::ST2_BYTES);
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(mbar + 8);

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int row = tid & (LTC_ROWS - 1);   // neighbour row of the tile this thread works on
    const int half = tid >> 7;              // which part of the channels / columns (0 .. NPART-1)

    // ---- once per CTA: weights, barriers, TMEM
    if (C::TRANS) {
        // score weight as the M operand: 128 rows (d = 64: the 64 channels twice, so that TMEM lanes
        // 64..127 serve the second half of the tile's points); source image is [D/8][D][8] hi, lo
        constexpr int CH = D / 8;
        for (int i = tid; i < 2 * CH * LTC_ROWS; i += NTH) {
            const int im = i / (CH * LTC_ROWS), rem = i % (CH * LTC_ROWS);
            const int kc = rem / LTC_ROWS, r = rem % LTC_ROWS;
            reinterpret_cast<uint4*>(b_hi)[i] = p.ws_img[(size_t)im * CH * D + kc * D + (r % D)];
        }
        for (int i = tid; i < CH * LTC_ROWS; i += NTH) {
            const int kc = i / LTC_ROWS, r = i % LTC_ROWS;
            const int j = (r % D) - kc * 8;        // position of the one inside this 8-wide chunk
            uint4 v = make_uint4(0u, 0u, 0u, 0u);
            if (j >= 0 && j < 8) {
                const uint32_t one = 0x3C00u << ((j & 1) * 16);
                if ((j >> 1) == 0) v.x = one;
                else if ((j >> 1) == 1) v.y = one;
                else if ((j >> 1) == 2) v.z = one;
                else v.w = one;
            }
            reinterpret_cast<uint4*>(i_hi)[i] = v;
        }
        if (C::MMA2)
            for (int i = tid; i < 2 * C::B2_BYTES / 16; i += NTH)
                reinterpret_cast<uint4*>(b2_hi)[i] = p.wl2_img[i];
    } else if (!C::STREAM) {
        for (int i = tid; i < 2 * C::B_BYTES / 16; i += NTH)
            reinterpret_cast<uint4*>(b_hi)[i] = p.ws_img[i];
        if (C::MMA2)
            for (int i = tid; i < 2 * C::B2_BYTES / 16; i += NTH)
                reinterpret_cast<uint4*>(b2_hi)[i] = p.wl2_img[i];
    }
    if (STAGE == 2) {
        for (int i = tid; i < H; i += NTH) {
            ST2[i] = p.s2[i];
            ST2[H + i] = p.t2[i];
        }
        if (H < 16)
            for (int i = tid; i < H * H; i += NTH) ST2[2 * H + i] = p.wl2t[i];
    }
    for (int i = tid; i < 10 * H; i += NTH) W10[i] = p.w10t[i];
    for (int i = tid; i < H; i += NTH) {
        W10[10 * H + i] = p.s10[i];
        W10[11 * H + i] = p.t10[i];
    }
    if (tid == 0) {
#pragma unroll
        for (int i = 0; i < 8; ++i) tc::mbar_init(&mbar[i], 1);
        tc::fence_mbar_init();
    }
    tc::fence_async_smem();
    __syncthreads();
    if (warp == 0) tc::tmem_alloc<C::TMEM_COLS>(tmem_slot);
    tc::tc_fence_before();
    __syncthreads();
    tc::tc_fence_after();
    const uint32_t tmem = *tmem_slot;
    const uint32_t tmem_lane = tmem + ((uint32_t)((warp & 3) * 32) << 16);
    // TRANS: the lse2 accumulator aliases the score columns (it is consumed before they are written)
    constexpr int LSE2_COL = C::TRANS ? 0 : D;
    uint32_t ph_main[2] = {0, 0};  // parities of mbar[0] (lse2) and mbar[1] (scores)
    uint32_t ph_ring[5] = {0, 0, 0, 0, 0};  // parities of mbar[2..6]: weight ring full / free and `done` (gemm_streamed)

    // The gathers are software-pipelined over tiles (d >= 64): the neighbour index of tile t+2 and the
    // coordinates / feature rows of tile t+1 are requested while tile t is worked on and land behind its
    // MMAs and epilogue (two dependent global round trips leave the per-tile critical path).  d = 256 holds 64
    // feature registers per tile: there the requests for tile t+1 go out after the rows of tile t have been stored
    // (LATE) and the index stays a raw loaded word until its tile comes up (RAW_INDEX, common.cuh RawIndex).  The
    // resident-weight kernels resolve the index of tile t+2 right behind its load: every warp of the CTA waits there
    // for one L2 round trip, 13-19 % of the stall samples (profiles/r02_lfa_stalls.md) -- and taking that wait away
    // made d = 64 SLOWER (2 x 188.6 / 217.3 us against 173.7 / 195.6 us per launch, same build otherwise; d = 128 equal):
    // with two CTAs per SM the wait is where the other CTA gets the issue slots and the shared-memory port.
    constexpr bool PREF = D >= 64;
    constexpr bool LATE = C::STREAM;
    constexpr bool RAW_INDEX = C::STREAM;
    constexpr int FCH = PREF ? (H / 8) / NPART : 1;      // feature chunks (8 channels) per thread
    int64_t g_nx = p.total, nb_nx = -1, g_n2 = p.total, base_n2 = -1;
    RawIndex raw_n2 = {0, 0};
    float qc_nx[6] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
    float4 f_nx[FCH][2];
    auto load_idx = [&](int64_t t, int64_t& g_, int64_t& base_, RawIndex& raw_) {
        g_ = p.total;
        base_ = -1;
        if (t < p.num_tiles) {
            g_ = t * (LTC_ROWS / LTC_K) + (row >> 4);
            if (g_ < p.total) {
                base_ = (g_ / p.n_per_batch) * p.n_per_batch;
                if (RAW_INDEX) load_index_raw(p.nidx, g_ * LTC_K + (row & 15), p.nidx_is64, raw_);
                else base_ += load_index(p.nidx, g_ * LTC_K + (row & 15), p.nidx_is64);
            }
        }
    };
    auto resolve = [&](int64_t base_, const RawIndex& raw_) -> int64_t {
        if (!RAW_INDEX) return base_;
        return base_ >= 0 ? base_ + index_value(raw_, p.nidx_is64) : (int64_t)-1;
    };
    auto load_data = [&](int64_t g_, int64_t nb_, float* qc, float4 (*f)[2]) {
        if (nb_ >= 0) {
            qc[0] = p.coords[3 * g_]; qc[1] = p.coords[3 * g_ + 1]; qc[2] = p.coords[3 * g_ + 2];
            qc[3] = p.coords[3 * nb_]; qc[4] = p.coords[3 * nb_ + 1]; qc[5] = p.coords[3 * nb_ + 2];
#pragma unroll
            for (int i = 0; i < FCH; ++i) {
                const float* src = p.feat + (size_t)nb_ * H + (half + i * NPART) * 8;
                f[i][0] = *reinterpret_cast<const float4*>(src);
                f[i][1] = *reinterpret_cast<const float4*>(src + 4);
            }
        } else {
#pragma unroll
            for (int i = 0; i < 6; ++i) qc[i] = 0.f;
#pragma unroll
            for (int i = 0; i < FCH; ++i) f[i][0] = f[i][1] = make_float4(0.f, 0.f, 0.f, 0.f);
        }
    };
    // requests for the tile after `tile` (index resolved now, one tile after its load) and the index of the one after
    auto advance = [&](int64_t tile) {
        g_nx = g_n2;
        nb_nx = resolve(base_n2, raw_n2);
        load_data(g_nx, nb_nx, qc_nx, f_nx);
        load_idx(tile + 2 * (int64_t)gridDim.x, g_n2, base_n2, raw_n2);
    };
    if (PREF) {
        load_idx(blockIdx.x, g_nx, base_n2, raw_n2);
        nb_nx = resolve(base_n2, raw_n2);
        load_data(g_nx, nb_nx, qc_nx, f_nx);
        load_idx((int64_t)blockIdx.x + gridDim.x, g_n2, base_n2, raw_n2);
    }

    // 10-channel relative position encoding of this thread's row (randlanet.py:586-600)
    auto encode = [&](int64_t nb_, const float* qc, float* e) {
#pragma unroll
        for (int q = 0; q < 10; ++q) e[q] = 0.f;
        if (nb_ >= 0) {
            const float dx = qc[0] - qc[3], dy = qc[1] - qc[4], dz = qc[2] - qc[5];
            e[0] = sqrtf(__fadd_rn(__fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy)), __fmul_rn(dz, dz)));
            e[1] = dx; e[2] = dy; e[3] = dz;
            e[4] = qc[0]; e[5] = qc[1]; e[6] = qc[2];
            e[7] = qc[3]; e[8] = qc[4]; e[9] = qc[5];
        }
    };
    // r1 = lrelu(BN(W10 . enc)), 8 outputs at a time, straight into an operand region of H channels (chunk-major,
    // chunk `ch` of the region at dst + ch * LTC_ROWS * 16):
    //   stage 1            -> channels [H, D) of A
    //   stage 2, tensor    -> channels [0, H) of A, the A operand of the lse2 GEMM
    //   stage 2, H < 16    -> r2 = lrelu(BN(Wl2 . r1)) in registers -> channels [H, D)
    auto locse = [&](const float* e, uint8_t* dst_hi, uint8_t* dst_lo) {
        for (int ch = half; ch < H / 8; ch += NPART) {
            float r[8];
#pragma unroll
            for (int j = 0; j < 8; ++j) r[j] = 0.f;
#pragma unroll
            for (int q = 0; q < 10; ++q) {   // warp-uniform LDS.128 of the weights
                const float4 wa = *reinterpret_cast<const float4*>(&W10[q * H + ch * 8]);
                const float4 wb = *reinterpret_cast<const float4*>(&W10[q * H + ch * 8 + 4]);
                ffma2(r[0], r[1], e[q], wa.x, wa.y);   // packed FFMA2: half the FMA instructions of the LocSE MLP
                ffma2(r[2], r[3], e[q], wa.z, wa.w);
                ffma2(r[4], r[5], e[q], wb.x, wb.y);
                ffma2(r[6], r[7], e[q], wb.z, wb.w);
            }
            {   // folded BN + LeakyReLU; scale / shift as four LDS.128
                const float4 sa = *reinterpret_cast<const float4*>(&W10[10 * H + ch * 8]);
                const float4 sb = *reinterpret_cast<const float4*>(&W10[10 * H + ch * 8 + 4]);
                const float4 ta = *reinterpret_cast<const float4*>(&W10[11 * H + ch * 8]);
                const float4 tb = *reinterpret_cast<const float4*>(&W10[11 * H + ch * 8 + 4]);
                const float sc[8] = {sa.x, sa.y, sa.z, sa.w, sb.x, sb.y, sb.z, sb.w};
                const float sh[8] = {ta.x, ta.y, ta.z, ta.w, tb.x, tb.y, tb.z, tb.w};
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                    const float a = fmaf(r[j], sc[j], sh[j]);
                    r[j] = a >= 0.f ? a : 0.2f * a;
                }
            }
            if (STAGE == 2 && !C::MMA2) {  // H == 8: one chunk holds all of r1
                float r2[8];
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                    float a = 0.f;
#pragma unroll
                    for (int i = 0; i < 8; ++i) a = fmaf(r[i], ST2[2 * H + i * H + j], a);
                    a = fmaf(a, ST2[j], ST2[H + j]);
                    r2[j] = a >= 0.f ? a : 0.2f * a;
                }
#pragma unroll
                for (int j = 0; j < 8; ++j) r[j] = r2[j];
            }
            uint4 hi, lo;
            tc::split8(r, hi, lo);
            *reinterpret_cast<uint4*>(dst_hi + tc::op_off(LTC_ROWS, row, ch)) = hi;
            *reinterpret_cast<uint4*>(dst_lo + tc::op_off(LTC_ROWS, row, ch)) = lo;
        }
    };
    // r1 goes to channels [0, H) when the tensor core computes lse2 from it, else (r1 of stage 1, r2 of the d = 16
    // register path) to channels [H, D)
    constexpr uint32_t R1_OFF = (STAGE == 2 && C::MMA2) ? 0u : (uint32_t)(H / 8) * LTC_ROWS * 16;

    for (int64_t tile = blockIdx.x; tile < p.num_tiles; tile += gridDim.x) {
        // ---------------- neighbour id + encoding + LocSE MLP of this thread's row
        int64_t g = tile * (LTC_ROWS / LTC_K) + (row >> 4);
        int64_t nb = -1;
        float4 f_cur[FCH][2];
        if (PREF) {
            g = g_nx;
            nb = nb_nx;
            float qc[6];
#pragma unroll
            for (int i = 0; i < 6; ++i) qc[i] = qc_nx[i];
#pragma unroll
            for (int i = 0; i < FCH; ++i) { f_cur[i][0] = f_nx[i][0]; f_cur[i][1] = f_nx[i][1]; }
            if (!LATE) advance(tile);        // tile t+1: data in flight from here; tile t+2: index
            float e[10];
            encode(nb, qc, e);
            locse(e, a_hi + R1_OFF, a_lo + R1_OFF);
        } else {
            float qc[6] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
            if (g < p.total) {
                const int64_t b = g / p.n_per_batch;
                nb = b * p.n_per_batch + load_index(p.nidx, g * LTC_K + (row & 15), p.nidx_is64);
                qc[0] = p.coords[3 * g]; qc[1] = p.coords[3 * g + 1]; qc[2] = p.coords[3 * g + 2];
                qc[3] = p.coords[3 * nb]; qc[4] = p.coords[3 * nb + 1]; qc[5] = p.coords[3 * nb + 2];
            }
            float e[10];
            encode(nb, qc, e);
            locse(e, a_hi + R1_OFF, a_lo + R1_OFF);
        }
        // gathered neighbour features -> channels [0, H) of A
        auto store_features = [&]() {
#pragma unroll
            for (int ch = half, fi = 0; ch < H / 8; ch += NPART, ++fi) {
                float x[8];
                if (PREF) {
                    const float4 v0 = f_cur[fi < FCH ? fi : 0][0], v1 = f_cur[fi < FCH ? fi : 0][1];
                    x[0] = v0.x; x[1] = v0.y; x[2] = v0.z; x[3] = v0.w;
                    x[4] = v1.x; x[5] = v1.y; x[6] = v1.z; x[7] = v1.w;
                } else if (nb >= 0) {
                    const float4 v0 = *reinterpret_cast<const float4*>(p.feat + (size_t)nb * H + ch * 8);
                    const float4 v1 = *reinterpret_cast<const float4*>(p.feat + (size_t)nb * H + ch * 8 + 4);
                    x[0] = v0.x; x[1] = v0.y; x[2] = v0.z; x[3] = v0.w;
                    x[4] = v1.x; x[5] = v1.y; x[6] = v1.z; x[7] = v1.w;
                } else {
#pragma unroll
                    for (int j = 0; j < 8; ++j) x[j] = 0.f;
                }
                uint4 hi, lo;
                tc::split8(x, hi, lo);
                *reinterpret_cast<uint4*>(a_hi + tc::op_off(LTC_ROWS, row, ch)) = hi;
                *reinterpret_cast<uint4*>(a_lo + tc::op_off(LTC_ROWS, row, ch)) = lo;
            }
        };

        // ---------------- stage 2: r2 = lrelu(BN(Wl2 . r1)) on the tensor core -> channels [H, D)
        if (C::MMA2) {
            tc::fence_async_smem();
            tc::tc_fence_before();
            __syncthreads();
            tc::tc_fence_after();
            if (C::STREAM) {
                gemm_streamed<H, H>(tmem + LSE2_COL, a_hi, a_lo, p.wl2_img, ring, C::RING_SLOT, &mbar[2], ph_ring, tid);
            } else {
                if (tid == 0) {
                    issue_resident<H, H>(tmem + LSE2_COL, a_hi, a_lo, b2_hi, b2_lo);
                    tc::umma_commit(&mbar[0]);
                }
                tc::mbar_wait(&mbar[0], ph_main[0]);
                ph_main[0] ^= 1;
                tc::tc_fence_after();
            }
            constexpr int NR2 = H / (8 * NPART) > 0 ? H / (8 * NPART) : 1;   // 8-column groups of r2 per thread
            constexpr int NB = NR2 > 4 ? 4 : NR2;                            // loads behind one wait
#pragma unroll
            for (int b0 = 0; b0 < NR2; b0 += NB) {
                uint32_t vr[NB][8];
#pragma unroll
                for (int i = 0; i < NB; ++i)
                    tc::tmem_ld8_issue(tmem_lane + LSE2_COL + (half + (b0 + i) * NPART) * 8, vr[i]);
                tc::tmem_ld_wait();
#pragma unroll
                for (int i = 0; i < NB; ++i) {
                    const int c0 = (half + (b0 + i) * NPART) * 8;
                    float v[8];
                    const float4 sa = *reinterpret_cast<const float4*>(&ST2[c0]);
                    const float4 sb = *reinterpret_cast<const float4*>(&ST2[c0 + 4]);
                    const float4 ta = *reinterpret_cast<const float4*>(&ST2[H + c0]);
                    const float4 tb = *reinterpret_cast<const float4*>(&ST2[H + c0 + 4]);
                    const float sc[8] = {sa.x, sa.y, sa.z, sa.w, sb.x, sb.y, sb.z, sb.w};
                    const float sh[8] = {ta.x, ta.y, ta.z, ta.w, tb.x, tb.y, tb.z, tb.w};
#pragma unroll
                    for (int j = 0; j < 8; ++j) {
                        const float a = fmaf(tc::tmem_val(vr[i][j]), sc[j], sh[j]);
                        v[j] = a >= 0.f ? a : 0.2f * a;
                    }
                    uint4 hi, lo;
                    tc::split8(v, hi, lo);
                    *reinterpret_cast<uint4*>(a_hi + tc::op_off(LTC_ROWS, row, (H + c0) / 8)) = hi;
                    *reinterpret_cast<uint4*>(a_lo + tc::op_off(LTC_ROWS, row, (H + c0) / 8)) = lo;
                }
            }
        }
        // (the features overwrite r1 in stage 2: the lse2 MMAs that read it have completed)
        store_features();
        if (PREF && LATE) advance(tile);     // lands behind the score GEMM and the epilogue
        tc::fence_async_smem();
        tc::tc_fence_before();
        __syncthreads();
        tc::tc_fence_after();

        // ---------------- scores = X . Ws^T on the tensor core
        if (C::STREAM) {
            gemm_streamed<D, D>(tmem, a_hi, a_lo, p.ws_img, ring, C::RING_SLOT, &mbar[2], ph_ring, tid);
        } else {
            if (tid == 0) {
                if (C::TRANS) {
                    issue_resident<LTC_ROWS, D>(tmem, b_hi, b_lo, a_hi, a_lo);   // [channel][row]
                    issue_identity<D>(tmem + LTC_ROWS, i_hi, a_hi, a_lo);        // X^T
                } else {
                    issue_resident<D, D>(tmem, a_hi, a_lo, b_hi, b_lo);
                }
                tc::umma_commit(&mbar[1]);
            }
            tc::mbar_wait(&mbar[1], ph_main[1]);
            ph_main[1] ^= 1;
            tc::tc_fence_after();
        }

        // ---------------- softmax over the 16 rows of each point + weighted sum
        if (C::TRANS) {
            // thread = TMEM lane = score channel; its 2 points' 16 neighbours are 16 columns each
            const int tl = (warp & 3) * 32 + lane;
            const int c = tl % D;
            const int pbase = (D == 64 ? (tl >> 6) * 4 : 0) + (warp >> 2) * 2;
#pragma unroll
            for (int q = 0; q < 2; ++q) {
                const int pt = pbase + q;
                float s[16], x[16];
                {
                    uint32_t sr[16], xr[16];     // scores and X^T of the point behind one wait
                    tc::tmem_ld16_issue(tmem_lane + pt * LTC_K, sr);
                    tc::tmem_ld16_issue(tmem_lane + LTC_ROWS + pt * LTC_K, xr);
                    tc::tmem_ld_wait();
#pragma unroll
                    for (int j = 0; j < 16; ++j) {
                        s[j] = tc::tmem_val(sr[j]);
                        x[j] = tc::tmem_val(xr[j]);
                    }
                }
                float m = s[0];
#pragma unroll
                for (int j = 1; j < 16; ++j) m = fmaxf(m, s[j]);
                float num = 0.f, den = 0.f;
                const float ml = -m * kLog2e;
#pragma unroll
                for (int j = 0; j < 16; ++j) {
                    const float ev = ex2_ftz(fmaf(s[j], kLog2e, ml));
                    den += ev;
                    num = fmaf(ev, x[j], num);
                }
                const int64_t gp = tile * (LTC_ROWS / LTC_K) + pt;
                if (gp < p.total) p.agg[(size_t)gp * D + c] = num / den;
            }
        }
        const bool upper = (lane & 16) != 0;
        const int j16 = lane & 15;
        for (int c0 = half * 16; c0 < (C::TRANS ? 0 : D); c0 += 32) {
            float s[16], x[16];
            tc::tmem_ld16(tmem_lane + c0, s);
#pragma unroll
            for (int q = 0; q < 2; ++q) {
                const uint4 hq = *reinterpret_cast<const uint4*>(a_hi + tc::op_off(LTC_ROWS, row, c0 / 8 + q));
                const uint4 lq = *reinterpret_cast<const uint4*>(a_lo + tc::op_off(LTC_ROWS, row, c0 / 8 + q));
                const __half2* hh = reinterpret_cast<const __half2*>(&hq);
                const __half2* ll = reinterpret_cast<const __half2*>(&lq);
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                    const float2 fh = __half22float2(hh[u]), fl = __half22float2(ll[u]);
                    x[q * 8 + 2 * u] = fh.x + fl.x;
                    x[q * 8 + 2 * u + 1] = fh.y + fl.y;
                }
            }
            float den[16], num[16];
#pragma unroll
            for (int i = 0; i < 16; ++i) {
                int o = __float_as_int(s[i]);
                o ^= (o >> 31) & 0x7fffffff;              // order-preserving float -> int
                // per-half-warp max through two FULL-warp reductions (redux.sync with two different
                // sub-warp masks in one instruction returned the wrong group's maximum on B200)
                const int m_lo = __reduce_max_sync(0xffffffffu, upper ? INT_MIN : o);
                const int m_hi = __reduce_max_sync(0xffffffffu, upper ? o : INT_MIN);
                int m = upper ? m_hi : m_lo;
                m ^= (m >> 31) & 0x7fffffff;
                const float ev = ex2_ftz(fmaf(s[i], kLog2e, -__int_as_float(m) * kLog2e));
                den[i] = ev;
                num[i] = ev * x[i];
#ifdef O3DML_DEBUG_NAN
                if (!(ev <= 1.0f) || !(fabsf(x[i]) < 1e30f) || !(fabsf(s[i]) < 1e30f))
                    printf("DBG tile %lld row %d c0 %d i %d s %g m %g ev %g x %g o %d mi %d\n",
                           (long long)tile, row, c0, i, s[i], __int_as_float(m), ev, x[i], o, m);
#endif
            }
            // reduce-scatter over the 16 lanes of the group: afterwards lane j16 holds column c0+j16
#pragma unroll
            for (int w = 8; w >= 1; w >>= 1) {
                const bool up = (lane & w) != 0;
#pragma unroll
                for (int i = 0; i < w; ++i) {
                    const float sd = up ? den[i] : den[i + w];
                    const float sn = up ? num[i] : num[i + w];
                    const float rd = __shfl_xor_sync(0xffffffffu, sd, w);
                    const float rn = __shfl_xor_sync(0xffffffffu, sn, w);
                    den[i] = (up ? den[i + w] : den[i]) + rd;
                    num[i] = (up ? num[i + w] : num[i]) + rn;
                }
            }
            if (g < p.total) p.agg[(size_t)g * D + c0 + j16] = num[0] / den[0];
        }
        tc::tc_fence_before();
        __syncthreads();   // TMEM accumulators and the A tile are free for the next tile
        tc::tc_fence_after();
    }
    __syncthreads();
    if (warp == 0) tc::tmem_dealloc<C::TMEM_COLS>(tmem);
}

template <int D, int STAGE>
static int lfa_tc_launch(const LfaTcParams& p, cudaStream_t st) {
    using C = LtcCfg<D, STAGE>;
    static_assert(C::SMEM <= 227 * 1024, "shared memory budget");
    static PerDeviceOnce once;
    const int dev = current_device();
    if (once.need(dev)) {
        O3DML_CUDA(cudaFuncSetAttribute(lfa_pool_tc_kernel<D, STAGE>,
                                        cudaFuncAttributeMaxDynamicSharedMemorySize, (int)C::SMEM));
        once.done(dev);
    }
    int per_sm = (int)(224 * 1024 / (C::SMEM + 1024));
    if (per_sm < 1) per_sm = 1;
    if (per_sm * C::TMEM_COLS > 512) per_sm = 512 / C::TMEM_COLS;
    if (per_sm > 4) per_sm = 4;
    int64_t grid = (int64_t)device_sm_count() * per_sm;
    if (grid > p.num_tiles) grid = p.num_tiles;
    lfa_pool_tc_kernel<D, STAGE><<<(unsigned)grid, C::NTH, C::SMEM, st>>>(p);
    O3DML_LAUNCH_CHECK();
    o3dml_count_launches(1);
    return O3DML_OK;
}

}  // namespace o3dml

using namespace o3dml;

extern "C" int o3dml_randla_lfa_pool_tc(int stage, int d, const float* coords, const void* neighbor_idx,
                                        int idx_is64, int num_neighbors, const float* feat, int64_t batch,
                                        int64_t n_per_batch, const float* w10_t, const float* s10,
                                        const float* t10, const void* wl2_image, const float* wl2_t,
                                        const float* s2, const float* t2, const void* wscore_image,
                                        float* agg, void* stream) {
    O3DML_CHECK(stage == 1 || stage == 2, "lfa_tc: stage must be 1 or 2");
    O3DML_CHECK(num_neighbors == LTC_K, "lfa_tc: built for 16 neighbours");
    O3DML_CHECK(batch * n_per_batch < ((int64_t)1 << 31), "lfa_tc: too many points");
    O3DML_CHECK(stage == 1 || (s2 && t2 && (d == 16 ? wl2_t != nullptr : wl2_image != nullptr)),
                "lfa_tc: stage 2 needs the lse2 weights");
    LfaTcParams p;
    p.coords = coords; p.nidx = neighbor_idx; p.nidx_is64 = idx_is64; p.feat = feat;
    p.total = batch * n_per_batch; p.n_per_batch = n_per_batch;
    p.w10t = w10_t; p.s10 = s10; p.t10 = t10;
    p.wl2_img = (const uint4*)wl2_image; p.wl2t = wl2_t; p.s2 = s2; p.t2 = t2;
    p.ws_img = (const uint4*)wscore_image; p.agg = agg;
    p.num_tiles = ceil_div<int64_t>(p.total, LTC_ROWS / LTC_K);
    if (p.total == 0) return O3DML_OK;
    cudaStream_t st = (cudaStream_t)stream;
#define LTC_CASE(DD) \
    case DD: return stage == 1 ? lfa_tc_launch<DD, 1>(p, st) : lfa_tc_launch<DD, 2>(p, st);
    switch (d) {
        LTC_CASE(16)
        LTC_CASE(32)
        LTC_CASE(64)
        LTC_CASE(128)
        LTC_CASE(256)
        default:
            O3DML_FAIL(O3DML_ERR_UNSUPPORTED, "lfa_tc: d_out %d not in {16,32,64,128,256}", d);
    }
#undef LTC_CASE
}

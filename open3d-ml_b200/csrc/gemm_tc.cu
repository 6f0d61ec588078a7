// gemm_tc.cu -- the gathered GEMM / implicit-GEMM convolution of gemm.cu on the tcgen05 tensor cores,
// round-2 design: 3xTF32 split, operands staged by the TMA engine.
//
//   D[128 x BN] = A[128 x K] * W[K x BN], fp32 in / fp32 out, accumulated in TMEM.
//
// Precision.  kind::tf32 keeps fp32's exponent, so -- unlike the fp16 split of round 1 -- no range
// pass, no power-of-two scaling and no clamp are needed.  x = hi + lo with hi = x & 0xFFFFE000
// (the 10 explicit mantissa bits TF32 keeps) and lo = x - hi (exact in fp32, <= 13 bits of which the
// tensor core keeps 11): A*W ~= Ah*Wh + Ah*Wl + Al*Wh, relative error ~2^-21 per product, i.e. the
// same 22 bits the fp16 split delivered (tests/test_split_numerics.py emulates it on the CPU).
// The weight side is split by the host (round-to-nearest, _lib.pack_linear).
//
// Data movement.  The raw fp32 A slice (128 rows x 32 channels = 128 B per row) IS the hi operand:
//   * identity row sources and the 3x3 convolution taps are fetched by ONE cp.async.bulk.tensor per
//     slice (2-D {channels, rows} map; 4-D {C, W, H, B} map whose box is a PW x PH patch of output
//     pixels shifted by the tap -- negative / overflowing coordinates are zero-filled by the TMA unit,
//     which is the convolution padding; stride-2 convolutions use four parity maps),
//   * gathered sources (index / batch-relative index / shadow rows) by 16-byte cp.async into the same
//     128-byte-swizzled layout,
//   * the weight slices (hi and lo image) by two more tensor copies.
// The 8 converter warps then only run  hi = x & mask, lo = x - hi  on their row (45 instructions per
// thread and slice against 357 + 686 in round 1) and store both parts into TENSOR MEMORY
// (tcgen05.st): the MMAs take A from TMEM (.kind::tf32 [d], [a], b-desc) and only W from shared memory.
// Why: an SS-mode 128x128x8 MMA reads 8 KB of shared memory in its 64 cycles, i.e. it saturates the
// 128 B/clk shared-memory port on its own; the first round-2 version (A hi/lo rewritten in shared
// memory) measured ~1 500 cycles per slice because the TMA fills (48 KB), the converter traffic (48 KB)
// and the operand reads (96 KB) all queue on that port.  With A in TMEM a slice moves 48 KB of fills,
// 16 KB of converter reads and 48 KB of W reads: 875 cycles against 768 of MMA issue.
// Shared-memory layout: K-major, SWIZZLE_128B (row r, 16-byte chunk c at r*128 + ((c ^ (r & 7)) << 4)),
// UMMA descriptors with SBO = 1024, K advanced by +32 B per MMA (K = 8 TF32).
// TMEM layout: columns [0, 2 BN) two accumulator buffers, then per stage 32 columns of A-hi and 32 of
// A-lo (lane = row, column = k: the M = 128 A-fragment layout of the TS-mode MMA).
//
// TMEM accumulation truncates (measured round 1), hence every GT_FLUSH slices the accumulator is folded
// into fp32 registers with round-to-nearest adds while the next chunk runs in the other TMEM buffer.
#include "../../include/o3dml_b200.h"
#include "common.cuh"
#include "tc.cuh"
#include <cuda.h>
#include <algorithm>

namespace o3dml {

#ifdef O3DML_DEBUG_TIMING
__device__ long long g_gt_dbg[8192];
#endif

constexpr int GT_ROWS = 128;
constexpr int GT_KS = 32;        // fp32 channels per k-slice (= one 128-byte swizzle row)
constexpr int GT_FLUSH = 4;      // k-slices (128 channels = 48 accumulating MMAs) per TMEM accumulation chunk
constexpr int GT_MAX_SRC = 3;
constexpr int GT_CONV_THREADS = 256;   // warps 0-7: converters + flush + epilogue
constexpr int GT_LOADERS = 128;        // warps 10-13 (GATHER kernels only)
constexpr int GT_A_BYTES = GT_ROWS * 128;

struct GtSrc {
    const float* data;
    const void* index;
    int64_t rows, out_rows_per_batch, src_rows_per_batch;
    int32_t channels, ld, index_is64, index_ld;
};

struct alignas(64) GemmTcParams {
    CUtensorMap mapA[4];   // rows mode: one per identity source; conv: stride 1 -> [0], stride 2 -> parity (py*2+px)
    CUtensorMap mapB;      // {Kpad, 2*Npad}: hi rows [0, Npad), lo rows [Npad, 2*Npad)
    int64_t N;
    int K, Kpad, Cout, Npad;
    int mode;  // 0 rows, 1 conv3x3
    int nsrc;
    GtSrc src[GT_MAX_SRC];
    int koff[GT_MAX_SRC + 1];
    int H, W, OH, OW, stride, C;
    int lpw, PH, tiles_x, tiles_y;   // conv: patch = (1 << lpw) x PH output pixels per CTA
    const float* scale;
    const float* shift;
    const float* residual;
    int res_ld;
    int act;
    float slope;
    float* out;
    int out_ld;
    int out_mode;   // 0 rows, 1 NCHW, 2 deconv pixel shuffle
    int64_t plane;
    int ds, dIH, dIW, dC;
};

__device__ __forceinline__ const float* gt_src_ptr(const GemmTcParams& p, int s, int64_t n) {
    const GtSrc& S = p.src[s];
    int64_t r = n;
    if (S.index) {
        r = load_index(S.index, n * S.index_ld, S.index_is64);
        if (r < 0) return nullptr;
        if (S.out_rows_per_batch > 0) {
            if (r >= S.src_rows_per_batch) return nullptr;
            r += (n / S.out_rows_per_batch) * S.src_rows_per_batch;
        }
        if (r >= S.rows) return nullptr;
    }
    return S.data + (size_t)r * S.ld;
}

// ---- async-copy primitives ---------------------------------------------------------------------
__device__ __forceinline__ void cp_async16(uint32_t smem_dst, const void* gsrc, int src_bytes) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(smem_dst), "l"(gsrc), "r"(src_bytes)
                 : "memory");
}
// the mbarrier gets one (pre-counted) arrival from this thread once all of its earlier cp.async have landed
__device__ __forceinline__ void cp_async_arrive(uint64_t* bar) {
    asm volatile("cp.async.mbarrier.arrive.noinc.shared::cta.b64 [%0];" ::"r"(tc::smem_u32(bar)) : "memory");
}
using tc::mbar_arrive_expect_tx;
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(tc::smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void named_bar_sync(int id, int nthreads) {
    asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}
__device__ __forceinline__ bool elect_one() {
    uint32_t pred;
    asm volatile("{\n\t.reg .pred p;\n\telect.sync _|p, 0xffffffff;\n\tselp.u32 %0, 1, 0, p;\n\t}" : "=r"(pred));
    return pred != 0;
}
// TMA tiled loads (cp.async.bulk.tensor), completion counted in bytes on the mbarrier
__device__ __forceinline__ void tma_load_2d(uint32_t smem_dst, const CUtensorMap* map, int c0, int c1, uint64_t* bar) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(
            smem_dst),
        "l"(map), "r"(tc::smem_u32(bar)), "r"(c0), "r"(c1)
        : "memory");
}
__device__ __forceinline__ void tma_load_4d(uint32_t smem_dst, const CUtensorMap* map, int c0, int c1, int c2, int c3,
                                            uint64_t* bar) {
    asm volatile(
        "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], "
        "[%2];" ::"r"(smem_dst),
        "l"(map), "r"(tc::smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
        : "memory");
}
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* map) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(map) : "memory");
}

// K-major SWIZZLE_128B operand descriptor: rows of 128 B, 8-row groups 1024 B apart (cute::UMMA::SmemDescriptor:
// start[0,14) lbo[16,30)=1 sbo[32,46)=64 version[46,48)=1 layout_type[61,64)=2)
__device__ __forceinline__ uint64_t smem_desc_sw128(uint32_t saddr) {
    uint64_t d = 0;
    d |= (uint64_t)((saddr >> 4) & 0x3fffu);
    d |= (uint64_t)1 << 16;
    d |= (uint64_t)(1024 >> 4) << 32;
    d |= (uint64_t)1 << 46;
    d |= (uint64_t)2 << 61;
    return d;
}
// kind::tf32 instruction descriptor: c_format[4,6)=1 (fp32), a_format[7,10)=b_format[10,13)=2 (TF32), both K-major
__host__ __device__ constexpr uint32_t idesc_tf32(int M, int N) {
    return (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}
__device__ __forceinline__ void umma_tf32(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                          uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}" ::"r"(tmem_d),
        "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}

// TS mode: A from tensor memory (lane = row, one column per TF32 element), B from shared memory
__device__ __forceinline__ void umma_tf32_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t bdesc, uint32_t idesc,
                                             uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], [%1], %2, %3, p;\n\t}" ::"r"(tmem_d),
        "r"(tmem_a), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}
// same, W descriptor passed as its two 32-bit words (only the low word varies between MMAs)
__device__ __forceinline__ void umma_tf32_ts2(uint32_t tmem_d, uint32_t tmem_a, uint32_t bdesc_lo, uint32_t bdesc_hi,
                                              uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t.reg .b64 d;\n\t"
        "mov.b64 d, {%2, %3};\n\t"
        "setp.ne.b32 p, %5, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], [%1], d, %4, p;\n\t}" ::"r"(tmem_d),
        "r"(tmem_a), "r"(bdesc_lo), "r"(bdesc_hi), "r"(idesc), "r"(accumulate)
        : "memory");
}
// registers -> TMEM: 32 lanes x 32 bit, 16 consecutive columns per thread (lane = 32 * (warp % 4) + lane id)
__device__ __forceinline__ void tmem_st16(uint32_t taddr, const uint32_t* r) {
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], "
        "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};" ::"r"(taddr),
        "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]), "r"(r[9]),
        "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15])
        : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// LITE: two stages and 256 TMEM columns instead of 4 - 6 stages and all 512, so that TWO CTAs share an SM.  A short
// product (K <= 512) is prologue (3.1 k cycles) + epilogue (3.5 - 6.4 k) around 0.7 k per 32-channel slice: with one CTA
// per SM the tensor pipe and the TMA unit idle through both; a sibling CTA fills them.
template <int BN, bool LITE = false>
struct GtCfg {
    static constexpr int B_BYTES = BN * 128;                       // one of hi/lo per stage
    static constexpr int STAGE = GT_A_BYTES + 2 * B_BYTES;         // raw A + W hi + W lo; multiples of 1024
    // bytes in flight = L2 bandwidth x latency: at BN = 64 a slice is consumed every ~430 cycles and takes ~2 500 to
    // arrive, i.e. ~190 KB must be outstanding (5 x 32 KB stages measured 648 cycles per slice, TMA-latency bound)
    static constexpr int STAGES = LITE ? 2 : BN >= 128 ? 4 : 6;
    static constexpr int A_COL0 = 2 * BN;                          // TMEM: accumulators first, then the A slots
    static constexpr int TMEM_COLS = LITE ? 256 : 512;             // 2 * BN + STAGES * 64 <= TMEM_COLS, power of two
    static_assert(2 * BN + STAGES * 64 <= TMEM_COLS, "TMEM budget");
    static_assert(!LITE || BN <= 64, "LITE is for the narrow tiles");
    static constexpr int TAIL = GT_MAX_SRC * GT_ROWS * 8 + GT_ROWS * 8 + 2 * BN * 4 + 256;
    static constexpr size_t SMEM = (size_t)STAGES * STAGE + TAIL + 1024;
    static_assert((size_t)STAGES * STAGE >= (size_t)GT_ROWS * (BN + 4) * 4, "epilogue staging lives in the stages");
};

// Pipeline (per CTA, one [128 x BN] output tile, k-slices of 32 channels through a ring of stages):
//   warps 0-7     converters: wait full[stage], split their row of the raw A tile into (hi, lo), tcgen05.st
//                 into the stage's TMEM slot, arrive conv[stage]; fold finished TMEM chunks into registers;
//                 epilogue (TMEM -> BN /
//                 residual / activation -> shared-memory staged, row-coalesced stores)
//   warp 8        MMA issuer: waits conv[stage], one elected lane issues 12 tcgen05.mma (4 k-steps x 3
//                 products), tcgen05.commit -> empty[stage] (+ chunk[] at chunk ends); owns the TMEM allocation
//   warp 9        TMA producer (one elected lane): waits empty[stage], arms full[stage] with the byte count
//                 and issues the weight-slice copies and -- for identity sources / convolution taps -- the A copy
//   warps 10-13   (GATHER kernels) loaders: 16-byte cp.async of gathered rows into the swizzled A tile,
//                 cp.async.mbarrier.arrive on full[stage]
template <int BN, bool GATHER, bool LITE>
__global__ void __launch_bounds__(GATHER ? 448 : 320, LITE ? 2 : 1)
gemm_tc_kernel(const __grid_constant__ GemmTcParams p) {
    using C = GtCfg<BN, LITE>;
    constexpr int S = C::STAGES;
    extern __shared__ uint8_t smem_raw[];
    const uint32_t raw_addr = tc::smem_u32(smem_raw);
    uint8_t* stages = smem_raw + ((1024u - (raw_addr & 1023u)) & 1023u);           // 1024-byte aligned
    const float** rowptr = reinterpret_cast<const float**>(stages + S * C::STAGE);   // [src][row]
    int64_t* rown = reinterpret_cast<int64_t*>(rowptr + GT_MAX_SRC * GT_ROWS);       // [row] output row or -1
    float* s_scale = reinterpret_cast<float*>(rown + GT_ROWS);                       // [BN] folded BN scale of this column tile
    float* s_shift = s_scale + BN;                                                   // [BN]
    uint64_t* mbar = reinterpret_cast<uint64_t*>(s_shift + BN);
    uint64_t* full_bar = mbar;                // [S] operands of the slice landed
    uint64_t* conv_bar = mbar + S;            // [S] A tile split + fenced
    uint64_t* empty_bar = mbar + 2 * S;       // [S] MMAs that read the stage are done
    uint64_t* chunk_bar = mbar + 3 * S;       // [2] accumulation chunk complete
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(mbar + 3 * S + 2);

    const int tid = threadIdx.x;
    const int warp = __shfl_sync(0xffffffffu, tid >> 5, 0);   // warp-uniform for the compiler
    const int col0 = blockIdx.y * BN;
    // rows mode: 128 consecutive output rows; conv mode: a PW x PH patch of output pixels of one image
    int64_t row0 = (int64_t)blockIdx.x * GT_ROWS;
    int cb = 0, oy0 = 0, ox0 = 0;
    if (p.mode == 1) {
        const int per = p.tiles_x * p.tiles_y;
        cb = blockIdx.x / per;
        const int t = blockIdx.x - cb * per;
        oy0 = (t / p.tiles_x) * p.PH;
        ox0 = (t % p.tiles_x) << p.lpw;
    }
#ifdef O3DML_DEBUG_TIMING
    const bool dbg = blockIdx.x == 0 && blockIdx.y == 0;
    if (dbg && tid == 0) g_gt_dbg[4000] = clock64();
#endif

    // ---- per-row bookkeeping
    for (int m = tid; m < GT_ROWS; m += blockDim.x) {
        int64_t n;
        if (p.mode == 0) {
            n = row0 + m;
            if (n >= p.N) n = -1;
        } else {
            const int oy = oy0 + (m >> p.lpw), ox = ox0 + (m & ((1 << p.lpw) - 1));
            n = (oy < p.OH && ox < p.OW) ? ((int64_t)cb * p.OH + oy) * p.OW + ox : -1;
        }
        rown[m] = n;
    }
    for (int i = tid; i < BN; i += blockDim.x) {      // per-column epilogue constants: read once, not per element
        const int c = col0 + i;
        s_scale[i] = (p.scale && c < p.Cout) ? p.scale[c] : 1.f;
        s_shift[i] = (p.shift && c < p.Cout) ? p.shift[c] : 0.f;
    }
    if (GATHER) {
        for (int i = tid; i < p.nsrc * GT_ROWS; i += blockDim.x) {
            const int s = i / GT_ROWS, m = i % GT_ROWS;
            const int64_t n = row0 + m;
            rowptr[s * GT_ROWS + m] = (n < p.N && p.src[s].index) ? gt_src_ptr(p, s, n) : nullptr;
        }
    }
    if (tid == 0) {
#pragma unroll
        for (int i = 0; i < S; ++i) {
            tc::mbar_init(&full_bar[i], GATHER ? 1 + GT_LOADERS : 1);
            tc::mbar_init(&conv_bar[i], GT_CONV_THREADS);
            tc::mbar_init(&empty_bar[i], 1);
        }
        tc::mbar_init(&chunk_bar[0], 1);
        tc::mbar_init(&chunk_bar[1], 1);
        tc::fence_mbar_init();
    }
    __syncthreads();
    if (warp == 8) tc::tmem_alloc<C::TMEM_COLS>(tmem_slot);
    tc::tc_fence_before();
    __syncthreads();
    tc::tc_fence_after();
    const uint32_t tmem = *tmem_slot;

    const int nsl = p.Kpad / GT_KS;
    const int last_chunk = (nsl - 1) / GT_FLUSH;
    const uint32_t stage0 = tc::smem_u32(stages);

    if (warp == 8) {
        // ================================================================= MMA issuer
        constexpr uint32_t idesc = idesc_tf32(GT_ROWS, BN);
        // descriptor words (smem_desc_sw128): high = sbo 1024 B | version 1 | SWIZZLE_128B; low = start >> 4 | lbo 1
        constexpr uint32_t DESC_HI = (1024u >> 4) | (1u << 14) | (2u << 29);
        const uint32_t desc_lo0 = (((stage0 + GT_A_BYTES) >> 4) & 0x3fffu) | (1u << 16);
        for (int s = 0; s < nsl; ++s) {
            const int stage = s % S, use = s / S, chunk = s / GT_FLUSH;
#ifdef O3DML_DEBUG_TIMING
            const long long tm0 = clock64();
#endif
            tc::mbar_wait(&conv_bar[stage], use & 1);
            tc::tc_fence_after();
#ifdef O3DML_DEBUG_TIMING
            const long long tm1 = clock64();
#endif
            if (elect_one()) {
                // only the 14-bit start-address field of the W descriptors changes: one add per MMA
                // (a lone thread retires ~1 dependent instruction per 4-6 cycles; rebuilding the 64-bit
                // descriptors cost 35-45 cycles per MMA, measured: 414 / 531 cycles to issue 12 MMAs)
                const uint32_t bh_lo = desc_lo0 + (uint32_t)stage * (C::STAGE >> 4);
                const uint32_t bl_lo = bh_lo + (C::B_BYTES >> 4);
                const uint32_t a_hi = tmem + (uint32_t)(C::A_COL0 + stage * 64);
                const uint32_t acc = tmem + (uint32_t)((chunk & 1) * BN);
                const uint32_t first_acc = (s % GT_FLUSH) != 0;
#pragma unroll
                for (int ks = 0; ks < GT_KS / 8; ++ks) {        // K = 8 TF32 = 8 TMEM columns / 32 bytes of W per MMA
                    umma_tf32_ts2(acc, a_hi + ks * 8, bh_lo + ks * 2, DESC_HI, idesc, ks == 0 ? first_acc : 1u);
                    umma_tf32_ts2(acc, a_hi + ks * 8, bl_lo + ks * 2, DESC_HI, idesc, 1u);
                    umma_tf32_ts2(acc, a_hi + 32 + ks * 8, bh_lo + ks * 2, DESC_HI, idesc, 1u);
                }
                tc::umma_commit(&empty_bar[stage]);
                if ((s % GT_FLUSH) == GT_FLUSH - 1 || s == nsl - 1) tc::umma_commit(&chunk_bar[chunk & 1]);
#ifdef O3DML_DEBUG_TIMING
                if (dbg && s < 300) { g_gt_dbg[2000 + 3 * s] = tm0; g_gt_dbg[2001 + 3 * s] = tm1; g_gt_dbg[2002 + 3 * s] = clock64(); }
#endif
            }
            __syncwarp();
        }
    } else if (warp == 9) {
        // ================================================================= TMA producer
        if (elect_one()) {
            tma_prefetch_desc(&p.mapB);
            const int spt = p.mode == 1 ? p.C / GT_KS : 1;      // slices per convolution tap
            int sidx = 0;
            for (int sl = 0; sl < nsl; ++sl) {
                const int stage = sl % S, use = sl / S;
                if (use >= 1) tc::mbar_wait(&empty_bar[stage], (use - 1) & 1);
                const int k0 = sl * GT_KS;
                bool a_tma = true;
                if (p.mode == 0) {
                    while (sidx + 1 < p.nsrc && k0 >= p.koff[sidx + 1]) ++sidx;
                    a_tma = p.src[sidx].index == nullptr;
                }
                const uint32_t ah = stage0 + (uint32_t)stage * C::STAGE;
                const uint32_t bh = ah + GT_A_BYTES;
                mbar_arrive_expect_tx(&full_bar[stage], 2 * C::B_BYTES + (a_tma ? GT_A_BYTES : 0));
                tma_load_2d(bh, &p.mapB, k0, col0, &full_bar[stage]);
                tma_load_2d(bh + C::B_BYTES, &p.mapB, k0, p.Npad + col0, &full_bar[stage]);
                if (a_tma) {
                    if (p.mode == 0) {
                        tma_load_2d(ah, &p.mapA[sidx], k0 - p.koff[sidx], (int)row0, &full_bar[stage]);
                    } else {
                        const int tap = sl / spt, cc = (sl - tap * spt) * GT_KS;
                        const int dy = tap / 3, dx = tap - dy * 3;
                        if (p.stride == 1) {
                            tma_load_4d(ah, &p.mapA[0], cc, ox0 - 1 + dx, oy0 - 1 + dy, cb, &full_bar[stage]);
                        } else {   // input pixel 2*o - 1 + d: odd parity for d = 0 (coordinate o - 1) and d = 2 (o)
                            const int py = dy != 1, px = dx != 1;
                            tma_load_4d(ah, &p.mapA[py * 2 + px], cc, ox0 - (dx == 0), oy0 - (dy == 0), cb,
                                        &full_bar[stage]);
                        }
                    }
                }
            }
        }
    } else if (GATHER && warp >= 10) {
        // ================================================================= gather loaders
        const int rt = tid - 320;
        int sidx = 0;
        for (int sl = 0; sl < nsl; ++sl) {
            const int stage = sl % S, use = sl / S;
            if (use >= 1) tc::mbar_wait(&empty_bar[stage], (use - 1) & 1);
            const int k0 = sl * GT_KS;
            while (sidx + 1 < p.nsrc && k0 >= p.koff[sidx + 1]) ++sidx;
            if (p.src[sidx].index != nullptr) {
                const uint32_t ah = stage0 + (uint32_t)stage * C::STAGE;
                const int kloc = k0 - p.koff[sidx];
                const int cs = p.src[sidx].channels;
#pragma unroll
                for (int j = 0; j < (GT_ROWS * 8) / GT_LOADERS; ++j) {     // 8 consecutive lanes = one row's 128 B
                    const int item = rt + j * GT_LOADERS;
                    const int m = item >> 3, c = item & 7;
                    const float* base = rowptr[sidx * GT_ROWS + m];
                    const int kk = kloc + c * 4;
                    const bool ok = base != nullptr && kk < cs;
                    cp_async16(ah + (uint32_t)m * 128u + (uint32_t)((c ^ (m & 7)) << 4),
                               ok ? (const void*)(base + kk) : (const void*)p.src[0].data, ok ? 16 : 0);
                }
                cp_async_arrive(&full_bar[stage]);
            } else {
                mbar_arrive(&full_bar[stage]);
            }
        }
    } else if (warp < 8) {
        // ================================================================= converters + flush + epilogue
        const int grp = warp >> 2;                     // column half
        const int rt = (warp & 3) * 32 + (tid & 31);   // output row = TMEM lane this thread can read
        const uint32_t tmem_lane = tmem + ((uint32_t)((warp & 3) * 32) << 16);
        constexpr int HB = BN / 2 < 16 ? 16 : BN / 2;  // columns owned by a group
        constexpr int NQ = HB / 16;
        float racc[HB];
#pragma unroll
        for (int i = 0; i < HB; ++i) racc[i] = 0.f;
        const bool owns_cols = (BN >= 32) || grp == 0;
        const int colbase = (BN >= 32) ? grp * HB : 0;
        uint32_t ph_chunk[2] = {0, 0};
        int next_flush = 0;                            // first chunk not folded yet
        auto fold = [&](int chunk) {                   // racc += accumulator of `chunk` (RN adds)
            tc::mbar_wait(&chunk_bar[chunk & 1], ph_chunk[chunk & 1]);
            ph_chunk[chunk & 1] ^= 1;
            tc::tc_fence_after();
            if (owns_cols) {
                uint32_t vr[NQ][16];       // all of this thread's columns behind one wait
#pragma unroll
                for (int q = 0; q < NQ; ++q) tc::tmem_ld16_issue(tmem_lane + (chunk & 1) * BN + colbase + q * 16, vr[q]);
                tc::tmem_ld_wait();
#pragma unroll
                for (int q = 0; q < NQ; ++q)
#pragma unroll
                    for (int j = 0; j < 16; ++j) racc[q * 16 + j] += tc::tmem_val(vr[q][j]);
            }
            tc::tc_fence_before();
        };
        for (int s = 0; s < nsl; ++s) {
            const int stage = s % S, use = s / S;
            // a chunk whose last slice is S slices behind has certainly drained (its stage was reused): fold it then,
            // and in any case before slice (chunk + 2) * GT_FLUSH reuses its TMEM buffer (the fold waits if it must)
            constexpr int LAG = (S - 1 < GT_FLUSH) ? S - 1 : GT_FLUSH;
            while (next_flush < last_chunk && s >= (next_flush + 1) * GT_FLUSH + LAG) fold(next_flush++);
#ifdef O3DML_DEBUG_TIMING
            const long long tq0 = clock64();
#endif
            tc::mbar_wait(&full_bar[stage], use & 1);
            tc::tc_fence_after();       // the MMAs that read this stage's TMEM slot completed (empty -> TMA -> full)
#ifdef O3DML_DEBUG_TIMING
            const long long tq1 = clock64();
#endif
            // this thread's row, k-half `grp` (4 of the row's 8 swizzled 16-byte chunks) -> hi / lo -> TMEM
            const uint8_t* a_row = stages + (size_t)stage * C::STAGE + (size_t)rt * 128;
            uint32_t hi[16], lo[16];
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const int cch = grp * 4 + j;
                const uint4 v = *reinterpret_cast<const uint4*>(a_row + (((cch ^ (rt & 7))) << 4));
                const uint32_t x[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                    hi[4 * j + u] = x[u] & 0xFFFFE000u;
                    lo[4 * j + u] = __float_as_uint(__uint_as_float(x[u]) - __uint_as_float(hi[4 * j + u]));
                }
            }
            const uint32_t a_slot = tmem_lane + (uint32_t)(C::A_COL0 + stage * 64 + grp * 16);
            tmem_st16(a_slot, hi);
            tmem_st16(a_slot + 32, lo);
            tmem_st_wait();
            tc::tc_fence_before();
            mbar_arrive(&conv_bar[stage]);
#ifdef O3DML_DEBUG_TIMING
            if (dbg && tid == 0 && s < 450) {
                g_gt_dbg[4 * s + 0] = tq0; g_gt_dbg[4 * s + 1] = tq1; g_gt_dbg[4 * s + 2] = clock64();
            }
#endif
        }
        while (next_flush < last_chunk) fold(next_flush++);
        tc::mbar_wait(&chunk_bar[last_chunk & 1], ph_chunk[last_chunk & 1]);
        tc::tc_fence_after();
#ifdef O3DML_DEBUG_TIMING
        if (dbg && tid == 0) g_gt_dbg[4002] = clock64();
#endif
        // ---- epilogue: thread = output row, this group's column half, 16 columns at a time.
        // Row-major and pixel-shuffle outputs are staged through the (now dead) pipeline stages so that the
        // global stores are whole rows written by consecutive lanes.
        const int64_t n = rown[rt];
        constexpr int SLD = BN + 4;                                  // staging row stride (floats)
        float* stg = reinterpret_cast<float*>(stages);
        const bool staged = p.out_mode == 0 || (p.out_mode == 2 && (p.dC & 3) == 0);
        if (owns_cols) {
#pragma unroll
            for (int q = 0; q < NQ; ++q) {
                const int c0 = colbase + 16 * q;
                float v[16];
                tc::tmem_ld16(tmem_lane + (last_chunk & 1) * BN + c0, v);   // warp-collective
                const int cbase = col0 + c0;
                if (n < 0 || cbase >= p.Cout) continue;
                // staged outputs get the residual and the activation in the row-coalesced copy-out below
#pragma unroll
                for (int j = 0; j < 16; ++j) {
                    float x = fmaf(v[j] + racc[q * 16 + j], s_scale[c0 + j], s_shift[c0 + j]);
                    if (!staged) {
                        const int c = cbase + j;
                        if (p.residual && c < p.Cout) x += p.residual[(size_t)n * p.res_ld + c];
                        x = apply_act(x, p.act, p.slope);
                    }
                    v[j] = x;
                }
                if (staged) {
#pragma unroll
                    for (int u = 0; u < 4; ++u)
                        *reinterpret_cast<float4*>(stg + rt * SLD + c0 + 4 * u) =
                            make_float4(v[4 * u], v[4 * u + 1], v[4 * u + 2], v[4 * u + 3]);
                } else if (p.out_mode == 1) {
                    const int64_t b = n / p.plane, pix = n % p.plane;
#pragma unroll
                    for (int j = 0; j < 16; ++j)
                        if (cbase + j < p.Cout) p.out[((size_t)b * p.Cout + cbase + j) * p.plane + pix] = v[j];
                } else {
                    const int64_t per = (int64_t)p.dIH * p.dIW;
                    const int64_t b = n / per;
                    const int r = (int)(n % per);
                    const int iy = r / p.dIW, ix = r % p.dIW;
                    const int OWd = p.dIW * p.ds;
#pragma unroll
                    for (int j = 0; j < 16; ++j) {
                        const int c = cbase + j;
                        if (c < p.Cout) {
                            const int sub = c / p.dC, co = c - sub * p.dC;
                            const int dy = sub / p.ds, dx = sub - dy * p.ds;
                            const size_t opix = ((size_t)b * p.dIH * p.ds + (size_t)iy * p.ds + dy) * OWd +
                                                (size_t)ix * p.ds + dx;
                            p.out[opix * p.out_ld + co] = v[j];
                        }
                    }
                }
            }
        }
        if (staged) {
            named_bar_sync(2, GT_CONV_THREADS);                        // the 8 epilogue warps
            constexpr int LPR = BN / 4;                                // lanes per output row
            const int c = (tid % LPR) * 4, cg = col0 + c;
            const bool vec = (p.out_ld & 3) == 0 && (reinterpret_cast<uintptr_t>(p.out) & 15) == 0;
            if (cg < p.Cout) {
                for (int r = tid / LPR; r < GT_ROWS; r += GT_CONV_THREADS / LPR) {
                    const int64_t nr = rown[r];
                    if (nr < 0) continue;
                    float4 v = *reinterpret_cast<const float4*>(stg + r * SLD + c);
                    if (p.residual) {
                        const float* rp = p.residual + (size_t)nr * p.res_ld + cg;
                        if (cg + 3 < p.Cout && (p.res_ld & 3) == 0 && (reinterpret_cast<uintptr_t>(p.residual) & 15) == 0) {
                            const float4 rv = *reinterpret_cast<const float4*>(rp);
                            v.x += rv.x; v.y += rv.y; v.z += rv.z; v.w += rv.w;
                        } else {
                            if (cg < p.Cout) v.x += rp[0];
                            if (cg + 1 < p.Cout) v.y += rp[1];
                            if (cg + 2 < p.Cout) v.z += rp[2];
                            if (cg + 3 < p.Cout) v.w += rp[3];
                        }
                    }
                    v.x = apply_act(v.x, p.act, p.slope); v.y = apply_act(v.y, p.act, p.slope);
                    v.z = apply_act(v.z, p.act, p.slope); v.w = apply_act(v.w, p.act, p.slope);
                    float* o;
                    if (p.out_mode == 0) {
                        o = p.out + (size_t)nr * p.out_ld + cg;
                    } else {
                        const int64_t per = (int64_t)p.dIH * p.dIW;
                        const int64_t b = nr / per;
                        const int rr = (int)(nr % per);
                        const int iy = rr / p.dIW, ix = rr % p.dIW;
                        const int sub = cg / p.dC, co = cg - sub * p.dC;
                        const int dy = sub / p.ds, dx = sub - dy * p.ds;
                        const size_t opix = ((size_t)b * p.dIH * p.ds + (size_t)iy * p.ds + dy) * (p.dIW * p.ds) +
                                            (size_t)ix * p.ds + dx;
                        o = p.out + opix * p.out_ld + co;
                    }
                    if (vec && cg + 3 < p.Cout) {
                        *reinterpret_cast<float4*>(o) = v;
                    } else {
                        const float e[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
                        for (int j = 0; j < 4; ++j)
                            if (cg + j < p.Cout) o[j] = e[j];
                    }
                }
            }
        }
    }
    tc::tc_fence_before();
    __syncthreads();
#ifdef O3DML_DEBUG_TIMING
    if (dbg && tid == 0) g_gt_dbg[4003] = clock64();
#endif
    if (warp == 8) tc::tmem_dealloc<C::TMEM_COLS>(tmem);
}

// ---- host side ---------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn encode_fn() {
    static EncodeTiledFn fn = nullptr;
    if (!fn) {
        void* ptr = nullptr;
        cudaDriverEntryPointQueryResult qres;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &ptr, cudaEnableDefault, &qres) == cudaSuccess &&
            qres == cudaDriverEntryPointSuccess)
            fn = (EncodeTiledFn)ptr;
    }
    return fn;
}

// fp32 tensor map with SWIZZLE_128B (inner box = 32 floats = 128 B), zero OOB fill
static int make_map(CUtensorMap* map, const void* base, int rank, const uint64_t* dims, const uint64_t* strides_bytes,
                    const uint32_t* box) {
    EncodeTiledFn fn = encode_fn();
    if (!fn) O3DML_FAIL(O3DML_ERR_CUDA, "linear_tc: cuTensorMapEncodeTiled is not available from the driver");
    cuuint64_t d[5], s[4];
    cuuint32_t b[5], e[5];
    for (int i = 0; i < rank; ++i) { d[i] = dims[i]; b[i] = box[i]; e[i] = 1; }
    for (int i = 0; i + 1 < rank; ++i) s[i] = strides_bytes[i];
    CUresult r = fn(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, (cuuint32_t)rank, const_cast<void*>(base), d, s, b, e,
                    CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                    CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) O3DML_FAIL(O3DML_ERR_CUDA, "linear_tc: cuTensorMapEncodeTiled failed (%d)", (int)r);
    return O3DML_OK;
}

static int g_num_sms = 0;
int gt_num_sms() {
    if (!g_num_sms) {
        int dev = 0, n = 0;
        if (cudaGetDevice(&dev) == cudaSuccess &&
            cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) == cudaSuccess && n > 0)
            g_num_sms = n;
        else
            g_num_sms = kNumSMs;
    }
    return g_num_sms;
}

template <int BN, bool GATHER, bool LITE = false>
static int gemm_tc_launch_bn(const GemmTcParams& p, unsigned grid_x, cudaStream_t st) {
    using C = GtCfg<BN, LITE>;
    // the opt-in shared-memory size is a per-device function attribute: set it once per device ordinal
    static unsigned long long configured = 0;
    int dev = 0;
    O3DML_CUDA(cudaGetDevice(&dev));
    if (dev >= 64 || !((configured >> dev) & 1ull)) {
        O3DML_CUDA(cudaFuncSetAttribute(gemm_tc_kernel<BN, GATHER, LITE>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                        (int)C::SMEM));
        if (dev < 64) configured |= 1ull << dev;
    }
    dim3 grid(grid_x, (unsigned)(p.Npad / BN));
    gemm_tc_kernel<BN, GATHER, LITE><<<grid, GATHER ? 448 : 320, C::SMEM, st>>>(p);
    O3DML_LAUNCH_CHECK();
    o3dml_count_launches(1);
    return O3DML_OK;
}

static int gemm_tc_launch(GemmTcParams& p, const void* wimg, cudaStream_t st) {
    if (p.N <= 0 || p.Cout <= 0) return O3DML_OK;
    O3DML_CHECK(p.Kpad % GT_KS == 0 && p.Kpad >= p.K, "linear_tc: weight image K padding must be a multiple of 32");
    O3DML_CHECK(p.Npad == 32 || p.Npad == 64 || p.Npad % 128 == 0,
                "linear_tc: weight image rows must be padded to 32, 64 or a multiple of 128");
    int bn = p.Npad == 32 ? 32 : (p.Npad == 64 ? 64 : 128);
    bool any_gather = false;
    if (p.mode == 0)
        for (int s = 0; s < p.nsrc; ++s) any_gather = any_gather || p.src[s].index != nullptr;
    int64_t row_tiles = ceil_div<int64_t>(p.N, GT_ROWS);
    if (p.mode == 1) {
        int best_tiles = 1 << 30;
        for (int l = 0; l <= 7; ++l) best_tiles = std::min(best_tiles, ceil_div(p.OW, 1 << l) * ceil_div(p.OH, GT_ROWS >> l));
        row_tiles = (p.N / ((int64_t)p.OH * p.OW)) * best_tiles;
    }
    // products of plain row sources, at most 16 k-slices long, that fill the SMs more than once as 64-column tiles run on
    // the LITE kernels, two CTAs per SM (GtCfg).  Measured (profiles/r02_gemm_lite.md): threshold 4 / 16 / 64 / none =
    // RandLA-Net 220.0 / 220.4 / 220.3 / 220.3, PointPillars 24.4 / 24.9 / 24.9 / 24.9, KPFCNN 48.8 / 49.1 / 48.6 / 48.1
    // M points/s against 217.1 / 24.0 / 46.5 without; LITE for the convolutions (K = 9 C) loses (PointPillars 24.5).
    const bool lite = p.mode == 0 && !any_gather && p.Kpad / GT_KS <= 16 &&
                      row_tiles * (p.Npad / (bn == 32 ? 32 : 64)) > gt_num_sms();
    if (lite && bn == 128) bn = 64;
    // a grid that fills less than half of the SMs (PointPillars block 3: 27 x 2 CTAs; one cloud per GPU: 6 - 88)
    // runs as 64-column tiles instead: twice the CTAs, 12 x 36 instead of 12 x 64 MMA cycles per slice each
    if (bn == 128 && 2 * row_tiles * (p.Npad / 128) <= gt_num_sms()) bn = 64;
    {   // weight image: fp32 [2 * Npad][Kpad] (TF32 hi rows, then lo rows)
        const uint64_t dims[2] = {(uint64_t)p.Kpad, (uint64_t)2 * p.Npad};
        const uint64_t str[1] = {(uint64_t)p.Kpad * 4};
        const uint32_t box[2] = {GT_KS, (uint32_t)bn};
        int rc = make_map(&p.mapB, wimg, 2, dims, str, box);
        if (rc) return rc;
    }
    bool gather = false;
    unsigned grid_x;
    if (p.mode == 0) {
        grid_x = (unsigned)ceil_div<int64_t>(p.N, GT_ROWS);
        for (int s = 0; s < p.nsrc; ++s) {
            if (p.src[s].index) { gather = true; continue; }
            const uint64_t rows = (uint64_t)(p.src[s].rows > 0 ? p.src[s].rows : p.N);
            const uint64_t dims[2] = {(uint64_t)p.src[s].channels, rows};
            const uint64_t str[1] = {(uint64_t)p.src[s].ld * 4};
            const uint32_t box[2] = {GT_KS, GT_ROWS};
            int rc = make_map(&p.mapA[s], p.src[s].data, 2, dims, str, box);
            if (rc) return rc;
        }
    } else {
        // patch of output pixels per CTA: PW x PH = 128, the shape with the fewest tiles
        int best = -1, best_tiles = 0;
        for (int l = 0; l <= 7; ++l) {
            const int pw = 1 << l, ph = GT_ROWS >> l;
            const int tiles = ceil_div(p.OW, pw) * ceil_div(p.OH, ph);
            if (best < 0 || tiles < best_tiles || (tiles == best_tiles && pw >= 8 && (1 << best) < 8)) {
                best = l;
                best_tiles = tiles;
            }
        }
        p.lpw = best;
        p.PH = GT_ROWS >> best;
        p.tiles_x = ceil_div(p.OW, 1 << best);
        p.tiles_y = ceil_div(p.OH, p.PH);
        const int64_t batch = p.N / ((int64_t)p.OH * p.OW);
        grid_x = (unsigned)(batch * p.tiles_x * p.tiles_y);
        const uint32_t box[4] = {GT_KS, (uint32_t)(1 << best), (uint32_t)p.PH, 1};
        const float* in = p.src[0].data;
        if (p.stride == 1) {
            const uint64_t dims[4] = {(uint64_t)p.C, (uint64_t)p.W, (uint64_t)p.H, (uint64_t)batch};
            const uint64_t str[3] = {(uint64_t)p.C * 4, (uint64_t)p.W * p.C * 4, (uint64_t)p.H * p.W * p.C * 4};
            int rc = make_map(&p.mapA[0], in, 4, dims, str, box);
            if (rc) return rc;
        } else {
            for (int py = 0; py < 2; ++py)
                for (int px = 0; px < 2; ++px) {
                    const uint64_t wp = (uint64_t)(p.W - px + 1) / 2, hp = (uint64_t)(p.H - py + 1) / 2;
                    if (wp == 0 || hp == 0) {      // a 1-pixel-wide image has no odd columns: never addressed in range
                        p.mapA[py * 2 + px] = p.mapA[0];
                        continue;
                    }
                    const uint64_t dims[4] = {(uint64_t)p.C, wp, hp, (uint64_t)batch};
                    const uint64_t str[3] = {(uint64_t)2 * p.C * 4, (uint64_t)2 * p.W * p.C * 4,
                                             (uint64_t)p.H * p.W * p.C * 4};
                    int rc = make_map(&p.mapA[py * 2 + px], in + ((size_t)py * p.W + px) * p.C, 4, dims, str, box);
                    if (rc) return rc;
                }
        }
    }
    if (gather) {
        if (bn == 32) return gemm_tc_launch_bn<32, true>(p, grid_x, st);
        if (bn == 64) return gemm_tc_launch_bn<64, true>(p, grid_x, st);
        return gemm_tc_launch_bn<128, true>(p, grid_x, st);
    }
    if (lite) {
        if (bn == 32) return gemm_tc_launch_bn<32, false, true>(p, grid_x, st);
        return gemm_tc_launch_bn<64, false, true>(p, grid_x, st);
    }
    if (bn == 32) return gemm_tc_launch_bn<32, false>(p, grid_x, st);
    if (bn == 64) return gemm_tc_launch_bn<64, false>(p, grid_x, st);
    return gemm_tc_launch_bn<128, false>(p, grid_x, st);
}

}  // namespace o3dml

using namespace o3dml;

static int gt_common(GemmTcParams& p, const void* wimg, int k_pad, int n_pad, const float* scale,
                     const float* shift, const float* residual, int residual_ld, int act, float slope,
                     float* out, int out_ld, int out_channels) {
    p.Kpad = k_pad;
    p.Npad = n_pad;
    p.scale = scale; p.shift = shift; p.residual = residual; p.res_ld = residual_ld;
    p.act = act; p.slope = slope; p.out = out; p.out_ld = out_ld; p.Cout = out_channels;
    O3DML_CHECK(act >= 0 && act <= 2, "linear_tc: unknown activation %d", act);
    O3DML_CHECK(wimg && out, "linear_tc: null weight image / out");
    O3DML_CHECK((reinterpret_cast<uintptr_t>(wimg) & 15) == 0, "linear_tc: weight image must be 16-byte aligned");
    O3DML_CHECK(n_pad >= out_channels, "linear_tc: weight image has fewer rows than out_channels");
    return O3DML_OK;
}

extern "C" int o3dml_linear_tc_supported(const o3dml_src_t* srcs, int num_srcs) {
    if (num_srcs < 1 || num_srcs > GT_MAX_SRC) return 0;
    for (int s = 0; s < num_srcs; ++s) {
        const o3dml_src_t& S = srcs[s];
        if (!S.data || S.channels <= 0 || (S.channels & 3) || (S.ld & 3) || (reinterpret_cast<uintptr_t>(S.data) & 15))
            return 0;
        if (s + 1 < num_srcs && (S.channels % GT_KS) != 0) return 0;   // a k-slice never straddles two sources
    }
    return 1;
}

extern "C" int o3dml_linear_tc(int64_t num_rows, const o3dml_src_t* srcs, int num_srcs,
                               const void* weight_image, int k_pad, int n_pad, const float* scale,
                               const float* shift, const float* residual, int residual_ld, int act,
                               float slope, float* out, int out_ld, int out_channels,
                               int out_nchw_plane, void* stream) {
    O3DML_CHECK(num_srcs >= 1 && num_srcs <= GT_MAX_SRC, "linear_tc: 1..3 sources");
    O3DML_CHECK(o3dml_linear_tc_supported(srcs, num_srcs),
                "linear_tc: sources need a multiple of 4 channels (32 for all but the last), 16-byte aligned rows");
    GemmTcParams p = {};
    p.N = num_rows;
    p.mode = 0;
    p.nsrc = num_srcs;
    int k = 0;
    for (int s = 0; s < num_srcs; ++s) {
        const o3dml_src_t& S = srcs[s];
        O3DML_CHECK(S.ld >= S.channels, "linear_tc: bad source %d", s);
        p.src[s].data = S.data; p.src[s].index = S.index; p.src[s].rows = S.rows;
        p.src[s].out_rows_per_batch = S.out_rows_per_batch;
        p.src[s].src_rows_per_batch = S.src_rows_per_batch;
        p.src[s].channels = S.channels; p.src[s].ld = S.ld; p.src[s].index_is64 = S.index_is64;
        p.src[s].index_ld = S.index ? (S.index_ld > 0 ? S.index_ld : 1) : 0;
        p.koff[s] = k;
        k += S.channels;
    }
    for (int s = num_srcs; s <= GT_MAX_SRC; ++s) p.koff[s] = k;
    p.K = k;
    int rc = gt_common(p, weight_image, k_pad, n_pad, scale, shift, residual, residual_ld, act, slope, out,
                       out_ld, out_channels);
    if (rc) return rc;
    if (out_nchw_plane > 0) {
        p.out_mode = 1;
        p.plane = out_nchw_plane;
    }
    return gemm_tc_launch(p, weight_image, (cudaStream_t)stream);
}

extern "C" int o3dml_conv3x3_nhwc_tc(const float* in, int batch, int H, int W, int C, int stride,
                                     const void* weight_image, int k_pad, int n_pad, const float* scale,
                                     const float* shift, int act, float slope, float* out,
                                     int out_channels, void* stream) {
    O3DML_CHECK(in && batch > 0 && H > 0 && W > 0, "conv3x3_tc: bad input");
    O3DML_CHECK((C % GT_KS) == 0, "conv3x3_tc: input channels must be a multiple of 32");
    O3DML_CHECK(stride == 1 || stride == 2, "conv3x3_tc: stride 1 or 2");
    O3DML_CHECK((reinterpret_cast<uintptr_t>(in) & 15) == 0, "conv3x3_tc: input must be 16-byte aligned");
    GemmTcParams p = {};
    p.mode = 1;
    p.nsrc = 1;
    p.src[0].data = in;
    p.H = H; p.W = W; p.C = C; p.stride = stride;
    p.OH = (H + 2 - 3) / stride + 1;
    p.OW = (W + 2 - 3) / stride + 1;
    p.N = (int64_t)batch * p.OH * p.OW;
    p.K = 9 * C;
    int rc = gt_common(p, weight_image, k_pad, n_pad, scale, shift, nullptr, 0, act, slope, out,
                       out_channels, out_channels);
    if (rc) return rc;
    return gemm_tc_launch(p, weight_image, (cudaStream_t)stream);
}

extern "C" int o3dml_deconv_nhwc_tc(const float* in, int batch, int H, int W, int C, int stride,
                                    const void* weight_image, int k_pad, int n_pad, const float* scale,
                                    const float* shift, int act, float slope, float* out, int out_ld,
                                    int out_channels, void* stream) {
    O3DML_CHECK(in && batch > 0 && H > 0 && W > 0 && stride >= 1, "deconv_tc: bad input");
    O3DML_CHECK((C % 4) == 0 && (reinterpret_cast<uintptr_t>(in) & 15) == 0, "deconv_tc: C % 4, aligned input");
    GemmTcParams p = {};
    p.N = (int64_t)batch * H * W;
    p.mode = 0;
    p.nsrc = 1;
    p.src[0].data = in; p.src[0].rows = p.N; p.src[0].channels = C; p.src[0].ld = C;
    p.koff[0] = 0;
    for (int i = 1; i <= GT_MAX_SRC; ++i) p.koff[i] = C;
    p.K = C;
    int rc = gt_common(p, weight_image, k_pad, n_pad, scale, shift, nullptr, 0, act, slope, out, out_ld,
                       stride * stride * out_channels);
    if (rc) return rc;
    p.out_mode = 2;
    p.ds = stride; p.dIH = H; p.dIW = W; p.dC = out_channels;
    return gemm_tc_launch(p, weight_image, (cudaStream_t)stream);
}

#ifdef O3DML_DEBUG_TIMING
extern "C" __attribute__((visibility("default"))) int o3dml_gt_debug_read(long long* host, int n) {
    return (int)cudaMemcpyFromSymbol(host, o3dml::g_gt_dbg, sizeof(long long) * n);
}
#endif

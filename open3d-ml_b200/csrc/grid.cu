// grid.cu -- uniform hash-grid neighbour search: exact k-NN and fixed-radius search,
// batched through row_splits.  Support points are counting-sorted into cells and
// stored as float4 (x, y, z, original index) so that every candidate is one
// coalesced 16-byte load; queries are processed in cell order so that the lanes
// of a warp walk the same cells.
//
// Replaces (reference call sites, /root/reference):
//   open3d.core.nns.NearestNeighborSearch.knn_search   ml3d/datasets/utils/dataprocessing.py:99-103
//                                                      (<- RandLANet.transform randlanet.py:218-229)
//   open3d.ml.torch.ops.knn_search                     ml3d/torch/models/point_transformer.py:724-734
//   open3d.ml.torch.layers.FixedRadiusSearch           ml3d/torch/models/kpconv.py:2021-2026
// Result order (implementation-defined upstream, fixed here): rows ascend by
// (squared distance, index); d2 = ((dx*dx + dy*dy) + dz*dz) in float32 without FMA
// (oracle/ops_ref.c).  HBM/latency-bound: 12 B/query in, 8*k (or 4*L) B/query out.
#include "../../include/o3dml_b200.h"
#include "prims.cuh"
#include <float.h>

namespace o3dml {

struct GridInfo {       // one per batch item, device resident
    float ox, oy, oz;   // origin (bbox min)
    float cs, inv_cs;   // cell size
    int dx, dy, dz;     // grid dims
    uint32_t cell_base; // first cell of this batch item in the global cell arrays
    uint32_t pad;
};

__device__ __forceinline__ unsigned f2ord(float f) {
    unsigned u = __float_as_uint(f);
    return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ float ord2f(unsigned u) {
    return __uint_as_float((u & 0x80000000u) ? (u & 0x7fffffffu) : ~u);
}

__device__ __forceinline__ int batch_of(int64_t i, const int64_t* splits, int batch) {
    int lo = 0, hi = batch;
    while (hi - lo > 1) {
        int mid = (lo + hi) >> 1;
        if (splits[mid] <= i) lo = mid; else hi = mid;
    }
    return lo;
}

// bbox[b][0..2] = ordered-uint min, [3..5] = ordered-uint max (initialised by grid_init_kernel)
__global__ void grid_init_kernel(unsigned* bbox, int batch) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < batch * 6) bbox[i] = (i % 6 < 3) ? 0xffffffffu : 0u;
}

__global__ void grid_bbox_kernel(const float* __restrict__ pts, int64_t n,
                                 const int64_t* __restrict__ splits, int batch, unsigned* bbox) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    int b = batch_of(i, splits, batch);
    // warp-aggregate when the whole warp is in the same batch item
    float x = pts[3 * i], y = pts[3 * i + 1], z = pts[3 * i + 2];
    unsigned act = __activemask();
    int b0 = __shfl_sync(act, b, __ffs(act) - 1);
    if (__all_sync(act, b == b0) && act == 0xffffffffu) {
        float mnx = x, mny = y, mnz = z, mxx = x, mxy = y, mxz = z;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            mnx = fminf(mnx, __shfl_xor_sync(0xffffffffu, mnx, o));
            mny = fminf(mny, __shfl_xor_sync(0xffffffffu, mny, o));
            mnz = fminf(mnz, __shfl_xor_sync(0xffffffffu, mnz, o));
            mxx = fmaxf(mxx, __shfl_xor_sync(0xffffffffu, mxx, o));
            mxy = fmaxf(mxy, __shfl_xor_sync(0xffffffffu, mxy, o));
            mxz = fmaxf(mxz, __shfl_xor_sync(0xffffffffu, mxz, o));
        }
        if ((threadIdx.x & 31) == 0) {
            atomicMin(&bbox[b * 6 + 0], f2ord(mnx)); atomicMin(&bbox[b * 6 + 1], f2ord(mny));
            atomicMin(&bbox[b * 6 + 2], f2ord(mnz)); atomicMax(&bbox[b * 6 + 3], f2ord(mxx));
            atomicMax(&bbox[b * 6 + 4], f2ord(mxy)); atomicMax(&bbox[b * 6 + 5], f2ord(mxz));
        }
    } else {
        atomicMin(&bbox[b * 6 + 0], f2ord(x)); atomicMin(&bbox[b * 6 + 1], f2ord(y));
        atomicMin(&bbox[b * 6 + 2], f2ord(z)); atomicMax(&bbox[b * 6 + 3], f2ord(x));
        atomicMax(&bbox[b * 6 + 4], f2ord(y)); atomicMax(&bbox[b * 6 + 5], f2ord(z));
    }
}

// One thread per batch item picks the cell size.  fixed_cs > 0: radius search (cs = radius);
// otherwise the k-NN heuristic: the radius expected to hold k points at the mean surface /
// volume density of the bounding box.  Cells per item are capped at 2*n_b + 64 so that the
// caller can size the cell arrays without a device->host sync.
__global__ void grid_setup_kernel(const unsigned* __restrict__ bbox,
                                  const int64_t* __restrict__ splits, int batch, float fixed_cs,
                                  int k, GridInfo* __restrict__ info, uint32_t* total_cells) {
    if (blockIdx.x != 0 || threadIdx.x != 0) return;
    uint32_t base = 0;
    for (int b = 0; b < batch; ++b) {
        int64_t nb = splits[b + 1] - splits[b];
        GridInfo g;
        if (nb <= 0) {
            g.ox = g.oy = g.oz = 0.f; g.cs = 1.f; g.inv_cs = 1.f; g.dx = g.dy = g.dz = 1;
        } else {
            float mn[3], mx[3], e[3];
            for (int d = 0; d < 3; ++d) {
                mn[d] = ord2f(bbox[b * 6 + d]);
                mx[d] = ord2f(bbox[b * 6 + 3 + d]);
                e[d] = fmaxf(mx[d] - mn[d], 1e-6f);
            }
            float cs = fixed_cs;
            if (!(cs > 0.f)) {
                float e0 = fmaxf(e[0], fmaxf(e[1], e[2]));
                float e2 = fminf(e[0], fminf(e[1], e[2]));
                float e1 = e[0] + e[1] + e[2] - e0 - e2;
                float kk = (float)(k < 4 ? 4 : k);
                float cs2 = sqrtf(kk * e0 * e1 / (3.14159265f * (float)nb));
                float cs3 = cbrtf(kk * e0 * e1 * e2 / (4.18879f * (float)nb));
                cs = fmaxf(fmaxf(cs2, cs3), 1e-6f);
            }
            const double cap = 2.0 * (double)nb + 64.0;
            for (int it = 0; it < 64; ++it) {
                double c = (floor((double)e[0] / cs) + 1) * (floor((double)e[1] / cs) + 1) *
                           (floor((double)e[2] / cs) + 1);
                if (c <= cap) break;
                cs *= 1.26f;
            }
            g.ox = mn[0]; g.oy = mn[1]; g.oz = mn[2];
            g.cs = cs; g.inv_cs = 1.0f / cs;
            g.dx = (int)floor((double)e[0] / cs) + 1;  // same arithmetic as the cap check above
            g.dy = (int)floor((double)e[1] / cs) + 1;
            g.dz = (int)floor((double)e[2] / cs) + 1;
        }
        g.cell_base = base;
        g.pad = 0;
        info[b] = g;
        base += (uint32_t)(g.dx * g.dy * g.dz);
    }
    *total_cells = base;
}

__device__ __forceinline__ void cell_coords(const GridInfo& g, float x, float y, float z, int& cx,
                                            int& cy, int& cz) {
    cx = min(max((int)floorf((x - g.ox) * g.inv_cs), 0), g.dx - 1);
    cy = min(max((int)floorf((y - g.oy) * g.inv_cs), 0), g.dy - 1);
    cz = min(max((int)floorf((z - g.oz) * g.inv_cs), 0), g.dz - 1);
}
__device__ __forceinline__ uint32_t cell_id(const GridInfo& g, int cx, int cy, int cz) {
    return g.cell_base + (uint32_t)((cz * g.dy + cy) * g.dx + cx);
}

__global__ void grid_count_kernel(const float* __restrict__ pts, int64_t n,
                                  const int64_t* __restrict__ splits, int batch,
                                  const GridInfo* __restrict__ info, uint32_t* __restrict__ cell_of,
                                  uint32_t* __restrict__ cell_count) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    int b = batch_of(i, splits, batch);
    GridInfo g = info[b];
    int cx, cy, cz;
    cell_coords(g, pts[3 * i], pts[3 * i + 1], pts[3 * i + 2], cx, cy, cz);
    uint32_t c = cell_id(g, cx, cy, cz);
    cell_of[i] = c;
    atomicAdd(&cell_count[c], 1u);
}

__global__ void grid_fill_kernel(const float* __restrict__ pts, int64_t n,
                                 const uint32_t* __restrict__ cell_of,
                                 const uint32_t* __restrict__ cell_start,
                                 uint32_t* __restrict__ cursor, float4* __restrict__ sorted) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    uint32_t c = cell_of[i];
    uint32_t pos = cell_start[c] + atomicAdd(&cursor[c], 1u);
    sorted[pos] = make_float4(pts[3 * i], pts[3 * i + 1], pts[3 * i + 2], __int_as_float((int)i));
}

// Order in which queries are processed: sort query ids by the support-grid cell they fall in
// (counting sort with atomics; order inside a cell is irrelevant).
__global__ void query_cell_kernel(const float* __restrict__ q, int64_t nq,
                                  const int64_t* __restrict__ qsplits, int batch,
                                  const GridInfo* __restrict__ info, uint32_t* __restrict__ qcell,
                                  uint32_t* __restrict__ qcount) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= nq) return;
    int b = batch_of(i, qsplits, batch);
    GridInfo g = info[b];
    int cx, cy, cz;
    cell_coords(g, q[3 * i], q[3 * i + 1], q[3 * i + 2], cx, cy, cz);
    uint32_t c = cell_id(g, cx, cy, cz);
    qcell[i] = c;
    atomicAdd(&qcount[c], 1u);
}
__global__ void query_order_kernel(int64_t nq, const uint32_t* __restrict__ qcell,
                                   const uint32_t* __restrict__ qstart,
                                   uint32_t* __restrict__ qcursor, uint32_t* __restrict__ order) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= nq) return;
    uint32_t c = qcell[i];
    order[qstart[c] + atomicAdd(&qcursor[c], 1u)] = (uint32_t)i;
}

__device__ __forceinline__ bool nb_less(float da, int ia, float db, int ib) {
    return da < db || (da == db && ia < ib);
}

// ------------------------------------------------------------------- k-NN ----
template <int KMAX>
__global__ void __launch_bounds__(128)
knn_kernel(const float* __restrict__ queries, int64_t nq, const int64_t* __restrict__ qsplits,
           const int64_t* __restrict__ psplits, int batch, const uint32_t* __restrict__ order,
           const GridInfo* __restrict__ info, const uint32_t* __restrict__ cell_start,
           const float4* __restrict__ sorted, int k, void* __restrict__ out_idx, int idx_is64,
           float* __restrict__ out_d2) {
    int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= nq) return;
    const int64_t qi = order ? (int64_t)order[t] : t;
    const int b = batch_of(qi, qsplits, batch);
    const GridInfo g = info[b];
    const float qx = queries[3 * qi], qy = queries[3 * qi + 1], qz = queries[3 * qi + 2];
    float bd[KMAX];
    int bi[KMAX];
#pragma unroll
    for (int j = 0; j < KMAX; ++j) { bd[j] = FLT_MAX; bi[j] = 0x7fffffff; }
    const int64_t nsup = psplits[b + 1] - psplits[b];
    const int kk = (int)(nsup < k ? nsup : k);  // neighbours that exist
    if (kk > 0) {
        int cx, cy, cz;
        cell_coords(g, qx, qy, qz, cx, cy, cz);
        const int rmax = max(max(max(cx, g.dx - 1 - cx), max(cy, g.dy - 1 - cy)), max(cz, g.dz - 1 - cz));
        for (int r = 0; r <= rmax; ++r) {
            const int z0 = max(cz - r, 0), z1 = min(cz + r, g.dz - 1);
            const int y0 = max(cy - r, 0), y1 = min(cy + r, g.dy - 1);
            for (int z = z0; z <= z1; ++z) {
                const bool zface = (z == cz - r) || (z == cz + r);
                for (int y = y0; y <= y1; ++y) {
                    const bool face = zface || (y == cy - r) || (y == cy + r);
                    // on a face row walk every x, otherwise only the two x-caps of the shell
                    const int xs = face ? 1 : max(2 * r, 1);
                    for (int x = cx - r; x <= cx + r; x += xs) {
                        if (x < 0 || x >= g.dx) continue;
                        const uint32_t c = cell_id(g, x, y, z);
                        const uint32_t s = cell_start[c], e = cell_start[c + 1];
                        for (uint32_t pi = s; pi < e; ++pi) {
                            const float4 pt = sorted[pi];
                            const float d = sqdist3(qx, qy, qz, pt.x, pt.y, pt.z);
                            const int id = __float_as_int(pt.w);
                            if (nb_less(d, id, bd[KMAX - 1], bi[KMAX - 1])) {
                                // replace the current worst (slot KMAX-1 holds the worst because
                                // unused slots are +inf) and bubble it up
                                bd[KMAX - 1] = d;
                                bi[KMAX - 1] = id;
#pragma unroll
                                for (int j = KMAX - 1; j > 0; --j) {
                                    if (nb_less(bd[j], bi[j], bd[j - 1], bi[j - 1])) {
                                        float td = bd[j]; bd[j] = bd[j - 1]; bd[j - 1] = td;
                                        int ti = bi[j]; bi[j] = bi[j - 1]; bi[j - 1] = ti;
                                    }
                                }
                            }
                        }
                    }
                }
            }
            // everything closer than r*cs has been seen (cells are >= cs wide, the query sits
            // inside its own cell or outside the grid on the far side); 1e-4 relative slack
            // covers the float rounding of the cell assignment
            const float cover = (float)r * g.cs * 0.9999f;
            float kth = FLT_MAX;  // the k-th best so far sits at slot kk-1 (slots are sorted)
#pragma unroll
            for (int j = 0; j < KMAX; ++j)
                if (j == kk - 1) kth = bd[j];
            if (kth != FLT_MAX && kth <= cover * cover) break;
        }
    }
#pragma unroll
    for (int j = 0; j < KMAX; ++j) {
        if (j < k) {
            const bool have = j < kk;
            if (idx_is64) ((int64_t*)out_idx)[qi * k + j] = have ? (int64_t)bi[j] : -1;
            else ((int32_t*)out_idx)[qi * k + j] = have ? bi[j] : -1;
            if (out_d2) out_d2[qi * k + j] = have ? bd[j] : __int_as_float(0x7f800000);
        }
    }
}

// ----------------------------------------------------------- fixed radius ----
// mode 0: count -> counts[qi]; mode 1: fill rows at row_splits[qi], kept sorted by (d2, idx)
template <int MODE>
__global__ void __launch_bounds__(128)
radius_kernel(const float* __restrict__ queries, int64_t nq, const int64_t* __restrict__ qsplits,
              int batch, const uint32_t* __restrict__ order, const GridInfo* __restrict__ info,
              const uint32_t* __restrict__ cell_start, const float4* __restrict__ sorted,
              float radius, uint32_t* __restrict__ counts, const int64_t* __restrict__ row_splits,
              int32_t* __restrict__ out_idx, float* __restrict__ out_d2) {
    int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= nq) return;
    const int64_t qi = order ? (int64_t)order[t] : t;
    const int b = batch_of(qi, qsplits, batch);
    const GridInfo g = info[b];
    const float qx = queries[3 * qi], qy = queries[3 * qi + 1], qz = queries[3 * qi + 2];
    const float r2 = __fmul_rn(radius, radius);
    // cell box that contains the ball, with slack for the float cell assignment
    const float rr = radius * 1.0001f + 1e-7f;
    int x0 = (int)floorf((qx - rr - g.ox) * g.inv_cs), x1 = (int)floorf((qx + rr - g.ox) * g.inv_cs);
    int y0 = (int)floorf((qy - rr - g.oy) * g.inv_cs), y1 = (int)floorf((qy + rr - g.oy) * g.inv_cs);
    int z0 = (int)floorf((qz - rr - g.oz) * g.inv_cs), z1 = (int)floorf((qz + rr - g.oz) * g.inv_cs);
    // points are clamped into the grid when binned, so clamp the box the same way
    x0 = min(max(x0, 0), g.dx - 1); x1 = min(max(x1, 0), g.dx - 1);
    y0 = min(max(y0, 0), g.dy - 1); y1 = min(max(y1, 0), g.dy - 1);
    z0 = min(max(z0, 0), g.dz - 1); z1 = min(max(z1, 0), g.dz - 1);
    uint32_t cnt = 0;
    int64_t row = 0, cap = 0;
    if (MODE == 1) { row = row_splits[qi]; cap = row_splits[qi + 1] - row; }
    for (int z = z0; z <= z1; ++z)
        for (int y = y0; y <= y1; ++y) {
            const uint32_t c0 = cell_id(g, x0, y, z);
            const uint32_t s = cell_start[c0], e = cell_start[c0 + (uint32_t)(x1 - x0) + 1];
            for (uint32_t pi = s; pi < e; ++pi) {  // x-adjacent cells are contiguous
                const float4 pt = sorted[pi];
                const float d = sqdist3(qx, qy, qz, pt.x, pt.y, pt.z);
                if (d <= r2) {
                    if (MODE == 1 && (int64_t)cnt < cap) {
                        const int id = __float_as_int(pt.w);
                        int64_t j = row + cnt;  // insertion keeps the row sorted
                        while (j > row && nb_less(d, id, out_d2[j - 1], out_idx[j - 1])) {
                            out_idx[j] = out_idx[j - 1];
                            out_d2[j] = out_d2[j - 1];
                            --j;
                        }
                        out_idx[j] = id;
                        out_d2[j] = d;
                    }
                    ++cnt;
                }
            }
        }
    if (MODE == 0) counts[qi] = cnt;
}

__global__ void widen_splits_kernel(const uint32_t* __restrict__ excl, int64_t n,
                                    const uint32_t* __restrict__ total,
                                    int64_t* __restrict__ out, int64_t* __restrict__ total64) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = excl[i];
    if (i == 0) { out[n] = *total; if (total64) *total64 = *total; }
}

struct GridBuf {
    unsigned* bbox; GridInfo* info; uint32_t* total_cells;
    uint32_t *cell_of, *cell_start, *cursor; float4* sorted;
    uint32_t *qcell, *qstart, *qcursor, *order;
    char* scan_tmp;
    int64_t max_cells;
};

static size_t grid_bytes(int64_t np, int64_t nq, int64_t batch) {
    int64_t max_cells = 2 * np + 128 * batch + 64;
    size_t s = 0;
    s += align_up(batch * 6 * 4) + align_up(batch * sizeof(GridInfo)) + align_up(64);
    s += align_up(np * 4) + 2 * align_up((max_cells + 1) * 4) + align_up(np * 16);
    s += align_up(nq * 4) + 2 * align_up((max_cells + 1) * 4) + align_up(nq * 4);
    s += scan_temp_bytes(max_cells + 1);
    return s + 4096;
}

static int grid_carve(Workspace& ws, int64_t np, int64_t nq, int64_t batch, GridBuf* g) {
    g->max_cells = 2 * np + 128 * batch + 64;
    g->bbox = ws.take<unsigned>(batch * 6);
    g->info = ws.take<GridInfo>(batch);
    g->total_cells = ws.take<uint32_t>(16);
    g->cell_of = ws.take<uint32_t>(np);
    g->cell_start = ws.take<uint32_t>(g->max_cells + 1);
    g->cursor = ws.take<uint32_t>(g->max_cells + 1);
    g->sorted = ws.take<float4>(np);
    g->qcell = ws.take<uint32_t>(nq);
    g->qstart = ws.take<uint32_t>(g->max_cells + 1);
    g->qcursor = ws.take<uint32_t>(g->max_cells + 1);
    g->order = ws.take<uint32_t>(nq);
    g->scan_tmp = ws.take<char>(scan_temp_bytes(g->max_cells + 1));
    return ws.ok ? 0 : 1;
}

// builds the support grid and the cell-ordered query permutation
static int grid_build(const float* pts, int64_t np, const int64_t* psplits, const float* q,
                      int64_t nq, const int64_t* qsplits, int batch, float fixed_cs, int k,
                      GridBuf& g, cudaStream_t st) {
    const int T = 256;
    grid_init_kernel<<<ceil_div(batch * 6, T), T, 0, st>>>(g.bbox, batch);
    if (np > 0) grid_bbox_kernel<<<(unsigned)ceil_div<int64_t>(np, T), T, 0, st>>>(pts, np, psplits, batch, g.bbox);
    grid_setup_kernel<<<1, 32, 0, st>>>(g.bbox, psplits, batch, fixed_cs, k, g.info, g.total_cells);
    O3DML_CUDA(cudaMemsetAsync(g.cell_start, 0, (g.max_cells + 1) * 4, st));
    O3DML_CUDA(cudaMemsetAsync(g.cursor, 0, (g.max_cells + 1) * 4, st));
    if (np > 0) grid_count_kernel<<<(unsigned)ceil_div<int64_t>(np, T), T, 0, st>>>(pts, np, psplits, batch, g.info, g.cell_of, g.cell_start);
    O3DML_CUDA(exclusive_scan_u32(g.cell_start, g.cell_start, g.max_cells + 1, nullptr, g.scan_tmp, st));
    if (np > 0) grid_fill_kernel<<<(unsigned)ceil_div<int64_t>(np, T), T, 0, st>>>(pts, np, g.cell_of, g.cell_start, g.cursor, g.sorted);
    if (nq > 0) {
        O3DML_CUDA(cudaMemsetAsync(g.qstart, 0, (g.max_cells + 1) * 4, st));
        O3DML_CUDA(cudaMemsetAsync(g.qcursor, 0, (g.max_cells + 1) * 4, st));
        query_cell_kernel<<<(unsigned)ceil_div<int64_t>(nq, T), T, 0, st>>>(q, nq, qsplits, batch, g.info, g.qcell, g.qstart);
        O3DML_CUDA(exclusive_scan_u32(g.qstart, g.qstart, g.max_cells + 1, nullptr, g.scan_tmp, st));
        query_order_kernel<<<(unsigned)ceil_div<int64_t>(nq, T), T, 0, st>>>(nq, g.qcell, g.qstart, g.qcursor, g.order);
    }
    O3DML_LAUNCH_CHECK();
    o3dml_count_launches(6 + (nq > 0 ? 3 : 0));
    return O3DML_OK;
}

}  // namespace o3dml

using namespace o3dml;

extern "C" size_t o3dml_knn_workspace_bytes(int64_t num_points, int64_t num_queries, int64_t batch) {
    return grid_bytes(num_points, num_queries, batch);
}

extern "C" int o3dml_knn_search(const float* points, int64_t num_points,
                                const int64_t* points_row_splits, const float* queries,
                                int64_t num_queries, const int64_t* queries_row_splits,
                                int64_t batch, int k, void* out_index, int index_is64,
                                float* out_distance2, void* workspace, size_t workspace_bytes,
                                void* stream) {
    cudaStream_t st = (cudaStream_t)stream;
    O3DML_CHECK(k >= 1 && k <= 64, "knn_search: k must be in 1..64 (got %d)", k);
    O3DML_CHECK(batch >= 1 && num_points >= 0 && num_queries >= 0, "knn_search: bad sizes");
    O3DML_CHECK(num_points < ((int64_t)1 << 30), "knn_search: too many points");
    if (num_queries == 0) return O3DML_OK;
    Workspace ws(workspace, workspace_bytes);
    GridBuf g;
    if (grid_carve(ws, num_points, num_queries, batch, &g))
        O3DML_FAIL(O3DML_ERR_WORKSPACE, "knn_search: workspace too small (%zu needed)", ws.off);
    int rc = grid_build(points, num_points, points_row_splits, queries, num_queries,
                        queries_row_splits, (int)batch, 0.f, k, g, st);
    if (rc) return rc;
    const unsigned nb = (unsigned)ceil_div<int64_t>(num_queries, 128);
#define KNN_LAUNCH(KM)                                                                           \
    knn_kernel<KM><<<nb, 128, 0, st>>>(queries, num_queries, queries_row_splits, points_row_splits, \
                                       (int)batch, g.order, g.info, g.cell_start, g.sorted, k,    \
                                       out_index, index_is64, out_distance2)
    if (k == 1) KNN_LAUNCH(1);
    else if (k <= 8) KNN_LAUNCH(8);
    else if (k <= 16) KNN_LAUNCH(16);
    else if (k <= 32) KNN_LAUNCH(32);
    else KNN_LAUNCH(64);
#undef KNN_LAUNCH
    O3DML_LAUNCH_CHECK();
    o3dml_count_launches(1);
    return O3DML_OK;
}

extern "C" size_t o3dml_radius_workspace_bytes(int64_t num_points, int64_t num_queries,
                                               int64_t batch) {
    return grid_bytes(num_points, num_queries, batch) + align_up((num_queries + 1) * 4) +
           scan_temp_bytes(num_queries + 1) + 1024;
}

// Phase 1: builds the grid (kept in the workspace for phase 2) and writes
// neighbors_row_splits int64 [Nq+1] plus the total (device int64).
extern "C" int o3dml_radius_count(const float* points, int64_t num_points,
                                  const int64_t* points_row_splits, const float* queries,
                                  int64_t num_queries, const int64_t* queries_row_splits,
                                  int64_t batch, float radius, int64_t* neighbors_row_splits,
                                  int64_t* d_total, void* workspace, size_t workspace_bytes,
                                  void* stream) {
    cudaStream_t st = (cudaStream_t)stream;
    O3DML_CHECK(radius > 0.f, "fixed_radius_search: radius must be positive");
    O3DML_CHECK(batch >= 1 && num_points >= 0 && num_queries >= 0, "fixed_radius_search: bad sizes");
    O3DML_CHECK(num_points < ((int64_t)1 << 30), "fixed_radius_search: too many points");
    Workspace ws(workspace, workspace_bytes);
    GridBuf g;
    int bad = grid_carve(ws, num_points, num_queries, batch, &g);
    uint32_t* counts = ws.take<uint32_t>(num_queries + 1);
    char* scan_tmp = ws.take<char>(scan_temp_bytes(num_queries + 1));
    uint32_t* total = ws.take<uint32_t>(16);
    if (bad || !ws.ok)
        O3DML_FAIL(O3DML_ERR_WORKSPACE, "fixed_radius_search: workspace too small (%zu needed)", ws.off);
    if (num_queries == 0) {
        O3DML_CUDA(cudaMemsetAsync(neighbors_row_splits, 0, sizeof(int64_t), st));
        if (d_total) O3DML_CUDA(cudaMemsetAsync(d_total, 0, sizeof(int64_t), st));
        return O3DML_OK;
    }
    int rc = grid_build(points, num_points, points_row_splits, queries, num_queries,
                        queries_row_splits, (int)batch, radius, 0, g, st);
    if (rc) return rc;
    const unsigned nb = (unsigned)ceil_div<int64_t>(num_queries, 128);
    radius_kernel<0><<<nb, 128, 0, st>>>(queries, num_queries, queries_row_splits, (int)batch, g.order,
                                         g.info, g.cell_start, g.sorted, radius, counts, nullptr,
                                         nullptr, nullptr);
    O3DML_CUDA(exclusive_scan_u32(counts, counts, num_queries, total, scan_tmp, st));
    widen_splits_kernel<<<(unsigned)ceil_div<int64_t>(num_queries, 256), 256, 0, st>>>(
        counts, num_queries, total, neighbors_row_splits, d_total);
    O3DML_LAUNCH_CHECK();
    o3dml_count_launches(3);
    return O3DML_OK;
}

// Phase 2: same workspace (untouched since phase 1), fills the rows.
extern "C" int o3dml_radius_fill(const float* queries, int64_t num_points, int64_t num_queries,
                                 const int64_t* queries_row_splits, int64_t batch, float radius,
                                 const int64_t* neighbors_row_splits, int32_t* neighbors_index,
                                 float* neighbors_distance2, void* workspace,
                                 size_t workspace_bytes, void* stream) {
    cudaStream_t st = (cudaStream_t)stream;
    if (num_queries == 0) return O3DML_OK;
    Workspace ws(workspace, workspace_bytes);
    GridBuf g;
    if (grid_carve(ws, num_points, num_queries, batch, &g))
        O3DML_FAIL(O3DML_ERR_WORKSPACE, "fixed_radius_search: workspace too small");
    O3DML_CHECK(neighbors_index != nullptr && neighbors_distance2 != nullptr,
                "fixed_radius_search: index and distance outputs are both required");
    const unsigned nb = (unsigned)ceil_div<int64_t>(num_queries, 128);
    radius_kernel<1><<<nb, 128, 0, st>>>(queries, num_queries, queries_row_splits, (int)batch, g.order,
                                         g.info, g.cell_start, g.sorted, radius, nullptr,
                                         neighbors_row_splits, neighbors_index, neighbors_distance2);
    O3DML_LAUNCH_CHECK();
    o3dml_count_launches(1);
    return O3DML_OK;
}

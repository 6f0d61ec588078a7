"""ctypes binding of libo3dml_b200.so (the C ABI declared in include/o3dml_b200.h).

There is NO CPU fallback: every entry point needs the CUDA library and a CUDA
device, and fails loudly otherwise.
"""
import ctypes
import math
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "libo3dml_b200.so")
_lib = None
ABI_VERSION = 2

c_void_p, c_int, c_int64, c_float, c_size_t = (ctypes.c_void_p, ctypes.c_int, ctypes.c_int64,
                                               ctypes.c_float, ctypes.c_size_t)


class Src(ctypes.Structure):
    """o3dml_src_t"""
    _fields_ = [("data", c_void_p), ("index", c_void_p), ("rows", c_int64),
                ("out_rows_per_batch", c_int64), ("src_rows_per_batch", c_int64),
                ("channels", ctypes.c_int32), ("ld", ctypes.c_int32),
                ("index_is64", ctypes.c_int32), ("index_ld", ctypes.c_int32)]


P, I, L, F, Z = c_void_p, c_int, c_int64, c_float, c_size_t
_SIGNATURES = {
    "o3dml_abi_version": (c_int, []),
    "o3dml_last_error": (ctypes.c_char_p, []),
    "o3dml_launch_count": (ctypes.c_ulonglong, []),
    "o3dml_launch_count_add": (None, [ctypes.c_ulonglong]),
    "o3dml_voxelize_workspace_bytes": (Z, [L, L]),
    "o3dml_voxelize": (I, [P, L, I, P, L, P, P, P, L, L, P, P, P, P, P, P, P, Z, P]),
    "o3dml_ragged_to_dense": (I, [P, I, L, P, L, L, L, L, P, P]),
    "o3dml_knn_workspace_bytes": (Z, [L, L, L]),
    "o3dml_knn_search": (I, [P, L, P, P, L, P, L, I, P, I, P, P, Z, P]),
    "o3dml_radius_workspace_bytes": (Z, [L, L, L]),
    "o3dml_radius_count": (I, [P, L, P, P, L, P, L, F, P, P, P, Z, P]),
    "o3dml_radius_fill": (I, [P, L, L, P, L, F, P, P, P, P, Z, P]),
    "o3dml_voxel_reduce": (I, [P, I, P, I, I, P, P, P, P, L, I, I, P, P, P, P]),
    "o3dml_reduce_subarrays_sum": (I, [P, P, L, P, P]),
    "o3dml_sparse_conv_workspace_bytes": (Z, [L]),
    "o3dml_sparse_conv_neighbors": (I, [P, L, P, L, F, P, P, I, P, P, P, Z, P]),
    "o3dml_continuous_conv": (I, [P, I, I, I, I, I, P, L, P, I, P, P, P, L, P, P, I, P, P, I, I, I, I, P, P]),
    "o3dml_nms_workspace_bytes": (Z, [L]),
    "o3dml_nms": (I, [P, P, L, F, P, P, P, Z, P]),
    "o3dml_iou_matrix": (I, [P, L, P, L, I, P, P]),
    "o3dml_pp_pfn_scatter": (I, [P, I, I, P, P, P, P, P, L, P, P, P, I, F, F, F, F, I, I, I, P, P,
                                 I, P]),
    "o3dml_linear": (I, [L, ctypes.POINTER(Src), I, P, P, P, P, I, I, F, P, I, I, I, P]),
    "o3dml_conv3x3_nhwc": (I, [P, I, I, I, I, I, P, P, P, I, F, P, I, P]),
    "o3dml_deconv_nhwc": (I, [P, I, I, I, I, I, P, P, P, I, F, P, I, I, P]),
    "o3dml_linear_tc_supported": (I, [ctypes.POINTER(Src), I]),
    "o3dml_linear_tc": (I, [L, ctypes.POINTER(Src), I, P, I, I, P, P, P, I, I, F, P, I, I, I, P]),
    "o3dml_conv3x3_nhwc_tc": (I, [P, I, I, I, I, I, P, I, I, P, P, I, F, P, I, P]),
    "o3dml_deconv_nhwc_tc": (I, [P, I, I, I, I, I, P, I, I, P, P, I, F, P, I, I, P]),
    "o3dml_randla_lfa_pool": (I, [I, I, P, P, I, I, P, L, L, P, P, P, P, P, P, P, P, P, P]),
    "o3dml_linear_rows_small_supported": (I, [I, I, I]),
    "o3dml_linear_rows_small": (I, [L, P, I, P, P, P, I, F, P, I, I, P]),
    "o3dml_randla_lfa16_pool": (I, [I, P, P, I, I, P, L, L, P, P, P]),
    "o3dml_randla_lfa_pool_tc": (I, [I, I, P, P, I, I, P, L, L, P, P, P, P, P, P, P, P, P, P]),
    "o3dml_randla_tail_supported": (I, [I, I, I, I, I, I]),
    "o3dml_randla_tail": (I, [P, I, P, I, L, P, I, L, L, L, P, P, P, F, I, P, P]),
    "o3dml_gather_max": (I, [P, L, I, I, P, I, L, I, L, L, I, P, I, P]),
    "o3dml_kpconv_gather": (I, [P, L, P, L, P, I, I, P, I, P, I, F, P, P]),
}
EXPORTS = tuple(_SIGNATURES)           # the product ABI: exactly what include/o3dml_b200.h declares
# bring-up / profiling hooks (include/o3dml_b200_bringup.h): exported by the library, not part of the product ABI
_BRINGUP_SIGNATURES = {
    "o3dml_tc_gemm_test": (I, [P, P, P, I, I, I, P]),
    "o3dml_tc_mma_rate": (I, [I, I, P, P]),
}


def lib():
    """Loads (building first if the .so is absent and nvcc is available)."""
    global _lib
    if _lib is None:
        from . import build as _build
        have_nvcc = os.path.exists(_build.NVCC)
        if have_nvcc or not os.path.exists(LIB_PATH):
            # build() is a cheap mtime check when the library is current: an edited csrc/ or header is never
            # served by a stale .so; without nvcc an existing library is used as it is
            try:
                _build.build()
            except Exception as e:  # noqa: BLE001
                if not os.path.exists(LIB_PATH):
                    raise RuntimeError(
                        "open3d_ml_b200: CUDA library %s is missing and could not be built (%s). "
                        "There is no CPU fallback." % (LIB_PATH, e)) from e
                raise
        h = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in list(_SIGNATURES.items()) + list(_BRINGUP_SIGNATURES.items()):
            fn = getattr(h, name)
            fn.restype, fn.argtypes = res, args
        if h.o3dml_abi_version() != ABI_VERSION:
            raise RuntimeError("open3d_ml_b200: ABI version mismatch")
        _lib = h
    return _lib


def check(rc):
    if rc != 0:
        raise RuntimeError("open3d_ml_b200: " + lib().o3dml_last_error().decode())


def require_cuda():
    if not torch.cuda.is_available():
        raise RuntimeError("open3d_ml_b200: no CUDA device visible; this library has no CPU path")


def ptr(t):
    return None if t is None else t.data_ptr()


def stream():
    return torch.cuda.current_stream().cuda_stream


def act_code(act):
    return {None: 0, "none": 0, "relu": 1, "leaky": 2}[act]


def make_src(data, index=None, index_ld=1, out_rows_per_batch=0, src_rows_per_batch=0,
             channels=None, ld=None, rows=None):
    """data: 2-D float32 CUDA tensor [rows, C] (row stride ld)."""
    s = Src()
    s.data = data.data_ptr()
    s.rows = data.shape[0] if rows is None else rows
    s.channels = data.shape[1] if channels is None else channels
    s.ld = data.stride(0) if ld is None else ld
    if index is not None:
        assert index.dtype in (torch.int64, torch.int32) and index.is_cuda
        s.index = index.data_ptr()
        s.index_is64 = 1 if index.dtype == torch.int64 else 0
        s.index_ld = index_ld
    s.out_rows_per_batch = out_rows_per_batch
    s.src_rows_per_batch = src_rows_per_batch
    return s


def tf32_round(x):
    """fp32 -> nearest TF32 (10 explicit mantissa bits, ties to even), returned as fp32."""
    u = x.contiguous().view(torch.int32).to(torch.int64) & 0xFFFFFFFF
    u = (u + 0xFFF + ((u >> 13) & 1)) & 0xFFFFE000
    u = torch.where(u >= 2 ** 31, u - 2 ** 32, u)
    return u.to(torch.int32).view(torch.float32)


def pack_tf32_image_host(w_nk):
    """fp32 [N, K] (K contiguous) -> fp32 CPU tensor [2 * N, K]: rows [0, N) = hi = tf32(w),
    rows [N, 2N) = lo = tf32(w - hi).  gemm_tc.cu fetches [BN x 32] boxes of it by TMA."""
    w = w_nk.detach().to(torch.float32).cpu().contiguous()
    hi = tf32_round(w)
    lo = tf32_round(w - hi)
    return torch.cat([hi, lo], 0).contiguous()


def _sw128_tile(b_n32):
    """fp32 [N, 32] (one 128-byte row per output channel) -> the same tile in the K-major SWIZZLE_128B shared-memory
    layout: 16-byte chunk c of row n sits at chunk position c ^ (n & 7)."""
    n = b_n32.shape[0]
    t = b_n32.reshape(n, 8, 4)
    out = torch.empty_like(t)
    rows = torch.arange(n)
    for c in range(8):
        out[rows, c ^ (rows & 7)] = t[:, c]
    return out.reshape(n, 32)


def pack_tail_image(weights_kn, n_pads):
    """rl_tail.cu weight image: for every layer ([K, N] fp32, in x out) the TF32 hi tiles of its 32-wide k-chunks, then the
    lo tiles, each [n_pad][32] floats in the SWIZZLE_128B layout; layers concatenated."""
    parts = []
    for w, n_pad in zip(weights_kn, n_pads):
        w = w.detach().to(torch.float32).cpu()
        k, n = w.shape
        assert k % 32 == 0 and n <= n_pad
        b = torch.zeros((n_pad, k), dtype=torch.float32)
        b[:n] = w.t()
        hi = tf32_round(b)
        lo = tf32_round(b - hi)
        for img in (hi, lo):
            for c in range(k // 32):
                parts.append(_sw128_tile(img[:, 32 * c:32 * c + 32].contiguous()).reshape(-1))
    return torch.cat(parts).contiguous()


class PackedWeight:
    """A dense-layer weight in both forms: fp32 [K, Cout] for the SIMT kernel (gemm.cu) and the
    zero-padded TF32 hi/lo image [2 * n_pad, k_pad] for the tcgen05 kernel (gemm_tc.cu)."""

    def __init__(self, w_kc):
        w = w_kc.detach().to(torch.float32).cpu().contiguous()
        self.k, self.cout = w.shape
        self.wt = w.cuda()
        self.k_pad = (self.k + 31) // 32 * 32
        self.n_pad = 32 if self.cout <= 32 else 64 if self.cout <= 64 else (self.cout + 127) // 128 * 128
        wp = torch.zeros((self.n_pad, self.k_pad), dtype=torch.float32)
        wp[:self.cout, :self.k] = w.t()
        self.img = pack_tf32_image_host(wp).cuda()
        self.host = w                      # fp32 [K, Cout] on the host: rowmlp.cu takes it by value
        self._host_affine = {}

    def host_affine(self, scale, shift):
        """Host copies of the folded-BN scale / shift of this layer (made once, at first use).  The cache
        entry keeps the device tensors alive (so their addresses cannot be reused by other tensors) and is
        keyed by their version counters (an in-place update invalidates it)."""
        def k(t):
            return (0, 0) if t is None else (t.data_ptr(), t._version)
        key = (k(scale), k(shift))
        ent = self._host_affine.get(key)
        if ent is None:
            ent = (None if scale is None else scale.detach().float().cpu().contiguous(),
                   None if shift is None else shift.detach().float().cpu().contiguous(), scale, shift)
            if len(self._host_affine) > 8:      # a layer has one (scale, shift) pair; do not grow without bound
                self._host_affine.clear()
            self._host_affine[key] = ent
        return ent[0], ent[1]

    @property
    def shape(self):
        return (self.k, self.cout)


def pack_linear(w_kc):
    return PackedWeight(w_kc)


TC_MIN_K = 64


def _tc_ok(srcs):
    """Tensor-core kernel only where it pays (K >= TC_MIN_K) and where the operand contract of gemm_tc.cu
    holds: every source 4-channel aligned with 16-byte aligned rows, and every source but the last a
    multiple of 32 channels (a 32-channel k-slice never straddles two sources)."""
    if sum(s.channels for s in srcs) < TC_MIN_K:
        return False
    if any(s.channels % 32 for s in srcs[:-1]):
        return False
    return all((s.channels % 4 == 0) and (s.ld % 4 == 0) and (s.data % 16 == 0) for s in srcs)


USE_ROW_MLP = True
# one-thread-per-row layers need rows >= SMs x 256 x a few to fill the machine: below this the tensor-core kernel
# (128 rows per CTA, K >= TC_MIN_K) has the shorter critical path (1 cloud per GPU: 11 264 rows = 44 CTAs, 25 us
# against ~10 us; profiles/r02_launches_randlanet_1cloud.md)
ROW_MLP_MIN_ROWS = 40000


def _rows_small_ok(srcs, out, ld, co):
    """Alignment contract of rowmlp.cu: float4 access wherever a width is a multiple of 4."""
    for s in srcs:
        if s.channels % 4 == 0 and (s.ld % 4 or s.data % 16):
            return False
    return not (co % 4 == 0 and (ld % 4 or out.data_ptr() % 16))


def linear(srcs, weight, out, scale=None, shift=None, residual=None, act=None, slope=0.0,
           num_rows=None, out_channels=None, out_ld=None, out_nchw_plane=0):
    """out[n,:] = act(scale * (concat(srcs)[n] @ W) + shift + residual[n]).  `weight` is either an
    fp32 [K, Cout] tensor (SIMT kernel) or a PackedWeight (tensor-core kernel when the sources
    allow it)."""
    arr = (Src * len(srcs))(*srcs)
    n = out.shape[0] if num_rows is None else num_rows
    packed = isinstance(weight, PackedWeight)
    wt = weight.wt if packed else weight
    co = wt.shape[1] if out_channels is None else out_channels
    ld = (out.stride(0) if out_nchw_plane == 0 else co) if out_ld is None else out_ld
    res_ld = residual.stride(0) if residual is not None else 0
    prefer_tc = packed and n < ROW_MLP_MIN_ROWS and _tc_ok(srcs)
    if (packed and USE_ROW_MLP and not prefer_tc and residual is None and out_nchw_plane == 0 and len(srcs) <= 2 and
            lib().o3dml_linear_rows_small_supported(srcs[0].channels, srcs[1].channels if len(srcs) == 2 else 0,
                                                    co) and _rows_small_ok(srcs, out, ld, co)):
        hs, ht = weight.host_affine(scale, shift)
        check(lib().o3dml_linear_rows_small(n, arr, len(srcs), weight.host.data_ptr(), ptr(hs), ptr(ht),
                                            act_code(act), float(slope), ptr(out), ld, co, stream()))
    elif packed and _tc_ok(srcs):
        check(lib().o3dml_linear_tc(n, arr, len(srcs), ptr(weight.img), weight.k_pad, weight.n_pad,
                                    ptr(scale), ptr(shift), ptr(residual), res_ld, act_code(act),
                                    float(slope), ptr(out), ld, co, out_nchw_plane, stream()))
    else:
        check(lib().o3dml_linear(n, arr, len(srcs), ptr(wt), ptr(scale), ptr(shift), ptr(residual),
                                 res_ld, act_code(act), float(slope), ptr(out), ld, co, out_nchw_plane,
                                 stream()))
    return out


def graph_replay(cache, key, thunk, device):
    """Runs thunk() by replaying a CUDA graph captured at the first call with `key`, and returns clones of its
    outputs (a tensor or a tuple of tensors), since the next replay overwrites the graph's own.  thunk must not
    synchronise with the host and must reuse its buffers from call to call; key must identify every input address.

    The first call runs thunk() eagerly once: that sizes the cached buffers and makes the one-time
    cudaFuncSetAttribute calls, neither of which may happen under stream capture.  Then the whole device is
    synchronised, so that no work of it is in flight while capturing (capturing while the previous batch's all_gather
    was still running faulted with an illegal address in multi-GPU runs, DESIGN.md section 6), and the capture is
    thread_local, so that CUDA calls of other threads do not invalidate it.  The cache is emptied when it holds more
    than 8 graphs."""
    ent = cache.get(key)
    if ent is None:
        thunk()
        torch.cuda.synchronize(device)
        graph = torch.cuda.CUDAGraph()
        n0 = lib().o3dml_launch_count()
        with torch.cuda.graph(graph, capture_error_mode="thread_local"):
            out = thunk()
        if len(cache) > 8:
            cache.clear()
        ent = cache[key] = (graph, out, lib().o3dml_launch_count() - n0)
    graph, out, launches = ent
    graph.replay()
    lib().o3dml_launch_count_add(launches)
    return tuple(o.clone() for o in out) if isinstance(out, tuple) else out.clone()


def pack_operand_image_host(w_nk):
    """fp32 [N, K] (K contiguous, i.e. nn.Linear's [out, in]) -> uint8 CPU tensor holding the
    3xFP16 operand images of csrc/tc.cuh: [K/8][N][8 halves] of hi = fp16(w), then the same
    layout of lo = fp16(w - hi)."""
    w = w_nk.detach().to(torch.float32).cpu().clamp(-65504.0, 65504.0)
    n, k = w.shape
    assert k % 8 == 0 and n % 8 == 0
    hi = w.to(torch.float16)
    lo = (w - hi.to(torch.float32)).to(torch.float16)

    def img(h):
        return h.view(n, k // 8, 8).permute(1, 0, 2).contiguous().view(-1)
    return torch.cat([img(hi), img(lo)]).view(torch.uint8)


def pack_operand_image(w_nk):
    """pack_operand_image_host, moved to the device."""
    return pack_operand_image_host(w_nk).cuda()

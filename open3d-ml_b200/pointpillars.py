"""PointPillars forward on the sm_100a kernels: the fused replacement of
``PointPillars.forward`` (ml3d/torch/models/point_pillars.py:102-134):

    voxelize (all frames in ONE batched call, no per-frame Python loop, :112-128, :328-382)
    -> pillar gather + decoration + PFN + max + scatter-to-BEV in one kernel (:417-616),
       reading the CSR voxel lists directly (the [M,32,4] pillar tensor never exists)
    -> SECOND / SECONDFPN / Anchor3DHead as NHWC implicit-GEMM convolutions (:619-841)

No device->host synchronisation happens inside forward(): the voxel count stays on
the device (the reference syncs at :106 and once per frame inside the op).
The dense part (20 launches of 20-60 us each at one KITTI frame) is launch-bound from
Python, so it is captured once per canvas shape into a CUDA graph and replayed
(`use_graph=False` keeps the eager launches).
Built from a reference ``state_dict``; returns (cls, reg, dir) in NCHW like the
reference head.
"""
import numpy as np
import torch

from . import _lib as L
from . import ops

BN_EPS = 1e-3  # point_pillars.py:409,648,724


def _fold_bn(sd, prefix, eps=BN_EPS):
    s = sd[prefix + ".weight"].double() / torch.sqrt(sd[prefix + ".running_var"].double() + eps)
    t = sd[prefix + ".bias"].double() - s * sd[prefix + ".running_mean"].double()
    return s.float(), t.float()


class PointPillarsB200:
    """cfg keys: point_cloud_range, voxel_size, max_num_points, max_voxels (eval value),
    output_shape [ny, nx], layer_nums, layer_strides, upsample_strides."""

    def __init__(self, state_dict, cfg, device=None, use_graph=True):
        L.require_cuda()
        self.use_graph = bool(use_graph)
        self._graphs = {}
        self.device = dev = torch.device(device or "cuda")
        self.cfg = cfg
        sd = {k: v.detach().to("cpu", torch.float32) if v.is_floating_point() else v.cpu()
              for k, v in state_dict.items()}
        w = self.w = {}

        def put(name, t):
            w[name] = t.to(dev, torch.float32).contiguous()

        # PFN (single layer): linear.weight [64, C+5]
        lw = sd["voxel_encoder.pfn_layers.0.linear.weight"]
        if "voxel_encoder.pfn_layers.1.linear.weight" in sd:
            raise RuntimeError("PointPillarsB200: only single-layer PillarFeatureNet is fused")
        self.pfn_out = lw.shape[0]
        self.point_channels = lw.shape[1] - 5
        put("pfn.wt", lw.t())
        s, t = _fold_bn(sd, "voxel_encoder.pfn_layers.0.norm")
        put("pfn.s", s), put("pfn.t", t)
        # backbone
        self.blocks = []
        for i, (n, stride) in enumerate(zip(cfg["layer_nums"], cfg["layer_strides"])):
            p = "backbone.blocks.%d" % i
            layers = [(p + ".0", p + ".1", stride)]
            layers += [("%s.%d" % (p, 3 + 3 * j), "%s.%d" % (p, 4 + 3 * j), 1) for j in range(n)]
            for conv, bn, st in layers:
                cw = sd[conv + ".weight"]  # [co, ci, 3, 3]
                w[conv + ".wt"] = L.pack_linear(cw.permute(2, 3, 1, 0).reshape(9 * cw.shape[1], cw.shape[0]))
                s, t = _fold_bn(sd, bn)
                put(conv + ".s", s), put(conv + ".t", t)
            self.blocks.append([(c, st, sd[c + ".weight"].shape[1], sd[c + ".weight"].shape[0])
                                for c, _, st in layers])
        # neck
        self.deblocks = []
        for i, us in enumerate(cfg["upsample_strides"]):
            p = "neck.deblocks.%d" % i
            dw = sd[p + ".0.weight"]  # ConvTranspose2d [ci, co, k, k]
            if dw.shape[2] != us or dw.shape[3] != us:
                raise RuntimeError("PointPillarsB200: deblock kernel must equal its stride")
            co = dw.shape[1]
            w[p + ".wt"] = L.pack_linear(dw.permute(0, 2, 3, 1).reshape(dw.shape[0], us * us * co))
            s, t = _fold_bn(sd, p + ".1")
            put(p + ".s", s.repeat(us * us)), put(p + ".t", t.repeat(us * us))
            self.deblocks.append((p, us, dw.shape[0], co))
        self.neck_channels = sum(d[3] for d in self.deblocks)
        # head: three 1x1 convs as one GEMM
        hw = [sd["bbox_head.%s.weight" % h][:, :, 0, 0] for h in ("conv_cls", "conv_reg", "conv_dir_cls")]
        hb = [sd["bbox_head.%s.bias" % h] for h in ("conv_cls", "conv_reg", "conv_dir_cls")]
        self.head_split = [x.shape[0] for x in hw]
        w["head.wt"] = L.pack_linear(torch.cat(hw, 0).t())
        put("head.t", torch.cat(hb, 0))
        r = cfg["point_cloud_range"]
        self.vx, self.vy = float(cfg["voxel_size"][0]), float(cfg["voxel_size"][1])
        # same float64->float32 path as PillarFeatureNet.__init__ (:506-509)
        self.x_off = float(self.vx / 2 + r[0])
        self.y_off = float(self.vy / 2 + r[1])
        self.ny, self.nx = cfg["output_shape"]
        self._buf = {}

    def _get(self, name, shape, dtype=torch.float32):
        key = (name, tuple(shape), dtype)
        t = self._buf.get(key)
        if t is None:
            t = torch.empty(shape, dtype=dtype, device=self.device)
            self._buf[key] = t
        return t

    # ------------------------------------------------------------- front end
    def front_end(self, frames, want_feat=False, canvas_nchw=False):
        """frames: list of [N_i, C] float32 tensors (CPU or CUDA).  Returns the zero-initialised
        canvas with the pillar features scattered, plus the raw voxel buffers."""
        cfg, dev = self.cfg, self.device
        B = len(frames)
        pts = torch.cat([f.to(dev, non_blocking=True) for f in frames], 0).contiguous()
        lens = [0] + [int(f.shape[0]) for f in frames]
        rs = torch.tensor(np.cumsum(lens), dtype=torch.int64).to(dev, non_blocking=True)
        r = cfg["point_cloud_range"]
        coords, pidx, vrs, bsp, bid, counts = ops.voxelize_raw(
            pts[:, :3], rs, cfg["voxel_size"], r[:3], r[3:], cfg["max_num_points"],
            cfg["max_voxels"], want_batch_id=True)
        C = self.pfn_out
        shape = (B, C, self.ny, self.nx) if canvas_nchw else (B, self.ny, self.nx, C)
        canvas = self._get("canvas", shape)
        canvas.zero_()
        bound = min(pts.shape[0], B * int(cfg["max_voxels"]))
        feat = torch.empty((bound, C), dtype=torch.float32, device=dev) if want_feat else None
        L.check(L.lib().o3dml_pp_pfn_scatter(
            L.ptr(pts), pts.stride(0), self.point_channels, L.ptr(coords), L.ptr(vrs), L.ptr(pidx),
            L.ptr(bid), L.ptr(counts), bound, L.ptr(self.w["pfn.wt"]), L.ptr(self.w["pfn.s"]),
            L.ptr(self.w["pfn.t"]), C, self.vx, self.vy, self.x_off, self.y_off, self.nx, self.ny,
            int(cfg["max_num_points"]), L.ptr(feat), L.ptr(canvas), 1 if canvas_nchw else 0,
            L.stream()))
        return canvas, dict(coords=coords, point_indices=pidx, row_splits=vrs, batch_splits=bsp,
                            batch_id=bid, counts=counts, feat=feat, points=pts)

    # ---------------------------------------------------------- dense layers
    def _conv(self, x, B, H, W, name, stride, cin, cout):
        OH, OW = (H - 1) // stride + 1, (W - 1) // stride + 1
        out = self._get(name, (B, OH, OW, cout))
        pw = self.w[name + ".wt"]
        if cin % 32 == 0:
            L.check(L.lib().o3dml_conv3x3_nhwc_tc(L.ptr(x), B, H, W, cin, stride, L.ptr(pw.img), pw.k_pad,
                                                  pw.n_pad, L.ptr(self.w[name + ".s"]),
                                                  L.ptr(self.w[name + ".t"]), 1, 0.0, L.ptr(out), cout,
                                                  L.stream()))
        else:
            L.check(L.lib().o3dml_conv3x3_nhwc(L.ptr(x), B, H, W, cin, stride, L.ptr(pw.wt),
                                               L.ptr(self.w[name + ".s"]), L.ptr(self.w[name + ".t"]),
                                               1, 0.0, L.ptr(out), cout, L.stream()))
        return out, OH, OW

    def backbone_neck_head(self, canvas):
        """SECOND + SECONDFPN + Anchor3DHead on the NHWC canvas -> (cls, reg, dir) in NCHW."""
        if not self.use_graph:
            return self._bnh_eager(canvas)
        return L.graph_replay(self._graphs, (canvas.data_ptr(), tuple(canvas.shape)),
                              lambda: self._bnh_eager(canvas), self.device)

    def _bnh_eager(self, canvas):
        B, H, W = canvas.shape[0], canvas.shape[1], canvas.shape[2]
        x = canvas
        feats = []
        for layers in self.blocks:
            for name, stride, cin, cout in layers:
                x, H, W = self._conv(x, B, H, W, name, stride, cin, cout)
            feats.append((x, H, W))
        us0 = self.deblocks[0][1]
        OH, OW = feats[0][1] * us0, feats[0][2] * us0
        neck = self._get("neck", (B, OH, OW, self.neck_channels))
        off = 0
        for (p, us, cin, co), (f, h, w_) in zip(self.deblocks, feats):
            if h * us != OH or w_ * us != OW:
                raise RuntimeError("PointPillarsB200: neck scales do not line up")
            pw = self.w[p + ".wt"]
            if cin % 4 == 0:
                L.check(L.lib().o3dml_deconv_nhwc_tc(L.ptr(f), B, h, w_, cin, us, L.ptr(pw.img), pw.k_pad,
                                                     pw.n_pad, L.ptr(self.w[p + ".s"]), L.ptr(self.w[p + ".t"]),
                                                     1, 0.0, neck.data_ptr() + 4 * off, self.neck_channels,
                                                     co, L.stream()))
            else:
                L.check(L.lib().o3dml_deconv_nhwc(L.ptr(f), B, h, w_, cin, us, L.ptr(pw.wt),
                                                  L.ptr(self.w[p + ".s"]), L.ptr(self.w[p + ".t"]), 1, 0.0,
                                                  neck.data_ptr() + 4 * off, self.neck_channels, co,
                                                  L.stream()))
            off += co
        ch = sum(self.head_split)
        out = torch.empty((B, ch, OH, OW), dtype=torch.float32, device=self.device)
        L.linear([L.make_src(neck.view(B * OH * OW, self.neck_channels))], self.w["head.wt"], out,
                 None, self.w["head.t"], act=None, num_rows=B * OH * OW, out_channels=ch,
                 out_nchw_plane=OH * OW)
        a, b_, _ = self.head_split
        return out[:, :a], out[:, a:a + b_], out[:, a + b_:]

    def forward(self, frames):
        if hasattr(frames, "point"):
            frames = frames.point
        canvas, _ = self.front_end(frames)
        return self.backbone_neck_head(canvas)

    __call__ = forward


def cfg_from_reference(model_cfg):
    """Builds the cfg dict from a reference yml `model:` section (pointpillars_kitti.yml:7-66)."""
    return dict(point_cloud_range=list(model_cfg["point_cloud_range"]),
                voxel_size=list(model_cfg["voxelize"]["voxel_size"]),
                max_num_points=model_cfg["voxelize"]["max_num_points"],
                max_voxels=model_cfg["voxelize"]["max_voxels"][1],
                output_shape=list(model_cfg["scatter"]["output_shape"]),
                layer_nums=list(model_cfg["backbone"]["layer_nums"]),
                layer_strides=list(model_cfg["backbone"]["layer_strides"]),
                upsample_strides=list(model_cfg["neck"]["upsample_strides"]))

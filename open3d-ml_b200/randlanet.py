"""RandLA-Net forward on the sm_100a kernels: the fused replacement of
``RandLANet.forward`` (ml3d/torch/models/randlanet.py:241-298) and of the layers it
calls (SharedMLP :471-518, LocalSpatialEncoding :521-605, AttentivePooling :608-639,
LocalFeatureAggregation :642-692, random_sample :300-327, nearest_interpolation
:329-350).

The module is built from a reference ``state_dict`` (same keys as the model-zoo
checkpoints), folds the eval-mode BatchNorms, and keeps every activation in
point-major [B*N, C] float32 buffers.  Per LFA block:

    linear(mlp1) -> lfa_pool(stage 1) -> linear(pool1.mlp) -> lfa_pool(stage 2)
    -> linear(pool2.mlp) -> linear([p2 | feat] -> mlp2 + shortcut, LeakyReLU 0.01)
    -> gather_max(random_sample)

Inputs are exactly the reference's ``inputs`` dict (CPU or CUDA tensors, int64
indices); the output is ``[B, N, num_classes]`` like the reference.
"""
import torch

from . import _lib as L

BN_EPS = 1e-6  # randlanet.py:77,499
# d_out values served by the tcgen05 kernel (lfa_tc.cu).  d = 16 stays on the FP32 SIMT kernel: its
# 16x16 score product is too small to pay for the per-tile MMA round trip (0.84 vs 1.23 ms measured);
# d = 512 (fifth encoder of the 5-level configs, a few hundred points) runs on the tiled SIMT kernel (lfa.cu).
TC_DIMS = (32, 64, 128, 256)
SUPPORTED_DIMS = (16, 32, 64, 128, 256, 512)


def _fold_bn(sd, prefix, bias=None, eps=BN_EPS):
    s = sd[prefix + ".weight"].double() / torch.sqrt(sd[prefix + ".running_var"].double() + eps)
    t = sd[prefix + ".bias"].double() - s * sd[prefix + ".running_mean"].double()
    if bias is not None:
        t = t + s * bias.double()
    return s.float(), t.float()


class RandLANetB200:
    def __init__(self, state_dict, num_layers=4, num_neighbors=16, device=None, sub_sampling_ratio=None,
                 use_graph=True):
        L.require_cuda()
        self.sub_sampling_ratio = list(sub_sampling_ratio or [4] * num_layers)
        self.use_graph = bool(use_graph)
        self._graphs = {}
        self._splits = {}
        self.device = torch.device(device or "cuda")
        self.num_layers = num_layers
        self.k = num_neighbors
        sd = {k: v.detach().to("cpu", torch.float32) if v.is_floating_point() else v.cpu()
              for k, v in state_dict.items()}
        self.w = {}
        dev = self.device

        def put(name, t):
            self.w[name] = t.to(dev, torch.float32).contiguous()

        def shared_mlp(p, transpose=False, bn=True, raw=False):
            w = sd[p + ".conv.weight"][:, :, 0, 0]
            w = w if transpose else w.t()
            if raw:      # consumed by the fused LFA kernels as plain fp32 [in, out]
                put(p + ".wt", w)
            else:        # dense layer: fp32 + tensor-core operand image
                self.w[p + ".wt"] = L.pack_linear(w)
            if bn:
                s, t = _fold_bn(sd, p + ".batch_norm", sd[p + ".conv.bias"])
                put(p + ".s", s)
                put(p + ".t", t)
            else:
                put(p + ".t", sd[p + ".conv.bias"])

        self.w["fc0.wt"] = L.pack_linear(sd["fc0.weight"].t())
        s, t = _fold_bn(sd, "bn0", sd["fc0.bias"])
        put("fc0.s", s), put("fc0.t", t)
        self.d_out = []
        for i in range(num_layers):
            p = "encoder.%d" % i
            shared_mlp(p + ".mlp1")
            shared_mlp(p + ".lse1.mlp", raw=True)
            shared_mlp(p + ".lse2.mlp", raw=True)
            shared_mlp(p + ".pool1.mlp")
            shared_mlp(p + ".pool2.mlp")
            for pool in ("pool1", "pool2"):
                put("%s.%s.score.wt" % (p, pool), sd["%s.%s.score_fn.0.weight" % (p, pool)].t())
                put("%s.%s.score.b" % (p, pool), sd["%s.%s.score_fn.0.bias" % (p, pool)])
            d = sd[p + ".pool2.mlp.conv.weight"].shape[0]
            if d not in SUPPORTED_DIMS:
                raise RuntimeError("RandLANetB200: encoder %d has dim_output %d; the fused LFA kernels serve %s"
                                   % (i, d, SUPPORTED_DIMS))
            self.d_out.append(d)
            if d in TC_DIMS:   # tcgen05 path: host-packed fp16 hi/lo operand images ([out][in])
                for pool in ("pool1", "pool2"):
                    self.w["%s.%s.score.img" % (p, pool)] = L.pack_operand_image(
                        sd["%s.%s.score_fn.0.weight" % (p, pool)])
                if d >= 32:
                    self.w[p + ".lse2.mlp.img"] = L.pack_operand_image(sd[p + ".lse2.mlp.conv.weight"][:, :, 0, 0])
            if d == 16:   # lfa16c_kernel: weights travel in the kernel parameter block (HOST memory)
                for stage, pool in ((1, "pool1"), (2, "pool2")):
                    hw = torch.zeros(448, dtype=torch.float32)
                    hw[0:80] = self.w[p + ".lse1.mlp.wt"].cpu().reshape(-1)
                    hw[80:88] = self.w[p + ".lse1.mlp.s"].cpu()
                    hw[88:96] = self.w[p + ".lse1.mlp.t"].cpu()
                    hw[96:160] = self.w[p + ".lse2.mlp.wt"].cpu().reshape(-1)
                    hw[160:168] = self.w[p + ".lse2.mlp.s"].cpu()
                    hw[168:176] = self.w[p + ".lse2.mlp.t"].cpu()
                    hw[176:432] = self.w["%s.%s.score.wt" % (p, pool)].cpu().reshape(-1)
                    hw[432:448] = self.w["%s.%s.score.b" % (p, pool)].cpu()
                    self.w["%s.lfa16.%d" % (p, stage)] = hw.contiguous()
            # mlp2 + shortcut as ONE gemm over [p2 | feat] with the BN scales folded into the rows
            s2, t2 = _fold_bn(sd, p + ".mlp2.batch_norm", sd[p + ".mlp2.conv.bias"])
            ss, ts = _fold_bn(sd, p + ".shortcut.batch_norm", sd[p + ".shortcut.conv.bias"])
            w2 = sd[p + ".mlp2.conv.weight"][:, :, 0, 0] * s2[:, None]
            ws = sd[p + ".shortcut.conv.weight"][:, :, 0, 0] * ss[:, None]
            self.w[p + ".out.wt"] = L.pack_linear(torch.cat([w2.t(), ws.t()], 0))
            put(p + ".out.t", t2 + ts)
        shared_mlp("mlp")
        for i in range(num_layers):
            shared_mlp("decoder.%d" % i, transpose=True)
        shared_mlp("fc1.0")
        shared_mlp("fc1.1")
        shared_mlp("fc1.3", bn=False)
        self.num_classes = sd["fc1.3.conv.weight"].shape[0]
        self.in_channels = sd["fc0.weight"].shape[1]
        self._buf = {}
        # ---- fused tail (rl_tail.cu): last decoder layer + fc1 stack chained through tensor memory
        self.tail = None
        pl = "decoder.%d" % (num_layers - 1)
        wd = sd[pl + ".conv.weight"][:, :, 0, 0]                          # ConvTranspose2d [in, out]
        w0, w1, w3 = (sd["fc1.%d.conv.weight" % j][:, :, 0, 0].t() for j in (0, 1, 3))
        skip_c = 2 * self.d_out[0]
        if L.lib().o3dml_randla_tail_supported(skip_c, wd.shape[0] - skip_c, wd.shape[1], w0.shape[1], w1.shape[1],
                                               self.num_classes):
            img = L.pack_tail_image([wd, w0, w1, w3], [32, 64, 32, 32]).to(dev)
            sc, sh = torch.ones(4, 64), torch.zeros(4, 64)
            for li, name in enumerate((pl, "fc1.0", "fc1.1")):
                s_, t_ = _fold_bn(sd, name + ".batch_norm", sd[name + ".conv.bias"])
                sc[li, :s_.numel()], sh[li, :t_.numel()] = s_, t_
            sh[3, :self.num_classes] = sd["fc1.3.conv.bias"]
            self.tail = (img, sc.contiguous(), sh.contiguous())

    # ------------------------------------------------------------------ buffers
    def _get(self, name, shape, dtype=torch.float32):
        key = (name, tuple(shape), dtype)
        t = self._buf.get(key)
        if t is None:
            t = torch.empty(shape, dtype=dtype, device=self.device)
            self._buf[key] = t
        return t

    def _mlp(self, p, srcs, out, act="leaky", slope=0.2):
        return L.linear(srcs, self.w[p + ".wt"], out, self.w.get(p + ".s"), self.w[p + ".t"],
                        act=act, slope=slope)

    def _lfa_pool(self, stage, d, coords, nidx, feat, B, N, p, agg):
        w = self.w
        pool = "pool1" if stage == 1 else "pool2"
        if d in TC_DIMS:
            L.check(L.lib().o3dml_randla_lfa_pool_tc(
                stage, d, L.ptr(coords), L.ptr(nidx), 1 if nidx.dtype == torch.int64 else 0, self.k,
                L.ptr(feat), B, N, L.ptr(w[p + ".lse1.mlp.wt"]), L.ptr(w[p + ".lse1.mlp.s"]),
                L.ptr(w[p + ".lse1.mlp.t"]),
                L.ptr(w.get(p + ".lse2.mlp.img")) if stage == 2 else None,
                L.ptr(w[p + ".lse2.mlp.wt"]) if stage == 2 else None,
                L.ptr(w[p + ".lse2.mlp.s"]) if stage == 2 else None,
                L.ptr(w[p + ".lse2.mlp.t"]) if stage == 2 else None,
                L.ptr(w["%s.%s.score.img" % (p, pool)]), L.ptr(agg), L.stream()))
            return
        if d == 16:
            L.check(L.lib().o3dml_randla_lfa16_pool(
                stage, L.ptr(coords), L.ptr(nidx), 1 if nidx.dtype == torch.int64 else 0, self.k,
                L.ptr(feat), B, N, w["%s.lfa16.%d" % (p, stage)].data_ptr(), L.ptr(agg), L.stream()))
            return
        L.check(L.lib().o3dml_randla_lfa_pool(
            stage, d, L.ptr(coords), L.ptr(nidx), 1 if nidx.dtype == torch.int64 else 0, self.k,
            L.ptr(feat), B, N, L.ptr(w[p + ".lse1.mlp.wt"]), L.ptr(w[p + ".lse1.mlp.s"]),
            L.ptr(w[p + ".lse1.mlp.t"]),
            L.ptr(w[p + ".lse2.mlp.wt"]) if stage == 2 else None,
            L.ptr(w[p + ".lse2.mlp.s"]) if stage == 2 else None,
            L.ptr(w[p + ".lse2.mlp.t"]) if stage == 2 else None,
            L.ptr(w["%s.%s.score.wt" % (p, pool)]), L.ptr(w["%s.%s.score.b" % (p, pool)]),
            L.ptr(agg), L.stream()))

    # ------------------------------------------------------------------ forward
    def to_device(self, inputs):
        """The H2D step of RandLANet.forward (randlanet.py:254-264)."""
        dev = self.device

        def mv(t):
            return t.to(dev, non_blocking=True).contiguous()
        return dict(features=mv(inputs["features"]),
                    coords=[mv(a) for a in inputs["coords"]],
                    neighbor_indices=[mv(a) for a in inputs["neighbor_indices"]],
                    sub_idx=[mv(a) for a in inputs["sub_idx"]],
                    interp_idx=[mv(a) for a in inputs["interp_idx"]])

    def forward(self, inputs, taps=None):
        inp = self.to_device(inputs)
        feats = inp["features"]
        B, N0, cin = feats.shape
        x = self._get("fc0", (B * N0, self.w["fc0.wt"].shape[1]))
        L.linear([L.make_src(feats.view(B * N0, cin))], self.w["fc0.wt"], x, self.w["fc0.s"],
                 self.w["fc0.t"], act="leaky", slope=0.2)
        skips = []
        for i in range(self.num_layers):
            p = "encoder.%d" % i
            d = self.d_out[i]
            h = d // 2
            coords = inp["coords"][i]
            nidx = inp["neighbor_indices"][i]
            N = coords.shape[1]
            rows = B * N
            cflat = coords.view(rows, 3)
            f1 = self._mlp(p + ".mlp1", [L.make_src(x)], self._get(p + ".f1", (rows, h)))
            agg1 = self._get(p + ".agg1", (rows, d))
            self._lfa_pool(1, d, cflat, nidx, f1, B, N, p, agg1)
            p1 = self._mlp(p + ".pool1.mlp", [L.make_src(agg1)], self._get(p + ".p1", (rows, h)))
            agg2 = self._get(p + ".agg2", (rows, d))
            self._lfa_pool(2, d, cflat, nidx, p1, B, N, p, agg2)
            p2 = self._mlp(p + ".pool2.mlp", [L.make_src(agg2)], self._get(p + ".p2", (rows, d)))
            enc = self._get(p + ".enc", (rows, 2 * d))
            L.linear([L.make_src(p2), L.make_src(x)], self.w[p + ".out.wt"], enc, None,
                     self.w[p + ".out.t"], act="leaky", slope=0.01)
            if taps is not None:
                taps[p + ".pool1"] = p1.view(B, N, h)
                taps[p] = enc.view(B, N, 2 * d)
            sub = inp["sub_idx"][i]
            ns = sub.shape[1]
            pooled = self._get(p + ".sub", (B * ns, 2 * d))
            L.check(L.lib().o3dml_gather_max(L.ptr(enc), rows, 2 * d, 2 * d, L.ptr(sub),
                                             1 if sub.dtype == torch.int64 else 0, B * ns,
                                             sub.shape[2], ns, N, 0, L.ptr(pooled), 2 * d,
                                             L.stream()))
            if i == 0:
                skips.append((enc, N))
            skips.append((pooled, ns))
            x = pooled
        nlast = skips[-1][1]
        x = self._mlp("mlp", [L.make_src(x)], self._get("mlp", x.shape))
        ncoarse = nlast
        use_tail = self.tail is not None and taps is None
        for i in range(self.num_layers):
            skip, nup = skips[-i - 2]
            interp = inp["interp_idx"][-i - 1]  # [B, nup, 1] ids into the coarse level
            p = "decoder.%d" % i
            if use_tail and i == self.num_layers - 1:
                img, sc, sh = self.tail
                logits = torch.empty((B * nup, self.num_classes), dtype=torch.float32, device=self.device)
                iv = interp.view(-1)
                L.check(L.lib().o3dml_randla_tail(
                    L.ptr(skip), skip.stride(0), L.ptr(x), x.stride(0), x.shape[0], L.ptr(iv),
                    1 if iv.dtype == torch.int64 else 0, nup, ncoarse, B * nup, L.ptr(img), sc.data_ptr(), sh.data_ptr(),
                    0.2, self.num_classes, L.ptr(logits), L.stream()))
                return logits.view(B, N0, self.num_classes)
            cout = self.w[p + ".wt"].shape[1]
            out = self._get(p, (B * nup, cout))
            self._mlp(p, [L.make_src(skip),
                          L.make_src(x, index=interp.view(-1), index_ld=1, out_rows_per_batch=nup,
                                     src_rows_per_batch=ncoarse)], out)
            if taps is not None:
                taps[p] = out.view(B, nup, cout)
            x, ncoarse = out, nup
        y = self._mlp("fc1.0", [L.make_src(x)], self._get("fc1.0", (x.shape[0], 64)))
        y = self._mlp("fc1.1", [L.make_src(y)], self._get("fc1.1", (x.shape[0], 32)))
        logits = torch.empty((B * N0, self.num_classes), dtype=torch.float32, device=self.device)
        self._mlp("fc1.3", [L.make_src(y)], logits, act=None)
        return logits.view(B, N0, self.num_classes)

    __call__ = forward

    # ------------------------------------------------------ device-side transform
    def _row_splits(self, B, n):
        key = (B, n)
        t = self._splits.get(key)
        if t is None:
            t = torch.arange(0, (B + 1) * n, n, dtype=torch.int64, device=self.device)
            self._splits[key] = t
        return t

    def _knn(self, points, queries, k, ps, qs, name):
        """o3dml_knn_search into cached int32 buffers (global row ids), no host synchronisation."""
        nq = queries.shape[0]
        idx = self._get(name, (nq, k), torch.int32)
        batch = ps.numel() - 1
        wsb = L.lib().o3dml_knn_workspace_bytes(points.shape[0], nq, batch)
        ws = self._get(name + ".ws", (wsb,), torch.uint8)
        L.check(L.lib().o3dml_knn_search(L.ptr(points), points.shape[0], L.ptr(ps), L.ptr(queries), nq,
                                         L.ptr(qs), batch, k, L.ptr(idx), 0, None, L.ptr(ws), wsb, L.stream()))
        return idx

    def build_pyramid(self, points):
        """The index pyramid of RandLANet.transform (randlanet.py:218-229: per level k-NN of the cloud in
        itself, the first N/ratio points as the sub-sampled cloud, 1-NN of every point in the sub-sampled
        cloud) for a [B, N, 3] CUDA tensor, built on the device with the batched grid k-NN
        (o3dml_knn_search, bit-exact against the oracle).  Indices are int32 GLOBAL row ids of the stacked
        [B*N, ...] buffers (the reference ships int64 batch-relative ids over PCIe: 80 of its 90 MB per
        SemanticKITTI batch), so the batch is presented to forward() as ONE cloud of B*N points:
        sub_idx is the per-cloud prefix of neighbor_indices, nothing is searched twice."""
        B, n, _ = points.shape
        pc = points.to(self.device, torch.float32).contiguous()
        out = dict(coords=[], neighbor_indices=[], sub_idx=[], interp_idx=[])
        for i in range(self.num_layers):
            flat = pc.view(B * n, 3)
            rs = self._row_splits(B, n)
            nb = self._knn(flat, flat, self.k, rs, rs, "pyr.nb.%d" % i)
            ns = n // self.sub_sampling_ratio[i]
            sub = self._get("pyr.sub.%d" % i, (B * ns, 3)).view(B, ns, 3)
            sub.copy_(pc[:, :ns])
            pool = self._get("pyr.pool.%d" % i, (B * ns, self.k), torch.int32)
            pool.view(B, ns, self.k).copy_(nb.view(B, n, self.k)[:, :ns])
            up = self._knn(sub.view(B * ns, 3), flat, 1, self._row_splits(B, ns), rs, "pyr.up.%d" % i)
            out["coords"].append(flat.view(1, B * n, 3))
            out["neighbor_indices"].append(nb.view(1, B * n, self.k))
            out["sub_idx"].append(pool.view(1, B * ns, self.k))
            out["interp_idx"].append(up.view(1, B * n, 1))
            pc, n = sub, ns
        return out

    def forward_points(self, points, features=None):
        """transform + forward from raw clouds: points [B, N, 3] (host or device), features [B, N, C] or
        None (= the coordinates, randlanet.py:204-207).  Only the points (and features) cross PCIe."""
        pts = points.to(self.device, non_blocking=True)
        B, N, _ = pts.shape
        inp = self.build_pyramid(pts)
        feat = pts if features is None else torch.cat([pts, features.to(self.device, non_blocking=True)], -1)
        inp["features"] = feat.reshape(1, B * N, -1)
        return self.forward(inp).view(B, N, self.num_classes)

    # ------------------------------------------------------------- CUDA graph
    def _graphed(self, name, tensors, thunk):
        """Replays thunk() from a CUDA graph captured at first use for these tensor addresses (the
        forward is ~40 launches of 5-60 us: launch-bound from Python at one cloud per GPU).  thunk must
        be sync-free and allocation-stable (cached buffers); the result is cloned."""
        if not self.use_graph:
            return thunk()
        key = (name,) + tuple((t.data_ptr(), tuple(t.shape), t.dtype) for t in tensors)
        return L.graph_replay(self._graphs, key, thunk, self.device)

    def forward_graphed(self, inputs):
        """forward() for DEVICE-resident inputs, replayed from a CUDA graph keyed by their addresses."""
        flat = [inputs["features"]] + [t for k in ("coords", "neighbor_indices", "sub_idx", "interp_idx")
                                       for t in inputs[k]]
        if not all(t.is_cuda for t in flat):
            return self.forward(inputs)
        return self._graphed("forward", flat, lambda: self.forward(inputs))

    def forward_points_graphed(self, points, features=None):
        """forward_points() for DEVICE-resident clouds, replayed from a CUDA graph (pyramid + forward)."""
        if not points.is_cuda or (features is not None and not features.is_cuda):
            return self.forward_points(points, features)
        ts = [points] + ([features] if features is not None else [])
        return self._graphed("forward_points", ts, lambda: self.forward_points(points, features))


def patch_reference_model(model):
    """Drop-in: make an (unmodified) reference ``RandLANet`` instance run its forward on the
    fused CUDA path (keeps preprocess/transform/losses).  BN must be in eval mode."""
    fused = RandLANetB200(model.state_dict(), model.cfg.num_layers, model.cfg.num_neighbors,
                          sub_sampling_ratio=list(model.cfg.sub_sampling_ratio))

    def forward(inputs):
        if model.training:
            raise RuntimeError("open3d_ml_b200: the fused RandLA-Net path is inference-only")
        return fused.forward(inputs)
    model.forward = forward
    return model

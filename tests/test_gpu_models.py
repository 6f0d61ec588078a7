"""Model-level parity of the fused CUDA forwards:
  (a) against the golden fixtures produced by the UNMODIFIED reference classes
      (tests/golden/make_golden.py), weights rebuilt from (manifest, seed);
  (b) against the torch port (oracle/models_torch.py) at the BASELINE.json sizes.
Tolerance: 1e-4 relative to the tensor scale for float features/logits (north_star);
indices bit-exact."""
import numpy as np
import pytest
import torch

from oracle import models_torch as MT, ops as O
from open3d_ml_b200 import synth
import open3d_ml_b200 as M
from conftest import rel_err, elem_err
import helpers as H

pytestmark = pytest.mark.gpu
TOL = 1e-4


# ------------------------------------------------------------------ RandLA-Net
def test_randlanet_vs_golden_reference():
    g = H.golden("randlanet_small.npz")
    sd, _ = H.state_dict("randlanet_semantickitti.manifest.json", g["weight_seed"])
    inp = H.randla_inputs(int(g["B"]), int(g["N"]), int(g["seed0"]))
    net = M.RandLANetB200(sd)
    taps = {}
    out = net(inp, taps=taps)
    for i in range(4):
        for k in ("encoder.%d.pool1" % i, "encoder.%d" % i):
            assert rel_err(H.tap_rows(taps[k], g, k), g["tap." + k]) < TOL, k
    assert out.shape == g["logits"].shape
    assert rel_err(out, g["logits"]) < TOL
    assert elem_err(out, g["logits"]) < 1e-2      # no regression hiding in the small-magnitude logits
    assert torch.equal(out.argmax(-1).cpu(), torch.from_numpy(g["logits"]).argmax(-1))


def test_randlanet_full_size_vs_port_with_gpu_knn_pyramid():
    """SemanticKITTI shape (45 056 pts), B=2; the KNN pyramid itself comes from the CUDA
    knn_search (bit-exact to the oracle, test_gpu_ops.py), then the fused forward is compared
    with the CPU port on identical inputs."""
    def gpu_knn(s, q, k):
        r = M.knn_search(torch.from_numpy(s).cuda(), torch.from_numpy(q).cuda(), k, index_dtype=torch.int64)
        return r.neighbors_index.reshape(len(q), k).cpu().numpy()
    sd, _ = H.state_dict("randlanet_semantickitti.manifest.json", 7)
    inp = H.randla_inputs(2, 45056, 500, knn=gpu_knn)
    ref_nb = O.c_knn(inp["coords"][1][0].numpy(), inp["coords"][1][0].numpy(), 16)[0]
    assert np.array_equal(inp["neighbor_indices"][1][0].numpy(), ref_nb)
    net = M.RandLANetB200(sd)
    out = net(inp)
    torch.set_num_threads(max(torch.get_num_threads(), 8))
    with torch.no_grad():
        ref = MT.randlanet_forward(sd, inp)
    assert out.shape == (2, 45056, 19)
    assert rel_err(out, ref) < TOL
    out2 = net(inp)                                         # buffers are reused: idempotent
    assert torch.equal(out, out2)


def test_randlanet_accepts_cuda_inputs_and_int32_indices():
    sd, _ = H.state_dict("randlanet_semantickitti.manifest.json", 3)
    inp = H.randla_inputs(1, 1024, 40)
    net = M.RandLANetB200(sd)
    a = net(inp)
    inp32 = {k: ([t.cuda().to(torch.int32) if t.dtype == torch.int64 else t.cuda() for t in v]
                 if isinstance(v, list) else v.cuda()) for k, v in inp.items()}
    assert torch.equal(a, net(inp32))


# ---------------------------------------------------------------- PointPillars
def test_pointpillars_vs_golden_reference_kitti():
    g = H.golden("pointpillars_kitti.npz")
    sd, extra = H.state_dict("pointpillars_kitti.manifest.json", g["weight_seed"])
    frames = [torch.from_numpy(synth.lidar_frame(int(g["frame_sizes"][0]), int(g["frame_seeds"][0]))),
              torch.from_numpy(synth.uniform_frame(int(g["frame_sizes"][1]), int(g["frame_seeds"][1])))]
    net = M.PointPillarsB200(sd, extra["cfg"])
    canvas, vox = net.front_end(frames, want_feat=True)
    m = int(vox["counts"][0])
    # index-level parity with the reference's voxelize + post-processing (z,y,x order, batch id first)
    co = torch.cat([vox["batch_id"][:m, None], vox["coords"][:m][:, [2, 1, 0]]], 1).cpu().numpy()
    cnt = (vox["row_splits"][1:m + 1] - vox["row_splits"][:m]).cpu().numpy()
    keep = (co[:, 2] < 496) & (co[:, 3] < 432)
    assert np.array_equal(co[keep], g["coords"]) and np.array_equal(cnt[keep], g["counts"])
    feat = vox["feat"][:m][torch.from_numpy(keep).cuda()]
    assert rel_err(feat[torch.from_numpy(g["pfn_rows"]).cuda()], g["pfn_vals"]) < TOL
    assert abs(canvas.double().sum().item() - float(g["canvas_sum"])) < 1e-5 * float(g["canvas_abs_sum"])
    outs = net.backbone_neck_head(canvas)
    for name, o in zip(("cls", "reg", "dir"), outs):
        assert tuple(o.shape) == tuple(g[name + "_shape"])
        assert rel_err(o.reshape(-1)[torch.from_numpy(g[name + "_idx"]).cuda()], g[name + "_vals"]) < TOL, name


def test_pointpillars_small_full_tensors_and_nchw_canvas():
    g = H.golden("pointpillars_small.npz")
    sd, extra = H.state_dict("pointpillars_kitti.manifest.json", g["weight_seed"])
    cfg = dict(extra["cfg"], point_cloud_range=[0, -10.24, -3, 20.48, 10.24, 1], output_shape=[128, 128])
    f = [torch.from_numpy(synth.lidar_frame(int(g["frame_size"]), int(g["frame_seed"]), tuple(cfg["point_cloud_range"])))]
    net = M.PointPillarsB200(sd, cfg)
    outs = net(f)
    for name, o in zip(("cls", "reg", "dir"), outs):
        assert tuple(o.shape) == tuple(g[name + "_shape"])
        assert rel_err(o.reshape(-1)[torch.from_numpy(g[name + "_idx"]).cuda()], g[name + "_vals"]) < TOL, name
    nhwc = net.front_end(f)[0].clone()
    nchw = net.front_end(f, canvas_nchw=True)[0]            # layout of PointPillarsScatter.forward
    assert torch.equal(nchw, nhwc.permute(0, 3, 1, 2))
    taps = {}
    with torch.no_grad():
        MT.pointpillars_forward(sd, f, cfg, taps=taps)
    assert rel_err(nchw, taps["canvas"]) < TOL


def test_pointpillars_waymo_shape_vs_port():
    sd, extra = H.state_dict("pointpillars_waymo.manifest.json", 11)
    frames = [torch.from_numpy(synth.lidar_frame(60000, 30 + i, synth.WAYMO_RANGE)) for i in range(2)]
    net = M.PointPillarsB200(sd, extra["cfg"])
    outs = net(frames)
    with torch.no_grad():
        ref = MT.pointpillars_forward(sd, frames, extra["cfg"])
    for o, r in zip(outs, ref):
        assert o.shape == r.shape and rel_err(o, r) < TOL


def test_pointpillars_graph_replay_equals_eager_launches():
    """The dense part is replayed from a CUDA graph by default: same bits as the eager launches,
    and results of consecutive calls do not alias."""
    g = H.golden("pointpillars_small.npz")
    sd, extra = H.state_dict("pointpillars_kitti.manifest.json", g["weight_seed"])
    cfg = dict(extra["cfg"], point_cloud_range=[0, -10.24, -3, 20.48, 10.24, 1], output_shape=[128, 128])
    fa = [torch.from_numpy(synth.lidar_frame(6000, 3, tuple(cfg["point_cloud_range"])))]
    fb = [torch.from_numpy(synth.lidar_frame(5000, 4, tuple(cfg["point_cloud_range"])))]
    eager = M.PointPillarsB200(sd, cfg, use_graph=False)
    graph = M.PointPillarsB200(sd, cfg, use_graph=True)
    ea, eb = eager(fa), eager(fb)
    ga = graph(fa)          # capture + first replay
    gb = graph(fb)          # replay on new data
    ga2 = graph(fa)
    for x, y, z, w in zip(ea, eb, ga, gb):
        assert torch.equal(x, z) and torch.equal(y, w)
    for x, z in zip(ea, ga2):
        assert torch.equal(x, z)
    assert not torch.equal(ga[0], gb[0])


# --------------------------------------------------------------------- KPConv
def test_kpfcnn_vs_golden_reference():
    g = H.golden("kpconv_small.npz")
    sd, extra = H.state_dict("kpconv_s3dis.manifest.json", g["weight_seed"])
    clouds = [synth.room_cloud(int(n), int(s), room=H.KP_SMALL_ROOM) for n, s in zip(g["cloud_sizes"], g["cloud_seeds"])]
    bd = H.kp_batch(clouds, extra["cfg"])
    net = M.KPFCNNB200(sd, extra["cfg"])
    taps = {}
    out = net(H.kp_batch_tensors(bd), taps=taps)
    for k in ("encoder_blocks.0", "encoder_blocks.1", "encoder_blocks.2", "encoder_blocks.12"):
        assert rel_err(taps[k][torch.from_numpy(g["tap.%s.rows" % k]).cuda()], g["tap." + k]) < TOL, k
    assert rel_err(out, g["logits"]) < TOL


def test_kpfcnn_medium_vs_port_with_gpu_radius_pyramid():
    """20 000-pt room cloud; the 13 radius searches of KPConvBatch (concat_batcher.py:186-305)
    run on the GPU (bit-exact to the oracle), the fused forward is compared with the port."""
    def gpu_radius(supports, queries, radius, ss, qs):
        r = M.fixed_radius_search(torch.from_numpy(supports).cuda(), torch.from_numpy(queries).cuda(), radius,
                                  torch.from_numpy(ss).cuda(), torch.from_numpy(qs).cuda())
        return r.neighbors_index.cpu().numpy(), r.neighbors_row_splits.cpu().numpy(), None
    sd, extra = H.state_dict("kpconv_s3dis.manifest.json", 5)
    clouds = [synth.room_cloud(12000, 70, room=(3.0, 2.5, 2.0)), synth.room_cloud(8000, 71, room=(3.0, 2.5, 2.0))]
    bd = H.kp_batch(clouds, extra["cfg"], radius_search=gpu_radius)
    ref_nb = MT.kp_batch_neighbors(bd["points"][1], bd["points"][1], bd["lengths"][1], bd["lengths"][1], 0.2)
    assert np.array_equal(bd["neighbors"][1], ref_nb)
    net = M.KPFCNNB200(sd, extra["cfg"])
    tb = H.kp_batch_tensors(bd)
    out = net(tb)
    with torch.no_grad():
        ref = MT.kpfcnn_forward(sd, tb, extra["cfg"])
    assert out.shape == ref.shape and rel_err(out, ref) < TOL


# ------------------------------------------------------------------ pipelined runner
def test_pipelined_runner_matches_direct_calls():
    """PipelinedRunner overlaps copies with the forward; results must equal the plain call,
    batch by batch and in order, including when consecutive batches differ."""
    sd, _ = H.state_dict("randlanet_semantickitti.manifest.json", 3)
    net = M.RandLANetB200(sd)
    batches = [H.randla_inputs(2, 2048, 50 + 10 * i) for i in range(5)]
    pinned = [{k: ([t.pin_memory() for t in v] if isinstance(v, list) else v.pin_memory())
               for k, v in b.items()} for b in batches]
    want = [net(b).cpu().clone() for b in batches]
    runner = M.PipelinedRunner(net)
    got = [r.clone() for r in runner.run(iter(pinned))]
    assert len(got) == len(want)
    for g, w in zip(got, want):
        assert torch.equal(g, w)
    # second pass reuses the slots
    got2 = [r.clone() for r in runner.run(iter(pinned[::-1]))]
    for g, w in zip(got2, want[::-1]):
        assert torch.equal(g, w)


# ------------------------------------------------------------------ device-side transforms (f1)
def test_kpconv_build_batch_on_device_matches_oracle_pyramid():
    """kpconv.build_batch = KPConvBatch.segmentation_inputs on the GPU (radius searches + grid
    subsampling): points of every level and the three index matrices equal the CPU oracle's."""
    from open3d_ml_b200.kpconv import build_batch
    from oracle import ops as O
    _, extra = H.state_dict("kpconv_s3dis.manifest.json", 5)
    cfg = extra["cfg"]
    clouds = [synth.room_cloud(9000, 80, room=(3.0, 2.5, 2.0)), synth.room_cloud(6000, 81, room=(3.0, 2.5, 2.0))]
    b = build_batch(clouds, cfg)
    P = np.concatenate([c[0] for c in clouds])
    lens = [len(c[0]) for c in clouds]
    r = cfg["first_subsampling_dl"] * cfg["conv_radius"]
    for lvl in range(cfg["num_layers"]):
        assert np.array_equal(b["points"][lvl].cpu().numpy(), P)
        assert list(b["lengths"][lvl].cpu().numpy()) == list(lens)
        assert np.array_equal(b["neighbors"][lvl].cpu().numpy(), MT.kp_batch_neighbors(P, P, lens, lens, r))
        if lvl < cfg["num_layers"] - 1:
            Q, ql = O.c_subsample_batch(P, lens, None, None, 2 * r / cfg["conv_radius"])
            assert np.array_equal(b["pools"][lvl].cpu().numpy(), MT.kp_batch_neighbors(Q, P, ql, lens, r))
            assert np.array_equal(b["upsamples"][lvl].cpu().numpy(), MT.kp_batch_neighbors(P, Q, lens, ql, 2 * r))
            P, lens, r = Q, list(ql), 2 * r


def test_randlanet_forward_points_builds_the_reference_pyramid():
    """forward_points (device k-NN pyramid, int32 global ids, one stacked cloud) == forward on the
    reference-shaped inputs built by the CPU oracle (int64 batch-relative ids), and the CUDA-graph
    replay of both equals the eager result bit for bit."""
    sd, _ = H.state_dict("randlanet_semantickitti.manifest.json", 4)
    net = M.RandLANetB200(sd)
    B, N = 3, 4096
    inp = H.randla_inputs(B, N, 90)
    want = net(inp).clone()
    pts = inp["coords"][0].cuda()
    pyr = net.build_pyramid(pts)
    for i in range(4):
        n = inp["coords"][i].shape[1]
        off = (torch.arange(B).view(B, 1, 1) * n).cuda()
        assert torch.equal(pyr["neighbor_indices"][i].view(B, n, 16).long(), inp["neighbor_indices"][i].cuda() + off)
        ns = inp["sub_idx"][i].shape[1]
        assert torch.equal(pyr["sub_idx"][i].view(B, ns, 16).long(), inp["sub_idx"][i].cuda() + off)
        offc = (torch.arange(B).view(B, 1, 1) * ns).cuda()
        assert torch.equal(pyr["interp_idx"][i].view(B, n, 1).long(), inp["interp_idx"][i].cuda() + offc)
    got = net.forward_points(inp["coords"][0])
    assert got.shape == want.shape and torch.equal(got, want)
    g1 = net.forward_points_graphed(pts)
    g2 = net.forward_points_graphed(pts)
    assert torch.equal(g1, want) and torch.equal(g2, want)
    dev_inp = net.to_device(inp)
    assert torch.equal(net.forward_graphed(dev_inp), want) and torch.equal(net.forward_graphed(dev_inp), want)


def test_randlanet_five_level_config_vs_golden_reference():
    """randlanet_s3dis.yml (also semantic3d / toronto3d / parislille3d): 5 encoders, d_out up to 512, ratios
    [4, 4, 4, 4, 2], 6 input channels -- golden logits of the unmodified reference class."""
    g = H.golden("randlanet_s3dis_small.npz")
    sd, extra = H.state_dict("randlanet_s3dis.manifest.json", g["weight_seed"])
    cfg = extra["cfg"]
    B, N = int(g["B"]), int(g["N"])
    per = [MT.randlanet_build_inputs(synth.semantickitti_cloud(N, int(g["seed0"]) + b), num_layers=5,
                                     ratios=cfg["sub_sampling_ratio"]) for b in range(B)]
    inp = {k: [torch.from_numpy(np.stack([q[k][i] for q in per])) for i in range(5)]
           for k in ("coords", "neighbor_indices", "sub_idx", "interp_idx")}
    inp["features"] = torch.cat([inp["coords"][0], torch.from_numpy(g["extra_feat"])], -1)
    net = M.RandLANetB200(sd, num_layers=5, sub_sampling_ratio=cfg["sub_sampling_ratio"])
    out = net(inp)
    assert out.shape == g["logits"].shape and rel_err(out, g["logits"]) < TOL
    assert bool((out.argmax(-1).cpu() == torch.from_numpy(g["logits"]).argmax(-1)).float().mean() > 0.999)
    # the device-side pyramid honours the per-level ratios
    got = net.forward_points(inp["coords"][0], torch.from_numpy(g["extra_feat"]))
    assert rel_err(got, g["logits"]) < TOL


def test_randlanet_fused_tail_matches_the_layerwise_path():
    """rl_tail.cu (last decoder layer + fc1 stack chained through tensor memory) against the four separate launches,
    on reference-shaped inputs (int64 batch-relative interp_idx, ragged last tile) and on the device pyramid."""
    sd, _ = H.state_dict("randlanet_semantickitti.manifest.json", 6)
    net = M.RandLANetB200(sd)
    assert net.tail is not None
    B, N = 3, 4096 + 64 * 3            # not a multiple of 128 per cloud: exercises the row tail
    inp = H.randla_inputs(B, N, 120)
    fused = net(inp).clone()
    n0 = M._lib.lib().o3dml_launch_count()
    net(inp)
    fused_launches = M._lib.lib().o3dml_launch_count() - n0
    tail, net.tail = net.tail, None
    n0 = M._lib.lib().o3dml_launch_count()
    ref = net(inp).clone()
    assert M._lib.lib().o3dml_launch_count() - n0 == fused_launches + 3      # four launches became one
    net.tail = tail
    assert rel_err(fused, ref) < 1e-5, rel_err(fused, ref)
    with torch.no_grad():
        port = MT.randlanet_forward(sd, inp)
    assert rel_err(fused, port) < TOL
    pts = inp["coords"][0].cuda()
    assert torch.equal(net.forward_points(pts), fused)


# ------------------------------------------------------------------ BASELINE sizes (configs[3], configs[4])
def test_kpfcnn_full_size_vs_port():
    """KPFCNN at the BASELINE configs[3] cloud size (65 536 points per cloud, S3DIS config; two clouds bound the CPU
    port's time): batch built on the device (kpconv.build_batch), fused forward against the torch port on the SAME
    index tensors."""
    from open3d_ml_b200.kpconv import build_batch
    sd, extra = H.state_dict("kpconv_s3dis.manifest.json", 5)
    cfg = extra["cfg"]
    clouds = [synth.room_cloud(65536, 200 + i) for i in range(2)]
    b = build_batch(clouds, cfg)
    net = M.KPFCNNB200(sd, cfg)
    out = net(b)
    tb = {k: ([t.cpu() for t in v] if isinstance(v, list) else v.cpu()) for k, v in b.items() if k != "lengths"}
    with torch.no_grad():
        ref = MT.kpfcnn_forward(sd, tb, cfg)
    assert out.shape == ref.shape == (2 * 65536, ref.shape[1])
    assert rel_err(out, ref) < TOL and elem_err(out, ref) < 1e-2


def test_pointpillars_waymo_full_frame_vs_port():
    """PointPillars at the BASELINE configs[4] frame size (180 000 points, 468 x 468 BEV)."""
    sd, extra = H.state_dict("pointpillars_waymo.manifest.json", 11)
    frames = [torch.from_numpy(synth.lidar_frame(180000, 77, synth.WAYMO_RANGE))]
    net = M.PointPillarsB200(sd, extra["cfg"])
    outs = net(frames)
    with torch.no_grad():
        ref = MT.pointpillars_forward(sd, frames, extra["cfg"])
    for o, r in zip(outs, ref):
        assert o.shape == r.shape and rel_err(o, r) < TOL

"""Generates the golden fixtures under tests/golden/ by running the UNMODIFIED
reference model classes from /root/reference (through oracle/refshim.py, torch
CPU) on seeded synthetic inputs with seeded weights.

    python tests/golden/make_golden.py

Only runs in the build container (needs /root/reference).  The fixtures it
writes are committed; the GPU box only reads them.  Inputs are NOT stored: they
are pure functions of the seeds below (open3d_ml_b200.synth + oracle/ops.py),
re-derived by the tests.
"""
import json
import os
import sys
import tempfile

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))

from oracle import refshim, weights, models_torch as MT, ops as O  # noqa: E402
from open3d_ml_b200 import synth  # noqa: E402

SEED = 1234
TAP_CAP = 16 * 1024      # values kept per RandLA-Net tap


def sample_idx(n, m, seed):
    return np.sort(np.random.default_rng(seed).choice(n, size=min(m, n), replace=False))


def sample_rows(t, cap, seed):
    """[..., C] -> (indices into its [rows, C] view, those rows): at most `cap` values, so that every fixture file
    stays under 1 MB."""
    flat = np.asarray(t).reshape(-1, t.shape[-1])
    rows = sample_idx(flat.shape[0], max(1, cap // flat.shape[1]), seed)
    return rows, flat[rows]


def sample_flat(t, m, seed):
    """Any tensor -> (its shape, m indices into the flattened tensor, the values there)."""
    flat = np.asarray(t).reshape(-1)
    idx = sample_idx(flat.size, m, seed)
    return np.array(t.shape), idx, flat[idx]


# ------------------------------------------------------------------ RandLA-Net
def randla_inputs(B, N, seed0):
    per = [MT.randlanet_build_inputs(synth.semantickitti_cloud(N, seed0 + b)) for b in range(B)]
    inp = {k: [torch.from_numpy(np.stack([p[k][i] for p in per])) for i in range(4)]
           for k in ("coords", "neighbor_indices", "sub_idx", "interp_idx")}
    inp["features"] = inp["coords"][0].clone()
    return inp


def make_randlanet():
    from ml3d.torch.models import RandLANet
    cfg = refshim.load_cfg("randlanet_semantickitti.yml")
    net = RandLANet(**cfg.model)
    net.device = "cpu"
    net.eval()
    man = weights.manifest_from_state_dict(net.state_dict())
    weights.save_manifest(os.path.join(HERE, "randlanet_semantickitti.manifest.json"), man,
                          dict(source="ml3d/configs/randlanet_semantickitti.yml"))
    sd = weights.seeded_state_dict(man, SEED)
    net.load_state_dict(sd, strict=True)
    B, N = 2, 2048
    inp = randla_inputs(B, N, 100)
    taps = {}
    hooks = []
    for i in range(4):
        hooks.append(net.encoder[i].register_forward_hook(
            lambda m, a, o, i=i: taps.__setitem__("encoder.%d" % i, o)))
        hooks.append(net.encoder[i].pool1.register_forward_hook(
            lambda m, a, o, i=i: taps.__setitem__("encoder.%d.pool1" % i, o)))
    with torch.no_grad():
        out = net(inp)
    for h in hooks:
        h.remove()
    # the port must agree with the real reference before we trust it elsewhere
    ptaps = {}
    with torch.no_grad():
        port = MT.randlanet_forward(sd, inp, taps=ptaps)
    err = (port - out).abs().max().item() / out.abs().max().item()
    print("randlanet: port vs reference rel err %.3e" % err)
    assert err < 1e-5
    save = dict(logits=out.numpy(), B=B, N=N, seed0=100, weight_seed=SEED)
    for k, v in taps.items():  # [B,C,N,1] -> [B,N,C], a sample of its B * N rows
        save["tap." + k + ".rows"], save["tap." + k] = sample_rows(v.squeeze(3).transpose(1, 2).numpy(), TAP_CAP, 4)
    np.savez_compressed(os.path.join(HERE, "randlanet_small.npz"), **save)

    # a second shape and weight seed: one cloud of 1024 points
    sd = weights.seeded_state_dict(man, 77)
    net.load_state_dict(sd, strict=True)
    inp = randla_inputs(1, 1024, 900)
    with torch.no_grad():
        out = net(inp)
    np.savez_compressed(os.path.join(HERE, "randlanet_other_shape.npz"), logits=out.numpy(), B=1, N=1024, seed0=900,
                        weight_seed=77)


def make_randlanet_s3dis():
    """5-level config (dim_output [16, 64, 128, 256, 512], ratios [4, 4, 4, 4, 2], 6 input channels):
    manifest + a small golden forward of the unmodified class."""
    from ml3d.torch.models import RandLANet
    cfg = refshim.load_cfg("randlanet_s3dis.yml")
    net = RandLANet(**cfg.model)
    net.device = "cpu"
    net.eval()
    man = weights.manifest_from_state_dict(net.state_dict())
    ratios = list(cfg.model["sub_sampling_ratio"])
    weights.save_manifest(os.path.join(HERE, "randlanet_s3dis.manifest.json"), man,
                          dict(source="ml3d/configs/randlanet_s3dis.yml",
                               cfg=dict(num_layers=int(cfg.model["num_layers"]), sub_sampling_ratio=ratios,
                                        in_channels=int(cfg.model["in_channels"]))))
    sd = weights.seeded_state_dict(man, SEED)
    net.load_state_dict(sd, strict=True)
    B, N = 2, 8192
    per = [MT.randlanet_build_inputs(synth.semantickitti_cloud(N, 300 + b), num_layers=5, ratios=ratios) for b in range(B)]
    inp = {k: [torch.from_numpy(np.stack([q[k][i] for q in per])) for i in range(5)]
           for k in ("coords", "neighbor_indices", "sub_idx", "interp_idx")}
    rng = np.random.default_rng(7)
    inp["features"] = torch.cat([inp["coords"][0], torch.from_numpy(rng.random((B, N, 3)).astype(np.float32))], -1)
    with torch.no_grad():
        out = net(inp)
        port = MT.randlanet_forward(sd, inp, num_layers=5)
    err = (port - out).abs().max().item() / out.abs().max().item()
    print("randlanet_s3dis: port vs reference rel err %.3e" % err)
    assert err < 1e-5
    np.savez_compressed(os.path.join(HERE, "randlanet_s3dis_small.npz"), logits=out.numpy(), B=B, N=N, seed0=300,
                        weight_seed=SEED, extra_feat=inp["features"][..., 3:].numpy())


# ------------------------------------------------------------------ PointPillars
PP_SMALL = dict(point_cloud_range=[0, -10.24, -3, 20.48, 10.24, 1], output_shape=[128, 128])


def pp_cfg_dict(cfg_model):
    return dict(point_cloud_range=list(cfg_model["point_cloud_range"]),
                voxel_size=list(cfg_model["voxelize"]["voxel_size"]),
                max_num_points=cfg_model["voxelize"]["max_num_points"],
                max_voxels=cfg_model["voxelize"]["max_voxels"][1],
                output_shape=list(cfg_model["scatter"]["output_shape"]),
                layer_nums=list(cfg_model["backbone"]["layer_nums"]),
                layer_strides=list(cfg_model["backbone"]["layer_strides"]),
                upsample_strides=list(cfg_model["neck"]["upsample_strides"]))


def make_pointpillars():
    from ml3d.torch.models import PointPillars

    class Batch:
        pass

    for tag, yml in (("kitti", "pointpillars_kitti.yml"), ("waymo", "pointpillars_waymo.yml")):
        cfg = refshim.load_cfg(yml)
        m = cfg.model.to_dict() if hasattr(cfg.model, "to_dict") else dict(cfg.model)
        net = PointPillars(device="cpu", **cfg.model)
        net.eval()
        man = weights.manifest_from_state_dict(net.state_dict())
        weights.save_manifest(os.path.join(HERE, "pointpillars_%s.manifest.json" % tag), man,
                              dict(source="ml3d/configs/" + yml, cfg=pp_cfg_dict(m)))
        if tag != "kitti":
            continue
        sd = weights.seeded_state_dict(man, SEED)
        net.load_state_dict(sd, strict=True)
        # (1) full KITTI config, 2 frames (LiDAR-like 20k + uniform 6k); sampled outputs
        frames = [torch.from_numpy(synth.lidar_frame(20000, 200)),
                  torch.from_numpy(synth.uniform_frame(6000, 201))]
        b = Batch()
        b.point = frames
        tp = {}
        h = net.voxel_encoder.register_forward_hook(lambda mod, a, o: tp.__setitem__("pfn", o))
        h2 = net.middle_encoder.register_forward_hook(lambda mod, a, o: tp.__setitem__("canvas", o))
        with torch.no_grad():
            vox = net.voxelize(frames)
            outs = net(b)
        h.remove(), h2.remove()
        pt = {}
        with torch.no_grad():
            port = MT.pointpillars_forward(sd, frames, pp_cfg_dict(m), taps=pt)
        for a, bb in zip(port, outs):
            e = (a - bb).abs().max().item() / bb.abs().max().item()
            print("pointpillars: port vs reference rel err %.3e" % e)
            assert e < 1e-5
        assert torch.equal(pt["coords"], vox[2]) and torch.equal(pt["counts"], vox[1])
        save = dict(weight_seed=SEED, frame_seeds=[200, 201], frame_sizes=[20000, 6000],
                    coords=vox[2].numpy().astype(np.int32), counts=vox[1].numpy().astype(np.int32))
        rows = sample_idx(tp["pfn"].shape[0], 1024, 1)
        save["pfn_rows"], save["pfn_vals"] = rows, tp["pfn"][rows].numpy()
        save["canvas_sum"] = tp["canvas"].double().sum().item()
        save["canvas_abs_sum"] = tp["canvas"].double().abs().sum().item()
        for name, o in zip(("cls", "reg", "dir"), outs):
            flat = o.reshape(-1)
            idx = sample_idx(flat.numel(), 20000, 2)
            save[name + "_shape"] = np.array(o.shape)
            save[name + "_idx"], save[name + "_vals"] = idx, flat[idx].numpy()
            save[name + "_abs_mean"] = flat.double().abs().mean().item()
        np.savez_compressed(os.path.join(HERE, "pointpillars_kitti.npz"), **save)

        # (2) reduced range (128x128 grid), same architecture: full output tensors
        m2 = json.loads(json.dumps(m))
        m2["point_cloud_range"] = PP_SMALL["point_cloud_range"]
        m2["scatter"]["output_shape"] = PP_SMALL["output_shape"]
        net2 = PointPillars(device="cpu", **refshim._AttrDict(m2))
        net2.eval()
        net2.load_state_dict(sd, strict=True)
        f2 = [torch.from_numpy(synth.lidar_frame(6000, 210, tuple(PP_SMALL["point_cloud_range"])))]
        b.point = f2
        with torch.no_grad():
            o2 = net2(b)
        save = dict(weight_seed=SEED, frame_seed=210, frame_size=6000)
        for name, o in zip(("cls", "reg", "dir"), o2):    # half of every output
            save[name + "_shape"], save[name + "_idx"], save[name + "_vals"] = sample_flat(o.numpy(), o.numel() // 2, 5)
        np.savez_compressed(os.path.join(HERE, "pointpillars_small.npz"), **save)


# ------------------------------------------------------------------ KPConv
KP_SMALL_ROOM = (1.6, 1.2, 1.0)


def kp_batch(clouds, cfg):
    """5-level pyramid like KPConvBatch.segmentation_inputs (concat_batcher.py:186-305) with the
    grid subsampling replaced by open3d_ml_b200.synth.grid_subsample (inputs only)."""
    pts = [np.concatenate([c[0] for c in clouds])]
    lens = [[len(c[0]) for c in clouds]]
    feats = np.concatenate([c[1] for c in clouds])
    r = cfg["first_subsampling_dl"] * cfg["conv_radius"]
    dl = cfg["first_subsampling_dl"]
    out = dict(features=feats, points=[], neighbors=[], pools=[], upsamples=[], lengths=[])
    cur = [c[0] for c in clouds]
    for L in range(cfg["num_layers"]):
        P = np.concatenate(cur)
        ln = [len(c) for c in cur]
        out["points"].append(P)
        out["lengths"].append(ln)
        out["neighbors"].append(MT.kp_batch_neighbors(P, P, ln, ln, r).astype(np.int64))
        if L < cfg["num_layers"] - 1:
            dl2 = 2 * dl
            nxt = [synth.grid_subsample(c, dl2) for c in cur]
            Q = np.concatenate(nxt)
            lq = [len(c) for c in nxt]
            out["pools"].append(MT.kp_batch_neighbors(Q, P, lq, ln, r).astype(np.int64))
            out["upsamples"].append(MT.kp_batch_neighbors(P, Q, ln, lq, 2 * r).astype(np.int64))
            cur, dl, r = nxt, dl2, r * 2
        else:
            out["pools"].append(np.zeros((0, 1), np.int64))
            out["upsamples"].append(np.zeros((0, 1), np.int64))
    return out


def make_kpconv():
    from ml3d.torch.models import KPFCNN
    cfg = refshim.load_cfg("kpconv_s3dis.yml")
    cwd = os.getcwd()
    with tempfile.TemporaryDirectory() as td:
        os.chdir(td)  # load_kernels writes kernels/dispositions/*.npy into the CWD (SURVEY A8)
        np.random.seed(0)
        net = KPFCNN(**cfg.model)
        os.chdir(cwd)
    net.device = "cpu"
    net.eval()
    man = weights.manifest_from_state_dict(net.state_dict())
    m = cfg.model.to_dict() if hasattr(cfg.model, "to_dict") else dict(cfg.model)
    keep = ("architecture", "first_subsampling_dl", "conv_radius", "KP_extent", "in_features_dim",
            "first_features_dim", "num_layers", "use_batch_norm", "num_kernel_points", "num_classes")
    kcfg = {k: m[k] for k in keep}
    kcfg["l_relu"] = 0.1
    weights.save_manifest(os.path.join(HERE, "kpconv_s3dis.manifest.json"), man,
                          dict(source="ml3d/configs/kpconv_s3dis.yml", cfg=kcfg))
    sd = weights.seeded_state_dict(man, SEED)
    net.load_state_dict(sd, strict=True)
    clouds = [synth.room_cloud(3000, 300, room=KP_SMALL_ROOM), synth.room_cloud(2000, 301, room=KP_SMALL_ROOM)]
    bd = kp_batch(clouds, kcfg)

    class B:
        pass
    b = B()
    b.features = torch.from_numpy(bd["features"])
    for k in ("points", "neighbors", "pools", "upsamples"):
        setattr(b, k, [torch.from_numpy(a) for a in bd[k]])
    b.lengths = [torch.tensor(x) for x in bd["lengths"]]
    taps = {}
    hooks = [blk.register_forward_hook(lambda mod, a, o, i=i: taps.__setitem__("encoder_blocks.%d" % i, o))
             for i, blk in enumerate(net.encoder_blocks)]
    with torch.no_grad():
        out = net(b)
    for h in hooks:
        h.remove()
    tb = dict(features=b.features, points=b.points, neighbors=b.neighbors, pools=b.pools,
              upsamples=b.upsamples)
    with torch.no_grad():
        port = MT.kpfcnn_forward(sd, tb, kcfg)
    err = (port - out).abs().max().item() / out.abs().max().item()
    print("kpconv: port vs reference rel err %.3e" % err, tuple(out.shape),
          [len(p) for p in bd["points"]], [n.shape[1] for n in bd["neighbors"]])
    assert err < 1e-5
    save = dict(logits=out.numpy(), weight_seed=SEED, cloud_seeds=[300, 301],
                cloud_sizes=[3000, 2000])
    for k in ("encoder_blocks.0", "encoder_blocks.1", "encoder_blocks.2", "encoder_blocks.12"):
        rows = sample_idx(taps[k].shape[0], 256, 3)
        save["tap." + k + ".rows"], save["tap." + k] = rows, taps[k][rows].numpy()
    np.savez_compressed(os.path.join(HERE, "kpconv_small.npz"), **save)


if __name__ == "__main__":
    refshim.install()
    torch.set_num_threads(8)
    which = sys.argv[1:] or ["randlanet", "pointpillars", "kpconv"]
    if "randlanet" in which:
        make_randlanet()
    if "randlanet_s3dis" in which:
        make_randlanet_s3dis()
    if "pointpillars" in which:
        make_pointpillars()
    if "kpconv" in which:
        make_kpconv()
    for f in sorted(os.listdir(HERE)):
        print("%9d  %s" % (os.path.getsize(os.path.join(HERE, f)), f))

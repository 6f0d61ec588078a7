"""The torch port in oracle/models_torch.py pinned against the committed golden
fixtures, which tests/golden/make_golden.py produced by running the UNMODIFIED reference
classes."""
import numpy as np
import torch

from oracle import models_torch as MT
from open3d_ml_b200 import synth
from conftest import rel_err
import helpers as H

TOL = 2e-5  # float32 re-association between two CPU implementations


def test_randlanet_port_vs_golden():
    g = H.golden("randlanet_small.npz")
    sd, _ = H.state_dict("randlanet_semantickitti.manifest.json", g["weight_seed"])
    inp = H.randla_inputs(int(g["B"]), int(g["N"]), int(g["seed0"]))
    taps = {}
    with torch.no_grad():
        out = MT.randlanet_forward(sd, inp, taps=taps)
    assert out.shape == g["logits"].shape
    assert rel_err(out, g["logits"]) < TOL
    for i in range(4):
        for k in ("encoder.%d" % i, "encoder.%d.pool1" % i):
            assert rel_err(H.tap_rows(taps[k], g, k), g["tap." + k]) < TOL, k


def test_pointpillars_port_vs_golden():
    g = H.golden("pointpillars_kitti.npz")
    sd, extra = H.state_dict("pointpillars_kitti.manifest.json", g["weight_seed"])
    frames = [torch.from_numpy(synth.lidar_frame(int(g["frame_sizes"][0]), int(g["frame_seeds"][0]))),
              torch.from_numpy(synth.uniform_frame(int(g["frame_sizes"][1]), int(g["frame_seeds"][1])))]
    taps = {}
    with torch.no_grad():
        outs = MT.pointpillars_forward(sd, frames, extra["cfg"], taps=taps)
    assert np.array_equal(taps["coords"].numpy(), g["coords"])      # index-level parity
    assert np.array_equal(taps["counts"].numpy(), g["counts"])
    assert rel_err(taps["pfn"][g["pfn_rows"]], g["pfn_vals"]) < TOL
    assert abs(taps["canvas"].double().sum().item() - float(g["canvas_sum"])) < 1e-6 * float(g["canvas_abs_sum"])
    for name, o in zip(("cls", "reg", "dir"), outs):
        assert tuple(o.shape) == tuple(g[name + "_shape"])
        assert rel_err(o.reshape(-1)[g[name + "_idx"]], g[name + "_vals"]) < TOL


def test_pointpillars_small_port_vs_golden():
    g = H.golden("pointpillars_small.npz")
    sd, extra = H.state_dict("pointpillars_kitti.manifest.json", g["weight_seed"])
    cfg = dict(extra["cfg"], point_cloud_range=[0, -10.24, -3, 20.48, 10.24, 1], output_shape=[128, 128])
    f = [torch.from_numpy(synth.lidar_frame(int(g["frame_size"]), int(g["frame_seed"]),
                                            tuple(cfg["point_cloud_range"])))]
    with torch.no_grad():
        outs = MT.pointpillars_forward(sd, f, cfg)
    for name, o in zip(("cls", "reg", "dir"), outs):
        assert tuple(o.shape) == tuple(g[name + "_shape"])
        assert rel_err(o.reshape(-1)[g[name + "_idx"]], g[name + "_vals"]) < TOL


def test_kpconv_port_vs_golden():
    g = H.golden("kpconv_small.npz")
    sd, extra = H.state_dict("kpconv_s3dis.manifest.json", g["weight_seed"])
    clouds = [synth.room_cloud(int(n), int(s), room=H.KP_SMALL_ROOM)
              for n, s in zip(g["cloud_sizes"], g["cloud_seeds"])]
    bd = H.kp_batch(clouds, extra["cfg"])
    taps = {}
    with torch.no_grad():
        out = MT.kpfcnn_forward(sd, H.kp_batch_tensors(bd), extra["cfg"], taps=taps)
    assert rel_err(out, g["logits"]) < TOL
    for k in ("encoder_blocks.0", "encoder_blocks.1", "encoder_blocks.2", "encoder_blocks.12"):
        assert rel_err(taps[k][g["tap.%s.rows" % k]], g["tap." + k]) < TOL


def test_randlanet_port_vs_live_reference_other_shape():
    """A second shape/seed than the fixture, against the logits the reference class computed for it
    (randlanet_other_shape.npz, written by tests/golden/make_golden.py)."""
    g = H.golden("randlanet_other_shape.npz")
    sd, _ = H.state_dict("randlanet_semantickitti.manifest.json", g["weight_seed"])
    inp = H.randla_inputs(int(g["B"]), int(g["N"]), int(g["seed0"]))
    with torch.no_grad():
        out = MT.randlanet_forward(sd, inp)
    assert out.shape == g["logits"].shape and rel_err(out, g["logits"]) < TOL

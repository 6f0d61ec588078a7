"""Shared builders for the model parity tests: seeded weights + seeded inputs,
re-derived exactly as tests/golden/make_golden.py derived them."""
import os

import numpy as np
import torch

from oracle import weights, models_torch as MT
from open3d_ml_b200 import synth

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
KP_SMALL_ROOM = (1.6, 1.2, 1.0)


def golden(name):
    return np.load(os.path.join(GOLDEN, name), allow_pickle=False)


def tap_rows(tap, g, key):
    """The rows of a [..., C] tap that fixture g keeps for `key` (make_golden.py:sample_rows)."""
    rows = torch.from_numpy(g["tap.%s.rows" % key]).to(tap.device)
    return tap.reshape(-1, tap.shape[-1])[rows]


def state_dict(manifest_name, seed):
    man, extra = weights.load_manifest(os.path.join(GOLDEN, manifest_name))
    return weights.seeded_state_dict(man, int(seed)), extra


def randla_inputs(B, N, seed0, knn=None):
    per = [MT.randlanet_build_inputs(synth.semantickitti_cloud(N, seed0 + b), knn=knn) for b in range(B)]
    inp = {k: [torch.from_numpy(np.stack([p[k][i] for p in per])) for i in range(4)]
           for k in ("coords", "neighbor_indices", "sub_idx", "interp_idx")}
    inp["features"] = inp["coords"][0].clone()
    return inp


def kp_batch(clouds, cfg, radius_search=None):
    """Same pyramid as tests/golden/make_golden.py:kp_batch."""
    r = cfg["first_subsampling_dl"] * cfg["conv_radius"]
    dl = cfg["first_subsampling_dl"]
    out = dict(features=np.concatenate([c[1] for c in clouds]), points=[], neighbors=[], pools=[],
               upsamples=[], lengths=[])
    cur = [c[0] for c in clouds]
    for lvl in range(cfg["num_layers"]):
        P = np.concatenate(cur)
        ln = [len(c) for c in cur]
        out["points"].append(P)
        out["lengths"].append(ln)
        out["neighbors"].append(MT.kp_batch_neighbors(P, P, ln, ln, r, radius_search).astype(np.int64))
        if lvl < cfg["num_layers"] - 1:
            nxt = [synth.grid_subsample(c, 2 * dl) for c in cur]
            Q = np.concatenate(nxt)
            lq = [len(c) for c in nxt]
            out["pools"].append(MT.kp_batch_neighbors(Q, P, lq, ln, r, radius_search).astype(np.int64))
            out["upsamples"].append(MT.kp_batch_neighbors(P, Q, ln, lq, 2 * r, radius_search).astype(np.int64))
            cur, dl, r = nxt, 2 * dl, r * 2
        else:
            out["pools"].append(np.zeros((0, 1), np.int64))
            out["upsamples"].append(np.zeros((0, 1), np.int64))
    return out


def kp_batch_tensors(bd):
    tb = dict(features=torch.from_numpy(bd["features"]))
    for k in ("points", "neighbors", "pools", "upsamples"):
        tb[k] = [torch.from_numpy(a) for a in bd[k]]
    return tb

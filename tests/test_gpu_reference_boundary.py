"""Row (b) of SURVEY.md section 8: UNMODIFIED reference code driven through the drop-in boundary
(open3d_ml_b200.shim) on the GPU -- the reference's own torch smoke tests, its PointPillars / RandLANet /
KPFCNN classes against the fused forwards built from their state_dicts, and SemanticSegmentation.run_inference.
The reference tree comes from /root/reference here and from the git-ignored snapshot oracle/_ref on the GPU box
(oracle/make_ref_snapshot.py, run by __graft_entry__.build()).  Every case runs in a fresh process because the
shim owns sys.modules['open3d']."""
import json
import os
import subprocess
import sys

import pytest

from conftest import ROOT

pytestmark = pytest.mark.gpu
TOL = 1e-4


def run_case(case, timeout=900):
    from oracle.make_ref_snapshot import ref_root
    if ref_root() is None:
        pytest.skip("needs the Open3D-ML source tree, which is not part of this repository: point $OPEN3D_ML_ROOT at "
                    "it, or copy it to oracle/_ref with oracle/make_ref_snapshot.py")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "ref_boundary_cases.py"), case], cwd=ROOT,
                       capture_output=True, text=True, timeout=timeout)
    assert r.returncode == 0, (r.stdout[-3000:], r.stderr[-3000:])
    line = [l for l in r.stdout.splitlines() if l.startswith("RESULT ")][-1]
    res = json.loads(line[len("RESULT "):])
    assert res["ops"] == "b200" and res["device"] == "cuda"
    return res


def test_reference_torch_smoke_tests_run_unmodified_through_the_shim():
    """/root/reference/tests/test_models.py: test_randlanet_torch, test_kpconv_torch, test_pointpillars_torch."""
    assert run_case("ref_tests")["pytest_rc"] == 0


def test_unmodified_pointpillars_class_matches_fused_forward_and_runs_inference_end():
    res = run_case("pointpillars_class")
    assert res["ref_shapes"] == [[2, 18, 248, 216], [2, 42, 248, 216], [2, 12, 248, 216]]
    assert all(e < TOL for e in res["rel_err"]), res
    assert all(n > 0 for n in res["boxes_per_frame"]), res       # anchors + top-k + decode + rotated NMS ran


def test_patch_reference_model_randlanet_matches_the_cpu_class():
    res = run_case("randlanet_patch")
    assert res["ref_shape"] == [1, 8192, 19] and res["rel_err"] < TOL and res["argmax_agree"] > 0.999, res


def test_semantic_segmentation_run_inference_unchanged_pipeline():
    res = run_case("semseg_inference")
    assert res["labels_shape"] == [20000] and res["scores_shape"] == [20000, 19] and res["finite"]
    assert res["fused_labels_shape"] == [20000] and res["fused_finite"]


def test_unmodified_kpfcnn_class_matches_fused_forward():
    res = run_case("kpconv_class")
    assert res["levels"][0] >= 1000 and res["ref_shape"][1] == 5 and res["rel_err"] < TOL, res

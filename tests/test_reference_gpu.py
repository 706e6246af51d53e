"""-m gpu: the CUDA path against the REFERENCE ITSELF (not the restatement).

The reference's outputs on these inputs were produced by running the unmodified reference code on the CPU
(oracle/ref_harness.py, tools/make_reference_golden.py) and are stored in tests/golden/reference_product.npz; arrays over the
5023 vertices keep a fixed sample of vertex columns, the encoder outputs a fixed sample of elements.  Every comparison here is
product (libdad3d.so through the C ABI) vs the unmodified reference code; tolerances are north_star's 1e-4 relative.
"""
import hashlib
import json
import os
import warnings

import numpy as np
import pytest
import torch

from dad_3dheads_b200.encoder_weights import synthetic_state_dict
from oracle.flame_oracle import sample_params

pytestmark = pytest.mark.gpu
GOLDEN = os.path.join(os.path.dirname(__file__), "golden")
warnings.filterwarnings("ignore", message="Using torch.cross")


def _rel(a, b):
    a, b = torch.as_tensor(a).double().cpu(), torch.as_tensor(b).double().cpu()
    return ((a - b).norm() / b.norm()).item()


def _contract(got, ref):
    """north_star: element-wise within 1e-4 relative fp32 (absolute floor 1e-4 for values near zero) -> max violation."""
    got, ref = torch.as_tensor(got).double().cpu(), torch.as_tensor(ref).double().cpu()
    return ((got - ref).abs() / (1e-4 * ref.abs() + 1e-4)).max().item()


@pytest.fixture(scope="module")
def ref():
    return np.load(os.path.join(GOLDEN, "reference_product.npz"))


@pytest.fixture(scope="module")
def product(cuda_device):
    from dad_3dheads_b200.predictor import FaceMeshPredictor
    return FaceMeshPredictor.dad_3dnet(state_dict=synthetic_state_dict(0))


@pytest.mark.parametrize("B", [1, 2, 64, 129])
def test_decode_vs_reference_headmesh(product, cuda_device, ref, B):
    vs = torch.from_numpy(ref["decode_vertex_sample"])
    p = sample_params(B, seed=40 + B)
    assert hashlib.sha256(p.numpy().tobytes()).hexdigest() == str(ref[f"decode_params_sha256_b{B}"])     # the reference's input
    want_v = torch.from_numpy(ref[f"decode_vertices3d_b{B}"])
    want_p = torch.from_numpy(ref[f"decode_projected2d_b{B}"])
    q = p.clone()
    q[:, 411] = torch.from_numpy(ref[f"decode_tz_after_reproject_b{B}"])   # the reference's in-place side effect
    for hilo, tol, l2 in ((False, 5e-5, 1e-4), (True, 2e-6, 1e-6)):      # default one-product kernel / strict hi-lo blend
        v3, pj = product.head_mesh.decode(p.to(cuda_device), to_2d=True, hilo=hilo)
        v3, pj = v3[:, vs], pj[:, vs]
        assert _rel(v3, want_v) < tol and _rel(pj, want_p) < tol, (hilo, _rel(v3, want_v), _rel(pj, want_p))
        assert _contract(v3, want_v) < 1.0 and _contract(pj, want_p) < 1.0
        assert (v3.cpu() - want_v).norm(dim=-1).max().item() < l2        # vertex L2 (m); north_star target < 1e-4
    # the reference-facing methods on CPU tensors, side effect included
    q2 = p.clone()
    got_p = product.head_mesh.reprojected_vertices(q2, to_2d=True)
    assert torch.equal(q2, q) and _rel(got_p[:, vs], want_p) < 2e-6


def test_encoder_vs_reference_flame_regression(cuda_device, ref):
    from dad_3dheads_b200.encoder import Dad3dEncoder
    sd = synthetic_state_dict(4)
    x = torch.randn(3, 3, 256, 256, generator=torch.Generator().manual_seed(31))
    keys = ("OUTPUT_2D_LANDMARKS", "OUTPUT_3DMM_PARAMS", "OUTPUT_LANDMARKS_HEATMAP")
    for mode, tol in (("fp32", 3e-5), ("fp16x2", 3e-5)):
        got = Dad3dEncoder(sd, cuda_device, precision=mode)(x.to(cuda_device))
        assert set(got) == set(keys), mode
        for k in keys:
            idx = torch.from_numpy(ref[f"encoder_{k}_index"]).to(cuda_device)
            assert _rel(got[k].reshape(-1)[idx], ref[f"encoder_{k}"]) < tol, (mode, k)
        assert ref["encoder_OUTPUT_3DMM_PARAMS"].size == got["OUTPUT_3DMM_PARAMS"].numel()    # kept whole
        assert _contract(got["OUTPUT_3DMM_PARAMS"].reshape(-1), ref["encoder_OUTPUT_3DMM_PARAMS"]) < 1.0, mode


def test_predictor_call_vs_reference_predictor(product, ref):
    """FaceMeshPredictor.__call__ (predictor.py:78-83) on the demo image and on odd sizes: same keys, dtypes, shapes,
    in-place semantics; values within the contract; integer landmark pixels within 1."""
    import cv2
    vs = ref["vertex_sample"]
    imgs = [cv2.cvtColor(cv2.imread(os.path.join(GOLDEN, "demo_head_1.jpeg")), cv2.COLOR_BGR2RGB)]
    g = np.random.default_rng(1)
    imgs += [g.integers(0, 256, s + (3,), dtype=np.uint8) for s in ((300, 517), (641, 203), (256, 256))]
    for i, img in enumerate(imgs):
        meta, got = json.loads(str(ref[f"predictor_{i}_meta"])), product(img.copy())
        assert set(got) == set(meta)
        for k, m in meta.items():
            assert list(got[k].shape) == m["shape"], (k, got[k].shape, m["shape"])
            if m["tensor"]:            # the reference pins its outputs to the CPU (oracle/ref_harness.cpu_only)
                assert torch.is_tensor(got[k]) and str(got[k].dtype) == m["dtype"] and got[k].device.type == "cpu", k
            else:
                assert isinstance(got[k], np.ndarray) and got[k].dtype.kind == m["kind"], (k, got[k].dtype)
        want = {"3dmm_params": ref[f"predictor_{i}_params"], "3d_vertices": ref[f"predictor_{i}_vertices3d"],
                "projected_vertices": ref[f"predictor_{i}_projected"]}
        got_s = {"3dmm_params": got["3dmm_params"], "3d_vertices": got["3d_vertices"][..., vs, :],
                 "projected_vertices": got["projected_vertices"][..., vs, :]}
        errs = {k: _rel(got_s[k], want[k]) for k in want}
        dpx = int(np.abs(got["points"] - ref[f"predictor_{i}_points"]).max())
        assert all(v < 5e-5 for v in errs.values()) and dpx <= 1, (img.shape, errs, dpx)


def test_predictor_fixture(product):
    """Same check against the committed output of the reference predictor (tests/golden/reference_predictor.npz)."""
    import cv2
    z = np.load(os.path.join(GOLDEN, "reference_predictor.npz"))
    img = cv2.cvtColor(cv2.imread(os.path.join(GOLDEN, "demo_head_1.jpeg")), cv2.COLOR_BGR2RGB)
    got = product(img)
    assert _rel(got["3dmm_params"], z["params_3dmm"]) < 5e-5
    assert _rel(got["3d_vertices"], z["vertices_3d"]) < 5e-5
    assert _rel(got["projected_vertices"], z["projected_vertices"]) < 5e-5
    assert np.abs(got["points"] - z["points"]).max() <= 1

"""-m gpu: the reference-facing API (FaceMeshPredictor) end to end against the oracle restatement of predictor.py."""
import os

import numpy as np
import pytest
import torch

from dad_3dheads_b200.encoder_weights import synthetic_state_dict
from oracle.predictor_oracle import PredictorOracle

pytestmark = pytest.mark.gpu
GOLDEN = os.path.join(os.path.dirname(__file__), "golden")


def _rel(a, b):
    a, b = torch.as_tensor(a).double().cpu(), torch.as_tensor(b).double().cpu()
    return ((a - b).norm() / b.norm()).item()


@pytest.fixture(scope="module")
def predictor(cuda_device):
    from dad_3dheads_b200.predictor import FaceMeshPredictor
    return FaceMeshPredictor.dad_3dnet(state_dict=synthetic_state_dict(0))


@pytest.fixture(scope="module")
def oracle():
    return PredictorOracle(synthetic_state_dict(0), dtype=torch.float64)


def _demo_image():
    import cv2
    return cv2.cvtColor(cv2.imread(os.path.join(GOLDEN, "demo_head_1.jpeg")), cv2.COLOR_BGR2RGB)


def test_single_image_call_matches_reference_semantics(predictor, oracle):
    """BASELINE configs[0]: FaceMeshPredictor.__call__ on images/demo_heads/1.jpeg (954x766 -> letter-boxed 256x206)."""
    img = _demo_image()
    got = predictor(img)
    want = oracle(img)
    assert set(got) == {"points", "projected_vertices", "3d_vertices", "3dmm_params"}
    assert got["points"].shape == (68, 2) and got["points"].dtype.kind == "i"
    assert got["projected_vertices"].shape == (1, 5023, 2) and got["projected_vertices"].device.type == "cpu"
    assert got["3d_vertices"].shape == (5023, 3) and got["3dmm_params"].shape == (1, 413)
    assert got["3dmm_params"][0, 411].item() == 0.0                      # tz zeroed in place (head_mesh.py:41)
    assert _rel(got["3dmm_params"], want["3dmm_params"]) < 5e-5
    assert _rel(got["3d_vertices"], want["3d_vertices"]) < 5e-5
    assert (got["projected_vertices"].double() - want["projected_vertices"]).abs().max() < 0.25   # input-image pixels (~1e3)
    assert np.abs(got["points"] - want["points"]).max() <= 1              # int truncation of pixel coordinates


def test_predict_batch_matches_oracle(predictor, oracle, cuda_device):
    x = torch.randn(4, 3, 256, 256, generator=torch.Generator().manual_seed(5))
    got = predictor.predict_batch(x, landmark_subset="445")
    want = oracle.predict_batch(x)
    for k in ("3dmm_params", "points", "3d_vertices", "projected_vertices"):
        assert got[k].is_cuda
        assert _rel(got[k], want[k]) < 5e-5, k
    idx = torch.from_numpy(np.load(os.path.join(os.path.dirname(GOLDEN), "..", "dad_3dheads_b200", "assets",
                                                "flame_static.npz"))["keypoints_445"].astype(np.int64))
    assert got["landmarks_445"].shape == (4, 445, 2)
    assert torch.equal(got["landmarks_445"].cpu(), got["projected_vertices"].cpu()[:, idx])


def test_vertex_l2_error_target(predictor, oracle):
    """north_star: vertex L2 error < 1e-4 vs reference (metres, per vertex) through the whole pipeline."""
    x = torch.randn(3, 3, 256, 256, generator=torch.Generator().manual_seed(6))
    got = predictor.predict_batch(x, landmark_subset=None)
    want = oracle.predict_batch(x)
    l2 = (got["3d_vertices"].double().cpu() - want["3d_vertices"]).norm(dim=-1)
    assert l2.max().item() < 1e-4, l2.max().item()


def test_graph_replay_equals_eager(predictor, cuda_device):
    """predict_batch_graphed replays predict_batch from a CUDA graph: bit-identical outputs, for fp32 and raw uint8
    input, and across consecutive calls with different data (static input buffer refreshed every call)."""
    g = torch.Generator().manual_seed(5)
    for make in (lambda: torch.randn(3, 3, 256, 256, generator=g),
                 lambda: torch.randint(0, 256, (3, 256, 256, 3), generator=g, dtype=torch.uint8)):
        for _ in range(2):
            x = make()
            want = {k: v.clone() for k, v in predictor.predict_batch(x).items()}
            got = predictor.predict_batch_graphed(x)
            torch.cuda.synchronize()
            for k in want:
                assert torch.equal(got[k], want[k]), k


def test_config2_batch_512_bf16_encoder(cuda_device):
    """BASELINE configs[2]: batch 512, bf16 encoder, fp32-class FLAME decode + 445-landmark projection.  Size-independent
    checks: finite everywhere, and (eval-mode network: images are independent) a sub-batch run on its own reproduces the
    corresponding rows bit for bit."""
    from dad_3dheads_b200.predictor import FaceMeshPredictor
    pred = FaceMeshPredictor.dad_3dnet(state_dict=synthetic_state_dict(0), precision="bf16")
    x = torch.randn(512, 3, 256, 256, generator=torch.Generator().manual_seed(512))
    out = {k: v.clone() for k, v in pred.predict_batch(x, landmark_subset="445").items()}
    assert out["3d_vertices"].shape == (512, 5023, 3) and out["landmarks_445"].shape == (512, 445, 2)
    assert all(torch.isfinite(v).all() for v in out.values())
    sub = pred.predict_batch(x[300:364], landmark_subset="445")
    for k in out:
        assert torch.equal(out[k][300:364], sub[k]), k
    # parity at the full size: a bf16-EMULATING oracle (folded CPU executor with every stored operand rounded to bf16 like the
    # engine's single-piece mode) on a subset of the 512 images; the plain fp32 oracle is ~6e-3 away from this mode, the
    # emulation must be clearly closer (what remains is accumulation order / rounding-boundary flips)
    from dad_3dheads_b200.encoder import fold_state_dict
    from tests.folded_ref import bf16_round, run_folded
    rows = [0, 137, 300, 511]
    layers, fw = fold_state_dict(synthetic_state_dict(0))
    emu = run_folded(x[rows], layers, fw, dtype=torch.float32, quant=bf16_round)
    ref = run_folded(x[rows], layers, fw, dtype=torch.float32)
    got = out["3dmm_params"][rows].cpu()
    e_emu, e_ref = _rel(got, emu["params"]), _rel(got, ref["params"])
    print(f"bf16 B=512 params: relL2 vs bf16-emulating oracle {e_emu:.2e}, vs fp32 oracle {e_ref:.2e}")
    assert e_emu < 5e-3 and e_emu < 0.7 * e_ref, (e_emu, e_ref)


def test_heatmap_fallback_branch_matches_reference(predictor):
    """predictor.py:109-113: when the model output has no OUTPUT_2D_LANDMARKS the landmarks come from the heat-map arg-max
    (``unravel_index`` -- which divides by H for both axes, model/utils.py:38-52) times the stride; same values as the
    reference's own ``_parse_output`` on the same tensors (tests/golden/reference_product.npz), and the 3DMM-only branch when
    neither key is present."""
    import os
    g = torch.Generator().manual_seed(3)
    hm = torch.randn(1, 68, 64, 64, generator=g)
    p = torch.randn(1, 413, generator=g)
    lm, p3 = predictor._parse_output({"OUTPUT_3DMM_PARAMS": p.clone(), "OUTPUT_LANDMARKS_HEATMAP": hm.clone()})
    flat = torch.sigmoid(hm).view(1, 68, -1).argmax(-1)
    want = torch.stack((flat % 64, flat // 64), -1)[0].numpy().astype(np.float64) * 4.0        # (x, y) * stride
    assert np.array_equal(lm, want) and torch.equal(p3, p)
    only = predictor._parse_output({"OUTPUT_3DMM_PARAMS": p.clone()})
    assert torch.is_tensor(only) and torch.equal(only, p)
    z = np.load(os.path.join(os.path.dirname(__file__), "golden", "reference_product.npz"))
    assert np.array_equal(lm, z["heatmap_fallback_landmarks"]) and np.array_equal(p3.numpy(), z["heatmap_fallback_params"])

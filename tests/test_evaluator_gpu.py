"""-m gpu: the GPU evaluator (csrc/evaluator.cu through the C ABI) against the oracle restatement of DADEvaluator (itself pinned
to the unmodified reference by tests/test_evaluator_cpu.py) and against the reference evaluator's own results on the same pairs
(tests/golden/reference_evaluator.json)."""
import json
import os

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_gpu_evaluator_matches_oracle_and_reference(cuda_device, tmp_path):
    from dad_3dheads_b200.evaluator import DADEvaluatorGPU
    from dad_3dheads_b200.flame import load_flame_static
    from oracle.evaluator_oracle import EvaluatorOracle
    from tests.eval_fixtures import make_pairs
    gts, sub = make_pairs(5, seed=2)
    json.dump(gts, open(tmp_path / "gt.json", "w"))
    json.dump(sub, open(tmp_path / "sub.json", "w"))
    overall, attrs = DADEvaluatorGPU(str(tmp_path / "gt.json"), str(tmp_path / "sub.json"))()
    st = load_flame_static()
    want = EvaluatorOracle(st, st["head_indices"], st["flame_indices_face"])(gts, sub)
    assert set(overall) == set(want) == {"pose_error", "nme_reprojection", "z5_accuracy", "chamfer"}
    for k in want:
        tol = 5e-3 if k == "z5_accuracy" else 1e-4           # z5 is ill-conditioned: torch.cdist's cancellation noise (~3e-4 m at
        # 0.8 m from the origin) reorders millimetre-scale neighbours, so even the reference differs by ~2e-3 between two CPUs
        assert abs(overall[k] - want[k]) <= tol * abs(want[k]) + 1e-6, (k, overall[k], want[k])
    assert set(attrs["chamfer"]) == {"pose", "occlusions"} and set(attrs["chamfer"]["pose"]) == {"front", "side"}
    ref = json.load(open(os.path.join(ROOT, "tests", "golden", "reference_evaluator.json")))["pairs_5_seed_2"]
    for k, v in ref["overall"].items():
        tol = 5e-3 if k == "z5_accuracy" else 1e-4
        assert abs(overall[k] - v) <= tol * abs(v) + 1e-6, (k, overall[k], v)
    for k, d in ref["attributes"]["nme_reprojection"].items():
        for kk, v in d.items():
            got = {str(a): b for a, b in attrs["nme_reprojection"][k].items()}[kk]
            assert abs(got - v) <= 1e-4 * abs(v) + 1e-6


def test_zn_kernel_exact_on_well_separated_points(cuda_device):
    """calc_zn bit-for-bit on inputs without near-ties (random points: distinct distances)."""
    from dad_3dheads_b200.evaluator import DADEvaluatorGPU
    from oracle.evaluator_oracle import calc_zn
    ev = DADEvaluatorGPU()
    g = torch.Generator().manual_seed(0)
    for K in (64, 1000, 3669):
        gt = torch.randn(3, K, 3, generator=g)
        pred = gt + 0.3 * torch.randn(3, K, 3, generator=g)
        got = ev.calc_zn(pred.to(cuda_device), gt.to(cuda_device), 5).cpu()
        want = torch.tensor([calc_zn(pred[b], gt[b], 5) for b in range(3)])
        assert (got - want).abs().max() < 5e-4, (K, got, want)


def test_chamfer_kernel(cuda_device):
    from dad_3dheads_b200.evaluator import DADEvaluatorGPU
    ev = DADEvaluatorGPU()
    g = torch.Generator().manual_seed(1)
    a = torch.randn(4, 2094, 3, generator=g)
    b = torch.randn(4, 5023, 3, generator=g)
    got = ev.chamfer_one_sided(a.to(cuda_device), b.to(cuda_device)).cpu()
    want = (torch.cdist(a.double(), b.double()) ** 2).min(dim=2).values.mean(dim=1)
    assert ((got.double() - want).abs() / want).max() < 1e-5

"""-m "not gpu": the evaluator oracle (oracle/evaluator_oracle.py) against the UNMODIFIED reference evaluator
(dad_3dheads_benchmark/benchmark.py::DADEvaluator, run by oracle/run_ref_benchmark.py with shims for fire / smplx / kaolin; its
results on these pairs are stored in tests/golden/reference_evaluator.json by tools/make_reference_golden.py)."""
import json
import os

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_evaluator_oracle_matches_reference():
    from dad_3dheads_b200.flame import load_flame_static
    from oracle.evaluator_oracle import EvaluatorOracle
    from tests.eval_fixtures import make_pairs
    gts, sub = make_pairs(3, seed=1)
    ref = json.load(open(os.path.join(ROOT, "tests", "golden", "reference_evaluator.json")))["pairs_3_seed_1"]["overall"]
    st = load_flame_static()
    got = EvaluatorOracle(st, st["head_indices"], st["flame_indices_face"])(gts, sub)
    assert set(got) == set(ref)
    for k in ref:
        assert abs(got[k] - ref[k]) <= 1e-5 * abs(ref[k]) + 1e-6, (k, got[k], ref[k])
    assert 0.5 < ref["z5_accuracy"] <= 1.0 and ref["chamfer"] > 0 and ref["nme_reprojection"] > 0

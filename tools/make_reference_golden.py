#!/usr/bin/env python
"""Generate tests/golden/reference_*.npz by RUNNING THE UNMODIFIED REFERENCE (oracle/ref_harness.py) in this container.

These are reference outputs, not oracle outputs: /root/reference's own predictor.py / head_mesh.py / flame.py /
model/utils.py / flame_regression.py / bifpn.py / encoders.py executed on the CPU, with shims only for the third-party
packages that are absent (oracle/ref_shims/README.md).  They pin the oracle (tests/test_oracle_pinned.py) and, on the GPU
box where /root/reference does not exist, the CUDA path (tests -m gpu).

  reference_flame.npz      HeadMesh.vertices_3d / reprojected_vertices, fp32 and fp64, B in {1, 3 (torch.cross quirk), 6}
  reference_encoder.npz    FlameRegression.forward, seed-0 synthetic weights, 2 seeded images, fp32 and fp64
  reference_predictor.npz  FaceMeshPredictor.__call__ on images/demo_heads/1.jpeg through a traced .trcd (batch-1 trace)
  reference_assets.npz     sha256 of every FLAMELayer buffer (flame.pkl -> fp32) + the landmark index sets
  reference_live.npz       the oracle-pinning cases: HeadMesh fp64 (3 seeds), rot_mat_from_6dof (incl. B=3), FlameRegression
                           fp64 per stage, FaceMeshPredictor.__call__ on odd sizes, the module's state-dict names, the pncc
                           estimator over the reference's C++ rasteriser
  reference_product.npz    the CUDA-path cases: HeadMesh decode at B in {1, 2, 64, 129}, FlameRegression fp64 on 3 images,
                           FaceMeshPredictor.__call__ on the demo image and odd sizes, the heat-map fallback of _parse_output
  reference_rasterizer.npz Sim3DR rasterize / get_normal (rasterize_kernel.cpp) on the rasteriser tests' scenes
  reference_evaluator.json DADEvaluator on the evaluator tests' seeded pairs
Arrays over 5023 vertices keep the VERTEX_SAMPLE columns and large activations a seeded sample of elements, so that every
file stays well under 1 MB.
"""
import hashlib
import json
import os
import sys
import warnings

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import ref_harness as R  # noqa: E402
from oracle.flame_oracle import sample_params  # noqa: E402

GOLD = os.path.join(ROOT, "tests", "golden")
N_VERTEX_SAMPLE, N_ELEMENT_SAMPLE = 256, 4096
warnings.filterwarnings("ignore", message="Using torch.cross")


def sha(a) -> str:
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def flame_golden():
    out = {}
    for name, dt in (("f32", torch.float32), ("f64", torch.float64)):
        hm = R.head_mesh(dtype=dt if dt is torch.float64 else None)
        for B, seed in ((1, 11), (3, 12), (6, 13)):
            p = sample_params(B, seed=seed)
            if B == 6:
                p[0] = 0
                p[0, 403:409] = torch.tensor([1.0, 0, 0, 0, 1.0, 0])
            out[f"params_b{B}"] = p.numpy().copy()
            q = p.clone().to(dt)
            v = hm.vertices_3d(q)                           # head_mesh.py:28-31
            vz = hm.vertices_3d(q, zero_rotation=True)
            q2 = q.clone()
            pr = hm.reprojected_vertices(q2, to_2d=False)   # head_mesh.py:33-46 (zeroes tz through the view)
            out[f"vertices3d_{name}_b{B}"] = v.to(torch.float64).numpy() if dt is torch.float64 else v.numpy()
            out[f"vertices3d_zero_rot_{name}_b{B}"] = vz.numpy()
            out[f"projected3_{name}_b{B}"] = pr.numpy()
            out[f"params_after_reproject_{name}_b{B}"] = q2.numpy()
    # keep the file small: fp64 arrays only for B=1 and B=6 vertices, stored as float64; everything else float32
    keep = {}
    for k, v in out.items():
        if "_f64_" in k and not (k.startswith("vertices3d_f64") or k.startswith("projected3_f64")):
            continue
        keep[k] = v
    np.savez_compressed(os.path.join(GOLD, "reference_flame.npz"), **keep)
    print("reference_flame.npz", os.path.getsize(os.path.join(GOLD, "reference_flame.npz")))


def encoder_golden():
    from dad_3dheads_b200.encoder_weights import synthetic_state_dict
    sd = synthetic_state_dict(0)
    x = torch.randn(2, 3, 256, 256, generator=torch.Generator().manual_seed(777))
    out = {"image_seed": np.int64(777), "weight_seed": np.int64(0)}
    for name, dt in (("f32", torch.float32), ("f64", torch.float64)):
        m = R.flame_regression(sd, dtype=dt)
        with torch.no_grad():
            o = m(x.to(dt))
        out[f"params_{name}"] = o["OUTPUT_3DMM_PARAMS"].numpy()
        out[f"landmarks_{name}"] = o["OUTPUT_2D_LANDMARKS"].numpy()
        hm = o["OUTPUT_LANDMARKS_HEATMAP"]
        out[f"heatmap_sum_{name}"] = hm.sum(dim=(2, 3)).numpy()
        out[f"heatmap_corner_{name}"] = hm[:, :, :4, :4].numpy()
    np.savez_compressed(os.path.join(GOLD, "reference_encoder.npz"), **out)
    print("reference_encoder.npz", os.path.getsize(os.path.join(GOLD, "reference_encoder.npz")))


def predictor_golden():
    import cv2
    from dad_3dheads_b200.encoder_weights import synthetic_state_dict
    pred = R.predictor(synthetic_state_dict(0))
    img = cv2.cvtColor(cv2.imread(os.path.join(GOLD, "demo_head_1.jpeg"), cv2.IMREAD_COLOR), cv2.COLOR_BGR2RGB)
    res = pred(img)
    cache = {}
    x = pred.preprocess(img, cache)
    np.savez_compressed(os.path.join(GOLD, "reference_predictor.npz"), weight_seed=np.int64(0),
                        input_sha256=sha(img), network_input_sha256=sha(x.numpy()),
                        points=res["points"], projected_vertices=res["projected_vertices"].numpy(),
                        vertices_3d=res["3d_vertices"].numpy(), params_3dmm=res["3dmm_params"].numpy())
    print("reference_predictor.npz", os.path.getsize(os.path.join(GOLD, "reference_predictor.npz")),
          {k: tuple(v.shape) for k, v in res.items()})


def assets_golden():
    buf = R.flame_buffers()
    out = {k + "_sha256": sha(v) for k, v in buf.items()}
    out.update({k + "_shape": np.asarray(v.shape) for k, v in buf.items()})
    R.activate()
    from model_training.utils import get_list_of_npy_files, load_indices_from_npy   # model_training/utils.py:81-105
    base = os.path.join(R.root(), "model_training", "model", "static", "face_keypoints")
    for sub, excl in (("191", None), ("445", "cheeks"), ("445", None)):
        files = get_list_of_npy_files({"2d_subset_path": os.path.join(base, f"keypoints_{sub}"), "2d_keys_exclude": excl})
        idx = []
        for f in sorted(files):
            idx += load_indices_from_npy(f)
        out["keypoints_" + (sub if excl or sub == "191" else "565")] = np.asarray(idx, dtype=np.int32)
    np.savez_compressed(os.path.join(GOLD, "reference_assets.npz"), **out)
    print("reference_assets.npz", os.path.getsize(os.path.join(GOLD, "reference_assets.npz")))


def vertex_sample(n=N_VERTEX_SAMPLE):
    """The vertex indices golden vertex arrays keep (stored beside them; tests index their own full outputs with them)."""
    return np.sort(np.random.default_rng(0).choice(5023, n, replace=False))


def element_sample(n, seed):
    return np.sort(np.random.default_rng(seed).choice(n, min(n, N_ELEMENT_SAMPLE), replace=False))


def _save(name, out):
    path = os.path.join(GOLD, name)
    np.savez_compressed(path, **out)
    print(name, os.path.getsize(path))
    assert os.path.getsize(path) < 1 << 20, name


def live_golden():
    from dad_3dheads_b200.encoder_weights import synthetic_state_dict
    vs = vertex_sample()
    out = {"vertex_sample": vs}
    hm = R.head_mesh(dtype=torch.float64)
    for B, seed in ((1, 101), (2, 102), (5, 103)):
        p = sample_params(B, seed=seed).double()
        q = p.clone()
        out[f"flame_params_b{B}"] = p.numpy()
        out[f"flame_vertices3d_b{B}"] = hm.vertices_3d(p.clone())[:, vs].numpy()
        out[f"flame_vertices3d_zero_rot_b{B}"] = hm.vertices_3d(p.clone(), zero_rotation=True)[:, vs].numpy()
        out[f"flame_projected2d_b{B}"] = hm.reprojected_vertices(q, to_2d=True)[:, vs].numpy()
        out[f"flame_params_after_reproject_b{B}"] = q.numpy()
    R.activate()
    from model_training.model.utils import rot_mat_from_6dof as ref_rot      # model/utils.py:92-101
    g = torch.Generator().manual_seed(5)
    for B in (1, 2, 4, 7, 3):
        v = torch.randn(B, 6, generator=g, dtype=torch.float64)
        out[f"rot6d_in_b{B}"], out[f"rot6d_out_b{B}"] = v.numpy(), ref_rot(v).numpy()
    # FlameRegression fp64: outputs and the reference-owned intermediates (BiFPN levels, fusion layer)
    sd = synthetic_state_dict(3)
    m = R.flame_regression(sd, dtype=torch.float64)
    x = torch.randn(1, 3, 256, 256, generator=torch.Generator().manual_seed(9)).double()
    grabbed = {}
    hooks = [m.bifpn.register_forward_hook(lambda mod, i, o: grabbed.__setitem__("bifpn", o)),
             m.fusion_layer.register_forward_hook(lambda mod, i, o: grabbed.__setitem__("fusion", o))]
    with torch.no_grad():
        ref = m(x)
    for h in hooks:
        h.remove()
    stages = dict(ref)
    stages.update({f"p{i + 3}_out": t for i, t in enumerate(grabbed["bifpn"])})
    stages["fusion"] = grabbed["fusion"]
    for i, (k, t) in enumerate(sorted(stages.items())):
        idx = element_sample(t.numel(), 100 + i)
        out[f"encoder_{k}_shape"] = np.asarray(t.shape)
        out[f"encoder_{k}_index"] = idx
        out[f"encoder_{k}"] = t.reshape(-1)[idx].numpy()
    # FaceMeshPredictor.__call__ on landscape / portrait / tiny / square inputs
    pred = R.predictor(synthetic_state_dict(0))
    g = np.random.default_rng(0)
    for (h, w) in ((300, 517), (641, 203), (97, 131), (256, 256)):
        img = g.integers(0, 256, (h, w, 3), dtype=np.uint8)
        res = pred(img.copy())
        tag = f"{h}x{w}"
        out[f"predictor_{tag}_params"] = res["3dmm_params"].numpy()
        out[f"predictor_{tag}_projected"] = res["projected_vertices"][..., vs, :].numpy()
        out[f"predictor_{tag}_vertices3d"] = res["3d_vertices"][..., vs, :].numpy()
        out[f"predictor_{tag}_points"] = res["points"]
    own = sorted(k for k in R.flame_regression(synthetic_state_dict(1)).state_dict() if not k.endswith("num_batches_tracked"))
    out["state_dict_names"] = np.asarray(own)
    # inference/pncc_estimator.py over the reference's own C++ rasteriser (oracle/_ref/libsim3dr_ref.so)
    import importlib
    est = importlib.import_module("inference.pncc_estimator").PNCCEstimator()
    import Sim3DR
    assert "ref_shims" in Sim3DR.__file__
    z = np.load(os.path.join(GOLD, "reference_predictor.npz"))
    image = np.full((640, 420, 3), 7, np.uint8)
    out["pncc_image"] = est(image, {"3dmm_params": torch.from_numpy(z["params_3dmm"]).clone()}, with_background=True)
    out["pncc_colors"] = np.asarray(est.colors, np.float32)
    out["pncc_faces"] = np.asarray(est.faces_wo_back_remapped)
    _save("reference_live.npz", out)


def product_golden():
    import cv2
    from dad_3dheads_b200.encoder_weights import synthetic_state_dict
    vs, dvs = vertex_sample(), vertex_sample(N_VERTEX_SAMPLE // 2)
    out = {"vertex_sample": vs, "decode_vertex_sample": dvs}
    hm = R.head_mesh()
    for B in (1, 2, 64, 129):
        p = sample_params(B, seed=40 + B)                       # stored as a checksum: the test draws the same params
        q = p.clone()
        out[f"decode_params_sha256_b{B}"] = sha(p.numpy())
        out[f"decode_vertices3d_b{B}"] = hm.vertices_3d(p.clone())[:, dvs].numpy()
        out[f"decode_projected2d_b{B}"] = hm.reprojected_vertices(q, to_2d=True)[:, dvs].numpy()
        changed = (q != p).any(0).nonzero().flatten().tolist()
        assert set(changed) <= {411}, changed                  # head_mesh.py:41 zeroes tz in place, nothing else
        out[f"decode_tz_after_reproject_b{B}"] = q[:, 411].numpy()
    m = R.flame_regression(synthetic_state_dict(4), dtype=torch.float64)
    x = torch.randn(3, 3, 256, 256, generator=torch.Generator().manual_seed(31))
    with torch.no_grad():
        want = m(x.double())
    for i, (k, t) in enumerate(sorted(want.items())):
        idx = element_sample(t.numel(), 200 + i)
        out[f"encoder_{k}_index"], out[f"encoder_{k}"] = idx, t.reshape(-1)[idx].numpy()
    pred = R.predictor(synthetic_state_dict(0))
    imgs = [cv2.cvtColor(cv2.imread(os.path.join(GOLD, "demo_head_1.jpeg")), cv2.COLOR_BGR2RGB)]
    g = np.random.default_rng(1)
    imgs += [g.integers(0, 256, s + (3,), dtype=np.uint8) for s in ((300, 517), (641, 203), (256, 256))]
    for i, img in enumerate(imgs):
        res = pred(img.copy())
        meta = {k: {"shape": list(v.shape), "tensor": torch.is_tensor(v), "dtype": str(v.dtype),
                    "kind": None if torch.is_tensor(v) else v.dtype.kind} for k, v in res.items()}
        out[f"predictor_{i}_meta"] = np.asarray(json.dumps(meta))
        out[f"predictor_{i}_params"] = res["3dmm_params"].numpy()
        out[f"predictor_{i}_vertices3d"] = res["3d_vertices"][..., vs, :].numpy()
        out[f"predictor_{i}_projected"] = res["projected_vertices"][..., vs, :].numpy()
        out[f"predictor_{i}_points"] = res["points"]
    # predictor.py:109-113: the heat-map arg-max branch of _parse_output
    g = torch.Generator().manual_seed(3)
    hmap = torch.randn(1, 68, 64, 64, generator=g)
    p = torch.randn(1, 413, generator=g)
    lm, p3 = pred._parse_output({"OUTPUT_3DMM_PARAMS": p.clone(), "OUTPUT_LANDMARKS_HEATMAP": hmap.clone()})
    out["heatmap_fallback_landmarks"], out["heatmap_fallback_params"] = np.asarray(lm), p3.numpy()
    _save("reference_product.npz", out)


def rasterizer_golden():
    """Sim3DR's rasterize / get_normal (the reference's rasterize_kernel.cpp, oracle/_ref/libsim3dr_ref.so) on the scenes of
    tests/test_rasterizer_{cpu,gpu}.py.  Images are stored as XOR with their seeded background, which compresses to the head."""
    from tests import test_rasterizer_gpu as T
    from tests.test_rasterizer_cpu import small_scene
    out = {}
    v, t, c = small_scene()
    img, depth = T._ref_rasterize(v, t, c, np.zeros((24, 28, 3), np.uint8))
    out["small_image"], out["small_depth"] = img, depth
    for size, reverse, seed in T.RASTER_CASES:
        v, faces, _ = T._mesh(seed, size)
        colors, bg = T._scene(v, seed, size)
        want, _ = T._ref_rasterize(v, faces, colors, bg, reverse)
        out[f"raster_{size}_vertices"] = v
        out[f"raster_{size}_xor_bg"] = want ^ bg
        out[f"raster_{size}_one_channel"], _ = T._ref_rasterize(v, faces, colors[:, :1].copy(),
                                                                np.zeros((size, size, 1), np.uint8), reverse)
    v, t, c = T.tie_scene()
    out["ties_image"], out["ties_depth"] = T._ref_rasterize(v, t, c, np.zeros((32, 32, 3), np.uint8))
    v, faces, _ = T._mesh(4, 256)
    want = np.zeros_like(v)
    T._ref().sim3dr_ref_get_normal(want.ctypes.data, np.ascontiguousarray(v).ctypes.data,
                                   np.ascontiguousarray(faces).ctypes.data, v.shape[0], faces.shape[0])
    out["normals_vertices"], out["normals"] = v, want
    _save("reference_rasterizer.npz", out)


def evaluator_golden():
    """DADEvaluator (dad_3dheads_benchmark/benchmark.py, through oracle/run_ref_benchmark.py) on make_pairs(3, seed=1) and
    make_pairs(5, seed=2)."""
    import subprocess
    import tempfile
    from tests.eval_fixtures import make_pairs
    out = {}
    for n, seed in ((3, 1), (5, 2)):
        gts, sub = make_pairs(n, seed=seed)
        with tempfile.TemporaryDirectory() as d:
            json.dump(gts, open(os.path.join(d, "gt.json"), "w"))
            json.dump(sub, open(os.path.join(d, "sub.json"), "w"))
            subprocess.run([sys.executable, "-W", "ignore", os.path.join(ROOT, "oracle", "run_ref_benchmark.py"),
                            os.path.join(d, "gt.json"), os.path.join(d, "sub.json"), os.path.join(d, "ref.json")], check=True)
            out[f"pairs_{n}_seed_{seed}"] = json.load(open(os.path.join(d, "ref.json")))
    with open(os.path.join(GOLD, "reference_evaluator.json"), "w") as f:
        json.dump(out, f, indent=1, sort_keys=True)


if __name__ == "__main__":
    assert R.available(), "needs /root/reference or oracle/_ref"
    print("reference:", R.root(), R.kind())
    flame_golden()
    encoder_golden()
    predictor_golden()
    assets_golden()
    live_golden()
    product_golden()
    rasterizer_golden()
    evaluator_golden()

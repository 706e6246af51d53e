"""-m "not gpu": host-side pieces of the rasteriser row (SURVEY 8f row 4) -- the CSR adjacency the GPU vertex-normal kernel walks,
and the oracle itself: the output of the reference's own C++ rasteriser (Sim3DR/lib/rasterize_kernel.cpp, stored in
tests/golden/reference_rasterizer.npz) agrees with a plain numpy restatement of its per-pixel rule on a small scene
(rasterize_kernel.cpp:219-292: barycentric inside test, depth = weighted vertex depth, strictly-greater z test, colour = weighted
vertex colours)."""
import os

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = os.path.join(ROOT, "tests", "golden", "reference_rasterizer.npz")


def test_vertex_adjacency_is_the_ascending_incidence_list():
    from dad_3dheads_b200.rasterizer import vertex_adjacency
    g = np.random.default_rng(0)
    tri = g.integers(0, 40, (200, 3)).astype(np.int32)          # repeated vertices inside a triangle included
    off, adj = vertex_adjacency(tri, 50)
    assert off.dtype == np.int32 and adj.dtype == np.int32 and off[0] == 0 and off[-1] == 600 and len(off) == 51
    for v in range(50):
        want = sorted(t for t in range(200) for k in range(3) if tri[t, k] == v)
        assert list(adj[off[v]:off[v + 1]]) == want


def _weights(px, py, p0, p1, p2):
    v0, v1, v2 = p2 - p0, p1 - p0, np.array([px, py], np.float32) - p0
    d00, d01, d02, d11, d12 = v0 @ v0, v0 @ v1, v0 @ v2, v1 @ v1, v1 @ v2
    den = d00 * d11 - d01 * d01
    inv = 0.0 if den == 0 else 1.0 / den
    u, v = (d11 * d02 - d01 * d12) * inv, (d00 * d12 - d01 * d02) * inv
    return np.array([1 - u - v, v, u], np.float32)


def small_scene():
    """Two overlapping triangles over a 24x28 image, with per-vertex colours."""
    v = np.array([[2, 3, 1.0], [20, 4, 2.0], [6, 19, 3.0], [25, 22, 0.5], [3, 21, 5.0], [22, 2, 4.0]], np.float32)
    t = np.array([[0, 1, 2], [3, 4, 5]], np.int32)
    c = np.random.default_rng(1).random((6, 3)).astype(np.float32)
    return v, t, c


def test_reference_rasteriser_matches_its_per_pixel_rule():
    h, w = 24, 28
    v, t, c = small_scene()
    z = np.load(GOLD)
    img, depth = z["small_image"], z["small_depth"]
    want = np.zeros((h, w, 3), np.float32)
    zbuf = np.zeros((h, w), np.float32) - 1e8
    for tri in t:
        p = v[tri]
        x0, x1 = max(int(np.ceil(p[:, 0].min())), 0), min(int(np.floor(p[:, 0].max())), w - 1)
        y0, y1 = max(int(np.ceil(p[:, 1].min())), 0), min(int(np.floor(p[:, 1].max())), h - 1)
        for y in range(y0, y1 + 1):
            for x in range(x0, x1 + 1):
                wt = _weights(x, y, p[0, :2], p[1, :2], p[2, :2])
                if wt[0] > 0 and wt[1] > 0 and wt[2] > 0:
                    z = float(wt @ p[:, 2])
                    if z > zbuf[y, x]:
                        zbuf[y, x] = z
                        want[y, x] = 255.0 * (wt @ c[tri])
    covered = zbuf > -1e8
    assert covered.sum() > 150 and np.array_equal(covered, depth > -1e8)
    assert np.abs(img.astype(np.float32)[covered] - want[covered]).max() <= 1.0       # uint8 truncation of the same float
    assert np.allclose(depth[covered], zbuf[covered], rtol=1e-6)

"""-m gpu: the GPU rasteriser (csrc/rasterize.cu through the C ABI) against the reference's own C++ rasteriser -- the unmodified
Sim3DR/lib/rasterize_kernel.cpp compiled by oracle/build_ref.py into oracle/_ref/libsim3dr_ref.so, whose outputs on these scenes
are stored in tests/golden/reference_rasterizer.npz (tools/make_reference_golden.py).  Bit-exact: image bytes, depth buffer bits
and vertex-normal bits are identical."""
import ctypes as C
import os

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF_SO = os.path.join(ROOT, "oracle", "_ref", "libsim3dr_ref.so")
GOLD = os.path.join(ROOT, "tests", "golden", "reference_rasterizer.npz")
RASTER_CASES = [(256, False, 1), (512, True, 2), (700, False, 3)]


def _ref():
    lib = C.CDLL(REF_SO)
    lib.sim3dr_ref_rasterize.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int,
                                         C.c_int, C.c_float, C.c_int]
    lib.sim3dr_ref_get_normal.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int]
    return lib


def _ref_rasterize(v, t, c, bg, reverse=False):
    lib = _ref()
    h, w, ch = bg.shape
    img = np.ascontiguousarray(bg.copy())
    depth = np.zeros((h, w), np.float32) - 1e8
    v, t, c = np.ascontiguousarray(v, np.float32), np.ascontiguousarray(t, np.int32), np.ascontiguousarray(c, np.float32)
    lib.sim3dr_ref_rasterize(img.ctypes.data, v.ctypes.data, t.ctypes.data, c.ctypes.data, depth.ctypes.data, t.shape[0], h, w, ch,
                             1.0, 1 if reverse else 0)
    return img, depth


def _mesh(seed, size):
    """A posed FLAME head projected into a size x size image (what pncc_estimator.py:72-79 feeds the rasteriser)."""
    from dad_3dheads_b200.flame import load_flame_static
    from oracle.flame_oracle import FlameOracle, sample_params
    st = load_flame_static()
    p = sample_params(1, seed=seed)
    p[:, 409:411] *= 0.3
    v = FlameOracle(st, image_size=size).reprojected_vertices(p, to_2d=False)[0].numpy().astype(np.float32)
    v[:, 2] *= -1
    return v, st["faces"].astype(np.int32), st


def _scene(v, seed, size):
    """Per-vertex colours and a random background for a rasteriser case."""
    g = np.random.default_rng(seed)
    colors = g.random((v.shape[0], 3)).astype(np.float32)
    bg = g.integers(0, 256, (size, size + 17, 3), dtype=np.uint8)
    return colors, bg


def tie_scene():
    """Coplanar duplicate triangles, a zero-area triangle, one outside the image and a plain one over 32x32."""
    v = np.array([[2, 2, 5], [30, 3, 5], [4, 28, 5], [2, 2, 5], [30, 3, 5], [4, 28, 5], [10, 10, 1], [10, 10, 1], [10, 10, 1],
                  [-50, -50, 9], [-40, -50, 9], [-50, -40, 9], [5, 5, 7], [20, 6, 2], [6, 22, 9]], np.float32)
    t = np.array([[3, 4, 5], [0, 1, 2], [6, 7, 8], [9, 10, 11], [12, 13, 14]], np.int32)
    c = np.random.default_rng(0).random((15, 3)).astype(np.float32)
    return v, t, c


@pytest.mark.parametrize("size,reverse,seed", RASTER_CASES)
def test_rasterize_bit_exact(cuda_device, size, reverse, seed):
    from dad_3dheads_b200.rasterizer import rasterize
    z = np.load(GOLD)
    v, faces, st = _mesh(seed, size)
    assert np.array_equal(v, z[f"raster_{size}_vertices"])                # the scene the reference rasterised
    colors, bg = _scene(v, seed, size)
    want = z[f"raster_{size}_xor_bg"] ^ bg
    got = rasterize(v, faces, colors, bg=bg.copy(), reverse=reverse)
    assert got.dtype == np.uint8 and np.array_equal(got, want)
    assert (want != bg).mean() > 0.003                                    # the head covers a visible part of the image
    # black background by size, one channel
    c1 = colors[:, :1].copy()
    got1 = rasterize(v, faces, c1, height=size, width=size, channel=1, reverse=reverse)
    assert np.array_equal(got1, z[f"raster_{size}_one_channel"])


def test_rasterize_depth_ties_and_degenerate_triangles(cuda_device):
    """Coplanar duplicate triangles (equal depth: the lowest index must win, as in the sequential loop), zero-area triangles,
    triangles outside the image, and the depth buffer itself."""
    from dad_3dheads_b200 import _lib
    lib = _lib.load()
    v, t, c = tie_scene()
    z = np.load(GOLD)
    want, want_depth = z["ties_image"], z["ties_depth"]
    dev = torch.device("cuda", 0)
    img = torch.zeros(32, 32, 3, dtype=torch.uint8, device=dev)
    depth = torch.full((32, 32), -1e8, dtype=torch.float32, device=dev)
    key = torch.empty(32 * 32, dtype=torch.int64, device=dev)
    tv, tt, tc = torch.from_numpy(v).to(dev), torch.from_numpy(t).to(dev), torch.from_numpy(c).to(dev)
    _lib.check(lib.dad3d_rasterize(tv.data_ptr(), tt.data_ptr(), tc.data_ptr(), 5, img.data_ptr(), depth.data_ptr(), key.data_ptr(),
                                   32, 32, 3, 0, torch.cuda.current_stream(dev).cuda_stream), "dad3d_rasterize")
    assert np.array_equal(img.cpu().numpy(), want)
    assert np.array_equal(depth.cpu().numpy().view(np.uint32), want_depth.view(np.uint32))


def test_vertex_normals_bit_exact(cuda_device):
    from dad_3dheads_b200.rasterizer import get_normal
    v, faces, _ = _mesh(4, 256)
    z = np.load(GOLD)
    assert np.array_equal(v, z["normals_vertices"])
    want = z["normals"]
    got = get_normal(v, faces)
    assert np.array_equal(got.view(np.uint32), want.view(np.uint32))
    assert np.allclose(np.linalg.norm(got, axis=1), 1.0, atol=1e-5)

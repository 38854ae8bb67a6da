"""Pins the C oracle (oracle/raster_oracle.c): against the committed golden fixtures produced by running
the reference (tests/golden/make_golden.py), and bit-for-bit against the reference's own C++ CPU ops (their outputs'
digests, stored by tests/golden/make_reference_outputs.py)."""
import numpy as np
import pytest
import torch

import oracle
from helpers import case_key, digest, rand_faces, rand_points, reference_outputs, upstream

MESH_CPP = lambda g: sorted(k for k in g if k.startswith("mesh/") and "/cpp" in k)  # noqa: E731
MESH_PY = lambda g: sorted(k for k in g if k.startswith("mesh/") and "/python" in k)  # noqa: E731
POINTS = lambda g: sorted(k for k in g if k.startswith("points/"))  # noqa: E731


def _run_mesh(c, **kw):
    H, W, K, persp, clip, cull = (int(v) for v in c["args"])
    return oracle.rasterize_meshes(c["face_verts"], c["first"], c["num"], (H, W), float(c["blur"][0]), K, persp,
                                   clip, cull, **kw)


def test_golden_mesh_cpp_bit_exact(golden):
    """Every reference known-answer scene + seeded random scene, C++ CPU op outputs: bit-exact."""
    names = MESH_CPP(golden)
    assert len(names) >= 10
    for name in names:
        c = golden[name]
        o = _run_mesh(c, arith=oracle.ARITH_CPU, select=oracle.SELECT_CPU)
        assert np.array_equal(o[0], c["pix_to_face"]), name
        assert np.array_equal(o[1], c["zbuf"]), name
        assert np.array_equal(o[2], c["bary"]), name
        assert np.array_equal(o[3], c["dists"]), name


def test_golden_mesh_python_impl(golden):
    """The reference's pure-python implementation agrees on indices; floats to its own test tolerance."""
    for name in MESH_PY(golden):
        c = golden[name]
        o = _run_mesh(c, arith=oracle.ARITH_CPU, select=oracle.SELECT_CPU)
        assert np.array_equal(o[0], c["pix_to_face"]), name
        np.testing.assert_allclose(o[1], c["zbuf"], rtol=1e-4, atol=1e-6, err_msg=name)
        np.testing.assert_allclose(o[2], c["bary"], rtol=1e-3, atol=1e-5, err_msg=name)
        np.testing.assert_allclose(o[3], c["dists"], rtol=6e-3, atol=1e-6, err_msg=name)


def test_golden_mesh_cuda_flavour_same_indices(golden):
    """The CUDA-flavoured arithmetic / queue must agree with the goldens on these razor-free scenes
    (the reference's own CUDA tests assert exactly this)."""
    for name in MESH_CPP(golden):
        c = golden[name]
        o = _run_mesh(c, arith=oracle.ARITH_CUDA, select=oracle.SELECT_CUDA)
        assert np.array_equal(o[0], c["pix_to_face"]), name
        np.testing.assert_allclose(o[1], c["zbuf"], rtol=1e-4, atol=1e-6, err_msg=name)
        np.testing.assert_allclose(o[3], c["dists"], rtol=6e-3, atol=1e-6, err_msg=name)


def test_golden_mesh_backward(golden):
    for name in MESH_CPP(golden):
        c = golden[name]
        if "grad_face_verts" not in c:
            continue
        _, _, K, persp, clip, _ = (int(v) for v in c["args"])
        g = oracle.rasterize_meshes_backward(c["face_verts"], c["pix_to_face"], c["grad_zbuf"], c["grad_bary"],
                                             c["grad_dists"], persp, clip, arith=oracle.ARITH_CPU)
        assert np.array_equal(g, c["grad_face_verts"]), name


def test_golden_points(golden):
    names = POINTS(golden)
    assert len(names) >= 5
    for name in names:
        c = golden[name]
        H, W, K = (int(v) for v in c["args"])
        o = oracle.rasterize_points(c["points"], c["first"], c["num"], (H, W), c["radius"], K,
                                    arith=oracle.ARITH_CPU, select=oracle.SELECT_CPU)
        assert np.array_equal(o[0], c["idx"]), name
        assert np.array_equal(o[1], c["zbuf"]), name
        assert np.array_equal(o[2], c["dists"]), name
        if "grad_points" in c:
            g = oracle.rasterize_points_backward(c["points"], c["idx"], c["grad_zbuf"], c["grad_dists"])
            assert np.array_equal(g, c["grad_points"]), name


REF_MESH_CASES = [  # persp, clip, cull, blur, K, H, W
    (0, 0, 0, 0.0, 4, 32, 32), (1, 0, 0, 1e-3, 8, 33, 47), (0, 1, 1, 1e-2, 3, 64, 40), (1, 1, 0, 1e-4, 8, 48, 48),
    (1, 1, 1, 0.05, 150, 16, 16)]
REF_POINT_CASES = [(1, 16, 16), (5, 32, 48), (10, 40, 24)]  # K, H, W


def neighbor_table():
    nb = torch.full((300,), -1, dtype=torch.int64)
    nb[0:100:2] = torch.arange(1, 100, 2)
    nb[1:100:2] = torch.arange(0, 100, 2)
    return nb


@pytest.fixture(scope="module")
def ref_cpu():
    """Digests of the reference's C++ CPU ops on these seeded scenes (tests/golden/make_reference_outputs.py cpu)."""
    return reference_outputs("reference_cpu")


@pytest.mark.parametrize("persp,clip,cull,blur,K,H,W", REF_MESH_CASES)
def test_oracle_equals_reference_cpu_meshes(ref_cpu, persp, clip, cull, blur, K, H, W):
    want = ref_cpu[case_key("meshes", persp, clip, cull, blur, K, H, W)]
    fv, first, num = rand_faces(400, 2, seed=K + H)
    o = oracle.rasterize_meshes(fv.numpy(), first.numpy(), num.numpy(), (H, W), blur, K, persp, clip, cull)
    assert digest(*o) == str(want["forward"])
    gz, gb, gd = upstream([o[1].shape, o[2].shape, o[3].shape])
    og = oracle.rasterize_meshes_backward(fv.numpy(), o[0], gz.numpy(), gb.numpy(), gd.numpy(), persp, clip)
    assert digest(og) == str(want["backward"])


def test_oracle_equals_reference_cpu_neighbors(ref_cpu):
    """clipped_faces_neighbor_idx semantics (rasterize_meshes_cpu.cpp:249-277)."""
    fv, first, num = rand_faces(300, 1, seed=7, scale=0.35)
    o = oracle.rasterize_meshes(fv.numpy(), first.numpy(), num.numpy(), (32, 32), 1e-2, 4,
                                clipped_faces_neighbor_idx=neighbor_table().numpy())
    assert digest(*o) == str(ref_cpu["neighbors"]["forward"])


@pytest.mark.parametrize("K,H,W", REF_POINT_CASES)
def test_oracle_equals_reference_cpu_points(ref_cpu, K, H, W):
    want = ref_cpu[case_key("points", K, H, W)]
    pts, first, num, rad = rand_points(1500, 2, seed=K)
    o = oracle.rasterize_points(pts.numpy(), first.numpy(), num.numpy(), (H, W), rad.numpy(), K)
    assert digest(*o) == str(want["forward"])
    gz, gd = upstream([o[1].shape, o[2].shape])
    og = oracle.rasterize_points_backward(pts.numpy(), o[0], gz.numpy(), gd.numpy())
    assert digest(og) == str(want["backward"])


def test_oracle_flavours_agree_without_ties():
    """CPU-form and CUDA-form queues select the same faces when no z tie straddles the K-th slot."""
    fv, first, num = rand_faces(300, 2, seed=3)
    a = oracle.rasterize_meshes(fv.numpy(), first.numpy(), num.numpy(), (24, 24), 1e-3, 3, arith=oracle.ARITH_CUDA,
                                select=oracle.SELECT_CPU)
    b = oracle.rasterize_meshes(fv.numpy(), first.numpy(), num.numpy(), (24, 24), 1e-3, 3, arith=oracle.ARITH_CUDA,
                                select=oracle.SELECT_CUDA)
    for x, y in zip(a, b):
        assert np.array_equal(x, y)


def test_oracle_row_ranges_compose():
    fv, first, num = rand_faces(200, 1, seed=5)
    full = oracle.rasterize_meshes(fv.numpy(), first.numpy(), num.numpy(), (20, 20), 1e-3, 2)
    top = oracle.rasterize_meshes(fv.numpy(), first.numpy(), num.numpy(), (20, 20), 1e-3, 2, rows=(0, 7))
    assert np.array_equal(full[0][:, :7], top[0][:, :7])
    assert (top[0][:, 7:] == -1).all()

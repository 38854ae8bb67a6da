"""Parity of the CUDA path (called through the C ABI) with the oracle, the golden fixtures and the reference's own CUDA
kernels (their outputs on these seeded inputs, stored by tests/golden/make_reference_outputs.py).

Bar: pix_to_face / idx bit-exact; zbuf / bary / dists bit-exact too against the CUDA-flavoured oracle
(identical arithmetic), <= 1e-5 against fixtures produced by the reference's CPU build; gradients within
the reference's own cross-implementation tolerances (tests/test_rasterize_meshes.py:543-594)."""
import numpy as np
import pytest
import torch

import oracle
from helpers import assert_frag_equal, case_key, digest, rand_faces, rand_points, reference_outputs, split, upstream

pytestmark = pytest.mark.gpu

CUDA = dict(arith=oracle.ARITH_CUDA, select=oracle.SELECT_CUDA)


@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch.device("cuda:0")


@pytest.fixture(scope="module")
def ops(built_lib):
    from pytorch3d_b200 import _C
    return _C


@pytest.fixture(scope="module")
def ref_cuda():
    return reference_outputs("reference_cuda")


def run_mesh(ops, dev, fv, first, num, size, blur, K, persp=0, clip=0, cull=0, nb=None):
    if nb is None:
        nbt = torch.full((fv.shape[0],), -1, dtype=torch.int64, device=dev)
        nbt._b200_all_minus_one = True
    else:
        nbt = nb.to(dev)
    return ops.rasterize_meshes(fv.to(dev), first.to(dev), num.to(dev), nbt, size, blur, K, 0, 0, bool(persp),
                                bool(clip), bool(cull))


MESH_MATRIX = [  # persp, clip, cull, blur, K, H, W, F, N
    (0, 0, 0, 0.0, 4, 32, 32, 500, 2),
    (1, 0, 0, 1e-3, 8, 33, 47, 500, 2),
    (0, 1, 1, 1e-2, 3, 64, 40, 500, 2),
    (1, 1, 0, 1e-4, 8, 48, 48, 500, 2),
    (0, 0, 0, 1e-4, 8, 128, 128, 6000, 3),
    (0, 0, 1, 0.0, 1, 17, 100, 800, 1),
    (0, 0, 0, 1e-3, 2, 100, 17, 800, 4),
    (1, 1, 1, 0.05, 20, 40, 40, 300, 1),
    (0, 0, 0, 1e-3, 150, 24, 24, 400, 1),
    (0, 0, 0, 1e-2, 5, 31, 31, 300, 1),
    (0, 0, 0, 1e-2, 7, 16, 16, 300, 1),
    (0, 0, 0, 1e-2, 9, 16, 16, 300, 1),
    # no blur (scan-conversion path) on images with partial tiles and odd widths: paired stores, empty tiles
    (0, 0, 0, 0.0, 8, 33, 47, 500, 2),
    (1, 0, 0, 0.0, 4, 31, 45, 800, 3),
    (0, 1, 0, 0.0, 2, 50, 19, 400, 1),
    (0, 0, 0, 0.0, 8, 100, 70, 30, 2),
    (0, 0, 1, 0.0, 6, 70, 100, 2000, 2),
    # 8 < K <= 32: queue keys in shared memory (mesh_fine_smemq_kernel); K % 8 == 0 takes the paired group stores
    (0, 0, 0, 1e-3, 16, 48, 48, 600, 2),
    (1, 0, 0, 0.0, 16, 33, 47, 500, 2),
    (0, 1, 0, 1e-2, 32, 40, 40, 400, 1),
    (0, 0, 0, 0.0, 24, 64, 64, 1500, 1),
    (1, 1, 1, 1e-2, 12, 31, 45, 600, 3),
    (0, 0, 0, 1e-3, 40, 24, 24, 300, 1),
    # tile lists longer than one chunk: sorted by the CTA in shared memory (3000 faces on 4 tiles) ...
    (0, 0, 0, 1e-2, 8, 32, 32, 3000, 1),
    (0, 0, 0, 0.0, 4, 32, 32, 3000, 1),
    (0, 0, 0, 1e-2, 16, 32, 32, 3000, 1),
    # ... or, beyond the kernel's shared memory, in place in global memory (20000 faces on one tile)
    (0, 0, 0, 1e-3, 2, 16, 16, 20000, 1),
    (0, 0, 0, 1e-3, 40, 16, 16, 6000, 1),
]


@pytest.mark.parametrize("persp,clip,cull,blur,K,H,W,F,N", MESH_MATRIX)
def test_mesh_forward_equals_oracle(ops, dev, persp, clip, cull, blur, K, H, W, F, N):
    fv, first, num = rand_faces(F, N, seed=K + H)
    mine = run_mesh(ops, dev, fv, first, num, (H, W), blur, K, persp, clip, cull)
    o = oracle.rasterize_meshes(fv.numpy(), first.numpy(), num.numpy(), (H, W), blur, K, persp, clip, cull, **CUDA)
    assert_frag_equal(mine, o, "mine vs oracle")


def test_mesh_forward_structured_with_z_ties(ops, dev, ref_cuda):
    """Two tori at 256^2, blur 1e-4, K=8: hundreds of exact z ties straddle the K-th slot here; the
    reference-CUDA queue semantics + ascending face order must still be reproduced bit-for-bit."""
    from pytorch3d_b200 import synthetic
    m = synthetic.torus_batch(2, 54, 54, seed=0)
    fv, first, num = synthetic.face_verts_of(m), m.mesh_to_faces_packed_first_idx(), m.num_faces_per_mesh()
    mine = run_mesh(ops, dev, fv, first, num, (256, 256), 1e-4, 8)
    o = oracle.rasterize_meshes(fv.numpy(), first.numpy(), num.numpy(), (256, 256), 1e-4, 8, **CUDA)
    assert_frag_equal(mine, o, "torus vs oracle")
    lex = oracle.rasterize_meshes(fv.numpy(), first.numpy(), num.numpy(), (256, 256), 1e-4, 8,
                                  arith=oracle.ARITH_CUDA, select=oracle.SELECT_CPU)
    assert (lex[0] != o[0]).sum() > 0, "scene is expected to contain ties (guards the test's purpose)"
    assert digest(*mine) == str(ref_cuda["torus_ties"]["forward"]), "torus vs reference CUDA (naive)"


def test_config1_ico_sphere(ops, dev):
    """BASELINE config 1: ico_sphere(level=4), batch 1, 64^2, K=1."""
    from pytorch3d_b200 import synthetic
    m = synthetic.ico_sphere_batch(1, 4)
    fv, first, num = synthetic.face_verts_of(m), m.mesh_to_faces_packed_first_idx(), m.num_faces_per_mesh()
    mine = run_mesh(ops, dev, fv, first, num, (64, 64), 0.0, 1)
    o = oracle.rasterize_meshes(fv.numpy(), first.numpy(), num.numpy(), (64, 64), 0.0, 1, **CUDA)
    assert_frag_equal(mine, o)
    assert (mine[0] >= 0).sum() > 1000


def test_mesh_golden_fixtures(ops, dev, golden):
    names = sorted(k for k in golden if k.startswith("mesh/") and "/cpp" in k)
    for name in names:
        c = golden[name]
        H, W, K, persp, clip, cull = (int(v) for v in c["args"])
        mine = run_mesh(ops, dev, torch.from_numpy(c["face_verts"]), torch.from_numpy(c["first"]),
                        torch.from_numpy(c["num"]), (H, W), float(c["blur"][0]), K, persp, clip, cull)
        assert np.array_equal(mine[0].cpu().numpy(), c["pix_to_face"]), name
        for got, want in zip(mine[1:], (c["zbuf"], c["bary"], c["dists"])):
            err = np.abs(got.cpu().numpy() - want)
            # Known-answer scenes of the reference: 1e-5 absolute (the north-star bar).  The seeded random
            # scenes contain sliver faces and (with perspective correction, no clipping) extrapolated
            # barycentrics up to 1e10; the fixtures come from the reference's non-FMA CPU arithmetic, so there
            # the reference's own cross-implementation tolerance applies (test_rasterize_meshes.py:543-594).
            if "/random/" in name:
                tol = 1e-5 + 1e-3 * np.abs(want)
            else:
                tol = np.full_like(want, 1e-5)
            assert (err <= tol).all(), name


@pytest.mark.parametrize("persp,clip,cull,blur,K,H,W,F,N", MESH_MATRIX[:6])
def test_mesh_forward_equals_reference_cuda(ops, dev, ref_cuda, persp, clip, cull, blur, K, H, W, F, N):
    fv, first, num = rand_faces(F, N, seed=K + H)
    mine = run_mesh(ops, dev, fv, first, num, (H, W), blur, K, persp, clip, cull)
    want = ref_cuda[case_key("mesh_forward", persp, clip, cull, blur, K, H, W, F, N)]["forward"]
    assert digest(*mine) == str(want), "mine vs reference CUDA naive"


def test_mesh_edge_cases(ops, dev):
    # empty mesh in the middle of the batch, faces behind the camera, degenerate faces, huge faces
    fv, _, _ = rand_faces(200, 1, seed=11, scale=0.3)
    fv[10:20, :, 2] = -1.0                       # behind the camera
    fv[20:30, 1] = fv[20:30, 0]                  # zero area
    fv[30] = torch.tensor([[-5.0, -5.0, 1.0], [5.0, -5.0, 1.2], [0.0, 6.0, 1.4]])  # covers everything
    fv[31] = torch.tensor([[-5.0, -5.0, 0.9], [0.0, 6.0, 1.1], [5.0, -5.0, 1.3]])  # back-facing twin
    first = torch.tensor([0, 100, 100], dtype=torch.int64)
    num = torch.tensor([100, 0, 100], dtype=torch.int64)
    for cull in (0, 1):
        mine = run_mesh(ops, dev, fv, first, num, (40, 56), 1e-3, 4, cull=cull)
        o = oracle.rasterize_meshes(fv.numpy(), first.numpy(), num.numpy(), (40, 56), 1e-3, 4, cull_backfaces=cull,
                                    **CUDA)
        assert_frag_equal(mine, o, "edge cases cull=%d" % cull)
        assert (mine[0][1] == -1).all()  # the empty mesh renders nothing
    # no faces at all / zero-size outputs
    e = run_mesh(ops, dev, torch.zeros(0, 3, 3), torch.zeros(1, dtype=torch.int64), torch.zeros(1, dtype=torch.int64),
                 (8, 8), 0.0, 2)
    assert e[0].shape == (1, 8, 8, 2) and (e[0] == -1).all() and (e[1] == -1).all() and (e[2] == -1).all()
    z = run_mesh(ops, dev, fv, first, num, (8, 8), 0.0, 0)
    assert z[0].shape == (3, 8, 8, 0)


def test_mesh_pair_overflow_falls_back_exactly(ops, dev):
    """With a deliberately tiny pair buffer most tiles overflow and rasterise from the full mesh range:
    the result must not change (the reference drops faces in this situation, rasterize_coarse.cu:186-201)."""
    fv, first, num = rand_faces(600, 2, seed=5, scale=0.5)
    full = run_mesh(ops, dev, fv, first, num, (64, 64), 1e-3, 4)
    ops.PAIR_CAPACITY = 64
    try:
        small = run_mesh(ops, dev, fv, first, num, (64, 64), 1e-3, 4)
    finally:
        ops.PAIR_CAPACITY = 0
    assert_frag_equal(full, small, "overflow fallback")


def test_mesh_clipped_neighbors(ops, dev):
    fv, first, num = rand_faces(300, 1, seed=7, scale=0.35)
    nb = torch.full((300,), -1, dtype=torch.int64)
    nb[0:100:2] = torch.arange(1, 100, 2)
    nb[1:100:2] = torch.arange(0, 100, 2)
    for K in (4, 12):
        mine = run_mesh(ops, dev, fv, first, num, (32, 32), 1e-2, K, nb=nb)
        o = oracle.rasterize_meshes(fv.numpy(), first.numpy(), num.numpy(), (32, 32), 1e-2, K,
                                    clipped_faces_neighbor_idx=nb.numpy(), **CUDA)
        assert_frag_equal(mine, o, "neighbours K=%d" % K)


def test_more_images_than_grid_z(ops, dev):
    """The fine / backward kernels use grid = (tiles x, tiles y, images): batches of more than 65535 images are
    rendered in slices.  65538 one-triangle meshes / one-point clouds on 16x16 images (one tile each)."""
    N, g = 65535 + 3, torch.Generator().manual_seed(7)
    fv = torch.rand(N, 3, 3, generator=g) * 2 - 1
    fv[..., 2] = 0.5 + torch.rand(N, 3, generator=g)
    first, num = torch.arange(N), torch.ones(N, dtype=torch.int64)
    got = run_mesh(ops, dev, fv, first, num, (16, 16), 0.0, 2)
    want = oracle.rasterize_meshes(fv.numpy(), first.numpy(), num.numpy(), (16, 16), 0.0, 2, **CUDA)
    assert_frag_equal(got, want, "65538 images")
    assert (got[0][-1] >= 0).any() or (want[0][-1] < 0).all()
    gz, gb, gd = (t.to(dev) for t in upstream([want[1].shape, want[2].shape, want[3].shape]))
    grad = ops.rasterize_meshes_backward(fv.to(dev), got[0], gz, gb, gd, False, False).cpu().numpy()
    gref = oracle.rasterize_meshes_backward(fv.numpy(), want[0], gz.cpu().numpy(), gb.cpu().numpy(), gd.cpu().numpy(),
                                            0, 0, arith=oracle.ARITH_CUDA)
    assert np.abs(grad - gref).max() <= 2e-3 * max(np.abs(gref).max(), 1e-6)
    pts = torch.rand(N, 3, generator=g) * 1.6 - 0.8
    pts[:, 2] = 0.5 + torch.rand(N, generator=g)
    rad = torch.full((N,), 0.3)
    pgot = ops.rasterize_points(pts.to(dev), first.to(dev), num.to(dev), (16, 16), rad.to(dev), 1, 0, 0)
    pwant = oracle.rasterize_points(pts.numpy(), first.numpy(), num.numpy(), (16, 16), rad.numpy(), 1, **CUDA)
    assert_frag_equal(pgot, pwant, "65538 clouds")
    pgz, pgd = (t.to(dev) for t in upstream([pwant[1].shape, pwant[2].shape]))
    pgrad = ops.rasterize_points_backward(pts.to(dev), pgot[0], pgz, pgd).cpu().numpy()
    pref = oracle.rasterize_points_backward(pts.numpy(), pwant[0], pgz.cpu().numpy(), pgd.cpu().numpy())
    assert np.abs(pgrad - pref).max() <= 1e-4 * max(np.abs(pref).max(), 1e-6)


BACKWARD_CASES = [(0, 0, 1e-3), (1, 0, 1e-3), (0, 1, 1e-3), (1, 1, 0.0), (1, 1, 1e-3)]  # persp, clip, blur


@pytest.mark.parametrize("persp,clip,blur", BACKWARD_CASES)
def test_mesh_backward(ops, dev, ref_cuda, persp, clip, blur):
    from pytorch3d_b200 import synthetic
    m = synthetic.torus_batch(2, 24, 24, seed=3)
    fv, first, num = synthetic.face_verts_of(m), m.mesh_to_faces_packed_first_idx(), m.num_faces_per_mesh()
    frag = run_mesh(ops, dev, fv, first, num, (64, 64), blur, 4, persp, clip)
    gz, gb, gd = upstream([frag[1].shape, frag[2].shape, frag[3].shape])
    mine = ops.rasterize_meshes_backward(fv.to(dev), frag[0], gz.to(dev), gb.to(dev), gd.to(dev), bool(persp),
                                         bool(clip)).cpu().numpy()
    want = oracle.rasterize_meshes_backward(fv.numpy(), frag[0].cpu().numpy(), gz.numpy(), gb.numpy(), gd.numpy(),
                                            persp, clip, arith=oracle.ARITH_CUDA)
    nf = len(want)
    err = np.abs(mine - want).reshape(nf, -1).max(1)
    mag = np.abs(want).reshape(nf, -1).max(1)
    if persp and clip and blur > 0:
        # Pixels in the blur band of a face are arbitrarily ill-conditioned with BOTH flags (perspective-
        # corrected then clipped barycentrics with near-zero denominators): even the reference's own two
        # arithmetics (FMA / no FMA) disagree by 100% on a few faces.  Require agreement on >= 98% of faces.
        ok = err <= 2e-3 * np.maximum(mag, 1e-3 * np.median(mag))
        assert ok.mean() >= 0.98
        # second witness: the reference's own C++ CPU backward (rasterize_meshes_cpu.cpp:391-532), which applies the clip
        # backward to the corrected barycentrics like this build (its CUDA kernel does not: DESIGN.md 5)
        rc = ref_cuda[case_key("mesh_backward", persp, clip, blur)]["grad_face_verts"]
        err_c = np.abs(mine - rc).reshape(nf, -1).max(1)
        mag_c = np.abs(rc).reshape(nf, -1).max(1)
        ok_c = err_c <= 2e-3 * np.maximum(mag_c, 1e-3 * np.median(mag_c))
        assert ok_c.mean() >= 0.98
        return
    scale = mag.max()
    assert err.max() <= 2e-3 * scale
    np.testing.assert_allclose(mine, want, rtol=2e-3, atol=2e-4 * scale)
    if not (persp and clip):
        # (with both flags the reference CUDA kernel feeds the uncorrected barycentrics to the clip
        # backward, rasterize_meshes.cu:527-529; we follow the forward-consistent CPU form)
        r = ref_cuda[case_key("mesh_backward", persp, clip, blur)]["grad_face_verts"]
        np.testing.assert_allclose(mine, r, rtol=2e-3, atol=2e-4 * scale)


def test_mesh_autograd_wrapper(ops, dev):
    import pytorch3d_b200 as p3b
    from pytorch3d_b200 import synthetic
    m = synthetic.torus_batch(2, 16, 16, seed=1, device=dev)
    m.requires_grad_(True)
    p2f, zbuf, bary, dists = p3b.rasterize_meshes(m, 48, blur_radius=1e-3, faces_per_pixel=3)
    gz, gb, gd = (t.to(dev) for t in upstream([zbuf.shape, bary.shape, dists.shape]))
    ((zbuf * gz).sum() + (bary * gb).sum() + (dists * gd).sum()).backward()
    grad_verts = m.verts_packed().grad
    fv = synthetic.face_verts_of(m).detach().cpu()
    want_fv = oracle.rasterize_meshes_backward(fv.numpy(), p2f.cpu().numpy(), gz.cpu().numpy(), gb.cpu().numpy(),
                                               gd.cpu().numpy(), 0, 0, arith=oracle.ARITH_CUDA)
    want = torch.zeros_like(m.verts_packed().detach().cpu())
    want.index_put_((m.faces_packed().cpu().reshape(-1),), torch.from_numpy(want_fv).reshape(-1, 3), accumulate=True)
    scale = want.abs().max()
    assert (grad_verts.cpu() - want).abs().max() <= 2e-3 * scale
    assert not p2f.requires_grad
    # a loss that uses only one of the outputs: the other gradients arrive as None
    m2 = synthetic.torus_batch(2, 16, 16, seed=1, device=dev)
    m2.requires_grad_(True)
    _, zbuf2, _, _ = p3b.rasterize_meshes(m2, 48, blur_radius=1e-3, faces_per_pixel=3)
    (zbuf2 * gz).sum().backward()
    fv_g = oracle.rasterize_meshes_backward(fv.numpy(), p2f.cpu().numpy(), gz.cpu().numpy(), np.zeros_like(gb.cpu().numpy()),
                                            np.zeros_like(gd.cpu().numpy()), 0, 0, arith=oracle.ARITH_CUDA)
    want2 = torch.zeros_like(want)
    want2.index_put_((m.faces_packed().cpu().reshape(-1),), torch.from_numpy(fv_g).reshape(-1, 3), accumulate=True)
    assert (m2.verts_packed().grad.cpu() - want2).abs().max() <= 2e-3 * max(float(want2.abs().max()), 1e-6)


def test_mesh_indexed_entry_points(ops, dev):
    """The fused (verts, faces) entry points against gather -> op -> scatter done with torch (SURVEY.md 8 f-4)."""
    from pytorch3d_b200 import synthetic
    m = synthetic.torus_batch(3, 20, 14, seed=5, device=dev)
    verts, faces = m.verts_packed(), m.faces_packed()
    first, num = m.mesh_to_faces_packed_first_idx(), m.num_faces_per_mesh()
    V = verts.shape[0]
    for blur, K, persp, clip in [(0.0, 4, 0, 0), (1e-3, 3, 1, 1), (0.0, 12, 0, 0)]:
        fv = verts[faces]
        nb = torch.full((fv.shape[0],), -1, dtype=torch.int64, device=dev)
        want = ops.rasterize_meshes(fv, first, num, nb, (40, 56), blur, K, 0, 0, bool(persp), bool(clip), False)
        got = ops.rasterize_meshes_indexed(verts, faces, first, num, (40, 56), blur, K, bool(persp), bool(clip), False)
        for a, b in zip(got[:4], want):
            assert torch.equal(a, b)
        assert torch.equal(got[4], fv)
        gz, gb, gd = (t.to(dev) for t in upstream([want[1].shape, want[2].shape, want[3].shape]))
        g_fv = ops.rasterize_meshes_backward(fv, want[0], gz, gb, gd, bool(persp), bool(clip))
        g_want = torch.zeros(V, 3, device=dev).index_add_(0, faces.reshape(-1), g_fv.reshape(-1, 3))
        g_got = ops.rasterize_meshes_backward_indexed(got[4], faces, V, got[0], gz, gb, gd, bool(persp), bool(clip))
        assert (g_got - g_want).abs().max() <= 1e-4 * g_want.abs().max()
    # a face with an out-of-range vertex index is never hit; empty inputs
    bad = faces.clone()
    bad[7, 1] = V + 5
    out = ops.rasterize_meshes_indexed(verts, bad, first, num, (32, 32), 0.0, 2, False, False, False)
    assert not (out[0] == 7).any() and torch.isnan(out[4][7, 1]).all()
    e = ops.rasterize_meshes_indexed(verts[:0], faces[:0], first[:0], num[:0], (8, 8), 0.0, 2, False, False, False)
    assert e[0].shape == (0, 8, 8, 2) and e[4].shape == (0, 3, 3)
    z = ops.rasterize_meshes_indexed(verts, faces[:0], torch.zeros(1, dtype=torch.int64, device=dev),
                                     torch.zeros(1, dtype=torch.int64, device=dev), (8, 8), 0.0, 2, False, False, False)
    assert (z[0] == -1).all()
    g0 = ops.rasterize_meshes_backward_indexed(z[4], faces[:0], V, z[0], z[1], z[2], z[3], False, False)
    assert g0.shape == (V, 3) and (g0 == 0).all()


# ------------------------------------------------------------------------------------ points

POINT_MATRIX = [(2000, 2, 32, 48, 5), (5000, 1, 64, 64, 10), (3000, 3, 40, 24, 1), (3000, 1, 50, 50, 40),
                (3000, 1, 20, 20, 150), (20000, 2, 128, 128, 8), (1000, 1, 17, 33, 3),
                # row segments that are / are not 16-byte multiples (W * K % 4), partial tiles, K = 32
                (4000, 2, 40, 50, 10), (4000, 1, 33, 47, 7), (3000, 1, 31, 36, 32), (2000, 1, 24, 20, 2),
                # tile lists longer than one chunk: in-kernel sort in shared / global memory
                (3000, 1, 32, 32, 6), (12000, 1, 16, 16, 3), (5000, 1, 16, 16, 40)]


@pytest.mark.parametrize("P,N,H,W,K", POINT_MATRIX)
def test_points_forward_equals_oracle(ops, dev, ref_cuda, P, N, H, W, K):
    pts, first, num, rad = rand_points(P, N, seed=P + K, z_ties=True)
    mine = ops.rasterize_points(pts.to(dev), first.to(dev), num.to(dev), (H, W), rad.to(dev), K, 0, 0)
    o = oracle.rasterize_points(pts.numpy(), first.numpy(), num.numpy(), (H, W), rad.numpy(), K, **CUDA)
    assert_frag_equal(mine, o, "points vs oracle")
    want = ref_cuda[case_key("points_forward", P, N, H, W, K)]["forward"]
    assert digest(*mine) == str(want), "points vs reference CUDA naive"


def test_points_golden_fixtures(ops, dev, golden):
    for name in sorted(k for k in golden if k.startswith("points/")):
        c = golden[name]
        H, W, K = (int(v) for v in c["args"])
        mine = ops.rasterize_points(torch.from_numpy(c["points"]).to(dev), torch.from_numpy(c["first"]).to(dev),
                                    torch.from_numpy(c["num"]).to(dev), (H, W),
                                    torch.from_numpy(c["radius"]).to(dev), K, 0, 0)
        assert np.array_equal(mine[0].cpu().numpy(), c["idx"]), name
        assert np.array_equal(mine[1].cpu().numpy(), c["zbuf"]), name
        assert np.abs(mine[2].cpu().numpy() - c["dists"]).max() <= 1e-5, name


def test_points_backward_and_edge_cases(ops, dev):
    pts, first, num, rad = rand_points(4000, 2, seed=9)
    pts[:50, 2] = -0.5  # behind the camera
    frag = ops.rasterize_points(pts.to(dev), first.to(dev), num.to(dev), (48, 48), rad.to(dev), 6, 0, 0)
    assert not np.isin(np.arange(50), frag[0].cpu().numpy()).any()
    gz, gd = upstream([frag[1].shape, frag[2].shape])
    mine = ops.rasterize_points_backward(pts.to(dev), frag[0], gz.to(dev), gd.to(dev)).cpu().numpy()
    want = oracle.rasterize_points_backward(pts.numpy(), frag[0].cpu().numpy(), gz.numpy(), gd.numpy(),
                                            arith=oracle.ARITH_CUDA)
    assert np.abs(mine - want).max() <= 5e-5  # reference tolerance is 2e-6 per unit gradient sum
    # empty cloud + empty outputs
    first2 = torch.tensor([0, 2000, 2000], dtype=torch.int64)
    num2 = torch.tensor([2000, 0, 2000], dtype=torch.int64)
    a = ops.rasterize_points(pts.to(dev), first2.to(dev), num2.to(dev), (24, 24), rad.to(dev), 3, 0, 0)
    o = oracle.rasterize_points(pts.numpy(), first2.numpy(), num2.numpy(), (24, 24), rad.numpy(), 3, **CUDA)
    assert_frag_equal(a, o)
    assert (a[0][1] == -1).all()


def test_points_autograd_wrapper(ops, dev):
    import pytorch3d_b200 as p3b
    from pytorch3d_b200 import synthetic
    pc = synthetic.random_pointclouds(2, 3000, seed=2, device=dev)
    pc.points_packed().requires_grad_(True)
    idx, zbuf, dists = p3b.rasterize_points(pc, (40, 56), radius=0.05, points_per_pixel=4)
    gz, gd = (t.to(dev) for t in upstream([zbuf.shape, dists.shape]))
    ((zbuf * gz).sum() + (dists * gd).sum()).backward()
    want = oracle.rasterize_points_backward(pc.points_packed().detach().cpu().numpy(), idx.cpu().numpy(),
                                            gz.cpu().numpy(), gd.cpu().numpy(), arith=oracle.ARITH_CUDA)
    assert np.abs(pc.points_packed().grad.cpu().numpy() - want).max() <= 5e-5
    assert idx.dtype == torch.int32


# ------------------------------------------------------------------------------------ full size

def test_full_size_properties(ops, dev, ref_cuda):
    """North-star size (8 x 69,938 faces, 512^2, K=8): size-independent properties, plus exact equality
    with the reference CUDA op."""
    from pytorch3d_b200 import synthetic
    m = synthetic.torus_batch(8, 187, 187, seed=0)
    fv = synthetic.face_verts_of(m).to(dev)
    first, num = m.mesh_to_faces_packed_first_idx().to(dev), m.num_faces_per_mesh().to(dev)
    a = run_mesh(ops, dev, fv, first, num, (512, 512), 0.0, 8)
    b = run_mesh(ops, dev, fv, first, num, (512, 512), 0.0, 8)
    for x, y in zip(a, b):
        assert torch.equal(x, y), "forward must be deterministic"
    p2f, zbuf, bary, dists = a
    valid = p2f >= 0
    assert valid.sum() > 1_000_000
    assert torch.equal(valid, zbuf >= 0) and (zbuf[~valid] == -1).all() and (dists[~valid] == -1).all()
    # valid entries first, sorted by depth
    assert (valid[..., :-1] | ~valid[..., 1:]).all()
    both = valid[..., :-1] & valid[..., 1:]
    assert (zbuf[..., :-1][both] <= zbuf[..., 1:][both]).all()
    # every index belongs to the mesh of its image; barycentrics sum to 1; inside hits have dist <= 0
    lo = first.view(-1, 1, 1, 1)
    hi = (first + num).view(-1, 1, 1, 1)
    assert ((p2f >= lo) & (p2f < hi) | ~valid).all()
    # barycentrics sum to area / (area + 1e-8): the reference's kEpsilon in the denominator
    # (geometry_utils.cuh:81) visibly biases sub-pixel faces, so compare against that, not against 1
    fvd = fv.double()
    area = ((fvd[:, 2, 0] - fvd[:, 0, 0]) * (fvd[:, 1, 1] - fvd[:, 0, 1])
            - (fvd[:, 2, 1] - fvd[:, 0, 1]) * (fvd[:, 1, 0] - fvd[:, 0, 0]))
    predicted = (area / (area + 1e-8))[p2f.clamp_min(0)]
    dev_sum = (bary.sum(-1).double() - predicted)[valid].abs()
    assert dev_sum.median() < 1e-5 and dev_sum.max() < 2e-2
    assert (dists[valid] <= 0).all()  # blur_radius = 0: only pixels inside a face are kept
    # z is the barycentric interpolation of the face's vertex depths
    zi = (bary * fv[p2f.clamp_min(0)][..., 2]).sum(-1)
    assert (zi - zbuf)[valid].abs().max() < 1e-5
    assert digest(*a) == str(ref_cuda["full_size"]["forward"]), "north-star vs reference CUDA (coarse-to-fine)"
    # backward: linear in the upstream gradients
    gz, gb, gd = (t.to(dev) for t in upstream([zbuf.shape, bary.shape, dists.shape]))
    g1 = ops.rasterize_meshes_backward(fv, p2f, gz, gb, gd, False, False)
    g2 = ops.rasterize_meshes_backward(fv, p2f, 2 * gz, 2 * gb, 2 * gd, False, False)
    assert torch.isfinite(g1).all()
    assert (g2 - 2 * g1).abs().max() <= 1e-3 * g1.abs().max()


def test_side_stream_and_noncontiguous(ops, dev):
    fv, first, num = rand_faces(400, 2, seed=21)
    base = run_mesh(ops, dev, fv, first, num, (32, 32), 1e-3, 4)
    s = torch.cuda.Stream(device=dev)
    big = torch.zeros(400, 3, 6)
    big[..., ::2] = fv
    with torch.cuda.stream(s):
        other = run_mesh(ops, dev, big.to(dev)[..., ::2], first, num, (32, 32), 1e-3, 4)
    s.synchronize()
    assert_frag_equal(base, other)


def test_ranges_with_gaps(ops, dev):
    """`first` / `num` that do not cover the packed array (unowned elements before, between and after the ranges):
    unowned elements are never drawn; the private-histogram binning of the point path starts a chunk in a gap."""
    pts, _, _, rad = rand_points(6000, 1, seed=11)
    pfirst = torch.tensor([100, 2600], dtype=torch.int64)
    pnum = torch.tensor([2000, 2500], dtype=torch.int64)
    mine = ops.rasterize_points(pts.to(dev), pfirst.to(dev), pnum.to(dev), (40, 56), rad.to(dev), 6, 0, 0)
    o = oracle.rasterize_points(pts.numpy(), pfirst.numpy(), pnum.numpy(), (40, 56), rad.numpy(), 6, **CUDA)
    assert_frag_equal(mine, o, "points with gaps vs oracle")
    fv, _, _ = rand_faces(3000, 1, seed=12)
    ffirst = torch.tensor([50, 1500], dtype=torch.int64)
    fnum = torch.tensor([1000, 1200], dtype=torch.int64)
    for blur, K in ((0.0, 4), (1e-3, 6)):
        mine = run_mesh(ops, dev, fv, ffirst, fnum, (48, 40), blur, K, 0, 0)
        o = oracle.rasterize_meshes(fv.numpy(), ffirst.numpy(), fnum.numpy(), (48, 40), blur, K, **CUDA)
        assert_frag_equal(mine, o, "meshes with gaps vs oracle")


def test_setup_pass_many_blocks_ragged_unaligned(ops, dev):
    """The setup pass on many blocks of 256 faces: a ragged last block whose word count is not a multiple of four (plain
    loads after the bulk copy), blocks that straddle two meshes (owner lookup per block + per-face fallback), and the same
    faces from a source that is only 4-byte aligned (no bulk copy at all)."""
    F = 400003
    fv, first, num = rand_faces(F, 2, seed=31, scale=0.01)
    mine = run_mesh(ops, dev, fv, first, num, (24, 40), 0.0, 4)
    o = oracle.rasterize_meshes(fv.numpy(), first.numpy(), num.numpy(), (24, 40), 0.0, 4, **CUDA)
    assert_frag_equal(mine, o, "many setup blocks vs oracle")
    assert int((mine[0] >= 0).sum()) > 100
    shifted = torch.zeros(F * 9 + 1, device=dev)
    shifted[1:] = fv.to(dev).reshape(-1)
    view = shifted[1:].view(F, 3, 3)
    assert view.data_ptr() % 16 != 0 and view.is_contiguous()
    nb = torch.full((F,), -1, dtype=torch.int64, device=dev)
    nb._b200_all_minus_one = True
    for blur, K in ((0.0, 4), (1e-3, 2)):
        a = ops.rasterize_meshes(fv.to(dev), first.to(dev), num.to(dev), nb, (24, 40), blur, K, 0, 0, False, False, False)
        b = ops.rasterize_meshes(view, first.to(dev), num.to(dev), nb, (24, 40), blur, K, 0, 0, False, False, False)
        assert_frag_equal(a, b, "unaligned source")

"""Parity at the sizes of BASELINE.json's configs (C3, C4, C5), the reference's tie-order test, the clipped
path against the reference's CUDA kernels, and the host-buffer C ABI.

Witnesses: the reference's own CUDA kernels rebuilt for sm_100a (their outputs on these seeded inputs, stored by
tests/golden/make_reference_outputs.py: digests, seeded samples of large outputs) wherever the oracle would take minutes
on the CPU; the C oracle otherwise."""
import ctypes

import numpy as np
import pytest
import torch

import oracle
from helpers import (assert_equal_up_to_ties, assert_frag_equal, case_key, digest, rand_faces, rand_points,
                     reference_outputs, upstream)

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


CLIP_SETTINGS = [(4, 1e-3), (12, 1e-3), (4, 0.0)]  # K, blur
NS_VARIANTS = [(1e-4, 8), (1e-4, 16), (0.0, 16)]  # blur, K
COARSE_SETTINGS = [((64, 64), 16, 0.0), ((48, 80), 8, 1e-3), ((33, 47), 16, 1e-2)]  # image size, bin size, blur


@pytest.fixture(scope="module")
def ref_cuda():
    return reference_outputs("reference_cuda")


@pytest.fixture(scope="module")
def ref_ties():
    return reference_outputs("reference_cuda_ties")


def seeded_randn(dev, *shapes, seed=231):
    g = torch.Generator(device=dev).manual_seed(seed)
    return [torch.randn(s, generator=g, device=dev) for s in shapes]


def _minus_one(n, dev, tagged=True):
    nb = torch.full((n,), -1, dtype=torch.int64, device=dev)
    if tagged:
        nb._b200_all_minus_one = True
    return nb


def test_config3_points_full_size(ops, dev, ref_cuda):
    """BASELINE config 3: 8 x 100k points, 512^2, K = 10, r = 0.01: size-independent properties, bit-exact against the
    reference's CUDA naive kernel (idx, zbuf, dists) and its backward on a seeded sample of the points."""
    from pytorch3d_b200 import synthetic
    pc = synthetic.random_pointclouds(8, 100000, seed=0)
    pts = pc.points_packed().to(dev)
    first, num = pc.cloud_to_packed_first_idx().to(dev), pc.num_points_per_cloud().to(dev)
    rad = torch.full((pts.shape[0],), 0.01, device=dev)
    idx, zbuf, dists = ops.rasterize_points(pts, first, num, (512, 512), rad, 10, 0, 0)
    valid = idx >= 0
    assert valid.sum() > 10_000_000
    assert (valid[..., :-1] | ~valid[..., 1:]).all()  # valid entries first
    both = valid[..., :-1] & valid[..., 1:]
    assert (zbuf[..., :-1][both] <= zbuf[..., 1:][both]).all()  # sorted by depth
    assert (zbuf[~valid] == -1).all() and (dists[~valid] == -1).all()
    assert (dists[valid] < 0.01 * 0.01).all() and (dists[valid] >= 0).all()
    lo, hi = first.view(-1, 1, 1, 1), (first + num).view(-1, 1, 1, 1)
    assert (((idx >= lo) & (idx < hi)) | ~valid).all()
    assert (pts[idx.clamp_min(0).long()][..., 2] == zbuf)[valid].all()
    gz, gd = seeded_randn(dev, zbuf.shape, dists.shape)
    grad = ops.rasterize_points_backward(pts, idx, gz, gd)
    assert torch.isfinite(grad).all()
    # grad_z of a point = sum of the upstream zbuf gradients of the slots it owns (exact up to summation order)
    want_z = torch.zeros(pts.shape[0], device=dev, dtype=torch.float64).index_add_(
        0, idx[valid].long(), gz[valid].double())
    assert (grad[:, 2].double() - want_z).abs().max() < 1e-4
    ref = ref_cuda["config3"]
    assert digest(idx, zbuf, dists) == str(ref["forward"]), "config 3 vs reference CUDA naive"
    sel = torch.from_numpy(ref["grad_points_idx"]).to(dev)
    rg = torch.from_numpy(ref["grad_points"]).to(dev)
    assert (grad[sel] - rg).abs().max() <= 2e-6 * max(1.0, float(ref["grad_scale"]))  # test_rasterize_points.py:201-234


def test_config5_stress_full_size(ops, dev, ref_cuda, ref_ties):
    """BASELINE config 5: one 999,698-face torus, 1024^2, K = 16, blur 1e-3 (thousands of blur-band candidates per
    pixel; the shared-memory-queue kernel with in-kernel sorting of ~5000-face tile lists)."""
    from pytorch3d_b200 import synthetic
    m = synthetic.torus_batch(1, 707, 707, seed=0)
    fv = synthetic.face_verts_of(m).to(dev)
    first, num = m.mesh_to_faces_packed_first_idx().to(dev), m.num_faces_per_mesh().to(dev)
    assert fv.shape[0] == 999698
    a = ops.rasterize_meshes(fv, first, num, _minus_one(fv.shape[0], dev), (1024, 1024), 1e-3, 16, 0, 0, False, False,
                             False)
    b = ops.rasterize_meshes(fv, first, num, _minus_one(fv.shape[0], dev), (1024, 1024), 1e-3, 16, 0, 0, False, False,
                             False)
    for x, y in zip(a, b):
        assert torch.equal(x, y), "forward must be deterministic"
    p2f, zbuf, bary, dists = a
    valid = p2f >= 0
    assert valid.sum() > 4_000_000
    assert torch.equal(valid, zbuf >= 0)
    assert (valid[..., :-1] | ~valid[..., 1:]).all()
    both = valid[..., :-1] & valid[..., 1:]
    assert (zbuf[..., :-1][both] <= zbuf[..., 1:][both]).all()
    assert (dists[valid] < 1e-3).all()
    # z is the barycentric interpolation of the vertex depths (the barycentrics of sliver faces extrapolate to ~1e4
    # in the blur band: bound the error relative to the magnitudes that were summed)
    terms = bary * fv[p2f.clamp_min(0)][..., 2]
    assert ((terms.sum(-1) - zbuf).abs() <= 1e-5 + 2e-6 * terms.abs().sum(-1))[valid].all()
    gz, gb, gd = seeded_randn(dev, zbuf.shape, bary.shape, dists.shape)
    g1 = ops.rasterize_meshes_backward(fv, p2f, gz, gb, gd, False, False)
    assert torch.isfinite(g1).all()
    # the reference with its own heuristics (bin_size 64 at 1024^2, max_faces_per_bin = F / 5)
    n_tie = assert_equal_up_to_ties(a, ref_ties["config5"], "config 5 vs reference CUDA coarse-to-fine",
                                    max_tie_pixels=2e-2)
    print("config 5: %d tie pixels of %d sampled" % (n_tie, len(ref_ties["config5"]["pixels"])))
    # the reference's backward on these Fragments, on a seeded sample of the faces
    ref = ref_cuda["config5"]
    sel = torch.from_numpy(ref["grad_faces_idx"]).to(dev)
    rg = torch.from_numpy(ref["grad_face_verts"]).to(dev)
    assert (g1[sel] - rg).abs().max() <= 5e-3 * float(ref["grad_scale"])  # atomics in a different order on ~16.8 M


def c4_face_counts(n=32, seed=0):
    """BASELINE config 4: face counts log-uniform in [5k, 100k] (SURVEY.md 8d)."""
    g = torch.Generator().manual_seed(seed)
    u = torch.rand(n, generator=g)
    return [int(v) for v in torch.exp(np.log(5e3) + u * (np.log(1e5) - np.log(5e3)))]


def test_config4_heterogeneous_batch_shards_exactly(ops, dev, ref_ties):
    """BASELINE config 4 (32 meshes, 5k-100k faces, 512^2, K = 8) rendered as ONE batch equals the same meshes
    rendered shard by shard with parallel.ShardPlan (the 8-rank LPT plan, local packing, pix_to_face re-based) --
    the multi-GPU data path minus the transport -- and equals the reference's CUDA kernels."""
    from pytorch3d_b200 import parallel, synthetic
    m = synthetic.torus_batch_hetero(c4_face_counts(), seed=0)
    fv = synthetic.face_verts_of(m).to(dev)
    first, num = m.mesh_to_faces_packed_first_idx(), m.num_faces_per_mesh()
    full = ops.rasterize_meshes(fv, first.to(dev), num.to(dev), _minus_one(fv.shape[0], dev), (512, 512), 0.0, 8, 0, 0,
                                False, False, False)
    plan = parallel.ShardPlan.build(first.tolist(), num.tolist(), 8)
    loads = [sum(plan.num[i] for i in ids) for ids in plan.assignment]
    assert max(loads) <= 1.25 * (sum(loads) / 8), "LPT plan is badly balanced: %r" % loads
    assert sorted(i for ids in plan.assignment for i in ids) == list(range(32))
    for rank in range(8):
        loc = plan.local_inputs(fv, rank)
        part = ops.rasterize_meshes(loc.face_verts, loc.first, loc.num, _minus_one(loc.face_verts.shape[0], dev),
                                    (512, 512), 0.0, 8, 0, 0, False, False, False)
        p2f = plan.rebase(part[0], rank)
        for j, i in enumerate(plan.assignment[rank]):
            assert torch.equal(p2f[j], full[0][i]), "mesh %d (rank %d)" % (i, rank)
            for a, b in zip(part[1:], full[1:]):
                assert torch.equal(a[j], b[i])
    # the reference with bin_size 32, max_faces_per_bin = max(10000, max faces of a mesh / 5)
    assert_equal_up_to_ties(full, ref_ties["config4"], "config 4 vs reference CUDA coarse-to-fine", max_tie_pixels=1e-4)


@pytest.mark.parametrize("K", [100, 32, 16, 8])
def test_order_of_ties(ops, dev, K):
    """tests/test_rasterize_meshes.py:1165-1185 of the reference: 100 copies of one triangle; every covered pixel
    must list the faces in index order (K = 100: thread-local queue; 32 / 16: shared-memory queue; 8: registers)."""
    tri = torch.tensor([[-0.9, -0.8, 1.5], [0.9, -0.7, 1.5], [0.1, 0.9, 1.5]])
    fv = tri.expand(100, 3, 3).contiguous().to(dev)
    first, num = torch.zeros(1, dtype=torch.int64, device=dev), torch.full((1,), 100, dtype=torch.int64, device=dev)
    for blur in (0.0, 1e-4):
        p2f, zbuf, _, _ = ops.rasterize_meshes(fv, first, num, _minus_one(100, dev), (28, 28), blur, K, 0, 0, False,
                                               False, False)
        covered = p2f[0, :, :, 0] >= 0
        assert covered.sum() > 100
        want = torch.arange(K, device=dev).expand(int(covered.sum()), K)
        assert torch.equal(p2f[0][covered], want)
        assert (p2f[0][~covered] == -1).all()


def test_clipped_faces_against_reference_cuda(ops, dev, ref_cuda, golden):
    """The faces produced by clip_faces (with their clipped-quad neighbour table) through our kernels and through
    the reference's CUDA kernels: bit-identical Fragments."""
    from pytorch3d_b200 import clip as mclip
    names = sorted(k for k in golden if k.startswith("clip/"))
    checked = 0
    for name in names:
        c = golden[name]
        persp, cull, has_z = (int(v) for v in c["args"])
        zc = float(c["z_clip"][0]) if has_z > 0 else None
        fr = mclip.ClipFrustum(left=-1, right=1, top=-1, bottom=1, perspective_correct=bool(persp), z_clip_value=zc,
                               cull=bool(cull))
        out = mclip.clip_faces(torch.from_numpy(c["face_verts"]).to(dev), torch.from_numpy(c["first"]).to(dev),
                               torch.from_numpy(c["num"]).to(dev), fr)
        nb = out.clipped_faces_neighbor_idx
        if nb is None:
            nb = _minus_one(out.face_verts.shape[0], dev, tagged=False)
        for K, blur in CLIP_SETTINGS:
            mine = ops.rasterize_meshes(out.face_verts, out.mesh_to_face_first_idx, out.num_faces_per_mesh, nb,
                                        (24, 32), blur, K, 0, 0, bool(persp), False, False)
            assert digest(*mine) == str(ref_cuda[case_key(name, K, blur)]["forward"]), \
                "%s K=%d blur=%g vs reference CUDA" % (name, K, blur)
            checked += 1
    assert checked >= 6


def test_host_abi_round_trip(ops, dev, built_lib):
    """The four `_host` entry points (host pointers in, host pointers out) against the device-pointer path."""
    from pytorch3d_b200 import _lib
    lib = _lib.load()
    fv, first, num = rand_faces(700, 2, seed=3)
    H, W, K, blur = 40, 56, 4, 1e-3
    slots = 2 * H * W * K
    p2f = torch.empty(slots, dtype=torch.int64)
    z, d, b = torch.empty(slots), torch.empty(slots), torch.empty(slots * 3)
    rc = lib.b200r_rasterize_meshes_forward_host(fv.data_ptr(), 700, first.data_ptr(), num.data_ptr(), None, 2, H, W,
                                                 blur, K, 1, 0, 0, p2f.data_ptr(), z.data_ptr(), b.data_ptr(),
                                                 d.data_ptr())
    assert rc == 0, _lib.last_error()
    want = ops.rasterize_meshes(fv.to(dev), first.to(dev), num.to(dev), _minus_one(700, dev), (H, W), blur, K, 0, 0,
                                True, False, False)
    got = (p2f.view(2, H, W, K), z.view(2, H, W, K), b.view(2, H, W, K, 3), d.view(2, H, W, K))
    assert_frag_equal(got, want, "meshes forward_host")
    gz, gb, gd = upstream([(2, H, W, K), (2, H, W, K, 3), (2, H, W, K)])
    grad = torch.empty(700, 3, 3)
    rc = lib.b200r_rasterize_meshes_backward_host(fv.data_ptr(), 700, p2f.data_ptr(), gz.data_ptr(), gb.data_ptr(),
                                                  gd.data_ptr(), 2, H, W, K, 1, 0, grad.data_ptr())
    assert rc == 0, _lib.last_error()
    gwant = ops.rasterize_meshes_backward(fv.to(dev), want[0], gz.to(dev), gb.to(dev), gd.to(dev), True, False).cpu()
    assert (grad - gwant).abs().max() <= 1e-4 * gwant.abs().max()
    # a neighbour table that carries information selects the kernel variant with the clipped-face rule
    nb = torch.full((700,), -1, dtype=torch.int64)
    nb[0:100:2] = torch.arange(1, 100, 2)
    nb[1:100:2] = torch.arange(0, 100, 2)
    rc = lib.b200r_rasterize_meshes_forward_host(fv.data_ptr(), 700, first.data_ptr(), num.data_ptr(), nb.data_ptr(),
                                                 2, H, W, blur, K, 0, 0, 0, p2f.data_ptr(), z.data_ptr(), b.data_ptr(),
                                                 d.data_ptr())
    assert rc == 0, _lib.last_error()
    o = oracle.rasterize_meshes(fv.numpy(), first.numpy(), num.numpy(), (H, W), blur, K,
                                clipped_faces_neighbor_idx=nb.numpy(), **CUDA)
    assert_frag_equal(got, o, "meshes forward_host with neighbours")
    # points
    pts, pfirst, pnum, rad = rand_points(3000, 2, seed=4)
    Kp = 6
    pslots = 2 * H * W * Kp
    idx = torch.empty(pslots, dtype=torch.int32)
    pz, pd = torch.empty(pslots), torch.empty(pslots)
    rc = lib.b200r_rasterize_points_forward_host(pts.data_ptr(), 3000, pfirst.data_ptr(), pnum.data_ptr(),
                                                 rad.data_ptr(), 2, H, W, Kp, idx.data_ptr(), pz.data_ptr(),
                                                 pd.data_ptr())
    assert rc == 0, _lib.last_error()
    pwant = ops.rasterize_points(pts.to(dev), pfirst.to(dev), pnum.to(dev), (H, W), rad.to(dev), Kp, 0, 0)
    assert_frag_equal((idx.view(2, H, W, Kp), pz.view(2, H, W, Kp), pd.view(2, H, W, Kp)), pwant, "points forward_host")
    pgz, pgd = upstream([(2, H, W, Kp), (2, H, W, Kp)])
    pgrad = torch.empty(3000, 3)
    rc = lib.b200r_rasterize_points_backward_host(pts.data_ptr(), 3000, idx.data_ptr(), pgz.data_ptr(),
                                                  pgd.data_ptr(), 2, H, W, Kp, pgrad.data_ptr())
    assert rc == 0, _lib.last_error()
    pgwant = ops.rasterize_points_backward(pts.to(dev), pwant[0], pgz.to(dev), pgd.to(dev)).cpu()
    assert (pgrad - pgwant).abs().max() <= 5e-5


def test_blur_and_k16_north_star_variants(ops, dev, ref_ties):
    """The north-star batch with a blur band (the soft-rasterization setting) and with K = 16, against the
    reference's CUDA coarse-to-fine kernels (bin_size 32, max_faces_per_bin 14000; equal up to its own tie
    nondeterminism)."""
    from pytorch3d_b200 import synthetic
    m = synthetic.torus_batch(2, 187, 187, seed=0)
    fv = synthetic.face_verts_of(m).to(dev)
    first, num = m.mesh_to_faces_packed_first_idx().to(dev), m.num_faces_per_mesh().to(dev)
    for blur, K in NS_VARIANTS:
        mine = ops.rasterize_meshes(fv, first, num, _minus_one(fv.shape[0], dev), (512, 512), blur, K, 0, 0, False,
                                    False, False)
        assert_equal_up_to_ties(mine, ref_ties[case_key("ns", blur, K)], "ns blur=%g K=%d vs reference CUDA" % (blur, K),
                                max_tie_pixels=2e-2)


def test_both_bindings_of_the_c_abi_agree(ops, dev):
    """The hot ops through the torch C++ extension (csrc/torch_ext.cpp, the default) and through ctypes: same library,
    same kernels -- forward outputs bit-identical, gradients equal up to the order of the atomic additions; and the
    extension's error behaviour mirrors the reference ops (RuntimeError)."""
    from pytorch3d_b200 import build
    build.build_ext()
    assert ops.binding() == "torch-extension", "the torch extension must be the binding in use on a GPU box"
    fv, first, num = rand_faces(3000, 2, seed=3)
    fv, first, num = fv.to(dev), first.to(dev), num.to(dev)
    pts, pfirst, pnum, rad = (t.to(dev) for t in rand_points(4000, 2, seed=5))
    nb_plain = _minus_one(fv.shape[0], dev, tagged=False)
    results = {}
    for use_ext in (True, False):
        ops.USE_EXT = use_ext
        try:
            assert ops.binding() == ("torch-extension" if use_ext else "ctypes")
            out = {}
            for name, nb in (("tagged", _minus_one(fv.shape[0], dev)), ("plain", nb_plain)):
                f = ops.rasterize_meshes(fv, first, num, nb, (48, 64), 1e-3, 5, 0, 0, True, True, False)
                g = upstream([tuple(t.shape) for t in f[1:]])
                out[name] = (f, ops.rasterize_meshes_backward(fv, f[0], g[0].to(dev), g[1].to(dev), g[2].to(dev), True,
                                                              True))
            p = ops.rasterize_points(pts, pfirst, pnum, (40, 56), rad, 6, 0, 0)
            gp = upstream([tuple(t.shape) for t in p[1:]])
            out["points"] = (p, ops.rasterize_points_backward(pts, p[0], gp[0].to(dev), gp[1].to(dev)))
            results[use_ext] = out
            with pytest.raises(RuntimeError, match="face_verts must have dimensions"):
                ops.rasterize_meshes(fv[:, :2], first, num, nb_plain, (8, 8), 0.0, 2, 0, 0, False, False, False)
            with pytest.raises(RuntimeError, match="CUDA tensor"):
                ops.rasterize_points(pts.cpu(), pfirst, pnum, (8, 8), rad, 2, 0, 0)
        finally:
            ops.USE_EXT = True
    for key in ("tagged", "plain", "points"):
        (fa, ga), (fb, gb) = results[True][key], results[False][key]
        for a, b in zip(fa, fb):
            assert a.dtype == b.dtype and a.shape == b.shape and torch.equal(a, b), key
        assert torch.allclose(ga, gb, rtol=1e-4, atol=1e-5), key
    assert torch.equal(results[True]["tagged"][0][0], results[True]["plain"][0][0])


def test_reference_test_hooks(ops, dev, ref_cuda):
    """The hooks the reference exports for its own tests (ext.cpp:69-73): coarse bin tables equal the reference's CUDA
    coarse stage (both sorted inside a bin), the hand-written expectation of tests/test_rasterize_meshes.py:1096-1163,
    and naive / fine give the result of the public op."""
    # the reference's own coarse test scene (16 x 16, bin_size 8, M = 3)
    verts = torch.tensor([[-0.5, 0.1, 0.1], [-0.3, 0.6, 0.1], [-0.1, 0.1, 0.1], [-0.3, -0.1, 0.4], [0.3, 0.5, 0.4],
                          [0.75, -0.1, 0.4], [0.2, -0.3, 0.9], [0.3, -0.7, 0.9], [0.6, -0.3, 0.9], [-0.4, 0.0, -1.5],
                          [0.6, 0.6, -1.5], [0.8, 0.0, -1.5]], device=dev)
    faces = torch.tensor([[1, 0, 2], [4, 3, 5], [7, 6, 8], [10, 9, 11]], dtype=torch.int64, device=dev)
    fv = verts[faces]
    first, num = torch.zeros(1, dtype=torch.int64, device=dev), torch.tensor([4], dtype=torch.int64, device=dev)
    want = torch.full((1, 2, 2, 3), -1, dtype=torch.int32, device=dev)
    want[0, 1, 1, 0] = 1
    want[0, 0, 1, 0:2] = torch.tensor([1, 2], dtype=torch.int32, device=dev)
    want[0, 1, 0, 0:2] = torch.tensor([0, 1], dtype=torch.int32, device=dev)
    want[0, 0, 0, 0] = 1
    got = ops._rasterize_meshes_coarse(fv, first, num, (16, 16), 0.0, 8, 3)
    assert torch.equal(got, want)
    # random scenes against the reference's CUDA coarse stage
    fv, first, num = rand_faces(3000, 2, seed=21)
    fv, first, num = fv.to(dev), first.to(dev), num.to(dev)
    pts, pfirst, pnum, rad = (t.to(dev) for t in rand_points(4000, 2, seed=22))
    for size, bs, blur in COARSE_SETTINGS:
        mine = ops._rasterize_meshes_coarse(fv, first, num, size, blur, bs, 3000)
        minep = ops._rasterize_points_coarse(pts, pfirst, pnum, size, rad, bs, 4000)
        assert mine.dtype == torch.int32 and mine.shape[1:3] == (1 + (size[0] - 1) // bs, 1 + (size[1] - 1) // bs)
        # the reference's bin tables, sorted inside every bin like ours
        for kind, m_ in (("meshes", mine), ("points", minep)):
            assert digest(m_) == str(ref_cuda[case_key("coarse", kind, size[0], size[1], bs, blur)]["bins"]), kind
        # naive and fine hooks = the public op
        nb = _minus_one(fv.shape[0], dev)
        pub = ops.rasterize_meshes(fv, first, num, nb, size, blur, 4, 0, 0, False, False, False)
        nai = ops._rasterize_meshes_naive(fv, first, num, nb, size, blur, 4, False, False, False)
        fin = ops._rasterize_meshes_fine(fv, mine, nb, size, blur, bs, 4, False, False, False)
        for a, b, c in zip(pub, nai, fin):
            assert torch.equal(a, b) and torch.equal(a, c)
        pp = ops.rasterize_points(pts, pfirst, pnum, size, rad, 5, 0, 0)
        pn = ops._rasterize_points_naive(pts, pfirst, pnum, size, rad, 5)
        for a, b in zip(pp, pn):
            assert torch.equal(a, b)

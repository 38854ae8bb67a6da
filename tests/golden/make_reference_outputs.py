"""Stores what the tests compare against the reference: the outputs of the UNMODIFIED reference ops, built from its
sources by oracle/build_ref.py into oracle/_ref/, on the same seeded inputs as the tests.

    python tests/golden/make_reference_outputs.py cpu  [OUTDIR]   # reference C++ CPU ops  -> reference_cpu.npz
    python tests/golden/make_reference_outputs.py cuda [OUTDIR]   # reference CUDA kernels -> reference_cuda.npz,
                                                                  # reference_cuda_ties.npz (on a B200, with the
                                                                  # product built)

Bit-exact comparisons are stored as SHA-256 digests (helpers.digest); comparisons with a tolerance as arrays, on a
fixed seeded sample of pixels / faces / points where the full output is large.  Nothing from the reference's sources is
stored; only its computed outputs.
"""
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
TESTS = os.path.dirname(HERE)
ROOT = os.path.dirname(TESTS)
sys.path[:0] = [ROOT, TESTS]

import oracle  # noqa: E402
from helpers import case_key, digest, rand_faces, rand_points, upstream  # noqa: E402

store = {}  # file name -> {"case/field": array}


def put(case, file="reference_cuda", **fields):
    for name, value in fields.items():
        store.setdefault(file, {})["%s/%s" % (case, name)] = np.asarray(value)


def _sample(n, size, seed):
    g = np.random.default_rng(seed)
    return np.sort(g.choice(n, size=min(size, n), replace=False)).astype(np.int64)


# ------------------------------------------------------------------------------------------------ C++ CPU ops

def cpu_outputs():
    import test_compositing as tc
    import test_oracle_vs_reference as tovr
    ref = oracle.load_reference(cuda=False)
    assert ref is not None, "oracle/_ref/ref_raster_cpu.so missing: run python oracle/build_ref.py --cpu-only"

    def put_cpu(case, **fields):
        put(case, file="reference_cpu", **fields)

    for persp, clip, cull, blur, K, H, W in tovr.REF_MESH_CASES:
        fv, first, num = rand_faces(400, 2, seed=K + H)
        nb = torch.full((fv.shape[0],), -1, dtype=torch.int64)
        r = ref.rasterize_meshes(fv, first, num, nb, (H, W), blur, K, 0, 0, bool(persp), bool(clip), bool(cull))
        gz, gb, gd = upstream([r[1].shape, r[2].shape, r[3].shape])
        rg = ref.rasterize_meshes_backward(fv, r[0], gz, gb, gd, bool(persp), bool(clip))
        put_cpu(case_key("meshes", persp, clip, cull, blur, K, H, W), forward=digest(*r), backward=digest(rg))
    fv, first, num = rand_faces(300, 1, seed=7, scale=0.35)
    put_cpu("neighbors", forward=digest(*ref.rasterize_meshes(fv, first, num, tovr.neighbor_table(), (32, 32), 1e-2, 4,
                                                              0, 0, False, False, False)))
    for K, H, W in tovr.REF_POINT_CASES:
        pts, first, num, rad = rand_points(1500, 2, seed=K)
        r = ref.rasterize_points(pts, first, num, (H, W), rad, K, 0, 0)
        gz, gd = upstream([r[1].shape, r[2].shape])
        put_cpu(case_key("points", K, H, W), forward=digest(*r),
                backward=digest(ref.rasterize_points_backward(pts, r[0], gz, gd)))
    for N, K, H, W, C, P in tc.REF_CASES:
        feats, alphas, idx = tc.scene(N, K, H, W, C, P, seed=K)
        want = ref.accum_alphacomposite(feats, alphas, idx)
        go = torch.rand(want.shape, generator=torch.Generator().manual_seed(1))
        put_cpu(case_key("alpha", N, K, H, W, C, P), forward=digest(want),
                backward=digest(*ref.accum_alphacomposite_backward(go, feats, alphas, idx)))
        for norm in (False, True):
            feats, alphas, idx = tc.scene(N, K, H, W, C, P, seed=K + 7)
            if norm:
                alphas[:, :, 0, 0] = 1e-6
            fwd = ref.accum_weightedsumnorm if norm else ref.accum_weightedsum
            bwd = ref.accum_weightedsumnorm_backward if norm else ref.accum_weightedsum_backward
            want = fwd(feats, alphas, idx)
            go = torch.rand(want.shape, generator=torch.Generator().manual_seed(1))
            put_cpu(case_key("weighted_sum", norm, N, K, H, W, C, P), forward=digest(want),
                    backward=digest(*bwd(go, feats, alphas, idx)))


# ------------------------------------------------------------------------------------------------ CUDA kernels

def tie_case(case, r, pixels_seed, n_pixels):
    """zbuf in full (digest) + indices, barycentrics and distances of a seeded sample of pixels (see
    helpers.assert_equal_up_to_ties)."""
    from helpers import sample_pixels
    N, H, W = r[0].shape[:3]
    pixels = _sample(N * H * W, n_pixels, pixels_seed)
    p2f, bary, dists = sample_pixels((r[0], r[2], r[3]), pixels)
    put(case, file="reference_cuda_ties", zbuf_digest=digest(r[1]), pixels=pixels, pix_to_face=p2f.astype(np.int32),
        bary=bary, dists=dists)


def cuda_outputs():
    import test_compositing as tc
    import test_gpu_configs as tg
    import test_gpu_parity as tp
    import test_interp_face_attrs as ti
    from pytorch3d_b200 import _C, synthetic
    from pytorch3d_b200 import clip as mclip
    ref = oracle.load_reference(cuda=True)
    ref_cpu = oracle.load_reference(cuda=False)
    assert ref is not None and ref_cpu is not None, "oracle/_ref/ missing: run python oracle/build_ref.py"
    dev = torch.device("cuda:0")

    def minus_one(n):
        return torch.full((n,), -1, dtype=torch.int64, device=dev)

    # ---- test_gpu_parity
    m = synthetic.torus_batch(2, 54, 54, seed=0)
    fv, first, num = synthetic.face_verts_of(m).to(dev), m.mesh_to_faces_packed_first_idx().to(dev), \
        m.num_faces_per_mesh().to(dev)
    put("torus_ties", forward=digest(*ref.rasterize_meshes(fv, first, num, minus_one(fv.shape[0]), (256, 256), 1e-4, 8,
                                                           0, 0, False, False, False)))
    for persp, clip, cull, blur, K, H, W, F, N in tp.MESH_MATRIX[:6]:
        fv, first, num = rand_faces(F, N, seed=K + H)
        r = ref.rasterize_meshes(fv.to(dev), first.to(dev), num.to(dev), minus_one(F), (H, W), blur, K, 0, 0,
                                 bool(persp), bool(clip), bool(cull))
        put(case_key("mesh_forward", persp, clip, cull, blur, K, H, W, F, N), forward=digest(*r))
    for persp, clip, blur in tp.BACKWARD_CASES:
        if persp and clip and blur == 0:  # the test has no reference witness there
            continue
        m = synthetic.torus_batch(2, 24, 24, seed=3)
        fv, first, num = synthetic.face_verts_of(m), m.mesh_to_faces_packed_first_idx(), m.num_faces_per_mesh()
        frag = tp.run_mesh(_C, dev, fv, first, num, (64, 64), blur, 4, persp, clip)
        gz, gb, gd = upstream([frag[1].shape, frag[2].shape, frag[3].shape])
        if persp and clip and blur > 0:  # the reference's C++ CPU backward is the witness here (see the test)
            g = ref_cpu.rasterize_meshes_backward(fv, frag[0].cpu(), gz, gb, gd, True, True)
        else:
            g = ref.rasterize_meshes_backward(fv.to(dev), frag[0], gz.to(dev), gb.to(dev), gd.to(dev), bool(persp),
                                              bool(clip))
        put(case_key("mesh_backward", persp, clip, blur), grad_face_verts=g.cpu().numpy())
    for P, N, H, W, K in tp.POINT_MATRIX:
        pts, first, num, rad = rand_points(P, N, seed=P + K, z_ties=True)
        r = ref.rasterize_points(pts.to(dev), first.to(dev), num.to(dev), (H, W), rad.to(dev), K, 0, 0)
        put(case_key("points_forward", P, N, H, W, K), forward=digest(*r))
    m = synthetic.torus_batch(8, 187, 187, seed=0)
    fv, first, num = synthetic.face_verts_of(m).to(dev), m.mesh_to_faces_packed_first_idx().to(dev), \
        m.num_faces_per_mesh().to(dev)
    put("full_size", forward=digest(*ref.rasterize_meshes(fv, first, num, minus_one(fv.shape[0]), (512, 512), 0.0, 8,
                                                          32, 14000, False, False, False)))
    del fv

    # ---- test_gpu_configs
    pc = synthetic.random_pointclouds(8, 100000, seed=0)
    pts = pc.points_packed().to(dev)
    first, num = pc.cloud_to_packed_first_idx().to(dev), pc.num_points_per_cloud().to(dev)
    rad = torch.full((pts.shape[0],), 0.01, device=dev)
    r = ref.rasterize_points(pts, first, num, (512, 512), rad, 10, 0, 0)
    gz, gd = tg.seeded_randn(dev, r[1].shape, r[2].shape)
    rg = ref.rasterize_points_backward(pts, r[0], gz, gd)
    sel = _sample(pts.shape[0], 8192, 3)
    put("config3", forward=digest(*r), grad_points_idx=sel, grad_points=rg.cpu().numpy()[sel],
        grad_scale=float(rg.abs().max()))
    del r, gz, gd, rg

    m = synthetic.torus_batch(1, 707, 707, seed=0)
    fv = synthetic.face_verts_of(m).to(dev)
    first, num = m.mesh_to_faces_packed_first_idx().to(dev), m.num_faces_per_mesh().to(dev)
    r = ref.rasterize_meshes(fv, first, num, minus_one(fv.shape[0]), (1024, 1024), 1e-3, 16, 64, int(fv.shape[0] / 5),
                             False, False, False)
    tie_case("config5", r, 5, 512)
    del r
    nb = minus_one(fv.shape[0])
    nb._b200_all_minus_one = True
    p2f = _C.rasterize_meshes(fv, first, num, nb, (1024, 1024), 1e-3, 16, 0, 0, False, False, False)[0]
    gz, gb, gd = tg.seeded_randn(dev, p2f.shape, p2f.shape + (3,), p2f.shape)
    rg = ref.rasterize_meshes_backward(fv, p2f, gz, gb, gd, False, False)
    sel = _sample(fv.shape[0], 8192, 6)
    put("config5", grad_faces_idx=sel, grad_face_verts=rg.cpu().numpy()[sel], grad_scale=float(rg.abs().max()))
    del fv, p2f, gz, gb, gd, rg

    m = synthetic.torus_batch_hetero(tg.c4_face_counts(), seed=0)
    fv = synthetic.face_verts_of(m).to(dev)
    first, num = m.mesh_to_faces_packed_first_idx(), m.num_faces_per_mesh()
    r = ref.rasterize_meshes(fv, first.to(dev), num.to(dev), minus_one(fv.shape[0]), (512, 512), 0.0, 8, 32,
                             max(10000, int(num.max()) // 5), False, False, False)
    tie_case("config4", r, 4, 1024)
    del fv, r

    golden = np.load(os.path.join(HERE, "clip_golden.npz"))
    for name in sorted({k.rsplit("/", 1)[0] for k in golden.files if k.startswith("clip/")}):
        persp, cull, has_z = (int(v) for v in golden[name + "/args"])
        zc = float(golden[name + "/z_clip"][0]) if has_z > 0 else None
        fr = mclip.ClipFrustum(left=-1, right=1, top=-1, bottom=1, perspective_correct=bool(persp), z_clip_value=zc,
                               cull=bool(cull))
        out = mclip.clip_faces(torch.from_numpy(golden[name + "/face_verts"]).to(dev),
                               torch.from_numpy(golden[name + "/first"]).to(dev),
                               torch.from_numpy(golden[name + "/num"]).to(dev), fr)
        nb = out.clipped_faces_neighbor_idx
        if nb is None:
            nb = minus_one(out.face_verts.shape[0])
        for K, blur in tg.CLIP_SETTINGS:
            r = ref.rasterize_meshes(out.face_verts, out.mesh_to_face_first_idx, out.num_faces_per_mesh, nb, (24, 32),
                                     blur, K, 0, 0, bool(persp), False, False)
            put(case_key(name, K, blur), forward=digest(*r))

    m = synthetic.torus_batch(2, 187, 187, seed=0)
    fv = synthetic.face_verts_of(m).to(dev)
    first, num = m.mesh_to_faces_packed_first_idx().to(dev), m.num_faces_per_mesh().to(dev)
    for blur, K in tg.NS_VARIANTS:
        r = ref.rasterize_meshes(fv, first, num, minus_one(fv.shape[0]), (512, 512), blur, K, 32, 14000, False, False,
                                 False)
        tie_case(case_key("ns", blur, K), r, K, 512)
    del fv, r

    fv, first, num = rand_faces(3000, 2, seed=21)
    fv, first, num = fv.to(dev), first.to(dev), num.to(dev)
    pts, pfirst, pnum, rad = (t.to(dev) for t in rand_points(4000, 2, seed=22))
    big = torch.iinfo(torch.int32).max
    for size, bs, blur in tg.COARSE_SETTINGS:
        for kind, bins in (("meshes", ref._rasterize_meshes_coarse(fv, first, num, size, blur, bs, 3000)),
                           ("points", ref._rasterize_points_coarse(pts, pfirst, pnum, size, rad, bs, 4000))):
            rs = torch.where(bins < 0, torch.full_like(bins, big), bins).sort(dim=-1).values
            rs = torch.where(rs == big, torch.full_like(rs, -1), rs)
            put(case_key("coarse", kind, size[0], size[1], bs, blur), bins=digest(rs))

    # ---- test_compositing, test_interp_face_attrs
    for N, K, H, W, C, P, _ in tc.CUDA_CASES:
        feats, alphas, idx = tc.scene(N, K, H, W, C, P, seed=N + K)
        put(case_key("alpha_cuda", N, K, H, W, C, P),
            forward=digest(ref.accum_alphacomposite(feats.to(dev), alphas.to(dev), idx.to(dev))))
        for norm in (False, True):
            feats, alphas, idx = tc.scene(N, K, H, W, C, P, seed=N + K + 3)
            if norm:
                alphas[:, :, 0, 0] = 1e-6
            fwd = ref.accum_weightedsumnorm if norm else ref.accum_weightedsum
            put(case_key("weighted_sum_cuda", norm, N, K, H, W, C, P),
                forward=digest(fwd(feats.to(dev), alphas.to(dev), idx.to(dev))))
    for N, H, W, K, F, D in ti.CUDA_CASES:
        p2f, bary, attrs, _ = ti.scene(N, H, W, K, F, D)
        put(case_key("interp", N, H, W, K, F, D),
            forward=digest(ref.interp_face_attrs_forward(p2f.reshape(-1).to(dev), bary.reshape(-1, 3).to(dev),
                                                         attrs.to(dev))))


if __name__ == "__main__":
    which = sys.argv[1]
    out_dir = sys.argv[2] if len(sys.argv) > 2 else HERE
    {"cpu": cpu_outputs, "cuda": cuda_outputs}[which]()
    os.makedirs(out_dir, exist_ok=True)
    for name, arrays in store.items():
        path = os.path.join(out_dir, name + ".npz")
        np.savez_compressed(path, **arrays)
        print("wrote %s: %d cases, %.1f KB" % (path, len({k.rsplit("/", 1)[0] for k in arrays}),
                                               os.path.getsize(path) / 1024))

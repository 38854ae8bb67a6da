"""Generates tests/golden/*.npz by RUNNING THE REFERENCE (PyTorch3D v0.7.9) in this container.

How the reference was made importable (no network; done once, outside the repo):
    cp -r /root/reference /tmp/p3d_build && cd /tmp/p3d_build && \
    PYTORCH3D_FORCE_NO_CUDA=1 python setup.py build_ext --inplace        # 3.5 min, CPU-only _C
Then:  python tests/golden/make_golden.py [/tmp/p3d_build]

What is recorded
  * The reference's own known-answer scenes: the scene builders of the reference test-suite
    (tests/test_rasterize_meshes.py: _simple_triangle_raster :853, _simple_blurry_raster :1005,
    _test_perspective_correct :596, _test_barycentric_clipping :708, _test_behind_camera :784,
    _test_back_face_culling :468;  tests/test_rasterize_points.py: _simple_test_case :278,
    _test_behind_camera :243, _test_variable_size_radius :541) are executed with a capturing
    rasterize function that calls the reference implementation.  The reference methods assert the
    outputs against their hand-written golden tensors while we record the operator-level inputs and
    outputs, so every recorded case is one the reference's goldens accept.  Each scene is run through
    the reference's C++ CPU op; the mesh scenes also through its pure-Python implementation
    (rasterize_meshes_python), whose outputs are stored under "<name>/python/...".
  * Seeded random scenes through the reference C++ CPU op, forward and backward (upstream grads
    seed 231 like tests/test_rasterize_meshes.py:563).

Nothing from the reference's sources is copied; only its computed outputs are stored.
"""
import os
import sys

import numpy as np
import torch

REF = sys.argv[1] if len(sys.argv) > 1 else "/tmp/p3d_build"
sys.path.insert(0, REF)

from pytorch3d.renderer.mesh.rasterize_meshes import rasterize_meshes, rasterize_meshes_python  # noqa: E402
from pytorch3d.renderer.points.rasterize_points import rasterize_points  # noqa: E402
from pytorch3d import _C  # noqa: E402
from tests.test_rasterize_meshes import TestRasterizeMeshes  # noqa: E402
from tests.test_rasterize_points import TestRasterizePoints  # noqa: E402

OUT = os.path.dirname(os.path.abspath(__file__))
store = {}
counter = {}


def _key(prefix):
    counter[prefix] = counter.get(prefix, 0) + 1
    return "%s_%02d" % (prefix, counter[prefix])


def _np(t):
    return t.detach().cpu().numpy()


class MeshCapture:
    def __init__(self, scene, fn, tag):
        self.scene, self.fn, self.tag = scene, fn, tag

    def __call__(self, meshes, image_size=256, blur_radius=0.0, faces_per_pixel=8, bin_size=None,
                 max_faces_per_bin=None, perspective_correct=False, clip_barycentric_coords=False,
                 cull_backfaces=False, **kw):
        if self.fn is rasterize_meshes:
            out = self.fn(meshes, image_size, blur_radius, faces_per_pixel, 0, max_faces_per_bin,
                          perspective_correct, clip_barycentric_coords, cull_backfaces)
        else:
            out = self.fn(meshes, image_size, blur_radius, faces_per_pixel, perspective_correct,
                          clip_barycentric_coords, cull_backfaces)
        k = _key("mesh/%s/%s" % (self.scene, self.tag))
        im = (image_size, image_size) if isinstance(image_size, int) else tuple(image_size)
        store[k + "/face_verts"] = _np(meshes.verts_packed()[meshes.faces_packed()]).astype(np.float32)
        store[k + "/first"] = _np(meshes.mesh_to_faces_packed_first_idx()).astype(np.int64)
        store[k + "/num"] = _np(meshes.num_faces_per_mesh()).astype(np.int64)
        store[k + "/args"] = np.array([im[0], im[1], faces_per_pixel, int(perspective_correct),
                                       int(clip_barycentric_coords), int(cull_backfaces)], np.int64)
        store[k + "/blur"] = np.array([blur_radius], np.float64)
        for name, t in zip(("pix_to_face", "zbuf", "bary", "dists"), out):
            store[k + "/" + name] = _np(t)
        return out


class PointCapture:
    def __init__(self, scene):
        self.scene = scene

    def __call__(self, pointclouds, image_size=256, radius=0.01, points_per_pixel=8, bin_size=None,
                 max_points_per_bin=None):
        out = rasterize_points(pointclouds, image_size, radius, points_per_pixel, 0, max_points_per_bin)
        from pytorch3d.renderer.points.rasterize_points import _format_radius
        k = _key("points/%s" % self.scene)
        im = (image_size, image_size) if isinstance(image_size, int) else tuple(image_size)
        store[k + "/points"] = _np(pointclouds.points_packed()).astype(np.float32)
        store[k + "/first"] = _np(pointclouds.cloud_to_packed_first_idx()).astype(np.int64)
        store[k + "/num"] = _np(pointclouds.num_points_per_cloud()).astype(np.int64)
        store[k + "/radius"] = _np(_format_radius(radius, pointclouds)).astype(np.float32)
        store[k + "/args"] = np.array([im[0], im[1], points_per_pixel], np.int64)
        for name, t in zip(("idx", "zbuf", "dists"), out):
            store[k + "/" + name] = _np(t)
        return out


def reference_scenes():
    cpu = torch.device("cpu")
    tm = TestRasterizeMeshes()
    for scene in ("_simple_triangle_raster", "_simple_blurry_raster", "_test_behind_camera",
                  "_test_perspective_correct", "_test_back_face_culling"):
        getattr(tm, scene)(MeshCapture(scene, rasterize_meshes, "cpp"), cpu, bin_size=0)
        getattr(tm, scene)(MeshCapture(scene, rasterize_meshes_python, "python"), cpu, bin_size=-1)
    # the reference runs the barycentric clipping goldens through its python implementation only
    tm._test_barycentric_clipping(MeshCapture("_test_barycentric_clipping", rasterize_meshes_python, "python"), cpu,
                                  bin_size=-1)
    tm._test_barycentric_clipping(MeshCapture("_test_barycentric_clipping", rasterize_meshes, "cpp"), cpu, bin_size=0)
    tp = TestRasterizePoints()
    tp._simple_test_case(PointCapture("_simple_test_case"), cpu)
    tp._test_behind_camera(PointCapture("_test_behind_camera"), cpu)
    tp._test_variable_size_radius(PointCapture("_test_variable_size_radius"), cpu)


def random_scenes():
    def rand_faces(F, N, seed, scale=0.2):
        g = torch.Generator().manual_seed(seed)
        c = torch.rand(F, 1, 3, generator=g) * 2 - 1
        v = c + (torch.rand(F, 3, 3, generator=g) - 0.5) * scale * 2
        v[..., 2] = 0.5 + 2.5 * torch.rand(F, 3, generator=g)
        per = F // N
        first = torch.arange(N) * per
        num = torch.full((N,), per)
        num[-1] = F - first[-1]
        return v.contiguous(), first.long(), num.long()

    cases = [  # F, N, H, W, blur, K, persp, clip, cull
        (200, 2, 24, 24, 0.0, 4, 0, 0, 0),
        (200, 2, 20, 32, 1e-3, 8, 1, 0, 0),
        (200, 1, 32, 20, 1e-2, 3, 0, 1, 1),
        (200, 2, 24, 24, 1e-3, 5, 1, 1, 0),
    ]
    for ci, (F, N, H, W, blur, K, persp, clip, cull) in enumerate(cases):
        fv, first, num = rand_faces(F, N, 100 + ci)
        nb = torch.full((F,), -1, dtype=torch.int64)
        out = _C.rasterize_meshes(fv, first, num, nb, (H, W), blur, K, 0, 0, bool(persp), bool(clip), bool(cull))
        g = torch.Generator().manual_seed(231)
        gz, gb, gd = (torch.randn(out[i].shape, generator=g) for i in (1, 2, 3))
        grad = _C.rasterize_meshes_backward(fv, out[0], gz, gb, gd, bool(persp), bool(clip))
        k = "mesh/random/cpp_%02d" % ci
        store[k + "/face_verts"], store[k + "/first"], store[k + "/num"] = _np(fv), _np(first), _np(num)
        store[k + "/args"] = np.array([H, W, K, persp, clip, cull], np.int64)
        store[k + "/blur"] = np.array([blur], np.float64)
        for name, t in zip(("pix_to_face", "zbuf", "bary", "dists"), out):
            store[k + "/" + name] = _np(t)
        store[k + "/grad_zbuf"], store[k + "/grad_bary"], store[k + "/grad_dists"] = _np(gz), _np(gb), _np(gd)
        store[k + "/grad_face_verts"] = _np(grad)
    for ci, (P, N, H, W, K) in enumerate([(300, 2, 24, 24, 5), (300, 1, 20, 36, 10)]):
        g = torch.Generator().manual_seed(200 + ci)
        pts = torch.rand(P, 3, generator=g) * 2 - 1
        pts[:, 2] = torch.rand(P, generator=g) * 2 - 0.2
        rad = torch.rand(P, generator=g) * 0.15 + 0.03
        per = P // N
        first = (torch.arange(N) * per).long()
        num = torch.full((N,), per).long()
        out = _C.rasterize_points(pts, first, num, (H, W), rad, K, 0, 0)
        g2 = torch.Generator().manual_seed(231)
        gz, gd = torch.randn(out[1].shape, generator=g2), torch.randn(out[2].shape, generator=g2)
        grad = _C.rasterize_points_backward(pts, out[0], gz, gd)
        k = "points/random/cpp_%02d" % ci
        store[k + "/points"], store[k + "/first"], store[k + "/num"], store[k + "/radius"] = (
            _np(pts), _np(first), _np(num), _np(rad))
        store[k + "/args"] = np.array([H, W, K], np.int64)
        for name, t in zip(("idx", "zbuf", "dists"), out):
            store[k + "/" + name] = _np(t)
        store[k + "/grad_zbuf"], store[k + "/grad_dists"], store[k + "/grad_points"] = _np(gz), _np(gd), _np(grad)


def clip_scenes():
    """clip_faces (renderer/mesh/clip.py:324-615) and the end-to-end rasterize_meshes(z_clip_value, cull_to_frustum)
    of the reference's C++ CPU path, on seeded scenes with faces crossing the clipping plane."""
    from pytorch3d.renderer.mesh import clip as rclip
    from pytorch3d.structures import Meshes

    def scene(F, seed):
        g = torch.Generator().manual_seed(seed)
        c = torch.rand(F, 1, 3, generator=g) * 2.4 - 1.2
        v = c + (torch.rand(F, 3, 3, generator=g) - 0.5) * 0.9
        v[..., 2] = torch.rand(F, 3, generator=g) * 3 - 0.8
        return v

    ci = 0
    for persp in (False, True):
        for cull in (False, True):
            for zc in (None, 0.3):
                if zc is None and not cull:
                    continue
                fv = scene(300, 40 + ci)
                first, num = torch.tensor([0, 120, 120]), torch.tensor([120, 0, 180])
                fr = rclip.ClipFrustum(left=-1, right=1, top=-1, bottom=1, perspective_correct=persp,
                                       z_clip_value=zc, cull=cull)
                r = rclip.clip_faces(fv, first, num, fr)
                k = "clip/faces_%02d" % ci
                store[k + "/face_verts"], store[k + "/first"], store[k + "/num"] = _np(fv), _np(first), _np(num)
                store[k + "/args"] = np.array([int(persp), int(cull), -1 if zc is None else 1], np.int64)
                store[k + "/z_clip"] = np.array([0.0 if zc is None else zc], np.float64)
                store[k + "/out_face_verts"] = _np(r.face_verts)
                store[k + "/out_first"], store[k + "/out_num"] = _np(r.mesh_to_face_first_idx), _np(r.num_faces_per_mesh)
                store[k + "/out_c2u"] = _np(r.faces_clipped_to_unclipped_idx)
                if r.clipped_faces_neighbor_idx is not None:
                    store[k + "/out_neighbor"] = _np(r.clipped_faces_neighbor_idx)
                # end to end through the reference wrapper (verts == face corners, faces = arange)
                verts = [fv[:120].reshape(-1, 3), torch.zeros(0, 3), fv[120:].reshape(-1, 3)]
                faces = [torch.arange(360).reshape(-1, 3), torch.zeros(0, 3, dtype=torch.int64),
                         torch.arange(540).reshape(-1, 3)]
                meshes = Meshes(verts=verts, faces=faces)
                out = rasterize_meshes(meshes, (24, 32), 1e-3, 4, 0, None, persp, False, False, zc, cull)
                for name, t in zip(("pix_to_face", "zbuf", "bary", "dists"), out):
                    store[k + "/e2e_" + name] = _np(t)
                ci += 1


def interp_scenes():
    """interpolate_face_attributes through the reference's CPU path (ops/interp_face_attrs.py:83-102)."""
    from pytorch3d.ops.interp_face_attrs import interpolate_face_attributes
    for ci, (N, H, W, K, F, D) in enumerate([(2, 5, 7, 3, 40, 3), (1, 4, 4, 1, 6, 1), (1, 6, 5, 2, 30, 8)]):
        g = torch.Generator().manual_seed(300 + ci)
        p2f = torch.randint(-1, F, (N, H, W, K), generator=g)
        bary = torch.rand(N, H, W, K, 3, generator=g)
        attrs = torch.randn(F, 3, D, generator=g)
        out = interpolate_face_attributes(p2f, bary, attrs)
        k = "interp/case_%02d" % ci
        store[k + "/pix_to_face"], store[k + "/bary"], store[k + "/attrs"] = _np(p2f), _np(bary), _np(attrs)
        store[k + "/out"] = _np(out)


if __name__ == "__main__":
    torch.manual_seed(0)
    reference_scenes()
    random_scenes()
    clip_scenes()
    interp_scenes()
    for name, keep in (("raster_golden.npz", lambda k: not k.startswith("clip/")),
                       ("clip_golden.npz", lambda k: k.startswith("clip/"))):  # (each file stays under 1 MB)
        part = {k: v for k, v in store.items() if keep(k)}
        path = os.path.join(OUT, name)
        np.savez_compressed(path, **part)
        cases = sorted({k.rsplit("/", 1)[0] for k in part})
        print("wrote %s: %d cases, %.1f KB" % (path, len(cases), os.path.getsize(path) / 1024))
        for c in cases:
            print("  ", c)

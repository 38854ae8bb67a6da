"""Backward kernels against plain float64 references (tests/f64_reference.py), element by element:

    |g32 - g64| <= tau * scale64 + TINY,

scale64 = that element's own sum of |terms| (never the largest value of the array).  tau is a multiple of the number
of float32 roundings an element goes through, times 2**-24:

* compositing, weighted sums, interpolation, points: TAU_ULPS * (terms per pixel + atomic contributions to the
  element) * 2**-24.  The C oracle, a float32 restatement of the reference ops, stays below 0.35 of that count on every
  case here, so TAU_ULPS = 4 leaves a factor of ~10.
* meshes: MESH_TAU + 2 * (slots on the face) * 2**-24.  The first term covers one slot's chain rule (~60 float32
  operations through edge functions, perspective correction, clipping and the segment distance); the oracle in
  ARITH_CUDA, the kernel's arithmetic on the CPU, reaches 2.5e-5 on the scenes below, so MESH_TAU = 1e-4.  The second
  term is the accumulation of the per-slot gradients into the face (atomics, any order).

CPU tests pin the references to the oracle and show that the comparison rejects plausible kernel bugs; the GPU tests
run every dispatch branch of the backward kernels against the references."""
import ctypes

import numpy as np
import pytest
import torch

import f64_reference as R
import oracle
from helpers import rand_faces, rand_points, split, upstream

TAU_ULPS = 4.0
MESH_TAU = 1e-4
MAX_SINGULAR = 0.05  # at most this fraction of a test's slots may be left out as singular


def tau_terms(n_terms):
    return TAU_ULPS * R.ULP * (n_terms if torch.is_tensor(n_terms) else float(n_terms))


def mesh_tau(slots_per_face):
    return MESH_TAU + 2.0 * R.ULP * slots_per_face.to(torch.float64).view(-1, 1, 1)


def hits_per(idx, n):
    """Number of valid slots that land on each of n targets (points / faces / vertices)."""
    i = idx.reshape(-1).long().cpu()
    i = i[i >= 0]
    return torch.bincount(i, minlength=n).to(torch.float64)


# ------------------------------------------------------------------------------------------------ scenes

REGIMES = {  # name -> alpha sampler
    "uniform": lambda g, s: torch.rand(s, generator=g),
    "deep": lambda g, s: 0.4 + 0.2 * torch.rand(s, generator=g),              # K = 150: the product underflows
    "opaque": lambda g, s: 1 - (1e-5 + 9e-5 * torch.rand(s, generator=g)),   # near-opaque splats
}


def comp_scene(N, K, H, W, C, P, regime, seed, hole=False, exact01=False, contention=False):
    g = torch.Generator().manual_seed(seed)
    feats = torch.rand(C, P, generator=g) * 2 - 1
    alphas = REGIMES[regime](g, (N, K, H, W)).float()
    idx = torch.randint(0, P, (N, K, H, W), generator=g)
    if hole:  # -1 in the middle of every pixel's list, and a few pixels with no point at all
        idx[:, K // 2] = -1
        idx[:, :, 0, 0] = -1
    if exact01:
        alphas[:, ::3] = 0.0
        alphas[:, 1::4] = 1.0
    if contention:
        idx[:, 0] = 0
    go = torch.randn(N, C, H, W, generator=g)
    return feats, alphas, idx, go


def feature_layout(feats, layout, dev):
    """(C,P) features as the kernels see them: 'contig' (C,P) array; 'pm' a (P,C).permute(1,0) view (point-major, the
    renderer's layout); 'pm_off' the same view starting 4 bytes into its allocation."""
    C, P = feats.shape
    if layout == "contig":
        return feats.to(dev)
    if layout == "pm":
        return feats.t().contiguous().to(dev).permute(1, 0)
    buf = torch.empty(P * C + 1, device=dev)
    view = buf[1:].view(P, C)
    view.copy_(feats.t())
    return view.permute(1, 0)


def old_division_scheme(feats, alphas, idx, go):
    """grad_alphas as the compositing backward computed them before: the full transmittance product, then cum_k
    recovered by dividing by (1 - alpha_k) walking backwards (O(K^2) recompute when |1 - alpha_k| <= 1e-6), in
    float32 -- the mutant the comparison must reject."""
    f, a, gout = feats.numpy(), alphas.numpy(), go.numpy()
    i = idx.numpy()
    N, K, H, W = i.shape
    valid = i >= 0
    G = f[:, np.clip(i, 0, None)]                                          # (C,N,K,H,W)
    A = (gout.transpose(1, 0, 2, 3)[:, :, None] * G).sum(0, dtype=np.float32)
    cum = np.ones((N, H, W), np.float32)
    for k in range(K):
        cum = np.where(valid[:, k], cum * (np.float32(1) - a[:, k]), cum).astype(np.float32)
    ga = np.zeros_like(a)
    suffix = np.zeros((N, H, W), np.float32)
    for k in range(K - 1, -1, -1):
        om = (np.float32(1) - a[:, k]).astype(np.float32)
        with np.errstate(divide="ignore", invalid="ignore"):
            ck = (cum / om).astype(np.float32)
        rec = np.ones((N, H, W), np.float32)
        for l in range(k):
            rec = np.where(valid[:, l], rec * (np.float32(1) - a[:, l]), rec).astype(np.float32)
        ck = np.where(np.abs(om) > 1e-6, ck, rec)
        gk = (ck * A[:, k] - suffix / (om + np.float32(1e-9))).astype(np.float32)
        ga[:, k] = np.where(valid[:, k], gk, 0)
        suffix = np.where(valid[:, k], suffix + ck * a[:, k] * A[:, k], suffix).astype(np.float32)
        cum = np.where(valid[:, k], ck, cum)
    return torch.from_numpy(ga)


def mesh_scene(F, H, W, K, blur, persp, clip, seed, empty_middle=True):
    """N = 3 meshes, the middle one empty; pix_to_face from the oracle in the kernels' arithmetic."""
    fv, _, _ = rand_faces(F, 2, seed)
    F1 = F // 2
    first = torch.tensor([0, F1, F1])
    num = torch.tensor([F1, 0, F - F1])
    if not empty_middle:
        first, num = split(F, 3)
    p2f, zb, bary, d = oracle.rasterize_meshes(fv.numpy(), first.numpy(), num.numpy(), (H, W), blur, K, persp, clip,
                                               arith=oracle.ARITH_CUDA, select=oracle.SELECT_CUDA)
    return fv, first, num, torch.from_numpy(p2f), (zb.shape, bary.shape, d.shape)


def masked_upstream(fv, p2f, shapes, persp, clip, seed=231):
    """Seeded upstream gradients with the singular slots zeroed (both sides get the same inputs)."""
    gz, gb, gd = upstream(shapes, seed)
    dev = fv.device
    gz, gb, gd = gz.to(dev), gb.to(dev), gd.to(dev)
    _, _, sing = R.rasterize_meshes_backward(fv, p2f, gz, gb, gd, persp, clip)
    gz[sing] = 0
    gb[sing] = 0
    gd[sing] = 0
    n_valid = int((p2f >= 0).sum())
    frac = float(sing.sum()) / max(n_valid, 1)
    assert frac <= MAX_SINGULAR, "%.3f of the slots are singular: the mask would hollow the test out" % frac
    return gz, gb, gd, frac


def check_mesh(got, fv, p2f, gz, gb, gd, persp, clip, what):
    ref, scale, _ = R.rasterize_meshes_backward(fv, p2f, gz, gb, gd, persp, clip)
    tau = mesh_tau(hits_per(p2f, fv.shape[0]))
    return R.check_close(got, ref, scale, tau, what)


# ------------------------------------------------------------------------------------------------ CPU: references

COMP_REF_CASES = [  # name, N, K, H, W, C, P, regime, hole, exact01
    ("uniform", 2, 10, 9, 11, 3, 40, "uniform", False, False),
    ("deep_chain", 1, 150, 4, 5, 3, 60, "deep", False, False),
    ("near_opaque", 2, 12, 6, 5, 4, 30, "opaque", False, False),
    ("exact_0_1", 1, 10, 6, 7, 5, 30, "uniform", False, True),
    ("hole", 2, 32, 5, 6, 9, 50, "uniform", True, False),
]


@pytest.mark.parametrize("name,N,K,H,W,C,P,regime,hole,exact01", COMP_REF_CASES)
def test_alpha_composite_reference_matches_oracle(name, N, K, H, W, C, P, regime, hole, exact01):
    feats, alphas, idx, go = comp_scene(N, K, H, W, C, P, regime, seed=K, hole=hole, exact01=exact01)
    ref = R.alpha_composite(feats, alphas, idx, go)
    out = oracle.alpha_composite(feats.numpy(), alphas.numpy(), idx.numpy(), arith=oracle.ARITH_CUDA)
    of, oa = oracle.alpha_composite_backward(go.numpy(), feats.numpy(), alphas.numpy(), idx.numpy())
    R.check_close(torch.from_numpy(out), ref["out"], ref["out_scale"], tau_terms(K + C), name + " forward")
    n = hits_per(idx, P).view(1, -1) + K + C
    R.check_close(torch.from_numpy(of), ref["grad_features"], ref["grad_features_scale"], tau_terms(n), name + " gf")
    R.check_close(torch.from_numpy(oa), ref["grad_alphas"], ref["grad_alphas_scale"], tau_terms(K + C), name + " ga")


@pytest.mark.parametrize("name", ["deep_chain", "near_opaque"])
def test_transmittance_by_division_is_rejected(name):
    """The backward's former scheme (cum_k recovered by division from the full product) loses slot 0 once the product
    underflows; the comparison must see it."""
    case = [c for c in COMP_REF_CASES if c[0] == name][0]
    _, N, K, H, W, C, P, regime, hole, exact01 = case
    feats, alphas, idx, go = comp_scene(N, K, H, W, C, P, regime, seed=K, hole=hole, exact01=exact01)
    ref = R.alpha_composite(feats, alphas, idx, go)
    with pytest.raises(AssertionError):
        R.check_close(old_division_scheme(feats, alphas, idx, go), ref["grad_alphas"], ref["grad_alphas_scale"],
                      tau_terms(K + C), name)


def test_transmittance_by_division_is_fine_for_short_chains():
    """... and is not rejected where it was right (K = 10, alpha in (0, 1)): the rejection above is the underflow."""
    _, N, K, H, W, C, P, regime, hole, exact01 = COMP_REF_CASES[0]
    feats, alphas, idx, go = comp_scene(N, K, H, W, C, P, regime, seed=K)
    ref = R.alpha_composite(feats, alphas, idx, go)
    R.check_close(old_division_scheme(feats, alphas, idx, go), ref["grad_alphas"], ref["grad_alphas_scale"],
                  tau_terms(K + C), "short chain")


@pytest.mark.parametrize("norm", [False, True])
def test_weighted_sum_reference_matches_oracle(norm):
    N, K, H, W, C, P = 2, 12, 7, 6, 5, 40
    feats, alphas, idx, go = comp_scene(N, K, H, W, C, P, "uniform", seed=3, hole=True)
    alphas[:, :, 1, :] = 1e-6  # the 1e-4 floor of the normalisation
    ref = R.weighted_sum(feats, alphas, idx, go, norm)
    out = oracle.weighted_sum(feats.numpy(), alphas.numpy(), idx.numpy(), norm=norm)
    of, oa = oracle.weighted_sum_backward(go.numpy(), feats.numpy(), alphas.numpy(), idx.numpy(), norm=norm)
    R.check_close(torch.from_numpy(out), ref["out"], ref["out_scale"], tau_terms(2 * K + C), "forward")
    n = hits_per(idx, P).view(1, -1) + 2 * K + C
    R.check_close(torch.from_numpy(of), ref["grad_features"], ref["grad_features_scale"], tau_terms(n), "gf")
    R.check_close(torch.from_numpy(oa), ref["grad_alphas"], ref["grad_alphas_scale"], tau_terms(2 * K + C), "ga")


def test_interp_face_attrs_reference_matches_oracle():
    g = torch.Generator().manual_seed(5)
    P, F, D = 500, 30, 17
    p2f = torch.randint(-1, F, (P,), generator=g)
    bary = torch.rand(P, 3, generator=g)
    attrs = torch.randn(F, 3, D, generator=g)
    go = torch.randn(P, D, generator=g)
    ref = R.interp_face_attrs(p2f, bary, attrs, go)
    out = oracle.interp_face_attrs(p2f.numpy(), bary.numpy(), attrs.numpy(), arith=oracle.ARITH_CUDA)
    gb, ga = oracle.interp_face_attrs_backward(p2f.numpy(), bary.numpy(), attrs.numpy(), go.numpy())
    R.check_close(torch.from_numpy(out), ref["out"], ref["out_scale"], tau_terms(3), "forward")
    R.check_close(torch.from_numpy(gb), ref["grad_bary"], ref["grad_bary_scale"], tau_terms(D), "grad_bary")
    n = hits_per(p2f, F).view(-1, 1, 1) + 3
    R.check_close(torch.from_numpy(ga), ref["grad_attrs"], ref["grad_attrs_scale"], tau_terms(n), "grad_attrs")


def test_points_backward_reference_matches_oracle():
    pts, first, num, rad = rand_points(300, 2, seed=4)
    H, W, K = 21, 27, 6
    idx, zb, d = oracle.rasterize_points(pts.numpy(), first.numpy(), num.numpy(), (H, W), rad.numpy(), K,
                                         arith=oracle.ARITH_CUDA, select=oracle.SELECT_CUDA)
    gz, gd = upstream([zb.shape, d.shape])
    ref, scale = R.rasterize_points_backward(pts, torch.from_numpy(idx), gz, gd)
    got = oracle.rasterize_points_backward(pts.numpy(), idx, gz.numpy(), gd.numpy(), arith=oracle.ARITH_CUDA)
    R.check_close(torch.from_numpy(got), ref, scale, tau_terms(hits_per(torch.from_numpy(idx), 300).view(-1, 1) + 4),
                  "grad_points")


@pytest.mark.parametrize("blur", [0.0, 1e-3])
@pytest.mark.parametrize("persp,clip", [(0, 0), (0, 1), (1, 0), (1, 1)])
def test_mesh_reference_matches_oracle(persp, clip, blur):
    fv, first, num, p2f, shapes = mesh_scene(240, 40, 36, 5, blur, persp, clip, seed=1)
    gz, gb, gd, _ = masked_upstream(fv, p2f, shapes, persp, clip)
    got = oracle.rasterize_meshes_backward(fv.numpy(), p2f.numpy(), gz.numpy(), gb.numpy(), gd.numpy(), persp, clip,
                                           arith=oracle.ARITH_CUDA)
    check_mesh(torch.from_numpy(got), fv, p2f, gz, gb, gd, persp, clip, "oracle")


# ------------------------------------------------------------------------------------------------ CPU: mutants

@pytest.fixture(scope="module")
def mesh_case():
    persp, clip, blur = 1, 1, 1e-3
    fv, first, num, p2f, shapes = mesh_scene(240, 40, 36, 5, blur, persp, clip, seed=1)
    gz, gb, gd, _ = masked_upstream(fv, p2f, shapes, persp, clip)
    good = oracle.rasterize_meshes_backward(fv.numpy(), p2f.numpy(), gz.numpy(), gb.numpy(), gd.numpy(), persp, clip,
                                            arith=oracle.ARITH_CUDA)
    return fv, p2f, gz, gb, gd, persp, clip, good


def test_mutant_dropped_pixel_is_rejected(mesh_case):
    fv, p2f, gz, gb, gd, persp, clip, _ = mesh_case
    active = (p2f >= 0) & ((gz != 0) | (gd != 0))
    slot = tuple(int(i) for i in torch.nonzero(active)[len(torch.nonzero(active)) // 2])
    gz2, gb2, gd2 = gz.clone(), gb.clone(), gd.clone()
    gz2[slot] = 0
    gb2[slot] = 0
    gd2[slot] = 0  # the kernel forgets this pixel's contribution to its face
    bad = oracle.rasterize_meshes_backward(fv.numpy(), p2f.numpy(), gz2.numpy(), gb2.numpy(), gd2.numpy(), persp, clip,
                                           arith=oracle.ARITH_CUDA)
    with pytest.raises(AssertionError):
        check_mesh(torch.from_numpy(bad), fv, p2f, gz, gb, gd, persp, clip, "dropped pixel")


def test_mutant_vertex_xy_swap_on_odd_face_is_rejected(mesh_case):
    """x and y of one vertex exchanged on an odd-indexed face: what a wrong parity choice of the 8-byte reductions
    would write."""
    fv, p2f, gz, gb, gd, persp, clip, good = mesh_case
    bad = good.copy()
    counts = hits_per(p2f, fv.shape[0])
    f = int([i for i in torch.argsort(counts, descending=True).tolist() if i % 2 == 1][0])
    bad[f, 1, [0, 1]] = bad[f, 1, [1, 0]]
    with pytest.raises(AssertionError):
        check_mesh(torch.from_numpy(bad), fv, p2f, gz, gb, gd, persp, clip, "xy swap")


def test_mutant_uncorrected_clip_backward_is_rejected(mesh_case):
    """The reference CUDA kernel's clip backward on the uncorrected barycentrics (DESIGN.md section 5)."""
    fv, p2f, gz, gb, gd, persp, clip, _ = mesh_case
    bad = oracle.rasterize_meshes_backward(fv.numpy(), p2f.numpy(), gz.numpy(), gb.numpy(), gd.numpy(), persp, clip,
                                           arith=oracle.ARITH_CUDA, clip_bwd_uncorrected=True)
    with pytest.raises(AssertionError):
        check_mesh(torch.from_numpy(bad), fv, p2f, gz, gb, gd, persp, clip, "uncorrected clip")


# ------------------------------------------------------------------------------------------------ GPU: meshes

DEV = "cuda:0"


def _gpu_mesh_forward(fv, first, num, H, W, blur, K, persp, clip):
    from pytorch3d_b200 import _C
    nb = torch.full((fv.shape[0],), -1, dtype=torch.int64, device=DEV)
    nb._b200_all_minus_one = True
    return _C.rasterize_meshes(fv.to(DEV), first.to(DEV), num.to(DEV), nb, (H, W), blur, K, 0, 0, bool(persp),
                               bool(clip), False)


# K -> the backward kernel it selects: K % 8 == 0 -> GV 8, K % 4 == 0 -> GV 4, else GV 0
MESH_GPU_CASES = [(K, pc, blur) for K, pc, blur in [
    (1, (0, 0), 0.0), (2, (1, 1), 1e-3), (3, (0, 1), 0.0), (5, (1, 0), 1e-3), (150, (1, 1), 1e-3),
    (4, (0, 0), 1e-3), (12, (1, 1), 0.0),
    (16, (0, 1), 1e-3), (40, (1, 0), 0.0)]] + [(8, pc, blur) for pc in [(0, 0), (0, 1), (1, 0), (1, 1)]
                                              for blur in [0.0, 1e-3]]


@pytest.mark.gpu
@pytest.mark.parametrize("K,pc,blur", MESH_GPU_CASES)
def test_mesh_backward_f64(built_lib, K, pc, blur):
    """_C.rasterize_meshes_backward on a 33 x 47 image (partial tiles), N = 3 with an empty middle mesh."""
    from pytorch3d_b200 import _C
    persp, clip = pc
    H, W = 33, 47
    fv, first, num, _, _ = mesh_scene(400, H, W, K, blur, persp, clip, seed=K)
    fvd = fv.to(DEV)
    p2f, zb, bary, d = _gpu_mesh_forward(fv, first, num, H, W, blur, K, persp, clip)
    gz, gb, gd, frac = masked_upstream(fvd, p2f, (zb.shape, bary.shape, d.shape), persp, clip)
    got = _C.rasterize_meshes_backward(fvd, p2f, gz, gb, gd, bool(persp), bool(clip))
    worst = check_mesh(got, fvd, p2f, gz, gb, gd, persp, clip, "mesh backward K=%d" % K)
    print("mesh K=%d persp=%d clip=%d blur=%g: singular %.4f, max |err|/scale %.3g" % (K, persp, clip, blur, frac, worst))


def _cover_faces(z_list, extent=2.0):
    """Two triangles per depth covering [-extent, extent]^2 (the diagonal runs off the pixel grid's centres)."""
    fs = []
    for z in z_list:
        fs.append([[-extent, -extent * 1.01, z], [extent, -extent, z + 0.1], [extent * 0.99, extent, z + 0.2]])
        fs.append([[-extent, -extent * 1.01, z], [extent * 0.99, extent, z + 0.2], [-extent, extent, z + 0.1]])
    return torch.tensor(fs, dtype=torch.float32)


def _stripe_faces(W, H, z=1.0):
    """One quad per pixel column, edges halfway between pixel centres: neighbouring lanes hit different faces."""
    _, xs = R.pixel_centres(H, W)
    xs = xs.numpy()
    edges = np.concatenate([[xs[0] + 0.5 * (xs[0] - xs[1])], 0.5 * (xs[1:] + xs[:-1]), [xs[-1] - 0.5 * (xs[0] - xs[1])]])
    fs = []
    for i in range(W):
        xa, xb = float(edges[i]), float(edges[i + 1])
        y0, y1 = -1.3, 1.31
        fs.append([[xa, y0, z], [xb, y0, z + 0.05], [xb, y1, z + 0.1]])
        fs.append([[xa, y0, z], [xb, y1, z + 0.1], [xa, y1, z + 0.05]])
    return torch.tensor(fs, dtype=torch.float32)


@pytest.mark.gpu
@pytest.mark.parametrize("pattern", ["cover", "stripes"])
def test_mesh_backward_warp_merge_f64(built_lib, pattern):
    """'cover': a few faces over the whole image, so all 32 lanes of a warp share each face and the pointer jumping
    runs all 5 rounds; 'stripes': neighbouring lanes alternate faces."""
    from pytorch3d_b200 import _C
    H, W, K = 40, 64, 8
    fv = _cover_faces([1.0, 1.5, 2.0, 2.5]) if pattern == "cover" else torch.cat(
        [_stripe_faces(W, H), _cover_faces([2.0])])
    first, num = torch.tensor([0]), torch.tensor([fv.shape[0]])
    fvd = fv.to(DEV)
    for persp, clip in [(0, 0), (1, 1)]:
        p2f, zb, bary, d = _gpu_mesh_forward(fv, first, num, H, W, 0.0, K, persp, clip)
        assert int((p2f >= 0).sum()) >= H * W
        gz, gb, gd, frac = masked_upstream(fvd, p2f, (zb.shape, bary.shape, d.shape), persp, clip)
        got = _C.rasterize_meshes_backward(fvd, p2f, gz, gb, gd, bool(persp), bool(clip))
        worst = check_mesh(got, fvd, p2f, gz, gb, gd, persp, clip, pattern)
        print("%s persp=%d clip=%d: singular %.4f, max |err|/scale %.3g" % (pattern, persp, clip, frac, worst))


@pytest.mark.gpu
@pytest.mark.parametrize("blur", [0.0, 1e-4])
def test_mesh_backward_north_star_f64(built_lib, blur):
    """The north-star batch (8 tori x 69,938 faces, 512 x 512, K = 8), every face compared, one image at a time."""
    from pytorch3d_b200 import _C, synthetic
    meshes = synthetic.torus_batch(8, 187, 187, seed=0)
    fv = synthetic.face_verts_of(meshes)
    first, num = meshes.mesh_to_faces_packed_first_idx(), meshes.num_faces_per_mesh()
    H = W = 512
    fvd = fv.to(DEV)
    p2f, zb, bary, d = _gpu_mesh_forward(fv, first, num, H, W, blur, 8, 0, 0)
    gz, gb, gd = (t.to(DEV) for t in upstream([zb.shape, bary.shape, d.shape]))
    n_sing = n_valid = 0
    for n in range(8):  # the mask, image by image
        _, _, sing = R.rasterize_meshes_backward(fvd, p2f[n:n + 1], gz[n:n + 1], gb[n:n + 1], gd[n:n + 1], 0, 0)
        gz[n][sing[0]] = 0
        gb[n][sing[0]] = 0
        gd[n][sing[0]] = 0
        n_sing += int(sing.sum())
        n_valid += int((p2f[n] >= 0).sum())
    assert n_sing <= MAX_SINGULAR * n_valid
    got = _C.rasterize_meshes_backward(fvd, p2f, gz, gb, gd, False, False)
    ref = torch.zeros_like(fvd, dtype=torch.float64)
    scale = torch.zeros_like(ref)
    for n in range(8):  # each image only touches its own mesh's faces
        r, s, _ = R.rasterize_meshes_backward(fvd, p2f[n:n + 1], gz[n:n + 1], gb[n:n + 1], gd[n:n + 1], 0, 0)
        ref += r
        scale += s
    worst = R.check_close(got, ref, scale, mesh_tau(hits_per(p2f, fv.shape[0])), "north-star blur=%g" % blur)
    print("north-star blur=%g: singular %.4f, max |err|/scale %.3g" % (blur, n_sing / n_valid, worst))


@pytest.mark.gpu
@pytest.mark.parametrize("persp,clip", [(0, 0), (1, 1)])
def test_mesh_backward_indexed_f64(built_lib, persp, clip):
    """rasterize_meshes_backward_indexed at K = 8: tori share every vertex among six faces, the grid mixes odd and even
    vertex indices, so both parities of the 8-byte vector reductions into grad_verts run."""
    from pytorch3d_b200 import _C, synthetic
    meshes = synthetic.torus_batch(2, 24, 24, seed=3)
    verts, faces = meshes.verts_packed().to(DEV), meshes.faces_packed().to(DEV)
    first, num = meshes.mesh_to_faces_packed_first_idx().to(DEV), meshes.num_faces_per_mesh().to(DEV)
    H, W, K = 72, 56, 8
    p2f, zb, bary, d, fv = _C.rasterize_meshes_indexed(verts, faces, first, num, (H, W), 1e-4, K, bool(persp),
                                                       bool(clip), False)
    gz, gb, gd, frac = masked_upstream(fv, p2f, (zb.shape, bary.shape, d.shape), persp, clip)
    got = _C.rasterize_meshes_backward_indexed(fv, faces, verts.shape[0], p2f, gz, gb, gd, bool(persp), bool(clip))
    _check_verts(got, fv, faces, verts.shape[0], p2f, gz, gb, gd, persp, clip, "indexed")
    print("indexed persp=%d clip=%d: singular %.4f" % (persp, clip, frac))


def _check_verts(got, fv, faces, V, p2f, gz, gb, gd, persp, clip, what):
    ref_f, scale_f, _ = R.rasterize_meshes_backward(fv, p2f, gz, gb, gd, persp, clip)
    fl = faces.reshape(-1)
    ref = torch.zeros((V, 3), dtype=torch.float64, device=fv.device).index_add_(0, fl, ref_f.reshape(-1, 3))
    scale = torch.zeros_like(ref).index_add_(0, fl, scale_f.reshape(-1, 3))
    slots_f = hits_per(p2f, fv.shape[0]).to(fv.device)
    slots_v = torch.zeros(V, dtype=torch.float64, device=fv.device).index_add_(0, fl, slots_f.repeat_interleave(3))
    return R.check_close(got, ref, scale, MESH_TAU + 2.0 * R.ULP * slots_v.view(-1, 1).cpu(), what)


@pytest.mark.gpu
def test_mesh_public_autograd_f64(built_lib):
    """pytorch3d_b200.rasterize_meshes(meshes, faces_per_pixel=8): the gradient w.r.t. the packed vertices."""
    import pytorch3d_b200 as p3b
    from pytorch3d_b200 import synthetic
    meshes = synthetic.torus_batch(2, 24, 24, seed=4, device=DEV)
    verts = meshes.verts_packed()
    meshes.requires_grad_(True)
    frags = p3b.rasterize_meshes(meshes, image_size=(64, 80), blur_radius=0.0, faces_per_pixel=8)
    p2f = frags[0]
    fv = verts.detach()[meshes.faces_packed()]
    gz, gb, gd, frac = masked_upstream(fv, p2f, (frags[1].shape, frags[2].shape, frags[3].shape), 0, 0)
    ((frags[1] * gz).sum() + (frags[2] * gb).sum() + (frags[3] * gd).sum()).backward()
    _check_verts(verts.grad, fv, meshes.faces_packed(), verts.shape[0], p2f, gz, gb, gd, 0, 0, "public autograd")


# ------------------------------------------------------------------------------------------------ GPU: C ABI fallbacks

def _p(t, offset_floats=0):
    return ctypes.c_void_p(t.data_ptr() + 4 * offset_floats)


@pytest.mark.gpu
def test_mesh_backward_unaligned_output_f64(built_lib):
    """The gradient buffer 4 bytes into a larger allocation: scalar reductions instead of the 8-byte vector ones, for
    both mesh entry points of the C ABI."""
    from pytorch3d_b200 import _C, _lib, synthetic
    lib = _lib.load()
    meshes = synthetic.torus_batch(2, 24, 24, seed=5)
    verts, faces = meshes.verts_packed().to(DEV), meshes.faces_packed().to(DEV)
    first, num = meshes.mesh_to_faces_packed_first_idx().to(DEV), meshes.num_faces_per_mesh().to(DEV)
    H, W, K = 48, 40, 8
    p2f, zb, bary, d, fv = _C.rasterize_meshes_indexed(verts, faces, first, num, (H, W), 0.0, K, False, False, False)
    gz, gb, gd, _ = masked_upstream(fv, p2f, (zb.shape, bary.shape, d.shape), 0, 0)
    F, V = fv.shape[0], verts.shape[0]
    stream = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    buf = torch.full((F * 9 + 1,), float("nan"), device=DEV)
    _lib.check(lib.b200r_rasterize_meshes_backward(_p(fv), F, _p(p2f), _p(gz), _p(gb), _p(gd), 2, H, W, K, 0, 0,
                                                   _p(buf, 1), stream))
    check_mesh(buf[1:].view(F, 3, 3), fv, p2f, gz, gb, gd, 0, 0, "face_verts, unaligned")
    vbuf = torch.full((V * 3 + 1,), float("nan"), device=DEV)
    _lib.check(lib.b200r_rasterize_meshes_backward_indexed(_p(fv), _p(faces), F, V, _p(p2f), _p(gz), _p(gb), _p(gd), 2,
                                                           H, W, K, 0, 0, _p(vbuf, 1), None, stream))
    _check_verts(vbuf[1:].view(V, 3), fv, faces, V, p2f, gz, gb, gd, 0, 0, "verts, unaligned")


# ------------------------------------------------------------------------------------------------ GPU: points

def _points_check(got, pts, idx, gz, gd, what):
    ref, scale = R.rasterize_points_backward(pts, idx, gz, gd)
    n = hits_per(idx, pts.shape[0]).view(-1, 1) + 4
    return R.check_close(got, ref, scale, tau_terms(n), what)


@pytest.mark.gpu
@pytest.mark.parametrize("K", [1, 7, 10, 32, 40, 150])
def test_points_backward_f64(built_lib, K):
    """K = 7 (W K % 4 != 0) and K > 32 take the unstaged kernel, the others the staged one; odd W, N = 2, and one hot
    point whose disc covers the whole image."""
    from pytorch3d_b200 import _C
    pts, first, num, rad = rand_points(2000, 2, seed=K)
    pts[0] = torch.tensor([0.0, 0.0, 1e-3])  # in front of (almost) every other point
    rad[0] = 3.0
    H, W = 30, 45
    pd, rd = pts.to(DEV), rad.to(DEV)
    idx, zb, d = _C.rasterize_points(pd, first.to(DEV), num.to(DEV), (H, W), rd, K, 0, 0)
    assert int((idx == 0).sum()) >= 0.9 * H * W
    gz, gd = (t.to(DEV) for t in upstream([zb.shape, d.shape]))
    got = _C.rasterize_points_backward(pd, idx, gz, gd)
    worst = _points_check(got, pd, idx, gz, gd, "points K=%d" % K)
    print("points K=%d: max |err|/scale %.3g" % (K, worst))


@pytest.mark.gpu
@pytest.mark.parametrize("which", ["grad_points", "grad_zbuf"])
def test_points_backward_unaligned_f64(built_lib, which):
    """Through the C ABI with grad_points 4 bytes into its allocation (scalar reductions), or grad_zbuf 4 bytes into
    its allocation (the unstaged kernel); every other buffer aligned."""
    from pytorch3d_b200 import _C, _lib
    lib = _lib.load()
    pts, first, num, rad = rand_points(1500, 2, seed=11)
    H, W, K = 31, 37, 8
    pd = pts.to(DEV)
    idx, zb, d = _C.rasterize_points(pd, first.to(DEV), num.to(DEV), (H, W), rad.to(DEV), K, 0, 0)
    gz, gd = (t.to(DEV) for t in upstream([zb.shape, d.shape]))
    P = pd.shape[0]
    stream = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    zbuf_in = torch.empty(gz.numel() + 1, device=DEV)
    zbuf_in[1:] = gz.reshape(-1)
    out = torch.full((P * 3 + 1,), float("nan"), device=DEV)
    if which == "grad_points":
        _lib.check(lib.b200r_rasterize_points_backward(_p(pd), P, _p(idx), _p(gz), _p(gd), 2, H, W, K, _p(out, 1),
                                                       stream))
        got = out[1:].view(P, 3)
    else:
        _lib.check(lib.b200r_rasterize_points_backward(_p(pd), P, _p(idx), _p(zbuf_in, 1), _p(gd), 2, H, W, K,
                                                       _p(out), stream))
        got = out[:P * 3].view(P, 3)
    _points_check(got, pd, idx, gz, gd, which + " unaligned")


# ------------------------------------------------------------------------------------------------ GPU: compositing

COMP_GPU_CASES = [  # id, N, K, H, W, C, P, regime, layout, hole, exact01, contention
    ("K1", 2, 1, 17, 23, 3, 300, "uniform", "contig", False, False, False),
    ("K10", 2, 10, 17, 23, 3, 300, "uniform", "contig", False, False, False),
    ("K32", 2, 32, 17, 23, 3, 300, "uniform", "contig", False, False, False),
    ("K100", 1, 100, 17, 23, 3, 300, "uniform", "contig", False, False, False),
    ("K150", 1, 150, 17, 23, 3, 300, "uniform", "contig", False, False, False),
    ("deep_chain", 1, 150, 16, 20, 4, 300, "deep", "pm", False, False, False),
    ("deep_chain_C3", 1, 150, 16, 20, 3, 300, "deep", "contig", False, False, False),
    ("near_opaque", 2, 12, 16, 20, 4, 300, "opaque", "pm", False, False, False),
    ("near_opaque_C9", 2, 12, 16, 20, 9, 300, "opaque", "contig", False, False, False),
    ("exact_0_1", 2, 10, 16, 20, 5, 300, "uniform", "contig", False, True, False),
    ("hole", 2, 32, 16, 20, 8, 300, "uniform", "pm", True, False, False),
    ("C1", 2, 10, 16, 20, 1, 300, "uniform", "contig", False, False, False),
    ("C4_contig", 2, 10, 16, 20, 4, 300, "uniform", "contig", False, False, False),
    ("C4_pm", 2, 10, 16, 20, 4, 300, "uniform", "pm", False, False, False),
    ("C4_pm_offset", 2, 10, 16, 20, 4, 300, "uniform", "pm_off", False, False, False),
    ("C5_pm", 2, 10, 16, 20, 5, 300, "uniform", "pm", False, False, False),
    ("C9_pm", 2, 10, 16, 20, 9, 300, "uniform", "pm", False, False, False),
    ("C16", 2, 10, 16, 20, 16, 300, "uniform", "contig", False, False, False),
    ("contention", 2, 10, 32, 40, 4, 300, "uniform", "pm", False, False, True),
    ("above_grid_cap", 5, 4, 512, 512, 3, 5000, "uniform", "contig", False, False, False),
]


def _comp_inputs(case, seed):
    _, N, K, H, W, C, P, regime, layout, hole, exact01, contention = case
    feats, alphas, idx, go = comp_scene(N, K, H, W, C, P, regime, seed, hole=hole, exact01=exact01,
                                        contention=contention)
    return feats, alphas, idx, go, layout


@pytest.mark.gpu
@pytest.mark.parametrize("case", COMP_GPU_CASES, ids=[c[0] for c in COMP_GPU_CASES])
def test_alpha_composite_f64(built_lib, case):
    """accum_alphacomposite + _backward and the alpha_composite autograd wrapper."""
    from pytorch3d_b200 import _C, compositing
    feats, alphas, idx, go, layout = _comp_inputs(case, seed=len(case[0]))
    N, K, H, W = idx.shape
    C, P = feats.shape
    fd = feature_layout(feats, layout, DEV)
    ad, idd, god = alphas.to(DEV), idx.to(DEV), go.to(DEV)
    ref = R.alpha_composite(fd, ad, idd, god)
    out = _C.accum_alphacomposite(fd, ad, idd)
    R.check_close(out, ref["out"], ref["out_scale"], tau_terms(K + C), "forward")
    gf, ga = _C.accum_alphacomposite_backward(god, fd, ad, idd)
    n_f = hits_per(idx, P).view(1, -1) + K + C
    w1 = R.check_close(gf, ref["grad_features"], ref["grad_features_scale"], tau_terms(n_f), "grad_features")
    w2 = R.check_close(ga, ref["grad_alphas"], ref["grad_alphas_scale"], tau_terms(K + C), "grad_alphas")
    fa = fd.detach().clone().requires_grad_(True) if layout == "contig" else fd.detach().requires_grad_(True)
    aa = ad.clone().requires_grad_(True)
    (compositing.alpha_composite(idd, aa, fa) * god).sum().backward()
    R.check_close(fa.grad, ref["grad_features"], ref["grad_features_scale"], tau_terms(n_f), "autograd features")
    R.check_close(aa.grad, ref["grad_alphas"], ref["grad_alphas_scale"], tau_terms(K + C), "autograd alphas")
    print("alpha_composite %s: max |err|/scale gf %.3g ga %.3g" % (case[0], w1, w2))


@pytest.mark.gpu
@pytest.mark.parametrize("case", COMP_GPU_CASES, ids=[c[0] for c in COMP_GPU_CASES])
def test_points_alpha_render_f64(built_lib, case):
    """The fused op on the rasterizer's (N,H,W,K) int32 / float32 layout, d = r^2 (1 - alpha)."""
    from pytorch3d_b200 import _C
    feats, alphas, idx, go, layout = _comp_inputs(case, seed=len(case[0]) + 1)
    r = 0.05
    C, P = feats.shape
    K = idx.shape[1]
    dists = (r * r * (1 - alphas.double())).float().permute(0, 2, 3, 1).contiguous()
    i32 = idx.permute(0, 2, 3, 1).contiguous().int()
    fd = feature_layout(feats, layout, DEV)
    dd, idd, god = dists.to(DEV), i32.to(DEV), go.to(DEV)
    ref = R.points_alpha_render(fd, idd, dd, r, god)
    out = _C.points_alpha_render(fd, idd, dd, r)
    R.check_close(out, ref["out"], ref["out_scale"], tau_terms(K + C), "forward")
    gf, gdist = _C.points_alpha_render_backward(god, fd, idd, dd, r)
    n_f = hits_per(idx, P).view(1, -1) + K + C
    w1 = R.check_close(gf, ref["grad_features"], ref["grad_features_scale"], tau_terms(n_f), "grad_features")
    w2 = R.check_close(gdist, ref["grad_dists"], ref["grad_dists_scale"], tau_terms(K + C), "grad_dists")
    print("points_alpha_render %s: max |err|/scale gf %.3g gd %.3g" % (case[0], w1, w2))


WS_GPU_CASES = [  # id, N, K, H, W, C, P
    ("K1", 2, 1, 17, 23, 3, 300), ("K32", 2, 32, 17, 23, 4, 300), ("K150", 1, 150, 16, 20, 5, 300),
    ("C1", 2, 10, 16, 20, 1, 300), ("C8", 2, 10, 16, 20, 8, 300), ("C9", 2, 10, 16, 20, 9, 300),
    ("C16", 2, 10, 16, 20, 16, 300), ("above_grid_cap", 5, 4, 512, 512, 3, 5000)]


@pytest.mark.gpu
@pytest.mark.parametrize("norm", [False, True])
@pytest.mark.parametrize("case", WS_GPU_CASES, ids=[c[0] for c in WS_GPU_CASES])
def test_weighted_sums_f64(built_lib, case, norm):
    """accum_weightedsum[norm] + _backward; a row of pixels has its alphas below the 1e-4 floor."""
    from pytorch3d_b200 import _C
    _, N, K, H, W, C, P = case
    feats, alphas, idx, go = comp_scene(N, K, H, W, C, P, "uniform", seed=K + C, hole=True)
    alphas[:, :, 1, :] = 1e-7
    fd, ad, idd, god = feats.to(DEV), alphas.to(DEV), idx.to(DEV), go.to(DEV)
    ref = R.weighted_sum(fd, ad, idd, god, norm)
    out = (_C.accum_weightedsumnorm if norm else _C.accum_weightedsum)(fd, ad, idd)
    R.check_close(out, ref["out"], ref["out_scale"], tau_terms(2 * K + C), "forward")
    gf, ga = (_C.accum_weightedsumnorm_backward if norm else _C.accum_weightedsum_backward)(god, fd, ad, idd)
    n_f = hits_per(idx, P).view(1, -1) + 2 * K + C
    R.check_close(gf, ref["grad_features"], ref["grad_features_scale"], tau_terms(n_f), "grad_features")
    R.check_close(ga, ref["grad_alphas"], ref["grad_alphas_scale"], tau_terms(2 * K + C), "grad_alphas")


@pytest.mark.gpu
@pytest.mark.parametrize("P,F,D", [(4000, 60, 1), (4000, 60, 3), (4000, 60, 4), (4000, 60, 17), (4000, 60, 64),
                                   (1_300_000, 5000, 3)])
def test_interp_face_attrs_backward_f64(built_lib, P, F, D):
    """interp_face_attrs_backward with -1 slots and one hot face (a quarter of all slots); the last case has more
    slots than the grid holds threads (148 * 32 blocks of 256)."""
    from pytorch3d_b200 import _C
    g = torch.Generator().manual_seed(D)
    p2f = torch.randint(-1, F, (P,), generator=g)
    p2f[::4] = 7
    bary = torch.rand(P, 3, generator=g)
    attrs = torch.randn(F, 3, D, generator=g)
    go = torch.randn(P, D, generator=g)
    pd, bd, ad, gd = p2f.to(DEV), bary.to(DEV), attrs.to(DEV), go.to(DEV)
    ref = R.interp_face_attrs(pd, bd, ad, gd)
    out = _C.interp_face_attrs_forward(pd, bd, ad)
    R.check_close(out, ref["out"], ref["out_scale"], tau_terms(3), "forward")
    gb, ga = _C.interp_face_attrs_backward(pd, bd, ad, gd)
    R.check_close(gb, ref["grad_bary"], ref["grad_bary_scale"], tau_terms(D), "grad_bary")
    n = hits_per(p2f, F).view(-1, 1, 1) + 3
    R.check_close(ga, ref["grad_attrs"], ref["grad_attrs_scale"], tau_terms(n), "grad_attrs")

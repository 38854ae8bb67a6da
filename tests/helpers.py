"""Shared scene builders for the tests (seeded, tiny) and the stored outputs of the reference."""
import hashlib
import os

import numpy as np
import torch

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def rand_faces(F, N, seed, scale=0.2, zlo=0.5, zhi=3.0):
    g = torch.Generator().manual_seed(seed)
    c = torch.rand(F, 1, 3, generator=g) * 2 - 1
    v = c + (torch.rand(F, 3, 3, generator=g) - 0.5) * scale * 2
    v[..., 2] = zlo + (zhi - zlo) * torch.rand(F, 3, generator=g)
    first, num = split(F, N)
    return v.contiguous(), first, num


def split(E, N):
    per = E // N
    first = (torch.arange(N) * per).long()
    num = torch.full((N,), per).long()
    num[-1] = E - first[-1]
    return first, num


def rand_points(P, N, seed, rlo=0.03, rhi=0.15, z_ties=False):
    g = torch.Generator().manual_seed(seed)
    pts = torch.rand(P, 3, generator=g) * 2 - 1
    pts[:, 2] = torch.rand(P, generator=g) * 2 - 0.2
    if z_ties:
        pts[::5, 2] = 0.5
    rad = torch.rand(P, generator=g) * (rhi - rlo) + rlo
    first, num = split(P, N)
    return pts.contiguous(), first, num, rad.contiguous()


def upstream(shapes, seed=231):
    """Seeded upstream gradients (the reference's own seed, tests/test_rasterize_meshes.py:563)."""
    g = torch.Generator().manual_seed(seed)
    return [torch.randn(s, generator=g) for s in shapes]


def _np(x):
    return x.detach().cpu().numpy() if torch.is_tensor(x) else np.asarray(x)


def digest(*arrays):
    """SHA-256 over the dtype, shape and bytes of each array: equal digests <=> bit-identical arrays.  Bit-exact
    comparisons with the reference store this instead of the (large) outputs themselves."""
    h = hashlib.sha256()
    for a in arrays:
        a = np.ascontiguousarray(_np(a))
        h.update(("%s%r" % (a.dtype.str, a.shape)).encode())
        h.update(a.tobytes())
    return h.hexdigest()


def case_key(*parts):
    return "_".join(str(p) for p in parts)


_REFERENCE = {}


def reference_outputs(name):
    """tests/golden/<name>.npz -- outputs of the unmodified reference ops on the tests' seeded inputs, written by
    tests/golden/make_reference_outputs.py -- as {case: {field: array}}."""
    if name not in _REFERENCE:
        data = np.load(os.path.join(GOLDEN, name + ".npz"))
        cases = {}
        for key in data.files:
            case, field = key.rsplit("/", 1)
            cases.setdefault(case, {})[field] = data[key]
        _REFERENCE[name] = cases
    return _REFERENCE[name]


def sample_pixels(frags, pixels):
    """The slots of the given flat (image, row, column) pixel indices of every (N, H, W, K[, 3]) output, on the host."""
    out = []
    for t in frags:
        n_pix = t.shape[0] * t.shape[1] * t.shape[2]
        flat = t.reshape((n_pix,) + tuple(t.shape[3:]))
        out.append(_np(flat[torch.from_numpy(pixels).to(t.device)] if torch.is_tensor(t) else flat[pixels]))
    return out


def assert_equal_up_to_ties(mine, ref, what, max_tie_pixels=1e-3):
    """Fragments equal to the reference's coarse-to-fine kernels wherever those agree with its own naive kernel: its
    fine kernel visits a bin's faces in a nondeterministic order, so slots that hold DIFFERENT faces must hold the SAME
    depth (an exact z tie at the K-th place); floats bit-equal everywhere else.  zbuf is therefore bit-equal in full
    (`ref["zbuf_digest"]`, which makes every index mismatch a z tie); indices, barycentrics and distances are compared
    on the stored seeded sample of pixels (`ref["pixels"]`), where at most a fraction `max_tie_pixels` may hold tied
    faces.  Returns the number of such pixels."""
    assert digest(mine[1]) == str(ref["zbuf_digest"]), "%s: zbuf differs from the reference" % what
    n = len(ref["pixels"])
    p2f, bary, dists = sample_pixels((mine[0], mine[2], mine[3]), ref["pixels"])
    diff = p2f != ref["pix_to_face"]
    n_diff_px = int(diff.any(-1).sum())
    assert n_diff_px <= max_tie_pixels * n, "%s: %d of %d sampled pixels differ" % (what, n_diff_px, n)
    same = ~diff
    assert np.array_equal(dists[same], ref["dists"][same]) and np.array_equal(bary[same], ref["bary"][same]), \
        "%s: float outputs differ" % what
    return n_diff_px


def assert_frag_equal(a, b, what=""):
    """idx bit-exact; floats bit-exact as well (same arithmetic) unless tol is given."""
    a = [x.detach().cpu().numpy() if torch.is_tensor(x) else np.asarray(x) for x in a]
    b = [x.detach().cpu().numpy() if torch.is_tensor(x) else np.asarray(x) for x in b]
    assert np.array_equal(a[0], b[0]), "%s: index mismatch in %d slots" % (what, int((a[0] != b[0]).sum()))
    for i, (x, y) in enumerate(zip(a[1:], b[1:])):
        assert np.array_equal(x, y), "%s: float output %d differs, max abs %g" % (
            what, i, float(np.abs(x.astype(np.float64) - y).max()))

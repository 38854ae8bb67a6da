"""Plain float64 restatements of the differentiable ops, for checking the CUDA backward kernels.

Every function takes the op's float32 inputs (torch tensors, on any device), widens them to float64 and returns the
outputs and gradients together with, per output element, `scale`: the float64 sum of the absolute values of the terms
that make up that element.  A float32 implementation that rounds each term and each partial sum is within a small
multiple of (number of terms) * 2**-24 of `scale`, whatever the cancellation between the terms, so the tests compare
element by element with

    |g32 - g64| <= tau * scale64 + TINY

and never against the largest value of the array, which would let an element with small gradients be entirely wrong.

Gradients come from autograd of the float64 forward, except where the op is *defined* by a closed form that is not the
derivative of its forward (the compositing ops' grad_alphas, which follow the reference kernels' formulas, including
their epsilons and floors); those are written out explicitly.
"""
import numpy as np
import torch

F64 = torch.float64
ULP = 2.0 ** -24
TINY = 1e-30  # above every float32 denormal error (<= 1.4e-45 times the factors in these ops), below any real value

COMP_EPS = 1e-9      # alpha_composite.cu:20: grad_alpha divides by (1 - alpha + eps)
NORM_EPS = 1e-4      # norm_weighted_sum.cu:20: floor of the sum of the alphas


def check_close(got, want, scale, tau, what, tiny=TINY):
    """Assert |got - want| <= tau * scale + tiny element by element; return the largest (|err| - tiny) / scale, where
    scale > 0 (elements whose whole scale is denormal pass on `tiny` and count as 0)."""
    got = got.detach().to(F64).cpu()
    want, scale = want.detach().cpu(), scale.detach().cpu()
    err = (got - want).abs()
    tau = torch.as_tensor(tau, dtype=F64).cpu().expand_as(scale)
    bound = tau * scale + tiny
    bad = ~(err <= bound)  # (NaN fails too)
    if bool(bad.any()):
        i = int(torch.nonzero(bad.reshape(-1))[0])
        n_bad = int(bad.sum())
        raise AssertionError("%s: %d of %d elements outside tau; first at flat index %d: tau %.3g, got %.9g want %.9g "
                             "(scale %.3g, |err| / scale %.3g)" % (
                                 what, n_bad, bad.numel(), i, float(tau.reshape(-1)[i]), float(got.reshape(-1)[i]),
                                 float(want.reshape(-1)[i]), float(scale.reshape(-1)[i]),
                                 float(err.reshape(-1)[i] / max(float(scale.reshape(-1)[i]), 1e-300))))
    pos = scale > 0
    return float(((err[pos] - tiny).clamp(min=0) / scale[pos]).max()) if bool(pos.any()) else 0.0


# ------------------------------------------------------------------------------------------------ pixel centres

def ndc_range(S1, S2):
    r = np.float32(2.0)
    if S1 > S2:
        r = np.float32(np.float32(S1) * r / np.float32(S2))
    return r


def pix_to_ndc(i, S1, S2):
    """DESIGN.md section 4: h = rn(range * 0.5), p = rn(rn(fma(range, i, h) / S1) - h), in float32, for integer array i."""
    rng = ndc_range(S1, S2)
    h = np.float32(rng * np.float32(0.5))
    t = (np.float64(rng) * np.asarray(i, np.float64) + np.float64(h)).astype(np.float32)  # the fma: one rounding
    return (t / np.float32(S1)).astype(np.float32) - h


def pixel_centres(H, W):
    """float32 NDC centres of the pixel rows and columns (row y -> +Y up, column x -> +X left), as float64 tensors."""
    ys = pix_to_ndc(H - 1 - np.arange(H), H, W)
    xs = pix_to_ndc(W - 1 - np.arange(W), W, H)
    return torch.from_numpy(ys.astype(np.float64)), torch.from_numpy(xs.astype(np.float64))


# ------------------------------------------------------------------------------------------------ compositing

def alpha_composite(features, alphas, points_idx, grad_out):
    """result[n,c] = sum_k f[c, idx_k] cum_k alpha_k, cum_k = prod_{l<k, idx_l >= 0} (1 - alpha_l) (a -1 slot is skipped
    wherever it sits).  grad_features by autograd; grad_alphas by the reference's formula
    grad_alpha_k = cum_k A_k - sum_{t>k} cum_t alpha_t A_t / (1 - alpha_k + 1e-9),  A_t = sum_c g_c f[c, idx_t]
    (alpha_composite.cu:112-134), which near alpha = 1 is the defined op rather than the derivative.

    Returns dict(out, out_scale, grad_features, grad_features_scale, grad_alphas, grad_alphas_scale)."""
    dev = alphas.device
    valid = points_idx >= 0
    a = torch.where(valid, alphas.to(F64), torch.zeros((), dtype=F64, device=dev))
    go = grad_out.to(F64)
    feats = features.detach().to(F64).requires_grad_(True)
    idx = points_idx.clamp(min=0)
    G = feats[:, idx] * valid.to(F64)                               # (C,N,K,H,W)
    one_m = 1.0 - a                                                  # 1 on invalid slots: skipped by the product
    cum = torch.cat([torch.ones_like(one_m[:, :1]), torch.cumprod(one_m, 1)[:, :-1]], 1)
    w = cum * a                                                      # (N,K,H,W)
    out = (G * w).sum(2).permute(1, 0, 2, 3)                         # (N,C,H,W)
    out_scale = (G.abs() * w.abs()).sum(2).permute(1, 0, 2, 3)
    (gf,) = torch.autograd.grad(out, feats, go)
    Gd = G.detach()
    gop = go.permute(1, 0, 2, 3).unsqueeze(2)                        # (C,N,1,H,W)
    A = (gop * Gd).sum(0)                                            # (N,K,H,W)
    A_abs = (gop * Gd).abs().sum(0)
    gf_scale = torch.zeros_like(feats, dtype=F64).index_put_(
        (torch.arange(feats.shape[0], device=dev).view(-1, 1, 1, 1, 1), idx.unsqueeze(0).expand_as(Gd)),
        (gop.abs() * w.abs() * valid), accumulate=True)
    wA, wA_abs = w * A, w.abs() * A_abs
    S = wA.flip(1).cumsum(1).flip(1) - wA                           # sum over t > k
    S_abs = wA_abs.flip(1).cumsum(1).flip(1) - wA_abs
    den = 1.0 - a + COMP_EPS
    ga = torch.where(valid, cum * A - S / den, torch.zeros_like(A))
    ga_scale = torch.where(valid, cum.abs() * A_abs + S_abs / den.abs(), torch.zeros_like(A))
    return dict(out=out.detach(), out_scale=out_scale, grad_features=gf, grad_features_scale=gf_scale,
                grad_alphas=ga, grad_alphas_scale=ga_scale)


def points_alpha_render(features, idx, dists, radius, grad_images):
    """The fused point rendering: alpha = 1 - d * (1 / r^2) evaluated in float32 exactly as the kernel does (torch
    divides a tensor by a scalar as a product with the float reciprocal), then `alpha_composite` in float64 on the
    (N,H,W,K) layout.  grad_dists = -grad_alpha * (1 / r^2).  Returns dict(out, out_scale, grad_features,
    grad_features_scale, grad_dists, grad_dists_scale, alphas)."""
    r2 = torch.tensor(float(radius) * float(radius), dtype=torch.float32)
    inv = (torch.tensor(1.0, dtype=torch.float32) / r2).to(dists.device)
    alpha32 = 1.0 - dists * inv                                      # float32: one product, one difference
    perm = (0, 3, 1, 2)
    res = alpha_composite(features, alpha32.permute(*perm), idx.long().permute(*perm), grad_images)
    inv64 = inv.to(F64)
    return dict(out=res["out"], out_scale=res["out_scale"], grad_features=res["grad_features"],
                grad_features_scale=res["grad_features_scale"],
                grad_dists=(-res["grad_alphas"] * inv64).permute(0, 2, 3, 1),
                grad_dists_scale=(res["grad_alphas_scale"] * inv64).permute(0, 2, 3, 1), alphas=alpha32)


def weighted_sum(features, alphas, points_idx, grad_out, norm):
    """result[n,c] = sum_k alpha_k f[c, idx_k] (/ max(sum_k alpha_k, 1e-4) when norm).  grad_features by autograd;
    grad_alphas by the reference's formula (norm_weighted_sum.cu:147-153: (f S - sum_t alpha_t f_t) / S^2 with the
    floored S, weighted_sum.cu: f), summed over the channels."""
    dev = alphas.device
    valid = points_idx >= 0
    a = torch.where(valid, alphas.to(F64), torch.zeros((), dtype=F64, device=dev))
    go = grad_out.to(F64)
    feats = features.detach().to(F64).requires_grad_(True)
    idx = points_idx.clamp(min=0)
    G = feats[:, idx] * valid.to(F64)                               # (C,N,K,H,W)
    if norm:
        S = a.sum(1, keepdim=True).clamp(min=NORM_EPS)              # (N,1,H,W)
    else:
        S = torch.ones_like(a[:, :1])
    out = ((G * a).sum(2) / S[:, 0]).permute(1, 0, 2, 3)
    out_scale = ((G.abs() * a.abs()).sum(2) / S[:, 0]).permute(1, 0, 2, 3)
    (gf,) = torch.autograd.grad(out, feats, go)
    Gd = G.detach()
    gop = go.permute(1, 0, 2, 3).unsqueeze(2)
    A = (gop * Gd).sum(0)
    A_abs = (gop * Gd).abs().sum(0)
    gf_scale = torch.zeros_like(feats, dtype=F64).index_put_(
        (torch.arange(feats.shape[0], device=dev).view(-1, 1, 1, 1, 1), idx.unsqueeze(0).expand_as(Gd)),
        (gop.abs() * (a.abs() / S) * valid), accumulate=True)
    if norm:
        T = (a * A).sum(1, keepdim=True)
        T_abs = (a.abs() * A_abs).sum(1, keepdim=True)
        ga = A / S - T / (S * S)
        ga_scale = A_abs / S + T_abs / (S * S)
    else:
        ga, ga_scale = A, A_abs
    zero = torch.zeros_like(ga)
    return dict(out=out.detach(), out_scale=out_scale, grad_features=gf, grad_features_scale=gf_scale,
                grad_alphas=torch.where(valid, ga, zero), grad_alphas_scale=torch.where(valid, ga_scale, zero))


# ------------------------------------------------------------------------------------------------ interpolation

def interp_face_attrs(pix_to_face, bary, attrs, grad_out):
    """out[p] = sum_i bary[p,i] attrs[f_p, i] (0 where f_p < 0); gradients by autograd."""
    valid = (pix_to_face >= 0).to(F64).unsqueeze(1)
    f = pix_to_face.clamp(min=0)
    b = bary.detach().to(F64).requires_grad_(True)
    at = attrs.detach().to(F64).requires_grad_(True)
    g = grad_out.to(F64)
    terms = b.unsqueeze(2) * at[f] * valid.unsqueeze(2)              # (P,3,D)
    out = terms.sum(1)
    gb, ga = torch.autograd.grad(out, (b, at), g)
    gb_scale = (at.detach()[f].abs() * g.abs().unsqueeze(1)).sum(2) * valid
    ga_scale = torch.zeros_like(at.detach()).index_add_(
        0, f, b.detach().abs().unsqueeze(2) * g.abs().unsqueeze(1) * valid.unsqueeze(2))
    return dict(out=out.detach(), out_scale=terms.detach().abs().sum(1), grad_bary=gb, grad_bary_scale=gb_scale,
                grad_attrs=ga, grad_attrs_scale=ga_scale)


# ------------------------------------------------------------------------------------------------ point rasterizer

def rasterize_points_backward(points, idx, grad_zbuf, grad_dists):
    """dists = (x - px)^2 + (y - py)^2 and zbuf = z per (pixel, slot) with a point; gradient w.r.t. points (P,3) by
    autograd.  Pixel centres as the kernels compute them (float32), widened."""
    N, H, W, K = idx.shape
    dev = points.device
    ys, xs = (t.to(dev) for t in pixel_centres(H, W))
    sel = idx >= 0
    n, y, x, k = torch.nonzero(sel, as_tuple=True)
    p = idx[sel].long()
    pts = points.detach().to(F64).requires_grad_(True)
    q = pts[p]
    dx, dy = q[:, 0] - xs[x], q[:, 1] - ys[y]
    gd, gz = grad_dists[sel].to(F64), grad_zbuf[sel].to(F64)
    loss = (gd * (dx * dx + dy * dy)).sum() + (gz * q[:, 2]).sum()
    (g,) = torch.autograd.grad(loss, pts)
    terms = torch.stack([2 * gd.abs() * dx.detach().abs(), 2 * gd.abs() * dy.detach().abs(), gz.abs()], 1)
    scale = torch.zeros_like(g).index_add_(0, p, terms)
    return g, scale


# ------------------------------------------------------------------------------------------------ mesh rasterizer

# Slots whose derivative is discontinuous or ill-conditioned at the pixel: a float32 kernel can legitimately land on the
# other side of the kink, so the tests give these slots zero upstream gradient on both sides (see `mesh_slot_geometry`).
SLIVER_RATIO = 1e-3      # |area| < 1e-3 * longest_edge^2: the barycentrics lose ~10 bits to the division by the area
BARY_EDGE_ULPS = 2.0 ** -9    # |E_i| < 2^-9 of its two products: the float32 barycentric's relative error reaches
                              # 2^9 ulps (3e-5), and it can flip the inside test; tiny faces (tori) need this bound
BARY_ZERO = 1e-6         # |w_i| < 1e-6: the inside test / clip kink, whatever the magnitude of the products
PERSP_FLOOR = 2e-8       # sum of the perspective terms within 2x of the max(., 1e-8) floor
CLIP_FLOOR = 2e-5        # sum of the clipped barycentrics within 2x of the max(., 1e-5) floor
SEG_TIE = 1e-4           # the two nearest segments within 1e-4 (relative): float32 may pick the other one ...
SEG_SAME_POINT = 1e-12   # ... unless both nearest points are the same (the shared vertex), where the gradient agrees
SEG_T_EDGE = 1e-5        # segment parameter t within 1e-5 of 0 or 1: nearest point at a vertex, where segments meet
DEGENERATE_L2 = 1e-6     # an edge shorter than 1e-3: the reference's l2 <= 1e-8 special case is close


class _AbsBack(torch.autograd.Function):
    """Identity whose backward passes |adjoint|.  Wrapped around every operand of the forward, a backward pass with
    non-negative upstream gradients then sums |local derivative products| over every path of the chain rule: the sum
    of the absolute values of the terms of each gradient element, cancellation inside the chain included."""

    @staticmethod
    def forward(ctx, x):
        return x.view_as(x)

    @staticmethod
    def backward(ctx, g):
        return g.abs()


def _plain(x):
    return x


def _ops(P):
    return (lambda a, b: P(a) + P(b), lambda a, b: P(a) - P(b), lambda a, b: P(a) * P(b), lambda a, b: P(a) / P(b))


def _edge_terms(px, py, ax, ay, bx, by):
    return ((px - ax) * (by - ay)).abs() + ((py - ay) * (bx - ax)).abs()


def mesh_slot_forward(v, px, py, persp, clip, P=_plain):
    """The per-(pixel, face) forward of rasterize_meshes.cu / geometry_utils.cuh in float64 for M slots: v (M,3,3),
    px, py (M,).  Returns (z, bary (M,3), signed dist, info) -- info holds the quantities the singular-slot mask needs.
    P is applied to every operand (`_AbsBack` for the scale pass)."""
    add, sub, mul, div = _ops(P)

    def edge(px, py, ax, ay, bx, by):  # E(p, a, b) = (p.x - a.x)(b.y - a.y) - (p.y - a.y)(b.x - a.x)
        return sub(mul(sub(px, ax), sub(by, ay)), mul(sub(py, ay), sub(bx, ax)))

    def seg_dist(px, py, ax, ay, bx, by):  # squared distance to the segment ab, t clamped to [0, 1]
        bax, bay = sub(bx, ax), sub(by, ay)
        l2 = add(mul(bax, bax), mul(bay, bay))
        l2_safe = torch.where(l2.detach() > 0, l2, torch.ones_like(l2))
        t_raw = div(add(mul(bax, sub(px, ax)), mul(bay, sub(py, ay))), l2_safe)
        t = P(t_raw).clamp(0.0, 1.0)
        qx, qy = add(ax, mul(t, bax)), add(ay, mul(t, bay))
        dx, dy = sub(qx, px), sub(qy, py)
        d = add(mul(dx, dx), mul(dy, dy))
        ex, ey = sub(px, bx), sub(py, by)
        d_degen = add(mul(ex, ex), mul(ey, ey))  # l2 <= 1e-8: distance to b (geometry_utils.cuh)
        return torch.where(l2.detach() <= 1e-8, d_degen, d), t_raw.detach(), l2.detach(), qx.detach(), qy.detach()

    x0, y0, z0 = v[:, 0, 0], v[:, 0, 1], v[:, 0, 2]
    x1, y1, z1 = v[:, 1, 0], v[:, 1, 1], v[:, 1, 2]
    x2, y2, z2 = v[:, 2, 0], v[:, 2, 1], v[:, 2, 2]
    area = P(edge(x2, y2, x0, y0, x1, y1)) + 1e-8
    E = [edge(px, py, x1, y1, x2, y2), edge(px, py, x2, y2, x0, y0), edge(px, py, x0, y0, x1, y1)]
    w = [div(e, area) for e in E]
    info = {"area": area.detach(), "E": torch.stack([e.detach() for e in E], 1),
            "E_terms": torch.stack([_edge_terms(px, py, x1, y1, x2, y2), _edge_terms(px, py, x2, y2, x0, y0),
                                    _edge_terms(px, py, x0, y0, x1, y1)], 1).detach(),
            "w": torch.stack([t.detach() for t in w], 1)}
    if persp:
        t0, t1, t2 = mul(mul(w[0], z1), z2), mul(mul(z0, w[1]), z2), mul(mul(z0, z1), w[2])
        tsum = add(add(t0, t1), t2)
        info["persp_sum"] = tsum.detach()
        den = P(tsum).clamp(min=1e-8)
        b = [div(t0, den), div(t1, den), div(t2, den)]
    else:
        b = w
    inside = (b[0].detach() > 0) & (b[1].detach() > 0) & (b[2].detach() > 0)
    if clip:
        c = [P(t).clamp(min=0.0) for t in b]
        s = add(add(c[0], c[1]), c[2])
        info["clip_sum"] = s.detach()
        s = P(s).clamp(min=1e-5)
        bc = [div(t, s) for t in c]
    else:
        bc = b
    z = add(add(mul(bc[0], z0), mul(bc[1], z1)), mul(bc[2], z2))
    segs = [seg_dist(px, py, x0, y0, x1, y1), seg_dist(px, py, x0, y0, x2, y2), seg_dist(px, py, x1, y1, x2, y2)]
    D = torch.stack([s[0] for s in segs], 1)
    j = D.detach().argmin(1, keepdim=True)                      # first minimum: the e01, e02, e12 order of the kernel
    dist = D.gather(1, j).squeeze(1)
    info.update(D=D.detach(), T=torch.stack([s[1] for s in segs], 1), L2=torch.stack([s[2] for s in segs], 1),
                Q=torch.stack([torch.stack([s[3], s[4]], 1) for s in segs], 1), seg=j.squeeze(1), inside=inside)
    signed = torch.where(inside, -dist, dist)
    return z, torch.stack(bc, 1), signed, info


def mesh_singular_slots(v, info, persp, clip):
    """Boolean (M,) mask of the slots at a kink or an ill-conditioned point of the forward (thresholds above)."""
    e = v.detach()[:, [1, 2, 2], :2] - v.detach()[:, [0, 0, 1], :2]
    longest2 = (e * e).sum(-1).max(1).values
    m = info["area"].abs() < SLIVER_RATIO * longest2
    m |= (info["E"].abs() <= BARY_EDGE_ULPS * info["E_terms"]).any(1)
    m |= (info["w"].abs() < BARY_ZERO).any(1)
    if persp:
        m |= info["persp_sum"] < PERSP_FLOOR
    if clip:
        m |= info["clip_sum"] < CLIP_FLOOR
    Ds, order = info["D"].sort(1)
    Q = info["Q"].gather(1, order[:, :2, None].expand(-1, -1, 2))
    same_point = ((Q[:, 0] - Q[:, 1]) ** 2).sum(1) <= SEG_SAME_POINT  # both at their shared vertex: same gradient
    m |= ((Ds[:, 1] - Ds[:, 0]) <= SEG_TIE * Ds[:, 1]) & ~same_point
    t = info["T"].gather(1, info["seg"].unsqueeze(1)).squeeze(1)
    m |= ((t.abs() < SEG_T_EDGE) | ((t - 1).abs() < SEG_T_EDGE))
    m |= (info["L2"] < DEGENERATE_L2).any(1)
    return m


def rasterize_meshes_backward(face_verts, pix_to_face, grad_zbuf, grad_bary, grad_dists, persp, clip,
                              chunk=1 << 21):
    """Gradient w.r.t. face_verts (F,3,3) of sum(grad_zbuf * zbuf + grad_bary * bary + grad_dists * dists) for a fixed
    pix_to_face (N,H,W,K), by autograd of the float64 forward (DESIGN.md section 5: forward-consistent perspective +
    clip convention).  Returns (grad, scale, singular) -- `singular` (N,H,W,K) marks the slots of
    `mesh_singular_slots`; the caller zeroes their upstream gradients on both sides and calls again (the mask does
    not depend on the upstream gradients).  Slots are processed `chunk` at a time."""
    N, H, W, K = pix_to_face.shape
    dev = face_verts.device
    ys, xs = (t.to(dev) for t in pixel_centres(H, W))
    fv64 = face_verts.detach().to(F64)
    grad = torch.zeros_like(fv64)
    scale = torch.zeros_like(fv64)
    singular = torch.zeros(pix_to_face.shape, dtype=torch.bool, device=dev)
    flat_sel = torch.nonzero((pix_to_face >= 0).reshape(-1)).squeeze(1)
    gz_all, gd_all = grad_zbuf.reshape(-1), grad_dists.reshape(-1)
    gb_all = grad_bary.reshape(-1, 3)
    p2f_flat = pix_to_face.reshape(-1)
    for s in range(0, flat_sel.numel(), chunk):
        sl = flat_sel[s:s + chunk]
        f = p2f_flat[sl]
        pix = sl // K
        x, y = pix % W, (pix // W) % H
        v = fv64[f].clone().requires_grad_(True)
        px, py = xs[x], ys[y]
        z, bc, sd, info = mesh_slot_forward(v, px, py, persp, clip)
        singular.view(-1)[sl] = mesh_singular_slots(v, info, persp, clip)
        gz, gd, gb = gz_all[sl].to(F64), gd_all[sl].to(F64), gb_all[sl].to(F64)
        loss = (gz * z).sum() + (gb * bc).sum() + (gd * sd).sum()
        (total,) = torch.autograd.grad(loss, v)
        va = fv64[f].clone().requires_grad_(True)
        za, bca, sda, _ = mesh_slot_forward(va, px, py, persp, clip, P=_AbsBack.apply)
        loss_abs = (gz.abs() * za).sum() + (gb.abs() * bca).sum() + (gd.abs() * sda).sum()
        (per_slot_abs,) = torch.autograd.grad(loss_abs, va)
        grad.index_add_(0, f, total)
        scale.index_add_(0, f, per_slot_abs.abs())
    return grad, scale, singular

"""Compositing of point features (SURVEY.md 8f-2: alpha, weighted sum, normalised weighted sum): oracle pinned to the
reference CPU ops; CUDA path against oracle / reference (stored outputs, tests/golden/make_reference_outputs.py)."""
import numpy as np
import pytest
import torch

import oracle
from helpers import case_key, digest, reference_outputs


def scene(N, K, H, W, C, P, seed, frac_empty=0.3):
    g = torch.Generator().manual_seed(seed)
    feats = torch.rand(C, P, generator=g)
    alphas = torch.rand(N, K, H, W, generator=g)
    idx = torch.randint(0, P, (N, K, H, W), generator=g)
    # z-buffer style padding: once a slot is empty all later slots of that pixel are empty too
    n_valid = (torch.rand(N, 1, H, W, generator=g) * (K + 1) * (1 + frac_empty)).long().clamp(max=K)
    empty = torch.arange(K).view(1, K, 1, 1) >= n_valid
    idx[empty] = -1
    return feats, alphas, idx


REF_CASES = [(2, 5, 9, 11, 3, 40), (1, 1, 4, 4, 1, 5), (1, 10, 16, 8, 4, 100)]  # N, K, H, W, C, P
CUDA_CASES = [(2, 5, 9, 11, 3, 40, False), (2, 10, 33, 17, 4, 500, True), (1, 1, 4, 4, 1, 5, False),
              (3, 8, 20, 20, 8, 300, True)]  # N, K, H, W, C, P, permuted


@pytest.fixture(scope="module")
def ref_cpu():
    """Digests of the reference's C++ CPU ops on these seeded scenes (tests/golden/make_reference_outputs.py cpu)."""
    return reference_outputs("reference_cpu")


@pytest.mark.parametrize("N,K,H,W,C,P", REF_CASES)
def test_oracle_equals_reference_cpu(ref_cpu, N, K, H, W, C, P):
    want = ref_cpu[case_key("alpha", N, K, H, W, C, P)]
    feats, alphas, idx = scene(N, K, H, W, C, P, seed=K)
    got = oracle.alpha_composite(feats.numpy(), alphas.numpy(), idx.numpy(), arith=oracle.ARITH_CPU)
    assert digest(got) == str(want["forward"])
    go = torch.rand(got.shape, generator=torch.Generator().manual_seed(1))
    of, oa = oracle.alpha_composite_backward(go.numpy(), feats.numpy(), alphas.numpy(), idx.numpy())
    assert digest(of, oa) == str(want["backward"])


def test_oracle_closed_form():
    """Single pixel, two points: result = a0 f0 + (1-a0) a1 f1; an empty first slot is skipped."""
    feats = torch.tensor([[2.0, 3.0]])
    alphas = torch.tensor([0.25, 0.5]).view(1, 2, 1, 1)
    idx = torch.tensor([0, 1]).view(1, 2, 1, 1)
    out = oracle.alpha_composite(feats.numpy(), alphas.numpy(), idx.numpy())
    assert out.item() == pytest.approx(0.25 * 2 + 0.75 * 0.5 * 3)
    idx2 = torch.tensor([-1, 1]).view(1, 2, 1, 1)
    assert oracle.alpha_composite(feats.numpy(), alphas.numpy(), idx2.numpy()).item() == pytest.approx(0.5 * 3)


@pytest.mark.gpu
@pytest.mark.parametrize("N,K,H,W,C,P,permuted", CUDA_CASES)
def test_cuda_forward_backward(built_lib, N, K, H, W, C, P, permuted):
    from pytorch3d_b200 import _C, compositing
    dev = torch.device("cuda:0")
    feats, alphas, idx = scene(N, K, H, W, C, P, seed=N + K)
    fd = feats.to(dev)
    if permuted:  # the renderer's layout: (N,H,W,K) tensors viewed as (N,K,H,W)
        ad = alphas.permute(0, 2, 3, 1).contiguous().to(dev).permute(0, 3, 1, 2)
        idd = idx.permute(0, 2, 3, 1).contiguous().to(dev).permute(0, 3, 1, 2)
        assert not ad.is_contiguous()
    else:
        ad, idd = alphas.to(dev), idx.to(dev)
    out = _C.accum_alphacomposite(fd, ad, idd)
    want = oracle.alpha_composite(feats.numpy(), alphas.numpy(), idx.numpy(), arith=oracle.ARITH_CUDA)
    assert np.array_equal(out.cpu().numpy(), want), "forward must be bit-identical to the CUDA-form oracle"
    ref = reference_outputs("reference_cuda")[case_key("alpha_cuda", N, K, H, W, C, P)]
    assert digest(out) == str(ref["forward"]), "forward must be bit-identical to the reference CUDA kernel"
    go = torch.rand(out.shape, generator=torch.Generator().manual_seed(1))
    gf, ga = _C.accum_alphacomposite_backward(go.to(dev), fd, ad, idd)
    of, oa = oracle.alpha_composite_backward(go.numpy(), feats.numpy(), alphas.numpy(), idx.numpy())
    np.testing.assert_allclose(gf.cpu().numpy(), of, rtol=1e-4, atol=1e-5)
    # the reference formula divides by (1 - alpha_t + 1e-9): near alpha = 1 it is ill-conditioned, so compare
    # where alphas stay away from 1 and require everything finite
    ok = (alphas < 0.99).all(1, keepdim=True).expand_as(alphas).numpy()
    np.testing.assert_allclose(ga.cpu().numpy()[ok], oa[ok], rtol=2e-3, atol=1e-4)
    assert torch.isfinite(ga).all()
    # autograd wrapper
    fa = fd.clone().requires_grad_(True)
    aa = ad.clone().requires_grad_(True)
    img = compositing.alpha_composite(idd, aa, fa)
    (img * go.to(dev)).sum().backward()
    np.testing.assert_allclose(fa.grad.cpu().numpy(), of, rtol=1e-4, atol=1e-5)


@pytest.mark.gpu
def test_points_renderer_pipeline(built_lib):
    """rasterize_points -> weights 1 - d/r^2 -> alpha_composite, as PointsRenderer does (points/renderer.py:56-76)."""
    import pytorch3d_b200 as p3b
    from pytorch3d_b200 import compositing, synthetic
    dev = torch.device("cuda:0")
    pc = synthetic.random_pointclouds(2, 5000, seed=3, device=dev)
    r = 0.05
    idx, zbuf, dists = p3b.rasterize_points(pc, (48, 64), radius=r, points_per_pixel=6)
    weights = (1 - dists / (r * r)).permute(0, 3, 1, 2)
    feats = torch.rand(4, pc.points_packed().shape[0], device=dev)
    img = compositing.AlphaCompositor(background_color=(0.0, 0.0, 0.0))(idx.long().permute(0, 3, 1, 2), weights, feats)
    want = oracle.alpha_composite(feats.cpu().numpy(), weights.contiguous().cpu().numpy(),
                                  idx.long().permute(0, 3, 1, 2).contiguous().cpu().numpy(), arith=oracle.ARITH_CUDA)
    covered = (idx[..., 0] >= 0).cpu().numpy()
    got = img.cpu().numpy()
    assert np.array_equal(got.transpose(0, 2, 3, 1)[covered][:, :4], want.transpose(0, 2, 3, 1)[covered])
    assert (got.transpose(0, 2, 3, 1)[~covered][:, :3] == 0).all()


# ------------------------------------------------------------------------------------ weighted sums

@pytest.mark.parametrize("norm", [False, True])
@pytest.mark.parametrize("N,K,H,W,C,P", REF_CASES)
def test_weighted_sum_oracle_equals_reference_cpu(ref_cpu, norm, N, K, H, W, C, P):
    want = ref_cpu[case_key("weighted_sum", norm, N, K, H, W, C, P)]
    feats, alphas, idx = scene(N, K, H, W, C, P, seed=K + 7)
    if norm:
        alphas[:, :, 0, 0] = 1e-6  # total below the 1e-4 floor
    got = oracle.weighted_sum(feats.numpy(), alphas.numpy(), idx.numpy(), norm=norm)
    assert digest(got) == str(want["forward"])
    go = torch.rand(got.shape, generator=torch.Generator().manual_seed(1))
    of, oa = oracle.weighted_sum_backward(go.numpy(), feats.numpy(), alphas.numpy(), idx.numpy(), norm=norm)
    assert digest(of, oa) == str(want["backward"])


@pytest.mark.gpu
@pytest.mark.parametrize("norm", [False, True])
@pytest.mark.parametrize("N,K,H,W,C,P,permuted", CUDA_CASES)
def test_weighted_sum_cuda_forward_backward(built_lib, norm, N, K, H, W, C, P, permuted):
    from pytorch3d_b200 import _C, compositing
    dev = torch.device("cuda:0")
    feats, alphas, idx = scene(N, K, H, W, C, P, seed=N + K + 3)
    if norm:
        alphas[:, :, 0, 0] = 1e-6
    fd = feats.to(dev)
    if permuted:
        ad = alphas.permute(0, 2, 3, 1).contiguous().to(dev).permute(0, 3, 1, 2)
        idd = idx.permute(0, 2, 3, 1).contiguous().to(dev).permute(0, 3, 1, 2)
    else:
        ad, idd = alphas.to(dev), idx.to(dev)
    fwd = _C.accum_weightedsumnorm if norm else _C.accum_weightedsum
    bwd = _C.accum_weightedsumnorm_backward if norm else _C.accum_weightedsum_backward
    out = fwd(fd, ad, idd)
    want = oracle.weighted_sum(feats.numpy(), alphas.numpy(), idx.numpy(), norm=norm)
    assert np.array_equal(out.cpu().numpy(), want), "forward must be bit-identical to the oracle"
    ref = reference_outputs("reference_cuda")[case_key("weighted_sum_cuda", norm, N, K, H, W, C, P)]
    assert digest(out) == str(ref["forward"]), "forward must equal the reference CUDA kernel"
    go = torch.rand(out.shape, generator=torch.Generator().manual_seed(1))
    gf, ga = bwd(go.to(dev), fd, ad, idd)
    of, oa = oracle.weighted_sum_backward(go.numpy(), feats.numpy(), alphas.numpy(), idx.numpy(), norm=norm)
    np.testing.assert_allclose(gf.cpu().numpy(), of, rtol=1e-4, atol=1e-4 * np.abs(of).max())
    np.testing.assert_allclose(ga.cpu().numpy(), oa, rtol=2e-4, atol=2e-4 * max(np.abs(oa).max(), 1e-2))
    # autograd wrappers + compositor module
    fa = fd.clone().requires_grad_(True)
    aa = ad.clone().requires_grad_(True)
    img = (compositing.norm_weighted_sum if norm else compositing.weighted_sum)(idd, aa, fa)
    (img * go.to(dev)).sum().backward()
    np.testing.assert_allclose(fa.grad.cpu().numpy(), of, rtol=1e-4, atol=1e-4 * np.abs(of).max())
    np.testing.assert_allclose(aa.grad.cpu().numpy(), oa, rtol=2e-4, atol=2e-4 * max(np.abs(oa).max(), 1e-2))
    if norm:
        img2 = compositing.NormWeightedCompositor(background_color=(0.5,) * C)(idd, ad, fd)
        bg = (idx[:, 0] < 0).to(dev)
        assert torch.equal(img2.permute(0, 2, 3, 1)[~bg], out.permute(0, 2, 3, 1)[~bg])
        assert (img2.permute(0, 2, 3, 1)[bg] == 0.5).all()


# ------------------------------------------------------------------------------------ fused point rendering

@pytest.mark.gpu
@pytest.mark.parametrize("P,N,size,K,C,r", [(3000, 2, (40, 56), 6, 4, 0.08), (20000, 3, (64, 64), 10, 3, 0.03),
                                           (500, 1, (17, 33), 1, 1, 0.2), (2000, 2, (32, 48), 5, 7, 0.1),
                                           (1500, 1, (24, 24), 4, 12, 0.1)])
def test_fused_point_rendering_equals_the_unfused_chain(built_lib, P, N, size, K, C, r):
    """`render_points_alpha(fragments, features, r)` = what PointsRenderer does with an AlphaCompositor
    (pytorch3d/renderer/points/renderer.py:63-73): weights = 1 - dists / r^2 (torch), idx.long(), two permutes and
    alpha_composite -- forward bit for bit, gradients w.r.t. features and dists to rounding (different summation order
    of the atomics only)."""
    from pytorch3d_b200 import _C, compositing, synthetic
    dev = torch.device("cuda:0")
    pc = synthetic.random_pointclouds(N, P, seed=P)
    pts = pc.points_packed().to(dev)
    rad = torch.full((pts.shape[0],), r, device=dev)
    idx, zbuf, dists = _C.rasterize_points(pts, pc.cloud_to_packed_first_idx().to(dev),
                                           pc.num_points_per_cloud().to(dev), size, rad, K, 0, 0)
    g = torch.Generator().manual_seed(7)
    if K != 6:  # the renderer's layout: features_packed() is (P, C); the compositor gets its (C, P) view
        feats = torch.rand(pts.shape[0], C, generator=g).to(dev).permute(1, 0)
    else:       # a plain contiguous (C, P) array
        feats = torch.rand(C, pts.shape[0], generator=g).to(dev)
    go = torch.rand((N, C) + tuple(size), generator=g).to(dev)
    # the unfused chain, as the reference renderer writes it
    d1 = dists.clone().requires_grad_(True)
    f1 = feats.clone().requires_grad_(True)
    weights = 1 - d1.permute(0, 3, 1, 2) / (r * r)
    img1 = compositing.alpha_composite(idx.long().permute(0, 3, 1, 2), weights, f1)
    (img1 * go).sum().backward()
    # fused
    d2 = dists.clone().requires_grad_(True)
    f2 = feats.clone().requires_grad_(True)
    img2 = compositing.render_points_alpha((idx, zbuf, d2), f2, r)
    (img2 * go).sum().backward()
    assert torch.equal(img1, img2), "fused forward must be bit-identical to the unfused chain"
    assert torch.allclose(f1.grad, f2.grad, rtol=1e-4, atol=1e-5 * float(f1.grad.abs().max()))
    assert torch.allclose(d1.grad, d2.grad, rtol=1e-4, atol=1e-5 * float(d1.grad.abs().max()))
    assert int((idx >= 0).sum()) > 0

"""interpolate_face_attributes (SURVEY.md 8f-3): oracle vs fixtures from the reference's CPU path; CUDA path vs oracle
and vs the reference's CUDA op (stored outputs, tests/golden/make_reference_outputs.py)."""
import numpy as np
import pytest
import torch

import oracle
from helpers import case_key, digest, reference_outputs

CUDA_CASES = [(2, 9, 11, 3, 50, 3), (1, 4, 4, 1, 6, 1), (2, 16, 16, 4, 300, 16)]  # N, H, W, K, F, D


def scene(N, H, W, K, F, D):
    """(pix_to_face, bary, attrs) and the generator that made them (it seeds the upstream gradient next)."""
    g = torch.Generator().manual_seed(F + D)
    p2f = torch.randint(-1, F, (N, H, W, K), generator=g)
    bary = torch.rand(N, H, W, K, 3, generator=g)
    attrs = torch.randn(F, 3, D, generator=g)
    return p2f, bary, attrs, g


def test_oracle_matches_reference_fixtures(golden):
    names = sorted(k for k in golden if k.startswith("interp/"))
    assert len(names) == 3
    for name in names:
        c = golden[name]
        got = oracle.interp_face_attrs(c["pix_to_face"], c["bary"], c["attrs"], arith=oracle.ARITH_CPU)
        want = c["out"].reshape(got.shape)
        # the reference's CPU path is a torch expression (broadcast multiply + sum over 3 terms)
        np.testing.assert_allclose(got, want, rtol=1e-6, atol=1e-7)
        assert (got[c["pix_to_face"].reshape(-1) < 0] == 0).all()


def test_invalid_shapes_raise(built_lib):
    from pytorch3d_b200.interp_face_attrs import interpolate_face_attributes
    with pytest.raises(ValueError, match="Faces can only have three vertices"):
        interpolate_face_attributes(torch.zeros(1, 2, 2, 1, dtype=torch.int64), torch.zeros(1, 2, 2, 1, 3),
                                    torch.zeros(5, 4, 2))
    with pytest.raises(ValueError, match="pix_to_face must have shape"):
        interpolate_face_attributes(torch.zeros(1, 2, 3, 1, dtype=torch.int64), torch.zeros(1, 2, 2, 1, 3),
                                    torch.zeros(5, 3, 2))


@pytest.mark.gpu
@pytest.mark.parametrize("N,H,W,K,F,D", CUDA_CASES)
def test_cuda_forward_backward(built_lib, N, H, W, K, F, D):
    from pytorch3d_b200 import _C
    from pytorch3d_b200.interp_face_attrs import interpolate_face_attributes
    dev = torch.device("cuda:0")
    p2f, bary, attrs, g = scene(N, H, W, K, F, D)
    out = _C.interp_face_attrs_forward(p2f.reshape(-1).to(dev), bary.reshape(-1, 3).to(dev), attrs.to(dev))
    want = oracle.interp_face_attrs(p2f.numpy(), bary.numpy(), attrs.numpy(), arith=oracle.ARITH_CUDA)
    assert np.array_equal(out.cpu().numpy(), want), "forward must be bit-identical to the CUDA-form oracle"
    ref = reference_outputs("reference_cuda")[case_key("interp", N, H, W, K, F, D)]
    assert digest(out) == str(ref["forward"]), "forward must be bit-identical to the reference CUDA kernel"
    go = torch.randn(out.shape, generator=g)
    gb, ga = _C.interp_face_attrs_backward(p2f.reshape(-1).to(dev), bary.reshape(-1, 3).to(dev), attrs.to(dev),
                                           go.to(dev))
    ob, oa = oracle.interp_face_attrs_backward(p2f.numpy(), bary.numpy(), attrs.numpy(), go.numpy())
    np.testing.assert_allclose(gb.cpu().numpy(), ob, rtol=1e-5, atol=1e-5)
    np.testing.assert_allclose(ga.cpu().numpy(), oa, rtol=1e-4, atol=1e-4)
    # autograd wrapper
    b2 = bary.to(dev).requires_grad_(True)
    a2 = attrs.to(dev).requires_grad_(True)
    vals = interpolate_face_attributes(p2f.to(dev), b2, a2)
    assert vals.shape == (N, H, W, K, D)
    (vals * go.to(dev).view_as(vals)).sum().backward()
    np.testing.assert_allclose(b2.grad.cpu().numpy().reshape(-1, 3), ob, rtol=1e-5, atol=1e-5)
    np.testing.assert_allclose(a2.grad.cpu().numpy(), oa, rtol=1e-4, atol=1e-4)

"""Decoder epilogue (next-row, SURVEY 8f rank 4): MLP output -> contiguous Gaussian-parameter tensors.

* CPU: the torch restatement is pinned bit-exactly against what the reference's own ``Decoder.forward_coarse`` +
  ``Network.get_offseted_pt`` (lightning/network.py) compute with an identity MLP (tests/golden/reference, made by
  tests/golden/make_reference_golden.py).
* GPU: the fused kernel vs the restatement -- forward values bit-exact except the sigmoid path (<= 2 ulp), backward
  to 1e-6."""
import pytest
import torch

from helpers import Reference, rel_err

def decoder_inputs():
    """MLP output features (identity MLP), group centres, K, sh_dim, opacity and scaling shifts."""
    B, N, K, sh_dim = 2, 27, 2, 12
    g = torch.Generator().manual_seed(0)
    feats = torch.randn((B, N, K * (10 + sh_dim)), generator=g)
    centers_grid = torch.rand((1, N, 3), generator=g) - 0.5
    return feats, centers_grid, K, sh_dim, -2.1792, -4.2


def test_decoder_restatement_matches_reference_on_cpu():
    from oracle.torch_restatements import decoder_layout_torch
    feats, centers_grid, K, sh_dim, opacity_shift, scaling_shift = decoder_inputs()
    mine = decoder_layout_torch(feats, centers_grid, K, sh_dim, opacity_shift, scaling_shift, 0.5 * 1.0 / 16)
    ref = Reference("decoder_layout")       # centres, sh, scaling, rotation, opacity
    for i, t in enumerate(mine):
        assert ref.equal(str(i), t), i


@pytest.mark.gpu
@pytest.mark.parametrize("B,N,K,sh_dim", [(1, 1000, 2, 12), (3, 4097, 1, 12), (2, 515, 2, 48), (1, 200, 3, 3)])
def test_decoder_layout_kernel_matches_restatement(cuda_device, B, N, K, sh_dim):
    from lara_b200.decoder_layout import gaussians_from_decoder
    from oracle.torch_restatements import decoder_layout_torch
    dev = cuda_device
    g = torch.Generator().manual_seed(N)
    C = 10 + sh_dim
    feats = (torch.randn((B, N, K * C), generator=g) * 2).to(dev)
    grid = (torch.rand((N, 3), generator=g) - 0.5).to(dev)
    ups = None
    res = []
    for fn in (gaussians_from_decoder, decoder_layout_torch):
        x = feats.clone().requires_grad_(True)
        out = fn(x, grid, K, sh_dim, -2.1792, -4.2, 0.03125)
        if ups is None:
            ups = [torch.randn(o.shape, generator=g).to(dev) for o in out]
        torch.autograd.backward(out, ups)
        res.append(([o.detach() for o in out], x.grad.detach()))
    (o1, g1), (o2, g2) = res
    for k, (a, b) in enumerate(zip(o1, o2)):
        assert a.shape == b.shape and a.is_contiguous(), k
        if k == 0:
            assert rel_err(a.cpu().numpy(), b.cpu().numpy()) < 1e-6       # sigmoid: torch's CUDA kernel vs expf-based, <= 2 ulp
        else:
            assert torch.equal(a, b), k
    assert rel_err(g1.cpu().numpy(), g2.cpu().numpy()) < 1e-6

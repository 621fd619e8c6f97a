"""GPU parity: distCUDA2 against the reference's SimpleKNN::knn (its outputs on these inputs are stored in
tests/golden/parity_test_knn_parity.npz, see tests/ref_golden.py).
The result is order-independent (exact 3-NN), so the bar is bit-exact."""
import pytest
import torch

from ref_golden import Golden

pytestmark = pytest.mark.gpu


import os
# BASELINE.json C5 initialises 5M points: always run at that size too (the reference kernel needs a few seconds there)
_FULL = [1000000, 5000000]          # BASELINE.json C3 / C5 point counts


@pytest.mark.parametrize("P", [1, 2, 3, 4, 7, 33, 1000, 1025, 50000, 262144] + _FULL)
def test_dist2_bit_exact_uniform(P, request):
    from simple_knn._C import distCUDA2
    g = torch.Generator().manual_seed(P)
    pts = (torch.rand(P, 3, generator=g) * 3 - 1.5).cuda()
    ours = distCUDA2(pts)
    torch.cuda.synchronize()
    assert Golden(request).equal("dist2", ours)


def test_dist2_clustered_and_duplicates(request):
    from simple_knn._C import distCUDA2
    g = torch.Generator().manual_seed(11)
    a = torch.randn(30000, 3, generator=g) * 0.01 + torch.tensor([1.0, 2.0, -3.0])
    b = torch.randn(30000, 3, generator=g) * 2.0
    c = a[:5000].clone()                      # exact duplicates -> zero distances
    d = torch.zeros(100, 3)                   # many coincident points
    e = torch.rand(1, 3, generator=g) * 1e4   # a far outlier
    pts = torch.cat([a, b, c, d, e]).cuda()
    pts = pts[torch.randperm(pts.shape[0], generator=g).cuda()]
    assert Golden(request).equal("dist2", distCUDA2(pts))


def test_dist2_grid_depth_image_like(request):
    # the real pipeline initialises from a 512x512 depth un-projection (gaussian_renderer/__init__.py:86)
    from simple_knn._C import distCUDA2
    n = 256
    ys, xs = torch.meshgrid(torch.linspace(-1, 1, n), torch.linspace(-1, 1, n), indexing="ij")
    z = 2 + 0.3 * torch.sin(3 * xs) * torch.cos(2 * ys)
    pts = torch.stack([xs * z, ys * z, z], -1).reshape(-1, 3).cuda()
    assert Golden(request).equal("dist2", distCUDA2(pts))

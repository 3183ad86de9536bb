"""ops.search_order (CPU): the k-d order of the culled search with every leaf in ascending caller index -- a permutation
with the same leaves as kd_order, which the ordered search relies on to return the lowest caller index among ties."""
import pytest
import torch

from reart_b200 import ops


@pytest.mark.parametrize("B,N,leaf", [(1, 300, 256), (3, 5000, 32), (2, 4096, 256), (1, 31, 32)])
def test_search_order_keeps_the_kd_leaves_and_sorts_inside_them(B, N, leaf):
    pts = torch.randn(B, N, 3, generator=torch.Generator().manual_seed(N))
    kd = ops.kd_order(pts, leaf)
    so = ops.search_order(pts, leaf)
    assert so.shape == (B, N)
    assert torch.equal(so.sort(dim=1).values, torch.arange(N)[None].expand(B, N))
    for s in range(0, N, leaf):
        blk = so[:, s:s + leaf]
        assert torch.equal(blk, kd[:, s:s + leaf].sort(dim=1).values)

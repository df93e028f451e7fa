"""twig/padded.py on the host: packing, per-image views and the size checks that run before any launch."""
import pytest
import torch

import common


def _cls():
    common.package()
    from dgtd_b200.twig.padded import PaddedBatch
    return PaddedBatch


def test_from_list_packs_top_left_and_unbind_returns_views():
    PaddedBatch = _cls()
    maps = [torch.rand(1, 5, 9), torch.rand(7, 3), torch.rand(1, 2, 2)]
    p = PaddedBatch.from_list(maps)
    assert p.data.shape == (3, 1, 7, 9) and p.data.dtype == torch.float32 and p.sizes == ((5, 9), (7, 3), (2, 2))
    views = p.unbind()
    for v, m in zip(views, maps):
        assert torch.equal(v, m.reshape(1, *m.shape[-2:])) and v.data_ptr() >= p.data.data_ptr()
    views[1].fill_(2.0)
    assert float(p.data[1, 0, :7, :3].min()) == 2.0
    sizes = p.device_sizes()
    assert sizes.dtype == torch.int32 and sizes.tolist() == [[5, 9], [7, 3], [2, 2]]
    q = p.empty_like()
    assert q.sizes == p.sizes and q.data.shape == p.data.shape and q.device_sizes() is sizes


@pytest.mark.parametrize("sizes, match", [([(1, 9), (7, 3)], "at least 2"), ([(5, 1), (7, 3)], "at least 2"),
                                          ([(8, 9), (7, 3)], "fit the 7 x 9"), ([(5, 10), (7, 3)], "fit the 7 x 9"),
                                          ([(5, 9)], "1 sizes for 2 images")])
def test_bad_sizes_raise(sizes, match):
    PaddedBatch = _cls()
    with pytest.raises(ValueError, match=match):
        PaddedBatch(torch.zeros(2, 1, 7, 9), sizes)


def test_from_list_rejects_multichannel_and_one_pixel_maps():
    PaddedBatch = _cls()
    with pytest.raises(ValueError, match=r"\(1, H, W\) or \(H, W\)"):
        PaddedBatch.from_list([torch.rand(3, 4, 4)])
    with pytest.raises(ValueError, match="at least 2"):
        PaddedBatch.from_list([torch.rand(1, 4, 4), torch.rand(1, 1, 4)])
    with pytest.raises(ValueError, match="no maps"):
        PaddedBatch.from_list([])

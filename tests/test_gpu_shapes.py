"""GPU parity of the tcgen05 correlation build + pooled lookup on EVERY shape BASELINE.json names
(SURVEY §8 head: cfg1 48x64, Replica 40x80, ScanNet 30x40, EuRoC 40x60 stereo, 640x480 -> 60x80)
against the CPU oracle — not only against the SIMT twin.  The irregular ones are what matters:
40x60 has w % 16 != 0 (ragged x-tile + padded tiles), 60x80 has h % 8 == 4 (ragged last band)
and 4800 / 128 = 37.5 (ragged last m-tile), 48x64 is the one CPU-shaped config."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from oracle import corr_oracle  # noqa: E402

SHAPES = [(48, 64), (40, 80), (30, 40), (40, 60), (60, 80)]


def dev():
    return torch.device("cuda:0")


def _coords(N, h, w, g):
    base = torch.stack(torch.meshgrid(torch.arange(w).float(), torch.arange(h).float(), indexing="xy"), -1)
    c = base[None, None].repeat(1, N, 1, 1, 1) + 3.0 * torch.randn(1, N, h, w, 2, generator=g)
    c[0, :, 0, :3] = torch.tensor([-5.5, 2.25])                  # windows hanging over every border
    c[0, :, 1, :3] = torch.tensor([w + 1.5, h - 2.0])
    c[0, :, 2, :3] = torch.tensor([w / 2.0, -3.75])
    c[0, :, 3, :3] = torch.tensor([w - 1.0, h - 1.0])            # integer coordinates at the last pixel
    return c


def _check_pyramid(got_levels, want_levels):
    for i, (got, want) in enumerate(zip(got_levels, want_levels)):
        got = got.float().cpu().numpy()
        want = want.float().numpy()
        assert got.shape == want.shape, (i, got.shape, want.shape)
        # fp32 accumulation in a different order, one rounding to half per level: <= 1 half-ulp,
        # and identical almost everywhere
        np.testing.assert_allclose(got, want, rtol=1.5e-3, atol=1e-3, err_msg="level %d" % i)
        assert (got == want).mean() > 0.97, (i, (got == want).mean())


@pytest.mark.parametrize("hw", SHAPES)
def test_tcgen05_build_vs_oracle(hw):
    """CorrBlock(fmap1, fmap2, impl=1) — the reference-layout tensor-core build — and the fused
    lookup on it, against the oracle (bit-exact for the half-precision lookup)."""
    from goslam_b200.modules import CorrBlock
    h, w = hw
    N = 2
    g = torch.Generator().manual_seed(100 + h)
    f1 = torch.randn(1, N, 128, h, w, generator=g).half()
    f2 = torch.randn(1, N, 128, h, w, generator=g).half()
    blk = CorrBlock(f1.to(dev()), f2.to(dev()), impl=1)
    _check_pyramid(blk.corr_pyramid, corr_oracle.corr_build(f1[0], f2[0], 4))
    coords = _coords(N, h, w, g)
    out = blk(coords.to(dev()))
    want = corr_oracle.corr_pyramid_lookup([p.cpu().numpy() for p in blk.corr_pyramid], coords[0].numpy(), 3)
    np.testing.assert_array_equal(out[0].cpu().numpy().astype(np.float32), want.astype(np.float32))


@pytest.mark.parametrize("layout", ["tiled", "rowmajor"])
@pytest.mark.parametrize("hw,rig", [((48, 64), 1), ((40, 80), 1), ((30, 40), 1), ((40, 60), 2), ((60, 80), 1),
                                    ((24, 96), 1)])
def test_pool_build_and_lookup_vs_oracle(hw, rig, layout):
    """FactorGraph's path: video-level K-major maps -> pooled (tiled / row-major) tensor-core build ->
    pooled 4-level lookup; stereo rigs use the right image for self-edges (src/factor_graph.py:108-111)."""
    from goslam_b200.modules import CorrBlock
    from goslam_b200.modules.corr import CorrPool, fmaps_to_kmajor
    h, w = hw
    g = torch.Generator().manual_seed(200 + h + rig)
    fmaps = torch.randn(4, rig, 128, h, w, generator=g).half()
    if rig == 2:
        ii = torch.tensor([0, 1, 2, 3, 1])
        jj = torch.tensor([1, 0, 2, 1, 1])            # (2,2) and (1,1) are stereo self-edges
    else:
        ii = torch.tensor([0, 1, 3])
        jj = torch.tensor([1, 0, 2])
    N = ii.numel()
    c = (ii == jj).long() if rig == 2 else torch.zeros_like(ii)
    want_pyr = corr_oracle.corr_build(fmaps[ii, 0], fmaps[jj, c], 4)
    km = fmaps_to_kmajor(fmaps.to(dev()))
    pool = CorrPool(N + 3, h, w, device=dev(), layout=layout)
    pool.alloc(2)                                       # edges do not start at slot 0
    blk = CorrBlock.from_video(km, ii.to(dev()), jj.to(dev()), h, w, rig=rig, pool=pool)
    got_pyr = blk.gather_pyramid()
    _check_pyramid(got_pyr, want_pyr)
    coords = _coords(N, h, w, g)
    out = blk(coords.to(dev()))
    want = corr_oracle.corr_pyramid_lookup([p.cpu().numpy() for p in got_pyr], coords[0].numpy(), 3)
    np.testing.assert_array_equal(out[0].cpu().numpy().astype(np.float32), want.astype(np.float32))

"""CPU: the oracle restatement reproduces the unmodified reference's outputs on the same seeded inputs
(tests/golden/pins_reference.npz, written by ``tools/make_golden.py pins`` from the reference itself).

Volumes and regressions must match BIT FOR BIT.  The hourglasses (3D convolutions), the geometry lookup (a batched matmul)
and the context up-sampling (9-tap windowed sums) run through CPU kernels whose summation order depends on the host CPU,
so against vectors stored on another host they are compared to within fp32 reordering: REORDER of the output's largest
magnitude (on the host that wrote them they are bit-equal)."""
import pytest
import torch

from oracle import aggregation as oagg
from oracle import cost_volume as ocv
from oracle import geo_lookup as ogeo
from oracle import regression as oreg
from oracle import seeded_init as si

from conftest import load_golden

REORDER = 1e-5


@pytest.fixture(scope="module")
def ref():
    return load_golden("pins_reference")


def rnd(seed, *shape):
    return torch.randn(*shape, generator=torch.Generator().manual_seed(seed))


def assert_pinned(got, g, key, exact=True):
    """got vs the reference output stored under `key`: whole, or a seeded sample plus the whole tensor's sums."""
    if key in g:
        want = g[key]
        assert got.shape == want.shape, key
        if exact:
            assert torch.equal(got, want), key
        else:
            assert (got - want).abs().max().item() <= REORDER * want.abs().max().item(), key
        return
    assert list(got.shape) == g[key + "__shape"].tolist(), key
    flat, want = got.reshape(-1)[g[key + "__idx"].long()], g[key + "__val"]
    if exact:
        assert torch.equal(flat, want), key
    else:
        assert (flat - want).abs().max().item() <= REORDER * want.abs().max().item(), key
    for name, total in (("__sum", got.double().sum()), ("__abssum", got.double().abs().sum())):
        assert total.item() == pytest.approx(g[key + name], rel=1e-9 if exact else REORDER, abs=1e-9), key + name


@pytest.mark.parametrize("b,c,h,w,d,g", [(2, 24, 4, 19, 7, 3), (1, 40, 3, 33, 40, 5), (1, 8, 2, 6, 9, 8)])
def test_volume_functions(ref, b, c, h, w, d, g):
    tag = "%d_%d_%d_%d_%d_%d" % (b, c, h, w, d, g)
    l, r = rnd(1, b, c, h, w), rnd(2, b, c, h, w)
    assert_pinned(ocv.build_gwc_volume(l, r, d, g), ref, "gwc_" + tag)
    assert_pinned(ocv.build_concat_volume(l, r, d), ref, "concat_" + tag)
    assert_pinned(ocv.correlation_volume(l, r, d), ref, "corr_" + tag)
    assert_pinned(ocv.cat_fms(l, r, max_disp=d), ref, "concat_" + tag)     # the reference's cat_fms equals its concat volume


def test_regression_functions(ref):
    p = torch.softmax(rnd(3, 2, 20, 5, 6) * 3, 1)
    assert_pinned(oreg.disparity_regression(p, 20), ref, "regression")
    assert_pinned(oreg.faster_soft_argmin(rnd(4, 2, 20, 5, 6), 20, alpha=2.0), ref, "faster_softargmin")


def test_hourglass_modules(ref):
    with torch.no_grad():
        mine = oagg.GwcHourglass(8).eval()
        mine.load_state_dict(si.seeded_state_dict(mine.state_dict(), seed=5))
        x = rnd(6, 1, 8, 4, 8, 8)
        assert_pinned(mine(x), ref, "gwc_hourglass", exact=False)
        mine = oagg.PSMHourglass(8).eval()
        mine.load_state_dict(si.seeded_state_dict(mine.state_dict(), seed=7))
        pre, post = rnd(8, 1, 16, 2, 4, 4), rnd(9, 1, 16, 2, 4, 4)
        for i, t in enumerate(mine(x, pre, post)):
            assert_pinned(t, ref, "psm_hourglass_%d" % i, exact=False)


@pytest.mark.parametrize("b,cf,cg,d,h,w,levels,radius", [(1, 5, 8, 24, 4, 30, 2, 4), (2, 3, 2, 9, 2, 11, 1, 3)])
def test_geo_lookup_classes(ref, b, cf, cg, d, h, w, levels, radius):
    f1, f2, vol = rnd(70, b, cf, h, w), rnd(71, b, cf, h, w), rnd(72, b, cg, d, h, w)
    disp = torch.rand(b, 1, h, w, generator=torch.Generator().manual_seed(73)) * (d + 4) - 2
    coords = torch.arange(w).float().reshape(1, 1, w, 1).repeat(b, h, 1, 1)
    mine = ogeo.GeoEncodingVolume(f1, f2, vol, num_levels=levels, radius=radius)(disp, coords)
    # the reference's IGEV and StereoBase classes gave the same output (checked when the vectors were written)
    assert_pinned(mine, ref, "geo_%d_%d_%d_%d_%d_%d_%d_%d" % (b, cf, cg, d, h, w, levels, radius), exact=False)


def test_context_upsample_function(ref):
    low, wts = rnd(74, 2, 1, 6, 9).abs() * 30, torch.softmax(rnd(75, 2, 9, 24, 36), dim=1)
    assert_pinned(ogeo.context_upsample(low, wts), ref, "context_upsample", exact=False)

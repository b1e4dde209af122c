"""CPU: host side of the opt-in fp16 route of StereoBase's hourglass -- the hi-only weight pack of the fp16-activation kernels and
the validation of patch(precision=...)."""
import pytest
import torch

import __graft_entry__

__graft_entry__.build()
from openstereo_b200 import ops                    # noqa: E402
from openstereo_b200.patch import patch            # noqa: E402


def rnd(seed, *shape):
    return torch.randn(*shape, generator=torch.Generator().manual_seed(seed))


@pytest.mark.parametrize("order", [(0, 1, 2), (1, 0, 2)])
def test_pack_tc_weight_h16_is_hi_only(order):
    """h16=True: the same power-of-two scaling per output channel as the split pack (max |w| 2^e in [2^14, 2^15), so no weight is
    flushed to a subnormal), hi = rn_fp16(w 2^e), lo halves zero, inv = 2^-e (no activation scale)."""
    cout, cin, kc = 8, 32, 16
    w = rnd(1, cout, cin, 3, 3, 3) * torch.logspace(-6, 6, cout).view(cout, 1, 1, 1, 1)
    p = ops.pack_tc_weight(w, kc, kw_order=order, h16=True)
    assert p.h16 and not ops.pack_tc_weight(w, kc, kw_order=order).h16
    assert p.data.shape == (3, cin // kc, 3, 3 * cout, 2 * kc) and p.data.dtype == torch.float16
    cpr = 2 * kc // 8
    key = (torch.arange(3 * cout) >> 1) & 3
    src = (torch.arange(cpr).view(1, cpr) ^ key.view(-1, 1)).view(1, 1, 1, 3 * cout, cpr, 1).expand(3, cin // kc, 3, 3 * cout, cpr, 8)
    lin = torch.gather(p.data.view(3, cin // kc, 3, 3 * cout, cpr, 8), 4, src).reshape(3, cin // kc, 3, 3 * cout, 2 * kc)
    t = lin.view(3, cin // kc, 3, 3, cout, 2, kc).permute(5, 4, 1, 6, 0, 2, 3).reshape(2, cout, cin, 3, 3, 3)
    hi, lo = t[0], t[1]
    assert (lo == 0).all()
    e = -torch.log2(p.inv.double())
    assert torch.equal(e, e.round())
    want = torch.ldexp(w[..., list(order)], e.round().to(torch.int32).view(-1, 1, 1, 1, 1)).to(torch.float16)
    assert torch.equal(hi, want)
    top = hi.double().abs().amax(dim=(1, 2, 3, 4))
    assert (top >= 2.0 ** 14).all() and (top <= 2.0 ** 15).all()
    split = ops.pack_tc_weight(w, kc, kw_order=order)
    assert torch.equal(split.inv, p.inv * 2.0 ** -ops.TC_ACT_SCALE_LOG2)
    d = ops.pack_tc_deconv_weight(rnd(2, 32, 16, 4, 4, 4), h16=True)
    assert d.h16 and d.ksize == 4


def test_patch_precision_validation():
    with pytest.raises(ValueError, match="precision"):
        patch(type("StereoBase", (torch.nn.Module,), {})(), precision="bf16")
    for name in ("GwcNet", "PSMNet", "LightStereo", "IGEVStereo"):
        with pytest.raises(ValueError, match=r"precision='fp16' is implemented for StereoBase only"):
            patch(type(name, (torch.nn.Module,), {})(), precision="fp16")


def test_engine_precision_validation():
    from openstereo_b200 import aggregation
    with pytest.raises(ValueError, match="precision"):
        aggregation.StereoBaseAggregation(torch.nn.Module(), precision="half")


def test_ops_refuse_a_mismatched_pack():
    w = rnd(3, 16, 16, 3, 3, 3)
    with pytest.raises(ValueError, match="h16=True"):
        ops._is_h16(torch.zeros(1, dtype=torch.float16), ops.pack_tc_weight(w, 16))
    with pytest.raises(ValueError, match="h16=False"):
        ops._is_h16(torch.zeros(1), ops.pack_tc_weight(w, 16, h16=True))
    with pytest.raises(TypeError):
        ops._is_h16(torch.zeros(1, dtype=torch.bfloat16))

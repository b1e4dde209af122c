"""CPU: patch() on the UNMODIFIED reference GwcNet / PSMNet classes (those tests need the reference tree and skip without it).

What can be checked without a GPU is the drop-in contract itself: the rebinding leaves parameters and state_dict keys
alone, strict=False hands CPU calls back to the reference's own methods bit for bit, strict=True refuses them loudly (no
silent CPU path in the product), and unsupported objects are rejected.  The CUDA side of the same engines is covered by
tests/test_models_gpu.py through the host mirrors (the reference package cannot travel to the GPU box)."""
import os

import numpy as np
import pytest
import torch

from oracle import _reference_shim as shim
from oracle import seeded_init as si

from conftest import GOLDEN

needs_reference = pytest.mark.skipif(not shim.available(), reason="reference tree not present")


def _gwcnet():
    cfg = shim.load_cfg("cfgs/gwcnet/gwcnet_sceneflow.yaml").MODEL
    m = shim.load("stereo.modeling.models.gwcnet.gwcnet").GwcNet(cfg).eval()
    m.load_state_dict(si.seeded_state_dict(m.state_dict(), seed=1, scale=si.GWCNET_SCALE))
    return m


def _inputs(h, w, seed):
    g = torch.Generator().manual_seed(seed)
    return {"left": torch.randn(1, 3, h, w, generator=g), "right": torch.randn(1, 3, h, w, generator=g)}


@needs_reference
def test_patch_gwcnet_contract():
    from openstereo_b200.patch import patch
    m = _gwcnet()
    keys = list(m.state_dict().keys())
    x = _inputs(64, 128, 3)
    with torch.no_grad():
        want = m(dict(x))["disp_pred"]
        assert patch(m, strict=False) is m and m._osb_patched
        assert patch(m, strict=False) is m                              # idempotent
        assert list(m.state_dict().keys()) == keys                      # checkpoints / cfgs untouched
        assert torch.equal(m(dict(x))["disp_pred"], want)               # CPU call delegated to the reference's own methods
        strict = patch(_gwcnet())
        with pytest.raises(RuntimeError, match="CUDA inference only"):
            strict(dict(x))
        # the volume builders keep the reference's bound-method signature and refuse CPU tensors (no silent fallback)
        with pytest.raises((RuntimeError, ValueError, AssertionError)):
            strict.CostProcessor.build_gwc_volume(torch.randn(1, 40, 4, 8), torch.randn(1, 40, 4, 8))


@needs_reference
def test_patch_psmnet_contract():
    from openstereo_b200.patch import patch
    cfg = shim.load_cfg("cfgs/psmnet/psmnet_sceneflow.yaml").MODEL
    m = shim.load("stereo.modeling.models.psmnet.psmnet").PSMNet(cfg).eval()
    m.load_state_dict(si.seeded_state_dict(m.state_dict(), seed=1, scale=si.PSMNET_SCALE, keep=si.PSMNET_KEEP))
    keys = list(m.state_dict().keys())
    x = _inputs(256, 256, 4)
    with torch.no_grad():
        want = m(dict(x))["disp_pred"]
        patch(m, strict=False)
        assert list(m.state_dict().keys()) == keys
        assert torch.equal(m(dict(x))["disp_pred"], want)


def test_patch_rejects_unknown():
    from openstereo_b200.patch import patch
    with pytest.raises(TypeError):
        patch("not a module")
    with pytest.raises(NotImplementedError, match="no hot-path drop-in"):
        patch(torch.nn.Linear(2, 2))


@needs_reference
def test_patch_strict_false_keeps_autograd():
    """ADVICE r1: strict=False must hand every call autograd is recording back to the reference's own code -- gradients have to
    reach the Backbone through the volume builders (the kernels have no backward and detach their inputs)."""
    from openstereo_b200.patch import patch
    m = patch(_gwcnet(), strict=False)
    x = _inputs(64, 128, 5)
    out = m(dict(x))["disp_pred"]
    assert out.requires_grad
    out.mean().backward()
    grads = [p.grad for n, p in m.named_parameters() if n.startswith("Backbone.")]
    assert all(g is not None for g in grads) and any(g.abs().sum() > 0 for g in grads)
    cfg = shim.load_cfg("cfgs/psmnet/psmnet_sceneflow.yaml").MODEL
    p = shim.load("stereo.modeling.models.psmnet.psmnet").PSMNet(cfg).eval()
    p.load_state_dict(si.seeded_state_dict(p.state_dict(), seed=1, scale=si.PSMNET_SCALE, keep=si.PSMNET_KEEP))
    patch(p, strict=False)
    out = p(dict(_inputs(256, 256, 6)))["disp_pred"]
    out.mean().backward()
    assert any(q.grad is not None and q.grad.abs().sum() > 0 for n, q in p.named_parameters() if n.startswith("Backbone."))


def test_stereobase_rebinding_is_per_instance():
    """The StereoBase drop-in must not rebind the reference module's globals (every other instance would change behaviour):
    patched instances get private method copies with their own globals.  The names the reference's StereoBase.forward and
    upsample_disp reach as module globals are stored in tests/golden/stereobase_globals.npz."""
    from openstereo_b200 import patch as P
    ns = {}
    exec("def helper(x):\n    return x + 1\n\nclass Net:\n    def forward(self, x):\n        return helper(x)\n"
         "    def other(self, x):\n        return x * 2\n", ns)
    a, b = ns["Net"](), ns["Net"]()
    P._rebind_methods(a, {"helper": lambda x: x + 100})
    assert a.forward(1) == 101 and b.forward(1) == 2 and ns["helper"](1) == 2       # module namespace and class untouched
    assert "other" not in vars(a)                                                    # only methods that use the name are copied
    with np.load(os.path.join(GOLDEN, "stereobase_globals.npz")) as g:
        names = set(g["names"].tolist())
    assert {"build_gwc_volume", "build_concat_volume", "disparity_regression", "CombinedGeoEncodingVolume", "context_upsample"} <= names

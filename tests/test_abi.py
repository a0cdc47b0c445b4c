"""CPU-side checks of the boundary: the C-ABI library loads and exports every symbol the
header declares; host-side module logic (constructors, state_dict schema, loud failure)."""
import ctypes
import importlib
import json
import os
import re
import sys

import numpy as np
import pytest
import torch

import smaat_unet_b200 as S
from oracle.cases import CASES, case_schema

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _header_symbols():
    src = open(os.path.join(ROOT, "include", "smaat_b200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(smaat_[a-z0-9_]+)\s*\(", src)))


def test_library_exports_every_declared_symbol():
    lib = ctypes.CDLL(S._lib.LIB_PATH)
    syms = _header_symbols()
    assert len(syms) >= 15
    for s in syms:
        assert hasattr(lib, s), f"{s} declared in include/smaat_b200.h but not exported"


def test_binding_table_matches_header():
    assert _header_symbols() == S._lib.EXPORTED


def test_abi_version_and_error_string():
    lib = S._lib.load()
    assert lib.smaat_abi_version() == 1
    # argument validation happens on the host before any CUDA call: usable without a GPU
    rc = lib.smaat_maxpool2_fwd(None, None, 1, 4, 4, None)
    assert rc == -1 and b"maxpool2" in lib.smaat_last_error()
    rc = lib.smaat_cbam_gate_fwd(1, 1, None, 1, None, 1, 8, 8, 5, None)
    assert rc == -1 and b"kernel size must be 3 or 7" in lib.smaat_last_error()


@pytest.mark.parametrize("args", [(12, 1, 2, 16), (3, 21, 1, 8)])
def test_model_state_dict_schema_matches_reference_schema(args):
    n_ch, n_cls, k, r = args
    from oracle.cases import smaat_unet_schema
    m = S.SmaAt_UNet(n_ch, n_cls, kernels_per_layer=k, reduction_ratio=r)
    sd = m.state_dict()
    schema = smaat_unet_schema(n_ch, n_cls, k, r)
    assert set(sd) == set(schema)
    for key, shape in schema.items():
        assert tuple(sd[key].shape) == tuple(shape), key


def test_block_schemas_match():
    for name, c in CASES.items():
        schema = case_schema(c)
        kind = c["kind"]
        if kind == "dsconv":
            m = S.DepthwiseSeparableConv(c["cin"], c["cout"], 3, padding=1, kernels_per_layer=c["k"])
        elif kind == "doubleconv":
            m = S.DoubleConvDS(c["cin"], c["cout"], c["mid"], kernels_per_layer=c["k"])
        elif kind == "down":
            m = S.DownDS(c["cin"], c["cout"], kernels_per_layer=c["k"])
        elif kind == "up":
            m = S.UpDS(c["cin"], c["cout"], c.get("bilinear", True), kernels_per_layer=c["k"])
        elif kind == "cbam":
            m = S.CBAM(c["c"], reduction_ratio=c["r"], kernel_size=c["ks"])
        elif kind == "outconv":
            m = S.OutConv(c["cin"], c["cout"])
        else:
            continue
        got = {"m." + k: tuple(v.shape) for k, v in m.state_dict().items()}
        assert got == {k: tuple(v) for k, v in schema.items()}, name


def test_no_cpu_fallback_fails_loudly():
    m = S.SmaAt_UNet(12, 1).eval()
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        m(torch.zeros(1, 12, 32, 32))
    with pytest.raises(RuntimeError, match="no CPU fallback"), torch.no_grad():      # the ConvTranspose2d branch too
        S.UpDS(8, 4, bilinear=False).eval()(torch.zeros(1, 8, 4, 4), torch.zeros(1, 4, 8, 8))


def test_product_package_never_imports_oracle():
    pkg = os.path.join(ROOT, "smaat_unet_b200")
    for fn in os.listdir(pkg):
        if fn.endswith(".py"):
            src = open(os.path.join(pkg, fn)).read()
            assert "oracle" not in src.replace("# oracle", ""), f"{fn} references the oracle"


# One module of the stand-in `models` package.  It binds the same nn.Module class names as the reference module of that
# name; its model classes make the reference constructors' block calls, looking each name up when the constructor runs.
_STANDIN_MODULE = '''\
from torch import nn

_LAYOUT = {layout!r}


class _NotRebound(nn.Module):
    def __init__(self, *args, **kwargs):
        raise AssertionError(type(self).__name__ + " was built but patch_reference() did not rebind it")


for _n in _LAYOUT["binds"]:
    globals()[_n] = type(_n, (_NotRebound,), {{}})


def _model_class(name, calls):
    def __init__(self):
        nn.Module.__init__(self)
        for attr, block, args, kwargs in calls:
            setattr(self, attr, globals()[block](*args, **kwargs))
    return type(name, (nn.Module,), {{"__init__": __init__}})


for _n, _m in _LAYOUT["models"].items():
    globals()[_n] = _model_class(_n, _m["calls"])
'''


def _drop_models_package():
    for name in [m for m in sys.modules if m == "models" or m.startswith("models.")]:
        del sys.modules[name]


@pytest.fixture
def reference_layout(tmp_path, monkeypatch):
    """A stand-in for the reference checkout's `models` package, written from tests/golden/patch_layout.json (recorded from
    the unmodified reference by oracle/make_golden_patch.py).  Yields (root to pass to patch_reference, the layout)."""
    with open(os.path.join(ROOT, "tests", "golden", "patch_layout.json")) as f:
        layout = json.load(f)
    pkg = tmp_path / "models"
    pkg.mkdir()
    (pkg / "__init__.py").write_text("")
    for modname, entry in layout["modules"].items():
        (pkg / (modname.split(".", 1)[1] + ".py")).write_text(_STANDIN_MODULE.format(layout=entry))
    monkeypatch.setattr(sys, "path", list(sys.path))
    _drop_models_package()
    importlib.invalidate_caches()
    yield str(tmp_path), layout
    _drop_models_package()


def test_patch_reference_rebinds_names(reference_layout):
    root, layout = reference_layout
    done = S.patch_reference(root)
    assert {k: sorted(v) for k, v in done.items()} == layout["patched"]
    import models.SmaAt_UNet as msu
    m = msu.SmaAt_UNet()                                  # the reference's SmaAt_UNet(12, 1)
    assert type(m.inc) is S.DoubleConvDS and type(m.cbam3) is S.CBAM and type(m.up2) is S.UpDS and type(m.outc) is S.OutConv
    assert len(m.state_dict()) == 214


def test_patch_reference_reaches_the_lightning_wrappers(reference_layout):
    """The Lightning wrapper classes (models/unet_precip_regression_lightning.py:86-208) import the block classes by name;
    after patch_reference() their UNCHANGED constructors build B200 blocks and keep the reference's state_dict schema."""
    from oracle.cases import smaat_unet_schema
    root, layout = reference_layout
    done = S.patch_reference(root, strict=True)
    assert "models.unet_precip_regression_lightning" in done
    import models.unet_precip_regression_lightning as L
    for cls, n_cbams in (("UNetDSAttention", 5), ("UNetDSAttention4CBAMs", 4), ("UNetDS", 0)):
        m = getattr(L, cls)()                             # built with hparams(n_channels=12, n_classes=1, kernels_per_layer=2)
        assert type(m.inc) is S.DoubleConvDS and type(m.down4) is S.DownDS and type(m.up1) is S.UpDS and type(m.outc) is S.OutConv
        if n_cbams:
            assert type(m.cbam1) is S.CBAM
        sd = m.state_dict()
        schema = smaat_unet_schema(12, 1, 2, n_cbams=n_cbams)
        assert set(sd) == set(schema)
        assert all(tuple(sd[k].shape) == tuple(schema[k]) for k in schema)

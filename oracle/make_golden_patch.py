"""Generate tests/golden/patch_layout.json from the UNMODIFIED reference -- TEST INFRASTRUCTURE ONLY.

    python -m oracle.make_golden_patch /path/to/SmaAt-UNet

patch_reference() works because the reference's modules bind the block classes by name at module scope and its model
constructors look those names up when they run.  For every module patch_reference() targets this records

* ``binds``: the nn.Module classes the module binds at module scope (defined there or imported by name);
* ``models``: for the model classes the tests build (SmaAt_UNet(12, 1) and the Lightning wrappers made of DS blocks),
  every block constructor call, in order: attribute, class name, positional and keyword arguments.  The calls are
  captured by rebinding the imported block names to recorders and running the reference constructors unmodified;

and ``patched``: what patch_reference() rebinds in the real reference.  tests/test_abi.py rebuilds a stand-in package
with this layout, so the patch tests run where the reference checkout does not exist.
"""
from __future__ import annotations

import inspect
import json
import os
import sys

import torch

OUT =os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden", "patch_layout.json")

LIT = ("UNetDSAttention", "UNetDSAttention4CBAMs", "UNetDS")


class Call(torch.nn.Module):
    """Stands in for an imported block class: remembers how the constructor called it."""

    def __init__(self, *args, **kwargs):
        super().__init__()
        self.call = [type(self).__name__, list(args), kwargs]


def main():
    if len(sys.argv) != 2:
        raise SystemExit("usage: python -m oracle.make_golden_patch <checkout of the reference SmaAt-UNet>")
    from oracle import ref_stubs
    import smaat_unet_b200 as S
    from smaat_unet_b200.patch import _TARGETS
    ref_stubs.install()
    patched = S.patch_reference(sys.argv[1], strict=True)
    hp = ref_stubs.hparams(12, 1, 2)
    builds = {"models.SmaAt_UNet": {"SmaAt_UNet": ("SmaAt_UNet(12, 1)", lambda cls: cls(12, 1))},
              "models.unet_precip_regression_lightning": {
                  c: (f"{c}(hparams=ref_stubs.hparams(12, 1, 2))", lambda cls: cls(hparams=hp)) for c in LIT}}
    modules = {}
    for modname in _TARGETS:
        mod = sys.modules[modname]
        binds = sorted(n for n, v in vars(mod).items() if inspect.isclass(v) and issubclass(v, torch.nn.Module))
        for n in binds:                      # imported names only: the classes defined here are the ones being built
            if vars(mod)[n].__module__ != modname:
                setattr(mod, n, type(n, (Call,), {}))
        models = {}
        for cls, (built_as, make) in builds.get(modname, {}).items():
            m = make(getattr(mod, cls))
            kids = list(m.named_children())
            assert all(isinstance(c, Call) or not c.state_dict() for _, c in kids), (cls, "a child with state is not a block")
            models[cls] = {"built_as": built_as, "calls": [[a] + c.call for a, c in kids if isinstance(c, Call)]}
        modules[modname] = {"binds": binds, "models": models}
    out = {"reference": "HansBambel/SmaAt-UNet", "torch": torch.__version__, "modules": modules,
           "patched": {k: sorted(v) for k, v in patched.items()}}
    with open(OUT, "w") as f:
        json.dump(out, f, indent=1, sort_keys=True)
    print("wrote", OUT, {k: (len(v["binds"]), {c: len(d["calls"]) for c, d in v["models"].items()}) for k, v in modules.items()})


if __name__ == "__main__":
    main()

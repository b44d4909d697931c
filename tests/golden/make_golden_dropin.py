#!/usr/bin/env python
"""Golden record of the drop-in check (tests/test_host.py::test_unchanged_reference_model_imports_our_operators),
taken from an UNCHANGED reference ``pointmvsnet/model.py`` after ``install_as_pointmvsnet(<checkout>)`` and from its
pretrained checkpoint, which must load strictly into that model (nothing copied, only names and shapes stored):

    python tests/golden/make_golden_dropin.py <PointMVSNet checkout>

writes dropin_model.json:
  imports     name in model.py's namespace that resolved to this package -> our object ("module:qualname") and the
              reference modules that hand it out
  submodules  PointMVSNet submodule built from one of our classes -> class ("module:qualname") and the shapes of its
              checkpoint entries (keys relative to the submodule)
  reference_modules  the checkout's modules that were loaded -> "package" or "module" (names only)
"""
import json
import os
import sys

import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))


def qualified(obj):
    return "%s:%s" % (obj.__module__, obj.__qualname__)


def ours(obj):
    return isinstance(getattr(obj, "__module__", None), str) and obj.__module__.startswith("pointmvsnet_b200")


def main(ref_root):
    import pointmvsnet_b200
    from pointmvsnet_b200.point_flow import PointFlow
    pointmvsnet_b200.install_as_pointmvsnet(ref_root)
    import pointmvsnet.model as m

    modules = {}
    for name, mod in list(sys.modules.items()):
        f = getattr(mod, "__file__", None)
        if f and os.path.abspath(f).startswith(ref_root + os.sep):
            modules[name] = "package" if hasattr(mod, "__path__") else "module"
    imports = {}
    for name, obj in sorted(vars(m).items()):
        if ours(obj) and callable(obj):
            providers = sorted(k for k, mod in sys.modules.items()
                               if k.startswith("pointmvsnet.") and k != "pointmvsnet.model" and getattr(mod, name, None) is obj)
            imports[name] = {"object": qualified(obj), "from": providers}

    net = m.PointMVSNet()
    sd = torch.load(os.path.join(ref_root, "outputs", "dtu_wde3", "model_pretrained.pth"), map_location="cpu",
                    weights_only=False)["model"]
    sd = {k[len("module."):] if k.startswith("module.") else k: v for k, v in sd.items()}
    net.load_state_dict(sd)  # strict: every checkpoint entry has its place in the model with our modules inside
    submodules = {}
    for path, mod in net.named_modules():
        if path and ours(type(mod)):
            state = {k: list(v.shape) for k, v in mod.state_dict().items()}
            assert all(list(sd[path + "." + k].shape) == s for k, s in state.items()), path
            submodules[path] = {"class": qualified(type(mod)), "state": state}
    # PointFlow runs on the reference model's own hot-path modules
    pf = PointFlow(flow_edge_conv=net.flow_edge_conv, flow_mlp=net.flow_mlp)
    assert pf.flow_mlp[1].weight is net.flow_mlp[1].weight

    out = os.path.join(HERE, "dropin_model.json")
    with open(out, "w") as f:
        json.dump({"imports": imports, "submodules": submodules, "reference_modules": modules}, f, indent=1,
                  sort_keys=True)
        f.write("\n")
    print("wrote", out, "%d imports, %d submodules" % (len(imports), len(submodules)))


if __name__ == "__main__":
    if len(sys.argv) != 2:
        sys.exit("usage: make_golden_dropin.py <PointMVSNet checkout>")
    main(os.path.abspath(sys.argv[1]))

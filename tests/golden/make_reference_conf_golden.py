"""Records, from a checkout of the reference (tijiang13/InstantAvatar@3cdfd49), what
tests/test_reference_import_surface.py checks the B200 mirror against, into tests/golden/reference_conf.json:

 * every `_target_` string of confs/{renderer,deformer,network}/*.yaml and of the top-level run configurations;
 * the tiny-cuda-nn modules the reference's models/networks/ngp.py builds (attribute, class, keyword arguments), its
   buffers and parameter sizes, captured by constructing its NeRFNGPNet on the in-repo `tinycudann` module.

Only configuration values are stored, no reference source.  CPU only:

    python tests/golden/make_reference_conf_golden.py <reference checkout>
"""
import importlib.util
import json
import os
import re
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
TOP_LEVEL = ("SNARF_NGP.yaml", "SNARF_NGP_refine.yaml", "SNARF_NGP_fitting.yaml", "demo.yaml")


def targets(path):
    return [m.group(1) for m in re.finditer(r"_target_:\s*(\S+)", open(path).read())]


def conf_targets(ref):
    found = []
    for sub in ("renderer", "deformer", "network"):
        d = os.path.join(ref, "confs", sub)
        for f in sorted(os.listdir(d)):
            found += [[f"confs/{sub}/{f}", t] for t in targets(os.path.join(d, f))]
    return found, {f: targets(os.path.join(ref, "confs", f)) for f in TOP_LEVEL}


def ngp_modules(ref):
    """construct the reference's NeRFNGPNet with the tinycudann classes wrapped to record their constructor calls"""
    import tinycudann
    from instantavatar_b200.config import Cfg
    calls = []
    originals = {n: getattr(tinycudann, n) for n in ("Network", "NetworkWithInputEncoding")}

    def recording(name, cls):
        def make(**kwargs):
            m = cls(**kwargs)
            calls.append((name, kwargs, m))
            return m
        return make

    for n, cls in originals.items():
        setattr(tinycudann, n, recording(n, cls))
    try:
        spec = importlib.util.spec_from_file_location("_ref_ngp", os.path.join(ref, "instant_avatar", "models", "networks", "ngp.py"))
        mod = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(mod)
        net = mod.NeRFNGPNet(Cfg({"center": [0, -0.3, 0], "scale": [2.5, 2.5, 2.5]}))
    finally:
        for n, cls in originals.items():
            setattr(tinycudann, n, cls)
    attr = {id(m): n for n, m in net.named_children()}
    return {"modules": [{"attr": attr[id(m)], "class": n, "kwargs": kw} for n, kw, m in calls],
            "buffers": sorted(dict(net.named_buffers())),
            "parameters": {k: v.numel() for k, v in net.named_parameters()}}


def main(ref):
    conf, top = conf_targets(ref)
    out = {"reference": "tijiang13/InstantAvatar@3cdfd49", "conf_targets": conf, "top_level_targets": top,
           "ngp": ngp_modules(ref)}
    path = os.path.join(ROOT, "tests", "golden", "reference_conf.json")
    with open(path, "w") as f:
        json.dump(out, f, indent=1)
        f.write("\n")
    print("wrote", path)


if __name__ == "__main__":
    main(sys.argv[1])

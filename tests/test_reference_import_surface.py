"""CPU: the reference's module paths resolve to the B200 mirror classes (SURVEY.md §8b).

Every `_target_` string of the reference's confs/{renderer,deformer,network}/*.yaml and of the `model` / `loss` nodes of
confs/SNARF_NGP*.yaml is resolved with importlib (no Hydra) through the `instant_avatar` alias package, the classes are
checked to be the instantavatar_b200 ones, and the classes that construct without a GPU are instantiated from the
reference's own YAML argument sets.  What the reference's files hold is recorded in tests/golden/reference_conf.json
(tests/golden/make_reference_conf_golden.py)."""
import importlib
import json
import os

import pytest

# (config file of the reference, _target_, kwargs given in that file after `${}` interpolation)
TARGETS = [
    ("confs/renderer/raymarcher_acc.yaml", "instant_avatar.renderers.raymarcher_acc.Raymarcher", {"MAX_SAMPLES": 256, "MAX_BATCH_SIZE": 291600}),
    ("confs/deformer/fast_snarf.yaml", "instant_avatar.deformers.snarf_deformer.SNARFDeformer", None),
    ("confs/deformer/fast_snarf_debug.yaml", "instant_avatar.deformers.snarf_deformer.SNARFDeformer", None),
    ("confs/deformer/smpl.yaml", "instant_avatar.deformers.smpl_deformer.SMPLDeformer", None),
    ("confs/network/ngp.yaml", "instant_avatar.models.networks.ngp.NeRFNGPNet",
     {"opt": {"use_viewdir": False, "cond_dim": 0, "center": [0, -0.3, 0], "scale": [2.5, 2.5, 2.5]}}),
    ("confs/SNARF_NGP.yaml", "instant_avatar.models.DNeRF.DNeRFModel", None),
    ("confs/SNARF_NGP.yaml", "instant_avatar.utils.loss.NeRFLoss", {"opt": {"w_rgb": 1.0, "w_alpha": 0.1, "w_reg": 0.1}}),
    ("confs/SNARF_NGP_refine.yaml", "instant_avatar.utils.loss.NGPLoss", None),
]
MIRROR = {
    "instant_avatar.renderers.raymarcher_acc.Raymarcher": "instantavatar_b200.renderers.raymarcher_acc.Raymarcher",
    "instant_avatar.deformers.snarf_deformer.SNARFDeformer": "instantavatar_b200.deformers.snarf_deformer.SNARFDeformer",
    "instant_avatar.deformers.smpl_deformer.SMPLDeformer": "instantavatar_b200.deformers.smpl_deformer.SMPLDeformer",
    "instant_avatar.models.networks.ngp.NeRFNGPNet": "instantavatar_b200.models.networks.ngp.NeRFNGPNet",
    "instant_avatar.models.DNeRF.DNeRFModel": "instantavatar_b200.models.dnerf.DNeRFModel",
    "instant_avatar.utils.loss.NeRFLoss": "instantavatar_b200.utils_loss.NeRFLoss",
    "instant_avatar.utils.loss.NGPLoss": "instantavatar_b200.utils_loss.NGPLoss",
}


def _resolve(path):
    mod, _, name = path.rpartition(".")
    return getattr(importlib.import_module(mod), name)


@pytest.mark.parametrize("conf,target,kwargs", TARGETS)
def test_target_resolves_to_the_mirror(conf, target, kwargs):
    from instantavatar_b200.config import resolve
    cls = resolve(target)
    assert cls is _resolve(MIRROR[target]), (target, cls)


@pytest.fixture(scope="module")
def reference_conf(golden_dir):
    with open(os.path.join(golden_dir, "reference_conf.json")) as f:
        return json.load(f)


def test_targets_are_the_reference_files_targets(reference_conf):
    """the committed list above equals what the reference's YAML files hold"""
    found = {tuple(ct) for ct in reference_conf["conf_targets"]}
    committed = {(c, t) for c, t, _ in TARGETS if c.split("/")[1] in ("renderer", "deformer", "network")}
    assert found == committed, found ^ committed
    assert set(reference_conf["top_level_targets"]) == {"SNARF_NGP.yaml", "SNARF_NGP_refine.yaml", "SNARF_NGP_fitting.yaml", "demo.yaml"}
    for f, targets in reference_conf["top_level_targets"].items():
        assert targets, f
        for t in targets:
            assert t in MIRROR, (f, t)


def test_instantiate_cpu_constructible_targets():
    """hydra.utils.instantiate(cfg, _recursive_=False) semantics on the YAML argument sets that need no GPU"""
    import torch
    from instantavatar_b200.config import instantiate
    net = instantiate({"_target_": "instant_avatar.models.networks.ngp.NeRFNGPNet",
                       "opt": {"use_viewdir": False, "cond_dim": 0, "center": [0, -0.3, 0], "scale": [2.5, 2.5, 2.5]}})
    assert torch.allclose(net.center, torch.tensor([0.0, -0.3, 0.0])) and torch.allclose(net.scale, torch.tensor([2.5, 2.5, 2.5]))
    # the reference's optimiser grouping keys on these names (DNeRF.py:34-45) and tcnn's flat fp32 parameter sizes
    names = dict(net.named_parameters())
    assert set(names) == {"encoder.params", "color_net.params"}
    assert names["encoder.params"].numel() == 3072 + 2 * 6513496 and names["color_net.params"].numel() == 6144
    loss = instantiate({"_target_": "instant_avatar.utils.loss.NeRFLoss", "opt": {"w_rgb": 1.0, "w_alpha": 0.1, "w_reg": 0.1}})
    assert (loss.w_rgb, loss.w_alpha, loss.w_reg) == (1.0, 0.1, 0.1)
    r = instantiate({"_target_": "instant_avatar.renderers.raymarcher_acc.Raymarcher", "MAX_SAMPLES": 256, "MAX_BATCH_SIZE": 291600},
                    smpl_init=False, device="cpu")
    r.initialize(3)
    assert r.MAX_BATCH_SIZE == 291600 and r.density_grid_train.grid_size == 64
    with pytest.raises(NotImplementedError):  # demo.yaml's smpl_init needs kaolin: loud, not silently different
        instantiate({"_target_": "instant_avatar.renderers.raymarcher_acc.Raymarcher", "MAX_SAMPLES": 256, "MAX_BATCH_SIZE": 291600},
                    smpl_init=True, device="cpu")


def test_reference_import_statements():
    """the `from instant_avatar... import ...` lines of the reference's own modules and scripts"""
    from instant_avatar.deformers.fast_snarf.deformer_torch import ForwardDeformer  # snarf_deformer.py:2
    from instant_avatar.models.structures.body_model_param import SMPLParamEmbedding  # DNeRF.py:1
    from instant_avatar.models.structures.density_grid import DensityGrid  # raymarcher_acc.py:4
    from instant_avatar.models.structures.utils import Rays  # DNeRF.py:3
    import instantavatar_b200.models.dnerf as m
    assert Rays is m.Rays and ForwardDeformer.__module__.startswith("instantavatar_b200")
    assert DensityGrid.__module__.startswith("instantavatar_b200") and SMPLParamEmbedding.__module__.startswith("instantavatar_b200")


def test_reference_ngp_file_runs_on_the_tinycudann_shim(reference_conf):
    """the tinycudann modules the reference's OWN models/networks/ngp.py builds (class and keyword arguments recorded from
    that file) construct on the in-repo `tinycudann` module: same sub-module names and flat parameter sizes (CPU:
    construction only; the forward is a GPU test)"""
    import torch
    import tinycudann
    assert "ia_b200" in tinycudann.__version__
    ngp = reference_conf["ngp"]
    net = torch.nn.Module()
    for m in ngp["modules"]:
        setattr(net, m["attr"], getattr(tinycudann, m["class"])(**m["kwargs"]))
    sizes = {k: v.numel() for k, v in net.named_parameters()}
    assert sizes == ngp["parameters"] == {"encoder.params": 3072 + 2 * 6513496, "color_net.params": 6144}
    assert ngp["buffers"] == ["center", "scale"]

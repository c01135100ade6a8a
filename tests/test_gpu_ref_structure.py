"""GPU: end-to-end comparison with the REFERENCE'S OWN KERNELS.  tests/golden/ref_structure_golden.npz holds what the
reference's raymarcher, fuse_broyden, filter and precompute extensions, driven by the reference's host loop
(oracle/ref_structure.py; only tiny-cuda-nn is replaced, by ia_ngp_forward), computed for this scene on a B200
(tests/golden/make_ref_structure_golden.py).  The fused kernel must reproduce that pipeline's image."""
import hashlib
import os

import numpy as np
import pytest

from oracle import scene as oscene
from oracle import testing as scene_util

pytestmark = pytest.mark.gpu


def test_fused_render_matches_reference_kernels_pipeline(golden_dir):
    import torch
    from instantavatar_b200 import ops
    g = np.load(os.path.join(golden_dir, "ref_structure_golden.npz"))
    sc = scene_util.oracle_scene(0)
    scene, extra = scene_util.upload(sc)
    fr = sc["frame"]
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()
    # the reference's precompute kernel vs ours (voxel-major, padded): bit-equal
    vJ = scene.field[..., :12].contiguous().cpu().numpy()
    assert vJ.shape == tuple(g["voxel_J_shape"])
    assert np.array_equal(vJ.reshape(-1)[g["voxel_J_sample_index"]], g["voxel_J_sample"])
    assert hashlib.sha256(vJ.tobytes()).hexdigest() == str(g["voxel_J_sha256"])
    # occupancy grid vs the reference structure's, with the same jitter
    field_ref = np.unpackbits(g["density_field_bits"])[:64 ** 3].reshape(64, 64, 64).astype(bool)
    jit = t(sc["occ_jitter"])
    dens = ops.occupancy_query(scene, jit, t(fr["bbox_deformed"].reshape(6)))
    field, bits = ops.occupancy_build(dens)
    assert (field.cpu().numpy() != field_ref).mean() < 5e-4
    # render a 128x192 crop with BOTH grids equal to the reference's
    o, d, near, far = oscene.camera_rays(fr, 512, 512)
    ys, xs = np.arange(160, 352), np.arange(192, 320)
    idx = (ys[:, None] * 512 + xs[None]).ravel()
    assert np.array_equal(g["pixel_index"], idx)
    import dataclasses
    scene2 = dataclasses.replace(scene, occ_bits=ops.pack_occupancy(t(field_ref)), occ_aabb=t(g["aabb"]))
    out = ops.render_fwd(scene2, t(o[idx]), t(d[idx]), t(near[idx]), t(far[idx]), None, 128)
    torch.cuda.synchronize()
    ref = {"rgb": t(g["rgb"]), "alpha": t(g["alpha"])}
    e_rgb = (out["rgb"] - ref["rgb"]).abs().max(-1).values
    e_a = (out["alpha"] - ref["alpha"]).abs()
    assert (ref["alpha"] > 0.5).sum().item() > 3000
    # the reference's Broyden differs from the oracle's in the last bits (nvcc fma contraction), which moves roots by
    # <= 1e-5 and, rarely, flips an fp16 rounding inside the network: allow the north_star tolerance on all but a few rays
    assert (e_rgb > 1e-3).float().mean().item() < 2e-3, ((e_rgb > 1e-3).sum().item(), e_rgb.max().item())
    assert (e_a > 1e-3).float().mean().item() < 2e-3
    assert e_rgb.max().item() < 5e-2

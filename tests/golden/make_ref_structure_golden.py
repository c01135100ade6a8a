"""Runs the reference's structure on a B200 -- its own raymarcher, fuse_broyden, filter and precompute extensions (built
into oracle/_ref by oracle/build_ref.py) driven by its host loop (oracle/ref_structure.py; tiny-cuda-nn replaced by
ia_ngp_forward) -- on the scene of tests/test_gpu_ref_structure.py, and stores what that test compares the product with:

 * the skinning-transform field of the reference's precompute kernel, voxel-major [32,128,128,12] (25 MB): its SHA-256
   and a seeded sample of 8192 entries;
 * the occupancy field of the reference's DensityGrid.initialize on the scene's jitter (bit-packed) and its AABB;
 * the reference pipeline's render_test of a 128x192 crop of the demo camera with that grid (rgb, alpha).

Needs a GPU and oracle/_ref:   python tests/golden/make_ref_structure_golden.py [OUT.npz]
(default OUT: tests/golden/ref_structure_golden.npz)."""
import hashlib
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from instantavatar_b200 import ops  # noqa: E402
from oracle import ref_structure, scene as oscene, testing as scene_util  # noqa: E402

CROP = (np.arange(160, 352)[:, None] * 512 + np.arange(192, 320)[None]).ravel()  # rows 160..351, columns 192..319


def main(path):
    sc = scene_util.oracle_scene(0)
    scene, _ = scene_util.upload(sc)
    subj, fr = sc["subj"], sc["frame"]
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()
    rs = ref_structure.RefStructure(t(subj.lbs_voxel)[None], t(subj.offset_kernel), t(subj.scale_kernel),
                                    lambda x: ops.ngp_forward(scene, x))
    rs.precompute(t(fr["tfs"])[None])
    vJ = rs.voxel_J[0].permute(1, 2, 3, 0).contiguous().cpu().numpy()
    sample = np.sort(np.random.default_rng(0).choice(vJ.size, 8192, replace=False))
    field = rs.density_grid_initialize(t(sc["occ_jitter"]))
    o, d, near, far = oscene.camera_rays(fr, 512, 512)
    ref = rs.render_test(t(o[CROP]), t(d[CROP]), t(near[CROP]), t(far[CROP]))
    torch.cuda.synchronize()
    out = {"voxel_J_shape": np.array(vJ.shape), "voxel_J_sha256": np.array(hashlib.sha256(vJ.tobytes()).hexdigest()),
           "voxel_J_sample_index": sample, "voxel_J_sample": vJ.reshape(-1)[sample],
           "density_field_bits": np.packbits(field.cpu().numpy().reshape(-1)),
           "aabb": torch.cat(rs.aabb).cpu().numpy(), "pixel_index": CROP,
           "rgb": ref["rgb"].cpu().numpy(), "alpha": ref["alpha"].cpu().numpy()}
    np.savez_compressed(path, **out)
    print("saved", path, {k: v.shape for k, v in out.items()})


if __name__ == "__main__":
    main(sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "tests", "golden", "ref_structure_golden.npz"))

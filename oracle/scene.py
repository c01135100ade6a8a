"""ORACLE-side assembly of the synthetic benchmark scene (SURVEY.md §8d) from instantavatar_b200.synthetic
data: subject -> frame -> network -> occupancy grid -> rays.  Test infrastructure."""
from __future__ import annotations

import os
import tempfile

import numpy as np

from instantavatar_b200 import synthetic
from . import frame as oframe
from . import render as orender

f32 = np.float32
# per user: a cache directory another account created in the shared temporary directory would not be writable
_CACHE_DIR = os.environ.get("IA_ORACLE_CACHE", os.path.join(tempfile.gettempdir(), f"ia_oracle_cache-{os.getuid()}"))


def build_subject(resolution=128, track="male-3-casual", cache=True):
    if track == "aist_demo":  # animate.py:100: the animation is rendered with the training subject's shape
        track = "male-3-casual"
    pose0 = synthetic.load_pose(synthetic.track_frames(track)[0], track)
    data = synthetic.smpl_dict_cached(0)
    lbs = None
    path = os.path.join(_CACHE_DIR, f"lbs_voxel_{track}_{resolution}.npy")
    if cache and os.path.exists(path):
        lbs = np.load(path)
    subj = oframe.SubjectOracle(data, pose0["betas"], resolution, lbs_voxel=lbs)
    if cache and lbs is None:
        os.makedirs(_CACHE_DIR, exist_ok=True)
        np.save(path, subj.lbs_voxel)
    return subj


def build_net(subj, seed=1337, sigma_in=100.0, emulate=True):
    c = ((subj.bbox[0] + subj.bbox[1]) / f32(2)).astype(f32)
    s = (subj.bbox[1] - subj.bbox[0]).astype(f32)
    enc, col = synthetic.analytic_avatar_params(subj.joints_cano, c.astype(np.float64), s.astype(np.float64), seed, sigma_in)
    return orender.Net(enc, col, c, s, emulate)


def camera_rays(fr, H=512, W=512, sub=None):
    """demo camera rays transformed to the SMPL root frame; `sub` = (y0, y1, x0, x1) crop."""
    o, d = synthetic.demo_camera_rays(H, W)
    if sub is not None:
        y0, y1, x0, x1 = sub
        o = o.reshape(H, W, 3)[y0:y1, x0:x1].reshape(-1, 3)
        d = d.reshape(H, W, 3)[y0:y1, x0:x1].reshape(-1, 3)
    return oframe.transform_rays_w2s(o, d, fr["w2s"])


def build_occupancy(subj, fr, net, seed=42, iters=5, G=64):
    rng = np.random.default_rng(seed)
    jit = rng.random((iters, G, G, G, 3), dtype=f32)
    aabb = fr["bbox_deformed"]
    field, density = orender.density_grid_initialize(lambda p: orender.deform_query(p, fr, subj, net, True), aabb, jit, G)
    return field, density, jit

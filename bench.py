#!/usr/bin/env python
"""bench.py -- rays/s of a 512x512 avatar render (BASELINE.json metric) on N B200s.

A "step" is one complete frame of the reference's `render_image_fast` (DNeRF.py:72-97) on the synthetic
PeopleSnapshot-shaped scene (SURVEY.md §8d): SMPL forward -> bone transforms -> skinning-transform field ->
5-pass occupancy-grid initialisation (+ connected component) -> 262 144 rays through the fused march / Broyden /
hash-grid / MLP / compositing kernel.

  value : rays/s with the frame's inputs (rays, SMPL pose) resident in HBM.
  e2e   : the same frame through the public API with HOST buffers: pinned rays + pose -> device, render, RGBA -> host.
  --impl reference : the CPU oracle (C port of the reference's kernels + numpy host loop, all host threads) on the same
                     frame -- the reference's own GPU path needs tiny-cuda-nn, which cannot be built (BASELINE.md §2).
N > 1: one process per GPU (torchrun), each rank renders whole frames of different poses; no data-path collective
("scaling": "weak").
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

H = W = 512
N_RAYS = H * W
FRAMES = [0, 20, 57, 100]
METRIC = "rays/sec at 512x512 render"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--rays-per-warp", type=int, default=0)
    ap.add_argument("--no-graph", action="store_true", help="eager launches instead of CUDA-graph replay")
    ap.add_argument("--train-rays-per-warp", type=int, default=0)
    ap.add_argument("--render-warps", type=int, default=0, help="warps per CTA of the fused renderer (12)")
    ap.add_argument("--query-warps", type=int, default=0, help="warps per CTA of the point-query kernel (12 / 16 / 20)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the frame of the last timed step (rgb, depth, alpha, counter of rank 0) as DIR/<name>.npy, float32")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs records the GPU frame (--impl ours)")
    return args


def dump_outputs(out_dir: str, arrays: dict) -> None:
    """--dump-outputs: one float32 DIR/<name>.npy per array, so that two builds can be compared output for output"""
    arrays = {k: np.asarray(v, dtype=np.float32) for k, v in arrays.items()}
    assert sum(a.nbytes for a in arrays.values()) <= 64 << 20, "outputs above 64 MB: store a seeded sample instead"
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), a)


# ------------------------------------------------------------------------------------------------
# clocks sampler (B200_PROFILING.md recipe)
# ------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = "index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index: int):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                                          "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")] + [time.monotonic()])

    def count_between(self, t0, t1):
        return sum(1 for r in self.rows if len(r) >= 9 and t0 <= r[-1] <= t1)

    def stop(self, t0=None, t1=None) -> dict:
        """summary of the samples received in [t0, t1] (the timed region); all samples if no window is given"""
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        if t0 is not None:
            self.rows = [r for r in self.rows if len(r) >= 9 and t0 <= r[-1] <= t1]
        sm = [float(r[1]) for r in self.rows if len(r) >= 8 and r[1].replace(".", "").isdigit()]
        mx = [float(r[2]) for r in self.rows if len(r) >= 8 and r[2].replace(".", "").isdigit()]
        reasons = set()
        for r in self.rows:
            if len(r) >= 8:
                for name, v in zip(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"], r[4:8]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------------
# scene
# ------------------------------------------------------------------------------------------------
def host_batch(frame: int):
    from instantavatar_b200 import synthetic
    pose = synthetic.load_pose(frame)
    o, d = synthetic.demo_camera_rays(H, W)
    dist = np.linalg.norm(pose["transl"], axis=-1).astype(np.float32)
    near = np.full((1, N_RAYS), dist[0] - 1, np.float32)  # peoplesnapshot dataset convention; overridden by w2s
    far = np.full((1, N_RAYS), dist[0] + 1, np.float32)
    return {"rays_o": o[None], "rays_d": d[None], "near": near, "far": far, **pose}


def build_model(device, frame: int):
    import torch
    from instantavatar_b200 import synthetic
    from instantavatar_b200.models.dnerf import DNeRFModel
    model = DNeRFModel(smpl_data=synthetic.smpl_dict_cached(0), device=device).eval()
    hb = host_batch(frame)
    batch = {k: torch.from_numpy(v).to(device) for k, v in hb.items()}
    model.deformer.prepare_deformer(batch)  # subject initialisation (KNN skinning-weight voxelisation etc.), untimed
    model.net_coarse.initialize(model.deformer.bbox)
    bbox = model.deformer.bbox.cpu().numpy().astype(np.float64)
    c, s = (bbox[0] + bbox[1]) / 2, bbox[1] - bbox[0]
    enc, col = synthetic.analytic_avatar_params(model.deformer.joints_cano[0].cpu().numpy(), c, s)
    model.net_coarse.load_flat_params(torch.from_numpy(enc).to(device), torch.from_numpy(col).to(device))
    return model, hb, batch


# ------------------------------------------------------------------------------------------------
# CPU oracle frame (cpu_baseline leg and --impl reference): the only place bench.py executes oracle/
# ------------------------------------------------------------------------------------------------
class CpuFrame:
    def __init__(self, frame: int):
        from oracle import capi, scene as oscene
        from instantavatar_b200 import synthetic
        self.capi = capi
        capi.set_num_threads(os.cpu_count() or 1)  # torchrun exports OMP_NUM_THREADS=1; the CPU arm uses every host thread
        self.subj = oscene.build_subject()
        self.net = oscene.build_net(self.subj)
        self.pose = synthetic.load_pose(frame)
        self.threads = capi.num_threads()

    def step(self):
        from oracle import render as orender, scene as oscene
        fr = self.subj.prepare_frame(self.pose)
        occ, _, _ = oscene.build_occupancy(self.subj, fr, self.net)
        o, d, near, far = oscene.camera_rays(fr, H, W)
        out = orender.render_test(o, d, near, far, occ, fr["bbox_deformed"][0], fr["bbox_deformed"][1],
                                  lambda p: orender.deform_query(p, fr, self.subj, self.net, True))
        return out


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cf = CpuFrame(FRAMES[0])
    for _ in range(min(args.warmup, 1)):
        cf.step()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        cf.step()
    dt = time.perf_counter() - t0
    v = N_RAYS * args.steps / dt
    line = {"impl": "reference", "metric": METRIC, "value": v, "unit": "rays/s", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": min(args.warmup, 1), "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": "male-3-casual-shaped synthetic frame, 512x512 rays, full render_image_fast on host cores"},
            "cpu_baseline": {"value": v, "unit": "rays/s", "cores": cf.threads, "kind": "port",
                             "sample": "complete 512x512 frame per step (prep + 5-pass occupancy init + march), C oracle with OpenMP"},
            "e2e": {"value": v, "unit": "rays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------------
def bench_frame_sharded(model, batch, device, rank, world, flush, steps=20, warmup=5):
    """BASELINE.json config 3 (one frame, rays sharded over the GPUs): latency of ONE 512x512 frame rendered cooperatively
    (strong scaling).  Two exchange paths, both measured, both checked bit-equal to the single-GPU frame:
      nccl : occupancy queries sharded + 1 MB max-all-reduce, ray tiles round-robin, RGBA all-gather (+ un-permute);
      peer : the same exchanges INSIDE the kernels over NVLink peer memory (parallel.PeerFrame: atomics into every rank's
             density grid, RGBA stores into every rank's image) -- two barriers, no collective."""
    import torch
    import torch.distributed as dist
    from instantavatar_b200 import parallel
    model.eval()
    torch.manual_seed(99)  # identical jitter on every rank
    jit = torch.rand((5, 64, 64, 64, 3), device=device)
    # every rank renders the SAME frame here: broadcast rank 0's pose
    b = {k: v.clone() for k, v in batch.items()}
    for k in ("betas", "body_pose", "global_orient", "transl"):
        dist.broadcast(b[k], 0)
    rgb, _, alpha, _ = model.render_image_fast(dict(b), (H, W), jit)
    single = torch.cat([rgb.reshape(-1, 3), alpha.reshape(-1, 1)], dim=1).clone()
    peer, peer_err = None, None
    try:
        peer = parallel.PeerFrame(H * W, device)
    except Exception as exc:  # platform without peer mapping: NCCL path only
        peer_err = f"{type(exc).__name__}: {exc}"[:200]
    ok = torch.tensor([1.0 if peer is not None else 0.0], device=device)
    dist.all_reduce(ok, op=dist.ReduceOp.MIN)
    if ok.item() == 0:
        peer = None
    res = {"scaling": "strong", "tile_rays": 2048}
    for name, pf in (("nccl", None), ("peer", peer)):
        if name == "peer" and pf is None:
            res["peer_unavailable"] = peer_err or "another rank could not map peer memory"
            continue
        graphed = None
        try:
            from instantavatar_b200.graphs import GraphedShardedFrame
            graphed = GraphedShardedFrame(model, b, (H, W), rank, world, jit, peer=pf)
        except Exception as exc:  # capture unavailable: eager launches
            if rank == 0:
                print(f"[bench] sharded-frame graph capture failed for {name} ({type(exc).__name__}: {exc}), running eagerly", file=sys.stderr)
            torch.cuda.synchronize()
        run = (lambda: graphed()) if graphed is not None else (lambda: model.render_image_sharded(b, (H, W), rank, world, jit, peer=pf))
        for _ in range(warmup):
            img = run()
        dist.barrier(); torch.cuda.synchronize()
        equal = torch.tensor([1.0 if (img is not None and torch.equal(img, single)) else 0.0], device=device)
        dist.all_reduce(equal, op=dist.ReduceOp.MIN)
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        for a, e in ev:
            flush.zero_()
            a.record(); run(); e.record()
        dist.barrier(); torch.cuda.synchronize()
        ms = torch.tensor([sum(a.elapsed_time(e) for a, e in ev) / steps], device=device, dtype=torch.float64)
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        res[name] = {"ms_per_frame": float(ms.item()), "rays_per_s": N_RAYS / (float(ms.item()) * 1e-3), "bit_equal_all_ranks": bool(equal.item() == 1.0),
                     "cuda_graph": graphed is not None}
    best = min((k for k in ("nccl", "peer") if k in res), key=lambda k: res[k]["ms_per_frame"])
    res.update({"ms_per_frame": res[best]["ms_per_frame"], "rays_per_s": res[best]["rays_per_s"], "path": best,
                "bit_equal": all(res[k]["bit_equal_all_ranks"] for k in ("nccl", "peer") if k in res)})
    return res


def bench_ref_structure(model, batch, device, iters=5):
    """The reference's own CUDA kernels (oracle/_ref, built from /root/reference) + the reference's host loop, with this
    repo's hash-grid/MLP standing in for tiny-cuda-nn, on the same frame: per-frame time of precompute +
    DensityGrid.initialize + render_test (bench infrastructure; see oracle/ref_structure.py)."""
    import torch
    try:
        from oracle import ref_structure
        if not ref_structure.available():
            return {"unavailable": "oracle/_ref not built"}
        from instantavatar_b200.models.dnerf import Rays
        dfm = model.deformer
        rs = ref_structure.RefStructure(dfm.deformer.lbs_voxel_final, dfm.deformer.offset_kernel, dfm.deformer.scale_kernel,
                                        lambda x: model.net_coarse(x))
        model.eval()
        dfm.prepare_deformer(batch)
        r = Rays(o=batch["rays_o"].clone(), d=batch["rays_d"].clone(), near=batch["near"].clone(), far=batch["far"].clone())
        dfm.transform_rays_w2s(r)
        o, d = r.o.reshape(-1, 3).contiguous(), r.d.reshape(-1, 3).contiguous()
        near, far = r.near.reshape(-1).contiguous(), r.far.reshape(-1).contiguous()
        ev = lambda: torch.cuda.Event(enable_timing=True)
        t_all, t_march = [], []
        for i in range(iters + 2):
            e0, e1, e2 = ev(), ev(), ev()
            e0.record()
            rs.precompute(dfm.tfs)
            rs.density_grid_initialize()
            e1.record()
            out = rs.render_test(o, d, near, far)
            e2.record()
            torch.cuda.synchronize()
            if i >= 2:
                t_all.append(e0.elapsed_time(e2)); t_march.append(e1.elapsed_time(e2))
        ms = float(np.median(t_all))
        return {"ms_per_frame": ms, "rays_per_s": N_RAYS / (ms * 1e-3), "ms_render_test_only": float(np.median(t_march)),
                "alpha_sum": float(out["alpha"].sum().item()),
                "what": "reference kernels (raymarcher.cu, fuse_cuda_kernel_fast.cu, filter.cu, precompute.cu built for sm_100) + "
                        "reference host loop; tiny-cuda-nn replaced by ia_ngp_forward; SMPL forward excluded"}
    except Exception as e:  # the checker must never take the bench down
        return {"unavailable": f"{type(e).__name__}: {e}"}


def bench_train(model, batch, device, rank, world, flush, steps=40, warmup=25, use_graph=True, train_rays_per_warp=None,
                rays_cap=None):
    """second half of BASELINE.json's metric: ms per training step (DNeRF.py:112-161) at 4096 rays per step
    (4 patches of 32x32, confs/sampler/patch.yaml), rays sharded over the ranks, one gradient all-reduce per step;
    includes the every-20-steps occupancy-grid refresh amortised over the timed steps."""
    import torch
    import torch.distributed as dist
    from instantavatar_b200 import parallel
    model.eval()
    rgb_gt, _, alpha_gt, _ = model.render_image_fast(dict(batch), (H, W))
    rgb_gt, alpha_gt = rgb_gt.reshape(-1, 3), alpha_gt.reshape(-1)
    torch.manual_seed(1234)  # identical on every rank: replicated grid refresh needs identical jitter
    idx = []
    for (y0, x0) in ((150, 240), (200, 232), (250, 236), (300, 240)):
        ys, xs = torch.arange(y0, y0 + 32), torch.arange(x0, x0 + 32)
        idx.append((ys[:, None] * W + xs[None]).reshape(-1))
    idx = torch.cat(idx)
    if rays_cap:  # sweeps only: a smaller step (every 4096 // rays_cap-th ray of the four patches)
        idx = idx[:: len(idx) // rays_cap][:rays_cap]
    sl = parallel.shard_train_rays(len(idx), rank, world)
    pick = idx[sl].to(device)
    n = len(pick)
    b = dict(batch)
    for k in ("rays_o", "rays_d", "near", "far"):
        b[k] = batch[k][:, pick].contiguous()
    a = alpha_gt[pick][None]
    model.configure_parallel(world)
    if train_rays_per_warp:  # sweeps (scripts/train_scaling.py) override the tile size configure_parallel picked
        from instantavatar_b200 import ops as _ops
        _ops.set_option("train_rays_per_warp", train_rays_per_warp)
    model.global_step = 2000  # steady state: no density noise, grid refresh uses the previous field as `valid`
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    graphed = None
    if use_graph:
        from instantavatar_b200.graphs import GraphedTrainStep
        b["bg_color"], b["alpha"], b["rgb"] = torch.rand((1, n, 3), device=device), a, rgb_gt[pick][None].clone()
        graphed = GraphedTrainStep(model, b)

    # per-step data (random background per pixel, peoplesnapshot.py:109-114 -- the reference composes it in the CPU data
    # loader, off the step's critical path): a pool of prebuilt device batches; a step copies three small tensors
    pool = []
    for _ in range(8):
        bg = torch.rand((1, n, 3), device=device)
        pool.append({"bg_color": bg, "rgb": rgb_gt[pick][None] - (1 - a[..., None]) + (1 - a[..., None]) * bg})
    counter = [0]

    def one():
        cur = pool[counter[0] % len(pool)]
        counter[0] += 1
        if graphed is not None:
            return graphed(cur)   # copies bg_color / rgb into the graph's static buffers, replays
        b["bg_color"], b["rgb"], b["alpha"] = cur["bg_color"], cur["rgb"], a
        return model.training_step(b)

    for _ in range(warmup):
        one()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    ev0.record()
    for _ in range(steps):
        out = one()
    ev1.record()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    ms = torch.tensor([ev0.elapsed_time(ev1) / steps], device=device, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    return {"ms_per_step": float(ms.item()), "rays_per_step": int(len(idx)), "rays_per_rank": int(n), "steps": steps,
            "cuda_graph": bool(use_graph), "grid_refresh_every": 20,
            "collective": ("reduce-scatter (52 MB fp32 gradient) + sharded Adam + all-gather (26 MB fp16 image): inside two kernels over NVLink "
                           "peer memory when available (config.train_exchange_path), else NCCL") if world > 1 else "none",
            "final_loss": float(out["loss"].item()), "scaling": "strong"}


def bench_next_rows(model, batch, device, steps=20, warmup=5):
    """SURVEY.md 8f rows 3 and 4, measured like the hot path (CUDA events after warm-up): one pose-refinement step
    (frozen network, SMPL parameters optimised through ia_pose_grad; eval.py / SNARF_NGP_refine.yaml) on 4096 rays, and
    the once-per-subject skinning-weight voxelisation (ia_voxelize_weights, 524 288 voxels x 6890 vertices, K = 30)."""
    import torch
    from instantavatar_b200 import ops
    out = {}
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    # ---- f4: voxelisation ----
    d = model.deformer
    fd = d.deformer
    dd, hh, ww = fd.lbs_voxel_final.shape[-3:]
    lin = lambda n: torch.linspace(-1, 1, steps=n, device=device)
    args_v = (d.vs_template[0].float(), d.body_model.lbs_weights.float(), lin(ww), lin(hh), lin(dd), fd.offset.reshape(3).float(),
              fd.scale.reshape(1).float(), float(fd.ratio))
    ops.voxelize_weights(*args_v)
    torch.cuda.synchronize()
    ev0.record(); ops.voxelize_weights(*args_v); ev1.record()
    torch.cuda.synchronize()
    out["voxelize_weights_ms"] = ev0.elapsed_time(ev1)
    # ---- f3: pose refinement step ----
    model.eval()
    rgb_gt, _, alpha_gt, _ = model.render_image_fast(dict(batch), (H, W))
    rgb_gt, alpha_gt = rgb_gt.reshape(-1, 3), alpha_gt.reshape(-1)
    idx = []
    for (y0, x0) in ((150, 240), (200, 232), (250, 236), (300, 240)):
        ys, xs = torch.arange(y0, y0 + 32), torch.arange(x0, x0 + 32)
        idx.append((ys[:, None] * W + xs[None]).reshape(-1))
    pick = torch.cat(idx).to(device)
    b = dict(batch)
    for k in ("rays_o", "rays_d", "near", "far"):
        b[k] = batch[k][:, pick].contiguous()
    a = alpha_gt[pick][None]
    b["bg_color"] = torch.rand((1, len(pick), 3), device=device)
    b["alpha"] = a
    b["rgb"] = rgb_gt[pick][None] - (1 - a[..., None]) + (1 - a[..., None]) * b["bg_color"]
    b["idx"] = torch.zeros(1, dtype=torch.long, device=device)
    world_before = model.world_size
    model.world_size = 1
    model.enable_pose_optimisation({k: batch[k].clone() for k in ("betas", "global_orient", "body_pose", "transl")}, lr=1e-5, is_refine=True)
    model.freeze_network()
    model.global_step = 2000
    def timed(fn, warmup, steps):
        for _ in range(warmup):
            fn()
        torch.cuda.synchronize()
        ev0.record()
        for _ in range(steps):
            fn()
        ev1.record()
        torch.cuda.synchronize()
        return ev0.elapsed_time(ev1) / steps

    eager_ms = timed(lambda: model.training_step(b), warmup, steps)
    graph_ms = None
    try:  # the refinement step is sync-free (device-state Adam, fused bone-transform backward): capture and replay it
        from instantavatar_b200.graphs import GraphedTrainStep
        model.global_step = 2000
        graphed = GraphedTrainStep(model, b)
        graph_ms = timed(lambda: graphed(), 25, 40)  # warm-up captures both variants (with / without the grid refresh)
    except Exception as exc:
        print(f"[bench] pose-refinement graph capture failed ({type(exc).__name__}: {exc}), eager number only", file=sys.stderr)
    out["pose_refine"] = {"ms_per_step": graph_ms if graph_ms is not None else eager_ms, "ms_per_step_eager": eager_ms,
                          "rays_per_step": int(len(pick)), "steps": 40 if graph_ms is not None else steps, "cuda_graph": graph_ms is not None,
                          "what": "frozen network: fused bone transforms (+ reverse mode), train_fwd, loss, composite_bwd, ngp_backward "
                                  "(features only), pose_grad, device Adam on the pose tables; grid refresh amortised"}
    model.freeze_network(False)
    model.SMPL_param, model.pose_optimizer, model.is_refine = None, None, False
    model.world_size = world_before
    return out


def multi_gpu_checks(model, batch, device, rank, world):
    """multi-GPU correctness the driver can see (body of tests/test_gpu_multi.py): the cooperative frame equals the
    single-GPU frame bit for bit, and the ray-sharded gradient (sum over ranks / world) equals the full-batch gradient"""
    import torch
    import torch.distributed as dist
    from instantavatar_b200 import ops, parallel
    from instantavatar_b200.autograd import GRAD_SCALE
    from instantavatar_b200.models.dnerf import Rays
    model.eval()
    b = {k: v.clone() for k, v in batch.items()}
    for k in ("betas", "body_pose", "global_orient", "transl"):
        dist.broadcast(b[k], 0)
    torch.manual_seed(99)
    jit = torch.rand((5, 64, 64, 64, 3), device=device)
    img = model.render_image_sharded(dict(b), (H, W), rank, world, jit)
    rgb, _, alpha, _ = model.render_image_fast(dict(b), (H, W), jit)
    out = {}
    if rank == 0:
        out["frame_bit_equal"] = bool(torch.equal(img, torch.cat([rgb.reshape(-1, 3), alpha.reshape(-1, 1)], dim=1)))
    # gradient of 4096 rays: full batch on every rank vs shard + sum over ranks
    ys, xs = torch.arange(200, 264), torch.arange(224, 288)
    pick = (ys[:, None] * W + xs[None]).reshape(-1).to(device)
    n = len(pick)
    tb = {k: b[k][:, pick].contiguous() for k in ("rays_o", "rays_d", "near", "far")}
    torch.manual_seed(11)
    tgt_rgb, tgt_a, bg = torch.rand((n, 3), device=device), torch.ones(n, device=device), torch.rand((n, 3), device=device)
    jitter, noise = torch.rand((n, 256), device=device), torch.zeros((n, 256), device=device)
    grid = model.renderer.density_grid_test
    g_enc, g_col = model.net_coarse.grad_buffers()

    def grads(sl, reduce):
        g_enc.zero_(); g_col.zero_()
        rr = Rays(o=tb["rays_o"][:, sl], d=tb["rays_d"][:, sl], near=tb["near"][:, sl], far=tb["far"][:, sl])
        model.deformer.transform_rays_w2s(rr)
        scene = model.deformer.scene(model.net_coarse, grid.occupancy_bits(), grid.aabb6())
        o_, d_ = rr.o.reshape(-1, 3).contiguous(), rr.d.reshape(-1, 3).contiguous()
        ne, fa = rr.near.reshape(-1).contiguous(), rr.far.reshape(-1).contiguous()
        out_, saved = ops.train_fwd(scene, o_, d_, ne, fa, bg[sl].contiguous(), jitter[sl].contiguous(), noise[sl].contiguous())
        _, g_rgb, g_alpha, g_w = ops.nerf_loss(out_, tgt_rgb[sl], tgt_a[sl])
        l = ops.composite_bwd(ne, fa, bg[sl].contiguous(), noise[sl].contiguous(), saved, g_rgb, None, g_alpha, g_w)
        ops.ngp_backward(scene, l[0], l[1], l[2], l[3], g_enc, g_col, GRAD_SCALE)
        ge = g_enc.clone()
        if reduce:
            dist.all_reduce(ge)
            ge /= world
        return ge

    full = grads(slice(0, n), False)
    shard = grads(parallel.shard_train_rays(n, rank, world), True)
    g_enc.zero_(); g_col.zero_()
    out["train_grad_rel_err"] = float(((shard - full).norm() / full.norm()).item())
    return out


def bench_collectives(model, device, rank, world, iters=20):
    """BASELINE.md B5: the step's gradient collective alone -- reduce-scatter (sum) of the flat fp32 gradient + all-gather of
    the fp16 image -- device time (max over ranks) and bus bandwidth: per-rank bytes on the wire = (G-1)/G x (52 MB + 26 MB)"""
    import torch
    import torch.distributed as dist
    from instantavatar_b200 import parallel
    from instantavatar_b200.optim import shard_layout
    opt = model.optimizer
    S, L = shard_layout(opt.n, world)
    g = torch.zeros(L, device=device); sh = torch.zeros(S, device=device); h = torch.zeros(L, device=device, dtype=torch.float16)
    for _ in range(5):
        parallel.reduce_scatter_sum(sh, g); parallel.all_gather_inplace(h)
    dist.barrier(); torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        parallel.reduce_scatter_sum(sh, g); parallel.all_gather_inplace(h)
    e1.record()
    dist.barrier(); torch.cuda.synchronize()
    ms = torch.tensor([e0.elapsed_time(e1) / iters], device=device, dtype=torch.float64)
    dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    nbytes = L * 4 + L * 2
    wire = (world - 1) / world * nbytes
    return {"ms": float(ms.item()), "bytes": int(nbytes), "bus_GBps": wire / (float(ms.item()) * 1e-3) / 1e9,
            "what": "reduce_scatter(fp32 flat gradient) + all_gather(fp16 image), NCCL over NVLink"}


def bench_optimizer_step(model, device, world, iters=30):
    """the sharded optimiser step alone (gradient exchange + Adam on the shard + fp16 image exchange), captured in a CUDA
    graph, device time max over ranks; says which exchange path ran (NVLink peer memory or NCCL)"""
    import torch
    import torch.distributed as dist
    opt = model.optimizer
    opt.zero_grad()
    fn = lambda: opt.step(model.scaler, world)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        for _ in range(3):
            fn()
    torch.cuda.current_stream().wait_stream(s)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        fn()
    for _ in range(3):
        g.replay()
    dist.barrier(); torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        g.replay()
    e1.record()
    dist.barrier(); torch.cuda.synchronize()
    ms = torch.tensor([e0.elapsed_time(e1) / iters], device=device, dtype=torch.float64)
    dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    return {"ms": float(ms.item()), "path": "peer" if getattr(opt, "_peer", None) else "nccl"}


def run_ours(args):
    import torch
    import torch.distributed as dist
    from instantavatar_b200 import _lib, ops

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    device = torch.device("cuda", local)
    # the occupancy-grid jitter of every frame is drawn inside the captured graph: seeded, the same arguments give the
    # same frames from run to run
    torch.manual_seed(0)
    if world > 1:
        dist.init_process_group("nccl", device_id=device)
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    if args.rays_per_warp:
        ops.set_option("render_rays_per_warp", args.rays_per_warp)
    if args.train_rays_per_warp:
        ops.set_option("train_rays_per_warp", args.train_rays_per_warp)
    if args.render_warps:
        ops.set_option("render_warps", args.render_warps)
    if args.query_warps:
        ops.set_option("query_warps", args.query_warps)

    frame = FRAMES[rank % len(FRAMES)]
    model, hb, batch = build_model(device, frame)
    pinned = {k: torch.from_numpy(v).pin_memory() for k, v in hb.items()}
    h2d_bytes = sum(v.numel() * v.element_size() for v in pinned.values())
    out_host = torch.empty((N_RAYS, 4), dtype=torch.float32).pin_memory()
    d2h_bytes = out_host.numel() * 4
    flush = torch.empty(192 * 1024 * 1024, dtype=torch.uint8, device=device)  # > 126 MB L2

    from instantavatar_b200.graphs import GraphedFrame
    use_graph = not args.no_graph
    frame_graph = GraphedFrame(model, batch, (H, W)) if use_graph else None

    def step_resident():
        if use_graph:
            return frame_graph()  # inputs already resident in the graph's static buffers
        return model.render_image_fast(dict(batch), (H, W))

    def step_e2e():
        if use_graph:
            rgb, depth, alpha, counter = frame_graph(pinned)  # pinned host -> static device buffers, replay
        else:
            b = {k: v.to(device, non_blocking=True) for k, v in pinned.items()}
            rgb, depth, alpha, counter = model.render_image_fast(b, (H, W))
        out_host.copy_(torch.cat([rgb.reshape(-1, 3), alpha.reshape(-1, 1)], dim=1), non_blocking=True)
        return rgb

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps, warmup):
        for _ in range(warmup):
            fn()
        barrier()
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        out = None
        for a, b in ev:
            flush.zero_()  # L2 flush between timed iterations (outside the event bracket)
            a.record(); out = fn(); b.record()
        barrier()
        ms = [a.elapsed_time(b) for a, b in ev]
        tot = torch.tensor([sum(ms)], device=device, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(tot, op=dist.ReduceOp.MAX)
        return float(tot.item()), ms, out

    # nvidia-smi needs a few hundred ms before its first row: the sampler was started before the model was built
    t_load0 = time.monotonic()
    _lib.LAUNCHES = 0
    total_ms, per, last = timed(step_resident, args.steps, max(args.warmup, 3))
    launches = getattr(_lib, "LAUNCHES", 0)
    # the graph's output buffers are overwritten by every later replay: keep the last timed frame
    last = dict(zip(("rgb", "depth", "alpha", "counter"), (t.clone() for t in last))) if args.dump_outputs else None
    e2e_ms, _, _ = timed(step_e2e, args.steps, 3)
    t_load1 = time.monotonic()
    clocks = None
    if rank == 0:
        window = "timed regions (device-resident + e2e)"
        if sampler.count_between(t_load0, t_load1) < 5:
            # the timed regions are shorter than a few 100-ms sampling periods: keep the GPU under the identical load
            # (same step, untimed) until enough rows have arrived
            while sampler.proc is not None and sampler.count_between(t_load0, time.monotonic()) < 5 and time.monotonic() - t_load1 < 3.0:
                step_resident()
            torch.cuda.synchronize()
            t_load1 = time.monotonic()
            window = "timed regions + the same step repeated untimed until 5 samples (100 ms period)"
        clocks = sampler.stop(t_load0, t_load1)
        clocks["window"] = window

    # ---- kernel-only timings + work counters for the rooflines of the two frame kernels ----
    rays = model.renderer
    stats = ops.new_stats(device)
    from instantavatar_b200.models.dnerf import Rays
    from instantavatar_b200.renderers.raymarcher_acc import BoundModel
    r = Rays(o=batch["rays_o"].clone(), d=batch["rays_d"].clone(), near=batch["near"].clone(), far=batch["far"].clone())
    model.deformer.transform_rays_w2s(r)
    bm = BoundModel(model.deformer, model.net_coarse, True)
    rays.image_width = W
    rays.render_test(r, bm, None, stats)
    torch.cuda.synchronize()
    st = ops.stats_dict(stats)

    def kernel_ms(fn, n=10):
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(n)]
        for a, b in ev:
            flush.zero_()
            a.record(); fn(); b.record()
        torch.cuda.synchronize()
        return float(np.median([a.elapsed_time(b) for a, b in ev]))

    k_ms = kernel_ms(lambda: rays.render_test(r, bm, None))
    # occupancy-init point queries (5 x 64^3 points): the query kernel alone, then the whole initialisation
    grid = rays.density_grid_test
    scene_q = model.deformer.scene(model.net_coarse)
    qjit = torch.rand((5, 64, 64, 64, 3), device=device)
    qstats = ops.new_stats(device)
    ops.occupancy_query(scene_q, qjit, grid.aabb6(), None, qstats)
    torch.cuda.synchronize()
    qst = ops.stats_dict(qstats)
    q_ms = kernel_ms(lambda: ops.occupancy_query(scene_q, qjit, grid.aabb6(), None, None), 8)
    occ_ms = kernel_ms(lambda: grid.initialize(model.deformer, model.net_coarse), 5)
    # measured ceiling of the kernels' gather shape on this GPU, same process, same table (ia_gather_ceiling)
    fld = model.deformer.deformer.field
    ceil_k = ops.gather_ceiling(fld, 200, 12, True)     # at the kernels' residency (12 warps / SM), coherent batches
    ceil_best = max([ceil_k] + [ops.gather_ceiling(fld, 200, w, c) for w, c in ((12, False), (32, True), (32, False))],
                    key=lambda d: d["sectors_per_s"])

    sharded = bench_frame_sharded(model, batch, device, rank, world, flush) if world > 1 else None
    checks = multi_gpu_checks(model, batch, device, rank, world) if world > 1 else None
    ref_struct = bench_ref_structure(model, batch, device) if rank == 0 else None
    train = bench_train(model, batch, device, rank, world, flush, use_graph=use_graph)
    comm = bench_collectives(model, device, rank, world) if world > 1 else None
    opt_step = bench_optimizer_step(model, device, world) if world > 1 else None
    next_rows = None
    if rank == 0:
        try:
            next_rows = bench_next_rows(model, batch, device)
        except Exception as exc:  # reported, never fatal for the headline numbers
            next_rows = {"error": f"{type(exc).__name__}: {exc}"}

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    if last is not None:
        dump_outputs(args.dump_outputs, {k: v.cpu().numpy() for k, v in last.items()})
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    hbm_peak, peak_src = (peaks.get("hbm_gbs"), "measured") if peaks.get("hbm_gbs") else (6650.0, "fallback")
    # Sectors the kernels REQUEST (kernel counters; exact-zero footprints and early-out solves issue nothing and are not
    # counted): 12 x 32 B per field footprint that loaded, one sector per hash-table load a lane issues (128 per network
    # evaluation: 16 levels x 8 corners).  The ceiling is the same shape in isolation (lane = footprint, 12 LDG.E.256, next
    # address data-dependent) measured in this run: frac = requested sectors / s over that.
    q_sect = qst["field_loads"] * 12 + qst["hash_loads"]
    r_sect = st["field_loads"] * 12 + st["hash_loads"]
    q_gbs, r_gbs = q_sect * 32 / (q_ms * 1e-3) / 1e9, r_sect * 32 / (k_ms * 1e-3) / 1e9
    ceil_gbs = ceil_best["GBps"]
    field_bytes = fld.numel() * 4
    table_bytes = 6513496 * 4
    value = world * N_RAYS * args.steps / (total_ms * 1e-3)
    e2e = world * N_RAYS * args.steps / (e2e_ms * 1e-3)
    cfg = {"workload": "male-3-casual-shaped synthetic avatar, one 512x512 frame per step per GPU (SMPL prep, 5-pass occupancy init, fused render)",
           "rays_per_step_per_gpu": N_RAYS, "l2_flush_between_steps": True, "cuda_graph": bool(use_graph),
           # scalar keys (the driver's record keeps scalars of `config`): per-kernel times of the frame, then the second half of
           # BASELINE.json's metric (train-step ms, 4096 rays strong-scaled over the ranks) and the strong-scaled single frame
           "ms_occupancy_query_kernel": q_ms, "ms_occupancy_init": occ_ms, "ms_render_kernel": k_ms, "ms_frame": total_ms / args.steps,
           "train_ms_per_step": train["ms_per_step"], "train_rays_per_step": train["rays_per_step"], "train_scaling": "strong",
           "train_forward": "split (march -> sample list -> point query -> compositing)" if ops.get_option("train_split") else "fused (one kernel)"}
    if sharded is not None:
        cfg.update({"frame_sharded_ms": sharded["ms_per_frame"], "frame_sharded_rays_per_s": sharded["rays_per_s"],
                    "frame_sharded_path": sharded["path"], "frame_sharded_nccl_ms": sharded["nccl"]["ms_per_frame"],
                    "frame_sharded_peer_ms": sharded["peer"]["ms_per_frame"] if "peer" in sharded else None,
                    "frame_sharded_bit_equal": bool(sharded["bit_equal"] and checks["frame_bit_equal"]),
                    "train_grad_rel_err": checks["train_grad_rel_err"]})
        from instantavatar_b200.models.dnerf import sharded_rays_per_warp
        cfg["frame_sharded_render_rays_per_warp"] = sharded_rays_per_warp(ops.get_option("render_rays_per_warp"), world)
    if comm is not None:
        cfg.update({"grad_collective_ms": comm["ms"], "grad_collective_bus_GBps": comm["bus_GBps"], "grad_collective_bytes": comm["bytes"]})
    if opt_step is not None:
        # the step's real exchange: reduce + finite agreement + Adam on 1/G + fp16 image exchange, on the path the step used
        cfg.update({"train_optimizer_step_ms": opt_step["ms"], "train_exchange_path": opt_step["path"],
                    "train_rays_per_warp": ops.get_option("train_rays_per_warp")})
    line = {
        "metric": METRIC, "value": value, "unit": "rays/s", "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
        "ms_per_step": total_ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32 geometry + f16 hash-grid/MLP (fp32 accumulate)", "data": "synthetic",
        "config": cfg,
        "clocks": clocks,
        "e2e": {"value": e2e, "unit": "rays/s", "h2d_bytes_per_step": h2d_bytes, "d2h_bytes_per_step": d2h_bytes,
                "ms_per_step": e2e_ms / args.steps},
        "gpu_launches": launches,
        # dominant kernel of the step = the occupancy-init point query; second = the fused renderer (flat `render_*` keys)
        "roofline": {"kernel": "deform_query_kernel", "bound": "hbm", "achieved": q_gbs, "peak": ceil_gbs, "unit": "GB/s",
                     "frac": q_gbs / ceil_gbs, "traffic": None, "kernel_ms": q_ms, "sectors_requested": q_sect,
                     "peak_source": f"measured in this run: ia_gather_ceiling, {ceil_best['warps']} warps/SM, coherent={ceil_best['coherent']}",
                     "peak_at_kernel_residency_GBps": ceil_k["GBps"], "hbm_peak_GBps": hbm_peak, "hbm_peak_source": peak_src,
                     "compulsory_dram_bytes": field_bytes + table_bytes,
                     "render_kernel": "render_fwd_kernel", "render_achieved": r_gbs, "render_frac": r_gbs / ceil_gbs,
                     "render_kernel_ms": k_ms, "render_sectors_requested": r_sect,
                     "note": "gather-bound on L2-resident tables (76 MB): achieved = 32 B x sectors the kernel requests / CUDA-event time; peak = the same access shape in isolation (L1 data pipe + L2), not HBM; DRAM traffic is the compulsory table read (ncu captures in profiles/)"},
        "work_per_frame": st, "work_per_occupancy_init": qst,
        "train": train, "grad_collective": comm, "frame_sharded": sharded, "multi_gpu_checks": checks,
        "next_rows": next_rows, "ref_structure": ref_struct,
    }
    if not args.no_cpu_baseline:
        cf = CpuFrame(frame)
        cf.step()
        t0 = time.perf_counter(); n = 2
        for _ in range(n):
            cf.step()
        dt = (time.perf_counter() - t0) / n
        line["cpu_baseline"] = {"value": N_RAYS / dt, "unit": "rays/s", "cores": cf.threads, "kind": "port",
                                "sample": f"{n} complete 512x512 frames (prep + occupancy init + march) on the C/numpy oracle, OpenMP"}
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    a = parse()
    if a.impl == "reference":
        run_reference(a)
    else:
        run_ours(a)

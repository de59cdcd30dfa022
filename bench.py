"""Benchmark of the PonderV2 pretraining hot path on B200 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload c2|c3|c4|c1]
                    [--dump-outputs DIR]

One "step" = one full pretraining iteration on one synthetic scene per GPU: SpUNet backbone forward/backward (rulebooks
rebuilt every step), densify, dense projection, NeuS render of R rays x S samples with its second-order backward,
the losses, the gradient all-reduce (N > 1; slices overlapped with backward) and the optimizer step.  Prints ONE JSON
line on rank 0.  Three separate timed loops (the same K steps each, barrier + synchronize on both sides):

  value    rays/s with inputs resident in HBM, NO per-call instrumentation (device-timed, CUDA events, max over ranks)
  e2e      same metric through the host-facing call: inputs in pinned host memory, H2D inside the timed region,
           loss read back (D2H) every step
  roofline third loop with one CUDA-event pair around every sparse-conv C-ABI call: dominant hand-written kernel family
           (gather-GEMM, forward + data gradient of all 59 layers): algorithmic bytes / event time vs the measured copy
           bandwidth in MEASURED_PEAKS.json; `traffic` = DRAM bytes per launch from the newest committed ncu launch list
           (profiles/*_traffic.json, written by tools/traffic_from_launches.py)
  cpu_baseline  the CPU oracle (port of the reference path: backbone + densify + projection + renderer + SGD update)
           timed on the host cores on a bounded sample, extrapolated linearly; the sample and both numbers are stated

Workloads (BASELINE.json configs): c2 = configs[1] (default: the single-GPU configuration the metric is quoted on),
c3 = configs[2] (200 k voxels, 8192 rays, bf16 autocast backbone), c4 = configs[3] (outdoor, 80 k voxels, 2048 rays x
(192 + 64) samples), c1 = configs[0] (plumbing size).

`--impl reference` times the reference's own algorithm on the CPU (oracle port: spconv is not installable offline and
smooth_sampler is CUDA-only, see DESIGN.md) with every host thread; each step is a bounded sample of the workload sized
from a calibration step so that the whole run stays within a few minutes.

`--dump-outputs DIR` writes what the last step of the device-resident loop computed (see `dump_outputs`) as
DIR/<name>.npy.  Scene, model and jitter are seeded, so two builds run with the same arguments can be compared output
for output.  The outputs are not bitwise reproducible: the sparse convolutions reduce with fp32 atomics, and every
training step amplifies the reordering.  Two runs of one build with --steps 20 --warmup 3 (B200, 1000 W power limit)
differed by 3e-3 relative in the loss and by 3e-3 relative L2 in param_sample, so compare with a tolerance above that.
"""
from __future__ import annotations

import argparse
import gc
import json
import os
import statistics
import subprocess
import sys
import tempfile
import threading
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

import numpy as np
import torch

WORKLOADS = {
    # BASELINE.json configs[1]: ScanNet-shape, ~100 k active voxels, 4096 rays x 128 samples, fp32, 1 x B200
    "c2": dict(name="ScanNet-shape synthetic: 100k voxels SpUNet-v1m1, 4096 rays x 128 samples (96+32), fp32",
               voxels=100_000, rays=4096, s0=96, si=32, grid_shape=(128, 128, 32), cfg_id=2),
    # BASELINE.json configs[0]: plumbing-size case
    "c1": dict(name="synthetic 1 scene, 2k voxels, 128 rays x 32 samples (24+8), fp32",
               voxels=2_000, rays=128, s0=24, si=8, grid_shape=(32, 32, 16), cfg_id=1),
    # BASELINE.json configs[2]: Structured3D-shape, ~200 k voxels, 8192 rays x 128, bf16 (reference: fp16 autocast), DDP
    "c3": dict(name="Structured3D-shape synthetic: 200k voxels SpUNet-v1m1, 8192 rays x 128 samples (96+32), bf16 autocast",
               voxels=200_000, rays=8192, s0=96, si=32, grid_shape=(128, 128, 32), cfg_id=3, dtype="bf16"),
    # BASELINE.json configs[3]: nuScenes-shape outdoor, ~80 k voxels over 108 x 108 x 8 m, 2048 rays x 256 samples
    "c4": dict(name="nuScenes-shape synthetic outdoor: 80k voxels, 2048 rays x 256 samples (192+64), fp32",
               voxels=80_000, rays=2048, s0=192, si=64, grid_shape=(180, 180, 5), cfg_id=4, outdoor=True),
}
for _w in WORKLOADS.values():
    _w.setdefault("dtype", "f32")
    _w.setdefault("outdoor", False)


def renderer_cfg(s0: int, si: int) -> dict:
    """configs/scannet/pretrain-ponder-spunet-v1m1-0-base.py:31-93 (semantic branch off: no CLIP offline)."""
    return dict(
        type="NeuSModel",
        field=dict(type="SDFField",
                   sdf_decoder=dict(in_dim=64, out_dim=65, hidden_size=128, n_blocks=1, points_factor=0.0),
                   rgb_decoder=dict(in_dim=134, out_dim=3, hidden_size=128, n_blocks=0, points_factor=0.0),
                   beta_init=0.3, use_gradient=True, volume_type="default", padding_mode="zeros", share_volume=False,
                   norm_pts=True, norm_padding=0.1),
        collider=dict(type="AABBBoxCollider", near_plane=0.01, bbox=[-0.55] * 3 + [0.55] * 3),
        sampler=dict(type="NeuSSampler", initial_sampler="UniformSampler", num_samples=s0, num_samples_importance=si,
                     num_upsample_steps=1, train_stratified=True, single_jitter=False),
        loss=dict(sensor_depth_truncation=0.05, temperature=0.01,
                  weights=dict(eikonal_loss=0.01, free_space_loss=1.0, sdf_loss=10.0, depth_loss=1.0, rgb_loss=10.0,
                               semantic_loss=0.0)))


def outdoor_renderer_cfg(s0: int, si: int) -> dict:
    """configs/nuscenes/pretrain-ponder-spunet-v1m1-0-base.py:31-74."""
    return dict(
        type="NeuSModel",
        field=dict(type="SDFField", sdf_decoder=dict(in_dim=32, out_dim=17, hidden_size=16, n_blocks=5),
                   beta_init=0.3, use_gradient=True, volume_type="default", padding_mode="zeros", share_volume=True),
        collider=dict(type="AABBBoxCollider", near_plane=0.01, bbox=[0.0, 0.0, 0.0, 1.0, 1.0, 1.0]),
        sampler=dict(type="NeuSSampler", initial_sampler="UniformSampler", num_samples=s0, num_samples_importance=si,
                     num_upsample_steps=1, train_stratified=True, single_jitter=False),
        loss=dict(sensor_depth_truncation=0.01, weights=dict(depth_loss=10.0)))


OUTDOOR_BBOX = (-54.0, -54.0, -5.0, 54.0, 54.0, 3.0)


def make_scene(wl: dict, seed: int) -> dict:
    """Host (numpy) scene: voxel cloud + ray batch, in the layout the dataloader/collate hands to the model."""
    from ponderv2_b200 import synth
    if wl["outdoor"]:
        c = synth.outdoor_cloud(wl["voxels"], seed)
        rng = np.random.default_rng(seed + 7)
        R = wl["rays"]
        lo, hi = np.array(OUTDOOR_BBOX[:3]), np.array(OUTDOOR_BBOX[3:])
        # lidar-like rays: from the sensor (scene centre, 1.8 m above the bbox floor) to points 5-50 m away
        start = np.tile((lo + hi) / 2 + np.array([0.0, 0.0, -2.2]), (R, 1))
        th, rr = rng.random(R) * 2 * np.pi, rng.uniform(5.0, 50.0, R)
        end = start + np.stack([rr * np.cos(th), rr * np.sin(th), rng.uniform(-1.5, 2.0, R)], 1)
        coord = c["coord"] + lo.astype(np.float32)          # sensor frame: metres inside the scene bbox
        return dict(grid_coord=c["grid_coord"], coord=coord.astype(np.float32), feat=c["feat"], offset=c["offset"],
                    ray_start=start.astype(np.float32), ray_end=end.astype(np.float32),
                    ray_offset=np.array([R], dtype=np.int64))
    c = synth.indoor_cloud(wl["voxels"], seed)
    r = synth.ray_batch(wl["rays"], seed + 7)
    gc = c["grid_coord"]
    # to_unit_cube (ponder_indoor_base.py:344-444) maps the scene into the renderer's +-0.5 cube; the densify step
    # only needs the voxel-frame coordinates and the longest bbox edge in voxels ("resolution", :622-627)
    return dict(grid_coord=gc, coord=c["coord"], feat=c["feat"], offset=c["offset"],
                resolution=np.array([int(gc.max())], dtype=np.int64),
                ray_o=r["rays_o"][None], ray_d=r["rays_d"][None], rgb=r["rgb"], depth=r["depth"])


# ------------------------------------------------------------------------------------------------------------
class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms while the timed region runs."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.proc, self.path = index, None, None

    def start(self):
        try:
            f = tempfile.NamedTemporaryFile("w", suffix=".csv", delete=False)
            self.path = f.name
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "200"], stdout=f,
                                         stderr=subprocess.DEVNULL)
        except OSError:
            self.proc = None

    def wait_first_sample(self, timeout: float = 5.0) -> None:
        """Block until nvidia-smi has written its first line (its start-up is over), at most `timeout` seconds."""
        t0 = time.time()
        while self.proc is not None and time.time() - t0 < timeout:
            try:
                if os.path.getsize(self.path) > 0:
                    return
            except OSError:
                return
            time.sleep(0.05)

    def stop(self) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in Path(self.path).read_text().splitlines():
            parts = [p.strip() for p in line.split(",")]
            if len(parts) < 7:
                continue
            try:
                sm.append(float(parts[0])); mx.append(float(parts[1]))
            except ValueError:
                continue
            for nm, val in zip(names, parts[3:7]):
                if val.lower().startswith("active"):
                    reasons.add(nm)
        os.unlink(self.path)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


T_START = time.time()


def log(msg: str) -> None:
    print(f"[bench +{time.time() - T_START:6.1f}s] {msg}", file=sys.stderr, flush=True)


def host_threads() -> int:
    """Threads for the CPU arm: every core up to 32 (torch's intra-op pool stops scaling on these small ops)."""
    return max(1, min(os.cpu_count() or 1, 32))


def profiled_traffic(kernel_prefix: str):
    """DRAM bytes per launch of `kernel_prefix` from the newest committed ncu launch list (profiles/*_traffic.json,
    written by tools/traffic_from_launches.py); None when no profile has been committed."""
    best = None
    for f in sorted((ROOT / "profiles").glob("*_traffic.json")):
        try:
            d = json.loads(f.read_text())
        except ValueError:
            continue
        tot_b = tot_n = 0
        for name, v in d.get("kernels", {}).items():
            if name.startswith(kernel_prefix) and "[render linear]" not in name:
                tot_b += v["dram_bytes_total"]; tot_n += v["launches"]
        if tot_n:
            best = dict(bytes_per_launch=tot_b / tot_n, source=f"profiles/{f.name}")
    return best


def measured_peaks() -> dict:
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        d = json.loads(p.read_text())
        return dict(hbm_gbs=float(d["hbm_gbs"]), bf16_tflops=float(d["bf16_tflops"]), source="measured")
    return dict(hbm_gbs=6650.0, bf16_tflops=1590.0, source="fallback")


# ------------------------------------------------------------------------------------------------------------
def cpu_oracle_step(wl: dict, frac: float, threads: int) -> dict:
    """Times the CPU oracle (port of the reference path) on a bounded sample of the workload: `frac` of the voxels, of the
    rays and of the dense volume's Z extent.  Stages: SpUNet forward+backward, densify, Conv3d+BN+ReLU projection
    forward+backward (torch CPU), NeuS render forward+backward (second order), one SGD update of every parameter.
    Returns the seconds of each stage and the whole-step time extrapolated linearly to the full workload."""
    from oracle import densify_oracle as do
    from oracle import spconv_oracle as so
    from oracle.render_oracle import NeusOracle, RenderConfig
    from ponderv2_b200 import synth
    from ponderv2_b200.backbone import SpUNetBase
    from ponderv2_b200.render import build_renderer

    torch.set_num_threads(threads)
    torch.manual_seed(0)
    outdoor = wl["outdoor"]
    sv = max(int(wl["voxels"] * frac), 1000)
    sr = max(int(wl["rays"] * frac), 16)
    X, Y, Z = wl["grid_shape"]
    zs = max(int(round(Z * frac)), 2) if not outdoor else Z
    ys = Y if not outdoor else max(int(round(Y * frac)), 4)
    cloud = (synth.outdoor_cloud if outdoor else synth.indoor_cloud)(sv, 4242)
    bb = SpUNetBase(in_channels=cloud["feat"].shape[1], num_classes=0)
    sd = {k: v.detach().clone().requires_grad_(v.is_floating_point() and v.dim() > 0 and "running" not in k)
          for k, v in bb.state_dict().items()}
    t0 = time.perf_counter()
    feats = so.spunet_forward(sd, cloud["grid_coord"], torch.from_numpy(cloud["feat"]), cloud["offset"])
    t_fwd = time.perf_counter() - t0
    # densify + projection on the sampled slab of the dense grid
    t0 = time.perf_counter()
    cproj = 32 if outdoor else 128
    cell = torch.randint(0, zs * ys * X, (sv,))
    vol = torch.zeros(zs * ys * X, feats.shape[1]).index_add_(0, cell, feats.float())
    cnt = torch.zeros(zs * ys * X).index_add_(0, cell, torch.ones(sv)).clamp(min=1)
    vol = (vol / cnt[:, None]).view(1, zs, ys, X, -1).permute(0, 4, 1, 2, 3)
    conv = torch.nn.Conv3d(96, cproj, 3, padding=1)
    bn = torch.nn.BatchNorm3d(cproj)
    vol_p = torch.relu(bn(conv(vol)))
    t_proj_fwd = time.perf_counter() - t0

    rcfg = outdoor_renderer_cfg(wl["s0"], wl["si"]) if outdoor else renderer_cfg(wl["s0"], wl["si"])
    rm = build_renderer(rcfg)
    rsd = {k: v.detach().clone().requires_grad_(v.requires_grad) for k, v in rm.state_dict().items()}
    for k, p in rm.named_parameters():
        rsd[k].requires_grad_(p.requires_grad)
    if outdoor:
        cfg = RenderConfig(bbox=[0, 0, 0, 1, 1, 1], near_plane=0.01, num_samples=wl["s0"], num_samples_importance=wl["si"],
                           share_volume=True, norm_pts=False, norm_padding=0.0, sdf_points_factor=1.0, has_rgb=False,
                           loss_weights=rcfg["loss"]["weights"], sensor_depth_truncation=0.01)
        rays = synth.ray_batch(sr, 99, bbox=(0, 0, 0, 1, 1, 1))
    else:
        cfg = RenderConfig(bbox=[-0.55] * 3 + [0.55] * 3, near_plane=0.01, num_samples=wl["s0"],
                           num_samples_importance=wl["si"], share_volume=False, norm_pts=True, norm_padding=0.1,
                           loss_weights=rcfg["loss"]["weights"])
        rays = synth.ray_batch(sr, 99)
    noise = {"uniform": torch.rand(sr, wl["s0"] + 1), "pdf": torch.rand(sr, wl["si"] + 1)}
    orc = NeusOracle(rsd, cfg)
    t0 = time.perf_counter()
    out = orc.render(torch.from_numpy(rays["rays_o"]), torch.from_numpy(rays["rays_d"]), [vol_p[0]], noise, True)
    ld = orc.loss(out, torch.from_numpy(rays["depth"]), None if outdoor else torch.from_numpy(rays["rgb"]))
    loss = orc.total_loss(ld)
    t_r_fwd = time.perf_counter() - t0
    t0 = time.perf_counter()
    loss.backward()                 # renderer (2nd order) -> projection -> densify -> backbone, one graph
    t_bwd = time.perf_counter() - t0
    t0 = time.perf_counter()
    with torch.no_grad():           # SGD(momentum, weight decay) over every parameter of the step
        for t in list(sd.values()) + list(rsd.values()) + list(conv.parameters()) + list(bn.parameters()):
            if t.grad is not None:
                buf = t.grad + 1e-4 * t
                t.add_(buf, alpha=-5e-4)
    t_opt = time.perf_counter() - t0
    sample_s = t_fwd + t_proj_fwd + t_r_fwd + t_bwd + t_opt
    return dict(sample_s=sample_s, full_step_s=sample_s / frac, frac=frac, voxels=sv, rays=sr,
                stages=dict(backbone_fwd=t_fwd, densify_projection_fwd=t_proj_fwd, render_fwd=t_r_fwd, backward=t_bwd,
                            optimizer=t_opt))


def config_dict(wl: dict, world: int) -> dict:
    """Identical keys from both arms."""
    return {"workload": wl["name"], "scenes_per_gpu_per_step": 1, "parallelism": f"dp{world}",
            "projection": ("UNet3D-v1m2 (the ScanNet config's projection, SURVEY 8f-1; cuDNN)"
                           if wl.get("projection") == "UNet3D-v1m2" else
                           "SimpleConv3D-v1m1 (the nuScenes config's projection; --projection unet3d runs the ScanNet "
                           "config's UNet3D-v1m2, SURVEY 8f-1)"),
            "l2": "per-step working set (dense volumes, render activations) exceeds the 126 MB L2"}


def run_reference(args, wl: dict) -> None:
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    threads = host_threads()
    n = args.warmup + args.steps
    # calibration on 5 % of the workload, then a sample fraction that keeps the whole run within ~4 minutes
    cal = cpu_oracle_step(wl, 0.05, threads)
    budget = 240.0 / max(n, 1)
    frac = min(1.0, max(0.05, 0.05 * budget / max(cal["sample_s"], 1e-3)))
    log(f"cpu arm: calibration {cal['sample_s']:.1f} s at 5 % -> sample fraction {frac:.3f} per step")
    times, last = [], None
    for i in range(n):
        last = cpu_oracle_step(wl, frac, threads)
        if i >= args.warmup:
            times.append(last["full_step_s"])
    per_step = statistics.mean(times)
    value = wl["rays"] / per_step  # one host: the CPU arm does not scale with N
    sample = (f"{frac:.3f} of the step per timed step ({last['voxels']} voxels, {last['rays']} rays x "
              f"{wl['s0'] + wl['si']} samples, the same fraction of the dense grid): SpUNet fwd+bwd, densify, Conv3d "
              f"projection, NeuS render fwd+bwd (2nd order), SGD update; measured {last['sample_s']:.1f} s, "
              f"extrapolated linearly x{1 / frac:.1f}")
    print(json.dumps({
        "impl": "reference", "metric": "pretrain_rays_per_sec", "value": value, "unit": "rays/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": per_step * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": wl["dtype"], "data": "synthetic",
        "config": config_dict(wl, args.gpus),
        "cpu_baseline": {"value": value, "unit": "rays/s", "cores": threads, "kind": "port", "sample": sample,
                         "stages_s": last["stages"], "run_to_run": [wl["rays"] / t for t in times]},
        "e2e": {"value": value, "unit": "rays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "scenes_per_sec": 1.0 / per_step, "voxels_per_sec": wl["voxels"] / per_step,
    }))


# ------------------------------------------------------------------------------------------------------------
def build_model(wl: dict, dev, overlap: bool = True):
    """Model (identical replicas: fixed seed), flat parameter/gradient buffers, SGD as in the reference configs
    (configs/scannet/pretrain-ponder-spunet-v1m1-0-base.py:96-98)."""
    from ponderv2_b200.dist import FlatParameters, broadcast_parameters
    from ponderv2_b200.pretrain import PonderIndoorStep, PonderOutdoorStep
    torch.manual_seed(1234)
    if wl["outdoor"]:
        model = PonderOutdoorStep(backbone=dict(in_channels=4, num_classes=0),
                                  renderer=outdoor_renderer_cfg(wl["s0"], wl["si"]),
                                  projection=dict(in_channels=96, out_channels=32),
                                  mask=dict(ratio=0.8, size=8, channel=4), scene_bbox=OUTDOOR_BBOX,
                                  grid_shape=wl["grid_shape"], grid_size=(0.6, 0.6, 1.6)).to(dev).train()
    else:
        model = PonderIndoorStep(backbone=dict(in_channels=6, num_classes=0), renderer=renderer_cfg(wl["s0"], wl["si"]),
                                 projection=dict(type=wl.get("projection", "SimpleConv3D-v1m1"), in_channels=96,
                                                 out_channels=128), grid_shape=wl["grid_shape"],
                                 grid_size=0.02).to(dev).train()
    # flat buffers in backward-completion order: renderer, projection, then the backbone back to front
    flat = FlatParameters(model, order=model.grad_completion_order(), num_chunks=4)
    flat.freeze_untouched([n for n, _ in model.named_parameters() if "laplace_density" in n])
    broadcast_parameters(flat)
    if overlap:
        flat.enable_overlap()
    opt = flat.make_optimizer(torch.optim.SGD, lr=5e-4, momentum=0.9, weight_decay=1e-4, nesterov=True)
    return model, flat, opt


def dump_outputs(path: str, out: dict, flat, sample: int = 1 << 22) -> None:
    """What a caller of the training step receives from its last run, as float32 .npy files under `path`: every entry of
    the step's output dict (the loss and its terms) and the parameters after the optimizer step.  The flat parameter
    buffer holds ~40 M values, so `param_sample` is the value at `sample` positions drawn with a fixed seed (16 MB)."""
    d = Path(path)
    d.mkdir(parents=True, exist_ok=True)
    for k, v in out.items():
        np.save(d / f"{k}.npy", v.float().cpu().numpy())
    n = flat.flat_param.numel()
    idx = np.sort(np.random.default_rng(0).choice(n, size=min(n, sample), replace=False))
    idx = torch.from_numpy(idx).to(flat.flat_param.device)
    np.save(d / "param_sample.npy", flat.flat_param[idx].float().cpu().numpy())


def nccl_summary(path_glob: str) -> dict:
    """Algorithm / protocol / transport lines NCCL logged for the all-reduce (NCCL_DEBUG=INFO to per-rank files)."""
    import glob
    import re
    found = {"nvls": False, "channels": None, "algos": set(), "version": None, "ranks_logged": 0, "lines": []}
    for f in sorted(glob.glob(path_glob)):
        try:
            txt = Path(f).read_text(errors="ignore")
        except OSError:
            continue
        found["ranks_logged"] += 1
        if not found["lines"]:   # a few verbatim lines of one rank: transport, channel count, tuning choice
            keep = [ln.split(" NCCL INFO ", 1)[-1][:160] for ln in txt.splitlines()
                    if re.search(r"NVLS|coll channels|via P2P|Connected all|AllReduce.*(Algo|algo)|comm 0x.* rank .* nranks", ln)]
            seen, uniq = set(), []
            for ln in keep:
                key = re.sub(r"0x[0-9a-f]+|\d+", "#", ln)
                if key not in seen:
                    seen.add(key); uniq.append(ln)
            found["lines"] = uniq[:12]
        if re.search(r"NVLS", txt):
            found["nvls"] = True
        m = re.search(r"NCCL version ([0-9.+a-z]+)", txt)
        if m:
            found["version"] = m.group(1)
        m = re.search(r"(\d+) coll channels", txt)
        if m:
            found["channels"] = int(m.group(1))
        for a in re.findall(r"Algo(?:rithm)?[ =:]+(\w+)", txt):
            found["algos"].add(a)
        for a in ("Ring", "Tree", "NVLS", "CollNet"):
            if re.search(rf"\b{a}\b", txt):
                found["algos"].add(a)
    found["algos"] = sorted(found["algos"])
    return found


def run_ours(args, wl: dict) -> None:
    import torch.distributed as dist
    from ponderv2_b200 import _lib

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py --impl ours needs a CUDA device: ponderv2_b200 has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    nccl_log = None
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        # NCCL's INFO log (algorithm, channels, NVLS) goes to per-rank files, never to the JSON line on stdout
        nccl_log = tempfile.mkdtemp(prefix="pv2_nccl_")
        # (forced, not setdefault: with an inherited NCCL_DEBUG=VERSION/WARN NCCL printf's its version line to stdout)
        os.environ["NCCL_DEBUG"] = "INFO"
        os.environ["NCCL_DEBUG_SUBSYS"] = "INIT,GRAPH,TUNING"
        os.environ["NCCL_DEBUG_FILE"] = os.path.join(nccl_log, "rank%h.%p.log")
        dist.init_process_group("nccl", device_id=dev)
    lib = _lib.load()

    model, flat, opt = build_model(wl, dev, overlap=not args.no_overlap)
    autocast = (lambda: torch.autocast("cuda", dtype=torch.bfloat16)) if wl["dtype"] == "bf16" else \
               (lambda: torch.autocast("cuda", enabled=False))

    # per-rank scene (seed = 1000*config + scene index, SURVEY §8d), kept in pinned host memory
    scene = make_scene(wl, 1000 * wl["cfg_id"] + rank)
    host = {k: torch.from_numpy(np.ascontiguousarray(v)).pin_memory() for k, v in scene.items()}
    h2d_bytes = sum(t.numel() * t.element_size() for t in host.values())
    resident = {k: v.to(dev) for k, v in host.items()}
    shape = (torch.from_numpy(scene["grid_coord"]).max(0).values + 96).tolist()
    loss_host = torch.zeros(1).pin_memory()

    def step(inputs: dict) -> dict:
        data = dict(inputs)
        data["sparse_shape"] = shape
        opt.zero_grad()                     # the flat gradient buffer is zeroed, views stay attached
        with autocast():
            out = model(data)
        out["loss"].backward()              # gradient slices are all-reduced from hooks while this runs (N > 1)
        flat.all_reduce_mean()
        opt.step()
        return {k: v.detach() for k, v in out.items()}

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed_loop(from_host: bool, profile: bool):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        if from_host:
            # two untimed steps of THIS path first: the per-step input tensors are new allocations, and the caching
            # allocator's first blocks for them are cudaMallocs (device-synchronising; slower still with NCCL peer
            # mappings alive), which otherwise land in the first timed steps (r2o: c3 at N = 2, 43.8 vs 37.7 ms/step)
            for _ in range(2):
                step({k: v.to(dev, non_blocking=True) for k, v in host.items()})
        # the host enqueues ~1000 launches per step and is within 20 % of the device time: a generation-2 garbage collection
        # inside the K steps (tens of ms) shows up as +2 ms/step (r2y: 30.2 vs 27.9 ms in two runs of the same binary), so
        # collect before and keep the collector off for the timed region, as training loops that manage GC themselves do
        gc.collect()
        gc.disable()
        barrier()
        l0 = lib.pv2_launch_count()
        if profile:
            _lib.PROFILE.start(["pv2_spconv_gather_gemm", "pv2_spconv_wgrad"])
        e0.record()
        for _ in range(args.steps):
            if from_host:
                inputs = {k: v.to(dev, non_blocking=True) for k, v in host.items()}
                out = step(inputs)
                loss_host.copy_(out["loss"].reshape(1), non_blocking=True)
            else:
                out = step(resident)
        e1.record()
        barrier()
        gc.enable()
        _lib.PROFILE.stop()
        ms = e0.elapsed_time(e1)
        t = torch.tensor([ms], device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return t.item(), lib.pv2_launch_count() - l0, out

    log(f"model + scene ready on rank {rank}/{world}: {wl['voxels']} voxels, {wl['rays']} rays")
    # The clock sampler is started BEFORE the warm-up: nvidia-smi's start-up (fork + NVML attaching to the device)
    # stalls kernel launches for a few hundred ms, which used to land inside the first timed loop (r2l: 34.9 ms/step
    # device-resident vs 27.2 ms/step host-fed in the same run); its steady 200 ms polling does not.
    clocks = ClockSampler(local_rank)
    if rank == 0 and not args.profile_step:
        clocks.start()
    for _ in range(max(args.warmup, 3)):
        step(resident)
    torch.cuda.synchronize()
    log("warm-up done")
    if args.profile_step:
        # for `ncu --profile-from-start off`: exactly one warmed-up step inside cudaProfilerStart/Stop, no timing
        torch.cuda.profiler.start()
        step(resident)
        torch.cuda.synchronize()
        torch.cuda.profiler.stop()
        return
    if rank == 0:
        clocks.wait_first_sample()
    ms_dev, launches, last_out = timed_loop(from_host=False, profile=False)       # `value`: un-instrumented
    log(f"device-resident loop: {ms_dev / args.steps:.2f} ms/step")
    last_loss = float(last_out["loss"])
    if args.dump_outputs and rank == 0:
        # before the two loops below move the parameters on
        dump_outputs(args.dump_outputs, last_out, flat)
        log(f"outputs of the last device-resident step written to {args.dump_outputs}")
    ms_e2e, _, _ = timed_loop(from_host=True, profile=False)
    log(f"host-fed loop: {ms_e2e / args.steps:.2f} ms/step")
    clk = clocks.stop() if rank == 0 else None
    ms_prof, _, _ = timed_loop(from_host=False, profile=True)                     # per-kernel events: roofline only
    prof = _lib.PROFILE.summary()
    log(f"instrumented loop: {ms_prof / args.steps:.2f} ms/step")

    rays_per_step = wl["rays"] * world
    value = rays_per_step * args.steps / (ms_dev * 1e-3)
    e2e = rays_per_step * args.steps / (ms_e2e * 1e-3)

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        threads = host_threads()
        log(f"cpu baseline on {threads} threads ({os.cpu_count()} cores) ...")
        cal = cpu_oracle_step(wl, 0.05, threads)
        frac = min(1.0, max(0.05, 0.05 * 20.0 / max(cal["sample_s"], 1e-3)))        # ~20 s of CPU work
        t = cpu_oracle_step(wl, frac, threads)
        log(f"cpu baseline done: {t}")
        cpu = {"value": wl["rays"] / t["full_step_s"], "unit": "rays/s", "cores": threads, "kind": "port",
               "sample": f"{frac:.3f} of the step ({t['voxels']} voxels, {t['rays']} rays, same fraction of the dense "
                         f"grid): oracle SpUNet + densify + projection + NeuS fwd+bwd + SGD measured {t['sample_s']:.1f} s, "
                         f"extrapolated linearly x{1 / frac:.1f}; the 5 % calibration sample extrapolates to "
                         f"{wl['rays'] / cal['full_step_s']:.1f} rays/s",
               "stages_s": t["stages"]}
    if rank == 0:
        peaks = measured_peaks()
        gg = prof.get("pv2_spconv_gather_gemm", dict(calls=0, ms=0.0, bytes=0))
        achieved = gg["bytes"] / max(gg["ms"], 1e-9) * 1e-6 if gg["calls"] else 0.0  # GB/s
        traffic = profiled_traffic("umma_gather_gemm")
        line = {
            "metric": "pretrain_rays_per_sec", "value": value, "unit": "rays/s", "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms_dev / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": wl["dtype"], "data": "synthetic",
            "config": config_dict(wl, world),
            "scenes_per_sec": world * args.steps / (ms_dev * 1e-3),
            "voxels_per_sec": wl["voxels"] * world * args.steps / (ms_dev * 1e-3),
            "e2e": {"value": e2e, "unit": "rays/s", "h2d_bytes_per_step": h2d_bytes, "d2h_bytes_per_step": 4,
                    "ms_per_step": ms_e2e / args.steps},
            "gpu_launches": int(launches),
            "roofline": {"kernel": "pv2_spconv_gather_gemm (fwd + dgrad, all layers)", "bound": "hbm",
                         "achieved": achieved, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                         "frac": achieved / peaks["hbm_gbs"],
                         "traffic": traffic["bytes_per_launch"] if traffic else None,
                         "traffic_source": traffic["source"] if traffic else None,
                         "algorithmic_bytes_per_launch": gg["bytes"] / max(gg["calls"], 1),
                         "peak_source": peaks["source"],
                         "launches": gg["calls"], "kernel_ms_per_step": gg["ms"] / args.steps,
                         "share_of_step": gg["ms"] / max(ms_prof, 1e-9),
                         "timed_in": "separate instrumented loop (CUDA events around each C-ABI call)"},
            "kernel_ms_per_step": {k: v["ms"] / args.steps for k, v in prof.items()},
            "instrumented_ms_per_step": ms_prof / args.steps,
            "cpu_baseline": cpu, "clocks": clk, "loss": last_loss,
        }
        if nccl_log is not None:
            line["nccl"] = nccl_summary(os.path.join(nccl_log, "*.log"))
            line["nccl"]["overlap"] = not args.no_overlap
            if os.environ.get("PV2_NCCL_LOG_COPY"):      # dev switch: keep the raw per-rank NCCL logs
                import shutil
                shutil.copytree(nccl_log, os.environ["PV2_NCCL_LOG_COPY"], dirs_exist_ok=True)
            log("nccl: " + json.dumps(line["nccl"]))
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c2", choices=sorted(WORKLOADS))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--projection", default="simple", choices=["simple", "unet3d"],
                    help="indoor workloads: dense projection network. simple = SimpleConv3D-v1m1 (default, the step the "
                         "round-1 numbers and the CPU arm are quoted on); unet3d = UNet3D-v1m2, the ScanNet config's own "
                         "(configs/scannet/pretrain-ponder-spunet-v1m1-0-base.py:26-30; cuDNN, GPU arm only)")
    ap.add_argument("--no-overlap", action="store_true",
                    help="N > 1: one all-reduce of the whole flat gradient buffer after backward instead of chunked "
                         "all-reduces overlapped with it (A/B switch)")
    ap.add_argument("--profile-step", action="store_true",
                    help="run one warmed-up step inside cudaProfilerStart/Stop and exit (for ncu --profile-from-start off)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the outputs of the last timed device-resident step to DIR/<name>.npy (float32)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl == "reference" or args.profile_step):
        ap.error("--dump-outputs needs the timed loops of --impl ours (not --profile-step)")
    wl = dict(WORKLOADS[args.workload])
    if args.projection == "unet3d":
        if wl["outdoor"] or args.impl == "reference":
            raise SystemExit("--projection unet3d: indoor workloads, GPU arm only")
        wl["projection"] = "UNet3D-v1m2"
        wl["name"] += ", UNet3D-v1m2 projection"
        args.no_cpu_baseline = True
    if args.impl == "reference":
        run_reference(args, wl)
    else:
        run_ours(args, wl)


if __name__ == "__main__":
    main()

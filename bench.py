#!/usr/bin/env python
"""bench.py — benchmark of the rasterizer / fusion hot path on the BASELINE.json configs (DESIGN.md §7).

  --config K3 (default)  configs[2], the one the metric is quoted on: 1 M Gaussians x 256-ch features, 1920x1080,
                         one view per rank per step, forward + backward (+ gradient exchange at N > 1)
  --config K2            configs[1]: 1 M Gaussians, RGB + median depth (rgbd path), 1920x1080, forward only
  --config K4            configs[3]: 3 M Gaussians x 512 ch, 1296x968, a batch of 32 views per step sharded over the
                         ranks through the batched native path, ONE gradient exchange per step (strong scaling)
  --config K5            configs[4]: fusion of 300 views x 512-ch fp16 maps at 640x480 onto 2 M Gaussians per step,
                         views strided over the ranks, one all-reduce of the (P, C) sums (strong scaling)

One JSON line on stdout (rank 0):
  value          Mviews/s, whole job, inputs resident in HBM, CUDA-event timed, max over ranks
  e2e            the same metric through the public Python API with HOST buffers (pinned H2D inputs, D2H result)
  roofline       dominant kernel: algorithmic bytes / CUDA-event duration against the measured HBM peak
  cpu_baseline   the CPU port of the reference algorithm on a bounded sample (rank 0, N = 1)
  --impl reference   times that CPU port alone (rank 0 only), same JSON contract
  --dump-outputs DIR   after the timed steps, rank 0 writes what the device-resident timed path computed in its last
                       step (images, radii, parameter gradients / fused features) to DIR/<name>.npy; see dump_outputs()
"""
from __future__ import annotations

import argparse
import hashlib
import json
import math
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

NVIEWS = 8            # cycling views of K2 / K3
NUM_CLASSES = 20
METRIC = "Mviews/s + HBM GB/s, 1M Gaussians, 256-ch features, 1080p, fwd+bwd"

CONFIGS = {
    "K2": dict(P=1_000_000, C=3, W=1920, H=1080, kind="blob", views_per_step=None,
               metric="Mviews/s + HBM GB/s, 1M Gaussians, RGB + depth (rgbd path), 1080p, fwd",
               workload="K2: 1M Gaussians, SH RGB + median depth, 1920x1080, 1 view/rank/step, fwd only (configs[1])"),
    "K3": dict(P=1_000_000, C=256, W=1920, H=1080, kind="blob", views_per_step=None, metric=METRIC,
               workload="K3: 1M Gaussians x 256-ch features, 1920x1080, 1 view/step, fwd+bwd (configs[2])"),
    "K4": dict(P=3_000_000, C=512, W=1296, H=968, kind="room", views_per_step=32,
               metric="Mviews/s + HBM GB/s, 3M Gaussians, 512-ch features, 1296x968, batch of 32 views, fwd+bwd + grad exchange",
               workload="K4: 3M Gaussians x 512-ch features, 1296x968, 32 views/step sharded over the ranks (batched "
                        "native path), fwd+bwd, one gradient exchange per step (configs[3])"),
    "K5": dict(P=2_000_000, C=512, W=640, H=480, kind="room", views_per_step=300,
               metric="Mviews/s + HBM GB/s, fusion of 512-ch fp16 maps at 640x480 onto 2M Gaussians, 300 views",
               workload="K5: fusion 300 views x 512-ch fp16 @ 640x480 -> 2M Gaussians per step, views strided over "
                        "the ranks, one all-reduce of the sums (configs[4])"),
}


def env_int(name, default):
    try:
        return int(os.environ.get(name, default))
    except ValueError:
        return default


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        try:
            return float(json.load(open(path))["hbm_gbs"]), "MEASURED_PEAKS.json (of measured)"
        except Exception:
            pass
    return 6650.0, "B200_PROFILING.md fallback (of fallback)"


def build_info():
    """Identity of the library that is being measured: the hash baked into the .so at build time against the hash
    of the sources next to it (a stale prebuilt libsgb200.so must not be benchmarked as the current code)."""
    import importlib.util
    from semantic_gaussians_b200 import _lib
    spec = importlib.util.spec_from_file_location("sgb200_build", os.path.join(ROOT, "semantic-gaussians_b200", "build.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    src = mod.source_hash()
    baked = _lib.build_id()
    try:
        h = hashlib.sha256(open(_lib.LIB_PATH, "rb").read()).hexdigest()[:16]
    except Exception:
        h = None
    return {"library": baked, "source_sha256_16": src, "lib_sha256_16": h, "matches_sources": baked.endswith(src)}


# The contract is ONE JSON line on stdout.  Libraries write there too (NCCL prints "NCCL version ..." to fd 1 on some
# boxes), so main() points fd 1 at stderr for the whole run and the result goes to a private duplicate of the real stdout.
_RESULT_OUT = None


def claim_stdout():
    global _RESULT_OUT
    sys.stdout.flush()
    _RESULT_OUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)


def emit_line(line):
    out = _RESULT_OUT or sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


def traffic_for(kernel, src_hash):
    """Measured DRAM bytes per launch (ncu --set full), only when the capture was taken from THIS source tree."""
    tpath = os.path.join(ROOT, "profiles", "dram_traffic.json")
    try:
        t = json.load(open(tpath))
    except Exception:
        return None, "no profiles/dram_traffic.json"
    if t.get("_src_sha256_16") != src_hash:
        return None, (f"profiles/dram_traffic.json was captured from sources {t.get('_src_sha256_16')}, "
                      f"not {src_hash}: stale, ignored")
    return t.get(kernel), t.get("_source")


# ------------------------------------------------------------------------------ clocks sampler
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu = gpu_index
        self.proc = None
        self.path = None

    def start(self):
        try:
            fd, self.path = tempfile.mkstemp(prefix="clocks_", suffix=".csv")
            os.close(fd)
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100", "-i",
                 str(self.gpu)], stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self) -> dict:
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.proc is None:
            return out
        try:
            self.proc.terminate()
            self.proc.wait(timeout=5)
        except Exception:
            pass
        sm, mx, reasons = [], [], set()
        try:
            for line in open(self.path):
                f = [x.strip() for x in line.split(",")]
                if len(f) < 9:
                    continue
                try:
                    sm.append(float(f[1]))
                    mx.append(float(f[2]))
                except ValueError:
                    continue
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"),
                                   f[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            os.unlink(self.path)
        except Exception:
            pass
        if sm:
            out.update(sm_mhz=float(np.median(sm)), sm_max_mhz=float(max(mx)), reasons=sorted(reasons),
                       samples=len(sm))
        return out


# ------------------------------------------------------------------------------ CPU arms
def host_threads():
    n = os.cpu_count() or 1
    try:
        n = len(os.sched_getaffinity(0))
    except Exception:
        pass
    return n


def cpu_raster_sample(cfg, scene, cam, band_tile_rows=1, backward=True, want_depth=False):
    """One bounded sample of a rasterizer config on the host cores with the CPU oracle (a port of the reference's
    algorithm — the reference has no CPU rasterizer): full per-Gaussian preprocess, then binning + blend forward
    (+ backward) of THREE bands of tile rows (top quarter, middle, bottom quarter of the image), each scaled to the
    full view.  Returns the per-band estimates so the spread is visible."""
    from oracle import oracle as orc
    threads = orc.set_num_threads(host_threads())      # torchrun exports OMP_NUM_THREADS=1: set it explicitly
    W, H, C = cam.image_width, cam.image_height, cfg["C"]
    use_feat = C > 3
    gy = (H + 15) // 16
    cd = orc.cam_dict(cam)
    bg = np.zeros(C, np.float32)
    t0 = time.perf_counter()
    pre = orc.preprocess(scene.xyz, scene.scales, scene.rotations, scene.opacity, cd["viewmatrix"], cd["projmatrix"],
                         cd["campos"], W, H, cd["tanfovx"], cd["tanfovy"],
                         shs=None if use_feat else scene.shs, colors_precomp=scene.features if use_feat else None)
    t_pre = time.perf_counter() - t0
    colors = scene.features if use_feat else pre["rgb"]
    bands, est = [], []
    for frac_y in (0.25, 0.5, 0.75):
        r0 = min(gy - band_tile_rows, max(0, int(gy * frac_y) - band_tile_rows // 2))
        r1 = min(gy, r0 + band_tile_rows)
        rows = (r0 * 16, min(H, r1 * 16))
        t1 = time.perf_counter()
        b = orc.bin_instances(pre, W, H, tile_rows=(r0, r1))
        f = orc.render_forward(pre, b, colors, bg, W, H, rows=rows, want_depth=True) if want_depth else \
            orc.render_forward(pre, b, colors, bg, W, H, rows=rows)
        if backward:
            fwd = dict(pre=pre, bin=b, colors=colors, **f)
            dL = np.full((C, H, W), 1.0 / (H * W), np.float32)
            orc.backward(fwd, orc.scene_dict(scene), cd, W, H, bg, dL, features=scene.features if use_feat else None,
                         rows=rows)
        t2 = time.perf_counter()
        frac = (rows[1] - rows[0]) / H
        bands.append(dict(rows=list(rows), seconds=t2 - t1, frac=frac))
        est.append((t2 - t1) / frac)
    full = t_pre + float(np.mean(est))
    return dict(seconds_sample=t_pre + sum(b["seconds"] for b in bands), seconds_full_view_est=full,
                preprocess_s=t_pre, band_full_view_est_s=[t_pre + e for e in est], bands=bands, threads=threads)


def cpu_fusion_sample(cfg, scene, cams, nviews=2):
    """The reference's own fusion step on the host: numpy compute_mapping (single-threaded by construction,
    dataset/fusion_utils.py:30-78) + the torch-CPU gather / accumulate of fusion.py:136-144, per view."""
    import torch
    from oracle import fusion_oracle as fo
    torch.set_num_threads(host_threads())
    P, C, w, h = cfg["P"], cfg["C"], cfg["W"], cfg["H"]
    rng = np.random.default_rng(0)
    fm = torch.from_numpy(rng.standard_normal((C, h, w)).astype(np.float16))
    depth = np.full((h, w), 2.5, np.float32)
    fs = torch.zeros((P, C))
    cnt = torch.zeros(P)
    t_map = t_acc = 0.0
    for i in range(nviews):
        K = fo.rescale_intrinsics(cams[i].intrinsics(), [w, h])
        t0 = time.perf_counter()
        m = fo.compute_mapping(cams[i].world_view_transform, scene.xyz, [w, h], K, 0.25, 10, depth)
        t1 = time.perf_counter()
        mt = torch.from_numpy(m)
        mask = mt[:, 2] != 0
        g = fm[:, mt[:, 0], mt[:, 1]].permute(1, 0)          # fusion.py:139-140
        cnt[mask] += 1
        fs[mask] += g[mask]
        t2 = time.perf_counter()
        t_map += t1 - t0
        t_acc += t2 - t1
    return dict(seconds_sample=t_map + t_acc, seconds_per_view=(t_map + t_acc) / nviews, mapping_s=t_map / nviews,
                accumulate_s=t_acc / nviews, threads=torch.get_num_threads(), nviews=nviews)


def cpu_torch_preprocess_leg(P=1_000_000):
    """north_star: the reference's pure-PyTorch preprocess alternatives on the host cores — eval_sh
    (utils/sh_utils.py:56-115 via pipe.convert_shs_python, model/renderer.py:100-105) and
    build_covariance_from_scaling_rotation (model/gaussian_model.py:34-38 via pipe.compute_cov3d_python,
    renderer.py:82-83) — at 1 M Gaussians with torch-CPU (this repo's device-agnostic restatements of the two
    functions; the reference's own hard-code device='cuda', utils/general_utils.py:67,87,107)."""
    import torch
    from semantic_gaussians_b200.gaussian_model import build_scaling_rotation, strip_symmetric
    from semantic_gaussians_b200.sh_utils import eval_sh
    torch.set_num_threads(host_threads())
    g = torch.Generator().manual_seed(0)
    xyz = torch.rand((P, 3), generator=g) * 2.6 - 1.3
    shs = torch.randn((P, 16, 3), generator=g) * 0.1
    scales = torch.rand((P, 3), generator=g) * 0.05 + 0.002
    rot = torch.nn.functional.normalize(torch.randn((P, 4), generator=g))
    campos = torch.tensor([3.0, 0.0, 0.4])

    def sh_leg():
        shs_view = shs.transpose(1, 2).view(-1, 3, 16)
        dir_pp = xyz - campos.repeat(P, 1)
        dir_pp = dir_pp / dir_pp.norm(dim=1, keepdim=True)
        return torch.clamp_min(eval_sh(3, shs_view, dir_pp) + 0.5, 0.0)

    def cov_leg():
        L = build_scaling_rotation(scales, rot)
        return strip_symmetric(L @ L.transpose(1, 2))
    out = {}
    for name, fn in (("eval_sh_ms", sh_leg), ("build_covariance_ms", cov_leg)):
        fn()
        t0 = time.perf_counter()
        for _ in range(3):
            fn()
        out[name] = 1e3 * (time.perf_counter() - t0) / 3
    out.update(P=P, threads=torch.get_num_threads(), kind="torch-CPU, port of utils/sh_utils.py:56-115 and "
               "model/gaussian_model.py:34-38 (reference versions hard-code device='cuda')")
    return out


def run_cpu_reference(args, rank, world):
    """--impl reference: the CPU port of the reference algorithm for the selected config on all host threads
    (rank 0 only; the other ranks exit without work)."""
    if rank != 0:
        return
    from semantic_gaussians_b200.scene_synth import make_scene, orbit_cameras, room_cameras
    cfg = CONFIGS[args.config]
    P, C, W, H = cfg["P"], cfg["C"], cfg["W"], cfg["H"]
    line_cfg = {"workload": cfg["workload"], "P": P, "C": C, "W": W, "H": H,
                "note": "CPU port of the reference algorithm (oracle/raster_oracle.c, oracle/fusion_oracle.py); the "
                        "reference itself has no CPU rasterizer"}
    if args.config == "K5":
        scene = make_scene(P, seed=0, kind="room")
        cams = room_cameras(8, W, H)
        for _ in range(min(args.warmup, 1)):
            cpu_fusion_sample(cfg, scene, cams, 1)
        t0 = time.perf_counter()
        per_view, last = [], None
        for _ in range(args.steps):
            last = cpu_fusion_sample(cfg, scene, cams, 1)
            per_view.append(last["seconds_per_view"])
        wall = time.perf_counter() - t0
        sec_per_step = float(np.mean(per_view)) * cfg["views_per_step"]
        views_per_s = cfg["views_per_step"] / sec_per_step
        sample = (f"per step: 1 fused view of the {cfg['views_per_step']} (numpy compute_mapping {last['mapping_s']:.2f} s on 1 core "
                  f"+ torch-CPU gather/accumulate {last['accumulate_s']:.2f} s on {last['threads']} threads), scaled to the scene")
        cores, spread = last["threads"], [min(per_view), max(per_view)]
    else:
        scene = make_scene(P, seed=0, kind=cfg["kind"], sh=C == 3, channels=C if C > 3 else 0)
        cams = (orbit_cameras if cfg["kind"] == "blob" else room_cameras)(NVIEWS, W, H)
        backward = args.config != "K2"
        for i in range(min(args.warmup, 1)):
            cpu_raster_sample(cfg, scene, cams[i % NVIEWS], backward=backward, want_depth=args.config == "K2")
        t0 = time.perf_counter()
        ests, last = [], None
        for i in range(args.steps):
            last = cpu_raster_sample(cfg, scene, cams[i % NVIEWS], backward=backward, want_depth=args.config == "K2")
            ests.append(last["seconds_full_view_est"])
        wall = time.perf_counter() - t0
        vps = cfg["views_per_step"] or 1
        sec_per_step = float(np.mean(ests)) * vps
        views_per_s = vps / sec_per_step
        pct = 100 * sum(b["frac"] for b in last["bands"])
        sample = (f"per step: full preprocess of {P} Gaussians + binning/blend {'fwd+bwd' if backward else 'fwd'} of 3 bands of "
                  f"16 image rows (top quarter / middle / bottom quarter, {pct:.1f}% of the pixels), each scaled to the "
                  f"full view; band estimates of the last step {['%.1f s' % b for b in last['band_full_view_est_s']]}")
        cores, spread = last["threads"], [float(min(ests)), float(max(ests))]
    value = views_per_s * 1e-6
    line_cfg["wall_s"] = wall
    line_cfg["full_view_estimate_spread_s"] = spread
    line = {
        "impl": "reference", "metric": cfg["metric"], "value": value, "unit": "Mviews/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * sec_per_step,
        "higher_is_better": True, "scaling": "weak" if cfg["views_per_step"] is None else "strong",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": line_cfg,
        "cpu_baseline": {"value": value, "unit": "Mviews/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": "Mviews/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit_line(line)


# ------------------------------------------------------------------------------ roofline helpers
def algorithmic_bytes(P, P_vis, R, C, W, H):
    """SURVEY.md §8(d) / BASELINE.md §4 compulsory traffic, split by kernel (DESIGN.md §3)."""
    px = W * H
    # per kernel: every input read once, every output written once
    alpha = 4 * R + 32 * P_vis + 8 * px                       # ids + splat records in, final_T / n_contrib out
    fwd_blend = 4 * C * P_vis + 4 * C * px + 4 * px           # features in, image out (+ final_T in)
    chain = 4 * C * px + 4 * C * P_vis + 32 * P_vis + 4 * px + 28 * P_vis   # dL/dout + features in, 7 geometry grads out
    dfeat = 4 * C * px + 4 * C * P_vis                        # dL/dout in, dL/dfeature out
    fwd_total = 44 * P + 4 * C * P_vis + 4 * C * px + 8 * px + 24 * R
    bwd_total = 4 * C * px + 8 * C * P_vis + 4 * R + 8 * px + 80 * P + 44 * P
    # RGB(-D) path (C <= 4): one fused blend kernel; the tile sort moves (16-bit key + 32-bit id) once in, once out
    rgb_blend = 4 * R + 32 * P_vis + 4 * (C + 1) * px + 8 * px
    tile_sort = 12 * R
    return dict(alpha_pass=alpha, blend_fwd=fwd_blend if C > 4 else rgb_blend, blend_bwd=chain, dfeature=dfeat,
                tile_sort=tile_sort, fwd=fwd_total + (4 * px if C <= 4 else 0), bwd=bwd_total)


FMA_PEAK_TFLOPS = 70.5   # dependent-free FFMA loop on this pool's B200s (tools/microbench.cu, BASELINE.md §6)


def fma_roofline(C, blended_pairs, per_stage):
    """fp32 CUDA-core roof of the three C-wide contractions (DESIGN.md §3): achieved = algorithmic flops
    (2*C per blended pair and contraction, zero-weight padding not counted) / stage time."""
    out = {"peak_tflops": FMA_PEAK_TFLOPS, "peak_source": "measured FFMA micro-benchmark (tools/microbench.cu)",
           "algorithmic_flops_per_contraction": 2 * C * blended_pairs, "kernels": {}}
    for k in ("blend_fwd", "blend_bwd", "dfeature"):
        ms = per_stage.get(k)
        if ms:
            tf = 2 * C * blended_pairs / (ms * 1e-3) * 1e-12
            out["kernels"][k] = {"ms": ms, "achieved_tflops": tf, "frac": tf / FMA_PEAK_TFLOPS}
    tot = sum(per_stage.get(k, 0.0) for k in ("blend_fwd", "blend_bwd", "dfeature", "alpha_pass"))
    if tot:
        out["achieved_tflops"] = 6 * C * blended_pairs / (tot * 1e-3) * 1e-12
        out["frac"] = out["achieved_tflops"] / FMA_PEAK_TFLOPS
    return out


# ------------------------------------------------------------------------------ GPU arm: shared pieces
DUMP_BYTES = 64 << 20


def dump_outputs(path, arrays):
    """Write each output tensor as path/<name>.npy: float32 when it is floating point, float64 otherwise (exact for
    the integer and boolean outputs).  Together the files stay within DUMP_BYTES: an output with more elements than
    its share is written as the flat values at a fixed seeded sample of positions (the same positions for every
    output of that size), so two builds run with the same arguments can be compared output for output."""
    import torch
    os.makedirs(path, exist_ok=True)
    cap = DUMP_BYTES // 8 // max(len(arrays), 1)
    for name, t in arrays.items():
        t = t.detach()
        if t.numel() > cap:
            idx = np.unique(np.random.default_rng(t.numel()).integers(0, t.numel(), cap))
            t = t.reshape(-1)[torch.as_tensor(idx, device=t.device)]
        t = t.to(torch.float32 if t.is_floating_point() else torch.float64)
        np.save(os.path.join(path, f"{name}.npy"), t.cpu().numpy())


def render_outputs(out, prefix=""):
    """The tensors a render()/render_chn() call hands its caller (viewspace_points through its gradient)."""
    d = {prefix + k: v for k, v in out.items() if k != "viewspace_points"}
    if out["viewspace_points"].grad is not None:
        d[prefix + "viewspace_points_grad"] = out["viewspace_points"].grad
    return d


class Pipe:
    convert_shs_python = False
    compute_cov3d_python = False
    debug = False


class Cam:
    pass


class Harness:
    """Process-group setup, device timing (barrier + synchronize on both sides, CUDA events, MAX over ranks)."""

    def __init__(self, args, rank, world, local_rank):
        import torch
        import torch.distributed as dist
        from semantic_gaussians_b200 import _lib
        if not torch.cuda.is_available():
            raise SystemExit("bench.py needs a CUDA device: the rasterizer has no CPU path")
        self.torch, self.dist, self._lib = torch, dist, _lib
        self.args, self.rank, self.world, self.local_rank = args, rank, world, local_rank
        torch.cuda.set_device(local_rank)
        self.dev = torch.device("cuda", local_rank)
        if world > 1:
            from semantic_gaussians_b200.distributed import nccl_overlap_options
            dist.init_process_group("nccl", device_id=self.dev, pg_options=nccl_overlap_options())
        _lib.load()
        self.stream = torch.cuda.current_stream(self.dev).cuda_stream
        self.ctx = _lib.ctx_for(local_rank, self.stream)
        self.warmup = max(args.warmup, 3)

    def dev_cam(self, c):
        torch = self.torch
        v = Cam()
        v.image_width, v.image_height, v.FoVx, v.FoVy = c.image_width, c.image_height, c.FoVx, c.FoVy
        v.world_view_transform = torch.as_tensor(c.world_view_transform, device=self.dev)
        v.full_proj_transform = torch.as_tensor(c.full_proj_transform, device=self.dev)
        v.camera_center = torch.as_tensor(c.camera_center, device=self.dev)
        return v

    def timed(self, fn, steps, finish=None):
        """(max-over-ranks ms, this rank's ms) for `steps` calls of fn(i)."""
        torch, dist = self.torch, self.dist
        if self.world > 1:
            dist.barrier()
        torch.cuda.synchronize(self.dev)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(steps):
            fn(i)
        if finish is not None:
            finish(steps - 1)      # the last step's result is read inside the timed region
        e1.record()
        torch.cuda.synchronize(self.dev)
        if self.world > 1:
            dist.barrier()
        mine = float(e0.elapsed_time(e1))
        ms = torch.tensor([mine], device=self.dev)
        if self.world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item()), mine

    def gather_floats(self, x):
        """list over ranks of a python float."""
        if self.world == 1:
            return [float(x)]
        t = self.torch.tensor([float(x)], device=self.dev)
        out = [self.torch.zeros_like(t) for _ in range(self.world)]
        self.dist.all_gather(out, t)
        return [float(o.item()) for o in out]

    def profiled(self, fn, steps, finish=None):
        """timed() with library stage tracing and (rank 0) clock sampling around it."""
        _lib = self._lib
        l0 = _lib.launch_count(self.ctx)
        _lib.profile_enable(self.ctx, True)
        sampler = ClockSampler(self.local_rank)
        if self.rank == 0:
            sampler.start()
        ms, mine = self.timed(fn, steps, finish)
        clocks = sampler.stop() if self.rank == 0 else {}
        stages = _lib.profile_read(self.ctx)
        _lib.profile_enable(self.ctx, False)
        l1 = _lib.launch_count(self.ctx)
        per_stage = {k: (v[0] / max(v[1], 1)) for k, v in stages.items() if v[1] > 0}
        counts = {k: v[1] for k, v in stages.items() if v[1] > 0}
        return ms, mine, per_stage, counts, clocks, (int(l1[0] - l0[0]), int(l1[1] - l0[1]))

    def finish(self):
        if self.world > 1:
            self.dist.destroy_process_group()

    def base_line(self, cfg, value, ms_per_step, steps, scaling):
        return {
            "metric": cfg["metric"], "value": value, "unit": "Mviews/s", "n_gpus": self.world, "steps": steps,
            "warmup": self.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": scaling,
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        }


def view_stats(h, cfg, pc, feats_or_none, cam, bg):
    """P_vis, R, mean list lengths of one view (reported with every timing, BASELINE.md §3)."""
    torch, _lib = h.torch, h._lib
    from semantic_gaussians_b200.rasterizer import _C_chn, _C_rgbd
    P, C, W, H = cfg["P"], cfg["C"], cfg["W"], cfg["H"]
    tiles = ((W + 15) // 16) * ((H + 15) // 16)
    e = torch.Tensor([])
    with torch.no_grad():
        if C > 3:
            Rn, _, radii, _, _, img = _C_chn.rasterize_gaussians(
                bg, pc.get_xyz, feats_or_none.detach(), pc.get_opacity, pc.get_scaling, pc.get_rotation, 1.0, e,
                cam.world_view_transform, cam.full_proj_transform, math.tan(cam.FoVx / 2), math.tan(cam.FoVy / 2), H, W,
                e, 0, cam.camera_center, False, False, C)
        else:
            Rn, _, radii, _, _, img, _ = _C_rgbd.rasterize_gaussians(
                bg, pc.get_xyz, e, pc.get_opacity, pc.get_scaling, pc.get_rotation, 1.0, e, cam.world_view_transform,
                cam.full_proj_transform, math.tan(cam.FoVx / 2), math.tan(cam.FoVy / 2), H, W, pc.get_features,
                pc.active_sh_degree, cam.camera_center, False)
        P_vis = int((radii > 0).sum())
        nc = torch.zeros(H * W, dtype=torch.int32, device=h.dev)
        _lib.load().sgb_state_field(b"n_contrib", P, Rn, W, H, None, None, img.data_ptr(), nc.data_ptr(), h.stream)
        out = {"P_vis": P_vis, "R": int(Rn), "gaussians_per_tile_mean": Rn / tiles,
               "n_contrib_mean": float(nc.float().mean())}
        if C > 3:
            out["blended_pairs"] = _lib.view_stat(h.ctx, 0)
            out["n_blended_mean"] = out["blended_pairs"] / (W * H)
            out["tile_entries_mean"] = _lib.view_stat(h.ctx, 1) * 16 / tiles
    return out


def roofline_block(per_stage, ab, candidates, src_hash, note=None, config="K3"):
    peak, peak_src = measured_peaks()
    dom = max(candidates, key=lambda k: per_stage.get(k, 0.0))
    dom_ms = per_stage.get(dom, float("nan"))
    achieved = ab[dom] / (dom_ms * 1e-3) * 1e-9
    traffic, tsrc = traffic_for(f"{config}.{dom}", src_hash)   # captures are per config: K2 and K3 blend different kernels
    r = {"bound": "hbm", "kernel": dom, "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
         "traffic": traffic, "traffic_source": tsrc, "algorithmic_bytes": ab[dom], "kernel_ms": dom_ms,
         "peak_source": peak_src}
    if note:
        r["note"] = note
    return r


# ------------------------------------------------------------------------------ K3 (default) and K2
def run_k3(args, rank, world, local_rank):
    cfg = CONFIGS["K3"]
    h = Harness(args, rank, world, local_rank)
    torch, dist, _lib, dev = h.torch, h.dist, h._lib, h.dev
    from semantic_gaussians_b200.gaussian_model import GaussianModel
    from semantic_gaussians_b200.renderer import render_chn
    from semantic_gaussians_b200.scene_synth import make_scene, orbit_cameras
    from semantic_gaussians_b200.semantic import distill_loss_and_grad
    P, C, W, H = cfg["P"], cfg["C"], cfg["W"], cfg["H"]

    scene = make_scene(P, seed=0, channels=C)
    cams_np = orbit_cameras(NVIEWS, W, H)
    pc = GaussianModel.from_activated(scene.xyz, scene.scales, scene.rotations, scene.opacity, device=dev)
    pc.active_sh_degree = 0
    feats = torch.as_tensor(scene.features, device=dev).contiguous().requires_grad_(True)
    for t in (pc._xyz, pc._scaling, pc._rotation, pc._opacity):
        t.requires_grad_(True)
    params = [feats, pc._xyz, pc._scaling, pc._rotation, pc._opacity]
    bg = torch.zeros(C, device=dev)
    cams = [h.dev_cam(c) for c in cams_np]
    # host side of the e2e arm: pinned camera blocks (35 floats) and per-view label maps
    host_cam = [torch.from_numpy(np.concatenate([c.world_view_transform.ravel(), c.full_proj_transform.ravel(),
                                                 c.camera_center.ravel()]).astype(np.float32)).pin_memory()
                for c in cams_np]
    rng = np.random.default_rng(1234 + rank)
    host_labels = [torch.from_numpy(rng.integers(0, NUM_CLASSES, size=(H, W), dtype=np.int64)
                                    .astype(np.int32)).pin_memory() for _ in range(2)]
    # identical on every rank (explicit seeds: the multi-GPU parity check compares against a single-GPU sum)
    gen = torch.Generator(device=dev).manual_seed(20260924)
    class_emb = torch.nn.functional.normalize(torch.randn(NUM_CLASSES, C, device=dev, generator=gen), dim=1)
    dL_fixed = torch.randn((C, H, W), device=dev, generator=gen) / (H * W)

    def zero_grads():
        for p in params:
            p.grad = None

    overlap = None
    if world > 1:
        from semantic_gaussians_b200.distributed import OverlappedFeatureGradReduce
        overlap = OverlappedFeatureGradReduce(dev)        # dL/dfeature is final before the chain kernels run

    def allreduce_grads():
        if world == 1:
            return None
        overlap.start(feats.grad)                         # (P, C) fp32, 1 GB: reduced under the chain/geometry kernels
        small = torch.cat([p.grad.reshape(-1) for p in params[1:]])
        dist.all_reduce(small)
        overlap.finish()
        return small

    def view_of(i):
        # every rank walks through all NVIEWS views (offset by its rank): N = 1 and N = 8 average the same view set,
        # and at every step the `world` ranks render `world` DIFFERENT views
        return (i + rank) % NVIEWS

    last = {}

    def step_device(i, exchange=True, keep=False):
        out = render_chn(cams[view_of(i)], pc, Pipe, bg, num_channels=C, override_color=feats)
        if overlap is not None:
            overlap.arm(feats)
        out["render"].backward(dL_fixed)
        if exchange:
            allreduce_grads()
        if keep:
            last.update(render_outputs(out))
            last.update({f"{n}_grad": p.grad for n, p in zip(("features", "xyz", "scaling", "rotation", "opacity"),
                                                              params)})
        zero_grads()

    cam_dev = Cam()
    cam_dev.image_width, cam_dev.image_height = W, H
    cam_dev.FoVx, cam_dev.FoVy = cams_np[0].FoVx, cams_np[0].FoVy
    cam_buf = torch.empty(35, device=dev)
    label_buf = torch.empty((H, W), dtype=torch.int32, device=dev)
    # the loss is read back the way training loops do it: an asynchronous 8-byte copy into pinned memory each
    # step, consumed one step later (and the last one inside the timed region), so the host keeps launching
    loss_host = [torch.zeros(1, dtype=torch.float64).pin_memory() for _ in range(2)]
    loss_ev = [torch.cuda.Event() for _ in range(2)]
    e2e_losses = []

    def step_e2e(i):
        k = view_of(i)
        cam_buf.copy_(host_cam[k], non_blocking=True)                      # H2D 140 B
        label_buf.copy_(host_labels[i % 2], non_blocking=True)             # H2D 8.3 MB
        cam_dev.world_view_transform = cam_buf[0:16].view(4, 4)
        cam_dev.full_proj_transform = cam_buf[16:32].view(4, 4)
        cam_dev.camera_center = cam_buf[32:35]
        out = render_chn(cam_dev, pc, Pipe, bg, num_channels=C, override_color=feats)
        # open-vocabulary distillation loss  L = -mean <render[:, p], E[label(p)]>  and its gradient, one fused pass
        loss, dL = distill_loss_and_grad(out["render"], class_emb, label_buf)
        loss_host[i % 2].copy_(loss.reshape(1), non_blocking=True)            # D2H 8 B (float64 scalar)
        loss_ev[i % 2].record()
        if overlap is not None:
            overlap.arm(feats)
        out["render"].backward(dL)
        allreduce_grads()
        zero_grads()
        if i > 0:
            finish_e2e(i - 1)

    def finish_e2e(i):
        loss_ev[i % 2].synchronize()
        e2e_losses.append(float(loss_host[i % 2]))

    # ---- warm-up
    for i in range(h.warmup):
        step_device(i)
    torch.cuda.synchronize(dev)

    # ---- N > 1: the exchanged gradients must equal the single-GPU sum over the same views (parity on hardware)
    parity = None
    if world > 1:
        def grads_of(view_ids):
            zero_grads()
            for k in view_ids:
                render_chn(cams[k % NVIEWS], pc, Pipe, bg, num_channels=C, override_color=feats)["render"].backward(dL_fixed)
            g = [p.grad.detach().clone() for p in params]
            zero_grads()
            return g
        mine = grads_of([rank])
        for g in mine:
            dist.all_reduce(g)
        # the production exchange path (overlapped feature-gradient all-reduce + flat small message) as well
        out = render_chn(cams[rank % NVIEWS], pc, Pipe, bg, num_channels=C, override_color=feats)
        overlap.arm(feats)
        out["render"].backward(dL_fixed)
        small = allreduce_grads()
        prod = [feats.grad.detach().clone(), small.clone()]
        zero_grads()
        if rank == 0:
            single = grads_of(list(range(world)))
            names = ["features", "xyz", "scaling", "rotation", "opacity"]
            errs = {}
            for n, a, b in zip(names, mine, single):
                errs[n] = float((a - b).abs().max() / (b.abs().max() + 1e-30))
            errs["features_overlapped_path"] = float((prod[0] - single[0]).abs().max() / (single[0].abs().max() + 1e-30))
            flat_single = torch.cat([g.reshape(-1) for g in single[1:]])
            errs["small_flat_path"] = float((prod[1] - flat_single).abs().max() / (flat_single.abs().max() + 1e-30))
            # features: pure fp32 re-association of the cross-rank sum; geometry gradients: each side sums its per-tile
            # partials with red.global in scheduling order, so two runs of the SAME view already differ by ~1e-5
            parity = {"views": world, "max_rel_err": errs, "tolerance": 1e-4, "ok": all(v <= 1e-4 for v in errs.values()),
                      "what": "all-reduced gradients of N ranks x 1 view vs rank 0 rendering the same N views alone"}
            if not parity["ok"]:   # reported in the JSON line (never fatal: the line must still be printed)
                print(f"WARNING: multi-GPU gradient parity outside tolerance: {errs}", file=sys.stderr, flush=True)
            del single
        del mine, prod
        torch.cuda.empty_cache()

    # ---- per-view cost spread on rank 0 (separates view skew from exchange cost in the scaling numbers)
    view_ms = []
    if rank == 0 and not args.quick:
        for k in range(NVIEWS):
            def one(i, k=k):
                render_chn(cams[k], pc, Pipe, bg, num_channels=C, override_color=feats)["render"].backward(dL_fixed)
                zero_grads()
            one(0)
            torch.cuda.synchronize(dev)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            one(0)
            one(1)
            e1.record()
            torch.cuda.synchronize(dev)
            view_ms.append(e0.elapsed_time(e1) / 2)
    stats = view_stats(h, cfg, pc, feats, cams[rank % NVIEWS], bg)

    # ---- device-resident timed region (stage tracing + clock sampling), then the same without the exchange
    ms_dev, ms_mine, per_stage, _, clocks, launches = h.profiled(
        lambda i: step_device(i, keep=args.dump_outputs is not None and i == args.steps - 1), args.steps)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, last)
    last.clear()
    rank_ms = h.gather_floats(ms_mine / args.steps)
    ms_nocomm = None
    if world > 1:
        ms_nc, _ = h.timed(lambda i: step_device(i, exchange=False), args.steps)
        ms_nocomm = ms_nc / args.steps

    # ---- end-to-end arm through the public API with host buffers
    for i in range(2):
        step_e2e(i)
    finish_e2e(1)
    e2e_losses.clear()
    ms_e2e, _ = h.timed(step_e2e, args.steps, finish=finish_e2e)
    assert len(e2e_losses) == args.steps and all(math.isfinite(v) for v in e2e_losses)

    if rank != 0:
        h.finish()
        return

    views = args.steps * world
    value = views / (ms_dev * 1e-3) * 1e-6
    e2e_value = views / (ms_e2e * 1e-3) * 1e-6
    peak, _ = measured_peaks()
    ab = algorithmic_bytes(P, stats["P_vis"], stats["R"], C, W, H)
    binfo = build_info()
    eff_gbs = (ab["fwd"] + ab["bwd"]) / (ms_dev / args.steps * 1e-3) * 1e-9
    line = h.base_line(cfg, value, ms_dev / args.steps, args.steps, "weak")
    line.update({
        "config": {"workload": cfg["workload"], "P": P, "C": C, "W": W, "H": H,
                   "views_per_step": world, "parallelism": f"view-sharded x{world}" + (
                       " + NCCL all-reduce of per-Gaussian grads (feature grad overlapped with the chain backward)" if world > 1 else ""),
                   "view_schedule": f"rank r renders view (step + r) % {NVIEWS}: every rank cycles all {NVIEWS} views",
                   "l2": "inputs larger than L2 (1.0 GB feature table, 2.1 GB dL/dout, 2.1 GB output per step; 8 cycling views)",
                   **{k: v for k, v in stats.items() if k != "blended_pairs"}},
        "views_per_s": value * 1e6, "hbm_gbs_effective": eff_gbs, "hbm_frac_effective": eff_gbs / peak,
        "stage_ms": per_stage, "kernel_ms_per_step": sum(per_stage.values()),
        "roofline": roofline_block(per_stage, ab, ("blend_fwd", "blend_bwd", "dfeature", "alpha_pass"),
                                   binfo["source_sha256_16"],
                                   "C=256 blend is fp32-FMA bound by design (no tensor cores, north_star); see fma_roofline and DESIGN.md"),
        # the C = 256 blend is three fp32 contractions on the CUDA cores (north_star rules out tensor cores):
        # algorithmic flops = 2*C per blended (pixel, Gaussian) pair for each of forward, s-pass, dL/dfeature
        "fma_roofline": fma_roofline(C, stats["blended_pairs"], per_stage),
        "e2e": {"value": e2e_value, "unit": "Mviews/s", "ms_per_step": ms_e2e / args.steps,
                "h2d_bytes_per_step": 35 * 4 + H * W * 4, "d2h_bytes_per_step": 8,
                "api": "render_chn() + semantic.distill_loss_and_grad() + backward; camera + label map from pinned host memory; "
                       "loss read back every step (async 8-byte copy to pinned memory, consumed one step later)"},
        "gpu_launches": launches[0], "cub_calls": launches[1], "clocks": clocks, "build": binfo,
        "per_rank_ms_per_step": rank_ms,
    })
    if view_ms:
        line["view_ms"] = {"per_view": view_ms, "mean": float(np.mean(view_ms)), "max": float(max(view_ms)),
                           "note": "fwd+bwd device time of each of the cycling views alone on rank 0; a synchronous "
                                   "step of N ranks costs the slowest of its N views"}
    if world > 1:
        line["exchange"] = {"ms_per_step_without_exchange": ms_nocomm,
                            "exposed_ms_per_step": ms_dev / args.steps - ms_nocomm,
                            "bytes_feature_grad": 4 * P * C, "bytes_small": 4 * P * 11, "collective": "all-reduce (sum)"}
        line["multi_gpu_parity"] = parity

    # ---- reference CUDA path on the same GPU (compiled unmodified reference, oracle/_ref) and the CPU legs
    if world == 1 and not args.no_baselines:
        with torch.no_grad():   # the reference gets exactly the tensors our rasterizer sees (activated parameters)
            sc_ref = dict(means3D=pc.get_xyz.detach().contiguous(), opacities=pc.get_opacity.detach().contiguous(),
                          scales=pc.get_scaling.detach().contiguous(), rotations=pc.get_rotation.detach().contiguous(),
                          features=feats.detach())
        line["reference_cuda"] = reference_cuda_times(
            torch, dev, sc_ref, cams_np[1], dL_fixed, C, W, H, cam_dev=cams[1],
            ours=lambda cam: render_chn(cam, pc, Pipe, bg, num_channels=C, override_color=feats))
        try:
            smp = cpu_raster_sample(cfg, scene, cams_np[0])
            v = 1.0 / smp["seconds_full_view_est"] * 1e-6
            line["cpu_baseline"] = {
                "value": v, "unit": "Mviews/s", "cores": smp["threads"], "kind": "port",
                "band_full_view_estimates_s": smp["band_full_view_est_s"],
                "sample": f"full preprocess of 1M Gaussians + binning/blend fwd+bwd of 3 bands of 16 rows (top quarter, middle, "
                          f"bottom quarter) each scaled to the view, mean of the three; {smp['seconds_sample']:.1f} s of CPU work"}
        except Exception as ex:  # pragma: no cover
            line["cpu_baseline"] = {"value": None, "error": repr(ex)}
        try:
            line["cpu_preprocess_torch"] = cpu_torch_preprocess_leg(P)
        except Exception as ex:  # pragma: no cover
            line["cpu_preprocess_torch"] = {"error": repr(ex)}
    emit_line(line)
    h.finish()


def reference_cuda_times(torch, dev, sc, cam, dL, C, W, H, ours=None, cam_dev=None):
    """The reference's channel-rasterization CUDA path recompiled for sm_100a, timed on this GPU: forward by the
    stock library, forward as render_chn() ships it (debug=True: a CPU deep copy of every argument before the
    call, channel_rasterization/__init__.py:86-87, model/renderer.py:181), backward by the NUM_CHANNELS=C rebuild
    (SURVEY.md 2d-1).  Also compares our image with the reference's on this exact view."""
    out = {}
    try:
        from oracle import ref as refmod
        sys.path.insert(0, os.path.join(ROOT, "tests"))
        from util import dev_cam
        cm = dev_cam(cam, dev)
        bg = torch.zeros(C, device=dev)
        kw = dict(bg=bg, means3D=sc["means3D"], opacities=sc["opacities"], viewmatrix=cm["viewmatrix"],
                  projmatrix=cm["projmatrix"], campos=cm["campos"], tanfovx=cm["tanfovx"], tanfovy=cm["tanfovy"],
                  W=W, H=H, colors_precomp=sc["features"], scales=sc["scales"], rotations=sc["rotations"],
                  num_channels=C)

        def ev_time(fn, n):
            fn()
            torch.cuda.synchronize(dev)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(n):
                fn()
            e1.record()
            torch.cuda.synchronize(dev)
            return e0.elapsed_time(e1) / n
        if refmod.available("chn"):
            r = refmod.RefRasterizer("chn")
            out["fwd_ms"] = ev_time(lambda: r.forward(**kw), 3)

            def fwd_debug():
                # cpu_deep_copy_tuple(args): every tensor argument is cloned to the host before the native call
                _ = [t.cpu().clone() for t in kw.values() if isinstance(t, torch.Tensor)]
                r.forward(**kw)
            t0 = time.perf_counter()
            fwd_debug()
            torch.cuda.synchronize(dev)
            out["fwd_as_shipped_debug_true_ms"] = 1e3 * (time.perf_counter() - t0)
            if ours is not None:
                ref_img = r.forward(**kw)
                with torch.no_grad():
                    mine = ours(cam_dev)
                out["parity_this_view"] = {
                    "color_max_rel_err": float((mine["render"] - ref_img["color"]).abs().max() / ref_img["color"].abs().max()),
                    "radii_equal": bool(torch.equal(mine["radii"], ref_img["radii"])), "tolerance": 1e-4}
                del ref_img, mine
        if refmod.available(f"chn_c{C}"):
            r2 = refmod.RefRasterizer(f"chn_c{C}")
            r2.forward(**kw)
            out["bwd_ms"] = ev_time(lambda: r2.backward(dL), 1)
        out["kind"] = "unmodified reference cuda_rasterizer compiled for sm_100a (oracle/_ref), debug=False unless named"
    except Exception as ex:  # pragma: no cover
        out["error"] = repr(ex)
    return out


def run_k2(args, rank, world, local_rank):
    cfg = CONFIGS["K2"]
    h = Harness(args, rank, world, local_rank)
    torch, dev = h.torch, h.dev
    from semantic_gaussians_b200.gaussian_model import GaussianModel
    from semantic_gaussians_b200.renderer import render
    from semantic_gaussians_b200.scene_synth import make_scene, orbit_cameras
    P, C, W, H = cfg["P"], cfg["C"], cfg["W"], cfg["H"]
    scene = make_scene(P, seed=0, sh=True)
    cams_np = orbit_cameras(NVIEWS, W, H)
    pc = GaussianModel.from_activated(scene.xyz, scene.scales, scene.rotations, scene.opacity, scene.shs, device=dev)
    bg = torch.zeros(3, device=dev)
    cams = [h.dev_cam(c) for c in cams_np]

    last = {}

    def step_device(i, keep=False):
        with torch.no_grad():
            out = render(cams[(i + rank) % NVIEWS], pc, Pipe, bg)
        if keep:
            last.update(render_outputs(out))

    host_cam = [torch.from_numpy(np.concatenate([c.world_view_transform.ravel(), c.full_proj_transform.ravel(),
                                                 c.camera_center.ravel()]).astype(np.float32)).pin_memory()
                for c in cams_np]
    cam_dev = Cam()
    cam_dev.image_width, cam_dev.image_height, cam_dev.FoVx, cam_dev.FoVy = W, H, cams_np[0].FoVx, cams_np[0].FoVy
    cam_buf = torch.empty(35, device=dev)
    host_img = [torch.empty((4, H, W), dtype=torch.float32).pin_memory() for _ in range(2)]
    img_ev = [torch.cuda.Event() for _ in range(2)]

    def step_e2e(i):
        cam_buf.copy_(host_cam[(i + rank) % NVIEWS], non_blocking=True)
        cam_dev.world_view_transform = cam_buf[0:16].view(4, 4)
        cam_dev.full_proj_transform = cam_buf[16:32].view(4, 4)
        cam_dev.camera_center = cam_buf[32:35]
        with torch.no_grad():
            out = render(cam_dev, pc, Pipe, bg)
        host_img[i % 2][:3].copy_(out["render"], non_blocking=True)       # D2H: the rendered RGB image and depth
        host_img[i % 2][3:].copy_(out["depth"], non_blocking=True)
        img_ev[i % 2].record()
        if i > 0:
            img_ev[(i - 1) % 2].synchronize()

    for i in range(h.warmup):
        step_device(i)
    stats = view_stats(h, cfg, pc, None, cams[rank % NVIEWS], bg)
    ms_dev, ms_mine, per_stage, _, clocks, launches = h.profiled(
        lambda i: step_device(i, keep=args.dump_outputs is not None and i == args.steps - 1), args.steps)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, last)
    last.clear()
    for i in range(2):
        step_e2e(i)
    ms_e2e, _ = h.timed(step_e2e, args.steps, finish=lambda i: img_ev[i % 2].synchronize())
    if rank != 0:
        h.finish()
        return
    views = args.steps * world
    value = views / (ms_dev * 1e-3) * 1e-6
    peak, _ = measured_peaks()
    ab = algorithmic_bytes(P, stats["P_vis"], stats["R"], C, W, H)
    binfo = build_info()
    eff = ab["fwd"] / (ms_dev / args.steps * 1e-3) * 1e-9
    line = h.base_line(cfg, value, ms_dev / args.steps, args.steps, "weak")
    line.update({
        "config": {"workload": cfg["workload"], "P": P, "C": C, "W": W, "H": H, "views_per_step": world,
                   "parallelism": f"view-sharded x{world}, no exchange (forward only)",
                   "l2": "8 cycling views; 45 M-instance sort streams (0.5 GB) exceed L2", **stats},
        "views_per_s": value * 1e6, "hbm_gbs_effective": eff, "hbm_frac_effective": eff / peak,
        "stage_ms": per_stage, "kernel_ms_per_step": sum(per_stage.values()),
        "roofline": roofline_block(per_stage, ab, ("blend_fwd", "tile_sort"), binfo["source_sha256_16"], config="K2"),
        "e2e": {"value": views / (ms_e2e * 1e-3) * 1e-6, "unit": "Mviews/s", "ms_per_step": ms_e2e / args.steps,
                "h2d_bytes_per_step": 35 * 4, "d2h_bytes_per_step": 16 * W * H,
                "api": "render(): camera from pinned host memory, RGB image + median depth copied back to pinned memory"},
        "gpu_launches": launches[0], "cub_calls": launches[1], "clocks": clocks, "build": binfo,
    })
    if world == 1 and not args.no_baselines:
        try:
            smp = cpu_raster_sample(cfg, scene, cams_np[0], backward=False, want_depth=True)
            line["cpu_baseline"] = {"value": 1.0 / smp["seconds_full_view_est"] * 1e-6, "unit": "Mviews/s",
                                    "cores": smp["threads"], "kind": "port",
                                    "sample": f"full preprocess + 3 bands of 16 rows fwd, scaled; {smp['seconds_sample']:.1f} s"}
        except Exception as ex:  # pragma: no cover
            line["cpu_baseline"] = {"value": None, "error": repr(ex)}
    emit_line(line)
    h.finish()


# ------------------------------------------------------------------------------ K4: batched views + one exchange
def run_k4(args, rank, world, local_rank):
    cfg = CONFIGS["K4"]
    h = Harness(args, rank, world, local_rank)
    torch, dist, _lib, dev = h.torch, h.dist, h._lib, h.dev
    from semantic_gaussians_b200.distributed import OverlappedFeatureGradReduce, shard_range
    from semantic_gaussians_b200.gaussian_model import GaussianModel
    from semantic_gaussians_b200.renderer import render_chn, render_chn_batch
    from semantic_gaussians_b200.scene_synth import make_scene, room_cameras
    from semantic_gaussians_b200.semantic import distill_loss_and_grad
    P, C, W, H, VT = cfg["P"], cfg["C"], cfg["W"], cfg["H"], cfg["views_per_step"]
    VT = env_int("SGB_K4_VIEWS", VT)
    scene = make_scene(P, seed=0, kind="room", channels=C)
    cams_np = room_cameras(VT, W, H)
    pc = GaussianModel.from_activated(scene.xyz, scene.scales, scene.rotations, scene.opacity, device=dev)
    pc.active_sh_degree = 0
    feats = torch.as_tensor(scene.features, device=dev).contiguous().requires_grad_(True)
    scene.features = None
    for t in (pc._xyz, pc._scaling, pc._rotation, pc._opacity):
        t.requires_grad_(True)
    params = [feats, pc._xyz, pc._scaling, pc._rotation, pc._opacity]
    bg = torch.zeros(C, device=dev)
    mine = list(shard_range(VT, rank, world))
    cams = {k: h.dev_cam(cams_np[k]) for k in mine}
    gen = torch.Generator(device=dev).manual_seed(20260924)
    dL_fixed = torch.randn((C, H, W), device=dev, generator=gen) / (H * W)
    MB = _lib.MAX_BATCH
    subs = [mine[i:i + MB] for i in range(0, len(mine), MB)]
    overlap = OverlappedFeatureGradReduce(dev) if world > 1 else None

    def zero_grads():
        for p in params:
            p.grad = None

    def exchange():
        if world == 1:
            return
        # one sub-batch: the (P, C) buffer written by sgb_backward_batch IS .grad and is final right after the batch's
        # dL/dfeature kernels -> the 6.1 GB all-reduce runs under the chain kernels of the whole batch
        overlap.start(feats.grad, fresh=len(subs) == 1)
        small = torch.cat([p.grad.reshape(-1) for p in params[1:]])
        dist.all_reduce(small)
        overlap.finish()

    last = {}

    def step_device(i, batched=True, do_exchange=True, keep=False):
        for sub in subs:
            if batched:
                outs = render_chn_batch([cams[k] for k in sub], pc, Pipe, bg, num_channels=C, override_color=feats)
                torch.autograd.backward([o["render"] for o in outs], [dL_fixed] * len(outs))
                if keep:
                    for k, o in zip(sub, outs):
                        last.update(render_outputs(o, f"view{k:02d}_"))
            else:
                for k in sub:
                    render_chn(cams[k], pc, Pipe, bg, num_channels=C, override_color=feats)["render"].backward(dL_fixed)
        if do_exchange:
            exchange()
        if keep:
            last.update({f"{n}_grad": p.grad for n, p in zip(("features", "xyz", "scaling", "rotation", "opacity"),
                                                              params)})
        zero_grads()

    rng = np.random.default_rng(99 + rank)
    host_labels = [torch.from_numpy(rng.integers(0, NUM_CLASSES, size=(H, W), dtype=np.int64).astype(np.int32)).pin_memory()
                   for _ in range(2)]
    host_cam = {k: torch.from_numpy(np.concatenate([cams_np[k].world_view_transform.ravel(),
                                                    cams_np[k].full_proj_transform.ravel(),
                                                    cams_np[k].camera_center.ravel()]).astype(np.float32)).pin_memory()
                for k in mine}
    class_emb = torch.nn.functional.normalize(torch.randn(NUM_CLASSES, C, device=dev, generator=gen), dim=1)
    loss_host = torch.zeros(1, dtype=torch.float64).pin_memory()

    def step_e2e(i):
        total = torch.zeros((), dtype=torch.float64, device=dev)
        for sub in subs:
            cs, labels = [], []
            for j, k in enumerate(sub):
                buf = torch.empty(35, device=dev)
                buf.copy_(host_cam[k], non_blocking=True)                      # H2D 140 B per view
                lb = torch.empty((H, W), dtype=torch.int32, device=dev)
                lb.copy_(host_labels[(i + j) % 2], non_blocking=True)          # H2D 5 MB per view
                c = Cam()
                c.image_width, c.image_height, c.FoVx, c.FoVy = W, H, cams_np[k].FoVx, cams_np[k].FoVy
                c.world_view_transform, c.full_proj_transform = buf[0:16].view(4, 4), buf[16:32].view(4, 4)
                c.camera_center = buf[32:35]
                cs.append(c)
                labels.append(lb)
            outs = render_chn_batch(cs, pc, Pipe, bg, num_channels=C, override_color=feats)
            grads = []
            for o, lb in zip(outs, labels):
                loss, dL = distill_loss_and_grad(o["render"], class_emb, lb)
                total = total + loss
                grads.append(dL)
            torch.autograd.backward([o["render"] for o in outs], grads)
        exchange()
        zero_grads()
        loss_host.copy_(total.reshape(1), non_blocking=False)                  # D2H 8 B: the step's loss

    for i in range(h.warmup):
        step_device(i)
    torch.cuda.synchronize(dev)
    stats = view_stats(h, cfg, pc, feats, cams[mine[0]], bg)
    steps = args.steps
    ms_dev, ms_mine, per_stage, counts, clocks, launches = h.profiled(
        lambda i: step_device(i, keep=args.dump_outputs is not None and i == steps - 1), steps)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, last)
    last.clear()
    rank_ms = h.gather_floats(ms_mine / steps)
    ms_nc, _ = h.timed(lambda i: step_device(i, do_exchange=False), steps)
    nloop = max(1, steps // 2)
    ms_loop, _ = h.timed(lambda i: step_device(i, batched=False, do_exchange=False), nloop)
    step_e2e(0)
    ms_e2e, _ = h.timed(step_e2e, steps)
    if rank != 0:
        h.finish()
        return
    value = VT * steps / (ms_dev * 1e-3) * 1e-6
    peak, _ = measured_peaks()
    ab = algorithmic_bytes(P, stats["P_vis"], stats["R"], C, W, H)
    binfo = build_info()
    nloc = len(mine)
    # per batch the shared buffers are touched once (zero-fill + final read of the (P, C) gradient), per view the rest
    batch_bytes = nloc * (ab["fwd"] + ab["bwd"]) + 8 * P * C
    line = h.base_line(cfg, value, ms_dev / steps, steps, "strong")
    line.update({
        "config": {"workload": cfg["workload"], "P": P, "C": C, "W": W, "H": H, "views_per_step": VT,
                   "views_per_rank": nloc, "sub_batches_per_rank": [len(s) for s in subs],
                   "parallelism": f"view-sharded x{world}: {nloc} views per rank through sgb_*_batch (<= {MB} per call), "
                                  "gradients summed in place over the local views, ONE all-reduce per step",
                   "l2": "6.1 GB feature table, 2.6 GB image and dL/dout per view: far beyond L2",
                   **{k: v for k, v in stats.items() if k != "blended_pairs"}},
        "views_per_s": value * 1e6, "stage_ms": per_stage, "stage_counts_per_step": {k: v / steps for k, v in counts.items()},
        "bytes": {"per_view_algorithmic": ab["fwd"] + ab["bwd"], "per_rank_batch_algorithmic": batch_bytes,
                  "hbm_gbs_effective": batch_bytes / (ms_nc / steps * 1e-3) * 1e-9,
                  "hbm_frac_effective": batch_bytes / (ms_nc / steps * 1e-3) * 1e-9 / peak},
        "roofline": roofline_block(per_stage, ab, ("blend_fwd", "blend_bwd", "dfeature", "alpha_pass"),
                                   binfo["source_sha256_16"], "C=512 blend: fp32-FMA bound by design; see fma_roofline",
                                   config="K4"),
        "fma_roofline": fma_roofline(C, stats["blended_pairs"], per_stage),
        "batched_vs_loop": {"batched_ms_per_step_no_exchange": ms_nc / steps,
                            "per_view_loop_ms_per_step_no_exchange": ms_loop / nloop,
                            "note": "same views through render_chn() one by one (V x zero-fill of the (P, C) gradient, "
                                    "V-way autograd accumulation, 2 syncs per view) vs render_chn_batch()"},
        "exchange": {"bytes_feature_grad": 4 * P * C,
                     "collective": ("all-reduce (sum), overlapped with the batch's chain kernels" if len(subs) == 1
                                    else "all-reduce (sum)") if world > 1 else "none (1 rank)",
                     "ms_per_step_without_exchange": ms_nc / steps, "exposed_ms_per_step": (ms_dev - ms_nc) / steps},
        "e2e": {"value": VT * steps / (ms_e2e * 1e-3) * 1e-6, "unit": "Mviews/s", "ms_per_step": ms_e2e / steps,
                "h2d_bytes_per_step": nloc * (35 * 4 + H * W * 4), "d2h_bytes_per_step": 8,
                "api": "render_chn_batch() + distill_loss_and_grad() per view + backward + exchange; cameras and label maps "
                       "from pinned host memory, summed loss read back every step"},
        "gpu_launches": launches[0], "cub_calls": launches[1], "clocks": clocks, "build": binfo,
        "per_rank_ms_per_step": rank_ms,
    })
    emit_line(line)
    h.finish()


# ------------------------------------------------------------------------------ K5: fusion
def run_k5(args, rank, world, local_rank):
    cfg = CONFIGS["K5"]
    t_start = time.perf_counter()
    h = Harness(args, rank, world, local_rank)
    torch, dev = h.torch, h.dev
    from semantic_gaussians_b200.distributed import allreduce_sums, shard_strided
    from semantic_gaussians_b200.fusion import PointCloudToImageMapper, normalize_fused
    from semantic_gaussians_b200.gaussian_model import GaussianModel
    from semantic_gaussians_b200.renderer import render
    from semantic_gaussians_b200.scene_synth import make_scene, room_cameras
    P, C, w, hh, VT = cfg["P"], cfg["C"], cfg["W"], cfg["H"], cfg["views_per_step"]
    VT = env_int("SGB_K5_VIEWS", VT)
    scene = make_scene(P, seed=0, kind="room", sh=True)
    cams_np = room_cameras(VT, w, hh)
    pc = GaussianModel.from_activated(scene.xyz, scene.scales, scene.rotations, scene.opacity, scene.shs, device=dev)
    xyz = pc.get_xyz
    mine = list(shard_strided(VT, rank, world))
    NM = 4                                                  # device-resident maps cycled (4 x 315 MB > L2)
    g = torch.Generator(device=dev).manual_seed(7)
    maps = [torch.randn((C, hh, w), device=dev, generator=g).half() for _ in range(NM)]
    host_maps = [torch.randn((C, hh, w)).half().pin_memory() for _ in range(2)]
    bg3 = torch.zeros(3, device=dev)
    # Visibility rule.  Default: the reference's `depth: none` branch (fusion_utils.py:70-72 — every Gaussian in front of
    # the camera and inside the cut image is visible): on a synthetic random cloud the rendered-depth test
    # (fusion.py:106-120) leaves < 100 of 2 M Gaussians visible per view (measured), which would benchmark nothing.
    # SGB_K5_DEPTH=render selects the rendered median depth (rendered once, outside the timed region).
    use_render = os.environ.get("SGB_K5_DEPTH", "none") == "render"
    depth, mappers = {}, {}
    with torch.no_grad():
        for k in mine:
            depth[k] = (render(h.dev_cam(cams_np[k]), pc, Pipe, bg3, override_shape=[w, hh])["depth"][0].contiguous()
                        if use_render else None)
            mappers[k] = PointCloudToImageMapper([w, hh], 0.25, 10, cams_np[k].intrinsics(), device=dev)
    w2c = {k: torch.as_tensor(cams_np[k].world_view_transform, device=dev) for k in mine}
    fs = torch.zeros((P, C), device=dev)
    cnt = torch.zeros(P, device=dev)
    nvis_acc = []

    def step_device(i, record=False):
        fs.zero_()
        cnt.zero_()
        for j, k in enumerate(mine):
            nv = mappers[k].accumulate(w2c[k], xyz, maps[j % NM], fs, cnt, depth[k])
            if record:
                nvis_acc.append(nv)
        allreduce_sums([fs, cnt])
        normalize_fused(fs, cnt)

    out_host = torch.empty((P, C), dtype=torch.float16).pin_memory()
    stage = torch.empty((C, hh, w), dtype=torch.float16, device=dev)

    def step_e2e(i):
        fs.zero_()
        cnt.zero_()
        for j, k in enumerate(mine):
            stage.copy_(host_maps[j % 2], non_blocking=True)           # H2D: this view's 2D feature map (315 MB)
            mappers[k].accumulate(w2c[k], xyz, stage, fs, cnt, depth[k])
        allreduce_sums([fs, cnt])
        normalize_fused(fs, cnt)
        if rank == 0:
            out_host.copy_(fs.half(), non_blocking=False)               # D2H: fused features as saved (fp16)

    def note(msg):
        if rank == 0:
            print(f"[K5 {time.perf_counter() - t_start:7.1f} s] {msg}", file=sys.stderr, flush=True)
    note("setup done")
    for i in range(min(h.warmup, 3)):
        step_device(i)
        torch.cuda.synchronize(dev)
        note(f"warm-up step {i}")
    step_device(0, record=True)
    nvis = [int(v) for v in nvis_acc]
    steps = args.steps
    ms_dev, ms_mine, per_stage, counts, clocks, launches = h.profiled(step_device, steps)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"fused_features": fs, "counts": cnt})   # the last step's, untouched since
    rank_ms = h.gather_floats(ms_mine / steps)

    def no_exchange(i):
        fs.zero_()
        cnt.zero_()
        for j, k in enumerate(mine):
            mappers[k].accumulate(w2c[k], xyz, maps[j % NM], fs, cnt, depth[k])
    note("device-resident region timed")
    ms_nc, _ = h.timed(no_exchange, steps)
    ne2e = max(1, steps // 2)
    step_e2e(0)
    note("e2e warm-up done")
    ms_e2e, _ = h.timed(step_e2e, ne2e)
    note("e2e timed")
    if rank != 0:
        h.finish()
        return
    value = VT * steps / (ms_dev * 1e-3) * 1e-6
    peak, peak_src = measured_peaks()
    binfo = build_info()
    nv_mean = float(np.mean(nvis)) if nvis else 0.0
    # SURVEY.md §8(d): xyz + depth in, one C-vector gathered per visible Gaussian, fp32 accumulator read-modify-write
    per_view = 12 * P + 4 * w * hh + nv_mean * C * 2 + nv_mean * C * 8 + nv_mean * 8
    kernel_view_ms = sum(v for k, v in per_stage.items() if k.startswith("fusion"))
    achieved = per_view / (kernel_view_ms * 1e-3) * 1e-9 if kernel_view_ms else float("nan")
    line = h.base_line(cfg, value, ms_dev / steps, steps, "strong")
    line.update({
        "config": {"workload": cfg["workload"], "P": P, "C": C, "W": w, "H": hh, "views_per_step": VT,
                   "views_per_rank": len(mine), "feature_dtype": "float16", "visibility_threshold": 0.25, "cut_boundary": 10,
                   "depth": "rendered median depth (fusion.py:106-120)" if use_render else
                            "none: every Gaussian in front of the camera inside the cut image is visible (fusion_utils.py:70-72)",
                   "N_vis_per_view": {"mean": nv_mean, "min": min(nvis) if nvis else 0, "max": max(nvis) if nvis else 0},
                   "parallelism": f"views strided over {world} ranks, one all-reduce of the (P, C) sums + counts, then normalise",
                   "l2": "4 cycling 315 MB maps and a 4.1 GB accumulator: beyond L2"},
        "views_per_s": value * 1e6, "stage_ms": per_stage,
        "bytes": {"per_view_algorithmic": per_view, "final_normalise": 8 * P * C},
        "roofline": {"bound": "hbm", "kernel": "fusion view (project + sort + gather/accumulate kernels)", "achieved": achieved,
                     "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                     "traffic": traffic_for("K5.fusion_gather", binfo["source_sha256_16"])[0],
                     "traffic_source": "gather/accumulate kernel alone (the dominant launch of the view), " +
                                       str(traffic_for("K5.fusion_gather", binfo["source_sha256_16"])[1]),
                     "algorithmic_bytes": per_view, "kernel_ms": kernel_view_ms, "peak_source": peak_src},
        "exchange": {"bytes": 4 * P * C + 4 * P, "ms_per_step_without_exchange_and_normalise": ms_nc / steps,
                     "exposed_ms_per_step": (ms_dev - ms_nc) / steps},
        "e2e": {"value": VT * ne2e / (ms_e2e * 1e-3) * 1e-6, "unit": "Mviews/s", "ms_per_step": ms_e2e / ne2e,
                "h2d_bytes_per_step": len(mine) * C * hh * w * 2, "d2h_bytes_per_step": 2 * P * C,
                "api": "PointCloudToImageMapper.accumulate() per view with the (C,h,w) fp16 map copied from pinned host "
                       "memory, all-reduce, normalize_fused(), fused features copied back as fp16"},
        "gpu_launches": launches[0], "cub_calls": launches[1], "clocks": clocks, "build": binfo,
        "per_rank_ms_per_step": rank_ms,
    })
    if world == 1 and not args.no_baselines:
        try:
            smp = cpu_fusion_sample(cfg, scene, cams_np, 2)
            line["cpu_baseline"] = {"value": 1.0 / smp["seconds_per_view"] * 1e-6, "unit": "Mviews/s", "cores": smp["threads"],
                                    "kind": "port", "sample": f"2 views: numpy compute_mapping {smp['mapping_s']:.2f} s/view (1 core) + "
                                                              f"torch-CPU gather/accumulate {smp['accumulate_s']:.2f} s/view"}
        except Exception as ex:  # pragma: no cover
            line["cpu_baseline"] = {"value": None, "error": repr(ex)}
    emit_line(line)
    h.finish()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="K3", choices=sorted(CONFIGS))
    ap.add_argument("--no-baselines", action="store_true", help="skip the reference-CUDA and CPU legs")
    ap.add_argument("--quick", action="store_true", help="skip the per-view cost spread")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the timed path computed in its last step to DIR/<name>.npy (float32 / float64, "
                         "64 MB at most: larger outputs as a fixed seeded sample of their values)")
    args = ap.parse_args()
    if args.steps is not None and args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs is not None and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of the CUDA path (--impl ours)")
    claim_stdout()
    if args.steps is None:
        args.steps = {"K2": 40, "K3": 20, "K4": 3, "K5": 3}[args.config] if args.impl == "ours" else 2
    rank, world, local_rank = env_int("RANK", 0), env_int("WORLD_SIZE", 1), env_int("LOCAL_RANK", 0)
    if args.impl == "reference":
        run_cpu_reference(args, rank, world)
        return
    {"K2": run_k2, "K3": run_k3, "K4": run_k4, "K5": run_k5}[args.config](args, rank, world, local_rank)


if __name__ == "__main__":
    main()

"""Config 4 (BASELINE.json): full-scene nDSM inference on a synthetic Munich-density scene.

python tools/bench_infer.py [--scale 0.45] [--tiles-per-batch 4] [--image]
Munich configuration (ALTO depth 6, footprint head, z range 134 m), 512 m tiles at 256 m stride, 1 m
pixels, ~1.93 points / m^2 (100 M points over 9050 m x 5730 m; --scale shrinks the scene edge lengths,
keeping the density).  Forward only, tiles batched as ragged clouds, everything on the device.
--image: the cloud + image model (use_image, image U-Net depth 6) with a seeded synthetic 3-band float32 orthophoto
covering the scene at the output's 1 m pixels; the line adds the summed CUDA-event time of the t2h_raster_windows
calls (the window cut) and their algorithmic bytes.
"""
import argparse, json, os, subprocess, sys, time
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))
import torch
import oracle
import tomosar2height_b200 as t2h
from tomosar2height_b200 import _lib
from tomosar2height_b200.generator import OrthoImage, SceneGenerator

ap = argparse.ArgumentParser()
ap.add_argument("--scale", type=float, default=0.45)
ap.add_argument("--tiles-per-batch", type=int, default=4)
ap.add_argument("--image", action="store_true", help="cloud + image model with a synthetic orthophoto")
args = ap.parse_args()
torch.backends.cudnn.allow_tf32 = False
cfg = t2h.munich_config(use_image=args.image)
params = oracle.synth_state_dict(oracle.reference_param_shapes(cfg), seed=0)
model = t2h.TomoSAR2Height(cfg); model.load_state_dict(params); model = model.cuda().eval()
W, H = 9050.0 * args.scale, 5730.0 * args.scale
n_pts = int(1.93 * W * H)
g = torch.Generator(device="cuda").manual_seed(0)
pts = torch.rand(n_pts, 3, generator=g, device="cuda", dtype=torch.float64)
# 70 % of the points on line-like "facades"
n_c = int(0.7 * n_pts); n_seg = max(int(W * H / 6500), 1)
a = torch.rand(n_seg, 2, generator=g, device="cuda", dtype=torch.float64)
d = (torch.rand(n_seg, 2, generator=g, device="cuda", dtype=torch.float64) - 0.5) * (100.0 / max(W, H))
which = torch.randint(0, n_seg, (n_c,), generator=g, device="cuda")
tt = torch.rand(n_c, 1, generator=g, device="cuda", dtype=torch.float64)
pts[:n_c, :2] = (a[which] + tt * d[which] + torch.randn(n_c, 2, generator=g, device="cuda", dtype=torch.float64) * (1.0 / max(W, H))).clamp(0, 1)
lo = torch.tensor([686167.0, 5331627.0], dtype=torch.float64, device="cuda")
pts[:, 0] = lo[0] + pts[:, 0] * W; pts[:, 1] = lo[1] + pts[:, 1] * H; pts[:, 2] = 465.5 + pts[:, 2] * 60.0
gen = SceneGenerator(model, lo.tolist(), [lo[0].item() + W, lo[1].item() + H], cfg.dataset.normalize.z_bound,
                     tiles_per_batch=args.tiles_per_batch)
warm = SceneGenerator(model, lo.tolist(), [lo[0].item() + 1024, lo[1].item() + 1024], cfg.dataset.normalize.z_bound, tiles_per_batch=args.tiles_per_batch)
image = None
if args.image:
    # the scene's raster grid (upper-left corner = the scene's), 3 bands uniform in [0, 255); one row and column more
    # than the nDSM, whose bottom / right tiles reach one pixel past it when the scene edge is not a whole number of pixels
    bands = torch.rand(3, gen.n_rows + 1, gen.n_cols + 1, generator=g, device="cuda") * 255.0
    image = OrthoImage(bands, gen.l, gen.t, 1.0, [127.5] * 3, [73.6] * 3)
    del bands

# CUDA events around the window cuts only (two events per batch: the timed pass is otherwise untouched)
win_events, _call = [], _lib.call
def _timed_call(name, *a):
    if name != "t2h_raster_windows":
        return _call(name, *a)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(); _call(name, *a); e1.record()
    win_events.append((e0, e1, 2 * 4 * a[6] * a[7] * a[7] * a[1]))  # read + write B*S*S*C floats
if args.image:
    _lib.call = _timed_call

warm.generate(pts, image=image)  # warm-up on a corner of the scene
torch.cuda.synchronize(); win_events.clear(); t0 = time.perf_counter()
dsm, weight = gen.generate(pts, image=image)
torch.cuda.synchronize(); dt = time.perf_counter() - t0
try:
    power = float(subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader,nounits", "-i",
                                  str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30).stdout)
except (OSError, ValueError, subprocess.TimeoutExpired):
    power = None
line = {"config": f"munich cloud-{'+image' if args.image else 'only'} inference, depth 6 + footprint head, 512 m tiles @ 256 m stride",
        "scene_m": [W, H], "scene_points": n_pts, "tiles": len(gen.anchors), "seconds": round(dt, 3),
        "scene_points_per_s": round(n_pts / dt), "ndsm_px_per_s": round(dsm.numel() / dt),
        "tile_px_per_s": round(len(gen.anchors) * 512 * 512 / dt),
        "covered_fraction": float((weight > 0).double().mean()), "n_gpus": 1,
        "gpu": torch.cuda.get_device_name(), "power_limit_w": power}
if args.image:
    ms = sum(e0.elapsed_time(e1) for e0, e1, _ in win_events)
    nbytes = sum(b for _, _, b in win_events)
    line["orthophoto"] = {"shape": list(image.bands.shape), "bytes": image.bands.numel() * 4}
    line["raster_windows"] = {"calls": len(win_events), "ms_total": round(ms, 3), "bytes": nbytes,
                              "gbs": round(nbytes / 1e9 / (ms / 1e3), 1) if ms > 0 else None,
                              "share_of_scene": round(ms / 1e3 / dt, 5)}
print(json.dumps(line))

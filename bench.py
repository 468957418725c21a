#!/usr/bin/env python
"""bench.py -- throughput of the TomoSAR2Height hot path on B200 (BASELINE.json configs 2, 3, 4).

--workload train        (default, the headline; config 2) point-cloud-only training step: batch of 32 synthetic
                        Berlin-shaped tiles (N = 262 144 points each, R = 256, ALTO depth 5, conv decoder, 512^2
                        nDSM), fp32, forward + L1 loss + backward in micro-batches (CUDA-graph replay), AdamW.
                        N GPUs = weak scaling, ONE flat fp32 gradient all-reduce (SUM) per step.
--workload train_image  (config 3) the same step with use_image=true: synthetic orthophoto tiles (B, 3, 512, 512)
                        through the image U-Net (stock PyTorch / cuDNN), tile-sharded data parallel.
--workload infer        (config 4) full-scene nDSM inference on a synthetic Munich-density scene (--scene-scale
                        1.0 = 9050 m x 5730 m, 100 M points, 770 tiles of 512 m at 256 m stride), Munich
                        configuration (depth 6, footprint head).  N GPUs = STRONG scaling: contiguous blocks of the
                        tile list per rank, no collective; value = scene points/s.

One process per GPU.  Prints ONE JSON line (driver contract): value = whole-job throughput with inputs resident in
HBM, e2e = the same work through the public API from pinned host buffers (H2D inside the timed region, result read
back), roofline = the dominant hand-written kernel of the step, cpu_baseline = the CPU oracle on this box's cores
with the oracle's heights compared against the CUDA path on the same tile (`parity`).  With the default workload
the line also carries `workloads`: configs 3 and 4 measured on bounded samples in the same run.

`--impl reference` times the reference's own CPU path on the host cores: the REAL reference (stub-imported, as
tests/golden/make_golden.py does) when /root/reference is mounted, else the oracle port.
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))

import numpy as np  # noqa: E402
import torch  # noqa: E402


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="train", choices=["train", "train_image", "infer"])
    ap.add_argument("--tiles", type=int, default=32, help="tiles per step per GPU (batch)")
    ap.add_argument("--points", type=int, default=262144, help="points per tile")
    ap.add_argument("--micro-batch", type=int, default=4, help="tiles per forward/backward")
    ap.add_argument("--scene-scale", type=float, default=0.3, help="infer: edge-length scale of the Munich scene (1.0 = 100 M points)")
    ap.add_argument("--tiles-per-batch", type=int, default=4, help="infer: tiles per forward")
    ap.add_argument("--no-extras", action="store_true", help="skip the bounded config-3 / config-4 measurements of the default run")
    ap.add_argument("--no-cudnn-benchmark", action="store_true", help="skip cuDNN autotuning (use under ncu)")
    ap.add_argument("--no-graph", action="store_true", help="issue every micro-batch eagerly instead of replaying a CUDA graph")
    ap.add_argument("--conv-tf32", action="store_true", help="let the retained cuDNN convs use TF32 (reference GPU default)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--cpu-points", type=int, default=262144, help="points of the CPU-baseline tile")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step returned as DIR/<name>.npy (train: loss, gradients, updated "
                         "parameters; infer: the summed height and weight rasters), a fixed sample of it beyond 60 MB")
    args = ap.parse_args()
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs applies to --impl b200")
    return args


def synthetic_batch(tiles, points, seed, with_image=False):
    from cases import synthetic_cloud, synthetic_targets
    cloud = synthetic_cloud(tiles, points, seed, clustered=True)
    dsm, image = synthetic_targets(tiles, 512, seed, with_image=with_image)
    return cloud, dsm, image


DUMP_BYTES = 60 << 20  # array data of --dump-outputs: the .npy files stay under 64 MB together


def dump_outputs(out_dir, arrays):
    """Write every name -> float32 / float64 CPU tensor as out_dir/<name>.npy.  When they hold more than DUMP_BYTES
    together, every array of more than one element is cut to the same fraction of its flat elements, taken in order
    at positions drawn from a fixed seed: runs with the same arguments store the same elements."""
    os.makedirs(out_dir, exist_ok=True)
    total = sum(t.numel() * t.element_size() for t in arrays.values())
    for name, t in arrays.items():
        assert t.dtype in (torch.float32, torch.float64), (name, t.dtype)
        if total > DUMP_BYTES and t.numel() > 1:
            pos = torch.randperm(t.numel(), generator=torch.Generator().manual_seed(0))[:t.numel() * DUMP_BYTES // total]
            t = t.flatten()[pos.sort().values]
        np.save(os.path.join(out_dir, name + ".npy"), t.numpy())


def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as fh:
            d = json.load(fh)
        return d.get("hbm_gbs", 6650.0), d.get("bf16_tflops_sustained", 1400.0), "measured"
    return 6650.0, 1590.0, "fallback"


class ClockSampler:
    QUERY = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.proc = None
        self.gpu_index = gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.QUERY}", "--format=csv,noheader,nounits",
                                          "-i", str(self.gpu_index), "-lms", "200"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
        except OSError:
            self.proc = None

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            out, _ = self.proc.communicate(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
            out, _ = self.proc.communicate()
        sm, mx, reasons = [], 0.0, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in out.strip().splitlines():
            f = [x.strip() for x in line.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx = max(mx, float(f[2]))
            except ValueError:
                continue
            for name, val in zip(names, f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx or None, "reasons": sorted(reasons),
                "samples": len(sm)}


# ------------------------------------------------------------------------------------------------------------
# reference arm (CPU)
# ------------------------------------------------------------------------------------------------------------
def cpu_oracle_step(cfg, params, cloud, dsm, image=None):
    """One tile through the CPU oracle: forward + L1 loss + backward (trainer.py:61-70)."""
    import oracle
    P = {k: v.clone().requires_grad_(True) for k, v in params.items()}
    t0 = time.perf_counter()
    pa, pb = oracle.oracle_forward(P, cfg, cloud, image)
    loss = oracle.oracle_loss(pa, pb, dsm, False)
    loss.backward()
    return time.perf_counter() - t0, float(loss.detach()), pa.detach()


def real_reference_model(cfg, params):
    """The UNMODIFIED reference model classes from /root/reference when it is mounted (this container; the GPU box
    has no copy): model.py / pointnet.py / alto.py / pixel.py / resnet.py run as they are.  Their absent third-party
    imports are stubbed as tests/golden/make_golden.py does; ``torch_scatter`` (absent, un-vendored) is served by
    the oracle's vectorised scatter_max / scatter_mean so that its cost is that of a compiled op, not of a python loop."""
    if not os.path.isdir(os.environ.get("T2H_REFERENCE", "/root/reference")):
        return None
    try:
        import make_golden
        import oracle
        Model, _ = make_golden.import_reference()

        def scatter_max(src, index, dim=-1, out=None, dim_size=None):
            return oracle.segment_max(src, index, dim_size)

        def scatter_mean(src, index, dim=-1, out=None, dim_size=None):
            return oracle.segment_mean(src, index, out.shape[-1] if out is not None else dim_size)

        for name in ("tomosar2height.encoder.pointnet", "tomosar2height.encoder.alto"):
            mod = sys.modules.get(name)
            if mod is not None:
                mod.scatter_max, mod.scatter_mean = scatter_max, scatter_mean
        model = Model(cfg)
        model.load_state_dict(params)
        return model
    except Exception:
        return None


def run_reference(args):
    """Reference arm: the reference's CPU implementation of the path on the host cores (rank 0 only)."""
    if int(os.environ.get("RANK", "0")) != 0:
        return
    import oracle
    import tomosar2height_b200 as t2h
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    use_image = args.workload == "train_image"
    cfg = t2h.munich_config() if args.workload == "infer" else t2h.berlin_config(use_image=use_image)
    params = oracle.synth_state_dict(oracle.reference_param_shapes(cfg), seed=0)
    n = args.cpu_points
    cloud, dsm, image = synthetic_batch(1, n, seed=0, with_image=use_image)
    real = real_reference_model(cfg, params)
    kind = "reference" if real is not None else "port"

    def step():
        t0 = time.perf_counter()
        if args.workload == "infer":
            with torch.no_grad():
                (real(input_cloud=cloud) if real is not None else oracle.oracle_forward(params, cfg, cloud))
        elif real is not None:
            real.zero_grad()
            pa, _ = real(input_cloud=cloud, input_image=image)
            torch.nn.functional.l1_loss(pa.squeeze(), dsm.squeeze()).backward()
        else:
            return cpu_oracle_step(cfg, params, cloud, dsm, image)[0]
        return time.perf_counter() - t0

    for _ in range(min(args.warmup, 1)):
        step()
    times = [step() for _ in range(args.steps)]
    t = sum(times) / len(times)
    value = n / t
    names = {"train": ("fwd+bwd points/s", "cloud-only training step (fwd+L1+bwd), Berlin-shaped tiles, R=256, ALTO depth 5"),
             "train_image": ("fwd+bwd points/s", "cloud+image training step (fwd+L1+bwd), Berlin-shaped tiles + 512^2 orthophoto"),
             "infer": ("scene points/s", "nDSM inference forward, Munich configuration (depth 6, footprint head), one tile")}
    metric, workload = names[args.workload]
    line = {
        "impl": "reference", "metric": metric, "value": value, "unit": "points/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": min(args.warmup, 1), "ms_per_step": t * 1e3, "higher_is_better": True,
        "scaling": "strong" if args.workload == "infer" else "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "ndsm_px_per_s": 512 * 512 / t,
        "config": {"workload": workload, "tiles_per_step": 1, "points_per_tile": n},
        "cpu_baseline": {"value": value, "unit": "points/s", "cores": cores, "kind": kind,
                         "sample": f"1 tile of {n} points per step through {'the unmodified reference (stub imports)' if kind == 'reference' else 'oracle/'} (torch CPU, {cores} threads)"},
        "e2e": {"value": value, "unit": "points/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------------------------
# B200 arm
# ------------------------------------------------------------------------------------------------------------
class Ctx:
    """process-wide state of the B200 arm"""

    def __init__(self, args):
        import torch.distributed as dist
        self.dist = dist
        self.rank = int(os.environ.get("RANK", "0"))
        self.local_rank = int(os.environ.get("LOCAL_RANK", "0"))
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        if not torch.cuda.is_available():
            raise RuntimeError("bench.py needs a CUDA device; the B200 path has no CPU fallback")
        torch.cuda.set_device(self.local_rank)
        self.dev = torch.device("cuda", self.local_rank)
        if self.world > 1:
            os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
            dist.init_process_group("nccl", device_id=self.dev)
        torch.backends.cudnn.allow_tf32 = bool(args.conv_tf32)
        torch.backends.cuda.matmul.allow_tf32 = False
        torch.backends.cudnn.benchmark = not args.no_cudnn_benchmark

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(self, values):
        t = torch.tensor(values, device=self.dev, dtype=torch.float64)
        if self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return t.tolist()

    def timed(self, fn, steps):
        """EXACTLY `steps` calls bracketed by barrier + synchronize; device time (CUDA events), max over ranks."""
        self.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        out = None
        for _ in range(steps):
            out = fn()
        e1.record()
        self.barrier()
        return self.max_over_ranks([e0.elapsed_time(e1)])[0], out


def build_model(cfg, dev, seed=0):
    """Random-init weights of the named architecture: the model's own rule (model.py:46-52, Xavier-uniform weights,
    zero biases), seeded; identical on every rank."""
    import tomosar2height_b200 as t2h
    torch.manual_seed(seed)
    return t2h.TomoSAR2Height(cfg).to(dev)


def run_train(args, ctx, use_image, tiles, steps, warmup, want_kernels, want_outputs=False):
    import tomosar2height_b200 as t2h
    from tomosar2height_b200 import _lib
    from tomosar2height_b200.trainer import Trainer
    dev = ctx.dev
    cfg = t2h.berlin_config(use_image=use_image)
    model = build_model(cfg, dev).train()
    opt = torch.optim.AdamW(model.parameters(), lr=1e-4)  # train.py:97
    N, mb = args.points, args.micro_batch
    trainer = Trainer(model, opt, micro_batch=mb, use_cuda_graph=not args.no_graph)
    cloud_h, dsm_h, image_h = synthetic_batch(tiles, N, seed=100 + ctx.rank, with_image=use_image)
    host = [t.pin_memory() for t in (cloud_h, dsm_h) + ((image_h,) if use_image else ())]
    resident = [t.to(dev) for t in host]

    def step_resident():
        return trainer.train_batch(*resident)

    def step_e2e():
        batch = [t.to(dev, non_blocking=True) for t in host]
        return trainer.train_batch(*batch).item()  # device -> host read of the step's loss

    for _ in range(warmup):
        step_resident()
    clocks = ClockSampler(ctx.local_rank)
    clocks.start()
    ctx.barrier()
    torch.cuda.profiler.start()  # ncu --profile-from-start off captures exactly the timed steps
    ms, _ = ctx.timed(step_resident, steps)
    torch.cuda.profiler.stop()
    clock_info = clocks.stop()
    ms_e2e, last = ctx.timed(step_e2e, steps)
    res = {"ms": ms, "ms_e2e": ms_e2e, "loss": last, "clocks": clock_info, "cfg": cfg, "model": model,
           "points": ctx.world * tiles * N * steps, "px": ctx.world * tiles * 512 * 512 * steps,
           "h2d": sum(t.numel() * t.element_size() for t in host), "d2h": 4,
           "grad_bytes": trainer.flat.nbytes, "allreduce_ms": trainer.last_allreduce_ms()}
    if want_outputs:  # taken before the kernel-timing step below moves the model on
        res["outputs"] = {"loss": torch.tensor(last, dtype=torch.float32), "gradients": trainer.flat.flat.cpu(),
                          "parameters": torch.cat([p.detach().flatten() for p in model.parameters()]).cpu()}
    if want_kernels:
        # per-kernel device times (roofline): the same step issued eagerly with CUDA events around every C-ABI call --
        # a graph replay has no host-visible launch boundaries; kernel durations are the same
        from tomosar2height_b200.profiling import KernelTimer
        calls0 = _lib.launch_count
        with KernelTimer(n_rows=mb * N) as kt:
            trainer.train_batch(*resident, eager=True)
            ctx.barrier()
        res["launches"] = (_lib.launch_count - calls0) * steps  # C-ABI calls replayed per timed step x steps
        res["kernels"] = kt.summary()
    return res


def munich_scene(scale, dev, seed=0):
    """Synthetic Munich-density scene (SURVEY §8d config 4): 1.93 points / m^2 over (9050 * scale) x (5730 * scale) m,
    70 % of the points on line-like facades, UTM-like float64 coordinates."""
    W, H = 9050.0 * scale, 5730.0 * scale
    n_pts = int(1.93 * W * H)
    g = torch.Generator(device=dev).manual_seed(seed)
    pts = torch.rand(n_pts, 3, generator=g, device=dev, dtype=torch.float64)
    n_c, n_seg = int(0.7 * n_pts), max(int(W * H / 6500), 1)
    a = torch.rand(n_seg, 2, generator=g, device=dev, dtype=torch.float64)
    d = (torch.rand(n_seg, 2, generator=g, device=dev, dtype=torch.float64) - 0.5) * (100.0 / max(W, H))
    which = torch.randint(0, n_seg, (n_c,), generator=g, device=dev)
    tt = torch.rand(n_c, 1, generator=g, device=dev, dtype=torch.float64)
    noise = torch.randn(n_c, 2, generator=g, device=dev, dtype=torch.float64) * (1.0 / max(W, H))
    pts[:n_c, :2] = (a[which] + tt * d[which] + noise).clamp(0, 1)
    lo = (686167.0, 5331627.0)
    pts[:, 0] = lo[0] + pts[:, 0] * W
    pts[:, 1] = lo[1] + pts[:, 1] * H
    pts[:, 2] = 465.5 + pts[:, 2] * 60.0
    return pts, lo, (lo[0] + W, lo[1] + H)


def run_infer(args, ctx, scale, steps, warmup, want_outputs=False):
    import tomosar2height_b200 as t2h
    from tomosar2height_b200.generator import SceneGenerator
    dev = ctx.dev
    cfg = t2h.munich_config()
    model = build_model(cfg, dev).eval()
    pts_d, lo, hi = munich_scene(scale, dev)
    pts_h = pts_d.cpu().pin_memory()
    gen = SceneGenerator(model, lo, hi, cfg.dataset.normalize.z_bound, tiles_per_batch=args.tiles_per_batch)
    # every rank takes a contiguous block of the anchor list (= a strip of the scene) with a balanced number of
    # candidate points, derived from the bin table each rank computes anyway: no communication
    def step_resident():
        return gen.generate(pts_d, rank=ctx.rank, world=ctx.world)

    def step_e2e():
        dsm, weight = gen.generate(pts_h.to(dev, non_blocking=True), rank=ctx.rank, world=ctx.world)
        rows = [gen.raster_window(*gen.anchors[i])[0] for i in gen.last_tile_range] or [0]
        r_lo, r_hi = max(min(rows), 0), min(max(rows) + 512, gen.n_rows)
        step_e2e.d2h = 2 * (r_hi - r_lo) * gen.n_cols * 8
        return dsm[r_lo:r_hi].cpu(), weight[r_lo:r_hi].cpu()  # the rank's strip of the partial rasters

    for _ in range(warmup):
        step_resident()
    ms, _ = ctx.timed(step_resident, steps)
    ms_e2e, out = ctx.timed(step_e2e, steps)
    res = {"ms": ms, "ms_e2e": ms_e2e, "points": pts_d.shape[0] * steps, "px": gen.n_rows * gen.n_cols * steps,
           "tiles": len(gen.anchors), "scene_m": [hi[0] - lo[0], hi[1] - lo[1]], "scene_points": pts_d.shape[0],
           "h2d": pts_h.numel() * 8, "d2h": getattr(step_e2e, "d2h", 0),
           "covered_fraction": float((out[1] > 0).double().mean()) if out is not None else None}
    if want_outputs:
        res["outputs"] = {"dsm_sum": out[0], "weight_sum": out[1]}
    return res


def roofline_of(kernels, ms_step):
    hbm_peak, tf_peak, peak_src = load_peaks()
    mine = {k: v for k, v in kernels.items() if v["bytes_per_launch"] > 0}
    if not mine:
        return None
    top = max(mine, key=lambda k: mine[k]["ms_total"])
    k = mine[top]
    if k.get("tflops", 0.0) > 0:
        # per-point MLP GEMMs: the only dense contraction -> tensor pipe.  Algorithmic FLOPs (2MKN, one pass) over
        # the MEASURED dense bf16 peak; the 3xFP16 kernels (*_f16) issue 3 fp16 MMAs per algorithmic product at the
        # bf16 rate (ceiling 1/3), the 3xTF32 ones 3 TF32 MMAs at half that rate (ceiling 1/6) -- DESIGN.md §4.
        passes = 3.0 if top.endswith("_f16") else 6.0
        roof = {"bound": "tensor", "kernel": top, "achieved": k["tflops"], "peak": tf_peak, "unit": "TFLOP/s",
                "frac": k["tflops"] / tf_peak, "traffic": None, "peak_source": peak_src + " bf16 sustained",
                "scheme": "3xFP16" if passes == 3.0 else "3xTF32", "scheme_ceiling_frac": 1.0 / passes,
                "frac_of_scheme_ceiling": k["tflops"] * passes / tf_peak, "hbm_gbs": k["gbs"], "hbm_frac": k["gbs"] / hbm_peak}
    else:
        roof = {"bound": "hbm", "kernel": top, "achieved": k["gbs"], "peak": hbm_peak, "unit": "GB/s",
                "frac": k["gbs"] / hbm_peak, "traffic": None, "peak_source": peak_src}
    roof.update({"launches": k["launches"], "ms_avg": k["ms_avg"], "bytes_per_launch": k["bytes_per_launch"],
                 "share_of_step": k["ms_total"] / ms_step})
    # measured DRAM traffic of ONE profiled launch of this kernel (ncu --set full, committed under profiles/); the
    # launches of a step have many shapes, so the capture's own shape and algorithmic bytes ride along
    try:
        with open(os.path.join(ROOT, "profiles", "ncu_traffic.json")) as f:
            cap = json.load(f)
        if cap.get("kernel") == top:
            roof["traffic"] = cap["dram_bytes"]
            roof["traffic_capture"] = {k2: cap[k2] for k2 in ("capture", "algorithmic_bytes", "note") if k2 in cap}
    except (OSError, ValueError, KeyError):
        pass
    # the HBM-bound operators of the path against the measured copy bandwidth (north star: >= 0.6)
    roof["hbm_kernels"] = {n: round(v["gbs"] / hbm_peak, 3) for n, v in kernels.items()
                           if n.startswith(("t2h_seg_", "t2h_bilinear_", "t2h_upsample_")) and v["gbs"] > 0}
    return roof


def run_b200(args):
    ctx = Ctx(args)
    rank, world = ctx.rank, ctx.world
    wl = args.workload
    extras = {}
    if wl in ("train", "train_image"):
        res = run_train(args, ctx, wl == "train_image", args.tiles, args.steps, args.warmup, want_kernels=True,
                        want_outputs=bool(args.dump_outputs))
        ms_step = res["ms"] / args.steps
        line = {
            "metric": "fwd+bwd points/s", "value": res["points"] / (res["ms"] / 1e3), "unit": "points/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic", "ndsm_px_per_s": res["px"] / (res["ms"] / 1e3),
            "config": {"workload": ("cloud+image" if wl == "train_image" else "cloud-only") +
                       " training step (fwd+L1+bwd+AdamW), Berlin-shaped tiles, R=256, ALTO depth 5, conv decoder",
                       "tiles_per_step_per_gpu": args.tiles, "points_per_tile": args.points, "micro_batch_tiles": args.micro_batch,
                       "parallelism": f"dp{world}", "conv_tf32": bool(args.conv_tf32), "cuda_graph": not args.no_graph,
                       "hand_written_kernel_ms_per_step": sum(v["ms_total"] for v in res["kernels"].values()),
                       "gradient_allreduce": {"bytes": res["grad_bytes"], "ms": res["allreduce_ms"]},
                       "l2": "inputs+activations per step >> 126 MB L2 (no flush needed)"},
            "e2e": {"value": res["points"] / (res["ms_e2e"] / 1e3), "unit": "points/s", "h2d_bytes_per_step": res["h2d"],
                    "d2h_bytes_per_step": res["d2h"], "ms_per_step": res["ms_e2e"] / args.steps, "loss": res["loss"]},
            "gpu_launches": res["launches"], "clocks": res["clocks"], "roofline": roofline_of(res["kernels"], ms_step),
            "kernels": {k: {kk: round(vv, 4) if isinstance(vv, float) else vv for kk, vv in v.items()} for k, v in res["kernels"].items()},
        }
        cfg, model, outputs = res["cfg"], res["model"], res.get("outputs")
        if wl == "train" and not args.no_extras:
            # configs 3 and 4 on bounded samples, so that the driver's BENCH / SCALE records carry them too
            del res
            torch.cuda.empty_cache()
            r3 = run_train(args, ctx, True, max(args.micro_batch, args.tiles // 4), 2, 3, want_kernels=False)
            extras["train_image"] = {
                "metric": "fwd+bwd points/s", "value": r3["points"] / (r3["ms"] / 1e3), "ms_per_step": r3["ms"] / 2, "scaling": "weak",
                "e2e": r3["points"] / (r3["ms_e2e"] / 1e3), "sample": f"{max(args.micro_batch, args.tiles // 4)} tiles x {args.points} points + (3, 512, 512) images per step per GPU, 2 steps after 3 warm-ups",
                "gradient_allreduce": {"bytes": r3["grad_bytes"], "ms": r3["allreduce_ms"]}}
            del r3
            torch.cuda.empty_cache()
            r4 = run_infer(args, ctx, 0.2, 2, 3)
            extras["infer"] = {
                "metric": "scene points/s", "value": r4["points"] / (r4["ms"] / 1e3), "ndsm_px_per_s": r4["px"] / (r4["ms"] / 1e3),
                "ms_per_step": r4["ms"] / 2, "scaling": "strong", "e2e": r4["points"] / (r4["ms_e2e"] / 1e3),
                "sample": f"Munich configuration, scene scale 0.2 ({r4['scene_points']} points, {r4['tiles']} tiles of 512 m at 256 m stride), "
                          f"tile list split over {world} GPU(s), 2 passes after 3 warm-ups"}
            line["workloads"] = extras
    else:
        res = run_infer(args, ctx, args.scene_scale, args.steps, args.warmup, want_outputs=bool(args.dump_outputs))
        outputs = res.get("outputs")
        line = {
            "metric": "scene points/s", "value": res["points"] / (res["ms"] / 1e3), "unit": "points/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": res["ms"] / args.steps, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "ndsm_px_per_s": res["px"] / (res["ms"] / 1e3),
            "config": {"workload": "full-scene nDSM inference, Munich configuration (ALTO depth 6, footprint head), 512 m tiles at 256 m stride, 1 m pixels",
                       "scene_scale": args.scene_scale, "scene_m": res["scene_m"], "scene_points": res["scene_points"], "tiles": res["tiles"],
                       "tiles_per_forward": args.tiles_per_batch, "parallelism": f"tile blocks over {world} GPU(s), no collective",
                       "covered_fraction": res["covered_fraction"], "l2": "scene cloud and activations >> 126 MB L2 (no flush needed)"},
            "e2e": {"value": res["points"] / (res["ms_e2e"] / 1e3), "unit": "points/s", "h2d_bytes_per_step": res["h2d"],
                    "d2h_bytes_per_step": res["d2h"], "ms_per_step": res["ms_e2e"] / args.steps},
        }
        cfg = model = None
    if rank == 0:
        if not args.no_cpu_baseline and cfg is not None:
            import oracle  # the checker: cpu_baseline leg only
            cores = os.cpu_count() or 1
            torch.set_num_threads(cores)
            n_cpu = args.cpu_points
            use_image = wl == "train_image"
            c1, d1, i1 = synthetic_batch(1, n_cpu, seed=0, with_image=use_image)
            torch.manual_seed(0)
            import tomosar2height_b200 as t2h
            fresh = t2h.TomoSAR2Height(cfg)  # the benchmark model's initial weights, for both implementations
            params = {k: v.detach().clone() for k, v in fresh.state_dict().items()}
            t_cpu, loss_cpu, pa_cpu = cpu_oracle_step(cfg, params, c1, d1, i1)
            line["cpu_baseline"] = {"value": n_cpu / t_cpu, "unit": "points/s", "cores": cores, "kind": "port",
                                    "sample": f"1 tile of {n_cpu} points, fwd+L1+bwd once through oracle/ (torch CPU, {cores} threads), {t_cpu:.1f} s"}
            # the same tile through the CUDA path: the checker's result is compared, not thrown away
            model.load_state_dict(params)
            model.eval()
            with torch.no_grad():
                pa_gpu, _ = model(input_cloud=c1.to(ctx.dev), input_image=None if i1 is None else i1.to(ctx.dev))
            loss_gpu = torch.nn.functional.l1_loss(pa_gpu.squeeze(), d1.to(ctx.dev).squeeze()).item()
            line["parity"] = {"tile_points": n_cpu, "heights_rel": float((pa_gpu.cpu() - pa_cpu).abs().max() / pa_cpu.abs().max()),
                              "loss_rel": abs(loss_gpu - loss_cpu) / abs(loss_cpu), "tolerance": 1e-4}
        if outputs is not None:
            dump_outputs(args.dump_outputs, outputs)
        print(json.dumps(line))
    if world > 1:
        ctx.dist.destroy_process_group()


if __name__ == "__main__":
    a = parse_args()
    if a.impl == "reference":
        run_reference(a)
    else:
        run_b200(a)

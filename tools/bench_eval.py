"""Evaluation of a Munich-size scene nDSM (9050 x 5730 = 51.9 Mpx) against its ground truth: residual_stats on the
device against the same statistics with numpy on the host.

python tools/bench_eval.py [--calls 30] [--warmup 3]
Seeded synthetic pair (tests_support.synthetic_eval_rasters): float64 nDSM with a 64-pixel NaN border, float32 ground
truth with -9999 no-data patches, masks building = gt > 2.5 and ground = ~building.  The inputs (0.9 GB as the kernels
read them) are larger than L2, so every timed call streams them from HBM.  Prints one JSON line:
  call_ms    CUDA-event median of whole residual_stats calls (float32 -> float64 cast of gt, mask packing, the kernels and
             the read-back of the results)
  kernel_ms  CUDA-event median around the t2h_residual_stats call alone; GB/s against the bytes its passes read and
             against the 17 B/px a single pass would need
  host       wall time of the numpy statistics incl. the device-to-host copy of the inputs, and the host core count
"""
import argparse, json, os, subprocess, sys, time
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch
from tomosar2height_b200 import _lib, residual_stats
from tomosar2height_b200.evaluation import DATA_PASSES
from tomosar2height_b200.tests_support import numpy_residual_stats, synthetic_eval_rasters

ap = argparse.ArgumentParser()
ap.add_argument("--calls", type=int, default=30)
ap.add_argument("--warmup", type=int, default=3)
args = ap.parse_args()
if not torch.cuda.is_available():
    sys.exit("bench_eval.py needs a CUDA device")

ROWS, COLS = 5730, 9050
pred, gt, masks, nodata = synthetic_eval_rasters(ROWS, COLS, seed=0)
n_px = pred.numel()

kernel_events, _call = [], _lib.call
def _timed_call(name, *a):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(); _call(name, *a); e1.record()
    kernel_events.append((e0, e1))
_lib.call = _timed_call

for _ in range(args.warmup):
    got = residual_stats(pred, gt, masks, nodata)
torch.cuda.synchronize(); kernel_events.clear()
call_ms = []
for _ in range(args.calls):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(); got = residual_stats(pred, gt, masks, nodata); e1.record()
    e1.synchronize(); call_ms.append(e0.elapsed_time(e1))
kernel_ms = [e0.elapsed_time(e1) for e0, e1 in kernel_events]
median = lambda v: sorted(v)[len(v) // 2]

t0 = time.perf_counter()
host = numpy_residual_stats(pred.cpu().numpy(), gt.cpu().numpy(), {k: v.cpu().numpy() for k, v in masks.items()}, nodata)
host_s = time.perf_counter() - t0

exact = ("count", "min", "max", "median", "medae", "nmad")
mismatch = [(c, f) for c in host for f in exact if not (got[c][f] == host[c][f])]
rel = max(abs(got[c][f] - host[c][f]) / abs(host[c][f]) for c in host for f in ("mean", "mae", "rmse") if host[c][f])
try:
    power = float(subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader,nounits", "-i",
                                  str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30).stdout)
except (OSError, ValueError, subprocess.TimeoutExpired):
    power = None
bytes_per_pass = n_px * (8 + 8 + 1)  # float64 pred and gt, one mask byte
moved = DATA_PASSES * bytes_per_pass
k_ms = median(kernel_ms)
line = {"config": "nDSM evaluation, 9050 x 5730 px, 2 masks (building = gt > 2.5, ground), float32 gt with no-data",
        "pixels": n_px, "valid": got["all"]["count"], "calls": args.calls,
        "call_ms": round(median(call_ms), 3), "kernel_ms": round(k_ms, 3),
        "kernel_ms_min_max": [round(min(kernel_ms), 3), round(max(kernel_ms), 3)],
        "passes": DATA_PASSES, "bytes_read": moved,
        "gbs_moved": round(moved / 1e9 / (k_ms / 1e3), 1), "gbs_17b_per_px": round(bytes_per_pass / 1e9 / (k_ms / 1e3), 1),
        "host": {"seconds": round(host_s, 3), "cores": os.cpu_count(),
                 "cores_usable": len(os.sched_getaffinity(0)), "what": "numpy fp64 incl. D2H of pred, gt, masks"},
        "agreement": {"exact_fields_equal": not mismatch, "mismatches": mismatch, "sums_max_rel_diff": rel},
        "stats": got, "gpu": torch.cuda.get_device_name(), "power_limit_w": power}
print(json.dumps(line))

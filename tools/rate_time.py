"""Cost of the rate curve (byte-budget encoding) per 1920x1080x64 chunk, for the three wavelets, on the GPU:

  * rate_curve_device: the whole call (CUDA events on the caller's stream around a synchronous call), and its split
    from torch.profiler kernel times in a separate pass: front-end with the coefficient dump, value histogram, and step
    histograms + tables + estimate;
  * one plain front-end pass (the batch API's CUDA-event front-end time) for comparison;
  * one trial encode at quality 80 (front-end + tables + rANS, the batch API's CUDA-event stage times);
  * predicted - actual .alc bytes at a handful of steps (how tight the bound is).
Card name and power limit are read in the same run.  Writes the records to --out (JSON) and prints them.

    python tools/rate_time.py [--reps 5] [--out rate_time.json]
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402
from __graft_entry__ import load_package  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--reps", type=int, default=5)
ap.add_argument("--width", type=int, default=1920)
ap.add_argument("--height", type=int, default=1080)
ap.add_argument("--out", default=None)
a = ap.parse_args()
if not torch.cuda.is_available():
    sys.exit("rate_time.py measures on a CUDA device; none is visible")
pkg = load_package()
api = pkg.default_api()
api.set_device(0)
W, H, F = a.width, a.height, 64
STEPS = (1, 8, 16, 30, 45, 64)
FRONT = ("k_fwd", "k_hist_zero")
VALUE = ("k_coef_value_hist",)
REST = ("k_step_hists", "k_build_tables", "k_estimate_stream_bytes", "k_rate_sizes")

smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                     capture_output=True, text=True).stdout.strip().splitlines()
card = {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi": smi[0] if smi else "unavailable"}
st = torch.cuda.current_stream()
rgb = torch.empty(W * H * F * 3, dtype=torch.uint8, device="cuda")
api._chk(api.lib.alice_codec_synth_rgb_device(1, 0x5EED0001, W, H, F, C.c_void_p(rgb.data_ptr()), C.c_void_p(st.cuda_stream)))
torch.cuda.synchronize()
records = []


def median(v):
    v = sorted(v)
    return v[len(v) // 2]


def kernel_split(enc, calls=3):
    """device time per call of each kernel rate_curve_device launches (torch.profiler, CUDA activities; a kernel's total
    over the `calls` calls divided by its launch count, since the profiler may miss the first launches of a session)"""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(calls):
            enc.rate_curve_device(rgb.data_ptr(), W, H, F, stream=st.cuda_stream)
        torch.cuda.synchronize()
    groups = {"frontend_dump": 0.0, "value_hist": 0.0, "step_hists_tables_estimate": 0.0, "other": 0.0}
    names = {}
    for e in prof.key_averages():
        us = getattr(e, "self_device_time_total", None)
        if us is None:
            us = e.self_cuda_time_total
        if not us or not e.count:
            continue
        n = e.key
        # every kernel runs once per call; copies and memsets (several per call, microseconds) are averaged over calls
        per_call = us / 1000.0 / (e.count if "alice::" in n else calls)
        g = ("frontend_dump" if any(k in n for k in FRONT) else "value_hist" if any(k in n for k in VALUE)
             else "step_hists_tables_estimate" if any(k in n for k in REST) else "other")
        groups[g] += per_call
        names[n[:80]] = {"ms_per_launch": round(us / 1000.0 / e.count, 4), "launches": e.count}
    return {k: round(v, 4) for k, v in groups.items()}, names


for wavelet in ("cdf53", "cdf97", "haar"):
    enc = pkg.FrameEncoder(80, wavelet, api=api)
    enc.rate_curve_device(rgb.data_ptr(), W, H, F, stream=st.cuda_stream)   # warm-up (allocates the rate buffers)
    t = []
    for _ in range(a.reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(st)
        curve = enc.rate_curve_device(rgb.data_ptr(), W, H, F, stream=st.cuda_stream)
        e1.record(st)
        e1.synchronize()
        t.append(e0.elapsed_time(e1))
    try:
        split, kernels = kernel_split(enc)
    except Exception as ex:   # the split is an extra; the event timings above stand on their own
        split, kernels = {"not measured": repr(ex)}, {}
    # plain front-end and a trial encode (batch API CUDA-event stage times: [0] front-end, [1] tables, [2] rANS)
    b = pkg.ChunkBatch(80, wavelet, W, H, F, 1, stream=st.cuda_stream, api=api)
    fe, trial = [], []
    for _ in range(a.reps):
        b.encode_device([rgb.data_ptr()])
        ms = b.timings()
        fe.append(ms[0])
        trial.append(ms[0] + ms[1] + ms[2])
    b.close()
    tight = []
    for s in STEPS:
        q = pkg.quality_for_step(s)
        bs = pkg.ChunkBatch(q, wavelet, W, H, F, 1, stream=st.cuda_stream, api=api)
        bs.encode_device([rgb.data_ptr()])
        actual = len(bs.get_chunk(0).to_bytes())
        bs.close()
        tight.append({"step": s, "quality": q, "predicted": curve[q], "actual": actual,
                      "predicted_minus_actual": None if curve[q] is None else curve[q] - actual})
    rec = {"wavelet": wavelet, "shape": [W, H, F], "input": "G1 (synth seed 0x5EED0001)", "card": card,
           "rate_curve_ms": [round(x, 4) for x in t], "rate_curve_ms_median": round(median(t), 4),
           "rate_curve_split_ms": split, "rate_curve_kernels_ms": kernels,
           "rate_curve_ms_outside_kernels": (round(median(t) - sum(v for v in split.values() if isinstance(v, float)), 4)
                                             if "not measured" not in split else None),
           "plain_frontend_ms_median": round(median(fe), 4), "trial_encode_q80_ms_median": round(median(trial), 4),
           "bound_tightness": tight}
    records.append(rec)
    print(json.dumps(rec), flush=True)

if a.out:
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(records, f, indent=1)

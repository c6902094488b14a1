"""PSNR curve cost per 1920x1080x64 G1 chunk, for the three wavelets, on the GPU:

  * the whole psnr_curve_device call (host clock around the call, which ends in a synchronisation; median of --reps);
  * its kernels, from torch.profiler in a pass of its own: the dump front-end (k_fwd_fused with the coefficient dump)
    and the SSE launch (k_inv_fused in SSE mode, all 64 steps), device time per launch;
  * the same call for an input one byte off alignment, which takes the general path (64 x symbols, two-kernel
    back-end, squared-difference sum), median of --reps;
  * one trial encode + decode at quality 80 with the well-formed tables (host clock; the library's FrameEncoder /
    FrameDecoder on host buffers), for comparison.
The curve is checked against the trial: its PSNR at quality 80 equals the PSNR of the trial's decode.  Card name and
power limit are read in the same run.  Writes the records to --out (JSON) and prints them.

    python tools/psnr_curve_time.py [--reps 5] [--out profiles/r05_psnr_curve.json]
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402
from __graft_entry__ import load_package  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--reps", type=int, default=5)
ap.add_argument("--out", default=None)
a = ap.parse_args()
if not torch.cuda.is_available():
    sys.exit("psnr_curve_time.py measures on a CUDA device; none is visible")
pkg = load_package()
api = pkg.default_api()
api.set_device(0)
W, H, F = 1920, 1080, 64
N = W * H * F * 3

smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                     capture_output=True, text=True).stdout.strip().splitlines()
card = {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi": smi[0] if smi else "unavailable"}
st = torch.cuda.current_stream()
buf = torch.empty(N + 16, dtype=torch.uint8, device="cuda")
rgb = buf[:N]
api._chk(api.lib.alice_codec_synth_rgb_device(1, 0x5EED0001, W, H, F, C.c_void_p(rgb.data_ptr()), C.c_void_p(st.cuda_stream)))
torch.cuda.synchronize()
shifted = buf[1:N + 1]
shifted.copy_(rgb.clone())
rgb_aligned = torch.empty(N, dtype=torch.uint8, device="cuda")
rgb_aligned.copy_(shifted)
torch.cuda.synchronize()
host_rgb = rgb_aligned.cpu().numpy()


def median(v):
    v = sorted(v)
    return v[len(v) // 2]


def timed_curve(enc, ptr):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    curve, sse = enc.psnr_curve_device(ptr, W, H, F, stream=st.cuda_stream, with_sse=True)
    return (time.perf_counter() - t0) * 1e3, curve, sse


def kernel_us(enc, names=("k_fwd_fused", "k_inv_fused")):
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        enc.psnr_curve_device(rgb_aligned.data_ptr(), W, H, F, stream=st.cuda_stream)
        torch.cuda.synchronize()
    res = {}
    for e in prof.key_averages():
        us = getattr(e, "self_device_time_total", None)
        if us is None:
            us = e.self_cuda_time_total
        for n in names:
            if n in e.key and e.count:
                res[e.key[:80]] = {"us_per_launch": round(us / e.count, 1), "launches": e.count}
    return res


records = []
for wavelet in ("cdf53", "cdf97", "haar"):
    enc = pkg.FrameEncoder(80, wavelet, api=api, well_formed_tables=True)
    timed_curve(enc, rgb_aligned.data_ptr())                      # warm-up: buffers, module load
    fused = [timed_curve(enc, rgb_aligned.data_ptr()) for _ in range(a.reps)]
    timed_curve(enc, shifted.data_ptr())
    general = [timed_curve(enc, shifted.data_ptr()) for _ in range(a.reps)]
    assert all((r[2] == fused[0][2]).all() for r in fused + general), wavelet
    kern = kernel_us(enc)
    t0 = time.perf_counter()
    chunk = enc.encode(host_rgb, W, H, F)
    t1 = time.perf_counter()
    dec = pkg.FrameDecoder(api).decode(chunk)
    t2 = time.perf_counter()
    trial_psnr = api.psnr(host_rgb, dec)
    curve = fused[0][1]
    assert curve[80] == trial_psnr, (wavelet, curve[80], trial_psnr)
    rec = {"wavelet": wavelet, "shape": [W, H, F], "input": "G1 (synth seed 0x5EED0001)", "card": card,
           "curve_call_ms_median": round(median([r[0] for r in fused]), 3),
           "curve_call_ms_all": [round(r[0], 3) for r in fused],
           "general_path_call_ms_median": round(median([r[0] for r in general]), 3),
           "general_path_call_ms_all": [round(r[0], 3) for r in general],
           "kernels": kern,
           "trial_q80": {"encode_ms": round((t1 - t0) * 1e3, 1), "decode_ms": round((t2 - t1) * 1e3, 1),
                         "alc_bytes": len(chunk.to_bytes()), "psnr_db": trial_psnr},
           "curve_db": {str(q): round(v, 3) for q, v in curve.items() if q in (100, 98, 90, 80, 60, 40, 1)}}
    records.append(rec)
    print(json.dumps(rec), flush=True)

if a.out:
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(records, f, indent=1)

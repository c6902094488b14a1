"""Well-formed-tables encoding against the default encode, per 1920x1080x64 G1 chunk, for the three wavelets at a few
qualities, on the GPU:

  * .alc size of both modes;
  * PSNR of the real decode of each (the library's decode of the chunk it just encoded, psnr_device against the input);
  * the batch API's CUDA-event stage times of both modes: [0] front-end, [1] tables (in the well-formed mode this
    includes k_well_formed_hists), [2] rANS encode, [3] tables (decode), [4] rANS decode, [5] back-end;
  * the device time of k_well_formed_hists and k_build_tables in one encode (torch.profiler, a pass of its own).
The two modes run alternately.  Card name and power limit are read in the same run.  Writes the records to --out
(JSON) and prints them.

    python tools/well_formed_time.py [--reps 2] [--out profiles/r04_well_formed.json]
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
ap.add_argument("--reps", type=int, default=2)
ap.add_argument("--qualities", default="90,80,60,40")
ap.add_argument("--out", default=None)
a = ap.parse_args()
if not torch.cuda.is_available():
    sys.exit("well_formed_time.py measures on a CUDA device; none is visible")
pkg = load_package()
api = pkg.default_api()
api.set_device(0)
W, H, F = 1920, 1080, 64
N = W * H * F * 3

smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                     capture_output=True, text=True).stdout.strip().splitlines()
card = {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi": smi[0] if smi else "unavailable"}
st = torch.cuda.current_stream()
rgb = torch.empty(N, dtype=torch.uint8, device="cuda")
out = torch.empty(N, dtype=torch.uint8, device="cuda")
api._chk(api.lib.alice_codec_synth_rgb_device(1, 0x5EED0001, W, H, F, C.c_void_p(rgb.data_ptr()), C.c_void_p(st.cuda_stream)))
torch.cuda.synchronize()
STAGES = ("frontend", "tables_enc", "rans_encode", "tables_dec", "rans_decode", "backend")


def median(v):
    v = sorted(v)
    return v[len(v) // 2]


def run(batch):
    """one encode + decode on the batch: (.alc bytes, psnr, stage ms) or (None, None, error) where the encode aborts"""
    try:
        batch.encode_device([rgb.data_ptr()])
    except pkg.CodecError as e:
        return None, None, str(e)
    size = len(batch.get_chunk(0).to_bytes())
    enc_ms = batch.timings()[:3]
    batch.decode_device([out.data_ptr()])
    ms = enc_ms + batch.timings()[3:6]
    return size, api.psnr_device(rgb.data_ptr(), out.data_ptr(), N, st.cuda_stream), ms


def kernel_ms(batch, names=("k_well_formed_hists", "k_build_tables")):
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        batch.encode_device([rgb.data_ptr()])
        torch.cuda.synchronize()
    res = {}
    for e in prof.key_averages():
        us = getattr(e, "self_device_time_total", None)
        if us is None:
            us = e.self_cuda_time_total
        for n in names:
            if n in e.key and e.count:
                res[n] = {"us_per_launch": round(us / e.count, 2), "launches": e.count}
    return res


records = []
for wavelet in ("cdf53", "cdf97", "haar"):
    for q in [int(x) for x in a.qualities.split(",")]:
        batches = {m: pkg.ChunkBatch(q, wavelet, W, H, F, 1, stream=st.cuda_stream, api=api, well_formed_tables=m)
                   for m in (False, True)}
        res = {False: [], True: []}
        for _ in range(a.reps):
            for m in (False, True):
                res[m].append(run(batches[m]))
        rec = {"wavelet": wavelet, "quality": q, "step": pkg.quality_to_step(q), "shape": [W, H, F],
               "input": "G1 (synth seed 0x5EED0001)", "card": card}
        for m, name in ((False, "default"), (True, "well_formed")):
            size, psnr, ms = res[m][-1]
            if size is None:
                rec[name] = {"alc_bytes": None, "error": ms}
                continue
            stage = {s: round(median([r[2][i] for r in res[m]]), 4) for i, s in enumerate(STAGES)}
            rec[name] = {"alc_bytes": size, "psnr_db": round(psnr, 3), "stage_ms_median": stage,
                         "stage_ms_all": [[round(x, 4) for x in r[2]] for r in res[m]]}
        if q == 80:
            try:
                rec["well_formed_kernels"] = kernel_ms(batches[True])
            except Exception as ex:   # an extra; the event timings stand on their own
                rec["well_formed_kernels"] = {"not measured": repr(ex)}
        for b in batches.values():
            b.close()
        records.append(rec)
        print(json.dumps(rec), flush=True)

if a.out:
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(records, f, indent=1)

#!/usr/bin/env python
"""bench.py — BASELINE.json's metric on BASELINE.json's configs, measured on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload cfg2] [--impl reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N --steps K --warmup W

Workloads (config.workload; SURVEY.md §8d).  The default, and the one the driver runs, is cfg2:
    cfg1  CDF 5/3 q=90  1920x1080x64 chunks, encode + decode                      (BASELINE.json configs[0])
    cfg2  CDF 9/7 q=80  1920x1080x64 chunks, encode + decode                      (configs[1], the metric's config)
    cfg3  Haar   q=75  3840x2160x64 chunks, encode + decode, single GPU           (configs[2])
    cfg4  lossless (src/lossless.rs) 1920x1080x64: 2-D CDF 5/3 per frame + rANS   (configs[3])
    cfg5  8 chunks of 3840x2160x64, CDF 9/7 q=80, sharded over the GPUs (STRONG scaling), host gather of the
          .alc blobs inside the timed region                                      (configs[4])
One *step* = one pass of the hot path over a batch of independent chunks per GPU:
    encode : RGB -> YCoCg-R -> 3-D lifting -> quantise -> symbols + histograms -> frequency tables -> 3B rANS lanes
    decode : tables -> 3B rANS lanes -> dequantise -> inverse lifting -> RGB
`value`  = frames/s with the RGB inputs resident in HBM (whole job, all GPUs).  A chunk's symbol planes live in the RGB
           buffer of the previous chunk and its decode lands in its own, so a chunk in flight costs its RGB + its
           payload and a step leaves no input behind: the inputs are regenerated on the device INSIDE the timed region
           at the start of every step (config.inputs says so).
`e2e`    = the same metric through the C-ABI batch calls with HOST buffers (pinned): H2D of every RGB chunk, D2H of
           the .alc payloads, H2D of the payloads again for decode, D2H of every decoded RGB chunk; a few host threads
           each drive their own batch so that one batch's copies run under the other batches' rANS kernels.
`roofline` = the dominant kernel of the step by device time (a rANS launch: latency bound, symbols/s is its figure);
           `roofline_by_kernel` lists all four stages, incl. the wavelet/quantise front-end and back-end, whose
           algorithmic traffic is 6 B per pixel (3 in + 3 out, SURVEY.md §8d); achieved = algorithmic bytes /
           CUDA-event time on the launch stream, peak = measured HBM copy bandwidth (MEASURED_PEAKS.json).
`cpu_baseline` / `--impl reference` = the C oracle (a port of the reference's single-threaded Rust CPU path; no Rust
           toolchain exists in this image) on this box's host cores, on FULL chunks of the same workload.
Multi-GPU: chunks are independent, so each rank runs its own batch (weak scaling; cfg5: a fixed set of 8 chunks, strong
scaling), no collective on the data path; torch.distributed (NCCL) is used only for the barrier and the max-over-ranks
of the timed region, gloo for the host-side gather of cfg5.
"""
from __future__ import annotations

import argparse
import ctypes as C
import hashlib
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

SEED = 0x5EED0001
BYTES_PER_PX_ALG = 6.0          # SURVEY.md §8(d): 3 B in + 3 B out per RGB pixel, front-end or back-end
WORKLOADS = {
    "cfg1": dict(w=1920, h=1080, f=64, q=90, wavelet="cdf53", wbyte=0, golden="cfg1_cdf53_q90_1080p64",
                 name="CDF 5/3 q=90 1920x1080x64 encode+decode (BASELINE.json configs[0])"),
    "cfg2": dict(w=1920, h=1080, f=64, q=80, wavelet="cdf97", wbyte=1, golden="cfg2_cdf97_q80_1080p64",
                 name="CDF 9/7 q=80 1920x1080x64 encode+decode (BASELINE.json configs[1])"),
    "cfg3": dict(w=3840, h=2160, f=64, q=75, wavelet="haar", wbyte=2, golden="cfg3_haar_q75_4k64",
                 name="Haar q=75 3840x2160x64 encode+decode, single GPU (BASELINE.json configs[2])"),
    "cfg4": dict(w=1920, h=1080, f=64, q=None, wavelet="cdf53", wbyte=0, golden="cfg4_lossless_1080p64",
                 name="lossless (src/lossless.rs) 1920x1080x64: 2-D CDF 5/3 per frame, symbols, rANS per (64-frame set, "
                      "channel) stream, encode+decode (BASELINE.json configs[3])"),
    "cfg5": dict(w=3840, h=2160, f=64, q=80, wavelet="cdf97", wbyte=1, golden="cfg5_cdf97_q80_4k64_chunk0", total_chunks=8,
                 name="3840x2160x512 stream = 8 chunks of 64 frames, CDF 9/7 q=80, sharded over the GPUs "
                      "(BASELINE.json configs[4])"),
}


def _peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def _golden(name):
    p = os.path.join(ROOT, "tests", "golden", "fullsize.json")
    if not os.path.exists(p):
        return None
    return json.load(open(p)).get(name)


def sha(b):
    return hashlib.sha256(b).hexdigest()


# ------------------------------------------------------------------------------------------ --dump-outputs
# What the timed path returned in its last step, written so that two builds run with the same arguments can be compared
# output for output.  A chunk holds hundreds of MB, so each dumped chunk contributes its whole .alc header and a fixed,
# seeded sample of its payload and decoded bytes; the samples depend only on the chunk, never on the batch size.
DUMP_SEED = 20261020
DUMP_SAMPLES = 1 << 19                  # decoded bytes per dumped chunk (cfg4: decoded samples per channel)
DUMP_PAYLOAD_SAMPLES = 1 << 17          # payload bytes per dumped chunk (cfg4: per channel stream)
DUMP_MAX_BYTES = 64 * 10**6
ALC_HEADER_BYTES = 3138


def dump_chunk_ids(n):
    """Chunks 0-15 and every power of two below n: the same rows whatever batch size free memory allows."""
    return sorted(set(range(min(n, 16))) | {1 << k for k in range(n.bit_length()) if (1 << k) < n})


def dump_positions(n, count, key):
    """`count` sorted positions in [0, n), drawn with replacement from a generator seeded by DUMP_SEED and `key`."""
    import numpy as np
    return np.sort(np.random.default_rng([DUMP_SEED, key]).integers(0, n, count))


def payload_sample(blob, key):
    """DUMP_PAYLOAD_SAMPLES bytes of an encoded stream at seeded positions, as float32."""
    import numpy as np
    a = np.frombuffer(blob, dtype=np.uint8)
    return a[dump_positions(a.size, DUMP_PAYLOAD_SAMPLES, key)].astype(np.float32)


def write_dump(out_dir, arrays):
    """One DIR/<name>.npy per array (float32 or float64), DUMP_MAX_BYTES at most in all."""
    import numpy as np
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_MAX_BYTES:
        raise RuntimeError(f"--dump-outputs: {total} bytes exceed the {DUMP_MAX_BYTES}-byte limit")
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        assert a.dtype in (np.float32, np.float64), (name, a.dtype)
        np.save(os.path.join(out_dir, name + ".npy"), a)


# ------------------------------------------------------------------------------------------ clocks
class ClockSampler(threading.Thread):
    """Samples SM clock and throttle reasons of one GPU every 200 ms while the timed region runs."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.stop_flag, self.max_mhz, self.err = index, [], set(), False, None, None

    def run(self):
        try:
            import pynvml as nv
            nv.nvmlInit()
            h = nv.nvmlDeviceGetHandleByIndex(self.index)
            self.max_mhz = nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)
            names = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap",
                     0x80: "hw_power_brake_slowdown", 0x2: "applications_clocks_setting"}
            while not self.stop_flag:
                self.samples.append(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM))
                try:
                    mask = nv.nvmlDeviceGetCurrentClocksEventReasons(h)
                except Exception:
                    mask = nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                for bit, name in names.items():
                    if mask & bit:
                        self.reasons.add(name)
                time.sleep(0.2)
        except Exception as e:  # noqa: BLE001
            self.err = repr(e)

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": [], "error": self.err or "no samples"}
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2], "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(s)}


# ------------------------------------------------------------------------------------------ CPU arms
def _oracle_lossless_seconds(wl, seed):
    """BASELINE config 4 on the CPU oracle: per channel, 2-D CDF 5/3 of each frame, symbols, histogram, table, rANS
    encode; then rANS decode and the inverse 2-D transform (tests/golden/make_golden.py::lossless_case)."""
    import numpy as np
    import oracle as O
    w, h, f = wl["w"], wl["h"], wl["f"]
    rgb = O.generate(O.G1, w, h, f, seed)
    t0 = time.perf_counter()
    planes = O.rgb_bytes_to_ycocg_r(rgb)
    fs = w * h
    for p in planes:
        co = np.empty(fs * f, dtype=np.int32)
        for t in range(f):
            co[t * fs:(t + 1) * fs] = O.wavelet2d_forward(0, p[t * fs:(t + 1) * fs].astype(np.int32), w, h)
        sy = O.to_symbols(co)
        table = O.freq_table_from_histogram(O.build_histogram(sy))
        stream = O.rans_encode(sy, table)
        O.rans_decode(stream, sy.size, table)
        for t in range(f):
            O.wavelet2d_inverse(0, co[t * fs:(t + 1) * fs], w, h)
    return time.perf_counter() - t0


def _oracle_chunk_seconds(wl, seed):
    """One encode+decode round trip of one FULL chunk of the workload through the CPU oracle; returns seconds."""
    if wl["q"] is None:
        return _oracle_lossless_seconds(wl, seed)
    import oracle as O
    rgb = O.generate(O.G1, wl["w"], wl["h"], wl["f"], seed)
    t0 = time.perf_counter()
    alc = O.encode(rgb, wl["w"], wl["h"], wl["f"], wl["q"], wl["wbyte"])
    out = O.decode(alc)
    dt = time.perf_counter() - t0
    assert out.size == rgb.size
    return dt


def cpu_baseline_single(wl):
    dt = _oracle_chunk_seconds(wl, SEED)
    return {"value": round(wl["f"] / dt, 3), "unit": "frames/s", "cores": 1, "kind": "port",
            "sample": f"one full {wl['w']}x{wl['h']}x{wl['f']} G1 chunk of the workload, encode+decode through the C oracle "
                      f"(single thread, like the reference; a port, not the Rust crate); {dt:.1f} s"}


def run_reference_arm(args, wl):
    """--impl reference: the reference's CPU path on all host threads.  The reference is a Rust crate and no Rust
    toolchain exists in this image, so this is the C oracle port; the reference is single-threaded, so the threads run
    independent FULL chunks of the workload in parallel, one chunk per worker per step."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import psutil
    from concurrent.futures import ThreadPoolExecutor
    px = wl["w"] * wl["h"] * wl["f"]
    per_worker_gb = px * 22 / 2**30 + 0.3            # rgb + i16 planes + i32 volume + quantised + symbols (+ copies)
    avail_gb = psutil.virtual_memory().available / 2**30
    workers = max(1, min(os.cpu_count() or 1, int(avail_gb * 0.7 / per_worker_gb), 256))
    if wl.get("total_chunks"):
        workers = min(workers, wl["total_chunks"])
    import oracle as O
    O.lib()
    times = []
    with ThreadPoolExecutor(workers) as ex:
        for step in range(args.warmup + args.steps):
            t0 = time.perf_counter()
            list(ex.map(lambda i: _oracle_chunk_seconds(wl, SEED + i), range(workers)))  # ctypes releases the GIL
            dt = time.perf_counter() - t0
            if step >= args.warmup:
                times.append(dt)
    total = sum(times)
    value = workers * wl["f"] * len(times) / total
    sample = (f"{workers} worker threads x one full {wl['w']}x{wl['h']}x{wl['f']} G1 chunk each per step "
              f"(seeds SEED+i), encode+decode through the C oracle (port of the reference's CPU path)")
    line = {"impl": "reference", "metric": "1080p encode+decode frames/s" if wl["w"] == 1920 else "encode+decode frames/s",
            "value": round(value, 3), "unit": "frames/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": round(1000 * total / len(times), 3), "higher_is_better": True,
            "scaling": "strong" if wl.get("total_chunks") else "weak",
            "vs_baseline": None, "dtype": "int32", "data": "synthetic",
            "config": {"workload": wl["name"], "sample": sample},
            "cpu_baseline": {"value": round(value, 3), "unit": "frames/s", "cores": workers, "kind": "port",
                             "sample": sample},
            "e2e": {"value": round(value, 3), "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------ GPU arm
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="cfg2", choices=sorted(WORKLOADS))
    ap.add_argument("--chunks", type=int, default=0, help="chunks in flight per GPU (0 = sized from free HBM)")
    ap.add_argument("--e2e-threads", type=int, default=6, help="host threads (batches in flight) of the e2e leg")
    ap.add_argument("--e2e-steps", type=int, default=0, help="timed e2e steps (0 = --steps)")
    ap.add_argument("--e2e-fused", action="store_true", help="e2e batches take the fused front-end / back-end kernels (default: the small-shared-memory kernels, which can start beside the other batches' resident rANS streams)")
    ap.add_argument("--host-ring", type=int, default=8, help="distinct pinned host input chunks the e2e leg cycles through")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--verbose", action="store_true")
    ap.add_argument("--lib", default=None, help="experiment build of libalice_codec (debugging aid)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last step returned (rank 0's chunks: .alc lengths and "
                         "headers, seeded samples of the payloads and of the decoded RGB) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the CUDA path (--impl b200)")
    if args.warmup < 3:
        args.warmup = 3                      # timing rule: at least 3 warm-up steps
    wl = WORKLOADS[args.workload]
    if args.impl == "reference":
        return run_reference_arm(args, wl)
    if args.workload == "cfg4":
        import bench_lossless
        return bench_lossless.main(args, wl)

    import numpy as np
    import torch
    import torch.distributed as dist
    from __graft_entry__ import load_package
    # encoded payloads land in page-locked host buffers that the library pools (include/alice_codec.h); a batch of
    # several hundred chunks needs more than the library's modest default to reuse them step after step
    try:
        import psutil
        host_avail = psutil.virtual_memory().available
    except Exception:  # noqa: BLE001
        host_avail = 64 << 30
    n_local = int(os.environ.get("LOCAL_WORLD_SIZE", os.environ.get("WORLD_SIZE", "1")))
    os.environ.setdefault("ALICE_CODEC_PINNED_POOL_MB", str(max(1024, min(49152, int(host_avail * 0.5 / n_local) >> 20))))
    pkg = load_package()

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: libalice_codec has no CPU fallback")
    torch.cuda.set_device(local)
    try:                                     # run this rank's host threads (and first-touch its pinned buffers) on the CPUs
        import pynvml as nv                  # next to its GPU: at N = 8 the host side of the copies is the e2e limiter
        nv.nvmlInit()
        nv.nvmlDeviceSetCpuAffinity(nv.nvmlDeviceGetHandleByIndex(local))
    except Exception:  # noqa: BLE001
        pass
    gloo = None
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        # NCCL may print its version banner on stdout when the communicator is created; stdout carries exactly one
        # JSON line, so route fd 1 to stderr until the first collective has run
        sys.stdout.flush()
        saved_fd = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=torch.device("cuda", local))
            dist.all_reduce(torch.zeros(1, device="cuda"))
            torch.cuda.synchronize()
            if wl.get("total_chunks"):
                gloo = dist.new_group(backend="gloo")      # host-side gather of the .alc blobs (no data-path collective)
        finally:
            sys.stdout.flush()
            os.dup2(saved_fd, 1)
            os.close(saved_fd)
    api = pkg.Api(args.lib) if args.lib else pkg.default_api()
    api.set_device(local)
    stream = torch.cuda.current_stream()
    W, H, F = wl["w"], wl["h"], wl["f"]
    n_px = W * H * F
    rgb_bytes = 3 * n_px
    n_sm = torch.cuda.get_device_properties(local).multi_processor_count
    free_b, total_b = torch.cuda.mem_get_info()
    strong = bool(wl.get("total_chunks"))
    # payload budget per chunk: measured on one trial chunk (outside the timed region) + 1.5 %; the batch places its streams
    # back to back in one arena, so this is all the payload memory a chunk in flight costs
    trial = torch.empty(rgb_bytes, dtype=torch.uint8, device="cuda")
    api._chk(api.lib.alice_codec_synth_rgb_device(1, SEED + rank, W, H, F, C.c_void_p(trial.data_ptr()), C.c_void_p(stream.cuda_stream)))
    tb = pkg.ChunkBatch(wl["q"], wl["wavelet"], W, H, F, 1, stream=stream.cuda_stream, api=api)
    tb.encode_device([trial.data_ptr()])
    pay_chunk = int(tb.get_chunk(0).compressed_size * 1.015) + 3 * 65536
    tb.close()
    del trial, tb
    torch.cuda.empty_cache()
    free_b, total_b = torch.cuda.mem_get_info()
    if strong:
        from alice_codec_b200 import sharding
        my_chunks = sharding.chunks_of_rank(wl["total_chunks"], rank, world)
        B = len(my_chunks)
        seeds = [SEED + c for c in my_chunks]
    else:
        # per chunk in flight: its RGB buffer (which later holds the next chunk's symbol planes and decode) + its payload
        # + tables; fixed: one spare RGB buffer, the 4-byte scratch volume, head-room.
        # Cap: eight rANS streams per SM = two per warp scheduler (profiles/r02_switches.md).
        per_chunk = rgb_bytes + pay_chunk + 3 * (16384 + 256 * 16 + 2048)
        fixed = rgb_bytes + 12 * n_px + (3 << 29)
        cap = (8 * n_sm) // 3
        B = args.chunks or max(1, min(cap, int((free_b - fixed) // per_chunk)))
        # chunk ids follow the round-robin sharding of alice_codec_b200.sharding: rank r holds chunks r, r+world, ...
        seeds = [SEED + rank + i * world for i in range(B)]
    bufs = [torch.empty(rgb_bytes, dtype=torch.uint8, device="cuda") for _ in range(B + 1)]
    rgb_ptrs = [t.data_ptr() for t in bufs[1:]]          # chunk i is generated into bufs[i + 1] ...
    ws_ptrs = [t.data_ptr() for t in bufs[:B]]           # ... its symbol planes go to bufs[i] (consumed input of chunk i - 1) ...

    def synth_inputs():
        for i in range(B):
            api._chk(api.lib.alice_codec_synth_rgb_device(1, seeds[i], W, H, F, C.c_void_p(rgb_ptrs[i]),
                                                          C.c_void_p(stream.cuda_stream)))
    batch = pkg.ChunkBatch(wl["q"], wl["wavelet"], W, H, F, B, stream=stream.cuda_stream, api=api, shared_workspace=True,
                           payload_bytes_per_chunk=pay_chunk)
    assert batch.workspace_bytes() == rgb_bytes
    blobs_len = [0]

    def step():
        synth_inputs()                                   # the previous step decoded over the inputs
        batch.encode_device(rgb_ptrs, ws_ptrs)
        if strong:                                       # cfg5: the container is part of the job
            blobs = [batch.get_chunk(i).to_bytes() for i in range(B)]
            out = sharding.gather_stream(blobs, wl["total_chunks"], rank, world, group=gloo)
            if out is not None:
                blobs_len[0] = sum(len(b) for b in out)
        batch.decode_device(rgb_ptrs)                    # ... and its decode lands back in bufs[i + 1] (descending order)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(args.warmup):
        step()
    sampler = ClockSampler(local)
    barrier()
    sampler.start()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    stage_ms = np.zeros(8)
    t_wall0 = time.perf_counter()
    ev0.record(stream)
    for _ in range(args.steps):
        step()
        stage_ms += np.array(batch.timings())
    ev1.record(stream)
    barrier()
    t_wall = time.perf_counter() - t_wall0
    sampler.stop_flag = True
    ms_total = ev0.elapsed_time(ev1)
    if strong:
        ms_total = max(ms_total, 1000.0 * t_wall)        # the host gather runs after the last kernel of the encode
    if world > 1:
        t = torch.tensor([ms_total], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_total = float(t.item())
    sampler.join(timeout=2)
    stage_ms /= args.steps
    ms_step = ms_total / args.steps
    frames_per_step = (wl["total_chunks"] if strong else B * world) * F
    value = frames_per_step / (ms_step / 1000.0)

    # ---- correctness of what was just timed (bit-exactness is part of the metric)
    bit_exact = None
    g = _golden(wl["golden"])
    if rank == 0 and g:
        alc = batch.get_chunk(0).to_bytes()
        bit_exact = (sha(alc) == g["sha256_alc"] and sha(bufs[1].cpu().numpy().tobytes()) == g["sha256_decoded"])
    if rank == 0 and args.dump_outputs:
        ids = dump_chunk_ids(B)
        alcs = [batch.get_chunk(i).to_bytes() for i in ids]
        decoded = [bufs[i + 1][torch.from_numpy(dump_positions(rgb_bytes, DUMP_SAMPLES, i)).cuda()] for i in ids]
        write_dump(args.dump_outputs, {
            "chunk_index": np.array(ids, dtype=np.float64),
            "alc_len": np.array([len(a) for a in alcs], dtype=np.float64),
            "alc_header": np.stack([np.frombuffer(a[:ALC_HEADER_BYTES], dtype=np.uint8) for a in alcs]).astype(np.float32),
            "alc_payload_sample": np.stack([payload_sample(a[ALC_HEADER_BYTES:], i) for i, a in zip(ids, alcs)]),
            "decoded_rgb_sample": torch.stack(decoded).float().cpu().numpy()})
        del alcs, decoded

    # ---- rooflines, from the library's own CUDA events on the launch stream (averaged over the timed steps)
    peak, peak_src = _peaks()
    fe_ms, be_ms = float(stage_ms[0]), float(stage_ms[5])
    enc_ms, dec_ms = float(stage_ms[2]), float(stage_ms[4])
    alg_bytes = BYTES_PER_PX_ALG * n_px * B
    n_sym = 3 * n_px * B
    payload_bytes = 0
    if rank == 0:
        payload_bytes = sum(batch.get_chunk(i).compressed_size for i in range(min(B, 4))) / min(B, 4) * B
    traffic = {}
    tp = os.path.join(ROOT, "profiles", "r02_traffic.json")
    if os.path.exists(tp):
        traffic = json.load(open(tp)).get(args.workload, {})

    def rl(kernel, bound, bytes_alg, ms, traffic_bytes=None, note=None):
        ach = bytes_alg / (ms / 1000.0) / 1e9 if ms > 0 else 0.0
        d = {"bound": bound, "kernel": kernel, "achieved": round(ach, 1), "peak": peak, "unit": "GB/s",
             "frac": round(ach / peak, 4), "traffic": traffic_bytes, "peak_source": peak_src,
             "algorithmic_bytes_per_launch": bytes_alg, "ms": round(ms, 3), "share_of_step": round(ms / ms_step, 5)}
        if note:
            d["note"] = note
        return d
    lat_note = ("a serial recurrence per stream: LATENCY bound, not HBM bound; symbols/s per lane and per SM (stages) are its "
                "figures of merit, the GB/s here only places it against the HBM peak")
    by_kernel = {
        "frontend": rl("encode front-end: k_fwd_fused (+ k_hist_zero_bin_batch), one launch per chunk", "hbm", alg_bytes, fe_ms,
                       traffic.get("frontend_dram_bytes_per_chunk", 0) * B or None,
                       "6 B/px algorithmic (3 in + 3 out); issue bound: DESIGN.md 4.1"),
        "backend": rl("decode back-end: k_inv_fused, one launch per chunk", "hbm", alg_bytes, be_ms,
                      traffic.get("backend_dram_bytes_per_chunk", 0) * B or None, "6 B/px algorithmic"),
        "rans_encode": rl("k_rans_encode (one launch, 3 streams per chunk)", "latency", n_sym + payload_bytes, enc_ms, None, lat_note),
        "rans_decode": rl("k_rans_decode (one launch, 3 streams per chunk)", "latency", n_sym + payload_bytes, dec_ms, None, lat_note),
    }
    dominant = max(by_kernel, key=lambda k: by_kernel[k]["ms"])
    roofline = dict(by_kernel[dominant])
    roofline["dominant_of"] = {k: v["share_of_step"] for k, v in by_kernel.items()}
    stages = {"frontend_ms": round(fe_ms, 3), "tables_enc_ms": round(float(stage_ms[1]), 3),
              "rans_encode_ms": round(enc_ms, 3), "tables_dec_ms": round(float(stage_ms[3]), 3),
              "rans_decode_ms": round(dec_ms, 3), "backend_ms": round(be_ms, 3),
              "frontend_ms_per_chunk": round(fe_ms / B, 4), "backend_ms_per_chunk": round(be_ms / B, 4),
              "rans_lanes": 3 * B, "rans_lanes_per_sm": round(3 * B / n_sm, 2),
              "rans_encode_msym_s_per_lane": round(n_px / (enc_ms / 1000.0) / 1e6, 2) if enc_ms > 0 else None,
              "rans_decode_msym_s_per_lane": round(n_px / (dec_ms / 1000.0) / 1e6, 2) if dec_ms > 0 else None,
              "rans_encode_msym_s_per_sm": round(n_sym / (enc_ms / 1000.0) / 1e6 / n_sm, 2) if enc_ms > 0 else None,
              "rans_decode_msym_s_per_sm": round(n_sym / (dec_ms / 1000.0) / 1e6 / n_sm, 2) if dec_ms > 0 else None}
    if strong:
        stages["alc_stream_bytes_gathered_per_step"] = blobs_len[0]
    batch.close()
    del bufs, rgb_ptrs, ws_ptrs
    torch.cuda.empty_cache()

    # ---- e2e: the same metric through the host-buffer C-ABI calls, copies inside the timed region
    e2e = None
    if not args.no_e2e:
        e2e = run_e2e(args, wl, pkg, api, B, seeds, local, rank, world, barrier, g, pay_chunk)

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cpu = cpu_baseline_single(wl)

    if rank == 0:
        launches_per_step = B * (1 + 2 + 1) + 2 + 2 + 1        # per chunk: synth, k_fwd_fused + zero-bin, k_inv_fused; tables x2, rANS x2, size estimate
        line = {"metric": "1080p encode+decode frames/s" if W == 1920 else "encode+decode frames/s",
                "value": round(value, 2), "unit": "frames/s",
                "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(ms_step, 3),
                "higher_is_better": True, "scaling": "strong" if strong else "weak", "vs_baseline": None, "dtype": "int32",
                "data": "synthetic",
                "config": {"workload": wl["name"], "chunks_per_gpu_per_step": B, "frames_per_step": frames_per_step,
                           "inputs": "G1 tri+hash volumes (SURVEY.md Appendix D), one seed per chunk, regenerated on the device "
                                     "inside every timed step (a chunk's symbol planes live in the previous chunk's input buffer, "
                                     "its decode lands in its own)",
                           "l2": "inputs (%.1f GB per step per GPU) are far larger than the 126 MB L2" % (B * rgb_bytes / 1e9),
                           "parallelism": f"chunks sharded over {world} GPU(s), no data-path collective"
                                          + ("; host-side gloo gather of the .alc blobs to rank 0 inside the step" if strong else "")},
                "e2e": e2e, "gpu_launches": args.steps * launches_per_step, "roofline": roofline, "roofline_by_kernel": by_kernel,
                "stages": stages,
                "cpu_baseline": cpu if cpu is not None else ({"note": "measured on rank 0 at N=1 only"} if world > 1 else None),
                "clocks": sampler.summary(), "bit_exact_vs_oracle_digest": bit_exact}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def run_e2e(args, wl, pkg, api, B, seeds, local, rank, world, barrier, golden, pay_chunk):
    """T host threads, each driving its own ChunkBatch (own CUDA stream) over its share of the chunks through the
    host-pointer batch calls, so one batch's PCIe copies run under another batch's rANS kernels.  Host memory: the RGB
    inputs cycle through `--host-ring` distinct pinned chunks (the copy of every chunk still happens), every thread
    reads its decoded chunks back into a small pinned ring of its own."""
    import torch
    import torch.distributed as dist
    W, H, F = wl["w"], wl["h"], wl["f"]
    rgb_bytes = 3 * W * H * F
    T = max(1, min(args.e2e_threads, B))
    steps = args.e2e_steps or args.steps
    warm = args.warmup
    K = max(1, min(args.host_ring, B))
    stream0 = torch.cuda.current_stream()
    d_tmp = torch.empty(rgb_bytes, dtype=torch.uint8, device="cuda")
    h_in = []
    for k in range(K):
        api._chk(api.lib.alice_codec_synth_rgb_device(1, seeds[k], W, H, F, C.c_void_p(d_tmp.data_ptr()), C.c_void_p(stream0.cuda_stream)))
        t = torch.empty(rgb_bytes, dtype=torch.uint8).pin_memory()
        t.copy_(d_tmp)
        h_in.append(t)
    torch.cuda.synchronize()
    # link probe: one pinned chunk each way, three times (explains run-to-run differences of the e2e figure)
    link = {}
    h_probe = torch.empty(rgb_bytes, dtype=torch.uint8).pin_memory()
    for name, fn in (("h2d", lambda: d_tmp.copy_(h_in[0], non_blocking=True)), ("d2h", lambda: h_probe.copy_(d_tmp, non_blocking=True))):
        fn()
        torch.cuda.synchronize()
        tp0 = time.perf_counter()
        for _ in range(3):
            fn()
        torch.cuda.synchronize()
        link[name + "_gbs"] = round(3 * rgb_bytes / (time.perf_counter() - tp0) / 1e9, 1)
    del d_tmp, h_probe
    torch.cuda.empty_cache()
    # chunks per thread: the device holds (n + 1) staging buffers + the payload budget per batch
    free_b, _ = torch.cuda.mem_get_info()
    n_px = W * H * F
    per_chunk = rgb_bytes + pay_chunk + 3 * (16384 + 256 * 16 + 2048)
    fixed_per_batch = rgb_bytes + 12 * n_px
    Be = max(T, min(B, int((free_b - (3 << 29) - T * fixed_per_batch) // per_chunk)))
    try:                                                # the encoded chunks of a step live in pinned host memory
        import psutil
        Be = max(T, min(Be, int(psutil.virtual_memory().available * 0.5 / max(1, int(os.environ.get("LOCAL_WORLD_SIZE", world))) // max(1, pay_chunk))))
    except Exception:  # noqa: BLE001
        pass
    shares = [list(range(t, Be, T)) for t in range(T)]
    streams = [torch.cuda.Stream() for _ in range(T)]
    batches = [pkg.ChunkBatch(wl["q"], wl["wavelet"], W, H, F, len(shares[t]), stream=streams[t].cuda_stream, api=api,
                              shared_workspace=True, payload_bytes_per_chunk=pay_chunk, small_smem_kernels=not args.e2e_fused)
               for t in range(T)]
    KO = 4
    h_out = [[torch.empty(rgb_bytes, dtype=torch.uint8).pin_memory() for _ in range(KO)] for _ in range(T)]
    payload = [0] * T
    t_start, t_end = [0.0] * T, [0.0] * T
    step_s = [0.0] * T
    go = threading.Barrier(T + 1)
    errors = []

    keep = [None]

    def worker(t):
        try:
            api.set_device(local)                       # cudaSetDevice is per host thread
            hin = [h_in[i % K].data_ptr() for i in shares[t]]
            hout = [h_out[t][j % KO].data_ptr() for j in range(len(shares[t]))]
            go.wait()
            for it in range(warm + steps):
                if it == 2 and t > 0:                   # warm-up: put the batches out of phase, so that the copies of
                    time.sleep(step_s[t] * t / T)       # one run under the rANS kernels of the others
                if it == warm:
                    t_start[t] = time.perf_counter()
                ta = time.perf_counter()
                chunks = batches[t].encode_host(hin)    # H2D RGB, kernels, D2H headers + payload
                tb = time.perf_counter()
                payload[t] = sum(c.compressed_size + 3138 for c in chunks)
                batches[t].decode_host(chunks, hout)    # H2D payload, kernels, D2H RGB
                if t == 0 and it == warm + steps - 1:
                    keep[0] = chunks[0]                 # global chunk 0, decoded once more after the timed region
                del chunks                              # payload buffers go back to the library's pinned pool
                tc = time.perf_counter()
                if it == 1:
                    step_s[t] = tc - ta
                if args.verbose:
                    ms = batches[t].timings()
                    sys.stderr.write(f"[e2e] thread {t} it {it}: encode_host {tb - ta:.2f} s (fe {ms[0] / 1e3:.2f} rans {ms[2] / 1e3:.2f}), "
                                     f"decode_host {tc - tb:.2f} s (rans {ms[4] / 1e3:.2f} be {ms[5] / 1e3:.2f})\n")
            t_end[t] = time.perf_counter()
        except Exception as e:  # noqa: BLE001
            errors.append(repr(e))
            try:
                go.abort()
            except Exception:  # noqa: BLE001
                pass
    threads = [threading.Thread(target=worker, args=(t,)) for t in range(T)]
    for th in threads:
        th.start()
    barrier()
    go.wait()
    for th in threads:
        th.join()
    barrier()
    if errors:
        raise RuntimeError("e2e leg failed: " + "; ".join(errors))
    # the timed window runs from the first thread's first timed iteration to the last thread's last one
    dt = max(t_end) - min(t_start)
    if world > 1:
        tt = torch.tensor([dt], device="cuda", dtype=torch.float64)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        dt = float(tt.item())
    e2e_ok = None
    if rank == 0 and golden and keep[0] is not None:    # outside the timed region: chunk 0 of the last step, decoded alone
        alc_ok = sha(keep[0].to_bytes()) == golden["sha256_alc"]
        batches[0].decode_host([keep[0]], [h_out[0][0].data_ptr()])
        e2e_ok = alc_ok and sha(h_out[0][0].numpy().tobytes()) == golden["sha256_decoded"]
    keep[0] = None
    res = {"value": round(Be * F * world * steps / dt, 2), "unit": "frames/s",
           "h2d_bytes_per_step": Be * rgb_bytes + sum(payload), "d2h_bytes_per_step": Be * rgb_bytes + sum(payload),
           "chunks_per_step_per_gpu": Be, "host_threads": T, "steps": steps, "warmup": warm,
           "ms_per_step": round(1000 * dt / steps, 1),
           "host_buffers": f"pinned; RGB inputs cycle through {K} distinct chunks, outputs through {KO} buffers per thread",
           "timed_with": "host wall clock around synchronous C-ABI batch calls",
           "kernels": "fused front-end / back-end" if args.e2e_fused else "two-kernel front-end / back-end (ALICE_BATCH_SMALL_SMEM_KERNELS: they start beside the other batches' resident rANS streams)",
           "decoded_matches_oracle_digest": e2e_ok, "pinned_link_probe": link}
    for bt in batches:
        bt.close()
    return res


if __name__ == "__main__":
    main()

"""bench.py --workload cfg4: BASELINE.json configs[3], the lossless module (src/lossless.rs) over 1920x1080x64 frame sets.

One *step* = one pass over a batch of B independent frame sets: rgb_bytes_to_ycocg_r, LosslessEncoder::transform_2d of
every frame of every channel, to_symbols, histograms, frequency tables, one rANS stream per (frame set, channel); then
RansDecoder and inverse_2d.  The rANS streams of a frame set (3 lanes) run concurrently; frame sets run one after another
(a set holds 4.4 GB of i32 stage buffers, so few fit), which makes this workload a per-stream latency report: the figures
of merit are the 2-D transform's HBM fraction and the rANS decode symbols/s per stream.
"""
import ctypes as C
import json
import os
import time


def main(args, wl):
    import numpy as np
    import torch
    import bench as B
    from __graft_entry__ import load_package
    pkg = load_package()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if world > 1:
        raise SystemExit("cfg4 is a single-GPU per-stream report; run it with --gpus 1")
    torch.cuda.set_device(0)
    api = pkg.Api(args.lib) if args.lib else pkg.default_api()
    api.set_device(0)
    stream = torch.cuda.current_stream()
    W, H, F = wl["w"], wl["h"], wl["f"]
    n = W * H * F
    nb = args.chunks or 2
    d_rgb = [torch.empty(3 * n, dtype=torch.uint8, device="cuda") for _ in range(nb)]
    for i, t in enumerate(d_rgb):
        api._chk(api.lib.alice_codec_synth_rgb_device(1, B.SEED + i, W, H, F, C.c_void_p(t.data_ptr()), C.c_void_p(stream.cuda_stream)))
    ls = pkg.LosslessSet(W, H, F, stream=stream.cuda_stream, api=api)

    def step():
        ms = np.zeros(8)
        for t in d_rgb:
            ls.encode_device(t.data_ptr())
            ls.decode_device()
            ms += np.array(ls.timings())
        return ms
    for _ in range(args.warmup):
        step()
    sampler = B.ClockSampler(0)
    torch.cuda.synchronize()
    sampler.start()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    stage = np.zeros(8)
    ev0.record(stream)
    for _ in range(args.steps):
        stage += step()
    ev1.record(stream)
    torch.cuda.synchronize()
    sampler.stop_flag = True
    ms_step = ev0.elapsed_time(ev1) / args.steps
    stage /= args.steps * nb                 # per frame set
    sampler.join(timeout=2)
    if args.dump_outputs:                    # what the last step returned for its last frame set (nb - 1)
        streams = [ls.stream(c) for c in range(3)]
        inverse = ls.fetch("inverse")
        B.write_dump(args.dump_outputs, {
            "stream_len": np.array([len(s) for s in streams], dtype=np.float64),
            "histogram": ls.fetch("hist").astype(np.float64),
            "stream_sample": np.stack([B.payload_sample(s, c) for c, s in enumerate(streams)]),
            "inverse_sample": np.stack([inverse[c][B.dump_positions(n, B.DUMP_SAMPLES, c)] for c in range(3)]).astype(np.float32)})
        del streams, inverse
    # correctness of what was just timed: digests of every stage of set 0 against the oracle's (tests/golden)
    g = B._golden(wl["golden"])
    ls.encode_device(d_rgb[0].data_ptr())
    ls.decode_device()
    exact = None
    if g:
        exact = True
        for what, key in (("coeffs", "sha256_coeffs"), ("symbols", "sha256_symbols"), ("hist", "sha256_hist"),
                          ("decoded", "sha256_decoded_symbols"), ("inverse", "sha256_inverse")):
            got = ls.fetch(what)
            exact = exact and all(B.sha(got[c].tobytes()) == g[key][c] for c in range(3))
        exact = exact and all(B.sha(ls.stream(c)) == g["sha256_streams"][c] for c in range(3))
    stream_lens = [len(ls.stream(c)) for c in range(3)]
    peak, peak_src = B._peaks()
    n_sm = torch.cuda.get_device_properties(0).multi_processor_count
    fwd_ms, inv_ms, enc_ms, dec_ms = float(stage[1]), float(stage[5]), float(stage[3]), float(stage[4])
    alg2d = 8.0 * 3 * n                      # 4 B in + 4 B out per sample, three channels (SURVEY.md 8d: 8 B/sample)

    def rl(kernel, bound, bytes_alg, ms, note):
        ach = bytes_alg / (ms / 1000.0) / 1e9 if ms > 0 else 0.0
        return {"bound": bound, "kernel": kernel, "achieved": round(ach, 1), "peak": peak, "unit": "GB/s", "frac": round(ach / peak, 4),
                "traffic": None, "peak_source": peak_src, "algorithmic_bytes_per_launch": bytes_alg, "ms": round(ms, 3),
                "share_of_step": round(ms * nb / ms_step, 5), "note": note}
    by_kernel = {
        "transform_2d": rl("k_wxy<cdf53, forward>: 3 channels x 64 frames", "hbm", alg2d, fwd_ms, "8 B/sample algorithmic, one out-of-place pass"),
        "inverse_2d": rl("k_wxy<cdf53, inverse>", "hbm", alg2d, inv_ms, "8 B/sample algorithmic"),
        "rans_encode": rl("k_rans_encode, 3 streams", "latency", 3 * n + sum(stream_lens), enc_ms, "serial recurrence per stream: symbols/s per stream is the figure of merit"),
        "rans_decode": rl("k_rans_decode, 3 streams", "latency", 3 * n + sum(stream_lens), dec_ms, "serial recurrence per stream: symbols/s per stream is the figure of merit"),
    }
    dominant = max(by_kernel, key=lambda k: by_kernel[k]["ms"])
    roofline = dict(by_kernel[dominant])
    cpu = None
    if not args.no_cpu_baseline:
        cpu = B.cpu_baseline_single(wl)
    line = {"metric": "1080p lossless transform+rANS round-trip frames/s", "value": round(nb * F / (ms_step / 1000.0), 2), "unit": "frames/s",
            "n_gpus": 1, "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(ms_step, 3), "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "int32", "data": "synthetic",
            "config": {"workload": wl["name"], "frame_sets_per_step": nb, "inputs": "G1 tri+hash volumes generated on the device",
                       "l2": "every stage buffer of a frame set (0.5 GB per channel) is larger than the 126 MB L2",
                       "parallelism": "frame sets one after another, the three channel streams of a set concurrently"},
            "e2e": None, "gpu_launches": args.steps * nb * 16, "roofline": roofline, "roofline_by_kernel": by_kernel,
            "stages": {"colour_ms": round(float(stage[0]), 3), "transform_2d_ms": round(fwd_ms, 3), "symbols_hist_tables_ms": round(float(stage[2]), 3),
                       "rans_encode_ms": round(enc_ms, 1), "rans_decode_ms": round(dec_ms, 1), "inverse_2d_ms": round(inv_ms, 3),
                       "rans_decode_msym_s_per_stream": round(n / (dec_ms / 1000.0) / 1e6, 2), "rans_encode_msym_s_per_stream": round(n / (enc_ms / 1000.0) / 1e6, 2),
                       "rans_streams_in_flight": 3, "rans_decode_msym_s_per_sm_hosting_a_stream": round(n / (dec_ms / 1000.0) / 1e6, 2),
                       "stream_bytes": stream_lens},
            "cpu_baseline": cpu, "clocks": sampler.summary(), "bit_exact_vs_oracle_digest": exact}
    print(json.dumps(line), flush=True)
    ls.close()

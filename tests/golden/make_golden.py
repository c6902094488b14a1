"""Generates tests/golden/fullsize.json: sha256 digests of the ORACLE's outputs at BASELINE.json's full sizes.

The reference is a Rust crate and cannot run in this image (no rustc/cargo), so these are digests of the CPU
oracle (oracle/alice_oracle.c), which is itself pinned by the reference's exact-value tests and the SURVEY
Appendix C vectors (tests/test_oracle.py).  Run on a CPU box:  python tests/golden/make_golden.py [names...]
The -m gpu tests compare the CUDA path's digests with these without re-running the oracle at full size.
"""
import hashlib
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
import oracle as O  # noqa: E402

OUT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "fullsize.json")
CASES = {
    # name: (kind, w, h, f, quality, wavelet, seed)        BASELINE.json configs
    "cfg1_cdf53_q90_1080p64": (O.G1, 1920, 1080, 64, 90, 0, O.SEED),
    "cfg2_cdf97_q80_1080p64": (O.G1, 1920, 1080, 64, 80, 1, O.SEED),
    "cfg3_haar_q75_4k64": (O.G1, 3840, 2160, 64, 75, 2, O.SEED),
    "cfg5_cdf97_q80_4k64_chunk0": (O.G1, 3840, 2160, 64, 80, 1, O.SEED),
    "cfg5_cdf97_q80_4k64_chunk1": (O.G1, 3840, 2160, 64, 80, 1, O.SEED + 1),
    "cfg5_cdf97_q80_4k64_chunk2": (O.G1, 3840, 2160, 64, 80, 1, O.SEED + 2),
    "cfg5_cdf97_q80_4k64_chunk3": (O.G1, 3840, 2160, 64, 80, 1, O.SEED + 3),
    "cfg5_cdf97_q80_4k64_chunk4": (O.G1, 3840, 2160, 64, 80, 1, O.SEED + 4),
    "cfg5_cdf97_q80_4k64_chunk5": (O.G1, 3840, 2160, 64, 80, 1, O.SEED + 5),
    "cfg5_cdf97_q80_4k64_chunk6": (O.G1, 3840, 2160, 64, 80, 1, O.SEED + 6),
    "cfg5_cdf97_q80_4k64_chunk7": (O.G1, 3840, 2160, 64, 80, 1, O.SEED + 7),
    "noise_cdf53_q90_1080p8": (O.G2, 1920, 1080, 8, 90, 0, O.SEED),
    "odd_cdf97_q80_1919x1079x63": (O.G1, 1919, 1079, 63, 80, 1, O.SEED),
}


def sha(b):
    return hashlib.sha256(b).hexdigest()


def lossless_case(w, h, f, seed):
    """BASELINE config 4 (SURVEY.md 8d-4): LosslessEncoder::transform_2d (= Wavelet2D::cdf53, lossless.rs:45-54) on
    every frame of the Y/Co/Cg planes, to_symbols of the coefficients (step 1, wrapping), histogram, table, one rANS
    stream per (64-frame set, channel), RansDecoder, and inverse_2d of the coefficients."""
    t0 = time.time()
    rgb = O.generate(O.G1, w, h, f, seed)
    planes = O.rgb_bytes_to_ycocg_r(rgb)
    out = {"kind": O.G1, "w": w, "h": h, "f": f, "seed": seed, "sha256_rgb_in": sha(rgb.tobytes()),
           "sha256_coeffs": [], "sha256_symbols": [], "sha256_hist": [], "stream_lens": [], "sha256_streams": [],
           "sha256_decoded_symbols": [], "sha256_inverse": [], "decoded_symbols_equal_encoded": []}
    fs = w * h
    for p in planes:
        co = np.empty(fs * f, dtype=np.int32)
        inv = np.empty(fs * f, dtype=np.int32)
        for t in range(f):
            img = p[t * fs:(t + 1) * fs].astype(np.int32)
            fw = O.wavelet2d_forward(0, img, w, h)
            co[t * fs:(t + 1) * fs] = fw
            inv[t * fs:(t + 1) * fs] = O.wavelet2d_inverse(0, fw, w, h)
        sy = O.to_symbols(co)
        hist = O.build_histogram(sy)
        table = O.freq_table_from_histogram(hist)
        stream = O.rans_encode(sy, table)
        dec = O.rans_decode(stream, sy.size, table)
        out["sha256_coeffs"].append(sha(co.tobytes()))
        out["sha256_symbols"].append(sha(sy.tobytes()))
        out["sha256_hist"].append(sha(np.asarray(hist, dtype=np.uint32).tobytes()))
        out["stream_lens"].append(len(stream))
        out["sha256_streams"].append(sha(stream))
        out["sha256_decoded_symbols"].append(sha(dec.tobytes()))
        out["sha256_inverse"].append(sha(inv.tobytes()))
        out["decoded_symbols_equal_encoded"].append(bool(np.array_equal(dec, sy)))
    out["oracle_seconds"] = {"total": round(time.time() - t0, 2)}
    return out


LOSSLESS_CASES = {"cfg4_lossless_1080p64": (1920, 1080, 64, O.SEED)}
BENCH_DUMP_OUT = os.path.join(os.path.dirname(OUT), "bench_dump_cfg2_chunk0.npz")


def bench_dump_case():
    """What `bench.py --dump-outputs` writes for chunk 0 of its default workload (cfg2), from the oracle, as uint8:
    the .alc header, and the payload and decoded RGB bytes at the bench's seeded sample positions."""
    import bench
    kind, w, h, f, q, wv, seed = CASES["cfg2_cdf97_q80_1080p64"]
    alc = O.encode(O.generate(kind, w, h, f, seed), w, h, f, q, wv)
    dec = O.decode(alc)
    payload = np.frombuffer(alc[bench.ALC_HEADER_BYTES:], dtype=np.uint8)
    np.savez_compressed(BENCH_DUMP_OUT, alc_len=np.array([len(alc)]),
                        alc_header=np.frombuffer(alc[:bench.ALC_HEADER_BYTES], dtype=np.uint8),
                        alc_payload_sample=payload[bench.dump_positions(payload.size, bench.DUMP_PAYLOAD_SAMPLES, 0)],
                        decoded_rgb_sample=dec[bench.dump_positions(dec.size, bench.DUMP_SAMPLES, 0)])


def main():
    names = sys.argv[1:] or list(CASES) + list(LOSSLESS_CASES) + ["bench_dump"]
    res = json.load(open(OUT)) if os.path.exists(OUT) else {}
    for name in names:
        if name == "bench_dump":
            bench_dump_case()
            continue
        if name in LOSSLESS_CASES:
            res[name] = lossless_case(*LOSSLESS_CASES[name])
            print(name, res[name]["stream_lens"], res[name]["oracle_seconds"], flush=True)
            json.dump(res, open(OUT, "w"), indent=1, sort_keys=True)
            continue
        kind, w, h, f, q, wv, seed = CASES[name]
        t0 = time.time()
        rgb = O.generate(kind, w, h, f, seed)
        t1 = time.time()
        alc, coeffs, syms = O.encode(rgb, w, h, f, q, wv, stages=True)
        t2 = time.time()
        dec = O.decode(alc)
        t3 = time.time()
        lens = [int.from_bytes(alc[18 + c * 1040:18 + c * 1040 + 4], "little") for c in range(3)]
        res[name] = {
            "kind": kind, "w": w, "h": h, "f": f, "quality": q, "wavelet": wv, "seed": seed,
            "sha256_rgb_in": sha(rgb.tobytes()), "alc_len": len(alc), "stream_lens": lens,
            "sha256_alc": sha(alc), "sha256_header": sha(alc[:3138]),
            "sha256_coeffs": [sha(c.tobytes()) for c in coeffs], "sha256_symbols": [sha(s.tobytes()) for s in syms],
            "sha256_decoded": sha(dec.tobytes()),
            "oracle_seconds": {"generate": round(t1 - t0, 2), "encode": round(t2 - t1, 2), "decode": round(t3 - t2, 2)},
        }
        print(name, res[name]["alc_len"], res[name]["oracle_seconds"], flush=True)
        del rgb, alc, coeffs, syms, dec
        json.dump(res, open(OUT, "w"), indent=1, sort_keys=True)


if __name__ == "__main__":
    main()

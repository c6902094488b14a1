"""Parity checks shared by the CPU (SIMT-emulator) and GPU test tiers.

Every function takes an `Api` (one loaded libalice_codec build) and compares it, through the
C ABI, with the CPU oracle (oracle/alice_oracle.c) on the same seeded inputs.  The bar is
bit-exact equality at every stage: wavelet coefficients, symbol planes, histograms, rANS
streams, .alc bytes and decoded RGB (the path is integer/byte work throughout).
"""
import hashlib
import os

import numpy as np

import oracle as O
from __graft_entry__ import load_package

pkg = load_package()
WV = {0: "cdf53", 1: "cdf97", 2: "haar"}
EMUL_BUILD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "emul", "_build")


def device_of(api):
    """torch device of the buffers that `api`'s device-pointer calls take.  The emulator builds (tests/emul/_build) run
    their kernels on the host and treat host memory as device memory, also on a machine that has a GPU."""
    return "cpu" if os.path.abspath(api.path).startswith(EMUL_BUILD + os.sep) else "cuda"


def check_encode_decode(api, kind, w, h, f, quality, wavelet, seed=O.SEED, stages=True):
    """FrameEncoder::encode -> to_bytes -> from_bytes -> FrameDecoder::decode vs the oracle, stage by stage."""
    rgb = O.generate(kind, w, h, f, seed)
    enc = pkg.FrameEncoder(quality, WV[wavelet], api=api)
    if stages:
        chunk, coeffs, syms = enc.encode_stages(rgb, w, h, f)
        ralc, rco, rsy = O.encode(rgb, w, h, f, quality, wavelet, stages=True)
        for c in range(3):
            assert np.array_equal(coeffs[c], rco[c]), f"wavelet coefficients differ (channel {c})"
            assert np.array_equal(syms[c], rsy[c]), f"symbol plane differs (channel {c})"
            hdr = chunk.channel_header(c)
            assert np.array_equal(hdr["histogram"], O.build_histogram(rsy[c])), f"histogram differs (channel {c})"
            assert hdr["quant_step"] == hdr["quant_dead_zone"] == O.quality_to_step(quality)
    else:
        chunk = enc.encode(rgb, w, h, f)
        ralc = O.encode(rgb, w, h, f, quality, wavelet)
    alc = chunk.to_bytes()
    assert len(alc) == len(ralc), f".alc length {len(alc)} != oracle {len(ralc)}"
    assert alc == ralc, ".alc bytes differ"
    assert (chunk.width, chunk.height, chunk.frames, chunk.wavelet) == (w, h, f, WV[wavelet])
    back = pkg.EncodedChunk.from_bytes(ralc, api=api)
    dec = pkg.FrameDecoder(api=api)
    if stages:
        out, dsyms = dec.decode_stages(back)
        rrgb, rdsy = O.decode(ralc, stages=True)
        for c in range(3):
            assert np.array_equal(dsyms[c], rdsy[c]), f"decoded symbol plane differs (channel {c})"
    else:
        out = dec.decode(back)
        rrgb = O.decode(ralc)
    assert out.size == w * h * f * 3
    assert np.array_equal(out, rrgb), "decoded RGB differs"
    return alc, out


def check_kat(api, row):
    kind, w, h, f, q, wv, alen, sha_alc, sha_rgb = row
    alc, out = check_encode_decode(api, kind, w, h, f, q, wv)
    assert len(alc) == alen
    assert hashlib.sha256(alc).hexdigest() == sha_alc
    assert hashlib.sha256(out.tobytes()).hexdigest() == sha_rgb


def check_wavelet_api(api, rng, shapes_1d, shapes_2d, shapes_3d, amplitude=1 << 20):
    for wv in (0, 1, 2):
        for n in shapes_1d:
            x = rng.integers(-amplitude, amplitude, n, dtype=np.int64).astype(np.int32)
            fw = api.wavelet1d(wv, x)
            assert np.array_equal(fw, O.wavelet1d_forward(wv, x)), (wv, n)
            assert np.array_equal(api.wavelet1d(wv, fw, inverse=True), O.wavelet1d_inverse(wv, fw)), (wv, n)
        for (w, h) in shapes_2d:
            x = rng.integers(-amplitude, amplitude, w * h, dtype=np.int64).astype(np.int32)
            fw = api.wavelet2d(wv, x, w, h)
            assert np.array_equal(fw, O.wavelet2d_forward(wv, x, w, h)), (wv, w, h)
            assert np.array_equal(api.wavelet2d(wv, fw, w, h, inverse=True), O.wavelet2d_inverse(wv, fw, w, h))
        for (w, h, d) in shapes_3d:
            x = rng.integers(-amplitude, amplitude, w * h * d, dtype=np.int64).astype(np.int32)
            fw = api.wavelet3d(wv, x, w, h, d)
            assert np.array_equal(fw, O.wavelet3d_forward(wv, x, w, h, d)), (wv, w, h, d)
            assert np.array_equal(api.wavelet3d(wv, fw, w, h, d, inverse=True),
                                  O.wavelet3d_inverse(wv, fw, w, h, d))


def check_wavelet_fast_path(api, shapes_2d=((8, 2), (16, 10), (128, 6), (244, 8), (480, 34)),
                            shapes_3d=((8, 2, 2), (16, 6, 4), (124, 8, 6), (256, 4, 64), (132, 36, 10))):
    """Shapes with w % 4 == 0 and even h (and d) take the per-pass kernels of k_wavelet_i32.cu (strips with and without
    interior lanes, several row segments, full-range i32 data for the i64 lifting product)."""
    rng = np.random.default_rng(11)
    check_wavelet_api(api, rng, [], shapes_2d, shapes_3d, amplitude=1 << 20)
    check_wavelet_api(api, rng, [], shapes_2d[:3], shapes_3d[:3], amplitude=(1 << 31) - 1)


def check_wavelet_extremes(api):
    """i32 wrap-around and the i64 lifting product (wavelet.rs:193-195): full-range inputs."""
    rng = np.random.default_rng(7)
    x = rng.integers(-(1 << 31), (1 << 31) - 1, 4096, dtype=np.int64).astype(np.int32)
    for wv in (0, 1, 2):
        fw = api.wavelet1d(wv, x)
        assert np.array_equal(fw, O.wavelet1d_forward(wv, x))
        assert np.array_equal(api.wavelet1d(wv, fw, inverse=True), O.wavelet1d_inverse(wv, fw))


def check_quant_api(api, rng, n=20000):
    vals = rng.integers(-70000, 70000, n, dtype=np.int64).astype(np.int32)
    vals[:8] = [0, 1, -1, 2147483647, -2147483647, -2147483648, 127, -128]
    for step, dz in [(1, 1), (8, 8), (14, 14), (17, 17), (33, 49), (64, 64), (5, 0), (128, 192), (1000, 1500)]:
        assert np.array_equal(api.quantize_buffer(step, dz, vals), O.quantize_buffer(step, dz, vals)), (step, dz)
        assert np.array_equal(api.fast_quantize_buffer(step, dz, vals), O.fast_quantize_buffer(step, dz, vals))
        q = O.quantize_buffer(step, dz, vals)
        assert np.array_equal(api.dequantize_buffer(step, q), O.dequantize_buffer(step, q))
    small = np.arange(-10000, 10001, dtype=np.int32)
    for step in (1, 2, 3, 7, 8, 14, 17, 33, 64, 100, 127, 128):  # quant.rs:1145-1150
        assert np.array_equal(api.fast_quantize_buffer(step, step, small), api.quantize_buffer(step, step, small))
    coeffs = rng.integers(-300, 300, n, dtype=np.int64).astype(np.int32)
    sy = api.to_symbols(coeffs)
    assert np.array_equal(sy, O.to_symbols(coeffs))                      # incl. the `as u8` wrap (quant.rs:555-560)
    assert np.array_equal(api.from_symbols(sy), O.from_symbols(sy))
    assert np.array_equal(api.build_histogram(sy), O.build_histogram(sy))
    for bad in (0, -5):                                                   # quant.rs:1116-1122
        try:
            api.fast_quantize_buffer(bad, bad, [1])
            raise AssertionError("InvalidQuantStep expected")
        except pkg.CodecError as e:
            assert e.kind == "InvalidQuantStep"


def check_rdo(api, rng):
    for q in (0, 10, 50, 75, 90, 100, 200):
        assert api.rdo_bpp_from_quality(q) == O.rdo_bpp_from_quality(q)
    for n in (0, 1, 7, 1000, 4097):
        x = rng.integers(-500, 500, n, dtype=np.int64).astype(np.int32)
        for sb in range(8):
            for bpp in (0.1, 1.0, O.rdo_bpp_from_quality(75)):
                assert api.rdo_compute_quantizer(bpp, x, sb) == O.rdo_compute_quantizer(bpp, x, sb), (n, sb, bpp)


def _octants(vol, w, h, d):
    """the 8 sub-band slices of a forward-transformed volume in SubBand3D order (x, y, t letters), row-major"""
    v = np.asarray(vol).reshape(d, h, w)
    hx, hy, ht = w // 2, h // 2, d // 2
    out = []
    for sb in range(8):
        x0, y0, t0 = (hx if sb & 4 else 0), (hy if sb & 2 else 0), (ht if sb & 1 else 0)
        out.append(np.ascontiguousarray(v[t0:t0 + ht, y0:y0 + hy, x0:x0 + hx]).reshape(-1))
    return out


def check_rdo_exact_variance(api, rng, sizes=(1, 2, 31, 1024, 1025, 5000, 40000)):
    """AnalyticalRDO::estimate_variance (quant.rs:415-435): the f64 sum is order dependent; the device result must
    equal the sequential loop bit for bit, across binade changes, exact ties and absorbed terms."""
    cases = []
    for n in sizes:
        cases.append(rng.integers(-500, 500, n, dtype=np.int64))
        cases.append(rng.integers(-(1 << 31), 1 << 31, n, dtype=np.int64))                 # full i32 range
        cases.append(np.where(rng.random(n) < 0.97, 0, rng.integers(-40000, 40000, n)))    # sparse, leading zeros
        cases.append(rng.integers(0, 2, n, dtype=np.int64) * 2 - 1)                        # +-1: mean ~ 0, many ties
        x = rng.integers(-3, 4, n, dtype=np.int64)
        x[n // 2:] *= 1 << 20                                                              # small terms absorbed later
        cases.append(x)
        t = np.empty(n + (n & 1), np.int64)
        t[0::2], t[1::2] = 1 << 20, 1 - (1 << 20)                                          # mean 0.5: every term ends in .25,
        cases.append(t)                                                                    # exact ties once ulp = 0.5
        cases.append(np.full(n, 7))                                                        # variance 0 -> floor 1.0
        cases.append(np.concatenate([np.full(n // 2, 1 << 30), np.zeros(n - n // 2, np.int64)]))
    for x in cases:
        x = np.asarray(x, dtype=np.int64).astype(np.int32)
        got, want = api.rdo_estimate_variance(x), O.rdo_estimate_variance(x)
        assert np.float64(got).tobytes() == np.float64(want).tobytes(), (x.size, got, want)


def check_rdo_octants(api, rng, shapes=((8, 6, 4), (16, 10, 6), (9, 7, 5), (2, 2, 2), (32, 18, 64))):
    for (w, h, d) in shapes:
        vol = (rng.standard_normal(w * h * d) * rng.choice([3, 50, 3000], w * h * d)).astype(np.int32)
        for bpp in (0.1, O.rdo_bpp_from_quality(75), 24.0):
            want = [O.rdo_compute_quantizer(bpp, o, sb) for sb, o in enumerate(_octants(vol, w, h, d))]
            assert api.rdo_compute_all_quantizers(bpp, vol, w, h, d) == want, (w, h, d, bpp)
            q, quants = api.rdo_quantize_volume(bpp, vol, w, h, d)
            assert quants == want
            # FastQuantizer == Quantizer (quant.rs:1145-1150), so the oracle's plain quantiser is the check
            v3 = vol.reshape(d, h, w)
            ref = np.empty_like(v3)
            hx, hy, ht = w // 2, h // 2, d // 2
            for t in range(d):
                for y in range(h):
                    for xs, sbx in ((slice(0, hx), 0), (slice(hx, w), 4)):
                        sb = sbx | (2 if y >= hy else 0) | (1 if t >= ht else 0)
                        ref[t, y, xs] = O.fast_quantize_buffer(want[sb][0], want[sb][1], v3[t, y, xs])
            assert np.array_equal(q.reshape(d, h, w), ref), (w, h, d, bpp)


def check_colour(api, rng, n=5000):
    rgb = rng.integers(0, 256, 3 * n, dtype=np.int64).astype(np.uint8)
    rgb[:12] = [0, 0, 0, 255, 255, 255, 255, 0, 0, 0, 0, 255]
    y, co, cg = api.rgb_to_ycocg_r(rgb)
    ry, rco, rcg = O.rgb_bytes_to_ycocg_r(rgb)
    assert np.array_equal(y, ry) and np.array_equal(co, rco) and np.array_equal(cg, rcg)
    assert np.array_equal(api.ycocg_r_to_rgb(y, co, cg), rgb)            # color.rs:429-461 exact round trip
    wild = [rng.integers(-32768, 32768, n, dtype=np.int64).astype(np.int16) for _ in range(3)]
    assert np.array_equal(api.ycocg_r_to_rgb(*wild), O.ycocg_r_to_rgb_bytes(*wild))   # i16 wrap + clamp


def _check_rans(api, sy, hist):
    hist = np.asarray(hist, np.uint32)
    t = O.freq_table_from_histogram(hist)
    cum, freq, lut = api.freq_table_from_histogram(hist)
    n = hist.size
    assert np.array_equal(cum, t.cum_np()[:n]) and np.array_equal(freq, t.freq_np()[:n])
    assert np.array_equal(lut, t.lut_np())
    try:
        ref = O.rans_encode(sy, t)
    except O.OracleError:
        try:
            api.rans_encode(sy, hist)
            raise AssertionError("reference panics (zero frequency); CUDA path must report it")
        except pkg.CodecError as e:
            assert e.kind == "ReferencePanic"
        return
    got = api.rans_encode(sy, hist)
    assert got == ref, "rANS stream differs"
    assert np.array_equal(api.rans_decode(ref, sy.size, hist), O.rans_decode(ref, sy.size, t)), "rANS decode differs"
    # decoders must also agree on truncated / empty input (rans.rs:341-347, 363-368)
    for cut in (0, 3, 4, len(ref) // 2):
        assert np.array_equal(api.rans_decode(ref[:cut], min(sy.size, 300), hist),
                              O.rans_decode(ref[:cut], min(sy.size, 300), t))


def check_rans_api(api, rng, n=6000):
    # well-formed skewed table, low-numbered symbols (rans.rs:738-787)
    p = np.array([0.7, 0.1, 0.08, 0.05, 0.04, 0.02, 0.01])
    sy = rng.choice(7, n, p=p).astype(np.uint8)
    _check_rans(api, sy, O.build_histogram(sy))
    # 4-bin histogram (rans.rs:819-830) and a uniform table via an all-zero histogram (rans.rs:158-189)
    sy4 = rng.integers(0, 4, n).astype(np.uint8)
    _check_rans(api, sy4, [100, 200, 300, 400])
    syu = rng.integers(0, 256, n).astype(np.uint8)
    _check_rans(api, syu, np.zeros(256, np.uint32))
    _check_rans(api, rng.integers(0, 16, 500).astype(np.uint8), np.zeros(16, np.uint32))
    # gappy histogram -> malformed table, freq[255] wraps (SURVEY §0.7): streams must still be identical
    sy = (rng.choice(60, n, p=np.r_[0.5, np.full(59, 0.5 / 59)]) * 2 + 1).astype(np.uint8)
    sy[rng.integers(0, n, n // 4)] = 0
    _check_rans(api, sy, O.build_histogram(sy))
    # symbol 255 in use with the wrapped frequency; full-range noise; single dominant symbol; tiny inputs
    sy = rng.integers(0, 256, n).astype(np.uint8)
    _check_rans(api, sy, O.build_histogram(sy))
    sy = np.where(rng.random(n) < 0.97, 0, rng.integers(1, 256, n)).astype(np.uint8)
    _check_rans(api, sy, O.build_histogram(sy))
    sy = np.full(n, 100, np.uint8)
    _check_rans(api, sy, O.build_histogram(sy))
    for m in (0, 1, 2, 15, 16, 17, 511, 512, 513, 1025):
        sy = rng.integers(0, 9, m).astype(np.uint8)
        _check_rans(api, sy, O.build_histogram(rng.integers(0, 9, 64).astype(np.uint8)) if m == 0 else O.build_histogram(sy))


def check_rans_interleaved(api, rng, sizes=(0, 1, 2, 3, 4, 5, 7, 1024, 4099, 70001)):
    """InterleavedRansEncoder / Decoder (rans.rs:393-524): container bytes and decoded symbols equal the oracle's,
    including partial decodes, hand-made containers with unequal counts (round-robin skipping) and malformed tables."""
    # the reference's own test (rans.rs:790-803): uniform(256), 1024 symbols i % 256
    sy = (np.arange(1024) % 256).astype(np.uint8)
    zero_hist = np.zeros(256, np.uint32)                    # all-zero histogram -> FrequencyTable::uniform(256)
    t = O.freq_table_from_histogram(zero_hist)
    blob = api.rans_encode_interleaved(sy, zero_hist)
    assert blob == O.rans_encode_interleaved(sy, t)
    assert np.array_equal(api.rans_decode_interleaved(blob, sy.size, zero_hist), sy)
    for n in sizes:
        for kind in ("skewed", "flat", "malformed"):
            if kind == "skewed":
                sy = np.minimum(rng.geometric(0.35, n) - 1, 255).astype(np.uint8)
            elif kind == "flat":
                sy = rng.integers(0, 256, n, dtype=np.int64).astype(np.uint8)
            else:   # only odd symbols in the upper range: from_histogram pushes used symbols past 4096 (SURVEY 0.7)
                sy = (rng.integers(60, 128, n, dtype=np.int64) * 2 + 1).astype(np.uint8)
            hist = np.bincount(sy, minlength=256).astype(np.uint32)
            t = O.freq_table_from_histogram(hist)
            try:
                want = O.rans_encode_interleaved(sy, t)
            except O.OracleError as e:          # a used symbol whose wrapped frequency is 0: the reference divides by zero
                assert e.code == O.ERR_PANIC
                try:
                    api.rans_encode_interleaved(sy, hist)
                    raise AssertionError("ReferencePanic expected")
                except pkg.CodecError as ce:
                    assert ce.kind == "ReferencePanic", ce.kind
                continue
            got = api.rans_encode_interleaved(sy, hist)
            assert got == want, (n, kind)
            for m in sorted({n, n // 2, max(n - 1, 0), min(n, 5)}):
                assert np.array_equal(api.rans_decode_interleaved(got, m, hist), O.rans_decode_interleaved(want, m, t)), (n, kind, m)
    # hand-made container: unequal counts, so the decoder's skip rule (rans.rs:511-513) shapes the order
    hist = np.bincount(np.minimum(rng.geometric(0.3, 4000) - 1, 255), minlength=256).astype(np.uint32)
    t = O.freq_table_from_histogram(hist)
    parts, counts = [], (700, 3, 0, 1291)
    for c in counts:
        parts.append(O.rans_encode(np.minimum(rng.geometric(0.3, c) - 1, 255).astype(np.uint8), t))
    blob = b"".join(len(p).to_bytes(4, "little") for p in parts) + b"".join(c.to_bytes(4, "little") for c in counts) + b"".join(parts)
    for m in (sum(counts), 1000, 13, 12, 11, 4, 1, 0):
        assert np.array_equal(api.rans_decode_interleaved(blob, m, hist), O.rans_decode_interleaved(blob, m, t)), m
    # error behaviour: short header, lengths past the end, more symbols than the container holds
    for bad, m in ((blob[:31], 1), (blob[:40], 1), (blob, sum(counts) + 1)):
        with np.testing.assert_raises(O.OracleError):
            O.rans_decode_interleaved(bad, m, t)
        try:
            api.rans_decode_interleaved(bad, m, hist)
            raise AssertionError("ReferencePanic expected")
        except pkg.CodecError as e:
            assert e.kind == "ReferencePanic", e.kind


def check_errors(api):
    """Error contract of FrameEncoder::encode / from_bytes / decode (pipeline.rs:384-427, 235-313, 562-579)."""
    enc = pkg.FrameEncoder(90, "cdf53", api=api)
    for (n, w, h, f, kind) in [(10, 4, 4, 2, "InvalidBufferSize"), (3, 0, 4, 2, "InvalidBufferSize"),
                               (0, 4, 4, 2, "InvalidBufferSize"), (12, 0xFFFFFFFF, 0xFFFFFFFF, 0xFFFFFFFF, "DimensionOverflow")]:
        try:
            enc.encode(np.zeros(n, np.uint8), w, h, f)
            raise AssertionError(f"{kind} expected")
        except pkg.CodecError as e:
            assert e.kind == kind, (e.kind, kind)
        try:
            O.encode(np.zeros(n, np.uint8), w, h, f, 90, 0)
            raise AssertionError("oracle accepted it")
        except O.OracleError as e:
            assert O.ERR_NAMES[e.code] == kind
    # empty chunk (pipeline.rs:391-412): 3138-byte .alc, decodes to nothing
    ck = enc.encode(np.zeros(0, np.uint8), 0, 0, 0)
    alc = ck.to_bytes()
    assert alc == O.encode(np.zeros(0, np.uint8), 0, 0, 0, 90, 0) and len(alc) == 3138
    assert pkg.FrameDecoder(api=api).decode(pkg.EncodedChunk.from_bytes(alc, api=api)).size == 0
    good = O.encode(O.generate(O.G0, 4, 4, 2), 4, 4, 2, 90, 0)
    bad_inputs = [good[:100], b"XLCC" + good[4:], good[:4] + b"\x02" + good[5:], good[:5] + b"\x03" + good[6:],
                  good[:-1]]
    for b in bad_inputs:
        try:
            pkg.EncodedChunk.from_bytes(b, api=api)
            raise AssertionError("InvalidBitstream expected")
        except pkg.CodecError as e:
            assert e.kind == "InvalidBitstream"
    assert pkg.EncodedChunk.from_bytes(good + b"junk", api=api).to_bytes() == good     # trailing bytes ignored
    # num_symbols mismatch is caught by decode, not from_bytes (pipeline.rs:566-570)
    tampered = bytearray(good)
    tampered[18 + 12] ^= 1
    ck = pkg.EncodedChunk.from_bytes(bytes(tampered), api=api)
    try:
        pkg.FrameDecoder(api=api).decode(ck)
        raise AssertionError("InvalidBitstream expected")
    except pkg.CodecError as e:
        assert e.kind == "InvalidBitstream"


def check_decode_foreign_headers(api, rng):
    """The decoder takes step/dead-zone/histograms from the header (pipeline.rs:582-595): tamper and compare."""
    w, h, f = 20, 12, 6
    alc = bytearray(O.encode(O.generate(O.G1, w, h, f), w, h, f, 80, 1))
    for c, step in enumerate((3, 1000, -7)):
        off = 18 + c * 1040 + 4
        alc[off:off + 4] = int(step).to_bytes(4, "little", signed=True)
    off = 18 + 1040 + 16                               # Co histogram: shuffle some counts -> other table, garbage symbols
    hist = np.frombuffer(bytes(alc[off:off + 1024]), np.uint32).copy()
    hist[:16] = hist[:16][::-1]
    alc[off:off + 1024] = hist.tobytes()
    out = pkg.FrameDecoder(api=api).decode(pkg.EncodedChunk.from_bytes(bytes(alc), api=api))
    assert np.array_equal(out, O.decode(bytes(alc)))
    # largest coefficients the 32-bit / i16 decode variant accepts (128 * |step| <= 15000) on full-range symbols
    # (noise at step 1 wraps through all 256 symbols), and just beyond it (wide variant), for every wavelet
    # (the 64-frame shape runs the compile-time-depth variants of the temporal kernels)
    for wv in (0, 1, 2):
        for (w, h, f) in ((36, 20, 8), (12, 4, 64)):
            base = O.encode(O.generate(O.G2, w, h, f), w, h, f, 100, wv)
            for steps in ((117, -117, 110), (118, 117, 117), (64, 64, 64)):
                alc = bytearray(base)
                for c, step in enumerate(steps):
                    off = 18 + c * 1040 + 4
                    alc[off:off + 4] = int(step).to_bytes(4, "little", signed=True)
                out = pkg.FrameDecoder(api=api).decode(pkg.EncodedChunk.from_bytes(bytes(alc), api=api))
                assert np.array_equal(out, O.decode(bytes(alc))), (wv, steps, f)


def check_reference_abi(api):
    """The 20 reference symbols used the way a consumer of the reference's cdylib does (ffi.rs tests :325-484)."""
    L = api.lib
    abi = pkg.ReferenceAbi(api)
    assert api.version() == "0.1.2"                                        # ffi.rs:311
    w, h, f = 16, 10, 4
    rgb = O.generate(O.G0, w, h, f)
    alc = abi.encode_to_bytes(rgb, w, h, f, quality=90)
    assert alc == O.encode(rgb, w, h, f, 90, 0)                            # encoder_create is always CDF 5/3 (ffi.rs:92)
    assert np.array_equal(abi.decode_from_bytes(alc), O.decode(alc))
    assert abi.encode_to_bytes(rgb[:-1], w, h, f) is None                  # errors are a null return
    assert abi.decode_from_bytes(alc[:50]) is None
    # null safety (ffi.rs:325-484)
    L.alice_codec_wavelet1d_destroy(None)
    L.alice_codec_encoder_destroy(None)
    L.alice_codec_chunk_destroy(None)
    L.alice_codec_data_free(None, 0)
    L.alice_codec_string_free(None)
    assert L.alice_codec_chunk_width(None) == 0 and L.alice_codec_chunk_height(None) == 0
    assert L.alice_codec_chunk_frames(None) == 0
    assert L.alice_codec_encode(None, None, 0, 1, 1, 1) is None
    import ctypes as C
    n = C.c_uint32()
    assert L.alice_codec_decode(None, C.byref(n)) is None
    assert L.alice_codec_chunk_to_bytes(None, C.byref(n)) is None
    assert L.alice_codec_chunk_from_bytes(None, 0) is None
    assert L.alice_codec_psnr(None, None, 0) == -1.0
    a = np.arange(30, dtype=np.uint8)
    assert api.psnr(a, a) == float("inf")
    b = a.copy(); b[3] += 9
    assert abs(api.psnr(a, b) - O.psnr(a, b)) < 1e-12
    # wavelet1d through the reference handles, incl. len < 2 no-op and odd length (wavelet.rs:133-137, 220-233)
    for wv in (0, 1, 2):
        for n_ in (0, 1, 2, 3, 9, 64):
            x = (np.arange(n_, dtype=np.int32) * 37 - 100) % 251
            assert np.array_equal(api.wavelet1d(wv, x), O.wavelet1d_forward(wv, x))


def check_shared_workspace_batch(api, shapes=((20, 12, 6), (21, 13, 5)), n=3):
    """ALICE_BATCH_SHARED_WORKSPACE: symbol planes live in caller buffers (device API; here the decode outputs and,
    for one chunk, the RGB input itself) or in the staging buffers (host API).  Needs torch for device memory."""
    import torch
    for (w, h, f) in shapes:
        for q, wv in ((80, 1), (90, 0)):
            rgbs = [O.generate(O.G1 if i else O.G2, w, h, f, O.SEED + i) for i in range(n)]
            refs = [O.encode(r, w, h, f, q, wv) for r in rgbs]
            outs_ref = [O.decode(r) for r in refs]
            batch = pkg.ChunkBatch(q, WV[wv], w, h, f, n, stream=0, api=api, shared_workspace=True)
            ws = batch.workspace_bytes()
            pw, ph, pf = O.padded_dims(w, h, f)
            assert ws == 3 * pw * ph * pf
            dev = device_of(api)
            d_in = [torch.zeros(max(ws, r.size), dtype=torch.uint8, device=dev) for r in rgbs]
            for t, r in zip(d_in, rgbs):
                t[:r.size] = torch.from_numpy(r).to(dev)
            d_out = [torch.zeros(max(ws, r.size), dtype=torch.uint8, device=dev) for r in rgbs]
            work = [d_out[0], d_out[1], d_in[2]]                         # chunk 2: in place over its own input
            batch.encode_device([t.data_ptr() for t in d_in], [t.data_ptr() for t in work])
            for i in range(n):
                assert batch.get_chunk(i).to_bytes() == refs[i], (w, h, f, q, wv, i)
            batch.decode_device([t.data_ptr() for t in work])            # decode over the workspaces
            if dev == "cuda":
                torch.cuda.synchronize()
            for i in range(n):
                assert np.array_equal(work[i][:rgbs[i].size].cpu().numpy(), outs_ref[i]), (w, h, f, q, wv, i)
            # host API: staging buffers double as the workspace
            h_in = [torch.from_numpy(r.copy()) for r in rgbs]
            h_out = [torch.zeros(r.size, dtype=torch.uint8) for r in rgbs]
            if dev == "cuda":
                h_in = [t.pin_memory() for t in h_in]
                h_out = [t.pin_memory() for t in h_out]
            chunks = batch.encode_host([t.data_ptr() for t in h_in])
            assert [c.to_bytes() for c in chunks] == refs
            batch.decode_host(chunks, [t.data_ptr() for t in h_out])
            for i in range(n):
                assert np.array_equal(h_out[i].numpy(), outs_ref[i])
            # a plain batch refuses the workspace call; a shared one refuses to run without workspaces
            try:
                batch.encode_device([t.data_ptr() for t in d_in])
                raise AssertionError("workspace pointers required")
            except pkg.CodecError as e:
                assert e.kind == "NullArgument"
            batch.close()


def check_payload_arena(api, w=48, h=20, f=8, n=4):
    """The batch places its rANS streams back to back in one payload arena, each with the upper bound its histogram gives
    (k_estimate_stream_bytes): with a budget just above the real payload everything fits, with a budget far below it the
    streams that find no room go through the worst-case retry -- the output is the oracle's either way."""
    import torch
    dev = device_of(api)
    rgbs = [O.generate(O.G2 if i == 1 else O.G1, w, h, f, O.SEED + i) for i in range(n)]
    for q, wv in ((80, 1), (100, 0)):
        refs = [O.encode(r, w, h, f, q, wv) for r in rgbs]
        outs = [O.decode(r) for r in refs]
        avg = sum(len(r) - 3138 for r in refs) // n
        for budget in (avg + 4096, avg // 2, 64):
            batch = pkg.ChunkBatch(q, WV[wv], w, h, f, n, stream=0, api=api, payload_bytes_per_chunk=budget)
            d_in = [torch.from_numpy(r.copy()).to(dev) for r in rgbs]
            d_out = [torch.zeros_like(t) for t in d_in]
            batch.encode_device([t.data_ptr() for t in d_in])
            for i in range(n):
                assert batch.get_chunk(i).to_bytes() == refs[i], (q, wv, budget, i)
            batch.decode_device([t.data_ptr() for t in d_out])
            if dev == "cuda":
                torch.cuda.synchronize()
            for i in range(n):
                assert np.array_equal(d_out[i].cpu().numpy(), outs[i]), (q, wv, budget, i)
            # foreign payloads through the same arena (decode_host places them back to back as well)
            chunks = [pkg.EncodedChunk.from_bytes(r, api=api) for r in refs]
            h_out = [torch.zeros(r.size, dtype=torch.uint8) for r in rgbs]
            batch.decode_host(chunks, [t.data_ptr() for t in h_out])
            for i in range(n):
                assert np.array_equal(h_out[i].numpy(), outs[i]), (q, wv, budget, i)
            batch.close()


def lossless_oracle(rgb, w, h, f):
    """BASELINE config 4 on the oracle (tests/golden/make_golden.py::lossless_case), every stage returned"""
    planes = O.rgb_bytes_to_ycocg_r(rgb)
    fs = w * h
    out = {"coeffs": [], "symbols": [], "hist": [], "streams": [], "decoded": [], "inverse": []}
    for p in planes:
        co = np.empty(fs * f, dtype=np.int32)
        inv = np.empty(fs * f, dtype=np.int32)
        for t in range(f):
            fw = O.wavelet2d_forward(0, p[t * fs:(t + 1) * fs].astype(np.int32), w, h)
            co[t * fs:(t + 1) * fs] = fw
            inv[t * fs:(t + 1) * fs] = O.wavelet2d_inverse(0, fw, w, h)
        sy = O.to_symbols(co)
        hist = O.build_histogram(sy)
        table = O.freq_table_from_histogram(hist)
        stream = O.rans_encode(sy, table)
        out["coeffs"].append(co); out["symbols"].append(sy); out["hist"].append(np.asarray(hist, dtype=np.uint32))
        out["streams"].append(stream); out["decoded"].append(O.rans_decode(stream, sy.size, table)); out["inverse"].append(inv)
    return out


def check_lossless_set(api, shapes=((16, 6, 4), (21, 9, 3), (128, 8, 6))):
    """alice_codec_lossless_* against the oracle's stages (fast 2-D kernels and the step-by-step path)"""
    import torch
    dev = device_of(api)
    for (w, h, f) in shapes:
        rgb = O.generate(O.G1, w, h, f)
        ref = lossless_oracle(rgb, w, h, f)
        d_rgb = torch.from_numpy(rgb.copy()).to(dev)
        ls = pkg.LosslessSet(w, h, f, api=api)
        ls.encode_device(d_rgb.data_ptr())
        ls.decode_device()
        for what in ("coeffs", "symbols", "hist", "decoded", "inverse"):
            got = ls.fetch(what)
            for c in range(3):
                assert np.array_equal(got[c], ref[what][c]), (w, h, f, what, c)
        for c in range(3):
            assert ls.stream(c) == ref["streams"][c], (w, h, f, c)
        ls.close()


def check_submit_collect(api, shapes=((48, 20, 8), (96, 4, 64)), n=4):
    """alice_codec_batch_submit_host / _collect: chunk-at-a-time encode through ONE reused host buffer equals the oracle
    (plain and shared-workspace batches), and out-of-order submits are refused."""
    for (w, h, f) in shapes:
        rgbs = [O.generate(O.G1, w, h, f, O.SEED + i) for i in range(n)]
        refs = [O.encode(r, w, h, f, 80, 1) for r in rgbs]
        for shared in (False, True):
            batch = pkg.ChunkBatch(80, "cdf97", w, h, f, n, stream=0, api=api, shared_workspace=shared)
            buf = np.empty_like(rgbs[0])
            for i in range(n):
                buf[:] = rgbs[i]
                batch.submit_host(i, buf.ctypes.data)
                batch.sync()                       # the copy has completed: the buffer may be overwritten
            chunks = batch.collect(n)
            assert [c.to_bytes() for c in chunks] == refs, (w, h, f, shared)
            outs = [np.zeros(r.size, dtype=np.uint8) for r in rgbs]
            batch.decode_host(chunks, [o.ctypes.data for o in outs])
            for i in range(n):
                assert np.array_equal(outs[i], O.decode(refs[i])), (w, h, f, shared, i)
            batch.submit_host(0, rgbs[0].ctypes.data)
            try:
                batch.submit_host(2, rgbs[2].ctypes.data)
                raise AssertionError("out-of-order submit accepted")
            except pkg.CodecError as e:
                assert e.kind == "InvalidBufferSize"
            batch.close()


def check_shifted_in_place(api, shapes=((20, 12, 6), (96, 4, 64)), n=3):
    """The memory plan of bench.py: n + 1 RGB-sized buffers; chunk i is read from bufs[i + 1], its symbol planes go to
    bufs[i] (the consumed input of chunk i - 1) and its decode lands back in bufs[i + 1] (the back-end runs the chunks in
    descending order).  Both fused kernels run in this plan (no buffer is read and written by the same launch)."""
    import torch
    dev = device_of(api)
    for (w, h, f) in shapes:
        for q, wv in ((80, 1), (90, 0), (75, 2)):
            rgbs = [O.generate(O.G1, w, h, f, O.SEED + i) for i in range(n)]
            refs = [O.encode(r, w, h, f, q, wv) for r in rgbs]
            # (CDF 5/3 also with ALICE_BATCH_SMALL_SMEM_KERNELS: the same plan on the two-kernel paths)
            batch = pkg.ChunkBatch(q, WV[wv], w, h, f, n, stream=0, api=api, shared_workspace=True, small_smem_kernels=(wv == 0))
            size = max(batch.workspace_bytes(), rgbs[0].size)
            bufs = [torch.zeros(size, dtype=torch.uint8, device=dev) for _ in range(n + 1)]
            for i, r in enumerate(rgbs):
                bufs[i + 1][:r.size] = torch.from_numpy(r).to(dev)
            rgb_ptrs = [t.data_ptr() for t in bufs[1:]]
            batch.encode_device(rgb_ptrs, [t.data_ptr() for t in bufs[:n]])
            for i in range(n):
                assert batch.get_chunk(i).to_bytes() == refs[i], (w, h, f, q, wv, i)
            batch.decode_device(rgb_ptrs)
            if dev == "cuda":
                torch.cuda.synchronize()
            for i in range(n):
                assert np.array_equal(bufs[i + 1][:rgbs[i].size].cpu().numpy(), O.decode(refs[i])), (w, h, f, q, wv, i)
            batch.close()


def check_stream_device(api, shapes=((20, 12, 6), (96, 4, 64)), n=4):
    """Device-pointer streaming (bench.py's memory plan): every chunk's RGB passes through ONE device buffer on the way in
    (submit_device) and ONE on the way out (decode_next_device); what stays per chunk is its symbol planes and payload.
    The decoded chunk is copied out on the same stream before the buffer is handed to the next chunk."""
    import torch
    dev = device_of(api)
    cuda = dev == "cuda"
    for (w, h, f) in shapes:
        for q, wv, small in ((80, 1, False), (90, 0, True), (75, 2, False)):
            rgbs = [O.generate(O.G1, w, h, f, O.SEED + i) for i in range(n)]
            refs = [O.encode(r, w, h, f, q, wv) for r in rgbs]
            st = torch.cuda.current_stream().cuda_stream if cuda else 0
            batch = pkg.ChunkBatch(q, WV[wv], w, h, f, n, stream=st, api=api, small_smem_kernels=small)
            rot_in = torch.zeros(rgbs[0].size, dtype=torch.uint8, device=dev)
            rot_out = torch.zeros(rgbs[0].size, dtype=torch.uint8, device=dev)
            for i, r in enumerate(rgbs):
                rot_in.copy_(torch.from_numpy(r).to(dev))      # stream-ordered: after the front-end of chunk i - 1
                batch.submit_device(i, rot_in.data_ptr())
            try:
                batch.submit_device(n - 2, rot_in.data_ptr())  # out of order
                raise AssertionError("out-of-order submit accepted")
            except pkg.CodecError:
                pass
            batch.encode_finish(n)
            for i in range(n):
                assert batch.get_chunk(i).to_bytes() == refs[i], (w, h, f, q, wv, i)
            try:
                batch.decode_next_device(0, rot_out.data_ptr())     # before decode_begin
                raise AssertionError("decode_next before decode_begin accepted")
            except pkg.CodecError:
                pass
            batch.decode_begin(n)
            outs = []
            for i in (2, 0, 3, 1)[:n]:
                batch.decode_next_device(i, rot_out.data_ptr())
                outs.append((i, rot_out.clone()))              # the consumer, on the same stream
            batch.decode_end()
            for i, t in outs:
                assert np.array_equal(t.cpu().numpy(), O.decode(refs[i])), (w, h, f, q, wv, i)
            batch.close()

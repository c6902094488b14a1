"""PSNR-target encoding: FrameEncoder.psnr_curve / psnr_curve_device / encode_to_psnr, ChunkBatch.encode_host_to_psnr and
`encode --min-psnr`.

A well-formed-tables chunk decodes to exactly the symbols it encodes, so the decode at every step follows from the
front-end's coefficients without rANS work, and the curve is exact.  Checked against the oracle: sse[s-1] equals the sum
of squared differences between the input and the oracle's decode of the well-formed blob at step s (built from the
oracle's stages by test_well_formed_tables.expected_blob), and the PSNR equals the oracle's psnr as a float.
encode_to_psnr must pick the largest step whose PSNR reaches the target and return the oracle's blob at that step.

CPU tier: the SIMT-emulator build (the general back-end path on the small shapes, the fused kernel's SSE mode on
80x2x64 and 112x40x64).  GPU tier (-m gpu): the product library."""
import json
import math
import os
import re
import subprocess
import sys

import numpy as np
import pytest

import oracle as O
import parity
from test_rate_control import SMALL_SHAPES, emul, gpu  # noqa: F401  (fixtures)
from test_well_formed_tables import expected_blob, oracle_coeffs

pkg = parity.pkg
WV = parity.WV
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ROUND_TRIP_STEPS = [1, 2, 8, 14, 27, 39, 64]


def wf(api, wavelet, quality=90):
    return pkg.FrameEncoder(quality, WV[wavelet], api=api, well_formed_tables=True)


def curve_list(curve):
    """{quality: dB} -> [dB] indexed by step - 1"""
    return [curve[pkg.quality_for_step(s)] for s in range(1, 65)]


def oracle_sse(rgb, blob):
    dec = O.decode(blob)
    return int(((dec.astype(np.int64) - rgb.astype(np.int64)) ** 2).sum()), O.psnr(rgb, dec)


def check_curve(api, kind, w, h, f, wavelet, steps=range(1, 65)):
    """sse and PSNR of the library's curve against the oracle's decode of the well-formed blob at each step"""
    rgb = O.generate(kind, w, h, f)
    curve, sse = wf(api, wavelet).psnr_curve(rgb, w, h, f, with_sse=True)
    assert len(curve) == 64 and sse.shape == (64,) and sse.dtype == np.uint64
    coeffs = oracle_coeffs(rgb, w, h, f, wavelet)
    for s in steps:
        blob, _, _ = expected_blob(coeffs, w, h, f, s, wavelet)
        want_sse, want_psnr = oracle_sse(rgb, blob)
        ctx = (w, h, f, wavelet, kind, s)
        assert int(sse[s - 1]) == want_sse, ctx + (int(sse[s - 1]), want_sse)
        assert curve[pkg.quality_for_step(s)] == want_psnr, ctx
    return rgb, curve


def check_round_trip(api, w, h, f, wavelet):
    """the library's own encode + decode at spread steps gives the curve's PSNR exactly"""
    rgb = O.generate(O.G1, w, h, f)
    curve = wf(api, wavelet).psnr_curve(rgb, w, h, f)
    dec = pkg.FrameDecoder(api)
    for s in ROUND_TRIP_STEPS:
        q = pkg.quality_for_step(s)
        out = dec.decode(wf(api, wavelet, q).encode(rgb, w, h, f))
        assert api.psnr(rgb, out) == curve[q] == O.psnr(rgb, out), (w, h, f, wavelet, s)


def check_path_selection(api, w, h, f, wavelet):
    """an input one byte off 4-byte alignment sends a fused shape down the general path: same sums"""
    import torch
    dev = parity.device_of(api)
    rgb = O.generate(O.G2, w, h, f)
    buf = torch.zeros(rgb.size + 16, dtype=torch.uint8, device=dev)
    buf[1:rgb.size + 1] = torch.from_numpy(rgb).to(dev)
    st = torch.cuda.current_stream().cuda_stream if dev == "cuda" else 0
    enc = wf(api, wavelet)
    shifted, sse_shifted = enc.psnr_curve_device(buf.data_ptr() + 1, w, h, f, stream=st, with_sse=True)
    buf[:rgb.size] = torch.from_numpy(rgb).to(dev)
    assert buf.data_ptr() % 16 == 0
    aligned, sse_aligned = enc.psnr_curve_device(buf.data_ptr(), w, h, f, stream=st, with_sse=True)
    assert np.array_equal(sse_shifted, sse_aligned) and shifted == aligned
    assert aligned == enc.psnr_curve(rgb, w, h, f)


def expected_psnr_step(psnr, target):
    ok = [s for s in range(1, 65) if psnr[s - 1] >= target]
    return max(ok) if ok else None


def check_encode_to_psnr(api, kind, w, h, f, wavelet, targets_per_step=True):
    rgb = O.generate(kind, w, h, f)
    enc = wf(api, wavelet, 7)                                         # the encoder's quality is not used
    psnr = curve_list(enc.psnr_curve(rgb, w, h, f))
    coeffs = oracle_coeffs(rgb, w, h, f, wavelet)
    blobs = {}
    steps = range(1, 65) if targets_per_step else (1, 2, 3, 8, 30, 64)
    targets = sorted({t for s in steps for v in [psnr[s - 1]] if math.isfinite(v)
                      for t in (v, math.nextafter(v, math.inf), math.nextafter(v, -math.inf))})
    for t in targets:
        want = expected_psnr_step(psnr, t)
        if want is None:
            continue
        chunk, q = enc.encode_to_psnr(rgb, w, h, f, t)
        assert q == pkg.quality_for_step(want), (w, h, f, wavelet, t, q, want)
        if want not in blobs:
            blobs[want] = expected_blob(coeffs, w, h, f, want, wavelet)[0]
            assert O.psnr(rgb, O.decode(blobs[want])) == psnr[want - 1]
        assert chunk.to_bytes() == blobs[want], (w, h, f, wavelet, t)
        assert psnr[want - 1] >= t
    best = max(psnr)
    for t in (math.nextafter(best, math.inf), best + 10, math.nan):
        with pytest.raises(pkg.CodecError) as ei:
            enc.encode_to_psnr(rgb, w, h, f, t)
        assert ei.value.kind == "InvalidQuantStep", t
        if not math.isnan(t):
            named = [float(x) for x in re.findall(r"best PSNR is (\S+) dB", str(ei.value))]
            assert named == [best], str(ei.value)
    return psnr


def check_not_monotone(psnr):
    """step 1 wraps symbols mod 256: a target that step 2 reaches and step 1 does not, so the steps that reach a
    target are not the top of the curve, and a rule that walks down from quality 100 would stop at the wrong step"""
    assert psnr[0] < psnr[1], psnr[:3]
    t = psnr[1]
    ok = [s for s in range(1, 65) if psnr[s - 1] >= t]
    assert 1 not in ok and 2 in ok and expected_psnr_step(psnr, t) >= 2


def check_empty_and_errors(api):
    enc = wf(api, 1)
    empty = np.zeros(0, np.uint8)
    curve, sse = enc.psnr_curve(empty, 0, 0, 0, with_sse=True)
    assert set(curve.values()) == {math.inf} and not sse.any()
    chunk, q = enc.encode_to_psnr(empty, 0, 0, 0, 60.0)
    assert q == pkg.quality_for_step(64) and chunk.to_bytes() == O.encode(empty, 0, 0, 0, q, 1)
    with pytest.raises(pkg.CodecError) as ei:                         # NaN is refused before any work
        enc.encode_to_psnr(empty, 0, 0, 0, math.nan)
    assert ei.value.kind == "InvalidQuantStep"
    with pytest.raises(pkg.CodecError) as ei:                         # the input is validated as encode does
        enc.psnr_curve(np.zeros(10, np.uint8), 4, 4, 2)
    assert ei.value.kind == "InvalidBufferSize"
    plain = pkg.FrameEncoder(90, "cdf97", api=api)                    # the curve describes the well-formed encode only
    rgb = O.generate(O.G1, 24, 10, 6)
    for call in (lambda: plain.psnr_curve(rgb, 24, 10, 6), lambda: plain.encode_to_psnr(rgb, 24, 10, 6, 20.0),
                 lambda: plain.psnr_curve_device(0, 24, 10, 6)):
        with pytest.raises(ValueError):
            call()


def check_batch(api, w, h, f, wavelet, n=3):
    """encode_host_to_psnr (owned and shared workspace) equals the single-chunk calls; a batch without
    well_formed_tables is refused"""
    rgbs = [O.generate(kind, w, h, f, O.SEED + 17 * i) for i, kind in enumerate((O.G1, O.G2, O.G0)[:n])]
    enc = wf(api, wavelet)
    curves = [curve_list(enc.psnr_curve(r, w, h, f)) for r in rgbs]
    finite = sorted(v for c in curves for v in c if math.isfinite(v))
    target = min(finite[len(finite) // 2], min(max(c) for c in curves))   # every chunk reaches it, at different steps
    singles = [enc.encode_to_psnr(r, w, h, f, target) for r in rgbs]
    for shared in (False, True):
        batch = pkg.ChunkBatch(3, WV[wavelet], w, h, f, n, stream=0, api=api, shared_workspace=shared,
                               well_formed_tables=True)
        chunks, qualities = batch.encode_host_to_psnr([r.ctypes.data for r in rgbs], target)
        assert qualities == [q for _, q in singles], (shared, qualities)
        for c, (sc, _) in zip(chunks, singles):
            assert c.to_bytes() == sc.to_bytes()
        with pytest.raises(pkg.CodecError) as ei:
            batch.encode_host_to_psnr([r.ctypes.data for r in rgbs], max(max(c) for c in curves) + 1)
        assert ei.value.kind == "InvalidQuantStep"
        batch.close()
    plain = pkg.ChunkBatch(3, WV[wavelet], w, h, f, n, stream=0, api=api)
    with pytest.raises(ValueError):
        plain.encode_host_to_psnr([r.ctypes.data for r in rgbs], target)
    import ctypes as C
    arr = plain._ptr_array([r.ctypes.data for r in rgbs])
    out = (C.c_void_p * n)()
    q = np.zeros(n, np.uint8)
    assert api.lib.alice_codec_batch_encode_host_to_psnr(plain._h, arr, n, target, out,
                                                         q.ctypes.data_as(pkg._capi.u8p)) == 2   # ALICE_ERR_DIMENSIONS
    plain.close()


# ------------------------------------------------------------------------------------------------ CPU tier
@pytest.mark.parametrize("shape", SMALL_SHAPES, ids=lambda s: "x".join(map(str, s)))
@pytest.mark.parametrize("wavelet", [0, 1, 2])
def test_curve_emul(emul, shape, wavelet):  # noqa: F811
    big = shape == (112, 40, 64)          # the emulator is slow at 112x40x64: one generator and spread steps there
    for kind in ((O.G1,) if big else (O.G0, O.G1, O.G2)):
        check_curve(emul, kind, *shape, wavelet, steps=ROUND_TRIP_STEPS if big else range(1, 65))


def test_round_trip_emul(emul):  # noqa: F811
    check_round_trip(emul, 24, 10, 6, 0)
    check_round_trip(emul, 80, 2, 64, 1)


def test_path_selection_emul(emul):  # noqa: F811
    check_path_selection(emul, 80, 2, 64, 2)


@pytest.mark.parametrize("wavelet", [0, 1, 2])
def test_encode_to_psnr_emul(emul, wavelet):  # noqa: F811
    # every call runs a whole curve: spread targets here, every step's on the GPU
    psnr = check_encode_to_psnr(emul, O.G1, 24, 10, 6, wavelet, targets_per_step=False)
    check_not_monotone(psnr)
    if wavelet == 2:
        check_encode_to_psnr(emul, O.G2, 80, 2, 64, wavelet, targets_per_step=False)


def test_empty_and_errors_emul(emul):  # noqa: F811
    check_empty_and_errors(emul)


def test_batch_emul(emul):  # noqa: F811
    check_batch(emul, 48, 20, 8, 1)


# ------------------------------------------------------------------------------------------------ GPU tier
@pytest.mark.gpu
@pytest.mark.parametrize("shape", SMALL_SHAPES, ids=lambda s: "x".join(map(str, s)))
@pytest.mark.parametrize("wavelet", [0, 1, 2])
def test_curve_gpu(gpu, shape, wavelet):  # noqa: F811
    for kind in (O.G0, O.G1, O.G2):
        check_curve(gpu, kind, *shape, wavelet)


@pytest.mark.gpu
@pytest.mark.parametrize("wavelet", [0, 1, 2])
def test_round_trip_gpu(gpu, wavelet):  # noqa: F811
    for shape in ((24, 10, 6), (80, 2, 64), (256, 128, 64), (640, 360, 16)):
        check_round_trip(gpu, *shape, wavelet)


@pytest.mark.gpu
def test_path_selection_gpu(gpu):  # noqa: F811
    check_path_selection(gpu, 80, 2, 64, 2)
    check_path_selection(gpu, 256, 128, 64, 1)


@pytest.mark.gpu
@pytest.mark.parametrize("wavelet", [0, 1, 2])
def test_encode_to_psnr_gpu(gpu, wavelet):  # noqa: F811
    psnr = check_encode_to_psnr(gpu, O.G1, 24, 10, 6, wavelet)
    check_not_monotone(psnr)
    check_encode_to_psnr(gpu, O.G2, 80, 2, 64, wavelet)
    check_empty_and_errors(gpu)


@pytest.mark.gpu
def test_batch_gpu(gpu):  # noqa: F811
    check_batch(gpu, 256, 128, 64, 0)
    check_batch(gpu, 48, 20, 8, 1)


@pytest.mark.gpu
@pytest.mark.parametrize("wavelet", [0, 1, 2])
def test_fullsize_gpu(gpu, wavelet):  # noqa: F811
    """one 1920x1080x64 G1 chunk: the curve at qualities 90/80/60/40 equals the PSNR of the library's own well-formed
    encode and decode, and the figures profiles/r04_well_formed.json recorded for the same chunks"""
    w, h, f = 1920, 1080, 64
    rgb = O.generate(O.G1, w, h, f)
    curve = wf(gpu, wavelet).psnr_curve(rgb, w, h, f)
    with open(os.path.join(ROOT, "profiles", "r04_well_formed.json")) as fh:
        r04 = {(r["wavelet"], r["quality"]): r["well_formed"]["psnr_db"] for r in json.load(fh)}
    for q in (90, 80, 60, 40):
        out = pkg.FrameDecoder(gpu).decode(wf(gpu, wavelet, q).encode(rgb, w, h, f))
        got = curve[pkg.quality_for_step(pkg.quality_to_step(q))]
        assert got == gpu.psnr(rgb, out), (wavelet, q)
        assert round(got, 3) == r04[(WV[wavelet], q)], (wavelet, q, got)


@pytest.mark.gpu
def test_cli_min_psnr(tmp_path):
    """encode --min-psnr with --chunk-frames: every chunk decodes to at least the target; the misuses exit 1"""
    w, h, f, cf = 64, 32, 20, 6                                        # three full chunks (one batch) + a 2-frame chunk
    rgb = O.generate(O.G1, w, h, f)
    src = tmp_path / "in.rgb"
    rgb.tofile(src)
    target = 25.0
    out = tmp_path / "out.alc"
    cli = [sys.executable, os.path.join(ROOT, "alice-codec_b200", "cli.py")]
    base = cli + ["encode", str(src), "-W", str(w), "-H", str(h), "-f", str(f), "-w", "cdf97", "-o", str(out)]
    r = subprocess.run(base + ["--chunk-frames", str(cf), "--min-psnr", str(target), "--well-formed-tables"],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    assert "min-psnr=25.0 dB" in r.stderr and "tables=well-formed" in r.stderr
    qualities = [int(x) for x in r.stderr.split("quality=")[1].split(",")[:4]]
    data, blobs = out.read_bytes(), []
    while data:
        n = 3138 + sum(int.from_bytes(data[18 + 1040 * c:22 + 1040 * c], "little") for c in range(3))
        blobs.append(data[:n])
        data = data[n:]
    assert len(blobs) == 4
    per = w * h * 3
    for i, (blob, q) in enumerate(zip(blobs, qualities)):
        nf = min(cf, f - i * cf)
        part = rgb[i * cf * per:(i * cf + nf) * per]
        assert O.psnr(part, O.decode(blob)) >= target, (i, q)
        assert blob == wf(pkg.default_api(), 1, q).encode(part, w, h, nf).to_bytes(), (i, q)
    for extra in (["--min-psnr", "25"], ["--min-psnr", "25", "--well-formed-tables", "--max-bytes", "9000"]):
        r = subprocess.run(base + extra, capture_output=True, text=True)
        assert r.returncode == 1 and r.stderr.startswith("error:"), r.stderr

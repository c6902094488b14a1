"""Byte-budget encoding: FrameEncoder.rate_curve / encode_to_size and ChunkBatch.encode_host_to_size.

The rate curve predicts the .alc size of every quantiser step from one transform pass and one histogram of the
coefficient values.  Checked against the oracle: the curve's symbol histograms equal the header histograms of the
oracle's encode at that step bit for bit, every prediction is >= the oracle's .alc length, and UINT64_MAX (None in
Python) marks exactly the steps where the oracle aborts.  encode_to_size must return the oracle's bytes at the quality
it reports, chosen by the rule "smallest step whose prediction fits".

CPU tier: the SIMT-emulator build (as in test_emul_parity.py).  GPU tier (-m gpu): the product library."""
import importlib.util
import os
import subprocess
import sys

import numpy as np
import pytest

import oracle as O
import parity

pkg = parity.pkg
WV = parity.WV
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HDR = 3138
SMALL_SHAPES = [(24, 10, 6), (3, 5, 1), (7, 2, 4), (80, 2, 64), (112, 40, 64)]   # the last two: fused front-end


@pytest.fixture(scope="module")
def emul():
    spec = importlib.util.spec_from_file_location("b", os.path.join(os.path.dirname(pkg.__file__), "build.py"))
    b = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(b)
    return pkg.Api(b.build_emul())


@pytest.fixture(scope="module")
def gpu():
    a = pkg.Api()
    assert a.device_count() >= 1, "no CUDA device visible to libalice_codec"
    a.set_device(0)
    return a


def steps_of(curve):
    """{quality: bytes} -> list of (step, quality, bytes) in step order"""
    return [(pkg.quality_to_step(q), q, b) for q, b in sorted(curve.items(), key=lambda kv: -kv[0])]


def header_hists(alc):
    return [np.frombuffer(alc[18 + c * 1040 + 16:18 + c * 1040 + 1040], np.uint32) for c in range(3)]


def oracle_step_hists(rgb, w, h, f, wavelet, steps):
    """the symbol histograms of the oracle's front-end at the given steps, from its coefficients (one transform)"""
    _, coeffs, _ = O.encode(rgb, w, h, f, 100, wavelet, stages=True)
    return {s: [O.build_histogram(O.to_symbols(O.quantize_buffer(s, s, coeffs[c]))) for c in range(3)] for s in steps}


def check_curve(api, kind, w, h, f, wavelet, seed=O.SEED):
    """all 64 steps against full oracle encodes"""
    rgb = O.generate(kind, w, h, f, seed)
    curve, hist = pkg.FrameEncoder(90, WV[wavelet], api=api).rate_curve(rgb, w, h, f, with_hist=True)
    assert len(curve) == 64 and hist.shape == (64, 3, 256)
    for s, q, pred in steps_of(curve):
        assert O.quality_to_step(q) == s
        assert q == 100 or O.quality_to_step(q + 1) != s            # the largest quality with this step
        try:
            ref = O.encode(rgb, w, h, f, q, wavelet)
        except O.OracleError as e:
            assert e.code == O.ERR_PANIC
            assert pred is None, (w, h, f, wavelet, kind, s)
            continue
        assert pred is not None, (w, h, f, wavelet, kind, s)
        for c, rh in enumerate(header_hists(ref)):
            assert np.array_equal(hist[s - 1, c], rh), (w, h, f, wavelet, kind, s, c)
        assert pred >= len(ref), (w, h, f, wavelet, kind, s, pred, len(ref))
    return rgb, curve


def expected_step(curve, budget):
    fits = [s for s, _, b in steps_of(curve) if b is not None and b <= budget]
    return min(fits) if fits else None


def check_encode_to_size(api, kind, w, h, f, wavelet, seed=O.SEED):
    rgb = O.generate(kind, w, h, f, seed)
    enc = pkg.FrameEncoder(7, WV[wavelet], api=api)                # the encoder's quality is not used
    curve = enc.rate_curve(rgb, w, h, f)
    preds = [b for _, _, b in steps_of(curve)]
    budgets = {10 ** 15}
    for s in (1, 2, 8, 30, 63, 64):
        if preds[s - 1] is not None:
            budgets |= {preds[s - 1], preds[s - 1] - 1}
    for budget in sorted(budgets):
        want = expected_step(curve, budget)
        if want is None:
            with pytest.raises(pkg.CodecError) as ei:
                enc.encode_to_size(rgb, w, h, f, budget)
            assert ei.value.kind == "InvalidBufferSize"
            continue
        chunk, q = enc.encode_to_size(rgb, w, h, f, budget)
        assert pkg.quality_to_step(q) == want and q == pkg.quality_for_step(want), (budget, q, want)
        alc = chunk.to_bytes()
        assert len(alc) <= budget
        assert alc == O.encode(rgb, w, h, f, q, wavelet), (w, h, f, wavelet, kind, budget, q)
    # a budget below every prediction
    smallest = min(b for b in preds if b is not None)
    with pytest.raises(pkg.CodecError) as ei:
        enc.encode_to_size(rgb, w, h, f, smallest - 1)
    assert ei.value.kind == "InvalidBufferSize" and str(smallest) in str(ei.value)


def check_empty(api):
    enc = pkg.FrameEncoder(50, "cdf97", api=api)
    empty = np.zeros(0, np.uint8)
    curve, hist = enc.rate_curve(empty, 0, 0, 0, with_hist=True)
    assert set(curve.values()) == {HDR} and not hist.any()
    chunk, q = enc.encode_to_size(empty, 0, 0, 0, HDR)
    assert q == 100 and chunk.to_bytes() == O.encode(empty, 0, 0, 0, 100, 1)
    with pytest.raises(pkg.CodecError) as ei:
        enc.encode_to_size(empty, 0, 0, 0, HDR - 1)
    assert ei.value.kind == "InvalidBufferSize"
    with pytest.raises(pkg.CodecError) as ei:                       # the input is validated as encode does
        enc.rate_curve(np.zeros(10, np.uint8), 4, 4, 2)
    assert ei.value.kind == "InvalidBufferSize"


def check_device_curve(api, dev, w, h, f, wavelet):
    import torch
    rgb = O.generate(O.G1, w, h, f)
    enc = pkg.FrameEncoder(90, WV[wavelet], api=api)
    curve, hist = enc.rate_curve(rgb, w, h, f, with_hist=True)
    d = torch.from_numpy(rgb.copy()).to(dev)
    st = torch.cuda.current_stream().cuda_stream if dev == "cuda" else 0
    dcurve, dhist = enc.rate_curve_device(d.data_ptr(), w, h, f, stream=st, with_hist=True)
    assert dcurve == curve and np.array_equal(dhist, hist)


def check_batch_to_size(api, w, h, f, wavelet, shared=False):
    """4 chunks of different content: the batch's qualities and bytes equal 4 single encode_to_size calls"""
    rgbs = [O.generate(kind, w, h, f, O.SEED + 17 * i) for i, kind in enumerate((O.G1, O.G2, O.G0, O.G1))]
    enc = pkg.FrameEncoder(90, WV[wavelet], api=api)
    curves = [enc.rate_curve(r, w, h, f) for r in rgbs]
    finite = sorted(b for c in curves for b in c.values() if b is not None)
    budget = finite[len(finite) // 2]                                # some chunks fit high qualities, others low
    budget = max(budget, max(min(b for b in c.values() if b is not None) for c in curves))
    singles = [enc.encode_to_size(r, w, h, f, budget) for r in rgbs]
    batch = pkg.ChunkBatch(3, WV[wavelet], w, h, f, 4, stream=0, api=api, shared_workspace=shared)
    bytes_plain = batch.device_bytes()
    chunks, qualities = batch.encode_host_to_size([r.ctypes.data for r in rgbs], budget)
    assert qualities == [q for _, q in singles]
    assert len(set(qualities)) > 1, qualities
    for c, (sc, q), r in zip(chunks, singles, rgbs):
        alc = c.to_bytes()
        assert alc == sc.to_bytes() == O.encode(r, w, h, f, q, wavelet) and len(alc) <= budget
    # the rate buffers are allocated by the first rate call, not before
    pw, ph, pf = O.padded_dims(w, h, f)
    assert batch.device_bytes() >= bytes_plain + 12 * pw * ph * pf
    # the batch still encodes at its own quality afterwards
    assert [c.to_bytes() for c in batch.encode_host([r.ctypes.data for r in rgbs])] == \
        [O.encode(r, w, h, f, 3, wavelet) for r in rgbs]
    with pytest.raises(pkg.CodecError) as ei:
        batch.encode_host_to_size([r.ctypes.data for r in rgbs], HDR)
    assert ei.value.kind == "InvalidBufferSize"
    batch.close()


def check_device_bytes_untouched(api, w, h, f):
    """a batch that never calls a rate function holds what it held before the feature existed"""
    rgbs = [O.generate(O.G1, w, h, f, O.SEED + i) for i in range(2)]
    a = pkg.ChunkBatch(80, "cdf53", w, h, f, 2, stream=0, api=api)
    b = pkg.ChunkBatch(80, "cdf53", w, h, f, 2, stream=0, api=api)
    before = a.device_bytes()
    a.encode_host([r.ctypes.data for r in rgbs])
    b.encode_host([r.ctypes.data for r in rgbs])
    assert a.device_bytes() == b.device_bytes()
    b.encode_host_to_size([r.ctypes.data for r in rgbs], 10 ** 12)
    pw, ph, pf = O.padded_dims(w, h, f)
    assert b.device_bytes() - a.device_bytes() >= 12 * pw * ph * pf
    assert a.device_bytes() - before < 12 * pw * ph * pf             # encode_host allocates only its staging buffer
    a.close()
    b.close()


def test_quality_for_step():
    for s in range(1, 65):
        q = pkg.quality_for_step(s)
        assert O.quality_to_step(q) == s and all(O.quality_to_step(x) != s for x in range(q + 1, 101))
    assert [pkg.quality_to_step(q) for q in range(256)] == [O.quality_to_step(q) for q in range(256)]


# ------------------------------------------------------------------------------------------------ CPU tier
@pytest.mark.parametrize("shape", SMALL_SHAPES, ids=lambda s: "x".join(map(str, s)))
@pytest.mark.parametrize("wavelet", [0, 1, 2])
@pytest.mark.parametrize("kind", [O.G0, O.G1, O.G2])
def test_curve_emul(emul, shape, wavelet, kind):
    check_curve(emul, kind, *shape, wavelet)


@pytest.mark.parametrize("shape", [(24, 10, 6), (3, 5, 1), (7, 3, 1), (80, 2, 64)], ids=lambda s: "x".join(map(str, s)))
@pytest.mark.parametrize("wavelet", [0, 1, 2])
def test_encode_to_size_emul(emul, shape, wavelet):
    for kind in (O.G1, O.G2):
        check_encode_to_size(emul, kind, *shape, wavelet)


def test_empty_and_errors_emul(emul):
    check_empty(emul)


def test_device_curve_emul(emul):
    for shape in ((24, 10, 6), (80, 2, 64)):
        check_device_curve(emul, "cpu", *shape, 1)


@pytest.mark.parametrize("shared", [False, True])
def test_batch_to_size_emul(emul, shared):
    check_batch_to_size(emul, 48, 20, 8, 1, shared)
    check_batch_to_size(emul, 96, 4, 64, 2, shared)


def test_device_bytes_emul(emul):
    check_device_bytes_untouched(emul, 48, 20, 8)


# ------------------------------------------------------------------------------------------------ GPU tier
@pytest.mark.gpu
@pytest.mark.parametrize("shape", SMALL_SHAPES, ids=lambda s: "x".join(map(str, s)))
@pytest.mark.parametrize("wavelet", [0, 1, 2])
def test_curve_gpu(gpu, shape, wavelet):
    for kind in (O.G0, O.G1, O.G2):
        check_curve(gpu, kind, *shape, wavelet)


@pytest.mark.gpu
@pytest.mark.parametrize("wavelet", [0, 1, 2])
def test_encode_to_size_and_empty_gpu(gpu, wavelet):
    for shape in ((24, 10, 6), (3, 5, 1), (7, 3, 1), (80, 2, 64)):
        check_encode_to_size(gpu, O.G1, *shape, wavelet)
    check_empty(gpu)


@pytest.mark.gpu
@pytest.mark.parametrize("shape", [(256, 128, 64), (640, 360, 16)], ids=lambda s: "x".join(map(str, s)))
@pytest.mark.parametrize("wavelet", [0, 1, 2])
def test_curve_medium_gpu(gpu, shape, wavelet):
    """every step's histograms against the oracle's coefficients, the bound against oracle encodes at spread steps"""
    w, h, f = shape
    rgb = O.generate(O.G1, w, h, f)
    curve, hist = pkg.FrameEncoder(90, WV[wavelet], api=gpu).rate_curve(rgb, w, h, f, with_hist=True)
    ref = oracle_step_hists(rgb, w, h, f, wavelet, range(1, 65))
    for s, q, pred in steps_of(curve):
        for c in range(3):
            assert np.array_equal(hist[s - 1, c], ref[s][c]), (shape, wavelet, s, c)
        if s in (1, 4, 16, 40, 64):
            assert pred >= len(O.encode(rgb, w, h, f, q, wavelet)), (shape, wavelet, s)
    if shape == (640, 360, 16) and wavelet == 0:
        check_encode_to_size(gpu, O.G1, w, h, f, wavelet)


@pytest.mark.gpu
@pytest.mark.parametrize("wavelet", [0, 1, 2])
def test_curve_fullsize_gpu(gpu, wavelet):
    """one 1920x1080x64 G1 chunk: histograms and bound against real encodes at steps 1, 8, 30, 64"""
    w, h, f = 1920, 1080, 64
    rgb = O.generate(O.G1, w, h, f)
    enc = pkg.FrameEncoder(90, WV[wavelet], api=gpu)
    curve, hist = enc.rate_curve(rgb, w, h, f, with_hist=True)
    for s in (1, 8, 30, 64):
        q = pkg.quality_for_step(s)
        chunk = pkg.FrameEncoder(q, WV[wavelet], api=gpu).encode(rgb, w, h, f)
        for c in range(3):
            assert np.array_equal(hist[s - 1, c], chunk.channel_header(c)["histogram"]), (wavelet, s, c)
        assert curve[q] >= len(chunk.to_bytes()), (wavelet, s)


@pytest.mark.gpu
def test_device_curve_gpu(gpu):
    for shape, wv in (((24, 10, 6), 1), ((256, 128, 64), 0), ((640, 360, 16), 2)):
        check_device_curve(gpu, "cuda", *shape, wv)


@pytest.mark.gpu
@pytest.mark.parametrize("shared", [False, True])
def test_batch_to_size_gpu(gpu, shared):
    check_batch_to_size(gpu, 256, 128, 64, 1, shared)
    check_batch_to_size(gpu, 48, 20, 8, 0, shared)


@pytest.mark.gpu
def test_device_bytes_gpu(gpu):
    check_device_bytes_untouched(gpu, 256, 128, 64)


@pytest.mark.gpu
def test_cli_max_bytes(tmp_path):
    """encode --max-bytes with --chunk-frames: every blob fits, each is the oracle's encode at the reported quality,
    and decode of the file equals the oracle's decode of those blobs"""
    w, h, f, cf = 64, 32, 20, 6                                        # three full chunks (one batch) + a 2-frame chunk
    rgb = O.generate(O.G1, w, h, f)
    src = tmp_path / "in.rgb"
    rgb.tofile(src)
    budget = 9000
    out = tmp_path / "out.alc"
    cli = [sys.executable, os.path.join(ROOT, "alice-codec_b200", "cli.py")]
    r = subprocess.run(cli + ["encode", str(src), "-W", str(w), "-H", str(h), "-f", str(f), "-w", "cdf97",
                              "--chunk-frames", str(cf), "--max-bytes", str(budget), "-o", str(out)],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    qualities = [int(x) for x in r.stderr.split("quality=")[1].split(",")[:4]]
    data, blobs = out.read_bytes(), []
    while data:
        n = HDR + sum(int.from_bytes(data[18 + 1040 * c:22 + 1040 * c], "little") for c in range(3))
        blobs.append(data[:n])
        data = data[n:]
    assert len(blobs) == 4
    per = w * h * 3
    for i, (blob, q) in enumerate(zip(blobs, qualities)):
        nf = min(cf, f - i * cf)
        assert len(blob) <= budget
        assert blob == O.encode(rgb[i * cf * per:(i * cf + nf) * per], w, h, nf, q, 1), (i, q)
    dec = tmp_path / "out.rgb"
    r = subprocess.run(cli + ["decode", str(out), "-o", str(dec)], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    assert np.array_equal(np.fromfile(dec, np.uint8), np.concatenate([O.decode(b) for b in blobs]))

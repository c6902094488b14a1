"""Well-formed-tables encoding: FrameEncoder(..., well_formed_tables=True), ChunkBatch(..., well_formed_tables=True) and
`encode --well-formed-tables`.

The default encode stores each channel's symbol counts, and FrequencyTable::from_histogram gives every empty bin a
frequency of 1: where empty bins lie below used symbols the high symbols' ranges run past 4096 and the chunk does not
decode to what was encoded.  In this mode a header stores a table specification H' derived from the counts by the rule
restated below (numpy, independent of the kernel), and the streams are rANS-coded with from_histogram(H').  Checked
against the oracle: the headers hold exactly H', the whole blob equals the oracle's rANS encode of the oracle's
symbols with that table, the oracle's decoder returns exactly the encoded symbols, and the library's decode equals the
oracle's.

CPU tier: the SIMT-emulator build (as in test_rate_control.py).  GPU tier (-m gpu): the product library."""
import importlib.util
import os
import struct
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
SHAPES = [(24, 10, 6), (3, 5, 1), (80, 2, 64), (112, 40, 64)]      # the last two take the fused paths
ALL_STEPS = list(range(1, 65))
SPREAD_STEPS = [1, 4, 13, 30, 45, 64]


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


# ------------------------------------------------------------------------------------------------ the rule
def table_is_clean(counts):
    """from_histogram(counts) gives every used symbol 1 <= f <= 4096 and cum + f <= 4096"""
    t = O.freq_table_from_histogram(counts)
    f, cum = t.freq_np().astype(np.int64), t.cum_np().astype(np.int64)
    used = np.asarray(counts) > 0
    return bool(np.all((f[used] >= 1) & (f[used] <= 4096) & (cum[used] + f[used] <= 4096)))


def well_formed_hist(counts):
    """(H', rule 1 applied) for one stream's symbol counts"""
    c = np.asarray(counts, np.uint64)
    if table_is_clean(c):
        return c.astype(np.uint32), True
    used = c > 0
    n = int(c.sum())
    scale = 4096 - int(np.count_nonzero(~used[:255]))
    prod = [int(x) * scale for x in c]
    f = [max(1, p // n) if u else 0 for p, u in zip(prod, used)]
    d = scale - sum(f)
    if d > 0:
        order = sorted(np.flatnonzero(used), key=lambda j: (-(prod[j] % n), j))
        for j in order[:d]:
            f[j] += 1
    while d < 0:
        j = max((j for j in range(256) if f[j] > 1), key=lambda j: (f[j], -j))
        f[j] -= 1
        d += 1
    h = np.array(f, np.uint32)
    h[255] = 4096 - sum(f[:255])
    return h, False


def test_rule_examples():
    """hand-checked cases of the restatement itself"""
    c = np.zeros(256, np.uint32)
    c[0], c[200] = 1000, 1
    h, clean = well_formed_hist(c)          # 199 empty bins below 200 push its range past 4096
    # S = 4096 - 253 empty bins: 3839 + 3 with remainders 161 and 840, so symbol 200 takes the spare slot
    assert not clean and h.sum() == 4096 and (h[0], h[200], h[255]) == (3839, 4, 253)
    t = O.freq_table_from_histogram(h)
    assert (t.freq_np()[0], t.freq_np()[200], t.cum_np()[200], t.freq_np()[255]) == (3839, 4, 4038, 0)
    c = np.zeros(256, np.uint32)
    c[:4] = [10, 20, 30, 40]
    h, clean = well_formed_hist(c)          # no empty bin below a used one
    assert clean and np.array_equal(h, c)
    c = np.full(256, 1, np.uint32)
    c[7] = 10 ** 6                          # every symbol used, D = -253 from max(1, .)
    h, clean = well_formed_hist(c)
    assert not clean and h.sum() == 4096 and h[7] == 4094 - 253 and np.all(np.delete(h, 7) == 1)


# ------------------------------------------------------------------------------------------------ oracle side
def oracle_coeffs(rgb, w, h, f, wavelet):
    """the oracle's wavelet coefficients (independent of the quality; an encode that aborts returns none)"""
    for q in (100, 0, 50, 90):
        try:
            return O.encode(rgb, w, h, f, q, wavelet, stages=True)[1]
        except O.OracleError as e:
            assert e.code == O.ERR_PANIC
    raise AssertionError("the oracle aborts at every tried quality")


def expected_blob(coeffs, w, h, f, step, wavelet):
    """(the well-formed .alc, per-channel symbols, per-channel rule-1 flags) from the oracle's stages"""
    pw, ph, pf = O.padded_dims(w, h, f)
    head = b"ALCC" + bytes([1, wavelet]) + struct.pack("<III", w, h, f)
    payload, syms, clean = b"", [], []
    for c in range(3):
        s = O.to_symbols(O.quantize_buffer(step, step, coeffs[c]))
        hw, cl = well_formed_hist(O.build_histogram(s))
        stream = O.rans_encode(s, O.freq_table_from_histogram(hw))
        head += struct.pack("<IiiI", len(stream), step, step, pw * ph * pf) + hw.astype("<u4").tobytes()
        payload += stream
        syms.append(s)
        clean.append(cl)
    return head + payload, syms, clean


def header_hists(alc):
    return [np.frombuffer(alc[18 + c * 1040 + 16:18 + c * 1040 + 1040], np.uint32) for c in range(3)]


def default_round_trips(rgb, w, h, f, q, wavelet, syms):
    try:
        _, dec = O.decode(O.encode(rgb, w, h, f, q, wavelet), stages=True)
    except O.OracleError:
        return False
    return all(np.array_equal(dec[c], syms[c]) for c in range(3))


def check_chunk(api, kind, w, h, f, wavelet, steps, lib_decode_steps, stats):
    """headers, whole blob, oracle round trip, library decode and the rate bound at the given steps"""
    rgb = O.generate(kind, w, h, f)
    coeffs = oracle_coeffs(rgb, w, h, f, wavelet)
    curve = pkg.FrameEncoder(90, WV[wavelet], api=api, well_formed_tables=True).rate_curve(rgb, w, h, f)
    assert None not in curve.values(), (w, h, f, wavelet, kind)
    for s in steps:
        q = pkg.quality_for_step(s)
        want, syms, clean = expected_blob(coeffs, w, h, f, s, wavelet)
        chunk = pkg.FrameEncoder(q, WV[wavelet], api=api, well_formed_tables=True).encode(rgb, w, h, f)
        alc = chunk.to_bytes()
        ctx = (w, h, f, wavelet, kind, s)
        for c, (got, hw) in enumerate(zip(header_hists(alc), header_hists(want))):
            assert np.array_equal(got, hw), ctx + (c,)
        assert alc == want, ctx
        rgb_dec, dec = O.decode(alc, stages=True)
        for c in range(3):
            assert np.array_equal(dec[c], syms[c]), ctx + (c,)
        if all(clean):
            assert alc == O.encode(rgb, w, h, f, q, wavelet), ctx
        if s in lib_decode_steps:
            assert np.array_equal(pkg.FrameDecoder(api).decode(pkg.EncodedChunk.from_bytes(alc, api=api)), rgb_dec), ctx
        assert curve[q] >= len(alc), ctx + (curve[q], len(alc))
        stats["clean"] += sum(clean)
        stats["rescaled"] += 3 - sum(clean)
        if not all(clean) and not default_round_trips(rgb, w, h, f, q, wavelet, syms):
            stats["default_fails"] += 1


def new_stats():
    return {"clean": 0, "rescaled": 0, "default_fails": 0}


def check_to_size(api, kind, w, h, f, wavelet):
    rgb = O.generate(kind, w, h, f)
    enc = pkg.FrameEncoder(7, WV[wavelet], api=api, well_formed_tables=True)
    curve = enc.rate_curve(rgb, w, h, f)
    preds = sorted(set(curve.values()))
    for budget in (preds[len(preds) // 2], preds[0], 10 ** 12):
        chunk, q = enc.encode_to_size(rgb, w, h, f, budget)
        fits = [pkg.quality_to_step(qq) for qq, b in curve.items() if b <= budget]
        assert pkg.quality_to_step(q) == min(fits), (budget, q)
        alc = chunk.to_bytes()
        assert len(alc) <= budget
        assert alc == pkg.FrameEncoder(q, WV[wavelet], api=api, well_formed_tables=True).encode(rgb, w, h, f).to_bytes()
    with pytest.raises(pkg.CodecError) as ei:
        enc.encode_to_size(rgb, w, h, f, preds[0] - 1)
    assert ei.value.kind == "InvalidBufferSize"


def check_batch(api, w, h, f, wavelet, n=3):
    """encode_host_to_size (owned and shared workspace), resident encode_device -> decode_device, and a default batch
    next to a well-formed one"""
    import torch
    dev = parity.device_of(api)
    rgbs = [O.generate(kind, w, h, f, O.SEED + 17 * i) for i, kind in enumerate((O.G1, O.G2, O.G0, O.G1)[:n])]
    wf = pkg.FrameEncoder(90, WV[wavelet], api=api, well_formed_tables=True)
    curves = [wf.rate_curve(r, w, h, f) for r in rgbs]
    budget = max(sorted(b for c in curves for b in c.values())[len(curves) * 32], max(min(c.values()) for c in curves))
    for shared in (False, True):
        batch = pkg.ChunkBatch(3, WV[wavelet], w, h, f, n, stream=0, api=api, shared_workspace=shared,
                               well_formed_tables=True)
        chunks, qualities = batch.encode_host_to_size([r.ctypes.data for r in rgbs], budget)
        for c, q, r in zip(chunks, qualities, rgbs):
            alc = c.to_bytes()
            assert len(alc) <= budget
            assert alc == pkg.FrameEncoder(q, WV[wavelet], api=api, well_formed_tables=True).encode(r, w, h, f).to_bytes()
        batch.close()
    q = 80
    refs = [pkg.FrameEncoder(q, WV[wavelet], api=api, well_formed_tables=True).encode(r, w, h, f).to_bytes() for r in rgbs]
    plain = pkg.ChunkBatch(q, WV[wavelet], w, h, f, n, stream=0, api=api)
    batch = pkg.ChunkBatch(q, WV[wavelet], w, h, f, n, stream=0, api=api, well_formed_tables=True)
    assert batch.device_bytes() == plain.device_bytes() + n * 3 * 256 * 4
    d_in = [torch.from_numpy(r.copy()).to(dev) for r in rgbs]
    d_out = [torch.zeros_like(t) for t in d_in]
    batch.encode_device([t.data_ptr() for t in d_in])
    for i in range(n):
        assert batch.get_chunk(i).to_bytes() == refs[i], (wavelet, i)
    batch.decode_device([t.data_ptr() for t in d_out])
    if dev == "cuda":
        torch.cuda.synchronize()
    for i in range(n):
        assert np.array_equal(d_out[i].cpu().numpy(), O.decode(refs[i])), (wavelet, i)
    # the default batch beside it: the oracle's encode, byte for byte
    assert [c.to_bytes() for c in plain.encode_host([r.ctypes.data for r in rgbs])] == \
        [O.encode(r, w, h, f, q, wavelet) for r in rgbs]
    batch.close()
    plain.close()


def check_flags(api):
    """unknown flag bits are refused; the default FrameEncoder still encodes what the oracle encodes"""
    assert not api.lib.alice_codec_encoder_create_ex(80, 0, 2)
    assert api.lib.alice_codec_last_error() == 2
    sizes = np.zeros(64, np.uint64)
    rgb = O.generate(O.G1, 24, 10, 6)
    assert api.lib.alice_codec_rate_curve_ex(0, rgb.ctypes.data_as(pkg._capi.u8p), rgb.size, 24, 10, 6,
                                             sizes.ctypes.data_as(pkg._capi.u64p), None, 8) == 2
    enc = pkg.FrameEncoder(80, "cdf97", api=api)
    assert not enc.well_formed_tables
    assert enc.encode(rgb, 24, 10, 6).to_bytes() == O.encode(rgb, 24, 10, 6, 80, 1)
    empty = np.zeros(0, np.uint8)
    wf = pkg.FrameEncoder(80, "cdf97", api=api, well_formed_tables=True)
    assert wf.encode(empty, 0, 0, 0).to_bytes() == O.encode(empty, 0, 0, 0, 80, 1)


# ------------------------------------------------------------------------------------------------ CPU tier
@pytest.mark.parametrize("shape", SHAPES, ids=lambda s: "x".join(map(str, s)))
@pytest.mark.parametrize("wavelet", [0, 1, 2])
def test_chunks_emul(emul, shape, wavelet):
    stats = new_stats()
    big = shape == (112, 40, 64)
    for kind in (O.G0, O.G1, O.G2):      # the emulator is slow at 112x40x64: spread steps there
        steps = SPREAD_STEPS if big else ALL_STEPS
        check_chunk(emul, kind, *shape, wavelet, steps, SPREAD_STEPS[:2] if big else SPREAD_STEPS, stats)
    assert stats["clean"] and stats["rescaled"], stats       # both branches of the rule met
    if shape in ((24, 10, 6), (112, 40, 64)):
        assert stats["default_fails"], stats                  # the default encode fails where this one decodes


@pytest.mark.parametrize("wavelet", [0, 1, 2])
def test_to_size_emul(emul, wavelet):
    for shape in ((24, 10, 6), (80, 2, 64)):
        check_to_size(emul, O.G1, *shape, wavelet)


def test_batch_emul(emul):
    check_batch(emul, 48, 20, 8, 1)
    check_batch(emul, 96, 4, 64, 2)


def test_flags_emul(emul):
    check_flags(emul)


# ------------------------------------------------------------------------------------------------ GPU tier
@pytest.mark.gpu
@pytest.mark.parametrize("shape", SHAPES, ids=lambda s: "x".join(map(str, s)))
@pytest.mark.parametrize("wavelet", [0, 1, 2])
def test_chunks_gpu(gpu, shape, wavelet):
    stats = new_stats()
    for kind in (O.G0, O.G1, O.G2):
        check_chunk(gpu, kind, *shape, wavelet, ALL_STEPS, ALL_STEPS, stats)
    assert stats["clean"] and stats["rescaled"], stats
    if shape in ((24, 10, 6), (112, 40, 64)):
        assert stats["default_fails"], stats


@pytest.mark.gpu
@pytest.mark.parametrize("wavelet", [0, 1, 2])
def test_to_size_gpu(gpu, wavelet):
    for shape in ((24, 10, 6), (80, 2, 64), (256, 128, 64)):
        check_to_size(gpu, O.G1, *shape, wavelet)


@pytest.mark.gpu
def test_batch_gpu(gpu):
    check_batch(gpu, 256, 128, 64, 1, n=4)
    check_batch(gpu, 48, 20, 8, 0)


@pytest.mark.gpu
def test_flags_gpu(gpu):
    check_flags(gpu)


@pytest.mark.gpu
@pytest.mark.parametrize("wavelet", [0, 1, 2])
def test_fullsize_gpu(gpu, wavelet):
    """one 1920x1080x64 G1 chunk at q=80: the symbols of encode_stages (pinned by the golden tests), each stream the
    oracle's rANS encode with the H' table, and the oracle's decode equal to the library's"""
    w, h, f, q = 1920, 1080, 64, 80
    rgb = O.generate(O.G1, w, h, f)
    _, _, syms = pkg.FrameEncoder(q, WV[wavelet], api=gpu).encode_stages(rgb, w, h, f, want_coeffs=False)
    chunk = pkg.FrameEncoder(q, WV[wavelet], api=gpu, well_formed_tables=True).encode(rgb, w, h, f)
    alc = chunk.to_bytes()
    off = HDR
    for c in range(3):
        hdr = chunk.channel_header(c)
        hw, _ = well_formed_hist(np.bincount(syms[c], minlength=256))
        assert np.array_equal(hdr["histogram"], hw), (wavelet, c)
        stream = O.rans_encode(syms[c], O.freq_table_from_histogram(hw))
        assert alc[off:off + hdr["compressed_len"]] == stream, (wavelet, c)
        off += hdr["compressed_len"]
    rgb_dec, dec = O.decode(alc, stages=True)
    for c in range(3):
        assert np.array_equal(dec[c], syms[c]), (wavelet, c)
    assert np.array_equal(pkg.FrameDecoder(gpu).decode(chunk), rgb_dec), wavelet


@pytest.mark.gpu
def test_cli_well_formed(tmp_path):
    """encode --well-formed-tables with --chunk-frames and --max-bytes: every blob fits, the oracle decodes each to its
    exact symbols, and decode of the file equals the oracle's decode of those blobs"""
    w, h, f, cf = 64, 32, 20, 6                                        # three full chunks (one batch) + a 2-frame chunk
    rgb = O.generate(O.G1, w, h, f)
    src = tmp_path / "in.rgb"
    rgb.tofile(src)
    budget = 9000
    out = tmp_path / "out.alc"
    cli = [sys.executable, os.path.join(ROOT, "alice-codec_b200", "cli.py")]
    r = subprocess.run(cli + ["encode", str(src), "-W", str(w), "-H", str(h), "-f", str(f), "-w", "cdf97",
                              "--chunk-frames", str(cf), "--max-bytes", str(budget), "--well-formed-tables",
                              "-o", str(out)], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    assert "tables=well-formed" in r.stderr
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
        part = rgb[i * cf * per:(i * cf + nf) * per]
        want, syms, _ = expected_blob(oracle_coeffs(part, w, h, nf, 1), w, h, nf, pkg.quality_to_step(q), 1)
        assert blob == want, (i, q)
        _, dec = O.decode(blob, stages=True)
        assert all(np.array_equal(dec[c], syms[c]) for c in range(3)), (i, q)
    dec = tmp_path / "out.rgb"
    r = subprocess.run(cli + ["decode", str(out), "-o", str(dec)], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    assert np.array_equal(np.fromfile(dec, np.uint8), np.concatenate([O.decode(b) for b in blobs]))
    # without the flag: the default encode, byte for byte
    r = subprocess.run(cli + ["encode", str(src), "-W", str(w), "-H", str(h), "-f", str(f), "-w", "cdf97", "-q", "80",
                              "-o", str(out)], capture_output=True, text=True)
    assert r.returncode == 0 and "tables=" not in r.stderr, r.stderr
    assert out.read_bytes() == O.encode(rgb, w, h, f, 80, 1)

"""`alice-codec encode | decode | info` over the C ABI — same sub-commands, flags, messages and exit codes as the
reference's CLI (src/bin/main.rs:36-196), plus multi-chunk streams (SURVEY.md §8f-1): with --chunk-frames N the input
is cut into N-frame chunks, the chunks run as one batch (all rANS streams concurrently) and the output is the
concatenation of self-delimiting .alc blobs; `decode` and `info` accept such streams.  With --max-bytes N every chunk
(the whole input without --chunk-frames) is encoded at the highest quality whose .alc blob is at most N bytes; the chunk
is byte-identical to an encode at that quality, and -q is not used.  With --well-formed-tables every chunk stores
rANS tables that decode exactly on any decoder of the format (DESIGN.md 4.8); without it the output is the reference's.
With --min-psnr DB (which needs --well-formed-tables) every chunk is encoded at the lowest quality whose decode reaches DB
dB of PSNR against the input (DESIGN.md 4.9); the chunk is byte-identical to a well-formed encode at that quality.

    python -m alice_codec_b200.cli encode raw.rgb -W 1920 -H 1080 -f 64 -q 90 -w cdf53 -o out.alc
    (from the repo root: python alice-codec_b200/cli.py ...)
"""
from __future__ import annotations

import argparse
import os
import sys

import numpy as np

if __package__ in (None, ""):                       # run as a script: make the hyphen-named package importable
    sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    from __graft_entry__ import load_package
    pkg = load_package()
else:                                               # pragma: no cover - imported as alice_codec_b200.cli
    import alice_codec_b200 as pkg
from alice_codec_b200 import sharding              # noqa: E402

WAVELET_LABEL = {"cdf53": "CDF 5/3", "cdf97": "CDF 9/7", "haar": "Haar"}   # main.rs:166-170


def cmd_encode(a) -> None:
    if a.wavelet not in pkg.WAVELET_NAMES:
        raise ValueError(f"unknown wavelet '{a.wavelet}'; expected cdf53, cdf97, or haar")     # main.rs:74-83
    target = a.min_psnr
    if target is not None and not a.well_formed_tables:
        raise ValueError("--min-psnr needs --well-formed-tables (the PSNR curve describes that encode only)")
    if target is not None and a.max_bytes is not None:
        raise ValueError("--min-psnr and --max-bytes cannot be combined")
    rgb = np.fromfile(a.input, dtype=np.uint8)
    enc = pkg.FrameEncoder(a.quality, a.wavelet, well_formed_tables=a.well_formed_tables)
    # --max-bytes / --min-psnr: every chunk is encoded at the quality that these calls choose for `goal`
    goal = None
    if a.max_bytes is not None:
        goal, single, batched, label = (a.max_bytes, enc.encode_to_size, pkg.ChunkBatch.encode_host_to_size,
                                        f"max-bytes={a.max_bytes} per chunk")
    elif target is not None:
        goal, single, batched, label = (target, enc.encode_to_psnr, pkg.ChunkBatch.encode_host_to_psnr,
                                        f"min-psnr={target} dB per chunk")
    qualities = []                                  # the quality chosen for each chunk

    def one(part, nf):
        if goal is None:
            return enc.encode(part, a.width, a.height, nf).to_bytes()
        chunk, q = single(part, a.width, a.height, nf, goal)
        qualities.append(q)
        return chunk.to_bytes()

    if a.chunk_frames and a.frames > a.chunk_frames:
        per = a.width * a.height * 3
        if rgb.size != per * a.frames:
            raise pkg.CodecError(1, f"buffer size mismatch: expected {per * a.frames}, got {rgb.size}")
        # the full-size chunks run as ONE batch (all their rANS streams concurrently); a shorter last chunk goes alone
        n_full, rest = divmod(a.frames, a.chunk_frames)
        blobs = []
        if n_full >= 2:
            batch = pkg.ChunkBatch(a.quality, a.wavelet, a.width, a.height, a.chunk_frames, n_full,
                                   well_formed_tables=a.well_formed_tables)
            cb = per * a.chunk_frames
            parts = [np.ascontiguousarray(rgb[i * cb:(i + 1) * cb]) for i in range(n_full)]
            if goal is None:
                chunks = batch.encode_host([p.ctypes.data for p in parts])
            else:
                chunks, qs = batched(batch, [p.ctypes.data for p in parts], goal)
                qualities.extend(qs)
            blobs = [c.to_bytes() for c in chunks]
            batch.close()
        else:
            n_full = 0
        for t0 in range(n_full * a.chunk_frames, a.frames, a.chunk_frames):
            nf = min(a.chunk_frames, a.frames - t0)
            blobs.append(one(rgb[t0 * per:(t0 + nf) * per], nf))
        data = sharding.concat_stream(blobs)
    else:
        data = one(rgb, a.frames)
    with open(a.output, "wb") as f:
        f.write(data)
    ratio = len(data) / rgb.size if rgb.size else 0.0
    setting = f"quality={a.quality}" if goal is None else f"{label}, quality={','.join(str(q) for q in qualities)}"
    tables = ", tables=well-formed" if a.well_formed_tables else ""
    sys.stderr.write(f"encoded {a.width}x{a.height}x{a.frames} ({rgb.size} bytes) -> {len(data)} bytes "
                     f"({ratio * 100:.1f}% ratio, {setting}, wavelet={a.wavelet}{tables})\n")


def _blobs(data: bytes):
    """The .alc blobs of a file: a multi-chunk stream is split; anything after the last well-formed blob is ignored, as
    EncodedChunk::from_bytes ignores trailing bytes (pipeline.rs:303).  A file that does not even hold one blob is
    handed to from_bytes as is, which reports the reference's error."""
    out, off = [], 0
    while len(data) - off >= 3138 and data[off:off + 4] == b"ALCC":
        n = 3138 + sum(int.from_bytes(data[off + 18 + 1040 * c:off + 22 + 1040 * c], "little") for c in range(3))
        if off + n > len(data):
            break
        out.append(data[off:off + n])
        off += n
    return out or [data]


def cmd_decode(a) -> None:
    data = open(a.input, "rb").read()
    blobs = _blobs(data)
    dec = pkg.FrameDecoder()
    with open(a.output, "wb") as f:
        total = 0
        for blob in blobs:
            chunk = pkg.EncodedChunk.from_bytes(blob)
            rgb = dec.decode(chunk)
            rgb.tofile(f)
            total += rgb.size
            sys.stderr.write(f"decoded {chunk.width}x{chunk.height}x{chunk.frames} -> {rgb.size} bytes (raw RGB)\n")


def cmd_info(a) -> None:
    data = open(a.input, "rb").read()
    chunk = pkg.EncodedChunk.from_bytes(data)              # the first blob (trailing bytes are ignored, pipeline.rs:303)
    raw = chunk.width * chunk.height * chunk.frames * 3
    ratio = chunk.compressed_size / raw if raw else 0.0
    print("ALICE-Codec Bitstream Info")
    print(f"  File:        {a.input}")
    print(f"  File size:   {len(data)} bytes")
    print(f"  Width:       {chunk.width}")
    print(f"  Height:      {chunk.height}")
    print(f"  Frames:      {chunk.frames}")
    print(f"  Wavelet:     {WAVELET_LABEL[chunk.wavelet]}")
    print(f"  Payload:     {chunk.compressed_size} bytes")
    print(f"  Raw size:    {raw} bytes (uncompressed RGB)")
    print(f"  Ratio:       {ratio * 100:.1f}%")
    n = len(_blobs(data))
    if n > 1:
        print(f"  Chunks:      {n} (multi-chunk stream)")


def main(argv=None) -> int:
    ap = argparse.ArgumentParser(prog="alice-codec", description="ALICE-Codec (.alc) on B200")
    sub = ap.add_subparsers(dest="command", required=True)
    e = sub.add_parser("encode", help="Encode raw RGB frames into an .alc bitstream")
    e.add_argument("input")
    e.add_argument("-o", "--output", required=True)
    e.add_argument("-W", "--width", type=int, required=True)
    e.add_argument("-H", "--height", type=int, required=True)
    e.add_argument("-f", "--frames", type=int, default=1)
    e.add_argument("-q", "--quality", type=int, default=90)
    e.add_argument("-w", "--wavelet", default="cdf53")
    e.add_argument("--chunk-frames", type=int, default=0, help="cut the input into chunks of this many frames (0 = one chunk)")
    e.add_argument("--max-bytes", type=int, default=None,
                   help="byte budget per chunk: encode each chunk at the highest quality whose .alc fits (-q is not used)")
    e.add_argument("--min-psnr", type=float, default=None, metavar="DB",
                   help="PSNR target per chunk: encode each chunk at the lowest quality whose decode reaches DB dB "
                        "(needs --well-formed-tables; -q is not used)")
    e.add_argument("--well-formed-tables", action="store_true",
                   help="store rANS tables that every .alc decoder decodes exactly (the header histograms become table "
                        "specifications instead of symbol counts)")
    d = sub.add_parser("decode", help="Decode an .alc bitstream back to raw RGB")
    d.add_argument("input")
    d.add_argument("-o", "--output", required=True)
    i = sub.add_parser("info", help="Show metadata of an .alc bitstream")
    i.add_argument("input")
    a = ap.parse_args(argv)
    try:
        if a.command == "encode" and not 0 <= a.quality <= 255:            # the reference's -q is a u8 (main.rs:54)
            raise ValueError(f"invalid value '{a.quality}' for '--quality': not in 0..=255")
        {"encode": cmd_encode, "decode": cmd_decode, "info": cmd_info}[a.command](a)
    except (ValueError, OSError) as ex:
        sys.stderr.write(f"error: {ex}\n")                 # main.rs:104-107
        return 1
    return 0


if __name__ == "__main__":
    sys.exit(main())

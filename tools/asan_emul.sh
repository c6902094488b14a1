#!/bin/bash
# Memory-safety check of the kernel sources where no GPU tool is available (compute-sanitizer is closed on this
# pool): the SIMT-emulator build (tests/emul/cuda_emul.h: device memory = malloc, shared memory = static arrays) is
# compiled with AddressSanitizer and driven through the same parity checks as tests/test_emul_parity.py.
set -e
ROOT=$(cd "$(dirname "$0")/.." && pwd)
OUT=$ROOT/tests/emul/_build/asan   # under tests/emul/_build: parity.device_of treats it as an emulator build
mkdir -p "$OUT"
for f in k_forward k_fwd_fused k_inv_fused k_inverse k_rans k_generic k_wavelet_i32 k_rdo k_rate k_synth engine lossless capi; do
  g++ -O1 -g -std=c++17 -fPIC -fwrapv -DALICE_EMUL -x c++ -Wno-unknown-pragmas -I "$ROOT/tests/emul" \
      -fsanitize=address -fno-omit-frame-pointer -c "$ROOT/alice-codec_b200/csrc/$f.cu" -o "$OUT/$f.o" &
done
wait
g++ -shared -fsanitize=address -o "$OUT/libalice_codec_asan.so" "$OUT"/*.o
cat > "$OUT/run.py" <<PY
import sys
sys.path.insert(0, "$ROOT"); sys.path.insert(0, "$ROOT/tests")
import numpy as np
import parity
from ref_vectors import SURVEY_KATS
import oracle as O
api = parity.pkg.Api("$OUT/libalice_codec_asan.so")
for row in SURVEY_KATS:
    parity.check_kat(api, row)
for shape in [(1, 1, 1), (3, 5, 1), (5, 3, 3), (7, 2, 4), (66, 6, 2), (130, 4, 2), (12, 6, 64), (256, 6, 2), (260, 4, 64)]:
    for wv in (0, 1, 2):
        parity.check_encode_decode(api, O.G1, *shape, 80, wv)
for kind, q in [(O.G2, 100), (O.G2, 0), (O.G0, 100)]:
    for wv in (0, 1, 2):
        parity.check_encode_decode(api, kind, 24, 10, 6, q, wv)
rng = np.random.default_rng(2)
parity.check_rans_api(api, rng, n=3000)
parity.check_errors(api)
parity.check_decode_foreign_headers(api, rng)
parity.check_shared_workspace_batch(api)
parity.check_wavelet_api(api, rng, [2, 3, 9, 31], [(5, 3), (16, 9)], [(5, 3, 2), (8, 6, 3)])
# interior strips of the xy / yx kernels (unchecked vector loads), 63/64/65-frame chunks (rolled temporal loops)
for shape in [(380, 10, 3), (512, 34, 2), (250, 30, 3), (260, 6, 63), (264, 4, 65), (16, 4, 64)]:
    for wv in (0, 1, 2):
        parity.check_encode_decode(api, O.G1, *shape, 80, wv)
parity.check_rdo_exact_variance(api, rng, sizes=(1, 31, 1025, 5000))
parity.check_rdo_octants(api, rng, shapes=((8, 6, 4), (9, 7, 5), (2, 2, 2)))
parity.check_rans_interleaved(api, rng, sizes=(0, 1, 5, 1024, 4099))
# the fused front-end / back-end kernels, the fast Wavelet2D/3D kernels, the lossless set, the payload arena, submit/collect
for shape in [(80, 2, 64), (128, 6, 64), (112, 40, 64)]:
    for wv in (0, 1, 2):
        parity.check_encode_decode(api, O.G1, *shape, 80, wv)
parity.check_wavelet_fast_path(api)
parity.check_lossless_set(api)
parity.check_payload_arena(api)
parity.check_submit_collect(api)
parity.check_stream_device(api)
parity.check_shifted_in_place(api)
# the PSNR curve: the SSE mode of the fused back-end (80x2x64) and the general path (24x10x6)
for shape in [(24, 10, 6), (80, 2, 64)]:
    for wv in (0, 1, 2):
        parity.pkg.FrameEncoder(80, parity.WV[wv], api=api, well_formed_tables=True).psnr_curve(O.generate(O.G1, *shape), *shape)
print("ASAN RUN OK")
PY
LD_PRELOAD=$(gcc -print-file-name=libasan.so) ASAN_OPTIONS=detect_leaks=0:detect_stack_use_after_return=0 python "$OUT/run.py"

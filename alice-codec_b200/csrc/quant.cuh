// quant.cuh — the pipeline's quantiser + zig-zag symbol map, shared by the encode front-end kernels.
//
// Reference: Quantizer::quantize (src/quant.rs:89-97) with dead_zone == step (Quantizer::new, quant.rs:70-75, the
// only form FrameEncoder::encode uses, pipeline.rs:469), then to_symbols (src/quant.rs:555-560, `as u8` wraps).
#pragma once
#include "compat.h"

namespace alice {

struct QuantDev {
    int step, dz, half_dz;
    uint32_t magic;  // ceil(2^32 / step) for step >= 2
};

ALICE_HD QuantDev make_quant_dev(int step) {
    QuantDev q;
    q.step = step;
    q.dz = step;
    q.half_dz = step / 2;
    q.magic = step >= 2 ? (uint32_t)((((uint64_t)1 << 32) + step - 1) / step) : 0;
    return q;
}

ALICE_D uint32_t quant_symbol(int v, const QuantDev &q) {
    // Without branches: for |v| < step the numerator |v| - step/2 is below step, so clamping it at 0 gives the dead
    // zone; the symbol 2q-1 (v > 0) / 2q (v < 0) is max(2q - 1 - (v >> 31), 0) because q == 0 when v == 0.
    const int a = v < 0 ? -v : v;
    const int n = max(a - q.half_dz, 0);
    const uint32_t qa = q.step == 1 ? (uint32_t)n : __umulhi((uint32_t)n, q.magic);   // exact: n < 2^26, magic = ceil(2^32/step)
    const int s = max((int)(2u * qa) - 1 - (v >> 31), 0);
    return (uint32_t)s & 0xffu;
}

}  // namespace alice

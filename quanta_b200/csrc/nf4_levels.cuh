// The 16 NF4 code values (Quanta/functional/quantization.py:105-110), used by the NF4 quantizer and dequantizer, the
// NF4 GEMM kernels and quanta_nf4_levels.  One initializer list serves the device table and the host copy.  Only the
// files that read the levels include this header: every module that defines the table carries it in its constant bank.
#pragma once

#define QUANTA_NF4_LEVELS                                                                              \
    {-1.0f, -0.6961928009986877f, -0.5250730514526367f, -0.39491748809814453f,                         \
     -0.28444138169288635f, -0.18477343022823334f, -0.09105003625154495f, 0.0f,                        \
     0.07958029955625534f, 0.16093020141124725f, 0.24611230194568634f, 0.33791524171829224f,           \
     0.44070982933044434f, 0.5626170039176941f, 0.7229568362236023f, 1.0f}

namespace quanta {
static __constant__ float kNf4Levels[16] = QUANTA_NF4_LEVELS;
}  // namespace quanta

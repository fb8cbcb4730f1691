/* Exhaustive CPU check of the division the int8 input-gradient kernel (csrc/gemm_dgrad.cu,
 * dequant_word8_row) uses for W16[n,k] = round_act(qw[n,k] / cw[n]):
 *
 *     y = rcp_rn(cw);  q0 = a * y;  r = fma(-cw, q0, a);  q = fma(y, r, q0)
 *
 * For every code a = 1..127 and every float cw in [2^-60, 2^60] (the window in which the kernel
 * takes this sequence, the window of affine_quotient in common.cuh; outside it the kernel divides
 * with __fdiv_rn), q must equal the IEEE quotient a / cw bit for bit.  Negative codes follow by
 * the symmetry of round-to-nearest-even, and a = 0 gives +0 both ways.  Prints the number of
 * cases and mismatches; exits 1 on a mismatch.
 *
 *     cc -O2 -fopenmp -ffp-contract=off tools/check_rowwise_div.c -o /tmp/check_rowwise_div -lm
 *     /tmp/check_rowwise_div            # ~1.3e11 cases */
#include <math.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

static float bits_to_float(uint32_t u) { float f; memcpy(&f, &u, 4); return f; }
static uint32_t float_to_bits(float f) { uint32_t u; memcpy(&u, &f, 4); return u; }

int main(void) {
    const uint32_t lo = float_to_bits(0x1p-60f), hi = float_to_bits(0x1p60f);
    long long cases = 0, bad = 0;
#pragma omp parallel for schedule(dynamic, 4096) reduction(+ : cases, bad)
    for (long long u = lo; u <= (long long)hi; ++u) {
        const float cw = bits_to_float((uint32_t)u);
        const float y = 1.0f / cw;
        for (int i = 1; i <= 127; ++i) {
            const float a = (float)i;
            const float q0 = a * y;
            const float r = fmaf(-cw, q0, a);
            const float q = fmaf(y, r, q0);
            const float ref = a / cw;
            bad += float_to_bits(q) != float_to_bits(ref);
            ++cases;
        }
    }
    printf("cw in [2^-60, 2^60], a = 1..127: %lld cases, %lld mismatches\n", cases, bad);
    return bad != 0;
}

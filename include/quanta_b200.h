/*
 * quanta_b200 — C ABI of the B200 (sm_100a) weight-quantization hot path.
 *
 * This is the drop-in boundary: a plain C shared library (libquanta_b200.so)
 * that a binding on the reference side (ctypes from
 * Quanta/backends/cuda/quantization.py, see INTEGRATION.md) calls with raw
 * device pointers.  Every entry point is
 *   - non-allocating (the caller owns inputs, outputs and the workspace),
 *   - asynchronous on the caller-supplied cudaStream_t (passed as void*),
 *   - non-throwing: returns 0 on success, a negative QUANTA_E* code for
 *     argument errors, or a positive cudaError_t from the launch.
 * No host synchronisation happens inside any call: the reference's host-side
 * decisions (`if max_val == min_val`, `torch.allclose(...)`) are evaluated on
 * the device.
 *
 * file:line citations are relative to the reference tree (ved1beta/Quanta).
 */
#ifndef QUANTA_B200_H
#define QUANTA_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define QUANTA_B200_ABI_VERSION 1

#if defined(__GNUC__)
#define QUANTA_API __attribute__((visibility("default")))
#else
#define QUANTA_API
#endif

/* reduction granularity of scale / zero_point */
#define QUANTA_MODE_TENSOR 0   /* per_channel=False : one scale for the whole tensor          */
#define QUANTA_MODE_DIM0   1   /* per_channel=True  : min/max over dim 0 -> one scale per column */
#define QUANTA_MODE_BLOCK  2   /* blockwise: per_channel applied to x.reshape(-1, block).t()    */

/* element types of floating-point buffers */
#define QUANTA_F32  0
#define QUANTA_F16  1
#define QUANTA_BF16 2

/* error codes (negative); positive return values are cudaError_t */
#define QUANTA_OK              0
#define QUANTA_EINVAL         -1   /* bad argument (null pointer, bits not 4/8, n % block != 0 ...) */
#define QUANTA_EUNSUPPORTED   -2   /* combination not implemented                                    */
#define QUANTA_EWORKSPACE     -3   /* workspace too small, see quanta_workspace_bytes                */
#define QUANTA_EDRIVER        -4   /* CUDA driver entry point (tensor-map encode) unavailable        */

/* workspace queries */
#define QUANTA_OP_QUANTIZE_AFFINE    0
#define QUANTA_OP_BACKEND_QUANTIZE   1
#define QUANTA_OP_BACKEND_DEQUANTIZE 2
#define QUANTA_OP_GEMM               3
#define QUANTA_OP_INT8_OUTLIER       4
#define QUANTA_OP_BASE_QUANTIZE      5   /* rows, cols as passed to quanta_base_quantize */

QUANTA_API int         quanta_abi_version(void);
QUANTA_API const char* quanta_error_string(int code);

/* Bytes of device workspace needed by `op` on a [rows, cols] problem
 * (QUANTA_OP_GEMM: rows = M, cols = N;  QUANTA_OP_INT8_OUTLIER: rows = M,
 * cols = K).  Always >= 256.  The first 64 KB of the QUANTA_OP_GEMM workspace
 * hold arrival counters: they must be zero before the first call and every
 * call leaves them zero (allocate the buffer zero-filled, once).  The same
 * holds for the first 256 bytes of the QUANTA_OP_QUANTIZE_AFFINE /
 * QUANTA_OP_BACKEND_QUANTIZE workspace (grid-barrier counters of the
 * single-launch per-tensor kernel): keep that buffer for these entries only.
 * Bytes 48-55 of that header are the one exception to "zero": they may hold the
 * device-visible address of a host-mapped int32 (cudaHostAlloc) error flag.  If
 * the grid barrier of a call cannot complete (stale counters, grid not
 * co-resident) the kernel gives up after ~1 s, stores 1 to that flag, leaves the
 * counters zero and finishes (the outputs of that call are undefined); the host
 * checks the flag before its next call.  With no flag registered the time-out is
 * silent.                                                                     */
QUANTA_API size_t quanta_workspace_bytes(int op, int64_t rows, int64_t cols);

/* ---- convention A: Quanta/functional/quantization.py "linear" -------------
 *
 * Replaces quantize_8bit / quantize_4bit -> quantize_{8,4}bit_linear
 * (functional/quantization.py:7-31, :73-99, :185-210):
 *     mn, mx = min, max         (all elements | over dim 0 | per block)
 *     if mx == mn: mx = mn + 1e-6
 *     scale = (mx - mn) / L ; zero_point = mn            (L = 255 or 15)
 *     q = clamp(round((x - mn) / scale), 0, L)           -> uint8
 * x is a contiguous [rows, cols] tensor (any shape flattened to rows x cols;
 * for TENSOR and BLOCK only rows*cols matters).  BLOCK: (rows*cols) % block
 * must be 0; block b covers flat elements [b*block, (b+1)*block).
 * Outputs: q_out uint8, one code per byte (values 0..L), or — when
 * pack4 != 0 (bits == 4 only) — nibble-packed exactly as pack_4bit_tensor
 * (utils/utils.py:23-35: even index -> low nibble, one zero pad if odd);
 * scale_out / zp_out float32: 1 value (TENSOR), cols values (DIM0),
 * rows*cols/block values (BLOCK).  x_dtype F16/BF16 inputs are widened to
 * fp32 first and then follow the fp32 arithmetic (declared deviation: the
 * reference would round every intermediate to the 16-bit type).          */
QUANTA_API int quanta_quantize_affine(const void* x, int x_dtype, int64_t rows, int64_t cols,
                           int mode, int64_t block, int bits, int pack4,
                           uint8_t* q_out, float* scale_out, float* zp_out,
                           void* workspace, size_t workspace_bytes, void* stream);

/* The same blockwise quantization (mode BLOCK) over `count` independent
 * tensors in as few launches as possible — the fused form of the per-parameter
 * loop of ModelQuantize.quantize (Quanta/functional/model.py:254-289, :60-71),
 * which calls quantize_*bit once per parameter.  xs / q_outs / scale_outs /
 * zp_outs are HOST arrays of device pointers, numels[i] the element count of
 * tensor i (a multiple of `block`); results are identical to `count` calls of
 * quanta_quantize_affine(..., QUANTA_MODE_BLOCK, ...).                        */
QUANTA_API int quanta_quantize_block_batch(const void* const* xs, const int64_t* numels, int count, int x_dtype,
                                int64_t block, int bits, int pack4,
                                uint8_t* const* q_outs, float* const* scale_outs, float* const* zp_outs,
                                void* stream);

/* Replaces dequantize_8bit / dequantize_4bit, quant_type="linear"
 * (functional/quantization.py:33-38, :53-58): out = q.float() * scale + zp,
 * multiply and add rounded separately.  packed4 != 0: q holds nibble-packed
 * codes (P1 layout) and rows*cols counts CODES.  out_dtype F32 is the
 * reference behaviour; F16/BF16 round the fp32 result once more.          */
QUANTA_API int quanta_dequantize_affine(const uint8_t* q, int packed4, int64_t rows, int64_t cols,
                             int mode, int64_t block, const float* scale, const float* zp,
                             void* out, int out_dtype, void* stream);

/* The same blockwise dequantization (mode BLOCK) over `count` tensors in
 * ceil(count / 16) launches — the fused form of calling
 * QuantizationState.dequantize_tensor (Quanta/functional/state.py:246-281),
 * i.e. dequantize_*bit, once per recorded tensor.  qs / scales / zps / outs are HOST arrays
 * of device pointers, numels[i] the CODE count of tensor i (a positive multiple
 * of `block`, block % 4 == 0); results are identical to `count` calls of
 * quanta_dequantize_affine(..., QUANTA_MODE_BLOCK, ...).                      */
QUANTA_API int quanta_dequantize_block_batch(const uint8_t* const* qs, const int64_t* numels, int count, int packed4,
                                  int64_t block, const float* const* scales, const float* const* zps,
                                  void* const* outs, int out_dtype, void* stream);

/* ---- NF4 codebook: Quanta/functional/quantization.py:101-118, :59-61 --------
 * quantize_4bit(tensor, quant_type="nf4"): abs_max = max|x|, normalized =
 * x / abs_max, code = argmin_l |normalized - level_l| (first index on ties,
 * NaN -> 0).  block = 0: one abs_max for the whole tensor (the reference);
 * block = 16 * 2^j <= 512: one abs_max per block of flat elements (the
 * reference function applied to every block), n % block == 0.  q_out: one
 * code per byte, or nibble-packed (P1 layout) when pack4 != 0; absmax_out: 1
 * or n / block floats.  dequantize: out = level[code] * abs_max.
 * quanta_nf4_levels writes the 16-entry table (host memory).               */
QUANTA_API int quanta_nf4_levels(float* out16);
QUANTA_API int quanta_quantize_nf4(const void* x, int x_dtype, int64_t n, int64_t block, int pack4,
                        uint8_t* q_out, float* absmax_out, void* stream);
QUANTA_API int quanta_dequantize_nf4(const uint8_t* q, int packed4, int64_t n, int64_t block,
                          const float* absmax, void* out, int out_dtype, void* stream);

/* ---- 4-bit nibble pack / unpack: Quanta/utils/utils.py:23-48 -------------
 * pack:   packed[i] = q[2i] | (q[2i+1] << 4) in uint8 arithmetic, one zero
 *         pad if n is odd; inputs > 15 are not masked (reference behaviour).
 *         packed holds (n+1)/2 bytes.
 * unpack: out[2i] = b & 0xF, out[2i+1] = b >> 4; out holds 2*nbytes codes. */
QUANTA_API int quanta_pack4(const uint8_t* q, int64_t n, uint8_t* packed, void* stream);
QUANTA_API int quanta_unpack4(const uint8_t* packed, int64_t nbytes, uint8_t* out, void* stream);
/* The opposite nibble order of ModelQuantize._pack_tensor / _unpack_tensor
 * (Quanta/functional/model.py:73-94): packed[i] = (q[2i] << 4) | q[2i+1] — the
 * first element goes to the HIGH nibble; one zero pad if n is odd.             */
QUANTA_API int quanta_pack4_hi(const uint8_t* q, int64_t n, uint8_t* packed, void* stream);
QUANTA_API int quanta_unpack4_hi(const uint8_t* packed, int64_t nbytes, uint8_t* out, void* stream);

/* ---- convention B: Quanta/backends/cpu/quantization.py -------------------
 *
 * Replaces quantize_8bit_cpu / quantize_4bit_cpu (:10-59, :86-135), i.e. the
 * semantics quantize_{8,4}bit_cuda must have behind
 * Quanta/backends/__init__.py:61,105.  per_channel reduces over dim 0 of the
 * [rows, cols] tensor.  symmetric: scale = rcp(absmax)*Q, zp = 0,
 * q = clamp(round(x*scale), -Q, Q) + OFF; asymmetric: scale = rcp(mx-mn)*L,
 * zp = round(-mn*scale), q = clamp(round(x*scale + zp), 0, L).  If
 * allclose(min, max) holds for ALL channels the reference's early-out is
 * reproduced: codes 0, scale 1, zp = min.  scale_out / zp_out: 1 or cols.  */
QUANTA_API int quanta_backend_quantize(const void* x, int x_dtype, int64_t rows, int64_t cols,
                            int per_channel, int symmetric, int bits,
                            uint8_t* q_out, float* scale_out, float* zp_out,
                            void* workspace, size_t workspace_bytes, void* stream);

/* Replaces dequantize_8bit_cpu / dequantize_4bit_cpu (:61-84, :137-160):
 * if allclose(zp, 0) for all channels, q' = int8(q) - OFF else q' = q;
 * out = (q'.float() - zp) / scale (true divide).  nchan = 1 or cols.       */
QUANTA_API int quanta_backend_dequantize(const uint8_t* q, int64_t rows, int64_t cols, int64_t nchan, int bits,
                              const float* scale, const float* zp, float* out,
                              void* workspace, size_t workspace_bytes, void* stream);

/* ---- convention C: Quanta/functional/base.py (BaseQuantizer, row N4) -------
 *
 * Replaces BaseQuantizer(num_bits, symmetric).quantize(tensor, per_channel)
 * (base.py:11-59): symmetric as convention B (scale = rcp(absmax)*Q, zp = 0,
 * codes offset by 2^(bits-1)); asymmetric scale = rcp(mx-mn)*L, zp = mn (a
 * float offset), q = clamp(round((x - zp)*scale), 0, L).  If allclose(min, max)
 * holds for ALL channels, scale = 1 and zp = min and the codes are still computed
 * with them (base.py:26-27).  bits = 8 or 4; per_channel reduces over dim 0 of
 * the [rows, cols] tensor; scale_out / zp_out: 1 or cols values.
 * quanta_base_dequantize replaces .dequantize (base.py:61-72): symmetric
 * (int8(q) - 2^(bits-1)) / scale, else q / scale + zp (true divides); the
 * branch is the quantizer's `symmetric`, not inferred from zp.                 */
QUANTA_API int quanta_base_quantize(const void* x, int x_dtype, int64_t rows, int64_t cols,
                         int per_channel, int symmetric, int bits,
                         uint8_t* q_out, float* scale_out, float* zp_out,
                         void* workspace, size_t workspace_bytes, void* stream);
QUANTA_API int quanta_base_dequantize(const uint8_t* q, int64_t rows, int64_t cols, int64_t nchan, int bits,
                           int symmetric, const float* scale, const float* zp, float* out, void* stream);

/* ---- the rest of the quant_type switch (row N4): nf8, fp4, fp8 ---------------
 *
 * quantize_8bit(..., quant_type="nf8")  Quanta/functional/quantization.py:170-183:
 *   256 levels tanh(2*linspace(-1,1,256)) (quanta_nf8_levels returns the reference's
 *   own float32 values), abs-max normalisation, nearest level (first index on ties);
 *   block = 0: whole tensor (the reference), block = 16 * 2^j <= 512: per block.
 * quantize_4bit(..., "fp4") / quantize_8bit(..., "fp8")  :120-168:
 *   code = sign | exponent field | mantissa, field = clamp(round(log2|x| + bias), 0, E)
 *   with bias 1 / 7, E = 3 / 15 and 1 / 3 mantissa bits; one code per byte; zero
 *   encodes as field = bias, mantissa 0 and decodes to 1.0 like the reference.
 * dequantize_*bit(..., quant_type=...)  :39-49, :62-69.                          */
QUANTA_API int quanta_nf8_levels(float* out256);
QUANTA_API int quanta_quantize_nf8(const void* x, int x_dtype, int64_t n, int64_t block,
                        uint8_t* q_out, float* absmax_out, void* stream);
QUANTA_API int quanta_dequantize_nf8(const uint8_t* q, int64_t n, int64_t block, const float* absmax,
                          void* out, int out_dtype, void* stream);
QUANTA_API int quanta_quantize_fp(const void* x, int x_dtype, int64_t n, int bits, uint8_t* q_out, void* stream);
QUANTA_API int quanta_dequantize_fp(const uint8_t* q, int64_t n, int bits, int bias,
                         void* out, int out_dtype, void* stream);

/* ---- convert_precision for per-tensor linear codes (row N3) ------------------
 * Replaces convert_precision(q, {type "linear", scalar scale / zero_point}, target_bits, "linear")
 * (utils/utils.py:216-279), i.e. dequantize_*bit + quantize_*bit per tensor, bit for bit, in two
 * passes over the CODES (3 B/element instead of 14): q holds n codes (one per byte, any source bit
 * depth), src_scale / src_zp are DEVICE pointers to one float each; q_out n codes, scale_out /
 * zp_out one float each.  workspace >= 256 bytes of scratch.                   */
QUANTA_API int quanta_convert_linear(const uint8_t* q, int64_t n, const float* src_scale, const float* src_zp,
                          int target_bits, uint8_t* q_out, float* scale_out, float* zp_out,
                          void* workspace, size_t workspace_bytes, void* stream);

/* ---- dequantize-then-matmul behind Quanta/nn/linear.py -------------------
 *
 * Replaces the placeholder F.linear in Linear4bit.forward (nn/linear.py:81-83)
 * and Linear8bitLt.forward (:43-45):  y[M,N] = x[M,K] . dequant(Wq)[N,K]^T + bias
 * with Wq in convention A, blockwise along K (block | K, block % 64 == 0):
 *   bits 8: wq uint8 [N, K];  bits 4: wq nibble-packed [N, K/2] (P1 layout)
 *   scale, zp float32 [N, K/block].
 * x, y, bias are `act_dtype` (F16 or BF16); accumulation is fp32 on the
 * tcgen05 tensor cores.  bias may be NULL.                                 */
QUANTA_API int quanta_gemm_wna16(const void* x, int act_dtype, const uint8_t* wq, int bits,
                      const float* scale, const float* zp, int64_t block,
                      const void* bias, void* y, int64_t M, int64_t N, int64_t K,
                      void* workspace, size_t workspace_bytes, void* stream);

/* Column-parallel form of quanta_gemm_wna16 (SURVEY 8(e), the tensor-parallel
 * Linear*: rank r holds rows [col0, col0+N) of the weight).  The tile epilogue
 * writes y[:, col0:col0+N] into EVERY buffer of `ys` (host array of n_out <= 8
 * device pointers, row pitch `ldy` elements >= col0 + N): the local y and the
 * peer-mapped y of the other ranks (CUDA IPC / symmetric memory over NVLink),
 * so the output all-gather happens inside the GEMM.  The caller orders the
 * ranks afterwards (one cross-rank barrier) before reading y.              */
QUANTA_API int quanta_gemm_wna16_scatter(const void* x, int act_dtype, const uint8_t* wq, int bits,
                              const float* scale, const float* zp, int64_t block,
                              const void* bias, void* const* ys, int n_out, int64_t ldy, int64_t col0,
                              int64_t M, int64_t N, int64_t K,
                              void* workspace, size_t workspace_bytes, void* stream);

/* quanta_gemm_wna16_scatter with the ranks' synchronisation INSIDE the kernel
 * (decode-sized batches: the separate barrier kernel costs as much as the GEMM).
 * peer_flags: host array of `world` device pointers, peer_flags[r] = rank r's
 * flag array of `world` unsigned ints in peer-mapped (symmetric) memory,
 * zero-initialised once; epoch_counter: one unsigned int in this rank's own
 * device memory, zero-initialised once, owned by the layer (the kernel
 * increments it: replaying the launch from a CUDA graph advances the epoch
 * like an eager call; every rank must run the same sequence of calls).  The
 * last CTA of this rank's grid stores the new epoch into
 * peer_flags[r][rank] of every peer after all of the grid's output stores are
 * performed system-wide, and leaves only when peer_flags[rank][r] has reached
 * that epoch for every r: completion of the kernel on a rank means that every
 * rank's columns are in that rank's y.  Returns QUANTA_EUNSUPPORTED when the
 * shape is outside the small-batch kernel (M > 16, block != 64, K % 256 != 0);
 * the caller then falls back to quanta_gemm_wna16_scatter + its own barrier. */
QUANTA_API int quanta_gemm_wna16_scatter_sync(const void* x, int act_dtype, const uint8_t* wq, int bits,
                              const float* scale, const float* zp, int64_t block,
                              const void* bias, void* const* ys, int n_out, int64_t ldy, int64_t col0,
                              int64_t M, int64_t N, int64_t K,
                              void* workspace, size_t workspace_bytes,
                              void* const* peer_flags, int rank, int world, unsigned int* epoch_counter, void* stream);

/* The cross-rank barrier behind quanta_gemm_wna16_scatter as one tiny kernel
 * that overlaps with the NEXT layer: it is launched with programmatic stream
 * serialization and releases its dependents at once, so the next GEMM's weight
 * stream starts while the ranks are still meeting; that GEMM's activation
 * loads and writes wait for the barrier.  peer_flags / epoch_counter as in
 * quanta_gemm_wna16_scatter_sync (the two may share them).                   */
QUANTA_API int quanta_peer_barrier(void* const* peer_flags, int rank, int world, unsigned int* epoch_counter,
                                   void* stream);

/* The same for NF4 weights — Linear4bit's default quant_type="nf4"
 * (nn/linear.py:58): wq nibble-packed NF4 codes [N, K/2], absmax float32
 * [N, K/block] (quanta_quantize_nf4 with block | K, block % 64 == 0);
 * y = x . (level[code] * absmax)[N,K]^T + bias.                            */
QUANTA_API int quanta_gemm_nf4a16(const void* x, int act_dtype, const uint8_t* wq, const float* absmax,
                       int64_t block, const void* bias, void* y, int64_t M, int64_t N, int64_t K,
                       void* workspace, size_t workspace_bytes, void* stream);

/* Input gradient of quanta_gemm_wna16 (the backward of Linear4bit /
 * Linear8bitLt for a frozen quantized weight):
 *     dx[M,K] = dy[M,N] . dequant(Wq)[N,K]
 * with wq / scale / zp / block exactly as passed to the forward; the
 * weights are dequantized to bit-for-bit the 16-bit values the forward
 * multiplies with.  dy, dx are `act_dtype` (F16 or BF16), fp32 accumulation.
 * dy rows have a pitch of round_up(N, 8) elements (16-byte aligned rows for
 * TMA); columns N .. pitch-1 are never read.  dx is [M, K] contiguous.
 * workspace: quanta_workspace_bytes(QUANTA_OP_GEMM, M, K), the same
 * zero-initialised buffer as the forward's (the counters are left zero).  */
QUANTA_API int quanta_gemm_wna16_dgrad(const void* dy, int act_dtype, const uint8_t* wq, int bits,
                            const float* scale, const float* zp, int64_t block, void* dx,
                            int64_t M, int64_t N, int64_t K,
                            void* workspace, size_t workspace_bytes, void* stream);

/* The same for NF4 weights (quanta_gemm_nf4a16):
 * dx = dy . (level[code] * absmax)[N,K].                                    */
QUANTA_API int quanta_gemm_nf4a16_dgrad(const void* dy, int act_dtype, const uint8_t* wq, const float* absmax,
                             int64_t block, void* dx, int64_t M, int64_t N, int64_t K,
                             void* workspace, size_t workspace_bytes, void* stream);

/* Input gradient of quanta_int8_outlier_matmul (the backward of
 * Linear8bitLt(outlier_split=True) for a frozen weight), straight-through:
 *     dx[M,K] = dy[M,N] . W16[N,K],   W16[n,k] = round_act(qw[n,k] / cw[n])
 * (an IEEE divide, then one rounding to act_dtype): bit for bit the weights
 * the forward multiplies its outlier columns with.  The threshold, the
 * outlier set and the int8 quantization of x do not enter.  qw / cw as
 * passed to the forward; K % 16 == 0.  dy, dx are `act_dtype` (F16 or BF16),
 * fp32 accumulation; dy rows have a pitch of round_up(N, 8) elements and dx
 * is [M, K] contiguous.  workspace: quanta_workspace_bytes(QUANTA_OP_GEMM,
 * M, K), the zero-initialised buffer of quanta_gemm_wna16_dgrad.          */
QUANTA_API int quanta_int8_outlier_dgrad(const void* dy, int act_dtype, const int8_t* qw, const float* cw, void* dx,
                              int64_t M, int64_t N, int64_t K,
                              void* workspace, size_t workspace_bytes, void* stream);

/* LLM.int8()-style outlier-split matmul for Linear8bitLt.threshold
 * (nn/linear.py:20,25; unused by the reference — semantics defined by this
 * repository, see oracle/oracle_np.py:int8_outlier_matmul).
 *   qw int8 [N,K] row-wise symmetric codes, cw float32 [N] multipliers
 *   (127/absmax), x/y/bias `act_dtype`.                                    */
QUANTA_API int quanta_int8_outlier_matmul(const void* x, int act_dtype, const int8_t* qw, const float* cw,
                               float threshold, const void* bias, void* y,
                               int64_t M, int64_t N, int64_t K,
                               void* workspace, size_t workspace_bytes, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* QUANTA_B200_H */

/* tfcb200.h -- C ABI of libtfcb200.so: the B200-native replacement for the data-parallel hot path of
 * tensorflow/compression (range coder ops, PmfToQuantizedCdf, GDN/IGDN forward + backward).
 *
 * This is the drop-in boundary: plain pointers and sizes, no torch / TF types.  Every entry point
 * names the reference interface it replaces (paths relative to /root/reference).
 *
 * Conventions
 *   - `_dev` pointers are CUDA device pointers on the current device, `_host` pointers are host memory.
 *   - `stream` is a cudaStream_t passed as void* (NULL = legacy default stream).  Calls are
 *     asynchronous on that stream unless stated otherwise.
 *   - Return value: TFCB_OK (0), TFCB_INVALID_ARGUMENT (1; the analogue of TF's InvalidArgument
 *     status), TFCB_CUDA_ERROR (2), TFCB_OUT_OF_MEMORY (3).  A message is available through
 *     tfcb_last_error() (thread local).
 *   - Handles are not thread safe; one consumer per handle, as the reference documents for its
 *     DT_VARIANT handles (tensorflow_compression/cc/ops/range_coder_ops.cc:94-95,190-192).
 *   - There is NO CPU fallback: without a CUDA device every compute entry returns TFCB_CUDA_ERROR.
 */
#ifndef TFCB200_H_
#define TFCB200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define TFCB_OK 0
#define TFCB_INVALID_ARGUMENT 1
#define TFCB_CUDA_ERROR 2
#define TFCB_OUT_OF_MEMORY 3

#define TFCB_ABI_VERSION 1

/* Version of this ABI (TFCB_ABI_VERSION of the library that was loaded). */
int tfcb_abi_version(void);
/* Message of the last failing call on this thread ("" if none). */
const char* tfcb_last_error(void);

/* ------------------------------------------------------------------------------------------------
 * Range ENCODER.  Replaces CreateRangeEncoder / EntropyEncodeChannel / EntropyEncodeIndex /
 * EntropyEncodeFinalize:
 *   op contract   tensorflow_compression/cc/ops/range_coder_ops.cc:28-135
 *   CPU kernels   tensorflow_compression/cc/kernels/range_coder_kernels.cc:168-322,484-592
 *   coder         tensorflow_compression/cc/lib/range_coder.cc:37-307
 * One CTA per code stream (gather / chain / drain warps); streams = prod(handle shape); a stream holds < 2^31
 * 16-bit words (4 GB).
 * ---------------------------------------------------------------------------------------------- */
typedef struct tfcb_encoder tfcb_encoder;

/* `lookup_host`: the reference's `lookup` tensor, int32, either 1-D (lookup_cols == 0: rows
 * concatenated, each [+-precision, 0, c1, ..., 2^precision, (2^precision padding)*]) or 2-D
 * (lookup_cols == row width).  Negative precision enables the overflow (escape + Elias gamma)
 * code for that row.  Validated like ScanCDF / IndexCDFVector / IndexCDFMatrix
 * (range_coder_kernels.cc:110-164); violations -> TFCB_INVALID_ARGUMENT. */
int tfcb_encoder_create(const int32_t* lookup_host, int64_t lookup_len, int64_t lookup_cols,
                        int64_t n_streams, void* stream, tfcb_encoder** out);

/* EntropyEncodeChannel: `value_dev` is int32 [n_streams, n_per_stream] row-major; symbol j of every
 * stream uses lookup row (j mod n_rows), restarting at 0 for each call (range_coder_kernels.cc:
 * 244-267).  May be called repeatedly; the streams keep growing (state persists, :225-226). */
int tfcb_encode_channel(tfcb_encoder* h, const int32_t* value_dev, int64_t n_per_stream, void* stream);

/* EntropyEncodeIndex: `index_dev` has the shape of `value_dev`; row = index (range_coder_kernels.cc:
 * 219-242).  Out-of-range index / value are reported by tfcb_encode_finalize / tfcb_encoder_check as
 * TFCB_INVALID_ARGUMENT ("index=... not in range", "value=... not in range"), mirroring
 * REQUIRE_IN_RANGE (:204-210,231,235,260). */
int tfcb_encode_index(tfcb_encoder* h, const int32_t* index_dev, const int32_t* value_dev,
                      int64_t n_per_stream, void* stream);

/* Fused quantize + EntropyEncodeChannel: the symbol is
 *   int32(rintf(y - quant_offset[c])) - cdf_offset[c],   c = j mod n_rows
 * i.e. ContinuousBatchedEntropyModel.compress without materialising the int32 tensor
 * (tensorflow_compression/python/entropy_models/continuous_batched.py:375-382).
 * `quant_offset_dev` may be NULL (no offset). */
int tfcb_encode_channel_f32(tfcb_encoder* h, const float* y_dev, const float* quant_offset_dev,
                            const int32_t* cdf_offset_dev, int64_t n_per_stream, void* stream);

/* Fused quantize + EntropyEncodeIndex: symbol = int32(rintf(y - loc)) - cdf_offset[index]
 * (continuous_indexed.py:378-385; `loc_dev` may be NULL).  `index_dev` are already-clamped int32
 * table indexes. */
int tfcb_encode_index_f32(tfcb_encoder* h, const int32_t* index_dev, const float* y_dev,
                          const float* loc_dev, const int32_t* cdf_offset_dev, int64_t n_per_stream,
                          void* stream);

/* Synchronises `stream` and reports a pending device-side argument error, if any. */
int tfcb_encoder_check(tfcb_encoder* h, void* stream);

/* EntropyEncodeFinalize: flushes every stream exactly like RangeEncoder::Finalize
 * (range_coder.cc:266-307), packs all strings back to back and returns the total size.  Synchronises
 * `stream`.  After this call only the output accessors and destroy are valid. */
int tfcb_encode_finalize(tfcb_encoder* h, void* stream, int64_t* total_bytes_host);

/* Device views of the result: bytes [total], offsets int64 [n_streams + 1].  Valid until destroy. */
int tfcb_encoder_output(tfcb_encoder* h, const uint8_t** bytes_dev, const int64_t** offsets_dev);
/* Copies the result to host buffers (bytes [total], offsets [n_streams + 1]); synchronises. */
int tfcb_encoder_copy_output(tfcb_encoder* h, uint8_t* bytes_host, int64_t* offsets_host,
                             void* stream);
void tfcb_encoder_destroy(tfcb_encoder* h);

/* ------------------------------------------------------------------------------------------------
 * Range DECODER.  Replaces CreateRangeDecoder / EntropyDecodeChannel / EntropyDecodeIndex /
 * EntropyDecodeFinalize:
 *   op contract   tensorflow_compression/cc/ops/range_coder_ops.cc:137-247
 *   CPU kernels   tensorflow_compression/cc/kernels/range_coder_kernels.cc:334-471,597-700
 *   coder         tensorflow_compression/cc/lib/range_coder.h:79-83,144-169,193-282
 * ---------------------------------------------------------------------------------------------- */
typedef struct tfcb_decoder tfcb_decoder;

/* `bytes_dev` / `offsets_dev` (int64 [n_streams + 1]) describe the encoded strings; the memory is
 * BORROWED and must outlive the handle (the reference also only holds a reference,
 * range_coder_kernels.cc:475-478). */
int tfcb_decoder_create(const uint8_t* bytes_dev, const int64_t* offsets_dev, int64_t n_streams,
                        const int32_t* lookup_host, int64_t lookup_len, int64_t lookup_cols,
                        void* stream, tfcb_decoder** out);
/* EntropyDecodeChannel -> int32 [n_streams, n_per_stream]. */
int tfcb_decode_channel(tfcb_decoder* h, int32_t* out_dev, int64_t n_per_stream, void* stream);
/* EntropyDecodeIndex. */
int tfcb_decode_index(tfcb_decoder* h, const int32_t* index_dev, int32_t* out_dev,
                      int64_t n_per_stream, void* stream);
/* Fused decode + dequantize: out = float(sym + cdf_offset[c]) + quant_offset[c]
 * (continuous_batched.py:416-421); `quant_offset_dev` may be NULL. */
int tfcb_decode_channel_f32(tfcb_decoder* h, float* out_dev, const float* quant_offset_dev,
                            const int32_t* cdf_offset_dev, int64_t n_per_stream, void* stream);
/* Fused decode + dequantize, index mode: out = float(sym + cdf_offset[index]) + loc
 * (continuous_indexed.py:409-416); `loc_dev` may be NULL. */
int tfcb_decode_index_f32(tfcb_decoder* h, const int32_t* index_dev, float* out_dev,
                          const float* loc_dev, const int32_t* cdf_offset_dev, int64_t n_per_stream,
                          void* stream);
/* EntropyDecodeFinalize: ok_host[s] = RangeDecoder::Finalize() of stream s (range_coder.h:144-169).
 * Synchronises; also reports a pending out-of-range index as TFCB_INVALID_ARGUMENT. */
int tfcb_decode_finalize(tfcb_decoder* h, uint8_t* ok_host, void* stream);
void tfcb_decoder_destroy(tfcb_decoder* h);

/* ------------------------------------------------------------------------------------------------
 * Legacy single-stream ops RangeEncode / RangeDecode (int16 data, broadcastable N-D int32 CDF):
 *   op contract   tensorflow_compression/cc/ops/range_coding_ops.cc:30-124
 *   CPU kernels   tensorflow_compression/cc/kernels/range_coding_kernels.cc:60-379
 *   axis merging  tensorflow_compression/cc/kernels/range_coding_kernels_util.cc:34-91
 * Shapes are host arrays; `cdf_rank` must be `rank + 1`.  `debug_level` 1 validates the CDF values
 * and the data range (range_coding_kernels.cc:150-173,249-253).  Both calls synchronise.
 * ---------------------------------------------------------------------------------------------- */
/* Writes at most `out_cap` bytes to `out_host`; *n_bytes_host receives the string length. */
int tfcb_range_encode(const int16_t* data_dev, const int64_t* data_shape_host, int rank,
                      const int32_t* cdf_dev, const int64_t* cdf_shape_host, int cdf_rank,
                      int precision, int debug_level, uint8_t* out_host, int64_t out_cap,
                      int64_t* n_bytes_host, void* stream);
int tfcb_range_decode(const uint8_t* encoded_host, int64_t n_bytes, const int64_t* shape_host,
                      int rank, const int32_t* cdf_dev, const int64_t* cdf_shape_host, int cdf_rank,
                      int precision, int debug_level, int16_t* out_dev, void* stream);

/* ------------------------------------------------------------------------------------------------
 * PmfToQuantizedCdf:
 *   op contract   tensorflow_compression/cc/ops/pmf_to_cdf_ops.cc:28-57
 *   CPU kernel    tensorflow_compression/cc/kernels/pmf_to_cdf_kernels.cc:58-208
 * pmf float32 [rows, n] -> cdf int32 [rows, n + 1].  Exact ties between bins are broken by lowest
 * bin index (the reference uses an unstable std::sort; see DESIGN.md).  Synchronises (it must
 * report non-finite / negative mass as TFCB_INVALID_ARGUMENT, pmf_to_cdf_kernels.cc:77-86).
 * ---------------------------------------------------------------------------------------------- */
int tfcb_pmf_to_quantized_cdf(const float* pmf_dev, int64_t rows, int64_t n, int precision,
                              int32_t* cdf_dev, void* stream);

/* The per-row loop of ContinuousEntropyModelBase._build_tables in one launch
 * (tensorflow_compression/python/entropy_models/continuous_base.py:282-294): for row r take
 * pmf[r, :lens[r]], append the overflow mass max(1 - sum, 0), quantise, and emit
 * [-precision, cdf...] into a 1-D concatenated lookup.  `lens_host` int32 [rows];
 * `lookup_dev` must hold sum(lens[r] + 3) int32.  Synchronises. */
int tfcb_build_lookup(const float* pmf_dev, int64_t rows, int64_t max_len, const int32_t* lens_host,
                      int precision, int32_t* lookup_dev, void* stream);

/* ------------------------------------------------------------------------------------------------
 * RunLengthEncode / RunLengthDecode (and RunLengthGammaEncode/Decode = codes (-1, -1), use_run_length_for_non_zeros 0):
 *   op contract   tensorflow_compression/cc/ops/run_length_ops.cc:28-84
 *   CPU kernels   tensorflow_compression/cc/kernels/run_length_kernels.cc:52-262, bit packing cc/lib/bit_coder.cc:50-191
 * data int32 [n] (flattened) <-> one bit string.  run_length_code / magnitude_code >= 0: Rice code with that parameter,
 * < 0: Elias gamma.  Encode: `code_dev` has room for `capacity` bytes (a multiple of 4 is used); *n_bytes_host receives
 * the length of the code; TFCB_INVALID_ARGUMENT with the needed size in the message (and in *n_bytes_host) when it
 * does not fit.  The encoder is data parallel (scans + atomics); the decoder is serial, as in the reference.
 * Decode errors carry the reference's DataLoss messages.
 * ---------------------------------------------------------------------------------------------- */
int tfcb_run_length_encode(const int32_t* data_dev, int64_t n, int run_length_code, int magnitude_code,
                           int use_run_length_for_non_zeros, uint8_t* code_dev, int64_t capacity,
                           int64_t* n_bytes_host, void* stream);
int tfcb_run_length_decode(const uint8_t* code_dev, int64_t n_bytes, int run_length_code, int magnitude_code,
                           int use_run_length_for_non_zeros, int32_t* data_dev, int64_t n, void* stream);

/* ------------------------------------------------------------------------------------------------
 * StochasticRound:
 *   op contract   tensorflow_compression/cc/ops/quantization_ops.cc:28-53
 *   CPU kernel    tensorflow_compression/cc/kernels/quantization_kernels.cc:48-95
 * outputs[i] = floor(inputs[i] / step_size) + (u_i < frac), u_i the i-th draw of the reference's xoshiro256+
 * stream seeded through std::seed_seq(seed) -- the same integers as the CPU op for the same seed (the
 * sequential stream is entered in parallel through GF(2) jump matrices).  `dtype` 0 float32, 1 float16,
 * 2 bfloat16; `seed_host` int32 [seed_len] in host memory, seed_len == 0 seeds from the clock
 * (quantization_kernels.cc:71-78).
 * ---------------------------------------------------------------------------------------------- */
int tfcb_stochastic_round(const void* inputs_dev, int dtype, int64_t n, float step_size,
                          const int32_t* seed_host, int64_t seed_len, int32_t* outputs_dev, void* stream);

/* ------------------------------------------------------------------------------------------------
 * GDN / IGDN (tensorflow_compression/python/layers/gdn.py:371-421), channels-last:
 *   u = rectify ? relu(x) : x;  p = |u|^alpha;  n_i = beta_i + sum_j p_j gamma[j,i];
 *   y_i = u_i / n_i^eps  (GDN)   or   u_i * n_i^eps  (IGDN)
 * x, y: float32 [n_pix, C] row-major;  gamma float32 [C, C] (row j, column i);  beta float32 [C].
 * alpha in {1, 2} and eps in {1, 0.5} take the reference's fast paths; other values use powf.
 * C in {128, 192} with those alpha / eps (not trainable) and 16-byte aligned activations run on the tensor cores (bf16
 * split with fp32 accumulation: <= 1e-5 relative forward, <= 2e-5 of the largest gradient backward); every other
 * call runs the fp32 kernels.  The aligned pointers are x, y and beta forward, x, dy, dx and (C = 192) the workspace
 * backward; every kernel but the C = 128 forward also needs fewer than 2^31 pixels.  tfcb_gdn_native_16bit states the
 * rule.
 * The reference has no native GDN code (TF graph of abs / conv1x1 / bias_add / div); the backward
 * pass replaces TF autodiff of that graph.
 * ---------------------------------------------------------------------------------------------- */
#define TFCB_GDN_INVERSE 1
#define TFCB_GDN_RECTIFY 2
/* trainable exponents: compute `u ** alpha` / `n ** epsilon` literally even when the current value is 1, 2 or 1/2
 * (gdn.py:380-388,406-411 take the |u| / u^2 / sqrt shortcuts only for fixed exponents) */
#define TFCB_GDN_POW_ALPHA 4
#define TFCB_GDN_POW_EPSILON 8

int tfcb_gdn_forward(const float* x_dev, const float* gamma_dev, const float* beta_dev, float* y_dev,
                     int64_t n_pix, int C, int flags, float alpha, float epsilon, void* stream);

/* Mixed-precision variant (gdn_test.py:200-210: float32 variables, float16 / bfloat16 activations): x and y in
 * 16 bits (dtype 1 float16, 2 bfloat16), arithmetic in float32, y rounded once to nearest even -- 4 bytes of HBM
 * traffic per element instead of 8.  Runs the tensor-core kernels only; TFCB_INVALID_ARGUMENT where they do not take
 * the call (tfcb_gdn_native_16bit returns 0; the caller converts to float32). */
int tfcb_gdn_forward_16bit(const void* x_dev, const float* gamma_dev, const float* beta_dev, void* y_dev,
                           int64_t n_pix, int C, int dtype, int flags, float alpha, float epsilon, void* stream);

/* Gradients for upstream dy: dx [n_pix, C], dgamma [C, C], dbeta [C] (dgamma / dbeta are
 * OVERWRITTEN, reduced over all pixels).  `workspace_dev` must hold
 * tfcb_gdn_backward_workspace_bytes(n_pix, C) bytes. */
int64_t tfcb_gdn_backward_workspace_bytes(int64_t n_pix, int C);
int tfcb_gdn_backward(const float* x_dev, const float* gamma_dev, const float* beta_dev,
                      const float* dy_dev, float* dx_dev, float* dgamma_dev, float* dbeta_dev,
                      void* workspace_dev, int64_t n_pix, int C, int flags, float alpha,
                      float epsilon, void* stream);
/* Mixed-precision backward: x, dy and dx in 16 bits of the same dtype (1 float16, 2 bfloat16); gamma, beta, dgamma,
 * dbeta float32; arithmetic float32, dx rounded once to nearest even -- 6 bytes of HBM traffic per element for x, dy
 * and dx.  Same workspace as tfcb_gdn_backward.  Runs the tensor-core kernels only; TFCB_INVALID_ARGUMENT where they
 * do not take the call (the caller converts to float32).  n_pix == 0 zeroes dgamma and dbeta. */
int tfcb_gdn_backward_16bit(const void* x_dev, const float* gamma_dev, const float* beta_dev, const void* dy_dev,
                            void* dx_dev, float* dgamma_dev, float* dbeta_dev, void* workspace_dev, int64_t n_pix,
                            int C, int dtype, int flags, float alpha, float epsilon, void* stream);
/* 1 where tfcb_gdn_forward_16bit (backward = 0) or tfcb_gdn_backward_16bit (backward = 1) has a kernel for the call,
 * 0 otherwise, including n_pix == 0.  Host only: reads none of the pointers, only their alignment.  The forward looks
 * at x and beta, the backward at x and dy; y, dx and the workspace are taken to be 16-byte aligned, as fresh
 * allocations are. */
int tfcb_gdn_native_16bit(int backward, const void* x_dev, const void* beta_dev, const void* dy_dev, int64_t n_pix,
                          int C, int dtype, int flags, float alpha, float epsilon);

/* Number of kernel launches issued by this library since load (bench.py's `gpu_launches`). */
/* Gradients of the loss with respect to the scalar exponents alpha and epsilon (gdn.py:345-367 makes them
 * trainable GDNParameters; TF autodiff differentiates through pow): dalpha_depsilon_dev float32 [2].
 * workspace_dev: tfcb_gdn_exponent_grads_workspace_bytes() bytes. */
int64_t tfcb_gdn_exponent_grads_workspace_bytes(void);
int tfcb_gdn_exponent_grads(const float* x_dev, const float* gamma_dev, const float* beta_dev,
                            const float* dy_dev, float* dalpha_depsilon_dev, void* workspace_dev,
                            int64_t n_pix, int C, int flags, float alpha, float epsilon, void* stream);

int64_t tfcb_launch_count(void);

#ifdef __cplusplus
}
#endif
#endif /* TFCB200_H_ */

/*
 * dietgpu_b200.h -- C ABI of the B200-native batched rANS + float codec.
 *
 * This is the drop-in boundary for DietGPU's codec hot path.  The reference
 * (facebookresearch/dietgpu) has no C ABI of its own: its public surface is
 * the C++ API in dietgpu/ans/GpuANSCodec.h and dietgpu/float/GpuFloatCodec.h
 * plus torch.ops.dietgpu.* (dietgpu/DietGpu.cpp).  Each entry point below
 * names the reference C++ function it replaces (file:line relative to
 * /root/reference/dietgpu/); include/dietgpu_b200_compat.hpp re-creates those
 * exact C++ signatures on top of this ABI and INTEGRATION.md shows the
 * binding a maintainer would add.
 *
 * Conventions (all entry points):
 *   - plain pointers and sizes only; no C++ or torch types;
 *   - "host array" = an array in host memory, consumed before the call
 *     returns; "_dev" = device memory; `stream` is a cudaStream_t passed as
 *     void* (NULL = the legacy default stream);
 *   - all device work is enqueued on `stream`; calls are asynchronous unless
 *     a checksum has to be verified (decode with use_checksum != 0);
 *   - temp_dev/temp_bytes: caller-owned device scratch, 256 B aligned, at
 *     least dgb_*_temp_bytes(...) bytes; it may be reused by the next call on
 *     the same stream.  The library allocates nothing (no cudaMalloc);
 *   - compressed buffers must be 16 B aligned (as in the reference,
 *     ans/GpuANSEncode.cu:19-21); raw ANS inputs 4 B aligned
 *     (ans/GpuANSCodec.h:16); float data aligned to its word size;
 *   - return value: DGB_OK or a DGB_ERR_* code; never aborts, never throws.
 *     There is NO CPU fallback: without a usable CUDA device the calls fail
 *     with DGB_ERR_CUDA.
 *   - wire format: identical to the reference's (ans/GpuANSUtils.cuh:67-227,
 *     float/GpuFloatUtils.cuh:26-74); archives are interchangeable in both
 *     directions.  Bits the reference leaves undefined are written as zero.
 */
#ifndef DIETGPU_B200_H_
#define DIETGPU_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DGB_OK 0
#define DGB_ERR_INVALID_ARG 1     /* bad prob_bits / float type / alignment / NULL */
#define DGB_ERR_TEMP_TOO_SMALL 2  /* temp_bytes < dgb_*_temp_bytes(...) */
#define DGB_ERR_CUDA 3            /* a CUDA runtime call failed (see dgb_last_cuda_error) */
#define DGB_ERR_CHECKSUM 4        /* decode: stored checksum != recomputed checksum */
#define DGB_ERR_TOO_LARGE 5       /* a size exceeds the format's 32-bit limits */

/* float/GpuFloatCodec.h:18-23 FloatType */
#define DGB_FLOAT16 1
#define DGB_BFLOAT16 2
#define DGB_FLOAT32 3

/* ans/GpuANSCodec.h:16,20 */
#define DGB_ANS_REQUIRED_ALIGNMENT 4
#define DGB_ANS_DEFAULT_PROB_BITS 10

int dgb_version(void);
const char* dgb_error_string(int code);
/* cudaError_t of the most recent DGB_ERR_CUDA on this thread (0 if none). */
int dgb_last_cuda_error(void);

/* ---- size bounds -------------------------------------------------------- */

/* ans/GpuANSEncode.cu:13-25 getMaxCompressedSize (same value, same quirk). */
uint32_t dgb_ans_max_compressed_size(uint32_t uncompressed_bytes);
/* float/GpuFloatCompress.cu:23-45 getMaxFloatCompressedSize. */
uint32_t dgb_float_max_compressed_size(int float_type, uint32_t num_floats);

/* ---- scratch sizing (new; the reference sizes scratch implicitly through
 *      StackDeviceMemory and falls back to cudaMalloc) ---------------------- */
size_t dgb_ans_encode_temp_bytes(uint32_t num_in_batch, uint32_t max_uncompressed_bytes);
size_t dgb_ans_decode_temp_bytes(uint32_t num_in_batch);
size_t dgb_float_compress_temp_bytes(int float_type, uint32_t num_in_batch, uint32_t max_num_floats);
size_t dgb_float_decompress_temp_bytes(int float_type, uint32_t num_in_batch, uint32_t max_num_floats);

/* ---- byte rANS encode --------------------------------------------------- */

/* ans/GpuANSCodec.h:100-128 / ans/GpuANSEncode.cu:55-113 ansEncodeBatchPointer.
 * in/out: host arrays of num_in_batch device pointers; in_size: host array of
 * byte counts; out[i] must hold dgb_ans_max_compressed_size(in_size[i]) bytes.
 * histogram_dev: optional device [num_in_batch][256] u32 pre-computed counts.
 * out_size_dev: optional device u32[num_in_batch], receives archive sizes. */
int dgb_ans_encode_pointer(void* temp_dev, size_t temp_bytes, int prob_bits, int use_checksum,
                           uint32_t num_in_batch, const void* const* in, const uint32_t* in_size,
                           const uint32_t* histogram_dev, void* const* out,
                           uint32_t* out_size_dev, void* stream);

/* ans/GpuANSCodec.h:65-98 / ans/GpuANSEncode.cu:27-53 ansEncodeBatchStride. */
int dgb_ans_encode_stride(void* temp_dev, size_t temp_bytes, int prob_bits, int use_checksum,
                          uint32_t num_in_batch, const void* in_dev, uint32_t in_per_batch_size,
                          uint32_t in_per_batch_stride, const uint32_t* histogram_dev,
                          void* out_dev, uint32_t out_per_batch_stride,
                          uint32_t* out_size_dev, void* stream);

/* ans/GpuANSCodec.h:130-164 / ans/GpuANSEncode.cu:115-179 ansEncodeBatchSplitSize.
 * in_split_sizes: host array; member i starts at sum_{j<i} in_split_sizes[j];
 * interior sizes must be multiples of 4. */
int dgb_ans_encode_split_size(void* temp_dev, size_t temp_bytes, int prob_bits, int use_checksum,
                              uint32_t num_in_batch, const void* in_dev,
                              const uint32_t* in_split_sizes, const uint32_t* histogram_dev,
                              void* out_dev, uint32_t out_stride, uint32_t* out_size_dev,
                              void* stream);

/* ---- byte rANS decode --------------------------------------------------- */

/* ans/GpuANSCodec.h:228-263 / ans/GpuANSDecode.cu:47-120 ansDecodeBatchPointer.
 * out_capacity: host array (bytes).  out_success_dev (u8[n]) / out_size_dev
 * (u32[n]): optional device arrays; a member whose capacity is too small, or
 * whose header is not a valid archive of `prob_bits`, gets success=0 and is
 * skipped (size = required bytes, or 0 for an invalid header).
 * With use_checksum != 0 the call synchronises `stream`, compares checksums
 * and returns DGB_ERR_CHECKSUM on mismatch; checksum_mismatch_host (optional
 * host u8[n]) then flags the failing members. */
int dgb_ans_decode_pointer(void* temp_dev, size_t temp_bytes, int prob_bits, int use_checksum,
                           uint32_t num_in_batch, const void* const* in, void* const* out,
                           const uint32_t* out_capacity, uint8_t* out_success_dev,
                           uint32_t* out_size_dev, uint8_t* checksum_mismatch_host, void* stream);

/* ans/GpuANSCodec.h:170-226 / ans/GpuANSDecode.cu:20-45 ansDecodeBatchStride. */
int dgb_ans_decode_stride(void* temp_dev, size_t temp_bytes, int prob_bits, int use_checksum,
                          uint32_t num_in_batch, const void* in_dev, uint32_t in_per_batch_stride,
                          void* out_dev, uint32_t out_per_batch_stride,
                          uint32_t out_per_batch_capacity, uint8_t* out_success_dev,
                          uint32_t* out_size_dev, uint8_t* checksum_mismatch_host, void* stream);

/* ans/GpuANSCodec.h:265-303 / ans/GpuANSDecode.cu:122-193 ansDecodeBatchSplitSize. */
int dgb_ans_decode_split_size(void* temp_dev, size_t temp_bytes, int prob_bits, int use_checksum,
                              uint32_t num_in_batch, const void* const* in, void* out_dev,
                              const uint32_t* out_split_sizes, uint8_t* out_success_dev,
                              uint32_t* out_size_dev, uint8_t* checksum_mismatch_host,
                              void* stream);

/* ans/GpuANSCodec.h:309-341 / ans/GpuANSInfo.cu:14-49 ansGetCompressedInfo{,Device}.
 * out_sizes_dev receives each archive's UNCOMPRESSED size in bytes (what the
 * reference kernel reports, ans/GpuANSInfo.cuh:27-29), 0 for a bad header.
 * in_is_device_array != 0: `in` is a device array of device pointers. */
int dgb_ans_get_compressed_info(void* temp_dev, size_t temp_bytes, const void* const* in,
                                int in_is_device_array, uint32_t num_in_batch,
                                uint32_t* out_sizes_dev, uint32_t* out_checksum_dev, void* stream);

/* ---- float codec (fp16 / bf16 / fp32) ------------------------------------ */

/* float/GpuFloatCodec.h:103-139 / float/GpuFloatCompress.cu:47-101 floatCompress.
 * in_size counts float WORDS.  out[i] must hold
 * dgb_float_max_compressed_size(float_type, in_size[i]) bytes. */
int dgb_float_compress_pointer(void* temp_dev, size_t temp_bytes, int float_type, int prob_bits,
                               int use_checksum, uint32_t num_in_batch, const void* const* in,
                               const uint32_t* in_size, void* const* out, uint32_t* out_size_dev,
                               void* stream);

/* float/GpuFloatCodec.h:141-170 / float/GpuFloatCompress.cu:103-159 floatCompressSplitSize. */
int dgb_float_compress_split_size(void* temp_dev, size_t temp_bytes, int float_type, int prob_bits,
                                  int use_checksum, uint32_t num_in_batch, const void* in_dev,
                                  const uint32_t* in_split_sizes, void* out_dev,
                                  uint32_t out_stride, uint32_t* out_size_dev, void* stream);

/* float/GpuFloatCodec.h:176-208 / float/GpuFloatDecompress.cu:22-115 floatDecompress.
 * out_capacity / out_size_dev are in float WORDS.  The reference's
 * is16ByteAligned switch is not needed: one fused decode+join kernel handles
 * any word-aligned output. */
int dgb_float_decompress_pointer(void* temp_dev, size_t temp_bytes, int float_type, int prob_bits,
                                 int use_checksum, uint32_t num_in_batch, const void* const* in,
                                 void* const* out, const uint32_t* out_capacity,
                                 uint8_t* out_success_dev, uint32_t* out_size_dev,
                                 uint8_t* checksum_mismatch_host, void* stream);

/* float/GpuFloatCodec.h:210-246 / float/GpuFloatDecompress.cu:117-179 floatDecompressSplitSize. */
int dgb_float_decompress_split_size(void* temp_dev, size_t temp_bytes, int float_type,
                                    int prob_bits, int use_checksum, uint32_t num_in_batch,
                                    const void* const* in, void* out_dev,
                                    const uint32_t* out_split_sizes, uint8_t* out_success_dev,
                                    uint32_t* out_size_dev, uint8_t* checksum_mismatch_host,
                                    void* stream);

/* float/GpuFloatCodec.h:252-292 / float/GpuFloatInfo.cu:17-64 floatGetCompressedInfo{,Device}. */
int dgb_float_get_compressed_info(void* temp_dev, size_t temp_bytes, const void* const* in,
                                  int in_is_device_array, uint32_t num_in_batch,
                                  uint32_t* out_sizes_dev, uint32_t* out_types_dev,
                                  uint32_t* out_checksum_dev, void* stream);

/* ---- host front end helpers (new) ----------------------------------------- */
/* Plain asynchronous copies on `stream`, used by the host-buffer front end (dietgpu_b200.HostCodec)
 * to move whole member groups in one DMA each instead of one call per member.  dgb_copy_async is
 * cudaMemcpyAsync(cudaMemcpyDefault); dgb_copy_rows_async copies `rows` rows of `width_bytes` between
 * two pitched matrices (cudaMemcpy2DAsync), e.g. archives [n, cols] device <-> pinned host. */
int dgb_copy_async(void* dst, const void* src, size_t bytes, void* stream);
int dgb_copy_rows_async(void* dst, size_t dst_pitch, const void* src, size_t src_pitch,
                        size_t width_bytes, size_t rows, void* stream);

/* ---- archive mover (new; for the compressed collectives) -------------------- */
/* Copies num_in_batch archives from src[i] to dst[i] (host arrays of device pointers, 16 B aligned), each
 * exactly as long as its own header says and at most dst_capacity[i] bytes: float_type 0 = ANS archives
 * (ans/GpuANSUtils.cuh:67-227 header), DGB_FLOAT16/BFLOAT16/FLOAT32 = float archives
 * (float/GpuFloatUtils.cuh:26-74).  src may be memory of a peer GPU mapped into this process (NVLink):
 * sizes are read on the device, nothing travels to the host; out_bytes_dev (optional, device, [n]) receives
 * the archive sizes.  An archive with a bad header is copied as its first 32 bytes so that the decoder
 * which follows reports it.  The reference has no counterpart (it names the use, README.md:72,103-104). */
int dgb_archives_pull(int float_type, uint32_t num_in_batch, const void* const* src, void* const* dst,
                      const uint32_t* dst_capacity, uint32_t* out_bytes_dev, void* stream);

/* ---- tuning knob (benchmarks / tests only) ------------------------------- */
/* Selects an internal kernel variant by name ("parts", "encode_canonical", "decode_warps" ...; the list
 * is in INTEGRATION.md section 4).  Unknown names return DGB_ERR_INVALID_ARG.  Defaults are the tuned choice. */
int dgb_set_option(const char* name, int value);
int dgb_get_option(const char* name, int* value);
/* Per-thread override: the first call copies the process-wide set into a copy that only codec calls made by
 * THIS thread see (and dgb_get_option on this thread reports); dgb_clear_thread_options drops the copy.  Every
 * codec call snapshots its effective set at entry, so changing options never affects a call in flight. */
int dgb_set_thread_option(const char* name, int value);
int dgb_clear_thread_options(void);
/* With option "timing" = 1 every kernel launch is bracketed by CUDA events on the caller's
 * stream; this returns (and resets) the summed durations in ms and launch counts per kernel:
 * slot 0 stats (K1), 1 encode (K2), 2 retired (always 0), 3 decode, 4 checksum, 5 retired (always 0), 6 archive mover.
 * Synchronises the device. */
int dgb_kernel_times(float* ms, int* counts, int nslots);

#ifdef __cplusplus
}
#endif
#endif /* DIETGPU_B200_H_ */

// ref_harness.cu -- TEST INFRASTRUCTURE ONLY (written for this repo).
// A C-ABI veneer over the UNMODIFIED reference library so Python (ctypes) can
// drive the reference's own CUDA path: as the GPU-side parity oracle
// (tests/golden/make_ref_golden.py) and as the `--impl reference` arm of
// bench.py.  It is compiled together with the reference sources, where they
// lie under /root/reference, by build_ref.sh into oracle/_ref/ (git-ignored).
// No reference source is copied into this repository.
#include <cuda_runtime.h>
#include <cassert>
#include <cstdint>
#include <string>
#include <vector>
#include "dietgpu/ans/GpuANSCodec.h"
#include "dietgpu/float/GpuFloatCodec.h"
#include "dietgpu/utils/StackDeviceMemory.h"

using namespace dietgpu;

namespace {
StackDeviceMemory makeRes(void* temp, size_t bytes) {
  int dev = 0;
  cudaGetDevice(&dev);
  return StackDeviceMemory(dev, temp, bytes);
}
} // namespace

extern "C" {

uint32_t ref_ans_max_compressed_size(uint32_t bytes) {
  return getMaxCompressedSize(bytes);
}

uint32_t ref_float_max_compressed_size(int ft, uint32_t n) {
  return getMaxFloatCompressedSize(FloatType(ft), n);
}

int ref_ans_encode_pointer(void* temp, size_t tempBytes, int pb, int checksum,
                           uint32_t n, const void** in, const uint32_t* inSize,
                           void** out, uint32_t* outSize_dev, void* stream) {
  auto res = makeRes(temp, tempBytes);
  ansEncodeBatchPointer(res, ANSCodecConfig(pb, checksum != 0), n, in, inSize,
                        nullptr, out, outSize_dev, (cudaStream_t)stream);
  return 0;
}

int ref_ans_decode_pointer(void* temp, size_t tempBytes, int pb, int checksum,
                           uint32_t n, const void** in, void** out,
                           const uint32_t* outCapacity, uint8_t* outSuccess_dev,
                           uint32_t* outSize_dev, void* stream) {
  auto res = makeRes(temp, tempBytes);
  auto st = ansDecodeBatchPointer(res, ANSCodecConfig(pb, checksum != 0), n, in,
                                  out, outCapacity, outSuccess_dev, outSize_dev,
                                  (cudaStream_t)stream);
  return st.error == ANSDecodeError::None ? 0 : 1;
}

int ref_float_compress(void* temp, size_t tempBytes, int ft, int pb,
                       int checksum, uint32_t n, const void** in,
                       const uint32_t* inSize, void** out,
                       uint32_t* outSize_dev, void* stream) {
  auto res = makeRes(temp, tempBytes);
  FloatCompressConfig cfg(FloatType(ft), ANSCodecConfig(pb, false), false,
                          checksum != 0);
  floatCompress(res, cfg, n, in, inSize, out, outSize_dev, (cudaStream_t)stream);
  return 0;
}

int ref_float_decompress(void* temp, size_t tempBytes, int ft, int pb,
                         int checksum, int aligned16, uint32_t n,
                         const void** in, void** out,
                         const uint32_t* outCapacity, uint8_t* outSuccess_dev,
                         uint32_t* outSize_dev, void* stream) {
  auto res = makeRes(temp, tempBytes);
  FloatDecompressConfig cfg(FloatType(ft), ANSCodecConfig(pb, false),
                            aligned16 != 0, checksum != 0);
  auto st = floatDecompress(res, cfg, n, in, out, outCapacity, outSuccess_dev,
                            outSize_dev, (cudaStream_t)stream);
  return st.error == FloatDecompressError::None ? 0 : 1;
}

} // extern "C"

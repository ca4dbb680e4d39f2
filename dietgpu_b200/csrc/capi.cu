// capi.cu -- the extern "C" boundary declared in include/dietgpu_b200.h.
// Maps the reference's three batch-addressing forms (pointer / stride / split
// size; ans/BatchProvider.cuh) onto one internal member list, so every kernel
// sees a single descriptor table uploaded in one copy.
#include <algorithm>
#include <atomic>
#include <cstring>
#include <mutex>
#include <string>
#include <vector>

#include "common.cuh"

namespace dgb {

// Tuning options: one process-wide set (dgb_set_option) and an optional per-thread copy that overrides it
// (dgb_set_thread_option), so threads that drive different streams can run different variants without racing;
// every codec call snapshots the effective set at entry.
static Options gOptions;
static thread_local Options tlsOptions;
static thread_local bool tlsHasOptions = false;
Options& options() { return tlsHasOptions ? tlsOptions : gOptions; }

static thread_local cudaError_t tlsLastCuda = cudaSuccess;
void setLastCudaError(cudaError_t e) { tlsLastCuda = e; }

// ---- per-kernel timing -------------------------------------------------------
namespace {
struct TimedLaunch { int slot; cudaEvent_t a, b; };
std::vector<TimedLaunch>& timedLaunches() { static std::vector<TimedLaunch> v; return v; }
std::vector<cudaEvent_t>& eventPool() { static std::vector<cudaEvent_t> v; return v; }
std::mutex& timerMutex() { static std::mutex m; return m; }  // guards the two vectors above (calls may come from several host threads)
cudaEvent_t takeEvent() {
  {
    std::lock_guard<std::mutex> lock(timerMutex());
    auto& pool = eventPool();
    if (!pool.empty()) { cudaEvent_t e = pool.back(); pool.pop_back(); return e; }
  }
  cudaEvent_t e = nullptr;
  cudaEventCreate(&e);
  return e;
}
thread_local TimedLaunch tlsOpen[kNumSlots];
}  // namespace

// One pool per (host thread, device): the fork/join events of a call must not be shared with a call
// that another thread, or the same thread on another device, makes at the same time.
int streamPool(StreamPool** out) {
  constexpr int kMaxDevices = 64;
  struct Slot {
    StreamPool pool;
    bool ready = false;
  };
  static thread_local Slot slots[kMaxDevices];
  int dev = 0;
  DGB_CUDA_TRY(cudaGetDevice(&dev));
  if (dev < 0 || dev >= kMaxDevices) return DGB_ERR_INVALID_ARG;
  Slot& sl = slots[dev];
  if (!sl.ready) {
    // all or nothing: a partly created pool is torn down again, so a later call can retry cleanly
    StreamPool p{};
    bool ok = cudaEventCreateWithFlags(&p.start, cudaEventDisableTiming) == cudaSuccess;
    for (int i = 0; ok && i < kMaxParts; ++i) {
      ok = cudaStreamCreateWithFlags(&p.s[i], cudaStreamNonBlocking) == cudaSuccess &&
           cudaEventCreateWithFlags(&p.done[i], cudaEventDisableTiming) == cudaSuccess;
    }
    if (!ok) {
      setLastCudaError(cudaGetLastError());
      if (p.start) cudaEventDestroy(p.start);
      for (int i = 0; i < kMaxParts; ++i) {
        if (p.s[i]) cudaStreamDestroy(p.s[i]);
        if (p.done[i]) cudaEventDestroy(p.done[i]);
      }
      return DGB_ERR_CUDA;
    }
    sl.pool = p;
    sl.ready = true;
  }
  *out = &sl.pool;
  return DGB_OK;
}

void splitParts(const uint64_t* weight, uint32_t n, int parts, uint32_t* bounds) {
  uint64_t total = 0;
  for (uint32_t i = 0; i < n; ++i) total += weight[i];
  bounds[0] = 0;
  uint64_t acc = 0;
  uint32_t idx = 0;
  const uint64_t eq = total / (uint64_t)parts;
  for (int p = 1; p < parts; ++p) {
    const uint64_t target = eq * (uint64_t)p;
    const uint32_t mustLeave = (uint32_t)(parts - p);  // one member for every later part
    while (idx + mustLeave < n && (idx < bounds[p - 1] + 1 || acc + weight[idx] / 2 <= target)) acc += weight[idx++];
    bounds[p] = idx;
  }
  bounds[parts] = n;
}

int autoParts(int kind, uint32_t n, uint64_t totalBytes) {
  const Options& o = options();
  if (o.timing) return 1;  // per-kernel timing wants un-overlapped launches
  int p = o.parts;
  // measured on B200 (tools/walltime.py, 256 MiB batches): float encode is best with 4 sub-batches
  // (the bandwidth-bound statistics kernel of one sub-batch runs beside the issue-bound coder of the
  // previous one: c3 204 / 195 / 189 us for 1 / 2 / 4); byte inputs gain nothing
  if (p <= 0) {
    const bool big = kind != kKindBytes && totalBytes >= (64ull << 20);
    p = !big ? 1 : (n >= 16 ? 4 : (n >= 8 ? 2 : 1));
  }
  p = std::min(p, kMaxParts);
  return (int)std::max<uint32_t>(1, std::min<uint32_t>((uint32_t)p, n));
}

// kernels launched by this library since load (every codec launch site calls timerBegin first)
static std::atomic<int> gLaunches{0};

void timerBegin(int slot, cudaStream_t stream) {
  gLaunches.fetch_add(1, std::memory_order_relaxed);
  if (!options().timing) return;
  TimedLaunch t{slot, takeEvent(), takeEvent()};
  cudaEventRecord(t.a, stream);
  tlsOpen[slot] = t;
}
void timerEnd(int slot, cudaStream_t stream) {
  if (!options().timing) return;
  cudaEventRecord(tlsOpen[slot].b, stream);
  std::lock_guard<std::mutex> lock(timerMutex());
  timedLaunches().push_back(tlsOpen[slot]);
}

namespace {

bool validFloatType(int ft) { return ft == DGB_FLOAT16 || ft == DGB_BFLOAT16 || ft == DGB_FLOAT32; }
uint32_t wordBytes(int kind) { return kind == kKindF32 ? 4u : (kind == kKindBytes ? 1u : 2u); }

// pointer form
int buildPointer(uint32_t n, const void* const* in, const uint32_t* size, void* const* out,
                 std::vector<HostMember>& v) {
  if (n && (!in || !size || !out)) return DGB_ERR_INVALID_ARG;
  v.resize(n);
  for (uint32_t i = 0; i < n; ++i) v[i] = HostMember{in[i], out[i], size[i]};
  return DGB_OK;
}

}  // namespace
}  // namespace dgb

using namespace dgb;

extern "C" {

int dgb_version(void) { return 1; }

const char* dgb_error_string(int code) {
  switch (code) {
    case DGB_OK: return "ok";
    case DGB_ERR_INVALID_ARG: return "invalid argument";
    case DGB_ERR_TEMP_TOO_SMALL: return "temporary device memory too small";
    case DGB_ERR_CUDA: return "CUDA runtime error";
    case DGB_ERR_CHECKSUM: return "checksum mismatch";
    case DGB_ERR_TOO_LARGE: return "size exceeds format limits";
    default: return "unknown error";
  }
}

int dgb_last_cuda_error(void) { return (int)tlsLastCuda; }

uint32_t dgb_ans_max_compressed_size(uint32_t bytes) {
  // ans/GpuANSEncode.cu:13-25 (the header overhead is charged for a constant 4096 blocks)
  // The reference CHECKs rawSize <= INT32_MAX (process abort); this ABI returns 0 = "too large"
  // instead of a wrapped value a caller would size its output buffer from.
  uint64_t raw = ansOverhead(kBlockBytes);
  raw += (uint64_t)roundUp(kBlockBytes + kBlockBytes / 4u, 16u) * (((uint64_t)bytes + kBlockBytes - 1) / kBlockBytes);
  raw = roundUp64(raw, 16);
  return raw <= 0x7fffffffull ? (uint32_t)raw : 0u;
}

uint32_t dgb_float_max_compressed_size(int ft, uint32_t n) {
  if (!validFloatType(ft)) return 0;
  const uint32_t ans = dgb_ans_max_compressed_size(n);
  if (ans == 0u) return 0u;  // too large (see above)
  const uint64_t non = ft == DGB_FLOAT32 ? 2ull * roundUp64(n, 8) + roundUp64(n, 16) : roundUp64(n, 16);
  const uint64_t total = (uint64_t)kFloatHeaderBytes + ans + non;
  return total <= 0xffffffffull ? (uint32_t)total : 0u;
}

size_t dgb_ans_encode_temp_bytes(uint32_t n, uint32_t maxBytes) {
  return encodeTempBytes(kKindBytes, n, maxBytes);
}
size_t dgb_ans_decode_temp_bytes(uint32_t n) { return decodeTempBytes(kKindBytes, n); }
size_t dgb_float_compress_temp_bytes(int ft, uint32_t n, uint32_t maxFloats) {
  return validFloatType(ft) ? encodeTempBytes(ft, n, maxFloats) : 0;
}
size_t dgb_float_decompress_temp_bytes(int ft, uint32_t n, uint32_t /*maxFloats*/) {
  return validFloatType(ft) ? decodeTempBytes(ft, n) : 0;
}

// ---- encode ----------------------------------------------------------------

int dgb_ans_encode_pointer(void* temp, size_t tempBytes, int pb, int useChecksum, uint32_t n,
                           const void* const* in, const uint32_t* inSize,
                           const uint32_t* histogram_dev, void* const* out, uint32_t* outSize_dev,
                           void* stream) {
  std::vector<HostMember> v;
  int rc = buildPointer(n, in, inSize, out, v);
  if (rc) return rc;
  return encodeBatch(kKindBytes, temp, tempBytes, pb, useChecksum != 0, n, v.data(), histogram_dev,
                     outSize_dev, (cudaStream_t)stream);
}

int dgb_ans_encode_stride(void* temp, size_t tempBytes, int pb, int useChecksum, uint32_t n,
                          const void* in_dev, uint32_t inSize, uint32_t inStride,
                          const uint32_t* histogram_dev, void* out_dev, uint32_t outStride,
                          uint32_t* outSize_dev, void* stream) {
  if (n && (!out_dev || (inSize && !in_dev))) return DGB_ERR_INVALID_ARG;
  std::vector<HostMember> v(n);
  for (uint32_t i = 0; i < n; ++i)
    v[i] = HostMember{static_cast<const uint8_t*>(in_dev) + (size_t)i * inStride,
                      static_cast<uint8_t*>(out_dev) + (size_t)i * outStride, inSize};
  return encodeBatch(kKindBytes, temp, tempBytes, pb, useChecksum != 0, n, v.data(), histogram_dev,
                     outSize_dev, (cudaStream_t)stream);
}

int dgb_ans_encode_split_size(void* temp, size_t tempBytes, int pb, int useChecksum, uint32_t n,
                              const void* in_dev, const uint32_t* splitSizes,
                              const uint32_t* histogram_dev, void* out_dev, uint32_t outStride,
                              uint32_t* outSize_dev, void* stream) {
  if (n && (!splitSizes || !out_dev)) return DGB_ERR_INVALID_ARG;
  std::vector<HostMember> v(n);
  size_t off = 0;
  for (uint32_t i = 0; i < n; ++i) {
    // ans/GpuANSEncode.cu:132-140: interior splits must keep 4 B alignment
    if (i + 1 != n && (splitSizes[i] % DGB_ANS_REQUIRED_ALIGNMENT)) return DGB_ERR_INVALID_ARG;
    v[i] = HostMember{static_cast<const uint8_t*>(in_dev) + off,
                      static_cast<uint8_t*>(out_dev) + (size_t)i * outStride, splitSizes[i]};
    off += splitSizes[i];
  }
  return encodeBatch(kKindBytes, temp, tempBytes, pb, useChecksum != 0, n, v.data(), histogram_dev,
                     outSize_dev, (cudaStream_t)stream);
}

int dgb_float_compress_pointer(void* temp, size_t tempBytes, int ft, int pb, int useChecksum,
                               uint32_t n, const void* const* in, const uint32_t* inSize,
                               void* const* out, uint32_t* outSize_dev, void* stream) {
  if (!validFloatType(ft)) return DGB_ERR_INVALID_ARG;
  std::vector<HostMember> v;
  int rc = buildPointer(n, in, inSize, out, v);
  if (rc) return rc;
  return encodeBatch(ft, temp, tempBytes, pb, useChecksum != 0, n, v.data(), nullptr, outSize_dev,
                     (cudaStream_t)stream);
}

int dgb_float_compress_split_size(void* temp, size_t tempBytes, int ft, int pb, int useChecksum,
                                  uint32_t n, const void* in_dev, const uint32_t* splitSizes,
                                  void* out_dev, uint32_t outStride, uint32_t* outSize_dev,
                                  void* stream) {
  if (!validFloatType(ft)) return DGB_ERR_INVALID_ARG;
  if (n && (!splitSizes || !out_dev)) return DGB_ERR_INVALID_ARG;
  std::vector<HostMember> v(n);
  size_t off = 0;
  for (uint32_t i = 0; i < n; ++i) {
    v[i] = HostMember{static_cast<const uint8_t*>(in_dev) + off * wordBytes(ft),
                      static_cast<uint8_t*>(out_dev) + (size_t)i * outStride, splitSizes[i]};
    off += splitSizes[i];
  }
  return encodeBatch(ft, temp, tempBytes, pb, useChecksum != 0, n, v.data(), nullptr, outSize_dev,
                     (cudaStream_t)stream);
}

// ---- decode ----------------------------------------------------------------

static int decodePointerCommon(int kind, void* temp, size_t tempBytes, int pb, int useChecksum,
                               uint32_t n, const void* const* in, void* const* out,
                               const uint32_t* cap, uint8_t* outSuccess_dev, uint32_t* outSize_dev,
                               uint8_t* mismatchHost, void* stream) {
  if (n && (!in || !out || !cap)) return DGB_ERR_INVALID_ARG;
  std::vector<HostMember> v(n);
  for (uint32_t i = 0; i < n; ++i) v[i] = HostMember{in[i], out[i], cap[i]};
  return decodeBatch(kind, temp, tempBytes, pb, useChecksum != 0, n, v.data(), outSuccess_dev,
                     outSize_dev, mismatchHost, (cudaStream_t)stream);
}

static int decodeSplitCommon(int kind, void* temp, size_t tempBytes, int pb, int useChecksum,
                             uint32_t n, const void* const* in, void* out_dev,
                             const uint32_t* splitSizes, uint8_t* outSuccess_dev,
                             uint32_t* outSize_dev, uint8_t* mismatchHost, void* stream) {
  if (n && (!in || !splitSizes)) return DGB_ERR_INVALID_ARG;
  std::vector<HostMember> v(n);
  size_t off = 0;
  for (uint32_t i = 0; i < n; ++i) {
    v[i] = HostMember{in[i], static_cast<uint8_t*>(out_dev) + off * wordBytes(kind), splitSizes[i]};
    off += splitSizes[i];
  }
  return decodeBatch(kind, temp, tempBytes, pb, useChecksum != 0, n, v.data(), outSuccess_dev,
                     outSize_dev, mismatchHost, (cudaStream_t)stream);
}

int dgb_ans_decode_pointer(void* temp, size_t tempBytes, int pb, int useChecksum, uint32_t n,
                           const void* const* in, void* const* out, const uint32_t* cap,
                           uint8_t* outSuccess_dev, uint32_t* outSize_dev, uint8_t* mismatchHost,
                           void* stream) {
  return decodePointerCommon(kKindBytes, temp, tempBytes, pb, useChecksum, n, in, out, cap,
                             outSuccess_dev, outSize_dev, mismatchHost, stream);
}

int dgb_ans_decode_stride(void* temp, size_t tempBytes, int pb, int useChecksum, uint32_t n,
                          const void* in_dev, uint32_t inStride, void* out_dev, uint32_t outStride,
                          uint32_t outCapacity, uint8_t* outSuccess_dev, uint32_t* outSize_dev,
                          uint8_t* mismatchHost, void* stream) {
  if (n && !in_dev) return DGB_ERR_INVALID_ARG;
  std::vector<HostMember> v(n);
  for (uint32_t i = 0; i < n; ++i)
    v[i] = HostMember{static_cast<const uint8_t*>(in_dev) + (size_t)i * inStride,
                      static_cast<uint8_t*>(out_dev) + (size_t)i * outStride, outCapacity};
  return decodeBatch(kKindBytes, temp, tempBytes, pb, useChecksum != 0, n, v.data(), outSuccess_dev,
                     outSize_dev, mismatchHost, (cudaStream_t)stream);
}

int dgb_ans_decode_split_size(void* temp, size_t tempBytes, int pb, int useChecksum, uint32_t n,
                              const void* const* in, void* out_dev, const uint32_t* splitSizes,
                              uint8_t* outSuccess_dev, uint32_t* outSize_dev, uint8_t* mismatchHost,
                              void* stream) {
  return decodeSplitCommon(kKindBytes, temp, tempBytes, pb, useChecksum, n, in, out_dev, splitSizes,
                           outSuccess_dev, outSize_dev, mismatchHost, stream);
}

int dgb_float_decompress_pointer(void* temp, size_t tempBytes, int ft, int pb, int useChecksum,
                                 uint32_t n, const void* const* in, void* const* out,
                                 const uint32_t* cap, uint8_t* outSuccess_dev,
                                 uint32_t* outSize_dev, uint8_t* mismatchHost, void* stream) {
  if (!validFloatType(ft)) return DGB_ERR_INVALID_ARG;
  return decodePointerCommon(ft, temp, tempBytes, pb, useChecksum, n, in, out, cap, outSuccess_dev,
                             outSize_dev, mismatchHost, stream);
}

int dgb_float_decompress_split_size(void* temp, size_t tempBytes, int ft, int pb, int useChecksum,
                                    uint32_t n, const void* const* in, void* out_dev,
                                    const uint32_t* splitSizes, uint8_t* outSuccess_dev,
                                    uint32_t* outSize_dev, uint8_t* mismatchHost, void* stream) {
  if (!validFloatType(ft)) return DGB_ERR_INVALID_ARG;
  return decodeSplitCommon(ft, temp, tempBytes, pb, useChecksum, n, in, out_dev, splitSizes,
                           outSuccess_dev, outSize_dev, mismatchHost, stream);
}

// ---- info ------------------------------------------------------------------

int dgb_ans_get_compressed_info(void* temp, size_t tempBytes, const void* const* in,
                                int inIsDevice, uint32_t n, uint32_t* outSizes_dev,
                                uint32_t* outChecksum_dev, void* stream) {
  return getInfo(kKindBytes, temp, tempBytes, in, inIsDevice != 0, n, outSizes_dev, nullptr,
                 outChecksum_dev, (cudaStream_t)stream);
}

int dgb_float_get_compressed_info(void* temp, size_t tempBytes, const void* const* in,
                                  int inIsDevice, uint32_t n, uint32_t* outSizes_dev,
                                  uint32_t* outTypes_dev, uint32_t* outChecksum_dev, void* stream) {
  return getInfo(kKindF16, temp, tempBytes, in, inIsDevice != 0, n, outSizes_dev, outTypes_dev,
                 outChecksum_dev, (cudaStream_t)stream);
}

// ---- host front end helpers ---------------------------------------------------
int dgb_copy_async(void* dst, const void* src, size_t bytes, void* stream) {
  if (bytes == 0) return DGB_OK;
  if (!dst || !src) return DGB_ERR_INVALID_ARG;
  DGB_CUDA_TRY(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDefault, (cudaStream_t)stream));
  return DGB_OK;
}

int dgb_copy_rows_async(void* dst, size_t dst_pitch, const void* src, size_t src_pitch,
                        size_t width_bytes, size_t rows, void* stream) {
  if (width_bytes == 0 || rows == 0) return DGB_OK;
  if (!dst || !src || width_bytes > dst_pitch || width_bytes > src_pitch) return DGB_ERR_INVALID_ARG;
  DGB_CUDA_TRY(cudaMemcpy2DAsync(dst, dst_pitch, src, src_pitch, width_bytes, rows, cudaMemcpyDefault,
                                 (cudaStream_t)stream));
  return DGB_OK;
}

int dgb_archives_pull(int float_type, uint32_t num_in_batch, const void* const* src, void* const* dst,
                      const uint32_t* dst_capacity, uint32_t* out_bytes_dev, void* stream) {
  if (float_type != 0 && float_type != DGB_FLOAT16 && float_type != DGB_BFLOAT16 && float_type != DGB_FLOAT32)
    return DGB_ERR_INVALID_ARG;
  return dgb::pullArchives(float_type, num_in_batch, src, dst, dst_capacity, out_bytes_dev, (cudaStream_t)stream);
}

// ---- options ---------------------------------------------------------------

static int* optionSlot(Options& o, const char* name) {
  if (!name) return nullptr;
  if (!std::strcmp(name, "decode_warps")) return &o.decode_warps;
  if (!std::strcmp(name, "decode_slot_words")) return &o.decode_slot_words;
  if (!std::strcmp(name, "encode_warps")) return &o.encode_warps;
  if (!std::strcmp(name, "encode_canonical")) return &o.encode_canonical;
  if (!std::strcmp(name, "encode_wide_table")) return &o.encode_wide_table;
  if (!std::strcmp(name, "encode_slot_words")) return &o.encode_slot_words;
  if (!std::strcmp(name, "hist_slab_kb")) return &o.hist_slab_kb;
  if (!std::strcmp(name, "hist_ctas_per_sm")) return &o.hist_ctas_per_sm;
  if (!std::strcmp(name, "inline_members")) return &o.inline_members;
  if (!std::strcmp(name, "pull_ctas")) return &o.pull_ctas;
  if (!std::strcmp(name, "timing")) return &o.timing;
  if (!std::strcmp(name, "parts")) return &o.parts;
  return nullptr;
}

int dgb_set_option(const char* name, int value) {
  int* s = optionSlot(dgb::gOptions, name);
  if (!s) return DGB_ERR_INVALID_ARG;
  *s = value;
  return DGB_OK;
}

int dgb_set_thread_option(const char* name, int value) {
  dgb::Options probe;
  if (!optionSlot(probe, name)) return DGB_ERR_INVALID_ARG;
  if (!dgb::tlsHasOptions) {
    dgb::tlsOptions = dgb::gOptions;
    dgb::tlsHasOptions = true;
  }
  *optionSlot(dgb::tlsOptions, name) = value;
  return DGB_OK;
}

int dgb_clear_thread_options(void) {
  dgb::tlsHasOptions = false;
  return DGB_OK;
}

// Sum of the event-timed durations (ms) and launch counts per kernel slot since the last
// call; synchronises the device.  Slots: 0 stats(K1) 1 encode(K2) 3 decode 4 checksum 6 archive mover
// (2 and 5 are retired and always 0).
int dgb_kernel_times(float* ms, int* counts, int nslots) {
  if (cudaDeviceSynchronize() != cudaSuccess) return DGB_ERR_CUDA;
  std::lock_guard<std::mutex> lock(timerMutex());
  for (int i = 0; i < nslots; ++i) { if (ms) ms[i] = 0.f; if (counts) counts[i] = 0; }
  for (auto& t : timedLaunches()) {
    float e = 0.f;
    cudaEventElapsedTime(&e, t.a, t.b);
    if (t.slot < nslots) { if (ms) ms[t.slot] += e; if (counts) counts[t.slot] += 1; }
    eventPool().push_back(t.a);
    eventPool().push_back(t.b);
  }
  timedLaunches().clear();
  return DGB_OK;
}

int dgb_get_option(const char* name, int* value) {
  // read-only counter: hot-path kernels launched so far (stats, encode, decode, archive mover)
  if (name && value && !std::strcmp(name, "launches")) {
    *value = dgb::gLaunches.load(std::memory_order_relaxed);
    return DGB_OK;
  }
  int* s = optionSlot(dgb::options(), name);
  if (!s || !value) return DGB_ERR_INVALID_ARG;
  *value = *s;
  return DGB_OK;
}

}  // extern "C"

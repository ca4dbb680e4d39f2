// common.cuh -- wire-format constants, device helpers and the internal host
// interface shared by the codec translation units.
//
// Wire format: identical to the reference's (ans/GpuANSUtils.cuh:67-227 and
// float/GpuFloatUtils.cuh:26-74, paths relative to /root/reference/dietgpu/).
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

#include <algorithm>

#include "../../include/dietgpu_b200.h"

namespace dgb {

// ---- format constants ------------------------------------------------------
constexpr uint32_t kBlockBytes = 4096;   // ans/GpuANSUtils.cuh:37
constexpr uint32_t kRowsPerBlock = kBlockBytes / 32;
constexpr uint32_t kNumSymbols = 256;
constexpr uint32_t kStateMin = 1u << 15; // ans/GpuANSUtils.cuh:46-49
constexpr uint32_t kAnsMagicVersion = (0xd00du << 16) | 1u;   // :52-55,105-107
constexpr uint32_t kFloatMagicVersion = (0xf00fu << 16) | 1u; // float/GpuFloatUtils.cuh:20-29
constexpr uint32_t kAnsHeaderBytes = 32;
constexpr uint32_t kAnsPdfBytes = 512;
constexpr uint32_t kFloatHeaderBytes = 16;

__host__ __device__ constexpr uint32_t divUp(uint32_t a, uint32_t b) { return (a + b - 1) / b; }
__host__ __device__ constexpr uint32_t roundUp(uint32_t a, uint32_t b) { return divUp(a, b) * b; }
__host__ __device__ constexpr uint64_t roundUp64(uint64_t a, uint64_t b) { return (a + b - 1) / b * b; }

// ans/GpuANSUtils.cuh:68-81
__host__ __device__ constexpr uint32_t ansOverhead(uint32_t numBlocks) {
  return kAnsHeaderBytes + kAnsPdfBytes + 128u * numBlocks + 8u * roundUp(numBlocks, 2u);
}

// float/GpuFloatUtils.cuh:123-127,163-167,194-203 (bytes of the stored,
// non-compressed part, 16 B padded)
__host__ __device__ constexpr uint32_t floatNonCompBytes(int ft, uint32_t n) {
  return ft == DGB_FLOAT32 ? 2u * roundUp(n, 8u) + roundUp(n, 16u) : roundUp(n, 16u);
}

// Worst-case u16 words one 4 KiB block can emit: every symbol costs at most
// probBits bits (a symbol of pdf 1), so 4096*pb/16 words; +8 for 16 B padding.
__host__ __device__ constexpr uint32_t maxBlockWords(int pb) { return 256u * (uint32_t)pb + 8u; }

// ---- per-member descriptor (device), built on the host in one upload -------
enum CodecKind : int { kKindBytes = 0, kKindF16 = DGB_FLOAT16, kKindBF16 = DGB_BFLOAT16, kKindF32 = DGB_FLOAT32 };

struct MemberDesc {
  const void* in;     // encode: raw input (bytes / float words); decode: archive
  void* out;          // encode: archive; decode: output
  uint32_t size;      // encode: input size (bytes, or float WORDS); decode: capacity (same unit)
  uint32_t work0;     // encode: first flat 4 KiB block of this member; decode: bound on its block count
};
static_assert(sizeof(MemberDesc) == 24, "");

// Batches of up to kInlineMembers members travel to the default kernels INSIDE the kernel parameters
// (constant bank, 1.5 KB) instead of through a host-to-device copy in front of the first launch: one
// dependent DMA less per call, nothing of the caller's host memory is read after the call returns,
// and the whole call can be captured into a CUDA graph.  Larger batches (and the canonical encoder)
// read the same table from the scratch buffer.
constexpr uint32_t kInlineMembers = 64;
struct InlineMembers {
  uint32_t count;  // 0: the table is in global memory (scratch)
  uint32_t pad;
  MemberDesc m[kInlineMembers];
};
__device__ __forceinline__ MemberDesc memberAt(const InlineMembers& im, const MemberDesc* global, uint32_t i) {
  return im.count ? im.m[i] : global[i];
}
__device__ __forceinline__ uint32_t memberWork0(const InlineMembers& im, const MemberDesc* global, uint32_t i) {
  return im.count ? im.m[i].work0 : __ldg(&global[i].work0);
}

// ---- encoder symbol table entry (one per symbol, 8 B, shared memory) -------
// magic = ceil(2^(32+shift)/pdf): state / pdf == hi32(state * magic) >> shift for state < 2^31
//         (the quotient ans/GpuANSStatistics.cuh:343-358 computes, without its add; pdf == 1 uses
//         2^32 - 1, i.e. state - 1, and carries the missing 2^pb - 1 in the cdf term)
// pack  = shift (bits 0..4, consumed by shf.wrap) | 2^pb - pdf (bits 5..16) | cdf term (bits 20..31)
// The renormalisation threshold pdf << (31 - pb) is rebuilt from 2^pb - pdf (encode.cu ldsEntry).
struct __align__(8) EncEntry {
  uint32_t magic, pack;
};
constexpr uint32_t kEncKmpShift = 5, kEncKmpMask = 0xfffu, kEncCdfShift = 20;
// Wide form of the same entry: nothing to unpack, four wavefronts per lookup (see EncSym in encode.cu).
//   thr = pdf << (31 - pb), kmp = 2^pb - pdf, cdfShift = shift | cdf term << 5
struct __align__(16) EncEntryWide {
  uint32_t thr, magic, kmp, cdfShift;
};

// ---- tuning options (dgb_set_option) ---------------------------------------
struct Options {
  int decode_warps = 0;      // decoder warps per CTA: 8, or 20 for byte archives; 0 = auto
  int decode_slot_words = 0; // TMA staging slot per warp in u16 words; 0 = auto
  int encode_warps = 8;      // warps per encode CTA (each warp is an independent worker)
  int encode_slot_words = 0; // staging slot of the fast encoder in u16 words; 0 = auto
  int encode_canonical = 0;  // 1: streams packed in block order (byte-identical archives, slower)
  int encode_wide_table = -1;  // encoder table entries: 1 = 16 B, 0 = 8 B, -1 = by data kind (bf16/fp32 wide)
  int hist_slab_kb = 64;     // bytes of input per histogram CTA iteration
  int hist_ctas_per_sm = 32; // stats grid = this many CTAs per SM (each CTA loops over slabs)
  int parts = 0;             // encode sub-batches run on internal streams (0 = auto, 1 = off, max 8)
  int pull_ctas = 64;        // grid of the archive mover (dgb_archives_pull): enough loads in flight for NVLink, few SMs
  int inline_members = 1;   // 1: member table inside the kernel parameters when the batch has <= 64 members
  int timing = 0;            // 1: bracket every kernel launch with CUDA events (bench.py roofline pass)
};
Options& options();

// ---- host-side internal API (capi.cu -> *.cu) --------------------------------
struct HostMember {
  const void* in;
  void* out;
  uint32_t size;  // see MemberDesc::size
};

int encodeBatch(int kind, void* temp, size_t tempBytes, int pb, bool checksum, uint32_t n,
                const HostMember* members, const uint32_t* histogram_dev, uint32_t* outSize_dev,
                cudaStream_t stream);
int decodeBatch(int kind, void* temp, size_t tempBytes, int pb, bool checksum, uint32_t n,
                const HostMember* members, uint8_t* outSuccess_dev, uint32_t* outSize_dev,
                uint8_t* mismatchHost, cudaStream_t stream);
size_t encodeTempBytes(int kind, uint32_t n, uint32_t maxSize);
size_t decodeTempBytes(int kind, uint32_t n);
int getInfo(int kind, void* temp, size_t tempBytes, const void* const* in, bool inIsDevice,
            uint32_t n, uint32_t* outSizes, uint32_t* outTypes, uint32_t* outChecksum,
            cudaStream_t stream);
int pullArchives(int kind, uint32_t n, const void* const* src, void* const* dst, const uint32_t* capacity,
                 uint32_t* outBytes_dev, cudaStream_t stream);

void setLastCudaError(cudaError_t e);

// Per-kernel timing (options().timing): slots are stable indices reported by
// dgb_kernel_times() (C ABI).  Slots 2 and 5 are retired and always report 0.
// No-ops when timing is off.
enum TimerSlot : int { kSlotStats = 0, kSlotEncode = 1, kSlotDecode = 3, kSlotChecksum = 4, kSlotPull = 6, kNumSlots = 7 };
// Internal helper streams: a large encode batch is cut into up to kMaxParts contiguous sub-batches whose
// kernels run on separate streams (forked from / joined to the caller's stream with events), so the
// HBM-bound statistics kernel of one sub-batch overlaps the issue-bound coder of another.
constexpr int kMaxParts = 8;
struct StreamPool {
  cudaStream_t s[kMaxParts];
  cudaEvent_t start, done[kMaxParts];
};
int streamPool(StreamPool** out);  // lazily created; DGB_OK or DGB_ERR_CUDA
// cuts members [0,n) into `parts` contiguous ranges of roughly equal `weight`; bounds has parts+1 entries
void splitParts(const uint64_t* weight, uint32_t n, int parts, uint32_t* bounds);
int autoParts(int kind, uint32_t n, uint64_t totalBytes);

void timerBegin(int slot, cudaStream_t stream);
void timerEnd(int slot, cudaStream_t stream);

#define DGB_CUDA_TRY(expr)                    \
  do {                                        \
    cudaError_t _e = (expr);                  \
    if (_e != cudaSuccess) {                  \
      ::dgb::setLastCudaError(_e);            \
      return DGB_ERR_CUDA;                    \
    }                                         \
  } while (0)

inline size_t alignUp256(size_t v) { return (v + 255) & ~size_t(255); }

// SMs of the current device, cached per device (a process may drive several); racing first calls
// write the same value
inline int smCount() {
  static int cached[64] = {};
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return 148;
  if (!cached[dev]) {
    int v = 0;
    cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, dev);
    cached[dev] = v > 0 ? v : 148;
  }
  return cached[dev];
}

// CTAs of KERN that fit on one SM with `threads` threads and `smemBytes` of dynamic shared memory
// (at least 1).  Cached per host thread and kernel; queried again when the block size, the shared
// memory or the current device changes (function attributes are per device).
template <auto KERN>
int residentPerSm(int threads, size_t smemBytes, int maxSmemBytes, int* out) {
  static thread_local int perSm = 0, keyThreads = 0, keyDev = -1;
  static thread_local size_t keySmem = 0;
  int dev = 0;
  DGB_CUDA_TRY(cudaGetDevice(&dev));
  if (perSm == 0 || keyThreads != threads || keySmem != smemBytes || keyDev != dev) {
    DGB_CUDA_TRY(cudaFuncSetAttribute(KERN, cudaFuncAttributeMaxDynamicSharedMemorySize, maxSmemBytes));
    int occ = 0;
    DGB_CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, KERN, threads, smemBytes));
    perSm = std::max(occ, 1);
    keyThreads = threads; keySmem = smemBytes; keyDev = dev;
  }
  *out = perSm;
  return DGB_OK;
}

#ifdef __CUDACC__
// ---- small device helpers ---------------------------------------------------
__device__ __forceinline__ uint32_t laneId() {
  uint32_t l;
  asm("mov.u32 %0, %%laneid;" : "=r"(l));
  return l;
}
__device__ __forceinline__ uint32_t laneMaskLt() {
  uint32_t m;
  asm("mov.u32 %0, %%lanemask_lt;" : "=r"(m));
  return m;
}
__device__ __forceinline__ uint32_t laneMaskGe() {
  uint32_t m;
  asm("mov.u32 %0, %%lanemask_ge;" : "=r"(m));
  return m;
}
__device__ __forceinline__ uint32_t smemAddr(const void* p) {
  return (uint32_t)__cvta_generic_to_shared(p);
}

// ---- mbarrier + TMA 1-D bulk copy (cp.async.bulk), sm_90+/sm_100a ------------
__device__ __forceinline__ void mbarInit(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void fenceBarrierInit() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void fenceProxyAsync() {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void mbarExpectTx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void mbarWait(uint32_t bar, uint32_t parity) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "DGB_WAIT_%=:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
      "@p bra DGB_DONE_%=;\n"
      "bra DGB_WAIT_%=;\n"
      "DGB_DONE_%=:\n"
      "}\n" ::"r"(bar),
      "r"(parity)
      : "memory");
}
// global -> shared bulk copy; bytes % 16 == 0, both addresses 16 B aligned.
__device__ __forceinline__ void bulkLoad(uint32_t dstSmem, const void* src, uint32_t bytes,
                                         uint32_t bar) {
  asm volatile(
      "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::
          "r"(dstSmem),
      "l"(src), "r"(bytes), "r"(bar)
      : "memory");
}
// ---- cp.async (LDGSTS): 16 B global -> shared copies in commit groups --------
__device__ __forceinline__ void cpAsync16(uint32_t dstSmem, const void* src) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dstSmem), "l"(src) : "memory");
}
__device__ __forceinline__ void cpAsyncCommit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cpAsyncWait() {
  asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory");
}
template <int OFF>
__device__ __forceinline__ uint32_t ldsU8(uint32_t addr) {
  uint32_t v;
  asm volatile("ld.shared.u8 %0, [%1+%2];" : "=r"(v) : "r"(addr), "n"(OFF));
  return v;
}

// block-wide exclusive scan of one value per thread for THREADS threads
// (THREADS multiple of 32, <= 1024).  `warpSums` is smem of THREADS/32 words.
template <int THREADS>
__device__ __forceinline__ uint32_t blockExclusiveScan(uint32_t v, uint32_t* warpSums,
                                                       uint32_t* total) {
  const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  uint32_t incl = v;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    uint32_t t = __shfl_up_sync(0xffffffffu, incl, d);
    if (lane >= (uint32_t)d) incl += t;
  }
  if (lane == 31) warpSums[warp] = incl;
  __syncthreads();
  uint32_t base = 0, tot = 0;
#pragma unroll
  for (int w = 0; w < THREADS / 32; ++w) {
    uint32_t s = warpSums[w];
    if ((uint32_t)w < warp) base += s;
    tot += s;
  }
  if (total) *total = tot;
  __syncthreads();
  return base + incl - v;
}
#endif  // __CUDACC__

}  // namespace dgb

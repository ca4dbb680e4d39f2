// encode.cu -- batched rANS encode (bytes) and float compress (fp16/bf16/fp32)
// for sm_100a.  Two launches per call, whatever the batch size:
//
//   K1  stats*Kernel     a pure read of the raw input: 256-bin histogram of the coded byte, taken out of
//                        the raw bytes / float words with one shift and one mask per element (+ XOR
//                        checksum); float kinds also write the 16 B float header and zero the
//                        padding of the stored plane(s).  The LAST CTA of each member (atomic
//                        ticket) normalises the histogram, bit-identical to the reference
//                        (ans/GpuANSStatistics.cuh:178-367), writes the pdf into the archive and
//                        the encoder table to scratch.
//   K2  encodeKernelFast one resident wave of CTAs, each owning a contiguous range of 4 KiB
//                        blocks (one shared table load per member); each warp runs the
//                        32-lane interleaved rANS state machine of its block
//                        (ans/GpuANSEncode.cuh:49-211) over the member's RAW words (cp.async ring; float
//                        kinds write the stored plane(s) of the archive from the same ring slot, which
//                        replaces the reference's split pass, float/GpuFloatCompress.cuh:280-365)
//                        into a shared-memory staging slot and takes its place in the archive's data section with one 64-bit
//                        atomic, so the words go from shared memory straight to their final
//                        place (the reference's uncoalesced scratch, prefix-sum kernels and
//                        coalesce kernel -- ans/GpuANSEncode.cuh:515-672,
//                        ans/BatchPrefixSum.cuh -- do not exist here).  Streams land in
//                        completion order, which the format allows (the decoder follows
//                        blockWords[k].y).  Option encode_canonical selects encodeKernel:
//                        ordered per-warp tickets + a decoupled look-back, block order,
//                        byte-identical to the reference, slower.
//   Large float batches are cut by member into sub-batches on internal streams (capi.cu autoParts), so
//   that K1 of one sub-batch (HBM-bound) runs beside K2 of the previous one (issue-bound).
//
// The archive produced is field-for-field the reference's (A.4 of SURVEY.md);
// bits the reference leaves undefined are zero.
#include <algorithm>
#include <cstring>
#include <vector>

#include "common.cuh"
#include "../../include/dietgpu_b200_device.cuh"

namespace dgb {

namespace {

constexpr int kStatsThreads = 256;  // == kNumSymbols: thread <-> symbol in the epilogue
constexpr int kStatsWarps = kStatsThreads / 32;
#ifndef DGB_STATS_UNROLL
#define DGB_STATS_UNROLL 4
#endif
constexpr int kStatsUnroll = DGB_STATS_UNROLL;     // independent 16 B loads in flight per thread

__device__ __forceinline__ uint4 ldStream16(const uint4* p) {
  uint4 v;
  asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];"
               : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w)
               : "l"(p));
  return v;
}

struct EncodeScratch {
  MemberDesc* members;            // [n]
  uint32_t* hist;                 // [n][256]      (zeroed per call)
  uint32_t* histDone;             // [n]           (zeroed)
  uint32_t* checksum;             // [n]           (zeroed)
  uint32_t* ticket;               // [4]           (zeroed)
  unsigned long long* lookback;   // [totalTickets](zeroed)   canonical (ordered) layout only
  unsigned long long* allocDone;  // [n]           (zeroed)   low: words handed out, high: blocks placed
  uint8_t* spill;                 // [resident warps][maxBlockWords] u16: overflow of small staging slots
  uint4* table;                   // [n][256] slots of 16 B (packed entries use the first half)
  bool wideTable;                 // entry format: EncEntryWide (16 B) or EncEntry (8 B)
};

// ---------------------------------------------------------------------------
// Normalisation epilogue: 256 threads, thread t owns symbol t.
// Restates ans/GpuANSStatistics.cuh:178-367 (see SURVEY.md A.1); the sort is a
// rank-by-counting over the 256 unique keys (q << 16 | sym), descending.
// ---------------------------------------------------------------------------
__device__ void normalizeAndPublish(const uint32_t* __restrict__ histGlobal, uint32_t total,
                                    int pb, bool wideTable, uint4* __restrict__ tableOut,
                                    uint8_t* __restrict__ ansArchive) {
  const uint32_t t = threadIdx.x;
  const uint32_t K = 1u << pb;
  // the normalisation itself is the device-level API's routine (include/dietgpu_b200_device.cuh): one
  // implementation of the reference's quirks for the library and for user kernels
  uint32_t cdf;
  const uint32_t pdf = dietgpu_b200::device::blockNormalizedPdf(__ldcg(histGlobal + t), total, pb, &cdf);

  // Division constants.  The reference (:343-358) uses the round-up magic that needs
  // hi32(x * magic) + x; the coder state is always < 2^31 here, so the plain round-up
  // reciprocal M = ceil(2^(32+s) / pdf), s = ceil(log2 pdf) - 1, already gives the exact
  // quotient as hi32(x * M) >> s (x * (M * pdf - 2^(32+s)) < 2^31 * pdf <= 2^(32+s)), one add
  // and one register pair cheaper per symbol.  pdf == 1 has no such M below 2^32: it uses
  // M = 2^32 - 1 (quotient x - 1) and folds the missing (K - 1) into the cdf term.
  uint32_t shift = 0, magic = 0, cdfTerm = cdf;
  if (pdf > 1) {
    shift = 31u - (uint32_t)__clz((int)(pdf - 1));
    magic = (uint32_t)(((1ull << (32 + shift)) + pdf - 1) / pdf);
  } else if (pdf == 1) {
    magic = 0xffffffffu;
    cdfTerm = cdf + (K - 1u);
  }
  if (wideTable) {
    EncEntryWide e;
    e.thr = pdf << (31 - pb);
    e.magic = magic;
    e.kmp = K - pdf;
    e.cdfShift = shift | (cdfTerm << 5);
    reinterpret_cast<EncEntryWide*>(tableOut)[t] = e;
  } else {
    EncEntry e;
    e.magic = magic;
    e.pack = shift | ((K - pdf) << kEncKmpShift) | (cdfTerm << kEncCdfShift);
    reinterpret_cast<EncEntry*>(tableOut)[t] = e;
  }
  // archive: u16 pdf[256] right after the 32 B header (ans/GpuANSEncode.cuh:572-577)
  reinterpret_cast<uint16_t*>(ansArchive + kAnsHeaderBytes)[t] = (uint16_t)pdf;
}

// Header + empty pdf for a zero-sized member (ans/ANSTest.cu:243-246 ZeroSized).
__device__ void publishEmptyMember(uint8_t* ansArchive, int pb, bool useChecksum,
                                   uint32_t* outSize, uint32_t m, uint32_t extraBytes) {
  const uint32_t t = threadIdx.x;
  reinterpret_cast<uint16_t*>(ansArchive + kAnsHeaderBytes)[t] = 0;
  if (t == 0) {
    uint4* h = reinterpret_cast<uint4*>(ansArchive);
    h[0] = make_uint4(kAnsMagicVersion, 0u, 0u, 0u);
    h[1] = make_uint4((uint32_t)pb | ((useChecksum ? 1u : 0u) << 4), 0u, 0u, 0u);
    if (outSize) outSize[m] = ansOverhead(0) + extraBytes;
  }
}

__device__ __forceinline__ uint32_t foldXor(uint32_t v) {
  return (v ^ (v >> 8) ^ (v >> 16) ^ (v >> 24)) & 0xffu;
}

// Adds this CTA's per-warp histograms to the global one, takes the member's
// completion ticket and tells whether this CTA is the last one.
__device__ bool flushAndTicket(uint32_t (*sHist)[kNumSymbols], uint32_t* histGlobal,
                               uint32_t* histDone, uint32_t expected, bool doHist,
                               uint32_t xorAcc, uint32_t* checksumGlobal, bool doChecksum) {
  __shared__ uint32_t sLast;
  __syncthreads();
  const uint32_t t = threadIdx.x;
  if (doHist) {
    uint32_t s = 0;
#pragma unroll
    for (int w = 0; w < kStatsWarps; ++w) s += sHist[w][t];
    if (s) atomicAdd(histGlobal + t, s);
  }
  if (doChecksum) {
    uint32_t x = foldXor(xorAcc);
#pragma unroll
    for (int d = 16; d >= 1; d >>= 1) x ^= __shfl_xor_sync(0xffffffffu, x, d);
    if ((t & 31) == 0 && x) atomicXor(checksumGlobal, x);
  }
  __threadfence();
  __syncthreads();
  if (t == 0) sLast = (atomicAdd(histDone, 1u) == expected - 1u);
  __syncthreads();
  const bool last = sLast != 0;
  if (last) __threadfence();
  return last;
}

// ---------------------------------------------------------------------------
// K1 (bytes): histogram + checksum + normalisation epilogue.
// grid = (n, Y): CTA (m, y) walks slabs y, y+Y, ... of member m.
// ---------------------------------------------------------------------------
__device__ inline uint32_t bytesHeadLen(const void* in, uint32_t size) {
  const uint32_t mis = (uint32_t)(reinterpret_cast<uintptr_t>(in) & 15u);
  const uint32_t head = (16u - mis) & 15u;
  return size < head ? size : head;
}
__device__ inline uint32_t bytesSlabs(const void* in, uint32_t size, uint32_t slabVecs, bool doPass) {
  if (!doPass) return 0u;
  const uint32_t nVec = (size - bytesHeadLen(in, size)) / 16u;
  const uint32_t s = divUp(nVec, slabVecs);
  return s > 0u ? s : (size > 0u ? 1u : 0u);
}

// Work of CTA y of Y on member m.  Returns true in the CTA that finished the member (its table is
// published).
__device__ __forceinline__ bool statsBytesItem(const EncodeScratch& sc, uint32_t (*sHist)[kNumSymbols],
                                               const uint32_t* __restrict__ histogramGiven, int pb,
                                               bool useChecksum, uint32_t slabVecs, const MemberDesc& md,
                                               uint32_t m, uint32_t y,
                                               uint32_t Y, uint32_t* __restrict__ outSize) {
  // shuffle => the histogram base is provably warp-uniform (ATOMS [R + UR], no per-symbol add)
  const uint32_t t = threadIdx.x, warp = __shfl_sync(0xffffffffu, t >> 5, 0);
  const uint8_t* in = static_cast<const uint8_t*>(md.in);
  const uint32_t size = md.size;
  uint8_t* archive = static_cast<uint8_t*>(md.out);
  const bool doHist = histogramGiven == nullptr;
  const bool doPass = doHist || useChecksum;

  // member = [head bytes | 16 B vectors | tail bytes]
  const uint32_t head = bytesHeadLen(in, size);
  const uint32_t nVec = (size - head) / 16u;
  const uint32_t tail = size - head - nVec * 16u;
  const uint32_t nSlabs = bytesSlabs(in, size, slabVecs, doPass);
  const uint32_t participants = min(nSlabs, Y);

  if (participants == 0) {
    if (y != 0) return false;
  } else {
    if (y >= participants) return false;
    const uint4* vec = reinterpret_cast<const uint4*>(in + head);
#pragma unroll
    for (int w = 0; w < kStatsWarps; ++w) sHist[w][t] = 0;
    __syncthreads();
    uint32_t* wh = sHist[warp];
    uint32_t xorAcc = 0;
    if (y == 0) {
      if (t < head) { uint32_t b = in[t]; atomicAdd(&wh[b], 1u); xorAcc ^= b; }
      if (t < tail) { uint32_t b = in[head + nVec * 16u + t]; atomicAdd(&wh[b], 1u); xorAcc ^= b; }
    }
    for (uint32_t slab = y; slab < nSlabs; slab += Y) {
      const uint32_t v0 = slab * slabVecs, v1 = min(nVec, v0 + slabVecs);
      for (uint32_t i0 = v0 + t; i0 < v1; i0 += kStatsUnroll * kStatsThreads) {
        uint4 vv[kStatsUnroll];
#pragma unroll
        for (int k = 0; k < kStatsUnroll; ++k) {
          const uint32_t i = i0 + k * kStatsThreads;
          vv[k] = i < v1 ? ldStream16(vec + i) : make_uint4(0, 0, 0, 0);
        }
#pragma unroll
        for (int k = 0; k < kStatsUnroll; ++k) {
          if (i0 + k * kStatsThreads >= v1) break;
          const uint4 v = vv[k];
          xorAcc ^= v.x ^ v.y ^ v.z ^ v.w;
          if (doHist) {
            const uint32_t w4[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
            for (int q = 0; q < 4; ++q) {
              atomicAdd(&wh[w4[q] & 0xffu], 1u);
              atomicAdd(&wh[(w4[q] >> 8) & 0xffu], 1u);
              atomicAdd(&wh[(w4[q] >> 16) & 0xffu], 1u);
              atomicAdd(&wh[w4[q] >> 24], 1u);
            }
          }
        }
      }
    }
    if (!flushAndTicket(sHist, sc.hist + m * kNumSymbols, sc.histDone + m, participants, doHist,
                        xorAcc, sc.checksum + m, useChecksum))
      return false;
  }

  // ---- last CTA of the member ----
  if (size == 0) {
    publishEmptyMember(archive, pb, useChecksum, outSize, m, 0);
    return true;
  }
  const uint32_t* h = doHist ? sc.hist + m * kNumSymbols : histogramGiven + m * kNumSymbols;
  normalizeAndPublish(h, size, pb, sc.wideTable, sc.table + m * kNumSymbols, archive);
  return true;
}

__global__ void __launch_bounds__(kStatsThreads)
statsBytesKernel(EncodeScratch sc, const __grid_constant__ InlineMembers im, const uint32_t* __restrict__ histogramGiven, int pb,
                 bool useChecksum, uint32_t slabVecs, uint32_t memberBase, uint32_t* __restrict__ outSize) {
  __shared__ uint32_t sHist[kStatsWarps][kNumSymbols];
  const uint32_t m = blockIdx.x + memberBase;
  statsBytesItem(sc, sHist, histogramGiven, pb, useChecksum, slabVecs, memberAt(im, sc.members, m), m, blockIdx.y,
                        gridDim.y, outSize);
}

// ---------------------------------------------------------------------------
// K1 (floats): split + histogram of the comp byte + header + epilogue.
// float/GpuFloatCompress.cuh:280-365 (splitFloat), float/GpuFloatUtils.cuh:
// 100-204 (split rules), restated with packed-word bit tricks:
//   fp16 : comp = w >> 8,            non = w & 0xff
//   bf16 : w' = rotl16(w, 1); comp = w' >> 8, non = w' & 0xff
//   fp32 : w' = rotl32(w, 1); comp = w' >> 24, non = w' & 0xffffff
//          stored as a u16 plane (low 16 bits) then a u8 plane (bits 16..23)
// ---------------------------------------------------------------------------
template <int FT>
__device__ __forceinline__ uint32_t rot16x2(uint32_t w) {
  if (FT == DGB_BFLOAT16) {
    // rotate both 16-bit halves left by one: bitwise select between w << 1 and w >> 15 under one
    // mask, a single LOP3 (written as two AND/ORs, ptxas emits two LOP3s for the two constants)
    uint32_t r;
    asm("lop3.b32 %0, %1, %2, %3, 0xE4;" : "=r"(r) : "r"(w << 1), "r"(w >> 15), "r"(0xfffefffeu));
    return r;
  }
  return w;
}

// member = [head elements up to the first 16 B boundary | 16 B vectors | tail elements]
__device__ inline uint32_t floatHeadLen(const void* in, uint32_t size, uint32_t wordBytes) {
  const uint32_t mis = (uint32_t)(reinterpret_cast<uintptr_t>(in) & 15u);
  const uint32_t head = ((16u - mis) & 15u) / wordBytes;
  return size < head ? size : head;
}
__device__ inline uint32_t floatSlabs(const void* in, uint32_t size, uint32_t wordBytes, uint32_t slabVecs) {
  if (size == 0) return 0u;
  const uint32_t nVec = (size - floatHeadLen(in, size, wordBytes)) / (16u / wordBytes);
  const uint32_t s = divUp(nVec, slabVecs);
  return s > 0u ? s : 1u;
}

// Histogram index (x4, the byte offset into a 256-bin u32 histogram) of the coded byte of the
// element in bits [LO, LO + 16) of a packed 16-bit pair, or of a 32-bit word: one shift, one mask.
//   fp16 coded = w >> 8, bf16 coded = (w >> 7) & 0xff, fp32 coded = (w >> 23) & 0xff
template <int FT>
__device__ __forceinline__ uint32_t histOffLo(uint32_t w) {  // low half (or the whole fp32 word)
  return FT == DGB_FLOAT32 ? (w >> 21) & 0x3fcu : (w >> (FT == DGB_BFLOAT16 ? 5 : 6)) & 0x3fcu;
}
template <int FT>
__device__ __forceinline__ uint32_t histOffHi(uint32_t w) {  // high half of a 16-bit pair
  return (w >> (FT == DGB_BFLOAT16 ? 21 : 22)) & 0x3fcu;
}
__device__ __forceinline__ void histAdd(uint32_t* wh, uint32_t byteOff) {
  atomicAdd(reinterpret_cast<uint32_t*>(reinterpret_cast<uint8_t*>(wh) + byteOff), 1u);
}
template <int FT>
__device__ __forceinline__ uint32_t codedScalar(const uint8_t* in, uint32_t e) {
  if (FT == DGB_FLOAT32) return (reinterpret_cast<const uint32_t*>(in)[e] >> 23) & 0xffu;
  const uint32_t w = reinterpret_cast<const uint16_t*>(in)[e];
  return FT == DGB_BFLOAT16 ? (w >> 7) & 0xffu : w >> 8;
}

// The vector body of a float statistics slab: vectors [v0, v1) of the member, 16 B each: a pure
// read (the coder takes the coded byte out of the raw words itself and writes the stored planes).
template <int FT>
__device__ __forceinline__ void histVectors(const uint4* __restrict__ vec, uint32_t v0, uint32_t v1, uint32_t t,
                                            uint32_t* wh) {
  for (uint32_t i0 = v0 + t; i0 < v1; i0 += kStatsUnroll * kStatsThreads) {
    uint4 vv[kStatsUnroll];
#pragma unroll
    for (int k = 0; k < kStatsUnroll; ++k) {
      const uint32_t i = i0 + k * kStatsThreads;
      vv[k] = i < v1 ? ldStream16(vec + i) : make_uint4(0, 0, 0, 0);
    }
#pragma unroll
    for (int k = 0; k < kStatsUnroll; ++k) {
      const uint32_t i = i0 + k * kStatsThreads;
      if (i >= v1) break;
      const uint32_t w4[4] = {vv[k].x, vv[k].y, vv[k].z, vv[k].w};
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        histAdd(wh, histOffLo<FT>(w4[q]));
        if (FT != DGB_FLOAT32) histAdd(wh, histOffHi<FT>(w4[q]));
      }
    }
  }
}

// Work of CTA y of Y on member m; returns true in the CTA that finished the member.
template <int FT>
__device__ __forceinline__ bool statsFloatItem(const EncodeScratch& sc, uint32_t (*sHist)[kNumSymbols], int pb,
                                               bool useChecksum, uint32_t slabVecs, const MemberDesc& md,
                                               uint32_t m, uint32_t y,
                                               uint32_t Y, uint32_t* __restrict__ outSize) {
  constexpr uint32_t EPV = (FT == DGB_FLOAT32) ? 4u : 8u;  // elements per 16 B vector
  constexpr uint32_t WB = (FT == DGB_FLOAT32) ? 4u : 2u;   // word bytes
  // shuffle => the histogram base is provably warp-uniform (ATOMS [R + UR], no per-symbol add)
  const uint32_t t = threadIdx.x, warp = __shfl_sync(0xffffffffu, t >> 5, 0);
  const uint8_t* in = static_cast<const uint8_t*>(md.in);
  const uint32_t size = md.size;  // float words
  uint8_t* archive = static_cast<uint8_t*>(md.out);
  uint8_t* non = archive + kFloatHeaderBytes;
  const uint32_t nonBytes = floatNonCompBytes(FT, size);
  uint8_t* ansArchive = non + nonBytes;

  const uint32_t head = floatHeadLen(in, size, WB);
  const uint32_t nVec = (size - head) / EPV;
  const uint32_t nSlabs = floatSlabs(in, size, WB, slabVecs);
  const uint32_t participants = min(nSlabs, Y);

  if (participants == 0) {
    if (y != 0) return false;
  } else {
    if (y >= participants) return false;
    const uint4* vec = reinterpret_cast<const uint4*>(in + (size_t)head * WB);
#pragma unroll
    for (int w = 0; w < kStatsWarps; ++w) sHist[w][t] = 0;
    __syncthreads();
    uint32_t* wh = sHist[warp];
    uint32_t xorAcc = 0;

    // ---- vector body ----
    for (uint32_t slab = y; slab < nSlabs; slab += Y) {
      const uint32_t v0 = slab * slabVecs, v1 = min(nVec, v0 + slabVecs);
      // four independent 16 B loads per thread are issued before any of them is consumed: the
      // kernel is a pure stream and was latency-bound with one load in flight
      histVectors<FT>(vec, v0, v1, t, wh);
    }
    if (y == 0) {
      // ---- scalar head and tail (fewer than one vector each) ----
      const uint32_t tailStart = head + nVec * EPV;
      if (t < head) atomicAdd(&wh[codedScalar<FT>(in, t)], 1u);
      if (t < size - tailStart) atomicAdd(&wh[codedScalar<FT>(in, tailStart + t)], 1u);
      // float header (float/GpuFloatCompress.cuh:324-337) and zero padding of the planes
      if (t == 0) {
        // float-level checksum is patched in by the epilogue CTA
        *reinterpret_cast<uint4*>(archive) =
            make_uint4(kFloatMagicVersion, size, (uint32_t)FT | ((useChecksum ? 1u : 0u) << 4), 0u);
      }
      if (FT == DGB_FLOAT32) {
        const uint32_t p16 = 2u * roundUp(size, 8u);
        for (uint32_t i = 2u * size + t; i < p16; i += kStatsThreads) non[i] = 0;
        for (uint32_t i = p16 + size + t; i < nonBytes; i += kStatsThreads) non[i] = 0;
      } else {
        for (uint32_t i = size + t; i < nonBytes; i += kStatsThreads) non[i] = 0;
      }
    }
    if (useChecksum) {
      // SURVEY A.6 / B6: the float checksum covers the first `size` BYTES only
      const uint32_t cbytes = size;  // bytes, not words
      for (uint32_t i = y * kStatsThreads + t; i < cbytes; i += participants * kStatsThreads)
        xorAcc ^= in[i];
    }
    if (!flushAndTicket(sHist, sc.hist + m * kNumSymbols, sc.histDone + m, participants, true,
                        xorAcc, sc.checksum + m, useChecksum))
      return false;
  }

  // ---- last CTA of the member ----
  if (size == 0) {
    if (t == 0) {
      *reinterpret_cast<uint4*>(archive) =
          make_uint4(kFloatMagicVersion, 0u, (uint32_t)FT | ((useChecksum ? 1u : 0u) << 4), 0u);
    }
    publishEmptyMember(ansArchive, pb, false, outSize, m, kFloatHeaderBytes + nonBytes);
    return true;
  }
  if (useChecksum && t == 0) {
    reinterpret_cast<uint32_t*>(archive)[3] = __ldcg(sc.checksum + m);
  }
  normalizeAndPublish(sc.hist + m * kNumSymbols, size, pb, sc.wideTable, sc.table + m * kNumSymbols, ansArchive);
  return true;
}

template <int FT>
__global__ void __launch_bounds__(kStatsThreads)
statsFloatKernel(EncodeScratch sc, const __grid_constant__ InlineMembers im, int pb, bool useChecksum, uint32_t slabVecs,
                 uint32_t memberBase, uint32_t* __restrict__ outSize) {
  __shared__ uint32_t sHist[kStatsWarps][kNumSymbols];
  const uint32_t m = blockIdx.x + memberBase;
  statsFloatItem<FT>(sc, sHist, pb, useChecksum, slabVecs, memberAt(im, sc.members, m), m, blockIdx.y, gridDim.y,
                            outSize);
}

// ---------------------------------------------------------------------------
// K2: the rANS state machine + single-pass packing.
//
// Every WARP is an independent worker: it draws ORDERED tickets (one 4 KiB block
// each) from a global counter, keeps its own copy of the member's encoder table
// and its own staging slot in shared memory, streams the block's input bytes
// through a small cp.async ring, and resolves the packed offset of its block
// with a warp-wide decoupled look-back over the tickets of the same member.
// There is no CTA-wide barrier anywhere in the loop (the first version's
// per-ticket __syncthreads cost 27 % of all stall samples in ncu).
// ---------------------------------------------------------------------------
#ifndef DGB_ENC_GROUP_ROWS
#define DGB_ENC_GROUP_ROWS 16
#endif
constexpr int kEncGroupRows = DGB_ENC_GROUP_ROWS;  // rows per cp.async group

// ---------------------------------------------------------------------------
// Input side of the coder, per data kind.  The coder reads the member's RAW words (bytes, or the
// fp16 / bf16 / fp32 words themselves): for float kinds it takes the coded byte out of each word on
// the way to the table lookup and writes the stored plane(s) of the float archive from the same
// shared-memory copy of the input.  The reference (and round 1 here) splits in a separate pass that
// writes the coded bytes to scratch for the coder to read back (float/GpuFloatCompress.cuh:280-365):
// one byte per element written and one read, which is a quarter of the statistics pass's traffic;
// here the statistics pass is a pure read.
//   fp16 : coded = w >> 8,        stored = w & 0xff                     (float/GpuFloatUtils.cuh:111-119)
//   bf16 : coded = (w >> 7) & ff, stored = (w & 7f) << 1 | w >> 15      (:141-159)
//   fp32 : coded = (w >> 23) & ff, stored = low 24 bits of rotl(w, 1): u16 plane then u8 plane (:181-203)
// ---------------------------------------------------------------------------
struct StoredPlanes {
  uint8_t* non;   // fp16 / bf16: the stored byte plane; fp32: the u16 plane
  uint8_t* non1;  // fp32: the u8 plane
};

template <int KIND>
struct EncIn;

template <>
struct EncIn<kKindBytes> {
  static constexpr uint32_t kWordBytes = 1, kRingSlots = 4;
  template <int J, uint32_t STRIDE>
  static __device__ __forceinline__ uint32_t tabOffset(uint32_t ringLane) {
    return STRIDE * ldsU8<J * 32>(ringLane);
  }
  template <uint32_t STRIDE>
  static __device__ __forceinline__ uint32_t tabOffsetOf(uint32_t w) { return STRIDE * w; }
  static __device__ __forceinline__ uint32_t loadWord(const uint8_t* in, uint32_t e) { return in[e]; }
  static __device__ __forceinline__ void storeScalar(const StoredPlanes&, uint32_t, uint32_t) {}
  static __device__ __forceinline__ void storeGroup(uint32_t, const StoredPlanes&, uint32_t, uint32_t) {}
};

#ifndef DGB_ENC_RING16
#define DGB_ENC_RING16 3  // 3 slots = 3 KiB per warp: 4 CTAs per SM (4 slots: 3), c3 encode 195 -> 189 us
#endif
template <int KIND>
struct EncIn16 {
  static constexpr uint32_t kWordBytes = 2, kRingSlots = DGB_ENC_RING16;
  static constexpr uint32_t kCodedBit = KIND == kKindBF16 ? 7u : 8u;
  template <uint32_t STRIDE>
  static __device__ __forceinline__ uint32_t tabOffsetOf(uint32_t w) {
    // STRIDE * ((w >> kCodedBit) & 0xff) in one shift and one mask (STRIDE is 8 or 16)
    constexpr uint32_t lg = STRIDE == 16 ? 4u : 3u;
    return (w >> (kCodedBit - lg)) & (0xffu << lg);
  }
  template <int J, uint32_t STRIDE>
  static __device__ __forceinline__ uint32_t tabOffset(uint32_t ringLane) {
    uint32_t w;
    if (KIND == kKindF16) {
      // the coded byte of fp16 IS the word's high byte: read it alone, no shift / mask
      asm volatile("ld.shared.u8 %0, [%1+%2];" : "=r"(w) : "r"(ringLane), "n"(J * 64 + 1));
      return STRIDE * w;
    }
    asm volatile("ld.shared.u16 %0, [%1+%2];" : "=r"(w) : "r"(ringLane), "n"(J * 64));
    return tabOffsetOf<STRIDE>(w);
  }
  static __device__ __forceinline__ uint32_t loadWord(const uint8_t* in, uint32_t e) {
    return __ldg(reinterpret_cast<const uint16_t*>(in) + e);
  }
  static __device__ __forceinline__ uint32_t storedOf(uint32_t w) {
    return KIND == kKindBF16 ? (((w << 1) | (w >> 15)) & 0xffu) : (w & 0xffu);
  }
  static __device__ __forceinline__ void storeScalar(const StoredPlanes& pl, uint32_t e, uint32_t w) {
    pl.non[e] = (uint8_t)storedOf(w);
  }
  // stored bytes of one group of 16 rows (512 elements, 1 KiB in the ring slot at `slot`): lane l
  // handles the 16 B vectors l and l + 32 -> 8 stored bytes each, one 8 B store
  static __device__ __forceinline__ void storeGroup(uint32_t slot, const StoredPlanes& pl, uint32_t elem0,
                                                    uint32_t lane) {
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const uint32_t v = lane + 32u * h;
      uint4 x;
      asm volatile("ld.shared.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(x.x), "=r"(x.y), "=r"(x.z), "=r"(x.w) : "r"(slot + v * 16u));
      const uint32_t r0 = rot16x2<KIND>(x.x), r1 = rot16x2<KIND>(x.y), r2 = rot16x2<KIND>(x.z), r3 = rot16x2<KIND>(x.w);
      uint2 nn;
      nn.x = __byte_perm(r0, r1, 0x6420);
      nn.y = __byte_perm(r2, r3, 0x6420);
      *reinterpret_cast<uint2*>(pl.non + elem0 + v * 8u) = nn;
    }
  }
};
template <> struct EncIn<kKindF16> : EncIn16<kKindF16> {};
template <> struct EncIn<kKindBF16> : EncIn16<kKindBF16> {};

template <>
struct EncIn<kKindF32> {
  static constexpr uint32_t kWordBytes = 4, kRingSlots = 3;
  template <uint32_t STRIDE>
  static __device__ __forceinline__ uint32_t tabOffsetOf(uint32_t w) {
    constexpr uint32_t lg = STRIDE == 16 ? 4u : 3u;
    return (w >> (23u - lg)) & (0xffu << lg);
  }
  template <int J, uint32_t STRIDE>
  static __device__ __forceinline__ uint32_t tabOffset(uint32_t ringLane) {
    uint32_t w;
    asm volatile("ld.shared.u32 %0, [%1+%2];" : "=r"(w) : "r"(ringLane), "n"(J * 128));
    return tabOffsetOf<STRIDE>(w);
  }
  static __device__ __forceinline__ uint32_t loadWord(const uint8_t* in, uint32_t e) {
    return __ldg(reinterpret_cast<const uint32_t*>(in) + e);
  }
  static __device__ __forceinline__ void storeScalar(const StoredPlanes& pl, uint32_t e, uint32_t w) {
    const uint32_t r = __funnelshift_l(w, w, 1);
    reinterpret_cast<uint16_t*>(pl.non)[e] = (uint16_t)r;
    pl.non1[e] = (uint8_t)(r >> 16);
  }
  // one group of 16 rows = 512 words = 2 KiB in the ring slot: lane l handles vectors l + 32 h
  static __device__ __forceinline__ void storeGroup(uint32_t slot, const StoredPlanes& pl, uint32_t elem0,
                                                    uint32_t lane) {
#pragma unroll
    for (int h = 0; h < 4; ++h) {
      const uint32_t v = lane + 32u * h;
      uint4 x;
      asm volatile("ld.shared.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(x.x), "=r"(x.y), "=r"(x.z), "=r"(x.w) : "r"(slot + v * 16u));
      const uint32_t r0 = __funnelshift_l(x.x, x.x, 1), r1 = __funnelshift_l(x.y, x.y, 1);
      const uint32_t r2 = __funnelshift_l(x.z, x.z, 1), r3 = __funnelshift_l(x.w, x.w, 1);
      uint2 lo;
      lo.x = __byte_perm(r0, r1, 0x5410);
      lo.y = __byte_perm(r2, r3, 0x5410);
      *reinterpret_cast<uint2*>(pl.non + 2u * (size_t)(elem0 + v * 4u)) = lo;
      const uint32_t hi = __byte_perm(__byte_perm(r0, r1, 0x0062), __byte_perm(r2, r3, 0x0062), 0x5410);
      *reinterpret_cast<uint32_t*>(pl.non1 + elem0 + v * 4u) = hi;
    }
  }
};

__host__ __device__ constexpr uint32_t encRingBytes(int kind) {
  return kind == kKindBytes ? 4u * kEncGroupRows * 32u
                            : (kind == kKindF32 ? 3u * kEncGroupRows * 128u : (uint32_t)DGB_ENC_RING16 * kEncGroupRows * 64u);
}

// One rANS step for a full row (ans/GpuANSEncode.cuh:49-90 restated).  The
// update uses x' = (x / pdf) * (2^pb - pdf) + x + cdf, which equals
// (x / pdf) << pb + x % pdf + cdf, so the loop needs neither pdf nor pb.
// `wa` is the shared-memory BYTE address of the next free staging word.
// The emit half is PTX so that one predicate feeds the vote, the store and the
// shift (the compiler otherwise materialises the comparison twice).
// The emitted word gets its own register: the store waits for the POPC, and if it read the state
// register the in-place shift (and with it the whole serial chain) would wait too.  Two ways to
// make the copy, picked per table format by measurement (tools/sweep.py, K2 us, c3 / c2 / c4):
//   FMACOPY = false: plain copy, which ptxas folds into shift + select        (wide 124, packed 266 / 142)
//   FMACOPY = true : multiply by a 1 the compiler cannot see through (IMAD, FMA pipe) and shift the
//                    state in place under the predicate                        (wide 131, packed 259 / 137)
template <bool FMACOPY>
__device__ __forceinline__ void emitWords(uint32_t& state, uint32_t thr, uint32_t& wa, uint32_t ltMask,
                                          uint32_t one) {
  if (FMACOPY) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        ".reg .b32 v, t, a, w;\n"
        ".reg .b16 h;\n"
        "setp.ge.u32 p, %0, %2;\n"
        "mul.lo.u32 w, %0, %4;\n"
        "@p shr.u32 %0, %0, 16;\n"
        "vote.sync.ballot.b32 v, p, 0xffffffff;\n"
        "and.b32 t, v, %3;\n"
        "popc.b32 t, t;\n"
        "mad.lo.u32 a, t, 2, %1;\n"
        "cvt.u16.u32 h, w;\n"
        "@p st.shared.u16 [a], h;\n"
        "popc.b32 t, v;\n"
        "mad.lo.u32 %1, t, 2, %1;\n"
        "}\n"
        : "+r"(state), "+r"(wa)
        : "r"(thr), "r"(ltMask), "r"(one)
        : "memory");
  } else {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        ".reg .b32 v, t, a, w;\n"
        ".reg .b16 h;\n"
        "setp.ge.u32 p, %0, %2;\n"
        "mov.b32 w, %0;\n"
        "shr.u32 t, %0, 16;\n"
        "selp.b32 %0, t, %0, p;\n"
        "vote.sync.ballot.b32 v, p, 0xffffffff;\n"
        "and.b32 t, v, %3;\n"
        "popc.b32 t, t;\n"
        "mad.lo.u32 a, t, 2, %1;\n"
        "cvt.u16.u32 h, w;\n"
        "@p st.shared.u16 [a], h;\n"
        "popc.b32 t, v;\n"
        "mad.lo.u32 %1, t, 2, %1;\n"
        "}\n"
        : "+r"(state), "+r"(wa)
        : "r"(thr), "r"(ltMask)
        : "memory");
  }
}

// Table entry -> the values a row needs.  Two formats (common.cuh), chosen per call by what the
// ANS input is:
//  * EncEntryWide (16 B, LDS.128, four shared-memory wavefronts per row): every field is stored, the
//    row needs the fewest instructions.  Right when a row touches few distinct symbols, i.e. the
//    exponent bytes of bf16 / fp32 data (mostly broadcast reads).
//  * EncEntry (8 B, LDS.64, two wavefronts): the threshold pdf << (31 - pb) is rebuilt from 2^pb - pdf
//    with one multiply-add and the fields are unpacked with shifts and masks.  Right for byte data
//    and fp16, where the bank conflicts of the wide entry dominate (c2: 371 -> 266 us, c4: 162 ->
//    142 us; on c3 the wide entry wins, 126 vs 140 us).
// (Unpacking with IMAD.HI to move work from the ALU to the FMA pipe was measured slower.)
// Everything here is independent of the coder state, so it runs ahead of the serial chain.
struct EncRegs {
  uint32_t tabAddr, ltMask, thrNegScale;  // thrNegScale = -(2^(31 - pb)), packed format only
  uint32_t one;                           // 1, but not a compile-time constant (see emitWords)
};
__device__ __forceinline__ EncRegs makeEncRegs(uint32_t tabAddr, int pb) {
  EncRegs r;
  r.tabAddr = tabAddr;
  r.ltMask = laneMaskLt();
  r.thrNegScale = 0u - (1u << (31 - pb));
  r.one = 1u + ((uint32_t)pb >> 31);  // pb is a kernel argument
  return r;
}

template <bool WIDE>
struct EncSym;
template <>
struct EncSym<true> {
  static constexpr uint32_t kStride = 16;
  uint32_t thr, magic, kmpv, cdfShift;
  __device__ __forceinline__ void load(uint32_t addr, const EncRegs&) {
    // not volatile: the table is read-only while a block is encoded, so the scheduler may hoist it
    asm("ld.shared.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(thr), "=r"(magic), "=r"(kmpv), "=r"(cdfShift) : "r"(addr));
  }
  __device__ __forceinline__ uint32_t shiftReg() const { return cdfShift; }  // low 5 bits count
  __device__ __forceinline__ uint32_t kmp() const { return kmpv; }
  __device__ __forceinline__ uint32_t plusCdf(uint32_t x) const { return x + (cdfShift >> 5); }  // one LEA.HI
};
template <>
struct EncSym<false> {
  static constexpr uint32_t kStride = 8;
  uint32_t thr, magic, pack, kmpv;
  __device__ __forceinline__ void load(uint32_t addr, const EncRegs& rc) {
    asm("ld.shared.v2.u32 {%0,%1}, [%2];" : "=r"(magic), "=r"(pack) : "r"(addr));
    kmpv = (pack >> kEncKmpShift) & kEncKmpMask;
    thr = kmpv * rc.thrNegScale + 0x80000000u;                                          // pdf << (31 - pb)
  }
  __device__ __forceinline__ uint32_t shiftReg() const { return pack; }
  __device__ __forceinline__ uint32_t kmp() const { return kmpv; }
  __device__ __forceinline__ uint32_t plusCdf(uint32_t x) const { return x + (pack >> kEncCdfShift); }
};

template <bool WIDE>
__device__ __forceinline__ void encodeUpdate(uint32_t& state, const EncSym<WIDE>& e) {
  const uint32_t div = __funnelshift_r(__umulhi(state, e.magic), 0u, e.shiftReg());
  state = div * e.kmp() + e.plusCdf(state);
}

template <bool WIDE>
__device__ __forceinline__ void encodeStep(uint32_t& state, uint32_t tabOff, const EncRegs& rc, uint32_t& wa) {
  EncSym<WIDE> e;
  e.load(rc.tabAddr + tabOff, rc);
  emitWords<!WIDE>(state, e.thr, wa, rc.ltMask, rc.one);
  encodeUpdate(state, e);
}

template <bool WIDE>
__device__ __forceinline__ void encodeStepPartial(bool valid, uint32_t& state, uint32_t tabOff,
                                                  const EncRegs& rc, uint32_t& wa) {
  EncSym<WIDE> e;
  e.load(rc.tabAddr + tabOff, rc);
  // invalid lanes never emit: compare against an unreachable threshold
  emitWords<!WIDE>(state, valid ? e.thr : 0xffffffffu, wa, rc.ltMask, rc.one);
  uint32_t next = state;
  encodeUpdate(next, e);
  state = valid ? next : state;
}

// One group of kEncGroupRows rows.  The symbol bytes and the table entries do not depend on
// the coder state, so they are fetched ahead of the serial state chain: all symbols of the
// group first, then table entries kept kDepth rows ahead of the row being coded.
template <int KIND, int J, uint32_t STRIDE>
struct EncLoad {
  static __device__ __forceinline__ void syms(uint32_t ringLane, uint32_t tabAddr, uint32_t* addr) {
    EncLoad<KIND, J - 1, STRIDE>::syms(ringLane, tabAddr, addr);
    addr[J - 1] = tabAddr + EncIn<KIND>::template tabOffset<J - 1, STRIDE>(ringLane);
  }
};
template <int KIND, uint32_t STRIDE>
struct EncLoad<KIND, 0, STRIDE> {
  static __device__ __forceinline__ void syms(uint32_t, uint32_t, uint32_t*) {}
};

template <bool WIDE, int KIND>
__device__ __forceinline__ void encodeGroup(uint32_t& state, uint32_t ringLane, const EncRegs& rc,
                                            uint32_t& wa) {
  constexpr int U = kEncGroupRows;
  constexpr int kDepth = 4;
  uint32_t addr[U];
  EncLoad<KIND, U, EncSym<WIDE>::kStride>::syms(ringLane, rc.tabAddr, addr);
  EncSym<WIDE> e[kDepth];
#pragma unroll
  for (int j = 0; j < kDepth; ++j) e[j].load(addr[j], rc);
#pragma unroll
  for (int j = 0; j < U; ++j) {
    const EncSym<WIDE> cur = e[j % kDepth];
    if (j + kDepth < U) e[j % kDepth].load(addr[j + kDepth], rc);
    emitWords<!WIDE>(state, cur.thr, wa, rc.ltMask, rc.one);
    encodeUpdate(state, cur);
  }
}

// Staging slot smaller than the worst case: when it runs low, the words staged so far are moved
// to this warp's global spill area (16 B granules; the < 8 leftover words slide to the slot start).
struct Spill {
  uint16_t* area;       // global, maxBlockWords(pb) words, 16 B aligned (nullptr: slot is worst-case sized)
  uint32_t limitBytes;  // spill when more than this many bytes are staged
  uint32_t spilled;     // words already in `area` (multiple of 8)
};

__device__ __forceinline__ void spillOut(Spill& sp, uint32_t stageAddr, uint16_t* stage, uint32_t& wa,
                                         uint32_t lane) {
  __syncwarp();
  const uint32_t used = (wa - stageAddr) >> 1;
  const uint32_t k = used & ~7u;
  uint4* dst = reinterpret_cast<uint4*>(sp.area + sp.spilled);
  const uint4* src = reinterpret_cast<const uint4*>(stage);
  for (uint32_t i = lane; i < k / 8u; i += 32u) dst[i] = src[i];
  const uint32_t left = used - k;
  uint16_t v = 0;
  if (lane < left) v = stage[k + lane];
  __syncwarp();
  if (lane < left) stage[lane] = v;
  __syncwarp();
  sp.spilled += k;
  wa = stageAddr + 2u * left;
}

// Encodes elements [0, n) of one block (raw words of data kind KIND at `in`; `elem0` = index of the
// block's first element in its member) with one warp into the staging slot at shared byte address
// `stageAddr` (spilling to sp.area when the slot is small); float kinds also write the block's
// stored plane(s).  Returns the TOTAL word count; the words not yet spilled are
// stage[0 .. total - sp.spilled).
template <bool WIDE, int KIND>
__device__ __forceinline__ uint32_t encodeBlockWarp(const uint8_t* __restrict__ in, uint32_t n, uint32_t elem0,
                                                    const StoredPlanes& planes, uint32_t tabAddr, int pb,
                                                    uint32_t stageAddr, uint16_t* stage, Spill& sp,
                                                    uint32_t ringAddr, uint32_t lane, uint32_t& stateOut) {
  typedef EncIn<KIND> In;
  constexpr int U = kEncGroupRows;
  constexpr uint32_t WB = In::kWordBytes;
  constexpr uint32_t kGroupBytes = U * 32 * WB;     // 512 B, 1 KiB or 2 KiB
  constexpr uint32_t kChunks = kGroupBytes / 512u;  // 16 B copies per lane and group
  constexpr uint32_t kStride = EncSym<WIDE>::kStride;
  uint32_t state = kStateMin;
  uint32_t wa = stageAddr;
  const EncRegs rc = makeEncRegs(tabAddr, pb);
  const uint32_t fullRows = n >> 5;
  uint32_t r = 0;
  sp.spilled = 0;
  if ((reinterpret_cast<uintptr_t>(in) & 15u) == 0) {
    const uint32_t groups = fullRows / U;
    // input rows stream through the cp.async ring, two groups ahead of the encoder
    const uint8_t* src = in + lane * 16u;
    const uint32_t dst = ringAddr + lane * 16u;
    auto issue = [&](uint32_t g, uint32_t slot) {
#pragma unroll
      for (uint32_t c = 0; c < kChunks; ++c)
        cpAsync16(dst + slot * kGroupBytes + c * 512u, src + (size_t)g * kGroupBytes + c * 512u);
    };
    if (groups > 0) issue(0, 0);
    cpAsyncCommit();
    if (groups > 1) issue(1, 1);
    cpAsyncCommit();
    uint32_t slot = 0, slotNext = 2 % In::kRingSlots;
    for (uint32_t k = 0; k < groups; ++k) {
      if (sp.area && wa - stageAddr > sp.limitBytes) spillOut(sp, stageAddr, stage, wa, lane);
      cpAsyncWait<1>();  // group k has landed (group k + 1 may still be in flight)
      // one warp barrier does both jobs: every lane sees group k, and every lane is done reading group
      // k - 1, whose ring slot (three-slot ring) the request below overwrites
      __syncwarp();
      if (k + 2 < groups) issue(k + 2, slotNext);
      cpAsyncCommit();
      const uint32_t slotAddr = ringAddr + slot * kGroupBytes;
      if (KIND != kKindBytes) In::storeGroup(slotAddr, planes, elem0 + k * (U * 32), lane);
      encodeGroup<WIDE, KIND>(state, slotAddr + lane * WB, rc, wa);
      slot = slot + 1 == In::kRingSlots ? 0u : slot + 1;
      slotNext = slotNext + 1 == In::kRingSlots ? 0u : slotNext + 1;
    }
    r = groups * U;
  }
  // remaining rows (fewer than U, or all of them when the input is not 16 B aligned): every U rows
  // the same spill check as above
  uint32_t e = r * 32u + lane;
  for (uint32_t j = 0; r < fullRows; ++r, ++j, e += 32) {
    if (sp.area && (j % U) == 0 && wa - stageAddr > sp.limitBytes) spillOut(sp, stageAddr, stage, wa, lane);
    const uint32_t w = In::loadWord(in, e);
    In::storeScalar(planes, elem0 + e, w);
    encodeStep<WIDE>(state, In::template tabOffsetOf<kStride>(w), rc, wa);
  }
  const uint32_t rem = n & 31u;
  if (rem) {
    if (sp.area && wa - stageAddr > sp.limitBytes) spillOut(sp, stageAddr, stage, wa, lane);
    const bool valid = lane < rem;
    const uint32_t w = valid ? In::loadWord(in, e) : 0u;
    if (valid) In::storeScalar(planes, elem0 + e, w);
    encodeStepPartial<WIDE>(valid, state, In::template tabOffsetOf<kStride>(w), rc, wa);
  }
  stateOut = state;
  return sp.spilled + ((wa - stageAddr) >> 1);
}

// Pads the block's stream to a multiple of 8 words and copies it to `dst` (global, 16 B aligned).
__device__ __forceinline__ void placeStream(uint16_t* stage, Spill& sp, uint32_t words, uint32_t padded,
                                            uint8_t* dst8, uint32_t lane) {
  const uint32_t local = words - sp.spilled;        // words still in the slot
  if (local + lane < padded - sp.spilled) stage[local + lane] = 0;  // pad < 8 words
  __syncwarp();
  uint4* dst = reinterpret_cast<uint4*>(dst8);
  if (sp.spilled) {
    const uint4* g = reinterpret_cast<const uint4*>(sp.area);
    for (uint32_t i = lane; i < sp.spilled / 8u; i += 32u) dst[i] = __ldcg(g + i);
    dst += sp.spilled / 8u;
  }
  const uint4* src = reinterpret_cast<const uint4*>(stage);
  for (uint32_t i = lane; i < (padded - sp.spilled) / 8u; i += 32u) dst[i] = src[i];
}

constexpr unsigned long long kFlagAgg = 1ull << 32;
constexpr unsigned long long kFlagPrefix = 2ull << 32;

// Exclusive prefix of the per-ticket totals of this member (decoupled
// look-back, one warp).  first = first ticket of the member.
__device__ __forceinline__ uint32_t lookbackWarp(volatile unsigned long long* desc, uint32_t ticket,
                                                 uint32_t first, uint32_t lane) {
  uint32_t base = 0;
  int64_t idx = (int64_t)ticket - 1;
  while (idx >= (int64_t)first) {
    const int64_t mine = idx - lane;
    unsigned long long d = kFlagPrefix;  // lanes before `first`: neutral, terminates the walk
    if (mine >= (int64_t)first) {
      do { d = desc[mine]; } while ((d >> 32) == 0ull);
    }
    const bool isPrefix = (d >> 32) == 2ull;
    const uint32_t pmask = __ballot_sync(0xffffffffu, isPrefix);
    // lanes 0..firstPrefixLane contribute (lane 0 is the nearest predecessor)
    const uint32_t stop = pmask ? (uint32_t)__ffs((int)pmask) - 1u : 31u;
    uint32_t v = lane <= stop ? (uint32_t)d : 0u;
#pragma unroll
    for (int s = 16; s >= 1; s >>= 1) v += __shfl_xor_sync(0xffffffffu, v, s);
    base += v;
    if (pmask) break;
    idx -= 32;
  }
  return base;
}

// dynamic shared memory per warp: [table 2 KiB][input ring 2 KiB][staging slot]
__host__ __device__ constexpr uint32_t encWarpSmem(int pb, int kind) {
  return kNumSymbols * 8u + encRingBytes(kind) + maxBlockWords(pb) * 2u;
}

template <int KIND>
__global__ void encodeKernel(EncodeScratch sc, int pb, bool useChecksum,
                             uint32_t numMembers, uint32_t totalTickets,
                             uint32_t* __restrict__ outSize) {
  constexpr int kind = KIND;
  extern __shared__ __align__(16) uint8_t smem[];
  const uint32_t t = threadIdx.x, lane = t & 31u;
  // shuffle => provably warp-uniform (no divergence check around the votes in the hot loop)
  const uint32_t warp = __shfl_sync(0xffffffffu, t >> 5, 0);
  uint8_t* mine = smem + (size_t)warp * encWarpSmem(pb, kind);
  uint4* myTab = reinterpret_cast<uint4*>(mine);
  const uint32_t tabAddr = smemAddr(mine);
  const uint32_t ringAddr = tabAddr + kNumSymbols * 8u;
  uint16_t* myStage = reinterpret_cast<uint16_t*>(mine + kNumSymbols * 8u + encRingBytes(kind));
  const uint32_t stageAddr = smemAddr(myStage);
  volatile unsigned long long* desc = sc.lookback;
  uint32_t curMember = 0xffffffffu;

  for (;;) {
    uint32_t ticket = 0;
    if (lane == 0) ticket = atomicAdd(sc.ticket, 1u);
    ticket = __shfl_sync(0xffffffffu, ticket, 0);
    if (ticket >= totalTickets) break;
    // member m with work0[m] <= ticket < work0[m+1]  (uniform binary search, L1-cached)
    uint32_t lo = 0, hi = numMembers;
    while (hi - lo > 1) {
      const uint32_t mid = (lo + hi) >> 1;
      if (__ldg(&sc.members[mid].work0) <= ticket) lo = mid; else hi = mid;
    }
    const uint32_t m = lo;
    const MemberDesc md = sc.members[m];
    const uint32_t size = md.size;
    const uint32_t nb = divUp(size, kBlockBytes);
    const uint32_t block = ticket - md.work0;

    const uint8_t* ansIn;
    uint8_t* ansOut;
    uint32_t extraBytes = 0;
    StoredPlanes planes{nullptr, nullptr};
    ansIn = static_cast<const uint8_t*>(md.in);
    if (kind == kKindBytes) {
      ansOut = static_cast<uint8_t*>(md.out);
    } else {
      extraBytes = kFloatHeaderBytes + floatNonCompBytes(kind, size);
      ansOut = static_cast<uint8_t*>(md.out) + extraBytes;
      planes.non = static_cast<uint8_t*>(md.out) + kFloatHeaderBytes;
      planes.non1 = planes.non + 2u * roundUp(size, 8u);
      __builtin_assume(__isGlobal(planes.non));
      __builtin_assume(__isGlobal(planes.non1));
    }
    __builtin_assume(__isGlobal(ansIn));
    __builtin_assume(__isGlobal(ansOut));

    if (m != curMember) {
      // this member's encoder table -> my private copy (written by K1's epilogue)
      const uint4* src = sc.table + (size_t)m * kNumSymbols;
#pragma unroll
      for (uint32_t i = 0; i < kNumSymbols / 64; ++i) myTab[i * 32 + lane] = __ldcg(src + i * 32 + lane);
      curMember = m;
      __syncwarp();
    }

    // ---- encode the block into my staging slot ----
    const uint32_t start = block * kBlockBytes;
    const uint32_t blockLen = min(kBlockBytes, size - start);
    uint32_t state;
    Spill sp{nullptr, 0u, 0u};  // worst-case sized slot: never spills
    const uint32_t words = encodeBlockWarp<false, KIND>(ansIn + (size_t)start * EncIn<KIND>::kWordBytes, blockLen, start, planes,
                                                        tabAddr, pb, stageAddr, myStage, sp, ringAddr, lane, state);
    const uint32_t padded = roundUp(words, 8u);

    // ---- packed offset of this block: look-back over the member's earlier tickets ----
    uint32_t base = 0;
    if (block != 0) {
      if (lane == 0) desc[ticket] = kFlagAgg | padded;
      base = lookbackWarp(desc, ticket, md.work0, lane);
    }
    if (lane == 0) desc[ticket] = kFlagPrefix | (unsigned long long)(base + padded);
    __syncwarp();

    // ---- final placement: states, blockWords, packed stream ----
    uint8_t* pStates = ansOut + kAnsHeaderBytes + kAnsPdfBytes;
    uint8_t* pBlockWords = pStates + 128u * nb;
    uint8_t* pData = pBlockWords + 8u * roundUp(nb, 2u);
    reinterpret_cast<uint32_t*>(pStates)[block * 32u + lane] = state;
    if (lane == 0)
      reinterpret_cast<uint2*>(pBlockWords)[block] = make_uint2((blockLen << 16) | words, base);
    placeStream(myStage, sp, words, padded, pData + 2u * (size_t)base, lane);
    if (block == nb - 1 && lane == 0) {
      // ans/GpuANSEncode.cuh:553-569 header (undefined bits zeroed)
      const uint32_t totalWords = base + padded;
      uint4* h = reinterpret_cast<uint4*>(ansOut);
      h[0] = make_uint4(kAnsMagicVersion, nb, size, totalWords);
      const bool ansChecksum = useChecksum && kind == kKindBytes;
      h[1] = make_uint4((uint32_t)pb | ((ansChecksum ? 1u : 0u) << 4),
                        ansChecksum ? __ldcg(sc.checksum + m) : 0u, 0u, 0u);
      if (nb & 1u) reinterpret_cast<uint2*>(pBlockWords)[nb] = make_uint2(0u, 0u);
      if (outSize) outSize[m] = ansOverhead(nb) + 2u * totalWords + extraBytes;
    }
    __syncwarp();  // staging and ring are reused by the next ticket
  }
}

// ---------------------------------------------------------------------------
// K2, default flavour: no inter-block dependency at all.  The archive format
// addresses every block's stream through blockWords[k].y, so streams may sit in
// the data section in ANY order; here a block takes its place with one
// atomicAdd on the member's word counter when it has been encoded.  Sizes, the
// pdf, every lane state and every stream are identical to the canonical
// encoder's (and to the reference's); only the ORDER of the streams inside the
// data section (and hence the .y offsets) depends on completion order.  The
// ordered, byte-for-byte canonical layout is available as option
// "encode_canonical" (encodeKernel above, ~25 % slower: ncu shows its warps
// spend that time polling the look-back descriptors of slower predecessors).
//
// Work split is static: CTA c owns a contiguous range of flat blocks, walks it
// member by member (one shared table load per member) and its warps stride
// over the blocks of the member.
// ---------------------------------------------------------------------------
__host__ __device__ constexpr uint32_t encFastWarpSmem(uint32_t slotWords, int kind) {
  return encRingBytes(kind) + slotWords * 2u;  // ring + staging
}

// Per-warp view of the CTA's dynamic shared memory: [input ring | staging slot] per warp.  Input rows
// arrive by per-lane cp.async: a TMA bulk copy per group (one lane issuing, 32 lanes polling an
// mbarrier) measured slower on B200, encode call c3 185.7 vs 192.1 us, c4 209.5 vs 212.0, c2 358.0 vs
// 363.3 (profiles/r02_ab_tma_input_ring.txt).
struct WarpSmem {
  uint32_t ringAddr, stageAddr;
  uint16_t* stage;
  Spill sp;
};
__device__ __forceinline__ WarpSmem warpSmem(const EncodeScratch& sc, uint8_t* smem, uint32_t warp, uint32_t W,
                                             uint32_t slotWords, int pb, int kind, uint32_t spillWarpBase) {
  WarpSmem ws;
  uint8_t* mine = smem + (size_t)warp * encFastWarpSmem(slotWords, kind);
  ws.ringAddr = smemAddr(mine);
  ws.sp.area = slotWords < maxBlockWords(pb)
                   ? reinterpret_cast<uint16_t*>(sc.spill) + (size_t)(spillWarpBase + blockIdx.x * W + warp) * maxBlockWords(pb)
                   : nullptr;
  ws.sp.limitBytes = (slotWords - kEncGroupRows * 32u - 8u) * 2u;  // a group emits at most 16*32 words
  ws.sp.spilled = 0;
  ws.stage = reinterpret_cast<uint16_t*>(mine + encRingBytes(kind));
  ws.stageAddr = smemAddr(ws.stage);
  return ws;
}

// Loads member m's encoder table (written by the statistics epilogue) into the CTA's table slot.
template <bool WIDE>
__device__ __forceinline__ void loadTable(const EncodeScratch& sc, uint4* sTab, uint32_t m) {
  const uint4* src = sc.table + (size_t)m * kNumSymbols;
  for (uint32_t i = threadIdx.x; i < (WIDE ? kNumSymbols : kNumSymbols / 2); i += blockDim.x) sTab[i] = __ldcg(src + i);
}

// Warps of the CTA encode blocks [first, last) of member m (block k by warp (k - first) % W): the
// 32-lane rANS state machine per block, then the block takes its place in the archive's data
// section with one 64-bit atomic.
template <bool WIDE, int KIND>
__device__ __forceinline__ void encodeMemberBlocks(const EncodeScratch& sc, const MemberDesc& md, uint32_t m,
                                                   uint32_t first, uint32_t last, int pb,
                                                   bool useChecksum, uint32_t tabAddr, WarpSmem& ws,
                                                   uint32_t warp, uint32_t W, uint32_t lane,
                                                   uint32_t* __restrict__ outSize) {
  constexpr int kind = KIND;
  const uint32_t size = md.size;
  const uint32_t nb = divUp(size, kBlockBytes);
  const uint8_t* ansIn;
  uint8_t* ansOut;
  uint32_t extraBytes = 0;
  StoredPlanes planes{nullptr, nullptr};
  ansIn = static_cast<const uint8_t*>(md.in);
  if (kind == kKindBytes) {
    ansOut = static_cast<uint8_t*>(md.out);
  } else {
    extraBytes = kFloatHeaderBytes + floatNonCompBytes(kind, size);
    ansOut = static_cast<uint8_t*>(md.out) + extraBytes;
    planes.non = static_cast<uint8_t*>(md.out) + kFloatHeaderBytes;
    planes.non1 = planes.non + 2u * roundUp(size, 8u);
    __builtin_assume(__isGlobal(planes.non));
    __builtin_assume(__isGlobal(planes.non1));
  }
  __builtin_assume(__isGlobal(ansIn));
  __builtin_assume(__isGlobal(ansOut));
  uint8_t* pStates = ansOut + kAnsHeaderBytes + kAnsPdfBytes;
  uint8_t* pBlockWords = pStates + 128u * nb;
  uint8_t* pData = pBlockWords + 8u * roundUp(nb, 2u);

  for (uint32_t block = first + warp; block < last; block += W) {
    const uint32_t start = block * kBlockBytes;
    const uint32_t blockLen = min(kBlockBytes, size - start);
    uint32_t state;
    const uint32_t words = encodeBlockWarp<WIDE, KIND>(ansIn + (size_t)start * EncIn<KIND>::kWordBytes, blockLen, start,
                                                       planes, tabAddr, pb, ws.stageAddr, ws.stage, ws.sp, ws.ringAddr,
                                                       lane, state);
    const uint32_t padded = roundUp(words, 8u);
    // take a place in the data section: one 64-bit atomic hands out the word offset (low half)
    // and counts finished blocks (high half), so no fence is needed to order the two
    unsigned long long old = 0;
    if (lane == 0) old = atomicAdd(sc.allocDone + m, (1ull << 32) | (unsigned long long)padded);
    reinterpret_cast<uint32_t*>(pStates)[block * 32u + lane] = state;
    old = __shfl_sync(0xffffffffu, old, 0);
    const uint32_t base = (uint32_t)old;
    if (lane == 0)
      reinterpret_cast<uint2*>(pBlockWords)[block] = make_uint2((blockLen << 16) | words, base);
    placeStream(ws.stage, ws.sp, words, padded, pData + 2u * (size_t)base, lane);
    // the block that takes the last place knows the member's total and writes the header
    if (lane == 0 && (uint32_t)(old >> 32) == nb - 1u) {
      const uint32_t totalWords = base + padded;
      uint4* h = reinterpret_cast<uint4*>(ansOut);
      h[0] = make_uint4(kAnsMagicVersion, nb, size, totalWords);
      const bool ansChecksum = useChecksum && kind == kKindBytes;
      h[1] = make_uint4((uint32_t)pb | ((ansChecksum ? 1u : 0u) << 4),
                        ansChecksum ? __ldcg(sc.checksum + m) : 0u, 0u, 0u);
      if (nb & 1u) reinterpret_cast<uint2*>(pBlockWords)[nb] = make_uint2(0u, 0u);
      if (outSize) outSize[m] = ansOverhead(nb) + 2u * totalWords + extraBytes;
    }
    __syncwarp();  // staging and ring are reused by the next block
  }
}

template <bool WIDE, int KIND>
__global__ void
encodeKernelFast(EncodeScratch sc, const __grid_constant__ InlineMembers im, int pb, bool useChecksum,
                                 uint32_t numMembers, uint32_t blockBegin, uint32_t blockEnd,
                                 uint32_t slotWords, uint32_t spillWarpBase,
                                 uint32_t* __restrict__ outSize) {
  extern __shared__ __align__(16) uint8_t smem[];
  __shared__ __align__(16) uint4 sTab[WIDE ? kNumSymbols : kNumSymbols / 2];  // static: constant base for the hot LDS
  __shared__ uint32_t sMember;
  const uint32_t t = threadIdx.x, lane = t & 31u;
  const uint32_t warp = __shfl_sync(0xffffffffu, t >> 5, 0);
  const uint32_t W = blockDim.x >> 5;
  WarpSmem ws = warpSmem(sc, smem, warp, W, slotWords, pb, KIND, spillWarpBase);
  const uint32_t tabAddr = smemAddr(sTab);

  const uint64_t g = gridDim.x, span = blockEnd - blockBegin;
  uint32_t cur = blockBegin + (uint32_t)(span * blockIdx.x / g);
  const uint32_t end = blockBegin + (uint32_t)(span * (blockIdx.x + 1) / g);

  while (cur < end) {
    if (t == 0) {
      uint32_t lo = 0, hi = numMembers;
      while (hi - lo > 1) {
        const uint32_t mid = (lo + hi) >> 1;
        if (memberWork0(im, sc.members, mid) <= cur) lo = mid; else hi = mid;
      }
      sMember = lo;
    }
    __syncthreads();
    const uint32_t m = sMember;
    const MemberDesc md = memberAt(im, sc.members, m);
    const uint32_t nb = divUp(md.size, kBlockBytes);
    const uint32_t memberEnd = min(end, md.work0 + nb);
    loadTable<WIDE>(sc, sTab, m);
    __syncthreads();
    encodeMemberBlocks<WIDE, KIND>(sc, md, m, cur - md.work0, memberEnd - md.work0, pb, useChecksum, tabAddr, ws,
                                   warp, W, lane, outSize);
    cur = memberEnd;
    __syncthreads();  // table is replaced for the next member
  }
}

struct ScratchPlan {
  size_t members, zeroBegin, hist, histDone, checksum, ticket, allocDone, zeroEnd, lookback, lookbackEnd, table, spill,
      total;
  uint32_t spillWarps;
};

// Encoder warps that may need a spill slot (one slot = the worst-case stream of one block): never
// more than the device can hold resident (64 warps per SM), never more than the batch has work
// for, so small batches get small scratch (the reference's scratch scales with the batch too).
// The bound also caps the coder grid (spillWarpsPerPart / W in encodeBatch), so it is part of the
// launch configuration, not only of the scratch size.
uint32_t spillWarpBound(uint32_t n, uint64_t totalBlocks) {
  const uint64_t resident = 64ull * (uint64_t)smCount();
  // up to 8 warps per CTA; a coder grid has at most one CTA per block, plus a slack of two CTAs per member
  const uint64_t work = 8ull * ((uint64_t)n * 2ull + totalBlocks);
  return (uint32_t)std::min(resident, work);
}

ScratchPlan planScratch(int kind, uint32_t n, uint32_t maxSize, uint32_t totalTickets, uint32_t spillWarps) {
  ScratchPlan p{};
  size_t o = 0;
  p.members = o; o = alignUp256(o + sizeof(MemberDesc) * (size_t)n);  // uploaded unless the kernel parameters carry it
  p.zeroBegin = o;
  p.hist = o; o = alignUp256(o + sizeof(uint32_t) * kNumSymbols * (size_t)n);
  p.histDone = o; o = alignUp256(o + sizeof(uint32_t) * (size_t)n);
  p.checksum = o; o = alignUp256(o + sizeof(uint32_t) * (size_t)n);
  p.ticket = o; o = alignUp256(o + 16);
  p.allocDone = o; o = alignUp256(o + sizeof(unsigned long long) * (size_t)n);
  p.zeroEnd = o;
  // look-back descriptors: canonical (ordered) layout only; cleared only then
  p.lookback = o; o = alignUp256(o + sizeof(unsigned long long) * (size_t)totalTickets);
  p.lookbackEnd = o;
  p.table = o; o = alignUp256(o + sizeof(uint4) * kNumSymbols * (size_t)n);
  p.spillWarps = spillWarps;
  p.spill = o; o = alignUp256(o + (size_t)spillWarps * maxBlockWords(11) * 2u);
  p.total = o;
  return p;
}

uint32_t ticketsFor(uint32_t size) { return divUp(size, kBlockBytes); }

// Joins the internal streams on every exit path: the caller frees / reuses its scratch when the
// call returns, so work already queued on a helper stream must be ordered before whatever the
// caller enqueues next on its own stream -- also when a later launch of the same call failed.
struct ForkGuard {
  StreamPool* pool = nullptr;
  cudaStream_t stream = nullptr;
  bool forked[kMaxParts] = {};
  ~ForkGuard() {
    if (!pool) return;
    for (int k = 0; k < kMaxParts; ++k) {
      if (!forked[k]) continue;
      if (cudaEventRecord(pool->done[k], pool->s[k]) == cudaSuccess) cudaStreamWaitEvent(stream, pool->done[k], 0);
    }
  }
};

// per-thread reusable host staging (no allocation on the steady-state call path)
struct HostStage {
  std::vector<MemberDesc> desc;
  std::vector<uint64_t> weight;
};
HostStage& hostStage() {
  static thread_local HostStage h;
  return h;
}

// K2 for one data kind: variant 0 = canonical (ordered, packed table), 1 = fast + packed table,
// 2 = fast + wide table.
template <int KIND>
struct K2Launcher {
  static int residentPerSm(int variant, uint32_t W, size_t smemBytes, int* out) {
    const int threads = (int)(W * 32), maxSmem = 200 * 1024;
    if (variant == 0) return dgb::residentPerSm<encodeKernel<KIND>>(threads, smemBytes, maxSmem, out);
    if (variant == 1) return dgb::residentPerSm<encodeKernelFast<false, KIND>>(threads, smemBytes, maxSmem, out);
    return dgb::residentPerSm<encodeKernelFast<true, KIND>>(threads, smemBytes, maxSmem, out);
  }
  static void launch(int variant, uint32_t grid, uint32_t W, size_t smemBytes, cudaStream_t ps, const EncodeScratch& sc,
                     const InlineMembers& im, int pb, bool checksum, uint32_t n, uint32_t totalTickets, uint32_t blockBegin, uint32_t blockEnd,
                     uint32_t slotWords, uint32_t spillWarpBase, uint32_t* outSize_dev) {
    if (variant == 0) {
      encodeKernel<KIND><<<grid, W * 32, smemBytes, ps>>>(sc, pb, checksum, n, totalTickets, outSize_dev);
    } else if (variant == 1) {
      encodeKernelFast<false, KIND><<<grid, W * 32, smemBytes, ps>>>(sc, im, pb, checksum, n, blockBegin, blockEnd, slotWords,
                                                                    spillWarpBase, outSize_dev);
    } else {
      encodeKernelFast<true, KIND><<<grid, W * 32, smemBytes, ps>>>(sc, im, pb, checksum, n, blockBegin, blockEnd, slotWords,
                                                                   spillWarpBase, outSize_dev);
    }
  }
};

#define DGB_BY_KIND(kind, CALL)                             \
  ((kind) == kKindBytes ? K2Launcher<kKindBytes>::CALL      \
   : (kind) == kKindF16 ? K2Launcher<kKindF16>::CALL        \
   : (kind) == kKindBF16 ? K2Launcher<kKindBF16>::CALL      \
                         : K2Launcher<kKindF32>::CALL)

}  // namespace

size_t encodeTempBytes(int kind, uint32_t n, uint32_t maxSize) {
  // worst case over warps-per-CTA choices: tickets with W = 1
  const uint64_t tickets = (uint64_t)n * divUp(maxSize, kBlockBytes);
  if (tickets > 0xffffffffull) return ~size_t(0);
  return planScratch(kind, n, maxSize, (uint32_t)tickets, spillWarpBound(n, tickets)).total + 256;
}

int encodeBatch(int kind, void* temp, size_t tempBytes, int pb, bool checksum, uint32_t n,
                const HostMember* members, const uint32_t* histogram_dev, uint32_t* outSize_dev,
                cudaStream_t stream) {
  if (n == 0) return DGB_OK;
  if (pb < 9 || pb > 11) return DGB_ERR_INVALID_ARG;
  if (kind != kKindBytes && histogram_dev) return DGB_ERR_INVALID_ARG;
  const Options opt = options();  // one snapshot per call
  const uint32_t W = (uint32_t)std::max(1, std::min(opt.encode_warps, 8));  // warps per coder CTA
  const uint32_t elemBytes = kind == kKindF32 ? 4u : (kind == kKindBytes ? 1u : 2u);
  const bool canonical = opt.encode_canonical != 0;
  // staging slot of the fast encoder (spills to global scratch when a block needs more)
  uint32_t slotWords = opt.encode_slot_words > 0 ? (uint32_t)opt.encode_slot_words
                                                 : (kind == kKindBytes ? 2304u : 1536u);
  slotWords = std::max<uint32_t>(roundUp(slotWords, 8u), kEncGroupRows * 32u + 264u);
  slotWords = std::min(slotWords, maxBlockWords(pb));
  const uint32_t slabVecs = (uint32_t)std::max(1, opt.hist_slab_kb) * 1024u / 16u;  // statistics slab

  // ---- member table (host staging) ----
  HostStage& hs = hostStage();
  hs.desc.resize(n);
  MemberDesc* desc = hs.desc.data();
  uint32_t maxSize = 0;
  uint64_t tickets = 0;
  for (uint32_t i = 0; i < n; ++i) {
    const HostMember& hm = members[i];
    if ((hm.size && !hm.in) || !hm.out) return DGB_ERR_INVALID_ARG;
    if (reinterpret_cast<uintptr_t>(hm.out) & 15u) return DGB_ERR_INVALID_ARG;
    if (reinterpret_cast<uintptr_t>(hm.in) & (elemBytes - 1u)) return DGB_ERR_INVALID_ARG;
    // the reference refuses members whose worst-case archive does not fit 32 bits
    // (ans/GpuANSEncode.cu:13-25 CHECK_LE(rawSize, INT32_MAX)): the caller cannot have sized `out`
    if ((kind == kKindBytes ? dgb_ans_max_compressed_size(hm.size) : dgb_float_max_compressed_size(kind, hm.size)) == 0u)
      return DGB_ERR_TOO_LARGE;
    desc[i].in = hm.in;
    desc[i].out = hm.out;
    desc[i].size = hm.size;
    desc[i].work0 = (uint32_t)tickets;
    tickets += ticketsFor(hm.size);
    maxSize = std::max(maxSize, hm.size);
    if (tickets > 0x7fffffffull) return DGB_ERR_TOO_LARGE;
  }
  const uint32_t totalTickets = (uint32_t)tickets;
  const ScratchPlan sp = planScratch(kind, n, maxSize, totalTickets, spillWarpBound(n, tickets));
  if (!temp || tempBytes < sp.total || (reinterpret_cast<uintptr_t>(temp) & 255u))
    return temp && tempBytes >= sp.total ? DGB_ERR_INVALID_ARG : DGB_ERR_TEMP_TOO_SMALL;

  uint8_t* base = static_cast<uint8_t*>(temp);
  EncodeScratch sc;
  sc.members = reinterpret_cast<MemberDesc*>(base + sp.members);
  sc.hist = reinterpret_cast<uint32_t*>(base + sp.hist);
  sc.histDone = reinterpret_cast<uint32_t*>(base + sp.histDone);
  sc.checksum = reinterpret_cast<uint32_t*>(base + sp.checksum);
  sc.ticket = reinterpret_cast<uint32_t*>(base + sp.ticket);
  sc.lookback = reinterpret_cast<unsigned long long*>(base + sp.lookback);
  sc.allocDone = reinterpret_cast<unsigned long long*>(base + sp.allocDone);
  sc.spill = base + sp.spill;
  sc.table = reinterpret_cast<uint4*>(base + sp.table);

  // member table: inside the kernel parameters when it fits (the canonical encoder reads scratch), else one upload
  static thread_local InlineMembers im;
  const bool inlined = opt.inline_members != 0 && n <= kInlineMembers && !canonical;
  im.count = inlined ? n : 0u;
  if (inlined) {
    std::memcpy(im.m, desc, sizeof(MemberDesc) * n);
  } else {
    DGB_CUDA_TRY(cudaMemcpyAsync(sc.members, desc, sizeof(MemberDesc) * n, cudaMemcpyHostToDevice, stream));
  }
  DGB_CUDA_TRY(cudaMemsetAsync(base + sp.zeroBegin, 0, (canonical ? sp.lookbackEnd : sp.zeroEnd) - sp.zeroBegin, stream));

  const int sms = smCount();
  // encoder table format (see EncSym in this file): wide entries for exponent-byte planes
  const bool wideTable = !canonical && opt.encode_wide_table != 0 &&
                         (opt.encode_wide_table > 0 || kind == DGB_BFLOAT16 || kind == DGB_FLOAT32);
  sc.wideTable = wideTable;

  // ---- sub-batches on internal streams (the ordered canonical encoder stays on one) ----
  hs.weight.resize(n);
  uint64_t totalBytes = 0;
  for (uint32_t i = 0; i < n; ++i) { hs.weight[i] = (uint64_t)desc[i].size * elemBytes; totalBytes += hs.weight[i]; }
  // byte inputs measured slightly slower when split (their stats kernel is atomics-bound, not HBM-bound)
  const int parts = canonical ? 1 : autoParts(kind, n, totalBytes);
  uint32_t bounds[kMaxParts + 1];
  splitParts(hs.weight.data(), n, parts, bounds);
  ForkGuard guard;
  StreamPool* pool = nullptr;
  if (parts > 1) {
    int rc = streamPool(&pool);
    if (rc != DGB_OK) return rc;
    DGB_CUDA_TRY(cudaEventRecord(pool->start, stream));
    guard.pool = pool;
    guard.stream = stream;
  }

  // K2 launch configuration (same for every part)
  const size_t smemBytes = (size_t)W * (canonical ? encWarpSmem(pb, kind) : encFastWarpSmem(slotWords, kind));
  // 0: canonical kernel (packed table), 1: fast kernel + packed table, 2: fast kernel + wide table
  const int variant = canonical ? 0 : (wideTable ? 2 : 1);
  int perSm = 1;
  {
    const int rc = DGB_BY_KIND(kind, residentPerSm(variant, W, smemBytes, &perSm));
    if (rc != DGB_OK) return rc;
  }
  const uint64_t resident = (uint64_t)perSm * sms;
  const uint32_t spillWarpsPerPart = sp.spillWarps / (uint32_t)parts;

  for (int part = 0; part < parts; ++part) {
    const uint32_t m0 = bounds[part], m1 = bounds[part + 1];
    if (m1 == m0) continue;
    cudaStream_t ps = stream;
    if (parts > 1) {
      ps = pool->s[part];
      DGB_CUDA_TRY(cudaStreamWaitEvent(ps, pool->start, 0));
      guard.forked[part] = true;
    }
    // ---- K1 ----
    uint32_t partMax = 0;
    for (uint32_t i = m0; i < m1; ++i) partMax = std::max(partMax, desc[i].size);
    const uint64_t maxVecs = ((uint64_t)partMax * elemBytes) / 16u;
    uint32_t gridY = (uint32_t)std::max<uint64_t>(1, (maxVecs + slabVecs - 1) / slabVecs);
    // enough CTAs to fill the machine a few times, never more than the slabs
    const uint32_t wantY = std::max(1u, (uint32_t)(std::max(1, opt.hist_ctas_per_sm) * sms) / (m1 - m0));
    gridY = std::min(gridY, wantY);
    gridY = std::min(gridY, 65535u);
    dim3 grid1(m1 - m0, gridY);
    timerBegin(kSlotStats, ps);
    if (kind == kKindBytes) {
      statsBytesKernel<<<grid1, kStatsThreads, 0, ps>>>(sc, im, histogram_dev, pb, checksum, slabVecs, m0, outSize_dev);
    } else if (kind == kKindF16) {
      statsFloatKernel<DGB_FLOAT16><<<grid1, kStatsThreads, 0, ps>>>(sc, im, pb, checksum, slabVecs, m0, outSize_dev);
    } else if (kind == kKindBF16) {
      statsFloatKernel<DGB_BFLOAT16><<<grid1, kStatsThreads, 0, ps>>>(sc, im, pb, checksum, slabVecs, m0, outSize_dev);
    } else {
      statsFloatKernel<DGB_FLOAT32><<<grid1, kStatsThreads, 0, ps>>>(sc, im, pb, checksum, slabVecs, m0, outSize_dev);
    }
    DGB_CUDA_TRY(cudaGetLastError());
    timerEnd(kSlotStats, ps);

    // ---- K2 ----
    const uint32_t blockBegin = desc[m0].work0;
    const uint32_t blockEnd = m1 < n ? desc[m1].work0 : totalTickets;
    const uint32_t partBlocks = blockEnd - blockBegin;
    if (partBlocks > 0) {
      timerBegin(kSlotEncode, ps);
      uint32_t grid2;
      if (canonical) {
        grid2 = std::min<uint32_t>(divUp(totalTickets, W), (uint32_t)resident);
      } else {
        // one resident wave, every warp gets the same number of blocks (rounds) when the batch is large,
        // so no warp idles at the end waiting for a neighbour's extra block
        const uint64_t rounds = std::max<uint64_t>(1, (partBlocks + resident * W - 1) / (resident * W));
        const uint64_t want = ((uint64_t)partBlocks + W * rounds - 1) / (W * rounds);
        grid2 = (uint32_t)std::max<uint64_t>(1, std::min<uint64_t>(want, resident));
        grid2 = std::max(1u, std::min(grid2, spillWarpsPerPart / W));  // every warp owns a spill slot
      }
      DGB_BY_KIND(kind, launch(variant, grid2, W, smemBytes, ps, sc, im, pb, checksum, n, totalTickets, blockBegin, blockEnd,
                               slotWords, (uint32_t)part * spillWarpsPerPart, outSize_dev));
      DGB_CUDA_TRY(cudaGetLastError());
      timerEnd(kSlotEncode, ps);
    }
  }
  return DGB_OK;  // ~ForkGuard joins the helper streams
}

}  // namespace dgb

// decode.cu -- batched rANS decode (bytes) and fused float decompress
// (fp16/bf16/fp32) for sm_100a.  One launch per call (decodeFusedKernel, further down): a persistent grid
// whose CTAs lease members (header checks and the 2^pb LUT from the archive's own pdf happen inside the
// CTA) and whose warps claim 4 KiB blocks; lane states + compressed words of a block arrive by one TMA
// bulk copy (cp.async.bulk + mbarrier), the 32-lane interleaved rANS decode of ans/GpuANSDecode.cuh:55-217
// runs with table look-ups and the loop-carried refill load in shared memory, and float kinds join the
// decoded byte with the stored byte(s) (cp.async ring) and store the float word in the same loop, at any
// alignment (float/GpuFloatDecompress.cuh:22-179, float/GpuFloatUtils.cuh:100-204 join rules; the
// reference's two-pass path, float/GpuFloatDecompress.cuh:622-694, is not needed).  A batch is never
// cut into sub-batches: the persistent grid already balances the blocks of every member.
#include <algorithm>
#include <cstring>
#include <vector>

#include "common.cuh"

// rows per software-pipelined group and the resident-warp target that caps registers
#ifndef DGB_DECODE_UNROLL
#define DGB_DECODE_UNROLL 8
#endif
#ifndef DGB_DECODE_WARPS_PER_SM
#define DGB_DECODE_WARPS_PER_SM 40
#endif

namespace dgb {

namespace {

struct DecodeScratch {
  MemberDesc* members;   // [n]; work0 = upper bound of the member's block count (host, from capacity)
  uint32_t* next;        // [n] next unclaimed block of the member (zeroed)
  uint32_t* seen;        // [n] 1 once a CTA has reported the member (zeroed)
  uint32_t* checksum;    // [n] checksum of decoded output (use_checksum only; zeroed)
  uint32_t* archiveChecksum;  // [n]
  uint32_t* sizes;       // [n] decoded size in bytes (for the checksum pass)
};

// Where the ANS archive of member `md` starts, and the float-level fields.
struct ArchiveView {
  const uint8_t* ans;      // ANS archive base
  const uint8_t* non;      // float kinds: stored (non-compressed) plane(s)
  uint32_t floatWords;     // float kinds: size field of the float header
  bool ok;
};

template <int KIND>
__device__ __forceinline__ ArchiveView openArchive(const uint8_t* in) {
  ArchiveView v;
  if (KIND == kKindBytes) {
    v.ans = in;
    v.non = nullptr;
    v.floatWords = 0;
    v.ok = true;
  } else {
    // float/GpuFloatUtils.cuh:26-74 GpuFloatHeader
    const uint4 fh = __ldg(reinterpret_cast<const uint4*>(in));
    v.ok = fh.x == kFloatMagicVersion && (int)(fh.z & 0xfu) == KIND;
    v.floatWords = fh.y;
    v.non = in + kFloatHeaderBytes;
    v.ans = v.non + floatNonCompBytes(KIND, fh.y);
  }
  return v;
}

// ---------------------------------------------------------------------------
// Output writers (ans/BatchProvider.cuh:16-37 BatchWriter, float/
// GpuFloatDecompress.cuh:391-486 JoinFloatWriter restated).  A writer is bound
// to one 4 KiB block.  The float kinds need the stored ("non-compressed")
// byte(s) of every element: those are streamed into a small per-warp
// shared-memory ring with cp.async (LDGSTS) -- one 16 B copy per lane covers a
// whole group of 8 rows -- two groups ahead of the row being decoded, so the
// join reads them with an LDS and the HBM latency of the stored plane never
// meets the dependent decode chain (ncu, first version: 46 % of all stall
// samples were long-scoreboard waits on per-row LDG.U8 of these bytes; holding
// them in registers instead made ptxas sink the loads next to their use).
// ---------------------------------------------------------------------------
#ifndef DGB_DEC_GROUP_ROWS
#define DGB_DEC_GROUP_ROWS 16
#endif
constexpr int kGroupRows = DGB_DEC_GROUP_ROWS;  // rows per prefetch group (8 or 16)
constexpr uint32_t kRingSlots = 3;              // groups resident per warp: current + 2 in flight

template <int OFF>
__device__ __forceinline__ uint32_t ldsU16(uint32_t addr) {
  uint32_t v;
  asm volatile("ld.shared.u16 %0, [%1+%2];" : "=r"(v) : "r"(addr), "n"(OFF));
  return v;
}

template <int KIND>
struct RowWriter;

template <>
struct RowWriter<kKindBytes> {
  static constexpr uint32_t kRingSlotBytes = 0;
  uint8_t* out;
  struct Cursor { uint8_t* o; };
  __device__ __forceinline__ void setRing(uint32_t, uint32_t) {}
  __device__ __forceinline__ void setBlock(const ArchiveView&, void* outBase, uint32_t block, uint32_t lane) {
    out = static_cast<uint8_t*>(outBase) + (size_t)block * kBlockBytes + lane;
    __builtin_assume(__isGlobal(out));
  }
  __device__ __forceinline__ Cursor at(uint32_t row, uint32_t) const { return Cursor{out + row * 32u}; }
  __device__ __forceinline__ void issue(uint32_t, uint32_t) const {}
  template <int J>
  __device__ __forceinline__ void write(const Cursor& c, uint32_t entry) const {
    c.o[J * 32] = (uint8_t)entry;
  }
  // rows outside the pipelined groups
  __device__ __forceinline__ void writeSlow(uint32_t row, uint32_t entry) const { out[row * 32u] = (uint8_t)entry; }
};

template <int KIND>
struct RowWriter16 {
  static constexpr uint32_t kRingSlotBytes = kGroupRows * 32;  // one stored byte per element
  uint16_t* out;
  const uint8_t* non;      // this lane's byte of row 0 of the block
  const uint8_t* nonCopy;  // copy source of this lane (lanes 0..15 move 16 B each per group)
  uint32_t ring, lane;
  struct Cursor { uint16_t* o; uint32_t s; };
  __device__ __forceinline__ void setRing(uint32_t ringAddr, uint32_t l) { ring = ringAddr; lane = l; }
  __device__ __forceinline__ void setBlock(const ArchiveView& av, void* outBase, uint32_t block, uint32_t l) {
    out = static_cast<uint16_t*>(outBase) + (size_t)block * kBlockBytes + l;
    non = av.non + (size_t)block * kBlockBytes + l;
    nonCopy = av.non + (size_t)block * kBlockBytes + l * 16u;
    __builtin_assume(__isGlobal(out));
    __builtin_assume(__isGlobal(non));
    __builtin_assume(__isGlobal(nonCopy));
  }
  // cursor of the group starting at `row`, resident in ring slot `slot`
  __device__ __forceinline__ Cursor at(uint32_t row, uint32_t slot) const {
    return Cursor{out + row * 32u, ring + slot * kRingSlotBytes + lane};
  }
  // request rows [row, row + 8) into ring slot `slot`
  __device__ __forceinline__ void issue(uint32_t row, uint32_t slot) const {
    if (lane < (uint32_t)(kGroupRows * 2)) cpAsync16(ring + slot * kRingSlotBytes + lane * 16u, nonCopy + row * 32u);
  }
  static __device__ __forceinline__ uint32_t join(uint32_t entry, uint32_t nc) {
    if (KIND == kKindF16) {
      // float/GpuFloatUtils.cuh:117-119: comp * 256 + nonComp  (bytes: [non, comp])
      return __byte_perm(entry, nc, 0x4404);
    }
    // float/GpuFloatUtils.cuh:149-159: (comp:non) rotated right by one within 16 bits.
    // x = comp<<24 | non<<16 ; (non : x) >> 17 leaves comp<<7 | non>>1 | (non&1)<<15 in the
    // low 16 bits (higher bits are dropped by the 16-bit store)
    return __funnelshift_r(__byte_perm(entry, nc, 0x0444), nc, 17);
  }
  template <int J>
  __device__ __forceinline__ void write(const Cursor& c, uint32_t entry) const {
    c.o[J * 32] = (uint16_t)join(entry, ldsU8<J * 32>(c.s));
  }
  __device__ __forceinline__ void writeSlow(uint32_t row, uint32_t entry) const {
    out[row * 32u] = (uint16_t)join(entry, __ldg(non + row * 32u));
  }
};
template <> struct RowWriter<kKindF16> : RowWriter16<kKindF16> {};
template <> struct RowWriter<kKindBF16> : RowWriter16<kKindBF16> {};

template <>
struct RowWriter<kKindF32> {
  // per group: 8 rows x 64 B of the u16 plane, then 8 rows x 32 B of the u8 plane
  static constexpr uint32_t kRingSlotBytes = kGroupRows * 96;
  uint32_t* out;
  const uint16_t* non2;
  const uint8_t* non1;
  const uint8_t* copy2;
  const uint8_t* copy1;
  uint32_t ring, lane;
  struct Cursor { uint32_t* o; uint32_t s2, s1; };
  __device__ __forceinline__ void setRing(uint32_t ringAddr, uint32_t l) { ring = ringAddr; lane = l; }
  __device__ __forceinline__ void setBlock(const ArchiveView& av, void* outBase, uint32_t block, uint32_t l) {
    out = static_cast<uint32_t*>(outBase) + (size_t)block * kBlockBytes + l;
    const uint8_t* p2 = av.non + 2u * (size_t)block * kBlockBytes;
    const uint8_t* p1 = av.non + 2u * (size_t)roundUp(av.floatWords, 8u) + (size_t)block * kBlockBytes;
    non2 = reinterpret_cast<const uint16_t*>(p2) + l;
    non1 = p1 + l;
    copy2 = p2 + l * 16u;
    copy1 = p1 + l * 16u;
    __builtin_assume(__isGlobal(out));
    __builtin_assume(__isGlobal(non2));
    __builtin_assume(__isGlobal(non1));
    __builtin_assume(__isGlobal(copy2));
    __builtin_assume(__isGlobal(copy1));
  }
  __device__ __forceinline__ Cursor at(uint32_t row, uint32_t slot) const {
    const uint32_t base = ring + slot * kRingSlotBytes;
    return Cursor{out + row * 32u, base + lane * 2u, base + kGroupRows * 64 + lane};
  }
  __device__ __forceinline__ void issue(uint32_t row, uint32_t slot) const {
    const uint32_t base = ring + slot * kRingSlotBytes;
#pragma unroll
    for (int h = 0; h < kGroupRows / 8; ++h)  // 32 lanes x 16 B = 8 rows x 64 B per copy
      cpAsync16(base + h * 512 + lane * 16u, copy2 + row * 64u + h * 512);
    if (lane < (uint32_t)(kGroupRows * 2)) cpAsync16(base + kGroupRows * 64 + lane * 16u, copy1 + row * 32u);
  }
  static __device__ __forceinline__ uint32_t join(uint32_t entry, uint32_t lo, uint32_t hi) {
    // float/GpuFloatUtils.cuh:187-190: (comp << 24 | stored 24 bits) rotated right by one
    const uint32_t v = __byte_perm(lo, __byte_perm(hi, entry, 0x0040), 0x5410);
    return __funnelshift_r(v, v, 1);
  }
  template <int J>
  __device__ __forceinline__ void write(const Cursor& c, uint32_t entry) const {
    c.o[J * 32] = join(entry, ldsU16<J * 64>(c.s2), ldsU8<J * 32>(c.s1));
  }
  __device__ __forceinline__ void writeSlow(uint32_t row, uint32_t entry) const {
    out[row * 32u] = join(entry, __ldg(non2 + row * 32u), __ldg(non1 + row * 32u));
  }
};

// ---------------------------------------------------------------------------
// The compressed word stream of one block, read backwards.  Two flavours so the
// hot loop always knows the address space: staged in shared memory by the TMA
// bulk copy (LDS on the loop-carried path) or straight from global memory.
// ---------------------------------------------------------------------------
struct SmemStream {
  uint32_t addr;  // shared BYTE address one past the last unread word
  __device__ __forceinline__ uint32_t pop(uint32_t back) const {
    uint32_t v;
    asm volatile("ld.shared.u16 %0, [%1];" : "=r"(v) : "r"(addr - 2u * back));
    return v;
  }
  __device__ __forceinline__ void retreat(uint32_t cnt) { addr -= 2u * cnt; }
};
struct GmemStream {
  const uint16_t* p;  // one past the last unread word
  __device__ __forceinline__ uint32_t pop(uint32_t back) const { return __ldg(p - back); }
  __device__ __forceinline__ void retreat(uint32_t cnt) { p -= cnt; }
};

// ---------------------------------------------------------------------------
// Decode LUT, one u32 entry per state residue (never leaves shared memory):
//   [31:20] pdf  [19:8] s-cdf  [7:0] symbol
// (8-byte entries {pdf, (s-cdf) << 8 | symbol} save two ALU ops per row for the unpack, take twice
// the shared memory, and measured slower on every workload.)
// One decode step for a full row (ans/GpuANSDecode.cuh:55-105 restated); the
// returned word has the decoded symbol in its low byte.
// ---------------------------------------------------------------------------
template <int PB>
struct Lut {
  typedef uint32_t Entry;
  static __device__ __forceinline__ Entry make(uint32_t pdf, uint32_t c, uint32_t sym) {
    return (pdf << 20) | (c << 8) | sym;
  }
  static __device__ __forceinline__ uint32_t step(uint32_t& state, const Entry* __restrict__ lut) {
    const uint32_t e = lut[state & ((1u << PB) - 1u)];
    // e >> 8 = pdf * 4096 + (s - cdf): the multiple of pdf is taken back out of the quotient, so the
    // (s - cdf) field needs no mask (all arithmetic mod 2^32); the -4096 folds into the shift (LEA.HI)
    state = (e >> 20) * ((state >> PB) - 4096u) + (e >> 8);
    return e;
  }
};

// refill (ans/GpuANSDecode.cuh:89-101 restated): lanes whose state dropped below 2^15 pop one
// word each, highest lane first
template <typename Stream>
__device__ __forceinline__ void refill(uint32_t& state, Stream& st, uint32_t geMask) {
  const bool rd = state < kStateMin;
  const uint32_t vote = __ballot_sync(0xffffffffu, rd);
  if (rd) state = (state << 16) + st.pop(__popc(vote & geMask));
  st.retreat(__popc(vote));
}
// shared-memory flavour in PTX: one predicate feeds the vote and the state update.  The load itself is NOT
// predicated: a predicated load leaves its destination "maybe written", which ptxas turns into one
// loop-carried register per unrolled row (16 registers of dead values in the round-1 kernel, spills in the
// free-running one).  Lanes that do not refill read at most 64 B below the stream, i.e. inside the slot's
// lane-state area, and drop the value.
template <>
__device__ __forceinline__ void refill<SmemStream>(uint32_t& state, SmemStream& st, uint32_t geMask) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      ".reg .b32 v, t, a, w;\n"
      "setp.lt.u32 p, %0, 32768;\n"
      "vote.sync.ballot.b32 v, p, 0xffffffff;\n"
      "and.b32 t, v, %2;\n"
      "popc.b32 t, t;\n"
      "shl.b32 t, t, 1;\n"
      "sub.u32 a, %1, t;\n"
      "ld.shared.u16 w, [a];\n"  // unpredicated on purpose (see below)
      "@p mad.lo.u32 %0, %0, 65536, w;\n"
      "popc.b32 t, v;\n"
      "shl.b32 t, t, 1;\n"
      "sub.u32 %1, %1, t;\n"
      "}\n"
      : "+r"(state), "+r"(st.addr)
      : "r"(geMask));
}

template <int PB, typename Stream>
__device__ __forceinline__ uint32_t decodeStep(uint32_t& state,
                                               const typename Lut<PB>::Entry* __restrict__ lut,
                                               Stream& st, uint32_t geMask) {
  const uint32_t e = Lut<PB>::step(state, lut);
  refill(state, st, geMask);
  return e;
}

template <int PB, typename Stream>
__device__ __forceinline__ uint32_t decodeStepPartial(bool valid, uint32_t& state,
                                                      const typename Lut<PB>::Entry* __restrict__ lut,
                                                      Stream& st, uint32_t geMask) {
  uint32_t s2 = state;
  const uint32_t e = Lut<PB>::step(s2, lut);
  if (valid) state = s2;
  const bool rd = valid && state < kStateMin;
  const uint32_t vote = __ballot_sync(0xffffffffu, rd);
  if (rd) state = (state << 16) + st.pop(__popc(vote & geMask));
  st.retreat(__popc(vote));
  return e;
}

template <int KIND, int PB, typename Stream, int J>
struct RowGroup {
  typedef RowWriter<KIND> W;
  // rows J-1 .. 0 of the group, highest first (the decoder walks rows backwards)
  static __device__ __forceinline__ void run(uint32_t& state,
                                             const typename Lut<PB>::Entry* __restrict__ lut,
                                             Stream& st, uint32_t geMask, const W& wr,
                                             const typename W::Cursor& c) {
    const uint32_t e = decodeStep<PB>(state, lut, st, geMask);
    wr.template write<J - 1>(c, e);
    RowGroup<KIND, PB, Stream, J - 1>::run(state, lut, st, geMask, wr, c);
  }
};
template <int KIND, int PB, typename Stream>
struct RowGroup<KIND, PB, Stream, 0> {
  typedef RowWriter<KIND> W;
  static __device__ __forceinline__ void run(uint32_t&, const typename Lut<PB>::Entry* __restrict__, Stream&,
                                             uint32_t, const W&, const typename W::Cursor&) {}
};

template <int KIND, int PB, typename Stream>
__device__ __forceinline__ void decodeBlockWarp(uint32_t state, Stream st, uint32_t n,
                                                const typename Lut<PB>::Entry* __restrict__ lut,
                                                const RowWriter<KIND>& wr, uint32_t lane) {
  typedef typename RowWriter<KIND>::Cursor Cursor;
  constexpr int U = kGroupRows;
  typedef RowGroup<KIND, PB, Stream, U> G;
  const uint32_t geMask = laneMaskGe();
  uint32_t row = n >> 5;  // number of full rows; the partial row (if any) has this index
  const uint32_t rem = n & 31u;
  // groups of U full rows are walked from the top: group k covers rows [row0 - U*(k+1), row0 - U*k)
  const uint32_t row0 = row;
  const uint32_t groups = row0 / U;
  // stored bytes of the first two groups are requested before anything else (the barrier: every lane is done
  // reading the ring slots of the previous block)
  __syncwarp();
  if (groups > 0) wr.issue(row0 - U, 0);
  cpAsyncCommit();
  if (groups > 1) wr.issue(row0 - 2 * U, 1);
  cpAsyncCommit();
  if (rem) {
    const bool valid = lane < rem;
    const uint32_t e = decodeStepPartial<PB>(valid, state, lut, st, geMask);
    if (valid) wr.writeSlow(row, e);
  }
  uint32_t slot = 0, slotNext = 2;  // ring slots of group k and of group k + 2
  for (uint32_t k = 0; k < groups; ++k) {
    row -= U;
    cpAsyncWait<1>();  // group k has landed (group k + 1 may still be in flight)
    // one warp barrier does both jobs: every lane sees group k, and every lane is done reading group k - 1,
    // whose ring slot the request below overwrites (three slots: current + two in flight)
    __syncwarp();
    if (k + 2 < groups) wr.issue(row - 2 * U, slotNext);
    cpAsyncCommit();
    const Cursor c = wr.at(row, slot);
    G::run(state, lut, st, geMask, wr, c);
    slot = slot + 1 == kRingSlots ? 0u : slot + 1;
    slotNext = slotNext + 1 == kRingSlots ? 0u : slotNext + 1;
  }
  while (row > 0) {
    --row;
    const uint32_t e = decodeStep<PB>(state, lut, st, geMask);
    wr.writeSlow(row, e);
  }
}

// LUT build from the archive's u16 pdf[256] (ans/GpuANSDecode.cuh:405-476
// restated; runs inside the decode CTA).  blockDim.x == WARPS*32.
template <int PB, int WARPS>
__device__ void buildLut(const uint8_t* __restrict__ ans, typename Lut<PB>::Entry* __restrict__ lut,
                         uint32_t* sPdf, uint32_t* sCdf, uint32_t* sWarp) {
  constexpr int T = WARPS * 32;
  constexpr int PER = (kNumSymbols + T - 1) / T;
  const uint16_t* pdfIn = reinterpret_cast<const uint16_t*>(ans + kAnsHeaderBytes);
  // contiguous PER symbols per thread so one block scan gives the cdf
  uint32_t p[PER];
  uint32_t s = 0;
#pragma unroll
  for (int k = 0; k < PER; ++k) {
    const uint32_t sym = threadIdx.x * PER + k;
    p[k] = sym < kNumSymbols ? (uint32_t)__ldg(pdfIn + sym) : 0u;
    s += p[k];
  }
  uint32_t tot;
  uint32_t c = blockExclusiveScan<T>(s, sWarp, &tot);
#pragma unroll
  for (int k = 0; k < PER; ++k) {
    const uint32_t sym = threadIdx.x * PER + k;
    if (sym < kNumSymbols) { sPdf[sym] = p[k]; sCdf[sym] = c; }
    c += p[k];
  }
  __syncthreads();
  const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31u;
  for (uint32_t sym = warp; sym < kNumSymbols; sym += WARPS) {
    const uint32_t pdf = sPdf[sym], begin = sCdf[sym];
    for (uint32_t j = lane; j < pdf; j += 32u) {
      if (begin + j < (1u << PB)) lut[begin + j] = Lut<PB>::make(pdf, j, sym);
    }
  }
  __syncthreads();
}

// ---------------------------------------------------------------------------
// Single-launch decoder.  One persistent grid, one launch per call.  The host
// knows every member's capacity, hence an upper bound on its 4 KiB block count (work0; at least one
// so that every header is visited), and zeroes one claim counter per member.  A CTA LEASES a
// member: it reads and validates the header(s), builds the decode LUT once, and then each of its
// warps claims blocks of that member one at a time with an atomic (the next claim is issued before
// the current block is decoded, so its latency hides) until none are left; only then do the warps
// meet at a barrier and the CTA moves on to the next member that still has unclaimed blocks,
// starting from its home member.  Several CTAs lease the same member at once, so the work balances
// at block granularity and the kernel has no per-block or per-chunk CTA barrier (a static split of
// the flat blocks over the CTAs left SMs idle for ~15 % of the kernel, ncu r01).  The first CTA to lease a
// member reports outSuccess / outSize (ans/GpuANSDecode.cuh:326-341 semantics); claims past the
// archive's real block count, or of a member that failed, are dropped.
// Measured and rejected (profiles/r02_wall_experiments.txt, step L): a variant without the lease-end
// barrier -- two LUT buffers per CTA, a generation counter, the first warp to run dry builds the next
// LUT alone while the others keep decoding -- was slower on every workload (c3 151.8 vs 143.7 us,
// c2 319 vs 245): a member runs dry for all of its warps within one block time, so they all arrive
// together anyway and then wait for a single-warp LUT build instead of sharing it.
// ---------------------------------------------------------------------------
constexpr uint32_t kNoMember = 0xffffffffu;

template <int KIND, int PB, int WARPS>
__global__ void __launch_bounds__(WARPS * 32, DGB_DECODE_WARPS_PER_SM / WARPS)
decodeFusedKernel(DecodeScratch sc, const __grid_constant__ InlineMembers im, uint32_t n, uint32_t slotWords,
                  uint8_t* __restrict__ outSuccess, uint32_t* __restrict__ outSize, bool wantChecksum) {
  extern __shared__ __align__(128) uint8_t smem[];
  constexpr uint32_t K = 1u << PB;
  typedef typename Lut<PB>::Entry Entry;
  __shared__ __align__(16) Entry lut[K];  // static: constant base address for the hot LDS
  uint32_t* sPdf = reinterpret_cast<uint32_t*>(smem);
  uint32_t* sCdf = sPdf + kNumSymbols;
  uint32_t* sWarp = sCdf + kNumSymbols;           // 32 words
  uint32_t* sMisc = sWarp + 32;                   // 32 words
  unsigned long long* sBar = reinterpret_cast<unsigned long long*>(sMisc + 32);  // [WARPS]
  uint8_t* sRing = reinterpret_cast<uint8_t*>(sBar + ((WARPS + 1) & ~1));  // [WARPS] stored-byte rings
  constexpr uint32_t ringBytes = kRingSlots * RowWriter<KIND>::kRingSlotBytes;
  uint8_t* sSlots = sRing + WARPS * ringBytes;
  const uint32_t slotBytes = 128u + slotWords * 2u;  // lane states + stream

  const uint32_t t = threadIdx.x, lane = t & 31u;
  const uint32_t warp = __shfl_sync(0xffffffffu, t >> 5, 0);
  uint8_t* mySlot = sSlots + (size_t)warp * slotBytes;
  const uint32_t myBar = smemAddr(sBar + warp);
  uint32_t phase = 0;
  if (lane == 0) mbarInit(myBar, 1);
  fenceBarrierInit();
  __syncthreads();

  uint32_t cursor = (uint32_t)((uint64_t)blockIdx.x * n / gridDim.x);  // home member (used by warp 0)

  for (;;) {
    // ---- lease: the first member at or after the cursor of which this CTA can still claim a block
    //      (the claim comes first: a CTA that arrives when others have just taken the last blocks
    //      moves on without reading the header or building the LUT) ----
    if (warp == 0) {
      uint32_t pick = kNoMember, firstBlock = 0, tries = 0;
      while (tries < n) {
        // 32 members at a time
        uint32_t mm = cursor + lane;
        if (mm >= n) mm -= n;
        bool has = false;
        if (tries + lane < n) has = *reinterpret_cast<volatile uint32_t*>(sc.next + mm) < memberWork0(im, sc.members, mm);
        const uint32_t mask = __ballot_sync(0xffffffffu, has);
        if (mask == 0u) {
          tries += 32u;
          cursor = (cursor + 32u) % n;
          continue;
        }
        const uint32_t first = (uint32_t)__ffs((int)mask) - 1u;
        uint32_t cand = cursor + first;
        if (cand >= n) cand -= n;
        uint32_t c = 0;
        if (lane == 0) c = atomicAdd(sc.next + cand, 1u);
        c = __shfl_sync(0xffffffffu, c, 0);
        if (c < memberWork0(im, sc.members, cand)) {
          pick = cand;
          firstBlock = c;
          cursor = cand;
          break;
        }
        tries += first + 1u;  // lost the race for its last block
        cursor = cand + 1 == n ? 0u : cand + 1;
      }
      if (lane == 0) { sMisc[0] = pick; sMisc[1] = firstBlock; }
    }
    __syncthreads();
    const uint32_t m = sMisc[0];
    if (m == kNoMember) break;
    const MemberDesc md = memberAt(im, sc.members, m);
    const uint32_t blocksCap = md.work0;

    // ---- header(s), validity, LUT ----
    const ArchiveView av = openArchive<KIND>(static_cast<const uint8_t*>(md.in));
    bool ok = av.ok;
    uint32_t need = 0, storedChecksum = 0, nb = 0;
    if (ok) {
      const uint4 h0 = __ldg(reinterpret_cast<const uint4*>(av.ans));
      const uint4 h1 = __ldg(reinterpret_cast<const uint4*>(av.ans) + 1);
      nb = h0.y;
      need = h0.z;  // uncompressed bytes == float words for float kinds
      ok = h0.x == kAnsMagicVersion && (int)(h1.x & 0xfu) == PB && nb == divUp(need, kBlockBytes);
      if (KIND != kKindBytes) ok = ok && need == av.floatWords;
      storedChecksum = KIND == kKindBytes ? h1.y : __ldg(reinterpret_cast<const uint32_t*>(md.in) + 3);
    }
    // ans/GpuANSDecode.cuh:326-337: success iff capacity suffices; size reported regardless
    const bool memberOk = ok && md.size >= need;
    if (t == 0 && atomicExch(sc.seen + m, 1u) == 0u) {
      if (outSuccess) outSuccess[m] = memberOk ? 1 : 0;
      if (outSize) outSize[m] = ok ? need : 0u;
      if (wantChecksum) {
        sc.archiveChecksum[m] = storedChecksum;
        sc.sizes[m] = memberOk ? need : 0u;
      }
    }
    const bool work = memberOk && nb > 0;
    if (work) buildLut<PB, WARPS>(av.ans, lut, sPdf, sCdf, sWarp);

    const uint8_t* pStates = av.ans + kAnsHeaderBytes + kAnsPdfBytes;
    const uint2* pBlockWords = reinterpret_cast<const uint2*>(pStates + 128u * (size_t)nb);
    const uint16_t* pData = reinterpret_cast<const uint16_t*>(
        reinterpret_cast<const uint8_t*>(pBlockWords) + 8u * (size_t)roundUp(nb, 2u));
    const bool canStage = (reinterpret_cast<uintptr_t>(av.ans) & 15u) == 0;
    RowWriter<KIND> wr;
    wr.setRing(smemAddr(sRing + warp * ringBytes), lane);

    // ---- every warp claims blocks of the member until none are left ----
    uint32_t block = sMisc[1];  // warp 0 starts with the block claimed with the lease
    if (warp != 0) {
      if (lane == 0) block = atomicAdd(sc.next + m, 1u);
      block = __shfl_sync(0xffffffffu, block, 0);
    }
    while (block < blocksCap) {
      uint32_t nextBlock = 0;
      if (lane == 0) nextBlock = atomicAdd(sc.next + m, 1u);  // in flight while this block is decoded
      if (work && block < nb) {
        const uint2 bw = __ldg(pBlockWords + block);
        const uint32_t blockLen = bw.x >> 16, words = bw.x & 0xffffu;
        const uint16_t* stream = pData + bw.y;
        wr.setBlock(av, md.out, block, lane);
        // two call sites on purpose: each knows the address space of the stream
        if (canStage && words <= slotWords && (bw.y & 7u) == 0u) {
          const uint32_t streamBytes = roundUp(words, 8u) * 2u;
          __syncwarp();
          if (lane == 0) {
            mbarExpectTx(myBar, 128u + streamBytes);
            bulkLoad(smemAddr(mySlot), pStates + 128u * (size_t)block, 128u, myBar);
            if (streamBytes) bulkLoad(smemAddr(mySlot + 128), stream, streamBytes, myBar);
          }
          mbarWait(myBar, phase);
          phase ^= 1u;
          const uint32_t state = reinterpret_cast<const uint32_t*>(mySlot)[lane];
          SmemStream st{smemAddr(mySlot + 128) + 2u * words};
          decodeBlockWarp<KIND, PB>(state, st, blockLen, lut, wr, lane);
        } else {
          const uint32_t state = __ldg(reinterpret_cast<const uint32_t*>(pStates) + block * 32u + lane);
          GmemStream st{stream + words};
          decodeBlockWarp<KIND, PB>(state, st, blockLen, lut, wr, lane);
        }
      }
      block = __shfl_sync(0xffffffffu, nextBlock, 0);
    }
    __syncthreads();  // every warp is done with this member's LUT (and sMisc) before the next lease
  }
}

// XOR checksum of decoded outputs (ans/GpuChecksum.cuh:26-93 semantics: XOR of
// all bytes folded to 8 bits).  grid = (n, Y).
__global__ void __launch_bounds__(256)
checksumKernel(DecodeScratch sc) {
  const uint32_t m = blockIdx.x;
  const uint8_t* p = static_cast<const uint8_t*>(sc.members[m].out);
  const uint32_t size = sc.sizes[m];
  uint32_t x = 0;
  for (uint32_t i = blockIdx.y * blockDim.x + threadIdx.x; i < size; i += gridDim.y * blockDim.x)
    x ^= p[i];
#pragma unroll
  for (int d = 16; d >= 1; d >>= 1) x ^= __shfl_xor_sync(0xffffffffu, x, d);
  if ((threadIdx.x & 31) == 0 && x) atomicXor(sc.checksum + m, x & 0xffu);
}

struct DecodePlan {
  size_t members, next, checksum, archiveChecksum, sizes, total;
};

DecodePlan planDecodeScratch(uint32_t n) {
  DecodePlan p{};
  size_t o = 0;
  p.members = o; o = alignUp256(o + sizeof(MemberDesc) * (size_t)n);
  p.next = o; o = alignUp256(o + 8 * (size_t)n);  // next[n] then seen[n]
  p.checksum = o; o = alignUp256(o + 4 * (size_t)n);
  p.archiveChecksum = o; o = alignUp256(o + 4 * (size_t)n);
  p.sizes = o; o = alignUp256(o + 4 * (size_t)n);
  p.total = o;
  return p;
}

// member table of the call in flight on this thread (decodeBatch fills it; count == 0: table in scratch)
InlineMembers& decodeInline() {
  static thread_local InlineMembers im;
  return im;
}

template <int KIND, int PB, int WARPS>
int launchDecodeFusedW(const DecodeScratch& sc, uint32_t n, uint64_t totalChunks,
                       uint32_t slotWordsOpt, uint8_t* outSuccess, uint32_t* outSize, bool checksum,
                       cudaStream_t stream) {
  // staging slot per warp: worst case for raw bytes; float kinds code exponent-like bytes that
  // compress well, so a smaller slot (more resident warps) covers them and rare larger blocks
  // take the direct-from-global path inside the kernel
  uint32_t slotWords = slotWordsOpt > 0 ? slotWordsOpt : (KIND == kKindBytes ? maxBlockWords(PB) : 1536u);
  slotWords = std::min(roundUp(slotWords, 8u), maxBlockWords(PB));
  const size_t smemBytes = (2 * kNumSymbols + 64) * 4 + ((WARPS + 1) & ~1) * 8 +
                           (size_t)WARPS * kRingSlots * RowWriter<KIND>::kRingSlotBytes +
                           (size_t)WARPS * (128u + slotWords * 2u);
  int perSm = 1;
  const int rc = residentPerSm<decodeFusedKernel<KIND, PB, WARPS>>(WARPS * 32, smemBytes, 160 * 1024, &perSm);
  if (rc != DGB_OK) return rc;
  const uint64_t resident = (uint64_t)perSm * smCount();
  const uint32_t grid = (uint32_t)std::max<uint64_t>(1, std::min<uint64_t>(resident, totalChunks));
  timerBegin(kSlotDecode, stream);
  decodeFusedKernel<KIND, PB, WARPS><<<grid, WARPS * 32, smemBytes, stream>>>(sc, decodeInline(), n, slotWords, outSuccess, outSize, checksum);
  DGB_CUDA_TRY(cudaGetLastError());
  timerEnd(kSlotDecode, stream);
  return DGB_OK;
}

template <int KIND, int PB>
int launchDecodeFused(const DecodeScratch& sc, uint32_t n, uint64_t totalChunks,
                      uint32_t slotWordsOpt, uint8_t* outSuccess, uint32_t* outSize, bool checksum,
                      cudaStream_t stream) {
  // warps per CTA = warps that share one LUT and meet at the barrier when a lease ends.  Float kinds: 8 (4 and
  // 10 / 20 measured: c3 146.5 / 142.1 / 151.2 us against 143.3).  Byte archives need the worst-case staging slot
  // (5.1 KiB per warp), which caps 8-warp CTAs at 32 resident warps per SM; 20-warp CTAs reach 40 (c2: 242 ->
  // 233.5 us) -- used when the members are long enough to keep 20 warps busy through a lease.  Option values
  // other than 20 (byte archives) select 8.
  int w = options().decode_warps;
  // (at 11 bits the LUT is 8 KiB and the slot 5.6 KiB per warp: a 20-warp CTA needs 126 KiB and fits once per
  // SM -- bench detail c2p11 fell from 884 to 800 GB/s -- so the wide CTA is used up to 10 bits only)
  if (w == 0) w = (KIND == kKindBytes && PB <= 10 && totalChunks * 8u >= 160ull * n) ? 20 : 8;
  if constexpr (KIND == kKindBytes) {
    if (w == 20)
      return launchDecodeFusedW<KIND, PB, 20>(sc, n, totalChunks, slotWordsOpt, outSuccess, outSize, checksum, stream);
  }
  return launchDecodeFusedW<KIND, PB, 8>(sc, n, totalChunks, slotWordsOpt, outSuccess, outSize, checksum, stream);
}

template <int KIND>
int decodeFusedKind(const DecodeScratch& sc, int pb, uint32_t n, uint64_t totalChunks,
                    uint32_t slotWordsOpt, uint8_t* outSuccess, uint32_t* outSize, bool checksum,
                    cudaStream_t stream) {
  switch (pb) {
    case 9: return launchDecodeFused<KIND, 9>(sc, n, totalChunks, slotWordsOpt, outSuccess, outSize, checksum, stream);
    case 10: return launchDecodeFused<KIND, 10>(sc, n, totalChunks, slotWordsOpt, outSuccess, outSize, checksum, stream);
    case 11: return launchDecodeFused<KIND, 11>(sc, n, totalChunks, slotWordsOpt, outSuccess, outSize, checksum, stream);
    default: return DGB_ERR_INVALID_ARG;
  }
}

}  // namespace

size_t decodeTempBytes(int /*kind*/, uint32_t n) { return planDecodeScratch(n).total + 256; }

int decodeBatch(int kind, void* temp, size_t tempBytes, int pb, bool checksum, uint32_t n,
                const HostMember* members, uint8_t* outSuccess_dev, uint32_t* outSize_dev,
                uint8_t* mismatchHost, cudaStream_t stream) {
  if (n == 0) return DGB_OK;
  if (pb < 9 || pb > 11) return DGB_ERR_INVALID_ARG;
  const DecodePlan dp = planDecodeScratch(n);
  if (!temp || tempBytes < dp.total) return DGB_ERR_TEMP_TOO_SMALL;
  if (reinterpret_cast<uintptr_t>(temp) & 255u) return DGB_ERR_INVALID_ARG;

  const Options opt = options();  // one snapshot per call
  static thread_local std::vector<MemberDesc> descStage;  // reused: no allocation on the steady-state path
  descStage.resize(n);
  MemberDesc* desc = descStage.data();
  const uint32_t wordBytes = kind == kKindF32 ? 4u : (kind == kKindBytes ? 1u : 2u);
  uint64_t totalChunks = 0;
  for (uint32_t i = 0; i < n; ++i) {
    if (!members[i].in || (members[i].size && !members[i].out)) return DGB_ERR_INVALID_ARG;
    // headers are read as 16 B vectors; the reference imposes the same alignment
    if (reinterpret_cast<uintptr_t>(members[i].in) & 15u) return DGB_ERR_INVALID_ARG;
    if (reinterpret_cast<uintptr_t>(members[i].out) & (wordBytes - 1u)) return DGB_ERR_INVALID_ARG;
    desc[i].in = members[i].in;
    desc[i].out = members[i].out;
    desc[i].size = members[i].size;  // capacity
    // block count bound from the capacity (>= 1: every header is visited once)
    const uint32_t blocks = std::max(1u, divUp(members[i].size, kBlockBytes));
    desc[i].work0 = blocks;
    totalChunks += divUp(blocks, 8u);
  }
  uint8_t* base = static_cast<uint8_t*>(temp);
  DecodeScratch sc;
  sc.members = reinterpret_cast<MemberDesc*>(base + dp.members);
  sc.next = reinterpret_cast<uint32_t*>(base + dp.next);
  sc.seen = sc.next + n;
  sc.checksum = reinterpret_cast<uint32_t*>(base + dp.checksum);
  sc.archiveChecksum = reinterpret_cast<uint32_t*>(base + dp.archiveChecksum);
  sc.sizes = reinterpret_cast<uint32_t*>(base + dp.sizes);
  // member table: inside the kernel parameters when it fits (the checksum pass reads it from scratch)
  InlineMembers& im = decodeInline();
  const bool inlined = opt.inline_members != 0 && !checksum && n <= kInlineMembers;
  im.count = inlined ? n : 0u;
  if (inlined) {
    std::memcpy(im.m, desc, sizeof(MemberDesc) * n);
  } else {
    DGB_CUDA_TRY(cudaMemcpyAsync(sc.members, desc, sizeof(MemberDesc) * n, cudaMemcpyHostToDevice, stream));
  }
  if (checksum) DGB_CUDA_TRY(cudaMemsetAsync(sc.checksum, 0, 4 * (size_t)n, stream));

  DGB_CUDA_TRY(cudaMemsetAsync(sc.next, 0, 8 * (size_t)n, stream));
  const uint32_t slotOpt = opt.decode_slot_words > 0 ? (uint32_t)opt.decode_slot_words : 0u;
  int rc;
  switch (kind) {
    case kKindBytes: rc = decodeFusedKind<kKindBytes>(sc, pb, n, totalChunks, slotOpt, outSuccess_dev, outSize_dev, checksum, stream); break;
    case kKindF16: rc = decodeFusedKind<kKindF16>(sc, pb, n, totalChunks, slotOpt, outSuccess_dev, outSize_dev, checksum, stream); break;
    case kKindBF16: rc = decodeFusedKind<kKindBF16>(sc, pb, n, totalChunks, slotOpt, outSuccess_dev, outSize_dev, checksum, stream); break;
    case kKindF32: rc = decodeFusedKind<kKindF32>(sc, pb, n, totalChunks, slotOpt, outSuccess_dev, outSize_dev, checksum, stream); break;
    default: return DGB_ERR_INVALID_ARG;
  }
  if (rc != DGB_OK) return rc;

  if (checksum) {
    // ans/GpuANSDecode.cuh:555-591 / float/GpuFloatDecompress.cuh:698-733: checksum the
    // output, compare with the archive's on the host (this path synchronises).
    // Float kinds: the checksum covers the first `size` BYTES (SURVEY A.6/B6); sc.sizes holds
    // the word count, which is exactly that byte count.
    const int sms = smCount();
    dim3 grid(n, std::max(1, std::min(64, 4 * sms / (int)std::max(1u, n))));
    checksumKernel<<<grid, 256, 0, stream>>>(sc);
    DGB_CUDA_TRY(cudaGetLastError());
    std::vector<uint32_t> got(n), want(n), sizes(n);
    DGB_CUDA_TRY(cudaMemcpyAsync(got.data(), sc.checksum, 4 * (size_t)n, cudaMemcpyDeviceToHost, stream));
    DGB_CUDA_TRY(cudaMemcpyAsync(want.data(), sc.archiveChecksum, 4 * (size_t)n, cudaMemcpyDeviceToHost, stream));
    DGB_CUDA_TRY(cudaMemcpyAsync(sizes.data(), sc.sizes, 4 * (size_t)n, cudaMemcpyDeviceToHost, stream));
    DGB_CUDA_TRY(cudaStreamSynchronize(stream));
    bool bad = false;
    for (uint32_t i = 0; i < n; ++i) {
      // members that were skipped (capacity / bad header) are reported through outSuccess
      const bool mm = sizes[i] != 0 && got[i] != want[i];
      if (mismatchHost) mismatchHost[i] = mm ? 1 : 0;
      bad = bad || mm;
    }
    if (bad) return DGB_ERR_CHECKSUM;
  }
  return DGB_OK;
}

// ---------------------------------------------------------------------------
// Header queries (ans/GpuANSInfo.cuh:16-37, float/GpuFloatInfo.cuh:19-41)
// ---------------------------------------------------------------------------
namespace {
__global__ void infoKernel(int kind, const void* const* in, uint32_t n, uint32_t* outSizes,
                           uint32_t* outTypes, uint32_t* outChecksum) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const uint32_t* h = static_cast<const uint32_t*>(in[i]);
  if (kind == kKindBytes) {
    const bool ok = h[0] == kAnsMagicVersion;
    if (outSizes) outSizes[i] = ok ? h[2] : 0u;  // UNCOMPRESSED bytes (ans/GpuANSInfo.cuh:27-29)
    if (outChecksum) outChecksum[i] = ok ? h[5] : 0u;
  } else {
    const bool ok = h[0] == kFloatMagicVersion;
    if (outSizes) outSizes[i] = ok ? h[1] : 0u;  // float words
    if (outTypes) outTypes[i] = ok ? (h[2] & 0xfu) : 0u;
    if (outChecksum) outChecksum[i] = ok ? h[3] : 0u;
  }
}
}  // namespace

// ---------------------------------------------------------------------------
// Archive mover: copies each archive EXACTLY as long as its own header says (float header + stored planes +
// ANS header .. data section), never the padded row it sits in.  Meant for sources in peer memory
// (NVLink): the sizes never travel to the host, every thread keeps four 16 B loads in flight, and a
// small persistent grid (option "pull_ctas") saturates the link while the decode kernel of the
// previous group owns the rest of the SMs.  An archive with a bad header is copied as its first 32
// bytes, so the decoder that follows reports it; one that exceeds the destination capacity is cut
// (the decoder then fails its bounds checks on the member, never reads past the row).
// ---------------------------------------------------------------------------
namespace {
__device__ __forceinline__ uint4 ldgNc(const uint4* p) {
  uint4 v;
  asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(p));
  return v;
}
constexpr uint32_t kPullThreads = 512;
constexpr uint32_t kPullChunkVecs = 4096;  // 64 KiB work units

__device__ __forceinline__ uint32_t archiveBytes(int kind, const uint8_t* a) {
  uint32_t extra = 0;
  if (kind != kKindBytes) {
    const uint4 fh = __ldg(reinterpret_cast<const uint4*>(a));
    if (fh.x != kFloatMagicVersion) return 32u;
    extra = kFloatHeaderBytes + floatNonCompBytes(kind, fh.y);
  }
  const uint4 h = __ldg(reinterpret_cast<const uint4*>(a + extra));
  if (h.x != kAnsMagicVersion) return extra + 32u;
  const uint64_t total = (uint64_t)extra + ansOverhead(h.y) + 2ull * h.w;
  return total > 0xfffffff0ull ? 32u : (uint32_t)total;
}

__global__ void __launch_bounds__(kPullThreads)
pullArchivesKernel(const __grid_constant__ InlineMembers im, int kind, uint32_t* __restrict__ outBytes) {
  __shared__ uint32_t sFirst[kInlineMembers + 1];  // first chunk of member i
  __shared__ uint32_t sBytes[kInlineMembers];
  const uint32_t t = threadIdx.x, n = im.count;
  if (t < n) {
    const uint32_t want = archiveBytes(kind, static_cast<const uint8_t*>(im.m[t].in));
    const uint32_t b = min(want, im.m[t].size & ~15u);
    sBytes[t] = b;
    if (outBytes && blockIdx.x == 0) outBytes[t] = want;
  }
  __syncthreads();
  if (t == 0) {
    uint32_t c = 0;
    for (uint32_t i = 0; i < n; ++i) { sFirst[i] = c; c += divUp(sBytes[i] / 16u, kPullChunkVecs); }
    sFirst[n] = c;
  }
  __syncthreads();
  const uint32_t total = sFirst[n];
  uint32_t m = 0;
  for (uint32_t c = blockIdx.x; c < total; c += gridDim.x) {
    while (sFirst[m + 1] <= c) ++m;
    const uint32_t v0 = (c - sFirst[m]) * kPullChunkVecs;
    const uint32_t v1 = min(sBytes[m] / 16u, v0 + kPullChunkVecs);
    const uint4* __restrict__ src = static_cast<const uint4*>(im.m[m].in);
    uint4* __restrict__ dst = static_cast<uint4*>(im.m[m].out);
    uint32_t v = v0 + t;
    for (; v + 3u * kPullThreads < v1; v += 4u * kPullThreads) {
      const uint4 a = ldgNc(src + v), b = ldgNc(src + v + kPullThreads), cc = ldgNc(src + v + 2u * kPullThreads),
                  d = ldgNc(src + v + 3u * kPullThreads);
      dst[v] = a; dst[v + kPullThreads] = b; dst[v + 2u * kPullThreads] = cc; dst[v + 3u * kPullThreads] = d;
    }
    for (; v < v1; v += kPullThreads) dst[v] = ldgNc(src + v);
  }
}
}  // namespace

int pullArchives(int kind, uint32_t n, const void* const* src, void* const* dst, const uint32_t* capacity,
                 uint32_t* outBytes_dev, cudaStream_t stream) {
  if (n == 0) return DGB_OK;
  if (!src || !dst || !capacity) return DGB_ERR_INVALID_ARG;
  const int ctas = std::max(1, options().pull_ctas);
  static thread_local InlineMembers im;
  for (uint32_t i0 = 0; i0 < n; i0 += kInlineMembers) {
    const uint32_t k = std::min(kInlineMembers, n - i0);
    im.count = k;
    for (uint32_t i = 0; i < k; ++i) {
      if (!src[i0 + i] || !dst[i0 + i]) return DGB_ERR_INVALID_ARG;
      if ((reinterpret_cast<uintptr_t>(src[i0 + i]) | reinterpret_cast<uintptr_t>(dst[i0 + i])) & 15u) return DGB_ERR_INVALID_ARG;
      im.m[i].in = src[i0 + i];
      im.m[i].out = dst[i0 + i];
      im.m[i].size = capacity[i0 + i];
      im.m[i].work0 = 0;
    }
    timerBegin(kSlotPull, stream);
    pullArchivesKernel<<<ctas, kPullThreads, 0, stream>>>(im, kind, outBytes_dev ? outBytes_dev + i0 : nullptr);
    DGB_CUDA_TRY(cudaGetLastError());
    timerEnd(kSlotPull, stream);
  }
  return DGB_OK;
}

int getInfo(int kind, void* temp, size_t tempBytes, const void* const* in, bool inIsDevice,
            uint32_t n, uint32_t* outSizes, uint32_t* outTypes, uint32_t* outChecksum,
            cudaStream_t stream) {
  if (n == 0) return DGB_OK;
  if (!in) return DGB_ERR_INVALID_ARG;
  const void* const* in_dev = in;
  if (!inIsDevice) {
    if (!temp || tempBytes < sizeof(void*) * (size_t)n) return DGB_ERR_TEMP_TOO_SMALL;
    DGB_CUDA_TRY(cudaMemcpyAsync(temp, in, sizeof(void*) * (size_t)n, cudaMemcpyHostToDevice, stream));
    in_dev = static_cast<const void* const*>(temp);
  }
  infoKernel<<<divUp(n, 128), 128, 0, stream>>>(kind, in_dev, n, outSizes, outTypes, outChecksum);
  DGB_CUDA_TRY(cudaGetLastError());
  return DGB_OK;
}

}  // namespace dgb

/*
 * dietgpu_oracle.c -- TEST INFRASTRUCTURE ONLY.
 *
 * A plain-C, CPU restatement of the DietGPU batched byte-rANS codec and the
 * fp16/bf16/fp32 float codec built on it.  It exists to (1) check the CUDA
 * product path bit-for-bit in tests/, __graft_entry__.smoke() and (2) serve as
 * the `cpu_baseline` leg of bench.py.  NOTHING in dietgpu_b200/ (the product)
 * may link, import or call this file; the product path fails loudly when its
 * CUDA library is missing instead of falling back here.
 *
 * Parity pin: the restatement is checked (tests/test_oracle.py) against the
 * reference's own known-answer tests (ANSStatisticsTest.cu:127-167) and against
 * archives written by the reference itself, compiled for sm_100a
 * (tests/golden/ref_golden.npz, tests/test_reference_parity.py).
 *
 * Every function cites the reference file:line (relative to
 * /root/reference/dietgpu/) whose behaviour it restates.  The text below is a
 * scalar re-derivation of those algorithms, not a copy of the CUDA sources.
 */
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

#ifdef _OPENMP
#include <omp.h>
#endif

#define DGO_BLOCK 4096u      /* ans/GpuANSUtils.cuh:37  kDefaultBlockSize          */
#define DGO_LANES 32u        /* one warp = 32 interleaved rANS states              */
#define DGO_STATE_MIN 32768u /* ans/GpuANSUtils.cuh:46-49 kANSStartState/MinState */
#define DGO_ANS_MAGIC 0xd00du
#define DGO_FLOAT_MAGIC 0xf00fu
#define DGO_VERSION 1u

enum {
  DGO_OK = 0,
  DGO_ERR_BAD_MAGIC = 1,
  DGO_ERR_BAD_PROBBITS = 2,
  DGO_ERR_CAPACITY = 3,
  DGO_ERR_CHECKSUM = 4,
  DGO_ERR_BAD_FLOAT_TYPE = 5,
  DGO_ERR_CORRUPT = 6,
};

enum { DGO_F16 = 1, DGO_BF16 = 2, DGO_F32 = 3 }; /* float/GpuFloatCodec.h:18-23 */

static uint32_t div_up(uint32_t a, uint32_t b) { return (a + b - 1) / b; }
static uint32_t round_up(uint32_t a, uint32_t b) { return div_up(a, b) * b; }

static void put32(uint8_t* p, uint32_t v) { memcpy(p, &v, 4); }
static uint32_t get32(const uint8_t* p) { uint32_t v; memcpy(&v, p, 4); return v; }
static void put16(uint8_t* p, uint16_t v) { memcpy(p, &v, 2); }
static uint16_t get16(const uint8_t* p) { uint16_t v; memcpy(&v, p, 2); return v; }

/* ---------------------------------------------------------------- sizes -- */

/* ans/GpuANSUtils.cuh:68-81 ANSCoalescedHeader::getCompressedOverhead */
uint32_t dgo_ans_overhead(uint32_t num_blocks) {
  return 32u + 2u * 256u + 128u * num_blocks + 8u * round_up(num_blocks, 2u);
}

/* ans/GpuANSEncode.cu:13-25 getMaxCompressedSize, incl. its quirk of charging
 * the header overhead of a constant 4096 blocks (SURVEY B2). */
uint32_t dgo_ans_max_compressed_size(uint32_t bytes) {
  uint64_t raw = dgo_ans_overhead(DGO_BLOCK);
  raw += (uint64_t)round_up(DGO_BLOCK + DGO_BLOCK / 4u, 16u) * div_up(bytes, DGO_BLOCK);
  raw = (raw + 15u) / 16u * 16u;
  return (uint32_t)raw;
}

/* float/GpuFloatUtils.cuh:123-127,163-167,194-203 getUncompDataSize */
uint32_t dgo_float_noncomp_bytes(int ft, uint32_t n) {
  if (ft == DGO_F32) return 2u * round_up(n, 8u) + round_up(n, 16u);
  return round_up(n, 16u);
}

/* float/GpuFloatCompress.cu:23-45 getMaxFloatCompressedSize */
uint32_t dgo_float_max_compressed_size(int ft, uint32_t n) {
  return 16u + dgo_ans_max_compressed_size(n) + dgo_float_noncomp_bytes(ft, n);
}

/* ----------------------------------------------------------- statistics -- */

/* ans/GpuANSStatistics.cuh:21-134 (what histogramBatch computes) */
void dgo_histogram(const uint8_t* in, uint32_t n, uint32_t hist[256]) {
  memset(hist, 0, 256 * sizeof(uint32_t));
  for (uint32_t i = 0; i < n; ++i) hist[in[i]]++;
}

/* ans/GpuChecksum.cuh:26-93: XOR of every byte, an 8-bit value in a u32 */
uint32_t dgo_checksum(const uint8_t* in, uint32_t n) {
  uint8_t c = 0;
  for (uint32_t i = 0; i < n; ++i) c ^= in[i];
  return c;
}

static int cmp_desc_u32(const void* a, const void* b) {
  uint32_t x = *(const uint32_t*)a, y = *(const uint32_t*)b;
  return x < y ? 1 : (x > y ? -1 : 0);
}

/* ans/GpuANSStatistics.cuh:178-341 normalizeProbabilitiesFromHistogram.
 * Produces pdf[256] summing to 2^pb (for total > 0). */
void dgo_normalize(const uint32_t hist[256], uint32_t total, int pb, uint32_t pdf[256]) {
  const uint32_t K = 1u << pb;
  uint32_t key[256];
  int32_t sum = 0;
  memset(pdf, 0, 256 * sizeof(uint32_t));
  if (total == 0) return; /* :192-195 */

  for (uint32_t s = 0; s < 256; ++s) {
    /* :215 fp32 convert, IEEE fp32 divide, multiply by 2^pb, truncate */
    volatile float ratio = (float)hist[s] / (float)total;
    volatile float scaled = (float)K * ratio;
    uint32_t q = (uint32_t)scaled;
    if (hist[s] > 0 && q == 0) q = 1; /* :218 */
    sum += (int32_t)q;
    key[s] = (q << 16) | s; /* :234 */
  }
  qsort(key, 256, sizeof(uint32_t), cmp_desc_u32); /* :241 SortDescending */

  uint32_t q[256], sym[256];
  for (uint32_t r = 0; r < 256; ++r) { sym[r] = key[r] & 0xffffu; q[r] = key[r] >> 16; }

  int32_t diff = (int32_t)K - sum; /* :256 */
  if (diff > 0) {
    /* :258-273 -- +1 to every entry whose SYMBOL ID is < min(diff,256),
     * repeated until diff is exhausted (SURVEY B1: ids, not ranks) */
    while (diff > 0) {
      int32_t it = diff < 256 ? diff : 256;
      for (uint32_t r = 0; r < 256; ++r)
        if ((int32_t)sym[r] < it) q[r] += 1;
      diff -= it;
    }
  } else if (diff < 0) {
    /* :274-315 -- -1 from the smallest entries that are still > 1, by rank */
    diff = -diff;
    while (diff > 0) {
      int32_t g = 0;
      for (uint32_t r = 0; r < 256; ++r) g += (q[r] > 1);
      int32_t it = diff < g ? diff : g;
      if (it <= 0) break; /* reference asserts; cannot happen for valid input */
      for (int32_t r = g - it; r < g; ++r) q[r] -= 1;
      diff -= it;
    }
  }
  for (uint32_t r = 0; r < 256; ++r) pdf[sym[r]] = q[r]; /* :318-323 */
}

static void cdf_from_pdf(const uint32_t pdf[256], uint32_t cdf[256]) {
  uint32_t acc = 0; /* ans/GpuANSStatistics.cuh:336-341 exclusive scan */
  for (uint32_t s = 0; s < 256; ++s) { cdf[s] = acc; acc += pdf[s]; }
}

/* ------------------------------------------------------- block encoding -- */

/* ans/GpuANSEncode.cuh:49-211: one 32-lane interleaved rANS block.
 * Lane l of row r owns byte r+l; per row, lanes emit in ascending lane order,
 * then update.  Returns the number of u16 words written to w. */
static uint32_t encode_block(const uint8_t* in, uint32_t n, int pb,
                             const uint32_t pdf[256], const uint32_t cdf[256],
                             uint32_t state[DGO_LANES], uint16_t* w) {
  const uint32_t K = 1u << pb;
  uint32_t cnt = 0;
  for (uint32_t l = 0; l < DGO_LANES; ++l) state[l] = DGO_STATE_MIN;
  for (uint32_t r = 0; r < n; r += DGO_LANES) {
    uint32_t lanes = n - r < DGO_LANES ? n - r : DGO_LANES;
    for (uint32_t l = 0; l < lanes; ++l) {
      uint32_t s = in[r + l], p = pdf[s], x = state[l];
      if (x >= (p << (31 - pb))) { /* :63-75 renormalise */
        w[cnt++] = (uint16_t)(x & 0xffffu);
        x >>= 16;
      }
      state[l] = (x / p) * K + (x % p) + cdf[s]; /* :79-86 */
    }
  }
  return cnt;
}

/* ans/GpuANSDecode.cuh:55-217,274-297: inverse of encode_block.  Rows are
 * visited last to first; per row every lane decodes, then lanes refill in
 * DESCENDING lane order from the end of w. */
static int decode_block(const uint32_t state_in[DGO_LANES], const uint16_t* w,
                        uint32_t nwords, uint32_t n, int pb,
                        const uint32_t* lut /* 2^pb entries */, uint8_t* out) {
  const uint32_t mask = (1u << pb) - 1u;
  uint32_t x[DGO_LANES];
  uint32_t pos = nwords;
  memcpy(x, state_in, sizeof(x));
  uint32_t last_row = (n - 1) / DGO_LANES * DGO_LANES;
  for (int64_t r = last_row; r >= 0; r -= DGO_LANES) {
    uint32_t lanes = n - (uint32_t)r < DGO_LANES ? n - (uint32_t)r : DGO_LANES;
    for (uint32_t l = 0; l < lanes; ++l) {
      uint32_t e = lut[x[l] & mask]; /* :34-53 [31:20] s-cdf [19:8] pdf [7:0] sym */
      out[r + l] = (uint8_t)(e & 0xffu);
      x[l] = ((e >> 8) & 0xfffu) * (x[l] >> pb) + (e >> 20);
    }
    for (int32_t l = (int32_t)lanes - 1; l >= 0; --l) {
      if (x[l] < DGO_STATE_MIN) {
        if (pos == 0) return DGO_ERR_CORRUPT;
        x[l] = (x[l] << 16) + w[--pos];
      }
    }
  }
  if (pos != 0) return DGO_ERR_CORRUPT;
  for (uint32_t l = 0; l < DGO_LANES; ++l)
    if (x[l] != DGO_STATE_MIN) return DGO_ERR_CORRUPT;
  return DGO_OK;
}

/* ---------------------------------------------------------- ANS archive -- */

/*
 * ans/GpuANSEncode.cuh:515-628 + ans/GpuANSUtils.cuh:67-227 archive layout:
 *   [0,32) header | [32,544) u16 pdf[256] | 128*nb warp states |
 *   8*roundUp(nb,2) blockWords | per-block u16 streams padded to 16 B.
 * Bits the reference leaves undefined (SURVEY B3) are written as zero.
 * hist_opt may be NULL (histogram computed here) or a caller histogram.
 * Returns the archive size in bytes.  Blocks are encoded in parallel when
 * built with OpenMP (that is the multi-core CPU baseline of bench.py).
 */
uint32_t dgo_ans_encode(const uint8_t* in, uint32_t n, int pb, int use_checksum,
                        const uint32_t* hist_opt, uint8_t* out) {
  uint32_t hist[256], pdf[256], cdf[256];
  uint32_t nb = div_up(n, DGO_BLOCK);
  if (hist_opt) memcpy(hist, hist_opt, sizeof(hist)); else dgo_histogram(in, n, hist);
  dgo_normalize(hist, n, pb, pdf);
  cdf_from_pdf(pdf, cdf);

  uint8_t* p_pdf = out + 32;
  uint8_t* p_states = p_pdf + 512;
  uint8_t* p_bw = p_states + 128u * nb;
  uint8_t* p_data = p_bw + 8u * round_up(nb, 2u);

  for (uint32_t s = 0; s < 256; ++s) put16(p_pdf + 2 * s, (uint16_t)pdf[s]);
  if (nb & 1u) memset(p_bw + 8u * nb, 0, 8);

  /* worst case pb bits per symbol -> 4096*pb/16 words; pad for 16 B rounding */
  const uint32_t slot_words = DGO_BLOCK * 11u / 16u + 8u;
  uint16_t* slots = nb ? (uint16_t*)malloc((size_t)nb * slot_words * 2u) : NULL;
  uint32_t* words = nb ? (uint32_t*)malloc((size_t)nb * 4u) : NULL;

#pragma omp parallel for schedule(dynamic, 16)
  for (int64_t b = 0; b < (int64_t)nb; ++b) {
    uint32_t st[DGO_LANES];
    uint32_t start = (uint32_t)b * DGO_BLOCK;
    uint32_t len = n - start < DGO_BLOCK ? n - start : DGO_BLOCK;
    words[b] = encode_block(in + start, len, pb, pdf, cdf, st, slots + (size_t)b * slot_words);
    memcpy(p_states + 128u * (uint32_t)b, st, 128);
  }

  uint32_t off = 0; /* ans/GpuANSEncode.cuh:497-513,796-823: scan of roundUp(words,8) */
  for (uint32_t b = 0; b < nb; ++b) {
    uint32_t len = n - b * DGO_BLOCK < DGO_BLOCK ? n - b * DGO_BLOCK : DGO_BLOCK;
    put32(p_bw + 8u * b, (len << 16) | words[b]); /* :598-608 */
    put32(p_bw + 8u * b + 4, off);
    uint32_t padded = round_up(words[b], 8u);
    memcpy(p_data + 2u * off, slots + (size_t)b * slot_words, 2u * words[b]);
    memset(p_data + 2u * (off + words[b]), 0, 2u * (padded - words[b]));
    off += padded;
  }
  free(slots);
  free(words);

  put32(out + 0, (DGO_ANS_MAGIC << 16) | DGO_VERSION); /* ans/GpuANSUtils.cuh:105-107 */
  put32(out + 4, nb);
  put32(out + 8, n);
  put32(out + 12, off);
  put32(out + 16, (uint32_t)pb | ((use_checksum ? 1u : 0u) << 4));
  put32(out + 20, use_checksum ? dgo_checksum(in, n) : 0u);
  put32(out + 24, 0);
  put32(out + 28, 0);
  return dgo_ans_overhead(nb) + 2u * off; /* ans/GpuANSUtils.cuh:83-86 */
}

/* ans/GpuANSInfo.cuh:16-37 */
int dgo_ans_info(const uint8_t* in, uint32_t* size, uint32_t* uncompressed,
                 uint32_t* checksum, int* pb, int* has_checksum) {
  uint32_t mv = get32(in);
  if ((mv >> 16) != DGO_ANS_MAGIC || (mv & 0xffffu) != DGO_VERSION) return DGO_ERR_BAD_MAGIC;
  uint32_t nb = get32(in + 4);
  if (size) *size = dgo_ans_overhead(nb) + 2u * get32(in + 12);
  if (uncompressed) *uncompressed = get32(in + 8);
  if (checksum) *checksum = get32(in + 20);
  if (pb) *pb = (int)(get32(in + 16) & 0xfu);
  if (has_checksum) *has_checksum = (int)((get32(in + 16) >> 4) & 1u);
  return DGO_OK;
}

/* ans/GpuANSDecode.cuh:405-476 ansDecodeTable: pdf -> cdf -> 2^pb-entry LUT */
static int build_decode_lut(const uint8_t* p_pdf, int pb, uint32_t* lut) {
  uint32_t acc = 0;
  for (uint32_t s = 0; s < 256; ++s) {
    uint32_t p = get16(p_pdf + 2 * s);
    if (acc + p > (1u << pb)) return DGO_ERR_CORRUPT;
    for (uint32_t j = 0; j < p; ++j) lut[acc + j] = (j << 20) | (p << 8) | s;
    acc += p;
  }
  return acc == (1u << pb) ? DGO_OK : DGO_ERR_CORRUPT;
}

/* ans/GpuANSDecode.cuh:299-403 ansDecodeKernel (+ :555-591 checksum verify).
 * capacity semantics as the reference: out_size always reports the archive's
 * uncompressed size; DGO_ERR_CAPACITY when it does not fit. */
int dgo_ans_decode(const uint8_t* in, int pb, int verify_checksum, uint8_t* out,
                   uint32_t capacity, uint32_t* out_size) {
  uint32_t mv = get32(in);
  if ((mv >> 16) != DGO_ANS_MAGIC || (mv & 0xffffu) != DGO_VERSION) return DGO_ERR_BAD_MAGIC;
  uint32_t nb = get32(in + 4), n = get32(in + 8);
  if ((int)(get32(in + 16) & 0xfu) != pb) return DGO_ERR_BAD_PROBBITS;
  if (out_size) *out_size = n;
  if (capacity < n) return DGO_ERR_CAPACITY;
  if (n == 0) return DGO_OK;

  const uint8_t* p_states = in + 32 + 512;
  const uint8_t* p_bw = p_states + 128u * nb;
  const uint8_t* p_data = p_bw + 8u * round_up(nb, 2u);
  uint32_t* lut = (uint32_t*)malloc(sizeof(uint32_t) << pb);
  int rc = build_decode_lut(in + 32, pb, lut);
  if (rc != DGO_OK) { free(lut); return rc; }

  int err = DGO_OK;
#pragma omp parallel for schedule(dynamic, 16)
  for (int64_t b = 0; b < (int64_t)nb; ++b) {
    uint32_t st[DGO_LANES];
    uint32_t bw = get32(p_bw + 8u * (uint32_t)b), off = get32(p_bw + 8u * (uint32_t)b + 4);
    memcpy(st, p_states + 128u * (uint32_t)b, 128);
    int r = decode_block(st, (const uint16_t*)(p_data + 2u * (size_t)off), bw & 0xffffu,
                         bw >> 16, pb, lut, out + (size_t)b * DGO_BLOCK);
    if (r != DGO_OK) {
#pragma omp atomic write
      err = r;
    }
  }
  free(lut);
  if (err != DGO_OK) return err;
  if (verify_checksum && ((get32(in + 16) >> 4) & 1u) && dgo_checksum(out, n) != get32(in + 20))
    return DGO_ERR_CHECKSUM;
  return DGO_OK;
}

/* ---------------------------------------------------------- float codec -- */

static uint32_t rotl32(uint32_t v, int s) { return (v << s) | (v >> (32 - s)); }
static uint32_t rotr32(uint32_t v, int s) { return (v >> s) | (v << (32 - s)); }

/* float/GpuFloatUtils.cuh:111-115 (fp16), :141-147 (bf16) */
static void split16(int ft, uint16_t v, uint8_t* comp, uint8_t* non) {
  if (ft == DGO_F16) { *comp = (uint8_t)(v >> 8); *non = (uint8_t)(v & 0xffu); }
  else { *comp = (uint8_t)((v >> 7) & 0xffu); *non = (uint8_t)(((v & 0x7fu) << 1) | (v >> 15)); }
}

/* float/GpuFloatUtils.cuh:117-119 (fp16), :149-159 (bf16) */
static uint16_t join16(int ft, uint8_t comp, uint8_t non) {
  if (ft == DGO_F16) return (uint16_t)(((uint32_t)comp << 8) | non);
  return (uint16_t)(((((uint32_t)comp << 8) | non) >> 1) | (((uint32_t)non & 1u) << 15));
}

/*
 * float/GpuFloatCompress.cuh:280-365 (splitFloat), :420-427 (ANS placement),
 * :369-377 (reported size).  n counts float WORDS.  Archive =
 * 16 B GpuFloatHeader | non-compressed bytes | ANS archive of the comp bytes.
 * The float-level checksum covers only the first n BYTES of the input
 * (SURVEY A.6/B6), reproduced here.
 */
uint32_t dgo_float_compress(int ft, const void* in, uint32_t n, int pb,
                            int use_checksum, uint8_t* out) {
  uint8_t* comp = (uint8_t*)malloc(n ? n : 1);
  uint32_t nc_bytes = dgo_float_noncomp_bytes(ft, n);
  uint8_t* non = out + 16;
  memset(non, 0, nc_bytes);
  if (ft == DGO_F32) {
    const uint32_t* w = (const uint32_t*)in;
    uint8_t* non1 = non + 2u * round_up(n, 8u); /* float/GpuFloatUtils.cuh:194-203 */
    for (uint32_t i = 0; i < n; ++i) {
      uint32_t v = rotl32(w[i], 1); /* :181-185 */
      comp[i] = (uint8_t)(v >> 24);
      put16(non + 2u * i, (uint16_t)(v & 0xffffu));
      non1[i] = (uint8_t)((v >> 16) & 0xffu);
    }
  } else {
    const uint16_t* w = (const uint16_t*)in;
    for (uint32_t i = 0; i < n; ++i) split16(ft, w[i], &comp[i], &non[i]);
  }
  put32(out + 0, (DGO_FLOAT_MAGIC << 16) | DGO_VERSION);
  put32(out + 4, n);
  put32(out + 8, (uint32_t)ft | ((use_checksum ? 1u : 0u) << 4));
  put32(out + 12, use_checksum ? dgo_checksum((const uint8_t*)in, n) : 0u);
  uint32_t ans = dgo_ans_encode(comp, n, pb, 0, NULL, out + 16 + nc_bytes);
  free(comp);
  return 16u + nc_bytes + ans;
}

/* float/GpuFloatInfo.cuh:19-41 */
int dgo_float_info(const uint8_t* in, uint32_t* n, int* ft, uint32_t* checksum) {
  uint32_t mv = get32(in);
  if ((mv >> 16) != DGO_FLOAT_MAGIC || (mv & 0xffffu) != DGO_VERSION) return DGO_ERR_BAD_MAGIC;
  if (n) *n = get32(in + 4);
  if (ft) *ft = (int)(get32(in + 8) & 0xfu);
  if (checksum) *checksum = get32(in + 12);
  return DGO_OK;
}

/* float/GpuFloatDecompress.cuh:565-738 (+ JoinFloatWriter :391-486).
 * capacity / out_size are in float words. */
int dgo_float_decompress(int ft, const uint8_t* in, int pb, int verify_checksum,
                         void* out, uint32_t capacity, uint32_t* out_size) {
  uint32_t mv = get32(in);
  if ((mv >> 16) != DGO_FLOAT_MAGIC || (mv & 0xffffu) != DGO_VERSION) return DGO_ERR_BAD_MAGIC;
  uint32_t n = get32(in + 4);
  if ((int)(get32(in + 8) & 0xfu) != ft) return DGO_ERR_BAD_FLOAT_TYPE;
  uint32_t nc_bytes = dgo_float_noncomp_bytes(ft, n);
  const uint8_t* non = in + 16;
  uint8_t* comp = (uint8_t*)malloc(n ? n : 1);
  uint32_t got = 0;
  int rc = dgo_ans_decode(in + 16 + nc_bytes, pb, 0, comp, capacity, &got);
  if (out_size) *out_size = got;
  if (rc != DGO_OK) { free(comp); return rc; }
  if (ft == DGO_F32) {
    uint32_t* w = (uint32_t*)out;
    const uint8_t* non1 = non + 2u * round_up(n, 8u);
    for (uint32_t i = 0; i < n; ++i) {
      uint32_t v = ((uint32_t)comp[i] << 24) | ((uint32_t)non1[i] << 16) | get16(non + 2u * i);
      w[i] = rotr32(v, 1); /* float/GpuFloatUtils.cuh:187-190 */
    }
  } else {
    uint16_t* w = (uint16_t*)out;
    for (uint32_t i = 0; i < n; ++i) w[i] = join16(ft, comp[i], non[i]);
  }
  free(comp);
  if (verify_checksum && ((get32(in + 8) >> 4) & 1u) &&
      dgo_checksum((const uint8_t*)out, n) != get32(in + 12))
    return DGO_ERR_CHECKSUM;
  return DGO_OK;
}

/* ------------------------------------------------ whole-batch CPU baseline -- */

/*
 * The host-CPU baseline of bench.py: one call takes the WHOLE batch and spreads every phase over
 * all cores -- split + histogram over (member, slab) pairs, normalisation over members, block
 * coding over the flat list of 4 KiB blocks of all members, packing over members; decode likewise
 * (LUTs over members, blocks over the flat list, join over (member, slab) pairs).  Same algorithm
 * and same archives as dgo_ans_encode / dgo_float_compress above (tests/test_oracle.py compares
 * them byte for byte); the block coder divides with the reference's reciprocal
 * (ans/GpuANSStatistics.cuh:343-358 + ans/GpuANSEncode.cuh:79-86) instead of a hardware divide.
 * ft: 0 = raw bytes, else DGO_F16 / DGO_BF16 / DGO_F32.  sizes in bytes (ft 0) or float words.
 * t_sec[0] / t_sec[1] receive the wall time of the encode / decode phase.
 * Returns DGO_OK, or the first decode error.
 */
#define DGO_SLAB 65536u

static uint32_t encode_block_magic(const uint8_t* in, uint32_t n, int pb, const uint32_t* tab /* [256][4] */,
                                   uint32_t state[DGO_LANES], uint16_t* w) {
  const uint32_t K = 1u << pb;
  uint32_t cnt = 0;
  for (uint32_t l = 0; l < DGO_LANES; ++l) state[l] = DGO_STATE_MIN;
  for (uint32_t r = 0; r < n; r += DGO_LANES) {
    uint32_t lanes = n - r < DGO_LANES ? n - r : DGO_LANES;
    for (uint32_t l = 0; l < lanes; ++l) {
      const uint32_t* e = tab + 4u * in[r + l]; /* {pdf, cdf, magic, shift} */
      uint32_t x = state[l];
      if (x >= (e[0] << (31 - pb))) {
        w[cnt++] = (uint16_t)(x & 0xffffu);
        x >>= 16;
      }
      uint32_t t = (uint32_t)(((uint64_t)x * e[2]) >> 32);
      uint32_t div = (uint32_t)(((uint64_t)t + x) >> e[3]); /* ans/GpuANSEncode.cuh:79-86 */
      state[l] = div * K + (x - div * e[0]) + e[1];
    }
  }
  return cnt;
}

void dgo_div_magic(uint32_t pdf, uint32_t* magic, uint32_t* shift);

int dgo_batch_roundtrip(int ft, const void* const* in, const uint32_t* sizes, uint32_t n, int pb,
                        uint8_t* const* archives, uint32_t* archive_sizes, void* const* outs,
                        double* t_sec) {
  const uint32_t wb = ft == DGO_F32 ? 4u : (ft == 0 ? 1u : 2u);
  const uint32_t slot_words = DGO_BLOCK * 11u / 16u + 8u;
  /* flat indices: blocks and slabs of every member */
  uint64_t* blk0 = (uint64_t*)malloc(sizeof(uint64_t) * (n + 1));
  uint64_t* slab0 = (uint64_t*)malloc(sizeof(uint64_t) * (n + 1));
  blk0[0] = slab0[0] = 0;
  for (uint32_t m = 0; m < n; ++m) {
    blk0[m + 1] = blk0[m] + div_up(sizes[m], DGO_BLOCK);
    slab0[m + 1] = slab0[m] + (sizes[m] ? div_up(sizes[m], DGO_SLAB) : 0u);
  }
  const uint64_t nblocks = blk0[n], nslabs = slab0[n];
  uint32_t* blk_member = (uint32_t*)malloc(sizeof(uint32_t) * (nblocks ? nblocks : 1));
  uint32_t* slab_member = (uint32_t*)malloc(sizeof(uint32_t) * (nslabs ? nslabs : 1));
  for (uint32_t m = 0; m < n; ++m) {
    for (uint64_t b = blk0[m]; b < blk0[m + 1]; ++b) blk_member[b] = m;
    for (uint64_t s = slab0[m]; s < slab0[m + 1]; ++s) slab_member[s] = m;
  }
  uint32_t* hist = (uint32_t*)calloc((size_t)n * 256u, sizeof(uint32_t));
  uint32_t* tab = (uint32_t*)malloc((size_t)n * 1024u * sizeof(uint32_t));
  uint32_t* luts = (uint32_t*)malloc(((size_t)n << pb) * sizeof(uint32_t));
  uint16_t* slots = (uint16_t*)malloc((size_t)(nblocks ? nblocks : 1) * slot_words * 2u);
  uint32_t* words = (uint32_t*)malloc(sizeof(uint32_t) * (nblocks ? nblocks : 1));
  uint8_t** comp = (uint8_t**)malloc(sizeof(uint8_t*) * n);
  for (uint32_t m = 0; m < n; ++m)
    comp[m] = ft ? (uint8_t*)malloc(sizes[m] ? sizes[m] : 1) : (uint8_t*)in[m];
  int err = DGO_OK;
#ifdef _OPENMP
  double t0 = omp_get_wtime();
#else
  double t0 = 0;
#endif

  /* ---------------- encode ---------------- */
#pragma omp parallel
  {
    /* split + histogram, one slab of one member per task */
#pragma omp for schedule(dynamic, 4)
    for (int64_t s = 0; s < (int64_t)nslabs; ++s) {
      const uint32_t m = slab_member[s];
      const uint32_t e0 = (uint32_t)((uint64_t)s - slab0[m]) * DGO_SLAB;
      const uint32_t e1 = sizes[m] - e0 < DGO_SLAB ? sizes[m] : e0 + DGO_SLAB;
      uint32_t local[256];
      memset(local, 0, sizeof(local));
      uint8_t* c = comp[m];
      if (ft == 0) {
        for (uint32_t i = e0; i < e1; ++i) local[c[i]]++;
      } else {
        uint8_t* non = archives[m] + 16;
        if (ft == DGO_F32) {
          const uint32_t* w = (const uint32_t*)in[m];
          uint8_t* non1 = non + 2u * round_up(sizes[m], 8u);
          for (uint32_t i = e0; i < e1; ++i) {
            uint32_t v = rotl32(w[i], 1);
            c[i] = (uint8_t)(v >> 24);
            put16(non + 2u * i, (uint16_t)(v & 0xffffu));
            non1[i] = (uint8_t)((v >> 16) & 0xffu);
            local[c[i]]++;
          }
        } else {
          const uint16_t* w = (const uint16_t*)in[m];
          for (uint32_t i = e0; i < e1; ++i) {
            split16(ft, w[i], &c[i], &non[i]);
            local[c[i]]++;
          }
        }
      }
      for (uint32_t k = 0; k < 256; ++k)
        if (local[k]) {
#pragma omp atomic
          hist[(size_t)m * 256u + k] += local[k];
        }
    }
    /* per member: normalise, encoder table {pdf, cdf, magic, shift}, pdf + float header into the archive */
#pragma omp for schedule(dynamic, 1)
    for (int64_t m = 0; m < (int64_t)n; ++m) {
      uint32_t pdf[256], cdf[256];
      dgo_normalize(hist + (size_t)m * 256u, sizes[m], pb, pdf);
      cdf_from_pdf(pdf, cdf);
      uint32_t* t = tab + (size_t)m * 1024u;
      for (uint32_t k = 0; k < 256; ++k) {
        t[4 * k] = pdf[k];
        t[4 * k + 1] = cdf[k];
        dgo_div_magic(pdf[k], &t[4 * k + 2], &t[4 * k + 3]);
      }
      uint8_t* a = archives[m];
      if (ft) {
        const uint32_t ncb = dgo_float_noncomp_bytes(ft, sizes[m]);
        put32(a + 0, (DGO_FLOAT_MAGIC << 16) | DGO_VERSION);
        put32(a + 4, sizes[m]);
        put32(a + 8, (uint32_t)ft);
        put32(a + 12, 0);
        /* zero padding of the stored planes */
        if (ft == DGO_F32) {
          memset(a + 16 + 2u * sizes[m], 0, 2u * round_up(sizes[m], 8u) - 2u * sizes[m]);
          memset(a + 16 + 2u * round_up(sizes[m], 8u) + sizes[m], 0, round_up(sizes[m], 16u) - sizes[m]);
        } else {
          memset(a + 16 + sizes[m], 0, ncb - sizes[m]);
        }
        a += 16 + ncb;
      }
      for (uint32_t k = 0; k < 256; ++k) put16(a + 32 + 2 * k, (uint16_t)pdf[k]);
    }
    /* every 4 KiB block of every member */
#pragma omp for schedule(dynamic, 16)
    for (int64_t b = 0; b < (int64_t)nblocks; ++b) {
      const uint32_t m = blk_member[b];
      const uint32_t blk = (uint32_t)((uint64_t)b - blk0[m]);
      const uint32_t nb = (uint32_t)(blk0[m + 1] - blk0[m]);
      const uint32_t start = blk * DGO_BLOCK;
      const uint32_t len = sizes[m] - start < DGO_BLOCK ? sizes[m] - start : DGO_BLOCK;
      uint32_t st[DGO_LANES];
      words[b] = encode_block_magic(comp[m] + start, len, pb, tab + (size_t)m * 1024u, st, slots + (size_t)b * slot_words);
      uint8_t* a = archives[m] + (ft ? 16u + dgo_float_noncomp_bytes(ft, sizes[m]) : 0u);
      memcpy(a + 32 + 512 + 128u * blk, st, 128);
      (void)nb;
    }
    /* per member: scan of padded sizes, pack, header */
#pragma omp for schedule(dynamic, 1)
    for (int64_t m = 0; m < (int64_t)n; ++m) {
      const uint32_t nb = (uint32_t)(blk0[m + 1] - blk0[m]);
      const uint32_t extra = ft ? 16u + dgo_float_noncomp_bytes(ft, sizes[m]) : 0u;
      uint8_t* a = archives[m] + extra;
      uint8_t* p_bw = a + 32 + 512 + 128u * nb;
      uint8_t* p_data = p_bw + 8u * round_up(nb, 2u);
      if (nb & 1u) memset(p_bw + 8u * nb, 0, 8);
      uint32_t off = 0;
      for (uint32_t k = 0; k < nb; ++k) {
        const uint64_t b = blk0[m] + k;
        const uint32_t len = sizes[m] - k * DGO_BLOCK < DGO_BLOCK ? sizes[m] - k * DGO_BLOCK : DGO_BLOCK;
        put32(p_bw + 8u * k, (len << 16) | words[b]);
        put32(p_bw + 8u * k + 4, off);
        const uint32_t padded = round_up(words[b], 8u);
        memcpy(p_data + 2u * off, slots + (size_t)b * slot_words, 2u * words[b]);
        memset(p_data + 2u * (off + words[b]), 0, 2u * (padded - words[b]));
        off += padded;
      }
      put32(a + 0, (DGO_ANS_MAGIC << 16) | DGO_VERSION);
      put32(a + 4, nb);
      put32(a + 8, sizes[m]);
      put32(a + 12, off);
      put32(a + 16, (uint32_t)pb);
      put32(a + 20, 0);
      put32(a + 24, 0);
      put32(a + 28, 0);
      archive_sizes[m] = extra + dgo_ans_overhead(nb) + 2u * off;
    }
  }
#ifdef _OPENMP
  double t1 = omp_get_wtime();
#else
  double t1 = 0;
#endif

  /* ---------------- decode ---------------- */
#pragma omp parallel
  {
#pragma omp for schedule(dynamic, 1)
    for (int64_t m = 0; m < (int64_t)n; ++m) {
      const uint8_t* a = archives[m] + (ft ? 16u + dgo_float_noncomp_bytes(ft, sizes[m]) : 0u);
      if (sizes[m] && build_decode_lut(a + 32, pb, luts + ((size_t)m << pb)) != DGO_OK) {
#pragma omp atomic write
        err = DGO_ERR_CORRUPT;
      }
    }
#pragma omp for schedule(dynamic, 16)
    for (int64_t b = 0; b < (int64_t)nblocks; ++b) {
      const uint32_t m = blk_member[b];
      const uint32_t blk = (uint32_t)((uint64_t)b - blk0[m]);
      const uint32_t nb = (uint32_t)(blk0[m + 1] - blk0[m]);
      const uint8_t* a = archives[m] + (ft ? 16u + dgo_float_noncomp_bytes(ft, sizes[m]) : 0u);
      const uint8_t* p_states = a + 32 + 512;
      const uint8_t* p_bw = p_states + 128u * nb;
      const uint8_t* p_data = p_bw + 8u * round_up(nb, 2u);
      uint32_t st[DGO_LANES];
      const uint32_t bw = get32(p_bw + 8u * blk), off = get32(p_bw + 8u * blk + 4);
      memcpy(st, p_states + 128u * blk, 128);
      uint8_t* dst = ft ? comp[m] : (uint8_t*)outs[m];
      int r = decode_block(st, (const uint16_t*)(p_data + 2u * (size_t)off), bw & 0xffffu, bw >> 16, pb,
                           luts + ((size_t)m << pb), dst + (size_t)blk * DGO_BLOCK);
      if (r != DGO_OK) {
#pragma omp atomic write
        err = r;
      }
    }
    if (ft) {
#pragma omp for schedule(dynamic, 4)
      for (int64_t s = 0; s < (int64_t)nslabs; ++s) {
        const uint32_t m = slab_member[s];
        const uint32_t e0 = (uint32_t)((uint64_t)s - slab0[m]) * DGO_SLAB;
        const uint32_t e1 = sizes[m] - e0 < DGO_SLAB ? sizes[m] : e0 + DGO_SLAB;
        const uint8_t* non = archives[m] + 16;
        const uint8_t* c = comp[m];
        if (ft == DGO_F32) {
          uint32_t* w = (uint32_t*)outs[m];
          const uint8_t* non1 = non + 2u * round_up(sizes[m], 8u);
          for (uint32_t i = e0; i < e1; ++i) {
            uint32_t v = ((uint32_t)c[i] << 24) | ((uint32_t)non1[i] << 16) | get16(non + 2u * i);
            w[i] = rotr32(v, 1);
          }
        } else {
          uint16_t* w = (uint16_t*)outs[m];
          for (uint32_t i = e0; i < e1; ++i) w[i] = join16(ft, c[i], non[i]);
        }
      }
    }
  }
#ifdef _OPENMP
  double t2 = omp_get_wtime();
#else
  double t2 = 0;
#endif
  if (t_sec) { t_sec[0] = t1 - t0; t_sec[1] = t2 - t1; }
  if (ft) for (uint32_t m = 0; m < n; ++m) free(comp[m]);
  free(comp); free(words); free(slots); free(luts); free(tab); free(hist);
  free(slab_member); free(blk_member); free(slab0); free(blk0);
  (void)wb;
  return err;
}

/* --------------------------------------------------------------- extras -- */

/* Exposed for tests: the encoder division constants of
 * ans/GpuANSStatistics.cuh:343-358 so the CUDA table can be checked. */
void dgo_div_magic(uint32_t pdf, uint32_t* magic, uint32_t* shift) {
  uint32_t sh = 0;
  while (sh < 32 && (1ull << sh) < pdf) sh++; /* 32 - clz(pdf-1) */
  if (pdf <= 1) sh = 0;
  *shift = sh;
  *magic = pdf ? (uint32_t)((((uint64_t)1 << 32) * (((uint64_t)1 << sh) - pdf)) / pdf + 1) : 0;
}

int dgo_num_threads(void) {
#ifdef _OPENMP
  return omp_get_max_threads();
#else
  return 1;
#endif
}

void dgo_set_threads(int n) {
#ifdef _OPENMP
  omp_set_num_threads(n > 0 ? n : 1);
#else
  (void)n;
#endif
}

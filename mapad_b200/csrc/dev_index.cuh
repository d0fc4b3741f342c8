// dev_index.cuh — device-resident FMD index: block layout access, rank queries, bidirectional
// extension, SA locate.  Compiles for the device (nvcc) and, for the CPU emulation harness used by
// the non-GPU tests, as plain C++.
//
// Reference semantics restated here:
//   Occ::get / get_small_k      rust-bio fork, called from src/map/fmd_index.rs:22-25, src/index/mod.rs:181
//   FmdExtIterator              src/map/fmd_index.rs:117-182
//   backward_ext / forward_ext  src/map/fmd_index.rs:77-96
//   SampledSuffixArray::get     src/index/mod.rs:160-187
//   get_reference_identifier    src/index/mod.rs:55-75
//   OriginalSymbols::get        src/index/mod.rs:206-209
#pragma once
#include <cstdint>

#include "common.h"

#if defined(__CUDACC__)
#define MAPAD_HD __host__ __device__ __forceinline__
#define MAPAD_DEV __device__ __forceinline__
#define MAPAD_DEV_NOINLINE __device__ __noinline__
#else
#define MAPAD_HD inline
#define MAPAD_DEV inline
#define MAPAD_DEV_NOINLINE inline
#endif

namespace mapad {

struct U4 { uint32_t x, y, z, w; };

MAPAD_DEV U4 load16(const void* p) {
#if defined(__CUDA_ARCH__)
  uint4 v = __ldg(reinterpret_cast<const uint4*>(p));
  return U4{v.x, v.y, v.z, v.w};
#else
  const uint32_t* q = reinterpret_cast<const uint32_t*>(p);
  return U4{q[0], q[1], q[2], q[3]};
#endif
}
MAPAD_DEV int popc32(uint32_t x) {
#if defined(__CUDA_ARCH__)
  return __popc(x);
#else
  return __builtin_popcount(x);
#endif
}

struct DevIndex {
  IndexMeta m;
  const uint8_t* blob;
  MAPAD_DEV const uint8_t* occ() const { return blob + m.off_occ; }
  MAPAD_DEV const uint8_t* sa() const { return blob + m.off_sa; }
  MAPAD_DEV const uint64_t* extra() const { return reinterpret_cast<const uint64_t*>(blob + m.off_extra); }
  MAPAD_DEV const XRange* xranges() const { return reinterpret_cast<const XRange*>(blob + m.off_xranges); }
  MAPAD_DEV const uint64_t* contigs() const { return reinterpret_cast<const uint64_t*>(blob + m.off_contigs); }
  MAPAD_DEV const uint64_t* orig_pos() const { return reinterpret_cast<const uint64_t*>(blob + m.off_orig); }
  MAPAD_DEV const uint8_t* orig_sym() const { return blob + m.off_orig + 8 * m.n_orig; }
};

struct BiIv {  // RtBiInterval (fmd_index.rs:185-189)
  uint64_t lower, lower_rev, size;
};

// number of rows with bwt == 'X' in [0, r]
MAPAD_DEV_NOINLINE uint64_t x_rows_upto(const DevIndex& ix, uint64_t r) {
  const XRange* xr = ix.xranges();
  uint64_t lo = 0, hi = ix.m.n_xranges;  // first range with start > r
  while (lo < hi) {
    uint64_t mid = (lo + hi) >> 1;
    if (xr[mid].start <= r) lo = mid + 1; else hi = mid;
  }
  if (lo == 0) return 0;
  const XRange& g = xr[lo - 1];
  uint64_t upto = r + 1 < g.end ? r + 1 : g.end;
  return g.before + (upto - g.start);
}
MAPAD_DEV_NOINLINE bool is_x_row(const DevIndex& ix, uint64_t r) {
  uint64_t a = x_rows_upto(ix, r);
  uint64_t b = r == 0 ? 0 : x_rows_upto(ix, r - 1);
  return a != b;
}

MAPAD_DEV void count_word(uint32_t x, int npos, uint32_t& nC, uint32_t& nG, uint32_t& nT) {
  int np = npos < 0 ? 0 : (npos > 16 ? 16 : npos);
  uint32_t mask = np >= 16 ? 0x55555555u : (((1u << (2 * np)) - 1u) & 0x55555555u);
  uint32_t lo = x & mask, hi = (x >> 1) & mask, hl = hi & lo;
  int phl = popc32(hl);
  nT += phl;
  nG += popc32(hi) - phl;
  nC += popc32(lo) - phl;
}

// Ranks of A,C,G,T at row r: c[k] = #(rank k+1) in bwt[0..=r]   (Occ::get for the four bases at once).
// Split into the block fetch (occ_load) and the popcount arithmetic (occ_finish) so that callers can put
// independent work between the two.
template <bool WIDE>
struct OccRaw { U4 w[WIDE ? 4 : 2]; };

template <bool WIDE>
MAPAD_DEV void occ_load(const DevIndex& ix, uint64_t r, OccRaw<WIDE>& raw) {
  if (!WIDE) {
    const uint8_t* p = ix.occ() + (r >> 6) * 32;
    raw.w[0] = load16(p); raw.w[1] = load16(p + 16);
  } else {
    const uint8_t* p = ix.occ() + (r >> 7) * 64;
    raw.w[0] = load16(p); raw.w[1] = load16(p + 16); raw.w[2] = load16(p + 32); raw.w[3] = load16(p + 48);
  }
}

template <bool WIDE>
MAPAD_DEV void occ_finish(const DevIndex& ix, uint64_t r, const OccRaw<WIDE>& raw, uint64_t c[4]) {
  uint32_t nC = 0, nG = 0, nT = 0;
  uint64_t bstart;
  int npos;
  bool flagged;
  if (!WIDE) {
    bstart = (r >> 6) << 6;
    npos = (int)(r & 63) + 1;
    const U4 cn = raw.w[0], cd = raw.w[1];
    flagged = (cn.x >> 31) != 0;
    c[0] = cn.x & 0x7fffffffu; c[1] = cn.y; c[2] = cn.z; c[3] = cn.w;
    count_word(cd.x, npos, nC, nG, nT);
    count_word(cd.y, npos - 16, nC, nG, nT);
    count_word(cd.z, npos - 32, nC, nG, nT);
    count_word(cd.w, npos - 48, nC, nG, nT);
  } else {
    bstart = (r >> 7) << 7;
    npos = (int)(r & 127) + 1;
    const U4 c0 = raw.w[0], c1 = raw.w[1], d0 = raw.w[2], d1 = raw.w[3];
    uint64_t a0 = (uint64_t)c0.x | ((uint64_t)c0.y << 32);
    flagged = (a0 >> 63) != 0;
    c[0] = a0 & 0x7fffffffffffffffull;
    c[1] = (uint64_t)c0.z | ((uint64_t)c0.w << 32);
    c[2] = (uint64_t)c1.x | ((uint64_t)c1.y << 32);
    c[3] = (uint64_t)c1.z | ((uint64_t)c1.w << 32);
    count_word(d0.x, npos, nC, nG, nT);
    count_word(d0.y, npos - 16, nC, nG, nT);
    count_word(d0.z, npos - 32, nC, nG, nT);
    count_word(d0.w, npos - 48, nC, nG, nT);
    count_word(d1.x, npos - 64, nC, nG, nT);
    count_word(d1.y, npos - 80, nC, nG, nT);
    count_word(d1.z, npos - 96, nC, nG, nT);
    count_word(d1.w, npos - 112, nC, nG, nT);
  }
  uint32_t nA = (uint32_t)npos - nC - nG - nT;
  // '$' rows are stored with code 0: take them out of the A count
  uint64_t s0 = ix.m.sentinel_rows[0], s1 = ix.m.sentinel_rows[1];
  nA -= (uint32_t)(s0 >= bstart && s0 <= r);
  nA -= (uint32_t)(s1 >= bstart && s1 <= r);
  if (flagged) {  // so are 'X' rows (N-runs >= 20 bp in the reference, indexing.rs:96-106)
    uint64_t upto = x_rows_upto(ix, r);
    uint64_t before = bstart == 0 ? 0 : x_rows_upto(ix, bstart - 1);
    nA -= (uint32_t)(upto - before);
  }
  c[0] += nA; c[1] += nC; c[2] += nG; c[3] += nT;
}

template <bool WIDE>
MAPAD_DEV void occ4(const DevIndex& ix, uint64_t r, uint64_t c[4]) {
  OccRaw<WIDE> raw;
  occ_load<WIDE>(ix, r, raw);
  occ_finish<WIDE>(ix, r, raw, c);
}

// rank (0..5) of the BWT symbol at `row`
template <bool WIDE>
MAPAD_DEV uint32_t bwt_at(const DevIndex& ix, uint64_t row) {
  if (row == ix.m.sentinel_rows[0] || row == ix.m.sentinel_rows[1]) return 0;
  const uint32_t* blk;
  uint32_t within;
  bool flagged;
  if (!WIDE) {
    blk = reinterpret_cast<const uint32_t*>(ix.occ() + (row >> 6) * 32);
    within = (uint32_t)(row & 63);
    flagged = (blk[0] >> 31) != 0;
    blk += 4;
  } else {
    blk = reinterpret_cast<const uint32_t*>(ix.occ() + (row >> 7) * 64);
    within = (uint32_t)(row & 127);
    flagged = (blk[1] >> 31) != 0;
    blk += 8;
  }
  if (flagged && is_x_row(ix, row)) return 5;
  return ((blk[within >> 4] >> (2 * (within & 15))) & 3u) + 1u;
}

MAPAD_DEV uint64_t sentinels_upto(const DevIndex& ix, uint64_t pos) {  // fmd_index.rs:140-146
  return (uint64_t)(ix.m.sentinel_rows[0] <= pos) + (uint64_t)(ix.m.sentinel_rows[1] <= pos);
}

// FmdExtIterator: out[k] is the extension by rank 4-k (T,G,C,A).  extend_load issues the (at most) two
// block fetches, extend_finish turns them into the four child intervals.
template <bool WIDE>
struct ExtRaw { OccRaw<WIDE> lo, hi; };

template <bool WIDE>
MAPAD_DEV void extend_load(const DevIndex& ix, const BiIv& in, ExtRaw<WIDE>& raw) {
  if (in.lower != 0) occ_load<WIDE>(ix, in.lower - 1, raw.lo);
  occ_load<WIDE>(ix, in.lower + in.size - 1, raw.hi);
}
template <bool WIDE>
MAPAD_DEV void extend_finish(const DevIndex& ix, const BiIv& in, const ExtRaw<WIDE>& raw, BiIv out[4]) {
  uint64_t lo[4] = {0, 0, 0, 0}, hi[4];
  uint64_t s_lo = 0;
  if (in.lower != 0) { occ_finish<WIDE>(ix, in.lower - 1, raw.lo, lo); s_lo = sentinels_upto(ix, in.lower - 1); }
  occ_finish<WIDE>(ix, in.lower + in.size - 1, raw.hi, hi);
  uint64_t l = in.lower_rev + (sentinels_upto(ix, in.lower + in.size - 1) - s_lo);
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    int c = 3 - k;  // index into lo/hi (rank - 1)
    uint64_t s = hi[c] - lo[c];
    out[k].lower = ix.m.less[c + 1] + lo[c];
    out[k].lower_rev = l;
    out[k].size = s;
    l += s;
  }
}
template <bool WIDE>
MAPAD_DEV void extend_all(const DevIndex& ix, const BiIv& in, BiIv out[4]) {
  ExtRaw<WIDE> raw;
  extend_load<WIDE>(ix, in, raw);
  extend_finish<WIDE>(ix, in, raw, out);
}

// backward_ext by rank r (1..4); r == 0 means "not in the alphabet" -> empty interval (fmd_index.rs:79-85)
template <bool WIDE>
MAPAD_DEV BiIv backward_ext_rank(const DevIndex& ix, const BiIv& in, int r) {
  BiIv e{0, 0, 0};
  if (r < 1 || r > 4) return e;
  BiIv out[4];
  extend_all<WIDE>(ix, in, out);
  return out[4 - r];
}
template <bool WIDE>
MAPAD_DEV BiIv forward_ext_rank(const DevIndex& ix, const BiIv& in, int r) {  // fmd_index.rs:93-96
  BiIv sw{in.lower_rev, in.lower, in.size};
  BiIv o = backward_ext_rank<WIDE>(ix, sw, r == 0 ? 0 : 5 - r);  // complement: A<->T, C<->G
  return BiIv{o.lower_rev, o.lower, o.size};
}

MAPAD_DEV int base_rank(uint8_t b) {  // RankTransform over $ACGTX restricted to what a read may extend by
  switch (b) { case 'A': return 1; case 'C': return 2; case 'G': return 3; case 'T': return 4; default: return 0; }
}
MAPAD_DEV uint8_t rank_base(int r) { return (uint8_t)("$ACGTX"[r]); }  // get_rev (fmd_index.rs:103-105)
MAPAD_DEV uint8_t complement_base(uint8_t b) {
  switch (b) { case 'A': return 'T'; case 'T': return 'A'; case 'C': return 'G'; case 'G': return 'C'; default: return b; }
}
// bio::alphabets::dna::complement: also pairs the IUPAC codes (R-Y, K-M, B-V, D-H; S, W, N map to themselves).  MD reports
// the reference's original symbol (record.rs:301-321), complemented like a base on the reverse strand.
MAPAD_DEV uint8_t complement_iupac(uint8_t b) {
  switch (b) {
    case 'R': return 'Y'; case 'Y': return 'R'; case 'K': return 'M'; case 'M': return 'K';
    case 'B': return 'V'; case 'V': return 'B'; case 'D': return 'H'; case 'H': return 'D';
    default: return complement_base(b);
  }
}

// SampledSuffixArray::get.  `steps` counts LF steps + the final sample / extra-row read (W of SURVEY §8d).
template <bool WIDE>
MAPAD_DEV uint64_t sa_get(const DevIndex& ix, uint64_t row, uint32_t& steps) {
  uint64_t pos = row, offset = 0;
  const uint32_t rate = ix.m.sa_rate;
  while (true) {
    if (pos % rate == 0) {
      steps += 1;
      uint64_t s = WIDE ? reinterpret_cast<const uint64_t*>(ix.sa())[pos / rate]
                        : (uint64_t) reinterpret_cast<const uint32_t*>(ix.sa())[pos / rate];
      return s + offset;
    }
    uint32_t c = bwt_at<WIDE>(ix, pos);
    if (c == 0) {
      steps += 1;
      const uint64_t* ex = ix.extra();
      for (uint64_t i = 0; i < ix.m.n_extra; ++i)
        if (ex[2 * i] == pos) return ex[2 * i + 1] + offset;
      return 0;  // unreachable for a consistent index
    }
    uint64_t occ_c;
    if (c == 5) {
      occ_c = x_rows_upto(ix, pos - 1);
    } else {
      uint64_t cnt[4];
      occ4<WIDE>(ix, pos - 1, cnt);
      occ_c = cnt[c - 1];
    }
    pos = ix.m.less[c] + occ_c;
    offset += 1;
    steps += 1;
  }
}

// FastaIdPositions::get_reference_identifier; contigs are disjoint and sorted, so the first match of
// the reference's linear scan is the only candidate.
MAPAD_DEV bool reference_identifier(const DevIndex& ix, uint64_t position, uint64_t pattern_length, int32_t& tid, uint64_t& rel) {
  const uint64_t* ct = ix.contigs();  // (start, end) pairs
  uint64_t lo = 0, hi = ix.m.n_contigs;  // first contig with start > position
  while (lo < hi) {
    uint64_t mid = (lo + hi) >> 1;
    if (ct[2 * mid] <= position) lo = mid + 1; else hi = mid;
  }
  if (lo == 0) return false;
  uint64_t i = lo - 1;
  if (position + pattern_length - 1 <= ct[2 * i + 1]) { tid = (int32_t)i; rel = position - ct[2 * i]; return true; }
  return false;
}

MAPAD_DEV bool original_symbol(const DevIndex& ix, uint64_t pos, uint8_t& sym) {
  uint64_t n = ix.m.n_orig;
  if (n == 0) return false;
  const uint64_t* op = ix.orig_pos();
  uint64_t lo = 0, hi = n;
  while (lo < hi) {
    uint64_t mid = (lo + hi) >> 1;
    if (op[mid] < pos) lo = mid + 1; else hi = mid;
  }
  if (lo < n && op[lo] == pos) { sym = ix.orig_sym()[lo]; return true; }
  return false;
}

}  // namespace mapad

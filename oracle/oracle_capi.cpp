// oracle/oracle_capi.cpp — TEST INFRASTRUCTURE ONLY (see oracle.hpp).
// C entry points for the ctypes wrapper oracle/oracle.py.  Output PODs reuse the layouts declared
// in include/mapad_gpu.h so that tests compare the CUDA path and the oracle field by field.
#include "oracle.hpp"

#include <atomic>
#include <cstdarg>
#include <mutex>
#include <thread>

#include "../include/mapad_gpu.h"

using namespace ora;

namespace {

struct DrawState { const char* draws; size_t n, i; };
uint8_t draw_replace(uint8_t, void* u) {
  DrawState* s = (DrawState*)u;
  if (s->draws && s->i < s->n) return (uint8_t)s->draws[s->i++];
  return 'A';
}

struct BatchOut {
  std::vector<mapad_record> records;
  std::vector<mapad_hit> hits;
  std::vector<mapad_edit_op> edit_ops;
  std::vector<uint32_t> cigar;
  std::vector<char> text;
  std::vector<std::string> xa;
  std::vector<char> xa_flat;
  std::vector<uint64_t> xa_off;
};

uint32_t bam_cigar(const CigarOp& c) {
  uint32_t op = c.kind == 'M' ? 0 : (c.kind == 'I' ? 1 : 2);
  return c.len << 4 | op;
}

struct PerRead {
  mapad_record rec;
  std::vector<mapad_hit> hits;
  std::vector<mapad_edit_op> ops;
  std::vector<uint32_t> cigar;
  std::string text;
  std::string xa;
};

void map_one(const Index& ix, const Params& p, const uint8_t* seq, const uint8_t* qual, usize L, uint32_t seed,
             Scratch& scratch, PerRead& out, bool want_hits) {
  Counters ctr;
  BinaryHeap<Hit> hits = k_mismatch_search(seq, qual, L, p, ix, scratch, &ctr);
  memset(&out.rec, 0, sizeof out.rec);
  out.hits.clear(); out.ops.clear(); out.cigar.clear(); out.text.clear(); out.xa.clear();
  out.rec.n_hits = (uint32_t)hits.len();
  if (want_hits) {
    for (const Hit& h : hits.d) {
      mapad_hit mh;
      memset(&mh, 0, sizeof mh);
      mh.lower = h.interval.lower; mh.lower_rev = h.interval.lower_rev; mh.size = h.interval.size;
      mh.alignment_score = h.alignment_score;
      mh.edit_off = (uint32_t)out.ops.size();
      mh.edit_len = (uint32_t)h.edit_operations.size();
      for (const EditOp& o : h.edit_operations) out.ops.push_back(mapad_edit_op{o.pos, o.kind, o.base});
      out.hits.push_back(mh);
    }
  }
  Record r = intervals_to_record(std::move(hits), ix, p, seed, &ctr);
  mapad_record& m = out.rec;
  m.mapped = r.mapped ? 1 : 0;
  m.tid = r.mapped ? (int32_t)r.tid : -1;
  m.pos = r.mapped ? (int64_t)r.pos : -1;
  m.strand = r.backward ? 1 : 0;
  m.mapq = r.mapq;
  m.alignment_score = r.alignment_score;
  m.nm = r.nm;
  m.x0 = r.x0; m.x1 = r.x1; m.xs = r.xs; m.xt = r.mapped ? r.xt : 0;
  m.cigar_off = 0; m.cigar_len = (uint32_t)r.cigar.size();
  for (const CigarOp& c : r.cigar) out.cigar.push_back(bam_cigar(c));
  m.md_off = 0; m.md_len = (uint32_t)r.md.size();
  out.text += r.md;
  m.n_alts = (uint32_t)r.alts.size();
  for (size_t a = 0; a < r.alts.size() && a < 2; ++a) {
    const AltHit& ah = r.alts[a];
    mapad_alt& ma = m.alts[a];
    ma.tid = (int32_t)ah.tid; ma.strand = ah.backward ? 1 : 0; ma.pos = (int64_t)ah.relative_pos;
    ma.cigar_off = (uint32_t)out.cigar.size(); ma.cigar_len = (uint32_t)ah.cigar.size();
    for (const CigarOp& c : ah.cigar) out.cigar.push_back(bam_cigar(c));
    ma.md_off = (uint32_t)out.text.size(); ma.md_len = (uint32_t)ah.md.size();
    out.text += ah.md;
    ma.nm = ah.nm; ma.alignment_score = ah.score; ma.interval_size = ah.interval_size;
  }
  m.best_lower = r.best_interval.lower; m.best_lower_rev = r.best_interval.lower_rev; m.best_size = r.best_interval.size;
  m.absolute_pos = r.absolute_pos;
  m.frames_popped = (uint32_t)ctr.frames_popped;
  m.d_ext_steps = (uint32_t)ctr.d_ext_steps;
  m.lf_steps = (uint32_t)ctr.lf_steps;
  m.flags = ctr.limit_hit ? 1u : 0u;
  out.xa = r.xa;
}

// Runs f(lo, hi) over [0, n_items) in slices of `grain` on n_threads threads.
template <class F>
void parallel_slices(uint64_t n_items, uint64_t grain, int n_threads, F f) {
  std::atomic<uint64_t> next(0);
  auto worker = [&]() {
    for (;;) {
      uint64_t lo = next.fetch_add(grain);
      if (lo >= n_items) break;
      f(lo, std::min(lo + grain, n_items));
    }
  };
  std::vector<std::thread> th;
  for (int t = 1; t < n_threads; ++t) th.emplace_back(worker);
  worker();
  for (auto& t : th) t.join();
}

// First failure of a parallel check; later ones are dropped.
struct Failure {
  std::atomic<bool> hit{false};
  std::mutex mu;
  std::string what;
  void set(const char* fmt, ...) __attribute__((format(printf, 2, 3))) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    std::lock_guard<std::mutex> g(mu);
    if (!hit.load()) { what = buf; hit.store(true); }
  }
};

// Sets bit i; returns whether it was already set.
inline bool test_and_set(std::vector<uint64_t>& bits, uint64_t i) {
  const uint64_t m = 1ull << (i & 63);
  return __atomic_fetch_or(&bits[i >> 6], m, __ATOMIC_RELAXED) & m;
}

// #c in bwt[0, r) for c = 1..5: u64 totals every 2^32 rows, u32 counts relative to them every 64 rows.
struct RankTable {
  static constexpr int SYMS = 5;
  const uint8_t* bwt;
  std::vector<uint64_t> super;
  std::vector<uint32_t> block;
  uint64_t rank(uint8_t c, uint64_t r) const {
    uint64_t k = super[(r >> 32) * SYMS + c - 1] + block[(r >> 6) * SYMS + c - 1];
    for (uint64_t j = r & ~63ull; j < r; ++j) k += bwt[j] == c;
    return k;
  }
};

int verify_index(const uint8_t* text, uint64_t n, const uint8_t* bwt, const uint64_t* less, const uint64_t* sa_sample,
                 uint64_t n_samples, uint64_t rate, const uint64_t* extra_kv, uint64_t n_extra, int n_threads, std::string* msg) {
  Failure fail;
  auto failed = [&]() { *msg = fail.what; return 1; };
  if (n < 4 || n % 2 || n_threads < 1 || rate < 1) { *msg = "bad arguments"; return 1; }
  const uint64_t G = (n - 2) / 2;
  if (text[G] != 0 || text[n - 1] != 0) { *msg = "text is not fwd $ revcomp $"; return 1; }
  // symbol counts of the text and of the BWT, and the BWT's '$' rows
  const uint64_t n_blocks = (n + 63) / 64;
  RankTable rt{bwt, std::vector<uint64_t>(((n >> 32) + 1) * RankTable::SYMS), std::vector<uint32_t>(n_blocks * RankTable::SYMS)};
  std::mutex mu;
  uint64_t text_cnt[8] = {0}, bwt_cnt[8] = {0};
  std::vector<uint64_t> dollar_rows;
  parallel_slices(n_blocks, 1 << 14, n_threads, [&](uint64_t lo, uint64_t hi) {
    uint64_t tc[8] = {0}, bc[8] = {0};
    std::vector<uint64_t> dr;
    for (uint64_t b = lo; b < hi; ++b) {
      uint64_t in_block[8] = {0};
      for (uint64_t i = b * 64; i < std::min(n, b * 64 + 64); ++i) {
        tc[text[i] & 7] += 1;
        if (text[i] > 5) fail.set("text[%llu] = %u is not a symbol rank", (unsigned long long)i, text[i]);
        in_block[bwt[i] & 7] += 1;
        if (bwt[i] > 5) fail.set("row %llu: bwt = %u is not a symbol rank", (unsigned long long)i, bwt[i]);
        if (bwt[i] == 0) dr.push_back(i);
      }
      for (int c = 0; c < 8; ++c) bc[c] += in_block[c];
      for (int c = 1; c <= RankTable::SYMS; ++c) rt.block[b * RankTable::SYMS + c - 1] = (uint32_t)in_block[c];
    }
    std::lock_guard<std::mutex> g(mu);
    for (int c = 0; c < 8; ++c) { text_cnt[c] += tc[c]; bwt_cnt[c] += bc[c]; }
    dollar_rows.insert(dollar_rows.end(), dr.begin(), dr.end());
  });
  if (fail.hit) return failed();
  {  // block counts -> counts before each block, restarting every 2^32 rows
    uint64_t rel[RankTable::SYMS] = {0}, total[RankTable::SYMS] = {0};
    for (uint64_t b = 0; b < n_blocks; ++b) {
      if ((b & ((1ull << 26) - 1)) == 0)
        for (int s = 0; s < RankTable::SYMS; ++s) { rt.super[(b >> 26) * RankTable::SYMS + s] = total[s]; rel[s] = 0; }
      for (int s = 0; s < RankTable::SYMS; ++s) {
        const uint32_t v = rt.block[b * RankTable::SYMS + s];
        rt.block[b * RankTable::SYMS + s] = (uint32_t)rel[s];
        rel[s] += v;
        total[s] += v;
      }
    }
  }
  if (text_cnt[0] != 2) { *msg = "text has " + std::to_string(text_cnt[0]) + " sentinels, not 2"; return 1; }
  for (int c = 0; c < 8; ++c)
    if (bwt_cnt[c] != text_cnt[c]) {
      fail.set("bwt holds %llu symbols of rank %d, the text %llu", (unsigned long long)bwt_cnt[c], c, (unsigned long long)text_cnt[c]);
      return failed();
    }
  {
    uint64_t acc = 0;
    for (int c = 0; c < 8; ++c) {
      if (less[c] != acc) {
        fail.set("less[%d] = %llu, but the text has %llu symbols below rank %d", c, (unsigned long long)less[c], (unsigned long long)acc, c);
        return failed();
      }
      acc += text_cnt[c];
    }
  }
  // sampled rows and the unsampled '$' rows
  if (n_samples != (n + rate - 1) / rate) { fail.set("%llu SA samples, expected %llu", (unsigned long long)n_samples, (unsigned long long)((n + rate - 1) / rate)); return failed(); }
  if (sa_sample[0] != n - 1) { fail.set("row 0: SA sample = %llu, expected n - 1 = %llu", (unsigned long long)sa_sample[0], (unsigned long long)(n - 1)); return failed(); }
  std::vector<uint64_t> extra_rows, extra_pos;
  for (uint64_t i = 0; i < n_extra; ++i) {
    const uint64_t r = extra_kv[2 * i], p = extra_kv[2 * i + 1];
    if (r >= n || p >= n || r % rate == 0 || bwt[r] != 0 || (i && r <= extra_rows.back())) {
      fail.set("extra row %llu (text position %llu): not an unsampled '$' row in increasing order", (unsigned long long)r, (unsigned long long)p);
      return failed();
    }
    extra_rows.push_back(r);
    extra_pos.push_back(p);
  }
  for (uint64_t r : dollar_rows)
    if (r % rate != 0 && !std::binary_search(extra_rows.begin(), extra_rows.end(), r)) {
      fail.set("row %llu: unsampled '$' row missing from the extra rows", (unsigned long long)r);
      return failed();
    }
  // start rows: the samples, the extra rows and row 1 (the first sentinel's suffix G, which no LF step reaches)
  const bool start_row1 = rate > 1;
  const uint64_t n_starts = n_samples + n_extra + (start_row1 ? 1 : 0);
  auto start = [&](uint64_t k, uint64_t* r, uint64_t* p) {
    if (k < n_samples) { *r = k * rate; *p = sa_sample[k]; }
    else if (k < n_samples + n_extra) { *r = extra_rows[k - n_samples]; *p = extra_pos[k - n_samples]; }
    else { *r = 1; *p = G; }
  };
  auto known = [&](uint64_t r, uint64_t* p) {
    if (r % rate == 0) { *p = sa_sample[r / rate]; return true; }
    if (r == 1) { *p = G; return true; }
    auto it = std::lower_bound(extra_rows.begin(), extra_rows.end(), r);
    if (it != extra_rows.end() && *it == r) { *p = extra_pos[it - extra_rows.begin()]; return true; }
    return false;
  };
  std::vector<uint64_t> row_seen(n_blocks, 0), pos_seen(n_blocks, 0);
  enum { GOING, DONE, FAILED };
  // one LF step of a walk at row r, text position p
  auto step = [&](uint64_t& r, uint64_t& p) -> int {
    if (p >= n) { fail.set("row %llu: SA = %llu is past the text end", (unsigned long long)r, (unsigned long long)p); return FAILED; }
    if (test_and_set(row_seen, r)) { fail.set("row %llu reached twice (text position %llu)", (unsigned long long)r, (unsigned long long)p); return FAILED; }
    if (test_and_set(pos_seen, p)) { fail.set("text position %llu reached twice (row %llu)", (unsigned long long)p, (unsigned long long)r); return FAILED; }
    const uint8_t c = bwt[r], want = text[p ? p - 1 : n - 1];
    if (c != want) {
      fail.set("row %llu (text position %llu): bwt = %u, but the text before it is %u", (unsigned long long)r, (unsigned long long)p, c, want);
      return FAILED;
    }
    if (c == 0) return DONE;
    const uint64_t from = r;
    r = less[c] + rt.rank(c, r);
    p -= 1;
    uint64_t kp;
    if (r >= n) { fail.set("row %llu: LF leaves the table (%llu)", (unsigned long long)from, (unsigned long long)r); return FAILED; }
    if (known(r, &kp)) {
      if (kp != p) {
        fail.set("row %llu: SA = %llu, but LF from row %llu reaches it at text position %llu", (unsigned long long)r, (unsigned long long)kp,
                 (unsigned long long)from, (unsigned long long)p);
        return FAILED;
      }
      return DONE;
    }
    __builtin_prefetch(&bwt[r]);
    __builtin_prefetch(&rt.block[(r >> 6) * RankTable::SYMS]);
    __builtin_prefetch(&row_seen[r >> 6]);
    return GOING;
  };
  // each thread advances W walks in turn, so that the cache misses of one step overlap with the others' work
  parallel_slices(n_starts, 4096, n_threads, [&](uint64_t lo, uint64_t hi) {
    constexpr int W = 16;
    uint64_t wr[W], wp[W];
    int live = 0;
    for (; live < W && lo < hi; ++live) start(lo++, &wr[live], &wp[live]);
    while (live > 0) {
      if (fail.hit.load(std::memory_order_relaxed)) return;
      for (int i = 0; i < live;) {
        const int s = step(wr[i], wp[i]);
        if (s == FAILED) return;
        if (s == DONE) {
          if (lo < hi) start(lo++, &wr[i], &wp[i]);
          else { wr[i] = wr[live - 1]; wp[i] = wp[live - 1]; --live; continue; }
        }
        ++i;
      }
    }
  });
  if (fail.hit) return failed();
  for (uint64_t b = 0; b < n_blocks; ++b) {
    const uint64_t full = b + 1 < n_blocks || n % 64 == 0 ? ~0ull : (1ull << (n % 64)) - 1;
    if (row_seen[b] != full) {
      fail.set("row %llu is not reached from any sampled row", (unsigned long long)(b * 64 + __builtin_ctzll(~row_seen[b])));
      return failed();
    }
  }
  return 0;
}

}  // namespace

extern "C" {

// ---- index -------------------------------------------------------------------------------
void* ora_index_build(uint64_t n_contigs, const char* const* names, const char* const* seqs, const uint64_t* lens,
                      int with_x, uint32_t occ_k, uint64_t sa_rate, int keep_full_sa, const char* draws,
                      uint64_t n_draws) {
  GenomeInput g;
  for (uint64_t i = 0; i < n_contigs; ++i) {
    g.names.push_back(names && names[i] ? names[i] : "");
    g.seqs.push_back(std::string(seqs[i], seqs[i] + lens[i]));
  }
  Index* ix = new Index();
  DrawState ds{draws, (size_t)n_draws, 0};
  build_index(*ix, g, with_x != 0, occ_k, sa_rate, keep_full_sa != 0, draw_replace, &ds);
  return ix;
}
// Adopt arrays produced by the product's index builder (so large parity runs share one index).
void* ora_index_from_arrays(const uint8_t* bwt, uint64_t n, int with_x, uint32_t occ_k, const uint64_t* sa_sample,
                            uint64_t n_samples, uint64_t sa_rate, const uint64_t* extra_kv, uint64_t n_extra,
                            uint64_t n_contigs, const uint64_t* cstart, const uint64_t* cend, const char* const* cname,
                            const uint64_t* orig_pos, const uint8_t* orig_sym, uint64_t n_orig) {
  Index* ix = new Index();
  index_from_arrays(*ix, bwt, n, with_x != 0, occ_k, sa_sample, n_samples, sa_rate, extra_kv, n_extra);
  for (uint64_t i = 0; i < n_contigs; ++i) ix->contigs.push_back(Contig{cstart[i], cend[i], cname && cname[i] ? cname[i] : ""});
  for (uint64_t i = 0; i < n_orig; ++i) ix->original_symbols[orig_pos[i]] = orig_sym[i];
  return ix;
}
void ora_index_free(void* h) { delete (Index*)h; }
uint64_t ora_index_n(void* h) { return ((Index*)h)->n; }
const uint8_t* ora_index_bwt(void* h) { return ((Index*)h)->bwt.data(); }
uint64_t ora_index_less(void* h, uint64_t* out, uint64_t cap) {
  Index* ix = (Index*)h;
  for (size_t i = 0; i < ix->less.size() && i < cap; ++i) out[i] = ix->less[i];
  return ix->less.size();
}
void ora_index_sentinel_rows(void* h, uint64_t* out) { out[0] = ((Index*)h)->sentinel_occ[0]; out[1] = ((Index*)h)->sentinel_occ[1]; }
uint64_t ora_index_sa_samples(void* h, const uint64_t** out) { *out = ((Index*)h)->sa_sample.data(); return ((Index*)h)->sa_sample.size(); }
uint64_t ora_index_full_sa(void* h, const uint64_t** out) { *out = ((Index*)h)->full_sa.data(); return ((Index*)h)->full_sa.size(); }
uint64_t ora_index_extra_rows(void* h, uint64_t* kv_out, uint64_t cap_pairs) {
  Index* ix = (Index*)h;
  uint64_t i = 0;
  for (auto& kv : ix->extra_rows) { if (i < cap_pairs) { kv_out[2 * i] = kv.first; kv_out[2 * i + 1] = kv.second; } ++i; }
  return i;
}
uint64_t ora_index_original_symbols(void* h, uint64_t* pos_out, uint8_t* sym_out, uint64_t cap) {
  Index* ix = (Index*)h;
  uint64_t i = 0;
  for (auto& kv : ix->original_symbols) { if (i < cap) { pos_out[i] = kv.first; sym_out[i] = kv.second; } ++i; }
  return i;
}
uint64_t ora_index_occ(void* h, uint64_t r, uint8_t a) { return ((Index*)h)->occ(r, a); }
// Independent check of a BWT + sampled SA (any builder's) against the rank text `fwd $ revcomp $` ($ = 0, A..T = 1..4,
// X = 5).  It walks LF from every row whose text position is known (the sampled rows, the extra rows and row 1, the first
// sentinel's suffix) to the next known row or '$' row: each row it passes must hold the text symbol before its position,
// each row and each position must be reached exactly once, and every known row must be reached at its own position.
// With `less` equal to the text's symbol counts, these local conditions force the suffix order.  Uses its own rank
// table, no Index.  Returns 0 if the arrays are the index of `text`, else 1 and a message naming a wrong row.
int ora_verify_index(const uint8_t* text, uint64_t n, const uint8_t* bwt, const uint64_t* less8, const uint64_t* sa_sample,
                     uint64_t n_samples, uint64_t sa_rate, const uint64_t* extra_kv, uint64_t n_extra, int n_threads, char* msg,
                     uint64_t cap) {
  std::string m;
  int rc = verify_index(text, n, bwt, less8, sa_sample, n_samples, sa_rate, extra_kv, n_extra, n_threads, &m);
  snprintf(msg, cap, "%s", m.c_str());
  return rc;
}
int ora_index_sa_get(void* h, uint64_t row, uint64_t* out) { usize v = 0; bool ok = ((Index*)h)->sa_get(row, &v, nullptr); *out = v; return ok; }
void ora_index_extend(void* h, uint64_t lower, uint64_t lower_rev, uint64_t size, uint64_t* out12) {
  BiInterval o[4];
  ((Index*)h)->extend_all(BiInterval{lower, lower_rev, size}, o);
  for (int k = 0; k < 4; ++k) { out12[3 * k] = o[k].lower; out12[3 * k + 1] = o[k].lower_rev; out12[3 * k + 2] = o[k].size; }
}

// ---- params ------------------------------------------------------------------------------
void* ora_params_new() { return new Params(); }
void ora_params_free(void* p) { delete (Params*)p; }
void ora_params_model_simple(void* p, int library, float f, float t, float d, float s, float divergence, int ignore_q) {
  ((Params*)p)->sdm.init_simple(library, f, t, d, s, divergence, ignore_q != 0);
}
void ora_params_model_vindija(void* p) { ((Params*)p)->sdm = Sdm(); ((Params*)p)->sdm.kind = SDM_VINDIJA; }
void ora_params_model_test(void* p, float deam, float mm, float match) {
  Sdm& s = ((Params*)p)->sdm; s = Sdm(); s.kind = SDM_TEST; s.deam_score = deam; s.mm_score = mm; s.match_score = match;
}
float ora_params_repr_mm(void* p) { return ((Params*)p)->sdm.representative_mismatch_penalty(); }
void ora_params_bound_discrete(void* p, float thr, float rate, float repr_mm) { ((Params*)p)->mb.init_discrete(thr, rate, repr_mm); }
void ora_params_bound_continuous(void* p, float cutoff, float exponent, float repr_mm) { ((Params*)p)->mb.init_continuous(cutoff, exponent, repr_mm); }
void ora_params_bound_test(void* p, float thr, float rmb) { ((Params*)p)->mb.init_test(thr, rmb); }
void ora_params_gaps(void* p, float open, float extend, int dist_ends, int max_open, int abort_on_limit) {
  Params* q = (Params*)p;
  q->penalty_gap_open = open; q->penalty_gap_extend = extend;
  q->gap_dist_ends = (uint8_t)dist_ends; q->max_num_gaps_open = (uint8_t)max_open; q->stack_limit_abort = abort_on_limit != 0;
}
void ora_params_limits(void* p, uint32_t stack_limit, uint32_t tree_limit) {
  ((Params*)p)->stack_limit = stack_limit; ((Params*)p)->edit_tree_limit = tree_limit;
}
float ora_sdm_get(void* p, uint64_t i, uint64_t L, uint8_t from, uint8_t to, uint8_t q) { return ((Params*)p)->sdm.get(i, L, from, to, q); }
float ora_sdm_min_penalty(void* p, uint64_t i, uint64_t L, uint8_t to, uint8_t q, int only_mm) { return ((Params*)p)->sdm.get_min_penalty(i, L, to, q, only_mm != 0); }
int ora_sdm_alignment_start(void* p, uint64_t L) { return ((Params*)p)->sdm.find_alignment_start(L); }
float ora_bound_discrete_get(void* p, uint64_t L) { return ((Params*)p)->mb.discrete_get(L); }
int ora_bound_reject(void* p, float v, uint64_t L) { return ((Params*)p)->mb.reject(v, L); }
float ora_bound_remaining_frac(void* p, float v, uint64_t L) { return ((Params*)p)->mb.remaining_frac_of_repr_mm(v, L); }
float ora_log2f(float x) { return log2f(x); }
float ora_exp2f(float x) { return exp2f(x); }
float ora_log10f(float x) { return log10f(x); }

// ---- D array -------------------------------------------------------------------------------
// split < 0 => the model's find_alignment_start
uint64_t ora_d_array(void* ixh, void* ph, const uint8_t* seq, const uint8_t* qual, uint64_t L, int64_t split, float* out,
                     uint64_t* ext_steps) {
  Params* p = (Params*)ph;
  BiDArray d;
  Counters c;
  usize sp = split < 0 ? (usize)p->sdm.find_alignment_start(L) : (usize)split;
  d.build(seq, qual, L, sp, *p, *(Index*)ixh, &c);
  for (usize i = 0; i < L; ++i) out[i] = d.d_composite[i];
  if (ext_steps) *ext_steps = c.d_ext_steps;
  return sp;
}
float ora_d_array_get(void* ixh, void* ph, const uint8_t* seq, const uint8_t* qual, uint64_t L, int64_t split, int k, int l) {
  Params* p = (Params*)ph;
  BiDArray d;
  usize sp = split < 0 ? (usize)p->sdm.find_alignment_start(L) : (usize)split;
  d.build(seq, qual, L, sp, *p, *(Index*)ixh, nullptr);
  return d.get((int16_t)k, (int16_t)l);
}

// ---- heaps (exposed so tests can pin their order on plain float sequences) ---------------
struct FKey { float k; uint32_t id; float key() const { return k; } };
void* ora_mmheap_new() { return new MinMaxHeap<FKey>(); }
void ora_mmheap_free(void* h) { delete (MinMaxHeap<FKey>*)h; }
void ora_mmheap_push(void* h, float k, uint32_t id) { ((MinMaxHeap<FKey>*)h)->push(FKey{k, id}); }
int ora_mmheap_pop_max(void* h, float* k, uint32_t* id) { FKey f; if (!((MinMaxHeap<FKey>*)h)->pop_max(&f)) return 0; *k = f.k; *id = f.id; return 1; }
int ora_mmheap_pop_min(void* h, float* k, uint32_t* id) { FKey f; if (!((MinMaxHeap<FKey>*)h)->pop_min(&f)) return 0; *k = f.k; *id = f.id; return 1; }
uint64_t ora_mmheap_len(void* h) { return ((MinMaxHeap<FKey>*)h)->len(); }
uint64_t ora_mmheap_dump(void* h, float* keys, uint32_t* ids, uint64_t cap) {
  auto* m = (MinMaxHeap<FKey>*)h;
  for (size_t i = 0; i < m->d.size() && i < cap; ++i) { keys[i] = m->d[i].k; ids[i] = m->d[i].id; }
  return m->d.size();
}
void* ora_binheap_new() { return new BinaryHeap<FKey>(); }
void ora_binheap_free(void* h) { delete (BinaryHeap<FKey>*)h; }
void ora_binheap_push(void* h, float k, uint32_t id) { ((BinaryHeap<FKey>*)h)->push(FKey{k, id}); }
int ora_binheap_pop(void* h, float* k, uint32_t* id) { FKey f; if (!((BinaryHeap<FKey>*)h)->pop(&f)) return 0; *k = f.k; *id = f.id; return 1; }
uint64_t ora_binheap_dump(void* h, float* keys, uint32_t* ids, uint64_t cap) {
  auto* m = (BinaryHeap<FKey>*)h;
  for (size_t i = 0; i < m->d.size() && i < cap; ++i) { keys[i] = m->d[i].k; ids[i] = m->d[i].id; }
  return m->d.size();
}
uint64_t ora_binheap_into_sorted(void* h, float* keys, uint32_t* ids, uint64_t cap) {
  auto v = ((BinaryHeap<FKey>*)h)->into_sorted_vec();
  for (size_t i = 0; i < v.size() && i < cap; ++i) { keys[i] = v[i].k; ids[i] = v[i].id; }
  return v.size();
}

// ---- PrRange -------------------------------------------------------------------------------
// Returns the number of values written (<= cap); -1 if try_new returned None.
int64_t ora_prrange(uint64_t start, uint64_t end, uint64_t seed, uint64_t* out, uint64_t cap) {
  PrRange r = PrRange::try_new(start, end, seed);
  if (!r.valid) return -1;
  uint64_t n = 0;
  usize v;
  while (r.next(&v)) { if (n < cap) out[n] = v; ++n; }
  return (int64_t)n;
}
uint32_t ora_draw_u32(uint32_t seed, uint32_t k) { return draw_u32(seed, k); }

// ---- to_bam_fields on an explicit track ------------------------------------------------------
// ops: (pos, kind, base) triples.  Writes "CIGAR\tMD\tNM" into buf.
int ora_to_bam_fields(void* ixh, const mapad_edit_op* ops, uint64_t n, int backward, uint64_t absolute_pos, char* buf,
                      uint64_t cap) {
  std::vector<EditOp> t;
  for (uint64_t i = 0; i < n; ++i) { EditOp e; e.pos = ops[i].pos; e.kind = ops[i].kind; e.base = ops[i].base; t.push_back(e); }
  std::vector<CigarOp> c; std::string md; uint16_t nm;
  Index empty;
  to_bam_fields(t, backward != 0, absolute_pos, ixh ? *(Index*)ixh : empty, &c, &md, &nm);
  std::string s = cigar_string(c) + "\t" + md + "\t" + std::to_string(nm);
  snprintf(buf, cap, "%s", s.c_str());
  return (int)s.size();
}

// ---- batch mapping -------------------------------------------------------------------------
void* ora_map_batch(void* ixh, void* ph, uint64_t n_reads, const uint8_t* seq, const uint8_t* qual, const uint64_t* offsets,
                    const uint32_t* seeds, int n_threads, int want_hits) {
  const Index& ix = *(Index*)ixh;
  const Params& p = *(Params*)ph;
  std::vector<PerRead> per(n_reads);
  if (n_threads < 1) n_threads = 1;
  std::atomic<uint64_t> next(0);
  auto worker = [&]() {
    Scratch scratch;  // thread-local buffers like STACK_BUF / TREE_BUF (mapping.rs:146-149)
    while (true) {
      uint64_t lo = next.fetch_add(64);
      if (lo >= n_reads) break;
      uint64_t hi = std::min<uint64_t>(lo + 64, n_reads);
      for (uint64_t r = lo; r < hi; ++r)
        map_one(ix, p, seq + offsets[r], qual + offsets[r], offsets[r + 1] - offsets[r], seeds ? seeds[r] : 0u, scratch,
                per[r], want_hits != 0);
    }
  };
  std::vector<std::thread> th;
  for (int t = 1; t < n_threads; ++t) th.emplace_back(worker);
  worker();
  for (auto& t : th) t.join();
  BatchOut* out = new BatchOut();
  out->records.resize(n_reads);
  out->xa_off.push_back(0);
  for (uint64_t r = 0; r < n_reads; ++r) {
    PerRead& pr = per[r];
    mapad_record m = pr.rec;
    uint32_t cig_base = (uint32_t)out->cigar.size(), text_base = (uint32_t)out->text.size();
    m.cigar_off += cig_base; m.md_off += text_base;
    for (uint32_t a = 0; a < m.n_alts; ++a) { m.alts[a].cigar_off += cig_base; m.alts[a].md_off += text_base; }
    m.hit_off = (uint32_t)out->hits.size();
    uint32_t op_base = (uint32_t)out->edit_ops.size();
    for (mapad_hit h : pr.hits) { h.edit_off += op_base; out->hits.push_back(h); }
    out->edit_ops.insert(out->edit_ops.end(), pr.ops.begin(), pr.ops.end());
    out->cigar.insert(out->cigar.end(), pr.cigar.begin(), pr.cigar.end());
    out->text.insert(out->text.end(), pr.text.begin(), pr.text.end());
    out->xa_flat.insert(out->xa_flat.end(), pr.xa.begin(), pr.xa.end());
    out->xa_off.push_back(out->xa_flat.size());
    out->records[r] = m;
  }
  return out;
}
void ora_batch_free(void* b) { delete (BatchOut*)b; }
void ora_batch_view(void* b, mapad_results* out) {
  BatchOut* o = (BatchOut*)b;
  memset(out, 0, sizeof *out);
  out->n_reads = o->records.size();
  out->records = o->records.data();
  out->hits = o->hits.data(); out->n_hits = o->hits.size();
  out->edit_ops = o->edit_ops.data(); out->n_edit_ops = o->edit_ops.size();
  out->cigar = o->cigar.data(); out->n_cigar = o->cigar.size();
  out->text = o->text.data(); out->n_text = o->text.size();
}
uint64_t ora_batch_xa(void* b, const char** flat, const uint64_t** offs) {
  BatchOut* o = (BatchOut*)b;
  *flat = o->xa_flat.data(); *offs = o->xa_off.data();
  return o->xa_off.size();
}

}  // extern "C"

// epilogue_core.cuh — per-read epilogue: best-hit choice, SA locate in PrRange order, strand and
// contig coordinates, MAPQ, CIGAR / MD / NM, alternative-hit summary.  Dual-compilable.
//
// Reference functions restated (under /root/reference/src/map/):
//   intervals_to_bam            mapping.rs:402-567
//   interval2coordinate         mapping.rs:590-649
//   interval_cross_check        mapping.rs:651-653
//   estimate_mapping_quality    mapping.rs:658-718
//   PrRange                     prrange.rs:6-184
//   EditOperationsTrack::{to_bam_fields, effective_len}   record.rs:269-428
//   MismatchBound::remaining_frac_of_repr_mm   mismatch_bounds.rs:93-97,140-144,278-280
#pragma once
#include <cmath>
#include <cstdint>

#include "search_core.cuh"

namespace mapad {

MAPAD_DEV uint32_t atomic_add_u32(uint32_t* p, uint32_t v) {
#if defined(__CUDA_ARCH__)
  return atomicAdd(p, v);
#else
  uint32_t o = *p; *p += v; return o;
#endif
}

// The reference seeds PrRange from an UNSEEDED thread-local RNG (mapping.rs:273,605).  For
// reproducible parity the k-th draw of a read is derived from the per-read seed of the batch.
MAPAD_DEV uint32_t draw_u32(uint32_t read_seed, uint32_t k) {
  uint64_t z = (((uint64_t)read_seed << 32) | k) + 0x9E3779B97F4A7C15ull;
  z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
  z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
  z = z ^ (z >> 31);
  return (uint32_t)(z >> 32);
}

// ---- PrRange (prrange.rs) ---------------------------------------------------------------------
struct PrRangeDev {
  uint64_t start, l, m, a, x, seed, count;
  bool valid;
};
MAPAD_DEV bool pr_is_prime(uint64_t n) {
  if (n <= 1) return false;
  if (n <= 3) return true;
  if (n % 2 == 0 || n % 3 == 0) return false;
  for (uint64_t i = 5; i * i <= n; i += 6)
    if (n % i == 0 || n % (i + 2) == 0) return false;
  return true;
}
MAPAD_DEV uint64_t pr_next_prime(uint64_t n) {
  uint64_t p = n + 1;
  if (p <= 2) return 2;
  if (p % 2 == 0) p += 1;
  while (!pr_is_prime(p)) p += 2;
  return p;
}
MAPAD_DEV bool pr_pow_mod(uint64_t base, uint64_t exponent, uint64_t modulus, uint64_t& out) {
  if (modulus == 1) { out = 0; return true; }
  if (modulus - 1 > 0xffffffffull) return false;  // (modulus-1).checked_mul(modulus-1) overflows
  uint64_t result = 1;
  base %= modulus;
  while (exponent > 0) {
    if (exponent % 2 == 1) result = (result * base) % modulus;
    exponent >>= 1;
    base = (base * base) % modulus;
  }
  out = result;
  return true;
}
// is_primitive_root with the reference's PrimeFactorIterator (prrange.rs:107-159) unrolled into it
MAPAD_DEV bool pr_is_primitive_root(uint64_t a, uint64_t n, bool& ok) {
  const uint64_t phi = n - 1;
  uint64_t fn = phi, fi = 2, fstep = 1, flast = 0;
  ok = true;
  while (true) {
    // PrimeFactorIterator::next
    if (fn <= 3) return true;
    bool yielded = false;
    uint64_t pf = 0;
    while (fi * fi <= fn && !yielded) {
      while (fn > 1 && !yielded) {
        while (fn % fi == 0) {
          if (fi > flast) { pf = fi; flast = fi; yielded = true; break; }
          fn /= fi;
        }
        if (yielded) break;
        fi += fstep;
        fstep = 2;
      }
    }
    if (!yielded) return true;
    uint64_t r;
    if (!pr_pow_mod(a, phi / pf, n, r)) { ok = false; return false; }
    if (r == 1) return false;
  }
}
MAPAD_DEV PrRangeDev pr_new(uint64_t start, uint64_t end, uint64_t seed) {
  PrRangeDev r;
  r.valid = false; r.start = start; r.l = 0; r.m = 0; r.a = 0; r.x = 0; r.seed = 0; r.count = 0;
  uint64_t l = end > start ? end - start : 0;
  if (l == 0) return r;
  uint64_t m = pr_next_prime(l);
  uint64_t a = 2;
  while (true) {
    bool ok;
    bool pr = pr_is_primitive_root(a, m, ok);
    if (!ok) return r;
    if (pr) break;
    a += 1;
  }
  uint64_t sd = seed % l;
  if (sd < 1) sd = 1;
  r.l = l; r.m = m; r.a = a; r.x = sd; r.seed = sd; r.valid = true;
  return r;
}
MAPAD_DEV bool pr_next(PrRangeDev& r, uint64_t& out) {
  if (r.count == 0 && r.l == 1) { r.count += 1; out = r.start; return true; }
  while (true) {
    uint64_t prev_x = r.x;
    r.x = (r.a * r.x) % r.m;
    if (r.count > 0 && prev_x == r.seed) return false;
    if (prev_x <= r.l) { r.count += 1; out = prev_x - 1 + r.start; return true; }
  }
}

// ---- coordinates -------------------------------------------------------------------------------
struct CoordDev {
  int32_t tid;
  uint64_t rel, abs;
  int backward;
  uint64_t num_skipped;
};
struct CoordIterDev {
  PrRangeDev pr;
  uint64_t enum_i;
  uint64_t eff_len;
  uint32_t hit;  // index into the read's hit span
};
MAPAD_DEV uint32_t effective_len(const mapad_edit_op* ops, uint32_t n) {
  uint32_t e = 0;
  for (uint32_t i = 0; i < n; ++i) e += ops[i].kind != MAPAD_ED_INSERTION;
  return e;
}
template <bool WIDE>
MAPAD_DEV bool coord_next(const DevIndex& ix, CoordIterDev& it, CoordDev& out, uint32_t& lf_steps) {
  uint64_t row;
  while (it.pr.valid && pr_next(it.pr, row)) {
    uint64_t i = it.enum_i++;
    if (row >= ix.m.n) continue;
    uint64_t abs = sa_get<WIDE>(ix, row, lf_steps);
    const uint64_t strand_len = ix.m.n / 2;
    int backward = 0;
    if (abs >= strand_len) { abs = ix.m.n - abs - it.eff_len - 1; backward = 1; }
    int32_t tid; uint64_t rel;
    if (reference_identifier(ix, abs, it.eff_len, tid, rel)) {
      out.tid = tid; out.rel = rel; out.abs = abs; out.backward = backward; out.num_skipped = i;
      return true;
    }
  }
  return false;
}

// ---- CIGAR / MD / NM ---------------------------------------------------------------------------
struct OutPools {
  uint32_t* cigar; uint32_t cigar_cap; uint32_t* cigar_cursor;
  char* text; uint32_t text_cap; uint32_t* text_cursor;
  uint32_t* overflow;
};
MAPAD_DEV uint32_t dec_digits(uint32_t v) { uint32_t d = 1; while (v >= 10) { v /= 10; ++d; } return d; }
MAPAD_DEV void dec_write(char* dst, uint32_t v, uint32_t nd) { for (uint32_t i = nd; i-- > 0;) { dst[i] = (char)('0' + v % 10); v /= 10; } }

template <bool WRITE>
MAPAD_DEV void bam_fields_pass(const DevIndex& ix, const mapad_edit_op* ops, uint32_t n, int backward, uint64_t absolute_pos,
                               uint32_t* cig_out, char* md_out, uint32_t& n_cig, uint32_t& n_md, uint32_t& nm) {
  uint32_t num_matches = 0, num_operations = 1, edit_distance = 0;
  bool have_last = false;
  int last_kind = 0;  // class: 0 M, 1 I, 2 D
  bool last_is_del = false;
  n_cig = 0; n_md = 0;
  auto emit_cigar = [&](int cls, uint32_t len) {
    if (WRITE) cig_out[n_cig] = len << 4 | (uint32_t)cls;
    n_cig += 1;
  };
  auto emit_num = [&](uint32_t k) {
    uint32_t nd = dec_digits(k);
    if (WRITE) dec_write(md_out + n_md, k, nd);
    n_md += nd;
  };
  auto emit_char = [&](char ch) {
    if (WRITE) md_out[n_md] = ch;
    n_md += 1;
  };
  for (uint32_t i = 0; i < n; ++i) {
    mapad_edit_op op = backward ? ops[n - 1 - i] : ops[i];
    if (op.kind != MAPAD_ED_INSERTION && ix.m.n_orig != 0) {  // record.rs:301-321
      uint8_t orig;
      if (original_symbol(ix, absolute_pos + i, orig)) {
        if (op.kind == MAPAD_ED_MATCH) op.kind = MAPAD_ED_MISMATCH;
        op.base = orig;
      }
    }
    if (op.kind != MAPAD_ED_MATCH) edit_distance += 1;
    // add_md_edit_operation (record.rs:383-419); `last` is the first operation of the current CIGAR run
    if (op.kind == MAPAD_ED_MATCH) num_matches += 1;
    else if (op.kind == MAPAD_ED_MISMATCH) {
      emit_num(num_matches);
      emit_char((char)(backward ? complement_iupac(op.base) : op.base));
      num_matches = 0;
    } else if (op.kind == MAPAD_ED_DELETION) {
      char b = (char)(backward ? complement_iupac(op.base) : op.base);
      if (have_last && last_is_del) emit_char(b);
      else { emit_num(num_matches); emit_char('^'); emit_char(b); }
      num_matches = 0;
    }
    int cls = op.kind == MAPAD_ED_INSERTION ? 1 : (op.kind == MAPAD_ED_DELETION ? 2 : 0);
    if (have_last) {
      if (cls == last_kind) num_operations += 1;
      else { emit_cigar(last_kind, num_operations); num_operations = 1; last_kind = cls; last_is_del = cls == 2; }
    } else {
      have_last = true; last_kind = cls; last_is_del = cls == 2;
    }
  }
  if (have_last) emit_cigar(last_kind, num_operations);
  emit_num(num_matches);
  nm = edit_distance;
}

template <bool WIDE>
MAPAD_DEV void emit_bam_fields(const DevIndex& ix, const OutPools& pools, const mapad_edit_op* ops, uint32_t n, int backward,
                               uint64_t absolute_pos, uint32_t& cigar_off, uint32_t& cigar_len, uint32_t& md_off, uint32_t& md_len,
                               int32_t& nm_out) {
  uint32_t nc, nmd, nm;
  bam_fields_pass<false>(ix, ops, n, backward, absolute_pos, nullptr, nullptr, nc, nmd, nm);
  uint32_t co = atomic_add_u32(pools.cigar_cursor, nc);
  uint32_t to = atomic_add_u32(pools.text_cursor, nmd);
  cigar_off = co; cigar_len = nc; md_off = to; md_len = nmd; nm_out = (int32_t)nm;
  if ((uint64_t)co + nc > pools.cigar_cap || (uint64_t)to + nmd > pools.text_cap) { *pools.overflow = 1; return; }
  uint32_t a, b, c;
  bam_fields_pass<true>(ix, ops, n, backward, absolute_pos, pools.cigar + co, pools.text + to, a, b, c);
}

MAPAD_DEV bool interval_cross_check(const mapad_hit& a, const mapad_hit& b) {
  return a.size == b.size && (a.lower == b.lower || a.lower_rev == b.lower_rev);
}

MAPAD_DEV uint8_t round_to_u8(float v) {  // `.round() as u8`: half away from zero, saturating, NaN -> 0
  if (v != v) return 0;
  float r = roundf(v);
  if (r <= 0.0f) return 0;
  if (r >= 255.0f) return 255;
  return (uint8_t)r;
}

MAPAD_DEV float remaining_frac(const DevParams& P, const float* bound_table, float value, int read_length) {
  float tv = (uint32_t)read_length < P.bound_table_len ? bound_table[read_length] : 0.0f;
  if (P.bound_kind == BOUND_DISCRETE) return fdiv_rn(fma_rn(tv, P.repr_mm, -value), P.repr_mm);
  if (P.bound_kind == BOUND_CONTINUOUS) return fdiv_rn(fsub(P.cutoff, fdiv_rn(value, tv)), fdiv_rn(P.repr_mm, tv));
  return fdiv_rn(fsub(P.test_threshold, value), P.test_repr_mm);
}

struct SortKey { float score; uint32_t idx; };

// intervals_to_bam for one read.  `hits`/`ops_pool`: the read's hit span in BinaryHeap vector order.
template <bool WIDE>
MAPAD_DEV void epilogue_read(const DevIndex& ix, const DevParams& P, const float* bound_table, int L, uint32_t read_seed,
                             const mapad_hit* hits, uint32_t n_hits, const mapad_edit_op* ops_pool, const OutPools& pools,
                             mapad_record& rec) {
  rec.mapped = 0; rec.tid = -1; rec.pos = -1; rec.strand = 0; rec.mapq = 0; rec.alignment_score = 0.0f; rec.nm = 0;
  rec.x0 = 0; rec.x1 = 0; rec.xs = 0.0f; rec.xt = 0;
  rec.cigar_off = 0; rec.cigar_len = 0; rec.md_off = 0; rec.md_len = 0; rec.n_alts = 0;
  rec.best_lower = 0; rec.best_lower_rev = 0; rec.best_size = 0; rec.absolute_pos = 0;
  for (int a = 0; a < 2; ++a) {
    rec.alts[a].tid = 0; rec.alts[a].strand = 0; rec.alts[a].pos = 0; rec.alts[a].cigar_off = 0; rec.alts[a].cigar_len = 0;
    rec.alts[a].md_off = 0; rec.alts[a].md_len = 0; rec.alts[a].nm = 0; rec.alts[a].alignment_score = 0.0f; rec.alts[a].interval_size = 0;
  }
  uint32_t lf_steps = 0;
  SortKey sorted[MAPAD_MAX_HITS];
  uint32_t n = n_hits < MAPAD_MAX_HITS ? n_hits : MAPAD_MAX_HITS;
  for (uint32_t i = 0; i < n; ++i) sorted[i] = SortKey{hits[i].alignment_score, i};
  bh_into_sorted(sorted, n);  // into_sorted_vec (mapping.rs:419)
  uint32_t draw_k = 0;
  while (n > 0) {
    const uint32_t bi = sorted[n - 1].idx;  // intervals.pop()
    n -= 1;
    const mapad_hit& best = hits[bi];
    CoordIterDev best_it;
    best_it.eff_len = effective_len(ops_pool + best.edit_off, best.edit_len);
    best_it.enum_i = 0; best_it.hit = bi;
    best_it.pr = pr_new(best.lower, best.lower + best.size, (uint64_t)draw_u32(read_seed, draw_k++));
    CoordDev bc;
    if (!coord_next<WIDE>(ix, best_it, bc, lf_steps)) continue;  // mapping.rs:541-544
    const uint64_t updated_size = best.size - bc.num_skipped;
    // alternative hits (mapping.rs:436-491)
    {
      uint32_t n_alts = 0;
      uint32_t sub_idx = n;  // iterate the remaining (sub-optimal) intervals best-first
      CoordIterDev sub_it;
      sub_it.pr.valid = false; sub_it.enum_i = 0; sub_it.eff_len = 0; sub_it.hit = 0;
      bool sub_active = false, best_phase = true;
      while (n_alts < 2) {
        CoordDev c;
        bool got = false;
        uint32_t from_hit = bi;
        if (best_phase) {
          if (coord_next<WIDE>(ix, best_it, c, lf_steps)) got = true; else best_phase = false;
        }
        if (!got && !best_phase) {
          while (true) {
            if (sub_active) {
              if (coord_next<WIDE>(ix, sub_it, c, lf_steps)) { got = true; from_hit = sub_it.hit; break; }
              sub_active = false;
            }
            bool found = false;
            while (sub_idx > 0) {
              sub_idx -= 1;
              if (!interval_cross_check(best, hits[sorted[sub_idx].idx])) { found = true; break; }
            }
            if (!found) break;
            const mapad_hit& sh = hits[sorted[sub_idx].idx];
            sub_it.hit = sorted[sub_idx].idx;
            sub_it.eff_len = effective_len(ops_pool + sh.edit_off, sh.edit_len);
            sub_it.enum_i = 0;
            sub_it.pr = pr_new(sh.lower, sh.lower + sh.size, (uint64_t)draw_u32(read_seed, draw_k++));
            if (!sub_it.pr.valid) continue;
            sub_active = true;
          }
        }
        if (!got) break;
        const mapad_hit& ah = hits[from_hit];
        mapad_alt& alt = rec.alts[n_alts];
        alt.tid = c.tid; alt.strand = c.backward; alt.pos = (int64_t)c.rel;
        emit_bam_fields<WIDE>(ix, pools, ops_pool + ah.edit_off, ah.edit_len, c.backward, c.abs, alt.cigar_off, alt.cigar_len,
                              alt.md_off, alt.md_len, alt.nm);
        alt.alignment_score = ah.alignment_score;
        alt.interval_size = ah.size;
        n_alts += 1;
      }
      rec.n_alts = n_alts;
    }
    rec.x0 = updated_size > 0x7fffffffull ? 0x7fffffff : (int32_t)updated_size;
    uint64_t x1 = 0;
    for (uint32_t i = 0; i < n; ++i) {
      const mapad_hit& h = hits[sorted[i].idx];
      if (!interval_cross_check(best, h)) x1 += h.size;
    }
    rec.x1 = x1 > 0x7fffffffull ? 0x7fffffff : (int32_t)x1;
    rec.xs = n > 0 ? hits[sorted[n - 1].idx].alignment_score : 0.0f;
    rec.xt = updated_size == 0 ? 'N' : (updated_size == 1 ? 'U' : 'R');
    // estimate_mapping_quality (mapping.rs:658-718)
    {
      const float prob_best = emu::exp2f_glibc(best.alignment_score);
      float ap;
      if (updated_size > 1) ap = fdiv_rn(1.0f, (float)updated_size);
      else {
        float acc = 0.0f;
        for (uint32_t i = 0; i < n; ++i) {
          const mapad_hit& h = hits[sorted[i].idx];
          if (interval_cross_check(best, h)) continue;
          acc = fma_rn(emu::exp2f_glibc(h.alignment_score), (float)h.size, acc);
        }
        ap = fdiv_rn(prob_best, fadd(prob_best, acc));
      }
      if (ap < 0.0f) ap = 0.0f;
      if (ap > 1.0f) ap = 1.0f;
      float q = fmul(-10.0f, emu::log10f_glibc(fsub(1.0f, ap)));
      q = fmin_rs(q, 37.0f);
      uint8_t mq = round_to_u8(q);
      if (mq == 37) {
        float frac = fmin_rs(remaining_frac(P, bound_table, best.alignment_score, L), 1.0f);
        mq = round_to_u8(fma_rn(17.0f, frac, 20.0f));
      }
      rec.mapq = mq;
    }
    rec.mapped = 1;
    rec.tid = bc.tid; rec.pos = (int64_t)bc.rel; rec.strand = bc.backward; rec.absolute_pos = bc.abs;
    rec.alignment_score = best.alignment_score;
    rec.best_lower = best.lower; rec.best_lower_rev = best.lower_rev; rec.best_size = best.size;
    emit_bam_fields<WIDE>(ix, pools, ops_pool + best.edit_off, best.edit_len, bc.backward, bc.abs, rec.cigar_off, rec.cigar_len,
                          rec.md_off, rec.md_len, rec.nm);
    rec.lf_steps = lf_steps;
    return;
  }
  rec.lf_steps = lf_steps;
}

}  // namespace mapad

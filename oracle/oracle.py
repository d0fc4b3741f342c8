"""ctypes wrapper of the CPU oracle (oracle/libmapad_oracle.so).

TEST INFRASTRUCTURE ONLY: importable from tests/, __graft_entry__.smoke() and the cpu_baseline /
--impl reference legs of bench.py.  Nothing under mapad_b200/ may import this module.
"""
import ctypes as C
import os
import subprocess

import numpy as np

from mapad_b200 import abi

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB_PATH = os.path.join(_HERE, "libmapad_oracle.so")
_lib = None


def build(force=False):
    src = [os.path.join(_HERE, f) for f in ("oracle_capi.cpp", "oracle.hpp", "Makefile")]
    if force or not os.path.exists(_LIB_PATH) or any(
        os.path.getmtime(s) > os.path.getmtime(_LIB_PATH) for s in src if os.path.exists(s)
    ):
        subprocess.check_call(["make", "-C", _HERE, "-s"] + (["-B"] if force else []))
    return _LIB_PATH


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(_LIB_PATH):
            build()
        L = C.CDLL(_LIB_PATH)
        vp, u64, u32, f32, i32, u8 = C.c_void_p, C.c_uint64, C.c_uint32, C.c_float, C.c_int, C.c_uint8
        sig = {
            "ora_index_build": (vp, [u64, C.POINTER(C.c_char_p), C.POINTER(C.c_char_p), C.POINTER(u64), i32, u32, u64, i32, C.c_char_p, u64]),
            "ora_index_from_arrays": (vp, [vp, u64, i32, u32, vp, u64, u64, vp, u64, u64, vp, vp, C.POINTER(C.c_char_p), vp, vp, u64]),
            "ora_index_free": (None, [vp]),
            "ora_index_n": (u64, [vp]),
            "ora_index_bwt": (C.POINTER(u8), [vp]),
            "ora_index_less": (u64, [vp, C.POINTER(u64), u64]),
            "ora_index_sentinel_rows": (None, [vp, C.POINTER(u64)]),
            "ora_index_sa_samples": (u64, [vp, C.POINTER(C.POINTER(u64))]),
            "ora_index_full_sa": (u64, [vp, C.POINTER(C.POINTER(u64))]),
            "ora_index_extra_rows": (u64, [vp, C.POINTER(u64), u64]),
            "ora_index_original_symbols": (u64, [vp, C.POINTER(u64), C.POINTER(u8), u64]),
            "ora_index_occ": (u64, [vp, u64, u8]),
            "ora_index_sa_get": (i32, [vp, u64, C.POINTER(u64)]),
            "ora_index_extend": (None, [vp, u64, u64, u64, C.POINTER(u64)]),
            "ora_verify_index": (i32, [vp, u64, vp, vp, vp, u64, u64, vp, u64, i32, C.c_char_p, u64]),
            "ora_params_new": (vp, []),
            "ora_params_free": (None, [vp]),
            "ora_params_model_simple": (None, [vp, i32, f32, f32, f32, f32, f32, i32]),
            "ora_params_model_vindija": (None, [vp]),
            "ora_params_model_test": (None, [vp, f32, f32, f32]),
            "ora_params_repr_mm": (f32, [vp]),
            "ora_params_bound_discrete": (None, [vp, f32, f32, f32]),
            "ora_params_bound_continuous": (None, [vp, f32, f32, f32]),
            "ora_params_bound_test": (None, [vp, f32, f32]),
            "ora_params_gaps": (None, [vp, f32, f32, i32, i32, i32]),
            "ora_params_limits": (None, [vp, u32, u32]),
            "ora_sdm_get": (f32, [vp, u64, u64, u8, u8, u8]),
            "ora_sdm_min_penalty": (f32, [vp, u64, u64, u8, u8, i32]),
            "ora_sdm_alignment_start": (i32, [vp, u64]),
            "ora_bound_discrete_get": (f32, [vp, u64]),
            "ora_bound_reject": (i32, [vp, f32, u64]),
            "ora_bound_remaining_frac": (f32, [vp, f32, u64]),
            "ora_log2f": (f32, [f32]),
            "ora_exp2f": (f32, [f32]),
            "ora_log10f": (f32, [f32]),
            "ora_d_array": (u64, [vp, vp, vp, vp, u64, C.c_int64, vp, C.POINTER(u64)]),
            "ora_d_array_get": (f32, [vp, vp, vp, vp, u64, C.c_int64, i32, i32]),
            "ora_mmheap_new": (vp, []),
            "ora_mmheap_free": (None, [vp]),
            "ora_mmheap_push": (None, [vp, f32, u32]),
            "ora_mmheap_pop_max": (i32, [vp, C.POINTER(f32), C.POINTER(u32)]),
            "ora_mmheap_pop_min": (i32, [vp, C.POINTER(f32), C.POINTER(u32)]),
            "ora_mmheap_len": (u64, [vp]),
            "ora_mmheap_dump": (u64, [vp, vp, vp, u64]),
            "ora_binheap_new": (vp, []),
            "ora_binheap_free": (None, [vp]),
            "ora_binheap_push": (None, [vp, f32, u32]),
            "ora_binheap_pop": (i32, [vp, C.POINTER(f32), C.POINTER(u32)]),
            "ora_binheap_dump": (u64, [vp, vp, vp, u64]),
            "ora_binheap_into_sorted": (u64, [vp, vp, vp, u64]),
            "ora_prrange": (C.c_int64, [u64, u64, u64, vp, u64]),
            "ora_draw_u32": (u32, [u32, u32]),
            "ora_to_bam_fields": (i32, [vp, vp, u64, i32, u64, C.c_char_p, u64]),
            "ora_map_batch": (vp, [vp, vp, u64, vp, vp, vp, vp, i32, i32]),
            "ora_batch_free": (None, [vp]),
            "ora_batch_view": (None, [vp, C.POINTER(abi.Results)]),
            "ora_batch_xa": (u64, [vp, C.POINTER(C.c_char_p), C.POINTER(C.POINTER(u64))]),
        }
        for name, (res, args) in sig.items():
            fn = getattr(L, name)
            fn.restype = res
            fn.argtypes = args
        _lib = L
    return _lib


def _ptr(a):
    return a.ctypes.data_as(C.c_void_p) if a is not None else None


class OracleIndex:
    """In-memory index built by the oracle's own (simple) suffix sorter, or adopted from arrays."""

    def __init__(self, handle):
        self.h = handle

    @classmethod
    def build(cls, contigs, with_x=True, occ_k=128, sa_rate=32, keep_full_sa=False, draws=None):
        """contigs: list[(name:str, seq:str|bytes)].  Production settings by default
        (indexing.rs:32,163-188); tests of the reference use with_x=False, occ_k=3 and the raw SA."""
        n = len(contigs)
        names = (C.c_char_p * n)(*[c[0].encode() if isinstance(c[0], str) else c[0] for c in contigs])
        seqs_b = [c[1].encode() if isinstance(c[1], str) else bytes(c[1]) for c in contigs]
        seqs = (C.c_char_p * n)(*seqs_b)
        lens = (C.c_uint64 * n)(*[len(s) for s in seqs_b])
        d = draws.encode() if isinstance(draws, str) else draws
        h = lib().ora_index_build(n, names, seqs, lens, int(with_x), occ_k, sa_rate, int(keep_full_sa), d, len(d) if d else 0)
        return cls(h)

    @classmethod
    def test_index(cls, ref_seq):
        """utils::build_auxiliary_structures (utils.rs:12-33): alphabet $ACGT, Occ k=3, raw SA."""
        return cls.build([("ref", ref_seq)], with_x=False, occ_k=3, sa_rate=1, keep_full_sa=True)

    @classmethod
    def from_arrays(cls, bwt, sa_sample, sa_rate, extra_rows, contigs, orig_pos=None, orig_sym=None, with_x=True, occ_k=128):
        bwt = np.ascontiguousarray(bwt, dtype=np.uint8)
        sa_sample = np.ascontiguousarray(sa_sample, dtype=np.uint64)
        extra = np.ascontiguousarray(extra_rows, dtype=np.uint64).reshape(-1)
        n_c = len(contigs)
        cs = np.array([c[1] for c in contigs], dtype=np.uint64)
        ce = np.array([c[2] for c in contigs], dtype=np.uint64)
        names = (C.c_char_p * n_c)(*[c[0].encode() if isinstance(c[0], str) else c[0] for c in contigs])
        op = np.ascontiguousarray(orig_pos if orig_pos is not None else [], dtype=np.uint64)
        osym = np.ascontiguousarray(orig_sym if orig_sym is not None else [], dtype=np.uint8)
        h = lib().ora_index_from_arrays(_ptr(bwt), len(bwt), int(with_x), occ_k, _ptr(sa_sample), len(sa_sample), sa_rate,
                                        _ptr(extra), len(extra) // 2, n_c, _ptr(cs), _ptr(ce), names, _ptr(op), _ptr(osym), len(op))
        return cls(h)

    def __del__(self):
        try:
            if self.h:
                lib().ora_index_free(self.h)
                self.h = None
        except Exception:
            pass

    @property
    def n(self):
        return int(lib().ora_index_n(self.h))

    def bwt(self):
        p = lib().ora_index_bwt(self.h)
        return np.ctypeslib.as_array(p, shape=(self.n,)).copy()

    def less(self):
        buf = (C.c_uint64 * 8)()
        k = lib().ora_index_less(self.h, buf, 8)
        return [int(buf[i]) for i in range(k)]

    def sentinel_rows(self):
        buf = (C.c_uint64 * 2)()
        lib().ora_index_sentinel_rows(self.h, buf)
        return [int(buf[0]), int(buf[1])]

    def sa_samples(self):
        p = C.POINTER(C.c_uint64)()
        k = lib().ora_index_sa_samples(self.h, C.byref(p))
        return np.ctypeslib.as_array(p, shape=(k,)).copy() if k else np.zeros(0, np.uint64)

    def full_sa(self):
        p = C.POINTER(C.c_uint64)()
        k = lib().ora_index_full_sa(self.h, C.byref(p))
        return np.ctypeslib.as_array(p, shape=(k,)).copy() if k else np.zeros(0, np.uint64)

    def extra_rows(self):
        k = lib().ora_index_extra_rows(self.h, None, 0)
        buf = (C.c_uint64 * (2 * max(k, 1)))()
        lib().ora_index_extra_rows(self.h, buf, k)
        return [(int(buf[2 * i]), int(buf[2 * i + 1])) for i in range(k)]

    def original_symbols(self):
        k = lib().ora_index_original_symbols(self.h, None, None, 0)
        pb = (C.c_uint64 * max(k, 1))()
        sb = (C.c_uint8 * max(k, 1))()
        lib().ora_index_original_symbols(self.h, pb, sb, k)
        return {int(pb[i]): int(sb[i]) for i in range(k)}

    def occ(self, r, a):
        return int(lib().ora_index_occ(self.h, r, a))

    def sa_get(self, row):
        out = C.c_uint64()
        ok = lib().ora_index_sa_get(self.h, row, C.byref(out))
        return int(out.value) if ok else None

    def extend(self, lower, lower_rev, size):
        buf = (C.c_uint64 * 12)()
        lib().ora_index_extend(self.h, lower, lower_rev, size, buf)
        return [(int(buf[3 * k]), int(buf[3 * k + 1]), int(buf[3 * k + 2])) for k in range(4)]

    def positions(self, lower, size):
        """Interval::occ(&suffix_array): text positions of SA rows [lower, lower+size)."""
        return [self.sa_get(r) for r in range(lower, lower + size)]

    def arrays(self):
        """The index in the layout of mapad_b200.api.Index.arrays() (`less` padded to 8 entries)."""
        n = self.n
        less = self.less()
        orig = self.original_symbols()
        return dict(n=n, bwt=self.bwt(), less=less + [n] * (8 - len(less)), sentinel_rows=self.sentinel_rows(),
                    sa_sample=self.sa_samples(), sa_rate=32,
                    extra_rows=np.array(self.extra_rows(), dtype=np.uint64).reshape(-1, 2),
                    orig_pos=np.array(sorted(orig), dtype=np.uint64), orig_sym=np.array([orig[k] for k in sorted(orig)], dtype=np.uint8))


class IndexMismatch(AssertionError):
    """verify_index found that the arrays are not the index of the text."""


_RANK = np.zeros(256, dtype=np.uint8)  # 0: not a base
for _c, _r in zip(b"ACGTacgt", (1, 2, 3, 4, 1, 2, 3, 4)):
    _RANK[_c] = _r
_COMP_RANK = np.array([0, 4, 3, 2, 1, 5], dtype=np.uint8)


def text_ranks(seqs):
    """The rank text `fwd $ revcomp $` ($ = 0, A C G T = 1..4, X = 5) of the contig sequences `seqs` (str, bytes or uint8
    arrays, concatenated in order), as `mapad index` builds it: a run of >= 20 equal non-ACGT symbols becomes X.  Shorter
    runs are replaced by seeded draws that cannot be reproduced independently, so they are refused (ValueError)."""
    parts = [np.frombuffer(s.encode() if isinstance(s, str) else s, dtype=np.uint8) if not isinstance(s, np.ndarray) else s
             for s in seqs]
    g = parts[0] if len(parts) == 1 else np.concatenate(parts)
    G = len(g)
    out = np.empty(2 * G + 2, dtype=np.uint8)
    fwd = out[:G]
    np.take(_RANK, g, out=fwd)
    other = np.flatnonzero(fwd == 0)
    if len(other):
        sym = np.char.upper(g[other].view("S1")).view(np.uint8)
        # runs of one symbol over consecutive positions (runs cross contig boundaries, as in the indexer)
        new_run = np.ones(len(other), dtype=bool)
        new_run[1:] = (np.diff(other) != 1) | (sym[1:] != sym[:-1])
        run_id = np.cumsum(new_run) - 1
        run_len = np.bincount(run_id)
        short = run_len[run_id] < 20
        if short.any():
            raise ValueError("a run of %d non-ACGT symbols at %d is replaced by seeded draws" % (run_len[run_id[short][0]], other[short][0]))
        fwd[other] = 5
    out[G] = 0
    np.take(_COMP_RANK, fwd[::-1], out=out[G + 1:2 * G + 1])
    out[-1] = 0
    return out


def verify_index(text, arrays, n_threads=None):
    """Checks index arrays (the layout of mapad_b200.api.Index.arrays()) against the rank text from text_ranks() with the
    oracle's independent LF-walk verifier.  Raises IndexMismatch naming a wrong row."""
    a = arrays
    text = np.ascontiguousarray(text, dtype=np.uint8)
    bwt = np.ascontiguousarray(a["bwt"], dtype=np.uint8)
    if len(text) != a["n"] or len(bwt) != a["n"]:
        raise IndexMismatch("text of %d symbols, index of n = %d with %d BWT rows" % (len(text), a["n"], len(bwt)))
    less = np.ascontiguousarray(a["less"], dtype=np.uint64)
    if len(less) != 8:
        raise IndexMismatch("less has %d entries, expected 8" % len(less))
    ss = np.ascontiguousarray(a["sa_sample"], dtype=np.uint64)
    if len(ss) == 0:
        raise IndexMismatch("no SA samples")
    extra = np.ascontiguousarray(a["extra_rows"], dtype=np.uint64).reshape(-1)
    msg = C.create_string_buffer(512)
    rc = lib().ora_verify_index(_ptr(text), len(text), _ptr(bwt), _ptr(less), _ptr(ss), len(ss), a["sa_rate"], _ptr(extra), len(extra) // 2,
                                n_threads or os.cpu_count() or 1, msg, len(msg))
    if rc:
        raise IndexMismatch(msg.value.decode())


class OracleParams:
    def __init__(self):
        self.h = lib().ora_params_new()
        self.repr_mm = None

    def __del__(self):
        try:
            if self.h:
                lib().ora_params_free(self.h)
                self.h = None
        except Exception:
            pass

    # models
    def model_simple(self, library, f, t, d, s, divergence, ignore_q=False):
        lib().ora_params_model_simple(self.h, {"single_stranded": 0, "double_stranded": 1}.get(library, library), f, t, d, s, divergence, int(ignore_q))
        return self

    def model_vindija(self):
        lib().ora_params_model_vindija(self.h)
        return self

    def model_test(self, deam, mm, match):
        lib().ora_params_model_test(self.h, deam, mm, match)
        return self

    def representative_mismatch_penalty(self):
        return float(lib().ora_params_repr_mm(self.h))

    # bounds
    def bound_discrete(self, poisson_threshold, base_error_rate, repr_mm=None):
        lib().ora_params_bound_discrete(self.h, poisson_threshold, base_error_rate, self.representative_mismatch_penalty() if repr_mm is None else repr_mm)
        return self

    def bound_continuous(self, cutoff, exponent, repr_mm=None):
        lib().ora_params_bound_continuous(self.h, cutoff, exponent, self.representative_mismatch_penalty() if repr_mm is None else repr_mm)
        return self

    def bound_test(self, threshold, representative_mm_bound):
        lib().ora_params_bound_test(self.h, threshold, representative_mm_bound)
        return self

    def gaps(self, open_, extend, dist_ends, max_open, abort_on_limit=False):
        lib().ora_params_gaps(self.h, open_, extend, dist_ends, max_open, int(abort_on_limit))
        return self

    def limits(self, stack_limit, tree_limit):
        lib().ora_params_limits(self.h, stack_limit, tree_limit)
        return self

    def sdm_get(self, i, L, frm, to, q):
        return float(lib().ora_sdm_get(self.h, i, L, ord(frm) if isinstance(frm, str) else frm, ord(to) if isinstance(to, str) else to, q))

    def discrete_get(self, L):
        return float(lib().ora_bound_discrete_get(self.h, L))


def d_array(index, params, seq, qual, split=-1):
    seq = np.frombuffer(bytes(seq), dtype=np.uint8)
    qual = np.frombuffer(bytes(bytearray(qual)), dtype=np.uint8)
    out = np.zeros(len(seq), dtype=np.float32)
    steps = C.c_uint64()
    sp = lib().ora_d_array(index.h, params.h, _ptr(seq), _ptr(qual), len(seq), split, _ptr(out), C.byref(steps))
    return out, int(sp), int(steps.value)


def d_array_get(index, params, seq, qual, split, k, l):
    seq = np.frombuffer(bytes(seq), dtype=np.uint8)
    qual = np.frombuffer(bytes(bytearray(qual)), dtype=np.uint8)
    return float(lib().ora_d_array_get(index.h, params.h, _ptr(seq), _ptr(qual), len(seq), split, k, l))


def map_batch(index, params, seqs, quals, seeds=None, n_threads=1, want_hits=True, packed=None):
    """Runs k_mismatch_search + intervals_to_bam for every read.  Returns abi.BatchResult (+ .xa list)."""
    if packed is None:
        seq, qual, offsets = abi.pack_reads(seqs, quals)
    else:
        seq, qual, offsets = packed
    n = len(offsets) - 1
    sd = np.ascontiguousarray(seeds, dtype=np.uint32) if seeds is not None else None
    b = lib().ora_map_batch(index.h, params.h, n, _ptr(seq), _ptr(qual), _ptr(offsets), _ptr(sd), n_threads, int(want_hits))
    try:
        view = abi.Results()
        lib().ora_batch_view(b, C.byref(view))
        res = abi.BatchResult(view)
        flat = C.c_char_p()
        offs = C.POINTER(C.c_uint64)()
        k = lib().ora_batch_xa(b, C.byref(flat), C.byref(offs))
        raw = C.string_at(flat, int(offs[k - 1])) if k and offs[k - 1] else b""
        res.xa = [raw[int(offs[i]) : int(offs[i + 1])].decode() for i in range(k - 1)]
    finally:
        lib().ora_batch_free(b)
    return res


def prrange(start, end, seed):
    cap = max(end - start, 1) + 4
    out = np.zeros(cap, dtype=np.uint64)
    k = lib().ora_prrange(start, end, seed, _ptr(out), cap)
    if k < 0:
        return None
    return [int(v) for v in out[:k]]


def to_bam_fields(ops, backward=False, absolute_pos=0, index=None):
    arr = np.zeros(len(ops), dtype=abi.EDIT_OP_DTYPE)
    for i, (p, k, b) in enumerate(ops):
        arr[i] = (p, k, b)
    buf = C.create_string_buffer(65536)
    lib().ora_to_bam_fields(index.h if index else None, _ptr(arr), len(ops), int(backward), absolute_pos, buf, 65536)
    cigar, md, nm = buf.value.decode().split("\t")
    return cigar, md, int(nm)

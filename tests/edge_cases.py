"""A deterministic adversarial workload for the parity tests (plain module, no fixtures).

The other parity tests map simulated reads against i.i.d. random genomes, where almost every read is unique.  This workload
aims at the code those inputs never reach: multi-mappers (segmental duplications on both strands, tandem repeats and
homopolymers), N runs on both sides of the 20 bp 'X' threshold, short IUPAC runs (replacement draws and the original-symbol
MD path), contigs of 1 - 33 bp, reads across contig and N boundaries, read lengths 0 - 250, extreme base qualities and
ambiguous read bases.  `coverage()` measures on a mapping result that the workload reaches those paths, so that an edit to
the generator cannot silently turn it into another random-genome workload.
"""
import numpy as np

from helpers import ora, product_params, simulate_reads
from ref_cases import cli_params

ACGT = np.frombuffer(b"ACGT", dtype=np.uint8)
_COMP = np.arange(256, dtype=np.uint8)
for _a, _b in zip(b"ACGTRYKMSWBDHVN", b"TGCAYRMKSWVHDBN"):
    _COMP[_a] = _b

LENGTH_LADDER = (1, 2, 3, 8, 15, 16, 17, 31, 32, 33, 63, 64, 65, 150, 250)
IUPAC_RUNS = ("R", "YY", "KKK", "M", "S", "W", "B", "D", "H", "V", "RYKMSWBDHV")
N_RUNS = (19, 20, 21, 347)


def _rand(rng, n):
    return ACGT[rng.integers(0, 4, size=n)].copy()


def revcomp(a):
    return _COMP[np.asarray(a, dtype=np.uint8)[::-1]]


def _substitute(rng, a, k):
    a = a.copy()
    for p in rng.choice(len(a), size=k, replace=False):
        a[p] = ACGT[(int(np.nonzero(ACGT == a[p])[0][0]) + 1 + int(rng.integers(0, 3))) % 4]
    return a


class EdgeGenome:
    """contigs: list[(name, str)]; features: list[(kind, contig index, start, end)] in contig coordinates;
    text: the contigs concatenated (the forward strand of the index text); starts: contig offsets in `text`."""

    def __init__(self, contigs, features):
        self.contigs = contigs
        self.features = features
        self.starts = np.cumsum([0] + [len(s) for _, s in contigs])
        self.text = np.frombuffer("".join(s for _, s in contigs).encode(), dtype=np.uint8)

    def where(self, kind):
        return [(int(self.starts[c]) + a, int(self.starts[c]) + b) for k, c, a, b in self.features if k == kind]


def edge_genome(seed=0, scale=1.0):
    """A few contigs, about 1.1 Mbp at scale 1 (the repeat features are ~110 kbp at every scale; the random background
    between them shrinks with `scale`)."""
    rng = np.random.default_rng(seed)
    contigs, features = [], []
    cur, name = [], None

    def bg(n):
        put(_rand(rng, max(200, int(n * scale))))

    def put(a, kind=None):
        a = np.frombuffer(a.encode(), np.uint8) if isinstance(a, str) else np.asarray(a, np.uint8)
        off = sum(len(x) for x in cur)
        cur.append(a)
        if kind:
            features.append((kind, len(contigs), off, off + len(a)))

    def close():
        contigs.append((name, b"".join(x.tobytes() for x in cur).decode()))
        cur.clear()

    # segmental duplications: block A (1.5 kbp) x 40 and block B (2.5 kbp) x 3, some copies with 1 - 3 substitutions, about half
    # of them reverse-complemented; block C (1 kbp) x 6, one copy split across the chr1 | t1 | chr2 junction
    block_a, block_b, block_c = _rand(rng, 1500), _rand(rng, 2500), _rand(rng, 1000)
    copies_a = []
    for k in range(40):
        c = block_a if k % 4 else _substitute(rng, block_a, 1 + k % 3)
        copies_a.append(revcomp(c) if k % 2 else c)

    name = "chr1"
    bg(150_000)
    for k in range(20):
        put(copies_a[k], "segdup_a")
        bg(3_000)
    for run in N_RUNS:
        put("N" * run, "n_run_%d" % run)
        bg(20_000)
    put(block_b, "segdup_b")
    bg(40_000)
    put(block_c, "segdup_c")
    bg(20_000)
    for u in IUPAC_RUNS:
        put(u, "iupac")
        bg(4_000)
    for unit, reps in (("A", 500), ("AC", 150), ("AGT", 100), ("ACCTGAT", 60), ("C", 200), ("A", 60)):
        put(unit * reps, "tandem_%d" % len(unit))
        bg(10_000)
    put(block_c[:400], "segdup_c_split")
    close()
    name = "t1"
    put(block_c[400:401])
    close()
    name = "chr2"
    put(block_c[401:], "segdup_c_split")
    bg(100_000)
    for k in range(20, 40):
        put(copies_a[k], "segdup_a")
        bg(2_000)
    put(revcomp(block_b), "segdup_b")
    bg(30_000)
    for _ in range(3):
        put(block_c, "segdup_c")
        bg(7_000)
    put(_substitute(rng, block_b, 2), "segdup_b")
    bg(60_000)
    put("T" * 300, "tandem_1")
    bg(5_000)
    put("A" * 120, "homopolymer_end")  # the A run continues into the next contigs: alignments straddling them are skipped
    close()
    name = "t2"
    put("AA")
    close()
    name = "t31"
    put(_rand(rng, 31))
    close()
    name = "chr3"
    put("A" * 40)
    bg(150_000)
    put(block_c, "segdup_c")
    bg(50_000)
    close()
    for n_ in (32, 33):
        name = "t%d" % n_
        put(_rand(rng, n_))
        close()
    name = "chr4"
    bg(60_000)
    put(revcomp(block_c), "segdup_c")
    bg(20_000)
    put("N" * 150, "n_run_end")
    close()
    return EdgeGenome(contigs, features)


def _damage(rng, r, rate=0.02, deam=True):
    r = r.copy()
    L = len(r)
    mut = rng.random(L) < rate
    r[mut] = _rand(rng, int(mut.sum()))
    if deam and L:
        ends = np.zeros(L, bool)
        ends[:2] = True
        ends[-2:] = True
        r[(r == ord("C")) & ends & (rng.random(L) < 0.5)] = ord("T")
    return r


def edge_reads(genome, seed=0, n_sim=600, qual_lengths=(20, 45)):
    """(seq, qual, offsets, seeds) of a packed batch: the classes of the module docstring, shuffled into one batch (so that
    the length-sorted work list of the search mixes them) with empty reads interleaved.  Reads with qualities 0 / 1 cost
    nothing to mismatch, so their searches grow steeply with `qual_lengths` (45 bp: ~8e5 frames)."""
    rng = np.random.default_rng(seed)
    text = genome.text
    G = len(text)
    reads = []  # (bytes seq, bytes qual)

    def window(a, L):
        a = max(0, min(int(a), G - L))
        return text[a:a + L].copy()

    def qual(L, hi=40):
        return np.array([40, 30, 20, 2], np.uint8)[rng.choice(4, size=L, p=[0.7, 0.2, 0.08, 0.02])] if hi else np.full(L, 40, np.uint8)

    def add(r, q=None, strand=None):
        r = np.asarray(r, np.uint8)
        q = qual(len(r)) if q is None else np.asarray(q, np.uint8)
        if strand if strand is not None else rng.random() < 0.5:
            r, q = revcomp(r), q[::-1].copy()
        reads.append((r.tobytes(), q.tobytes()))

    # 1. repeats: exact and damaged copies of every segmental duplication and tandem repeat
    for kind, n_per in (("segdup_a", 4), ("segdup_b", 12), ("segdup_c", 8), ("segdup_c_split", 10), ("tandem_1", 6), ("tandem_2", 6),
                        ("tandem_3", 6), ("tandem_7", 6), ("homopolymer_end", 6)):
        for a, b in genome.where(kind):
            for k in range(n_per):
                L = int(rng.integers(20, 80))
                st = int(rng.integers(a - L // 2, b - L // 2)) if kind in ("segdup_c_split", "homopolymer_end") else int(rng.integers(a, max(a + 1, b - L)))
                w = window(st, L)
                add(w if k % 2 == 0 else _damage(rng, w), np.full(L, 40, np.uint8) if k % 2 == 0 else None)
    # 2. across N / X boundaries (N kept as N, or replaced as a sequencer would call it) and across contig boundaries
    for kind in ["n_run_%d" % r for r in N_RUNS] + ["n_run_end"]:
        for a, b in genome.where(kind):
            for edge in (a, b):
                for d in (-30, -12, -3, 3, 12):
                    L = int(rng.integers(30, 70))
                    w = window(edge + d - L // 2, L)
                    if d % 2:
                        n = w == ord("N")
                        w[n] = _rand(rng, int(n.sum()))
                    add(w)
    for s in genome.starts[1:-1]:
        for d in (-20, -5, 0, 5, 20):
            L = int(rng.integers(25, 60))
            add(window(s + d - L // 2, L), np.full(L, 40, np.uint8))
    # 3. over the short IUPAC runs (the index replaced them by drawn bases; MD reports the original symbol)
    for a, b in genome.where("iupac"):
        for k in range(4):
            L = int(rng.integers(30, 60))
            w = window(a - int(rng.integers(3, L - 12)), L)
            n = ~np.isin(w, ACGT)
            w[n] = _rand(rng, int(n.sum()))
            add(w, np.full(L, 40, np.uint8))
    # 4. the usual simulated mix, drawn from the whole text (IUPAC symbols read as N)
    sim_text = text.copy()
    sim_text[~np.isin(sim_text, ACGT) & (sim_text != ord("N"))] = ord("N")
    seqs, quals = simulate_reads(sim_text.tobytes().decode(), n_sim, (25, 100), seed=seed + 1)
    for k, (s_, q_) in enumerate(zip(seqs, quals)):
        if k % 50 == 5 and len(s_) > 20:
            s_ = s_[:10] + b"N" + s_[11:]
        reads.append((s_, q_))
    # 5. the length ladder, drawn from the genome with light damage
    for L in LENGTH_LADDER:
        for k in range(3):
            st = int(rng.integers(0, G - L))
            w = window(st, L)
            w[~np.isin(w, ACGT)] = ord("A")
            add(_damage(rng, w, rate=0.01 if L > 30 else 0.0), np.full(L, 40 if k else 30, np.uint8))
    # 6. extreme base qualities
    for qv in (0, 1, 93, 255, "alt"):
        for L in qual_lengths:
            st = int(rng.integers(0, G - L))
            w = window(st, L)
            w[~np.isin(w, ACGT)] = ord("C")
            q = np.tile(np.array([0, 255], np.uint8), L)[:L] if qv == "alt" else np.full(L, qv, np.uint8)
            add(_damage(rng, w, rate=0.03), q)
    # 7. ambiguous read bases: R / Y / N inside genomic reads, one all-N read
    for k in range(12):
        L = int(rng.integers(30, 60))
        w = window(int(rng.integers(0, G - L)), L)
        w[~np.isin(w, ACGT)] = ord("G")
        for p in rng.choice(L, size=1 + k % 3, replace=False):
            w[p] = b"RYN"[k % 3]
        add(w)
    add(np.full(36, ord("N"), np.uint8), np.full(36, 30, np.uint8), strand=False)

    order = rng.permutation(len(reads))
    out = []
    for k, i in enumerate(order):
        if k % 97 == 0:
            out.append((b"", b""))
        out.append(reads[i])
    seq = np.frombuffer(b"".join(s for s, _ in out), np.uint8).copy()
    qual_ = np.frombuffer(b"".join(q for _, q in out), np.uint8).copy()
    off = np.zeros(len(out) + 1, np.uint64)
    off[1:] = np.cumsum([len(s) for s, _ in out])
    seeds = (np.arange(len(out), dtype=np.uint64) * 2654435761 % (1 << 32)).astype(np.uint32)
    return seq, qual_, off, seeds


def index_arrays_have_x(arrays):
    """Number of 'X' rows of the index (N runs >= 20 bp)."""
    return int(np.count_nonzero(arrays["bwt"] == 5))


def coverage(res, arrays=None):
    """Counts on a mapping result (oracle or product) of the paths this workload exists for."""
    rec = res.records
    m = rec["mapped"] != 0
    c = dict(
        reads=len(rec),
        mapped=int(m.sum()),
        x0_gt1=int(np.count_nonzero(m & (rec["x0"] > 1))),
        n_alts_2=int(np.count_nonzero(m & (rec["n_alts"] == 2))),
        xt_r=int(np.count_nonzero(m & (rec["xt"] == ord("R")))),
        max_hits=int(rec["n_hits"].max()) if len(rec) else 0,
        hits_ge10=int(np.count_nonzero(rec["n_hits"] >= 10)),
        max_best_size=int(rec["best_size"][m].max()) if m.any() else 0,
        skipped=int(np.count_nonzero(m & (rec["x0"].astype(np.int64) < rec["best_size"].astype(np.int64)))),
        reverse=int(np.count_nonzero(m & (rec["strand"] == 1))),
        md_iupac=0,
    )
    for i in np.nonzero(m)[0]:
        md = res.md_str(int(rec["md_off"][i]), int(rec["md_len"][i]))
        if any(ch in md for ch in "RYKMSWBDHVN"):
            c["md_iupac"] += 1
    if arrays is not None:
        c["x_rows"] = index_arrays_have_x(arrays)
    return c


def assert_coverage(c, scale=1.0):
    """The workload reaches multi-mappers, alts, full hit heaps, huge intervals, skipped positions, IUPAC MD and X rows."""
    assert c["x0_gt1"] >= 30, c
    assert c["n_alts_2"] >= 5 and c["xt_r"] >= 5, c
    assert c["max_hits"] >= 10, c
    assert c["max_best_size"] > 1000, c
    assert c["skipped"] >= 1, c
    assert c["md_iupac"] >= 1, c
    assert c.get("x_rows", 1) > 0, c
    assert c["reverse"] > 0, c


# ---- scoring models the edge workload is mapped under ---------------------------------------------------------------------
# TestDifferenceModel (search starts at L / 2, forward and backward steps); MAPAD_MODEL_CUSTOM runs use the same semantics
TEST_SPEC = dict(model=("test", -1.0, -2.0, 0.0), bound=("test", -5.0, None), gaps=(-4.0, -1.0, 3, 2))


def model_specs():
    """name -> case spec (tests/ref_cases.py format) of every model / bound the device offers besides the two CLI libraries."""
    ss = cli_params("single_stranded")
    cont = dict(ss, bound=("continuous", -0.25, 1.0))
    ign = dict(ss, model=ss["model"][:7] + (True,))
    return dict(test=TEST_SPEC, vindija=dict(ss, model=("vindija",)), continuous=cont, ignore_quality=ign)


def _test_get(frm, to):
    if frm == ord("C") and to == ord("T"):
        return -1.0
    return 0.0 if frm == to else -2.0


def custom_params():
    """MAPAD_MODEL_CUSTOM with TEST_SPEC's semantics through the host callback (keep the returned object alive)."""
    from mapad_b200 import abi
    P = product_params(TEST_SPEC)
    P.model_kind = abi.MODEL_CUSTOM

    @abi.SDM_GET_FN
    def get(user, i, L, frm, to, q):
        return _test_get(frm, to)

    P.custom_get = get
    P._keep = get
    return P


def custom_penalty_table(seq):
    """MAPAD_MODEL_CUSTOM's precomputed penalties: get(i, L, b, read[i], q[i]) for b = A, C, G, T, 4 floats per base."""
    seq = np.asarray(seq, np.uint8)
    out = np.full((len(seq), 4), -2.0, np.float32)
    for k, b in enumerate(b"ACGT"):
        out[seq == b, k] = 0.0
    out[seq == ord("T"), 1] = -1.0
    return out.reshape(-1)


def oracle_index(index):
    a = index.arrays()
    return ora.OracleIndex.from_arrays(a["bwt"], a["sa_sample"], a["sa_rate"], a["extra_rows"], a["contigs"], a["orig_pos"], a["orig_sym"])


def sub_batch(packed, seeds, idx):
    """The reads `idx` of a packed batch, as a new packed batch (and their seeds)."""
    seq, qual, off = packed
    parts = [(seq[int(off[i]):int(off[i + 1])], qual[int(off[i]):int(off[i + 1])]) for i in idx]
    o = np.zeros(len(parts) + 1, np.uint64)
    o[1:] = np.cumsum([len(p[0]) for p in parts])
    cat = lambda xs: np.concatenate(xs).astype(np.uint8) if xs else np.zeros(0, np.uint8)
    return (cat([p[0] for p in parts]), cat([p[1] for p in parts]), o), np.asarray(seeds)[list(idx)].astype(np.uint32)

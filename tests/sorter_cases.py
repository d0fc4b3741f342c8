"""Deterministic texts at the corners of the device suffix sorter (mapad_b200/csrc/gpu_index_build.cu).

That sorter buckets suffixes by their first symbol and orders each bucket by the next 42 symbols, packed 21 to a 63-bit key
(offsets 1..21 and 22..42).  Two suffixes sharing 43 symbols, the bucket symbol included, tie: the sorter reports it and
the index is built by the host SA-IS instead.  i.i.d. random texts share about log4(n) symbols, so they never reach the key
boundaries.  Each text here is built to reach one: shared prefixes that end on either side of the boundary between the two
keys and at the last key symbol, the two sentinels (last '$' = code 0, first '$' = 1) as the first differing symbol, 'X'
runs, empty symbol buckets, texts shorter than one key or around one compaction tile (8 192 symbols), many and 1 bp
contigs, and the '$'-preceded suffixes on and off sampled rows.  `Case.check_reach` measures on the suffix array of the
oracle's own sorter that the text reaches what it was built for.

No text has a short IUPAC run: those are replaced by seeded draws that an independent text builder cannot reproduce.
"""
import numpy as np

TIE = 43  # shared symbols (bucket symbol included) at which the device sorter gives up
FALLBACK_MESSAGE = "falling back to the host SA-IS"

_COMP = {"A": "T", "C": "G", "G": "C", "T": "A"}


def revcomp(s):
    return "".join(_COMP[c] for c in reversed(s))


def lcp_codes(text):
    """Sort codes of a rank text (last '$' = 0, first '$' = 1, A..X = 2..6), padded past the end."""
    codes = text.astype(np.int16) + 1
    codes[-1] = 0
    return np.concatenate([codes, np.full(TIE + 1, -1, np.int16)])


def lcp(codes, a, b, cap=TIE + 1):
    """Shared prefix of the suffixes at a and b (arrays of positions), up to `cap` symbols."""
    eq = np.ones(len(a), dtype=bool)
    out = np.zeros(len(a), dtype=np.int64)
    for k in range(cap):
        eq &= codes[a + k] == codes[b + k]
        out += eq
    return out


class Case:
    """contigs: list[(name, str)].  pairs: (i, j, k) = the suffixes at text positions i and j share exactly k symbols.
    lcp_max: the exact maximum shared prefix of adjacent suffixes when the text is built to reach it (else only < TIE or
    >= TIE is checked).  n_extra: number of unsampled '$' rows, where the text was chosen for it."""

    def __init__(self, name, contigs, pairs=(), lcp_max=None, n_extra=None):
        self.name, self.contigs, self.pairs, self.lcp_max, self.n_extra = name, contigs, list(pairs), lcp_max, n_extra
        self.device_sorts = lcp_max is None or lcp_max < TIE

    def __repr__(self):
        return self.name

    @property
    def seqs(self):
        return [s for _, s in self.contigs]

    def check_reach(self, text, sa):
        codes = lcp_codes(text)
        for i, j, k in self.pairs:
            got = int(lcp(codes, np.array([i]), np.array([j]))[0])
            assert got == k, "%s: suffixes %d and %d share %d symbols, built for %d" % (self.name, i, j, got, k)
        sa = np.asarray(sa, dtype=np.int64)
        m = int(lcp(codes, sa[:-1], sa[1:]).max())
        if self.lcp_max is not None:
            assert m == self.lcp_max, "%s: longest shared prefix %d, built for %d" % (self.name, m, self.lcp_max)
        else:
            assert m < TIE, "%s: longest shared prefix %d" % (self.name, m)


class _Text:
    """A random forward strand to plant features in; positions are text (= forward strand) coordinates."""

    def __init__(self, G, seed, alphabet="ACGT"):
        self.rng = np.random.default_rng(seed)
        self.g = list(self.rand(G, alphabet))
        self.pairs = []

    def rand(self, n, alphabet="ACGT"):
        return "".join(alphabet[i] for i in self.rng.integers(0, len(alphabet), size=n))

    def other(self, *avoid):
        return self.rng.choice([c for c in "ACGT" if c not in avoid])

    def put(self, at, s):
        self.g[at:at + len(s)] = list(s)

    @property
    def G(self):
        return len(self.g)

    def mirror(self, at, length):
        """Text position of the reverse complement of forward interval [at, at + length)."""
        return self.G + 1 + self.G - at - length

    def pair(self, k, at1, at2):
        """Two copies of k symbols whose neighbours differ on both sides."""
        s = self.rand(k)
        x1, y1 = self.rand(1), self.rand(1)
        self.put(at1 - 1, x1 + s + y1)
        self.put(at2 - 1, self.other(x1) + s + self.other(y1))
        self.pairs.append((at1, at2, k))

    def palindrome(self, k, at):
        """k symbols equal to their reverse complement: the copy on the reverse strand shares exactly k."""
        h = self.rand(k // 2)
        x = self.rand(1)
        self.put(at - 1, x + h + revcomp(h) + self.other(_COMP[x]))
        self.pairs.append((at, self.mirror(at, k), k))

    def x_run(self, k, at):
        """k N (-> X) whose flanks make the forward and reverse-strand runs differ right after the run."""
        x = self.rand(1)
        self.put(at - 1, x + "N" * k + self.other(_COMP[x]))
        self.pairs.append((at, self.mirror(at, k), k))

    def sentinel(self, k):
        """The forward strand ends with the reverse complement of its first k symbols, so the reverse strand ends with them
        too: the suffixes before the two '$' share k symbols and then differ only in the sentinel."""
        self.put(self.G - k, revcomp("".join(self.g[:k])))
        self.g[self.G - 1 - k] = self.other(_COMP[self.g[k]])
        self.pairs.append((self.G - k, 2 * self.G + 1 - k, k))

    def contigs(self, n=1):
        s = "".join(self.g)
        cuts = [len(s) * i // n for i in range(n + 1)]
        return [("c%d" % i, s[cuts[i]:cuts[i + 1]]) for i in range(n)]


def assert_same_index(want, got, label):
    """Index arrays (api.Index.arrays() layout) equal field by field; orig_pos / orig_sym only where both have them."""
    assert want["n"] == got["n"], label
    assert list(want["less"]) == list(got["less"]), (label, want["less"], got["less"])
    assert list(want["sentinel_rows"]) == list(got["sentinel_rows"]), label
    assert want["sa_rate"] == got["sa_rate"], label
    assert np.array_equal(want["bwt"], got["bwt"]), (label, "bwt", int(np.argmax(want["bwt"] != got["bwt"])))
    assert np.array_equal(want["sa_sample"], got["sa_sample"]), (label, "sa_sample", int(np.argmax(want["sa_sample"] != got["sa_sample"])))
    assert np.array_equal(np.asarray(want["extra_rows"]).reshape(-1, 2), np.asarray(got["extra_rows"]).reshape(-1, 2)), (label, "extra_rows")
    for k in ("contigs", "orig_pos", "orig_sym"):
        if k in want and k in got:
            assert np.array_equal(np.asarray(want[k], dtype=object), np.asarray(got[k], dtype=object)), (label, k)


def contig_table(contigs):
    """(name, first, last) text positions of each contig, as the indexer records them."""
    out, start = [], 0
    for name, s in contigs:
        out.append((name, start, start + len(s) - 1))
        start += len(s)
    return out


def _one(name, G, seed, build, lcp_max=None, n_contigs=1):
    t = _Text(G, seed)
    build(t)
    return Case(name, t.contigs(n_contigs), t.pairs, lcp_max)


def cases():
    """The texts the device sorter must finish (lcp_max < TIE) and the ones it must hand to the host SA-IS."""
    out = []
    for k in (21, 22, 23, 42, 43):
        out.append(_one("pair%d" % k, 20_000, 100 + k, lambda t, k=k: t.pair(k, 5_000, 12_000), lcp_max=k))
    for k in (22, 42, 44):
        out.append(_one("palindrome%d" % k, 20_000, 200 + k, lambda t, k=k: t.palindrome(k, 7_000), lcp_max=k))
    for k in (1, 10, 21, 22, 41, 42, 43):
        out.append(_one("sentinel%d" % k, 20_000, 300 + k, lambda t, k=k: t.sentinel(k), lcp_max=k if k > 20 else None))
    for k in (20, 21, 42, 43, 44):
        out.append(_one("xrun%d" % k, 20_000, 400 + k, lambda t, k=k: t.x_run(k, 9_000), lcp_max=k))
    t = _Text(3_000, 500, alphabet="AT")  # C and G buckets empty
    out.append(Case("at_only", t.contigs()))
    for G in (1, 2, 20, 21, 42, 43, 4_095, 4_096, 4_097):  # n = 2G + 2: shorter than one key; one tile of 8 192 and just over
        out.append(Case("G%d" % G, _Text(G, 600 + G).contigs()))
    t = _Text(20_000, 700)
    lens = [1, 1, 2, 1, 3, 5, 1, 8, 13, 1, 21, 34, 1, 55]
    lens += [int(x) for x in t.rng.integers(1, 400, size=100)]
    lens.append(t.G - sum(lens))
    cuts = np.cumsum([0] + lens)
    s = "".join(t.g)
    out.append(Case("contigs%d" % len(lens), [("k%d" % i, s[cuts[i]:cuts[i + 1]]) for i in range(len(lens))]))
    # rows of the '$'-preceded suffixes (text positions 0 and G + 1): one of them sampled (row % 32 == 0), or neither
    for seed, n_extra in ((SEED_ONE_DOLLAR_ROW_SAMPLED, 1), (SEED_NO_DOLLAR_ROW_SAMPLED, 2)):
        out.append(Case("dollar_rows_extra%d" % n_extra, _Text(3_000, seed).contigs(), n_extra=n_extra))
    out.append(large())
    return out


# found with the host builder: G = 3 000 random texts whose '$'-preceded suffixes fall on 1 or 0 sampled rows
SEED_ONE_DOLLAR_ROW_SAMPLED = 1040
SEED_NO_DOLLAR_ROW_SAMPLED = 1000


def large(G=1_000_000, seed=800):
    """About 1 Mbp with every resolvable corner at once (three contigs): pairs sharing 21, 22, 23 and 42 symbols,
    palindromes of 22 and 42, X runs of 20, 21 and 42 and the sentinel order at 42.  Longest shared prefix: 42."""
    t = _Text(G, seed)
    for i, k in enumerate((21, 22, 23, 42)):
        t.pair(k, 10_000 + 50_000 * i, 500_000 + 50_000 * i)
    for i, k in enumerate((22, 42)):
        t.palindrome(k, 250_000 + 50_000 * i)
    for i, k in enumerate((20, 21, 42)):
        t.x_run(k, 750_000 + 50_000 * i)
    t.sentinel(42)
    return Case("large", t.contigs(3), t.pairs, lcp_max=42)

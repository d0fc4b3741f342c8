"""The oracle's independent index verifier (oracle.verify_index: LF walks from every known row against the text) on the
adversarial texts of sorter_cases, built by both CPU indexers (the oracle's prefix doubling and the product's SA-IS), and
on mutated indexes it must reject.  The device sorter's output is checked with the same verifier in
test_gpu_index_builder.py and, at 4.4 G rows, in test_gpu_parity.py::test_real_wide_index."""
import re

import numpy as np
import pytest

import sorter_cases as sc
from helpers import ora
from mapad_b200 import api

CASES = sc.cases()


@pytest.mark.parametrize("case", CASES, ids=[c.name for c in CASES])
def test_accepts_both_cpu_indexers(case):
    oix = ora.OracleIndex.build(case.contigs, keep_full_sa=True)
    text = ora.text_ranks(case.seqs)
    case.check_reach(text, oix.full_sa())
    want = oix.arrays()
    host = api.Index.build(case.contigs).arrays()
    assert host["contigs"] == sc.contig_table(case.contigs)
    sc.assert_same_index(want, host, "oracle vs host SA-IS")
    if case.n_extra is not None:
        assert len(host["extra_rows"]) == case.n_extra
    ora.verify_index(text, want)
    ora.verify_index(text, host)


def test_text_ranks():
    assert ora.text_ranks(["ACGT", "a"]).tolist() == [1, 2, 3, 4, 1, 0, 4, 1, 2, 3, 4, 0]
    t = ora.text_ranks(["AC" + "N" * 19, "N" + "T"])  # a run across a contig boundary counts as one
    assert t[:23].tolist() == [1, 2] + [5] * 20 + [4] and t[23] == 0 and t[24:-1].tolist() == [1] + [5] * 20 + [3, 4]
    with pytest.raises(ValueError):
        ora.text_ranks(["ACG" + "N" * 19 + "T"])
    with pytest.raises(ValueError):
        ora.text_ranks(["ACRT"])


@pytest.fixture(scope="module")
def base():
    """sentinel42: the two '$'-preceded suffixes share 42 symbols; both are unsampled (two extra rows)."""
    case = next(c for c in CASES if c.name == "sentinel42")
    a = api.Index.build(case.contigs).arrays()
    assert len(a["extra_rows"]) == 2
    return case, ora.text_ranks(case.seqs), a


def _rejects(text, a, pattern):
    for threads in (1, 8):
        with pytest.raises(ora.IndexMismatch) as e:
            ora.verify_index(text, a, n_threads=threads)
        assert re.search(pattern, str(e.value)), str(e.value)
    return str(e.value)


def test_rejects_swapped_bwt_symbols(base):
    _, text, a = base
    bwt = a["bwt"]
    i = next(i for i in range(1000, len(bwt) - 1) if bwt[i] and bwt[i + 1] and bwt[i] != bwt[i + 1])
    m = dict(a, bwt=bwt.copy())
    m["bwt"][[i, i + 1]] = bwt[[i + 1, i]]
    # rows before i are intact and LF ranks change only at i + 1, so every walk fails first at row i or i + 1
    _rejects(text, m, r"^row (%d|%d) \(text position \d+\): bwt = " % (i, i + 1))


@pytest.mark.parametrize("delta", [1, -1])
def test_rejects_shifted_sample(base, delta):
    _, text, a = base
    for k in (0, 7, len(a["sa_sample"]) - 1):
        m = dict(a, sa_sample=a["sa_sample"].copy())
        m["sa_sample"][k] = np.uint64(int(m["sa_sample"][k]) + delta)
        _rejects(text, m, r"row \d+")


def test_rejects_swapped_extra_rows(base):
    _, text, a = base
    m = dict(a, extra_rows=a["extra_rows"].copy())
    m["extra_rows"][:, 1] = a["extra_rows"][::-1, 1]
    rows = a["extra_rows"][:, 0].tolist()
    msg = _rejects(text, m, r"row \d+")
    assert any(re.search(r"row %d\b" % r, msg) for r in rows), msg
    m = dict(a, extra_rows=a["extra_rows"][:1])  # one left out
    _rejects(text, m, r"row %d\b.*missing" % rows[1])


def test_rejects_wrong_less(base):
    _, text, a = base
    for c, d in ((2, 1), (3, -1), (6, 1)):
        less = list(a["less"])
        less[c] += d
        _rejects(text, dict(a, less=less), r"less\[%d\]" % c)


def test_rejects_index_of_another_text(base):
    """The BWT and samples of a text with the same composition (two bases swapped) are not the index of the text."""
    case, text, a = base
    s = case.contigs[0][1]
    i, j = 4_000, next(j for j in range(9_000, len(s)) if s[j] != s[4_000])
    other = s[:i] + s[j] + s[i + 1:j] + s[i] + s[j + 1:]
    b = api.Index.build([("c0", other)]).arrays()
    assert b["less"] == a["less"] and not np.array_equal(b["bwt"], a["bwt"])
    _rejects(text, b, r"row \d+")
    _rejects(text, dict(a, bwt=b["bwt"]), r"row \d+")


def test_rejects_wrong_text(base):
    _, text, a = base
    _rejects(text[:-2], a, r"text of \d+ symbols")
    t = text.copy()
    t[100] = 5 - t[100] if t[100] != 5 else 1  # a base complemented: the composition changes
    _rejects(t, a, r"symbols|row \d+")


def test_accepts_cfg3_host_index():
    """The host SA-IS index of the benchmark's cfg3 genome (50 Mbp, 8 contigs, 100 M rows): ten times the size the
    oracle's own sorter is compared at."""
    from mapad_b200 import workloads
    cfg = workloads.CONFIGS["cfg3"]
    genome = workloads.random_genome_array(cfg["genome_bp"], seed=42)
    contigs = workloads.split_contigs(genome, cfg["n_contigs"])
    a = api.Index.build(contigs, seed=1234).arrays()
    assert a["n"] == 2 * cfg["genome_bp"] + 2
    ora.verify_index(ora.text_ranks([genome]), a)

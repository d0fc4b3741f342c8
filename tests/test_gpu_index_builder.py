"""`-m gpu`: the device suffix sorter (mapad_index_build_on_device, mapad_b200/csrc/gpu_index_build.cu) on the adversarial
texts of sorter_cases.  Each resolvable text must be sorted on the device (no fallback message) into exactly the arrays of
the host SA-IS and of the oracle's own sorter, and pass the independent verifier; each text with a 43-symbol tie must be
handed to the host SA-IS, with the same result."""
import os

import numpy as np
import pytest

import sorter_cases as sc
from compare import compare_results
from helpers import ora, oracle_params, product_params, random_genome, simulate_reads
from ref_cases import cli_params

pytestmark = pytest.mark.gpu
CASES = sc.cases()


@pytest.fixture(scope="module")
def api():
    from mapad_b200 import api as _api
    _api.lib()
    return _api


def build_on_device(api, contigs, capfd, **kw):
    """Device-built index arrays, and whether the sorter fell back to the host SA-IS."""
    capfd.readouterr()
    a = api.Index.build(contigs, device=0, **kw).arrays()
    return a, sc.FALLBACK_MESSAGE in capfd.readouterr().err


@pytest.mark.parametrize("case", CASES, ids=[c.name for c in CASES])
def test_device_sorter_case(api, case, capfd):
    oix = ora.OracleIndex.build(case.contigs, keep_full_sa=True)
    text = ora.text_ranks(case.seqs)
    case.check_reach(text, oix.full_sa())
    want = oix.arrays()
    del oix
    host = api.Index.build(case.contigs).arrays()
    dev, fell_back = build_on_device(api, case.contigs, capfd)
    assert fell_back == (not case.device_sorts), case.name
    assert dev["contigs"] == host["contigs"] == sc.contig_table(case.contigs)
    sc.assert_same_index(host, dev, "host SA-IS vs device")
    sc.assert_same_index(want, dev, "oracle vs device")
    if case.n_extra is not None:
        assert len(dev["extra_rows"]) == case.n_extra
    ora.verify_index(text, dev)


def test_device_sorter_iupac_runs(api, capfd):
    """Short IUPAC runs (seeded replacement draws) and N runs: the device-built index equals the host one, original symbols
    included."""
    g = random_genome(30_000, seed=31)
    g = g[:1000] + "R" + g[1000:2000] + "YYK" + g[2000:5000] + "N" * 19 + g[5000:9000] + "N" * 20 + g[9000:20000] + "BDHVNSWM" + g[20000:]
    contigs = [("a", g[:12_000]), ("b", g[12_000:])]
    host = api.Index.build(contigs, seed=77).arrays()
    dev, fell_back = build_on_device(api, contigs, capfd, seed=77)
    assert not fell_back
    assert len(dev["orig_pos"]) == 1 + 3 + 19 + 8
    sc.assert_same_index(host, dev, "host SA-IS vs device")


@pytest.mark.parametrize("library", ["single_stranded", "double_stranded"])
def test_map_on_device_built_adversarial_index(api, library, capfd):
    """Simulated reads mapped on the device-built ~1 Mbp adversarial index, against the oracle on the index of its own
    suffix sorter (not on the device's arrays)."""
    case = sc.large()
    index = api.Index.build(case.contigs, device=0)
    assert sc.FALLBACK_MESSAGE not in capfd.readouterr().err
    oix = ora.OracleIndex.build(case.contigs)
    genome = "".join(case.seqs)
    spec = cli_params(library)
    seqs, quals = simulate_reads(genome, 2000, (25, 90), seed=1234, library=library)
    # reads over the planted corners: both copies of each pair, the palindromes, the X-run flanks and the text's ends
    for k, (i, _, L) in enumerate(case.pairs):
        if i < len(genome):
            a = max(0, min(i - 10, len(genome) - L - 20))
            seqs[k] = genome[a:a + L + 20].encode()
            quals[k] = bytes([40] * len(seqs[k]))
    seeds = np.arange(len(seqs), dtype=np.uint32)
    want = ora.map_batch(oix, oracle_params(spec), seqs, quals, seeds=seeds, n_threads=os.cpu_count() or 4, want_hits=True)
    m = api.Mapper(index, product_params(spec))
    got = m.map_batch(seqs, quals, seeds=seeds, want_hits=True, with_xa=True)
    m.close()
    compare_results(want, got)
    assert got.records["mapped"].mean() > 0.6

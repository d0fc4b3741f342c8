"""Non-GPU check of the shared device logic (search_group.cuh, epilogue_core.cuh, dev_index.cuh) on the adversarial edge
workload of tests/edge_cases.py: the group kernel under the SIMT emulator for G = 1, 4, 8, 32 on both block layouts and
under every scoring model, bit for bit against the oracle.  The same workload runs on the device in tests/test_gpu_edges.py."""
import numpy as np
import pytest

import edge_cases as ec
from compare import compare_results
from helpers import oracle_params, product_params, ora
from mapad_b200 import api
from ref_cases import cli_params
from emu import emu

FRAMES_CAP = 3000  # the emulator runs lanes as coroutines: reads above this many popped frames are left to the GPU tests


@pytest.fixture(scope="module")
def small_world():
    """The edge genome with its random background shrunk to 30 % (the repeat features stay), fewer simulated reads, the
    quality-0 / -1 reads at 12 and 20 bp, and only reads the oracle maps within FRAMES_CAP frames."""
    g = ec.edge_genome(0, scale=0.3)
    index = api.Index.build(g.contigs)
    oix = ec.oracle_index(index)
    seq, qual, off, seeds = ec.edge_reads(g, 0, n_sim=150, qual_lengths=(12, 20))
    spec = cli_params("single_stranded")
    full = ora.map_batch(oix, oracle_params(spec), None, None, seeds=seeds, n_threads=4, want_hits=True, packed=(seq, qual, off))
    keep = np.nonzero(full.records["frames_popped"] <= FRAMES_CAP)[0]
    packed, seeds = ec.sub_batch((seq, qual, off), seeds, keep)
    want = ora.map_batch(oix, oracle_params(spec), None, None, seeds=seeds, n_threads=4, want_hits=True, packed=packed)
    ec.assert_coverage(ec.coverage(want, index.arrays()))
    return index, oix, packed, seeds, want


def test_edge_workload_coverage():
    """The full-size workload reaches what it exists for (multi-mappers, alts, full hit heaps, huge intervals, skipped
    positions, IUPAC symbols in MD, X rows), and the product's indexer agrees with the oracle's on its text."""
    g = ec.edge_genome(0)
    assert 500_000 < len(g.text) < 2_000_000
    index = api.Index.build(g.contigs)
    a = index.arrays()
    seq, qual, off, seeds = ec.edge_reads(g, 0)
    lengths = set(np.diff(off.astype(np.int64)).tolist())
    assert set(ec.LENGTH_LADDER) | {0} <= lengths and max(lengths) == 250
    for library in ("single_stranded", "double_stranded"):
        want = ora.map_batch(ec.oracle_index(index), oracle_params(cli_params(library)), None, None, seeds=seeds, n_threads=4,
                             want_hits=True, packed=(seq, qual, off))
        c = ec.coverage(want, a)
        print(library, c)
        ec.assert_coverage(c)
    # the two independent indexers on this text, with the same replacement draws for the short IUPAC / N runs
    draws = "ACGTTGCAAGCT" * 20
    index = api.Index.build(g.contigs, draws=draws)
    oix = ora.OracleIndex.build(g.contigs, draws=draws)
    a = index.arrays()
    assert a["n"] == oix.n == 2 * len(g.text) + 2
    assert np.array_equal(a["bwt"], oix.bwt())
    assert a["less"][: len(oix.less())] == oix.less()
    assert a["sentinel_rows"] == oix.sentinel_rows()
    assert np.array_equal(a["sa_sample"], oix.sa_samples())
    assert [tuple(x) for x in a["extra_rows"].tolist()] == oix.extra_rows()
    assert dict(zip(a["orig_pos"].tolist(), a["orig_sym"].tolist())) == oix.original_symbols()


@pytest.mark.parametrize("G", [1, 4, 8, 32])
@pytest.mark.parametrize("layout", [-1, 1], ids=["narrow", "wide"])
def test_edge_group_shapes(small_world, G, layout):
    index, oix, packed, seeds, want = small_world
    got = emu.map_batch(index, product_params(cli_params("single_stranded")), seeds=seeds, packed=packed, layout=layout,
                        group=dict(G=G, n_groups=4, pool_chunks=64))
    compare_results(want, got)


@pytest.mark.parametrize("model", ["double_stranded", "test", "vindija", "continuous", "ignore_quality", "custom_callback", "custom_table"])
def test_edge_models(small_world, model):
    """Every scoring model; the custom model (TestDifferenceModel semantics, callback or precomputed penalties) must equal
    the oracle's TEST model."""
    index, oix, packed, seeds, _ = small_world
    specs = dict(ec.model_specs(), double_stranded=cli_params("double_stranded"))
    spec = ec.TEST_SPEC if model.startswith("custom") else specs[model]
    want = ora.map_batch(oix, oracle_params(spec), None, None, seeds=seeds, n_threads=4, want_hits=True, packed=packed)
    P = ec.custom_params() if model.startswith("custom") else product_params(spec)
    table = ec.custom_penalty_table(packed[0]) if model == "custom_table" else None
    got = emu.map_batch(index, P, seeds=seeds, packed=packed, group=dict(G=8, n_groups=4, pool_chunks=64), custom_penalties=table)
    compare_results(want, got)
    assert got.records["mapped"].sum() > 0.3 * len(got)

"""`-m gpu`: the CUDA path, called through the C ABI (mapad_b200/libmapad_gpu.so), against the oracle
and against the reference's own known-answer expectations.  Bit-exact on hit intervals, scores,
edit operations, position, strand, CIGAR, MD, NM, MAPQ, X0/X1/XS/XT and the alternative hits."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from compare import compare_results
from helpers import oracle_params, product_params, ora, revcomp, random_genome, simulate_reads
from ref_cases import BENCH_PARAMS, INTEGRATION_PARAMS, SEARCH_CASES, cli_params

pytestmark = pytest.mark.gpu
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def oracle_index_from_product(index, occ_k=128):
    a = index.arrays()
    return ora.OracleIndex.from_arrays(a["bwt"], a["sa_sample"], a["sa_rate"], a["extra_rows"], a["contigs"], a["orig_pos"], a["orig_sym"],
                                       with_x=True, occ_k=occ_k)


@pytest.fixture(scope="module")
def api():
    from mapad_b200 import api as _api
    _api.lib()
    return _api


def test_reference_known_answers(api):
    """Every search known-answer case of src/map/mapping.rs:1401-2665 through the GPU."""
    for case in SEARCH_CASES:
        index = api.Index.build([("ref", case["ref"])])
        oix = oracle_index_from_product(index)
        pat = case["pattern"].encode()
        q = bytes([case["qual"]] * len(pat))
        want = ora.map_batch(oix, oracle_params(case), [pat], [q], seeds=[7], want_hits=True)
        m = api.Mapper(index, product_params(case))
        got = m.map_batch([pat], [q], seeds=[7], want_hits=True, with_xa=True)
        m.close()
        try:
            compare_results(want, got)
        except AssertionError as e:
            raise AssertionError("%s: %s" % (case["name"], e))
        e = case["expect"]
        hits = got.hits_of(0)
        if "scores_iter" in e:
            assert [np.float32(h["score"]) for h in hits] == [np.float32(s) for s in e["scores_iter"]], case["name"]
        if "n_hits" in e:
            assert len(hits) == e["n_hits"]


def test_bench_reads(api):
    data = json.load(open(os.path.join(GOLDEN, "ref_test_bench.json")))
    index = api.Index.build([("ref", data["ref_seq"])])
    oix = oracle_index_from_product(index)
    seqs = [r["pattern"].encode() for r in data["reads"]]
    quals = [bytes([40] * len(s)) for s in seqs]
    want = ora.map_batch(oix, oracle_params(BENCH_PARAMS), seqs, quals, want_hits=True)
    m = api.Mapper(index, product_params(BENCH_PARAMS))
    got = m.map_batch(seqs, quals, want_hits=True, with_xa=True)
    compare_results(want, got)
    assert [int(r["n_hits"]) for r in got.records] == [r["n_hits"] for r in data["reads"]]
    m.close()


def test_integration_fixture(api):
    """tests/integration_tests.rs: 17 reads, 4 contigs, N in the reference, multi-mappers, indels."""
    data = json.load(open(os.path.join(GOLDEN, "ref_integration.json")))
    index = api.Index.build([(n, s) for n, s in data["contigs"]], draws="A")
    oix = ora.OracleIndex.build([(n, s) for n, s in data["contigs"]], draws="A")
    seqs, quals = [], []
    for r in data["reads"]:
        s, q = r["seq"], bytes(c - 33 for c in r["qual"].encode())
        if r["flag"] & 16:
            s, q = revcomp(s), q[::-1]
        seqs.append(s.encode())
        quals.append(q)
    seeds = list(range(100, 100 + len(seqs)))
    want = ora.map_batch(oix, oracle_params(INTEGRATION_PARAMS), seqs, quals, seeds=seeds, want_hits=True)
    m = api.Mapper(index, product_params(INTEGRATION_PARAMS))
    got = m.map_batch(seqs, quals, seeds=seeds, want_hits=True, with_xa=True)
    m.close()
    compare_results(want, got)
    exp = {e["name"]: e for e in data["expectation"]}
    for i, r in enumerate(data["reads"]):
        e = exp[r["name"]]
        s = got.record_summary(i)
        if e["tid"] is None:
            assert not s["mapped"] and s["mapq"] == 0
        else:
            assert (s["tid"], s["pos"] + 1, s["mapq"], s["cigar"], s["md"], s["x0"], s["x1"], s["xt"]) == \
                   (e["tid"], e["pos"], e["mq"], e["cigar"], e["md"], e["x0"], e["x1"], e["xt"]), r["name"]
            assert got.xa[i] == (e["xa"] or "")
            if e["xs"] is not None:
                assert np.float32(s["xs"]) == np.float32(e["xs"])


@pytest.mark.parametrize("library,len_range,n_reads,gsize", [("single_stranded", (50, 50), 3000, 1_000_000),
                                                             ("double_stranded", (30, 75), 2000, 400_000)])
def test_simulated_reads_vs_oracle(api, library, len_range, n_reads, gsize):
    genome = random_genome(gsize, seed=42)
    cut = gsize // 3
    index = api.Index.build([("chr1", genome[:cut]), ("chr2", genome[cut:])])
    oix = oracle_index_from_product(index)
    spec = cli_params(library)
    seqs, quals = simulate_reads(genome, n_reads, len_range, seed=1001, library=library)
    seqs[5] = seqs[5][:10] + b"N" + seqs[5][11:]
    seqs[6] = b""
    quals[6] = b""
    seeds = (np.arange(len(seqs), dtype=np.uint64) * 2654435761 % (1 << 32)).astype(np.uint32)
    want = ora.map_batch(oix, oracle_params(spec), seqs, quals, seeds=seeds, n_threads=os.cpu_count() or 4, want_hits=True)
    m = api.Mapper(index, product_params(spec))
    got = m.map_batch(seqs, quals, seeds=seeds, want_hits=True, with_xa=True)
    compare_results(want, got)
    mapped = sum(int(r["mapped"]) for r in got.records)
    assert mapped > 0.6 * n_reads, mapped
    # idempotence: a second pass over the resident batch returns identical records
    from mapad_b200 import abi
    res2 = abi.BatchResult(m.map_raw(None, abi.BATCH_RESIDENT | abi.BATCH_WANT_HITS))
    compare_results(got, res2, label_a="pass1", label_b="pass2")
    m.close()


def _run_child(code, env_extra):
    env = dict(os.environ)
    env.update(env_extra)
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, "-c", code], env=env, cwd=os.path.join(root, "tests"), capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout + r.stderr
    return r.stdout


CHILD = r"""
import numpy as np, os, sys
sys.path.insert(0, os.path.dirname(os.getcwd())); sys.path.insert(0, os.getcwd())
from compare import compare_results
from helpers import oracle_params, product_params, ora, random_genome, simulate_reads
from ref_cases import cli_params
from mapad_b200 import api
genome = random_genome(200000, seed=43)
index = api.Index.build([("chr1", genome)])
a = index.arrays()
oix = ora.OracleIndex.from_arrays(a["bwt"], a["sa_sample"], a["sa_rate"], a["extra_rows"], a["contigs"], a["orig_pos"], a["orig_sym"])
spec = cli_params("single_stranded")
SPEC_EXTRA
seqs, quals = simulate_reads(genome, 600, (30, 90), seed=77)
seeds = np.arange(len(seqs), dtype=np.uint32)
want = ora.map_batch(oix, oracle_params(spec), seqs, quals, seeds=seeds, n_threads=os.cpu_count() or 4, want_hits=True)
m = api.Mapper(index, product_params(spec))
got = m.map_batch(seqs, quals, seeds=seeds, want_hits=True, with_xa=True)
compare_results(want, got)
print("deferred", int(sum(1 for r in got.records if r["flags"] & 2)), "limit", int(sum(1 for r in got.records if r["flags"] & 1)))
"""


def test_wide_layout_and_retry_launch(api):
    """64-bit block layout forced on a small index, and a chunk pool so small that it runs dry: reads are handed back
    and re-run with fewer groups in flight; results must not change.  Also every group size the library is built for."""
    out = _run_child(CHILD.replace("SPEC_EXTRA", ""), {"MAPAD_FORCE_WIDE": "1"})
    for g in ("1", "4", "16", "32"):
        _run_child(CHILD.replace("SPEC_EXTRA", ""), {"MAPAD_GROUP": g})
    # latency-hiding variants of the one-read-per-warp kernel: heap-line + occ prefetch, 171 heap lines in shared memory,
    # kernels compiled for 20 / 24 resident warps per SM
    _run_child(CHILD.replace("SPEC_EXTRA", ""), {"MAPAD_FORCE_WIDE": "1", "MAPAD_TRICKLE_PREFETCH": "3", "MAPAD_TOPL": "171"})
    _run_child(CHILD.replace("SPEC_EXTRA", ""), {"MAPAD_FORCE_WIDE": "1", "MAPAD_TRICKLE_PREFETCH": "3", "MAPAD_GROUPS_PER_SM": "24"})
    _run_child(CHILD.replace("SPEC_EXTRA", ""), {"MAPAD_FORCE_WIDE": "1", "MAPAD_TRICKLE_PREFETCH": "2", "MAPAD_GROUPS_PER_SM": "20"})
    _run_child(CHILD.replace("SPEC_EXTRA", ""), {"MAPAD_FORCE_WIDE": "1", "MAPAD_TOPL": "11"})
    # 16 groups own 32 of the 72 chunks (256 KiB each); the largest of these reads pops 3e5 frames, so the 40 pooled chunks
    # run dry while several groups grow at once (calibrated with the emulation: tests/test_group_kernel.py)
    out = _run_child(CHILD.replace("SPEC_EXTRA", "").replace("(30, 90)", "(50, 70)").replace("genome = random_genome(200000, seed=43)", "genome = random_genome(3000000, seed=43)"),
                     {"MAPAD_GROUPS": "16", "MAPAD_TEST_POOL_CHUNKS": "72"})
    assert int(out.split("deferred")[1].split()[0]) > 0, out


def test_search_limits_eviction(api):
    """STACK_LIMIT / EDIT_TREE_LIMIT recovery (mapping.rs:1358-1380) with small limits: pop_min eviction and
    slab key reuse must match the oracle."""
    out = _run_child(CHILD.replace("SPEC_EXTRA", "spec['limits'] = (300, 700)"), {})
    assert int(out.split("limit")[1].split()[0]) > 20, out
    out = _run_child(CHILD.replace("SPEC_EXTRA", "spec['limits'] = (300, 700); spec['abort'] = True"), {})
    assert int(out.split("limit")[1].split()[0]) > 20, out
    # pop_min descents with the speculative line prefetch (heaps reaching below the shared-memory top)
    out = _run_child(CHILD.replace("SPEC_EXTRA", "spec['limits'] = (300, 700)"), {"MAPAD_TRICKLE_PREFETCH": "3", "MAPAD_GROUP": "8"})
    assert int(out.split("limit")[1].split()[0]) > 20, out
    out = _run_child(CHILD.replace("SPEC_EXTRA", "spec['limits'] = (2000, 5000)"), {"MAPAD_TRICKLE_PREFETCH": "3", "MAPAD_FORCE_WIDE": "1"})
    assert int(out.split("limit")[1].split()[0]) > 0, out


def test_cfg3_size_index(api):
    """The benchmarked cfg3 index itself (50 Mbp, 8 contigs, host SA-IS) with reads simulated exactly like bench.py's chunks."""
    from mapad_b200 import workloads
    cfg = workloads.CONFIGS["cfg3"]
    genome = workloads.random_genome_array(cfg["genome_bp"], seed=42)
    index = api.Index.build(workloads.split_contigs(genome, cfg["n_contigs"]), seed=1234)
    oix = oracle_index_from_product(index)
    spec = cli_params(cfg["library"])
    n = 4000
    packed = workloads.simulate_batch(genome, n, cfg["len_range"], seed=cfg["seed"] * 1000 + 20_000, library=cfg["library"])
    seeds = np.arange(n, dtype=np.uint32)
    want = ora.map_batch(oix, oracle_params(spec), None, None, seeds=seeds, n_threads=os.cpu_count() or 4, want_hits=True, packed=packed)
    m = api.Mapper(index, product_params(spec))
    got = m.map_batch(seeds=seeds, want_hits=True, packed=packed)
    m.close()
    compare_results(want, got)
    assert got.records["mapped"].mean() > 0.8 and got.records["tid"].max() == 7


def test_continuous_bound(api):
    """Continuous mismatch bound (-c / -e of older mapAD versions, mismatch_bounds.rs:77-121) on the device."""
    genome = random_genome(1_000_000, seed=5)
    index = api.Index.build([("c1", genome[:400_000]), ("c2", genome[400_000:])])
    oix = oracle_index_from_product(index)
    spec = dict(cli_params("single_stranded"))
    spec["bound"] = ("continuous", -0.25, 1.0)
    seqs, quals = simulate_reads(genome, 1500, (25, 80), seed=17)
    seeds = np.arange(len(seqs), dtype=np.uint32)
    want = ora.map_batch(oix, oracle_params(spec), seqs, quals, seeds=seeds, n_threads=os.cpu_count() or 4, want_hits=True)
    m = api.Mapper(index, product_params(spec))
    got = m.map_batch(seqs, quals, seeds=seeds, want_hits=True)
    m.close()
    compare_results(want, got)
    assert 0.3 < got.records["mapped"].mean() <= 1.0


def test_cfg5_cell(api):
    """One cell of the BASELINE cfg5 stress sweep (L = 100, -p 0.06: k(100) = 7 allowed mismatches) on a small index, so that
    the oracle finishes in seconds: deep heaps, pool growth and (with the small limits of the second pass) eviction."""
    genome = random_genome(1_500_000, seed=9)
    index = api.Index.build([("c", genome)])
    oix = oracle_index_from_product(index)
    spec = dict(cli_params("single_stranded"))
    spec["bound"] = ("discrete", 0.06, 0.02)
    seqs, quals = simulate_reads(genome, 300, (100, 100), seed=23)
    seeds = np.arange(len(seqs), dtype=np.uint32)
    m = api.Mapper(index, product_params(spec))
    for limits in (None, (3000, 9000)):
        if limits:
            spec["limits"] = limits
            m.set_params(product_params(spec))
        want = ora.map_batch(oix, oracle_params(spec), seqs, quals, seeds=seeds, n_threads=os.cpu_count() or 4, want_hits=True)
        got = m.map_batch(seqs, quals, seeds=seeds, want_hits=True)
        compare_results(want, got)
    assert sum(1 for r in got.records if r["flags"] & 1) > 5
    m.close()


def test_real_wide_index(api, capfd):
    """A reference whose text (2 G + 2 symbols) exceeds 2^32 rows: device suffix sorter, 64-byte occ blocks, u64 SA samples,
    40-bit tree nodes.  Reads from both strands, reads that straddle a contig boundary (must not be reported there), and
    rows / positions beyond 2^32.  The oracle maps on the device's own arrays, so they are first checked against the text
    by the independent verifier."""
    import time
    from mapad_b200 import workloads
    from sorter_cases import FALLBACK_MESSAGE
    gbp = 2_200_000_000
    genome = workloads.random_genome_array(gbp, seed=42)
    contigs = workloads.split_contigs(genome, 24)
    capfd.readouterr()
    index = api.Index.build(contigs, device=0)
    assert FALLBACK_MESSAGE not in capfd.readouterr().err
    del contigs
    a = index.arrays()
    assert a["n"] == 2 * gbp + 2 and a["n"] > 1 << 32
    t0 = time.time()
    ora.verify_index(ora.text_ranks([genome]), a)
    with capfd.disabled():
        print("\nverify_index: %d rows in %.1f s on %d threads" % (a["n"], time.time() - t0, os.cpu_count() or 1))
    oix = ora.OracleIndex.from_arrays(a["bwt"], a["sa_sample"], a["sa_rate"], a["extra_rows"], a["contigs"], a["orig_pos"], a["orig_sym"])
    del a
    spec = cli_params("single_stranded")
    n = 260
    seq, qual, off = workloads.simulate_batch(genome, n, (25, 60), seed=77)
    # 20 undamaged reads across contig boundaries (10 per strand): their only exact locus straddles two contigs
    cuts = [gbp * i // 24 for i in range(25)]  # workloads.split_contigs
    comp = {65: 84, 67: 71, 71: 67, 84: 65}
    for k in range(20):
        L = int(off[k + 1] - off[k])
        b = cuts[k % 23 + 1]  # boundary between contig (k % 23) and the next
        w = genome[b - L // 2: b - L // 2 + L].copy()
        if k % 2:
            w = np.array([comp[int(c)] for c in w[::-1]], dtype=np.uint8)
        seq[int(off[k]):int(off[k + 1])] = w
        qual[int(off[k]):int(off[k + 1])] = 40
    seeds = np.arange(n, dtype=np.uint32)
    want = ora.map_batch(oix, oracle_params(spec), None, None, seeds=seeds, n_threads=os.cpu_count() or 4, want_hits=True, packed=(seq, qual, off))
    m = api.Mapper(index, product_params(spec))
    got = m.map_batch(seeds=seeds, want_hits=True, packed=(seq, qual, off))
    m.close()
    compare_results(want, got)
    rec = got.records
    assert int(rec["best_lower"].max()) > 1 << 32 and int(rec["absolute_pos"].max()) > 1 << 31
    assert rec["strand"][rec["mapped"] != 0].sum() > 20
    for k in range(20):  # never reported at the locus it was cut from
        if rec["mapped"][k]:
            L = int(off[k + 1] - off[k])
            assert abs(int(rec["absolute_pos"][k]) - (cuts[k % 23 + 1] - L // 2)) > L, k


def test_device_index_builder_matches_host(api, capfd):
    """mapad_index_build_on_device (prefix-key radix sort on the GPU) must produce exactly the arrays of the host
    SA-IS builder; a repetitive text makes it fall back to the host builder (still identical)."""
    from sorter_cases import FALLBACK_MESSAGE
    for gsize, seed in ((300_000, 7), (65_537, 8)):
        genome = random_genome(gsize, seed=seed)
        contigs = [("a", genome[: gsize // 2]), ("b", genome[gsize // 2:])]
        host = api.Index.build(contigs).arrays()
        capfd.readouterr()
        dev = api.Index.build(contigs, device=0).arrays()
        assert FALLBACK_MESSAGE not in capfd.readouterr().err  # sorted on the device
        assert host["n"] == dev["n"] and host["less"] == dev["less"] and host["sentinel_rows"] == dev["sentinel_rows"]
        assert np.array_equal(host["bwt"], dev["bwt"])
        assert np.array_equal(host["sa_sample"], dev["sa_sample"])
        assert np.array_equal(host["extra_rows"], dev["extra_rows"])
    rep = [("r", "ACGT" * 200 + "N" * 30 + "GATTACA" * 50)]
    host = api.Index.build(rep).arrays()
    capfd.readouterr()
    dev = api.Index.build(rep, device=0).arrays()
    assert FALLBACK_MESSAGE in capfd.readouterr().err
    assert np.array_equal(host["bwt"], dev["bwt"]) and np.array_equal(host["sa_sample"], dev["sa_sample"])


def test_cli_fastq_to_bam(api, tmp_path):
    """`python -m mapad_b200.cli map` end to end on the GPU: FASTA + FASTQ.GZ in, BAM out, records in input order and
    identical to what the oracle decides for every read."""
    import gzip
    from bamio import read_bam
    genome = random_genome(120_000, seed=21)
    contigs = [("chrA", genome[:50_000]), ("chrB", genome[50_000:])]
    fa = tmp_path / "g.fa"
    with open(fa, "w") as f:
        for n, s in contigs:
            f.write(">%s test contig\n" % n)
            for i in range(0, len(s), 70):
                f.write(s[i:i + 70] + "\n")
    seqs, quals = simulate_reads(genome, 700, (30, 70), seed=5)
    fq = tmp_path / "r.fastq.gz"
    with gzip.open(fq, "wt") as f:
        for i, (s, q) in enumerate(zip(seqs, quals)):
            f.write("@read%d\n%s\n+\n%s\n" % (i, s.decode(), bytes(c + 33 for c in q).decode()))
    out = tmp_path / "o.bam"
    cmd = [sys.executable, "-m", "mapad_b200.cli", "map", "-r", str(fq), "-g", str(fa), "-o", str(out), "--library", "single_stranded",
           "-p", "0.03", "-f", "0.5", "-t", "0.5", "-d", "0.02", "-s", "1.0", "-i", "0.001", "-x", "0.5", "--batch_size", "150", "--seed", "99"]
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    # `index` writes the seven index files next to the FASTA; `map` then loads them instead of re-indexing
    r = subprocess.run([sys.executable, "-m", "mapad_b200.cli", "index", "-g", str(fa)], cwd=root, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout + r.stderr
    assert all(os.path.exists(str(fa) + "." + s) for s in ("tbw", "tle", "toc", "trt", "tsa", "tpi", "tos"))
    r = subprocess.run(cmd, cwd=root, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "indexing in memory" not in r.stderr
    text, refs, recs = read_bam(str(out))
    assert [x["name"] for x in recs] == ["read%d" % i for i in range(700)]
    assert refs == [("chrA", 50_000), ("chrB", 70_000)]
    # same seeds as the CLI draws (numpy generator seeded with --seed, one draw per read, chunk by chunk)
    rng = np.random.default_rng(99)
    seeds = np.concatenate([rng.integers(0, 1 << 32, size=min(150, 700 - k), dtype=np.uint64).astype(np.uint32) for k in range(0, 700, 150)])
    index = api.Index.build(contigs)
    oix = oracle_index_from_product(index)
    spec = cli_params("single_stranded")
    want = ora.map_batch(oix, oracle_params(spec), seqs, quals, seeds=seeds, n_threads=os.cpu_count() or 4, want_hits=False)
    for i, rec in enumerate(recs):
        s = want.record_summary(i)
        if not s["mapped"]:
            assert rec["flag"] & 4
            continue
        assert (rec["ref_id"], rec["pos"], rec["mapq"], rec["cigar"], rec["tags"]["MD"], rec["tags"]["NM"]) == \
               (s["tid"], s["pos"], s["mapq"], s["cigar"], s["md"], s["nm"]), i
        assert bool(rec["flag"] & 16) == bool(s["strand"])
        assert np.float32(rec["tags"]["AS"]) == np.float32(s["AS"])
    # the same reads as an unaligned BAM (the usual aDNA input): identical records, input tags carried over
    from bamio import write_bam
    src = tmp_path / "r.bam"
    write_bam(str(src), "@HD\tVN:1.6\n@PG\tID:leeHom\tPN:leeHom\n",
              [], [dict(name="read%d" % i, flag=4, seq=s_.decode(), qual=bytes(q_), aux=b"XYZorig\x00") for i, (s_, q_) in enumerate(zip(seqs, quals))])
    out2 = tmp_path / "o2.bam"
    cmd2 = [c if c != str(fq) else str(src) for c in cmd]
    cmd2[cmd2.index(str(out))] = str(out2)
    r = subprocess.run(cmd2, cwd=root, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout + r.stderr
    text2, refs2, recs2 = read_bam(str(out2))
    assert refs2 == refs and "@PG\tID:leeHom\tPN:leeHom\n" in text2 and "\tPP:leeHom\n" in text2
    assert len(recs2) == len(recs)
    for a, b in zip(recs, recs2):
        assert b["tags"].pop("XY") == "orig"
        b["tag_order"].remove("XY")
        assert a == b, a["name"]


def test_full_size_cfg1_properties(api):
    """BASELINE cfg1 at full size (1 Mbp reference, 100 000 x 50 bp reads): size-independent properties —
    chunking invariance (one chunk vs seven ragged chunks give identical records), internal consistency of every
    record (CIGAR query length = read length, NM = edits implied by CIGAR + MD, reference span inside the contig),
    exact-copy reads map to their origin — plus the oracle on a 4 000-read subset."""
    import re
    from mapad_b200 import abi, workloads
    cfg = workloads.CONFIGS["cfg1"]
    genome = workloads.random_genome_array(cfg["genome_bp"], seed=42)
    index = api.Index.build(workloads.split_contigs(genome, 1))
    spec = cli_params("single_stranded")
    m = api.Mapper(index, product_params(spec))
    seq, qual, off = workloads.simulate_batch(genome, cfg["n_reads"], cfg["len_range"], seed=cfg["seed"])
    n = len(off) - 1
    # plant 500 exact copies (forward strand, quality 40) at known positions
    rng = np.random.default_rng(1)
    planted = rng.integers(0, cfg["genome_bp"] - 60, size=500)
    for k, p in enumerate(planted):
        Lk = int(off[k + 1] - off[k])
        seq[int(off[k]):int(off[k + 1])] = genome[p:p + Lk]
        qual[int(off[k]):int(off[k + 1])] = 40
    seeds = np.arange(n, dtype=np.uint32)
    whole = m.map_batch(seeds=seeds, packed=(seq, qual, off))
    cuts = [0, 1, 17, 5000, 5001, 40000, 99999, n]
    parts = []
    for a, b in zip(cuts[:-1], cuts[1:]):
        sub = (seq[int(off[a]):int(off[b])], qual[int(off[a]):int(off[b])], (off[a:b + 1] - off[a]).astype(np.uint64))
        parts.append(m.map_batch(seeds=seeds[a:b], packed=sub))
    from mapad_b200 import sharding
    merged = sharding.merge_results(parts)
    compare_results(whole, merged, check_hits=False, label_a="one chunk", label_b="seven chunks")
    rec = whole.records
    assert rec["mapped"].mean() > 0.8
    for k, p in enumerate(planted):
        assert rec["mapped"][k] and rec["pos"][k] == p and rec["strand"][k] == 0 and rec["nm"][k] == 0, k
    for i in np.nonzero(rec["mapped"])[0][:20000]:
        cig = whole.cigar_str(int(rec["cigar_off"][i]), int(rec["cigar_len"][i]))
        md = whole.md_str(int(rec["md_off"][i]), int(rec["md_len"][i]))
        ops = [(int(a), b) for a, b in re.findall(r"(\d+)([MID])", cig)]
        assert sum(a for a, b in ops if b in "MI") == int(off[i + 1] - off[i]), (i, cig)
        ref_span = sum(a for a, b in ops if b in "MD")
        assert rec["pos"][i] >= 0 and rec["pos"][i] + ref_span <= cfg["genome_bp"]
        mism = len(re.findall(r"(?<![\^A-Z])[A-Z]", re.sub(r"\^[A-Z]+", "^", md)))
        dels = sum(a for a, b in ops if b == "D")
        ins = sum(a for a, b in ops if b == "I")
        assert rec["nm"][i] == mism + dels + ins, (i, cig, md, int(rec["nm"][i]))
    sub_n = 4000
    oix = oracle_index_from_product(index)
    sub = (seq[: int(off[sub_n])], qual[: int(off[sub_n])], off[: sub_n + 1])
    want = ora.map_batch(oix, oracle_params(spec), None, None, seeds=seeds[:sub_n], n_threads=os.cpu_count() or 4, want_hits=True, packed=sub)
    got = m.map_batch(seeds=seeds[:sub_n], want_hits=True, packed=sub)
    compare_results(want, got)
    m.close()

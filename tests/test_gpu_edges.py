"""`-m gpu`: the CUDA path on the adversarial edge workload of tests/edge_cases.py, against the oracle, bit for bit on records,
hits, edit operations, CIGAR, MD and XA: every group shape on both block layouts, every scoring model, output-pool growth,
one handle reused across batch shapes and parameter sets, and several handles competing for one dry chunk pool."""
import os
import time

import numpy as np
import pytest

import edge_cases as ec
from compare import compare_results
from helpers import oracle_params, product_params, ora
from ref_cases import cli_params
from test_gpu_parity import _run_child

pytestmark = pytest.mark.gpu
N_THREADS = os.cpu_count() or 4


@pytest.fixture(scope="module")
def world():
    from mapad_b200 import api
    api.lib()
    g = ec.edge_genome(0)
    index = api.Index.build(g.contigs)
    seq, qual, off, seeds = ec.edge_reads(g, 0)
    return api, g, index, ec.oracle_index(index), (seq, qual, off), seeds


def _oracle(oix, spec, packed, seeds):
    t = time.time()
    want = ora.map_batch(oix, oracle_params(spec), None, None, seeds=seeds, n_threads=N_THREADS, want_hits=True, packed=packed)
    print("oracle %.1f s for %d reads" % (time.time() - t, len(want)))
    return want


CHILD_SHAPES = r"""
import os, sys
sys.path.insert(0, os.path.dirname(os.getcwd())); sys.path.insert(0, os.getcwd())
import edge_cases as ec
from compare import compare_results
from helpers import oracle_params, product_params, ora
from ref_cases import cli_params
from mapad_b200 import api
g = ec.edge_genome(0)
index = api.Index.build(g.contigs)
oix = ec.oracle_index(index)
seq, qual, off, seeds = ec.edge_reads(g, 0)
for library in ("single_stranded", "double_stranded"):
    spec = cli_params(library)
    want = ora.map_batch(oix, oracle_params(spec), None, None, seeds=seeds, n_threads=os.cpu_count() or 4, want_hits=True, packed=(seq, qual, off))
    m = api.Mapper(index, product_params(spec))
    got = m.map_batch(seeds=seeds, want_hits=True, packed=(seq, qual, off), with_xa=True)
    m.close()
    compare_results(want, got)
    ec.assert_coverage(ec.coverage(got, index.arrays()))
    print(library, "ok", ec.coverage(got))
"""


@pytest.mark.parametrize("env", [{"MAPAD_GROUP": "1"}, {"MAPAD_GROUP": "4"}, {"MAPAD_GROUP": "8"}, {"MAPAD_GROUP": "16"}, {"MAPAD_GROUP": "32"},
                                 {"MAPAD_FORCE_WIDE": "1", "MAPAD_GROUP": "8"}, {"MAPAD_FORCE_WIDE": "1", "MAPAD_GROUP": "32"}],
                         ids=["narrow-G1", "narrow-G4", "narrow-G8", "narrow-G16", "narrow-G32", "wide-G8", "wide-G32"])
def test_edge_workload_group_shapes(env):
    """Both CLI libraries on every lane-group size; the wide 64-bit block layout at G = 8 and at G = 32 (the hg19-scale
    default).  The X-flagged occ blocks, the '$' corrections and the shuffles of extend_all_group run here on the device."""
    out = _run_child(CHILD_SHAPES, env)
    assert out.count(" ok ") == 2, out


@pytest.mark.parametrize("model", ["test", "vindija", "continuous", "ignore_quality", "custom_callback", "custom_table"])
def test_edge_workload_models(world, model):
    """Every scoring model on the device.  The custom model has TestDifferenceModel's semantics, through the host callback
    or through precomputed penalties, and must equal the oracle's TEST model."""
    api, g, index, oix, packed, seeds = world
    specs = ec.model_specs()
    spec = ec.TEST_SPEC if model.startswith("custom") else specs[model]
    want = _oracle(oix, spec, packed, seeds)
    P = ec.custom_params() if model.startswith("custom") else product_params(spec)
    m = api.Mapper(index, P)
    table = ec.custom_penalty_table(packed[0]) if model == "custom_table" else None
    got = m.map_batch(seeds=seeds, want_hits=True, packed=packed, with_xa=True, custom_penalties=table)
    m.close()
    compare_results(want, got)
    assert got.records["mapped"].sum() > 0.3 * len(got), model


def _pool_demand(res):
    """(hits, edit operations, MD / XA text bytes) a result occupies in the output pools."""
    r = res.records
    ops = sum(len(h["ops"]) for i in range(len(res)) for h in res.hits_of(i))
    text = int(r["md_len"].sum()) + int(r["alts"]["md_len"][r["n_alts"] >= 1, 0].sum()) + int(r["alts"]["md_len"][r["n_alts"] >= 2, 1].sum())
    return int(r["n_hits"].sum()), ops, text


def test_output_pool_growth(world):
    """The first batch on a fresh handle overflows the hit, edit-op and text pools (run_batch sizes them 4n + 1024 hits,
    4 bases + 64n + 1024 ops, 24n + 1024 bytes of text, each with the 25 % slack of DevBuf::reserve): K2 and K3 are re-run
    with grown pools.  The same batch on the grown handle needs fewer launches; both must equal the oracle."""
    api, g, index, oix, packed, seeds = world
    spec = cli_params("single_stranded")
    full = _oracle(oix, spec, packed, seeds)
    r = full.records
    # cheap reads with full hit heaps and long MD strings (the quality-0 / -1 reads of 20 bp), repeated
    heavy = [i for i in range(len(r)) if r["n_hits"][i] >= 10 and r["frames_popped"][i] < 50_000]
    assert len(heavy) >= 2, heavy
    idx = (heavy * (3000 // len(heavy) + 1))[:3000]
    sub, sub_seeds = ec.sub_batch(packed, np.arange(len(idx), dtype=np.uint32) * 7919, idx)
    want = _oracle(oix, spec, sub, sub_seeds)
    n, tb = len(idx), int(sub[2][-1])
    slack = lambda k: k + k // 4 + 64
    hits, ops, text = _pool_demand(want)
    assert hits > slack(4 * n + 1024) and ops > slack(4 * tb + 64 * n + 1024) and text > slack(24 * n + 1024), (hits, ops, text, n, tb)
    m = api.Mapper(index, product_params(spec))
    first = m.map_batch(seeds=sub_seeds, want_hits=True, packed=sub, with_xa=True)
    compare_results(want, first)
    second = m.map_batch(seeds=sub_seeds, want_hits=True, packed=sub, with_xa=True)
    compare_results(want, second)
    print("launches: fresh handle %d, grown handle %d" % (first.gpu_launches, second.gpu_launches))
    assert first.gpu_launches > second.gpu_launches
    m.close()


def _xa(api, index, res_struct, out):
    import ctypes as C
    buf = C.create_string_buffer(1 << 16)
    out.xa = []
    for i in range(len(out)):
        k = api.lib().mapad_format_xa(index.h, C.byref(res_struct), i, buf, 1 << 16)
        assert k >= 0
        out.xa.append(buf.raw[:k].decode())
    return out


def test_handle_reuse_across_shapes(world):
    """One handle: a large batch, a 1-read batch, a 0-read batch, the large batch again, switching the model in between; then
    bench.py's staging path (BATCH_UPLOAD_ONLY, then BATCH_RESIDENT).  Grow-only device buffers keep the data of larger
    batches, so a cursor or count that is not reset would show here."""
    from mapad_b200 import abi
    api, g, index, oix, packed, seeds = world
    ss, specs = cli_params("single_stranded"), ec.model_specs()
    want_ss = _oracle(oix, ss, packed, seeds)
    multi = int(np.nonzero((want_ss.records["n_alts"] == 2) & (want_ss.records["x1"] > 0))[0][0]) if \
        ((want_ss.records["n_alts"] == 2) & (want_ss.records["x1"] > 0)).any() else int(np.argmax(want_ss.records["n_alts"]))
    one, one_seeds = ec.sub_batch(packed, seeds, [multi])
    empty = (np.zeros(0, np.uint8), np.zeros(0, np.uint8), np.zeros(1, np.uint64))
    m = api.Mapper(index, product_params(ss))
    compare_results(want_ss, m.map_batch(seeds=seeds, want_hits=True, packed=packed, with_xa=True))
    m.set_params(product_params(specs["test"]))
    compare_results(_oracle(oix, specs["test"], one, one_seeds), m.map_batch(seeds=one_seeds, want_hits=True, packed=one, with_xa=True))
    m.set_params(product_params(specs["vindija"]))
    assert len(m.map_batch(seeds=np.zeros(0, np.uint32), want_hits=True, packed=empty, with_xa=True)) == 0
    m.set_params(product_params(ss))
    compare_results(want_ss, m.map_batch(seeds=seeds, want_hits=True, packed=packed, with_xa=True))
    # staging: upload one batch, run it later from HBM (with another model than the previous run)
    m.set_params(product_params(specs["continuous"]))
    want_c = _oracle(oix, specs["continuous"], packed, seeds)
    R, keep = api.make_reads(packed[0], packed[1], packed[2], seeds)
    assert m.map_raw(R, abi.BATCH_UPLOAD_ONLY).n_reads == len(seeds)
    res = m.map_raw(None, abi.BATCH_RESIDENT | abi.BATCH_WANT_HITS)
    compare_results(want_c, _xa(api, index, res, abi.BatchResult(res)))
    del keep
    m.close()


CHILD_CONCURRENT = r"""
import os, sys, threading, time
sys.path.insert(0, os.path.dirname(os.getcwd())); sys.path.insert(0, os.getcwd())
import numpy as np
import edge_cases as ec
from compare import compare_results
from helpers import oracle_params, product_params, ora, simulate_reads
from ref_cases import cli_params
from mapad_b200 import api
H = 6
g = ec.edge_genome(0)
index = api.Index.build(g.contigs)
oix = ec.oracle_index(index)
seq, qual, off, seeds = ec.edge_reads(g, 0)
n = len(seeds)
# six heavy chunks: the edge workload in two halves, and a cfg5-like slice (L = 100, -p 0.06: 7 allowed mismatches) twice
# without and twice with small search limits
ss = cli_params("single_stranded")
cfg5 = dict(ss, bound=("discrete", 0.06, 0.02))
sim_text = g.text.copy()
sim_text[~np.isin(sim_text, ec.ACGT)] = ord("N")
chunks = [ec.sub_batch((seq, qual, off), seeds, range(0, n // 2)) + (ss,), ec.sub_batch((seq, qual, off), seeds, range(n // 2, n)) + (ss,)]
for k in range(4):
    s_, q_ = simulate_reads(sim_text.tobytes().decode(), 120, (100, 100), seed=500 + k)
    from mapad_b200 import abi
    packed = abi.pack_reads(s_, q_)
    chunks.append((packed, np.arange(len(s_), dtype=np.uint32) + 1000 * k, cfg5 if k < 2 else dict(cfg5, limits=(3000, 9000))))
wants = [ora.map_batch(oix, oracle_params(sp), None, None, seeds=sd, n_threads=os.cpu_count() or 4, want_hits=True, packed=pk) for pk, sd, sp in chunks]
# Pool size.  A popped frame costs ~105 bytes of pool (2.5 tree nodes of 32 B + 1.5 heap entries of 8 B with their line
# overhead; 0.0257 chunks of 4 KiB per frame, calibrated with the emulation in tests/test_group_kernel.py), i.e. a 256 KiB
# chunk holds ~2500 frames.  The heaviest read must fit the pool on its own (else the batch fails by design), so the pool is
# 1.5 x that read's chunks + 16.  Each launch takes up to pool / 4 groups x 2 base chunks (search_with_groups), so two
# launches hold the whole pool in base chunks and the other four, and every read that grows, find it dry.
max_frames = max(int(w.records["frames_popped"].max()) for w in wants)
pool = int(max_frames * 105 / 262144 * 1.5) + 16
os.environ["MAPAD_TEST_POOL_CHUNKS"] = str(pool)
print("max frames", max_frames, "pool chunks", pool)
api.plan_handles(0, H)
m0 = api.Mapper(index, product_params(ss))
handles = [m0] + [m0.clone() for _ in range(H - 1)]
for h, (pk, sd, sp) in zip(handles, chunks):
    h.set_params(product_params(sp))
res, span, errs = [None] * H, [None] * H, []
def run(k):
    try:
        t0 = time.monotonic()
        pk, sd, sp = chunks[k]
        res[k] = handles[k].map_batch(seeds=sd, want_hits=True, packed=pk, with_xa=True)
        span[k] = (t0, time.monotonic())
    except Exception as e:
        errs.append((k, repr(e), api.lib().mapad_gpu_last_error(handles[k].h)))
threads = [threading.Thread(target=run, args=(k,)) for k in range(H)]
for t in threads: t.start()
for t in threads: t.join()
assert not errs, errs
handed_back, overlapped = [], 0
for k in range(H):
    compare_results(wants[k], res[k], label_b="handle %d" % k)
    hb = int(np.count_nonzero(res[k].records["flags"] & 2))
    handed_back.append(hb)
    if hb and any(j != k and span[j][0] < span[k][1] and span[k][0] < span[j][1] for j in range(H)):
        overlapped += 1
print("handed back", handed_back, "spans", [(round(a - span[0][0], 2), round(b - span[0][0], 2)) for a, b in span])
assert overlapped > 0, "no read was handed back in a launch that overlapped another handle's"
# each chunk alone on one handle: the same records (compare_results does not look at the flags)
for k, (pk, sd, sp) in enumerate(chunks):
    m0.set_params(product_params(sp))
    compare_results(res[k], m0.map_batch(seeds=sd, want_hits=True, packed=pk, with_xa=True), label_a="concurrent", label_b="alone")
for h in handles[::-1]:
    h.close()
print("concurrent ok")
"""


@pytest.mark.parametrize("env", [{}, {"MAPAD_FORCE_WIDE": "1", "MAPAD_GROUP": "32"}], ids=["narrow", "wide-G32"])
def test_concurrent_handles_dry_pool(env):
    """Six handles (clones sharing one index blob and the device-wide chunk pool) map six heavy chunks at once from six
    threads, with a pool so small that it runs dry across launches: reads are handed back and re-run.  Every chunk must
    equal the oracle and the same chunk mapped alone."""
    out = _run_child(CHILD_CONCURRENT, env)
    print(out)
    assert "concurrent ok" in out, out

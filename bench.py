#!/usr/bin/env python3
"""bench.py — reads mapped / second of the B200 hot path (BASELINE.json metric), per the driver contract.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload cfg4|cfg3|cfg2|cfg1]
                    [--batch READS_PER_STEP] [--scaling weak|strong] [--dump-outputs DIR]

Default workload: BASELINE cfg4, the metric's own configuration (3.1 Gbp hg19-scale synthetic reference, 25-100 bp
single-stranded damaged reads, -p 0.03); `--workload cfg3` etc. give the other BASELINE shapes.
One "step" = one pass of the hot path (penalties + D array + search + epilogue) over one chunk of `--batch` simulated reads
(the reference's --batch_size is 250 000, src/main.rs:229; hg19-scale steps use smaller chunks so that the driver's
K + W steps fit its time limit — stated in config.workload).  Every step uses a different chunk.
  One timed pass gives both numbers (the hg19-scale run is bounded below by its 1e7-frame reads, ~2 min per pass, so the
  pass is not repeated): phase U stages every chunk through the public C-ABI call (host buffers -> HBM), phase R runs them.
  value  reads/s with the chunks already resident in HBM: K chunks / phase R (device time from CUDA events on the library's
         streams, first launch to last completion, max over ranks), D2H of the records included
  e2e    reads/s through the public C-ABI calls with host buffers: K chunks / (phase U + phase R), i.e. H2D + kernels +
         D2H inside the timed region (host wall clock)
  parity the records of one timed end-to-end chunk are compared with the CPU oracle's on the same reads (bit-exact on
         position, strand, CIGAR, MD, NM, MAPQ, X0/X1/XS, best-hit interval, scores and the work counters);
         any mismatch makes the run exit non-zero
  --dump-outputs DIR  writes the records of the last timed chunk (rank 0) as DIR/<name>.npy, so that two builds can be
         compared output for output on identical inputs (see dump_outputs)
Multi-GPU: one process per GPU (torchrun), index built once on rank 0 and broadcast with NCCL, reads sharded per rank
(weak scaling: K chunks per rank; --scaling strong: the same K chunks split over the ranks), no data-path collective.
`--impl reference` times the CPU restatement of mapAD 0.45.0 (oracle/, all host threads): the reference itself is Rust and
cannot be built in this image (no rustc/cargo).  That arm obtains its index arrays from a helper process
(tools/index_arrays.py) and loads only oracle/libmapad_oracle.so itself.
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "32")  # one hardware queue per in-flight handle (see mapad_b200/__init__.py)

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from mapad_b200 import abi, workloads  # noqa: E402

# reads per step (chunk) and size of the CPU sample, per workload
DEFAULT_BATCH = {"cfg1": 100_000, "cfg2": 250_000, "cfg3": 250_000, "cfg4": 25_000}
DEFAULT_CPU_SAMPLE = {"cfg1": 20_000, "cfg2": 20_000, "cfg3": 20_000, "cfg4": 1_500}
DEFAULT_REF_SAMPLE = {"cfg1": 20_000, "cfg2": 20_000, "cfg3": 20_000, "cfg4": 250}
PARAMS_TEXT = "-p 0.03 -f 0.5 -t 0.5 -d 0.02 -s 1.0 -D 0.02 -i 0.001 -x 0.5 --gap_dist_ends 5 --max_num_gaps_open 2"
CPU_LABEL = "C++ restatement of mapAD 0.45.0 (reference binary not buildable here: no Rust toolchain)"


def cli_spec(library):
    from mapad_b200 import specs
    return specs.cli_spec(library)


class ClockSampler:
    QUERY = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.rows = []
        self.proc = None
        self.gpu = gpu_index
        self.thread = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.QUERY, "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None
            return

        def pump():
            for line in self.proc.stdout:
                self.rows.append(line.strip())
        self.thread = threading.Thread(target=pump, daemon=True)
        self.thread.start()

    def stop(self):
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=5)
            except Exception:
                self.proc.kill()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons), "samples": len(sm)}


def chunk_seed(cfg, chunk_id):
    return cfg["seed"] * 1000 + chunk_id


def simulate_chunks(cfg, genome, batch, chunk_ids):
    """At most MAPAD_BENCH_DISTINCT_CHUNKS different chunks are simulated (seconds of numpy each); longer runs cycle."""
    distinct = max(1, int(os.environ.get("MAPAD_BENCH_DISTINCT_CHUNKS", "12")))
    cache = {}
    out = {}
    for cid in chunk_ids:
        key = cid % distinct if len(chunk_ids) > distinct else cid
        if key not in cache:
            cache[key] = workloads.simulate_batch(genome, batch, cfg["len_range"], seed=chunk_seed(cfg, key), library=cfg["library"])
        out[cid] = cache[key]
    return out, len(cache)


def build_index(cfg):
    from mapad_b200 import api
    genome = workloads.random_genome_array(cfg["genome_bp"], seed=42)
    # references beyond ~0.5 Gbp are suffix-sorted on the GPU (mapad_index_build_on_device); smaller ones on the host (SA-IS)
    dev = int(os.environ.get("LOCAL_RANK", "0")) if cfg["genome_bp"] > 500_000_000 else None
    cache = os.environ.get("MAPAD_BENCH_INDEX_CACHE")  # tuning runs: keep the index files between invocations
    if cache and os.path.exists(cache + ".tbw"):
        index = api.Index.load(cache)
    else:
        index = api.Index.build(workloads.split_contigs(genome, cfg["n_contigs"]), seed=1234, device=dev)
        if cache:
            index.save(cache)
    return genome, index


def oracle_index_from_arrays(a):
    from oracle import oracle as ora
    return ora.OracleIndex.from_arrays(a["bwt"], a["sa_sample"], a["sa_rate"], a["extra_rows"], a["contigs"], a["orig_pos"], a["orig_sym"])


def run_cpu(oix, spec, packed, n_sample, threads):
    """Times the oracle on the first n_sample reads of a chunk; returns (reads/s, seconds, n, oracle BatchResult)."""
    from helpers import oracle_params
    from oracle import oracle as ora
    seq, qual, off = packed
    n = min(n_sample, len(off) - 1)
    sub = (seq[: int(off[n])], qual[: int(off[n])], off[: n + 1])
    p = oracle_params(spec)
    t0 = time.time()
    res = ora.map_batch(oix, p, None, None, seeds=np.arange(n, dtype=np.uint32), n_threads=threads, want_hits=False, packed=sub)
    dt = time.time() - t0
    return n / dt, dt, n, res


DUMP_MAX_READS = 100_000
DUMP_MAX_BYTES = 64 << 20


def _gather(pool, offs, lens):
    """pool[offs[0]:offs[0]+lens[0]], pool[offs[1]:...], ... concatenated"""
    offs, lens = offs.astype(np.int64).ravel(), lens.astype(np.int64).ravel()
    starts = np.cumsum(lens) - lens
    return pool[np.repeat(offs - starts, lens) + np.arange(int(lens.sum()))]


def dump_outputs(res, out_dir):
    """Writes what a caller of the timed path receives for one chunk as out_dir/<name>.npy: every per-read record field
    (integers as float64, f32 scores as float32; alternative hits as alt_<field>, shape (n, 2)) and, per read in read
    order, the CIGAR words and MD text of its primary alignment followed by those of its alternative hits (float32;
    the *_len fields split them).  Pool offsets are left out: they only say where the library put the strings.  Of
    flags only bit 0 (search limit hit) is kept: bit 1 (went through the retry lane) depends on what else was in flight.
    Chunks of more than DUMP_MAX_READS reads are sampled with a fixed seed; read_index holds the sampled reads."""
    rec = res.records
    n = len(rec)
    idx = np.arange(n) if n <= DUMP_MAX_READS else np.sort(np.random.default_rng(0).choice(n, DUMP_MAX_READS, replace=False))
    rec = rec[idx]
    alts = rec["alts"]
    out = {"read_index": idx.astype(np.float64)}
    for table, prefix in ((rec, ""), (alts, "alt_")):
        for f in table.dtype.names:
            if f in ("alts", "cigar_off", "md_off", "hit_off"):
                continue
            v = table[f] & 1 if f == "flags" else table[f]
            out[prefix + f] = v.astype(np.float32 if v.dtype == np.float32 else np.float64)
    for name, pool, off, ln in (("cigar", res.cigar, "cigar_off", "cigar_len"), ("md", np.frombuffer(res.text, np.uint8), "md_off", "md_len")):
        offs = np.concatenate([rec[off][:, None], alts[off]], axis=1)
        lens = np.concatenate([rec[ln][:, None], alts[ln]], axis=1)
        out[name] = _gather(pool, offs, lens).astype(np.float32)
    total = sum(a.nbytes for a in out.values())
    if total > DUMP_MAX_BYTES:
        raise SystemExit("bench.py: --dump-outputs would write %d bytes (limit %d)" % (total, DUMP_MAX_BYTES))
    os.makedirs(out_dir, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


# ---------------------------------------------------------------------------------------------------------------------
# reference arm (CPU restatement; this process never loads the product library)
# ---------------------------------------------------------------------------------------------------------------------
def reference_arm(args, cfg, spec, workload_name, threads):
    n_steps = args.steps + args.warmup
    sample = max(50, min(args.batch, int(os.environ.get("MAPAD_REF_SAMPLE", str(DEFAULT_REF_SAMPLE[args.workload])))))
    t0 = time.time()
    genome = workloads.random_genome_array(cfg["genome_bp"], seed=42)
    if cfg["genome_bp"] <= 5_000_000:
        # small references: the oracle's own indexer (cross-checked against the product's on 5 Mbp, tests/test_emulated_kernels.py)
        from oracle import oracle as ora
        oix = ora.OracleIndex.build(workloads.split_contigs(genome, cfg["n_contigs"]))
        index_txt = "built by the oracle's own indexer"
    else:
        # the oracle's suffix sorter does not scale to these texts: a helper PROCESS builds the arrays with the product's indexer
        # (host SA-IS, device suffix sorter beyond 0.5 Gbp); this process itself only loads oracle/libmapad_oracle.so
        tmp = tempfile.mkdtemp(prefix="mapad_ref_index_")
        subprocess.check_call([sys.executable, os.path.join(ROOT, "tools", "index_arrays.py"), args.workload, tmp])
        meta = json.load(open(os.path.join(tmp, "meta.json")))
        a = dict(sa_rate=meta["sa_rate"], contigs=[tuple(c) for c in meta["contigs"]])
        for k in ("bwt", "sa_sample", "extra_rows", "orig_pos", "orig_sym"):
            a[k] = np.load(os.path.join(tmp, k + ".npy"), mmap_mode="r")
        oix = oracle_index_from_arrays(a)
        del a
        for f in os.listdir(tmp):
            os.unlink(os.path.join(tmp, f))
        os.rmdir(tmp)
        index_txt = "arrays built by a helper process (tools/index_arrays.py)"
    t_index = time.time() - t0
    chunks, _ = simulate_chunks(cfg, genome, sample, list(range(n_steps)))
    times, n_done = [], 0
    for b in range(n_steps):
        rps, dt, n, _ = run_cpu(oix, spec, chunks[b], sample, threads)
        if b >= args.warmup:
            times.append(dt); n_done += n
    value = n_done / sum(times)
    sample_txt = "%s, %d reads per step (bounded sample of the %d-read chunk), %d threads" % (CPU_LABEL, sample, args.batch, threads)
    print(json.dumps({
        "impl": "reference", "metric": "reads mapped/sec", "value": value, "unit": "reads/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * sum(times) / len(times), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "u64 intervals + f32 scores", "data": "synthetic",
        "config": {"workload": workload_name, "params": PARAMS_TEXT, "sample": "%d reads per step" % sample,
                   "index": "%s, %.1f s" % (index_txt, t_index)},
        "cpu_baseline": {"value": value, "unit": "reads/s", "cores": threads, "kind": "port", "sample": sample_txt},
        "e2e": {"value": value, "unit": "reads/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }))


# ---------------------------------------------------------------------------------------------------------------------
# our arm (CUDA)
# ---------------------------------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours")
    ap.add_argument("--workload", default=os.environ.get("MAPAD_BENCH_WORKLOAD", "cfg4"))
    ap.add_argument("--batch", type=int, default=0)
    ap.add_argument("--cpu-sample", type=int, default=0)
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the records of the last timed step as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    cfg = dict(workloads.CONFIGS[args.workload])
    if not args.batch:
        args.batch = int(os.environ.get("MAPAD_BENCH_BATCH", str(DEFAULT_BATCH[args.workload])))
    if not args.cpu_sample:
        args.cpu_sample = DEFAULT_CPU_SAMPLE[args.workload]
    spec = cli_spec(cfg["library"])
    threads = os.cpu_count() or 1
    workload_name = "%s: %s; chunk of %d reads per step" % (args.workload, cfg["desc"], args.batch)

    if args.impl == "reference":
        if rank == 0:
            reference_arm(args, cfg, spec, workload_name, threads)
        return

    import torch
    import torch.distributed as dist
    from compare import mismatching_reads  # pure numpy record comparison (tests/compare.py)
    from mapad_b200 import api
    from mapad_b200.specs import product_params  # oracle-free: the oracle is only loaded by the CPU legs below (run_cpu)

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the product path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    params = product_params(spec)
    strong = args.scaling == "strong" and world > 1
    if strong and args.steps % world:
        raise SystemExit("--scaling strong needs --steps divisible by the number of GPUs")
    # chunk ids: warm-up chunks are private to the rank; timed chunks are K per rank (weak) or the same K split over the ranks (strong)
    warm_ids = [10_000 + rank * 100 + i for i in range(args.warmup)]
    if strong:
        timed_ids = [20_000 + i for i in range(args.steps)][rank::world]
    else:
        timed_ids = [20_000 + rank * 1000 + i for i in range(args.steps)]
    t0 = time.time()
    index = None
    if rank == 0:
        genome, index = build_index(cfg)
    else:
        genome = workloads.random_genome_array(cfg["genome_bp"], seed=42)
    t_index = time.time() - t0
    chunks, n_distinct = simulate_chunks(cfg, genome, args.batch, warm_ids + timed_ids)
    del genome
    t0 = time.time()
    free_b0, _ = torch.cuda.mem_get_info()
    inflight = max(1, min(len(timed_ids), int(os.environ.get("MAPAD_BENCH_INFLIGHT", "32"))))
    # search workspace: ONE chunk pool per GPU shared by all handles (75 % of the memory left after the index, sized by the
    # library when the first handle is created; MAPAD_WS_BYTES overrides)
    api.plan_handles(local_rank, inflight + 1)
    if world == 1:
        mapper = api.Mapper(index, params, device=local_rank)
        meta, blob_ptr, nbytes = mapper.export_index()
        keep_blob = mapper
    else:
        # index replicated per GPU: built + re-laid-out on rank 0, ONE NCCL broadcast of the device blob over NVLink
        if rank == 0:
            mapper0 = api.Mapper(index, params, device=local_rank)
            meta, _, nbytes = mapper0.export_index()
            hdr = [meta, nbytes]
        else:
            hdr = [None, None]
        dist.broadcast_object_list(hdr, src=0)
        meta, nbytes = hdr
        blob = torch.empty(nbytes, dtype=torch.uint8, device="cuda")
        if rank == 0:
            mapper0.copy_index_to(blob.data_ptr(), nbytes)
            torch.cuda.synchronize()
            mapper0.close()
        dist.broadcast(blob, src=0)
        torch.cuda.synchronize()
        blob_ptr, keep_blob = blob.data_ptr(), blob
    blob_bytes = nbytes
    t_upload = time.time() - t0
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    reads_structs = {cid: api.make_reads(c[0], c[1], c[2], np.arange(len(c[2]) - 1, dtype=np.uint32)) for cid, c in chunks.items()}

    # Chunks are pipelined: `inflight` handles share the index blob, each owns a stream and a workspace, so the straggler reads
    # of one chunk (per-read work is heavy-tailed over four orders of magnitude) overlap with the next chunks.  The timed region
    # spans from the first launch to the completion of the last chunk.
    mappers = [api.Mapper.from_device_blob(meta, blob_ptr, nbytes, index, params, device=local_rank) for _ in range(inflight)]
    streams = [torch.cuda.Stream() for _ in mappers]
    for mp, st in zip(mappers, streams):
        mp.set_stream(st.cuda_stream)
    keep_result = {}

    def run_pipelined(chunk_ids, resident, keep=()):
        """Maps the given chunks, round-robin over the handles, one host thread per handle.
        resident=True (one chunk per handle): phase U stages every chunk in HBM through the C ABI (timed on the host clock),
        phase R runs them from HBM (timed with CUDA events and on the host clock); otherwise a single phase maps from host buffers.
        keep: chunk ids whose full result (records + CIGAR/MD pools) is copied for the parity check and --dump-outputs.
        Returns (device seconds of phase R from first start to last end event, per-chunk stats, wall seconds of R, wall seconds of U)."""
        per = [[] for _ in mappers]
        for k, cid in enumerate(chunk_ids):
            per[k % len(mappers)].append(cid)
        flush.fill_(1)
        barrier()
        errors = []
        wall_u = 0.0
        if resident:
            assert all(len(p) <= 1 for p in per), "resident timing needs one handle per chunk"

            def stage(h):
                try:
                    torch.cuda.set_device(local_rank)
                    for cid in per[h]:
                        mappers[h].map_raw(reads_structs[cid][0], abi.BATCH_UPLOAD_ONLY)
                except Exception as e:  # noqa: BLE001
                    errors.append(e)
            u0 = time.perf_counter()
            ths = [threading.Thread(target=stage, args=(h,)) for h in range(len(mappers)) if per[h]]
            for t_ in ths:
                t_.start()
            for t_ in ths:
                t_.join()
            torch.cuda.synchronize()
            wall_u = time.perf_counter() - u0
            if errors:
                raise errors[0]
            barrier()
        ev0 = [torch.cuda.Event(enable_timing=True) for _ in mappers]
        ev1 = [torch.cuda.Event(enable_timing=True) for _ in mappers]
        results = {}

        def work(h):
            try:
                torch.cuda.set_device(local_rank)
                ev0[h].record(streams[h])
                for cid in per[h]:
                    if resident:
                        res = mappers[h].map_raw(None, abi.BATCH_RESIDENT)
                    else:
                        res = mappers[h].map_raw(reads_structs[cid][0], 0)
                    recs = abi._as_array(res.records, res.n_reads, abi.RECORD_DTYPE)
                    results[cid] = dict(recs=recs, ms_search=res.ms_search, ms_prologue=res.ms_prologue, ms_epilogue=res.ms_epilogue,
                                        ms_total=res.ms_total, launches=int(res.gpu_launches), n_cigar=int(res.n_cigar), n_text=int(res.n_text))
                    if cid in keep:
                        keep_result[cid] = abi.BatchResult(res)
                ev1[h].record(streams[h])
            except Exception as e:  # noqa: BLE001
                errors.append(e)

        w0 = time.perf_counter()
        threads_ = [threading.Thread(target=work, args=(h,)) for h in range(len(mappers)) if per[h]]
        for t_ in threads_:
            t_.start()
        for t_ in threads_:
            t_.join()
        torch.cuda.synchronize()
        wall = time.perf_counter() - w0
        if errors:
            raise errors[0]
        used = [h for h in range(len(mappers)) if per[h]]
        first = min(used, key=lambda h: ev0[used[0]].elapsed_time(ev0[h]))
        done_ms = sorted(ev0[first].elapsed_time(ev1[h]) for h in used)
        run_pipelined.done_s = [round(x * 1e-3, 2) for x in done_ms]  # per-handle completion times: shows the straggler tail
        return done_ms[-1] * 1e-3, results, wall, wall_u

    # ---- warm-up (untimed): W real steps, each on its own handle (kernels loaded, pool and buffers of those handles allocated;
    #      the other handles allocate their batch buffers — a few cudaMallocs each — inside the timed region) ----
    for k0 in range(0, len(warm_ids), len(mappers)):
        run_pipelined(warm_ids[k0:k0 + len(mappers)], resident=False)
    barrier()
    sampler = ClockSampler(local_rank)
    sampler.start()
    # ---- timed pass: phase U (host buffers -> HBM through the C ABI), phase R (run from HBM) ----
    resident_ok = len(timed_ids) <= len(mappers)
    keep = ({timed_ids[0], timed_ids[-1]} if args.dump_outputs else {timed_ids[0]}) if rank == 0 else ()
    dev_s, results, wall_r, wall_u = run_pipelined(timed_ids, resident=resident_ok, keep=keep)
    dev_ms = dev_s * 1e3
    wall_resident = wall_r
    e2e_wall = wall_u + wall_r
    done_resident = list(run_pipelined.done_s)
    results_e2e = results
    search_ms = sum(r["ms_search"] for r in results.values())
    launches = sum(r["launches"] for r in results.values())
    stats = dict(P=0, E=0, W=0, search_bytes=0, total_bytes=0, mapped=0, deferred=0, limit=0, max_frames=0)
    for cid, r in results.items():
        ab = workloads.algorithmic_bytes(r["recs"], int(chunks[cid][2][-1]))
        for k in ("P", "E", "W", "search_bytes", "total_bytes"):
            stats[k] += ab[k]
        stats["mapped"] += int(r["recs"]["mapped"].sum())
        stats["deferred"] += int(((r["recs"]["flags"] & 2) != 0).sum())
        stats["limit"] += int(((r["recs"]["flags"] & 1) != 0).sum())
        stats["max_frames"] = max(stats["max_frames"], int(r["recs"]["frames_popped"].max()))
    barrier()
    tb = int(chunks[timed_ids[0]][2][-1])
    h2d = 2 * tb + 8 * (args.batch + 1) + 4 * args.batch
    r0 = results_e2e[timed_ids[0]]
    d2h = args.batch * ctypes.sizeof(abi.Record) + 4 * r0["n_cigar"] + r0["n_text"]
    barrier()
    clocks = sampler.stop()

    n_local = len(timed_ids)
    t = torch.tensor([dev_ms, e2e_wall, search_ms], dtype=torch.float64, device="cuda")
    tot = torch.tensor([stats["P"], stats["E"], stats["W"], stats["search_bytes"], stats["total_bytes"], stats["mapped"], launches,
                        stats["deferred"], stats["limit"], n_local], dtype=torch.float64, device="cuda")
    mx = torch.tensor([stats["max_frames"]], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(tot, op=dist.ReduceOp.SUM)
        dist.all_reduce(mx, op=dist.ReduceOp.MAX)
    dev_ms_max, e2e_s_max, search_ms_max = [float(x) for x in t.tolist()]
    P, E, W, search_bytes, total_bytes, mapped, launches_all, deferred, limit_reads, n_chunks_all = [float(x) for x in tot.tolist()]
    total_reads = args.batch * n_chunks_all
    value = total_reads / (dev_ms_max * 1e-3)
    e2e_value = total_reads / e2e_s_max

    rc = 0
    if rank == 0:
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
        peak_src = "MEASURED_PEAKS.json hbm_gbs (measured)" if "hbm_gbs" in peaks else "fallback 6650 GB/s (B200_PROFILING.md)"
        # live denominator for random sector traffic: 64 B gathers over a table of the index size
        try:
            gather = api.gather_peak(local_rank, max(blob_bytes, 64 << 20), 64, 1 << 27)
            gather32 = api.gather_peak(local_rank, max(blob_bytes, 64 << 20), 32, 1 << 27)
        except Exception:
            gather = gather32 = None
        traffic, traffic_src = None, None
        try:  # DRAM bytes per popped frame of the search kernel from the committed `ncu` capture (profiles/)
            tj = json.load(open(os.path.join(ROOT, "profiles", "r2_traffic.json")))
            per_frame = tj.get("by_workload", {}).get(args.workload)
            if per_frame is not None:  # only a capture of THIS workload's index / heap regime is carried over
                traffic = per_frame * P / n_chunks_all
                traffic_src = tj.get("source_" + args.workload, tj["source"])
        except Exception:
            pass
        # the search launches of different chunks overlap on the device, so the dominant kernel's achieved rate is taken over
        # the whole timed region (it accounts for >98 % of it): algorithmic bytes of all its launches / elapsed device time
        achieved = (search_bytes / world) / (dev_ms_max * 1e-3) / 1e9
        out = {
            "metric": "reads mapped/sec", "value": value, "unit": "reads/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": dev_ms_max / max(1, n_local), "higher_is_better": True, "scaling": args.scaling if world > 1 else "weak", "vs_baseline": None,
            "dtype": "u64 intervals + f32 scores", "data": "synthetic",
            "config": {"workload": workload_name,
                       "l2": "256 MiB memset before each timed region; %d distinct chunks; per-read search state (GBs) far exceeds L2" % n_distinct,
                       "params": PARAMS_TEXT,
                       "index_bytes_hbm": blob_bytes, "index_build_s": round(t_index, 2), "index_upload_s": round(t_upload, 3),
                       "mapped_fraction": mapped / total_reads, "frames_popped_per_read": P / total_reads,
                       "d_ext_steps_per_read": E / total_reads, "lf_steps_per_read": W / total_reads, "max_frames_one_read": mx.item(),
                       "reads_at_search_limit": limit_reads, "retry_launch_reads": deferred, "wall_s_resident_loop": round(wall_resident, 3),
                       "chunks_in_flight": len(mappers), "handle_done_s": done_resident, "inputs_resident_for_value": bool(resident_ok),
                       "timed_pass": "phase U (stage K chunks through the C ABI, %.3f s) + phase R (run from HBM, %.3f s); value = K chunks / R (CUDA events), e2e = K chunks / (U + R) (host clock)" % (wall_u, wall_r),
                       "frames_per_s": P / (dev_ms_max * 1e-3) / world},
            "e2e": {"value": e2e_value, "unit": "reads/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h},
            "gpu_launches": int(launches_all),
            "clocks": clocks,
            "roofline": {"bound": "hbm", "kernel": "k_search_group (>98 % of device time)", "achieved": achieved,
                         "peak": hbm_peak, "unit": "GB/s", "frac": achieved / hbm_peak,
                         "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src,
                         "algorithmic_bytes_per_launch": search_bytes / n_chunks_all,
                         "kernel_ms_per_launch_wall": search_ms_max / max(1, n_local),
                         "kernel_ms_note": "per-chunk wall of the search launch; %d launches overlap on the device" % len(mappers),
                         "random_gather_peak_64B_gbs": gather, "random_gather_peak_32B_gbs": gather32,
                         "frac_of_gather_peak": (achieved / gather) if gather else None,
                         "path_algorithmic_gbs": (total_bytes / world) / (dev_ms_max * 1e-3) / 1e9},
        }
        if not args.no_cpu_baseline:
            # CPU restatement on a bounded sample of a timed chunk; the same reads' GPU records (end-to-end pass) are checked against it
            oix = oracle_index_from_arrays(index.arrays())
            cid = timed_ids[0]
            rps, dt, n, want = run_cpu(oix, spec, chunks[cid], args.cpu_sample, threads)
            del oix
            if world == 1:
                out["cpu_baseline"] = {"value": rps, "unit": "reads/s", "cores": threads, "kind": "port",
                                       "sample": "first %d reads of a timed chunk, %.1f s, %s" % (n, dt, CPU_LABEL)}
            got = keep_result.get(cid)
            if got is not None:
                bad = mismatching_reads(want, got, n=n)
                out["parity"] = {"reads_checked": n, "mismatches": len(bad), "against": "oracle (CPU restatement) on the same reads, records of the timed end-to-end pass",
                                 "first": bad[0][1] if bad else None}
                if bad:
                    rc = 3
        if args.dump_outputs:
            dump_outputs(keep_result[timed_ids[-1]], args.dump_outputs)
        print(json.dumps(out))
    for mp in mappers:
        mp.close()
    if world == 1:
        keep_blob.close()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    if rc:
        sys.exit(rc)


if __name__ == "__main__":
    main()

#!/usr/bin/env python3
"""Checks a benchmark index against its genome with the oracle's independent verifier (LF walks from every known row,
oracle/oracle_capi.cpp: ora_verify_index).

    python tools/verify_index.py [--workload cfg4] [--index PREFIX] [--threads T]

Without --index it builds the workload's index the way bench.py does (genome seed 42, contig split, replacement seed 1234,
the device suffix sorter above 0.5 Gbp).  With --index it loads the index files at PREFIX instead, e.g. a
MAPAD_BENCH_INDEX_CACHE that bench.py reuses without checking.  Either way the text is regenerated from the workload's
genome.  Prints rows, seconds and peak RSS as one JSON line; exits 1 if the index is not the one of the genome."""
import argparse
import json
import os
import resource
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from mapad_b200 import api, workloads  # noqa: E402
from oracle import oracle as ora  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workload", default="cfg4", choices=sorted(workloads.CONFIGS))
    ap.add_argument("--index", metavar="PREFIX", help="load the index files <PREFIX>.tbw ... instead of building the index")
    ap.add_argument("--threads", type=int, default=os.cpu_count() or 1)
    args = ap.parse_args()
    cfg = workloads.CONFIGS[args.workload]
    out = dict(workload=args.workload, genome_bp=cfg["genome_bp"], threads=args.threads)
    t0 = time.time()
    genome = workloads.random_genome_array(cfg["genome_bp"], seed=42)
    if args.index:
        index = api.Index.load(args.index)
        out["index"] = args.index
    else:
        dev = 0 if cfg["genome_bp"] > 500_000_000 else None
        index = api.Index.build(workloads.split_contigs(genome, cfg["n_contigs"]), seed=1234, device=dev)
        out["sorter"] = "device" if dev is not None else "host SA-IS"
    out["index_s"] = round(time.time() - t0, 1)
    a = index.arrays()
    del index
    t0 = time.time()
    text = ora.text_ranks([genome])
    del genome
    out["text_s"] = round(time.time() - t0, 1)
    out["rows"] = a["n"]
    t0 = time.time()
    try:
        ora.verify_index(text, a, n_threads=args.threads)
        out["result"] = "ok"
    except ora.IndexMismatch as e:
        out["result"] = "mismatch: %s" % e
    out["verify_s"] = round(time.time() - t0, 1)
    out["peak_rss_gb"] = round(resource.getrusage(resource.RUSAGE_SELF).ru_maxrss / 2**20, 1)
    print(json.dumps(out))
    return 0 if out["result"] == "ok" else 1


if __name__ == "__main__":
    sys.exit(main())

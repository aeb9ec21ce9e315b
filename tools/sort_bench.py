"""Unsorted versus coordinate-sorted, indexed BAM end to end on bench.py's default workload (c3: synthetic 3.1 Gbp
reference, 40 000-pair buckets).

Qualities are redrawn from four binned values as in tools/bam_bench.py.  One session runs the same K buckets through
emab_align_buckets, alternating `-O bam` (every call compresses its own members) and `-O bam -S` (calls hold raw records;
emab_session_finish sorts, compresses and indexes them once), three repetitions each.  Prints one JSON line: pairs/s of both,
the sorted run's finish phase split into device sort, host gather, compression and index build (medians over the
repetitions), the output sizes, and the card's name and power limit read in the same run.

--spill-bytes N adds a third arm, `-O bam -S -T` (bam_sorted_spill): the sorted run with a host-memory budget of N bytes,
spilled to files under --spill-dir (the node's local temporary directory by default) and merged at finish.  It reports the
align calls' spill_files, spill_bytes and spill_ms beside the finish split.

    python tools/sort_bench.py [--steps 12] [--workers 8] [--spill-bytes N]
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

import bench  # noqa: E402
from bam_bench import binned  # noqa: E402


def med(xs):
    return sorted(xs)[len(xs) // 2]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workload", default="c3", choices=sorted(bench.WORKLOADS))
    ap.add_argument("--steps", type=int, default=12)
    ap.add_argument("--workers", type=int, default=8)
    ap.add_argument("--threads", type=int, default=0, help="host threads (0 = all cores)")
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--data-dir", default=os.environ.get("EMAB_DATA", "/tmp/emab_data"))
    ap.add_argument("--spill-bytes", type=int, default=0, help="host-memory budget of the spilling arm (0: no such arm)")
    ap.add_argument("--spill-dir", default=tempfile.gettempdir())
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("sort_bench.py needs a CUDA device")
    smi = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
    n_buckets = bench.WORKLOADS[args.workload][1]
    bench.prepare_buckets(args.workload, args.data_dir, min(args.steps, n_buckets))
    fa, buckets, pairs = bench.prepare(args.workload, args.data_dir, min(args.steps, n_buckets))
    import ema_b200
    threads = args.threads or os.cpu_count()
    sess = ema_b200.Session(fa, "10x", threads=threads, output="bam")
    batch = [ema_b200.PinnedText(binned(open(buckets[i % len(buckets)], "rb").read(), 1000 + i)) for i in range(args.steps)]
    sess.set_workers(args.workers)
    hdr = sess.header(["ema", "align", "-O", "bam"])

    def unsorted():
        sess.set_sort(False)
        return sum(sess.align_buckets(batch, keep_text=False))

    def srt():
        sess.set_sort(True)
        sess.header(["ema", "align", "-O", "bam", "-S"])   # the index counts the header's bytes
        sess.align_buckets(batch, keep_text=False)
        body, bai = sess.finish()
        return len(body), len(bai), sess.stats

    spill_dir = tempfile.mkdtemp(prefix="emab_spill_", dir=args.spill_dir)

    def spilled():
        sess.set_spill(os.path.join(spill_dir, "run"))
        sess.set_sort(True, args.spill_bytes)
        sess.header(["ema", "align", "-O", "bam", "-S", "-T"])
        sess.align_buckets(batch, keep_text=False)
        calls = sess.stats
        body, bai = sess.finish()
        sess.set_spill(None)
        return len(body), len(bai), calls, sess.stats

    unsorted()   # warm every worker and shape of both modes
    srt()
    walls = {"bam": [], "bam_sorted": []}
    split = {k: [] for k in ("sort_ms", "gather_ms", "compress_ms", "index_ms", "finish_ms")}
    sizes = {}
    spill = {k: [] for k in ("spill_files", "spill_bytes", "spill_ms", "sort_ms", "gather_ms", "compress_ms", "index_ms", "finish_ms")}
    if args.spill_bytes:
        spilled()
        walls["bam_sorted_spill"] = []
    for _ in range(args.repeats):
        t0 = time.time()
        sizes["bam"] = unsorted()
        walls["bam"].append(time.time() - t0)
        t0 = time.time()
        n_body, n_bai, st = srt()
        walls["bam_sorted"].append(time.time() - t0)
        sizes["bam_sorted"], sizes["bai"] = n_body, n_bai
        for k in ("sort_ms", "gather_ms", "compress_ms", "index_ms"):
            split[k].append(getattr(st, k))
        split["finish_ms"].append(st.total_ms)
        if args.spill_bytes:
            t0 = time.time()
            n_body, _, calls, st = spilled()
            walls["bam_sorted_spill"].append(time.time() - t0)
            sizes["spill_body"] = n_body
            for k in ("spill_files", "spill_bytes", "spill_ms"):
                spill[k].append(getattr(calls, k))
            for k in ("sort_ms", "gather_ms", "compress_ms", "index_ms"):
                spill[k].append(getattr(st, k))
            spill["finish_ms"].append(st.total_ms)
    os.rmdir(spill_dir)
    rate = {f: args.steps * pairs / med(w) for f, w in walls.items()}
    extra = {}
    if args.spill_bytes:
        extra = {"spill_budget_bytes": args.spill_bytes,
                 "spill_median": {k: round(med(v), 2) for k, v in spill.items()}, "spill_body": sizes["spill_body"]}
    print(json.dumps({
        "workload": args.workload, "steps": args.steps, "workers": args.workers, "threads": threads, "pairs_per_bucket": pairs,
        "qualities": "redrawn from F : , # (seeded)",
        "pairs_per_s": {f: round(v) for f, v in rate.items()}, "sorted_over_unsorted_rate": round(rate["bam_sorted"] / rate["bam"], 3),
        "wall_s": walls,
        "finish_ms_median": {k: round(med(v), 2) for k, v in split.items()},
        "finish_ms_per_bucket": {k: round(med(v) / args.steps, 2) for k, v in split.items()},
        "bytes": {"header": len(hdr), "bam_body": sizes["bam"], "sorted_body": sizes["bam_sorted"], "bai": sizes["bai"]},
        "gpu": smi, **extra,
    }))


if __name__ == "__main__":
    main()

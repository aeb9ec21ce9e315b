"""`ema-b200 merge` (emab_bam_merge_files) and the device BGZF inflater (emab_bgzf_inflate) on bench.py's default workload
(c3: synthetic 3.1 Gbp reference, 40 000-pair buckets).

Qualities are redrawn from four binned values as in tools/bam_bench.py.  One session aligns K buckets with `-O bam -S` as
four sorted runs of K / 4 buckets each, written to four BAM files (header, body, EOF block) in a temporary directory, and
then all K buckets as one sorted run, whose finish phase (emab_session_finish: device sort, host gather, compression,
index) is the comparison.  Then, in the same process:
  inflate   the four files' bytes back to back through emab_bgzf_inflate; the rate is inflated bytes over the kernel's
            time from CUDA events (emab_last_kernel_ms), median of the repetitions
  merge     emab_bam_merge_files over the four files with an index: wall time, input MB/s, records/s and the ms[] split
            (inflate, rows, order, gather, compress, index), median of the repetitions
Prints one JSON line with the card's name and power limit read in the same run.

    python tools/merge_bench.py [--steps 12] [--workers 8]
"""
import argparse
import json
import os
import shutil
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
    ap.add_argument("--inputs", type=int, default=4)
    ap.add_argument("--workers", type=int, default=8)
    ap.add_argument("--threads", type=int, default=0, help="host threads (0 = all cores)")
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--data-dir", default=os.environ.get("EMAB_DATA", "/tmp/emab_data"))
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("merge_bench.py needs a CUDA device")
    smi = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
    n_buckets = bench.WORKLOADS[args.workload][1]
    bench.prepare_buckets(args.workload, args.data_dir, min(args.steps, n_buckets))
    fa, buckets, pairs = bench.prepare(args.workload, args.data_dir, min(args.steps, n_buckets))
    import ema_b200
    threads = args.threads or os.cpu_count()
    sess = ema_b200.Session(fa, "10x", threads=threads, output="bam")
    batch = [ema_b200.PinnedText(binned(open(buckets[i % len(buckets)], "rb").read(), 1000 + i)) for i in range(args.steps)]
    sess.set_workers(args.workers)
    eof = ema_b200.bgzf_eof()

    def sorted_run(part):
        sess.set_sort(True)
        hdr = sess.header(["ema", "align", "-O", "bam", "-S"])
        sess.align_buckets(part, keep_text=False)
        body, bai = sess.finish()
        return hdr + body + eof, sess.stats

    tmp = tempfile.mkdtemp(prefix="emab_merge_")
    try:
        paths = []
        per = (args.steps + args.inputs - 1) // args.inputs
        for k in range(args.inputs):
            data, _ = sorted_run(batch[k * per:(k + 1) * per])
            p = os.path.join(tmp, f"in{k}.bam")
            open(p, "wb").write(data)
            paths.append(p)
        finish = {k: [] for k in ("sort_ms", "gather_ms", "compress_ms", "index_ms", "finish_ms")}
        for _ in range(args.repeats):
            _, st = sorted_run(batch)
            for k in ("sort_ms", "gather_ms", "compress_ms", "index_ms"):
                finish[k].append(getattr(st, k))
            finish["finish_ms"].append(st.total_ms)
        # the inflater alone
        allz = b"".join(open(p, "rb").read() for p in paths)
        ctx = ema_b200.Context()
        ema_b200.bgzf_inflate(ctx, allz)   # warm-up
        kms, n_out = [], 0
        for _ in range(args.repeats):
            n_out = len(ema_b200.bgzf_inflate(ctx, allz))
            kms.append(ctx.last_kernel_ms)
        ctx.close()
        # the merge
        ema_b200.bam_merge(paths)   # warm-up
        walls, split = [], []
        st = {}
        for _ in range(args.repeats):
            st = {}
            t0 = time.time()
            body, bai = ema_b200.bam_merge(paths, stats=st)
            walls.append(time.time() - t0)
            split.append(st)
        in_bytes = sum(os.path.getsize(p) for p in paths)
        w = med(walls)
    finally:
        shutil.rmtree(tmp, ignore_errors=True)
    keys = ("inflate_ms", "rows_ms", "order_ms", "gather_ms", "compress_ms", "index_ms")
    print(json.dumps({
        "workload": args.workload, "steps": args.steps, "inputs": args.inputs, "workers": args.workers, "threads": threads,
        "pairs_per_bucket": pairs, "qualities": "redrawn from F : , # (seeded)",
        "inflate": {"compressed_bytes": len(allz), "inflated_bytes": n_out, "kernel_ms_median": round(med(kms), 3),
                    "gb_per_s": round(n_out / med(kms) / 1e6, 2)},
        "merge": {"wall_s": [round(x, 3) for x in walls], "input_mb_per_s": round(in_bytes / w / 1e6, 1),
                  "records": st["records"], "records_per_s": round(st["records"] / w), "windows": st["windows"],
                  "ms_median": {k: round(med([s[k] for s in split]), 2) for k in keys},
                  "ms_per_bucket": {k: round(med([s[k] for s in split]) / args.steps, 2) for k in keys},
                  "output_bytes": len(body) + len(eof), "bai_bytes": len(bai)},
        "sorted_finish_ms_median": {k: round(med(v), 2) for k, v in finish.items()},
        "sorted_finish_ms_per_bucket": {k: round(med(v) / args.steps, 2) for k, v in finish.items()},
        "gpu": smi,
    }))


if __name__ == "__main__":
    main()

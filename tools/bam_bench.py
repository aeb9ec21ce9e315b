"""SAM versus BAM output end to end on bench.py's default workload (c3: synthetic 3.1 Gbp reference, 40 000-pair buckets).

Qualities are redrawn from four binned values (F : , #, seeded): the synthetic buckets' constant qualities would flatter
every compression ratio, and qualities do not change the alignments.  One session runs the same K buckets through
emab_align_buckets, alternating SAM and BAM output, three repetitions each; prints one JSON line: pairs/s per format, bytes
per bucket (SAM text, raw BAM, BGZF), the BGZF size against zlib level 1 on the same raw bytes and chunking, the
formatting kernels' device time per bucket, and the card's name and power limit read in the same run.

    python tools/bam_bench.py [--steps 12] [--workers 8]
"""
import argparse
import json
import os
import random
import subprocess
import sys
import time
import zlib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import bench  # noqa: E402
from test_bam import inflate  # noqa: E402

CHUNK = 65280


def binned(raw: bytes, seed: int) -> bytes:
    r = random.Random(seed)
    table = b"F:,#"
    out = []
    for line in raw.split(b"\n"):
        if not line:
            continue
        f = line.split(b" ")
        for k in (3, 5):
            f[k] = bytes(table[r.getrandbits(2)] for _ in range(len(f[k])))
        out.append(b" ".join(f))
    return b"\n".join(out) + b"\n"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workload", default="c3", choices=sorted(bench.WORKLOADS))
    ap.add_argument("--steps", type=int, default=12)
    ap.add_argument("--workers", type=int, default=8)
    ap.add_argument("--threads", type=int, default=0, help="host threads (0 = all cores)")
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--data-dir", default=os.environ.get("EMAB_DATA", "/tmp/emab_data"))
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bam_bench.py needs a CUDA device")
    smi = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
    n_buckets = bench.WORKLOADS[args.workload][1]
    bench.prepare_buckets(args.workload, args.data_dir, min(args.steps, n_buckets))
    fa, buckets, pairs = bench.prepare(args.workload, args.data_dir, min(args.steps, n_buckets))
    import ema_b200
    threads = args.threads or os.cpu_count()
    sess = ema_b200.Session(fa, "10x", threads=threads)
    batch = [ema_b200.PinnedText(binned(open(buckets[i % len(buckets)], "rb").read(), 1000 + i)) for i in range(args.steps)]
    sess.set_workers(args.workers)
    # per-bucket sizes and formatting kernel time (one bucket at a time, untimed)
    per = {}
    for fmt in ("sam", "bam"):
        sess.set_output(fmt)
        out = sess.align_bucket(batch[0])
        per[fmt] = (out, sess.stats.format_kernel_ms)
        sess.align_buckets(batch, keep_text=False)   # warm every worker for this format
    raw = inflate(per["bam"][0])
    zl = 0
    for o in range(0, len(raw), CHUNK):
        c = zlib.compressobj(1, zlib.DEFLATED, -15)
        zl += len(c.compress(raw[o:o + CHUNK]) + c.flush()) + 26
    walls = {"sam": [], "bam": []}
    out_bytes = {}
    for _ in range(args.repeats):
        for fmt in ("sam", "bam"):
            sess.set_output(fmt)
            t0 = time.time()
            lens = sess.align_buckets(batch, keep_text=False)
            walls[fmt].append(time.time() - t0)
            out_bytes[fmt] = sum(lens) / len(lens)
    rate = {f: args.steps * pairs / sorted(w)[len(w) // 2] for f, w in walls.items()}
    print(json.dumps({
        "workload": args.workload, "steps": args.steps, "workers": args.workers, "threads": threads, "pairs_per_bucket": pairs,
        "qualities": "redrawn from F : , # (seeded)",
        "pairs_per_s": {"sam": round(rate["sam"]), "bam": round(rate["bam"])}, "bam_over_sam_rate": round(rate["bam"] / rate["sam"], 3),
        "wall_s": walls,
        "bytes_per_bucket": {"sam_text": len(per["sam"][0]), "bam_raw": len(raw), "bam_bgzf": len(per["bam"][0]),
                             "mean_returned_sam": out_bytes["sam"], "mean_returned_bam": out_bytes["bam"]},
        "bgzf_over_zlib1": round(len(per["bam"][0]) / zl, 4), "zlib1_bytes": zl,
        "bgzf_over_sam_text": round(len(per["bam"][0]) / len(per["sam"][0]), 4),
        "format_kernel_ms_per_bucket": {"sam": per["sam"][1], "bam": per["bam"][1]},
        "gpu": smi,
    }))


if __name__ == "__main__":
    main()

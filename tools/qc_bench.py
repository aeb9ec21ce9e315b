"""What `align -Q` costs end to end on bench.py's default workload (c3: synthetic 3.1 Gbp reference, 40 000-pair buckets).

One session runs the same K buckets through emab_align_buckets with SAM output, alternating QC off and QC on (every call
then counts its records with emab_qc_records after formatting them), three repetitions each.  Prints one JSON line: pairs/s of
both arms (medians), the QC kernels' device time per bucket (CUDA events around them, emab_session_qc_cost), the extra
host-to-device and device-to-host bytes per bucket, the report's size, and the card's name and power limit read in the same
run.

    python tools/qc_bench.py [--steps 12] [--workers 8]
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import bench  # noqa: E402


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
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("qc_bench.py needs a CUDA device")
    smi = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
    n_buckets = bench.WORKLOADS[args.workload][1]
    bench.prepare_buckets(args.workload, args.data_dir, min(args.steps, n_buckets))
    fa, buckets, pairs = bench.prepare(args.workload, args.data_dir, min(args.steps, n_buckets))
    import ema_b200
    threads = args.threads or os.cpu_count()
    sess = ema_b200.Session(fa, "10x", threads=threads)
    batch = [ema_b200.PinnedText(open(buckets[i % len(buckets)], "rb").read()) for i in range(args.steps)]
    sess.set_workers(args.workers)

    def run(qc):
        sess.set_qc(qc)
        t0 = time.time()
        n = sum(sess.align_buckets(batch, keep_text=False))
        return time.time() - t0, n

    run(False)   # warm every worker and shape of both arms
    run(True)
    walls = {"sam": [], "sam_qc": []}
    cost = {"kernel_ms": [], "h2d_bytes": [], "d2h_bytes": []}
    sizes = {}
    for _ in range(args.repeats):
        w, sizes["sam"] = run(False)
        walls["sam"].append(w)
        w, sizes["sam_qc"] = run(True)
        walls["sam_qc"].append(w)
        c = sess.qc_cost()
        assert c["calls"] == args.steps, c
        for k in cost:
            cost[k].append(c[k] / args.steps)
    assert sizes["sam"] == sizes["sam_qc"], "QC changes no output byte"
    report = sess.qc_report()
    sess.set_qc(False)
    rate = {f: args.steps * pairs / med(w) for f, w in walls.items()}
    print(json.dumps({
        "workload": args.workload, "steps": args.steps, "workers": args.workers, "threads": threads, "pairs_per_bucket": pairs,
        "pairs_per_s": {f: round(v) for f, v in rate.items()}, "qc_over_plain_rate": round(rate["sam_qc"] / rate["sam"], 4),
        "wall_s": walls,
        "qc_kernel_ms_per_bucket": round(med(cost["kernel_ms"]), 4),
        "qc_h2d_bytes_per_bucket": round(med(cost["h2d_bytes"])), "qc_d2h_bytes_per_bucket": round(med(cost["d2h_bytes"])),
        "sam_bytes": sizes["sam"], "report_bytes": len(report),
        "gpu": smi,
    }))


if __name__ == "__main__":
    main()

#!/usr/bin/env python
"""The target regime on one B200 (BASELINE configs[2] shape): a synthetic reference whose BWT does not fit L2
(--config g1 = 1 Gbp, c3 = 3.1 Gbp / hg38-sized), indexed on the GPU by emab_index_build, then `--buckets` buckets of
40 000 pairs aligned by ema_b200 and by the unmodified reference (`oracle/_ref/ema`) on the same index; SAM bodies must
be byte-identical (-d runs are compared under the pinned clock of tests/shims/faketime.c).  Prints one JSON line.

Measurement tooling (run through gpurun); not part of the product path."""
import argparse
import hashlib
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from tools import synth  # noqa: E402

REF_EMA = os.path.join(ROOT, "oracle", "_ref", "ema")


def log(*a):
    print(*a, file=sys.stderr, flush=True)


def body_md5(path_or_bytes):
    data = open(path_or_bytes, "rb").read() if isinstance(path_or_bytes, str) else path_or_bytes
    h = hashlib.md5()
    n = 0
    for line in data.splitlines(keepends=True):
        if not line.startswith(b"@"):
            h.update(line)
            n += 1
    return h.hexdigest(), n


def faketime_so(d):
    so = os.path.join(d, "faketime.so")
    if not os.path.exists(so):
        subprocess.run(["gcc", "-shared", "-fPIC", "-O2", os.path.join(ROOT, "tests", "shims", "faketime.c"), "-o", so], check=True)
    return so


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--config", default="c3")
    ap.add_argument("--buckets", type=int, default=2)
    ap.add_argument("--data-dir", default=os.environ.get("EMAB_DATA", "/tmp/emab_data"))
    ap.add_argument("--density", action="store_true", help="-d (density optimisation) under the pinned clock")
    ap.add_argument("--ref-threads", type=int, default=0, help="threads of the reference run (0 = 1: with more, the reference's MI cloud ids depend on scheduling)")
    ap.add_argument("--no-reference", action="store_true")
    args = ap.parse_args()
    import numpy as np
    import ema_b200
    n_contigs, clen, rseed, dup, _, _, indel = synth.CONFIGS[args.config]
    d = os.path.join(args.data_dir, "big_" + args.config)
    os.makedirs(d, exist_ok=True)
    fa = os.path.join(d, "ref.fa")
    out = {"config": args.config, "bp": n_contigs * clen}
    t0 = time.time()
    contigs = synth.make_reference(n_contigs, clen, rseed, dup)
    out["s_make_reference"] = time.time() - t0
    if not os.path.exists(fa + ".fai"):
        t0 = time.time()
        synth.write_fasta(fa, contigs)
        out["s_write_fasta"] = time.time() - t0
    if not os.path.exists(fa + ".sa"):
        st = ema_b200.index_build(fa)
        out["index_build"] = st
        log("[big] index built:", st)
    buckets = []
    t0 = time.time()
    for b in range(args.buckets):
        p = os.path.join(d, f"ema-bin-{b:03d}")
        if not os.path.exists(p):
            synth.write_bucket(p, synth.simulate_pairs(contigs, 200, 200, rseed + 1000 + b, indel=indel))
        buckets.append(p)
    out["s_buckets"] = time.time() - t0
    del contigs
    cores = os.cpu_count() or 1
    t0 = time.time()
    sess = ema_b200.Session(fa, "10x", device=0, threads=cores)
    out["s_session_open"] = time.time() - t0
    out["dense_sa_build_ms"] = sess.index_build_ms if hasattr(sess, "index_build_ms") else None
    env = dict(os.environ)
    res = []
    for p in buckets:
        data = open(p, "rb").read()
        # MI cloud ids continue across the calls of one session (as across the reference's buckets), so only the first
        # pass over each bucket is comparable with a fresh reference run per bucket: reopen the session per bucket
        if res:
            sess.close()
            sess = ema_b200.Session(fa, "10x", device=0, threads=cores)
        md5, n = body_md5(sess.align_bucket(data))
        t0 = time.time()
        sess.align_bucket(data)          # timed: warm
        dt = time.time() - t0
        st = sess.stats
        r = {"bucket": os.path.basename(p), "records": n, "md5": md5, "wall_ms": 1e3 * dt, "kernel_ms": st.kernel_ms,
             "ms_seed": st.ms_seed, "ms_chain": st.ms_chain, "ms_align1": st.ms_align1, "ms_rescue": st.ms_rescue, "ms_finalize": st.ms_finalize,
             "occ_touches": st.occ_touches, "seed_GBps": st.occ_touches * 64 / (st.ms_seed * 1e-3) / 1e9}
        if not args.no_reference and os.path.exists(REF_EMA):
            thr = args.ref_threads or 1   # MI cloud ids are scheduling-dependent in the reference with -t > 1
            o = os.path.join(d, "ref_out.sam")
            t0 = time.time()
            subprocess.run([REF_EMA, "align", "-s", p, "-r", fa, "-p", "10x", "-t", str(thr), "-o", o],
                           check=True, env=env, stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
            r["ref_wall_s"] = time.time() - t0
            r["ref_threads"] = thr
            r["ref_md5"], r["ref_records"] = body_md5(o)
            r["identical"] = r["ref_md5"] == md5 and r["ref_records"] == n
        res.append(r)
        log("[big]", r)
    out["buckets"] = res
    if args.density:
        # -d seeds rand() from time(): both command lines run under the pinned clock, the reference with -t 1
        sess.close()
        env["LD_PRELOAD"] = faketime_so(d)
        cli = os.path.join(ROOT, "ema_b200", "ema-b200")
        dres = []
        for p in buckets:
            o1, o2 = os.path.join(d, "d_ours.sam"), os.path.join(d, "d_ref.sam")
            t0 = time.time()
            subprocess.run([cli, "align", "-s", p, "-r", fa, "-p", "10x", "-t", str(cores), "-d", "-o", o1], check=True, env=env,
                           stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
            t1 = time.time()
            b = (None, None)
            if not args.no_reference and os.path.exists(REF_EMA):
                subprocess.run([REF_EMA, "align", "-s", p, "-r", fa, "-p", "10x", "-t", "1", "-d", "-o", o2], check=True, env=env,
                               stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
                b = body_md5(o2)
            t2 = time.time()
            a = body_md5(o1)
            dres.append({"bucket": os.path.basename(p), "ours_cli_s": t1 - t0, "ref_t1_s": t2 - t1, "md5": a[0], "ref_md5": b[0],
                         "records": a[1], "identical": a == b if b[0] is not None else None})
            log("[big -d]", dres[-1])
        out["density"] = dres
        out["density_identical"] = all(r["identical"] for r in dres) if dres and dres[0]["identical"] is not None else None
    out["all_identical"] = all(r.get("identical", False) for r in res) if res and "identical" in res[0] else None
    print(json.dumps(out))


if __name__ == "__main__":
    main()

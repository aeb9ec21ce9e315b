"""GPU tests (-m gpu) of the host's batch runner, which moves -x buckets, the -1/-2 stream's batches and the parts of a
split bucket through the pipeline: the stats a call reports are the sum of its batches' whatever the mode, and a failing
batch ends the call with its error instead of hanging it."""
import ctypes as C
import os
import subprocess

import pytest

import helpers
from test_gpu_sam import CLI

pytestmark = pytest.mark.gpu

# counters that depend only on the reads, not on how they are cut into batches (occ_touches does not qualify: a batch
# seeded again with more room counts differently from its parts)
PER_READ = ("n_pairs", "n_barcodes", "n_cands", "n_clouds", "sam_bytes", "extend_cells", "global_cells", "local_cells",
            "ext_planned_cells", "glob_planned_cells")


def _counters(st, names=PER_READ):
    return {n: getattr(st, n) for n in names}


def _c1_rep(platform="10x"):
    import ema_b200
    from tools import synth
    return synth.build_config("c1_rep", helpers.DATA_ROOT, indexer=ema_b200.index_build, platform=platform)


def _bucket_lines(p):
    return [l for l in open(p["bucket"], "rb").read().split(b"\n") if l]


def test_buckets_stats_are_the_sum_of_single_calls():
    """-x (emab_align_buckets, three workers): every counter is the sum of the same buckets aligned one call each, and
    the SAM kernels' time is reported."""
    import ema_b200
    p = _c1_rep()
    lines = _bucket_lines(p)
    parts = [b"\n".join(lines[i::5]) + b"\n" for i in range(5)]
    s1 = ema_b200.Session(p["fasta"], "10x", threads=8)
    want = dict.fromkeys(PER_READ + ("launches",), 0)
    serial = []
    for d in parts:
        serial.append(s1.align_bucket(d))
        for n, v in _counters(s1.stats, PER_READ + ("launches",)).items():
            want[n] += v
    s2 = ema_b200.Session(p["fasta"], "10x", threads=8)
    s2.set_workers(3)
    assert s2.align_buckets(parts) == serial
    st = s2.stats
    assert _counters(st, PER_READ + ("launches",)) == want
    assert want["ext_planned_cells"] > 0 and st.format_kernel_ms > 0 and st.total_ms > 0


def test_split_bucket_stats_match_serial():
    """one bucket cut over two index replicas (four workers): the per-read counters of the parts add up to the serial
    run's."""
    import torch
    import ema_b200
    p = _c1_rep()
    data = open(p["bucket"], "rb").read()
    s1 = ema_b200.Session(p["fasta"], "10x", threads=8)
    serial = s1.align_bucket(data)
    s2 = ema_b200.Session(p["fasta"], "10x", threads=8)
    s2.add_device(1 if torch.cuda.device_count() > 1 else 0)
    s2.set_workers(4)
    assert s2.align_bucket(data) == serial
    want = _counters(s1.stats)
    assert _counters(s2.stats) == want
    assert want["ext_planned_cells"] > 0 and s2.stats.format_kernel_ms > 0


READ_CB = C.CFUNCTYPE(C.c_int64, C.c_void_p, C.c_void_p, C.c_int64)
WRITE_CB = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_void_p, C.c_uint64)


def _stream(s, data, batch_pairs):
    """emab_align_fastq_stream over one interleaved input held in memory: (SAM body, stats)"""
    from ema_b200 import _lib
    at, out = [0], []

    def rd(_u, buf, cap):
        n = min(cap, len(data) - at[0])
        C.memmove(buf, data[at[0]:at[0] + n], n)
        at[0] += n
        return n

    def wr(_u, p, n):
        out.append(C.string_at(p, n))
        return 0
    r, w = READ_CB(rd), WRITE_CB(wr)
    _lib._check(_lib.lib().emab_align_fastq_stream(s._h, r, None, None, None, w, None, batch_pairs))
    return b"".join(out), s.stats


def test_stream_stats_match_one_batch():
    """the -1/-2 stream cut into batches of 500 pairs with four workers: the bytes and the per-read counters of the
    one-batch run."""
    import ema_b200
    p = _c1_rep("tru")
    data = open(p["bucket"], "rb").read()
    one = ema_b200.Session(p["fasta"], "tru", threads=8)
    body1, st1 = _stream(one, data, 0)
    many = ema_b200.Session(p["fasta"], "tru", threads=8)
    many.set_workers(4)
    body2, st2 = _stream(many, data, 500)
    assert body2 == body1 and body1.count(b"\n") > p["n_pairs"]
    want = _counters(st1)
    assert _counters(st2) == want
    assert want["n_pairs"] == p["n_pairs"] and want["ext_planned_cells"] > 0 and st2.format_kernel_ms > 0


def _run_cli(args, env):
    return subprocess.run([CLI, "align"] + args + ["-t", "8"], capture_output=True, text=True, timeout=600,
                          env=dict(os.environ, **env))


def test_buckets_error_ends_the_call(tmp_path):
    """-x with three workers, the middle of five buckets holding a read over 200 bp: the run fails with that error."""
    p = _c1_rep()
    lines = _bucket_lines(p)
    files = []
    for i in range(5):
        part = lines[i::5]
        if i == 2:
            f = part[len(part) // 2].split(b" ")
            f[2] += b"A" * 80
            f[3] += b"I" * 80
            part[len(part) // 2] = b" ".join(f)
        files.append(str(tmp_path / f"b{i}"))
        open(files[-1], "wb").write(b"\n".join(part) + b"\n")
    r = _run_cli(["-x", "-r", p["fasta"], "-p", "10x", "-o", str(tmp_path / "x.sam")] + files, {"EMAB_WORKERS": "3"})
    assert r.returncode != 0 and "error: read longer than MAX_READ_LEN (200)" in r.stderr, r.stderr[-2000:]


def test_stream_error_ends_the_call(tmp_path):
    """-1 in batches of 500 pairs over four workers, a late record holding a read over 200 bp: the run fails with that
    error."""
    p = _c1_rep("tru")
    lines = open(p["bucket"], "rb").read().split(b"\n")
    k = 4 * (len(lines) // 4 - 40)             # a record near the end of the input
    lines[k + 1] += b"A" * 80
    lines[k + 3] += b"I" * 80
    fq = tmp_path / "reads.fq"
    fq.write_bytes(b"\n".join(lines))
    r = _run_cli(["-1", str(fq), "-r", p["fasta"], "-p", "tru", "-o", str(tmp_path / "s.sam")],
                 {"EMAB_FASTQ_BATCH": "500", "EMAB_WORKERS": "4"})
    assert r.returncode != 0 and "error: read longer than MAX_READ_LEN (200)" in r.stderr, r.stderr[-2000:]

"""Sorted BAM past a host-memory budget: runs spilled to temporary files and merged on the device (`align -O bam -S -T`,
Session(sort=True, max_host_bytes=N, spill=prefix)).

CPU (-m "not gpu"): the CLI refuses -T without -S; the spill prefix is a session setting, passed through the binding as set.
GPU (-m gpu): with budgets small enough for several spill files and many merge windows, the body and the .bai equal the
in-memory -S run's over every input mode; equal keys spread over several files keep input order; one record per block
still gives the same bytes; the files are gone after finish, a failed call, set_sort and close; a spill file that cannot be
created fails the call with EMAB_ERR_IO naming the path."""
import glob
import os
import subprocess

import pytest

import helpers
from test_bam import CLI, EOF_BLOCK, _data
from test_bam_sort import _check_sorted, index_inputs, layout, header_len, records_of

ROOT = helpers.ROOT


# ---- CPU ----

def test_cli_spill_needs_sort():
    r = subprocess.run([CLI, "align", "-O", "bam", "-T", "/tmp/x", "-s", "x", "-r", "x.fa"], capture_output=True, text=True)
    assert r.returncode != 0 and "-T (spill prefix) needs -S" in r.stderr


class _Recorder:
    """stands in for libema_b200.so: records the session calls the binding makes"""

    def __init__(self):
        self.calls = []

    def __getattr__(self, name):
        def f(*args):
            self.calls.append((name, args))
            return 0
        return f


def test_spill_prefix_is_a_session_setting(monkeypatch):
    from ema_b200 import _lib
    rec = _Recorder()
    monkeypatch.setattr(_lib, "_lib", rec)
    s = _lib.Session("ref.fa", "10x", output="bam", spill="/scratch/run")
    names = [c[0] for c in rec.calls]
    assert "emab_session_sort_spill" in names and "emab_session_sort" not in names, "accepted while sorting is off"
    assert [c[1][1] for c in rec.calls if c[0] == "emab_session_sort_spill"] == [b"/scratch/run"]
    rec.calls.clear()
    s.set_sort(True, 1 << 20)
    s.set_sort(False)
    assert [c[0] for c in rec.calls] == ["emab_session_sort", "emab_session_sort"], "set_sort leaves the prefix alone"
    s.set_spill(None)
    assert rec.calls[-1][0] == "emab_session_sort_spill" and rec.calls[-1][1][1] is None
    rec.calls.clear()
    _lib.Session("ref.fa", "10x", output="bam", sort=True, max_host_bytes=5000, spill="p")
    names = [c[0] for c in rec.calls]
    assert names.index("emab_session_sort_spill") < names.index("emab_session_sort")
    s._h = None   # nothing to close on the stand-in
    monkeypatch.setattr(_lib, "_lib", None)
    assert _lib.lib().emab_session_sort_spill(None, b"x") == -3, "the C ABI refuses a null session"


# ---- GPU ----

def body_of(data: bytes) -> bytes:
    """the BGZF members after the header's"""
    assert data.endswith(EOF_BLOCK)
    offs, sizes, raw = layout(data[:-len(EOF_BLOCK)])
    hl, _ = header_len(raw)
    k, acc = 0, 0
    while acc < hl:
        acc += sizes[k]
        k += 1
    return data[offs[k]:-len(EOF_BLOCK)] if k < len(offs) else b""


def held_bytes(srt: bytes) -> int:
    """the bytes a sorted run holds: raw records plus a 24-byte row each"""
    _, placed, _, no_coor, allrecs = index_inputs(srt)
    raw = layout(srt[:-len(EOF_BLOCK)])[2]
    return len(raw) - header_len(raw)[0] + 24 * len(allrecs)


def _spill_case(args, tmp_path, tag, env=None, div=6, budget=None):
    """one CLI run unsorted, sorted in memory and sorted with -T at a budget of 1/div of the run: the spilled file's body
    equals the in-memory one's, its .bai is the restatement's, and no spill file is left"""
    env = dict(env or os.environ)
    u, m, s = tmp_path / f"u{tag}.bam", tmp_path / f"m{tag}.bam", tmp_path / f"s{tag}.bam"
    subprocess.run([CLI] + args + ["-O", "bam", "-o", str(u)], check=True, env=env, stderr=subprocess.DEVNULL)
    subprocess.run([CLI] + args + ["-O", "bam", "-S", "-o", str(m)], check=True, env=env, stderr=subprocess.DEVNULL)
    mem = m.read_bytes()
    budget = budget or held_bytes(mem) // div
    prefix = tmp_path / f"spill{tag}" / "run"
    prefix.parent.mkdir()
    r = subprocess.run([CLI] + args + ["-O", "bam", "-S", "-T", str(prefix), "-o", str(s)], env=dict(env, EMAB_SORT_HOST_BYTES=str(budget)),
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-2000:]
    n_files = int(r.stderr.split("[sort] ")[1].split(" ")[0])
    assert n_files >= 3, r.stderr[-500:]
    srt = s.read_bytes()
    assert body_of(srt) == body_of(mem)
    _check_sorted(u.read_bytes(), srt, (tmp_path / f"s{tag}.bam.bai").read_bytes())
    assert os.listdir(prefix.parent) == [], "spill files left after finish"
    return srt


@pytest.mark.gpu
def test_spill_equals_in_memory(tmp_path):
    from test_gpu_platforms import _faketime_env
    for cfg in ("c1", "c1_rep"):
        p = _data(cfg)
        _spill_case(["align", "-s", p["bucket"], "-r", p["fasta"], "-p", "10x", "-t", "8"], tmp_path, cfg)
    p = _data("c1_rep")
    lines = [l for l in open(p["bucket"], "rb").read().split(b"\n") if l]
    files = []
    for i in range(4):
        f = tmp_path / f"b{i}"
        f.write_bytes(b"\n".join(lines[i::4]) + b"\n")
        files.append(str(f))
    _spill_case(["align", "-x", "-r", p["fasta"], "-p", "10x", "-t", "8"] + files, tmp_path, "x", env=dict(os.environ, EMAB_WORKERS="3"))
    q = _data("c1_rep", "tru")
    fq = open(q["bucket"], "rb").read().split(b"\n")
    recs = [b"\n".join(fq[i:i + 4]) + b"\n" for i in range(0, len(fq) - 3, 4)]
    (tmp_path / "r1.fq").write_bytes(b"".join(recs[0::2]))
    (tmp_path / "r2.fq").write_bytes(b"".join(recs[1::2]))
    _spill_case(["align", "-1", str(tmp_path / "r1.fq"), "-2", str(tmp_path / "r2.fq"), "-r", q["fasta"], "-p", "tru", "-t", "6"], tmp_path, "12",
                env=dict(os.environ, EMAB_FASTQ_BATCH="700"))
    import random
    r = random.Random(5)   # every seventh pair with a random second read: unmapped mates
    fl = [l.split(b" ") for l in lines]
    for f in fl[::7]:
        f[4] = bytes(r.choice(b"ACGT") for _ in f[4])
    (tmp_path / "unmapped").write_bytes(b"\n".join(b" ".join(f) for f in fl) + b"\n")
    _spill_case(["align", "-s", str(tmp_path / "unmapped"), "-r", p["fasta"], "-p", "10x", "-t", "6"], tmp_path, "u")
    _spill_case(["align", "-s", p["bucket"], "-r", p["fasta"], "-p", "10x", "-t", "6", "-R", "@RG\\tID:rg7\\tSM:s", "-i", "7"], tmp_path, "rg")
    _spill_case(["align", "-s", p["bucket"], "-r", p["fasta"], "-p", "10x", "-t", "6", "-d"], tmp_path, "d", env=_faketime_env(tmp_path))


@pytest.mark.gpu
def test_equal_keys_across_files(tmp_path):
    """one pair repeated in many barcodes over four -x buckets: a large group of equal keys spans several spill files and
    still comes out in input order"""
    p = _data("c1_rep")
    lines = [l for l in open(p["bucket"], "rb").read().split(b"\n") if l]
    bcs = sorted({l.split(b" ")[0] for l in lines})[:40]
    tmpl = lines[len(lines) // 2].split(b" ")
    extra = []
    for k, bc in enumerate(bcs):
        for j in range(12):
            extra.append(b" ".join([bc, tmpl[1] + b"_dup%d_%d" % (k, j)] + tmpl[2:]))
    allx = sorted(lines + extra, key=lambda l: l.split(b" ")[0])
    files = []
    for i in range(4):
        f = tmp_path / f"e{i}"
        f.write_bytes(b"\n".join(sorted(allx[i::4], key=lambda l: l.split(b" ")[0])) + b"\n")
        files.append(str(f))
    group = 2 * len(extra) * 300
    srt = _spill_case(["align", "-x", "-r", p["fasta"], "-p", "10x", "-t", "8"] + files, tmp_path, "eq", env=dict(os.environ, EMAB_WORKERS="3"),
                      budget=group // 4)
    _, sl, refs = records_of(srt)
    names = [l.split(b"\t")[0] for l in sl if b"_dup" in l.split(b"\t")[0]]
    assert len(names) >= len(extra)


@pytest.mark.gpu
def test_one_record_per_block(tmp_path):
    """a budget of a few records: every block holds one record, so chunks, references and members straddle windows"""
    g = os.path.join(ROOT, "tests", "golden", "tiny_rep")
    _spill_case(["align", "-s", os.path.join(g, "ema-bin-000.10x"), "-r", os.path.join(g, "ref.fa"), "-p", "10x", "-t", "4"], tmp_path, "tiny",
                budget=3000)


def _session(p, budget, spill, threads=8):
    import ema_b200
    s = ema_b200.Session(p["fasta"], "10x", threads=threads, output="bam", sort=True, max_host_bytes=budget, spill=spill)
    s.set_workers(3)
    return s


@pytest.mark.gpu
def test_session_spill_bytes_and_stats(tmp_path):
    """the Session path at one and 64 chunks per slice: the same body and BAI as in memory; the stats count the files"""
    p = _data("c1")
    lines = [l for l in open(p["bucket"], "rb").read().split(b"\n") if l]
    parts = [b"\n".join(lines[i::3]) + b"\n" for i in range(3)]
    out = []
    for sc in (1, 64):
        os.environ["EMAB_SORT_SLICE_CHUNKS"] = str(sc)
        try:
            m = _session(p, 0, None)
            m.header(["ema", "align"])
            m.align_buckets(parts)
            want = m.finish()
            # cloud ids continue across the runs of one session: each run below has a session of its own
            s = _session(p, 0, str(tmp_path / "s"))   # a cap of 0: no limit, nothing spills
            s.header(["ema", "align"])
            s.align_buckets(parts)
            assert s.stats.spill_files == 0
            assert s.finish() == want
            import ema_b200
            s = ema_b200.Session(p["fasta"], "10x", threads=8, output="bam", spill=str(tmp_path / "s"))   # set while sorting is off
            s.set_workers(3)
            s.set_sort(True, len(want[0]) // 2)
            s.header(["ema", "align"])
            s.align_buckets(parts)
            st = s.stats
            assert st.spill_files >= 3 and st.spill_bytes > 0 and st.spill_ms > 0, st.spill_files
            assert glob.glob(str(tmp_path / "s.*.spill"))
            got = s.finish()
            assert got == want
            assert s.stats.sort_ms > 0 and not glob.glob(str(tmp_path / "s.*"))
            out.append(got)
        finally:
            del os.environ["EMAB_SORT_SLICE_CHUNKS"]
    assert out[0] == out[1]


@pytest.mark.gpu
def test_spill_cleanup_and_errors(tmp_path):
    import ema_b200
    p = _data("c1_rep")
    data = open(p["bucket"], "rb").read()
    pre = str(tmp_path / "k")
    # set_sort(False) mid-run, and close
    s = _session(p, 50_000, pre)
    s.align_bucket(data)
    assert glob.glob(pre + ".*.spill")
    s.set_sort(False)
    assert not glob.glob(pre + ".*")
    s.set_sort(True, 50_000)
    s.align_bucket(data)
    assert glob.glob(pre + ".*.spill")
    s.close()
    assert not glob.glob(pre + ".*")
    # a prefix in a missing directory
    bad = str(tmp_path / "missing" / "run")
    s = _session(p, 50_000, bad)
    with pytest.raises(ema_b200.EmabError, match="error -1.*" + bad.replace(".", r"\.")):
        s.align_bucket(data)
    with pytest.raises(ema_b200.EmabError):
        s.finish()
    out = tmp_path / "bad.bam"
    r = subprocess.run([CLI, "align", "-O", "bam", "-S", "-T", bad, "-s", p["bucket"], "-r", p["fasta"], "-p", "10x", "-t", "4", "-o", str(out)],
                       env=dict(os.environ, EMAB_SORT_HOST_BYTES="50000"), capture_output=True, text=True)
    assert r.returncode != 0 and bad in r.stderr
    assert out.read_bytes() == b"" and not os.path.exists(str(out) + ".bai")
    # a read over 200 bp in the last -x bucket, and in a late stream batch: the files of the failed run are removed
    lines = [l for l in data.split(b"\n") if l]
    files = []
    for i in range(4):
        part = lines[i::4]
        if i == 3:
            f = part[len(part) // 2].split(b" ")
            f[2] += b"A" * 80
            f[3] += b"I" * 80
            part[len(part) // 2] = b" ".join(f)
        files.append(str(tmp_path / f"f{i}"))
        open(files[-1], "wb").write(b"\n".join(part) + b"\n")
    r = subprocess.run([CLI, "align", "-O", "bam", "-S", "-T", pre, "-x", "-r", p["fasta"], "-p", "10x", "-t", "8", "-o", str(tmp_path / "x.bam")] + files,
                       env=dict(os.environ, EMAB_SORT_HOST_BYTES="50000", EMAB_WORKERS="3"), capture_output=True, text=True)
    assert r.returncode != 0 and "MAX_READ_LEN" in r.stderr
    assert not glob.glob(pre + ".*")
    q = _data("c1_rep", "tru")
    fq = open(q["bucket"], "rb").read().split(b"\n")
    k = 4 * (len(fq) // 4 - 40)
    fq[k + 1] += b"A" * 80
    fq[k + 3] += b"I" * 80
    (tmp_path / "long.fq").write_bytes(b"\n".join(fq))
    r = subprocess.run([CLI, "align", "-O", "bam", "-S", "-T", pre, "-1", str(tmp_path / "long.fq"), "-r", q["fasta"], "-p", "tru", "-t", "8",
                        "-o", str(tmp_path / "l.bam")],
                       env=dict(os.environ, EMAB_SORT_HOST_BYTES="50000", EMAB_FASTQ_BATCH="500", EMAB_WORKERS="4"), capture_output=True, text=True)
    assert r.returncode != 0 and "MAX_READ_LEN" in r.stderr
    assert not glob.glob(pre + ".*")

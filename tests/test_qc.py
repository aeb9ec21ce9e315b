"""Alignment and linked-read molecule QC (`align -Q FILE`, Session(qc=True), emab_qc_records).

CPU (-m "not gpu"): the report renderer (ema_b200/csrc/host/qc.hpp, built for the host) against the Python restatement of
report format 1 below, byte for byte, on hand-made and random accumulators; -Q in the CLI's option parsing and usage.
GPU (-m gpu): the -Q file equals the restatement computed from the run's own SAM text, over every input mode; the report is
the same bytes over output modes, worker counts, bucket splits and devices; -Q changes no output byte; emab_session_qc(s, 1)
starts afresh; an MI outside the batch's range is an argument error."""
import ctypes as C
import os
import random
import subprocess

import pytest

import helpers
from test_bam import CLI, _data

ROOT = helpers.ROOT
G = os.path.join(ROOT, "tests", "golden")
FS_NAMES = ["total", "primary", "secondary", "supplementary", "duplicates", "primary duplicates", "mapped", "primary mapped",
            "paired in sequencing", "read1", "read2", "properly paired", "with itself and mate mapped", "singletons",
            "with mate mapped to a different chr", "with mate mapped to a different chr (mapQ>=5)"]
MAPQ_BINS, ISIZE_BINS = 256, 8192


# ---- report format 1, restated ----

class Acc:
    def __init__(self, n_ref):
        self.fs = [[0, 0] for _ in FS_NAMES]
        self.mapq = [0] * MAPQ_BINS
        self.isize = [0] * ISIZE_BINS
        self.ref_mapped = [0] * (n_ref + 1)
        self.ref_unmapped = [0] * (n_ref + 1)
        self.molecules = []          # (length, reads, xf, multi_contig)
        self.n_barcodes = 0


def render(a: Acc, sq) -> bytes:
    o = ["# ema-b200 qc 1"]
    for k, name in enumerate(FS_NAMES):
        o.append(f"FS\t{name}\t{a.fs[k][0]}\t{a.fs[k][1]}")
    one = [m for m in a.molecules if not m[3]]
    lengths = sorted((m[0] for m in one), reverse=True)
    total, run, n50 = sum(lengths), 0, 0
    for l in lengths:
        run += l
        if 2 * run >= total:
            n50 = l
            break
    reads = sum(m[1] for m in one)

    def mean(x, y):
        return "%.2f" % (x / y if y else 0.0)
    o += [f"LR\tbarcodes\t{a.n_barcodes}", f"LR\tmolecules\t{len(a.molecules)}", f"LR\tmolecules_xf\t{sum(1 for m in a.molecules if m[2])}",
          f"LR\tmolecules_multi_contig\t{len(a.molecules) - len(one)}", f"LR\tmolecule_reads\t{reads}", f"LR\tmolecule_length_sum\t{total}",
          f"LR\tmolecule_length_mean\t{mean(total, len(one))}", f"LR\tmolecule_length_n50\t{n50}",
          f"LR\treads_per_molecule_mean\t{mean(reads, len(one))}", f"LR\tmolecules_per_barcode_mean\t{mean(len(one), a.n_barcodes)}"]
    o += [f"MQ\t{k}\t{n}" for k, n in enumerate(a.mapq) if n]
    o += [f"IS\t{k}\t{n}" for k, n in enumerate(a.isize) if n]
    bins, per = {}, {}
    for m in one:
        bins[m[0] // 1000 * 1000] = bins.get(m[0] // 1000 * 1000, 0) + 1
        per[m[1]] = per.get(m[1], 0) + 1
    o += [f"ML\t{k}\t{bins[k]}" for k in sorted(bins)]
    o += [f"RM\t{k}\t{per[k]}" for k in sorted(per)]
    o += [f"IX\t{name}\t{ln}\t{a.ref_mapped[i]}\t{a.ref_unmapped[i]}" for i, (name, ln) in enumerate(sq)]
    o.append(f"IX\t*\t0\t0\t{a.ref_mapped[len(sq)] + a.ref_unmapped[len(sq)]}")
    return ("\n".join(o) + "\n").encode()


def ref_len(cigar: bytes):
    n, out = 0, 0
    for ch in cigar:
        if 48 <= ch <= 57:
            n = n * 10 + ch - 48
        else:
            if ch in b"MDN=X":
                out += n
            n = 0
    return out


def report_from_sam(sam: bytes, haplotag=False) -> bytes:
    """every section of the report from SAM text by the rules of include/ema_b200.h (samtools >= 1.13 flagstat)"""
    lines = sam.split(b"\n")
    sq = []
    for l in lines:
        if l.startswith(b"@SQ"):
            f = dict(x.split(b":", 1) for x in l.split(b"\t")[1:])
            sq.append((f[b"SN"].decode(), int(f[b"LN"])))
    ix = {}
    for i, (name, _) in enumerate(sq):
        ix.setdefault(name.encode(), i)
    a = Acc(len(sq))
    mols, bcs = {}, set()
    for l in lines:
        if not l or l.startswith(b"@"):
            continue
        f = l.split(b"\t")
        flag, mapq = int(f[1]), int(f[4])
        ref = ix.get(f[2], -1)
        mref = ref if f[6] == b"=" else ix.get(f[6], -1)
        tags = {t[:2]: t[5:] for t in f[11:]}
        w = 1 if flag & 0x200 else 0
        unm, munm = flag & 4, flag & 8

        def cnt(k):
            a.fs[k][w] += 1
        cnt(0)
        if flag & 0x100:
            cnt(2)
        elif flag & 0x800:
            cnt(3)
        else:
            cnt(1)
            if flag & 1:
                cnt(8)
                if flag & 2 and not unm:
                    cnt(11)
                if flag & 0x40:
                    cnt(9)
                if flag & 0x80:
                    cnt(10)
                if munm and not unm:
                    cnt(13)
                if not unm and not munm:
                    cnt(12)
                    if mref != ref:
                        cnt(14)
                        if mapq >= 5:
                            cnt(15)
            if not unm:
                cnt(7)
                a.mapq[mapq] += 1
            if flag & 0x400:
                cnt(5)
        if not unm:
            cnt(6)
        if flag & 0x400:
            cnt(4)
        if flag & 0x40 and not unm and not munm and mref == ref:
            a.isize[min(abs(int(f[8])), ISIZE_BINS - 1)] += 1
        k = ref if ref >= 0 else len(sq)
        (a.ref_unmapped if unm else a.ref_mapped)[k] += 1
        bx = tags[b"BX"]
        bcs.add(bx if haplotag else bx.rsplit(b"-", 1)[0])
        if b"MI" in tags:
            pos = int(f[3]) - 1
            end = pos + max(ref_len(f[5]), 1)
            m = mols.setdefault(int(tags[b"MI"]), [pos, end, 0, 0, set()])
            m[0], m[1] = min(m[0], pos), max(m[1], end)
            m[2] += 1
            m[3] |= int(tags[b"XF"])
            m[4].add(ref)
    a.n_barcodes = len(bcs)
    a.molecules = [(m[1] - m[0], m[2], m[3], int(len(m[4]) > 1)) for m in mols.values()]
    return render(a, sq)


# ---- CPU: the renderer's host build ----

class Mol(C.Structure):
    _fields_ = [("length", C.c_uint32), ("reads", C.c_uint32), ("xf", C.c_uint8), ("multi_contig", C.c_uint8), ("pad", C.c_uint16)]


@pytest.fixture(scope="module")
def host_qc(tmp_path_factory):
    so = tmp_path_factory.mktemp("qc") / "qc_host.so"
    subprocess.run(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", os.path.join(ROOT, "tests", "qc_host", "qc_host.cpp"), "-o", str(so)], check=True)
    L = C.CDLL(str(so))
    L.qc_host_render.restype = C.c_uint64
    L.qc_host_render.argtypes = [C.c_void_p] * 3 + [C.c_int] + [C.c_void_p] * 5 + [C.c_uint64, C.c_uint64, C.c_void_p, C.c_uint64]
    assert L.qc_host_molecule_size() == C.sizeof(Mol)
    return L


def host_render(L, a: Acc, sq) -> bytes:
    u64 = lambda xs: (C.c_uint64 * max(len(xs), 1))(*xs)
    names = (C.c_char_p * max(len(sq), 1))(*[n.encode() for n, _ in sq])
    lens = (C.c_int32 * max(len(sq), 1))(*[l for _, l in sq])
    mols = (Mol * max(len(a.molecules), 1))(*[Mol(*m, 0) for m in a.molecules])
    args = [u64([x for p in a.fs for x in p]), u64(a.mapq), u64(a.isize), len(sq), names, lens, u64(a.ref_mapped), u64(a.ref_unmapped),
            mols, len(a.molecules), a.n_barcodes]
    n = L.qc_host_render(*args, None, 0)
    out = C.create_string_buffer(n)
    assert L.qc_host_render(*args, out, n) == n
    return out.raw[:n]


def _random_acc(r, sq):
    a = Acc(len(sq))
    for p in a.fs:
        p[0], p[1] = r.randrange(0, 1 << 40), r.choice([0, r.randrange(100)])
    for k in r.sample(range(MAPQ_BINS), r.randrange(0, 20)):
        a.mapq[k] = r.randrange(1, 1 << 33)
    for k in r.sample(range(ISIZE_BINS), r.randrange(0, 300)):
        a.isize[k] = r.randrange(1, 1000)
    for i in range(len(sq) + 1):
        a.ref_mapped[i], a.ref_unmapped[i] = r.randrange(0, 1 << 36), r.randrange(0, 50)
    a.molecules = [(r.choice([0, 1, 999, 1000, r.randrange(1 << 20), (1 << 32) - 1]), r.randrange(1, 500), r.randrange(2), int(r.random() < 0.05))
                   for _ in range(r.randrange(0, 2000))]
    a.n_barcodes = r.choice([0, r.randrange(1, 1 << 20)])
    return a


def test_renderer_matches_restatement(host_qc):
    sq2 = [("chr1", 60000), ("chr2", 60000)]
    cases = []
    cases.append(("empty run", Acc(2), sq2))
    a = Acc(2)
    a.fs[0] = [2, 0]
    a.molecules, a.n_barcodes = [(416, 2, 1, 0)], 1
    cases.append(("one molecule", a, sq2))
    a = Acc(1)
    a.molecules, a.n_barcodes = [(5000, 3, 0, 0), (5000, 4, 0, 0), (3000, 1, 0, 0), (2000, 2, 0, 0)], 2   # 2 x 5000 = 10000 = total
    cases.append(("N50 tie at the half", a, [("c", 10)]))
    a = Acc(1)
    a.molecules, a.n_barcodes = [(7, 1, 0, 0)] * 4, 3
    cases.append(("all lengths equal", a, [("c", 10)]))
    a = Acc(0)
    a.isize[ISIZE_BINS - 1], a.isize[0], a.isize[8190] = 17, 2, 1
    cases.append(("insert-size overflow bin, no @SQ", a, []))
    a = Acc(1)
    a.molecules, a.n_barcodes = [(100, 2, 1, 0)], 0
    cases.append(("molecules, no barcodes", a, [("c", 10)]))
    a = Acc(1)
    a.n_barcodes = 4
    cases.append(("barcodes, no molecules", a, [("c", 10)]))
    a = Acc(2)
    a.molecules, a.n_barcodes = [(0, 2, 1, 1)], 1
    cases.append(("only a multi-contig molecule", a, sq2))
    a = Acc(2)
    a.molecules, a.n_barcodes = [(123456, 9, 0, 1), (2500, 3, 1, 0), (1500, 3, 0, 0)], 2
    cases.append(("multi-contig molecule beside others", a, sq2))
    r = random.Random(23)
    for i in range(25):
        sq = [(f"contig_{j}", r.randrange(1, 1 << 31)) for j in range(r.randrange(0, 40))]
        cases.append((f"random {i}", _random_acc(r, sq), sq))
    for name, a, sq in cases:
        assert host_render(host_qc, a, sq) == render(a, sq), name
    assert render(Acc(2), sq2).startswith(b"# ema-b200 qc 1\nFS\ttotal\t0\t0\n")
    assert b"LR\tmolecule_length_n50\t5000\n" in render(cases[2][1], cases[2][2])


def test_cli_qc_option():
    r = subprocess.run([CLI, "help"], capture_output=True, text=True)
    assert r.returncode == 0 and "-Q <file>" in r.stdout
    # -Q takes its argument, and the file is opened before any GPU work
    r = subprocess.run([CLI, "align", "-Q", "/nonexistent-dir/qc.txt", "-s", "x", "-r", "x.fa"], capture_output=True, text=True)
    assert r.returncode != 0 and "file /nonexistent-dir/qc.txt could not be opened" in r.stderr
    r = subprocess.run([CLI, "align", "-Q", "q.txt", "-S", "-s", "x", "-r", "x.fa"], capture_output=True, text=True)
    assert r.returncode != 0 and "needs -O bam" in r.stderr


# ---- GPU ----

def _run(args, tmp_path, tag, env=None, out_args=()):
    """one CLI run with -Q -> (output bytes, report bytes)"""
    o, q = tmp_path / f"o{tag}", tmp_path / f"q{tag}.txt"
    subprocess.run([CLI] + args + list(out_args) + ["-o", str(o), "-Q", str(q)], check=True, env=env, stderr=subprocess.DEVNULL)
    return o.read_bytes(), q.read_bytes()


def _by_barcode(path):
    """the bucket's lines grouped by barcode (in order of first appearance), each group in file order"""
    groups = {}
    for l in open(path, "rb").read().split(b"\n"):
        if l:
            groups.setdefault(l.split(b" ", 1)[0], []).append(l)
    return list(groups.values())


def _split(tmp_path, path, k, tag):
    """the bucket cut into k bucket files of whole barcodes"""
    groups = _by_barcode(path)
    files = []
    for i in range(k):
        f = tmp_path / f"{tag}{i}"
        f.write_bytes(b"".join(b"\n".join(g) + b"\n" for g in groups[i::k]))
        files.append(str(f))
    return files


@pytest.mark.gpu
def test_report_equals_restatement_of_sam(tmp_path):
    from test_gpu_platforms import _faketime_env
    seen = {"xf": False, "singleton": False, "isize": False}

    def check(args, tag, env=None, haplotag=False):
        sam, rep = _run(args, tmp_path, tag, env)
        want = report_from_sam(sam, haplotag)
        assert rep == want, (tag, helpers.diff_msg(rep.split(b"\n"), want.split(b"\n")))
        seen["xf"] |= b"LR\tmolecules_xf\t0\n" not in rep
        seen["singleton"] |= b"FS\tsingletons\t0\t0\n" not in rep
        seen["isize"] |= b"\nIS\t" in rep
        assert b"LR\tmolecules\t0\n" not in rep, tag
    for cfg in ("c1", "c1_rep"):
        p = _data(cfg)
        check(["align", "-s", p["bucket"], "-r", p["fasta"], "-p", "10x", "-t", "8"], cfg)
    for platform, in_flag in (("10x", "-s"), ("haplotag", "-s"), ("dbs", "-s"), ("tru", "-1"), ("tellseq", "-1"), ("cpt", "-1")):
        p = _data("c1_rep", platform)
        check(["align", in_flag, p["bucket"], "-r", p["fasta"], "-p", platform, "-t", "6"], platform, haplotag=platform == "haplotag")
    p = _data("c1_rep")
    r = random.Random(5)   # every seventh pair with a random second read: unmapped mates and singletons
    lines = [l.split(b" ") for l in open(p["bucket"], "rb").read().split(b"\n") if l]
    for f in lines[::7]:
        f[4] = bytes(r.choice(b"ACGT") for _ in f[4])
    (tmp_path / "unmapped").write_bytes(b"\n".join(b" ".join(f) for f in lines) + b"\n")
    check(["align", "-s", str(tmp_path / "unmapped"), "-r", p["fasta"], "-p", "10x", "-t", "6"], "u")
    check(["align", "-s", p["bucket"], "-r", p["fasta"], "-p", "10x", "-t", "6", "-R", "@RG\\tID:rg7\\tSM:s", "-i", "7"], "rg")
    check(["align", "-s", p["bucket"], "-r", p["fasta"], "-p", "10x", "-t", "6", "-d"], "d", env=_faketime_env(tmp_path))
    lines = [l for l in open(p["bucket"], "rb").read().split(b"\n") if l]
    files = []
    for i in range(4):
        f = tmp_path / f"b{i}"
        f.write_bytes(b"\n".join(lines[i::4]) + b"\n")
        files.append(str(f))
    check(["align", "-x", "-r", p["fasta"], "-p", "10x", "-t", "8"] + files, "x", env=dict(os.environ, EMAB_WORKERS="3"))
    q = _data("c1_rep", "tru")
    fq = open(q["bucket"], "rb").read().split(b"\n")
    recs = [b"\n".join(fq[i:i + 4]) + b"\n" for i in range(0, len(fq) - 3, 4)]
    (tmp_path / "r1.fq").write_bytes(b"".join(recs[0::2]))
    (tmp_path / "r2.fq").write_bytes(b"".join(recs[1::2]))
    check(["align", "-1", str(tmp_path / "r1.fq"), "-2", str(tmp_path / "r2.fq"), "-r", q["fasta"], "-p", "tru", "-t", "6"], "12",
          env=dict(os.environ, EMAB_FASTQ_BATCH="700"))
    assert all(seen.values()), seen
    # -x without inputs: a zero report
    _, rep = _run(["align", "-x", "-r", p["fasta"], "-p", "10x"], tmp_path, "none")
    assert rep == report_from_sam(open(tmp_path / "onone", "rb").read())
    assert b"FS\ttotal\t0\t0\n" in rep


@pytest.mark.gpu
def test_report_invariance(tmp_path):
    import torch
    p = _data("c1_rep")
    base = ["align", "-r", p["fasta"], "-p", "10x", "-t", "6"]
    _, want = _run(base + ["-s", p["bucket"]], tmp_path, "s")
    assert b"LR\tmolecules\t0\n" not in want
    spill = dict(os.environ, EMAB_SORT_HOST_BYTES="300000")
    runs = {
        "bam": (base + ["-s", p["bucket"], "-O", "bam"], None),
        "bam -S": (base + ["-s", p["bucket"], "-O", "bam", "-S"], None),
        "bam -S -T": (base + ["-s", p["bucket"], "-O", "bam", "-S", "-T", str(tmp_path / "spill")], spill),
    }
    one, four = _split(tmp_path, p["bucket"], 1, "one"), _split(tmp_path, p["bucket"], 4, "four")
    for w in ("1", "3"):
        runs[f"-x 1 bucket, {w} workers"] = (base + ["-x"] + one, dict(os.environ, EMAB_WORKERS=w))
        runs[f"-x 4 buckets, {w} workers"] = (base + ["-x"] + four, dict(os.environ, EMAB_WORKERS=w))
    if torch.cuda.device_count() > 1:
        runs["-x 4 buckets, 2 devices"] = (base + ["-x"] + four, dict(os.environ, EMAB_DEVICES="0,1", EMAB_WORKERS="4"))
    for i, (name, (args, env)) in enumerate(runs.items()):
        _, got = _run(args, tmp_path, f"v{i}", env)
        assert got == want, (name, helpers.diff_msg(got.split(b"\n"), want.split(b"\n")))
    assert not [f for f in os.listdir(tmp_path) if f.endswith(".spill")]


@pytest.mark.gpu
def test_qc_changes_no_output_byte(tmp_path):
    import ema_b200
    p = _data("c1_rep")
    data = open(p["bucket"], "rb").read()
    halves = [b"".join(b"\n".join(g) + b"\n" for g in _by_barcode(p["bucket"])[i::2]) for i in range(2)]

    def run(qc, output, sort):
        s = ema_b200.Session(p["fasta"], "10x", threads=6, output=output, sort=sort, qc=qc)
        s.set_workers(2)
        hdr = s.header(["ema", "align"])
        body = s.align_bucket(data) + b"".join(s.align_buckets(halves))
        bai = b""
        if sort:
            tail, bai = s.finish()
            body += tail
        rep = s.qc_report()
        s.close()
        return hdr + body, bai, rep
    for output, sort in (("sam", False), ("bam", False), ("bam", True)):
        plain, qc = run(False, output, sort), run(True, output, sort)
        assert plain[:2] == qc[:2], (output, sort)
        assert b"FS\ttotal\t0\t0\n" in plain[2], "QC off counts nothing"
        if output == "sam":
            assert qc[2] == report_from_sam(qc[0])
            sam_rep = qc[2]
        else:
            assert qc[2] == sam_rep, (output, sort)
    # through the CLI: the SAM body is the same (the @PG line echoes the command line)
    a, _ = _run(["align", "-s", p["bucket"], "-r", p["fasta"], "-p", "10x", "-t", "6"], tmp_path, "cli")
    b = tmp_path / "plain.sam"
    subprocess.run([CLI, "align", "-s", p["bucket"], "-r", p["fasta"], "-p", "10x", "-t", "6", "-o", str(b)], check=True, stderr=subprocess.DEVNULL)
    strip = lambda t: [l for l in t.split(b"\n") if not l.startswith(b"@PG")]
    assert strip(a) == strip(b.read_bytes())


@pytest.mark.gpu
def test_session_qc_restarts():
    """two runs on one session with emab_session_qc(s, 1) between them: the report is the second run's alone"""
    import ema_b200
    p = _data("c1_rep")
    halves = [b"".join(b"\n".join(g) + b"\n" for g in _by_barcode(p["bucket"])[i::2]) for i in range(2)]
    s = ema_b200.Session(p["fasta"], "10x", threads=6, qc=True)
    hdr = s.header(["ema"])
    s.align_bucket(halves[0])
    first = s.qc_report()
    assert s.qc_cost()["calls"] == 1
    s.set_qc(True)
    assert s.qc_report() == report_from_sam(hdr) and s.qc_cost()["calls"] == 0
    sam = s.align_bucket(halves[1])
    second = s.qc_report()
    assert sam and b"LR\tmolecules\t0\n" not in second, "the second run counts records"
    assert second != first and second == report_from_sam(hdr + sam)
    assert s.qc_cost()["calls"] == 1 and s.qc_cost()["kernel_ms"] > 0
    fresh = ema_b200.Session(p["fasta"], "10x", threads=6, qc=True)
    fresh.align_bucket(halves[1])
    assert fresh.qc_report() == second
    s.set_qc(False)
    s.align_bucket(halves[0])
    assert s.qc_report() == second, "off: nothing more is counted"


class SamRec(C.Structure):
    _fields_ = [("pair", C.c_uint32), ("rec_cand", C.c_int32), ("mate_cand", C.c_int32), ("alt_cand", C.c_int32), ("mi", C.c_int32),
                ("bc", C.c_uint32), ("flag", C.c_uint16), ("which", C.c_uint8), ("mapq", C.c_uint8), ("xf", C.c_uint8),
                ("gamma_len", C.c_uint8), ("gamma", C.c_char * 14)]


class SamJob(C.Structure):
    _fields_ = [("n_recs", C.c_int32), ("n_bc", C.c_int32), ("recs", C.c_void_p), ("bc_off", C.c_void_p), ("bc_text", C.c_char_p),
                ("bx_index", C.c_char_p), ("rg_id", C.c_char_p), ("is_haplotag", C.c_int32), ("pad", C.c_int32)]


class Counts(C.Structure):
    _fields_ = [("flagstat", C.c_uint64 * 32), ("mapq", C.c_uint64 * MAPQ_BINS), ("isize", C.c_uint64 * ISIZE_BINS), ("n_molecules", C.c_int64)]


@pytest.mark.gpu
def test_mi_out_of_range_is_an_argument_error():
    import ema_b200
    L = ema_b200.lib()
    L.emab_session_ctx.restype = C.c_void_p
    L.emab_session_ctx.argtypes = [C.c_void_p]
    L.emab_qc_records.argtypes = [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32] + [C.c_void_p] * 5
    s = ema_b200.Session(os.path.join(G, "tiny_rep", "ref.fa"), "10x", threads=2)
    s.align_bucket(open(os.path.join(G, "tiny_rep", "ema-bin-000.10x"), "rb").read())   # the batch and candidates on the device
    ctx = L.emab_session_ctx(s._h)
    n_ref = s.header(["ema"]).count(b"@SQ")
    recs = (SamRec * 2)(SamRec(0, 0, -1, -1, 1, 0, 1 | 8 | 64, 0, 60, 0, 1, b"1"), SamRec(0, -1, 0, -1, 0, 0, 1 | 4 | 128, 1, 0, 0, 0, b""))
    bc_off = (C.c_int32 * 2)(0, 4)
    job = SamJob(2, 1, C.cast(recs, C.c_void_p), C.cast(bc_off, C.c_void_p), b"ACGT", b"1", None, 0, 0)
    counts, rm, ru = Counts(), (C.c_uint64 * (n_ref + 1))(), (C.c_uint64 * (n_ref + 1))()
    mol, has = (Mol * 4)(), (C.c_uint8 * 1)()

    def call(mi_lo, n_mi):
        return L.emab_qc_records(ctx, C.byref(job), mi_lo, n_mi, n_ref, C.byref(counts), rm, ru, mol, has)
    for mi_lo, n_mi in ((2, 4), (0, 1), (-5, 3)):
        assert call(mi_lo, n_mi) == -3
        assert b"record 0 (pair 0, read 1): MI 1 outside" in L.emab_last_error()
    assert L.emab_qc_records(ctx, C.byref(job), 0, 2, n_ref + 1, C.byref(counts), rm, ru, mol, has) == -3
    # in range, on the same ctx: two records, one molecule of one read, both under refID or '*'
    assert call(1, 1) == 0
    assert counts.flagstat[0] == 2 and counts.n_molecules == 1 and mol[0].reads == 1 and has[0] == 1
    assert sum(rm) == 1 and sum(ru) == 1 and ru[n_ref] == 1
    assert s.align_bucket(open(os.path.join(G, "tiny_rep", "ema-bin-000.10x"), "rb").read())

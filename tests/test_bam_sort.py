"""Coordinate-sorted BAM with a BAI index (`align -O bam -S`, Session(output="bam", sort=True)).

CPU (-m "not gpu"): reg2bin / reg2bins of the host build of csrc/bai.cuh against SAM spec v1 §5.3 restated in Python, at
bin edges; the BAI serializer on hand-made arrays against the Python writer below; the CLI's refusal of -S without -O bam.
GPU (-m gpu): the sorted file holds exactly the unsorted run's records, stably sorted by samtools' coordinate key, over every
input mode; the .bai equals the Python restatement of the index rules built from the decoded file; regions looked up through
the index find what a brute-force scan finds; slice size and repetition do not change a byte; the host-memory cap refuses."""
import ctypes as C
import os
import random
import struct
import subprocess

import numpy as np
import pytest

import helpers
from test_bam import CLI, EOF_BLOCK, _data, decode_bam, members, inflate

ROOT = helpers.ROOT
G = os.path.join(ROOT, "tests", "golden")
CHUNK = 65280
PSEUDO_BIN = 37450


# ---- SAM spec v1 §5.3, restated ----

def spec_reg2bin(beg, end):
    end -= 1
    if beg >> 14 == end >> 14:
        return ((1 << 15) - 1) // 7 + (beg >> 14)
    if beg >> 17 == end >> 17:
        return ((1 << 12) - 1) // 7 + (beg >> 17)
    if beg >> 20 == end >> 20:
        return ((1 << 9) - 1) // 7 + (beg >> 20)
    if beg >> 23 == end >> 23:
        return ((1 << 6) - 1) // 7 + (beg >> 23)
    if beg >> 26 == end >> 26:
        return ((1 << 3) - 1) // 7 + (beg >> 26)
    return 0


def spec_reg2bins(beg, end):
    end -= 1
    out = [0]
    for off, sh in ((1, 26), (9, 23), (73, 20), (585, 17), (4681, 14)):
        out += list(range(off + (beg >> sh), off + (end >> sh) + 1))
    return out


# ---- the index rules, restated (csrc/bai.cuh) ----

def key_of(rid, pos, flag):
    return (rid & 0xffffffff) << 32 | (pos + 1) << 1 | (1 if flag & 16 else 0)


def write_bai(n_ref, recs, voff_end, n_no_coor):
    """recs: placed records in file order as (rid, pos, end, bin, unmapped, voff); voff_end: the virtual offset of the record
    after the last placed one, or of the end of the data"""
    out = bytearray(b"BAI\1" + struct.pack("<i", n_ref))
    for r in range(n_ref):
        idx = [k for k, x in enumerate(recs) if x[0] == r]
        chunks = []   # (bin, beg, end) of maximal runs with the same bin
        for k in idx:
            nxt = recs[k + 1][5] if k + 1 < len(recs) else voff_end
            if chunks and chunks[-1][3] == k - 1 and chunks[-1][0] == recs[k][3]:
                chunks[-1] = (chunks[-1][0], chunks[-1][1], nxt, k)
            else:
                chunks.append((recs[k][3], recs[k][5], nxt, k))
        bins = {}
        for b, beg, end, _ in sorted(chunks, key=lambda c: c[0]):   # stable: file order within a bin
            bins.setdefault(b, []).append((beg, end))
        out += struct.pack("<i", len(bins) + (1 if idx else 0))
        for b in sorted(bins):
            out += struct.pack("<Ii", b, len(bins[b]))
            for beg, end in bins[b]:
                out += struct.pack("<QQ", beg, end)
        lin = []
        if idx:
            unm = sum(recs[k][4] for k in idx)
            last = idx[-1]
            out += struct.pack("<IiQQQQ", PSEUDO_BIN, 2, recs[idx[0]][5], recs[last + 1][5] if last + 1 < len(recs) else voff_end,
                               len(idx) - unm, unm)
            nwin = max((recs[k][2] - 1) >> 14 for k in idx) + 1
            lin = [None] * nwin
            for k in idx:
                for w in range(recs[k][1] >> 14, ((recs[k][2] - 1) >> 14) + 1):
                    if lin[w] is None or recs[k][5] < lin[w]:
                        lin[w] = recs[k][5]
            for w in range(nwin - 2, -1, -1):
                if lin[w] is None:
                    lin[w] = lin[w + 1]
        out += struct.pack("<i", len(lin)) + b"".join(struct.pack("<Q", v) for v in lin)
    return bytes(out + struct.pack("<Q", n_no_coor))


def read_bai(data):
    """a spec-level reader: [(bins {bin: [(beg, end)]}, pseudo (beg, end, mapped, unmapped) or None, linear)], n_no_coor"""
    assert data[:4] == b"BAI\1"
    n_ref, = struct.unpack_from("<i", data, 4)
    o, refs = 8, []
    for _ in range(n_ref):
        n_bin, = struct.unpack_from("<i", data, o)
        o += 4
        bins, pseudo = {}, None
        for _ in range(n_bin):
            b, n = struct.unpack_from("<Ii", data, o)
            o += 8
            ch = [struct.unpack_from("<QQ", data, o + 16 * k) for k in range(n)]
            o += 16 * n
            if b == PSEUDO_BIN:
                pseudo = (ch[0][0], ch[0][1], ch[1][0], ch[1][1])
            else:
                bins[b] = ch
        n_intv, = struct.unpack_from("<i", data, o)
        lin = list(struct.unpack_from(f"<{n_intv}Q", data, o + 4))
        o += 4 + 8 * n_intv
        refs.append((bins, pseudo, lin))
    n_no_coor, = struct.unpack_from("<Q", data, o)
    assert o + 8 == len(data)
    return refs, n_no_coor


# ---- the host build ----

class Ref(C.Structure):
    _fields_ = [("off_beg", C.c_uint64), ("off_end", C.c_uint64), ("n_mapped", C.c_uint64), ("n_unmapped", C.c_uint64),
                ("chunk0", C.c_uint32), ("n_chunk", C.c_uint32), ("lin0", C.c_uint32), ("n_lin", C.c_uint32)]


@pytest.fixture(scope="module")
def host_bai(tmp_path_factory):
    so = tmp_path_factory.mktemp("bai") / "bai_host.so"
    subprocess.run(["g++", "-O2", "-shared", "-fPIC", os.path.join(ROOT, "tests", "bai_host", "bai_host.cpp"), "-o", str(so)], check=True)
    L = C.CDLL(str(so))
    L.bai_host_serialize.restype = C.c_uint64
    L.bai_host_serialize.argtypes = [C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p]
    L.bai_host_reg2bin.argtypes = [C.c_longlong, C.c_longlong]
    L.bai_host_reg2bins.argtypes = [C.c_longlong, C.c_longlong, C.c_void_p]
    assert L.bai_host_ref_size() == C.sizeof(Ref)
    return L


def edges():
    out = []
    for sh in (14, 17, 20, 23, 26):
        for k in (1, 2, 3, 7):
            e = k << sh
            for beg in (e - 2, e - 1, e, e + 1):
                for ln in (1, 2, 100, (1 << sh) - 1, 1 << sh, (1 << sh) + 1):
                    if beg >= 0 and beg + ln <= 1 << 29:
                        out.append((beg, beg + ln))
    out += [(0, 1), (0, 1 << 29), ((1 << 29) - 1, 1 << 29), (-1, 0)]
    r = random.Random(3)
    out += [(b, b + r.randrange(1, 1 << 20)) for b in (r.randrange(0, (1 << 29) - (1 << 20)) for _ in range(300))]
    return out


def test_reg2bin_reg2bins_at_edges(host_bai):
    buf = (C.c_uint16 * 37450)()
    for beg, end in edges():
        assert host_bai.bai_host_reg2bin(beg, end) == spec_reg2bin(beg, end), (beg, end)
        if beg < 0:
            continue
        n = host_bai.bai_host_reg2bins(beg, end, buf)
        assert list(buf[:n]) == spec_reg2bins(beg, end), (beg, end)


def _serialize(L, n_ref, recs, voff_end, n_no_coor):
    """the arrays bam_sort.cu hands the serializer, made by hand from recs: chunks sorted by (ref, bin), windows filled"""
    chunks, refs, lin = [], [], []
    for r in range(n_ref):
        idx = [k for k, x in enumerate(recs) if x[0] == r]
        ch = []
        for k in idx:
            if ch and ch[-1][3] == k - 1 and ch[-1][0] == recs[k][3]:
                ch[-1] = (ch[-1][0], ch[-1][1], None, k)
            else:
                ch.append((recs[k][3], recs[k][5], None, k))
        # chunk ends: the next chunk's start, the first record after the reference, or the end of the data
        starts = [c[1] for c in ch]
        after = recs[idx[-1] + 1][5] if idx and idx[-1] + 1 < len(recs) else voff_end
        ch = [(c[0], c[1], starts[i + 1] if i + 1 < len(ch) else after) for i, c in enumerate(ch)]
        ch.sort(key=lambda c: c[0])
        ref = Ref(chunk0=len(chunks), n_chunk=len(ch), lin0=len(lin))
        chunks += ch
        if idx:
            unm = sum(recs[k][4] for k in idx)
            ref.off_beg, ref.off_end, ref.n_mapped, ref.n_unmapped = recs[idx[0]][5], after, len(idx) - unm, unm
            nwin = max((recs[k][2] - 1) >> 14 for k in idx) + 1
            w = [None] * nwin
            for k in idx:
                for x in range(recs[k][1] >> 14, ((recs[k][2] - 1) >> 14) + 1):
                    w[x] = recs[k][5] if w[x] is None else min(w[x], recs[k][5])
            for x in range(nwin - 2, -1, -1):
                w[x] = w[x + 1] if w[x] is None else w[x]
            lin += w
            ref.n_lin = nwin
        refs.append(ref)
    R = (Ref * max(1, n_ref))(*refs)
    b = np.array([c[0] for c in chunks] or [0], np.uint16)
    cb = np.array([c[1] for c in chunks] or [0], np.uint64)
    ce = np.array([c[2] for c in chunks] or [0], np.uint64)
    ln = np.array(lin or [0], np.uint64)
    args = [n_ref, R, b.ctypes.data, cb.ctypes.data, ce.ctypes.data, ln.ctypes.data, n_no_coor]
    n = L.bai_host_serialize(*args, None)
    out = C.create_string_buffer(n)
    assert L.bai_host_serialize(*args, out) == n
    return out.raw


def test_serializer_on_hand_made_arrays(host_bai):
    r = random.Random(17)
    cases = [(3, []), (1, [(0, 5, 6, spec_reg2bin(5, 6), 0)])]
    for n_ref in (1, 2, 4):
        recs = []
        for ref in sorted(r.randrange(n_ref) for _ in range(r.randrange(1, 80))):
            recs.append(ref)
        rows = []
        for ref in recs:
            pos = r.choice([r.randrange(0, 1 << 16), r.randrange(0, 1 << 22), (1 << 14) - 1, 1 << 14])
            end = pos + r.choice([1, 100, 20000, 1 << 17])
            rows.append((ref, pos, end, spec_reg2bin(pos, end), int(r.random() < 0.1)))
        rows.sort(key=lambda x: (x[0], x[1]))
        cases.append((n_ref, rows))
    for n_ref, rows in cases:
        voff = 7 << 16
        recs = []
        for x in rows:
            recs.append(x + (voff,))
            voff += r.randrange(40, 400)
        no_coor = r.randrange(5)
        got = _serialize(host_bai, n_ref, recs, voff, no_coor)
        assert got == write_bai(n_ref, recs, voff, no_coor)
        refs, nn = read_bai(got)
        assert nn == no_coor and len(refs) == n_ref


def test_cli_sort_needs_bam():
    r = subprocess.run([CLI, "align", "-S", "-s", "x", "-r", "x.fa"], capture_output=True, text=True)
    assert r.returncode != 0 and "-S (coordinate sort) needs -O bam" in r.stderr
    r = subprocess.run([CLI, "align", "-S", "-O", "sam", "-s", "x", "-r", "x.fa"], capture_output=True, text=True)
    assert r.returncode != 0 and "needs -O bam" in r.stderr


# ---- GPU ----

def layout(data: bytes):
    """(member file offsets, uncompressed sizes, raw bytes) of a BGZF file"""
    offs, sizes, raw, o = [], [], [], 0
    for m in members(data):
        offs.append(o)
        o += len(m)
        u = inflate(m)
        sizes.append(len(u))
        raw.append(u)
    return offs, sizes, b"".join(raw)


def walk_records(raw: bytes, o: int):
    """(start offset, rid, pos, flag, bin, reference length of the CIGAR) of every record from o"""
    out = []
    while o < len(raw):
        bs, rid, pos, lrn, _mapq, b, ncig, flag = struct.unpack_from("<iiiBBHHH", raw, o)
        cig = struct.unpack_from(f"<{ncig}I", raw, o + 36 + lrn)
        rl = sum(c >> 4 for c in cig if c & 15 in (0, 2, 3, 7, 8))
        out.append((o, rid, pos, flag, b, rl))
        o += 4 + bs
    assert o == len(raw)
    return out


def header_len(raw: bytes):
    l_text, = struct.unpack_from("<i", raw, 4)
    o = 8 + l_text
    n_ref, = struct.unpack_from("<i", raw, o)
    o += 4
    for _ in range(n_ref):
        ln, = struct.unpack_from("<i", raw, o)
        o += 8 + ln
    return o, n_ref


def index_inputs(data: bytes):
    """what the BAI is built from, read back from the file: n_ref, placed records (rid, pos, end, bin, unmapped, voff),
    the virtual offset after the last placed record, records without a reference, every record's (rid, pos, end, voff,
    unmapped)"""
    assert data.endswith(EOF_BLOCK)
    offs, sizes, raw = layout(data[:-len(EOF_BLOCK)])
    hl, n_ref = header_len(raw)
    # the body starts at a member boundary and is cut every 65 280 bytes
    k0, acc = 0, 0
    while acc < hl:
        acc += sizes[k0]
        k0 += 1
    assert acc == hl
    body_offs, body_sizes = offs[k0:] + [len(data) - len(EOF_BLOCK)], sizes[k0:]
    assert all(s == CHUNK for s in body_sizes[:-1])

    def voff(u):
        m = u // CHUNK
        return body_offs[m] << 16 | (u - m * CHUNK)
    recs = walk_records(raw, hl)
    placed, allrecs = [], []
    for o, rid, pos, flag, b, rl in recs:
        unm = 1 if flag & 4 else 0
        end = pos + (rl if rl and not unm else 1)
        assert rid < 0 or b == spec_reg2bin(pos, end), "the record's bin follows the end rule"
        allrecs.append((rid, pos, end, voff(o - hl), unm))
        if rid >= 0:
            assert len(placed) == len(allrecs) - 1, "records without a reference come last"
            placed.append((rid, pos, end, b, unm, voff(o - hl)))
    after = allrecs[len(placed)][3] if len(placed) < len(allrecs) else voff(len(raw) - hl)
    return n_ref, placed, after, len(recs) - len(placed), allrecs


def records_of(data: bytes):
    text, lines, refs = decode_bam(inflate(data))
    return text, lines, refs


def sorted_lines(lines, refs):
    ix = {r: i for i, r in enumerate(refs)}

    def key(l):
        f = l.split(b"\t")
        return key_of(ix.get(f[2], -1), int(f[3]) - 1, int(f[1]))
    return sorted(lines, key=key)


def _cli_sorted_pair(args, tmp_path, env=None, tag=""):
    """the same CLI run with -O bam and -O bam -S -o -> (unsorted BAM, sorted BAM, .bai bytes)"""
    u, s = tmp_path / f"u{tag}.bam", tmp_path / f"s{tag}.bam"
    subprocess.run([CLI] + args + ["-O", "bam", "-o", str(u)], check=True, env=env, stderr=subprocess.DEVNULL)
    subprocess.run([CLI] + args + ["-O", "bam", "-S", "-o", str(s)], check=True, env=env, stderr=subprocess.DEVNULL)
    return u.read_bytes(), s.read_bytes(), (tmp_path / f"s{tag}.bam.bai").read_bytes()


def _check_sorted(unsorted: bytes, srt: bytes, bai: bytes):
    ut, ul, refs = records_of(unsorted)
    st, sl, refs2 = records_of(srt)
    assert refs == refs2
    # the header differs only in SO: and the @PG line's argv (which has -S)
    assert [l for l in st.split(b"\n") if not l.startswith(b"@PG")] == \
        [l.replace(b"SO:unsorted", b"SO:coordinate") for l in ut.split(b"\n") if not l.startswith(b"@PG")]
    assert st.startswith(b"@HD\tVN:1.3\tSO:coordinate\n") and b" -S" in [l for l in st.split(b"\n") if l.startswith(b"@PG")][0]
    want = sorted_lines(ul, refs)
    assert sl == want, helpers.diff_msg(sl, want)
    n_ref, placed, vend, no_coor, _ = index_inputs(srt)
    assert bai == write_bai(n_ref, placed, vend, no_coor)
    return sl


@pytest.mark.gpu
def test_sorted_order_content_and_index(tmp_path):
    """every input mode: the sorted BAM is the unsorted run's records stably sorted by the coordinate key; the .bai is the
    restatement's file"""
    from test_gpu_platforms import _faketime_env
    seen = []
    for cfg in ("c1", "c1_rep"):
        p = _data(cfg)
        seen += _check_sorted(*_cli_sorted_pair(["align", "-s", p["bucket"], "-r", p["fasta"], "-p", "10x", "-t", "8"], tmp_path, tag=cfg))
    for platform, in_flag in (("10x", "-s"), ("haplotag", "-s"), ("dbs", "-s"), ("tru", "-1"), ("tellseq", "-1"), ("cpt", "-1")):
        p = _data("c1_rep", platform)
        seen += _check_sorted(*_cli_sorted_pair(["align", in_flag, p["bucket"], "-r", p["fasta"], "-p", platform, "-t", "6"], tmp_path, tag=platform))
    p = _data("c1_rep")
    r = random.Random(5)   # every seventh pair with a random second read: unmapped mates
    lines = [l.split(b" ") for l in open(p["bucket"], "rb").read().split(b"\n") if l]
    for f in lines[::7]:
        f[4] = bytes(r.choice(b"ACGT") for _ in f[4])
    (tmp_path / "unmapped").write_bytes(b"\n".join(b" ".join(f) for f in lines) + b"\n")
    seen += _check_sorted(*_cli_sorted_pair(["align", "-s", str(tmp_path / "unmapped"), "-r", p["fasta"], "-p", "10x", "-t", "6"], tmp_path, tag="u"))
    _check_sorted(*_cli_sorted_pair(["align", "-s", p["bucket"], "-r", p["fasta"], "-p", "10x", "-t", "6", "-R", "@RG\\tID:rg7\\tSM:s", "-i", "7"],
                                    tmp_path, tag="rg"))
    _check_sorted(*_cli_sorted_pair(["align", "-s", p["bucket"], "-r", p["fasta"], "-p", "10x", "-t", "6", "-d"], tmp_path,
                                    env=_faketime_env(tmp_path), tag="d"))
    # -x: several buckets, several workers
    lines = [l for l in open(p["bucket"], "rb").read().split(b"\n") if l]
    files = []
    for i in range(4):
        f = tmp_path / f"b{i}"
        f.write_bytes(b"\n".join(lines[i::4]) + b"\n")
        files.append(str(f))
    env = dict(os.environ, EMAB_WORKERS="3")
    seen += _check_sorted(*_cli_sorted_pair(["align", "-x", "-r", p["fasta"], "-p", "10x", "-t", "8"] + files, tmp_path, env=env, tag="x"))
    # -1/-2 streamed in small batches
    q = _data("c1_rep", "tru")
    fq = open(q["bucket"], "rb").read().split(b"\n")
    recs = [b"\n".join(fq[i:i + 4]) + b"\n" for i in range(0, len(fq) - 3, 4)]
    (tmp_path / "r1.fq").write_bytes(b"".join(recs[0::2]))
    (tmp_path / "r2.fq").write_bytes(b"".join(recs[1::2]))
    env = dict(os.environ, EMAB_FASTQ_BATCH="700")
    seen += _check_sorted(*_cli_sorted_pair(["align", "-1", str(tmp_path / "r1.fq"), "-2", str(tmp_path / "r2.fq"), "-r", q["fasta"], "-p", "tru",
                                             "-t", "6"], tmp_path, env=env, tag="12"))
    flags = [int(l.split(b"\t")[1]) for l in seen]
    assert any(f & 4 for f in flags) and any(f & 16 for f in flags), "unmapped mates and reverse-strand hits were sorted"
    # to stdout: sorted, no index
    r = subprocess.run([CLI, "align", "-O", "bam", "-S", "-s", p["bucket"], "-r", p["fasta"], "-p", "10x", "-t", "6"], check=True, capture_output=True)
    u = subprocess.run([CLI, "align", "-O", "bam", "-s", p["bucket"], "-r", p["fasta"], "-p", "10x", "-t", "6"], check=True, capture_output=True).stdout
    _, ul, refs = records_of(u)
    assert records_of(r.stdout)[1] == sorted_lines(ul, refs)


def _regions(rng, length, lin_len):
    out = [(0, length), (max(0, length - 1), length), (0, 1)]
    for w in range(min(lin_len, 40)):
        out += [(max(0, (w << 14) - 1), (w << 14) + 1), (w << 14, (w + 1) << 14)]
    for _ in range(300):
        b = rng.randrange(0, length)
        out.append((b, min(length, b + rng.choice([1, 50, 300, 5000, 1 << 16]))))
    return out


@pytest.mark.gpu
def test_index_finds_what_a_scan_finds(tmp_path):
    """independent of the rules: regions looked up through bins, chunks and the linear lower bound give the records a
    brute-force scan of the file gives; the pseudo-bins' counts and n_no_coor match the file"""
    p = _data("c1_rep")
    u, s, bai = _cli_sorted_pair(["align", "-s", p["bucket"], "-r", p["fasta"], "-p", "10x", "-t", "8"], tmp_path, tag="q")
    refs, n_no_coor = read_bai(bai)
    n_ref, placed, vend, no_coor, allrecs = index_inputs(s)
    assert n_no_coor == no_coor and len(refs) == n_ref
    raw = inflate(s)
    hl, _ = header_len(raw)
    lens = {}
    o = 8 + struct.unpack_from("<i", raw, 4)[0] + 4
    for i in range(n_ref):
        ln, = struct.unpack_from("<i", raw, o)
        lens[i] = struct.unpack_from("<i", raw, o + 4 + ln)[0]
        o += 8 + ln
    rng = random.Random(29)
    by_voff = {x[3]: k for k, x in enumerate(allrecs)}
    starts = sorted(by_voff)
    import bisect
    looked = 0
    for r in range(n_ref):
        bins, pseudo, lin = refs[r]
        mine = [k for k, x in enumerate(allrecs) if x[0] == r]
        if pseudo:
            unm = sum(allrecs[k][4] for k in mine)
            assert pseudo[2] + pseudo[3] == len(mine) and pseudo[3] == unm
            assert pseudo[0] == allrecs[mine[0]][3]
        else:
            assert not mine
        for beg, end in _regions(rng, lens[r], len(lin)):
            want = {k for k in mine if allrecs[k][1] < end and allrecs[k][2] > beg}
            lo = lin[beg >> 14] if (beg >> 14) < len(lin) else None
            got = set()
            for b in spec_reg2bins(beg, end):
                for cb, ce in bins.get(b, []):
                    if lo is not None and ce <= lo:
                        continue
                    for i in range(bisect.bisect_left(starts, cb), bisect.bisect_left(starts, ce)):
                        k = by_voff[starts[i]]
                        x = allrecs[k]
                        if x[0] == r and x[1] < end and x[2] > beg:
                            got.add(k)
            assert got == want, (r, beg, end)
            looked += 1
    assert looked > 300


def _session_sorted(p, parts, slice_chunks, threads=8):
    import ema_b200
    os.environ["EMAB_SORT_SLICE_CHUNKS"] = str(slice_chunks)
    try:
        s = ema_b200.Session(p["fasta"], "10x", threads=threads, output="bam", sort=True)
        s.set_workers(3)
        hdr = s.header(["ema", "align"])
        outs = s.align_buckets(parts)
        assert outs == [b""] * len(parts)
        body, bai = s.finish()
        st = s.stats
        assert st.sam_bytes == len(body) and st.sort_ms > 0 and st.compress_ms > 0 and st.index_ms > 0
        return hdr, body, bai
    finally:
        del os.environ["EMAB_SORT_SLICE_CHUNKS"]


@pytest.mark.gpu
def test_sorted_bytes_deterministic():
    """one 65 280-byte chunk per slice and 64 per slice give the same bytes; a second run gives the same BAM and BAI; the
    Session's file is the unsorted Session run, sorted"""
    import ema_b200
    p = _data("c1")
    lines = [l for l in open(p["bucket"], "rb").read().split(b"\n") if l]
    parts = [b"\n".join(lines[i::3]) + b"\n" for i in range(3)]
    a = _session_sorted(p, parts, 1)
    b = _session_sorted(p, parts, 64)
    c = _session_sorted(p, parts, 64)
    assert a == b == c
    hdr, body, bai = a
    assert len(members(body)) > 1, "more than one slice at one chunk per slice"
    u = ema_b200.Session(p["fasta"], "10x", threads=8, output="bam")
    u.set_workers(3)
    unsorted = u.header(["ema", "align"]) + b"".join(u.align_buckets(parts)) + ema_b200.bgzf_eof()
    _check_sorted_session(unsorted, hdr + body + ema_b200.bgzf_eof(), bai)


def _check_sorted_session(unsorted, srt, bai):
    ut, ul, refs = records_of(unsorted)
    st, sl, _ = records_of(srt)
    assert st == ut.replace(b"SO:unsorted", b"SO:coordinate", 1)
    assert sl == sorted_lines(ul, refs)
    n_ref, placed, vend, no_coor, _ = index_inputs(srt)
    assert bai == write_bai(n_ref, placed, vend, no_coor)


@pytest.mark.gpu
def test_host_memory_cap(tmp_path):
    import ema_b200
    p = _data("c1_rep")
    data = open(p["bucket"], "rb").read()
    s = ema_b200.Session(p["fasta"], "10x", threads=4, output="bam", sort=True, max_host_bytes=100_000)
    with pytest.raises(ema_b200.EmabError, match="error -4.*bytes of host memory"):
        s.align_bucket(data)
    with pytest.raises(ema_b200.EmabError, match="error -4"):
        s.finish()
    # the CLI: a failed exit, an empty file and no index
    out = tmp_path / "capped.bam"
    r = subprocess.run([CLI, "align", "-O", "bam", "-S", "-s", p["bucket"], "-r", p["fasta"], "-p", "10x", "-t", "4", "-o", str(out)],
                       env=dict(os.environ, EMAB_SORT_HOST_BYTES="100000"), capture_output=True, text=True)
    assert r.returncode != 0 and "host memory" in r.stderr
    assert out.read_bytes() == b"" and not os.path.exists(str(out) + ".bai")
    # sorting needs BAM output
    with pytest.raises(ema_b200.EmabError, match="needs BAM output"):
        ema_b200.Session(p["fasta"], "10x", sort=True)

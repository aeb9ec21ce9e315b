"""BAM output (`align -O bam`, Session(output="bam")): BAM records encoded and BGZF-compressed on the device.

CPU (-m "not gpu"): the host build of the block encoder (ema_b200/csrc/bgzf.cuh, compiled from tests/bgzf_host) on edge
inputs — every member well formed, inflated by zlib to its input, CRC-32 and ISIZE accepted by gzip — and the CLI's
refusal of an unknown format.  GPU (-m gpu): decoded BAM equals the SAM text of the same run; the device compressor makes
the host build's bytes; the compression ratio against zlib level 1; BAM's refusals."""
import ctypes as C
import gzip
import os
import random
import struct
import subprocess
import zlib

import pytest

import helpers

ROOT = helpers.ROOT
G = os.path.join(ROOT, "tests", "golden")
CLI = os.path.join(ROOT, "ema_b200", "ema-b200")
CHUNK = 65280
EOF_BLOCK = bytes.fromhex("1f8b08040000000000ff0600424302001b0003000000000000000000")


# ---- the decoder: BGZF members -> bytes, BAM -> SAM text as `samtools view -h` prints it ----

def members(data: bytes):
    """split into BGZF members, checking each one's framing"""
    out, o = [], 0
    while o < len(data):
        assert data[o:o + 4] == b"\x1f\x8b\x08\x04", "gzip magic / FEXTRA"
        xlen = struct.unpack_from("<H", data, o + 10)[0]
        assert xlen == 6 and data[o + 12:o + 14] == b"BC" and struct.unpack_from("<H", data, o + 14)[0] == 2, "BC subfield"
        bsize = struct.unpack_from("<H", data, o + 16)[0]
        out.append(data[o:o + bsize + 1])
        o += bsize + 1
    assert o == len(data), "a member runs past the end"
    return out


def inflate(data: bytes) -> bytes:
    raw = b""
    for m in members(data):
        body = zlib.decompressobj(-15)
        got = body.decompress(m[18:-8]) + body.flush()
        assert body.eof and not body.unused_data
        assert gzip.decompress(m) == got   # CRC-32 and ISIZE
        assert len(m) <= 65536
        raw += got
    return raw


def _z(b, o):
    e = b.index(b"\0", o)
    return b[o:e], e + 1


def decode_bam(raw: bytes):
    """(header text, [SAM lines without newline], reference names)"""
    assert raw[:4] == b"BAM\1"
    l_text = struct.unpack_from("<i", raw, 4)[0]
    text = raw[8:8 + l_text]
    o = 8 + l_text
    n_ref = struct.unpack_from("<i", raw, o)[0]
    o += 4
    refs = []
    for _ in range(n_ref):
        ln = struct.unpack_from("<i", raw, o)[0]
        refs.append(raw[o + 4:o + 4 + ln - 1])
        o += 8 + ln
    lines = []
    while o < len(raw):
        bs, rid, pos, lrn, mapq, _bin, ncig, flag, lseq, nrid, npos, tlen = struct.unpack_from("<iiiBBHHHiiii", raw, o)
        end = o + 4 + bs
        p = o + 36
        name = raw[p:p + lrn - 1]
        p += lrn
        cig = struct.unpack_from(f"<{ncig}I", raw, p)
        p += 4 * ncig
        seq = bytes(b"=ACMGRSVTWYHKDBN"[(raw[p + i // 2] >> (4 - 4 * (i % 2))) & 15] for i in range(lseq))
        p += (lseq + 1) // 2
        q = raw[p:p + lseq]
        p += lseq
        qual = b"*" if not lseq or q[0] == 0xff else bytes(c + 33 for c in q)
        tags = []
        while p < end:
            tg, ty = raw[p:p + 2], raw[p + 2:p + 3]
            p += 3
            if ty in b"cCsSiI":
                fmt = {b"c": "b", b"C": "B", b"s": "h", b"S": "H", b"i": "i", b"I": "I"}[ty]
                v = struct.unpack_from("<" + fmt, raw, p)[0]
                p += struct.calcsize(fmt)
                tags.append(tg + b":i:" + str(v).encode())
            elif ty == b"f":
                tags.append(tg + b":f:" + (b"%g" % struct.unpack_from("<f", raw, p)[0]))
                p += 4
            elif ty == b"A":
                tags.append(tg + b":A:" + raw[p:p + 1])
                p += 1
            elif ty in b"ZH":
                v, p = _z(raw, p)
                tags.append(tg + b":" + ty + b":" + v)
            else:
                raise AssertionError(f"tag type {ty!r}")
        assert p == end
        rname = b"*" if rid < 0 else refs[rid]
        rnext = b"*" if nrid < 0 else b"=" if nrid == rid else refs[nrid]
        cigar = b"".join(str(c >> 4).encode() + b"MIDNSHP=X"[c & 15:(c & 15) + 1] for c in cig) or b"*"
        lines.append(b"\t".join([name, b"%d" % flag, rname, b"%d" % (pos + 1), b"%d" % mapq, cigar, rnext, b"%d" % (npos + 1),
                                 b"%d" % tlen, seq or b"*", qual] + tags))
        o = end
    return text, lines, refs


def bam_to_sam(data: bytes) -> bytes:
    text, lines, _ = decode_bam(inflate(data))
    return text + b"".join(l + b"\n" for l in lines)


def without_pg(sam: bytes) -> bytes:
    return b"".join(l for l in sam.splitlines(keepends=True) if not l.startswith(b"@PG"))


# ---- the host build of the block encoder ----

@pytest.fixture(scope="module")
def host_encoder(tmp_path_factory):
    so = tmp_path_factory.mktemp("bgzf") / "bgzf_host.so"
    subprocess.run(["g++", "-O2", "-shared", "-fPIC", os.path.join(ROOT, "tests", "bgzf_host", "bgzf_host.cpp"), "-o", str(so)], check=True)
    L = C.CDLL(str(so))
    L.bgzf_host_compress.restype = C.c_longlong
    L.bgzf_host_compress.argtypes = [C.c_char_p, C.c_longlong, C.c_char_p, C.c_longlong]

    def compress(data: bytes) -> bytes:
        cap = len(data) + (len(data) // CHUNK + 2) * 64
        out = C.create_string_buffer(cap)
        n = L.bgzf_host_compress(data, len(data), out, cap)
        assert n >= 0
        return out.raw[:n]
    compress.lib = L
    return compress


def encoder_inputs():
    r = random.Random(20261020)
    blk = bytes(r.getrandbits(8) for _ in range(300))
    fib = [1, 1]
    while len(fib) < 26:
        fib.append(fib[-1] + fib[-2])
    # symbol k occurs fib[k] times (the length limit itself is pinned by test_length_limited_codes: matches flatten these counts)
    fibs = bytearray(b"".join(bytes([65 + k]) * f for k, f in enumerate(fib[:23])))
    r.shuffle(fibs)
    sam = open(os.path.join(G, "tiny_rep", "ref.sam"), "rb").read()
    return {
        "empty": b"",
        "one_byte": b"x",
        "random": bytes(r.getrandbits(8) for _ in range(CHUNK)),
        "zeros": bytes(CHUNK),
        "dist_32768": blk + bytes(32768 - len(blk)) + blk,
        "dist_32769": blk + bytes(32769 - len(blk)) + blk,
        "fibonacci": bytes(fibs[:CHUNK]),
        "sam_text": sam,
    }


def dynamic_code_lengths(member: bytes):
    """the literal/length and distance code lengths a dynamic block declares (None for another block type)"""
    data, pos = member[18:-8], 0

    def bits(n):
        nonlocal pos
        v = 0
        for k in range(n):
            v |= ((data[(pos + k) >> 3] >> ((pos + k) & 7)) & 1) << k
        pos += n
        return v
    bits(1)
    if bits(2) != 2:
        return None
    hlit, hdist, hclen = bits(5) + 257, bits(5) + 1, bits(4) + 4
    order = [16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15]
    cl = [0] * 19
    for k in range(hclen):
        cl[order[k]] = bits(3)
    # canonical decode table of the code-length code
    codes, code, nxt = {}, 0, {}
    for ln in range(1, 8):
        code = (code + sum(1 for x in cl if x == ln - 1 and ln > 1)) << 1 if ln > 1 else 0
        nxt[ln] = code
    for s in range(19):
        if cl[s]:
            codes[(cl[s], nxt[cl[s]])] = s
            nxt[cl[s]] += 1
    lens = []
    while len(lens) < hlit + hdist:
        v, ln = 0, 0
        while (ln, v) not in codes:
            v = (v << 1) | bits(1)
            ln += 1
            assert ln <= 7
        s = codes[(ln, v)]
        if s < 16:
            lens.append(s)
        elif s == 16:
            lens += [lens[-1]] * (3 + bits(2))
        elif s == 17:
            lens += [0] * (3 + bits(3))
        else:
            lens += [0] * (11 + bits(7))
    return lens[:hlit], lens[hlit:]


@pytest.mark.parametrize("name", list(encoder_inputs()))
def test_host_encoder_members(host_encoder, name):
    data = encoder_inputs()[name]
    z = host_encoder(data)
    ms = members(z)
    assert len(ms) == max(1, (len(data) + CHUNK - 1) // CHUNK)
    for m in ms:
        assert struct.unpack_from("<H", m, 16)[0] == len(m) - 1 and len(m) <= 65536
    assert inflate(z) == data
    if name == "random":
        assert ms[0][18] & 7 == 1, "incompressible input falls back to a stored block"
    if name == "zeros":
        assert len(z) < 200
    if name == "dist_32768":
        assert len(z) < len(host_encoder(encoder_inputs()["dist_32769"])), "a repeat at the window's edge is matched, one byte farther is not"
    if name in ("fibonacci", "sam_text"):
        lit, dist = dynamic_code_lengths(ms[0])
        assert max(lit) <= 15 and max(dist) <= 15



@pytest.mark.parametrize("limit,n_sym", [(15, 24), (7, 19)])
def test_length_limited_codes(host_encoder, limit, n_sym):
    """Fibonacci-weighted frequencies: an unlimited Huffman code would be n_sym - 1 bits deep; the limited one is complete
    (Kraft sum 1), reaches the limit, and gives no rarer symbol a shorter code than a more frequent one"""
    fib = [1, 1]
    while len(fib) < n_sym:
        fib.append(fib[-1] + fib[-2])   # fib[23] = 46 368: counts of one chunk stay below 65 536
    freq = (C.c_uint32 * n_sym)(*fib[:n_sym])
    lens = (C.c_uint8 * n_sym)()
    host_encoder.lib.bgzf_host_code_lengths(freq, n_sym, limit, lens)
    ln = list(lens)
    assert max(ln) == limit and min(ln) >= 1
    assert sum(2.0 ** -l for l in ln) == 1.0
    assert all(ln[k] >= ln[k + 1] for k in range(n_sym - 1))


def test_cli_unknown_output_format():
    r = subprocess.run([CLI, "align", "-O", "cram", "-s", "x", "-r", "x.fa"], capture_output=True, text=True)
    assert r.returncode != 0 and "unknown output format" in r.stderr


def test_bgzf_eof_block():
    import ema_b200
    assert ema_b200.bgzf_eof() == EOF_BLOCK
    assert gzip.decompress(EOF_BLOCK) == b""


# ---- GPU ----

def _cli_pair(args, tmp_path, env=None, tag=""):
    """the same CLI run with -O sam and -O bam -> (SAM text, BAM bytes)"""
    s, b = tmp_path / f"o{tag}.sam", tmp_path / f"o{tag}.bam"
    subprocess.run([CLI] + args + ["-o", str(s)], check=True, env=env, stderr=subprocess.DEVNULL)
    subprocess.run([CLI] + args + ["-O", "bam", "-o", str(b)], check=True, env=env, stderr=subprocess.DEVNULL)
    return s.read_bytes(), b.read_bytes()


def _same(sam: bytes, bam: bytes):
    assert bam.endswith(EOF_BLOCK)
    got = bam_to_sam(bam)
    assert without_pg(got) == without_pg(sam), helpers.diff_msg(without_pg(got).split(b"\n"), without_pg(sam).split(b"\n"))
    return [l for l in sam.split(b"\n") if l and not l.startswith(b"@")]


def _coverage(lines):
    flags = [int(l.split(b"\t")[1]) for l in lines]
    return any(f & 4 for f in flags), any(b"\tXA:Z:" in l for l in lines), any(f & 16 for f in flags)


def _data(cfg, platform="10x"):
    import ema_b200
    from tools import synth
    return synth.build_config(cfg, helpers.DATA_ROOT, indexer=ema_b200.index_build, platform=platform)


@pytest.mark.gpu
def test_cli_bam_golden_tiny(tmp_path):
    out = tmp_path / "out.bam"
    subprocess.run([CLI, "align", "-O", "bam", "-s", os.path.join(G, "tiny_rep", "ema-bin-000.10x"), "-r", os.path.join(G, "tiny_rep", "ref.fa"),
                    "-p", "10x", "-t", "4", "-o", str(out)], check=True)
    data = out.read_bytes()
    assert data.endswith(EOF_BLOCK)
    want = open(os.path.join(G, "tiny_rep", "ref.sam"), "rb").read()
    got = bam_to_sam(data)
    assert without_pg(got) == without_pg(want)
    # to stdout as well
    r = subprocess.run([CLI, "align", "-O", "bam", "-s", os.path.join(G, "tiny_rep", "ema-bin-000.10x"), "-r", os.path.join(G, "tiny_rep", "ref.fa"),
                        "-p", "10x", "-t", "4"], check=True, capture_output=True)
    assert without_pg(bam_to_sam(r.stdout)) == without_pg(want)


@pytest.mark.gpu
def test_bam_equals_sam(tmp_path):
    """decoded BAM equals the SAM text of the same settings, over every input mode and option that changes a record"""
    from test_gpu_platforms import _faketime_env
    seen = []
    for cfg in ("c1", "c1_rep"):
        p = _data(cfg)
        seen += _same(*_cli_pair(["align", "-s", p["bucket"], "-r", p["fasta"], "-p", "10x", "-t", "8"], tmp_path, tag=cfg))
    for platform, in_flag in (("10x", "-s"), ("haplotag", "-s"), ("dbs", "-s"), ("tru", "-1"), ("tellseq", "-1"), ("cpt", "-1")):
        p = _data("c1_rep", platform)
        lines = _same(*_cli_pair(["align", in_flag, p["bucket"], "-r", p["fasta"], "-p", platform, "-t", "6"], tmp_path, tag=platform))
        bx = [t for l in lines for t in l.split(b"\t") if t.startswith(b"BX:Z:")]
        assert bx and (platform != "haplotag") == any(t.endswith(b"-1") for t in bx)
        seen += lines
    p = _data("c1_rep")
    # every seventh pair with a random second read: unmapped mates (flag 4) next to mapped ones
    r = random.Random(5)
    lines = [l.split(b" ") for l in open(p["bucket"], "rb").read().split(b"\n") if l]
    for f in lines[::7]:
        f[4] = bytes(r.choice(b"ACGT") for _ in f[4])
    (tmp_path / "unmapped").write_bytes(b"\n".join(b" ".join(f) for f in lines) + b"\n")
    seen += _same(*_cli_pair(["align", "-s", str(tmp_path / "unmapped"), "-r", p["fasta"], "-p", "10x", "-t", "6"], tmp_path, tag="u"))
    _same(*_cli_pair(["align", "-s", p["bucket"], "-r", p["fasta"], "-p", "10x", "-t", "6", "-R", "@RG\\tID:rg7\\tSM:s", "-i", "7"], tmp_path, tag="rg"))
    _same(*_cli_pair(["align", "-s", p["bucket"], "-r", p["fasta"], "-p", "10x", "-t", "6", "-d"], tmp_path, env=_faketime_env(tmp_path), tag="d"))
    # -x: several buckets, several workers
    lines = [l for l in open(p["bucket"], "rb").read().split(b"\n") if l]
    files = []
    for i in range(4):
        f = tmp_path / f"b{i}"
        f.write_bytes(b"\n".join(lines[i::4]) + b"\n")
        files.append(str(f))
    env = dict(os.environ, EMAB_WORKERS="3")
    _same(*_cli_pair(["align", "-x", "-r", p["fasta"], "-p", "10x", "-t", "8"] + files, tmp_path, env=env, tag="x"))
    # -1/-2 streamed in small batches
    q = _data("c1_rep", "tru")
    fq = open(q["bucket"], "rb").read().split(b"\n")
    recs = [b"\n".join(fq[i:i + 4]) + b"\n" for i in range(0, len(fq) - 3, 4)]
    (tmp_path / "r1.fq").write_bytes(b"".join(recs[0::2]))
    (tmp_path / "r2.fq").write_bytes(b"".join(recs[1::2]))
    env = dict(os.environ, EMAB_FASTQ_BATCH="700")
    seen += _same(*_cli_pair(["align", "-1", str(tmp_path / "r1.fq"), "-2", str(tmp_path / "r2.fq"), "-r", q["fasta"], "-p", "tru", "-t", "6"],
                             tmp_path, env=env, tag="12"))
    assert all(_coverage(seen)), "the compared records include unmapped mates, XA tags and reverse-strand hits"


@pytest.mark.gpu
def test_session_bam_buckets_are_whole_members():
    """Session(output="bam"): header() and every bucket's bytes are whole BGZF members (blocks never span calls), also with
    several buckets in flight; concatenated with the EOF block they are one BAM file equal to the SAM run"""
    import ema_b200
    p = _data("c1_rep")
    lines = [l for l in open(p["bucket"], "rb").read().split(b"\n") if l]
    parts = [b"\n".join(lines[i::3]) + b"\n" for i in range(3)]
    s = ema_b200.Session(p["fasta"], "10x", threads=8)
    s.set_workers(3)
    sam = s.header(["ema", "align"]) + b"".join(s.align_buckets(parts))
    b = ema_b200.Session(p["fasta"], "10x", threads=8, output="bam")
    b.set_workers(3)
    outs = b.align_buckets(parts)
    hdr = b.header(["ema", "align"])
    for x in [hdr] + outs:
        members(x)
    assert b.stats.sam_bytes == sum(len(x) for x in outs)   # the compressed bytes returned
    assert bam_to_sam(hdr + b"".join(outs) + ema_b200.bgzf_eof()) == sam


@pytest.mark.gpu
def test_device_encoder_matches_host(host_encoder):
    import ema_b200
    ctx = ema_b200.Context()
    r = random.Random(7)
    sam = open(os.path.join(G, "tiny_rep", "ref.sam"), "rb").read()
    mix = bytearray()
    while len(mix) < 40 << 20:   # text, zeros, random bytes, binned qualities, in pieces that straddle chunks
        k = r.randrange(4)
        n = r.randrange(1, 200_000)
        mix += (sam[:n] if k == 0 else bytes(n) if k == 1 else r.randbytes(n) if k == 2 else bytes(r.choice(b"F:,#") for _ in range(n // 16)))
    for name, data in list(encoder_inputs().items()) + [("mix", bytes(mix))]:
        got = ema_b200.bgzf_compress(ctx, data)
        want = host_encoder(data) if data else b""
        assert got == want, name
    assert inflate(got) == bytes(mix)


def _binned_bucket(path, seed=11):
    """the bucket with every quality redrawn from four binned values (qualities do not change the alignments)"""
    r = random.Random(seed)
    out = []
    for l in open(path, "rb").read().split(b"\n"):
        if not l:
            continue
        f = l.split(b" ")
        for k in (3, 5):
            f[k] = bytes(r.choice(b"F:,#") for _ in f[k])
        out.append(b" ".join(f))
    return b"\n".join(out) + b"\n"


@pytest.mark.gpu
def test_compression_ratio_vs_zlib1():
    import ema_b200
    p = _data("c1")
    data = _binned_bucket(p["bucket"])
    b = ema_b200.Session(p["fasta"], "10x", threads=8, output="bam")
    z = b.align_bucket(data)
    raw = inflate(z)
    zl = 0
    for o in range(0, len(raw), CHUNK):
        c = zlib.compressobj(1, zlib.DEFLATED, -15)
        zl += len(c.compress(raw[o:o + CHUNK]) + c.flush()) + 26
    ratio = len(z) / zl
    sam = ema_b200.Session(p["fasta"], "10x", threads=8).align_bucket(data)
    print(f"\nBAM: {len(sam)} SAM bytes, {len(raw)} raw BAM bytes, {len(z)} BGZF bytes = {ratio:.3f} x zlib level 1 ({zl} bytes)")
    assert ratio <= 1.15


def _edit_bucket(edit):
    lines = [l for l in open(os.path.join(G, "tiny_rep", "ema-bin-000.10x"), "rb").read().split(b"\n") if l][:60]
    f = lines[10].split(b" ")
    edit(f)
    lines[10] = b" ".join(f)
    return b"\n".join(lines) + b"\n"


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["name_255", "qual_length", "qual_byte"])
def test_bam_refusals(case):
    import ema_b200

    def edit(f):
        if case == "name_255":
            f[1] = b"@" + b"r" * 255
        elif case == "qual_length":
            f[3] = f[3][:-1]
        else:
            f[3] = b"\x01" + f[3][1:]
    data = _edit_bucket(edit)
    ref = os.path.join(G, "tiny_rep", "ref.fa")
    assert ema_b200.Session(ref, "10x").align_bucket(data)   # SAM accepts it
    with pytest.raises(ema_b200.EmabError, match="emab_bam_format"):
        ema_b200.Session(ref, "10x", output="bam").align_bucket(data)

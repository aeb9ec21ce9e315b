"""Merging coordinate-sorted BAM files on the device (`ema-b200 merge`, ema_b200.bam_merge) and the BGZF decoder under it
(ema_b200/csrc/inflate.cuh, emab_bgzf_inflate).

CPU (-m "not gpu"): the host build of the decoder (tests/inflate_host, with AddressSanitizer and UBSan) against zlib on
members of every block kind, and on hand-made malformed members, every truncation and every single-bit flip; the merged
header's rules (emab_bam_merge_header, host code); the rows built from records read from a file and their refusals
(bam_row.cuh, tests/bam_row_host); the CLI's refusals before any device work.  GPU (-m gpu): the device decoder against
zlib; merging one sorted file reproduces it and its .bai byte for byte; several inputs, a BAM the project did not write,
recompressed inputs, small budgets with records cut across reads, region queries through the index against a scan, and
the refusals of unsorted and out-of-range records, truncated files and the missing-EOF warning."""
import ctypes as C
import os
import random
import struct
import subprocess
import zlib

import pytest

import helpers
from test_bam import CHUNK, CLI, EOF_BLOCK, encoder_inputs, host_encoder  # noqa: F401 (host_encoder is a fixture)

ROOT = helpers.ROOT

# the decoder's codes (inflate.cuh)
TRUNCATED, HEADER, BLOCK_TYPE, STORED_LEN, BAD_CODE, BAD_SYMBOL, DIST_FAR, OUTPUT, CRC, ISIZE = range(1, 11)


# ---- members made by zlib ----

def frame(deflate: bytes, data: bytes, extra: bytes = b"", fname: bytes | None = None, flg: int = 4,
          crc: int | None = None, isize: int | None = None) -> bytes:
    """a BGZF member around a raw DEFLATE stream: gzip header with FEXTRA (other subfields `extra` before BC), optional FNAME"""
    xlen = len(extra) + 6
    tail = b"" if fname is None else fname + b"\0"
    size = 12 + xlen + len(tail) + len(deflate) + 8
    hdr = bytes([31, 139, 8, flg | (8 if fname is not None else 0), 0, 0, 0, 0, 0, 255]) + struct.pack("<H", xlen) + extra + \
        b"BC" + struct.pack("<HH", 2, size - 1) + tail
    return hdr + deflate + struct.pack("<II", zlib.crc32(data) if crc is None else crc, len(data) if isize is None else isize)


def zmember(data: bytes, level: int = 6, strategy: int = zlib.Z_DEFAULT_STRATEGY, flushes=(), **kw) -> bytes:
    """data as one member made by zlib; `flushes`: (offset, mode) pairs where a Z_SYNC_FLUSH / Z_FULL_FLUSH cuts the stream"""
    z = zlib.compressobj(level, zlib.DEFLATED, -15, 9, strategy)
    out, at = b"", 0
    for off, mode in flushes:
        out += z.compress(data[at:off]) + z.flush(mode)
        at = off
    out += z.compress(data[at:]) + z.flush()
    return frame(out, data, **kw)


def zmembers(data: bytes, level=6, strategy=zlib.Z_DEFAULT_STRATEGY, cut=CHUNK) -> bytes:
    return b"".join(zmember(data[o:o + cut], level, strategy) for o in range(0, max(len(data), 1), cut))


@pytest.fixture(scope="module")
def host_inflate(tmp_path_factory):
    so = tmp_path_factory.mktemp("inflate") / "inflate_host.so"
    subprocess.run(["g++", "-O1", "-g", "-shared", "-fPIC", "-fsanitize=address,undefined", "-fno-sanitize-recover=all",
                    os.path.join(ROOT, "tests", "inflate_host", "inflate_host.cpp"), "-o", str(so)], check=True)
    return str(so)


_RUNNER = r"""
import ctypes as C, sys
L = C.CDLL(sys.argv[1])
L.inflate_host.restype = C.c_longlong
L.inflate_host.argtypes = [C.c_char_p, C.c_longlong, C.c_char_p, C.c_longlong, C.POINTER(C.c_longlong)]
data = sys.stdin.buffer.read()
out = sys.stdout.buffer
n = 0
while n < len(data):
    ln = int.from_bytes(data[n:n + 8], "little"); n += 8
    m = data[n:n + ln]; n += ln
    buf = C.create_string_buffer(max(1, 65536 * (len(m) // 18 + 1)))
    at = C.c_longlong(-1)
    r = L.inflate_host(m, len(m), buf, len(buf), C.byref(at))
    res = buf.raw[:r] if r >= 0 else b""
    out.write(r.to_bytes(8, "little", signed=True) + at.value.to_bytes(8, "little", signed=True) + len(res).to_bytes(8, "little") + res)
"""


def run_host(so, inputs):
    """[(rc, bad member offset, bytes)] of the host decoder over each input, in one sanitized process (ASan needs its
    runtime preloaded into Python); any sanitizer finding fails the process"""
    import sysconfig
    asan = subprocess.run(["g++", "-print-file-name=libasan.so"], capture_output=True, text=True).stdout.strip()
    ubsan = subprocess.run(["g++", "-print-file-name=libubsan.so"], capture_output=True, text=True).stdout.strip()
    env = dict(os.environ, LD_PRELOAD=f"{asan} {ubsan}", ASAN_OPTIONS="detect_leaks=0:abort_on_error=1",
               UBSAN_OPTIONS="halt_on_error=1:print_stacktrace=1")
    payload = b"".join(len(m).to_bytes(8, "little") + m for m in inputs)
    r = subprocess.run([sysconfig.get_config_var("BINDIR") + "/python3", "-c", _RUNNER, so], input=payload, capture_output=True, env=env)
    assert r.returncode == 0, r.stderr.decode(errors="replace")[-3000:]
    out, o = [], 0
    d = r.stdout
    while o < len(d):
        rc = int.from_bytes(d[o:o + 8], "little", signed=True)
        at = int.from_bytes(d[o + 8:o + 16], "little", signed=True)
        ln = int.from_bytes(d[o + 16:o + 24], "little")
        out.append((rc, at, d[o + 24:o + 24 + ln]))
        o += 24 + ln
    assert len(out) == len(inputs)
    return out


def zlib_of(m: bytes):
    """zlib's reading of one member (gzip framing, CRC and ISIZE checked), or None where it refuses"""
    try:
        d = zlib.decompressobj(31)
        got = d.decompress(m) + d.flush()
        return got if d.eof and not d.unused_data else None
    except zlib.error:
        return None


def valid_cases(host_encoder):
    r = random.Random(7)
    sam = open(os.path.join(ROOT, "tests", "golden", "tiny_rep", "ref.sam"), "rb").read()
    text = (sam * 2)[:CHUNK]
    rnd = bytes(r.getrandbits(8) for _ in range(20000))
    cases = {}
    for lv in (0, 1, 6, 9):
        cases[f"zlib_level{lv}"] = zmembers(sam, lv)
    for name, st in (("fixed", zlib.Z_FIXED), ("huffman_only", zlib.Z_HUFFMAN_ONLY), ("rle", zlib.Z_RLE)):
        cases[f"zlib_{name}"] = zmembers(sam, 6, st)
    cases["sync_flush"] = zmember(text, 6, flushes=[(100, zlib.Z_SYNC_FLUSH), (100, zlib.Z_SYNC_FLUSH), (30000, zlib.Z_SYNC_FLUSH)])
    cases["full_flush"] = zmember(text, 6, flushes=[(5000, zlib.Z_FULL_FLUSH), (40000, zlib.Z_FULL_FLUSH)])
    cases["stored_random"] = zmember(rnd, 0) + zmember(rnd, 9)
    for k, v in encoder_inputs().items():
        cases[f"encoder_{k}"] = host_encoder(v)
    cases["match_258"] = zmember(b"ACGT" * 16000, 9)   # runs of 258-byte matches
    cases["eof"] = EOF_BLOCK
    cases["fname_extra"] = zmember(text[:3000], 6, extra=b"XY" + struct.pack("<H", 3) + b"abc", fname=b"reads.bam")
    cases["empty_member"] = zmember(b"")
    return cases


def test_host_decoder_equals_zlib(host_inflate, host_encoder):
    cases = valid_cases(host_encoder)
    got = run_host(host_inflate, list(cases.values()))
    for (name, data), (rc, at, out) in zip(cases.items(), got):
        want = b"".join(zlib_of(m) for m in _split(data))
        assert rc >= 0, f"{name}: code {-rc} at {at}"
        assert out == want, name


def _split(data: bytes):
    out, o = [], 0
    while o < len(data):
        xlen = struct.unpack_from("<H", data, o + 10)[0]
        x, bs = o + 12, None
        while x < o + 12 + xlen:
            sl = struct.unpack_from("<H", data, x + 2)[0]
            if data[x:x + 2] == b"BC":
                bs = struct.unpack_from("<H", data, x + 4)[0]
            x += 4 + sl
        out.append(data[o:o + bs + 1])
        o += bs + 1
    return out


def _bits(fields):
    """a raw DEFLATE stream from (value, nbits) fields, LSB first"""
    acc, n, out = 0, 0, bytearray()
    for v, k in fields:
        acc |= v << n
        n += k
        while n >= 8:
            out.append(acc & 255)
            acc >>= 8
            n -= 8
    if n:
        out.append(acc & 255)
    return bytes(out)


def malformed_cases():
    good = zmember(b"hello hello hello hello", 6)
    d = b"abcabcabc"
    cases = {
        "truncated": (good[:-3], TRUNCATED),
        "bad_magic": (b"\x1f\x8c" + good[2:], HEADER),
        "no_bc": (good[:12] + b"XC" + good[14:], HEADER),
        "block_type_3": (frame(_bits([(1, 1), (3, 2)]) + b"\0", b""), BLOCK_TYPE),
        "stored_nlen": (frame(b"\x01" + struct.pack("<HH", 3, 0x1234) + b"abc", b"abc"), STORED_LEN),
        # dynamic block whose code-length code gives three symbols one bit each: over-subscribed
        "oversubscribed": (frame(_bits([(1, 1), (2, 2), (0, 5), (0, 5), (0, 4)] + [(1, 3)] * 4) + b"\0" * 4, b""), BAD_CODE),
        # fixed block: literal/length symbol 286 (8-bit code 11000110) then end
        "lit_286": (frame(_bits([(1, 1), (1, 2), (int("01100011", 2), 8)]) + b"\0", b""), BAD_SYMBOL),
        # fixed block: literal 'a', length 3 (symbol 257, 7-bit code 0000001), distance symbol 30 (11110)
        "dist_30": (frame(_bits([(1, 1), (1, 2), (_rev(0x30 + 97, 8), 8), (_rev(1, 7), 7), (_rev(30, 5), 5), (0, 7)]) + b"\0", b"aaaa"), BAD_SYMBOL),
        # fixed block: literal 'a', length 3 at distance 2
        "dist_far": (frame(_bits([(1, 1), (1, 2), (_rev(0x30 + 97, 8), 8), (_rev(1, 7), 7), (_rev(1, 5), 5), (0, 7)]) + b"\0", b"aaaa"), DIST_FAR),
        "output_past_isize": (zmember(d, 6, isize=5), OUTPUT),
        "crc": (zmember(d, 6, crc=zlib.crc32(d) ^ 1), CRC),
        "isize": (zmember(d, 6, isize=len(d) + 1), ISIZE),
    }
    return cases


def _rev(v, n):
    return int(format(v, f"0{n}b")[::-1], 2)


def test_malformed_members(host_inflate):
    cases = malformed_cases()
    got = run_host(host_inflate, [m for m, _ in cases.values()])
    for (name, (m, code)), (rc, at, _) in zip(cases.items(), got):
        assert name == "no_bc" or zlib_of(m) is None, f"{name}: zlib accepts the member"   # gzip needs no BC field
        assert rc == -code and at == 0, f"{name}: code {-rc}, want {code}"


def test_every_truncation_and_bit_flip(host_inflate):
    two = zmember(b"the quick brown fox " * 20, 6) + zmember(bytes(range(256)) * 2, 9, zlib.Z_FIXED)
    one = zmember(b"ACGTTGCA" * 40 + b"NNNN" * 10, 6)
    inputs = [two[:k] for k in range(1, len(two))]
    for i in range(len(one) * 8):
        b = bytearray(one)
        b[i >> 3] ^= 1 << (i & 7)
        inputs.append(bytes(b))
    got = run_host(host_inflate, inputs)
    first = len(_split(two)[0])
    for k, (rc, at, out) in enumerate(got[:len(two) - 1]):
        cut = k + 1
        if cut == first:
            assert rc >= 0 and out == zlib_of(two[:first]), "a cut at a member boundary is a whole member"
        else:
            assert rc < 0 and at == (0 if cut < first else first), f"truncation at {cut}: {rc}"
    for i, (rc, at, out) in enumerate(got[len(two) - 1:]):
        if rc >= 0:
            assert out == zlib_of(inputs[len(two) - 1 + i]), f"bit {i}: accepted bytes differ from zlib's"


# ---- BAM files made in Python ----

def bam_record(name, flag, rid, pos, cigar=(), seq=b"", mapq=60, nrid=-1, npos=-1, tlen=0, bin_=4680, tags=b""):
    cig = b"".join(struct.pack("<I", n << 4 | "MIDNSHP=X".index(op)) for op, n in cigar)
    nt = {c: i for i, c in enumerate(b"=ACMGRSVTWYHKDBN")}
    s = bytes(((nt[seq[i]] << 4) | (nt[seq[i + 1]] if i + 1 < len(seq) else 0)) for i in range(0, len(seq), 2))
    body = struct.pack("<iiBBHHHiiii", rid, pos, len(name) + 1, mapq, bin_, len(cigar), flag, len(seq), nrid, npos, tlen) + \
        name + b"\0" + cig + s + b"\x1e" * len(seq) + tags
    return struct.pack("<i", len(body)) + body


def bam_file(text: bytes, refs, records, level=6, cut=CHUNK, eof=True) -> bytes:
    raw = b"BAM\1" + struct.pack("<i", len(text)) + text + struct.pack("<i", len(refs))
    for name, ln in refs:
        raw += struct.pack("<i", len(name) + 1) + name + b"\0" + struct.pack("<i", ln)
    raw += b"".join(records)
    return zmembers(raw, level, cut=cut) + (EOF_BLOCK if eof else b"")


REFS = [(b"chr1", 50000), (b"chr2", 40000)]
HDR = b"@HD\tVN:1.6\tSO:coordinate\n@SQ\tSN:chr1\tLN:50000\n@SQ\tSN:chr2\tLN:40000\n"


def _merge_cli(tmp_path, files, out="m.bam"):
    o = tmp_path / out
    r = subprocess.run([CLI, "merge", "-o", str(o)] + [str(f) for f in files], capture_output=True, text=True)
    return r, o


@pytest.mark.parametrize("case", ["no_inputs", "not_bgzf", "not_bam", "sq_differ", "rg_clash", "truncated_header"])
def test_cli_refusals(tmp_path, case):
    a = tmp_path / "a.bam"
    a.write_bytes(bam_file(HDR + b"@RG\tID:x\tSM:one\n", REFS, [bam_record(b"r1", 0, 0, 10, [("M", 5)], b"ACGTA")]))
    b = tmp_path / "b.bam"
    if case == "not_bgzf":
        b.write_bytes(b"@HD\tVN:1.6\n" * 4)
    elif case == "not_bam":
        b.write_bytes(zmembers(b"CRAM" + bytes(100)) + EOF_BLOCK)
    elif case == "sq_differ":
        b.write_bytes(bam_file(HDR, [(b"chr1", 50000), (b"chr2", 40001)], []))
    elif case == "truncated_header":
        full = bam_file(HDR, REFS, [], level=0)
        b.write_bytes(full[:len(full) // 2])
    else:
        b.write_bytes(bam_file(HDR + b"@RG\tID:x\tSM:two\n", REFS, []))
    r, o = _merge_cli(tmp_path, [] if case == "no_inputs" else [a, b])
    assert r.returncode != 0, r.stderr
    assert not o.exists()
    if case == "no_inputs":
        assert "specify" in r.stderr
    else:
        assert str(b) in r.stderr, r.stderr
    want = {"not_bgzf": "not a BGZF file", "not_bam": "not a BAM file", "sq_differ": "reference 1", "rg_clash": "@RG ID:x",
            "truncated_header": "BGZF member at byte offset 0: truncated member"}
    if case in want:
        assert want[case] in r.stderr, r.stderr


@pytest.fixture(scope="module")
def host_rows(tmp_path_factory):
    so = tmp_path_factory.mktemp("bam_row") / "bam_row_host.so"
    subprocess.run(["g++", "-O1", "-g", "-shared", "-fPIC", "-fsanitize=address,undefined", "-fno-sanitize-recover=all",
                    os.path.join(ROOT, "tests", "bam_row_host", "bam_row_host.cpp"), "-o", str(so)], check=True)
    return str(so)


# the row refusals (bam_row.cuh)
ROW_NAME, ROW_FIELDS, ROW_REFID, ROW_POS, ROW_END = range(1, 6)

_ROW_RUNNER = r"""
import ctypes as C, sys, json
class Key(C.Structure):
    _fields_ = [("key", C.c_uint64), ("end", C.c_uint32), ("len", C.c_uint32), ("bin", C.c_uint16), ("unmapped", C.c_uint16), ("pad", C.c_uint32)]
L = C.CDLL(sys.argv[1])
lens = (C.c_int32 * 2)(50000, 40000)
out = []
for h in json.loads(sys.stdin.read()):
    r = bytes.fromhex(h)
    k = Key()
    why = L.bam_row_host(r, 2, lens, C.byref(k))
    out.append([why, k.key, k.end, k.len, k.bin, k.unmapped])
print(json.dumps(out))
"""


def row_cases():
    """(record, expected reason or the accepted row (key, end, bin, unmapped)) on REFS: chr1 50 000 bp, chr2 40 000 bp"""
    from test_bam_sort import spec_reg2bin
    no_name = bytearray(bam_record(b"r", 0, 0, 10, [("M", 5)], b"ACGTA"))
    no_name[12] = 0
    over = bytearray(bam_record(b"r", 0, 0, 10, [("M", 5)], b"ACGTA"))
    over[16] = 3   # three CIGAR operations where there is one
    return [
        (bam_record(b"ok", 16, 1, 100, [("S", 3), ("M", 40), ("N", 500), ("D", 2), ("M", 10), ("H", 4)], b"A" * 53),
         (1 << 32 | 101 << 1 | 1, 652, spec_reg2bin(100, 652), 0)),
        (bam_record(b"last_base", 0, 0, 49990, [("M", 10)], b"A" * 10), (49991 << 1, 50000, spec_reg2bin(49990, 50000), 0)),
        (bam_record(b"placed_unmapped", 4, 1, 39999, [("M", 10)], b"A" * 10), (1 << 32 | 40000 << 1, 40000, spec_reg2bin(39999, 40000), 1)),
        (bam_record(b"unplaced", 4, -1, -1, [], b"ACG"), (0xffffffff << 32, 0, 4680, 1)),
        (bytes(no_name), ROW_NAME),
        (bytes(over), ROW_FIELDS),
        (bam_record(b"r", 0, 2, 10, [("M", 5)], b"ACGTA"), ROW_REFID),
        (bam_record(b"r", 0, -2, 10, [("M", 5)], b"ACGTA"), ROW_REFID),
        (bam_record(b"mapped_pos_-1", 0, 0, -1, [("M", 10)], b"A" * 10), ROW_POS),
        (bam_record(b"pos_ln", 4, 1, 40000, [], b"A"), ROW_POS),
        (bam_record(b"pos_2^31-1", 0, 1, 0x7fffffff, [("M", 1)], b"A"), ROW_POS),
        (bam_record(b"unplaced_2^31-1", 4, -1, 0x7fffffff, [], b"A"), ROW_POS),
        (bam_record(b"unplaced_-2", 4, -1, -2, [], b"A"), ROW_POS),
        (bam_record(b"end_past_ln", 0, 0, 49990, [("M", 11)], b"A" * 11), ROW_END),
        (bam_record(b"huge_cigar", 0, 0, 10, [("N", (1 << 28) - 1)] * 20, b""), ROW_END),
    ]


def test_record_rows_and_refusals(host_rows):
    """the rows merge builds from records read from a file, and the refusals that keep the index's refID and window indices
    in range: a mapped record at POS -1, POS 2^31 - 1 (whose POS + 1 would carry into the refID bits), POS past LN, an end
    past LN"""
    import json
    cases = row_cases()
    asan = subprocess.run(["g++", "-print-file-name=libasan.so"], capture_output=True, text=True).stdout.strip()
    ubsan = subprocess.run(["g++", "-print-file-name=libubsan.so"], capture_output=True, text=True).stdout.strip()
    env = dict(os.environ, LD_PRELOAD=f"{asan} {ubsan}", ASAN_OPTIONS="detect_leaks=0:abort_on_error=1", UBSAN_OPTIONS="halt_on_error=1")
    import sysconfig
    r = subprocess.run([sysconfig.get_config_var("BINDIR") + "/python3", "-c", _ROW_RUNNER, host_rows], input=json.dumps([c.hex() for c, _ in cases]),
                       capture_output=True, text=True, env=env)
    assert r.returncode == 0, r.stderr[-2000:]
    for (rec, want), (why, key, end, ln, b, unm) in zip(cases, json.loads(r.stdout)):
        name = rec[36:36 + rec[12] - 1] if rec[12] else b"no_name"
        if isinstance(want, int):
            assert why == want, (name, why, want)
        else:
            assert why == 0, (name, why)
            assert (key, end, b, unm) == want and ln == len(rec), (name, (key, end, b, unm), want)


def test_merged_header_rules(tmp_path):
    """SO:coordinate set on @HD (or an @HD added), new @RG and @PG IDs appended, known @PG IDs dropped, @CO appended; an
    already sorted single input keeps its text byte for byte"""
    import ema_b200
    f = []
    texts = [b"@HD\tVN:1.6\tSO:unsorted\tGO:none\n@SQ\tSN:chr1\tLN:50000\n@SQ\tSN:chr2\tLN:40000\n@RG\tID:a\tSM:s\n@PG\tID:ema\tPN:ema\n",
             b"@SQ\tSN:chr1\tLN:50000\n@SQ\tSN:chr2\tLN:40000\n@RG\tID:a\tSM:s\n@RG\tID:b\tSM:t\n@PG\tID:ema\tPN:other\n@PG\tID:bwa\tPN:bwa\n@CO\thello\n",
             b"@SQ\tSN:chr1\tLN:50000\n@SQ\tSN:chr2\tLN:40000\n"]
    for k, t in enumerate(texts):
        p = tmp_path / f"h{k}.bam"
        p.write_bytes(bam_file(t, REFS, []))
        f.append(str(p))
    got = ema_b200.bam_merge_header(f)
    assert got == (b"@HD\tVN:1.6\tSO:coordinate\tGO:none\n@SQ\tSN:chr1\tLN:50000\n@SQ\tSN:chr2\tLN:40000\n@RG\tID:a\tSM:s\n"
                   b"@PG\tID:ema\tPN:ema\n@RG\tID:b\tSM:t\n@PG\tID:bwa\tPN:bwa\n@CO\thello\n")
    assert ema_b200.bam_merge_header([f[2]]).startswith(b"@HD\tVN:1.6\tSO:coordinate\n@SQ")
    p = tmp_path / "sorted.bam"
    p.write_bytes(bam_file(HDR + b"\0\0\0", REFS, []))
    assert ema_b200.bam_merge_header([str(p)]) == HDR + b"\0\0\0"


# ---- GPU ----

@pytest.mark.gpu
def test_device_decoder(host_encoder, tmp_path):
    """emab_bgzf_inflate equals zlib on the valid member sets, on a whole -O bam run of a 40 000-pair bucket recompressed at level 6, and names
    the offset and reason of a bad member"""
    import ema_b200
    from test_bam import _data
    ctx = ema_b200.Context()
    for name, data in valid_cases(host_encoder).items():
        assert ema_b200.bgzf_inflate(ctx, data) == b"".join(zlib_of(m) for m in _split(data)), name
    import ema_b200 as E
    from tools import synth
    p = synth.build_config("c1_rep", helpers.DATA_ROOT, indexer=E.index_build, n_barcodes=800, tag="_40k")   # 800 x 50 pairs
    assert sum(1 for _ in open(p["bucket"], "rb")) == 40000
    out = tmp_path / "big.bam"
    subprocess.run([CLI, "align", "-O", "bam", "-s", p["bucket"], "-r", p["fasta"], "-p", "10x", "-t", "8", "-o", str(out)], check=True,
                   stderr=subprocess.DEVNULL)
    raw = b"".join(zlib_of(m) for m in _split(out.read_bytes()))
    big = zmembers(raw, 6)
    assert len(raw) > 10 << 20
    assert ema_b200.bgzf_inflate(ctx, big) == raw
    good = zmember(b"hello hello hello", 6)
    bad = malformed_cases()
    for name, (m, _code) in [("truncated", (big[:len(big) // 2], None)), ("crc", bad["crc"]), ("block_type_3", bad["block_type_3"]),
                              ("dist_far", bad["dist_far"])]:
        with pytest.raises(ema_b200.EmabError) as e:
            ema_b200.bgzf_inflate(ctx, good + m)
        at = len(good) + (max(o for o in _offsets(big) if o <= len(big) // 2) if name == "truncated" else 0)
        assert f"byte offset {at}:" in str(e.value), (name, str(e.value))


def _offsets(data):
    out, o = [], 0
    for m in _split_partial(data):
        out.append(o)
        o += m
    return out


def _split_partial(data):
    o = 0
    while o + 18 <= len(data):
        bs = struct.unpack_from("<H", data, o + 16)[0]
        yield bs + 1
        o += bs + 1


def _sorted_run(tmp_path, args, tag, env=None):
    from test_bam_sort import _cli_sorted_pair
    return _cli_sorted_pair(args, tmp_path, env=env, tag=tag)


def _merge(paths, tmp_path, tag, env=None):
    out = tmp_path / f"merged{tag}.bam"
    r = subprocess.run([CLI, "merge", "-o", str(out)] + [str(p) for p in paths], capture_output=True, text=True, env=env)
    assert r.returncode == 0, r.stderr[-2000:]
    return out.read_bytes(), (tmp_path / f"merged{tag}.bam.bai").read_bytes()


def _records(data: bytes):
    """(header text, [raw records]) of a BAM file"""
    from test_bam_sort import header_len
    raw = b"".join(zlib_of(m) for m in _split(data))
    hl, _ = header_len(raw)
    recs, o = [], hl
    while o < len(raw):
        bs, = struct.unpack_from("<i", raw, o)
        recs.append(raw[o:o + 4 + bs])
        o += 4 + bs
    return raw[8:8 + struct.unpack_from("<i", raw, 4)[0]], recs


def _key(r):
    rid, pos = struct.unpack_from("<ii", r, 4)
    flag, = struct.unpack_from("<H", r, 18)
    return (rid & 0xffffffff) << 32 | (pos + 1) << 1 | (1 if flag & 16 else 0)


def _restated_bai(data: bytes):
    """the .bai write_bai gives for this file, with every bin recomputed from POS and the CIGAR"""
    from test_bam_sort import CHUNK as _C, layout, header_len, spec_reg2bin, write_bai
    offs, sizes, raw = layout(data[:-len(EOF_BLOCK)])
    hl, n_ref = header_len(raw)
    k0, acc = 0, 0
    while acc < hl:
        acc += sizes[k0]
        k0 += 1
    body_offs = offs[k0:] + [len(data) - len(EOF_BLOCK)]

    def voff(u):
        m = u // _C
        return body_offs[m] << 16 | (u - m * _C)
    placed, n_no, o, after = [], 0, hl, None
    while o < len(raw):
        bs, rid, pos, lrn, _mq, _b, ncig, flag = struct.unpack_from("<iiiBBHHH", raw, o)
        cig = struct.unpack_from(f"<{ncig}I", raw, o + 36 + lrn)
        unm = 1 if flag & 4 else 0
        rl = 0 if unm else sum(c >> 4 for c in cig if c & 15 in (0, 2, 3, 7, 8))
        if rid >= 0:
            end = pos + (rl if rl else 1)
            placed.append((rid, pos, end, spec_reg2bin(pos, end), unm, voff(o - hl)))
        else:
            n_no += 1
            if after is None:
                after = voff(o - hl)
        o += 4 + bs
    return write_bai(n_ref, placed, after if after is not None else voff(len(raw) - hl), n_no)


@pytest.mark.gpu
def test_merge_one_file_is_identity(tmp_path):
    """merge of one `align -O bam -S -o` output reproduces the file and its .bai byte for byte"""
    from test_bam import _data
    p = _data("c1")
    q = _data("c1_rep")
    lines = [l for l in open(q["bucket"], "rb").read().split(b"\n") if l]
    r = random.Random(5)   # every seventh pair with a random second read: unmapped mates
    fl = [l.split(b" ") for l in lines]
    for f in fl[::7]:
        f[4] = bytes(r.choice(b"ACGT") for _ in f[4])
    (tmp_path / "unmapped").write_bytes(b"\n".join(b" ".join(f) for f in fl) + b"\n")
    cases = [(["align", "-s", p["bucket"], "-r", p["fasta"]], "c1"), (["align", "-s", q["bucket"], "-r", q["fasta"]], "rep"),
             (["align", "-s", str(tmp_path / "unmapped"), "-r", q["fasta"]], "unm"),
             (["align", "-s", q["bucket"], "-r", q["fasta"], "-R", "@RG\\tID:rg7\\tSM:s", "-i", "7"], "rg")]
    for args, tag in cases:
        _, s, bai = _sorted_run(tmp_path, args + ["-p", "10x", "-t", "8"], tag)
        got, gbai = _merge([tmp_path / f"s{tag}.bam"], tmp_path, tag)
        assert got == s, tag
        assert gbai == bai, tag


def _four_way(tmp_path):
    """a c1_rep bucket split four ways and sorted piece by piece, plus a streamed -1/-2 run on the same reference"""
    from test_bam import _data
    p = _data("c1_rep")
    lines = [l for l in open(p["bucket"], "rb").read().split(b"\n") if l]
    files = []
    for i in range(4):
        f = tmp_path / f"b{i}"
        f.write_bytes(b"\n".join(lines[i::4]) + b"\n")
        _sorted_run(tmp_path, ["align", "-s", str(f), "-r", p["fasta"], "-p", "10x", "-t", "8"], f"p{i}")
        files.append(tmp_path / f"sp{i}.bam")
    q = _data("c1_rep", "tru")
    fq = open(q["bucket"], "rb").read().split(b"\n")
    recs = [b"\n".join(fq[i:i + 4]) + b"\n" for i in range(0, len(fq) - 3, 4)]
    (tmp_path / "r1.fq").write_bytes(b"".join(recs[0::2]))
    (tmp_path / "r2.fq").write_bytes(b"".join(recs[1::2]))
    _sorted_run(tmp_path, ["align", "-1", str(tmp_path / "r1.fq"), "-2", str(tmp_path / "r2.fq"), "-r", q["fasta"], "-p", "tru", "-t", "6"], "fq",
                env=dict(os.environ, EMAB_FASTQ_BATCH="700"))
    files.append(tmp_path / "sfq.bam")
    return files


def _check_merged(files, got, gbai):
    want = sorted([r for f in files for r in _records(f.read_bytes())[1]], key=_key)   # stable: argument order, then file order
    text, recs = _records(got)
    assert recs == want
    assert text.startswith(b"@HD\tVN:1.3\tSO:coordinate\n")
    assert gbai == _restated_bai(got)
    _regions_match_scan(got, gbai)


def _regions_match_scan(data: bytes, bai: bytes):
    """independent of the index's rules (as test_index_finds_what_a_scan_finds): regions looked up through bins, chunks and
    the linear lower bound give the records a brute-force scan of the file gives"""
    import bisect
    from test_bam_sort import CHUNK as _C, layout, header_len, read_bai, spec_reg2bins, _regions
    offs, sizes, raw = layout(data[:-len(EOF_BLOCK)])
    hl, n_ref = header_len(raw)
    k0, acc = 0, 0
    while acc < hl:
        acc += sizes[k0]
        k0 += 1
    body_offs = offs[k0:] + [len(data) - len(EOF_BLOCK)]
    lens, o = [], 8 + struct.unpack_from("<i", raw, 4)[0] + 4
    for _ in range(n_ref):
        ln, = struct.unpack_from("<i", raw, o)
        lens.append(struct.unpack_from("<i", raw, o + 4 + ln)[0])
        o += 8 + ln
    allrecs, o = [], hl
    while o < len(raw):
        bs, rid, pos, lrn, _mq, _b, ncig, flag = struct.unpack_from("<iiiBBHHH", raw, o)
        cig = struct.unpack_from(f"<{ncig}I", raw, o + 36 + lrn)
        rl = 0 if flag & 4 else sum(c >> 4 for c in cig if c & 15 in (0, 2, 3, 7, 8))
        m = (o - hl) // _C
        allrecs.append((rid, pos, pos + (rl if rl else 1), body_offs[m] << 16 | (o - hl - m * _C)))
        o += 4 + bs
    refs, _ = read_bai(bai)
    starts = [x[3] for x in allrecs]
    by_voff = {v: k for k, v in enumerate(starts)}
    rng = random.Random(29)
    looked = 0
    for r in range(n_ref):
        bins, _pseudo, lin = refs[r]
        mine = [k for k, x in enumerate(allrecs) if x[0] == r]
        for beg, end in _regions(rng, lens[r], len(lin))[:120]:
            want = {k for k in mine if allrecs[k][1] < end and allrecs[k][2] > beg}
            lo = lin[beg >> 14] if (beg >> 14) < len(lin) else None
            got = set()
            for b in spec_reg2bins(beg, end):
                for cb, ce in bins.get(b, []):
                    if lo is not None and ce <= lo:
                        continue
                    for i in range(bisect.bisect_left(starts, cb), bisect.bisect_left(starts, ce)):
                        x = allrecs[by_voff[starts[i]]]
                        if x[0] == r and x[1] < end and x[2] > beg:
                            got.add(by_voff[starts[i]])
            assert got == want, (r, beg, end)
            looked += 1
    assert looked > 100


@pytest.mark.gpu
def test_merge_several_inputs_budget_and_recompression(tmp_path):
    files = _four_way(tmp_path)
    got, gbai = _merge(files, tmp_path, "4")
    _check_merged(files, got, gbai)
    # an input listed twice: its records twice, ties in argument order
    got2, gbai2 = _merge(files + [files[0]], tmp_path, "dup")
    _check_merged(files + [files[0]], got2, gbai2)
    # small budgets, down to one record per block: the same bytes
    for budget in (200000, 3000):
        b, i = _merge(files, tmp_path, f"b{budget}", env=dict(os.environ, EMAB_SORT_HOST_BYTES=str(budget)))
        assert b == got and i == gbai, budget
    # the inputs recompressed by zlib with members of random sizes that cut records and the header anywhere
    r = random.Random(3)
    for level, strategy in ((0, zlib.Z_DEFAULT_STRATEGY), (1, zlib.Z_DEFAULT_STRATEGY), (6, zlib.Z_DEFAULT_STRATEGY),
                            (9, zlib.Z_DEFAULT_STRATEGY), (6, zlib.Z_FIXED)):
        re = []
        for k, f in enumerate(files):
            raw = b"".join(zlib_of(m) for m in _split(f.read_bytes()))
            out, o = b"", 0
            while o < len(raw):
                n = r.randint(1, 65280)
                out += zmember(raw[o:o + n], level, strategy)
                o += n
            g = tmp_path / f"z{level}_{strategy}_{k}.bam"
            g.write_bytes(out + EOF_BLOCK)
            re.append(g)
        b, i = _merge(re, tmp_path, f"z{level}{strategy}")
        assert b == got and i == gbai, (level, strategy)


@pytest.mark.gpu
def test_merge_foreign_bam(tmp_path):
    """a BAM written in Python (standing in for a bwa mem BAM of the no-barcode reads): unpaired and paired flags, no BX,
    CIGARs with N, D, S and H, records ending at a contig's last base, placed-unmapped and unplaced records, stale bins.
    Merged with an EMA output: the restatement's records (verbatim) and index (recomputed bins)."""
    from test_bam import _data
    p = _data("c1_rep")
    _, s, _ = _sorted_run(tmp_path, ["align", "-s", p["bucket"], "-r", p["fasta"], "-p", "10x", "-t", "8"], "ema")
    text, _ = _records(s)
    from test_bam_sort import layout, header_len
    raw = layout(s[:-len(EOF_BLOCK)])[2]
    hl, n_ref = header_len(raw)
    o, refs = 8 + struct.unpack_from("<i", raw, 4)[0] + 4, []
    for _ in range(n_ref):
        ln, = struct.unpack_from("<i", raw, o)
        refs.append((raw[o + 4:o + 3 + ln], struct.unpack_from("<i", raw, o + 4 + ln)[0]))
        o += 8 + ln
    rng = random.Random(17)
    recs = []
    for rid, (name, ln) in enumerate(refs):
        for k in range(60):
            pos = rng.randrange(0, ln - 300)
            cig = rng.choice([[("M", 100)], [("S", 5), ("M", 40), ("N", 1000), ("M", 55)], [("H", 7), ("M", 30), ("D", 4), ("M", 70)],
                              [("M", 50), ("I", 2), ("M", 48)]])
            cig = [(op, n) if op != "N" else (op, min(n, ln - pos - 200)) for op, n in cig]
            qlen = sum(n for op, n in cig if op in "MIS=X")
            flag = rng.choice([0, 16, 1 | 2 | 64 | 32, 1 | 2 | 128 | 16])
            recs.append((rid, pos, flag, cig, qlen))
        recs.append((rid, ln - 100, 0, [("M", 100)], 100))   # ends at the contig's last base
        recs.append((rid, ln // 2, 4 | 1 | 128, [], 50))     # placed, unmapped
    recs.sort(key=lambda x: (x[0], x[1], 1 if x[2] & 16 else 0))
    body = [bam_record(b"nobc%d" % i, fl, rid, pos, cig, b"ACGT" * (q // 4) + b"A" * (q % 4), bin_=1234 if i % 3 else 4680)
            for i, (rid, pos, fl, cig, q) in enumerate(recs)]
    body += [bam_record(b"unpl%d" % i, 4 | 1 | 8 | 64, -1, -1, [], b"ACGTAC") for i in range(5)]
    foreign = tmp_path / "nobc.bam"
    foreign.write_bytes(bam_file(b"@HD\tVN:1.6\tSO:coordinate\n" + b"".join(b"@SQ\tSN:%s\tLN:%d\n" % r for r in refs) +
                                 b"@PG\tID:bwa\tPN:bwa\tVN:0.7.17\n", refs, body))
    files = [tmp_path / "sema.bam", foreign]
    got, gbai = _merge(files, tmp_path, "f")
    want = sorted([r for f in files for r in _records(f.read_bytes())[1]], key=_key)
    mtext, mrecs = _records(got)
    assert mrecs == want
    assert mtext == text + b"@PG\tID:bwa\tPN:bwa\tVN:0.7.17\n"
    assert gbai == _restated_bai(got)
    _regions_match_scan(got, gbai)


@pytest.mark.gpu
def test_merge_refuses_unsorted(tmp_path):
    from test_bam import _data
    p = _data("c1")
    u = tmp_path / "u.bam"
    subprocess.run([CLI, "align", "-O", "bam", "-s", p["bucket"], "-r", p["fasta"], "-p", "10x", "-t", "8", "-o", str(u)], check=True,
                   stderr=subprocess.DEVNULL)
    recs = _records(u.read_bytes())[1]
    first_bad = next(i for i in range(1, len(recs)) if _key(recs[i]) < _key(recs[i - 1]))
    r, o = _merge_cli(tmp_path, [u])
    assert r.returncode != 0 and not o.exists() and not (tmp_path / "m.bam.bai").exists()
    assert f"{u}: record {first_bad}: not coordinate-sorted" in r.stderr, r.stderr


@pytest.mark.gpu
def test_records_cut_across_reads_at_small_budgets(tmp_path):
    """inputs recompressed into members of 1 to 300 bytes, merged at budgets of a few hundred bytes per input: a block
    often holds no whole record, and a record's bytes are carried over several reads.  Same file and .bai as the
    originals' merge at the default budget."""
    g = os.path.join(ROOT, "tests", "golden", "tiny_rep")
    lines = [l for l in open(os.path.join(g, "ema-bin-000.10x"), "rb").read().split(b"\n") if l]
    files = []
    for i in range(2):
        f = tmp_path / f"t{i}"
        f.write_bytes(b"\n".join(lines[i::2]) + b"\n")
        _sorted_run(tmp_path, ["align", "-s", str(f), "-r", os.path.join(g, "ref.fa"), "-p", "10x", "-t", "4"], f"t{i}")
        files.append(tmp_path / f"st{i}.bam")
    got, gbai = _merge(files, tmp_path, "t")
    _check_merged(files, got, gbai)
    r = random.Random(11)
    small = []
    for k, f in enumerate(files):
        raw = b"".join(zlib_of(m) for m in _split(f.read_bytes()))
        out, o = b"", 0
        while o < len(raw):
            n = r.randint(1, 300)
            out += zmember(raw[o:o + n], r.choice([0, 1, 6]))
            o += n
        p = tmp_path / f"small{k}.bam"
        p.write_bytes(out + EOF_BLOCK)
        small.append(p)
    for budget in (None, 20000, 3000):
        env = dict(os.environ, EMAB_SORT_HOST_BYTES=str(budget)) if budget else None
        b, i = _merge(small, tmp_path, f"s{budget}", env=env)
        assert b == got and i == gbai, budget


def _refs_of(data: bytes):
    raw = b"".join(zlib_of(m) for m in _split(data))
    o, refs = 8 + struct.unpack_from("<i", raw, 4)[0], []
    n_ref, = struct.unpack_from("<i", raw, o)
    o += 4
    for _ in range(n_ref):
        ln, = struct.unpack_from("<i", raw, o)
        refs.append((raw[o + 4:o + 3 + ln], struct.unpack_from("<i", raw, o + 4 + ln)[0]))
        o += 8 + ln
    return refs


@pytest.mark.gpu
def test_merge_record_refusals_and_file_ends(tmp_path):
    """records whose rows would index the BAI's arrays out of range are refused with the file and ordinal and leave no
    output; a file without the EOF block merges with a warning; a truncated last member is an error naming its offset"""
    good = [bam_record(b"a%d" % i, 0, 0, 100 * i, [("M", 50)], b"A" * 50) for i in range(1, 6)]
    for name, bad in (("pos_-1", bam_record(b"x", 0, 0, -1, [("M", 20)], b"A" * 20)),
                      ("pos_2^31-1", bam_record(b"x", 0, 1, 0x7fffffff, [("M", 1)], b"A")),
                      ("end_past_ln", bam_record(b"x", 0, 1, 39990, [("M", 20)], b"A" * 20))):
        recs = good[:3] + [bad] if name != "pos_-1" else [bad] + good
        f = tmp_path / f"{name}.bam"
        f.write_bytes(bam_file(HDR, REFS, recs))
        r, o = _merge_cli(tmp_path, [f])
        ordinal = 0 if name == "pos_-1" else 3
        assert r.returncode != 0 and not o.exists() and not (tmp_path / "m.bam.bai").exists(), (name, r.stderr)
        assert f"{f}: record {ordinal}:" in r.stderr and ("POS outside" in r.stderr or "past its reference" in r.stderr), (name, r.stderr)
    ok = tmp_path / "ok.bam"
    ok.write_bytes(bam_file(HDR, REFS, good))
    no_eof = tmp_path / "no_eof.bam"
    no_eof.write_bytes(bam_file(HDR, REFS, good, eof=False))
    r, o = _merge_cli(tmp_path, [ok, no_eof], "w.bam")
    assert r.returncode == 0, r.stderr
    assert f"warning: {no_eof} has no EOF block" in r.stderr and f"{ok} has no EOF" not in r.stderr
    assert _records(o.read_bytes())[1] == sorted(2 * good, key=_key)
    body = bam_file(HDR, REFS, good, cut=200, eof=False)
    last = _offsets(body)[-1]
    cut = tmp_path / "cut.bam"
    cut.write_bytes(body[:-5])
    r, o = _merge_cli(tmp_path, [ok, cut], "c.bam")
    assert r.returncode != 0 and not o.exists()
    assert f"{cut}: BGZF member at byte offset {last}: truncated member" in r.stderr, r.stderr

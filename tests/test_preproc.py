"""CPU tests (-m "not gpu"): `ema-b200 count` / `preproc` (host/preproc.cpp) against the reference binary (oracle/_ref/ema) on a
synthetic raw 10x FASTQ — whitelisted barcodes, one- and two-base errors with matching low qualities, N bases, barcodes not
on the list, short reads, a quality character below '!'.  Every output file must be byte-identical: the census (.ema-ncnt in
the reference's hash-map order, .ema-fcnt incl. block dumps), every ema-bin-NNN and ema-nobc, with and without -h / -b.
Where oracle/_ref is not built, the reference's files are represented by their recorded digests (tests/golden/reference)."""
import filecmp
import os
import subprocess

import numpy as np
import pytest

import helpers

CLI = os.path.join(helpers.ROOT, "ema_b200", "ema-b200")
REF = helpers.ref_bin("ema")
HAVE_REF = os.path.exists(REF)
ACGT = np.frombuffer(b"ACGT", dtype=np.uint8)


def make_raw_fastq(path, wl_path, n_pairs=6000, n_wl=400, n_used=60, seed=7):
    rng = np.random.default_rng(seed)
    wl = set()
    while len(wl) < n_wl:
        bc = rng.integers(0, 4, 16)
        if bc.any():
            wl.add(bytes(ACGT[bc]))
    wl = sorted(wl)
    order = rng.permutation(len(wl))
    with open(wl_path, "wb") as f:
        for i in order:
            f.write(wl[i] + b"\n")
    used = [wl[i] for i in order[:n_used]]
    with open(path, "wb") as f:
        for i in range(n_pairs):
            bc = bytearray(used[int(rng.integers(0, n_used))])
            qual = bytearray(b"I" * 16)
            kind = rng.random()
            if kind < 0.10:      # one substitution, low quality there
                k = int(rng.integers(0, 16)); bc[k] = b"ACGT"[(b"ACGT".index(bc[k]) + int(rng.integers(1, 4))) % 4]; qual[k] = ord("#") + int(rng.integers(0, 8))
            elif kind < 0.14:    # two substitutions
                for k in rng.choice(16, 2, replace=False):
                    bc[k] = b"ACGT"[(b"ACGT".index(bc[k]) + int(rng.integers(1, 4))) % 4]; qual[k] = ord("#") + int(rng.integers(0, 5))
            elif kind < 0.18:    # an N
                k = int(rng.integers(0, 16)); bc[k] = ord("N"); qual[k] = ord("#")
            elif kind < 0.20:    # two Ns
                for k in rng.choice(16, 2, replace=False):
                    bc[k] = ord("N"); qual[k] = ord("#")
            elif kind < 0.25:    # not on the list
                bc = bytearray(ACGT[rng.integers(0, 4, 16)].tobytes())
            elif kind < 0.27:    # substitution with HIGH quality (should not be corrected confidently when ambiguous)
                k = int(rng.integers(0, 16)); bc[k] = b"ACGT"[(b"ACGT".index(bc[k]) + 1) % 4]
            l1 = 16 + 7 + int(rng.integers(90, 128)) if rng.random() > 0.02 else int(rng.integers(5, 31))   # some reads too short
            r1 = bytes(bc) + ACGT[rng.integers(0, 4, max(0, l1 - 16))].tobytes()
            r1 = r1[:l1]
            q1 = (bytes(qual) + bytes(rng.integers(35, 75, max(0, l1 - 16)).astype(np.uint8)))[:l1]
            if rng.random() < 0.003 and l1 > 20:
                q1 = q1[:3] + b" " + q1[4:]      # a quality character below '!': the read is ignored
            if rng.random() < 0.01 and l1 > 20:
                q1 = q1[:5] + b"~" + q1[6:]      # above the cap: trimmed to 'B'
            l2 = int(rng.integers(100, 151))
            r2 = ACGT[rng.integers(0, 4, l2)].tobytes()
            q2 = bytes(rng.integers(35, 75, l2).astype(np.uint8))
            extra = b" 1:N:0:1" if i % 3 == 0 else b""
            f.write(b"@read%d%s\n%s\n+\n%s\n@read%d%s\n%s\n+\n%s\n" % (i, extra, r1, q1, i, extra.replace(b"1:N", b"2:N"), r2, q2))
    return wl_path


def run(cmd, stdin_path, cwd=None):
    with open(stdin_path, "rb") as fin:
        subprocess.run(cmd, stdin=fin, check=True, stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL, cwd=cwd)


@pytest.fixture(scope="module")
def raw(tmp_path_factory):
    if not os.path.exists(CLI):
        subprocess.run(["make", "-s", "-C", os.path.join(helpers.ROOT, "ema_b200", "csrc")], check=True)
    d = tmp_path_factory.mktemp("raw")
    fq, wl = str(d / "reads.fq"), str(d / "wl.txt")
    make_raw_fastq(fq, wl)
    return d, fq, wl


def same_as_reference(key, ours, ref=None):
    """this build's files {name: path} against the reference's files of the same names ({name: path}, where it ran) or,
    without oracle/_ref, against the recorded digests of the reference's files for case `key`"""
    assert ours
    if HAVE_REF:
        assert sorted(ref) == sorted(ours)
        for n in ours:
            assert filecmp.cmp(ref[n], ours[n], shallow=False), n
        return sorted(ours)
    names = sorted(ours)
    assert names == helpers.recorded_reference(f"{key}/names", names)
    for n in names:
        d = helpers.sha(open(ours[n], "rb").read())
        assert d == helpers.recorded_reference(f"{key}/{n}", d), n
    return names


def files(d):
    return {n: os.path.join(d, n) for n in os.listdir(d)}


def programs():
    """(tag, executable) of the runs to compare: the reference's where it is built, then this build's"""
    return ((("ref", REF),) if HAVE_REF else ()) + (("our", CLI),)


def test_count_files_identical(raw):
    d, fq, wl = raw
    for tag, exe in programs():
        run([exe, "count", "-w", wl, "-o", str(d / tag)], fq)
    exts = (".ema-ncnt", ".ema-fcnt")
    same_as_reference("count", {e: str(d / "our") + e for e in exts}, {e: str(d / "ref") + e for e in exts})
    assert os.path.getsize(str(d / "our") + ".ema-ncnt") > 8 + 12 * 30


@pytest.mark.parametrize("flags", [[], ["-h"], ["-b"], ["-h", "-t", "3", "-n", "5"]])
def test_preproc_buckets_identical(raw, flags, tmp_path):
    d, fq, wl = raw
    # the census both programs correct with: the reference's (this build's where the reference is not built; the two are
    # byte-identical, test_count_files_identical)
    census = str(d / ("ref" if HAVE_REF else "our"))
    if not os.path.exists(census + ".ema-ncnt"):
        run([REF if HAVE_REF else CLI, "count", "-w", wl, "-o", census], fq)
    n = ["-n", "7"] if "-n" not in flags else []
    for tag, exe in programs():
        run([exe, "preproc", "-w", wl, "-o", str(tmp_path / (tag + "_out"))] + n + flags + [census + ".ema-ncnt"], fq)
    names = same_as_reference("preproc" + "".join(flags), files(str(tmp_path / "our_out")),
                              files(str(tmp_path / "ref_out")) if HAVE_REF else None)
    assert "ema-nobc" in names and "ema-bin-000" in names
    assert sum(os.path.getsize(str(tmp_path / "our_out" / x)) for x in names if x.startswith("ema-bin")) > 500_000


def test_count_block_dumps(raw):
    """the full census written in several blocks (a small map budget), through the C ABI"""
    import ctypes as C
    d, fq, wl = raw
    lib = C.CDLL(os.path.join(helpers.ROOT, "ema_b200", "libema_b200.so"))
    libc = C.CDLL(None)
    libc.fopen.restype = C.c_void_p
    libc.fopen.argtypes = [C.c_char_p, C.c_char_p]
    libc.fclose.argtypes = [C.c_void_p]
    lib.emab_count.argtypes = [C.c_char_p, C.c_char_p, C.c_uint64, C.c_int, C.c_void_p]
    f = libc.fopen(fq.encode(), b"rb")
    assert lib.emab_count(wl.encode(), str(d / "blk").encode(), 72 * 400, 0, f) == 0
    libc.fclose(f)
    data = open(str(d / "blk.ema-fcnt"), "rb").read()
    blocks, pos, total = 0, 0, 0
    while pos < len(data):
        n = int.from_bytes(data[pos:pos + 8], "little"); pos += 8
        keys = [data[pos + 24 * i:pos + 24 * i + 16] for i in range(n)]
        assert keys == sorted(keys)
        total += sum(int.from_bytes(data[pos + 24 * i + 16:pos + 24 * i + 24], "little") for i in range(n))
        pos += 24 * n; blocks += 1
    assert blocks >= 3 and pos == len(data)
    # the one-block census of the same reads: the reference's, or where it is not built this build's (byte-identical to
    # the reference's, test_count_files_identical)
    tag, exe = programs()[0]
    if not os.path.exists(str(d / tag) + ".ema-fcnt"):
        run([exe, "count", "-w", wl, "-o", str(d / tag)], fq)
    ref = open(str(d / tag) + ".ema-fcnt", "rb").read()
    n = int.from_bytes(ref[:8], "little")
    assert total == sum(int.from_bytes(ref[8 + 24 * i + 16:8 + 24 * i + 24], "little") for i in range(n))


@pytest.mark.parametrize("case", ["empty", "no_final_newline", "one_pair"])
def test_preproc_edge_inputs(raw, case, tmp_path):
    """an empty stream, a last line without its newline, a single pair: same files as the reference"""
    d, fq, wl = raw
    text = open(fq, "rb").read()
    lines = text.split(b"\n")
    small = {"empty": b"", "no_final_newline": b"\n".join(lines[:8 * 50]), "one_pair": b"\n".join(lines[:8]) + b"\n"}[case]
    sfq = str(tmp_path / "s.fq")
    open(sfq, "wb").write(small)
    for tag, exe in programs():
        run([exe, "count", "-w", wl, "-o", str(tmp_path / tag)], sfq)
        run([exe, "preproc", "-w", wl, "-n", "4", "-o", str(tmp_path / (tag + "_out")), str(tmp_path / tag) + ".ema-ncnt"], sfq)
    exts = (".ema-ncnt", ".ema-fcnt")
    same_as_reference(f"edge_{case}_count", {e: str(tmp_path / "our") + e for e in exts}, {e: str(tmp_path / "ref") + e for e in exts})
    same_as_reference(f"edge_{case}_preproc", files(str(tmp_path / "our_out")), files(str(tmp_path / "ref_out")) if HAVE_REF else None)


def test_preproc_several_count_files(raw, tmp_path):
    """the census of two FASTQ halves counted separately and corrected together (`preproc ... a.ema-ncnt b.ema-ncnt`)"""
    d, fq, wl = raw
    lines = open(fq, "rb").read().split(b"\n")
    half = (len(lines) // 16) * 8
    parts = [b"\n".join(lines[:half]) + b"\n", b"\n".join(lines[half:])]
    for i, p in enumerate(parts):
        open(str(tmp_path / f"p{i}.fq"), "wb").write(p)
    for tag, exe in programs():
        for i in range(2):
            run([exe, "count", "-w", wl, "-o", str(tmp_path / f"{tag}{i}")], str(tmp_path / f"p{i}.fq"))
        run([exe, "preproc", "-w", wl, "-n", "6", "-t", "2", "-o", str(tmp_path / (tag + "_out")), str(tmp_path / f"{tag}0.ema-ncnt"), str(tmp_path / f"{tag}1.ema-ncnt")], fq)
    same_as_reference("several_count_files", files(str(tmp_path / "our_out")), files(str(tmp_path / "ref_out")) if HAVE_REF else None)


def make_haplotag_fastq(path, n_pairs=3000, seed=3):
    rng = np.random.default_rng(seed)
    tags = ["A%02dC%02dB%02dD%02d" % tuple(int(v) for v in rng.integers(1, 97, 4)) for _ in range(40)]
    with open(path, "wb") as f:
        for i in range(n_pairs):
            t = tags[int(rng.integers(0, len(tags)))]
            u = rng.random()
            if u < 0.03:
                hdr = b"@h%d" % i                                   # no tag at all
            elif u < 0.06:
                hdr = b"@h%d BX:Z:A00C00B00D00" % i                 # the "no barcode" tag: not one of the 96^4
            elif u < 0.08:
                hdr = b"@h%d RG:Z:x\tBX:Z:%s\tQX:Z:y" % (i, t.encode())   # other tags around it, tab separated
            else:
                hdr = b"@h%d BX:Z:%s" % (i, t.encode())
            l1 = int(rng.integers(100, 151)) if rng.random() > 0.02 else int(rng.integers(5, 31))
            l2 = int(rng.integers(100, 151))
            r1, r2 = ACGT[rng.integers(0, 4, l1)].tobytes(), ACGT[rng.integers(0, 4, l2)].tobytes()
            q1, q2 = bytes(rng.integers(35, 75, l1).astype(np.uint8)), bytes(rng.integers(35, 75, l2).astype(np.uint8))
            f.write(hdr + b"\n" + r1 + b"\n+\n" + q1 + b"\n" + hdr + b"\n" + r2 + b"\n+\n" + q2 + b"\n")


@pytest.mark.skipif(os.environ.get("EMAB_SLOW_TESTS") != "1", reason="builds the 96^4-entry haplotag maps four times (~2 minutes, ~6 GB); EMAB_SLOW_TESTS=1 runs it")
@pytest.mark.parametrize("flags", [[], ["-b"]])
def test_haplotag_count_and_preproc(flags, tmp_path):
    """-p: barcodes from the BX:Z: tag of the name line, all 96^4 combinations known, no correction, reads untrimmed — and
    the reference's quirks (the first pair is never bucketed, the tag is bounded by the previous pair's last line)"""
    fq = str(tmp_path / "h.fq")
    make_haplotag_fastq(fq)
    for tag, exe in programs():
        run([exe, "count", "-p", "-o", str(tmp_path / tag)], fq)
        run([exe, "preproc", "-p", "-n", "5", "-o", str(tmp_path / (tag + "_out"))] + flags + [str(tmp_path / tag) + ".ema-ncnt"], fq)
    key = "haplotag" + "".join(flags)
    same_as_reference(key + "_count", {"ncnt": str(tmp_path / "our.ema-ncnt")}, {"ncnt": str(tmp_path / "ref.ema-ncnt")})
    assert not os.path.exists(str(tmp_path / "our.ema-fcnt")) and not os.path.exists(str(tmp_path / "ref.ema-fcnt"))
    names = same_as_reference(key + "_preproc", files(str(tmp_path / "our_out")), files(str(tmp_path / "ref_out")) if HAVE_REF else None)
    assert sum(os.path.getsize(str(tmp_path / "our_out" / x)) for x in names if x.startswith("ema-bin")) > 300_000

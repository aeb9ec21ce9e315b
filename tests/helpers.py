"""ctypes front-ends for the two checkers used by the tests (never by the product):

* ``port()``  — oracle/liboracle.so, this repo's plain-C restatement (travels everywhere);
* ``ref()``   — oracle/_ref/libemaref.so, the unmodified reference compiled from /root/reference
                (present wherever oracle/Makefile's ``ref`` target was built; tests skip otherwise).
"""
from __future__ import annotations

import ctypes as C
import hashlib
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
ORACLE_DIR = os.path.join(ROOT, "oracle")
REF_DIR = os.path.join(ORACLE_DIR, "_ref")
DATA_ROOT = os.environ.get("EMAB_DATA", "/tmp/emab_data")

HREG_N = 18
REG_FIELDS = ["rb", "re", "qb", "qe", "rid", "score", "truesc", "sub", "csub", "sub_n", "w", "seedcov",
              "secondary", "seedlen0", "n_comp", "is_alt", "frac_rep_bits", "secondary_all"]

_p = lambda a, t: a.ctypes.data_as(C.POINTER(t))

# Where oracle/_ref is not built, the tests that compare with the reference's output compare with a digest of it recorded in
# tests/golden/reference/ (see its README).  EMAB_RECORD_REFERENCE=<dir> writes the recordings of cases that have none there.
RECORDED_DIR = os.path.join(ROOT, "tests", "golden", "reference")
RECORD_TO = os.environ.get("EMAB_RECORD_REFERENCE")


def nt4(seq: bytes | str) -> np.ndarray:
    if isinstance(seq, str):
        seq = seq.encode()
    tab = np.full(256, 4, dtype=np.uint8)
    for i, ch in enumerate(b"ACGT"):
        tab[ch] = i
        tab[ch + 32] = i
    return tab[np.frombuffer(seq, dtype=np.uint8)]


def read_fasta_nt4(path):
    """contigs of a FASTA file as nt4 arrays, in file order"""
    out, cur = [], []
    with open(path, "rb") as f:
        for ln in f:
            if ln.startswith(b">"):
                if cur:
                    out.append(nt4(b"".join(cur)))
                cur = []
            else:
                cur.append(ln.strip())
    if cur:
        out.append(nt4(b"".join(cur)))
    return out


def pack(seqs):
    """list of uint8 arrays -> (concatenated, int64 offsets[n+1])"""
    off = np.zeros(len(seqs) + 1, dtype=np.int64)
    if len(seqs):
        off[1:] = np.cumsum([len(s) for s in seqs])
    flat = np.concatenate(seqs).astype(np.uint8) if len(seqs) else np.zeros(0, np.uint8)
    return np.ascontiguousarray(flat), off


def build_port():
    subprocess.run(["make", "-s", "-C", ORACLE_DIR, "port"], check=True)


_port = None


def port():
    global _port
    if _port is None:
        so = os.path.join(ORACLE_DIR, "liboracle.so")
        if not os.path.exists(so):
            build_port()
        L = C.CDLL(so)
        L.orc_index_load.restype = C.c_void_p
        L.orc_index_load.argtypes = [C.c_char_p]
        L.orc_index_free.argtypes = [C.c_void_p]
        L.orc_sa.restype = C.c_uint64
        L.orc_sa.argtypes = [C.c_void_p, C.c_uint64]
        L.orc_touches.restype = C.c_int64
        L.orc_touches.argtypes = [C.c_void_p, C.c_int]
        for f in ("orc_collect_intv_flat", "orc_sa_batch", "orc_index_info", "orc_occ4"):
            getattr(L, f).argtypes = None
        _port = L
    return _port


_ref = None


def have_ref() -> bool:
    return os.path.exists(os.path.join(REF_DIR, "libemaref.so"))


def ref():
    global _ref
    if _ref is None:
        L = C.CDLL(os.path.join(REF_DIR, "libemaref.so"))
        L.ref_idx_load.restype = C.c_void_p
        L.ref_idx_load.argtypes = [C.c_char_p]
        L.ref_sa.restype = C.c_int64
        _ref = L
    return _ref


def ref_bin(name: str) -> str:
    return os.path.join(REF_DIR, name)


def sha(*parts) -> str:
    """SHA-256 over the parts (bytes as they are, anything else by repr)"""
    h = hashlib.sha256()
    for x in parts:
        h.update(x if isinstance(x, bytes) else repr(x).encode())
        h.update(b"\0")
    return h.hexdigest()


def recorded_reference(key: str, ours):
    """The recorded digest of the reference's output for case `key` (tests/golden/reference/digests.json).  In record mode a
    case without a recording is recorded as `ours` (this build's digest of the same output) into $EMAB_RECORD_REFERENCE."""
    path = os.path.join(RECORDED_DIR, "digests.json")
    rec = json.load(open(path)) if os.path.exists(path) else {}
    if key not in rec and RECORD_TO:
        os.makedirs(RECORD_TO, exist_ok=True)
        out = os.path.join(RECORD_TO, "digests.json")
        new = json.load(open(out)) if os.path.exists(out) else {}
        new[key] = ours
        json.dump(new, open(out, "w"), indent=1, sort_keys=True)
        return ours
    assert key in rec, f"no recorded reference output for {key} in {path}"
    return rec[key]


def split_sam(text: bytes):
    """SAM text -> (header lines minus @PG, which echoes argv; records)"""
    lines = text.split(b"\n")
    head = [l for l in lines if l.startswith(b"@") and not l.startswith(b"@PG")]
    body = [l for l in lines if l and not l.startswith(b"@")]
    return head, body


def diff_msg(a, b):
    for i, (x, y) in enumerate(zip(a, b)):
        if x != y:
            return f"first difference at record {i}:\n ours: {x[:300]!r}\n ref:  {y[:300]!r}"
    return f"record counts differ: {len(a)} vs {len(b)}"


def compare_sam_with_reference(key, ours: bytes, run_reference, tmp_path, min_records=1):
    """This build's SAM text against the reference's on the same input: the header minus @PG and every record, byte for
    byte.  run_reference(out_path) runs oracle/_ref/ema where it is built; elsewhere the recorded digest of the reference's
    output for case `key` stands in for it.  Returns this build's records."""
    h1, b1 = split_sam(ours)
    if os.path.exists(ref_bin("ema")):
        out = os.path.join(str(tmp_path), "ref.sam")
        run_reference(out)
        h2, b2 = split_sam(open(out, "rb").read())
        assert h1 == h2
        assert len(b2) >= min_records
        assert b1 == b2, diff_msg(b1, b2)
    else:
        assert len(b1) >= min_records
        d = sha(b"\n".join(h1), b"\n".join(b1))
        assert d == recorded_reference(key, d), f"{key}: SAM differs from the reference's recorded output"
    return b1


# ---- batched SW wrappers with one signature for both checkers -------------------------------------
def sw_extend(lib, prefix, qs, ts, h0, w=100, end_bonus=5, zdrop=100, threads=8):
    q, qo = pack(qs)
    t, to = pack(ts)
    h0 = np.ascontiguousarray(h0, dtype=np.int32)
    out = np.zeros((len(qs), 6), dtype=np.int32)
    if prefix == "orc":
        cells = C.c_int64(0)
        lib.orc_extend_batch(len(qs), _p(q, C.c_uint8), _p(qo, C.c_int64), _p(t, C.c_uint8), _p(to, C.c_int64),
                             _p(h0, C.c_int32), w, end_bonus, zdrop, _p(out, C.c_int32), C.byref(cells), threads)
        return out, cells.value
    lib.ref_extend_batch(len(qs), _p(q, C.c_uint8), _p(qo, C.c_int64), _p(t, C.c_uint8), _p(to, C.c_int64),
                         _p(h0, C.c_int32), w, end_bonus, zdrop, _p(out, C.c_int32), threads)
    return out, None


def sw_global(lib, prefix, qs, ts, ws, max_cigar=64, threads=8):
    q, qo = pack(qs)
    t, to = pack(ts)
    ws = np.ascontiguousarray(ws, dtype=np.int32)
    out = np.zeros((len(qs), 2), dtype=np.int32)
    cig = np.zeros((len(qs), max_cigar), dtype=np.uint32)
    if prefix == "orc":
        cells = C.c_int64(0)
        lib.orc_global_batch(len(qs), _p(q, C.c_uint8), _p(qo, C.c_int64), _p(t, C.c_uint8), _p(to, C.c_int64),
                             _p(ws, C.c_int32), _p(out, C.c_int32), _p(cig, C.c_uint32), max_cigar, C.byref(cells), threads)
        return out, cig, cells.value
    lib.ref_global_batch(len(qs), _p(q, C.c_uint8), _p(qo, C.c_int64), _p(t, C.c_uint8), _p(to, C.c_int64),
                         _p(ws, C.c_int32), _p(out, C.c_int32), _p(cig, C.c_uint32), max_cigar, threads)
    return out, cig, None


def sw_local(lib, prefix, qs, ts, threads=8):
    q, qo = pack(qs)
    t, to = pack(ts)
    out = np.zeros((len(qs), 7), dtype=np.int32)
    if prefix == "orc":
        cells = C.c_int64(0)
        lib.orc_local_batch(len(qs), _p(q, C.c_uint8), _p(qo, C.c_int64), _p(t, C.c_uint8), _p(to, C.c_int64),
                            _p(out, C.c_int32), C.byref(cells), threads)
        return out, cells.value
    lib.ref_local_batch(len(qs), _p(q, C.c_uint8), _p(qo, C.c_int64), _p(t, C.c_uint8), _p(to, C.c_int64),
                        _p(out, C.c_int32), threads)
    return out, None


# ---- random SW task generators (shared by oracle-vs-ref and GPU parity tests) ----------------------
def random_extend_tasks(n, seed, max_q=200, n_frac=0.02):
    """Mixed bag: related pairs with noise, unrelated pairs, tiny and empty-ish cases, Ns."""
    rng = np.random.default_rng(seed)
    qs, ts, h0 = [], [], []
    for i in range(n):
        ql = int(rng.integers(1, max_q + 1))
        q = rng.integers(0, 4, size=ql, dtype=np.uint8)
        mode = i % 5
        if mode == 0:  # unrelated target
            t = rng.integers(0, 4, size=int(rng.integers(1, ql + 120)), dtype=np.uint8)
        else:
            t = list(q)
            rate = [0.0, 0.01, 0.05, 0.15][mode - 1]
            j = 0
            out = []
            for b in t:
                r = rng.random()
                if r < rate * 0.25:
                    continue  # deletion from target
                if r < rate * 0.5:
                    out.append(int(rng.integers(0, 4)))  # insertion
                if r < rate:
                    out.append(int(rng.integers(0, 4)))
                else:
                    out.append(int(b))
            pad = int(rng.integers(0, 120))
            t = np.array(out + list(rng.integers(0, 4, size=pad)), dtype=np.uint8)
            if len(t) == 0:
                t = rng.integers(0, 4, size=3, dtype=np.uint8)
        if rng.random() < n_frac * 5:
            q = q.copy()
            q[rng.random(ql) < 0.03] = 4
        if rng.random() < n_frac * 5:
            t = t.copy()
            t[rng.random(len(t)) < 0.03] = 4
        qs.append(q)
        ts.append(np.asarray(t, dtype=np.uint8))
        h0.append(int(rng.integers(1, 160)))
    return qs, ts, np.array(h0, dtype=np.int32)


# ---- bucket files and candidate records ------------------------------------------------------------
def read_bucket(path, limit=None):
    """Lines of a preprocessed bucket -> list of (bc, name, read1, qual1, read2, qual2) strings."""
    out = []
    with open(path) as f:
        for ln in f:
            ln = ln.rstrip("\n")
            if ln:
                out.append(tuple(ln.split(" ")))
            if limit and len(out) >= limit:
                break
    return out


def cands_from_alns(alns, n1, n2, base=0):
    """emab_aln_t records of one pair (mate-1 regions then mate-2 regions) -> the tuples the reference's
    append_alignments would have kept: (chrom,pos1,rev,mate,mapq,score_mapq,clip,clip_edit_dist,NM,n_cigar,score,cigar)"""
    out = []
    for k in range(n1 + n2):
        x = alns[base + k]
        if x["keep"]:
            out.append((int(x["rid"]), int(x["pos"]) + 1, int(x["is_rev"]), 0 if k < n1 else 1, int(x["mapq"]), int(x["score_mapq"]),
                        int(x["clip"]), int(x["clip_edit_dist"]), int(x["NM"]), int(x["n_cigar"]), float(x["em_score"]),
                        tuple(int(c) for c in x["cigar"][:x["n_cigar"]])))
    return out


def cands_from_golden(g):
    """tests/golden/cand_golden.npz -> per-pair lists of the same tuples"""
    out, pos = [], 0
    for n in g["n"]:
        cur = []
        for i, s, c in zip(g["ints"][pos:pos + n], g["score"][pos:pos + n], g["cigar"][pos:pos + n]):
            cur.append((int(i[0]), int(i[1]), int(i[2]), int(i[3]), int(i[4]), int(i[5]), int(i[6]), int(i[7]), int(i[8]), int(i[9]),
                        float(s), tuple(int(x) for x in c[:i[9]])))
        out.append(cur)
        pos += n
    return out


_hs = None


def hostsim():
    """tests/hostsim/libhostsim.so: the scalar device logic compiled for the host (test tooling)."""
    global _hs
    if _hs is None:
        d = os.path.join(ROOT, "tests", "hostsim")
        subprocess.run(["make", "-s", "-C", d], check=True)
        L = C.CDLL(os.path.join(d, "libhostsim.so"))
        L.hs_index_load.restype = C.c_void_p
        L.hs_index_load.argtypes = [C.c_char_p]
        _hs = L
    return _hs

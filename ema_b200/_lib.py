"""ctypes binding of include/ema_b200.h (no compute here; see ema_b200/csrc)."""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_SO = os.path.join(_HERE, "libema_b200.so")


class EmabError(RuntimeError):
    pass


_lib = None


def lib():
    """Load libema_b200.so; there is no fallback if it is missing."""
    global _lib
    if _lib is None:
        if not os.path.exists(_SO):
            raise EmabError(f"{_SO} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                            "(ema_b200 has no CPU fallback)")
        L = C.CDLL(_SO)
        L.emab_last_error.restype = C.c_char_p
        L.emab_last_kernel_ms.restype = C.c_double
        L.emab_last_kernel_ms.argtypes = [C.c_void_p]
        L.emab_last_launches.argtypes = [C.c_void_p]
        L.emab_index_build_ms.restype = C.c_double
        L.emab_index_build_ms.argtypes = [C.c_void_p]
        L.emab_index_free.argtypes = [C.c_void_p]
        L.emab_ctx_free.argtypes = [C.c_void_p]
        L.emab_session_close.argtypes = [C.c_void_p]
        L.emab_free.argtypes = [C.c_void_p]
        L.emab_align_bucket.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.POINTER(C.c_void_p), C.POINTER(C.c_uint64)]
        L.emab_pinned_alloc.restype = C.c_void_p
        L.emab_pinned_alloc.argtypes = [C.c_uint64]
        L.emab_pinned_free.argtypes = [C.c_void_p]
        L.emab_align_fastq.argtypes = [C.c_void_p, C.c_char_p, C.c_uint64, C.c_char_p, C.c_uint64, C.POINTER(C.c_void_p), C.POINTER(C.c_uint64)]
        _lib = L
    return _lib


def _check(rc: int):
    if rc != 0:
        raise EmabError(f"libema_b200 error {rc}: {lib().emab_last_error().decode(errors='replace')}")


def _p(a: np.ndarray, t):
    return a.ctypes.data_as(C.POINTER(t))


def _pack(seqs):
    off = np.zeros(len(seqs) + 1, dtype=np.int64)
    if len(seqs):
        off[1:] = np.cumsum([len(s) for s in seqs])
    flat = np.concatenate([np.asarray(s, dtype=np.uint8) for s in seqs]) if len(seqs) and off[-1] else np.zeros(1, np.uint8)
    return np.ascontiguousarray(flat), off


class IndexBuildStats(C.Structure):
    _fields_ = [("l_pac", C.c_int64), ("primary", C.c_int64), ("n_seqs", C.c_int32), ("n_holes", C.c_int32), ("chunk_bits", C.c_int32),
                ("n_chunks", C.c_int32), ("max_chunk", C.c_int64), ("n_tied", C.c_int64), ("max_rounds", C.c_int32), ("pad", C.c_int32),
                ("ms_pack", C.c_double), ("ms_sort", C.c_double), ("ms_occ", C.c_double), ("ms_write", C.c_double), ("ms_total", C.c_double)]


def index_build(fasta: str, prefix: str | None = None, device: int = 0) -> dict:
    """emab_index_build: `bwa index` on the GPU; writes <prefix>.pac/.ann/.amb/.bwt/.sa and returns the build statistics."""
    st = IndexBuildStats()
    _check(lib().emab_index_build(fasta.encode(), prefix.encode() if prefix else None, device, C.byref(st)))
    return {n: getattr(st, n) for n, _ in IndexBuildStats._fields_ if n != "pad"}


def index_pack_fasta(fasta: str, prefix: str | None = None):
    """emab_index_pack_fasta: the host half of the index build (.pac/.ann/.amb); runs without a GPU."""
    _check(lib().emab_index_pack_fasta(fasta.encode(), prefix.encode() if prefix else None))


class Index:
    """FM index + packed reference resident in one GPU's HBM (emab_index_load)."""

    def __init__(self, prefix: str, device: int = 0):
        self._h = C.c_void_p()
        _check(lib().emab_index_load(prefix.encode(), device, C.byref(self._h)))
        info = np.zeros(12, dtype=np.int64)
        _check(lib().emab_index_info(self._h, _p(info, C.c_int64)))
        self.info = info
        self.l_pac, self.n_seqs, self.primary, self.seq_len = (int(x) for x in info[:4])
        self.contigs = []
        for i in range(self.n_seqs):
            off, ln, name = C.c_int64(), C.c_int32(), C.create_string_buffer(512)
            _check(lib().emab_index_contig(self._h, i, C.byref(off), C.byref(ln), name, 512))
            self.contigs.append((name.value.decode(), off.value, ln.value))

    @property
    def build_ms(self) -> float:
        return lib().emab_index_build_ms(self._h)

    def close(self):
        if self._h:
            lib().emab_index_free(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class Context:
    """One worker (CUDA stream + scratch) — emab_ctx_create."""

    def __init__(self, index: Index | None = None):
        self._h = C.c_void_p()
        self.index = index
        _check(lib().emab_ctx_create(index._h if index else None, C.byref(self._h)))

    @property
    def last_kernel_ms(self) -> float:
        return lib().emab_last_kernel_ms(self._h)

    @property
    def last_launches(self) -> int:
        return lib().emab_last_launches(self._h)

    def close(self):
        if self._h:
            lib().emab_ctx_free(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def extend_batch(ctx: Context, qs, ts, h0, w=100, end_bonus=5, zdrop=100):
    """ksw_extend2 over a batch -> (out[n,6] = score,qle,tle,gtle,gscore,max_off ; cells)"""
    q, qo = _pack(qs)
    t, to = _pack(ts)
    h0 = np.ascontiguousarray(h0, dtype=np.int32)
    out = np.zeros((len(qs), 6), dtype=np.int32)
    cells = C.c_int64(0)
    _check(lib().emab_extend_batch(ctx._h, len(qs), _p(q, C.c_uint8), _p(qo, C.c_int64), _p(t, C.c_uint8), _p(to, C.c_int64),
                                   _p(h0, C.c_int32), w, end_bonus, zdrop, _p(out, C.c_int32), C.byref(cells)))
    return out, cells.value


def set_sw_mode(ctx: Context, mode: int):
    """0 = one thread per task (ksw_lanes.cuh, default), 1 = one warp per task (ksw_warp.cuh)."""
    _check(lib().emab_set_sw_mode(ctx._h, mode))


def set_seed_mode(ctx: Context, mode: int):
    """5 (default) = seed_hot.cuh (x1 not carried); 1-4 = the exact forms; 0 = EMAB_SEED_MODE or the default."""
    _check(lib().emab_set_seed_mode(ctx._h, mode))


def extend_resident_load(ctx: Context, q2d: np.ndarray, t2d: np.ndarray, h0):
    """Upload n fixed-length tasks (q2d[n,qlen], t2d[n,tlen]) once for emab_extend_resident_run."""
    n = q2d.shape[0]
    q = np.ascontiguousarray(q2d, dtype=np.uint8).reshape(-1)
    t = np.ascontiguousarray(t2d, dtype=np.uint8).reshape(-1)
    qo = np.arange(n + 1, dtype=np.int64) * q2d.shape[1]
    to = np.arange(n + 1, dtype=np.int64) * t2d.shape[1]
    h0 = np.ascontiguousarray(h0, dtype=np.int32)
    _check(lib().emab_extend_resident_load(ctx._h, n, _p(q, C.c_uint8), _p(qo, C.c_int64), _p(t, C.c_uint8), _p(to, C.c_int64), _p(h0, C.c_int32)))
    return n


def extend_resident_run(ctx: Context, n, reps=1, w=100, end_bonus=5, zdrop=100, want_out=True):
    """-> (out[n,6] or None, visited cells per launch, device ms per launch)"""
    out = np.zeros((n, 6), dtype=np.int32) if want_out else None
    cells = C.c_int64(0)
    _check(lib().emab_extend_resident_run(ctx._h, w, end_bonus, zdrop, reps, _p(out, C.c_int32) if want_out else None, C.byref(cells)))
    return out, cells.value, ctx.last_kernel_ms / reps


def int_peak(ctx: Context, kind: int, iters: int = 2000):
    """Integer-pipe microbenchmark -> (1e9 lane-instructions/s, ms)"""
    g, ms = C.c_double(0), C.c_double(0)
    _check(lib().emab_int_peak(ctx._h, kind, iters, C.byref(g), C.byref(ms)))
    return g.value, ms.value


def global_batch(ctx: Context, qs, ts, ws, max_cigar=64):
    """ksw_global2 over a batch -> (out[n,2] = score,n_cigar ; cigar[n,max_cigar] ; cells)"""
    q, qo = _pack(qs)
    t, to = _pack(ts)
    ws = np.ascontiguousarray(ws, dtype=np.int32)
    out = np.zeros((len(qs), 2), dtype=np.int32)
    cig = np.zeros((len(qs), max_cigar), dtype=np.uint32)
    cells = C.c_int64(0)
    _check(lib().emab_global_batch(ctx._h, len(qs), _p(q, C.c_uint8), _p(qo, C.c_int64), _p(t, C.c_uint8), _p(to, C.c_int64),
                                   _p(ws, C.c_int32), _p(out, C.c_int32), _p(cig, C.c_uint32), max_cigar, C.byref(cells)))
    return out, cig, cells.value


def local_batch(ctx: Context, qs, ts):
    """ksw_align2 (mem_matesw flags) over a batch -> (out[n,7] = score,te,qe,score2,te2,tb,qb ; cells)"""
    q, qo = _pack(qs)
    t, to = _pack(ts)
    out = np.zeros((len(qs), 7), dtype=np.int32)
    cells = C.c_int64(0)
    _check(lib().emab_local_batch(ctx._h, len(qs), _p(q, C.c_uint8), _p(qo, C.c_int64), _p(t, C.c_uint8), _p(to, C.c_int64),
                                  _p(out, C.c_int32), C.byref(cells)))
    return out, cells.value


def smem_batch(ctx: Context, reads, max_intv=128):
    """mem_collect_intv over a batch of nt4 reads -> (list of (n_i,4) int64 arrays ; block touches)"""
    s, off = _pack(reads)
    n = len(reads)
    iv = np.zeros((n, max_intv, 4), dtype=np.int64)
    cnt = np.zeros(n, dtype=np.int32)
    touches = C.c_int64(0)
    _check(lib().emab_smem_batch(ctx._h, n, _p(s, C.c_uint8), _p(off, C.c_int64), _p(iv, C.c_int64), _p(cnt, C.c_int32),
                                 max_intv, C.byref(touches)))
    return [iv[i, :cnt[i]] for i in range(n)], touches.value


def sa_batch(ctx: Context, ks, mode=0):
    """bwt_sa for SA indices ks (mode 0: dense SA, 1: LF walk over the sampled SA)"""
    ks = np.ascontiguousarray(ks, dtype=np.int64)
    out = np.zeros_like(ks)
    _check(lib().emab_sa_batch(ctx._h, len(ks), _p(ks, C.c_int64), _p(out, C.c_int64), mode))
    return out


ALN_DTYPE = np.dtype([("pos", "<i8"), ("rid", "<i4"), ("is_rev", "<i4"), ("NM", "<i4"), ("n_cigar", "<i4"), ("score", "<i4"),
                      ("mapq", "<i4"), ("score_mapq", "<i4"), ("clip", "<i4"), ("clip_edit_dist", "<i4"), ("keep", "<i4"),
                      ("em_score", "<f8"), ("cigar", "<u4", (64,))])
CAND_DTYPE = np.dtype([("pos", "<i8"), ("em_score", "<f8"), ("rid", "<i4"), ("NM", "<i4"), ("score", "<i4"), ("mapq", "<i4"),
                       ("score_mapq", "<i4"), ("clip", "<i4"), ("clip_edit_dist", "<i4"), ("cigar_off", "<u4"), ("n_cigar", "<u2"),
                       ("is_rev", "u1"), ("keep", "u1"), ("pad", "<u4")])
assert CAND_DTYPE.itemsize == 56


PAIR_TEXT_DTYPE = np.dtype([("id_off", "<u4", 2), ("id_len", "<u4", 2), ("read_off", "<u4", 2), ("read_len", "<u4", 2),
                            ("qual_off", "<u4", 2), ("qual_len", "<u4", 2)])


def parse_bucket(ctx: Context, data: bytes, bc_len: int = 16, haplotag: bool = False):
    """emab_parse_bucket: the bucket reader on the device.  Returns (pair table as a structured array, barcode codes)."""
    n = C.c_int()
    pt, bc = C.c_void_p(), C.c_void_p()
    _check(lib().emab_parse_bucket(ctx._h, data, C.c_uint64(len(data)), bc_len, int(haplotag), C.byref(n), C.byref(pt), C.byref(bc)))
    if n.value == 0:
        return np.zeros(0, PAIR_TEXT_DTYPE), np.zeros(0, np.uint64)
    tab = np.frombuffer(C.string_at(pt, n.value * PAIR_TEXT_DTYPE.itemsize), dtype=PAIR_TEXT_DTYPE).copy()
    bcs = np.frombuffer(C.string_at(bc, n.value * 8), dtype=np.uint64).copy()
    return tab, bcs


class Stats(C.Structure):
    _fields_ = [("extend_cells", C.c_int64), ("global_cells", C.c_int64), ("local_cells", C.c_int64), ("occ_touches", C.c_int64),
                ("n_occ", C.c_int64), ("n_regs", C.c_int64), ("kernel_ms", C.c_double), ("ms_seed", C.c_double), ("ms_chain", C.c_double),
                ("ms_align1", C.c_double), ("ms_rescue", C.c_double), ("ms_finalize", C.c_double), ("h2d_bytes", C.c_int64),
                ("d2h_bytes", C.c_int64), ("launches", C.c_int32), ("pad", C.c_int32), ("rescue_planned_cells", C.c_int64), ("rescue_unplanned", C.c_int64),
                ("ext_planned_cells", C.c_int64), ("ext_unplanned", C.c_int64), ("glob_planned_cells", C.c_int64), ("glob_unplanned", C.c_int64),
                ("ms_ext_wave", C.c_double), ("ms_glob_wave", C.c_double)]


class PairsResult(C.Structure):
    _fields_ = [("n_cands", C.c_int64), ("n_cigar_ops", C.c_int64), ("n_regs", C.POINTER(C.c_int32)), ("cands", C.c_void_p),
                ("cigars", C.POINTER(C.c_uint32)), ("regs_dbg", C.POINTER(C.c_int64))]


def align_pairs(ctx: Context, reads, stage=3, want_regs=False):
    """emab_align_pairs over nt4 reads laid out pair0/mate1, pair0/mate2, pair1/mate1, ...
    Returns dict(n_regs[2n], alns (structured array with inline CIGARs, all regions incl. keep==0),
    regs (A,18) or None, stats)."""
    assert len(reads) % 2 == 0
    s, off = _pack(reads)
    R = len(reads)
    res = PairsResult()
    st = Stats()
    _check(lib().emab_align_pairs(ctx._h, R // 2, _p(s, C.c_uint8), _p(off, C.c_int64), stage, int(want_regs), C.byref(res), C.byref(st)))
    A = res.n_cands
    n_regs = np.ctypeslib.as_array(res.n_regs, shape=(R,)).copy() if R else np.zeros(0, np.int32)
    alns = np.zeros(A, dtype=ALN_DTYPE)
    if stage >= 3 and A:
        cands = np.frombuffer(C.string_at(res.cands, A * 56), dtype=CAND_DTYPE)
        pool = np.ctypeslib.as_array(res.cigars, shape=(max(int(res.n_cigar_ops), 1),)).copy()
        for f in ("pos", "rid", "is_rev", "NM", "n_cigar", "score", "mapq", "score_mapq", "clip", "clip_edit_dist", "keep", "em_score"):
            alns[f] = cands[f]
        for i in np.nonzero(cands["n_cigar"])[0]:
            n, o = int(cands["n_cigar"][i]), int(cands["cigar_off"][i])
            alns["cigar"][i, :n] = pool[o:o + n]
    regs = np.ctypeslib.as_array(res.regs_dbg, shape=(A, 18)).copy() if want_regs and A else (np.zeros((0, 18), np.int64) if want_regs else None)
    return dict(n_regs=n_regs, alns=alns, regs=regs, stats=st)


def bgzf_eof() -> bytes:
    """The 28-byte empty BGZF member that ends a BAM file (emab_bgzf_eof)."""
    p, n = C.c_void_p(), C.c_uint64()
    _check(lib().emab_bgzf_eof(C.byref(p), C.byref(n)))
    return C.string_at(p, n.value)


def bgzf_compress(ctx: Context, data: bytes) -> bytes:
    """emab_bgzf_compress: BGZF members of `data` (one per 65 280-byte chunk), compressed on the device."""
    cap = len(data) + (len(data) // 65280 + 1) * 64
    out = C.create_string_buffer(cap)
    n = C.c_uint64()
    _check(lib().emab_bgzf_compress(ctx._h, data, C.c_uint64(len(data)), out, C.c_uint64(cap), C.byref(n)))
    return out.raw[:n.value]


def bgzf_inflate(ctx: Context, data: bytes) -> bytes:
    """emab_bgzf_inflate: the content of the whole BGZF members in `data`, inflated on the device (one warp per member)"""
    n = C.c_uint64()
    rc = lib().emab_bgzf_inflate(ctx._h, data, C.c_uint64(len(data)), None, C.c_uint64(0), C.byref(n))
    if rc != -4:   # EMAB_ERR_OVERFLOW gives the size needed
        _check(rc)
        return b""
    out = C.create_string_buffer(max(n.value, 1))
    _check(lib().emab_bgzf_inflate(ctx._h, data, C.c_uint64(len(data)), out, C.c_uint64(n.value), C.byref(n)))
    return out.raw[:n.value]


_MERGE_CB = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_void_p, C.c_uint64)


def bam_merge(paths, budget: int = 4 << 30, index: bool = True, device: int = 0, slice_chunks: int = 0, stats: dict | None = None):
    """emab_bam_merge_files: the coordinate-sorted BAM files `paths` merged on the device into one sorted file ->
    (file bytes without the EOF block, .bai bytes; b"" with index=False).  budget: host bytes of records read per window.
    stats (optional) receives the wall times (ms) and the counts of the call."""
    ctx = Context.__new__(Context)
    ctx._h, ctx.index = C.c_void_p(), None
    _check(lib().emab_ctx_create_on(device, C.byref(ctx._h)))
    parts = []

    def write(_u, p, n):
        parts.append(C.string_at(p, n))
        return 0
    cb = _MERGE_CB(write)
    arr = (C.c_char_p * len(paths))(*[os.fsencode(p) for p in paths])
    bai, n = C.c_void_p(), C.c_uint64()
    ms, counts = (C.c_double * 6)(), (C.c_uint64 * 4)()
    _check(lib().emab_bam_merge_files(ctx._h, len(paths), arr, C.c_uint64(budget), slice_chunks, cb, None,
                                      C.byref(bai) if index else None, C.byref(n), ms, counts))
    idx = C.string_at(bai, n.value) if bai.value else b""
    if bai.value:
        lib().emab_free(bai)
    if stats is not None:
        stats.update(zip(("inflate_ms", "rows_ms", "order_ms", "gather_ms", "compress_ms", "index_ms"), list(ms)))
        stats.update(zip(("read_bytes", "inflated_bytes", "records", "windows"), list(counts)))
    return b"".join(parts), idx


def bam_merge_header(paths) -> bytes:
    """emab_bam_merge_header: the header text `bam_merge` writes for these inputs (host code, no device)"""
    arr = (C.c_char_p * len(paths))(*[os.fsencode(p) for p in paths])
    text, n = C.c_void_p(), C.c_uint64()
    _check(lib().emab_bam_merge_header(len(paths), arr, C.byref(text), C.byref(n)))
    out = C.string_at(text, n.value)
    lib().emab_free(text)
    return out


class RunStats(C.Structure):
    _fields_ = [(n, C.c_double) for n in ("parse_ms", "encode_ms", "align_ms", "kernel_ms", "cloud_ms", "flatten_ms", "em_ms",
                                          "em_kernel_ms", "format_ms", "total_ms", "ms_seed", "ms_chain", "ms_align1", "ms_rescue",
                                          "ms_finalize", "gate_wait_ms")] + [("h2d_bytes", C.c_int64), ("d2h_bytes", C.c_int64)] + \
               [(n, C.c_int64) for n in ("n_pairs", "n_barcodes", "n_cands", "n_clouds", "sam_bytes", "extend_cells", "global_cells",
                                         "local_cells", "occ_touches")] + [("launches", C.c_int32), ("pad", C.c_int32)] + \
               [(n, C.c_int64) for n in ("ext_planned_cells", "ext_unplanned", "glob_planned_cells", "glob_unplanned")] + \
               [("ms_ext_wave", C.c_double), ("ms_glob_wave", C.c_double), ("format_kernel_ms", C.c_double)] + \
               [(n, C.c_double) for n in ("sort_ms", "gather_ms", "compress_ms", "index_ms")] + \
               [("spill_files", C.c_int64), ("spill_bytes", C.c_int64), ("spill_ms", C.c_double)]


class PinnedText:
    """A host buffer in page-locked memory (emab_pinned_alloc) holding `data`: what a caller that reads its bucket files into
    pinned buffers hands to emab_align_bucket[s] — the library copies it to the device without a staging copy."""

    def __init__(self, data: bytes):
        self.n = len(data)
        self.ptr = lib().emab_pinned_alloc(max(self.n, 1))
        if not self.ptr:
            raise EmabError("emab_pinned_alloc failed")
        C.memmove(self.ptr, data, self.n)

    def __len__(self):
        return self.n

    def __del__(self):
        try:
            if self.ptr:
                lib().emab_pinned_free(self.ptr)
                self.ptr = None
        except Exception:
            pass


def _host_ptr(d):
    """(address, keep-alive object) of a bytes object or a PinnedText"""
    if isinstance(d, PinnedText):
        return d.ptr, d
    b = C.c_char_p(d)
    return C.cast(b, C.c_void_p).value, b


class Session:
    """The operator the reference's main() calls (find_clouds_and_align and friends) on one GPU:
    emab_session_open / emab_sam_header / emab_align_bucket / emab_align_fastq."""

    OUTPUTS = {"sam": 0, "bam": 1}
    SORT_OFF, SORT_COORD, SORT_COORD_NOINDEX = 0, 1, 2
    _WRITE_CB = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_void_p, C.c_uint64)

    def __init__(self, ref_path: str, platform: str = "10x", device: int = 0, rg: str | None = None, bx_index: str | None = None,
                 apply_opt: bool = False, threads: int = 1, output: str = "sam", sort: bool = False, max_host_bytes: int = 0,
                 spill: str | None = None, qc: bool = False):
        """output="bam": header() and every align call return BGZF members of BAM instead of SAM text
        (a BAM file is header, the calls' bytes in order, then bgzf_eof()).
        sort=True (BAM only): align calls return b"" and hold their records (at most max_host_bytes of host memory, 0: no
        cap); finish() returns them as one coordinate-sorted body and its BAI (file: header, body, bgzf_eof()).
        spill=PREFIX: with a nonzero max_host_bytes, reaching it writes the held records to PREFIX.*.spill files instead of
        failing, and finish() merges them (see set_spill).
        qc=True: the align calls count alignment and linked-read molecule QC on the device (see set_qc, qc_report)."""
        self._h = C.c_void_p()
        _check(lib().emab_session_open(ref_path.encode(), platform.encode(), device, C.byref(self._h)))
        _check(lib().emab_session_config(self._h, rg.encode() if rg else None, bx_index.encode() if bx_index else None,
                                         int(apply_opt), threads))
        self.set_output(output)
        if spill:
            self.set_spill(spill)
        if sort:
            self.set_sort(True, max_host_bytes)
        if qc:
            self.set_qc(True)

    def set_sort(self, on: bool, max_host_bytes: int = 0, index: bool = True):
        """emab_session_sort: coordinate-sorted BAM for the calls that follow (index=False: no BAI, any contig length)"""
        mode = (self.SORT_COORD if index else self.SORT_COORD_NOINDEX) if on else self.SORT_OFF
        _check(lib().emab_session_sort(self._h, mode, C.c_uint64(max_host_bytes)))

    def set_spill(self, prefix: str | None):
        """emab_session_sort_spill: the prefix of the temporary files a sorted run spills to when it reaches max_host_bytes
        (None: no spilling, the cap fails the run).  A session setting that set_sort keeps."""
        _check(lib().emab_session_sort_spill(self._h, prefix.encode() if prefix else None))

    def set_qc(self, on: bool):
        """emab_session_qc: True starts a fresh QC accumulation over the align calls that follow, False stops it"""
        _check(lib().emab_session_qc(self._h, int(on)))

    def qc_report(self) -> bytes:
        """emab_session_qc_report: the QC report (format version 1, include/ema_b200.h) of the calls since set_qc(True)"""
        text, n = C.c_void_p(), C.c_uint64()
        _check(lib().emab_session_qc_report(self._h, C.byref(text), C.byref(n)))
        return self._take(text, n)

    def qc_cost(self) -> dict:
        """emab_session_qc_cost: device time of the QC kernels, QC calls and their copies since set_qc(True)"""
        ms, calls, h2d, d2h = C.c_double(), C.c_int64(), C.c_int64(), C.c_int64()
        _check(lib().emab_session_qc_cost(self._h, C.byref(ms), C.byref(calls), C.byref(h2d), C.byref(d2h)))
        return dict(kernel_ms=ms.value, calls=calls.value, h2d_bytes=h2d.value, d2h_bytes=d2h.value)

    def finish(self) -> tuple[bytes, bytes]:
        """emab_session_finish: (sorted BGZF body without the EOF block, .bai bytes; b"" without an index)"""
        parts = []

        def write(_u, p, n):
            parts.append(C.string_at(p, n))
            return 0
        cb = self._WRITE_CB(write)
        bai, n = C.c_void_p(), C.c_uint64()
        _check(lib().emab_session_finish(self._h, cb, None, C.byref(bai), C.byref(n)))
        idx = C.string_at(bai, n.value) if bai.value else b""
        if bai.value:
            lib().emab_free(bai)
        return b"".join(parts), idx

    def set_output(self, output: str):
        """emab_session_output: "sam" or "bam" for the calls that follow"""
        if output not in self.OUTPUTS:
            raise ValueError(f"unknown output format {output!r} (sam or bam)")
        _check(lib().emab_session_output(self._h, self.OUTPUTS[output]))

    def header(self, argv) -> bytes:
        arr = (C.c_char_p * len(argv))(*[a.encode() for a in argv])
        text, n = C.c_void_p(), C.c_uint64()
        _check(lib().emab_sam_header(self._h, len(argv), arr, C.byref(text), C.byref(n)))
        out = C.string_at(text, n.value)
        lib().emab_free(text)
        return out

    def _take(self, text, n) -> bytes:
        out = C.string_at(text, n.value)
        lib().emab_free(text)
        return out

    def align_bucket(self, data) -> bytes:
        text, n = C.c_void_p(), C.c_uint64()
        addr, keep = _host_ptr(data)
        _check(lib().emab_align_bucket(self._h, addr, len(data), C.byref(text), C.byref(n)))
        del keep
        return self._take(text, n)

    def set_workers(self, n: int):
        _check(lib().emab_session_workers(self._h, n))

    def add_device(self, device: int):
        """emab_session_add_device: one more index replica; align_buckets spreads over all of them (call before set_workers)"""
        _check(lib().emab_session_add_device(self._h, device))

    def align_buckets(self, datas, keep_text=True):
        """emab_align_buckets (-x mode): up to `workers` buckets in flight; returns the SAM texts in input
        order (or only their lengths when keep_text is False, which skips the copy into Python objects)."""
        n = len(datas)
        ptrs = [_host_ptr(d) for d in datas]
        arr = (C.c_void_p * n)(*[a for a, _ in ptrs])
        lens = (C.c_uint64 * n)(*[len(d) for d in datas])
        outs = (C.c_void_p * n)()
        olens = (C.c_uint64 * n)()
        _check(lib().emab_align_buckets(self._h, n, arr, lens, outs, olens))
        res = []
        for i in range(n):
            res.append(C.string_at(outs[i], olens[i]) if keep_text else int(olens[i]))
            lib().emab_free(outs[i])
        return res

    def align_fastq(self, d1: bytes, d2: bytes | None = None) -> bytes:
        text, n = C.c_void_p(), C.c_uint64()
        _check(lib().emab_align_fastq(self._h, d1, len(d1), d2, len(d2) if d2 else 0, C.byref(text), C.byref(n)))
        return self._take(text, n)

    def dump_posteriors(self, path: str | None):
        _check(lib().emab_session_dump_posteriors(self._h, path.encode() if path else None))

    @property
    def stats(self) -> RunStats:
        st = RunStats()
        _check(lib().emab_session_stats(self._h, C.byref(st)))
        return st

    def close(self):
        if self._h:
            lib().emab_session_close(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

"""CPU tests (-m "not gpu") of the HOST-SIDE/control logic of the product: the thread-scalar
(__host__ __device__) code of ema_b200/csrc — seeding, chaining, filtering, extension scheduling,
de-duplication, mate rescue, CIGAR generation, candidate filters — compiled for the host by
tests/hostsim (DP steps supplied by the oracle), checked against golden vectors of the reference
and, where oracle/_ref is built, against the reference itself stage by stage."""
import ctypes as C
import os

import numpy as np
import pytest

import helpers
from helpers import _p

G = os.path.join(os.path.dirname(__file__), "golden")
ALN = np.dtype([("pos", "<i8"), ("rid", "<i4"), ("is_rev", "<i4"), ("NM", "<i4"), ("n_cigar", "<i4"), ("score", "<i4"),
                ("mapq", "<i4"), ("score_mapq", "<i4"), ("clip", "<i4"), ("clip_edit_dist", "<i4"), ("keep", "<i4"),
                ("em_score", "<f8"), ("cigar", "<u4", (64,))])


@pytest.fixture(scope="module")
def hs():
    helpers.build_port()
    return helpers.hostsim()


def hs_candidates(H, hi, s1, s2):
    al = np.zeros(8192, ALN)
    n1, n2 = C.c_int(), C.c_int()
    rc = H.hs_candidates(hi, C.c_double(0.001), len(s1), _p(s1, C.c_uint8), len(s2), _p(s2, C.c_uint8),
                         al.ctypes.data_as(C.c_void_p), C.byref(n1), C.byref(n2), 8192)
    assert rc == 0
    return helpers.cands_from_alns(al, n1.value, n2.value)


def test_layout(hs):
    assert hs.hs_sizeof_aln() == ALN.itemsize


def test_candidates_golden(hs):
    hi = C.c_void_p(hs.hs_index_load(os.path.join(G, "tiny_rep", "ref.fa").encode()))
    want = helpers.cands_from_golden(np.load(os.path.join(G, "cand_golden.npz")))
    lines = helpers.read_bucket(os.path.join(G, "tiny_rep", "ema-bin-000.10x"))
    assert len(lines) == len(want)
    n_multi = 0
    for f, w in zip(lines, want):
        got = hs_candidates(hs, hi, helpers.nt4(f[2]), helpers.nt4(f[4]))
        assert got == w, f[1]
        n_multi += len(w) > 2
    assert n_multi > 5, "fixture must contain multi-mapped pairs"


def test_seeding_golden(hs):
    g = np.load(os.path.join(G, "fm_golden.npz"))
    hi = C.c_void_p(hs.hs_index_load(os.path.join(G, "tiny_rep", "ref.fa").encode()))
    pos = 0
    for i, n in enumerate(g["n_intv"]):
        s = np.ascontiguousarray(g["reads"][g["roff"][i]:g["roff"][i + 1]])
        ob = np.zeros((256, 4), np.int64)
        nb = hs.hs_collect_intv(hi, len(s), _p(s, C.c_uint8), _p(ob, C.c_int64), 256)
        assert nb == n and np.array_equal(ob[:nb], g["intv"][pos:pos + n])
        pos += n


def test_seeding_flat_equals_nested(hs):
    """The device kernel's flattened one-extend-per-iteration form of mem_collect_intv against the
    reference-shaped nested form: same intervals and the same number of Occ-block loads, on reads
    with repeats, N bases and every length from 1 up."""
    hi = C.c_void_p(hs.hs_index_load(os.path.join(G, "tiny_rep", "ref.fa").encode()))
    hs.hs_collect_intv_touches.restype = C.c_int64
    lines = helpers.read_bucket(os.path.join(G, "tiny_rep", "ema-bin-000.10x"))
    rng = np.random.default_rng(11)
    reads = []
    for f in lines[:200]:
        for s in (helpers.nt4(f[2]), helpers.nt4(f[4])):
            reads.append(s)
            t = s.copy()
            t[rng.integers(0, len(t), size=int(rng.integers(1, 6)))] = 4
            reads.append(t)
            reads.append(np.ascontiguousarray(s[:int(rng.integers(1, len(s)))]))
    reads.append(np.full(30, 4, np.uint8))
    reads.append(np.zeros(150, np.uint8))
    for s in reads:
        s = np.ascontiguousarray(s)
        a, b = np.zeros((256, 4), np.int64), np.zeros((256, 4), np.int64)
        tb = C.c_int64()
        na = hs.hs_collect_intv(hi, len(s), _p(s, C.c_uint8), _p(a, C.c_int64), 256)
        nb = hs.hs_collect_intv_nested(hi, len(s), _p(s, C.c_uint8), _p(b, C.c_int64), 256, C.byref(tb))
        assert na == nb and np.array_equal(a, b)
        assert hs.hs_collect_intv_touches(hi, len(s), _p(s, C.c_uint8)) == tb.value


def _seed_reads(rng, n_lines=200):
    lines = helpers.read_bucket(os.path.join(G, "tiny_rep", "ema-bin-000.10x"))
    reads = []
    for f in lines[:n_lines]:
        for s in (helpers.nt4(f[2]), helpers.nt4(f[4])):
            reads.append(s)
            t = s.copy()
            t[rng.integers(0, len(t), size=int(rng.integers(1, 6)))] = 4
            reads.append(t)
            reads.append(np.ascontiguousarray(s[:int(rng.integers(1, len(s)))]))
            u = s.copy()   # substitutions: several SMEMs per read, backward sweeps that die at a mismatch
            u[rng.integers(0, len(u), size=int(rng.integers(1, 4)))] ^= 1
            reads.append(np.minimum(u, 3).astype(np.uint8))
    reads.append(np.full(30, 4, np.uint8))
    reads.append(np.zeros(150, np.uint8))
    reads.append(np.tile(np.array([0, 1], np.uint8), 75))
    reads.append(rng.integers(0, 4, 151).astype(np.uint8))   # matches nothing for long: empty table entries
    return [np.ascontiguousarray(r) for r in reads]


@pytest.mark.parametrize("K", [0, 1, 2, 5, -1, 9, 12])
def test_seeding_hot_equals_exact(hs, K):
    """The default device form (seed_hot.cuh: one-hot Occ blocks, k-mer start table, text comparison at a unique locus)
    against the exact restatement of mem_collect_intv: the same intervals on the coordinates mem_chain reads
    (x0, x2, info), x1 = 0, for every table depth incl. none, the index's default (-1) and deeper than any unique
    k-mer of this reference; reads with N, substitutions, all lengths from 1, ends of the text."""
    hi = C.c_void_p(hs.hs_index_load(os.path.join(G, "tiny_rep", "ref.fa").encode()))
    hs.hs_set_kmer_k(hi, K)
    reads = _seed_reads(np.random.default_rng(12))
    # reads cut from the very ends of the forward-reverse text and across the strand junction
    ref = helpers.read_fasta_nt4(os.path.join(G, "tiny_rep", "ref.fa"))
    cat = np.concatenate(ref)
    both = np.concatenate([cat, (3 - cat)[::-1]])
    L = len(cat)
    for a in (0, 1, L - 150, L - 75, L - 10, 2 * L - 151, 2 * L - 100):
        reads.append(np.ascontiguousarray(both[a:a + 151]))
    n_sec = 0
    for s in reads:
        a, b = np.zeros((256, 4), np.int64), np.zeros((256, 4), np.int64)
        sec = C.c_int64()
        na = hs.hs_collect_intv(hi, len(s), _p(s, C.c_uint8), _p(a, C.c_int64), 256)
        nb = hs.hs_collect_intv_hot(hi, len(s), _p(s, C.c_uint8), _p(b, C.c_int64), 256, C.byref(sec))
        assert na == nb
        assert np.array_equal(a[:na, [0, 2, 3]], b[:nb, [0, 2, 3]]) and not b[:nb, 1].any()
        n_sec += sec.value
    assert n_sec > 0


@pytest.mark.gpu
def test_seeding_hot_equals_exact_c1_rep(hs):
    """the same on the 5 Mbp reference with planted repeats and indel-bearing reads (BASELINE configs[0] variant), at
    the index's own table depth: 1400 reads, and the traffic of the two forms side by side.  The index is built by
    emab_index_build (files byte-identical to `bwa index`'s: tests/test_index_build.py), hence the GPU mark."""
    import ema_b200
    from tools import synth
    p = synth.build_config("c1_rep", helpers.DATA_ROOT, indexer=ema_b200.index_build)
    hi = C.c_void_p(hs.hs_index_load(p["fasta"].encode()))
    assert hs.hs_kmer_k(hi) >= 8
    hs.hs_collect_intv_touches.restype = C.c_int64
    sectors = touches = 0
    for f in helpers.read_bucket(p["bucket"], 700):
        for s in (helpers.nt4(f[2]), helpers.nt4(f[4])):
            a, b = np.zeros((256, 4), np.int64), np.zeros((256, 4), np.int64)
            sec = C.c_int64()
            na = hs.hs_collect_intv(hi, len(s), _p(s, C.c_uint8), _p(a, C.c_int64), 256)
            nb = hs.hs_collect_intv_hot(hi, len(s), _p(s, C.c_uint8), _p(b, C.c_int64), 256, C.byref(sec))
            assert na == nb and np.array_equal(a[:na, [0, 2, 3]], b[:nb, [0, 2, 3]])
            sectors += sec.value
            touches += hs.hs_collect_intv_touches(hi, len(s), _p(s, C.c_uint8))
    # bytes requested: 32-byte sectors here, 64-byte Occ blocks in the exact form
    assert sectors * 32 < 0.6 * touches * 64, (sectors, touches)


@pytest.mark.gpu
def test_seeding_hot_staircase(hs, tmp_path):
    """forward sweeps whose interval size changes 46 times (a staircase of planted prefixes): long prev/curr lists, every
    k-mer table level and several FM steps recorded, multi-step backward rounds — default form against the exact one
    (index by emab_index_build, hence the GPU mark)"""
    import ema_b200
    from tools import synth
    rng = np.random.default_rng(123)
    contigs = synth.make_reference(1, 80_000, 7, 0)
    S = rng.integers(0, 4, 70, dtype=np.uint8)
    c = contigs[0]
    for n, k in enumerate(range(25, 71)):
        pos = 1000 + 1500 * n
        c[pos:pos + k] = S[:k]
        c[pos - 1] = (S[0] + 1 + (n & 1)) & 3
        if k < 70:
            c[pos + k] = (S[k] + 1) & 3
    fa = str(tmp_path / "ref.fa")
    synth.write_fasta(fa, contigs)
    ema_b200.index_build(fa)
    hi = C.c_void_p(hs.hs_index_load(fa.encode()))
    n_long = 0
    for K in (-1, 0, 3):
        hs.hs_set_kmer_k(hi, K)
        for cut in (70, 60, 45):
            for lead in (0, 7, 30):
                r = np.concatenate([rng.integers(0, 4, lead, dtype=np.uint8), S[:cut], rng.integers(0, 4, 100 - cut, dtype=np.uint8)])
                for s in (np.ascontiguousarray(r), np.ascontiguousarray((3 - r)[::-1])):
                    a, b = np.zeros((512, 4), np.int64), np.zeros((512, 4), np.int64)
                    na = hs.hs_collect_intv(hi, len(s), _p(s, C.c_uint8), _p(a, C.c_int64), 512)
                    nb = hs.hs_collect_intv_hot(hi, len(s), _p(s, C.c_uint8), _p(b, C.c_int64), 512, None)
                    assert na == nb and na >= 1 and np.array_equal(a[:na, [0, 2, 3]], b[:nb, [0, 2, 3]])
                    n_long += int((a[:na, 2] > 5).any())
    assert n_long > 10, "the staircase should yield multi-copy intervals"


def test_scalar_patch_global_vs_oracle(hs, port_lib):
    """ScalarPatchDP::global (the score-only ksw_global2 the thread-per-read kernel runs inline for
    mem_patch_reg) against the oracle: same score and same visited cells, both strands, assorted bands."""
    hi = C.c_void_p(hs.hs_index_load(os.path.join(G, "tiny_rep", "ref.fa").encode()))
    rng = np.random.default_rng(3)
    l_pac = 120000
    qs, ts, ws, got, gcells = [], [], [], [], []
    for it in range(300):
        tlen = int(rng.integers(1, 230))
        rev = it % 2
        t0 = int(rng.integers(1000, l_pac - 1000)) + (l_pac if rev else 0)
        tstep = -1 if it % 3 == 0 else 1
        w = int(rng.choice([0, 1, 3, 10, 50, 100, 400]))
        tgt = np.zeros(tlen, np.uint8)
        # query = noisy copy of the window (filled after the bases are known), or unrelated
        probe = np.zeros(1, np.uint8)
        hs.hs_patch_global(hi, 1, _p(probe, C.c_uint8), C.c_int64(t0), tstep, tlen, w, _p(tgt, C.c_uint8), None)
        q = [int(b) for b in tgt]
        if it % 5 == 0:
            q = list(rng.integers(0, 4, size=int(rng.integers(1, 200))))
        else:
            for _ in range(int(rng.integers(0, 6))):
                pos = int(rng.integers(0, max(1, len(q))))
                r = rng.random()
                if r < 0.4 and len(q) > 1:
                    del q[pos]
                elif r < 0.7:
                    q.insert(pos, int(rng.integers(0, 4)))
                elif q:
                    q[pos] = int(rng.integers(0, 5))
        q = np.array(q[:200] or [0], np.uint8)
        cells = C.c_int64()
        sc = hs.hs_patch_global(hi, len(q), _p(q, C.c_uint8), C.c_int64(t0), tstep, tlen, w, _p(tgt, C.c_uint8), C.byref(cells))
        qs.append(q); ts.append(tgt.copy()); ws.append(w); got.append(sc); gcells.append(cells.value)
    want, _, wcells = helpers.sw_global(port_lib, "orc", qs, ts, ws)
    assert np.array_equal(np.array(got), want[:, 0])
    assert sum(gcells) == wcells


def _regs(lib, fn, idx, s, *extra):
    rg = np.zeros((4096, 18), np.int64)
    n = getattr(lib, fn)(idx, len(s), _p(s, C.c_uint8), _p(rg, C.c_int64), 4096, *extra)
    return rg[:n]


def _chains(lib, fn, idx, s, *flt):
    ch = np.zeros((4096, 8), np.int64)
    sd = np.zeros((65536, 4), np.int64)
    ns = C.c_int(0)
    n = getattr(lib, fn)(idx, len(s), _p(s, C.c_uint8), *flt, _p(ch, C.c_int64), 4096, _p(sd, C.c_int64), 65536, C.byref(ns))
    return ch[:n], sd[:ns.value]


@pytest.mark.parametrize("cfg,limit,device_like", [("tiny_rep", 480, 0), pytest.param("c1_rep", 700, 0, marks=pytest.mark.gpu),
                                                    pytest.param("c1_rep", 400, 1, marks=pytest.mark.gpu)])
def test_stages_vs_reference(hs, cfg, limit, device_like):
    """chains after mem_chain_flt, regions after mem_chain2aln, after mem_sort_dedup_patch, after
    mate rescue, and the final candidates: all bit-exact against the compiled reference.  device_like: with the data flow
    of the device pipeline's default forms — intervals of the seed_hot.cuh algorithm (x1 = 0) and the occurrences' SA
    values gathered ahead of the chaining, as k_sa_gather hands them to k_chain.  Where oracle/_ref is not built, all of
    it against the recorded digest of the reference's stage outputs on the same reads.  The c1_rep cases index their
    5 Mbp reference with emab_index_build (hence the GPU mark); tiny_rep uses the committed index."""
    from tools import synth
    hs.hs_set_device_like(device_like)
    if cfg == "tiny_rep":
        p = {"fasta": os.path.join(G, "tiny_rep", "ref.fa"), "bucket": os.path.join(G, "tiny_rep", "ema-bin-000.10x")}
    else:
        import ema_b200
        p = synth.build_config(cfg, helpers.DATA_ROOT, indexer=ema_b200.index_build)
    pre = p["fasta"].encode()
    hi = C.c_void_p(hs.hs_index_load(pre))
    ref_lib = helpers.ref() if helpers.have_ref() else None
    ri = C.c_void_p(ref_lib.ref_idx_load(pre)) if ref_lib else None
    parts = []
    rng = np.random.default_rng(5)
    for f in helpers.read_bucket(p["bucket"], limit):
        reads = [helpers.nt4(f[2]), helpers.nt4(f[4])]
        if rng.random() < 0.05:
            reads[0][rng.integers(0, len(reads[0]))] = 4
        for s in reads:
            a = _chains(hs, "hs_chain", hi, s)
            r0, r1 = _regs(hs, "hs_align1", hi, s, 0), _regs(hs, "hs_align1", hi, s, 1)
            if ref_lib:
                b = _chains(ref_lib, "ref_chain", ri, s, 1)
                assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1]), ("chain", f[1])
                assert np.array_equal(r0, _regs(ref_lib, "ref_chain2aln", ri, s)), ("chain2aln", f[1])
                assert np.array_equal(r1, _regs(ref_lib, "ref_align1", ri, s)), ("align1", f[1])
            else:
                parts += [x.tobytes() + str(x.shape).encode() for x in (a[0], a[1], r0, r1)]
    hs.hs_set_device_like(0)
    if not ref_lib:
        d = helpers.sha(*parts)
        assert d == helpers.recorded_reference(f"stages_{cfg}_{limit}", d)

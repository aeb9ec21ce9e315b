"""GPU parity tests (-m gpu) of the assembled device pipeline (emab_align_pairs, through the C ABI):
candidate alignments — positions, strands, CIGARs, NM, MAPQ inputs and the EM log-likelihood
score — must be bit-exact against the reference's append_alignments (golden vectors, and the
compiled reference where oracle/_ref exists)."""
import ctypes as C
import os

import numpy as np
import pytest

import helpers
from helpers import _p

pytestmark = pytest.mark.gpu
G = os.path.join(os.path.dirname(__file__), "golden")


@pytest.fixture(scope="module")
def emab():
    import ema_b200
    return ema_b200


def pipeline_candidates(emab, ctx, lines):
    reads = []
    for f in lines:
        reads += [helpers.nt4(f[2]), helpers.nt4(f[4])]
    res = emab.align_pairs(ctx, reads)
    off = np.zeros(len(reads) + 1, dtype=np.int64)
    off[1:] = np.cumsum(res["n_regs"])
    out = []
    for i in range(len(lines)):
        n1, n2 = int(res["n_regs"][2 * i]), int(res["n_regs"][2 * i + 1])
        out.append(helpers.cands_from_alns(res["alns"], n1, n2, int(off[2 * i])))
    return out, res


def test_candidates_golden(emab):
    ix = emab.Index(os.path.join(G, "tiny_rep", "ref.fa"))
    ctx = emab.Context(ix)
    want = helpers.cands_from_golden(np.load(os.path.join(G, "cand_golden.npz")))
    lines = helpers.read_bucket(os.path.join(G, "tiny_rep", "ema-bin-000.10x"))
    got, res = pipeline_candidates(emab, ctx, lines)
    bad = [i for i, (a, b) in enumerate(zip(got, want)) if a != b]
    assert not bad, f"{len(bad)} of {len(want)} pairs differ; first {lines[bad[0]][1]}: {got[bad[0]]} vs {want[bad[0]]}"
    st = res["stats"]
    assert st.launches >= 7 and st.kernel_ms > 0 and st.occ_touches > 0
    # determinism: a second run returns identical bytes
    got2, _ = pipeline_candidates(emab, ctx, lines)
    assert got2 == got


def test_candidates_golden_thread_per_read(emab):
    """the same golden comparison with mem_align1_core run one thread per read (emab_set_sw_mode 2,
    align_lanes.cuh) instead of one warp per read"""
    ix = emab.Index(os.path.join(G, "tiny_rep", "ref.fa"))
    ctx = emab.Context(ix)
    emab.set_sw_mode(ctx, 2)
    want = helpers.cands_from_golden(np.load(os.path.join(G, "cand_golden.npz")))
    lines = helpers.read_bucket(os.path.join(G, "tiny_rep", "ema-bin-000.10x"))
    got, res = pipeline_candidates(emab, ctx, lines)
    bad = [i for i, (a, b) in enumerate(zip(got, want)) if a != b]
    assert not bad, f"{len(bad)} of {len(want)} pairs differ; first {lines[bad[0]][1]}: {got[bad[0]]} vs {want[bad[0]]}"
    ctx1 = emab.Context(ix)
    got1, res1 = pipeline_candidates(emab, ctx1, lines)
    assert res["stats"].extend_cells == res1["stats"].extend_cells, "both kernels must visit the reference's DP cells"


def test_stage_regions_vs_hostsim(emab):
    """regions after mem_align1_core (stage 1) and after mate rescue (stage 2) against the host build of
    the same control logic driven by the oracle's scalar DP (itself pinned to the reference)."""
    hs = helpers.hostsim()
    pre = os.path.join(G, "tiny_rep", "ref.fa")
    ix = emab.Index(pre)
    ctx = emab.Context(ix)
    hi = C.c_void_p(hs.hs_index_load(pre.encode()))
    lines = helpers.read_bucket(os.path.join(G, "tiny_rep", "ema-bin-000.10x"))
    reads = []
    for f in lines:
        reads += [helpers.nt4(f[2]), helpers.nt4(f[4])]
    for stage in (1, 2):
        res = emab.align_pairs(ctx, reads, stage=stage, want_regs=True)
        off = np.zeros(len(reads) + 1, dtype=np.int64)
        off[1:] = np.cumsum(res["n_regs"])
        for i in range(len(lines)):
            s1, s2 = reads[2 * i], reads[2 * i + 1]
            if stage == 1:
                for k, s in ((2 * i, s1), (2 * i + 1, s2)):
                    rg = np.zeros((4096, 18), np.int64)
                    n = hs.hs_align1(hi, len(s), _p(s, C.c_uint8), _p(rg, C.c_int64), 4096, 1)
                    assert np.array_equal(res["regs"][off[k]:off[k + 1]], rg[:n]), (stage, lines[i][1])
            else:
                a1 = np.zeros((4096, 18), np.int64)
                a2 = np.zeros((4096, 18), np.int64)
                n1, n2 = C.c_int(), C.c_int()
                hs.hs_pair(hi, len(s1), _p(s1, C.c_uint8), len(s2), _p(s2, C.c_uint8), _p(a1, C.c_int64), C.byref(n1), _p(a2, C.c_int64), C.byref(n2), 4096)
                assert np.array_equal(res["regs"][off[2 * i]:off[2 * i + 1]], a1[:n1.value]), (stage, lines[i][1])
                assert np.array_equal(res["regs"][off[2 * i + 1]:off[2 * i + 2]], a2[:n2.value]), (stage, lines[i][1])


def test_candidates_vs_reference_c1(emab):
    """BASELINE config 1 with planted repeats + indels: 3000 pairs against the compiled reference (without oracle/_ref:
    against the recorded digest of the reference's candidates)."""
    from tools import synth
    p = synth.build_config("c1_rep", helpers.DATA_ROOT, indexer=emab.index_build)
    ix = emab.Index(p["fasta"])
    ctx = emab.Context(ix)
    lines = helpers.read_bucket(p["bucket"], 3000)
    got, res = pipeline_candidates(emab, ctx, lines)
    if not helpers.have_ref():
        d = helpers.sha(got)
        assert d == helpers.recorded_reference("candidates_c1_rep_3000", d), "candidates differ from the reference's recorded ones"
        return
    ref_lib = helpers.ref()
    ref_lib.ref_ema_init.argtypes = [C.c_char_p, C.c_char_p]
    assert ref_lib.ref_ema_init(p["fasta"].encode(), b"10x") == 0
    bad = 0
    for f, g in zip(lines, got):
        ints = np.zeros((4096, 11), np.int64)
        sc = np.zeros(4096, np.float64)
        cg = np.zeros((4096, 64), np.uint32)
        n = ref_lib.ref_ema_candidates(f[1][1:].encode(), f[2].encode(), f[3].encode(), f[4].encode(), f[5].encode(),
                                       _p(ints, C.c_int64), _p(sc, C.c_double), _p(cg, C.c_uint32), 64, 4096)
        want = [(int(i[0]), int(i[1]), int(i[2]), int(i[3]), int(i[4]), int(i[5]), int(i[6]), int(i[7]), int(i[8]), int(i[9]), float(s),
                 tuple(int(c) for c in c_[:i[9]])) for i, s, c_ in zip(ints[:n], sc[:n], cg[:n])]
        if g != want:
            bad += 1
            if bad == 1:
                first = (f[1], g, want)
    assert bad == 0, f"{bad} pairs differ, first: {first}"


def test_edge_cases(emab):
    ix = emab.Index(os.path.join(G, "tiny_rep", "ref.fa"))
    ctx = emab.Context(ix)
    res = emab.align_pairs(ctx, [])
    assert len(res["alns"]) == 0
    lines = helpers.read_bucket(os.path.join(G, "tiny_rep", "ema-bin-000.10x"), 4)
    r = helpers.nt4(lines[0][2])
    # all-N mate, too-short mate, ragged lengths in one batch
    reads = [r, np.full(150, 4, np.uint8), r[:15], helpers.nt4(lines[1][4]), helpers.nt4(lines[2][2])[:60], helpers.nt4(lines[2][4])]
    res = emab.align_pairs(ctx, reads)
    assert res["n_regs"][1] == 0 and res["n_regs"][2] == 0 and res["n_regs"][0] >= 1
    with pytest.raises(emab.EmabError):
        emab.align_pairs(ctx, [np.zeros(400, np.uint8), r])


def test_wide_dense_sa_branch(emab, monkeypatch):
    """hg38-sized indexes (2*l_pac >= 2^32, BASELINE configs[2]) keep the dense SA as u64; EMAB_SA64=1 forces
    that table on the small golden index: every SA slot and the golden candidates must be unchanged."""
    monkeypatch.setenv("EMAB_SA64", "1")
    ix = emab.Index(os.path.join(G, "tiny_rep", "ref.fa"))
    monkeypatch.delenv("EMAB_SA64")
    ctx = emab.Context(ix)
    allk = np.arange(0, ix.seq_len + 1, dtype=np.int64)
    assert np.array_equal(emab.sa_batch(ctx, allk, mode=0), emab.sa_batch(ctx, allk, mode=1)), "every SA slot (u64 table)"
    want = helpers.cands_from_golden(np.load(os.path.join(G, "cand_golden.npz")))
    lines = helpers.read_bucket(os.path.join(G, "tiny_rep", "ema-bin-000.10x"))
    got, _ = pipeline_candidates(emab, ctx, lines)
    assert got == want


def test_rescue_plan_is_transparent(emab, monkeypatch):
    """mate rescue as plan + batched ksw_align2 + replay (pipeline.cu) must return what the single sequential
    warp-per-pair kernel returns — candidates, regions per read and the DP cells the reference's loop visits —
    on the golden bucket and on the repeat/indel variant of BASELINE configs[0] (where rescues chain)."""
    from tools import synth
    cases = [(os.path.join(G, "tiny_rep", "ref.fa"), helpers.read_bucket(os.path.join(G, "tiny_rep", "ema-bin-000.10x")))]
    p = synth.build_config("c1_rep", helpers.DATA_ROOT, indexer=emab.index_build)
    cases.append((p["fasta"], helpers.read_bucket(p["bucket"])))
    for pre, lines in cases:
        ix = emab.Index(pre)
        monkeypatch.setenv("EMAB_RESCUE_PLAN", "0")
        ctx0 = emab.Context(ix)
        monkeypatch.delenv("EMAB_RESCUE_PLAN")
        ctx1 = emab.Context(ix)
        a, ra = pipeline_candidates(emab, ctx0, lines)
        b, rb = pipeline_candidates(emab, ctx1, lines)
        assert a == b
        assert np.array_equal(ra["n_regs"], rb["n_regs"])
        sa, sb = ra["stats"], rb["stats"]
        assert sa.local_cells == sb.local_cells and sa.local_cells > 0
        assert sa.rescue_planned_cells == 0 and sb.rescue_planned_cells > 0
        n_sw = max(1, sb.local_cells // 60000)  # ~ number of ksw_align2 calls
        assert sb.rescue_unplanned * 10 <= n_sw, f"the plan should foresee nearly every alignment ({sb.rescue_unplanned} of ~{n_sw} were not)"
        print(f"rescue plan: {sb.rescue_planned_cells} cells planned, {sb.local_cells} consumed, {sb.rescue_unplanned} alignments unplanned")


def test_wave_plans_are_transparent(emab, monkeypatch):
    """ksw_extend2 / ksw_global2 run ahead as bucket-wide thread-per-task waves (ext_wave.cuh, glob_wave.cuh) and replayed by the
    per-read control flow must give what the inline warp-per-task path gives: candidates, regions per read, and the
    DP cells the reference's loops visit — on the golden bucket and on the repeat/indel variant of BASELINE configs[0]."""
    from tools import synth
    cases = [(os.path.join(G, "tiny_rep", "ref.fa"), helpers.read_bucket(os.path.join(G, "tiny_rep", "ema-bin-000.10x")))]
    p = synth.build_config("c1_rep", helpers.DATA_ROOT, indexer=emab.index_build)
    cases.append((p["fasta"], helpers.read_bucket(p["bucket"])))
    for pre, lines in cases:
        ix = emab.Index(pre)
        monkeypatch.setenv("EMAB_EXT_PLAN", "0")
        monkeypatch.setenv("EMAB_GLOB_PLAN", "0")
        ctx0 = emab.Context(ix)
        monkeypatch.delenv("EMAB_EXT_PLAN")
        monkeypatch.delenv("EMAB_GLOB_PLAN")
        ctx1 = emab.Context(ix)
        a, ra = pipeline_candidates(emab, ctx0, lines)
        b, rb = pipeline_candidates(emab, ctx1, lines)
        assert a == b
        assert np.array_equal(ra["n_regs"], rb["n_regs"])
        sa, sb = ra["stats"], rb["stats"]
        assert sa.extend_cells == sb.extend_cells and sa.extend_cells > 0
        assert sa.global_cells == sb.global_cells
        assert sa.ext_planned_cells == 0 and sb.ext_planned_cells > 0
        print(f"ext plan: {sb.ext_planned_cells} cells planned, {sb.extend_cells} consumed, {sb.ext_unplanned} extensions inline; "
              f"glob plan: {sb.glob_planned_cells} planned, {sb.global_cells} consumed, {sb.glob_unplanned} inline")

"""Index construction (SURVEY.md §8 f4): emab_index_build replaces `bwa index` (bwa/bwtindex.c:255-323).

The bar is byte identity of all five files with the reference's own `bwa index` output:
  * without a GPU: the host half (FASTA -> .pac/.ann/.amb, bns_fasta2bntseq) against the committed index of
    tests/golden/tiny_rep and, where oracle/_ref/bwa exists, against `bwa index` on a FASTA with ambiguity runs,
    lower case, header comments, blank lines and CRLF line ends;
  * on the GPU (-m gpu): the whole build against the committed index and against `bwa index` on references
    with planted repeats, single- and multi-chunk, below and above the 50 Mbp switch of the reference's own
    BWT algorithm (bwa/bwtindex.c:276).
"""
import filecmp
import os
import shutil
import subprocess

import numpy as np
import pytest

import ema_b200
import helpers

GOLD = os.path.join(helpers.ROOT, "tests", "golden", "tiny_rep")
BWA = os.path.join(helpers.REF_DIR, "bwa")
EXTS = (".pac", ".ann", ".amb", ".bwt", ".sa")


def _messy_fasta(path, seed=5, n_contigs=3, ln=20011, crlf=False):
    rng = np.random.default_rng(seed)
    nl = b"\r\n" if crlf else b"\n"
    with open(path, "wb") as f:
        f.write(b"; leading junk before the first header\n")
        for c in range(n_contigs):
            seq = np.frombuffer(b"ACGT", dtype=np.uint8)[rng.integers(0, 4, ln + c)].copy()
            lower = rng.random(len(seq)) < 0.3
            seq[lower] += 32
            for _ in range(6):  # ambiguity runs: N, n, mixed codes, a run touching the contig end
                p = int(rng.integers(0, len(seq) - 40))
                seq[p:p + int(rng.integers(1, 30))] = rng.choice(np.frombuffer(b"NnRYK-", dtype=np.uint8))
            seq[-3:] = ord("N")
            if c == 1:
                seq[:2] = ord("N")
            f.write(b">ctg%d" % c + (b" some comment %d" % c if c != 1 else b"") + nl)
            w = 70 if c != 2 else 61
            for i in range(0, len(seq), w):
                f.write(seq[i:i + w].tobytes() + nl)
                if c == 0 and i == 140:
                    f.write(b"\n")  # a blank line inside a record


def test_pack_matches_committed_index(tmp_path):
    fa = str(tmp_path / "ref.fa")
    shutil.copy(os.path.join(GOLD, "ref.fa"), fa)
    ema_b200.index_pack_fasta(fa)
    for e in (".pac", ".ann", ".amb"):
        assert filecmp.cmp(fa + e, os.path.join(GOLD, "ref.fa" + e), shallow=False), e


@pytest.mark.parametrize("crlf", [False, True])
def test_pack_matches_bwa_on_messy_fasta(tmp_path, crlf):
    fa = str(tmp_path / "m.fa")
    _messy_fasta(fa, crlf=crlf)
    ema_b200.index_pack_fasta(fa, str(tmp_path / "ours"))
    _same_as_bwa(f"fa2pac_messy_crlf{int(crlf)}", ["fa2pac", "-f", fa, str(tmp_path / "theirs")], str(tmp_path / "ours"),
                 str(tmp_path / "theirs"), (".pac", ".ann", ".amb"))


def _same_index(a, b):
    for e in EXTS:
        assert filecmp.cmp(a + e, b + e, shallow=False), "%s differs" % e


def _same_as_bwa(key, bwa_args, ours, theirs, exts=EXTS):
    """ours.<ext> against what `bwa <bwa_args>` writes to theirs.<ext>: the files themselves where oracle/_ref/bwa is built,
    elsewhere the recorded digests of bwa's files for case `key`"""
    if os.path.exists(BWA):
        subprocess.run([BWA] + bwa_args, check=True, capture_output=True)
        for e in exts:
            assert filecmp.cmp(ours + e, theirs + e, shallow=False), "%s differs" % e
        return
    for e in exts:
        d = helpers.sha(open(ours + e, "rb").read())
        assert d == helpers.recorded_reference(key + e, d), "%s differs" % e


@pytest.mark.gpu
@pytest.mark.parametrize("chunk_bits", [None, "3"])
def test_build_matches_committed_index(tmp_path, chunk_bits, monkeypatch):
    if chunk_bits:
        monkeypatch.setenv("EMAB_INDEX_CHUNK_BITS", chunk_bits)
    fa = str(tmp_path / "ref.fa")
    shutil.copy(os.path.join(GOLD, "ref.fa"), fa)
    st = ema_b200.index_build(fa)
    assert st["n_chunks"] >= (1 if not chunk_bits else 2)
    _same_index(fa, os.path.join(GOLD, "ref.fa"))


@pytest.mark.gpu
def test_build_matches_bwa_messy_and_repeats(tmp_path):
    from tools import synth
    # (a) ambiguity codes etc.; (b) 5 Mbp with planted 2-10 kb repeats; (c) a text that is one long tandem repeat plus
    # a poly-A tail (deep ties, suffixes that run into the end of the text)
    fa_a = str(tmp_path / "a.fa")
    _messy_fasta(fa_a)
    fa_b = str(tmp_path / "b.fa")
    synth.write_fasta(fa_b, synth.make_reference(5, 1_000_000, 7, dup_every=100_000))
    fa_c = str(tmp_path / "c.fa")
    rng = np.random.default_rng(3)
    unit = rng.integers(0, 4, 97, dtype=np.uint8)
    synth.write_fasta(fa_c, [np.concatenate([np.tile(unit, 400), rng.integers(0, 4, 1000, dtype=np.uint8), np.zeros(300, np.uint8)]),
                             np.concatenate([np.zeros(200, np.uint8), np.tile(unit, 50)])])
    for tag, fa in (("a", fa_a), ("b", fa_b), ("c", fa_c)):
        ema_b200.index_build(fa, fa + ".ours")
        _same_as_bwa(f"bwa_index_messy_and_repeats_{tag}", ["index", "-p", fa + ".theirs", fa], fa + ".ours", fa + ".theirs")


@pytest.mark.gpu
def test_build_matches_bwa_above_50mbp(tmp_path):
    """above 50 Mbp the reference switches from SA-IS to bwtsw (bwa/bwtindex.c:276); the files must still be identical"""
    from tools import synth
    fa = str(tmp_path / "big.fa")
    synth.write_fasta(fa, synth.make_reference(4, 13_000_000, 11, dup_every=200_000))
    st = ema_b200.index_build(fa, fa + ".ours")
    _same_as_bwa("bwa_index_above_50mbp", ["index", "-p", fa + ".theirs", fa], fa + ".ours", fa + ".theirs")
    assert st["l_pac"] == 52_000_000

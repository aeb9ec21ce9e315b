"""GPU parity tests (-m gpu) of the cases the reference handles by growing a list or reading a stream, where this
implementation has capacities and batches (VERDICT r1 "what's weak" 2, "missing" 2):

* a read engineered to have far more than 128 SA intervals (the per-read capacity of one seeding pass): the bucket is
  seeded again with more room and the SAM must still be the reference's;
* -1 input cut into many small device batches (EMAB_FASTQ_BATCH) must give the bytes of the one-batch run and of the
  reference, cloud ids included;
* the full-size buckets of BASELINE configs[1] and the configs[2]-shaped run on the 3.1 Gbp reference (u64 suffix array),
  plain and -d, promoted from the round-1 tool logs to tests.
"""
import os
import subprocess

import numpy as np
import pytest

import helpers
from test_gpu_sam import CLI
from test_gpu_platforms import _faketime_env

pytestmark = pytest.mark.gpu
REF_EMA = helpers.ref_bin("ema")


def _compare(key, cmd_tail, tmp_path, env=None, ours_env=None, threads="8", min_records=1):
    our_sam = tmp_path / "ours.sam"
    e = dict(env or os.environ)
    e.update(ours_env or {})
    subprocess.run([CLI, "align"] + cmd_tail + ["-t", threads, "-o", str(our_sam)], check=True, env=e)
    return helpers.compare_sam_with_reference(
        key, our_sam.read_bytes(),
        lambda out: subprocess.run([REF_EMA, "align"] + cmd_tail + ["-t", "1", "-o", out], check=True, stderr=subprocess.DEVNULL, env=env),
        tmp_path, min_records=min_records)


def test_read_with_many_sa_intervals(tmp_path):
    """163 supermaximal exact matches of 28 bp tile one 190-bp read (each planted once in the reference with mismatching
    flanks): mem_collect_intv returns far more than EMAB_MAX_INTV = 128 intervals for it."""
    import ema_b200
    from tools import synth
    rng = np.random.default_rng(99)
    contigs = synth.make_reference(2, 150_000, 5, 0)
    L, K = 190, 28
    read = rng.integers(0, 4, L, dtype=np.uint8)
    spots = rng.permutation(np.arange(1000, 149_000, 400))[: L - K + 1]
    for i, pos in enumerate(spots):
        c = contigs[i & 1]
        c[pos:pos + K] = read[i:i + K]
        if i > 0:
            c[pos - 1] = (read[i - 1] + 1) & 3          # the match must not extend to the left ...
        if i + K < L:
            c[pos + K] = (read[i + K] + 2) & 3          # ... nor to the right
    fa = str(tmp_path / "ref.fa")
    synth.write_fasta(fa, contigs)
    ema_b200.index_build(fa)
    sim = synth.simulate_pairs(contigs, 6, 40, 17, r1_len=127, r2_len=150)
    bucket = str(tmp_path / "ema-bin-000")
    synth.write_bucket(bucket, sim)
    # one more pair in the first barcode: the engineered read and an ordinary mate
    lines = open(bucket, "rb").read().splitlines()
    bc = lines[0].split()[0]
    mate = synth.ACGT[contigs[0][5000:5150]].tobytes()
    lines.append(bc + b" @engineered " + synth.ACGT[read].tobytes() + b" " + b"I" * L + b" " + mate + b" " + b"I" * 150)
    open(bucket, "wb").write(b"\n".join(lines) + b"\n")
    ctx = ema_b200.Context(ema_b200.Index(fa))
    ivs, _ = ema_b200.smem_batch(ctx, [helpers.nt4(synth.ACGT[read].tobytes())], max_intv=8192)
    assert len(ivs[0]) > 128, "the construction should exceed the default capacity (got %d intervals)" % len(ivs[0])
    body = _compare("many_sa_intervals", ["-s", bucket, "-r", fa, "-p", "10x"], tmp_path, min_records=2 * 241)
    assert any(l.startswith(b"engineered\t") for l in body)


def test_seeding_long_interval_lists(tmp_path):
    """A staircase of planted prefixes (S[0:k] for k = 25..70, each once, each followed by a wrong base) makes the forward
    sweep over S change its interval size 46 times: bwt_smem1a's prev/curr lists outgrow the 24 entries the seeding kernel
    keeps in shared memory and continue in its global slab.  The default form must still equal the exact one."""
    import ema_b200
    from tools import synth
    rng = np.random.default_rng(123)
    contigs = synth.make_reference(1, 80_000, 7, 0)
    S = rng.integers(0, 4, 70, dtype=np.uint8)
    c = contigs[0]
    for n, k in enumerate(range(25, 71)):
        pos = 1000 + 1500 * n
        c[pos:pos + k] = S[:k]
        c[pos - 1] = (S[0] + 1 + (n & 1)) & 3           # nothing extends the copies to the left in step
        if k < 70:
            c[pos + k] = (S[k] + 1) & 3
    fa = str(tmp_path / "ref.fa")
    synth.write_fasta(fa, contigs)
    ema_b200.index_build(fa)
    ctx = ema_b200.Context(ema_b200.Index(fa))
    reads = []
    for cut in (70, 60, 45):
        for lead in (0, 7, 30):
            reads.append(np.concatenate([rng.integers(0, 4, lead, dtype=np.uint8), S[:cut], rng.integers(0, 4, 100 - cut, dtype=np.uint8)]))
            reads.append(np.ascontiguousarray((3 - reads[-1])[::-1]))
    got, _ = ema_b200.smem_batch(ctx, reads, max_intv=512)
    ema_b200.set_seed_mode(ctx, 3)
    want, _ = ema_b200.smem_batch(ctx, reads, max_intv=512)
    ema_b200.set_seed_mode(ctx, 0)
    assert max(len(w) for w in want) >= 3
    sizes = set()
    for a, b in zip(got, want):
        assert len(a) == len(b) and np.array_equal(a[:, [0, 2, 3]], b[:, [0, 2, 3]])
        sizes |= set(int(v) for v in b[:, 2])
    assert len(sizes) >= 3


@pytest.mark.parametrize("platform", ["tru", "10x"])
def test_fastq_stream_small_batches(platform, tmp_path):
    """-1 cut into ~20 device batches: same bytes as the reference (whose cloud ids run through the whole file)."""
    import ema_b200
    from tools import synth
    p = synth.build_config("c1_rep", helpers.DATA_ROOT, indexer=ema_b200.index_build, platform="tru")
    if platform == "10x":   # 10x ids in interleaved FASTQ
        n_contigs, clen, rseed, dup, nbc, ppb, indel = synth.CONFIGS["c1_rep"]
        contigs = synth.make_reference(n_contigs, clen, rseed, dup)
        sim = synth.simulate_pairs(contigs, 60, 50, rseed + 3000, indel=indel)
        fq = str(tmp_path / "reads.fq")
        synth.write_interleaved_fastq(fq, sim, platform="10x")
    else:
        fq = p["bucket"]
    _compare(f"fastq_stream_small_batches_{platform}", ["-1", fq, "-r", p["fasta"], "-p", platform], tmp_path, ours_env={"EMAB_FASTQ_BATCH": "500", "EMAB_WORKERS": "4"}, min_records=1000)


def test_full_size_c2_buckets_plain_and_density(tmp_path):
    """Two full 40 000-pair buckets of BASELINE configs[1] through -x, plain and with -d under the pinned clock (round 1:
    tools/verify_c2.sh, builder-run only)."""
    import ema_b200
    from tools import synth
    n_contigs, clen, rseed, dup, _, _, indel = synth.CONFIGS["c2"]
    d = os.path.join(helpers.DATA_ROOT, "c2_full")
    os.makedirs(d, exist_ok=True)
    fa = os.path.join(d, "ref.fa")
    buckets = [os.path.join(d, f"ema-bin-{b:03d}") for b in range(2)]
    if not all(os.path.exists(b) for b in buckets) or not os.path.exists(fa + ".sa"):
        contigs = synth.make_reference(n_contigs, clen, rseed, dup)
        if not os.path.exists(fa + ".fai"):
            synth.write_fasta(fa, contigs)
        if not os.path.exists(fa + ".sa"):
            ema_b200.index_build(fa)
        for b, path in enumerate(buckets):
            if not os.path.exists(path):
                synth.write_bucket(path, synth.simulate_pairs(contigs, 200, 200, rseed + 1000 + b, indel=indel))
    plain = tmp_path / "plain"; plain.mkdir()
    _compare("full_size_c2_plain", ["-x", "-r", fa, "-p", "10x"] + buckets, plain, threads="16", min_records=160000)
    dens = tmp_path / "dens"; dens.mkdir()
    _compare("full_size_c2_density", ["-x", "-d", "-r", fa, "-p", "10x"] + buckets, dens, env=_faketime_env(tmp_path), threads="16", min_records=160000)


def test_target_regime_3p1gbp(tmp_path):
    """BASELINE configs[2] shape: the 3.1 Gbp synthetic reference (2 * l_pac > 2^32: u64 suffix array, 64-bit coordinates
    everywhere), indexed by emab_index_build, one 40 000-pair bucket plain and one with -d, against the reference binary
    loading the same index.  Needs ~60 GB of HBM and ~25 GB of host memory; about two minutes."""
    import torch
    if torch.cuda.get_device_properties(0).total_memory < 100e9:
        pytest.skip("needs a GPU with > 100 GB")
    out = subprocess.run(["python", os.path.join(helpers.ROOT, "tools", "big_run.py"), "--config", "c3", "--buckets", "1", "--density",
                          "--data-dir", helpers.DATA_ROOT], capture_output=True, text=True, timeout=1500)
    assert out.returncode == 0, out.stderr[-2000:]
    import json
    res = json.loads(out.stdout.strip().splitlines()[-1])
    if os.path.exists(REF_EMA):
        assert res["all_identical"] is True, res["buckets"]
        assert res["density_identical"] is True, res["density"]
    else:   # the MD5s of the reference's SAM bodies, recorded
        for key, md5 in (("target_regime_c3_plain", res["buckets"][0]["md5"]), ("target_regime_c3_density", res["density"][0]["md5"])):
            assert md5 == helpers.recorded_reference(key, md5), key
    assert res["buckets"][0]["records"] == 80000

"""GPU parity tests (-m gpu) of the whole `ema align` path: SAM bytes.  The body must be
byte-identical to the reference's `ema align ... -t 1`; the header is compared minus @PG, which
echoes argv (src/align.c:208-211)."""
import os
import subprocess

import numpy as np
import pytest

import helpers
from helpers import diff_msg, split_sam

pytestmark = pytest.mark.gpu
G = os.path.join(os.path.dirname(__file__), "golden")
CLI = os.path.join(helpers.ROOT, "ema_b200", "ema-b200")


def test_cli_golden_tiny(tmp_path):
    out = tmp_path / "out.sam"
    subprocess.run([CLI, "align", "-s", os.path.join(G, "tiny_rep", "ema-bin-000.10x"), "-r", os.path.join(G, "tiny_rep", "ref.fa"),
                    "-p", "10x", "-t", "4", "-o", str(out)], check=True)
    h1, b1 = split_sam(out.read_bytes())
    h2, b2 = split_sam(open(os.path.join(G, "tiny_rep", "ref.sam"), "rb").read())
    assert h1 == h2
    assert b1 == b2, diff_msg(b1, b2)


def test_cli_errors(tmp_path):
    r = subprocess.run([CLI, "align", "-r", "x.fa"], capture_output=True, text=True)
    assert r.returncode != 0 and "exactly one" in r.stderr
    r = subprocess.run([CLI, "align", "-s", "nope", "-r", os.path.join(G, "tiny_rep", "ref.fa"), "-p", "bogus"], capture_output=True, text=True)
    assert r.returncode != 0 and "invalid platform name" in r.stderr
    r = subprocess.run([CLI, "align", "-s", "nope", "-r", "/nonexistent.fa"], capture_output=True, text=True)
    assert r.returncode != 0 and "could not be opened" in r.stderr


@pytest.mark.parametrize("cfg", ["c1", "c1_rep"])
def test_session_vs_reference_c1(cfg, tmp_path):
    """BASELINE config 1 (10k pairs, 200 barcodes, 5 Mbp) and its repeat/indel variant against the
    reference binary run on the same files."""
    import ema_b200
    from tools import synth
    p = synth.build_config(cfg, helpers.DATA_ROOT, indexer=ema_b200.index_build)
    s = ema_b200.Session(p["fasta"], "10x", threads=8)
    body = s.align_bucket(open(p["bucket"], "rb").read())
    helpers.compare_sam_with_reference(
        f"session_{cfg}", s.header(["ema", "align"]) + body,
        lambda out: subprocess.run([helpers.ref_bin("ema"), "align", "-s", p["bucket"], "-r", p["fasta"], "-p", "10x", "-t", "1", "-o", out],
                                   check=True, stderr=subprocess.DEVNULL), tmp_path, min_records=1)
    st = s.stats
    assert st.n_pairs == p["n_pairs"] and st.launches >= 8


def test_em_posteriors_vs_reference(tmp_path):
    """EM posteriors at full precision (the SAM only carries %.5g): within 1e-6 relative of the
    reference's, with identical chosen alignments (north_star tolerance).  Without oracle/_ref the reference's posteriors
    come from tests/golden/reference/em_posteriors_c1_rep.npz."""
    import ctypes as C
    import ema_b200
    from tools import synth
    p = synth.build_config("c1_rep", helpers.DATA_ROOT, indexer=ema_b200.index_build)
    s = ema_b200.Session(p["fasta"], "10x", threads=8)
    mine = tmp_path / "mine.tsv"
    s.dump_posteriors(str(mine))
    s.align_bucket(open(p["bucket"], "rb").read())
    rows = [ln.rstrip("\n").split("\t") for ln in open(mine)]
    want = {}
    if helpers.have_ref():
        R = helpers.ref()
        R.ref_ema_init.argtypes = [C.c_char_p, C.c_char_p]
        assert R.ref_ema_init(p["fasta"].encode(), b"10x") == 0
        dump = tmp_path / "gamma.tsv"
        R.ref_ema_run_bucket.argtypes = [C.c_char_p, C.c_char_p, C.c_char_p, C.c_int, C.c_int]
        assert R.ref_ema_run_bucket(p["bucket"].encode(), str(tmp_path / "r.sam").encode(), str(dump).encode(), 0, 1) == 0
        for ln in open(dump):
            f = ln.rstrip("\n").split("\t")
            chosen = f[-1].split(":")
            want[(f[0], int(f[1]))] = (int(chosen[0]), int(chosen[1]), float(chosen[2]))
    else:
        name = "em_posteriors_c1_rep.npz"
        path = os.path.join(helpers.RECORDED_DIR, name)
        if not os.path.exists(path) and helpers.RECORD_TO:
            os.makedirs(helpers.RECORD_TO, exist_ok=True)
            path = os.path.join(helpers.RECORD_TO, name)
            np.savez_compressed(path, ident=np.array([r[0] for r in rows], "S"), mate=np.array([int(r[1]) for r in rows], np.int8),
                                chrom=np.array([int(r[2]) for r in rows], np.int32), pos=np.array([int(r[3]) for r in rows], np.int64),
                                gamma=np.array([float(r[4]) for r in rows], np.float64))
        g = np.load(path)
        for i, m, c, q, y in zip(g["ident"], g["mate"], g["chrom"], g["pos"], g["gamma"]):
            want[(i.decode(), int(m))] = (int(c), int(q), float(y))
    n, worst = 0, 0.0
    for ident, mate, chrom, pos, gamma in rows:
        wc, wp, wg = want[(ident, int(mate))]
        assert (wc, wp) == (int(chrom), int(pos)), (ident, mate)
        rel = abs(float(gamma) - wg) / max(abs(wg), 1e-300)
        worst = max(worst, rel)
        n += 1
    assert n == len(want) and n > 15000
    assert worst <= 1e-6, worst


def test_multi_bucket_pipeline_matches_serial(tmp_path):
    """-x mode with several buckets in flight: same bytes as bucket-by-bucket, cloud ids in input order;
    and the CLI's -x output equals the concatenation."""
    import ema_b200
    from tools import synth
    p = synth.build_config("c1_rep", helpers.DATA_ROOT, indexer=ema_b200.index_build)
    lines = open(p["bucket"], "rb").read().split(b"\n")
    lines = [l for l in lines if l]
    parts = [b"\n".join(lines[i::4]) + b"\n" for i in range(4)] + [b""]
    s1 = ema_b200.Session(p["fasta"], "10x", threads=8)
    serial = [s1.align_bucket(d) for d in parts]
    s2 = ema_b200.Session(p["fasta"], "10x", threads=8)
    s2.set_workers(3)
    multi = s2.align_buckets(parts)
    assert multi == serial
    assert sum(len(x) for x in multi) > 1_000_000
    # the same buckets handed over in page-locked buffers (copied to the device without the staging copy), mixed with plain ones
    s3 = ema_b200.Session(p["fasta"], "10x", threads=8)
    s3.set_workers(3)
    mixed = [ema_b200.PinnedText(d) if i % 2 == 0 else d for i, d in enumerate(parts)]
    assert s3.align_buckets(mixed) == serial
    assert s3.align_bucket(ema_b200.PinnedText(parts[1])) is not None
    files = []
    for i, d in enumerate(parts[:4]):
        f = tmp_path / f"b{i}"
        f.write_bytes(d)
        files.append(str(f))
    out = tmp_path / "x.sam"
    subprocess.run([CLI, "align", "-x", "-r", p["fasta"], "-p", "10x", "-t", "8", "-o", str(out)] + files, check=True)
    _, body = split_sam(out.read_bytes())
    assert b"\n".join(body) + b"\n" == b"".join(serial)


def test_multi_device_session_matches_serial(tmp_path):
    """several index replicas in one process (emab_session_add_device / EMAB_DEVICES): workers on different replicas take
    buckets from one shared counter (host-side work stealing, SURVEY.md 8e).  On a one-GPU box the second replica is a
    second copy on cuda:0 — the same code path; with more GPUs visible the replicas go to different devices.  Output
    and cloud ids must be those of the serial run."""
    import torch
    import ema_b200
    from tools import synth
    p = synth.build_config("c1_rep", helpers.DATA_ROOT, indexer=ema_b200.index_build)
    lines = [l for l in open(p["bucket"], "rb").read().split(b"\n") if l]
    parts = [b"\n".join(lines[i::6]) + b"\n" for i in range(6)]
    s1 = ema_b200.Session(p["fasta"], "10x", threads=8)
    serial = [s1.align_bucket(d) for d in parts]
    second = 1 if torch.cuda.device_count() > 1 else 0
    s2 = ema_b200.Session(p["fasta"], "10x", threads=8)
    s2.add_device(second)
    s2.set_workers(4)
    assert s2.align_buckets(parts) == serial
    assert s2.align_bucket(parts[0])[:200] != b""          # single calls still work after the multi-device run
    files = []
    for i, d in enumerate(parts):
        f = tmp_path / f"b{i}"
        f.write_bytes(d)
        files.append(str(f))
    out = tmp_path / "x.sam"
    env = dict(os.environ, EMAB_DEVICES=f"0,{second}", EMAB_HOST_PROFILE="1")
    r = subprocess.run([CLI, "align", "-x", "-r", p["fasta"], "-p", "10x", "-t", "8", "-o", str(out)] + files, check=True, env=env,
                       capture_output=True, text=True)
    assert "buckets per device" in r.stderr, r.stderr[-500:]
    _, body = split_sam(out.read_bytes())
    assert b"\n".join(body) + b"\n" == b"".join(serial)


def test_single_bucket_split_over_replicas():
    """fewer buckets than GPUs (SURVEY.md 8e): one bucket is cut at barcode boundaries into one part per worker, the parts
    run on the session's index replicas concurrently, and the joined SAM — cloud ids included — is the serial run's."""
    import torch
    import ema_b200
    from tools import synth
    p = synth.build_config("c1_rep", helpers.DATA_ROOT, indexer=ema_b200.index_build)
    data = open(p["bucket"], "rb").read()
    serial = ema_b200.Session(p["fasta"], "10x", threads=8).align_bucket(data)
    s2 = ema_b200.Session(p["fasta"], "10x", threads=8)
    s2.add_device(1 if torch.cuda.device_count() > 1 else 0)
    s2.set_workers(4)
    split = s2.align_bucket(data)
    assert split == serial
    assert s2.align_bucket(data).count(b"\n") == serial.count(b"\n")


def test_raw_fastq_through_count_preproc_align(tmp_path):
    """From RAW 10x reads: `count` -> `preproc` -> `align` with this build against the same three steps of the reference —
    identical bucket files (host/preproc.cpp), identical SAM (the buckets carry corrected barcodes, trimmed read 1).
    Without oracle/_ref the reference's bucket files and SAM are represented by their recorded digests."""
    import filecmp
    import ema_b200
    from tools import synth
    p = synth.build_config("c1_rep", helpers.DATA_ROOT, indexer=ema_b200.index_build)
    n_contigs, clen, rseed, dup, nbc, ppb, indel = synth.CONFIGS["c1_rep"]
    contigs = synth.make_reference(n_contigs, clen, rseed, dup)
    sim = synth.simulate_pairs(contigs, 40, 60, rseed + 4242, indel=indel)
    fq, wl = str(tmp_path / "raw.fq"), str(tmp_path / "wl.txt")
    synth.write_raw_10x_fastq(fq, wl, sim)
    have_ref = os.path.exists(helpers.ref_bin("ema"))
    outs = {}
    for tag, exe in ((("ref", helpers.ref_bin("ema")),) if have_ref else ()) + (("our", CLI),):
        with open(fq, "rb") as f:
            subprocess.run([exe, "count", "-w", wl, "-o", str(tmp_path / tag)], stdin=f, check=True, stderr=subprocess.DEVNULL)
        with open(fq, "rb") as f:
            subprocess.run([exe, "preproc", "-w", wl, "-n", "3", "-t", "2", "-o", str(tmp_path / (tag + "_b")), str(tmp_path / tag) + ".ema-ncnt"],
                           stdin=f, check=True, stderr=subprocess.DEVNULL)
        outs[tag] = tmp_path / (tag + "_b")
    names = sorted(os.listdir(outs["our"]))
    assert names == ["ema-bin-000", "ema-bin-001", "ema-bin-002", "ema-nobc"]
    if have_ref:
        assert names == sorted(os.listdir(outs["ref"]))
        for n in names:
            assert filecmp.cmp(outs["ref"] / n, outs["our"] / n, shallow=False), n
    else:
        for n in names:
            d = helpers.sha((outs["our"] / n).read_bytes())
            assert d == helpers.recorded_reference(f"raw_fastq_preproc_{n}", d), n
    bucket = str(outs["our"] / "ema-bin-001")
    our_sam = tmp_path / "our.sam"
    subprocess.run([CLI, "align", "-s", bucket, "-r", p["fasta"], "-p", "10x", "-t", "8", "-o", str(our_sam)], check=True, stderr=subprocess.DEVNULL)
    helpers.compare_sam_with_reference(
        "raw_fastq_align", our_sam.read_bytes(),
        lambda out: subprocess.run([helpers.ref_bin("ema"), "align", "-s", bucket, "-r", p["fasta"], "-p", "10x", "-t", "1", "-o", out],
                                   check=True, stderr=subprocess.DEVNULL), tmp_path, min_records=1001)

"""GPU tests (-m gpu) of what a ctx keeps between calls: the resident SW inputs and outputs
(emab_extend_resident_load) are the ctx's own and outlive every other entry point run on it."""
import os

import numpy as np
import pytest

import helpers

pytestmark = pytest.mark.gpu
G = os.path.join(os.path.dirname(__file__), "golden")


@pytest.fixture(scope="module")
def emab():
    import ema_b200
    return ema_b200


@pytest.fixture(scope="module")
def tiny(emab):
    return emab.Index(os.path.join(G, "tiny_rep", "ref.fa"))


def resident_tasks(n, seed):
    """n fixed-length extension tasks: a 150-bp query, a 250-bp target that starts with it at 2 % substitutions"""
    rng = np.random.default_rng(seed)
    t = rng.integers(0, 4, size=(n, 250), dtype=np.uint8)
    q = t[:, :150].copy()
    flip = rng.random(q.shape) < 0.02
    q[flip] = (q[flip] + rng.integers(1, 4, size=int(flip.sum()), dtype=np.uint8)) % 4
    return q, t, np.full(n, 19, np.int32)


@pytest.mark.parametrize("sw_mode", [0, 1], ids=["lanes", "warp"])
def test_resident_survives_other_calls(emab, tiny, sw_mode):
    ctx = emab.Context(tiny)
    emab.set_sw_mode(ctx, sw_mode)
    q, t, h0 = resident_tasks(3000, 11)
    n = emab.extend_resident_load(ctx, q, t, h0)
    want, want_cells, _ = emab.extend_resident_run(ctx, n)
    assert (want[:, 0] > 0).all()
    # every other entry point that runs device work on the ctx, with batches of other sizes than the resident one
    lines = helpers.read_bucket(os.path.join(G, "tiny_rep", "ema-bin-000.10x"))
    reads = []
    for f in lines:
        reads += [helpers.nt4(f[2]), helpers.nt4(f[4])]
    assert emab.align_pairs(ctx, reads)["alns"].size > 0
    g = np.load(os.path.join(G, "fm_golden.npz"))
    emab.smem_batch(ctx, [g["reads"][g["roff"][i]:g["roff"][i + 1]] for i in range(len(g["roff"]) - 1)])
    emab.sa_batch(ctx, np.arange(0, tiny.seq_len + 1, dtype=np.int64))
    qs, ts, eh0 = helpers.random_extend_tasks(5000, 12, max_q=256)
    emab.extend_batch(ctx, qs, ts, eh0)
    ws = np.array([abs(len(a) - len(b)) + 20 for a, b in zip(qs, ts)], dtype=np.int32)
    emab.global_batch(ctx, qs, ts, ws, max_cigar=600)
    got, got_cells, _ = emab.extend_resident_run(ctx, n)
    assert np.array_equal(got, want) and got_cells == want_cells

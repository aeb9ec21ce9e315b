"""ema_b200 — B200-native (sm_100a CUDA) implementation of the `ema align` hot path.

The product is the C-ABI shared library ``libema_b200.so`` (include/ema_b200.h) and the
``ema-b200`` CLI built from ema_b200/csrc.  This package is the thin ctypes mirror used by the
tests and bench.py; it contains no compute of its own and no CPU fallback: every call fails loudly
when the CUDA library or a GPU is missing.
"""
from ._lib import (EmabError, Index, Context, lib, extend_batch, global_batch, local_batch,  # noqa: F401
                   smem_batch, sa_batch, align_pairs, ALN_DTYPE, Session, PinnedText, RunStats, set_sw_mode, set_seed_mode,
                   extend_resident_load, extend_resident_run, int_peak, index_build, index_pack_fasta, parse_bucket,
                   bgzf_eof, bgzf_compress, bgzf_inflate, bam_merge, bam_merge_header)

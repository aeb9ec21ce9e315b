/*
 * ema_b200.h — the C ABI of libema_b200.so: a B200-native (sm_100a CUDA) implementation of the
 * `ema align` hot path, exported as the drop-in for the reference's BWA bridge
 * (reference: include/bwabridge.h:19-22,92-106 as used from src/align.c:986-1061).
 *
 * Conventions
 *   - plain pointers and sizes only; every function returns EMAB_OK (0) or a negative error code,
 *     and never calls exit() (the reference bridge asserts / exits: src/bwabridge.c:81-84);
 *     emab_last_error() returns a message for the calling thread.
 *   - all buffers passed in are HOST buffers owned by the caller; host<->device copies happen
 *     inside the call.  Output buffers are caller-allocated with the stated capacities.
 *   - sequences are nt4 codes (A,C,G,T,other -> 0,1,2,3,4 : bwa/bntseq.c nst_nt4_table) unless a
 *     function says ASCII.
 *   - there is no CPU implementation behind any entry point: without a CUDA device every compute
 *     call fails with EMAB_ERR_CUDA.
 */
#ifndef EMA_B200_H
#define EMA_B200_H
#include <stdint.h>
#include <stdio.h>

#ifdef __cplusplus
extern "C" {
#endif

#define EMAB_OK 0
#define EMAB_ERR_IO (-1)
#define EMAB_ERR_CUDA (-2)
#define EMAB_ERR_ARG (-3)
#define EMAB_ERR_OVERFLOW (-4)
#define EMAB_ERR_NOMEM (-5)

typedef struct emab_index emab_index_t; /* FM index + packed reference resident in one GPU's HBM */
typedef struct emab_ctx emab_ctx_t;     /* one worker: a CUDA stream + its device scratch */

const char *emab_last_error(void);
int emab_version(void);
int emab_device_count(int *n);

/* ---- index: replaces load_reference / bwa_idx_load (src/bwabridge.c:76-96, bwa/bwa.c:271-316).
 * Reads <prefix>.bwt/.sa/.pac/.ann/.amb as written by `bwa index`, uploads them to `device` and
 * builds the dense suffix array there.  info[12] = l_pac, n_seqs, primary, seq_len, L2[0..4],
 * sa_intv, n_sa, bwt_size(u32) — the same fields bwt_t/bntseq_t expose. */
int emab_index_load(const char *prefix, int device, emab_index_t **out);
void emab_index_free(emab_index_t *ix);
int emab_index_info(const emab_index_t *ix, int64_t info[12]);
int emab_index_contig(const emab_index_t *ix, int i, int64_t *offset, int32_t *len, char *name, int name_cap);
double emab_index_build_ms(const emab_index_t *ix); /* device time spent densifying the SA */

/* ---- index construction: replaces `bwa index <fasta>` (bwa/bwtindex.c:255-323 bwa_idx_build =
 * bns_fasta2bntseq + is_bwt/bwt_bwtgen2 + bwt_bwtupdate_core + bwt_cal_sa), the step `ema align -r` depends on.
 * Reads the FASTA at fasta_path, sorts the suffixes of forward + reverse complement on `device` and writes
 * <prefix>.pac/.ann/.amb/.bwt/.sa byte-identical to the reference's (prefix NULL = fasta_path, as `bwa index` does).
 * Needs about 5 bytes of HBM per base of the reference on top of the chunk buffers (see csrc/indexbuild.cu). */
typedef struct {
	int64_t l_pac, primary;
	int32_t n_seqs, n_holes;
	int32_t chunk_bits, n_chunks;     /* the key space was cut into 2^chunk_bits chunks, n_chunks of them non-empty */
	int64_t max_chunk;                /* suffixes in the largest chunk */
	int64_t n_tied;                   /* suffixes that shared their first 29 bases with another one */
	int32_t max_rounds, pad;          /* tie-refinement rounds of the slowest chunk */
	double ms_pack, ms_sort, ms_occ, ms_write, ms_total;  /* FASTA -> pac (host) | suffix sort + BWT/SA emit | Occ | file writes */
} emab_index_build_stats_t;
int emab_index_build(const char *fasta_path, const char *prefix, int device, emab_index_build_stats_t *stats);
/* the host half on its own (= `bwa fa2pac -f`): <prefix>.pac/.ann/.amb only; needs no GPU */
int emab_index_pack_fasta(const char *fasta_path, const char *prefix);

/* ---- the producers of the bucket format (host code; need no GPU) ----------------------------
 * emab_count   = count()   (cpp/count.h, cpp/count.cc:38-182):   interleaved FASTQ (in: NULL = stdin) -> <prefix>.ema-ncnt, .ema-fcnt
 * emab_preproc = correct() (cpp/correct.h, cpp/correct.cc:271-633): the count files + the same FASTQ -> <dir>/ema-bin-NNN, ema-nobc
 * Files are byte-identical to the reference's (tests/test_preproc.py); is_haplotag as the reference's -p (whitelist_path may be NULL). */
int emab_count(const char *whitelist_path, const char *output_prefix, uint64_t max_map_bytes, int is_haplotag, FILE *in);
int emab_preproc(const char *whitelist_path, const char *const *count_files, int n_count_files, const char *output_dir,
                 int do_h2, uint64_t buffer_size, int do_bx_format, int n_threads, int n_buckets, int is_haplotag, FILE *in);

int emab_ctx_create(emab_index_t *ix, emab_ctx_t **out);  /* ix may be NULL for the sequence-only SW calls */
void emab_ctx_free(emab_ctx_t *ctx);
/* Makes the ctx's device current on the calling thread.  Every entry point that takes a ctx does this itself; a
 * thread that allocates pinned memory before its first ctx call uses it to stay off device 0. */
int emab_ctx_make_current(emab_ctx_t *ctx);
/* how the calling thread waits for the ctx's stream: 0 = poll briefly, then sleep between polls (frees the core: for hosts with
 * few cores per GPU), 1 = spin (lowest latency, the default of a bare ctx), 2 = blocking-sync event.  EMAB_SYNC=spin|block|nap overrides. */
int emab_ctx_set_wait(emab_ctx_t *ctx, int mode);
/* device time (ms, CUDA events on the ctx stream) of the kernels launched by the last call, and
 * the number of kernel launches it made */
double emab_last_kernel_ms(const emab_ctx_t *ctx);
int emab_last_launches(const emab_ctx_t *ctx);

/* ---- Smith-Waterman batches (sequence-only; one warp per task) -------------------------------
 * q/t are concatenated nt4 strings with n+1 int64 offsets.  Scoring is BWA-MEM's default
 * (a=1,b=4,o=6,e=1 both ways: bwa/bwamem.c:79-81).  *cells (optional) receives the number of DP
 * cells visited (the roofline unit of SURVEY.md §8d).
 *
 * emab_extend_batch  = ksw_extend2 (bwa/ksw.c:416) ; out[6n] = score,qle,tle,gtle,gscore,max_off
 * emab_global_batch  = ksw_global2 (bwa/ksw.c:540) ; out[2n] = score,n_cigar ; cigar[n*max_cigar]
 * emab_local_batch   = ksw_align2 with KSW_XSUBO|KSW_XSTART|19 (+KSW_XBYTE when qlen<250), the
 *                      mem_matesw call (bwa/bwamem_pair.c:176-177) ; out[7n] = score,te,qe,score2,te2,tb,qb
 */
int emab_extend_batch(emab_ctx_t *ctx, int n, const uint8_t *q, const int64_t *qoff, const uint8_t *t, const int64_t *toff,
                      const int32_t *h0, int w, int end_bonus, int zdrop, int32_t *out, int64_t *cells);
int emab_global_batch(emab_ctx_t *ctx, int n, const uint8_t *q, const int64_t *qoff, const uint8_t *t, const int64_t *toff,
                      const int32_t *w, int32_t *out, uint32_t *cigar, int max_cigar, int64_t *cells);
int emab_local_batch(emab_ctx_t *ctx, int n, const uint8_t *q, const int64_t *qoff, const uint8_t *t, const int64_t *toff,
                     int32_t *out, int64_t *cells);

/* which kernel family serves the SW work: 0 (default) = batch calls use one thread per task, 32 tasks per warp
 * advancing row by row (ksw_lanes.cuh), the pipeline one warp per read; 1 = one warp per task everywhere
 * (ksw_warp.cuh); 2 = thread-per-task everywhere, including mem_align1_core inside emab_align_pairs
 * (align_lanes.cuh).  Results are identical. */
int emab_set_sw_mode(emab_ctx_t *ctx, int mode);

/* device-resident variant used by bench.py for the kernel-only number: uploads once, then
 * emab_extend_resident_run launches the kernel `reps` times on resident inputs. */
int emab_extend_resident_load(emab_ctx_t *ctx, int n, const uint8_t *q, const int64_t *qoff, const uint8_t *t, const int64_t *toff, const int32_t *h0);
int emab_extend_resident_run(emab_ctx_t *ctx, int w, int end_bonus, int zdrop, int reps, int32_t *out, int64_t *cells);

/* Integer-pipe throughput of this GPU (the denominator of the SW roofline): kind 0 add, 1 max, 2 DPX viaddmax,
 * 3 DPX vimax3, 4 mad (FMA pipe), 5 add+mad on both pipes, 6 viaddmax.s16x2.  Result in 1e9 lane-instructions/s. */
int emab_int_peak(emab_ctx_t *ctx, int kind, int iters, double *gops_per_s, double *ms);

/* ---- FM index --------------------------------------------------------------------------------
 * emab_sa_batch      = bwt_sa (bwa/bwt.c:86) for n SA indices; mode 0 = dense SA, 1 = LF walk
 * emab_smem_batch    = mem_collect_intv (bwa/bwamem.c:140) for n reads: intervals[n*max_intv*4]
 *                      (x0,x1,x2,info), n_intv[n]
 * emab_set_seed_mode   which form of the seeding kernel a ctx runs (pipeline and emab_smem_batch alike):
 *                      5 (default; 0 = EMAB_SEED_MODE or 5): one-hot Occ blocks + k-mer start table + text comparison at
 *                        a unique locus (csrc/seed_hot.cuh).  Intervals carry the coordinates mem_chain reads — x0, x2,
 *                        info (bwa/bwamem.c:163-164,294-309) — and x1 = 0: x[1] is bwt_smem1a's forward working
 *                        coordinate, read by nothing after the forward sweep.  *touches = 32-byte sectors requested.
 *                      1-4: exact restatements over bwa's Occ layout (csrc/seed.cuh, seed_quad.cuh): x1 as the
 *                        reference leaves it; *touches = 64-byte Occ-block loads as the reference issues them.
 */
int emab_set_seed_mode(emab_ctx_t *ctx, int mode);
int emab_sa_batch(emab_ctx_t *ctx, int n, const int64_t *k, int64_t *out, int mode);
int emab_smem_batch(emab_ctx_t *ctx, int n, const uint8_t *seq, const int64_t *off, int64_t *intervals, int32_t *n_intv,
                    int max_intv, int64_t *touches);

/* ---- the pipeline: batched bwa_mem_mate_sw + bwa_smith_waterman + append_alignments ----------
 * (src/bwabridge.c:204-311, src/align.c:986-1061).  Reads are nt4, concatenated as
 * pair0/mate1, pair0/mate2, pair1/mate1, ... with 2*n_pairs+1 offsets.
 *
 * For every read the call returns its candidate regions IN THE ORDER the reference's
 * append_alignments visits them (region order of bwa_mem_mate_sw).  n_regs[r] regions of read r
 * start at cands[sum(n_regs[0..r))].  A record with keep == 0 was dropped by the reference's clip /
 * edit-distance filters (src/align.c:1017-1024) and must be ignored; the others carry exactly the
 * fields alignment_to_sam_rec stores in a SAMRecord (src/align.c:915-956).
 *
 * stage: 1 = stop after mem_align1_core, 2 = stop after mate rescue (regions only, via regs_dbg),
 *        3 = full.  regs_dbg (want_regs) holds 18 int64 per region: rb,re,qb,qe,rid,score,truesc,
 *        sub,csub,sub_n,w,seedcov,secondary,seedlen0,n_comp,is_alt,frac_rep(float bits),secondary_all.
 */
typedef struct {            /* one candidate region of one read: 56-byte wire record */
	int64_t pos;            /* 0-based leftmost reference position on contig rid */
	double em_score;        /* src/align.c:904-907 */
	int32_t rid;
	int32_t NM;
	int32_t score;          /* SW score of the region (mem_alnreg_t.score) */
	int32_t mapq;           /* mem_approx_mapq_se_insist (src/align.c:959-984) */
	int32_t score_mapq;     /* src/align.c:909-912 */
	int32_t clip;
	int32_t clip_edit_dist;
	uint32_t cigar_off;     /* first op in the CIGAR pool; BAM encoding len<<4|op, op 0..3 = M,I,D,S */
	uint16_t n_cigar;
	uint8_t is_rev;
	uint8_t keep;
} emab_cand_t;

typedef struct {            /* arrays are pinned host memory owned by the ctx, valid until its next call */
	int64_t n_cands, n_cigar_ops;
	const int32_t *n_regs;      /* [2*n_pairs] regions per read */
	const emab_cand_t *cands;   /* [n_cands] (stage 3) */
	const uint32_t *cigars;     /* [n_cigar_ops] (stage 3) */
	const int64_t *regs_dbg;    /* [n_cands*18] when want_regs */
} emab_pairs_result_t;

typedef struct {
	int64_t extend_cells, global_cells, local_cells;  /* DP cells visited */
	int64_t occ_touches;                              /* seeding form 5 (default): 32-byte sectors requested; forms 1-4: 64-byte Occ block loads as the reference issues them */
	int64_t n_occ, n_regs;
	double kernel_ms;                                 /* device time, first kernel to last (CUDA events on the ctx stream) */
	double ms_seed, ms_chain, ms_align1, ms_rescue, ms_finalize; /* per-kernel device time */
	int64_t h2d_bytes, d2h_bytes;                     /* bytes copied inside the call */
	int32_t launches;
	int32_t pad;
	int64_t rescue_planned_cells;                     /* local-SW cells computed ahead of the rescue replay (>= local_cells' share of them) */
	int64_t rescue_unplanned;                         /* mem_matesw alignments the plan did not foresee (computed inline by the replay) */
	/* the two planned waves (csrc/ext_wave.cuh, csrc/glob_wave.cuh): cells computed ahead by the thread-per-task kernels,
	 * calls the per-read replay had to compute inline, and the waves' device time (part of ms_align1 / ms_finalize) */
	int64_t ext_planned_cells, ext_unplanned, glob_planned_cells, glob_unplanned;
	double ms_ext_wave, ms_glob_wave;
} emab_stats_t;

int emab_set_error_rate(emab_ctx_t *ctx, double eps);  /* platform error_rate (src/techs.c:71-127); default 0.001 */
int emab_align_pairs(emab_ctx_t *ctx, int n_pairs, const uint8_t *seq, const int64_t *off, int stage, int want_regs,
                     emab_pairs_result_t *result, emab_stats_t *stats);
/* ---- the batch as text, and SAM text from the device ------------------------------------------------
 * emab_align_pairs_text = emab_align_pairs where the reads are not handed over as nt4 arrays but as positions inside the
 * batch's TEXT (the bucket file's contents, or FASTQ text): the text and one emab_pair_text_t per pair are uploaded, the
 * nt4 reads are derived on the device, and text + candidates stay resident for emab_sam_format.  res->cigars is NULL
 * (CIGARs are only needed for printing, which then happens on the device).
 * emab_sam_tables  = once per ctx: the .fai contig names (src/main.c:57-71) and the index-contig -> name map
 * emab_sam_format  = print_sam_record (src/samrecord.c:104-284) for n_recs records described by emab_sam_rec_t, into
 *                    `out` (host memory; pinned for speed), in the order given.  Everything the record copies — name,
 *                    bases (reverse-complemented for reverse-strand hits), qualities, CIGAR, contig names — comes from the
 *                    device-resident batch; the host supplies decisions only. */
typedef struct {
	uint32_t id_off[2], id_len[2];      /* read names without the leading '@' */
	uint32_t read_off[2], read_len[2];
	uint32_t qual_off[2], qual_len[2];
} emab_pair_text_t;
typedef struct {            /* one SAM record: 48 bytes */
	uint32_t pair;          /* pair index in the batch */
	int32_t rec_cand;       /* index of the candidate printed (into the call's candidates), -1: the read is unmapped */
	int32_t mate_cand;      /* its mate's chosen candidate, -1: none */
	int32_t alt_cand;       /* the XA:Z candidate, -1: none */
	int32_t mi;             /* MI:i */
	uint32_t bc;            /* index of the barcode's BX string */
	uint16_t flag;
	uint8_t which;          /* which read of the pair: 0 / 1 */
	uint8_t mapq;
	uint8_t xf;             /* XF:i */
	uint8_t gamma_len;
	char gamma[14];         /* the XG:f value as printed by %.5g */
} emab_sam_rec_t;
typedef struct {
	int32_t n_recs, n_bc;
	const emab_sam_rec_t *recs;
	const int32_t *bc_off;      /* [n_bc + 1] into bc_text */
	const char *bc_text;
	const char *bx_index;       /* -i suffix */
	const char *rg_id;          /* RG:Z value, NULL: no read group */
	int32_t is_haplotag, pad;
} emab_sam_job_t;
int emab_align_pairs_text(emab_ctx_t *ctx, int n_pairs, const char *text, uint64_t text_len, const emab_pair_text_t *pairs,
                          const int64_t *off, emab_pairs_result_t *result, emab_stats_t *stats);
/* emab_parse_bucket = read_special_fastq (src/align.c:759-806) on the device: uploads one preprocessed bucket's text, splits it
 * into lines, sorts them stably by their first bc_len bytes, tokenises them and encodes the barcodes.  Returns one
 * emab_pair_text_t and one barcode code per pair in sorted order (page-locked memory owned by the ctx) and leaves text and
 * table resident; emab_align_pairs_resident then runs the pipeline on them (off = prefix sums of the read lengths). */
int emab_parse_bucket(emab_ctx_t *ctx, const char *text, uint64_t text_len, int bc_len, int is_haplotag, int *n_pairs,
                      const emab_pair_text_t **pairs, const uint64_t **bcs);
int emab_align_pairs_resident(emab_ctx_t *ctx, int n_pairs, const int64_t *off, emab_pairs_result_t *result, emab_stats_t *stats);
int emab_sam_tables(emab_ctx_t *ctx, int n_chrom, const char *const *names, int n_rid, const int32_t *rid2chrom);
int emab_sam_format(emab_ctx_t *ctx, const emab_sam_job_t *job, char *out, uint64_t out_cap, uint64_t *out_len);
/* What the formatters read stays on the device until the next emab_align_pairs* or emab_parse_bucket call on the ctx: the
 * batch's text and pair table, and the candidates and CIGAR pool of the last align call (rec_cand, mate_cand and alt_cand
 * index them).  emab_em_batch, the formatters and the kernel-level calls leave them alone, so EM may run between the align
 * call and the formatters.
 * emab_bam_format = the same records as BAM (SAM spec v1 §4.2), compressed on the device into BGZF members; only the members
 *                    are copied to `out`.  Decoded the way `samtools view` prints them they are emab_sam_format's lines.
 *                    refID / next_refID: the first @SQ entry (contig of the index) with the .fai name the SAM line prints.
 *                    Fails with EMAB_ERR_ARG where BAM cannot hold the record: a read name longer than 254 bytes, a quality
 *                    string whose length differs from its read's, a quality byte outside '!'..'~'; and when a contig's
 *                    .fai name has no @SQ entry.
 * emab_bgzf_compress = the device compressor on its own: in[0..len) cut at multiples of 65 280 bytes, one BGZF member per
 *                    chunk (gzip header with the BC field, one raw DEFLATE block — LZ77 in the 32 KB window with dynamic
 *                    Huffman codes, or stored when that is smaller — CRC-32, ISIZE), packed into `out`.  The encoder is
 *                    deterministic: csrc/bgzf.cuh compiled for the host makes the same bytes.
 * emab_bgzf_eof     = the 28-byte empty member that ends a BGZF file (static storage; needs no GPU). */
int emab_bam_format(emab_ctx_t *ctx, const emab_sam_job_t *job, char *out, uint64_t out_cap, uint64_t *out_len);
/* emab_bam_records = emab_bam_format without the compression: the raw BAM records into `out`, and one sort row per record
 *                    into keys[n_recs], read from the same view of the record as the emitter.  The rows are what
 *                    emab_bam_sort orders and indexes:
 *                      key       (uint64)(uint32)refID << 32 | (uint64)(POS + 1) << 1 | reverse (samtools' coordinate key)
 *                      end       POS + the CIGAR's reference length; POS + 1 if that is 0 or the record is unmapped
 *                      len       the record's bytes (block_size + 4)
 *                      bin       reg2bin(POS, end), as the record holds it
 *                      unmapped  FLAG & 4 */
typedef struct {
	uint64_t key;
	uint32_t end, len;
	uint16_t bin, unmapped;
	uint32_t pad;
} emab_bam_key_t;
int emab_bam_records(emab_ctx_t *ctx, const emab_sam_job_t *job, char *out, uint64_t out_cap, uint64_t *out_len, emab_bam_key_t *keys);
/* emab_bam_sort = one coordinate-sorted BGZF body (and its BAI) from runs of raw records in input order.  A stable radix
 *                    sort of (key, record index) on the device gives the order; records are gathered on the host in that
 *                    order into page-locked slices of slice_chunks x 65 280 bytes (0 = 1 024 chunks), each compressed by the
 *                    device BGZF encoder and passed to w in order (no EOF block).  Members are cut every 65 280 bytes of
 *                    the whole body, so the bytes do not depend on the slice size.  With bai != NULL the index is built on
 *                    the device (csrc/bai.cuh states its rules) over n_ref references, with file offsets counted from
 *                    body_offset (the compressed header's size); free it with emab_free.  ms[4] (optional) receives the
 *                    wall time of the device sort, the host gather, the compression and the index build. */
typedef struct {
	const char *raw;                /* the run's records, back to back */
	const emab_bam_key_t *keys;     /* one row per record, in the same order */
	uint64_t n_recs;
} emab_bam_run_t;
typedef int (*emab_write_cb)(void *user, const char *text, uint64_t len);
int emab_bam_sort(emab_ctx_t *ctx, int n_runs, const emab_bam_run_t *runs, int n_ref, uint64_t body_offset, int slice_chunks,
                  emab_write_cb w, void *uw, char **bai, uint64_t *bai_len, double ms[4]);
/* emab_bam_spill = the runs in the order emab_bam_sort gives them, written to a new file at `path` (created with O_EXCL):
 *                    a 24-byte header ("EMABSPL1", records, record bytes), one 32-byte row per record (the emab_bam_key_t,
 *                    then its input position seq0[r] + the record's index in run r), then the raw records, all in that
 *                    order and uncompressed.  *file_bytes receives the file's size.  A failed create or write removes the
 *                    file and returns EMAB_ERR_IO with a message naming the path.
 * emab_bam_merge = emab_bam_sort over spill files and runs still in memory (seq0 as above), for runs larger than host
 *                    memory: the same bytes as emab_bam_sort over all the records in input order.  It works in windows: a
 *                    block of about budget / (2 (runs + 1)) bytes (at least one record) is read from each run, the device
 *                    takes every row up to the smallest last (key, input position) of the blocks that continue, orders
 *                    them and appends them to the body and the index.  ref_len[n_ref] (the @SQ lengths) sizes the linear
 *                    index.  ms[0] is the time of the device ordering; ms[1] includes reading the blocks. */
int emab_bam_spill(emab_ctx_t *ctx, int n_runs, const emab_bam_run_t *runs, const uint64_t *seq0, const char *path, uint64_t *file_bytes);
int emab_bam_merge(emab_ctx_t *ctx, int n_files, const char *const *paths, int n_runs, const emab_bam_run_t *runs, const uint64_t *seq0,
                   int n_ref, const int32_t *ref_len, uint64_t body_offset, int slice_chunks, uint64_t budget,
                   emab_write_cb w, void *uw, char **bai, uint64_t *bai_len, double ms[4]);
int emab_bgzf_compress(emab_ctx_t *ctx, const uint8_t *in, uint64_t len, uint8_t *out, uint64_t out_cap, uint64_t *out_len);
int emab_bgzf_eof(const uint8_t **p, uint64_t *len);
/* pinned host memory for callers that want their input buffers to take the fast H2D path */
void *emab_pinned_alloc(uint64_t bytes);
void emab_pinned_free(void *p);
int emab_is_pinned_host(const void *p);   /* 1 if p lies in page-locked host memory: such buffers are copied to the device without a staging copy */

/* ---- the barcode-cloud EM (src/align.c:410-543) ------------------------------------------------
 * The host groups candidates into clouds and links mates (the SAMDict bookkeeping of
 * src/samdict.c, src/align.c:354-408) and flattens every barcode of a bucket into the arrays
 * below; the device runs the initialisation and the 5 EM sweeps and returns the posteriors
 * gamma[n_cands] (double).  Lists are in the reference's iteration order (sd->head order for
 * entries, chain order for linked cloud sets) so the floating-point summation order is the
 * reference's.  Indices are global across the batch. */
typedef struct {
	int32_t n_bc, n_entries, n_cands, n_clouds, n_groups, n_units, many_clouds, pad;
	const int32_t *bc_entry_off, *bc_cloud_off, *bc_group_off, *bc_unit_off; /* [n_bc+1] */
	const int32_t *bc_full_em;       /* [n_bc] 1 if the barcode has >= 30 pairs (src/align.c:345) */
	const int32_t *entry_cand_off;   /* [n_entries+1] */
	const int32_t *entry_mate;       /* [n_entries] entry index of the mate, or -1 */
	const double *cand_score;        /* [n_cands] EM log-likelihood score */
	const int32_t *cand_cloud;       /* [n_cands] */
	const int32_t *cand_chrom;       /* [n_cands] */
	const uint32_t *cand_pos;        /* [n_cands] 1-based position */
	const uint8_t *cand_flags;       /* [n_cands] bit0 = reverse strand, bit1 = active */
	const int32_t *group_off;        /* [n_groups+1] */
	const int32_t *group_clouds;     /* [n_clouds] clouds of each linked set, chain order */
	const int32_t *cloud_contrib_off;/* [n_clouds+1] */
	const int32_t *cloud_contrib;    /* [n_cands] candidates of each cloud in entry-list order */
	const int32_t *unit_first, *unit_second; /* [n_units] the entries of a mate pair in list order (second = -1 if single) */
} emab_em_problem_t;

int emab_em_batch(emab_ctx_t *ctx, const emab_em_problem_t *problem, double *gamma_out);

/* ---- the operator the reference's main() calls: find_clouds_and_align --------------------------
 * (include/align.h:10-21; src/align.c:180-212,214-630).  A session replaces the reference's
 * process globals (ref, opts, tech, chroms, rg, bx_index: src/align.c:177-178, src/main.c:23-34):
 *   emab_session_open    = read_fai("<ref>.fai") + bwa_init(ref) + platform profile (-p)
 *   emab_session_config  = -R / -i / -d / -t
 *   emab_sam_header      = write_sam_header (argv is echoed into @PG as the reference does)
 *   emab_align_bucket    = find_clouds_and_align(NULL, NULL, fqx, ...) on the CONTENTS of one
 *                          preprocessed bucket file ("special FASTQ", -s / -x inputs)
 *   emab_align_fastq     = find_clouds_and_align(fq1, fq2, NULL, ...) on the contents of
 *                          barcode-sorted FASTQ(s); d2 == NULL means interleaved (-1 only)
 * SAM text is returned in a malloc'ed buffer the caller releases with emab_free().  Output is in
 * barcode order — byte-identical to the reference run with -t 1 (MI cloud ids included; they
 * continue across calls on one session like the reference's process-wide counter).
 *   emab_session_output  = EMAB_OUTPUT_SAM (default) or EMAB_OUTPUT_BAM.  In BAM mode emab_sam_header returns BGZF members
 *                          holding the BAM header (magic, the same header text, the @SQ names and lengths), and every align
 *                          call returns (or passes to its write callback) whole BGZF members of its records instead of SAM
 *                          text: blocks never span calls.  A BAM file is the header's bytes, every call's bytes in order,
 *                          then emab_bgzf_eof's block.  Fails when a contig's .fai name has no @SQ entry.  In BAM mode
 *                          emab_run_stats_t.sam_bytes counts the compressed bytes returned and format_kernel_ms includes
 *                          the compression kernels. */
#define EMAB_OUTPUT_SAM 0
#define EMAB_OUTPUT_BAM 1
typedef struct emab_session emab_session_t;

typedef struct {
	double parse_ms, encode_ms, align_ms, kernel_ms, cloud_ms, flatten_ms, em_ms, em_kernel_ms, format_ms, total_ms;
	double ms_seed, ms_chain, ms_align1, ms_rescue, ms_finalize;
	double gate_wait_ms;                              /* time spent waiting for a pipeline phase (emab_align_buckets) */
	int64_t h2d_bytes, d2h_bytes;
	int64_t n_pairs, n_barcodes, n_cands, n_clouds, sam_bytes;  /* sam_bytes: bytes returned (BAM: compressed) */
	int64_t extend_cells, global_cells, local_cells, occ_touches;
	int32_t launches, pad;
	int64_t ext_planned_cells, ext_unplanned, glob_planned_cells, glob_unplanned;
	double ms_ext_wave, ms_glob_wave;
	double format_kernel_ms;                          /* device time of the SAM text kernels (BAM: records + BGZF compression) */
	/* emab_session_finish (sorted BAM): wall time of the device sort, the host gather, the compression (slices to the device,
	 * BGZF kernels, members back and written) and the index build */
	double sort_ms, gather_ms, compress_ms, index_ms;
	/* sorted BAM with a spill prefix: the spill files this align call wrote, their bytes and the wall time spent on them */
	int64_t spill_files, spill_bytes;
	double spill_ms;
} emab_run_stats_t;

int emab_session_open(const char *ref_path, const char *platform, int device, emab_session_t **out);
void emab_session_close(emab_session_t *s);
int emab_session_config(emab_session_t *s, const char *rg, const char *bx_index, int apply_opt, int n_threads);
int emab_session_output(emab_session_t *s, int format);
/* Coordinate-sorted BAM (BAM output only).  emab_session_sort(s, on, max_host_bytes):
 *   EMAB_SORT_OFF        align calls return BGZF members as above (turning sorting off drops the records held so far)
 *   EMAB_SORT_COORD      align calls return zero bytes; their raw records and sort rows (emab_bam_records) are held in
 *                        host memory, in input order, until emab_session_finish writes them as one body sorted by
 *                        samtools' coordinate key (stable: equal keys keep input order, unplaced records last) and returns
 *                        its BAI.  Refused when a contig is longer than 2^29 - 1 bp, which a BAI cannot index.
 *   EMAB_SORT_COORD_NOINDEX  the same without the index (any contig length)
 * max_host_bytes caps the bytes held (raw records + 24 bytes per record; 0: no cap): without a spill prefix, the align call
 * that would go over it fails with EMAB_ERR_OVERFLOW, and so does emab_session_finish after it, which then writes nothing.
 * With a spill prefix (emab_session_sort_spill) and a nonzero cap, that call instead takes every held run and its own,
 * sorts them on its device and writes them to PREFIX.<session token>.<n>.spill (created with O_EXCL, raw and uncompressed;
 * emab_bam_spill); later calls start holding again while the file is written, so the run holds at most about twice the
 * cap in host memory.  emab_session_finish then merges the files and the held remainder on the device in windows bounded
 * by the cap (emab_bam_merge) into the same bytes, body and index, as without spilling.  The files are removed after
 * finish, when an align call of the run fails, on emab_session_sort and on emab_session_close.  A spill file that cannot
 * be created or written fails the align call with EMAB_ERR_IO naming the path, and finish then refuses the run.
 * emab_sam_header says SO:coordinate in sorted mode.
 * emab_session_finish(s, w, uw, bai, bai_len): the sorted BGZF body to w (without the EOF block) and, in EMAB_SORT_COORD,
 * the .bai in a buffer released with emab_free (bai may be NULL to skip it).  The index's file offsets count the bytes of
 * the header emab_sam_header returned last.  The held records are released; later calls start a new run. */
#define EMAB_SORT_OFF 0
#define EMAB_SORT_COORD 1
#define EMAB_SORT_COORD_NOINDEX 2
int emab_session_sort(emab_session_t *s, int on, uint64_t max_host_bytes);
/* the spill prefix of sorted runs (NULL: no spilling).  A session setting: it may be set while sorting is off or between
 * runs, and emab_session_sort keeps it. */
int emab_session_sort_spill(emab_session_t *s, const char *prefix);
int emab_session_finish(emab_session_t *s, emab_write_cb w, void *uw, char **bai, uint64_t *bai_len);
int emab_sam_header(emab_session_t *s, int argc, const char *const *argv, char **text, uint64_t *len);
int emab_align_bucket(emab_session_t *s, const char *data, uint64_t len, char **sam, uint64_t *sam_len);
int emab_align_fastq(emab_session_t *s, const char *d1, uint64_t l1, const char *d2, uint64_t l2, char **sam, uint64_t *sam_len);
/* -1/-2 as a stream (the reference reads barcode groups one at a time under a lock, src/align.c:296-341,653-744): the
 * callbacks supply barcode-sorted FASTQ text (read: up to cap bytes into buf, 0 at the end, < 0 on error; r2 == NULL means
 * one interleaved input) and receive the SAM body in input order.  Groups are cut into device batches of about batch_pairs
 * pairs (0 = 40 000) at barcode boundaries, up to `workers` batches in flight; memory is bounded by the batches in flight. */
typedef int64_t (*emab_read_cb)(void *user, char *buf, int64_t cap);
int emab_align_fastq_stream(emab_session_t *s, emab_read_cb r1, void *u1, emab_read_cb r2, void *u2, emab_write_cb w, void *uw, int batch_pairs);
/* -x (multi-input) mode: n buckets with up to `workers` of them in flight on this GPU (each worker is a
 * CUDA stream + scratch, so one bucket's kernels overlap another's host work and copies).  sam[i] /
 * sam_len[i] are per bucket, in input order; cloud ids continue in input order. */
int emab_session_workers(emab_session_t *s, int n_workers);
/* More GPUs of the box in one process: replicates the index on `device` (call before emab_session_workers).
 * emab_align_buckets then spreads its workers round-robin over the replicas and every worker takes the next
 * bucket from one shared counter, i.e. a bucket goes to whichever GPU is free (SURVEY.md 8e: host-side work
 * stealing, no collective); outputs and MI cloud ids stay in input order.  Up to 8 workers per device. */
int emab_session_add_device(emab_session_t *s, int device);
int emab_align_buckets(emab_session_t *s, int n, const char *const *data, const uint64_t *len, char **sam, uint64_t *sam_len);
int emab_session_stats(const emab_session_t *s, emab_run_stats_t *out);
/* test hook: write "ident<TAB>mate<TAB>chrom<TAB>pos<TAB>gamma(%.17g)" of every chosen alignment of later calls to path (NULL = off) */
int emab_session_dump_posteriors(emab_session_t *s, const char *path);
emab_ctx_t *emab_session_ctx(emab_session_t *s);
void emab_free(void *p);
void emab_abi_sizes(int32_t out[4]);  /* sizeof emab_cand_t, emab_stats_t, emab_run_stats_t, emab_index_build_stats_t: lets a binding check its mirror */
int emab_host_selftest(void);  /* host-side vector byte kernels checked against their scalar definitions; 0 = ok (no GPU needed) */

#ifdef __cplusplus
}
#endif
#endif

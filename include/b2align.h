/*
 * b2align.h -- C ABI of the B200-native pairwise alignment engine.
 *
 * Drop-in boundary for the hot path of gorkemsolun/Bioinformatics-Algorithms,
 * Local_Global_Alignment/hw2.cpp.  The reference has no FFI; its seam is the
 * per-pair function pair
 *     AlignmentResult* globalAlignmentNeedlemanWunsch(const string&, const string&, int, int, int)   hw2.cpp:118
 *     AlignmentResult* localAlignmentSmithWaterman   (const string&, const string&, int, int, int)   hw2.cpp:192
 * called from the serial batch loop hw2.cpp:328-338.  A GPU cannot be fed one
 * pair at a time, so the boundary is the BATCH: one call replaces the whole
 * loop hw2.cpp:328-338 plus, per pair, overlapLongestExactMatch (hw2.cpp:267-278).
 *
 * Plain C, no exceptions, caller-owned buffers, int status (0 = ok, <0 = error).
 * One b2a_ctx per host thread / GPU; a ctx is not thread-safe, the library is.
 * There is NO CPU fallback: every entry point that computes fails with
 * B2A_ERR_CUDA when no sm_100 device is usable.
 */
#ifndef B2ALIGN_H
#define B2ALIGN_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define B2A_VERSION 2   /* 2: B2A_MODE_SEMIGLOBAL */

/* status codes */
#define B2A_OK            0
#define B2A_ERR_ARG      -1   /* bad argument (null pointer, inconsistent offsets, ...)        */
#define B2A_ERR_CUDA     -2   /* CUDA runtime / no device; b2a_last_error() has the text      */
#define B2A_ERR_NOMEM    -3   /* host or device allocation failed                             */
#define B2A_ERR_RANGE    -4   /* scores outside the supported domain (SURVEY.md Appendix A.8) */
#define B2A_ERR_STATE    -5   /* call order violated (e.g. fetch before a batch was run)      */

/* alignment mode: hw2's -g / -l (hw2.cpp:292-295) */
#define B2A_MODE_GLOBAL   0   /* Needleman-Wunsch, hw2.cpp:118-190, tie order d > l > u      */
#define B2A_MODE_LOCAL    1   /* Smith-Waterman,   hw2.cpp:192-265, tie order 0 > d > u > l  */
/* Semi-global ("glocal", ends-free in the text; not in the reference): the WHOLE pattern against the substring of the text that
 * suits it best -- what a read against its reference window asks for.  Pattern = rows i, text = columns j, hw2's scoring.
 *   borders   H(0, j) = 0 for j = 0..n (leading text is free), H(i, 0) = i * gap;
 *   cells     hw2's NW recurrence and tie order d > l > u (hw2.cpp:140-153);
 *   end cell  (m, j*), j* = the smallest j in 0..n with H(m, j) = max_j H(m, j) (trailing text is free); score = H(m, j*);
 *   traceback from (m, j*) with hw2's NW test order, column 0 holding 'u', until row 0: no 'I' run along the free row.
 * Result: end = (m, j*), start = (0, column where the walk reached row 0), overlap = longest exact-match run as in global mode,
 * n_ops = alignment columns.  m = 0: score 0, end = start = (0,0), no ops.  n = 0: score m*gap, end (m,0), m 'D' ops.
 * Accepted by every batch entry point and in any run of b2a_align_batch_multi / _multi_seq2 / the device-resident calls, with
 * B2A_WANT_OPS or B2A_SCORE_ONLY (same score and end cell as the full call).  Not with B2A_TIE_HW4 or b2a_align_anchored
 * (B2A_ERR_ARG).  A pair whose traceback record exceeds B2A_OPT_CKPT_BYTES fails the batch with B2A_ERR_RANGE: the checkpointed
 * path serves global and local mode only. */
#define B2A_MODE_SEMIGLOBAL 2

/* b2a_params.flags */
#define B2A_WANT_OPS      1u  /* keep per-pair traceback ops on the device for b2a_fetch_ops / b2a_copy_ops */
#define B2A_TIE_HW4       4u  /* global mode only: break ties d > u > l as hw4's own needleman_wunsch does (hw4/hw4.cpp:37-46) instead of
                                 hw2's d > l > u (hw2.cpp:145-153); b2a_result.overlap then carries hw4's distance = number of alignment
                                 columns holding a gap or a mismatch (hw4/hw4.cpp:141-152) */
#define B2A_SCORE_ONLY    2u  /* fill only: results carry the score (hw2.cpp:186 / :225-229), no traceback record,
                                 no coordinates/overlap/ops -- the shape of hw3's distance stage (hw3.cpp:231-241) */

/* op codes, 2 bits each (the reference's own letters, hw2.cpp:164-180 / :240-256) */
#define B2A_OP_M          0u  /* 'M' diagonal: pattern base over text base            */
#define B2A_OP_D          1u  /* 'D' up:       pattern base over '-'                   */
#define B2A_OP_I          2u  /* 'I' left:     '-' over text base                      */

typedef struct b2a_ctx b2a_ctx;

/* hw2's "-s <match> <mismatch> <gap>" (hw2.cpp:302-305): linear gap, raw byte equality (hw2.cpp:142, :208) */
typedef struct b2a_params {
    int32_t  mode;       /* B2A_MODE_*            */
    int32_t  match;
    int32_t  mismatch;
    int32_t  gap;
    uint32_t flags;      /* B2A_WANT_OPS or 0     */
} b2a_params;

/* One record per pair: everything struct AlignmentResult (hw2.cpp:17-23) carries, in index form.
 * The aligned strings / CIGAR / MD:Z are rendered from (ops, raw sequences) by b2a_render_*. */
typedef struct b2a_result {
    int32_t  score;      /* hw2.cpp:186 dp[m][n] (global) / running max hw2.cpp:225-229 (local) / H(m,j*) (semi) */
    uint32_t end_i;      /* traceback start cell, 1-based rows (pattern) ...                         */
    uint32_t end_j;      /* ... and columns (text): (m,n) global, first row-major arg-max local, (m,j*) semi */
    uint32_t start_i;    /* cell where the traceback stopped: (0,0) global; H==0 or an edge local; row 0 semi */
    uint32_t start_j;
    int32_t  overlap;    /* overlapLongestExactMatch(alignedPattern, alignedReference), hw2.cpp:267;
                            with B2A_TIE_HW4: mismatch + gap columns of the alignment, hw4.cpp:141-152  */
    uint32_t n_ops;      /* alignment columns = length of the traceback op list                      */
    uint32_t path;       /* which kernel family served the pair: 1 = short16 (s16x2), 2 = wide32     */
} b2a_result;

/* ---- lifecycle ---------------------------------------------------------------------------- */
int         b2a_device_count(void);                 /* usable CUDA devices, 0 if none / no driver     */
b2a_ctx*    b2a_create(int device);                 /* NULL on failure (no CUDA device)               */
void        b2a_destroy(b2a_ctx* ctx);
const char* b2a_last_error(const b2a_ctx* ctx);     /* text of the last failure on this ctx           */

/* Pinned host memory for batch inputs/outputs (optional; pageable memory works, staged). */
void*       b2a_host_alloc(size_t bytes);
void        b2a_host_free(void* p);
/* Pin memory the caller already owns (e.g. a POSIX shared-memory segment several one-GPU processes write their result records
 * into: the "host gather" of a pair-sharded batch is then the device->host copies themselves).  Call after b2a_create. */
int         b2a_host_register(void* p, size_t bytes);
int         b2a_host_unregister(void* p);

/* ---- the batch call: replaces the loop hw2.cpp:328-338 ------------------------------------ */
/* Pair k aligns pattern bytes pat[pat_off[k] .. pat_off[k+1]) against text bytes
 * txt[txt_off[k] .. txt_off[k+1]) (index-wise zip, hw2.cpp:328-335).  All pointers are HOST
 * pointers; offsets arrays hold n_pairs+1 entries.  results receives n_pairs records.
 * Host->device copies, both kernels and the device->host copy of the records happen inside. */
int b2a_align_batch(b2a_ctx* ctx, const b2a_params* prm,
                    const uint8_t* pat, const uint64_t* pat_off,
                    const uint8_t* txt, const uint64_t* txt_off,
                    uint64_t n_pairs, b2a_result* results);

/* Several runs over ONE upload of the same pairs: run r aligns them under prm[r].  The runs share scoring and flags and differ in
 * mode -- hw2's -g and -l over one batch (BASELINE config 2 asks for both).  Per segment the sequences cross PCIe once and the
 * kernels of every run follow, so the copy is hidden behind n_runs times the work.  results[r] receives the n_pairs records of run r.
 * b2a_select_run chooses which run b2a_fetch_ops / b2a_copy_ops / b2a_batch_download read afterwards (run 0 after the call). */
#define B2A_MAX_RUNS 2
int b2a_align_batch_multi(b2a_ctx* ctx, const b2a_params* prm, uint32_t n_runs,
                          const uint8_t* pat, const uint64_t* pat_off,
                          const uint8_t* txt, const uint64_t* txt_off,
                          uint64_t n_pairs, b2a_result* const* results);
int b2a_select_run(b2a_ctx* ctx, uint32_t run);

/* ---- compact sequence input: 2 bits per base + an exception list (lossless) ----------------- */
/* The reference keeps every sequence as a std::string and compares raw bytes (hw2.cpp:142, :208), so any byte may occur.  A b2a_seq2
 * describes the SAME concatenated byte buffer `seq[0 .. n_bytes)` that b2a_align_batch takes, at a quarter of its size: byte p is
 * alphabet[c] with c = bits 2*(p%4) .. 2*(p%4)+1 of codes[p/4], except at the positions listed in exc_pos (ascending), where it is
 * exc_byte[] (an 'N' in a read, lower case, ...; the code stored there is 0).  Host->device traffic drops 4x; the device expands the
 * buffer back to bytes in HBM (one HBM-bound kernel per segment, < 1 % of the step) and everything downstream is unchanged, so the
 * results are those of the byte call bit for bit.  Offsets stay byte offsets. */
typedef struct b2a_seq2 {
    const uint8_t*  codes;        /* (n_bytes + 3) / 4 bytes                                        */
    uint64_t        n_bytes;      /* bytes the buffer stands for (= off[n_pairs] of its offsets)     */
    uint8_t         alphabet[4];  /* code c stands for byte alphabet[c]                              */
    uint32_t        reserved;     /* 0                                                              */
    const uint64_t* exc_pos;      /* n_exc ascending byte positions outside the alphabet ...         */
    const uint8_t*  exc_byte;     /* ... and the bytes that stand there                              */
    uint64_t        n_exc;
} b2a_seq2;
/* Host only, multi-threaded: packs seq[0 .. n_bytes) into codes ((n_bytes+3)/4 bytes) and lists the exceptions.  Returns the number
 * of exceptions the buffer holds (>= 0) and writes the first min(that, exc_cap) of them (snprintf style: call with exc_cap = 0 to
 * size the arrays, codes may then be NULL), or <0. */
int64_t b2a_seq2_pack(const uint8_t* seq, uint64_t n_bytes, const uint8_t alphabet[4],
                      uint8_t* codes, uint64_t* exc_pos, uint8_t* exc_byte, uint64_t exc_cap);
/* Host only: bytes [first, first + count) of the buffer a b2a_seq2 stands for (e.g. the winner's pattern and text for
 * b2a_render_mdz).  Returns B2A_OK or B2A_ERR_ARG. */
int b2a_seq2_unpack(const b2a_seq2* s, uint64_t first, uint64_t count, uint8_t* out);
/* b2a_align_batch_multi over compact inputs: same pairs, same results, a quarter of the upload.  As in every batch call the offsets
 * need not start at 0: several contexts (one per GPU) can share ONE b2a_seq2 pair and take consecutive slices off + first of the
 * offsets arrays; each context copies and expands only the bytes its slice covers. */
int b2a_align_batch_multi_seq2(b2a_ctx* ctx, const b2a_params* prm, uint32_t n_runs,
                               const b2a_seq2* pat, const uint64_t* pat_off,
                               const b2a_seq2* txt, const uint64_t* txt_off,
                               uint64_t n_pairs, b2a_result* const* results);

/* After a batch run with B2A_WANT_OPS: traceback ops of one pair as ASCII 'M'/'D'/'I', in
 * TRACEBACK order (alignment end -> start, exactly the reference's `tracebacks` vector,
 * hw2.cpp:161).  Returns the op count, or <0.  ops_cap must be >= results[pair].n_ops. */
int64_t b2a_fetch_ops(b2a_ctx* ctx, uint64_t pair, char* ops, uint64_t ops_cap);

/* All pairs' ops in device format: 2-bit codes, op t of pair k at bits 2*(t%16) of word
 * ops_words[ops_off[k] + t/16], traceback order.  ops_off (n_pairs+1 entries, may be NULL)
 * receives the per-pair word offsets.  Returns the total word count (>=0) or <0; call with
 * ops_words == NULL to query it. */
int64_t b2a_copy_ops(b2a_ctx* ctx, uint32_t* ops_words, uint64_t cap_words, uint64_t* ops_off);

/* Optional: have the NEXT b2a_align_batch / _multi / _multi_seq2 calls (with B2A_WANT_OPS) also deliver every pair's op list to host
 * memory, copied segment by segment under the kernels of the following segments instead of in one b2a_copy_ops afterwards.
 * ops_words[r] (cap_words 32-bit words each; pinned memory makes the copies asynchronous) receives run r's words in exactly the
 * b2a_copy_ops layout; the per-pair offsets come from b2a_copy_ops(ctx, NULL, 0, ops_off) after the call.  A batch whose op words
 * (sum over pairs of (m + n + 15) / 16 + 1) exceed cap_words fails with B2A_ERR_ARG.  NULL / n_runs = 0 switches the sink off. */
int b2a_set_ops_sink(b2a_ctx* ctx, uint32_t* const* ops_words, uint32_t n_runs, uint64_t cap_words);

/* ---- device-resident variant (kernel-only timing; inputs already in HBM) ------------------- */
int b2a_batch_upload(b2a_ctx* ctx, const b2a_params* prm,
                     const uint8_t* pat, const uint64_t* pat_off,
                     const uint8_t* txt, const uint64_t* txt_off, uint64_t n_pairs);
int b2a_batch_run(b2a_ctx* ctx, float* fill_ms, float* traceback_ms);   /* CUDA-event times of this run */
int b2a_batch_download(b2a_ctx* ctx, b2a_result* results);
/* times of the last b2a_batch_run: sums of the per-segment fill / traceback kernel times and the
 * device time from the first kernel's start to the last kernel's end (with two compute lanes the
 * kernels of neighbouring segments overlap, so total <= fill + traceback). */
int b2a_batch_times(const b2a_ctx* ctx, float* fill_ms, float* traceback_ms, float* total_ms);
/* counters of the last run: kernels launched, algorithmic cells, bytes written by the fill kernel */
int b2a_batch_stats(const b2a_ctx* ctx, uint64_t* kernel_launches, uint64_t* cells, uint64_t* fill_bytes,
                    uint64_t* h2d_bytes, uint64_t* d2h_bytes);

/* ---- hw3's distance stage: score-only 3-state affine global alignment ------------------------ */
/* Replaces affine_alignment(..., &alignmentScore) (Multiple_Sequence_Alignment/hw3.cpp:23-98) as it is
 * called from the all-vs-all loop hw3.cpp:231-241: V/F/E recurrences with hw3's "-s M:Mm:Go:Ge" scores,
 * the INT_MIN/2 sentinel (hw3.cpp:16), result max(V,F,E)[m][n].  Pair k aligns pat[k] (string1, rows)
 * against txt[k] (string2, columns); scores receives n_pairs ints. */
int b2a_affine_score_batch(b2a_ctx* ctx, int32_t match, int32_t mismatch, int32_t gap_open, int32_t gap_extend,
                           const uint8_t* pat, const uint64_t* pat_off, const uint8_t* txt, const uint64_t* txt_off,
                           uint64_t n_pairs, int32_t* scores);
/* The same alignment WITH its traceback (hw3.cpp:100-135), as hw3 runs it for the centre against every other
 * sequence (hw3.cpp:259-266): the op list (traceback order, hw2's letters: 'M' column of two bases, 'D' string1 base
 * over '-', 'I' '-' over string2 base) stays on the device for b2a_affine_fetch_ops; n_ops (may be NULL) receives the
 * alignment lengths.  Trace decisions are the reference's: V/F/E priority with strict '>' (hw3.cpp:59-82, :86-98). */
int b2a_affine_align_batch(b2a_ctx* ctx, int32_t match, int32_t mismatch, int32_t gap_open, int32_t gap_extend,
                           const uint8_t* pat, const uint64_t* pat_off, const uint8_t* txt, const uint64_t* txt_off,
                           uint64_t n_pairs, int32_t* scores, uint32_t* n_ops);
int64_t b2a_affine_fetch_ops(b2a_ctx* ctx, uint64_t pair, char* ops, uint64_t ops_cap);
/* The loop hw3.cpp:231-251 itself over one sequence set: pairs (i, j), i < j, in the reference's
 * row-major order; this call serves pairs [pair_first, pair_first + pair_count) of that order (so the
 * n(n-1)/2 pairs can be sharded over GPUs), writes their scores, the star sums sum_scores[n_seqs]
 * restricted to the range (add the ranges' sums, hw3.cpp:238-239) and the centre index hw3.cpp:243-251
 * (first strict maximum) when the range covers every pair, -1 otherwise (partial sums do not determine it).
 * Any output pointer may be NULL; the centre does not depend on sum_scores being requested. */
int b2a_affine_star_scores(b2a_ctx* ctx, int32_t match, int32_t mismatch, int32_t gap_open, int32_t gap_extend,
                           const uint8_t* seqs, const uint64_t* seq_off, uint32_t n_seqs,
                           uint32_t pair_first, uint32_t pair_count, int32_t* pair_scores, int32_t* sum_scores, int64_t* center);

/* ---- tuning knobs (defaults are what bench.py measures) -------------------------------------- */
/* A batch is cut into segments of consecutive pairs; the copy of segment k+1 overlaps the kernels
 * of segment k and the DP record of a lane is reused by every second segment. */
#define B2A_OPT_LANES      1   /* DP records (+ traceback streams) the launches alternate over: 1..8, 0 = automatic */
#define B2A_OPT_SEG_PAIRS  2   /* max pairs per segment                                                  */
#define B2A_OPT_SEG_FIRST  5   /* pairs of the first segment of b2a_align_batch (doubling up to the max) */
#define B2A_OPT_SEG_BYTES  3   /* DP-record bytes per segment                                            */
#define B2A_OPT_CKPT_BYTES 6   /* a long pair whose traceback record (0.5 byte per cell) would exceed this many bytes is walked from
                                  checkpoint rows instead (score pass + band groups re-filled bottom-up): default 48 GB              */
#define B2A_OPT_CKPT_GROUP 7   /* ... and this is the record size of one re-filled band group: default 1 GB                         */
#define B2A_OPT_CKPT_COLS  8   /* ... which is cut into tiles at every 2^value-th column (kept by the score pass too): default 13    */
int b2a_set_option(b2a_ctx* ctx, int option, int64_t value);

/* ---- result formatting: prepareCigarString hw2.cpp:59-78, prepareMDZString hw2.cpp:80-116 --- */
/* ops = ASCII list in traceback order (as returned by b2a_fetch_ops). Return the string
 * length (excluding NUL) or <0 if cap is too small. */
int64_t b2a_render_cigar(const char* ops, uint64_t n_ops, char* out, uint64_t cap);
int64_t b2a_render_mdz(const char* ops, uint64_t n_ops, const uint8_t* pattern, const uint8_t* text,
                       uint32_t start_i, uint32_t start_j, char* out, uint64_t cap);

/* Batch winner, hw2.cpp:326-357: key = overlap (global) / score (local and semi-global), strict '>' from
 * -1000000 so the lowest index wins ties; -1 for an empty batch. */
int64_t b2a_select_best(int32_t mode, const b2a_result* results, uint64_t n_pairs);

/* ---- hw4's tree stage: UPGMA over the all-vs-all distances + Newick text (hw4/hw4.cpp:154-228) ---- */
/* pair_dist holds the n(n-1)/2 distances of pairs (i, j), i < j, in row-major order (the order of the loop
 * hw4.cpp:138-139); names are the FASTA ids.  Writes the line hw4 writes to its tree file WITHOUT the trailing
 * newline ("(...):0.0;").  Host only.  Returns the length or <0 (buffer too small / bad argument). */
int64_t b2a_upgma_newick(const int32_t* pair_dist, uint32_t n_seqs, const char* const* names, char* out, uint64_t cap);

/* ---- hw3's assembly stage: centre-star merge + PHYLIP text (hw3.cpp:253-357) ------------------------------- */
/* ops[i] / n_ops[i] (ignored for i == centre): the op list of affine_alignment(seqs[centre], seqs[i]) in traceback
 * order as b2a_affine_fetch_ops returns it.  Writes the whole file hw3 writes (header line, one row per sequence with
 * the centre first, 10-character ids, blocks of 10).  Host only.  Returns the length or <0. */
int64_t b2a_center_star_phylip(uint32_t n_seqs, uint32_t centre, const char* const* names,
                               const uint8_t* const* seqs, const uint64_t* seq_len,
                               const char* const* ops, const uint64_t* n_ops, char* out, uint64_t cap);

/* ---- seed-anchored global alignment of one long pair (SURVEY.md 8 f4) ------------------------------------- */
/* Not in the reference's code: its report ("Performance Bottlenecks") names banded / seed-anchored alignment as the way out of the
 * O(mn) matrices of hw2.cpp:119-120.  An anchor is an exact match pattern[i .. i+len) == text[j .. j+len) (0-based).  The anchored
 * alignment is the global alignment CONSTRAINED to contain every anchor as a run of 'M' columns: the stretches between consecutive
 * anchors (and before the first / after the last) are independent Needleman-Wunsch problems with hw2's recurrences and tie order
 * (hw2.cpp:118-190), which the engine runs as ONE batch; score = sum of the stretch scores + match * sum(len).  m*n cells shrink to
 * sum(m_s * n_s).  The result is optimal among alignments through the anchors; it equals hw2's unconstrained score whenever some
 * optimal alignment passes through them (tests compare both). */
typedef struct b2a_anchor { uint32_t i, j, len; } b2a_anchor;
/* Host only.  Candidate anchors = k-mers that occur exactly once in the pattern and exactly once in the text (verified byte-wise);
 * the longest chain increasing in both coordinates is kept, thinned so that consecutive anchors start at least `spacing` pattern
 * bases apart and never overlap.  Returns the number of anchors of the chain (>= 0) and writes the first min(that, cap), or <0. */
int64_t b2a_find_anchors(const uint8_t* pattern, uint64_t m, const uint8_t* text, uint64_t n, uint32_t k, uint32_t spacing,
                         b2a_anchor* out, uint64_t cap);
/* prm->mode must be B2A_MODE_GLOBAL.  anchors must ascend strictly in i and j without overlapping (as b2a_find_anchors returns them)
 * and be exact matches (checked: B2A_ERR_ARG otherwise).  result receives one record (overlap = longest exact-match run of the whole
 * alignment, hw2.cpp:267-278; path = 3); ops (may be NULL: overlap is then -1, as it is when ops_cap is too small) receives the op list, ASCII
 * 'M'/'D'/'I' in traceback order like b2a_fetch_ops, at most ops_cap characters.  Returns the op count or <0.  The context's last batch is replaced and a sink set with
 * b2a_set_ops_sink is switched off. */
int64_t b2a_align_anchored(b2a_ctx* ctx, const b2a_params* prm, const uint8_t* pattern, uint64_t m, const uint8_t* text, uint64_t n,
                           const b2a_anchor* anchors, uint64_t n_anchors, b2a_result* result, char* ops, uint64_t ops_cap);

/* ---- measurement helper: sustained issue rate of the packed int16x2 DPX instructions ------- */
/* Runs the microbenchmark kernel on ctx's device; *gops = 1e9 lane-instructions/s sustained by
 * kind 0: VIADDMNMX.S16x2 only, 1: the fill kernel's ALU mix, 2: ALU mix + IMAD (both pipes). */
int b2a_microbench_int16x2(b2a_ctx* ctx, int kind, double* gops, float* sm_mhz);

/* ---- introspection for white-box tests: raw HBM record of the first short16 class --------- */
/* Copies the delta/anchor chunks (and, in local mode, the per-row maxima) the fill kernel wrote.
 * Returns the record size in bytes, or <0. */
int64_t b2a_debug_copy_record(b2a_ctx* ctx, void* chunks, uint64_t chunk_bytes_cap, void* rowbest, uint64_t rowbest_bytes_cap);

#ifdef __cplusplus
}
#endif
#endif /* B2ALIGN_H */

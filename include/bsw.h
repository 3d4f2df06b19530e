/*
 * bsw.h -- C ABI of the B200-native batched banded Smith-Waterman extension engine.
 *
 * This is the drop-in boundary for the one hot path of GenomicsBench `bsw`
 * (bwa-mem2's BandedPairWiseSW::getScores16 / getScores8, i.e. ksw_extend2
 * semantics over batches of SeqPair).  Every entry point below replaces a
 * piece of the reference interface; the citation next to each one is the
 * reference file:line (relative to /root/reference/benchmarks/bsw) it stands
 * in for.  Plain pointers and sizes only: no C++ or torch types cross this line.
 *
 * There is NO CPU fallback behind this ABI: every bsw_extend* call runs the
 * hand-written sm_100a kernels and fails with BSW_ERR_CUDA when no device or
 * no usable kernel image is present.
 */
#ifndef BSW_B200_H
#define BSW_B200_H

#include <stdint.h>
#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

/* ---- a1: SeqPair, layout identical to bandedSWA.h:91-100 (72 bytes) ------ */
#ifndef BSW_SEQPAIR_DEFINED
#define BSW_SEQPAIR_DEFINED
typedef struct dnaSeqPair {
    int64_t idr, idq, id;       /* byte offsets of ref / query in the sequence buffers; caller's id */
    int32_t len1, len2;         /* len1 = reference (target) length, len2 = query length          */
    int32_t h0;                 /* seed score, >= 0                                                */
    int32_t seqid, regid;       /* untouched                                                       */
    int32_t score, tle, gtle, qle;  /* outputs                                                     */
    int32_t gscore, max_off;        /* outputs                                                     */
} SeqPair;
#endif

/* ---- error codes (the reference has none: it exit()s, bandedSWA.cpp:94-99) */
enum {
    BSW_OK            =  0,
    BSW_ERR_PARAM     = -1,   /* parameter outside the supported domain                 */
    BSW_ERR_DOMAIN    = -2,   /* a pair violates 1<=len<=32767, h0>=0, scores<32768 ... */
    BSW_ERR_CUDA      = -3,   /* CUDA runtime / no device / kernel image missing        */
    BSW_ERR_NOMEM     = -4,
    BSW_ERR_STATE     = -5,   /* call sequence error (e.g. run before stage)            */
    BSW_ERR_IO        = -6
};

/* z-drop rule selector.  The reference's vector code (ZSCORE16, bandedSWA.cpp:323-336)
 * and its scalar code (bandedSWA.cpp:222-228) disagree when e_del/e_ins != 1 or
 * zdrop <= 0 (SURVEY Appendix B, Q1/Q2).  getScores16/getScores8 use VECTOR,
 * scalarBandedSWAWrapper uses SCALAR. */
enum { BSW_ZDROP_VECTOR = 0, BSW_ZDROP_SCALAR = 1 };

/* Thread-per-pair kernel of the short pairs.  PACKED16: two DP columns per DPX .S16x2
 * instruction (pairs with N or with (h0 + len2*match)*(1+match) > 32767 still take the 32-bit
 * kernel); WIDE32: the 32-bit kernel for every short pair (A/B measurements). */
enum { BSW_SHORT_PACKED16 = 0, BSW_SHORT_WIDE32 = 1 };

/* ---- a2: constructor arguments of BandedPairWiseSW (bandedSWA.cpp:51-100) -- */
typedef struct bsw_params {
    int32_t o_del, e_del, o_ins, e_ins;   /* gap open / extend, > 0 extend           */
    int32_t zdrop;                        /* 1..32767; 32767 == off (vector rule)    */
    int32_t end_bonus;
    int32_t match;                        /* w_match  (> 0)                          */
    int32_t mismatch;                     /* penalty, positive (ctor negates it)     */
    int32_t ambig;                        /* score of any cell touching base 4 (N); reference vector code hard-wires -1 (bandedSWA.cpp:69) */
    int32_t zdrop_mode;                   /* BSW_ZDROP_VECTOR | BSW_ZDROP_SCALAR     */
    int32_t n_devices;                    /* 0 => use the current CUDA device only   */
    int32_t devices[16];                  /* CUDA ordinals when n_devices > 0        */
    int32_t host_threads;                 /* packer threads per engine, 0 => auto    */
    int32_t long_min_qlen;                /* queries of at least this length use the warp-per-pair
                                             kernel; 0 => default (825, the short kernel's shared-
                                             memory limit + 1); 1 routes every pair to it          */
    int32_t short_variant;                /* BSW_SHORT_PACKED16 (default) | BSW_SHORT_WIDE32               */
    int32_t tiny_batch;                   /* latency route: calls with at most this many pairs skip bucketing and
                                             packing and run every pair on the warp-per-pair kernel (rows in shared
                                             memory), ~2x lower latency for batches that cannot fill the GPU one pair
                                             per thread; 0 = off (default).  The BandedPairWiseSW class sets 1536: the
                                             reference driver's habit is -b 512 (scripts/run-cpu.sh:30)              */
    int32_t warp_max_pairs;               /* pairs a device runs one per WARP at any moment (queries <= 255, no N, 16-bit
                                             scores; the row in registers, bsw_warp16.cuh): a call too small to fill the
                                             GPU one pair per thread is bound by one thread's time for one pair (~0.4 ms
                                             at 151 bp; a warp: ~0.14 ms, at ~10 x the issue slots).  The budget is shared
                                             by all calls and engines of the process: a call that fits takes its share
                                             while it runs, any other runs thread-per-pair.  0 = default (4096),
                                             -1 = never                                                               */
    int32_t reserved[4];
} bsw_params;

/* Per-call statistics (replaces the rdtsc counters behind getTicks(),
 * bandedSWA.cpp:108-122, and the commented-out GCUPS print main_banded.cpp:321-323). */
typedef struct bsw_stats {
    int64_t pairs;               /* pairs processed by the last call                     */
    int64_t cells_nominal;       /* sum len1*len2 (reference GCUPS convention)           */
    int64_t cells_effective;     /* inner-loop iterations actually executed (SW_cells)   */
    double  ms_sort;             /* unused (bucketing runs on the device)                */
    double  ms_pack;             /* host: streaming pass into pinned staging (pageable buffers only) */
    double  ms_h2d;              /* unused (copies overlap the kernels)                  */
    double  ms_kernel;           /* bsw_run_staged: device timeline of the DP launches (events);
                                    bsw_extend: sum of the chunks' device timelines      */
    double  ms_d2h;              /* unused                                               */
    double  ms_scatter;          /* host: results written into SeqPair[] (pageable buffers only) */
    double  ms_total;            /* host wall clock of the whole call                    */
    int64_t h2d_bytes, d2h_bytes;
    int32_t kernel_launches;     /* kernels launched by the last call (prep + DP + write-back) */
    int32_t n_short, n_long;     /* pairs routed to the thread-per-pair / warp-per-pair kernel */
    int32_t partitioned;         /* 1: the call ran with the SMs split into a service and a DP partition (PCIe-bound batch) */
    int32_t shards;              /* device ranges the call was cut into (multi-GPU partitioner): 1, or the engine's device count */
    int32_t reserved[3];
} bsw_stats;

typedef struct bsw_engine bsw_engine;

/* ---- engine lifetime ------------------------------------------------------ */
/* replaces: new BandedPairWiseSW(...)   main_banded.cpp:253-258, bandedSWA.cpp:51-100 */
bsw_engine* bsw_create(const bsw_params* params, int* err);
/* replaces: delete bsw[i]               main_banded.cpp:346-349, bandedSWA.cpp:103-106 */
void        bsw_destroy(bsw_engine* eng);
const char* bsw_last_error(const bsw_engine* eng);   /* also valid with eng == NULL (creation errors) */
void        bsw_default_params(bsw_params* p);       /* bwa defaults: main_banded.cpp:49-53,250 */

/* ---- the hot path ---------------------------------------------------------
 * replaces: getScores16 / getScores8 (bandedSWA.cpp:1124-1148 / :424-446) called
 * at main_banded.cpp:286.  Host buffers in, six result fields written in place,
 * input order preserved; pads are never written and pair.id is never read. */
int bsw_extend(bsw_engine* eng, SeqPair* pairs, const uint8_t* seq_ref,
               const uint8_t* seq_qer, int64_t n_pairs, int32_t w);

/* ---- long-read flanks --------------------------------------------------------
 * replaces: ksw_extend2 (tools/bwa/ksw.c:380-479) with its int32 arithmetic, for pairs outside bsw_extend's
 * 16-bit domain (long-read flanks).  Same SeqPair records, engine scoring, z-drop rule (zdrop_mode) and in-place
 * result fields as bsw_extend; pads never written, pair.id never read.  Runs on the engine's first device.
 * Domain (BSW_ERR_DOMAIN): 1 <= len1, len2 <= 2^24 - 1, h0 >= 0, h0 + len2 * mx + end_bonus <= 2^30
 * (mx = largest score of the matrix, as in the band clamp).  Pairs inside bsw_extend's domain give bsw_extend's
 * results. */
int bsw_extend32(bsw_engine* eng, SeqPair* pairs, const uint8_t* seq_ref, const uint8_t* seq_qer,
                 int64_t n_pairs, int32_t w);

/* ---- the packed host format ---------------------------------------------------
 * The reference keeps file parsing outside its timed region (main_banded.cpp:262-270 loadPairs, :306 readTim) and
 * layout conversion inside it (the AoS->SoA transposes of bandedSWA.cpp:1266-1326).  A loader that emits THIS layout
 * instead of SeqPair[] + one byte per base lets the engine DMA 2 bits per base and 16 bytes per descriptor
 * (~50 B/pair for 16-96 bp reads instead of 194) and return 24 bytes per pair (OutScore, the reference's own result
 * type, bandedSWA.h:103-107) instead of the whole 72-byte record.
 *   packed pair   bases 0-3, 16 per 32-bit word, base k of a sequence at bits [2k, 2k+2) of word k/16, every
 *                 sequence starts on a word; q_off / r_off = first word in q2 / r2
 *   RAW pair      (BSW_PAIR_RAW) one base code per byte (0-3, 4 = N) in raw_q / raw_r, q_off / r_off = first byte;
 *                 the builders use it for pairs that contain N and for queries longer than
 *                 BSW_PACKED_MAX_QLEN (the thread-per-pair kernel's limit)
 * `ordered` = 1 promises that offsets never decrease with the pair index (in q2, r2, and among the RAW pairs in
 * raw_q, raw_r) -- what the builders below emit; the engine then streams the buffers chunk by chunk.  Otherwise
 * all four buffers are copied before the first chunk runs. */
#define BSW_PACKED_MAX_QLEN 824
enum { BSW_PAIR_RAW = 1 };
typedef struct bsw_pair_desc {        /* 16 bytes */
    uint32_t q_off, r_off;
    uint16_t len2, len1;              /* query / reference (target) length, 1..32767     */
    uint16_t h0;                      /* seed score                                       */
    uint16_t flags;                   /* BSW_PAIR_RAW                                     */
} bsw_pair_desc;
typedef struct bsw_packed_batch {
    int64_t n_pairs;
    bsw_pair_desc* desc;
    uint32_t* q2; int64_t q2_words;
    uint32_t* r2; int64_t r2_words;
    uint8_t* raw_q; int64_t raw_q_bytes;
    uint8_t* raw_r; int64_t raw_r_bytes;
    int32_t ordered;
    int32_t reserved[3];
} bsw_packed_batch;
#ifndef BSW_OUTSCORE_DEFINED
#define BSW_OUTSCORE_DEFINED
typedef struct dnaOutScore {          /* bandedSWA.h:103-107 */
    int32_t score, tle, gtle, qle;
    int32_t gscore, max_off;
} OutScore;
#endif
typedef struct bsw_score16 {          /* the same six values in 16 bytes (all fit int16: bandedSWA.h:84) */
    int16_t score, qle, tle, gtle, gscore, max_off, reserved[2];
} bsw_score16;

/* Builders (host only; no CUDA call).  alloc / release = the allocator of the batch's five buffers: pass
 * bsw_host_alloc / bsw_host_free for page-locked memory (what the engine DMAs without staging), NULL / NULL for
 * malloc / free.  raw_min_qlen: queries of at least this length are stored RAW (0 = BSW_PACKED_MAX_QLEN + 1).
 *   bsw_batch_from_pairs   from the reference's layout (SeqPair[] + byte buffers): the packing loader
 *   bsw_batch_from_file    from the 3-line text format of main_banded.cpp:131-185
 *   bsw_batch_gen          the synthetic generator of SURVEY 8(d), straight into the packed layout
 *   bsw_batch_to_pairs     the inverse (tests, tools): pairs[] with idr / idq laid out consecutively, bytes in
 *                          ref / qer (capacities in bytes; BSW_ERR_NOMEM if too small)
 *   bsw_batch_release      frees the five buffers with `release` (NULL = free) and clears the struct */
typedef void* (*bsw_alloc_fn)(size_t bytes);
typedef void  (*bsw_release_fn)(void* p);
int  bsw_batch_from_pairs(const SeqPair* pairs, const uint8_t* seq_ref, const uint8_t* seq_qer, int64_t n_pairs,
                          int32_t raw_min_qlen, bsw_alloc_fn alloc, bsw_release_fn release, bsw_packed_batch* out);
int  bsw_batch_from_file(const char* path, int64_t max_pairs, int32_t raw_min_qlen, bsw_alloc_fn alloc,
                         bsw_release_fn release, bsw_packed_batch* out);
int  bsw_batch_to_pairs(const bsw_packed_batch* batch, SeqPair* pairs, uint8_t* seq_ref, int64_t ref_cap,
                        uint8_t* seq_qer, int64_t qer_cap);
void bsw_batch_release(bsw_packed_batch* batch, bsw_release_fn release);

/* replaces: getScores16 (bandedSWA.cpp:1124-1148) for a loader that emits the packed layout.  out[i] receives the
 * six result fields of pair i (input order).  Same kernels, same results as bsw_extend on the unpacked pairs.
 * Page-locked batch buffers and out (bsw_host_alloc) are DMA'd in place; pageable ones work, slower.
 * bsw_extend_packed16: the same call returning 16 bytes per pair. */
int bsw_extend_packed(bsw_engine* eng, const bsw_packed_batch* batch, int32_t w, OutScore* out);
int bsw_extend_packed16(bsw_engine* eng, const bsw_packed_batch* batch, int32_t w, bsw_score16* out);

/* ---- asynchronous submit + call coalescing (SURVEY 8(b)) -----------------------
 * replaces: the OpenMP loop of 512-pair getScores16 calls, main_banded.cpp:279-291 with scripts/run-cpu.sh:30.
 * bsw_extend_async queues the call and returns a ticket at once; a worker thread of the engine runs everything that is
 * queued at that moment -- calls of any threads, over any buffers, with the same w -- as ONE batch and writes every
 * call's six result fields into its own records; bsw_wait blocks until the ticket's results are there and returns
 * that call's status (cells_effective, optional: the call's share of the batch's effective DP cells).  Thread-safe:
 * any thread may submit and wait.  The buffers must stay valid until bsw_wait returns; every ticket must be waited for
 * exactly once.  The queue runs on a private child engine, so synchronous calls on `eng` may go on meanwhile.
 * bsw_async_stats: calls submitted / batches run so far (calls / batches = the coalescing factor). */
int bsw_extend_async(bsw_engine* eng, SeqPair* pairs, const uint8_t* seq_ref, const uint8_t* seq_qer, int64_t n_pairs,
                     int32_t w, int64_t* ticket);
int bsw_wait(bsw_engine* eng, int64_t ticket, int64_t* cells_effective);
int bsw_async_stats(const bsw_engine* eng, int64_t* calls, int64_t* batches);

/* ---- (f.1) band-doubling retry of the aligner ------------------------------
 * replaces: the MAX_BAND_TRY loops around ksw_extend2 in mem_chain2aln,
 * tools/bwa/bwamem.c:630,723-753 (left extension) and :770-800 (right extension):
 *     for (t = 0; t < max_try; ++t) { prev = score; w_t = w << t; extend with w_t;
 *                                     if (score == prev || max_off < (w_t>>1) + (w_t>>2)) break; }
 * batched: try t re-runs only the pairs that did not break at try t-1.  prev_score[i] is the
 * score before the first try (bwamem.c uses -1 for left extensions, :707, and the seed / left
 * score h0 for right extensions, :767); NULL means -1 for every pair.  band_used[i] (optional)
 * receives the band of the last try pair i ran (aw[] at bwamem.c:725,772).  The six result
 * fields hold the outcome of that last try. */
int bsw_extend_retry(bsw_engine* eng, SeqPair* pairs, const uint8_t* seq_ref,
                     const uint8_t* seq_qer, int64_t n_pairs, int32_t w, int32_t max_try,
                     const int32_t* prev_score, int32_t* band_used);

/* ---- (f.3) seed -> pair construction and the local / to-end decision --------
 * replaces: the body of mem_chain2aln, tools/bwa/bwamem.c:632-822 -- for every seed of a chain, in
 * the reference's order (by score, :661-665) and with its containment test (:667-700): the left
 * extension over the REVERSED query prefix and reference flank with h0 = len * match (:709-753),
 * the local-vs-to-end decision against pen_clip5 (:755-761), the right extension with h0 = the left
 * score (:765-800), its decision against pen_clip3 (:802-808), seedcov / w / seedlen0 (:812-822).
 * Batched over chains: round r extends the r-th surviving seed of every chain in two
 * bsw_extend_retry calls (all left flanks, then all right flanks); the containment test makes the
 * seeds of ONE chain -- and the chains of one read (bsw_chain.same_read) -- sequential; reads are
 * independent.
 *
 * bsw_seed = mem_seed_t (bwamem.c:168-172); coordinates are the reference's: rbeg in [0, 2 l_pac)
 * (forward strand, then the reverse complement), qbeg on the read.  A chain names its read
 * (query + query_off, l_query codes 0-4) and its reference window [rmax0, rmax1) -- what
 * bns_fetch_seq returned (bwamem.c:660) -- as ref + ref_off.  bsw_chain_window computes that
 * window (:643-659); the caller intersects it with the contig as bns_fetch_seq does
 * (bntseq.c:436-444) and fetches the bases.
 * out_regs must hold one bsw_alnreg per seed: the regions of chain c are written to
 * out_regs[chains[c].seed_first ...] in the order the reference pushes them, out_count[c] of them.
 * The engine's end_bonus must equal pen_clip5 and pen_clip3 (ksw_extend2 receives them as end_bonus,
 * :746,:793; bwa's default is 5 for all three).  zdrop_mode BSW_ZDROP_SCALAR reproduces ksw_extend2's
 * z-drop rule for e_del / e_ins != 1. */
typedef struct bsw_seed { int64_t rbeg; int32_t qbeg, len, score, reserved; } bsw_seed;
typedef struct bsw_chain {
    int64_t seed_first;          /* first seed of the chain in seeds[]                     */
    int32_t n_seeds, l_query;
    int64_t query_off;           /* the read: query[query_off .. query_off + l_query)      */
    int64_t rmax0, rmax1;        /* reference window, coordinates as rbeg                  */
    int64_t ref_off;             /* its bases: ref[ref_off .. ref_off + rmax1 - rmax0)     */
    int32_t same_read;           /* 1: same read as chains[c - 1] -- mem_align1_core pushes the regions of all
                                    chains of a read into ONE vector (bwamem.c:1105-1112), so this chain starts
                                    when the previous one is done and its containment test sees those regions */
    int32_t reserved;
} bsw_chain;
typedef struct bsw_alnreg {      /* the fields of mem_alnreg_t that mem_chain2aln computes (bwamem.h:71-91) */
    int64_t rb, re;
    int32_t qb, qe, score, truesc, w, seedcov, seedlen0, reserved;
} bsw_alnreg;
typedef struct bsw_chain_opt {
    int32_t w;                   /* opt->w                                                 */
    int32_t pen_clip5, pen_clip3;
    int32_t max_band_try;        /* MAX_BAND_TRY, bwamem.c:630 (2)                         */
} bsw_chain_opt;
int bsw_chain_window(const bsw_params* params, int32_t w, int64_t l_pac, const bsw_seed* seeds,
                     int32_t n_seeds, int32_t l_query, int64_t* rmax0, int64_t* rmax1);
int bsw_extend_chains(bsw_engine* eng, const bsw_chain* chains, int64_t n_chains, const bsw_seed* seeds,
                      const uint8_t* query, const uint8_t* ref, const bsw_chain_opt* opt,
                      bsw_alnreg* out_regs, int32_t* out_count);

/* ---- (f.4) banded global alignment with traceback -> CIGAR -------------------
 * replaces: ksw_global2 (tools/bwa/ksw.c:502-606, push_cigar :489-500) as bwa_gen_cigar2 (bwa.c:167) calls it for
 * every alignment region: global alignment of query[0, len2) against target[0, len1) inside the fixed
 * band |i - j| <= w[i], int32 scores, gap costs and scoring of the engine (match / -mismatch / ambig),
 * the reference's tie-breaking in every cell, its backtrack and its merged operation list.
 * pairs[i] supplies idr / idq / len1 / len2 (h0 and the result fields are not used).  Outputs:
 * score[i]; n_cigar[i]; the operations (len << 4 | op, op 0 = M, 1 = I, 2 = D, as in BAM and ksw.c) of
 * alignment i at cigar[cigar_off[i] .. cigar_off[i + 1]) -- cigar_off has n + 1 entries, cigar_cap is the
 * capacity of cigar in entries (sum of len1 + len2 always suffices; BSW_ERR_PARAM if it overflows).
 * Domain: |len1 - len2| <= w[i] (outside it the reference's backtrack leaves its matrix). */
int bsw_global(bsw_engine* eng, const SeqPair* pairs, const uint8_t* seq_ref, const uint8_t* seq_qer,
               int64_t n_pairs, const int32_t* w, int32_t* score, int32_t* n_cigar, uint32_t* cigar,
               int64_t cigar_cap, int64_t* cigar_off);

/* replaces: ksw_global2 (tools/bwa/ksw.c:502-606; push_cigar :489-500) with its int32 arithmetic, for alignment
 * regions beyond bsw_global's 32767-base lengths (bwa_gen_cigar2 on long-read regions).  Same arguments, outputs,
 * operation encoding, scoring and error codes as bsw_global; for any alignment inside bsw_global's domain the score
 * and the operations are bsw_global's.  One warp per alignment; runs on the engine's first device.
 * Domain (BSW_ERR_DOMAIN), checked for every alignment before any device work:
 *   1 <= len1, len2 <= 2^24 - 1, offsets >= 0, |len1 - len2| <= w[i] (a band wider than max(len1, len2) is that band);
 *   (len1 + len2 + 2) * c + o_del + o_ins <= 2^29, c = max(match, mismatch, |ambig|, e_del, e_ins): every real
 *     H / E / F of the alignment lies in [-2^29, 2^29], far above the reference's -2^30 sentinel, and no sum
 *     overflows (a path to any cell runs diagonally, then along one gap: at most max(len1, len2) + 2 steps of at most
 *     c each and one gap open);
 *   direction matrix len1 * 64 * ceil((min(len2, 2 w + 1) + 3) / 128) <= 2^31 bytes (4 bits per band cell). */
int bsw_global32(bsw_engine* eng, const SeqPair* pairs, const uint8_t* seq_ref, const uint8_t* seq_qer,
                 int64_t n_pairs, const int32_t* w, int32_t* score, int32_t* n_cigar, uint32_t* cigar,
                 int64_t cigar_cap, int64_t* cigar_off);

/* ---- (f.5) alignment regions -> alignment records (CIGAR, NM, MD) ---------------------------
 * replaces: the alignment part of mem_reg2aln (tools/bwa/bwamem.c, bwa 0.7.17) with infer_bw (bwamem.c) and
 * bwa_gen_cigar2 (tools/bwa/bwa.c), bns_depos (bntseq.h), for every region of bsw_extend_chains' output:
 *   w2 = max(infer_bw(qe-qb, re-rb, truesc, match, o_del, e_del), infer_bw(.., o_ins, e_ins)); if (w2 > w) w2 = min(w2, reg.w);
 *   up to three tries:  w2 = min(w2, w << 2); bwa_gen_cigar2 with band w2;  stop if score == last score or
 *                       w2 == w << 2;  else w2 <<= 1 and go on while score < truesc - match;
 *   bwa_gen_cigar2:     rseq = ref bytes of [rb, re); for rb >= l_pac query segment and rseq are both reversed (indels
 *                       come out leftmost in forward coordinates); l_query == re - rb and w2 == 0: one M run, score =
 *                       sum of the column scores, no DP; else ksw_global2 (bsw_global / bsw_global32) with band
 *                       max(min((max_gap + |rlen - l_query| + 1) >> 1, w2), |rlen - l_query| + 3), max_gap from
 *                       (((l_query + 1) >> 1) * match - o) / e + 1 for both gap kinds, at least 1;  NM and MD over the
 *                       (reversed) sequences, bases through "ACGTN" (rb < l_pac) or "TGCAN"; a D that is the first or
 *                       the last operation is not in MD or NM; an I does not reset the match run;
 *   then:               pos = rb < l_pac ? rb : 2 l_pac - 1 - (re - 1);  a leading D is dropped and moves pos, else a
 *                       trailing D is dropped (only one end);  soft clips (op 3) of qb and l_query - qe bases, swapped
 *                       when is_rev, are added at the ends.
 * Operations are len << 4 | op in bwa's internal order "MIDSH": 0 = M, 1 = I, 2 = D, 3 = SOFT CLIP (not BAM's 4).
 * regs[i].reg supplies rb re qb qe truesc w (the other fields are ignored); the read is
 * query[query_off .. + l_query) (codes 0-4), the reference bases ref[ref_off .. + re - rb) as bns_get_seq(rb, re) returns
 * them (for rb >= l_pac the reverse complement of the forward strand, i.e. D[rb, re) with D = G + revcomp(G)).  A region
 * with rb < 0 or re < 0 gives the unmapped record: pos = -1, no operations, empty MD, no work.
 * Outputs: out[i]; the operations of region i at cigar[cigar_off[i] .. cigar_off[i + 1]) (clips included); its MD at
 * md[md_off[i] .. md_off[i + 1]) without a NUL.  cigar_off / md_off have n + 1 entries.  Capacities that always suffice,
 * per region:  (qe - qb) + (re - rb) + 2 operations;  4 (qe - qb) + (re - rb) + 1 MD bytes (MD holds one number per
 * mismatch and per inner D plus the last one, at most n_mm + n_D + 1 numbers, each of at most u + 1 digits for a run of
 * u matches; the letters are n_mm mismatches and the deleted bases with one '^' per inner D; with
 * sum u + n_mm <= qe - qb, n_mm <= qe - qb, n_D <= qe - qb (two D runs are separated by an operation that consumes query)
 * and deleted bases <= re - rb the total is at most 4 (qe - qb) + (re - rb) + 1).  A buffer that cannot take the results
 * gives BSW_ERR_PARAM (cigar: before any device work; md: after the chunks that fit are written).
 * Domain (BSW_ERR_DOMAIN), checked for every region before any device work: 0 <= w <= 2^28; rb < re <= 2 l_pac, not
 * bridging the strands (rb < l_pac < re); 0 <= qb < qe <= l_query; 1 <= l_query, re - rb <= 2^24 - 1; offsets >= 0;
 * bsw_global32's value and direction-matrix bounds at the widest band the loop can reach.
 * DP tries run through bsw_global (max(len1, len2) <= 32767) or bsw_global32 (longer); the finishing pass (NM, MD, the
 * fast path's score) runs on the device.  Runs on the engine's first device.  Statistics: the sums over the call's DP
 * calls and the finishing pass; ms_kernel includes both, ms_sort is the finishing pass's device time alone. */
typedef struct bsw_reg_in {        /* one region to turn into an alignment record */
    bsw_alnreg reg;                /* from bsw_extend_chains: rb re qb qe truesc w are read, the rest ignored */
    int64_t query_off;             /* the read: query[query_off .. + l_query), codes 0-4 */
    int64_t ref_off;               /* ref[ref_off .. + re - rb): the bases bns_get_seq(rb, re) returns */
    int32_t l_query, reserved;
} bsw_reg_in;
typedef struct bsw_aln {           /* mem_aln_t's alignment fields */
    int64_t pos;                   /* forward-strand 0-based leftmost position after the squeeze; -1 = unmapped */
    int32_t is_rev, n_cigar, NM;
    int32_t gscore;                /* global score of the last try (mem_aln_t.score is reg.score, the caller has it) */
    int32_t w;                     /* band w2 of the last try */
    int32_t reserved;
} bsw_aln;
int bsw_reg2aln(bsw_engine* eng, const bsw_reg_in* regs, int64_t n, const uint8_t* query, const uint8_t* ref,
                int64_t l_pac, int32_t w, bsw_aln* out, uint32_t* cigar, int64_t cigar_cap, int64_t* cigar_off,
                char* md, int64_t md_cap, int64_t* md_off);

/* Pinned host memory.  bsw_extend takes any host pointers; when all three buffers (pairs,
 * seq_ref, seq_qer) are page-locked -- allocated here, or registered, or pinned by the caller's
 * own CUDA / torch allocator -- the engine DMAs them as they are and DMAs the records back with
 * the six result fields filled in ("direct" route: no host pass over the payload; the input
 * fields of pairs[] are rewritten with the values they had).  Pageable buffers
 * go through one streaming host pass into pinned staging instead.  A maintainer's binding swaps
 * the _mm_malloc calls of main_banded.cpp:244-246 for bsw_host_alloc (INTEGRATION.md). */
void* bsw_host_alloc(size_t bytes);                 /* NULL on failure */
void  bsw_host_free(void* p);
int   bsw_host_register(void* p, size_t bytes);     /* page-locks an existing allocation */
int   bsw_host_unregister(void* p);

/* Split form of the same call, so that a caller (and bench.py) can keep a batch
 * resident in HBM and time the DP kernels alone:
 *   stage  = bucket + 2-bit pack + H2D      (host buffers -> HBM)
 *   run    = DP kernels only on the staged batch (repeatable)
 *   fetch  = D2H + scatter into pairs[] in input order                       */
int bsw_stage(bsw_engine* eng, const SeqPair* pairs, const uint8_t* seq_ref,
              const uint8_t* seq_qer, int64_t n_pairs, int32_t w);
int bsw_run_staged(bsw_engine* eng);
int bsw_fetch(bsw_engine* eng, SeqPair* pairs, int64_t n_pairs);

int bsw_get_stats(const bsw_engine* eng, bsw_stats* out);

/* ---- a6 / (e): length bucketing and the multi-GPU partitioner --------------
 * replaces: sortPairsLen / sortPairsId (bandedSWA.cpp:368-420) and the OpenMP
 * batch loop (main_banded.cpp:279-291).
 * Inside bsw_extend / bsw_extend_packed an engine with several devices cuts the call's pairs, in input order, into one
 * contiguous range per device with equal estimated DP cost sum len1*min(len2, 2w+1) (bsw_split_by_cost is that cut,
 * exposed for callers that shard across processes), runs every range on its own host thread through its device's
 * chunk pipeline (length bucketing per chunk, on the device), and every result lands at its pair's input position.
 * bsw_bucket_order is the host-side mirror of sortPairsLen for callers that want the processing order themselves:
 * order[] receives indices into pairs[] sorted by (len2, h0, len1).  (Round 1's bsw_partition -- a global bucketing dealt
 * onto shards in blocks -- lost the comparison against the contiguous cut and is gone.) */
int bsw_split_by_cost(const SeqPair* pairs, int64_t n_pairs, int32_t w, int32_t n_shards, int64_t* shard_begin);
int bsw_bucket_order(const SeqPair* pairs, int64_t n_pairs, int64_t* order);

/* ---- synthetic-pair generator (SURVEY 8(d); the reference has no generator:
 * its inputs come from the dumper tools/bwa/bwamem.c:741-745,788-792) --------- */
typedef struct bsw_gen_config {
    uint64_t seed;
    int64_t  n_pairs;
    int32_t  qlen_min, qlen_max;     /* len2 ~ U[min,max]                               */
    int32_t  tail_min, tail_max;     /* random reference tail ~ U[min,max]              */
    int32_t  h0_min, h0_max;         /* h0 ~ U[min,max]                                 */
    int32_t  max_len1;               /* clip reference length (0 = none)                */
    int32_t  max_score8;             /* if > 0: clip h0 so that h0 + len2*match <= it   */
    double   error_rate;             /* total, split equally sub / ins / del            */
    double   n_rate;                 /* probability of an ambiguous base (code 4)       */
    int32_t  match;                  /* only used by max_score8                         */
    int32_t  reserved[7];
} bsw_gen_config;

/* Named configs of BASELINE.json: 0 small, 1 8-bit, 2 16-bit, 3 large, 4 sweep. */
int     bsw_gen_named_config(int32_t which, bsw_gen_config* out);
/* Upper bounds of the buffers bsw_gen_pairs needs for this config. */
int     bsw_gen_bounds(const bsw_gen_config* cfg, int64_t* ref_bytes, int64_t* qer_bytes);
/* Fills pairs[0..n), seq_ref, seq_qer (one base code per byte, 0-3, 4 = N).
 * Pairs first_pair .. first_pair+n of the config's stream are produced, so a
 * shard of a big config can be generated without the rest.  Returns bytes used
 * through *ref_used / *qer_used. */
int     bsw_gen_pairs(const bsw_gen_config* cfg, int64_t first_pair, int64_t n,
                      SeqPair* pairs, uint8_t* seq_ref, uint8_t* seq_qer,
                      int64_t* ref_used, int64_t* qer_used);

/* The same stream, straight into the packed layout (see bsw_batch_from_pairs for alloc / release). */
int     bsw_batch_gen(const bsw_gen_config* cfg, int64_t first_pair, int64_t n, int32_t raw_min_qlen,
                      bsw_alloc_fn alloc, bsw_release_fn release, bsw_packed_batch* out);

/* ---- dataset I/O: the 3-line text format of main_banded.cpp:131-185 --------- */
int64_t bsw_count_pairs_file(const char* path);
int     bsw_read_pairs_file(const char* path, int64_t max_pairs, SeqPair* pairs,
                            uint8_t* seq_ref, int64_t ref_cap, uint8_t* seq_qer, int64_t qer_cap,
                            int64_t* n_read);
int     bsw_write_pairs_file(const char* path, const SeqPair* pairs, int64_t n_pairs,
                             const uint8_t* seq_ref, const uint8_t* seq_qer);

/* ---- measured integer/DPX peak (roofline denominator, SURVEY 8(d)) ---------- */
/* Runs a dependency-free __viaddmax_s32 microbenchmark on the engine's first
 * device and returns lane-ops/s (0 on failure). */
double  bsw_measure_int_peak(bsw_engine* eng);

/* library identification: "bsw_b200 <version> sm_100a" */
const char* bsw_version(void);

#ifdef __cplusplus
}
#endif
#endif /* BSW_B200_H */

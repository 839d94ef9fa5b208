/*
 * lvc.h -- C-ABI of the B200-native live-variant-caller hot path (liblvc_b200.so).
 *
 * The reference (COVID-SpiNGS/covid-spings-variant-caller) is 100% Python and has NO FFI; the drop-in
 * boundary is the Python class variant_caller/live_variant_caller.py:21 `LiveVariantCaller`.  Each
 * entry point below cites the reference code it replaces; INTEGRATION.md shows the ctypes binding a
 * maintainer of the reference would add.  Plain pointers and sizes only -- no torch / numpy types.
 *
 * Conventions: every function returning int returns 0 on success and a negative LVC_E* code on
 * failure; lvc_last_error(h) gives the message.  A handle owns ONE contig's persistent device tables
 * (the reference's `self.memory`, live_variant_caller.py:31) and one CUDA stream.  Handles are not
 * thread-safe; the Python shim serialises calls with a lock (the reference calls the class from
 * un-locked daemon threads, client_server/vc_queue.py:99-111).
 */
#ifndef LVC_H_
#define LVC_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define LVC_OK 0
#define LVC_EINVAL (-1)     /* bad argument / malformed batch                                   */
#define LVC_ECUDA (-2)      /* CUDA runtime error (message has the cudaError string)            */
#define LVC_ENOMEM (-3)
#define LVC_EUNSORTED (-4)  /* reads not coordinate sorted (htslib errors out too, SURVEY B2)   */
#define LVC_ERANGE (-5)     /* a read extends past the reference / ordinal space exhausted      */
#define LVC_ENODEVICE (-6)  /* no CUDA device: there is NO CPU fallback                          */
#define LVC_EIO (-8)        /* file cannot be opened / read                                     */
#define LVC_EAGAIN (-7)     /* async pushes met a new (allele group, quality) key: redo synchronously */

#define LVC_MAX_DEPTH_DEFAULT 8000 /* pysam pileup() default max_depth [EXT], SURVEY B1/B4 */

typedef struct lvc_handle lvc_handle;

/*
 * One batch of alignments of ONE contig, coordinate sorted, structure-of-arrays (SURVEY F1).
 * This is what `pysam.AlignmentFile(...).pileup(...)` consumes inside process_bam
 * (live_variant_caller.py:54-60).  All pointers are host pointers for lvc_push_batch and device
 * pointers for lvc_push_batch_device.
 *
 *   seq_off[i]  = byte offset of read i's qualities in `qual`; MUST be even; the read's 4-bit bases
 *                 start at seq4[seq_off[i]/2] (BAM nibble codes "=ACMGRSVTWYHKDBN", high nibble first).
 *                 l_qseq of a read is the sum of its query-consuming CIGAR ops (BAM invariant).
 *   cigar       = BAM encoding  len<<4 | op,  op in MIDNSHP=X (0..8).
 *   keep[i]     bit0 = the read survives the host-side, order-dependent admission rules (htslib
 *                 max_depth rule, SURVEY B4; computed by lvc_admit); flag / mapq / orphan filters
 *                 (SURVEY B2) are re-evaluated on the device.  bit1 = hint: every base of the read
 *                 is A, C, G or T (set ONLY if true; reads without it take the general kernel).
 *   The payload arrays seq4 / qual must be readable for 16 bytes past their end (TMA stages whole
 *   16-byte groups) and 16-byte aligned at their start.
 *
 *   Quality codes (qual_bits = 2) [EXT]: instrument-binned base qualities (NovaSeq RTA3: 2, 12, 23, 37) take four
 *   values, so a batch whose qualities take at most four distinct values may carry them as 2-bit CODES, four bases
 *   per byte: the base with quality index x (x = seq_off[i] + k, the index it would have in the byte array) has its
 *   code in bits 2*(x & 3) of qual[x >> 2], and its phred value is qual_dict[code].  Offsets, seq4 and n_qual_bytes
 *   keep their meaning (`qual` then holds n_qual_bytes / 4 bytes); the tables, records and checkpoints that result
 *   are identical to those of the byte form.  The payload that crosses PCIe drops from 1.5 to 0.75 bytes per base.
 *   lvc_read_alignments produces this form by itself when a file qualifies (lvc_reads_batch; lvc_reads_batch_bytes
 *   always gives the byte form); lvc_pack_quality_codes converts a byte array.  Code batches run on the generation-5
 *   tiled kernel and the any-record kernel (impl 0, 1 or 5; other selections are refused with LVC_EINVAL).
 *
 *   Base codes (seq_form = 2 | threshold << 8) [EXT]: a quality-code batch may carry its bases as 2-bit codes too
 *   (A, C, G, T = 0..3, the base with quality index x in bits 2*(x & 3) of seq4[x >> 2]; `seq4` then holds
 *   n_qual_bytes / 4 bytes).  The pileup the reference iterates never shows a base whose quality is below
 *   min_base_quality (live_variant_caller.py:56-60), so such a base -- every no-call an Illumina instrument writes:
 *   N at quality 2 --, any base of a read the admission dropped and pad nibbles need no representation; a batch in
 *   which every OTHER base is A, C, G or T qualifies (lvc_pack_base_codes; lvc_reads_batch_for makes the codes for a
 *   given threshold).  Tables, records and checkpoints are identical; the payload over PCIe is 0.5 bytes per base.
 *   A handle whose threshold is lower than the one in seq_form refuses the batch (LVC_EINVAL).
 */
typedef struct lvc_batch {
    uint32_t n_reads;
    uint32_t qual_bits;    /* 0 or 8: one phred byte per base; 2: 2-bit codes into qual_dict */
    uint64_t n_cigar_ops;  /* == cigar_off[n_reads] */
    uint64_t n_qual_bytes; /* == seq_off[n_reads]   */
    const int32_t* pos;    /* [n_reads] 0-based leftmost reference position */
    const uint16_t* flag;  /* [n_reads] */
    const uint8_t* mapq;   /* [n_reads] */
    const uint8_t* keep;   /* [n_reads] */
    const uint32_t* cigar_off; /* [n_reads+1] */
    const uint32_t* cigar;     /* [n_cigar_ops] */
    const uint64_t* seq_off;   /* [n_reads+1] */
    const uint8_t* seq4;       /* [n_qual_bytes/2] */
    const uint8_t* qual;       /* [n_qual_bytes], or [n_qual_bytes/4] codes when qual_bits == 2 */
    uint8_t qual_dict[4];      /* qual_bits == 2: phred value of code 0..3 (unused entries 0) */
    uint32_t seq_form;         /* bits 0..7: width of a base in `seq4`: 0 or 4 = BAM nibbles, 2 = codes (below);
                                  bits 8..15: the base-quality threshold 2-bit codes were made for */
} lvc_batch;

/* Byte qualities -> 2-bit codes (no GPU needed).  Returns the number of distinct values found (1..4) after writing
 * dict_out[4] (ascending, unused entries 0) and codes_out[(n_qual_bytes + 3) / 4]; returns 0 and writes nothing useful
 * if the array holds more than four distinct values (the batch stays in the byte form); LVC_EINVAL on null arguments.
 * n_reads / keep / seq_off / cigar_off / cigar (optional, all or none): only the l_qseq qualities of the reads with keep
 * bit0 set decide -- the payload of reads the admission dropped is never read by any kernel, and the pad byte of an
 * odd-length read is not a quality.  Bytes that do not decide get code 0. */
int lvc_pack_quality_codes(const uint8_t* qual, uint64_t n_qual_bytes, uint32_t n_reads, const uint8_t* keep,
                           const uint64_t* seq_off, const uint32_t* cigar_off, const uint32_t* cigar, int n_threads,
                           uint8_t dict_out[4], uint8_t* codes_out);

/* 4-bit BAM base codes -> 2-bit codes (A, C, G, T = 0..3; the base with quality index x in bits 2*(x & 3) of
 * codes_out[x >> 2], like the quality codes) [EXT] (no GPU needed).  Only a batch with quality codes (qual_bits = 2) may
 * carry them: lvc_batch.seq4 = codes_out, lvc_batch.seq_form = 2 | min_base_quality << 8; its payload is then 0.5 bytes
 * per base.  Returns 1 if every base that can reach the tables is A, C, G or T -- a base of a read the admission dropped,
 * a base whose quality is below min_base_quality (pileup(min_base_quality=...) never shows it,
 * live_variant_caller.py:56-60: Illumina writes its N calls with quality 2) and the pad nibble of an odd-length read may be
 * anything, and get code 0 --, 0 if not (the batch keeps its nibbles); LVC_EINVAL on null arguments.  `qual`: the phred
 * bytes.  lvc_push_batch refuses such a batch on a handle whose threshold is LOWER than the one the codes were made for. */
int lvc_pack_base_codes(const uint8_t* seq4, const uint8_t* qual, uint64_t n_qual_bytes, uint32_t n_reads, const uint8_t* keep,
                        const uint64_t* seq_off, const uint32_t* cigar_off, const uint32_t* cigar, int min_base_quality,
                        int n_threads, uint8_t* codes_out);

/* One (position, allele) that passed the genotype-stage filters; the host finalises log10/round/
 * formatting with the host libm so the text matches the reference (SURVEY A6). */
typedef struct lvc_candidate {
    int32_t pos;       /* 0-based */
    uint8_t code;      /* BAM nibble code of the allele */
    uint8_t ref;       /* reference byte at pos (as stored in the FASTA) */
    uint16_t pad0;
    uint32_t ad;       /* allele depth  = len(snvs[allele])               (live_variant_caller.py:149) */
    uint32_t dp;       /* totalDepth                                      (live_variant_caller.py:179) */
    uint32_t first;    /* ordinal of the first read that deposited this allele (dict order, SURVEY A7) */
    uint32_t pad1;
    double L;          /* genotype_likelihood(allele, snvs)               (utils.py:16-24)  */
    double S;          /* sum of L over the alleles at pos, 1.0 if 0      (live_variant_caller.py:145-146) */
    double esum;       /* sum of error probabilities of the allele; qual = esum/ad (live_variant_caller.py:168) */
} lvc_candidate;

#define LVC_GENO_EMIT_ALL 1u /* flags: emit every allele of every gated site (tests / export) */

/* ---- lifetime -------------------------------------------------------------------------------
 * lvc_create  <- LiveVariantCaller.__init__ (live_variant_caller.py:22-32): thresholds that act at
 *                deposit time (min_base_quality, min_mapping_quality :57-58) are fixed per handle.
 *                `ref_bytes` = the contig as stored in the FASTA (case preserved, :78-81).
 *                `stream` = a cudaStream_t to launch on, or NULL to create a private one.
 * lvc_destroy <- __del__ (:34-35).      lvc_reset <- reset_memory (:37-38). */
int lvc_create(lvc_handle** out, int device, int64_t ref_len, const uint8_t* ref_bytes,
               int min_base_quality, int min_mapping_quality, void* stream);
void lvc_destroy(lvc_handle* h);
int lvc_reset(lvc_handle* h);
const char* lvc_last_error(const lvc_handle* h); /* h may be NULL: error of the last failed lvc_create */
int lvc_set_stream(lvc_handle* h, void* stream);
int lvc_sync(lvc_handle* h);

/* ---- host-side admission (no GPU needed) -------------------------------------------------------
 * Restates the order-dependent part of pysam's pileup engine that process_bam relies on
 * (live_variant_caller.py:56-60): read-level filter (SURVEY B2) + htslib bam_plp_push max_depth rule
 * (SURVEY B4).  Writes keep_out[i] in {0,1}.  Returns LVC_EUNSORTED for unsorted input. */
int lvc_admit(uint32_t n_reads, const int32_t* pos, const uint16_t* flag, const uint8_t* mapq,
              const uint32_t* cigar_off, const uint32_t* cigar, int min_mapping_quality, int max_depth,
              uint8_t* keep_out);

/* ---- mate overlaps (no GPU needed) --------------------------------------------------------------
 * The reference calls pileup() with pysam's default ignore_overlaps=True (live_variant_caller.py:56-60): htslib
 * rewrites the base qualities of the two reads of a proper pair where they cover the same reference positions
 * (bam_plp overlap hash + tweak_overlap_quality, SURVEY B5), and both pysam's base-quality filter and the phreds
 * the reference stores (:97-103) see the rewritten values.  lvc_admit_overlaps is lvc_admit plus that rewrite, done
 * IN PLACE on `qual` inside the same sequential pass (entries leave the hash when a read is swept or dropped by
 * max_depth, exactly as in the pileup engine).  htslib changed the rule between releases and pysam is unpinned in
 * the reference (requirements.txt:1): `overlap_model` selects the release line.
 *   name_off[n_reads+1] / names: concatenated QNAMEs (no terminators); mate_pos = PNEXT (0-based, -1 if absent);
 *   mate_ref: 1 = RNEXT is this contig, 0 = another contig, -1 = absent; tlen = TLEN.
 *   n_pairs / n_bases (optional): pairs whose qualities were rewritten / quality bytes rewritten. */
#define LVC_OVERLAP_OFF 0          /* pileup(ignore_overlaps=False) */
#define LVC_OVERLAP_HTSLIB_1_10 1  /* htslib <= 1.10: the later mate is zeroed */
#define LVC_OVERLAP_HTSLIB_1_13 2  /* htslib >= 1.13: mate chosen by a hash of the read name; deletions handled */
#define LVC_OVERLAP_DEFAULT LVC_OVERLAP_HTSLIB_1_13
int lvc_admit_overlaps(uint32_t n_reads, const int32_t* pos, const uint16_t* flag, const uint8_t* mapq,
                       const uint32_t* cigar_off, const uint32_t* cigar, const uint64_t* seq_off, const uint8_t* seq4,
                       uint8_t* qual, const uint32_t* name_off, const char* names, const int32_t* mate_pos,
                       const int8_t* mate_ref, const int32_t* tlen, int min_mapping_quality, int max_depth,
                       int overlap_model, uint8_t* keep_out, uint64_t* n_pairs, uint64_t* n_bases);

/* ---- native host ingest (no GPU needed): BAM (BGZF, multi-threaded inflate) or SAM text -> packed batch ----
 * Replaces pysam.AlignmentFile(inputBam, 'rb') + the region iterator (live_variant_caller.py:55-60) and, for SAM
 * input, pysam.sort's order (client_server/vc_queue.py:34).  Reads of `contig` (NULL / "" = first @SQ) are packed
 * into page-locked arrays when a CUDA device is present (lvc_push_batch then reads the payload in place), the keep
 * mask (lvc_admit_overlaps + the ACGT-only hint) is filled in and the qualities of overlapping mates are rewritten
 * (lvc_read_alignments uses LVC_OVERLAP_DEFAULT; lvc_read_alignments_ex takes the model).  Records the path cannot
 * reproduce (missing qualities, CG-tag CIGARs) are refused with LVC_EINVAL and a message in errbuf.  Re-entrant: any
 * number of threads may call it at once (the phase timer is per call).
 * n_threads <= 0: all host threads.  The page-locked arrays of a freed lvc_reads go to a process-wide pool (at most
 * 4 GiB parked) and are reused by later calls; LVC_INGEST_TIMING=1 in the environment prints the phase times.
 * BGZF blocks are inflated by the library's own DEFLATE decoder (csrc/inflate_fast.hpp: 64-bit bit buffer, one table
 * lookup per symbol, 2.3x zlib's inflate on BAM blocks) into a huge-page backed array, and the CRC-32 of every block is
 * checked (carry-less multiplication where the CPU has it, csrc/crc32_clmul.hpp), as htslib does; LVC_INFLATE=zlib
 * selects zlib's inflate() instead (A/B measurements).  A corrupt or truncated block fails the call.  The array the blocks
 * are inflated into (one mapping of the file's uncompressed size) is parked between calls, at most 2 GiB, so the next file
 * neither faults its pages in again nor unmaps them (config-2 BAM: 70 against 77 ms); LVC_INGEST_PARK=0 disables it. */
typedef struct lvc_reads lvc_reads;
int lvc_read_alignments(const char* path, const char* contig, int min_mapping_quality, int max_depth, int n_threads,
                        lvc_reads** out, char* errbuf, int errlen);
int lvc_read_alignments_ex(const char* path, const char* contig, int min_mapping_quality, int max_depth, int n_threads,
                           int overlap_model, lvc_reads** out, char* errbuf, int errlen);
int lvc_reads_overlap_stats(const lvc_reads* r, uint64_t* n_pairs, uint64_t* n_bases);
int lvc_reads_batch(const lvc_reads* r, lvc_batch* batch_out);   /* pointers stay valid until lvc_reads_free; the
                                                                    quality-code form when the file qualifies */
int lvc_reads_batch_bytes(const lvc_reads* r, lvc_batch* batch_out); /* always one phred byte per base */
/* lvc_reads_batch for a handle whose base-quality threshold is min_base_quality: a quality-code batch also gets 2-bit
 * base codes (lvc_pack_base_codes) when its bases allow it -- 0.5 instead of 0.75 payload bytes per base over PCIe.
 * LVC_BASE_CODES=0 in the environment keeps the nibbles. */
int lvc_reads_batch_for(const lvc_reads* r, int min_base_quality, lvc_batch* batch_out);
/* Leaves out the reads the admission dropped (keep bit0 clear: read-level filter, max_depth rule): no kernel reads them,
 * the tables that result are the same, and first-seen ordinals number the admitted reads in the same order.  The arrays
 * are re-packed (batches obtained before the call are invalid).  Returns 1 if reads were removed, 0 if the batch stays
 * as it was (nothing dropped, or no memory for the copy).  What lvc_push_batch moves over PCIe shrinks by the dropped
 * reads' per-read arrays: 60 % of the reads of an amplicon sample at 10,000x. */
int lvc_reads_compact(lvc_reads* r, int n_threads);
int lvc_reads_info(const lvc_reads* r, char* contig_name, int name_cap, int64_t* contig_len, int* n_contigs, int* pinned);
void lvc_reads_free(lvc_reads* r);

/* ---- deposit: process_bam / process_pileup_column / process_svn (live_variant_caller.py:54-103) ----
 * Walks every kept read's CIGAR on the device and adds its bases/qualities to the persistent
 * per-position tables.  Accumulates across calls (live batches).  `impl`: 0 = auto (the tiled kernel for short-read
 * batches, the long-read kernel 6 for batches averaging more than 4 CIGAR ops per read -- 3 if they average more than
 * 40), 1 = general kernel only (one thread per read), 2 = tiled kernel staging the raw payload with TMA, 3 = one warp
 * per read (any record, wide quality alphabets), 4 = tiled kernel staging 4-bit keys with SWAR counters, 5 = tiled
 * kernel with bit-sliced counters and per-task flush, 6 = long-read kernel (CTA of up to 32 reads: run units, compacted
 * passing bases, first-seen hints from the genotype pass).  The fast kernels use the warp path for the reads they cannot
 * take.  Device-resident batches (lvc_push_batch_device*): the kernels read `seq4` and `qual` in aligned 16-byte
 * groups, so both arrays must be READABLE up to the next 16-byte boundary past their last byte (any cudaMalloc
 * allocation is; a sub-allocation that ends exactly at the end of a mapped range is not).  NVTX ranges named after the
 * entry points (lvc_read_alignments, lvc_push_batch*, lvc_genotype*, lvc_reduce_tables) are emitted when a tool is
 * attached. */
/* How lvc_push_batch moves a host batch: the per-read arrays are copied; the payload (seq4 + qual) of a batch WITHOUT
 * dropped reads (lvc_reads_compact / every keep bit0 set) is copied in bulk, one copy per array; the payload of a batch
 * with dropped reads is read in place over PCIe when the caller's arrays are page-locked (only the chunks with admitted
 * reads are touched), else the byte ranges of the admitted reads are copied.  Environment switches for experiments:
 * LVC_ZERO_COPY=0 (never read in place), LVC_DENSE_BULK_COPY=0 (always read page-locked payload in place),
 * LVC_ZC_HEADERS=1 (per-read arrays other than `keep` read in place too), LVC_QUALITY_CODES=0 (the ingest keeps the byte
 * form). */
int lvc_push_batch(lvc_handle* h, const lvc_batch* host_batch);
int lvc_push_batch_device(lvc_handle* h, const lvc_batch* device_batch);
int lvc_set_impl(lvc_handle* h, int impl);
/* Stream-ordered variant for back-to-back live batches: enqueues the kernels and returns.  No replay is
 * possible, so every (allele group, quality) key must already have a plane (true after the first
 * synchronous push of a run with the same quality alphabet); lvc_check_async() synchronises and
 * reports LVC_EAGAIN if a key was missing, LVC_ERANGE if a read left the reference. */
int lvc_push_batch_device_async(lvc_handle* h, const lvc_batch* device_batch);
int lvc_check_async(lvc_handle* h);
/* pinned host memory for the SoA buffers (cudaHostAlloc) */
void* lvc_host_alloc(uint64_t bytes);
void lvc_host_free(void* p);

/* ---- genotype: prepare_variants (live_variant_caller.py:120-231) + utils.py:9-24 -----------------
 * e_lut[q] = math.pow(10, q/-10) and om_lut[q] = 1.0 - e_lut[q] MUST be built by the caller with the
 * host libm (SURVEY A6: never pow() on the device).  Writes up to `cap` candidates; *n_out is the
 * number found (may exceed cap: call again with a larger buffer).  Also refreshes the dense
 * per-position outputs (depth, A/C/G/T depth, A/C/G/T likelihood) readable by lvc_copy_dense. */
int lvc_genotype(lvc_handle* h, int64_t min_total_depth, int64_t min_allele_depth, double min_evidence_ratio,
                 const double* e_lut, const double* om_lut, uint32_t flags, lvc_candidate* out, uint32_t cap,
                 uint32_t* n_out);
/* device-only variant (no D2H, for timing); lvc_fetch_candidates reads the result back. */
int lvc_genotype_device(lvc_handle* h, int64_t min_total_depth, int64_t min_allele_depth,
                        double min_evidence_ratio, const double* e_lut, const double* om_lut, uint32_t flags);
int lvc_genotype_device_async(lvc_handle* h, int64_t min_total_depth, int64_t min_allele_depth,
                              double min_evidence_ratio, const double* e_lut, const double* om_lut, uint32_t flags);
int lvc_fetch_candidates(lvc_handle* h, lvc_candidate* out, uint32_t cap, uint32_t* n_out);
/* restrict the genotype pass to positions [p0, p1) (multi-GPU: each rank genotypes its slice of the reduced
 * tables); p1 < 0 restores the whole contig.  Dense outputs outside the range keep their previous values. */
int lvc_set_genotype_range(lvc_handle* h, int64_t p0, int64_t p1);
int lvc_copy_dense(lvc_handle* h, uint32_t* depth /*[G]*/, uint32_t* ad /*[G*4] A,C,G,T*/,
                   double* lik /*[G*4]*/);

/* ---- consensus genome and coverage summary [EXT] ------------------------------------------------
 * The reference gives neither; both are computed on the device from the count tables alone (no genotype pass, no
 * first-seen ordinals), so the result is the same for any deposit kernel, batch form, checkpoint load or reduction.
 * For each position p in [p0, p1):
 *   nA, nC, nG, nT = sums over the group-0 planes of slots 0..3;  nO = sum over the group-1..3 planes and all four
 *   slots (=, IUPAC letters, N read as bases);  nD = dels[p];  d = nA + nC + nG + nT + nO + nD (64-bit; the
 *   totalDepth of `memory`, 0 where p is not in it).
 *   d == 0 or d < min_depth                                         -> 'N'
 *   members = (count, rank) for rank, count in enumerate(nA, nC, nG, nT, nD) if count > 0, sorted by count descending,
 *             ties by rank (A < C < G < T < deletion); take members in that order until cum / d >= threshold (fp64
 *             division); never reached (the rest of the depth is in other codes)   -> 'N'
 *   deletion taken first                                            -> '-'
 *   else "=ACMGRSVTWYHKDBN"[mask], mask = OR of (1 << rank) of the taken bases (A=1 C=2 G=4 T=8: the BAM nibble
 *   alphabet is the IUPAC code of the mask; a deletion taken later is not in the mask).
 * threshold 0 is a plain majority call; 0.5-0.75 gives mixed positions ambiguity codes.  Letters are uppercase.
 * Insertions are not in these tables, so the letters contain none; unless counting is enabled (lvc_enable_insertions
 * below), the consensus has no insertions.
 * Statistics over the same range: n_positions, depth_sum, depth_max, n_low_depth (d < min_depth), n_N (every 'N'),
 * n_deleted (every '-'), n_ambiguous (two- and three-base codes), n_mismatch (a single-base call other than the reference
 * letter, where toupper(ref[p]) is A/C/G/T), depth_ge[i] (d >= depth_thresholds[i], i < n_thresholds; the rest 0).
 * p1 < 0: the whole contig.  threshold outside [0, 1] or NaN, n_thresholds outside 0..8 or a range outside [0, G):
 * LVC_EINVAL.  seq_out (p1 - p0 bytes) and stats_out may be NULL.  Synchronous: returns after the copy back.  The
 * kernel runs on the handle's stream after everything enqueued before (lvc_push_batch_device_async included).
 * After lvc_peer_attach or lvc_reduce_tables(LVC_REDUCE_SCATTER) a rank's tables hold its own slice only: call it with
 * the range of lvc_position_slice. */
typedef struct lvc_consensus_stats {
    uint64_t n_positions, depth_sum, depth_max, n_low_depth, n_N, n_deleted, n_ambiguous, n_mismatch;
    uint64_t depth_ge[8];
} lvc_consensus_stats;                                                   /* 128 bytes */
int lvc_consensus(lvc_handle* h, int64_t p0, int64_t p1, uint64_t min_depth, double threshold,
                  const uint32_t* depth_thresholds, int n_thresholds, uint8_t* seq_out, lvc_consensus_stats* stats_out);

/* ---- insertions in the consensus genome [EXT] ---------------------------------------------------
 * Opt-in: records, VCF, `memory` and checkpoints never contain insertions (the reference emits none), and nothing that
 * exists changes while counting is on, except that each push launches one more kernel.
 * Counting rule.  A read the deposit walks (it passes read_passes_filter, has a reference-consuming op and lies inside
 * [0, G); reads skipped with LVC_ERANGE count nothing) counts each I op that meets all of:
 *   - the op before it, ignoring P ops and ops of length 0, is a match op (M, =, X); an I op after S, D or N, or at the
 *     start of the read, is not counted.  [EXT] htslib also reports insertions on deletion anchors; this rule does not;
 *   - the anchor -- the last base of that match op, at reference position p -- has quality >= min_base_quality (the
 *     pileup entry on which htslib reports indel > 0 and which pysam's base-quality filter keeps).
 * Key: (p, len, seq) when len <= 32 and every inserted base is A/C/G/T with quality >= min_base_quality (seq = 2-bit
 * codes A,C,G,T = 0..3, base k in bits 2k); otherwise (p, 0, 0), an "unresolved" insertion that counts towards the
 * insertions at p but is never emitted.  The counts are the same for every batch form (byte or 2-bit qualities, 4-bit
 * bases or 2-bit base codes): the rule never needs a base below the threshold.  Mate-overlap rewrites need no special
 * case: the qualities are read as the batch carries them.  Once per batch, in a device hash table.
 * lvc_enable_insertions  only on empty tables (after lvc_create or lvc_reset, before any push or import), else
 *                        LVC_EINVAL; refused with peer tables attached (and lvc_peer_attach is refused on a handle that
 *                        counts).  The table has at least 2 * max_keys slots (a power of two); it holds at least
 *                        max_keys keys, and a key is dropped only when every slot holds another.  lvc_reset clears it and
 *                        keeps counting on.  Timer 4 of lvc_get_timing times the counting kernel.
 * Both queries fail with LVC_EINVAL after lvc_import_plane / _dels / _covdiff / _first or lvc_reduce_tables (the tables
 * then hold counts the insertion table does not cover) until lvc_reset, and with LVC_ENOMEM (the message gives the number)
 * if keys were dropped.  *n_out > cap: call again with a larger buffer.
 * lvc_copy_insertions    every key with its count (depth = 0), sorted by (pos, len, seq).
 * lvc_insertion_calls    for each anchor p in [p0, p1) (p1 < 0: the whole contig; arguments checked as lvc_consensus):
 *                        d = the consensus depth of p, I = the sum of every count at p (unresolved included),
 *                        none = d - I.  The resolved key s is emitted (count, depth = d) iff the consensus letter of p for
 *                        (min_depth, threshold) is neither 'N' nor '-', count(s) > none, count(s) > the unresolved count,
 *                        count(s) > every other resolved count at p, and count(s) / d >= threshold (fp64 division).
 *                        Every comparison is strict: a tie emits nothing.  Sorted by pos (at most one per position).
 * The splice: a called sequence follows the letter of its anchor. */
typedef struct lvc_insertion {
    int32_t pos;        /* anchor: 0-based position of the reference base the insertion follows */
    uint32_t len;       /* inserted bases; 0 = unresolved */
    uint64_t seq;       /* 2-bit codes A,C,G,T = 0..3, base k in bits 2k */
    uint32_t count;     /* reads carrying the key */
    uint32_t depth;     /* lvc_insertion_calls: consensus depth at pos; lvc_copy_insertions: 0 */
} lvc_insertion;        /* 24 bytes */
int lvc_enable_insertions(lvc_handle* h, uint32_t max_keys);
int lvc_copy_insertions(lvc_handle* h, lvc_insertion* out, uint32_t cap, uint32_t* n_out);
int lvc_insertion_calls(lvc_handle* h, int64_t p0, int64_t p1, uint64_t min_depth, double threshold,
                        lvc_insertion* out, uint32_t cap, uint32_t* n_out);

/* ---- table access: self.memory (live_variant_caller.py:31), checkpoints (:40-52), tests, NCCL ----
 * A "plane" holds, for one (allele group, quality) key, uint32 counts [G][4].  key = group<<8 | q;
 * group 0 = A,C,G,T (slots 0..3); groups 1..3 hold the other BAM nibble codes:
 * {=,M,R,S} {V,W,Y,H} {K,D,B,N}.  dels[G] counts deletion/ref-skip entries that passed the
 * base-quality rule (totalDepth = sum of all counts + dels).  covdiff[G+1] is a difference array of
 * read coverage (a site exists in `memory` iff its prefix sum is > 0).  first[group][G][4] is the
 * ordinal of the first read that deposited (pos, allele), 0xFFFFFFFF if never. */
int lvc_num_planes(lvc_handle* h);
int lvc_plane_keys(lvc_handle* h, uint16_t* keys_out /*[lvc_num_planes]*/);
int lvc_ensure_plane(lvc_handle* h, uint16_t key);
int lvc_copy_plane(lvc_handle* h, uint16_t key, uint32_t* dst /*[G*4]*/);
int lvc_import_plane(lvc_handle* h, uint16_t key, const uint32_t* src /*[G*4]*/, int accumulate);
int lvc_copy_dels(lvc_handle* h, uint32_t* dst /*[G]*/);
int lvc_import_dels(lvc_handle* h, const uint32_t* src, int accumulate);
int lvc_copy_covdiff(lvc_handle* h, int32_t* dst /*[G+1]*/);
int lvc_import_covdiff(lvc_handle* h, const int32_t* src, int accumulate);
int lvc_copy_first(lvc_handle* h, int group, uint32_t* dst /*[G*4]*/); /* LVC_EINVAL if group unallocated */
int lvc_import_first(lvc_handle* h, int group, const uint32_t* src);
uint64_t lvc_ordinal(lvc_handle* h);              /* reads consumed so far (next first-seen ordinal) */
int lvc_set_ordinal(lvc_handle* h, uint64_t ordinal);
/* raw device pointers for zero-copy collectives (torch.distributed all_reduce over NCCL) */
void* lvc_plane_devptr(lvc_handle* h, uint16_t key);
void* lvc_dels_devptr(lvc_handle* h);
void* lvc_covdiff_devptr(lvc_handle* h);
void* lvc_first_devptr(lvc_handle* h, int group);

/* ---- multi-GPU: the one exchange step of the read-chunk sharding (SURVEY 8e) -----------------------------
 * The reference is a single process (client_server/vc_queue.py:99); its state update is a commutative integer
 * add per (position, allele, quality) and a min per first-seen rank, so ranks that deposited different chunks
 * of one coordinate-sorted batch combine with ONE collective.  lvc_reduce_tables issues it as one NCCL group on
 * the handle's stream, on the device tables themselves: integer SUM for the count planes / deletion counts /
 * coverage, unsigned MIN for the first-seen ordinals; the set of (allele group, quality) planes is agreed first.
 *   LVC_REDUCE_ALL     all-reduce: every rank holds the complete tables afterwards.
 *   LVC_REDUCE_SCATTER reduce-scatter in place onto position slices (lvc_position_slice): rank r keeps the complete
 *                      history of its slice only, the rest of its tables is cleared, and its genotype range is set to
 *                      the slice.  Ranks must then keep owning the same slice for the lifetime of the handle.
 * `nccl_comm` is an ncclComm_t (from lvc_nccl_comm_create, or the caller's own).  NCCL is bound at run time
 * (dlopen of libnccl.so.2); without it these return LVC_EIO.  The max_depth keep mask must be computed over the
 * WHOLE batch before it is split, and each rank sets lvc_set_ordinal(base + first read index of its chunk). */
#define LVC_REDUCE_ALL 0
#define LVC_REDUCE_SCATTER 1
int lvc_nccl_unique_id(uint8_t id_out[128]);                       /* rank 0; ship the 128 bytes to the other ranks */
int lvc_nccl_comm_create(void** comm_out, int device, int n_ranks, int rank, const uint8_t id[128]);
void lvc_nccl_comm_destroy(void* comm);
int lvc_position_slice(const lvc_handle* h, int n_ranks, int rank, int64_t* p0, int64_t* p1);
int lvc_reduce_tables(lvc_handle* h, void* nccl_comm, int n_ranks, int rank, int mode);
uint64_t lvc_last_exchange_bytes(lvc_handle* h);    /* bytes this rank fed into the last lvc_reduce_tables */

/* ---- multi-GPU without an exchange step: position ownership over NVLink peer memory -------------------------------
 * Rank r owns the columns lvc_position_slice(h, n, r) and its tables hold the history of those columns only.  After
 * lvc_peer_attach the deposit kernels reduce a base of column c directly into the tables of the rank that OWNS c,
 * through that rank's peer-mapped pointers (CUDA IPC, one process per GPU): a RED that crosses NVLink / NVSwitch and is
 * resolved in the owner's L2.  A rank's chunk of a coordinate-sorted batch lies almost entirely inside its own slice,
 * so only the reads that straddle a slice border pay the link.  Per batch: every rank calls lvc_set_ordinal(base +
 * first read index of its chunk) and lvc_push_batch*, then lvc_stream_barrier (all ranks' reductions are complete),
 * then lvc_genotype* (its own slice; the range is set by lvc_peer_attach), then lvc_stream_barrier again before the
 * next batch (nobody deposits into tables a slower rank is still genotyping).
 *   lvc_peer_export  writes the handle's IPC blob (call with blob = NULL to get the size).  The (allele group, quality)
 *                    plane set must be identical on all ranks (ensure the union first); a plane added later makes
 *                    lvc_push_batch* fail with LVC_EINVAL until a new export / attach round.
 *   lvc_peer_attach  blobs[r] / lens[r] = rank r's blob (blobs[rank] is ignored).  At most 8 ranks.  Short-read batches
 *                    run the generation-5 tiled kernel, everything else the any-record kernels.
 *   lvc_peer_detach  closes the peer mappings (also done by lvc_destroy).
 * [EXT] the reference is one process (client_server/vc_queue.py:99); this replaces its in-order dict update
 * (live_variant_caller.py:77-103) for one sample spread over several GPUs. */
int lvc_peer_export(lvc_handle* h, void* blob, size_t cap, size_t* len);
int lvc_peer_attach(lvc_handle* h, int rank, int n_ranks, const void* const* blobs, const size_t* lens);
int lvc_peer_detach(lvc_handle* h);
int lvc_stream_barrier(lvc_handle* h, void* nccl_comm);

/* ---- introspection ---------------------------------------------------------------------------- */
/* number of kernels this library has launched on the handle since creation (bench gpu_launches) */
uint64_t lvc_launch_count(lvc_handle* h);
/* cumulative payload bytes (seq4 + qual) lvc_push_batch actually copied host->device: the bytes of reads the
 * host admission dropped are never shipped */
uint64_t lvc_h2d_payload_bytes(lvc_handle* h);
/* per-kernel device time from CUDA events recorded on the handle's stream around every launch while
 * timing is on.  which: 0 = tiled deposit, 1 = general deposit, 2 = genotype, 3 = consensus, 4 = insertion counts (only
 * on a handle that counts them, lvc_enable_insertions).  Reading resets. */
int lvc_set_timing(lvc_handle* h, int on);
int lvc_get_timing(lvc_handle* h, int which, double* ms_total, uint64_t* n_launches);
int lvc_version(void);

#ifdef __cplusplus
}
#endif
#endif /* LVC_H_ */

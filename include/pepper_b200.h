/*
 * pepper_b200.h — C-ABI of libpepper_b200.so (sm_100a).
 *
 * Drop-in boundary for PEPPER's pileup-summary encoders and recurrent-network
 * inference (SURVEY.md §8b).  Every entry point replaces one Python-visible
 * pybind class/method or predict function of the reference; the reference
 * interface it replaces is cited as file:line (relative to the reference repo).
 *
 * Conventions
 *   - plain pointers + sizes, no torch / STL types;
 *   - "d_" pointers are DEVICE pointers, "h_" pointers are HOST pointers;
 *   - every function returns 0 on success, <0 on error (pb_last_error() gives
 *     the message); nothing ever calls exit() (the reference does:
 *     region_summary.cpp:151, bam_handler.cpp:9-26);
 *   - caller owns every buffer; opaque handles own only library scratch;
 *   - `stream` is a cudaStream_t passed as void* (0 = legacy default stream);
 *   - there is NO CPU fallback: without a CUDA device every compute entry
 *     point fails with PB_ERR_CUDA.
 *
 * Read records ("post-get_reads" reads, i.e. what BAM_handler::get_reads
 * returns: pepper_variant/modules/cpp/bam_handler.cpp:115-451, struct
 * type_read pepper_variant/modules/cpp/read.h:60) are passed as a
 * structure-of-arrays in BAM-native packing:
 *   seq   4-bit codes "=ACMGRSVTWYHKDBN", two bases per byte, high nibble
 *         first; base i of read r is nibble (seq_off[r] + i)
 *   qual  one byte per base at qual[seq_off[r] + i]
 *   cigar uint32 (len << 4 | op), op in {0 M,1 I,2 D,3 N,4 S,5 H,6 P,7 =,8 X}
 */
#ifndef PEPPER_B200_H
#define PEPPER_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PB_OK             0
#define PB_ERR_ARG       -1
#define PB_ERR_CUDA      -2
#define PB_ERR_CAPACITY  -3   /* output capacity too small; *n_out holds the need */
#define PB_ERR_STATE     -4

#define PB_VARIANT_WINDOW   33   /* CANDIDATE_WINDOW_SIZE + 1, Options.py:9   */
#define PB_VARIANT_FEATURES 26   /* IMAGE_HEIGHT, Options.py:7                */
#define PB_ALLELE_STRIDE    64   /* key "1T" / "2ACG.." / "3ACG.." <=61 + NUL */
#define PB_POLISH_FEATURES  10   /* summary_generator.cpp:16-32               */
#define PB_POLISH_SEQ_LEN   1000 /* pepper Options.py SEQ_LENGTH              */
#define PB_POLISH_CLASSES   5

/* SoA read batch (host or device pointers depending on the entry point). */
typedef struct {
    int64_t         n_reads;
    const int64_t  *pos;        /* [n_reads]   0-based reference position of the first cigar op */
    const int64_t  *seq_off;    /* [n_reads+1] base (nibble) offset of each read in seq / byte offset in qual */
    const int64_t  *cigar_off;  /* [n_reads+1] */
    const uint8_t  *flags;      /* [n_reads]   bit0 = is_reverse (type_read_flags, read.h:13) */
    const uint8_t  *mapq;       /* [n_reads]   mapping_quality (read.h:69) */
    const uint8_t  *seq;        /* [(seq_off[n]+1)/2] */
    const uint8_t  *qual;       /* [seq_off[n]] */
    const uint32_t *cigar;      /* [cigar_off[n]] */
} pb_reads_t;

/* One encoder region == one RegionalSummaryGenerator / SummaryGenerator object. */
typedef struct {
    int64_t ref_start;      /* ctor region_start (inclusive)                     */
    int64_t ref_end;        /* ctor region_end   (inclusive)                     */
    int64_t cand_start;     /* generate_summary candidate_region_start (variant) */
    int64_t cand_end;       /* generate_summary candidate_region_end   (variant) */
    int64_t ref_off;        /* offset of this region's reference string in `ref` */
    int64_t ref_len;        /* its length (normally ref_end-ref_start+1)         */
    int64_t read_begin;     /* reads [read_begin, read_end) belong to the region */
    int64_t read_end;
} pb_region_t;

/* generate_summary arguments, region_summary.h:191-206 (same order). */
typedef struct {
    double  min_snp_baseq;
    double  min_indel_baseq;
    double  snp_freq_threshold;
    double  insert_freq_threshold;
    double  delete_freq_threshold;
    double  min_coverage_threshold;
    double  snp_candidate_freq_threshold;
    double  indel_candidate_freq_threshold;
    double  candidate_support_threshold;
    int32_t skip_indels;
    int32_t reserved;
} pb_variant_params_t;

const char *pb_last_error(void);
int  pb_version(void);
/* number of CUDA devices visible (0 on a CPU box); never fails */
int  pb_device_count(void);
/* synchronous device -> host copy of a library-owned device buffer (read-backs of device views, tests) */
int  pb_memcpy_to_host(void *h_dst, const void *d_src, int64_t bytes);

/* ------------------------------------------------------------------------
 * Region read fetch + trim (SURVEY 8a row a2).  Replaces the per-record body of
 *   BAM_handler::get_reads(chromosome, start, stop, include_supplementary,
 *                          min_mapq, min_baseq)
 * (pepper/modules/src/dataio/bam_handler.cpp:115-451; the pepper_variant copy
 * pepper_variant/modules/cpp/bam_handler.cpp is identical) for a BATCH of
 * region queries against one coordinate-sorted contig held in device memory:
 *   - which records a query returns: htslib 1.9 iterator overlap rule
 *     (pos < stop && pos + max(reference length of the CIGAR, n_cigar ? 0 : 1) > start)
 *   - flag / MAPQ filters                                   bam_handler.cpp:139-150
 *   - the CIGAR-walk trim to [start, stop] (inclusive stop, anchor on the first
 *     match base, I/S/D/N only after the anchor)             bam_handler.cpp:176-303
 *   - reads left without bases are dropped                  bam_handler.cpp:432
 * The trimmed reads come out as a pb_reads_t in HBM that feeds the encoders
 * directly.  Record fields the encoders never read (query_name, bad_indicies,
 * hp_tag; min_baseq only feeds bad_indicies) are not materialised.
 * ---------------------------------------------------------------------- */
typedef struct {
    int64_t         n_records;
    const int64_t  *pos;        /* [n]   bam1_core_t.pos, non-decreasing               */
    const int64_t  *seq_off;    /* [n+1] base (nibble) offsets into seq / byte offsets into qual */
    const int64_t  *cigar_off;  /* [n+1]                                               */
    const uint16_t *flag;       /* [n]   bam1_core_t.flag (SAM FLAG bits)              */
    const uint8_t  *mapq;       /* [n]   bam1_core_t.qual                              */
    const uint8_t  *seq;        /* 4-bit codes, bam_get_seq                            */
    const uint8_t  *qual;       /* bam_get_qual                                        */
    const uint32_t *cigar;      /* len<<4|op, bam_get_cigar                            */
} pb_records_t;

typedef struct { int64_t start, stop; } pb_interval_t;          /* get_reads(chrom, start, stop) */
typedef struct { int32_t include_supplementary, min_mapq, min_baseq, reserved; } pb_get_reads_options_t;

typedef struct pb_read_trimmer pb_read_trimmer_t;
int pb_read_trimmer_create(pb_read_trimmer_t **out, int device);
int pb_read_trimmer_destroy(pb_read_trimmer_t *t);

/* Phase 1: evaluate every query.  h_reads_per_interval[i] = len(get_reads(...)) of query i. */
int pb_get_reads_plan_device(pb_read_trimmer_t *t, const pb_records_t *d_records /* struct on host, pointers on device */,
                             const pb_interval_t *h_intervals, int64_t n_intervals,
                             const pb_get_reads_options_t *opt, int64_t *h_reads_per_interval, void *stream);
/* Phase 2: write the trimmed reads of the planned queries.  h_select (optional) lists, per query, indices into that
 * query's result in get_reads order - the reference's reservoir sample (AlignmentSummarizer.py:113-125) - NULL = all.
 * d_reads_out is a view of buffers owned by the trimmer (valid until its next plan/destroy); reads of query i are
 * [h_read_begin[i], h_read_end[i]).                                                                              */
int pb_get_reads_emit_device(pb_read_trimmer_t *t, const int64_t *h_select_off /* [n+1] or NULL */,
                             const int32_t *h_select, pb_reads_t *d_reads_out,
                             int64_t *h_read_begin, int64_t *h_read_end, void *stream);
/* sizes[3] = n_reads, n_bases, n_cigar of the last emit; fetch copies it to host arrays sized accordingly */
int pb_get_reads_sizes(pb_read_trimmer_t *t, int64_t *sizes);
int pb_get_reads_fetch(pb_read_trimmer_t *t, int64_t *pos, int64_t *seq_off, int64_t *cigar_off, uint8_t *flags,
                       uint8_t *mapq, uint8_t *seq, uint8_t *qual, uint32_t *cigar, void *stream);
/* Host-buffer convenience: upload the records, plan.  (emit/fetch as above) */
int pb_get_reads_plan_host(pb_read_trimmer_t *t, const pb_records_t *h_records,
                           const pb_interval_t *h_intervals, int64_t n_intervals,
                           const pb_get_reads_options_t *opt, int64_t *h_reads_per_interval, void *stream);

/* ------------------------------------------------------------------------
 * Read -> reference realignment (SURVEY 8f row f1).  Replaces
 *   ReadAligner(ref_start, ref_end, ref_seq).align_reads_to_reference(reads)
 * (pepper/modules/src/local_reassembly/simple_aligner.cpp:66-106 on top of the
 * vendored SSW library ssw.c / ssw_cpp.cpp; pybind_api.h ReadAligner) for every
 * region of a batch: region i is [ref_start, ...] with its reference string
 * ref[ref_off : ref_off + ref_len] (= get_reference_sequence(chrom,
 * region_start, region_end + ALIGNMENT_SAFE_BASES), AlignmentSummarizer.py:
 * 164-170) and its reads [read_begin, read_end).  Each read is aligned against
 * the reference suffix that starts at its own position; with sw_score > 1 it
 * takes the SSW CIGAR ('=' / 'X' -> M tuples, S, I, D) and
 * pos = pos + ref_begin, otherwise it is returned unchanged.  Sequences and
 * qualities are never modified: the output pb_reads_t aliases the input's
 * seq_off / flags / mapq / seq / qual and owns new pos / cigar_off / cigar
 * (valid until the realigner's next call).  The reference implementation drops
 * reads that start before the region start; here that is PB_ERR_ARG (fetch the
 * reads with get_reads(start = region start), as the reference's caller does).
 * ---------------------------------------------------------------------- */
typedef struct pb_realigner pb_realigner_t;
int pb_realigner_create(pb_realigner_t **out, int device);
int pb_realigner_destroy(pb_realigner_t *t);
int pb_realign_device(pb_realigner_t *t, const pb_reads_t *d_reads,
                      const pb_region_t *d_regions, const pb_region_t *h_regions, int64_t n_regions,
                      const char *d_ref, int64_t ref_bytes, pb_reads_t *d_out, void *stream);
/* host buffers in, new pos [n] / cigar_off [n+1] / cigar out; PB_ERR_CAPACITY (with *n_cigar set) if cigar_capacity is short */
int pb_realign_host(pb_realigner_t *t, const pb_reads_t *h_reads, const pb_region_t *h_regions, int64_t n_regions,
                    const char *h_ref, int64_t ref_bytes, int64_t *h_pos, int64_t *h_cigar_off, uint32_t *h_cigar,
                    int64_t cigar_capacity, int64_t *n_cigar, void *stream);
int pb_realign_stats(pb_realigner_t *t, int64_t *n_aligned, int64_t *n_realigned, float *ms_sw, float *ms_cigar);

/* ------------------------------------------------------------------------
 * File readers under BAM_handler / FASTA_handler (SURVEY 8f row f4).  Host code
 * written from the SAM/BAM/BAI and faidx specifications (the reference gets
 * these from htslib 1.9: sam_open / sam_index_load / sam_hdr_read /
 * sam_itr_queryi / sam_itr_next, bam_handler.cpp:6-28,127-135; fai_load /
 * faidx_fetch_seq, fasta_handler.cpp:7-50).
 * ---------------------------------------------------------------------- */
typedef struct pb_bam pb_bam_t;
/* BAM_handler(path): opens path and path + ".bai" (or name.bai); n_threads <= 0 = all cores (BGZF inflate pool) */
int pb_bam_open(pb_bam_t **out, const char *path, int n_threads);
int pb_bam_close(pb_bam_t *b);
int pb_bam_n_contigs(pb_bam_t *b);                              /* get_chromosome_sequence_names (bam_handler.cpp:103) */
const char *pb_bam_contig_name(pb_bam_t *b, int tid);
int64_t pb_bam_contig_length(pb_bam_t *b, int tid);            /* ..._with_length (:88)                              */
int pb_bam_contig_id(pb_bam_t *b, const char *name);           /* bam_name2id                                         */
const char *pb_bam_header_text(pb_bam_t *b, int64_t *len);     /* get_sample_names parses @RG SM from it (:30-56)     */
/* every record sam_itr_queryi(idx, tid, beg, end) / sam_itr_next would return, in file order, as a pb_records_t in
 * reader-owned host memory (page-locked when a GPU is present; valid until the next fetch / close)                   */
int pb_bam_fetch(pb_bam_t *b, int tid, int64_t beg, int64_t end, pb_records_t *h_view);
int pb_bam_io_stats(pb_bam_t *b, int64_t *compressed_bytes, int64_t *inflated_bytes);

/* GPU fetch (VERDICT r1 item 5): the same records as pb_bam_fetch, but only the COMPRESSED BGZF blocks are copied to the
 * device; DEFLATE inflate (one warp per BGZF block), the record-chain walk (one thread per BAI linear-index window start), the
 * record parse and the scatter into the structure-of-arrays are kernels.  `view` receives DEVICE pointers owned by the
 * reader (valid until its next pb_bam_fetch_device) — the input of pb_get_reads_plan_device.  Replaces bgzf_read / bam_read1 /
 * sam_itr_next under BAM_handler::get_reads (bam_handler.cpp:115-135).                                                        */
int pb_bam_fetch_device(pb_bam_t *bam, int tid, int64_t beg, int64_t end, int device, pb_records_t *view, void *stream);
/* device time (ms) of the last pb_bam_fetch_device: [H2D + inflate, record chains + parse, scatter] */
int pb_bam_fetch_device_timings(pb_bam_t *bam, float *ms3);
/* Hybrid inflate of pb_bam_fetch_device: `share` (0..1) of the BGZF blocks — runs of 16 consecutive blocks — is inflated by the
 * reader's host thread pool (zlib) WHILE the kernel inflates the rest; the host runs reach the same device buffer through a copy
 * stream, and the record kernels wait for both.  Default 0 (everything on the GPU); the environment variable
 * PB_INFLATE_HOST_SHARE overrides the default.  The records are identical for every share. */
int pb_bam_set_host_share(pb_bam_t *bam, double share);
/* blocks inflated by the host pool / by the kernel over all pb_bam_fetch_device calls of this reader */
int pb_bam_inflate_split(pb_bam_t *bam, int64_t *host_blocks, int64_t *device_blocks);
/* diagnostics: raw DEFLATE streams inflated by the GPU kernel (outputs concatenated; h_status[i] != 0 = rejected stream) */
int pb_inflate_blocks_host(const uint8_t *h_comp, int64_t comp_bytes, const int64_t *h_in_off, const int32_t *h_in_len,
                           const int32_t *h_out_len, int64_t n_blocks, uint8_t *h_out, int32_t *h_status, void *stream);

typedef struct pb_fasta pb_fasta_t;
int pb_fasta_open(pb_fasta_t **out, const char *path);          /* FASTA_handler(path): path + ".fai" must exist       */
int pb_fasta_close(pb_fasta_t *f);
int pb_fasta_n_contigs(pb_fasta_t *f);                          /* get_chromosome_names (fasta_handler.cpp:19)         */
const char *pb_fasta_contig_name(pb_fasta_t *f, int i);
int64_t pb_fasta_contig_length(pb_fasta_t *f, const char *name);/* get_chromosome_sequence_length (:52)                */
/* get_reference_sequence(region, start, stop) (:31-50) = faidx_fetch_seq(.., start, stop - 1, &len); *len = -2 when the
 * contig is absent; PB_ERR_CAPACITY (with *len set) when cap is too small                                            */
int pb_fasta_fetch(pb_fasta_t *f, const char *name, int64_t start, int64_t stop, char *out, int64_t cap, int64_t *len);

/* ------------------------------------------------------------------------
 * Variant encoder.  Replaces
 *   RegionalSummaryGenerator(contig, region_start, region_end, ref_seq)
 *     .generate_max_insert_summary(reads)
 *     .generate_summary(reads, ...16 args...) -> list[CandidateImageSummary]
 * (pepper_variant/modules/cpp/pybind_api.h:55-62, region_summary.cpp:568)
 * for a BATCH of regions in one call.
 * ---------------------------------------------------------------------- */
typedef struct pb_variant_encoder pb_variant_encoder_t;

int pb_variant_encoder_create(pb_variant_encoder_t **out, int device);
int pb_variant_encoder_destroy(pb_variant_encoder_t *enc);
/* keep the snp/insert/delete count vectors of the next encode calls for
 * pb_variant_encoder_debug_region (off by default: 12 B/position of traffic) */
int pb_variant_encoder_set_debug(pb_variant_encoder_t *enc, int on);

/* Host-buffer entry point (the one the PEPPER_VARIANT mirror classes call):
 * copies reads/ref to the device, encodes, copies the candidates back.
 * Outputs are ordered by region, then position, then allele key (std::set
 * order, region_summary.cpp:669-670).
 *   h_images     int8  [cap][33][26]   (DataStore.py:68 stores int8)
 *   h_positions  int64 [cap]
 *   h_depths     uint8 [cap]           min(coverage,125)  region_summary.cpp:682
 *   h_freqs      uint8 [cap]           min(allele_depth,125)          :862
 *   h_keys       char  [cap][64]       NUL-terminated allele key
 *   h_region_of  int32 [cap]
 *   h_n_per_region int64 [n_regions]   (may be NULL)
 *   n_out        total number of candidates (also set on PB_ERR_CAPACITY)   */
int pb_variant_encode_host(pb_variant_encoder_t *enc,
                           const pb_reads_t *h_reads,
                           const pb_region_t *h_regions, int64_t n_regions,
                           const char *h_ref, int64_t ref_bytes,
                           const pb_variant_params_t *params,
                           int64_t capacity,
                           int8_t *h_images, int64_t *h_positions,
                           uint8_t *h_depths, uint8_t *h_freqs,
                           char *h_keys, int32_t *h_region_of,
                           int64_t *h_n_per_region, int64_t *n_out,
                           void *stream);

/* Device-resident entry point: reads/regions/ref already in HBM, outputs stay
 * in HBM (feeds pb_variant_net_forward without a host round trip).           */
int pb_variant_encode_device(pb_variant_encoder_t *enc,
                             const pb_reads_t *d_reads,       /* struct on host, pointers on device */
                             const pb_region_t *d_regions, int64_t n_regions,
                             const pb_region_t *h_regions,    /* host copy of the same table */
                             const char *d_ref, int64_t ref_bytes,
                             const pb_variant_params_t *params,
                             int64_t capacity,
                             int8_t *d_images, int64_t *d_positions,
                             uint8_t *d_depths, uint8_t *d_freqs,
                             char *d_keys, int32_t *d_region_of,
                             int64_t *d_n_per_region, int64_t *n_out,
                             void *stream);

/* Debug/parity read-back of the intermediate of the LAST encode call:
 * the [L+1][26] count matrix after the clamp of region_summary.cpp:648-653
 * (int32, col 0 = reference code) and the coverage/snp/insert/delete vectors
 * (region_summary.cpp:586-589) of region `region`.                          */
int pb_variant_encoder_debug_region(pb_variant_encoder_t *enc, int64_t region,
                                    int32_t *h_matrix, int32_t *h_coverage,
                                    int32_t *h_snp, int32_t *h_ins, int32_t *h_del);

/* per-kernel device time (ms) of the last encode call, measured with CUDA
 * events on the call's stream: [prefix, count, sites, alleles, windows]      */
int pb_variant_encoder_timings(pb_variant_encoder_t *enc, float *ms5);
/* kernels launched by the last encode call */
int pb_variant_encoder_launches(pb_variant_encoder_t *enc, int64_t *n_launches);

/* ------------------------------------------------------------------------
 * Polish encoder.  Replaces
 *   SummaryGenerator(ref_seq, chrom, ref_start, ref_end)
 *     .generate_summary(reads, start, end);  .image  .genomic_pos
 * (pepper/modules/headers/pybind_api.h:18-25, summary_generator.cpp:370)
 * for a batch of regions.
 *   h_image   uint8 [cap_cols][10]
 *   h_pos     int64 [cap_cols]     genomic_pos.first
 *   h_idx     int32 [cap_cols]     genomic_pos.second
 *   h_col_off int64 [n_regions+1]  columns of region r are [off[r], off[r+1])
 * ---------------------------------------------------------------------- */
typedef struct pb_polish_encoder pb_polish_encoder_t;
int pb_polish_encoder_create(pb_polish_encoder_t **out, int device);
int pb_polish_encoder_destroy(pb_polish_encoder_t *enc);
int pb_polish_encode_host(pb_polish_encoder_t *enc,
                          const pb_reads_t *h_reads,
                          const pb_region_t *h_regions, int64_t n_regions,
                          int64_t capacity_cols,
                          uint8_t *h_image, int64_t *h_pos, int32_t *h_idx,
                          int64_t *h_col_off, int64_t *n_cols_out, void *stream);
int pb_polish_encode_device(pb_polish_encoder_t *enc,
                            const pb_reads_t *d_reads,
                            const pb_region_t *d_regions, int64_t n_regions,
                            const pb_region_t *h_regions,
                            int64_t capacity_cols,
                            uint8_t *d_image, int64_t *d_pos, int32_t *d_idx,
                            int64_t *d_col_off, int64_t *n_cols_out, void *stream);
int pb_polish_encoder_timings(pb_polish_encoder_t *enc, float *ms3);

/* ------------------------------------------------------------------------
 * Variant network (bi-LSTM x2 + 5x(Linear+SELU) + Linear + softmax).
 * Replaces TransducerGRU.forward, pepper_variant/modules/python/models/
 * simple_model.py:48-82, as driven by predict_distributed_gpu.py:58-70.
 * Weights are passed as the state_dict tensors (fp32, PyTorch layout) in the
 * order of pb_variant_net_param_names(); the handle keeps a packed copy.
 * ---------------------------------------------------------------------- */
typedef struct pb_variant_net pb_variant_net_t;
#define PB_VARIANT_NET_N_PARAMS 28
const char *pb_variant_net_param_name(int i);   /* state_dict key */
int64_t     pb_variant_net_param_numel(int i);
int pb_variant_net_create(pb_variant_net_t **out, int device,
                          const float *const *h_params /* [28] host fp32 */);
int pb_variant_net_destroy(pb_variant_net_t *net);
/* d_images int8 [n][33][26] on device -> d_probs float [n][3] on device.
 * d_hidden_dbg (optional, may be NULL): float [n][33][512] decoder output.   */
int pb_variant_net_forward_device(pb_variant_net_t *net, const int8_t *d_images,
                                  int64_t n, float *d_probs, float *d_hidden_dbg,
                                  void *stream);
/* The prediction record a rank-0 writer needs for one candidate (SURVEY 8e: 3 x f32 probabilities, i32 position, i32 region
 * id, u8 depth, u8 frequency, 62 B allele key = 84 B): what pepper_variant DataStorePredict.write_prediction stores per
 * candidate (DataStorePredict.py:49-66).  Written by the head kernel (512 -> 3 + softmax) itself when a record sink is
 * given, so that the buffer an NCCL all-gather sends needs no staging copy.                                               */
typedef struct {
    float   probs[3];
    int32_t position;          /* contig position (int32 as in the reference's HDF5 'contig_pos' dataset) */
    int32_t region;            /* global region (interval) id */
    uint8_t depth, freq;
    char    key[62];           /* NUL padded allele key, <= 61 characters */
} pb_pred_record_t;
/* the per-candidate columns the encoder produced for the candidates of one forward call (device pointers) */
typedef struct {
    const int64_t *positions;
    const int32_t *region_of;
    const uint8_t *depths, *freqs;
    const char    *keys;       /* [n][PB_ALLELE_STRIDE] */
} pb_candidate_columns_t;
/* as pb_variant_net_forward_device; additionally writes d_records[i] for every candidate (cols / d_records may be NULL) */
int pb_variant_net_forward_records_device(pb_variant_net_t *net, const int8_t *d_images, int64_t n, float *d_probs,
                                          const pb_candidate_columns_t *cols, pb_pred_record_t *d_records, void *stream);
int pb_variant_net_forward_host(pb_variant_net_t *net, const int8_t *h_images,
                                int64_t n, float *h_probs, float *h_hidden_dbg,
                                void *stream);
/* GEMM path: 0 = fp32 FFMA (reference-exact ordering), 1 = tcgen05 with the fp16 hi/lo operand split (2-3 products per GEMM,
 * see pb_variant_net_set_lo_mask; default)                                                                                       */
int pb_variant_net_set_mode(pb_variant_net_t *net, int mode);
int pb_variant_net_launches(pb_variant_net_t *net, int64_t *n_launches);

/* ------------------------------------------------------------------------
 * Polish network (bi-GRU x2 + Linear(256->5)), 19-window sliding loop with
 * carried hidden state, softmax accumulate, argmax, phred.  Replaces
 * TransducerGRU.forward (pepper/modules/python/models/simple_model.py:27-42)
 * and the loop of predict_distributed_cpu.py:50-90 / _gpu.py:63-105.
 * ---------------------------------------------------------------------- */
typedef struct pb_polish_net pb_polish_net_t;
#define PB_POLISH_NET_N_PARAMS 18
const char *pb_polish_net_param_name(int i);
int64_t     pb_polish_net_param_numel(int i);
int pb_polish_net_create(pb_polish_net_t **out, int device,
                         const float *const *h_params /* [18] host fp32 */);
int pb_polish_net_destroy(pb_polish_net_t *net);
/* d_images uint8 [n][1000][10] -> d_bases uint8 [n][1000], d_phred uint8 [n][1000]
 * d_hidden_dbg (optional): float [19][n][2][128] hidden state returned by each window
 * d_acc_dbg (optional): float [n][1000][5] accumulated softmax                */
int pb_polish_net_forward_device(pb_polish_net_t *net, const uint8_t *d_images,
                                 int64_t n, uint8_t *d_bases, uint8_t *d_phred,
                                 float *d_hidden_dbg, float *d_acc_dbg, void *stream);
int pb_polish_net_forward_host(pb_polish_net_t *net, const uint8_t *h_images,
                               int64_t n, uint8_t *h_bases, uint8_t *h_phred,
                               float *h_hidden_dbg, float *h_acc_dbg, void *stream);
int pb_polish_net_launches(pb_polish_net_t *net, int64_t *n_launches);
/* Products per GEMM on the tcgen05 path: every GEMM runs as a_hi*w_hi + a_hi*w_lo (+ a_lo*w_hi); the mask says which GEMMs keep the
 * third product.  variant bits: 0 encoder h-part, 1 decoder x-part, 2 decoder h-part, 3 linear_1, 4 linear_2-5 (default 0x1a: the
 * two recurrent GEMMs, which pass the parity gate with two products, run with two; the decoder's x-part and the head keep three);
 * polish bits: 0 encoder h, 1 decoder x, 2 decoder h (default 0x7: every polish GEMM needs three).  0x1f / 0x7 = three products
 * everywhere; DESIGN.md section 4 holds the measured error of every choice.                                                     */
int pb_variant_net_set_lo_mask(pb_variant_net_t *net, int mask);
int pb_polish_net_set_lo_mask(pb_polish_net_t *net, int mask);
/* Variant network, same bits as lo_mask: a set bit runs that GEMM's correction products (a_hi*w_lo, and a_lo*w_hi where lo_mask
 * keeps it) as e4m3 tensor-core MMAs (kind::f8f6f4) next to the fp16 main product; default 0x1f.  0 = the fp16 split everywhere. */
int pb_variant_net_set_f8_mask(pb_variant_net_t *net, int mask);
/* 0 = fp32 FFMA GEMMs, 1 = tcgen05 GEMMs with the fp16 hi/lo operand split x3 (fp32-equivalent, default) */
int pb_polish_net_set_mode(pb_polish_net_t *net, int mode);

/* diagnostics: C[M][N] = A[M][K] W[N][K]^T + bias through the tcgen05 kernel (N % 256 == 0, K % 32 == 0) */
int pb_test_tc_gemm(int M, int N, int K, const float *h_A, const float *h_W, const float *h_bias, float *h_out);
/* the same GEMM with the variant network's operand images: weights scaled by 2^(12-E) (max|w| = f * 2^E, f in [0.5, 1)) with
 * e4m3 copies; lo = 1 runs a_lo*w_hi, f8 = 1 runs the corrections in e4m3 */
int pb_test_tc_gemm_f8(int M, int N, int K, const float *h_A, const float *h_W, const float *h_bias, float *h_out, int lo, int f8);

/* ------------------------------------------------------------------------
 * Fused make_images + run_inference for the variant path: what
 * `pepper_variant call_variant` does between the BAM and the prediction HDF5
 * (CallVariant.py:12 steps 1+2) without the image HDF5 round trip.
 * Host entry point: H2D of the reads, encode, network, D2H of the candidate
 * records and probabilities (h_images may be NULL to skip the image copy).
 * Device entry point: everything already / still in HBM.
 * ---------------------------------------------------------------------- */
int pb_variant_call_host(pb_variant_encoder_t *enc, pb_variant_net_t *net,
                         const pb_reads_t *h_reads,
                         const pb_region_t *h_regions, int64_t n_regions,
                         const char *h_ref, int64_t ref_bytes,
                         const pb_variant_params_t *params, int64_t capacity,
                         int8_t *h_images /* optional */, int64_t *h_positions,
                         uint8_t *h_depths, uint8_t *h_freqs, char *h_keys,
                         int32_t *h_region_of, float *h_probs /* [cap][3] */,
                         int64_t *n_out, void *stream);
int pb_variant_call_device(pb_variant_encoder_t *enc, pb_variant_net_t *net,
                           const pb_reads_t *d_reads,
                           const pb_region_t *d_regions, int64_t n_regions,
                           const pb_region_t *h_regions,
                           const char *d_ref, int64_t ref_bytes,
                           const pb_variant_params_t *params, int64_t capacity,
                           int8_t *d_images, int64_t *d_positions,
                           uint8_t *d_depths, uint8_t *d_freqs, char *d_keys,
                           int32_t *d_region_of, float *d_probs,
                           int64_t *n_out, void *stream);

/* ------------------------------------------------------------------------
 * Streaming session over region GROUPS (the unit a multi-GPU job hands out; replaces the reference's file-chunk round
 * robin, pepper_variant/modules/python/RunInference.py:70-72,104-106 + ImageGenerationUI.py:307-316).  Candidates
 * accumulate in library-owned device buffers; the network runs over whole 9,472-candidate chunks as they fill, the tail
 * at _end.  Typical loop:  begin; stage(g0); { run(last?); stage(next); sync; }*; end; fetch / use d_records.
 *   d_records  optional device buffer [capacity] (e.g. this rank's slice of an all-gather buffer): the network's head
 *              kernel writes one pb_pred_record_t per candidate straight into it
 *   region_id0 global id of the group's first region (added to region_of / record.region)
 * pb_variant_stream_run returns while the network is still running; PB_ERR_CAPACITY ends the session (*n_total = need so far).
 * ---------------------------------------------------------------------- */
int pb_variant_stream_begin(pb_variant_encoder_t *enc, pb_variant_net_t *net, const pb_variant_params_t *params,
                            int64_t capacity, pb_pred_record_t *d_records, void *stream);
int pb_variant_stream_stage_host(pb_variant_encoder_t *enc, const pb_reads_t *h_reads, const pb_region_t *h_regions,
                                 int64_t g0, int64_t g1, const char *h_ref, int32_t region_id0);
int pb_variant_stream_stage_device(pb_variant_encoder_t *enc, const pb_reads_t *d_reads, const pb_region_t *h_regions,
                                   int64_t g0, int64_t g1, const char *d_ref, int32_t region_id0);
int pb_variant_stream_run(pb_variant_encoder_t *enc, pb_variant_net_t *net, int flush, int64_t *n_total);
int pb_variant_stream_sync(pb_variant_encoder_t *enc);
int pb_variant_stream_end(pb_variant_encoder_t *enc, pb_variant_net_t *net, int64_t *n_out);
/* encoder device time per phase (ms: cigar prefix, pileup count, site index, alleles, windows) and kernel launches
 * [encoder, network] of the last session, summed over its groups */
int pb_variant_stream_stats(pb_variant_encoder_t *enc, float *ms5, int64_t *launches2, int64_t *groups);
int pb_variant_stream_columns(pb_variant_encoder_t *enc, pb_candidate_columns_t *cols, const float **d_probs, const int8_t **d_images);
int pb_variant_stream_fetch(pb_variant_encoder_t *enc, int64_t n, int8_t *h_images, int64_t *h_positions, uint8_t *h_depths,
                            uint8_t *h_freqs, char *h_keys, int32_t *h_region_of, float *h_probs, void *stream);

/* Fused make_images + call_consensus for the polish path (polish.py:14 steps
 * 1+2): encode, chunk into 1000-column images with 50 overlap
 * (AlignmentSummarizer.py:19-56) on the device, run the network.
 *   h_bases / h_phred  uint8 [cap_images][1000]
 *   h_position int64 [cap_images][1000], h_index int32 [cap_images][1000]  ((-1,-1) padding)
 *   h_image_region int32 [cap_images], h_chunk_id int32 [cap_images]        */
int pb_polish_call_host(pb_polish_encoder_t *enc, pb_polish_net_t *net,
                        const pb_reads_t *h_reads,
                        const pb_region_t *h_regions, int64_t n_regions,
                        int64_t capacity_images,
                        uint8_t *h_bases, uint8_t *h_phred,
                        int64_t *h_position, int32_t *h_index,
                        int32_t *h_image_region, int32_t *h_chunk_id,
                        int64_t *n_images_out, void *stream);
int pb_polish_call_device(pb_polish_encoder_t *enc, pb_polish_net_t *net,
                          const pb_reads_t *d_reads,
                          const pb_region_t *d_regions, int64_t n_regions,
                          const pb_region_t *h_regions,
                          int64_t capacity_images,
                          uint8_t *d_bases, uint8_t *d_phred,
                          int64_t *d_position, int32_t *d_index,
                          int32_t *d_image_region, int32_t *d_chunk_id,
                          int64_t *n_images_out, void *stream);
/* device time (ms) of the last pb_*_call_*: [encode, network] */
int pb_variant_call_timings(pb_variant_encoder_t *enc, float *ms2);
int pb_polish_call_timings(pb_polish_encoder_t *enc, float *ms2);

/* ------------------------------------------------------------------------
 * Polish stitch (SURVEY 8f row f3).  Replaces small_chunk_stitch +
 * create_consensus_sequence (pepper/modules/python/Stitch.py:36-128) for one
 * contig: drops the padding columns (-1,-1), the first 200 positions of every
 * region that does not start at 0, the 50-column chunk overlap (the chunk whose
 * id sorts later AS A STRING wins, Stitch.py:50), label 0, and concatenates
 * A/C/G/T in (position, index) order.  Images must be ordered by region (regions
 * sorted by start, tiled with the reference's 2 x 100 overlap) then chunk id —
 * the order pb_polish_call_* produces.
 *   out  char [capacity] (not NUL terminated); n_out = consensus length
 * ---------------------------------------------------------------------- */
int pb_polish_stitch_device(const uint8_t *d_bases, const int64_t *d_position,
                            const int32_t *d_index, const int32_t *d_image_region,
                            const int32_t *d_chunk_id, const int64_t *d_region_starts,
                            int64_t n_images, char *d_out, int64_t capacity,
                            int64_t *n_out, void *stream);
int pb_polish_stitch_host(const uint8_t *h_bases, const int64_t *h_position,
                          const int32_t *h_index, const int32_t *h_image_region,
                          const int32_t *h_chunk_id, const int64_t *h_region_starts,
                          int64_t n_regions, int64_t n_images, char *h_out,
                          int64_t capacity, int64_t *n_out, void *stream);

/* ------------------------------------------------------------------------
 * Candidate selection (SURVEY 8f row f2).  Replaces the per-candidate logic of
 * small_chunk_stitch, pepper_variant/modules/python/CandidateFinder.py:356-530:
 * homopolymer context of the +-10 bp reference window (:393-406), genotype =
 * argmax of the prediction (:411), Margin list = SNP alleles with a non-ref
 * genotype (:427-449), DeepVariant list by the p-value / frequency thresholds
 * per allele type in and outside repeats (:460-519).  One allele per record
 * (what the encoder emits).
 *   flags  uint8 [n]: bit0 Margin record, bit1 DeepVariant record, bit2 in repeat,
 *                     bit3 delete ref/alt swap (:497-505), bit4 reference base valid
 *   genotype uint8 [n]: 0 hom-ref, 1 het, 2 hom-alt
 * ---------------------------------------------------------------------- */
typedef struct {
    double snp_p_value, insert_p_value, delete_p_value;
    double snp_p_value_in_lc, insert_p_value_in_lc, delete_p_value_in_lc;
    double report_snp_above_freq, report_indel_above_freq;
} pb_candidate_options_t;
int pb_variant_find_candidates_device(const int64_t *d_positions, const int32_t *d_region_of,
                                      const uint8_t *d_depths, const uint8_t *d_freqs,
                                      const char *d_keys, const float *d_probs, int64_t n,
                                      const pb_region_t *d_regions, const char *d_ref,
                                      const pb_candidate_options_t *opt,
                                      uint8_t *d_flags, uint8_t *d_genotype, void *stream);
int pb_variant_find_candidates_host(const int64_t *h_positions, const int32_t *h_region_of,
                                    const uint8_t *h_depths, const uint8_t *h_freqs,
                                    const char *h_keys, const float *h_probs, int64_t n,
                                    const pb_region_t *h_regions, int64_t n_regions,
                                    const char *h_ref, int64_t ref_bytes,
                                    const pb_candidate_options_t *opt,
                                    uint8_t *h_flags, uint8_t *h_genotype, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* PEPPER_B200_H */

/*
 * mega_reads_b200.h -- C ABI of the B200-native create_mega_reads / jf_aligner hot path.
 *
 * The reference (alekseyzimin/PacBio) has no FFI; the path lives behind three C++ class seams
 * inside one process.  Each entry point below replaces one of those seams (cited per function,
 * paths relative to the reference root) so that the host driver stays a transliteration of
 * src_jf_aligner/create_mega_reads.cc:25-167.
 *
 * Conventions
 *  - plain C types only; host buffers belong to the caller, all device memory to the library;
 *  - every call returns 0 on success, a negative MR_E* code otherwise; mr_last_error() gives text;
 *  - a context is bound to ONE GPU and is thread-compatible (one driver thread per context), the
 *    analogue of the reference's shared-const-index + per-thread-scratch model
 *    (coarse_aligner.hpp:126-148, overlap_graph.hpp:161-172);
 *  - there is NO CPU fallback: without a CUDA device mr_context_create fails with MR_ENODEV.
 */
#ifndef MEGA_READS_B200_H
#define MEGA_READS_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MR_OK        0
#define MR_EINVAL   -1   /* bad argument / unsupported option value          */
#define MR_ENODEV   -2   /* no usable CUDA device                            */
#define MR_ECUDA    -3   /* CUDA runtime error (text in mr_last_error)       */
#define MR_ENOMEM   -4   /* host or device allocation failed                 */
#define MR_ELIMIT   -5   /* input exceeds an implementation limit            */

typedef struct mr_context mr_context;
typedef struct mr_index   mr_index;
typedef struct mr_result  mr_result;

/* ---- context --------------------------------------------------------------------------------- */
int         mr_context_create(int device, mr_context** out);
void        mr_context_destroy(mr_context* ctx);
const char* mr_last_error(const mr_context* ctx);      /* ctx may be NULL: last creation error */
int         mr_context_device(const mr_context* ctx);
/* device seconds spent in each phase of the last mr_align_batch/mr_index_create call, for
 * profiling; names follow the reference's global_timer phases where they exist
 * (src_psa/mer_sa_imp.hpp:211-252, create_mega_reads.cc:130,154).  Returns number of entries. */
int         mr_context_timers(const mr_context* ctx, const char** names, double* seconds, int cap);
/* number of kernels this library launched on ctx since creation (bench.py's gpu_launches) */
uint64_t    mr_context_launches(const mr_context* ctx);

/* page-lock / unlock a caller-owned host buffer so that mr_align_batch's H2D copy runs at full PCIe
 * speed (optional; the reference has no counterpart) */
int         mr_host_pin(mr_context* ctx, const void* p, size_t bytes);
int         mr_host_unpin(mr_context* ctx, const void* p);

/* ---- index: replaces superread_parse() -> sequence_psa (superread_parser.hpp:212-224),
 *      i.e. sequence_psa::append_fasta (superread_parser.cc:12-46) output +
 *      PSA::PSA -> SA::create_mt (psa.hpp:130-140, mer_sa_imp.hpp:197-267).
 *  text2bit  : concatenated super-read bases, 2 bits each, A0 C1 G2 T3, base i at bits
 *              2*(i%32) of word i/32 (compact_dna layout), ceil(n/32) words
 *  sr_start  : nseq+1 offsets into the text (m_offsets[].sequence)
 *  unitig_ids/unitig_off : CSR of each super-read's forward unitig path, (id<<1)|ori, ori 1 = 'R'
 *              (super_read_name::u_id_ori, super_read_name.hpp:16-37); may be NULL when no -l/-u
 *  unitig_len: length of every k-unitig (misc.cc:11-37), may be NULL
 *  psa_min,k : --psa-min and -m.  Requires psa_min < k <= 31.                                    */
int  mr_index_create(mr_context* ctx, const uint64_t* text2bit, uint64_t n,
                     const uint64_t* sr_start, uint32_t nseq,
                     const uint32_t* unitig_ids, const uint64_t* unitig_off,
                     const int32_t* unitig_len, uint32_t n_unitigs,
                     uint32_t psa_min, uint32_t k, mr_index** out);
void mr_index_destroy(mr_index* idx);
uint64_t mr_index_sa_size(const mr_index* idx);                 /* n - psa_min + 1 (of the first part) */
/* A text of 2^32 bases or more (the reference switches to its 48-bit suffix array there,
 * src_psa/48bit_index.hpp) is indexed as several PARTS of fewer than 2^32 bases, cut at super-read
 * boundaries; mr_align_batch gives the same rows either way.  The calls that speak in ranks of one
 * suffix array (mr_index_export_*, mr_lookup_batch*) return MR_ELIMIT for an index of several
 * parts.
 * Environment: MR_INDEX_PART_BASES=<n> lowers the part limit (tests). */
uint32_t mr_index_parts(const mr_index* idx);
/* bytes of the tables a k-mer lookup reads at random (prefix counts + tails, all parts): what has to
 * stay in the L2 for lookups to hit there; bench.py sizes its random-access ceiling probe with it */
uint64_t mr_index_table_bytes(const mr_index* idx);
/* parity taps: suffix-array values in SA order and the 4^psa_min + 1 prefix counts
 * (mer_sa_imp.hpp:317-330), widened to 64 bit */
int  mr_index_export_sa(mr_index* idx, uint64_t* sa_out);
int  mr_index_export_counts(mr_index* idx, uint64_t* counts_out);

/* ---- index files.  The reference rebuilds the suffix array in every process
 *  (superread_parser.hpp:212-224 is called from main, create_mega_reads.cc:131), while the pipeline
 *  runs the tool many times over the same super-reads (array jobs,
 *  mega_reads_assemble_cluster2.sh:358-448).  mr_index_save writes a built index to one file,
 *  mr_index_load brings it back on any device without sorting.  mr_inputs_checksum hashes the
 *  arguments of mr_index_create on the host; mr_index_checksum returns the hash an index was built
 *  from (also after a load), so a caller can tell whether a file matches the inputs it parsed.    */
int      mr_index_save(mr_index* idx, const char* path);
int      mr_index_load(mr_context* ctx, const char* path, mr_index** out);
uint64_t mr_index_checksum(const mr_index* idx);
/* reads only the header of an index file: the checksum of the inputs it was built from, so that a
 * caller can skip a file made for other inputs without uploading gigabytes first.  mr_index_load
 * itself verifies a hash of the arrays against the header and fails on a corrupt or stale body. */
int      mr_index_peek_checksum(const char* path, uint64_t* checksum);
uint64_t mr_inputs_checksum(const uint64_t* text2bit, uint64_t n, const uint64_t* sr_start, uint32_t nseq,
                            const uint32_t* unitig_ids, const uint64_t* unitig_off, const int32_t* unitig_len,
                            uint32_t n_unitigs, uint32_t psa_min, uint32_t k);

/* ---- k-mer lookup: replaces PSA::search (psa.hpp:150-153 -> mer_sa_imp.hpp:369-479).
 *  mers[i] holds a k-mer as an integer, first base most significant.  index_out/nb_out get the
 *  rank of the first matching SA entry and the number of matches (index 0 when nb is 0).
 *  Host-pointer version copies in and out; the _device version takes device pointers and only
 *  enqueues the kernel on the context's stream (use mr_context_sync to wait).                  */
int  mr_lookup_batch(mr_index* idx, const uint64_t* mers, uint64_t q, uint64_t* index_out, uint64_t* nb_out);
int  mr_lookup_batch_device(mr_index* idx, const uint64_t* d_mers, uint64_t q, uint64_t* d_index_out, uint64_t* d_nb_out);
int  mr_context_sync(mr_context* ctx);
/* the CUDA stream (cudaStream_t) the context launches on, for callers that time with events */
void* mr_context_stream(mr_context* ctx);

/* ---- alignment parameters: the numeric arguments of coarse_aligner's constructor
 *      (coarse_aligner.hpp:55-72 as called from create_mega_reads.cc:140-146) and of
 *      overlap_graph (overlap_graph.hpp:90-95 as called from create_mega_reads.cc:155).        */
typedef struct mr_params {
  double   stretch_factor;     /* --stretch-factor   1.3   */
  double   stretch_constant;   /* --stretch-constant 10    */
  double   stretch_cap;        /* --stretch-cap      10000 */
  uint32_t window_size;        /* --window-size      1 (only 1 is implemented)        */
  int32_t  forward;            /* create_mega_reads: always 1; jf_aligner: -f          */
  int32_t  max_match;          /* --max-match                                         */
  int32_t  max_count;          /* --max-count, 0 means unlimited                      */
  double   matching_mers;      /* -M / 100                                            */
  double   matching_bases;     /* -B / 100                                            */
  uint32_t unitigs_k;          /* -k (0: no unitig information, kmers_info stay empty) */
  double   overlap_play;       /* -O 1.3   */
  double   errors;             /* -e 3.0   */
  int32_t  bases;              /* -b       */
  int32_t  run_graph;          /* 0: stop after coords (jf_aligner), 1: also run the overlap graph */
  uint32_t fine_mer;           /* -F: mer length of the fine pass (fine_aligner.cc:38-51), 0 = none; < -m    */
} mr_params;
void mr_params_default(mr_params* p);

/* ---- one batch of reads: replaces, for every read of the batch,
 *      coarse_aligner::thread::align_sequence_max + coords()  (coarse_aligner.cc:42-72,81-141,
 *      pb_aligner.cc:11-143, lis_align.hpp:139-204), the coords sort of
 *      create_mega_reads.cc:69-77 and overlap_graph::thread::{reset,traverse}
 *      (overlap_graph.hpp:177-196, overlap_graph.cc:7-59).
 *  bases      : reads concatenated, one ASCII character per base, as parsed (any case, non-ACGT
 *               breaks k-mers exactly like jf_aligner.hpp:41-52)
 *  read_start : nreads+1 offsets into bases
 *  The result object owns pinned host arrays, valid until mr_result_free.                       */
int  mr_align_batch(mr_context* ctx, mr_index* idx, const mr_params* p,
                    const char* bases, const uint64_t* read_start, uint32_t nreads, mr_result** out);
/* same, but with the batch already resident in device memory (bench.py's device-resident timing) */
int  mr_align_batch_device(mr_context* ctx, mr_index* idx, const mr_params* p,
                           const char* d_bases, const uint64_t* d_read_start, const uint64_t* h_read_start,
                           uint32_t nreads, mr_result** out);
/* ---- packed reads.  The library keeps a batch on the device 2-bit packed (the layout of the reference's
 *  compact_dna, src_psa/compact_dna.hpp:102-136: base g at bits 2 (g % 32) of word g / 32, A0 C1 G2 T3,
 *  non-ACGT as 0) next to a mask with bit g % 64 of word g / 64 set where the character was not one of
 *  ACGTacgt (those break k-mers, jf_aligner.hpp:41-52): 0.375 bytes per base over PCIe instead of one.
 *  mr_pack_reads fills caller-owned arrays of mr_packed_code_words(n) / mr_packed_mask_words(n) words (the
 *  counts include the padding the kernels may read); the _packed entry points take such arrays.  The
 *  entry points that take characters pack them on the device.                                        */
uint64_t mr_packed_code_words(uint64_t nbases);
uint64_t mr_packed_mask_words(uint64_t nbases);
int  mr_pack_reads(const char* bases, uint64_t nbases, uint64_t* codes, uint64_t* nmask);
/* the same for mask words [first_word, first_word + n_words) only (and their code words): lets several host
 * threads pack disjoint ranges of one batch */
int  mr_pack_reads_range(const char* bases, uint64_t nbases, uint64_t first_word, uint64_t n_words, uint64_t* codes, uint64_t* nmask);
int  mr_align_batch_packed(mr_context* ctx, mr_index* idx, const mr_params* p, const uint64_t* codes, const uint64_t* nmask,
                           const uint64_t* read_start, uint32_t nreads, mr_result** out);
int  mr_align_batch_device_packed(mr_context* ctx, mr_index* idx, const mr_params* p, const uint64_t* d_codes, const uint64_t* d_nmask,
                                  const uint64_t* d_read_start, const uint64_t* h_read_start, uint32_t nreads, mr_result** out);
void mr_result_free(mr_result* r);

/* Structure-of-arrays view of a result.  Coords of read r are rows
 * [read_coords[r], read_coords[r+1]) and are ordered by (rs, re, ql, super-read index): the
 * reference's (unstable) order of create_mega_reads.cc:74 with ties broken canonically.
 * One row == one align_pb::coords_info (pb_aligner.hpp:103-175) and, when run_graph, one
 * node_info (overlap_graph.hpp:9-40); node links (lstart, lprev) are row offsets inside the read. */
typedef struct mr_result_view {
  uint32_t nreads;
  uint64_t ncoords;
  const uint64_t* read_coords;      /* nreads + 1 */
  const int32_t  *rs, *re, *qs, *qe, *nb_mers;
  const uint32_t *pb_cons, *sr_cons, *pb_cover, *sr_cover;
  const uint32_t *ql;               /* super-read length */
  const uint32_t *sr;               /* super-read index (qfrag) */
  const uint8_t  *rn;               /* reverse match */
  const uint8_t  *use_bwd;          /* name_u == &qfrag->bwd */
  const double   *stretch, *offset, *avg_err;
  const uint64_t *info_off;         /* per row: start of its entries in kmers_info / bases_info */
  const uint32_t *info_len;         /* per row: 2*#unitigs-1, or 0 when empty (no -l/-u, bad name, error path) */
  const int32_t  *kmers_info, *bases_info;
  /* overlap graph (NULL unless run_graph) */
  const uint8_t  *start_node, *end_node;
  const int32_t  *lstart, *lprev, *lpath, *lunitigs;
  const int32_t  *component;        /* union-find root, row offset inside the read */
  /* work counters of the batch, for roofline arithmetic */
  uint64_t n_kmers_looked_up;       /* k-mers that reached the suffix-array lookup (x2 strands) */
  uint64_t n_tail_entries;          /* entries of the tail array those lookups scanned (buckets not held inline in their slot) */
  uint64_t n_hits;                  /* hits expanded into (read, super-read) lists */
  uint64_t n_groups;                /* (read, super-read) pairs chained */
  uint64_t n_lists;                 /* read positions whose k-mer kept a non-empty list after --max-count */
  uint64_t n_buckets;               /* non-empty prefix buckets those lookups went on to scan (second random access) */
} mr_result_view;
int  mr_result_get(const mr_result* r, mr_result_view* view);

/* ---- staged batches: mr_align_batch copies its input and only then starts the kernels.  A caller
 *  that knows the next batch can have it copied while the current one is aligned: mr_stage_batch
 *  starts the copy on the context's copy stream and returns (at once when the buffers are pinned,
 *  mr_host_pin; it may be called from another host thread than the aligning one),
 *  mr_align_staged waits for the copy on the device, aligns, and releases the staged batch
 *  (mr_staged_free does that for a batch that is never aligned).  `bases` must stay valid until
 *  mr_align_staged / mr_staged_free returns.                                                     */
typedef struct mr_staged mr_staged;
int  mr_stage_batch(mr_context* ctx, const char* bases, const uint64_t* read_start, uint32_t nreads, mr_staged** out);
int  mr_stage_batch_packed(mr_context* ctx, const uint64_t* codes, const uint64_t* nmask, const uint64_t* read_start, uint32_t nreads,
                           mr_staged** out);
int  mr_align_staged(mr_context* ctx, mr_index* idx, const mr_params* p, mr_staged* staged, mr_result** out);
void mr_staged_free(mr_staged* staged);

/* ---- overlap graph over rows the caller already has: replaces overlap_graph::thread::reset +
 *  traverse (overlap_graph.hpp:177-198, overlap_graph.cc:7-59) as longest_path_overlap_graph2.cc:46-49
 *  calls them on the rows of a coords file.  `rows` is an mr_result_view in HOST memory whose
 *  coords columns and kmers_info / bases_info are filled (graph pointers ignored); rows->sr[i]
 *  indexes the caller's table of unitig paths (path_ids[path_off[s] .. path_off[s + 1]) as
 *  id << 1 | (orientation == 'R'), rows->use_bwd[i] reads it reversed and flipped).  Rows keep
 *  their order; the result echoes them and adds the node arrays.                                   */
int  mr_graph_batch(mr_context* ctx, const mr_params* params, const mr_result_view* rows, const uint32_t* read_len,
                    const uint32_t* path_ids, const uint64_t* path_off, uint32_t npaths,
                    const int32_t* unitig_len, uint32_t n_unitigs, mr_result** out);

/* ---- mega-read records: replaces overlap_graph::thread's printing side, i.e. term_node_per_comp, trim_match,
 *  tile_greedy / tile_maximal and print_mega_reads (overlap_graph.cc:61-299, overlap_graph.hpp:198-262), on the
 *  device, over the rows and graph nodes a batch left there.
 *
 *  mr_unitigs: the k-unitig sequences of the -u file (misc.cc:11-37), uploaded once: `seq` holds every sequence
 *  back to back as in the file, off[i] .. off[i + 1] is unitig i (n + 1 offsets).  Read-only once created; any
 *  context of the same device may use it.                                                                     */
typedef struct mr_unitigs mr_unitigs;
int  mr_unitigs_create(mr_context* ctx, const char* seq, const uint64_t* off, uint32_t n, mr_unitigs** out);
void mr_unitigs_destroy(mr_unitigs* u);

/* the options of the printing side (create_mega_reads_cmdline.yaggo): -k, -O, -d, -L, -T, --trim */
typedef struct mr_records_params {
  uint32_t unitigs_k;          /* -k */
  double   overlap_play;       /* -O 1.3 */
  double   density;            /* -d 0.029 */
  double   min_length;         /* -L 100 */
  int32_t  tiling;             /* -T: 0 none, 1 greedy, 2 maximal, 3 weighted */
  int32_t  trim;               /* --trim: 0 none, non-zero trims as `match` does */
} mr_records_params;

/* The create_mega_reads text records of the reads of `r`, in read order: for every read with at least one
 *  mega-read a ">name" line, then one line per mega-read (numbers, unitig path, super-read length and, with
 *  `u`, the spliced sequence).  `r` must be the latest result of `ctx` and carry the overlap graph
 *  (mr_align_* with run_graph, or mr_graph_batch): the rows are read where that batch left them on the
 *  device; any other result gives MR_EINVAL.  u == NULL: no sequence column (-l).  names: the reads' names
 *  back to back, name_off[r] .. name_off[r + 1] for read r (nreads + 1 offsets).
 *  MR_EINVAL also for the inputs the reference rejects while printing: a unitig id of a super-read name
 *  that the -u file does not have, and a component root outside the read's rows (mr_last_error says which).
 *  The text lives in pinned host memory owned by the returned object: mr_text_get gives its bytes, valid
 *  until mr_text_free.                                                                                  */
typedef struct mr_text mr_text;
int  mr_records(mr_context* ctx, const mr_result* r, const mr_records_params* p, const mr_unitigs* u,
                const char* names, const uint64_t* name_off, mr_text** out);
int  mr_text_get(const mr_text* t, const char** bytes, uint64_t* size);
void mr_text_free(mr_text* t);

/* ---- jf_aligner coords records: replaces print_coords (jf_aligner.cc:41-70) on the device, over the rows a batch
 *  left there.
 *
 *  mr_sr_names: what a coords line names a super-read by (frag_info's fwd.name / bwd.name, super_reads::row_name):
 *  the FASTA header after '>' as it was read (names[name_off[s] .. name_off[s + 1])), and the unitig path as
 *  mr_index_create takes it (path_ids[path_off[s] .. path_off[s + 1]), (id << 1) | (ori == 'R'); path_ids may be
 *  NULL when every path is empty).  A backward row of a super-read with a path prints that path reversed, F and R
 *  swapped, as "<id><F|R>" joined by '_'; any other row prints the header.  The tools build it from their
 *  super-reads, whatever -l / -u say; for rows of mr_graph_batch it is built from the caller's path table that
 *  their `sr` indexes.  Read-only once created; any context of the same device may use it.                    */
typedef struct mr_sr_names mr_sr_names;
int  mr_sr_names_create(mr_context* ctx, const char* names, const uint64_t* name_off, const uint32_t* path_ids,
                        const uint64_t* path_off, uint32_t nseq, mr_sr_names** out);
void mr_sr_names_destroy(mr_sr_names* s);

/* the options of jf_aligner's printing: --compact (non-zero: the compact format, the tool's default) and -0 */
typedef struct mr_coords_params {
  int32_t compact;             /* ">N name" before a read's N rows; 0: the read's name before every row  */
  int32_t zero_match;          /* -0: a read without rows still gets its ">0 name" line (compact format) */
} mr_coords_params;

/* The jf_aligner coords text of the reads of `r`, in read order: one line per row ("Rstart Rend Qstart Qend Nmers
 *  Rcons Qcons Rcover Qcover Rlen Qlen Stretch Offset Err" as "%d %d %d %d %d %u %u %u %u %llu %u %g %g %g ", the
 *  super-read's name, then " kmers:bases" per kmers_info entry), under a ">N name" line per read (compact) or
 *  after the read's name and a blank (not compact).  The column header line is the caller's.  `r` must be the
 *  latest result of `ctx`, from any entry point (mr_align_*, with or without run_graph, -F, --max-match,
 *  --window-size, or mr_graph_batch); any other result gives MR_EINVAL, as do names made on another device and a
 *  row whose super-read index is not below the names' nseq (mr_last_error says which).  names / name_off: the
 *  reads' names as mr_records takes them.  The text comes back as mr_records' does (mr_text_get / mr_text_free). */
int  mr_coords_records(mr_context* ctx, const mr_result* r, const mr_coords_params* p, const mr_sr_names* s,
                       const char* names, const uint64_t* name_off, mr_text** out);

/* parity tap: per-(read, super-read) hit lists and chains of the last batch, in the layout of
 * tests/oracle_lib.py (groups[g] = {read, sr, n_fwd, n_bwd, lis_fwd, lis_bwd}); only filled when
 * mr_context_keep_taps(ctx, 1) was called before the batch.  With max_match the lists are the
 * ones the discard loop ends with: the hits of the chains it removed are gone from n_fwd / n_bwd
 * and the offsets, and each chain is the list's latest one (the chain that failed the filters, or
 * empty), as indices into that shortened list.  Not available with a fine pass (MR_EINVAL). */
int  mr_context_keep_taps(mr_context* ctx, int on);
int  mr_result_taps(const mr_result* r, uint64_t* ngroups, const int64_t** groups,
                    uint64_t* noffsets, const int32_t** offsets, uint64_t* nlis, const uint32_t** lis);

/* self test: the least-squares kernel divides by the running count through a shared reciprocal
 * (3 FP64 instructions); this sweeps `samples` random operands over counts 1..max_n and reports how
 * many quotients differ, bit for bit, from the IEEE division the reference executes (must be 0). */
int  mr_selftest_division(mr_context* ctx, uint64_t samples, uint64_t seed, uint32_t max_n, uint64_t* mismatches);

/* measurement aid (SURVEY.md 8d): the random 32-byte-sector ceiling of this GPU, the denominator the
 * k-mer lookup is judged against.  `loads` independent 16-byte loads (8 in flight per thread, no
 * pointer chasing) at uniformly random 16-byte-aligned places of a table of table_bytes; reports
 * sectors x 32 B per second of the best of three launches, in GB/s.  A table much larger than the
 * 126 MB L2 gives the HBM figure, a table of the index's size what the L2 adds. */
int  mr_selftest_random_gather(mr_context* ctx, uint64_t table_bytes, uint64_t loads, double* sector_gbs);

#ifdef __cplusplus
}
#endif
#endif /* MEGA_READS_B200_H */

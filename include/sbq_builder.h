/* sbq_builder.h - C ABI of the host class-table builder (part of libsbq.so).
 *
 * Host side of the hot path: turns one locus (collapsed fragments + candidate isoforms) into the
 * fragment-class x isoform CSR that sbq_submit() takes. It is a from-scratch implementation of what
 * the reference does in the LocusContext constructor (include/estimate.hpp:61-109):
 *
 *   a11  Contig::Contig(const PairedHit&)            src/contig.cpp:216-267   -> sbq_pair_features
 *   a12  IRanges<GenomicFeature,false>::disjoint()   include/interval.hpp:150-223
 *   a8   Isoform (segments contained in the isoform) include/isoform.h:40-86, src/contig.cpp:615-634
 *   a9   Contig::is_compatible(read, isoform)        src/contig.cpp:547-599
 *   a3   LocusContext::assign_exon_bin / overlap_exons / set_maps
 *                                                    src/estimate.cpp:115-198, include/estimate.hpp:29-52
 *   a7   ExonBin::read_count (float sum over the _frags set)   include/isoform.h:285-296
 *   a6   ExonBin::bin_under_iso / effective_len      include/isoform.h:363-516
 *   a13  InsertSize::emp_dist_pdf / normal_pdf       src/read.cpp:274-297, include/common.h:92-99
 *   a4/a5 set_theory_bin_weight / set_bin_weight_without_frag_dist    src/estimate.cpp:201-247
 *
 * Integer outputs (segments, class coordinates and ids, isoform->class map, counts) are bit-exact
 * with the reference; alpha is fp64 accumulated in increasing fragment length like the reference
 * (which is built with -Ofast, so its own last ulp is not defined).
 *
 * Feature codes follow the reference's Match_t (include/contig.h:27-32).
 */
#ifndef SBQ_BUILDER_H_
#define SBQ_BUILDER_H_
#include <stdint.h>
#include "sbq.h"

#ifdef __cplusplus
extern "C" {
#endif

enum { SBQ_FEAT_MATCH = 0, SBQ_FEAT_INTRON = 1, SBQ_FEAT_GAP = 2 };
/* CIGAR operation codes, BAM numbering (include/read.hpp:24-34) */
enum { SBQ_CIG_MATCH = 0, SBQ_CIG_INS = 1, SBQ_CIG_DEL = 2, SBQ_CIG_REF_SKIP = 3, SBQ_CIG_SOFT_CLIP = 4 };

/* InsertSize (include/read.hpp:176-192): empirical histogram with normal fallback, or plain normal. */
typedef struct {
   int32_t use_emp;          /* InsertSize::_use_emp                                              */
   int32_t start_offset;     /* smallest observed fragment length (_start_offset)                 */
   int32_t end_offset;       /* largest observed fragment length (_end_offset)                    */
   const double* emp_dist;   /* end_offset - start_offset + 1 counts (_emp_dist)                  */
   int32_t total_reads;      /* _total_reads                                                      */
   double mean, sd;          /* _mean, _sd                                                        */
} sbq_insert_model;

/* One locus as LocusContext sees it. Feature lists are flattened: element k of list i lives at
 * ptr[i] .. ptr[i+1]-1 of the off/len/code arrays. Transcripts alternate MATCH / INTRON features
 * (Contig 6-argument ctor, include/contig.h:164-181). Hits are Contig(PairedHit) feature lists in
 * HitCluster::uniq_hits() order (an empty list = ref_id -1 = dropped, include/estimate.hpp:71-79). */
typedef struct {
   int32_t n_iso;
   const int32_t* iso_feat_ptr;
   const uint32_t* iso_feat_off;
   const uint32_t* iso_feat_len;
   const uint8_t* iso_feat_code;
   int32_t n_hit;
   const int32_t* hit_feat_ptr;
   const uint32_t* hit_feat_off;
   const uint32_t* hit_feat_len;
   const uint8_t* hit_feat_code;
   const double* hit_mass;       /* PairedHit::collapse_mass()                                   */
   const int32_t* hit_ref_id;    /* Contig::ref_id(); may be NULL (all 0)                         */
   int32_t read_len;             /* ReadTable::read_len_mode()                                   */
   int32_t long_read;            /* long_read_sample: alpha = 1 / L_t (src/estimate.cpp:236-247) */
   int32_t defer_weights;        /* 1: do not evaluate the alpha sums on the host; emit per-entry descriptors instead */
                                 /*    (sbq_table_weight_desc) and let sbq_submit_deferred compute alpha on the GPU   */
} sbq_locus_input;

typedef struct sbq_table sbq_table;

/* Build the class table of one locus. Thread-safe (no shared state). */
int  sbq_build_locus(const sbq_locus_input* in, const sbq_insert_model* model, sbq_table** out);
void sbq_table_free(sbq_table*);

/* CSR view for sbq_submit(); pointers stay valid until sbq_table_free. */
int  sbq_table_locus(const sbq_table*, sbq_locus* out);

/* Sizes: segments S, classes R, isoforms T, non-zeros, total class coordinates, hits dropped. */
typedef struct { int32_t n_seg, n_class, n_iso; int64_t nnz; int64_t n_coord; int32_t n_dropped_hits; } sbq_table_dims;
int  sbq_table_get_dims(const sbq_table*, sbq_table_dims* out);

/* Copy-out accessors (caller-sized by sbq_table_dims; any pointer may be NULL):
 *   seg_left/right[S]                      disjoint exon segments (_exon_segs)
 *   iso_seg_ptr[T+1], iso_seg[...]         segment indices contained in each isoform (Isoform::_exon_segs)
 *   class_coord_ptr[R+1], class_coord[...] segment indices of each class (ExonBin::_coords), first-seen order
 *   class_count[R]                         (int)ExonBin::read_count()
 *   class_mass[R]                          ExonBin::read_count() as float
 *   class_nfrag[R]                         ExonBin::_frags.size()                                    */
int  sbq_table_segments(const sbq_table*, uint32_t* seg_left, uint32_t* seg_right);
int  sbq_table_iso_segments(const sbq_table*, int32_t* iso_seg_ptr, int32_t* iso_seg);
int  sbq_table_classes(const sbq_table*, int32_t* class_coord_ptr, int32_t* class_coord, int32_t* class_count,
                       float* class_mass, int32_t* class_nfrag);

/* Deferred weights: what the GPU needs to evaluate alpha_ct = sum_fl pdf(fl) * effective_len(fl) / (L_t - fl + 1)
 * (LocusContext::set_theory_bin_weight, src/estimate.cpp:201-234) for every CSR entry of the table. Entry k's segment
 * lengths are pool[seg_ptr[k] .. seg_ptr[k] + n_seg[k]); seg_ptr[k] = -1 means alpha[k] is already final (long-read
 * mode, or a class spanning more than 32 segments). Pointers stay valid until sbq_table_free. */
typedef struct {
   int64_t n_entry;
   const int64_t* seg_ptr;
   const uint8_t* n_seg;
   const uint32_t* implicit_mask;   /* bit i set = segment i of the span is implicit (include/isoform.h:363-411) */
   const int32_t* iso_len;          /* L_t of the entry's isoform */
   const uint32_t* pool;
   int64_t n_pool;
} sbq_weight_desc;
int  sbq_table_weight_desc(const sbq_table*, sbq_weight_desc* out);

/* GPU weights (SURVEY 8f.1, the weight half of the class-table build on the device). The insert model and read
 * length are per context; tables built with defer_weights = 1 are queued like sbq_submit, their alpha is computed by
 * weights_kernel during sbq_upload. A batch is either all deferred or all host-weighted. sbq_fetch_alpha copies the
 * device alpha (nnz doubles, CSR order of the batch) back, e.g. to fill ExonBin::_bin_weight_map for -f output.
 * Call it BEFORE the first sbq_solve of an upload: the one-off layout pass of the giant-locus tier re-sorts the weights
 * of giant loci inside each row's CSR range (bank order), after which they no longer line up with the host's columns. */
int  sbq_set_insert_model(sbq_ctx*, const sbq_insert_model* model, int32_t read_len);
int  sbq_submit_deferred(sbq_ctx*, const sbq_table* const* tables, int64_t n_tables);
int  sbq_fetch_alpha(sbq_ctx*, double* alpha);

/* Class assignment ON THE DEVICE (SURVEY 8f.1; strawberry_b200/csrc/sbq_rawbuild.cuh). sbq_submit_raw queues one locus as
 * the reference's LocusContext constructor receives it - the same sbq_locus_input sbq_build_locus takes (read_len and the
 * insert model come from sbq_set_insert_model; defer_weights is ignored) - and sbq_upload then builds the whole class table of
 * the batch on the GPU: compatibility (Contig::is_compatible), class coordinates (overlap_exons), first-seen class ids,
 * code-blind set semantics of ExonBin::_frags, float class masses, the class x isoform CSR and the weight descriptors that
 * weights_kernel turns into alpha. Integer results are bit-identical to sbq_build_locus (tests/test_gpu_rawbuild.py,
 * tests/test_gpu_rawbuild_long.py). A batch is either all raw loci or none. In a multi-GPU context (n_gpus > 1) every raw locus
 * is dealt to a device when it is submitted - the device with the least hits x isoforms so far; its non-zeros are not known
 * before the table exists - and the devices build their tables concurrently; results come back in submit order. A hit may
 * touch any number of exon segments and a class may span any number of an isoform's segments (long reads, exon-dense loci),
 * as in sbq_build_locus; a locus may have at most 65535 segments (sbq_submit_raw refuses more). What the kernels cannot
 * reproduce bit-exactly - in the default mass mode fragment masses that are not multiples of 1/2, a 64-bit hash collision
 * of two coordinate lists - and a class coordinate outside the isoform's segments (the reference asserts) make sbq_upload
 * return SBQ_ERR_UNSUPPORTED: use sbq_build_locus for such a batch. Fractional masses are accepted in SBQ_RAW_MASS_ANY mode (below).
 * sbq_fetch_raw_classes (tests, single-device contexts) copies the device-built table out; the CSR comes from sbq_fetch_batch.
 * Its hit_coords[n_hit][16] holds the first 16 segments a hit touches (zeros after the last) and hit_ncoord[n_hit] their
 * number, saturated at 255; for hits of at most 16 segments that is the whole list. sbq_fetch_raw_coords (tests,
 * single-device contexts) copies the full lists: hit h touches hit_coords[hit_coord_off[h] .. hit_coord_off[h + 1]), and
 * hit_coord_off[n_hit] is the length of hit_coords (fetch the offsets first, with hit_coords = NULL, to size it). */
int  sbq_submit_raw(sbq_ctx*, const sbq_locus_input* in, int64_t* locus_index /* may be NULL: position of the locus in the batch (submit order) */);
int  sbq_fetch_raw_classes(sbq_ctx*, int32_t* hit_class, uint8_t* hit_ncoord, uint16_t* hit_coords, int64_t* class_rep, float* class_mass,
                           int32_t* class_nfrag);
int  sbq_fetch_raw_coords(sbq_ctx*, int64_t* hit_coord_off /* [n_hit + 1] */, uint16_t* hit_coords);

/* How the device adds the masses of a raw batch's classes (n_c = (int) sum of float masses over ExonBin::_frags,
 * include/isoform.h:285-296; the sum runs in std::set<Contig> order: ref_id, then the feature lists lexicographically by
 * (offset, len), op codes ignored, a proper prefix first).
 *   SBQ_RAW_MASS_HALVES (default)  order-free atomic sum; exact, hence equal to the set-order sum, because every mass must be a
 *                                  multiple of 1/2 and every class sum below 2^23 (collapse masses without
 *                                  --allow-multimapped-hits); any other mass makes sbq_upload return SBQ_ERR_UNSUPPORTED.
 *   SBQ_RAW_MASS_ANY               any finite, non-negative mass (1/NH fractions of multimapped hits): the surviving members of
 *                                  every class are sorted in set order on the device and added in float in that order, bit for
 *                                  bit the reference's sum. A class sum of 2^31 or more is refused ((int) is undefined there).
 * The mode is per context, takes effect at the next sbq_upload and is forwarded to the devices of a multi-GPU context.
 * An unknown mode returns SBQ_ERR_INVALID. */
enum { SBQ_RAW_MASS_HALVES = 0, SBQ_RAW_MASS_ANY = 1 };
int  sbq_set_raw_mass_mode(sbq_ctx*, int32_t mode);

/* hit_class[n_hit]: class id of every input hit (the ExonBin whose _frags set it was offered to), -1 for hits
 * that were dropped (ref_id -1) or are compatible with no isoform. */
int  sbq_table_hit_classes(const sbq_table*, int32_t* hit_class);

/* a11: feature list of one collapsed fragment from its mates' CIGARs (Contig::Contig(const PairedHit&)).
 * A mate with n_cig == 0 is absent. Returns the number of features written (0 = inconsistent
 * overlapping mates => ref_id -1), or a negative sbq_error (SBQ_ERR_INVALID if cap is too small). */
int  sbq_pair_features(uint32_t left_pos, const uint8_t* left_cig_op, const uint32_t* left_cig_len, int32_t left_n_cig,
                       uint32_t right_pos, const uint8_t* right_cig_op, const uint32_t* right_cig_len, int32_t right_n_cig,
                       uint32_t* feat_off, uint32_t* feat_len, uint8_t* feat_code, int32_t cap);

/* a6 / a13 exposed for unit parity: ExonBin::effective_len and InsertSize::emp_dist_pdf. */
int32_t sbq_effective_len(const uint32_t* seg_lens, int32_t n_seg, const uint32_t* implicit_idx, int32_t n_implicit,
                          int32_t fl, int32_t rl);
double  sbq_insert_pdf(const sbq_insert_model* model, uint32_t insert_size);

#ifdef __cplusplus
}
#endif
#endif /* SBQ_BUILDER_H_ */

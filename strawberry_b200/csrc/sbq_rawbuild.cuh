// sbq_rawbuild.cuh - fragment-class assignment ON THE DEVICE (SURVEY section 8f.1, rows a3 / a7 / a9 of the scope table).
//
// What LocusContext::assign_exon_bin computes (reference src/estimate.cpp:135-198, with Contig::is_compatible
// src/contig.cpp:547-599, overlap_exons src/estimate.cpp:115-131, ExonBin::read_count include/isoform.h:285-296), for a whole
// batch of loci at once, from the collapsed hits' and the isoforms' feature lists:
//
//   raw_hit_kernel     one thread per hit: compatibility with every isoform of its locus (bit mask), the NUMBER of disjoint
//                      exon segments its aligned blocks touch (the class coordinates), hashes of both
//   raw_class_insert / raw_class_rep   hash table per locus keyed by the coordinate list: the FIRST hit (smallest index) of
//                      every distinct list is the class representative - the reference numbers classes in first-seen order,
//                      so class id = number of representatives before it (one prefix sum over the hits of the batch)
//   raw_coord_kernel   the coordinate lists themselves, into one u16 pool at the hit's offset (prefix sum of the counts): a
//                      full-length long read touches every segment of its gene, so no per-hit limit
//   raw_member_kernel  class of every hit, union of the members' isoform masks (iso_2_bins_map), second hash table keyed by
//                      (class, code-blind feature list): the reference keeps the members in a std::set under a comparator that
//                      ignores the op code, so of several equivalent hits only the first inserted one counts
//   raw_mass_kernel    class mass = sum of the surviving members' masses (float), member count
//   raw_member_*       RB_MASS_ANY only: the class mass summed in set order instead (scatter, sort, one thread per class)
//   raw_nnz_kernel / raw_fill_kernel   CSR rows (classes) x columns (isoforms, ascending), integer counts (int)mass, and per
//                      entry the descriptor of the class under the isoform (segment lengths of the span, implicit-segment mask,
//                      L_t: ExonBin::bin_under_iso, include/isoform.h:363-411) that weights_kernel turns into alpha. The
//                      nnz kernel also counts the segments a class's entries span; their prefix sum places each class's
//                      segment lengths in the descriptor pool (4 B per spanned segment, no per-entry limit)
//
// Everything is order-free, so atomics are safe: class ids come from a prefix sum, set semantics from atomicMin on the hit
// index. In the default mass mode (RB_MASS_HALVES) the float mass sum is EXACT (hence independent of the order the reference's
// std::set imposes) as long as every mass is a multiple of 1/2 and a class holds less than 2^23 of it - true for every BAM read
// without --allow-multimapped-hits (collapse masses are multiplicities of 0.5 + 0.5). With 1/NH masses the float sum depends on
// the order, so RB_MASS_ANY sorts every class's survivors in set order and adds them in that order. The kernels flag what they
// cannot reproduce bit-exactly (in the default mode a mass that is not a multiple of 1/2; in RB_MASS_ANY a NaN, infinite or
// negative mass; a 64-bit hash collision), a class mass (int) cannot hold, or what the reference asserts on (a class coordinate
// outside the isoform's segments), and the upload is refused with SBQ_ERR_UNSUPPORTED: the caller then uses the host builder.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace sbq {

enum : int { RB_FLAG_COLLISION = 2, RB_FLAG_MASS = 4, RB_FLAG_NSEG = 8 };
enum : int { RB_MASS_HALVES = 0, RB_MASS_ANY = 1 };   // SBQ_RAW_MASS_HALVES / SBQ_RAW_MASS_ANY
constexpr unsigned long long RB_EMPTY = 0xffffffffffffffffull;

struct RawBatch {
   int64_t n_hit;
   int32_t n_loci;
   int32_t long_read;
   int32_t mass_mode;              // RB_MASS_HALVES: order-free atomic sum of multiples of 1/2; RB_MASS_ANY: sum in set order
   // input (device copies of the staged batch)
   const int32_t* hit_locus;       // [H]
   const int64_t* hit_feat_ptr;    // [H + 1]
   const uint32_t* hf_off;
   const uint32_t* hf_len;
   const uint8_t* hf_code;
   const float* hit_mass;          // [H] (PairedHit::collapse_mass read back as float, src/contig.cpp:306-309)
   const int32_t* hit_ref;         // [H]
   const int64_t* loc_hit_off;     // [L + 1]
   const int64_t* loc_iso_off;     // [L + 1]
   const int64_t* loc_seg_off;     // [L + 1]
   const int64_t* iso_feat_ptr;    // [T + 1]
   const uint32_t* if_off;
   const uint32_t* if_len;
   const uint8_t* if_code;
   const uint32_t* seg_left;       // [S] disjoint exon segments of every locus (closed intervals)
   const uint32_t* seg_right;
   const int64_t* iso_seg_ptr;     // [T + 1]
   const int32_t* iso_seg;         // segment indices (local to the locus) contained in each isoform, ascending
   const int32_t* iso_len;         // [T]
   // workspace
   int32_t* ncoord;                // [H] number of segments the hit touches
   int64_t* coord_off;             // [H + 1] exclusive prefix sum of ncoord: the hit's list in coords
   uint16_t* coords;               // [coord_off[H]] segment indices (local) each hit touches, ascending (allocated once the total is known)
   int64_t n_coord;
   uint8_t* valid;                 // [H] compatible with at least one isoform and touches at least one segment
   unsigned long long* chash;      // [H] hash of the coordinate list
   unsigned long long* fhash;      // [H] hash of (ref_id, code-blind feature list)
   const int64_t* loc_cm_off;      // [L + 1] first compatibility-mask word of the locus (hit i of the locus: + i * W, W = ceil(T / 32))
   uint32_t* cm;
   const int64_t* loc_tab_off;     // [L + 1] first hash-table slot of the locus; the capacity (a power of two) is the difference
   unsigned long long* keys1;      // class table
   uint32_t* min1;
   uint32_t* slot1;                // [H]
   unsigned long long* keys2;      // member (dedup) table
   uint32_t* min2;
   uint32_t* slot2;                // [H]
   int32_t* is_rep;                // [H]
   int64_t* cls_prefix;            // [H + 1] exclusive prefix sum of is_rep = global class index of a representative
   int32_t* hit_class;             // [H] class id local to the locus, -1 for invalid hits
   int* flags;
   // class-level arrays (allocated once the number of classes is known)
   const int64_t* loc_cls_off;     // [L + 1] first class of the locus
   const int64_t* loc_cmask_off;   // [L + 1] first isoform-mask word of the locus' classes (class c: + c * W)
   int64_t* class_rep;             // [R] representative hit (global index)
   float* class_mass;              // [R]
   int32_t* class_nfrag;           // [R]
   uint32_t* cmask;
   int32_t* class_nnz;             // [R]
   int32_t* class_nseg;            // [R] segments spanned by the class's CSR entries, summed (descriptor pool length of the row)
};

__device__ __forceinline__ unsigned long long rb_mix(unsigned long long h, unsigned long long x) {
   h ^= x + 0x9E3779B97F4A7C15ull + (h << 6) + (h >> 2);
   h *= 0xBF58476D1CE4E5B9ull;
   return h ^ (h >> 29);
}

// Contig::is_compatible(read, isoform) (src/contig.cpp:547-599). Transcripts alternate MATCH / INTRON features
// (Contig 6-argument ctor), so exon k is feature 2 k and "the isoform's next intron" is feature 2 k + 1.
__device__ inline bool rb_compatible(const uint32_t* ro, const uint32_t* rl, const uint8_t* rc, int rn, const uint32_t* io, const uint32_t* il, const uint8_t* ic, int in) {
   const int ne = (in + 1) >> 1;
   if (rn == 0 || ne == 0) return false;
   const uint32_t fl = ro[0], fr = ro[0] + rl[0] - 1;
   int lo = 0, hi = ne;   // first exon with right >= first.left
   while (lo < hi) {
      const int mid = (lo + hi) >> 1;
      if (io[2 * mid] + il[2 * mid] - 1 < fl) lo = mid + 1; else hi = mid;
   }
   if (lo == ne) return false;
   if (!(io[2 * lo] <= fl && io[2 * lo] + il[2 * lo] - 1 >= fr)) return false;
   int it = lo;
   for (int i = 1; i < rn; ++i) {
      const uint8_t code = rc[i];
      if (code == 2) continue;                                   // S_GAP
      if (code == 1) {                                           // S_INTRON: must equal the isoform's next intron
         const int nx = 2 * it + 1;
         if (nx >= in) return false;
         if (!(ic[nx] == code && io[nx] == ro[i] && il[nx] == rl[i])) return false;
      } else {                                                   // S_MATCH: inside the current or a later exon
         const uint32_t l = ro[i], r = ro[i] + rl[i] - 1;
         while (it < ne && !(io[2 * it] <= l && io[2 * it] + il[2 * it] - 1 >= r)) ++it;
         if (it == ne) return false;
      }
   }
   return true;
}

// overlap_exons() (src/estimate.cpp:115-131): the segments [sl, sr] (closed, ascending, S of them) that any MATCH block of a
// hit touches, ascending; emit(i, s) for the i-th of them. Returns their number.
template <class Emit>
__device__ __forceinline__ int rb_overlap_exons(const uint32_t* ro, const uint32_t* rl, const uint8_t* rc, int rn, const uint32_t* sl, const uint32_t* sr, int S, Emit emit) {
   int nc = 0, next = 0;                                         // blocks are ascending: segments below `next` are listed already
   for (int k = 0; k < rn; ++k) {
      if (rc[k] != 0) continue;
      const uint32_t l_ = ro[k], r_ = ro[k] + rl[k] - 1;
      int lo = 0, hi = S;                                        // first segment with right >= block.left
      while (lo < hi) {
         const int mid = (lo + hi) >> 1;
         if (sr[mid] < l_) lo = mid + 1; else hi = mid;
      }
      for (int s = max(lo, next); s < S && sl[s] <= r_; ++s) { emit(nc++, s); next = s + 1; }
   }
   return nc;
}

__global__ void __launch_bounds__(128) raw_hit_kernel(RawBatch b) {
   for (int64_t h = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; h < b.n_hit; h += (int64_t)gridDim.x * blockDim.x) {
      const int l = b.hit_locus[h];
      const int64_t f0 = b.hit_feat_ptr[h];
      const int rn = (int)(b.hit_feat_ptr[h + 1] - f0);
      b.hit_class[h] = -1;
      b.is_rep[h] = 0;
      b.valid[h] = 0;
      b.ncoord[h] = 0;
      if (rn == 0) continue;                                     // Contig with ref_id == -1: dropped (include/estimate.hpp:71-79)
      const uint32_t *ro = b.hf_off + f0, *rl = b.hf_len + f0;
      const uint8_t* rc = b.hf_code + f0;
      const int64_t t0 = b.loc_iso_off[l];
      const int T = (int)(b.loc_iso_off[l + 1] - t0), W = (T + 31) >> 5;
      uint32_t* cm = b.cm + b.loc_cm_off[l] + (h - b.loc_hit_off[l]) * W;
      int ncompat = 0;
      for (int w = 0; w < W; ++w) {
         uint32_t bits = 0;
         for (int t = 32 * w; t < min(T, 32 * w + 32); ++t) {
            const int64_t i0 = b.iso_feat_ptr[t0 + t];
            const int in = (int)(b.iso_feat_ptr[t0 + t + 1] - i0);
            if (rb_compatible(ro, rl, rc, rn, b.if_off + i0, b.if_len + i0, b.if_code + i0, in)) { bits |= 1u << (t & 31); ++ncompat; }
         }
         cm[w] = bits;
      }
      unsigned long long ch = 1469598103934665603ull;
      const int nc = rb_overlap_exons(ro, rl, rc, rn, b.seg_left + b.loc_seg_off[l], b.seg_right + b.loc_seg_off[l],
                                      (int)(b.loc_seg_off[l + 1] - b.loc_seg_off[l]), [&](int, int s) { ch = rb_mix(ch, (uint16_t)s); });
      b.ncoord[h] = nc;
      b.chash[h] = ch == RB_EMPTY ? 0 : ch;
      unsigned long long fh = rb_mix(88172645463325252ull, (unsigned)b.hit_ref[h]);
      for (int k = 0; k < rn; ++k) fh = rb_mix(rb_mix(fh, ro[k]), rl[k]);
      b.fhash[h] = fh;
      const bool ok = ncompat > 0 && nc > 0;
      b.valid[h] = ok;
      if (ok) {
         const float m = b.hit_mass[h];
         const float m2 = m * 2.0f;
         if (b.mass_mode == RB_MASS_ANY) {
            if (!(m >= 0.0f && m <= 3.402823466e38f)) atomicOr(b.flags, RB_FLAG_MASS);                  // NaN, infinite or negative
         } else if (!(m >= 0.0f && m < 4194304.0f && m2 == floorf(m2))) {
            atomicOr(b.flags, RB_FLAG_MASS);                     // not a multiple of 1/2: the order of the sum would matter
         }
      }
   }
}

// open-addressing insert: returns the slot of `key` in the locus' table; min[slot] ends up as the smallest hit index with that key
__device__ __forceinline__ uint32_t rb_insert(unsigned long long* keys, uint32_t* mins, int64_t base, uint32_t cap, unsigned long long key, uint32_t h) {
   uint32_t s = (uint32_t)(key * 0x9E3779B97F4A7C15ull >> 32) & (cap - 1);
   for (;;) {
      const unsigned long long old = atomicCAS(&keys[base + s], RB_EMPTY, key);
      if (old == RB_EMPTY || old == key) {
         atomicMin(&mins[base + s], h);
         return s;
      }
      s = (s + 1) & (cap - 1);
   }
}

__global__ void __launch_bounds__(256) raw_class_insert_kernel(RawBatch b) {
   for (int64_t h = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; h < b.n_hit; h += (int64_t)gridDim.x * blockDim.x) {
      if (!b.valid[h]) continue;
      const int l = b.hit_locus[h];
      const int64_t base = b.loc_tab_off[l];
      const uint32_t cap = (uint32_t)(b.loc_tab_off[l + 1] - base);
      b.slot1[h] = rb_insert(b.keys1, b.min1, base, cap, b.chash[h], (uint32_t)(h - b.loc_hit_off[l]));
   }
}

__global__ void __launch_bounds__(256) raw_class_rep_kernel(RawBatch b) {
   for (int64_t h = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; h < b.n_hit; h += (int64_t)gridDim.x * blockDim.x) {
      if (!b.valid[h]) continue;
      const int l = b.hit_locus[h];
      if (b.loc_hit_off[l] + b.min1[b.loc_tab_off[l] + b.slot1[h]] == h) b.is_rep[h] = 1;
   }
}

__global__ void __launch_bounds__(128) raw_coord_kernel(RawBatch b) {
   for (int64_t h = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; h < b.n_hit; h += (int64_t)gridDim.x * blockDim.x) {
      if (b.ncoord[h] == 0) continue;
      const int l = b.hit_locus[h];
      const int64_t f0 = b.hit_feat_ptr[h];
      uint16_t* out = b.coords + b.coord_off[h];
      rb_overlap_exons(b.hf_off + f0, b.hf_len + f0, b.hf_code + f0, (int)(b.hit_feat_ptr[h + 1] - f0), b.seg_left + b.loc_seg_off[l],
                       b.seg_right + b.loc_seg_off[l], (int)(b.loc_seg_off[l + 1] - b.loc_seg_off[l]), [&](int i, int s) { out[i] = (uint16_t)s; });
   }
}

__global__ void __launch_bounds__(256) raw_member_kernel(RawBatch b) {
   for (int64_t h = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; h < b.n_hit; h += (int64_t)gridDim.x * blockDim.x) {
      if (!b.valid[h]) continue;
      const int l = b.hit_locus[h];
      const int64_t h0 = b.loc_hit_off[l];
      const int64_t rep = h0 + b.min1[b.loc_tab_off[l] + b.slot1[h]];
      const int64_t cg = b.cls_prefix[rep];                      // global class index = representatives before it
      const int cid = (int)(cg - b.loc_cls_off[l]);
      b.hit_class[h] = cid;
      if (rep == h) {
         b.class_rep[cg] = h;
      } else {                                                   // a 64-bit collision of two different lists: refuse rather than merge classes
         const int n = b.ncoord[h];
         const uint16_t *a = b.coords + b.coord_off[h], *r = b.coords + b.coord_off[rep];
         bool same = b.ncoord[rep] == n;
         for (int i = 0; same && i < n; ++i) same = a[i] == r[i];
         if (!same) atomicOr(b.flags, RB_FLAG_COLLISION);
      }
      const int T = (int)(b.loc_iso_off[l + 1] - b.loc_iso_off[l]), W = (T + 31) >> 5;
      const uint32_t* cm = b.cm + b.loc_cm_off[l] + (h - h0) * W;
      uint32_t* dst = b.cmask + b.loc_cmask_off[l] + (int64_t)cid * W;
      for (int w = 0; w < W; ++w)
         if (cm[w]) atomicOr(&dst[w], cm[w]);                    // iso_2_bins_map[t].insert(class) for every compatible (hit, isoform)
      const int64_t base = b.loc_tab_off[l];
      const uint32_t cap = (uint32_t)(b.loc_tab_off[l + 1] - base);
      unsigned long long key = rb_mix(b.fhash[h], (unsigned long long)cid + 1);
      if (key == RB_EMPTY) key = 0;
      b.slot2[h] = rb_insert(b.keys2, b.min2, base, cap, key, (uint32_t)(h - h0));
   }
}

__global__ void __launch_bounds__(256) raw_mass_kernel(RawBatch b) {
   for (int64_t h = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; h < b.n_hit; h += (int64_t)gridDim.x * blockDim.x) {
      if (!b.valid[h]) continue;
      const int l = b.hit_locus[h];
      const int64_t h0 = b.loc_hit_off[l];
      const int64_t first = h0 + b.min2[b.loc_tab_off[l] + b.slot2[h]];
      if (first != h) {
         // an equivalent hit (same class, same ref_id, same (offset, len) list - op codes ignored) was inserted first: this one is
         // not a new set element, its mass does not count. Verify the equivalence (a hash collision must not drop a real member).
         const int64_t a0 = b.hit_feat_ptr[h], b0 = b.hit_feat_ptr[first];
         const int n = (int)(b.hit_feat_ptr[h + 1] - a0);
         bool same = n == (int)(b.hit_feat_ptr[first + 1] - b0) && b.hit_ref[h] == b.hit_ref[first] && b.hit_class[first] == b.hit_class[h];
         for (int k = 0; same && k < n; ++k) same = b.hf_off[a0 + k] == b.hf_off[b0 + k] && b.hf_len[a0 + k] == b.hf_len[b0 + k];
         if (!same) atomicOr(b.flags, RB_FLAG_COLLISION);
         continue;
      }
      const int64_t cg = b.loc_cls_off[l] + b.hit_class[h];
      if (b.mass_mode == RB_MASS_HALVES) atomicAdd(&b.class_mass[cg], b.hit_mass[h]);   // exact: multiples of 1/2, class total checked against 2^23 below
      atomicAdd(&b.class_nfrag[cg], 1);
   }
}

// ---- RB_MASS_ANY: the class mass is the float sum of the surviving members in std::set<Contig> order (ExonBin::read_count,
// include/isoform.h:285-296). The survivors are scattered into per-class segments, the whole array is sorted by (global class,
// Contig::operator<) - a bitonic sort of 1024-element tiles in shared memory, then merge-path passes that double the sorted
// runs - and one thread per class adds the masses in that order. Survivors of one class are pairwise non-equivalent, so the
// order is total and does not depend on the scatter. An element is (k0, k1, hit): k0 = global class, k1 = (ref_id, offset of the
// first feature), which decide most comparisons; the full feature lists break the remaining ties.
constexpr int RB_SORT_TILE = 1024;
constexpr int RB_MERGE_PER_THREAD = 8;

// Contig::operator< (src/contig.cpp:342-347): ref_id, then the feature lists lexicographically by (offset, len), op codes
// ignored; a proper prefix sorts first
__device__ __forceinline__ bool rb_contig_less(const RawBatch& b, int64_t x, int64_t y) {
   if (x < 0 || y < 0) return false;                             // tile padding
   const int rx = b.hit_ref[x], ry = b.hit_ref[y];
   if (rx != ry) return rx < ry;
   const int64_t x0 = b.hit_feat_ptr[x], y0 = b.hit_feat_ptr[y];
   const int64_t nx = b.hit_feat_ptr[x + 1] - x0, ny = b.hit_feat_ptr[y + 1] - y0;
   for (int64_t k = 0; k < nx && k < ny; ++k) {
      const uint32_t ox = b.hf_off[x0 + k], oy = b.hf_off[y0 + k];
      if (ox != oy) return ox < oy;
      const uint32_t lx = b.hf_len[x0 + k], ly = b.hf_len[y0 + k];
      if (lx != ly) return lx < ly;
   }
   return nx < ny;
}

__device__ __forceinline__ bool rb_member_less(const RawBatch& b, unsigned long long a0, unsigned long long a1, int64_t ah, unsigned long long b0,
                                               unsigned long long b1, int64_t bh) {
   if (a0 != b0) return a0 < b0;
   if (a1 != b1) return a1 < b1;
   return rb_contig_less(b, ah, bh);
}

// survivors (as raw_mass_kernel finds them) into their class's segment [member_off[c], member_off[c + 1]), in any order
__global__ void __launch_bounds__(256) raw_member_scatter_kernel(RawBatch b, const int64_t* __restrict__ member_off, int32_t* __restrict__ cursor,
                                                                 unsigned long long* __restrict__ k0, unsigned long long* __restrict__ k1, int64_t* __restrict__ hit) {
   for (int64_t h = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; h < b.n_hit; h += (int64_t)gridDim.x * blockDim.x) {
      if (!b.valid[h]) continue;
      const int l = b.hit_locus[h];
      if (b.loc_hit_off[l] + b.min2[b.loc_tab_off[l] + b.slot2[h]] != h) continue;
      const int64_t cg = b.loc_cls_off[l] + b.hit_class[h];
      const int64_t k = member_off[cg] + atomicAdd(&cursor[cg], 1);
      k0[k] = (unsigned long long)cg;
      k1[k] = (unsigned long long)((uint32_t)b.hit_ref[h] ^ 0x80000000u) << 32 | b.hf_off[b.hit_feat_ptr[h]];
      hit[k] = h;
   }
}

// every 1024-element tile of the n = *n_member elements sorted in place (bitonic network, padded with elements that sort last)
__global__ void __launch_bounds__(RB_SORT_TILE / 2) raw_member_tile_sort_kernel(RawBatch b, const int64_t* __restrict__ n_member, unsigned long long* __restrict__ k0,
                                                                              unsigned long long* __restrict__ k1, int64_t* __restrict__ hit) {
   __shared__ unsigned long long s0[RB_SORT_TILE], s1[RB_SORT_TILE];
   __shared__ int64_t sh[RB_SORT_TILE];
   const int64_t n = *n_member;
   const int64_t base = (int64_t)blockIdx.x * RB_SORT_TILE;
   if (base >= n) return;
   for (int e = threadIdx.x; e < RB_SORT_TILE; e += blockDim.x) {
      const bool in = base + e < n;
      s0[e] = in ? k0[base + e] : ~0ull;
      s1[e] = in ? k1[base + e] : ~0ull;
      sh[e] = in ? hit[base + e] : -1;
   }
   __syncthreads();
   for (int k = 2; k <= RB_SORT_TILE; k <<= 1) {
      for (int j = k >> 1; j > 0; j >>= 1) {
         const int t = threadIdx.x;
         const int e = 2 * t - (t & (j - 1)), p = e + j;
         const bool asc = (e & k) == 0;
         if (asc ? rb_member_less(b, s0[p], s1[p], sh[p], s0[e], s1[e], sh[e]) : rb_member_less(b, s0[e], s1[e], sh[e], s0[p], s1[p], sh[p])) {
            const unsigned long long a0 = s0[e], a1 = s1[e];
            const int64_t ah = sh[e];
            s0[e] = s0[p]; s1[e] = s1[p]; sh[e] = sh[p];
            s0[p] = a0; s1[p] = a1; sh[p] = ah;
         }
         __syncthreads();
      }
   }
   for (int e = threadIdx.x; e < RB_SORT_TILE && base + e < n; e += blockDim.x) {
      k0[base + e] = s0[e];
      k1[base + e] = s1[e];
      hit[base + e] = sh[e];
   }
}

// one merge-path pass: sorted runs of `width` elements, pairwise merged into runs of 2 width (a run without a partner is copied)
__global__ void __launch_bounds__(256) raw_member_merge_kernel(RawBatch b, const int64_t* __restrict__ n_member, int64_t width,
                                                               const unsigned long long* __restrict__ i0, const unsigned long long* __restrict__ i1, const int64_t* __restrict__ ih,
                                                               unsigned long long* __restrict__ o0, unsigned long long* __restrict__ o1, int64_t* __restrict__ oh) {
   const int64_t n = *n_member;
   for (int64_t out = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) * RB_MERGE_PER_THREAD; out < n;
        out += (int64_t)gridDim.x * blockDim.x * RB_MERGE_PER_THREAD) {
      const int64_t start = out / (2 * width) * (2 * width);
      const int64_t a = start, na = min(width, n - start), bb = start + na, nb = min(width, n - bb);
      const int64_t diag = out - start;
      int64_t lo = max((int64_t)0, diag - nb), hi = min(diag, na);
      while (lo < hi) {                                          // smallest i with B[diag - 1 - i] < A[i]: A[0, i) and B[0, diag - i) come first
         const int64_t mid = (lo + hi) >> 1, y = bb + diag - 1 - mid;
         if (rb_member_less(b, i0[y], i1[y], ih[y], i0[a + mid], i1[a + mid], ih[a + mid])) hi = mid; else lo = mid + 1;
      }
      int64_t x = a + lo, y = bb + (diag - lo);
      const int64_t xe = a + na, ye = bb + nb;
      const int64_t end = min(out + RB_MERGE_PER_THREAD, start + na + nb);
      for (int64_t o = out; o < end; ++o) {
         const bool take_b = x == xe || (y < ye && rb_member_less(b, i0[y], i1[y], ih[y], i0[x], i1[x], ih[x]));
         const int64_t s = take_b ? y++ : x++;
         o0[o] = i0[s]; o1[o] = i1[s]; oh[o] = ih[s];
      }
   }
}

// one thread per class: float sum in set order, round to nearest at every step like the reference's `sum += mass`
__global__ void __launch_bounds__(256) raw_member_sum_kernel(RawBatch b, int64_t n_class, const int64_t* __restrict__ member_off, const int64_t* __restrict__ hit) {
   for (int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; c < n_class; c += (int64_t)gridDim.x * blockDim.x) {
      float s = 0.0f;
      for (int64_t k = member_off[c]; k < member_off[c + 1]; ++k) s = __fadd_rn(s, b.hit_mass[hit[k]]);
      b.class_mass[c] = s;
   }
}

// ExonBin::bin_under_iso (include/isoform.h:363-411): the isoform's segments from the class's first to its last coordinate are
// isegs[lo] .. isegs[lo + n - 1]. Returns n, or 0 when a coordinate lies past the isoform's last segment (the reference asserts).
__device__ __forceinline__ int rb_span(const int32_t* __restrict__ isegs, int nis, int first, int last, int& lo) {
   lo = 0;
   int hi = nis;
   while (lo < hi) { const int mid = (lo + hi) >> 1; if (isegs[mid] < first) lo = mid + 1; else hi = mid; }
   int up = 0;
   hi = nis;
   while (up < hi) { const int mid = (up + hi) >> 1; if (isegs[mid] < last) up = mid + 1; else hi = mid; }
   return lo >= nis || up >= nis ? 0 : up - lo + 1;
}

__global__ void __launch_bounds__(256) raw_nnz_kernel(RawBatch b, int64_t n_class, const int32_t* __restrict__ class_locus) {
   for (int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; c < n_class; c += (int64_t)gridDim.x * blockDim.x) {
      const int l = class_locus[c];
      const int64_t t0 = b.loc_iso_off[l];
      const int T = (int)(b.loc_iso_off[l + 1] - t0), W = (T + 31) >> 5;
      const uint32_t* m = b.cmask + b.loc_cmask_off[l] + (c - b.loc_cls_off[l]) * W;
      const int64_t rep = b.class_rep[c];
      const uint16_t* cc = b.coords + b.coord_off[rep];
      const int first = cc[0], last = cc[b.ncoord[rep] - 1];
      int n = 0, nseg = 0;
      for (int w = 0; w < W; ++w) {
         uint32_t bits = m[w];
         n += __popc(bits);
         while (bits && !b.long_read) {
            const int t = 32 * w + __ffs(bits) - 1;
            bits &= bits - 1;
            int lo;
            const int ns = rb_span(b.iso_seg + b.iso_seg_ptr[t0 + t], (int)(b.iso_seg_ptr[t0 + t + 1] - b.iso_seg_ptr[t0 + t]), first, last, lo);
            if (ns == 0) atomicOr(b.flags, RB_FLAG_NSEG);
            nseg += ns;
         }
      }
      b.class_nnz[c] = n;
      b.class_nseg[c] = nseg;
      // halves: the atomic sum is exact below 2^23; any: (int)mass is defined below 2^31
      if (!(b.class_mass[c] < (b.mass_mode == RB_MASS_ANY ? 2147483648.0f : 8388608.0f))) atomicOr(b.flags, RB_FLAG_MASS);
   }
}

// CSR rows of the batch + per-entry weight descriptors. row_ptr (exclusive scan of class_nnz) and pool_off (exclusive scan of
// class_nseg) are already in place. (The minimum of 8 blocks per SM keeps ptxas from spilling 16 B at the same 48 registers.)
__global__ void __launch_bounds__(128, 8)
raw_fill_kernel(RawBatch b, int64_t n_class, const int32_t* __restrict__ class_locus, const int64_t* __restrict__ row_ptr, const int64_t* __restrict__ pool_off,
                int32_t* __restrict__ col, double* __restrict__ alpha, int32_t* __restrict__ count, int64_t* __restrict__ w_seg, uint16_t* __restrict__ w_n,
                uint32_t* __restrict__ w_mask, int32_t* __restrict__ w_len, uint32_t* __restrict__ w_pool) {
   for (int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; c < n_class; c += (int64_t)gridDim.x * blockDim.x) {
      const int l = class_locus[c];
      const int64_t t0 = b.loc_iso_off[l];
      const int T = (int)(b.loc_iso_off[l + 1] - t0), W = (T + 31) >> 5;
      const uint32_t* m = b.cmask + b.loc_cmask_off[l] + (c - b.loc_cls_off[l]) * W;
      count[c] = (int32_t)b.class_mass[c];                       // n_c = (int) float sum (src/estimate.cpp:288)
      const int64_t rep = b.class_rep[c];
      const uint16_t* cc = b.coords + b.coord_off[rep];
      const int ncc = b.ncoord[rep];
      const int64_t s0 = b.loc_seg_off[l];
      int64_t k = row_ptr[c], p = pool_off[c];
      for (int w = 0; w < W; ++w) {
         uint32_t bits = m[w];
         while (bits) {
            const int t = 32 * w + __ffs(bits) - 1;
            bits &= bits - 1;
            col[k] = t;
            w_len[k] = b.iso_len[t0 + t];
            if (b.long_read) {                                   // set_bin_weight_without_frag_dist: alpha = 1 / L_t (src/estimate.cpp:236-247)
               alpha[k] = 1.0 / (double)b.iso_len[t0 + t];
               w_seg[k] = -1; w_n[k] = 0; w_mask[k] = 0;
            } else {
               // the span's inner segments that the class does not list are implicit. The mask aliases like the reference's
               // 32-bit one (1u << (i & 31), include/isoform.h:476-512), so spans of more than 32 segments weigh the same.
               const int32_t* isegs = b.iso_seg + b.iso_seg_ptr[t0 + t];
               int lo;
               const int nseg = rb_span(isegs, (int)(b.iso_seg_ptr[t0 + t + 1] - b.iso_seg_ptr[t0 + t]), cc[0], cc[ncc - 1], lo);
               uint32_t mask = 0;
               int cpos = 1;
               for (int i = 0; i < nseg; ++i) {
                  const int sg = isegs[lo + i];
                  w_pool[p + i] = b.seg_right[s0 + sg] - b.seg_left[s0 + sg] + 1;
                  if (i >= 1 && i + 1 < nseg) {
                     if (cpos < ncc && sg == (int)cc[cpos]) ++cpos; else mask |= 1u << (i & 31);
                  }
               }
               alpha[k] = 0.0;
               w_seg[k] = p;
               w_n[k] = (uint16_t)nseg;
               w_mask[k] = mask;
               p += nseg;
            }
            ++k;
         }
      }
   }
}

// ---- generic exclusive scan int32 -> int64 (three kernels, 4096 elements per block)
constexpr int RB_SCAN_BLOCK = 4096;
__global__ void __launch_bounds__(1024) rb_scan_sums_kernel(const int32_t* __restrict__ v, int64_t n, long long* __restrict__ block_sum) {
   __shared__ long long red[32];
   const int64_t base = (int64_t)blockIdx.x * RB_SCAN_BLOCK;
   long long s = 0;
   for (int x = threadIdx.x; x < RB_SCAN_BLOCK; x += 1024)
      if (base + x < n) s += v[base + x];
   for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
   if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
   __syncthreads();
   if (threadIdx.x == 0) {
      long long t = 0;
      for (int w = 0; w < 32; ++w) t += red[w];
      block_sum[blockIdx.x] = t;
   }
}
__global__ void __launch_bounds__(1024) rb_scan_fill_kernel(const int32_t* __restrict__ v, int64_t n, const long long* __restrict__ block_off, int64_t* __restrict__ out) {
   __shared__ long long wsum[32];
   const int64_t base = (int64_t)blockIdx.x * RB_SCAN_BLOCK + (int64_t)threadIdx.x * 4;
   int d[4];
   long long mine = 0;
#pragma unroll
   for (int e = 0; e < 4; ++e) { d[e] = base + e < n ? v[base + e] : 0; mine += d[e]; }
   long long incl = mine;
   const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
   for (int o = 1; o < 32; o <<= 1) {
      const long long u = __shfl_up_sync(0xffffffffu, incl, o);
      if (lane >= o) incl += u;
   }
   if (lane == 31) wsum[warp] = incl;
   __syncthreads();
   if (warp == 0) {
      long long w = wsum[lane], wi = w;
      for (int o = 1; o < 32; o <<= 1) {
         const long long u = __shfl_up_sync(0xffffffffu, wi, o);
         if (lane >= o) wi += u;
      }
      wsum[lane] = wi - w;
   }
   __syncthreads();
   long long run = block_off[blockIdx.x] + wsum[warp] + incl - mine;
#pragma unroll
   for (int e = 0; e < 4; ++e) {
      if (base + e < n) out[base + e] = run;
      run += d[e];
      if (base + e == n - 1) out[n] = run;
   }
}

__global__ void rb_gather_kernel(const int64_t* __restrict__ src, const int64_t* __restrict__ idx, int64_t n, int64_t* __restrict__ out) {
   const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
   if (i < n) out[i] = src[idx[i]];
}

}  // namespace sbq

// sbq_weights.cuh - class weights on the GPU (SURVEY 8f.1): alpha_ct = sum_{fl=lmin}^{lmax} pdf(fl) * eff_len(fl) / (L_t - fl + 1),
// what LocusContext::set_theory_bin_weight (reference src/estimate.cpp:201-234) evaluates with a scalar loop per
// (class, isoform) pair and what costs the reference ~12 % of its wall time on human-shaped data.
// One warp per CSR entry, lanes stride the fragment length; integer effective lengths follow
// ExonBin::effective_len (include/isoform.h:419-516) exactly, the insert pdf follows InsertSize::emp_dist_pdf
// (src/read.cpp:274-297). The fp64 sum is formed lane-strided + butterfly instead of sequentially, so alpha agrees
// with the host builder to ~1e-15 relative, not bitwise (the reference itself is -Ofast).
#pragma once
#include "sbq_kernels.cuh"

namespace sbq {

struct WeightModel {
   int use_emp, start_offset, end_offset, total_reads;
   const double* emp_dist;   // device copy of InsertSize::_emp_dist
   double mean, sd;
   int read_len;
};

__device__ __forceinline__ int w_no_gap_ef(int l_left, int l_right, int l_int, int fl) {
   if (fl < l_int + 2) return 0;
   if (fl > l_left + l_right + l_int) return 0;
   const int mid = fl - l_int - 1;
   return min(l_left, mid) + min(l_right, mid) - mid;
}
__device__ __forceinline__ int w_gap_ef(int l_left, int l_right, int l_int, int rl, int gap) {
   if (2 * rl + gap < l_int + 2) return 0;
   if (2 * rl + gap > l_left + l_right + l_int) return 0;
   const int start = max(rl, l_left + l_int - gap - 1);
   const int end = min(l_left, l_left + l_right + l_int - gap - rl);
   return max(0, end - start);
}

// s: the entry's segment lengths (global memory), mask: implicit segments, bit i & 31 for span index i (the reference's 32-bit
// masks alias the same way)
__device__ int w_effective_len(const uint32_t* __restrict__ s, int n, unsigned mask, int fl, int rl) {
   const int gap = fl - 2 * rl;
   if (n == 1) return (int)(s[0] - (uint32_t)fl + 1u);
   if (n == 2) return w_no_gap_ef((int)s[0], (int)s[1], 0, fl);
   const int n_imp = __popc(mask);
   if (n == 3) {
      if (n_imp == 1) return w_gap_ef((int)s[0], (int)s[2], (int)s[1], rl, gap);
      return w_no_gap_ef((int)s[0], (int)s[2], (int)s[1], fl) - w_gap_ef((int)s[0], (int)s[2], (int)s[1], rl, gap);
   }
   if (n == 4) {
      const int s0 = (int)s[0], s1 = (int)s[1], s2 = (int)s[2], s3 = (int)s[3];
      const int hit14 = w_gap_ef(s0, s3, s2 + s1, rl, gap);
      const int hit24 = w_gap_ef(s3, s1, s2, rl, gap);
      const int hit124 = w_gap_ef(s0 + s1, s3, s2, rl, gap);
      const int hit13 = w_gap_ef(s0, s2, s1, rl, gap);
      const int hit134 = w_gap_ef(s0, s2 + s3, s1, rl, gap);
      if (n_imp == 0) return w_no_gap_ef(s0, s3, s1 + s2, fl) - (hit124 - hit14 - hit24) - (hit134 - hit14 - hit13) - hit14;
      if (n_imp == 2) return hit14;
      if (mask & 2u) return hit134 - hit14 - hit13;   // first implicit index == 1
      return hit124 - hit14 - hit24;
   }
   const unsigned num_inners = (unsigned)n - 2;
   unsigned num_pos = 0;
   // the reference's target (uint32_t)(uint64_t)(pow(2, n) - 1) is all ones for 32 <= n <= 53 and 0 from n = 54 on, where
   // 2^n - 1 rounds to 2^n in a double
   const unsigned target = (n < 32 ? (1u << n) - 1u : n < 54 ? 0xffffffffu : 0u) & ~mask;
   if (target == 0) return 0;   // every hit mask has bit 0 set: no start offset can match
   int inner_sum = 0;
   for (int k = 1; k < n - 1; ++k) inner_sum += (int)s[k];
   const unsigned last = s[n - 1];
   for (int i = 1; i != (int)(s[0] + 1u); ++i) {
      unsigned hit = 1;
      const int bp_last = fl - i - inner_sum;
      if ((unsigned)bp_last > last) continue;
      if (bp_last == 0) break;
      hit |= 1u << ((unsigned)(n - 1) & 31u);
      int last_rest = rl - bp_last;
      unsigned j = num_inners;
      while (last_rest > 0 && j > 0) {
         hit |= 1u << (j & 31u);
         last_rest = (int)((unsigned)last_rest - s[j]);
         --j;
      }
      int first_rest = rl - i;
      j = 1;
      while (first_rest > 0 && j <= num_inners) {
         hit |= 1u << (j & 31u);
         first_rest = (int)((unsigned)first_rest - s[j]);
         ++j;
      }
      if (hit == target) ++num_pos;
   }
   return (int)num_pos;
}

__device__ __forceinline__ double w_insert_pdf(const WeightModel& m, unsigned fl) {
   if (m.use_emp) {
      double ret = 0.0;
      if (!(fl < (unsigned)m.start_offset || fl > (unsigned)m.end_offset)) ret = m.emp_dist[fl - (unsigned)m.start_offset] / m.total_reads;
      if (ret != 0.0) return ret;
   }
   const double a = ((double)fl - m.mean) / m.sd;
   const double p = 0.3989422804014327 / m.sd * exp(-0.5 * a * a);
   return p > 0 ? p : 0.0;
}

// NSeg: uint8_t for descriptors built on the host (sbq_weight_desc, spans of at most 32 segments), uint16_t for those the device
// class builder writes (a span may cover every segment of a locus, at most 65 535)
template <typename NSeg>
__global__ void __launch_bounds__(256)
weights_kernel(int64_t n_entry, const int64_t* __restrict__ seg_ptr, const NSeg* __restrict__ n_seg, const uint32_t* __restrict__ mask,
               const int32_t* __restrict__ iso_len, const uint32_t* __restrict__ pool, WeightModel m, double* __restrict__ alpha) {
   const int lane = threadIdx.x & 31;
   const int64_t wid = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5, nw = ((int64_t)gridDim.x * blockDim.x) >> 5;
   for (int64_t k = wid; k < n_entry; k += nw) {
      const int64_t sp = seg_ptr[k];
      if (sp < 0) continue;   // alpha[k] already final
      const uint32_t* s = pool + sp;
      const int n = n_seg[k];
      int lmax = 0, inner = 0;
      for (int i = 0; i < n; ++i) { lmax += (int)s[i]; if (i > 0 && i + 1 < n) inner += (int)s[i]; }
      int lmin = m.use_emp ? m.start_offset : m.read_len;
      if (n > 2) lmin = max(lmin, inner);
      const int L = iso_len[k];
      const unsigned mk = mask[k];
      double sum = 0.0;
      for (int fl = lmin + lane; fl <= lmax; fl += 32) {
         const double le_eff = (double)w_effective_len(s, n, mk, fl, m.read_len);
         sum += w_insert_pdf(m, (unsigned)fl) * le_eff / (double)(L - fl + 1);
      }
      sum = warp_sum(sum);
      if (lane == 0) alpha[k] = sum;
   }
}

}  // namespace sbq

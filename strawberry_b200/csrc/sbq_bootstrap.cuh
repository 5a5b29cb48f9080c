// sbq_bootstrap.cuh - bootstrap replicates of a resident batch (sbq_bootstrap, DESIGN.md "Bootstrap replicates"; our definition,
// the reference has none).
//
// Replicate b of locus l redraws the locus' N = sum_i n_i fragments from its own classes, conditional on N:
//   key     = sm64(sm64(sm64(seed ^ 0xD1B54A32D192ED03) + b) + l)          l = the locus' submit position
//   draw k  : h = sm64(key + k), r = umulhi64(h, N) = floor(h N / 2^64)      k = 0 .. N - 1
//             lands on the row i of the locus with C_i <= r < C_{i+1}      C = exclusive prefix of n over the locus' rows
//   n*_i    = number of draws that land on row i
// A pure integer function of (seed, b, l, the locus' counts): no tier, device, batch mate or chunking of the replicates changes
// it, and tests/bootstrap_ref.py restates it bit for bit. The replicate's EM is the existing launch sequence run with dp.count
// pointing at n*.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "sbq_synth.cuh"

namespace sbq {

__host__ __device__ __forceinline__ uint64_t boot_key(uint64_t seed, uint64_t rep, uint64_t locus) {
   return sm64(sm64(sm64(seed ^ 0xD1B54A32D192ED03ull) + rep) + locus);
}

// largest i in [lo, hi) with v[i] <= x, for ascending v and v[lo] <= x
__device__ __forceinline__ int64_t boot_last_le(const int64_t* __restrict__ v, int64_t lo, int64_t hi, int64_t x) {
   while (hi - lo > 1) {
      const int64_t mid = lo + ((hi - lo) >> 1);
      if (v[mid] <= x) lo = mid; else hi = mid;
   }
   return lo;
}

// One thread per draw, grid-stride over all sum N draws of the batch. draw_off[n_row + 1] is the exclusive prefix of the counts
// over the batch's rows, loc_draw_off[n_loci + 1] the same prefix at the locus boundaries; so draw g belongs to the last locus
// whose first draw is <= g (empty loci share their neighbour's offset and are skipped by "last"), and lands on the last row of that
// locus whose prefix is <= its first draw + r (rows with n_i = 0 likewise). locus_id: the hash position of every locus (multi-GPU
// children: its submit position in the parent), NULL = its own index. out[n_row] must be zero; lanes of a warp that hit the same
// row add once (one hot row of the headline batch holds 342 k fragments).
__global__ void __launch_bounds__(256) boot_resample_kernel(const int64_t* __restrict__ draw_off, const int64_t* __restrict__ loc_draw_off,
                                                            const int64_t* __restrict__ loc_row_off, int64_t n_loci, const int32_t* __restrict__ locus_id,
                                                            uint64_t seed, uint64_t rep, int32_t* __restrict__ out) {
   const int64_t total = loc_draw_off[n_loci];
   const int lane = threadIdx.x & 31;
   const int64_t stride = (int64_t)gridDim.x * blockDim.x;
   for (int64_t g0 = (int64_t)blockIdx.x * blockDim.x + (threadIdx.x & ~31); g0 < total; g0 += stride) {   // warp-uniform bound
      const int64_t g = g0 + lane;
      int64_t row = -1;
      if (g < total) {
         const int64_t l = boot_last_le(loc_draw_off, 0, n_loci, g);
         const int64_t base = loc_draw_off[l], N = loc_draw_off[l + 1] - base;
         const uint64_t id = locus_id ? (uint64_t)locus_id[l] : (uint64_t)l;
         const uint64_t h = sm64(boot_key(seed, rep, id) + (uint64_t)(g - base));
         row = boot_last_le(draw_off, loc_row_off[l], loc_row_off[l + 1], base + (int64_t)__umul64hi(h, (uint64_t)N));
      }
      const unsigned peers = __match_any_sync(0xffffffffu, (unsigned long long)row);
      if (row >= 0 && lane == __ffs(peers) - 1) atomicAdd(out + row, __popc(peers));
   }
}

// TPM of n replicates in place over their FPKM rows, each with its own denominator (same arithmetic as tpm_kernel)
__global__ void __launch_bounds__(256) boot_tpm_kernel(double* __restrict__ fpkm_tpm, int64_t n_iso, int64_t n_rep, const double* __restrict__ sums) {
   const int64_t n = n_iso * n_rep, stride = (int64_t)gridDim.x * blockDim.x;
   for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) fpkm_tpm[i] = 1e6 * fpkm_tpm[i] / sums[i / n_iso];
}

}  // namespace sbq

// sbq_grid.cuh - Tier 3: multi-CTA streaming EM for giant loci (one locus at a time on the whole GPU).
//
// Persistent cooperative kernel, one CTA of 16 warps per SM. The CSR of a giant locus (hundreds of MB)
// lives in HBM and is streamed once per EM iteration: 8 B alpha + 4 B column per non-zero, 8 B row
// pointer + 4 B count per row - exactly the algorithmic bytes of SURVEY section 8d. Rows are split
// over CTAs by non-zero count; inside a CTA each warp owns GT_RU consecutive rows at a time, keeps
// their non-zeros in registers between the normaliser pass (d_i, warp-shuffle reduction) and the
// expected-count pass, and adds u_ij into a WARP-PRIVATE accumulator row in shared memory (a row's
// columns are distinct, so no two lanes of the warp collide; no atomics). Per iteration:
//
//   row pass -> sum over warps (fixed order) -> partial[cta][T] in global scratch -> grid barrier
//   -> column owners sum the partials over CTAs in CTA order -> theta_next[T] -> grid barrier
//   -> every CTA reads theta_next, forms ||theta' - theta||_2 redundantly and takes the same decision.
//
// All reductions have a fixed shape, so results are bit-reproducible for a given grid size.
#pragma once
#include "sbq_kernels.cuh"

namespace sbq {

constexpr int GT_NT = 512;   // threads per CTA (16 warps)
constexpr int GT_RU = 4;     // rows a warp keeps in flight
constexpr int GT_EPL = 2;    // register-held elements per lane per row (rows up to 64 non-zeros)
constexpr size_t GT_SMEM_CAP = 200 * 1024;

__host__ __device__ inline int grid_tier_warps(int T) {
   long long budget = (long long)(GT_SMEM_CAP / sizeof(double)) - 3LL * T - 16;
   long long w = budget / (T > 0 ? T : 1);
   if (w > GT_NT / 32) w = GT_NT / 32;
   return (int)w;
}
inline bool grid_tier_supports(int T) { return grid_tier_warps(T) >= 4; }

struct GridScratch {
   double* partial;        // [n_cta][tstride]
   double* theta_next;     // [tstride]
   long long* ctr;         // [n_list][2]  total count, kept rows
   int* zero_flag;         // [n_list]
   int tstride;
};

// ---- per-locus frame shared by the three giant-tier kernels (em_grid_kernel, em_grid_tma_kernel, em_grid_dual_kernel)

// Rows [s_rows[0], s_rows[1]) of CTA b of nb: the locus's R rows split over the grid by non-zero count, inner boundaries rounded to
// the nearest multiple of `chunk` rows (1: not rounded). Threads 0 and 1 write s_rows; the caller synchronises before reading it.
__device__ __forceinline__ void grid_row_range(const int64_t* rp, int R, int chunk, int b, int nb, int* s_rows) {
   const int tid = threadIdx.x;
   if (tid < 2) {
      const int64_t base = rp[0], nnz = rp[R] - base;
      const int64_t target = base + (nnz * (int64_t)(b + tid)) / nb;
      int lo = 0, hi = R;
      if (b + tid >= nb) lo = R;
      else if (b + tid == 0) hi = 0;
      while (lo < hi) {
         const int mid = (lo + hi) >> 1;
         if (rp[mid] < target) lo = mid + 1; else hi = mid;
      }
      if (b + tid < nb) lo = min(R, (lo + chunk / 2) / chunk * chunk);
      s_rows[tid] = lo;
   }
}

// Adds the total / kept row counts of this warp's setup pass into the counters of list entry `item`.
__device__ __forceinline__ void grid_publish_counts(const GridScratch& gs, int item, long long tot, long long kept) {
   tot = warp_sum_ll(tot);
   kept = warp_sum_ll(kept);
   if ((threadIdx.x & 31) == 0 && (tot | kept)) {
      atomicAdd((unsigned long long*)&gs.ctr[2 * item], (unsigned long long)tot);
      atomicAdd((unsigned long long*)&gs.ctr[2 * item + 1], (unsigned long long)kept);
   }
}

// Called by every CTA once it has written its partial[cta][0, T): column owners sum the partials over the CTAs, in CTA order,
// into theta_next. Returns when theta_next is complete, on every CTA.
template <int NT>
__device__ __forceinline__ void grid_owner_reduce(cg::grid_group& grid, const GridScratch& gs, int T) {
   const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nb = gridDim.x;
   grid.sync();
   for (int j = blockIdx.x * (NT / 32) + warp; j < T; j += nb * (NT / 32)) {
      double sj = 0.0;
      for (int cta = lane; cta < nb; cta += 32) sj += __ldcg(gs.partial + (size_t)cta * gs.tstride + j);
      sj = warp_sum(sj);
      if (lane == 0) gs.theta_next[j] = sj;
   }
   grid.sync();
}

// Copies theta' (theta_next) into th[0, T) and returns ||theta' - cur||^2, the same value on every thread of every CTA.
template <int NT>
__device__ __forceinline__ double grid_read_next(const GridScratch& gs, const double* cur, double* th, int T, double* red) {
   double d2 = 0.0;
   for (int j = threadIdx.x; j < T; j += NT) {
      const double nj = __ldcg(gs.theta_next + j);
      const double diff = nj - cur[j];
      d2 += diff * diff;
      th[j] = nj;
   }
   return block_sum<NT>(d2, red);
}

__device__ __forceinline__ double ld_stream_f64(const double* p) {
   double v;
   asm volatile("ld.global.nc.L1::no_allocate.f64 %0, [%1];" : "=d"(v) : "l"(p));
   return v;
}
__device__ __forceinline__ int ld_stream_s32(const int32_t* p) {
   int v;
   asm volatile("ld.global.nc.L1::no_allocate.s32 %0, [%1];" : "=r"(v) : "l"(p));
   return v;
}

// One pass over this CTA's rows. SETUP: row filter + column sums of kept rows (+ total / kept counts).
// !SETUP: one E/M pass with the scaled theta in th[].
template <bool SETUP>
__device__ __forceinline__ void grid_row_pass(const DevParams& p, const int64_t* __restrict__ rp, int32_t* neff,
                                              const int32_t* __restrict__ cnt, int ra, int rb, int W, const double* th,
                                              double* acc, int T, long long& tot, long long& kept, int& zero) {
   const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
   if (warp >= W) return;
   double* my = acc + (size_t)warp * T;
   const int32_t* __restrict__ col = p.col;
   const double* __restrict__ al = p.alpha;
   for (int base = ra + warp * GT_RU; base < rb; base += W * GT_RU) {
      // row metadata: lanes 0..RU fetch row pointers, lanes 0..RU-1 fetch counts
      int64_t rpv = 0;
      int nev = -1;
      if (lane <= GT_RU) rpv = rp[min(base + lane, rb)];
      if (lane < GT_RU && base + lane < rb) nev = SETUP ? cnt[base + lane] : neff[base + lane];
      int64_t k0[GT_RU], k1[GT_RU];
      int ne[GT_RU];
      bool fast = true;
#pragma unroll
      for (int q = 0; q < GT_RU; ++q) {
         k0[q] = __shfl_sync(0xffffffffu, rpv, q);
         k1[q] = __shfl_sync(0xffffffffu, rpv, q + 1);
         ne[q] = __shfl_sync(0xffffffffu, nev, q);
         if (base + q >= rb || (!SETUP && ne[q] < 0)) k1[q] = k0[q];   // nothing to do for this slot
         fast &= (k1[q] - k0[q]) <= 32 * GT_EPL;
      }
      if (fast) {
         double a[GT_RU][GT_EPL];
         int c[GT_RU][GT_EPL];
#pragma unroll
         for (int q = 0; q < GT_RU; ++q)
#pragma unroll
            for (int e = 0; e < GT_EPL; ++e) {
               const int64_t k = k0[q] + lane + 32 * e;
               const bool v = k < k1[q];
               a[q][e] = v ? ld_stream_f64(al + k) : 0.0;
               c[q][e] = v ? ld_stream_s32(col + k) : -1;
            }
         if (SETUP) {
#pragma unroll
            for (int q = 0; q < GT_RU; ++q) {
               bool keep = false;
#pragma unroll
               for (int e = 0; e < GT_EPL; ++e) keep |= a[q][e] > p.row_eps;
               keep = __any_sync(0xffffffffu, keep);
               if (base + q < rb) {
                  if (lane == 0) { neff[base + q] = keep ? ne[q] : -1; tot += ne[q]; kept += keep; }
                  if (keep) {
#pragma unroll
                     for (int e = 0; e < GT_EPL; ++e)
                        if (c[q][e] >= 0) my[c[q][e]] += a[q][e];
                  }
               }
               __syncwarp();
            }
         } else {
            double t[GT_RU][GT_EPL], d[GT_RU];
#pragma unroll
            for (int q = 0; q < GT_RU; ++q) {
               d[q] = 0.0;
#pragma unroll
               for (int e = 0; e < GT_EPL; ++e) {
                  t[q][e] = c[q][e] >= 0 ? th[c[q][e]] : 0.0;
                  d[q] += a[q][e] * t[q][e];
               }
            }
#pragma unroll
            for (int q = 0; q < GT_RU; ++q) d[q] = warp_sum(d[q]);
            // one division per row: lane q divides for row q
            double rmine = 0.0;
#pragma unroll
            for (int q = 0; q < GT_RU; ++q)
               if (lane == q && k1[q] > k0[q]) {
                  if (d[q] == 0) zero = 1; else rmine = (double)ne[q] / d[q];
               }
#pragma unroll
            for (int q = 0; q < GT_RU; ++q) {
               const double r = __shfl_sync(0xffffffffu, rmine, q);
#pragma unroll
               for (int e = 0; e < GT_EPL; ++e)
                  if (c[q][e] >= 0) my[c[q][e]] += a[q][e] * t[q][e] * r;
               __syncwarp();   // the next row may touch the same accumulator column from another lane
            }
         }
      } else {
         // generic path for long rows: stream the row twice (second read hits L1/L2)
         for (int q = 0; q < GT_RU; ++q) {
            if (base + q >= rb) break;
            if (SETUP) {
               bool keep = false;
               for (int64_t k = k0[q] + lane; k < k1[q]; k += 32) keep |= al[k] > p.row_eps;
               keep = __any_sync(0xffffffffu, keep);
               if (lane == 0) { neff[base + q] = keep ? ne[q] : -1; tot += ne[q]; kept += keep; }
               if (keep)
                  for (int64_t k = k0[q] + lane; k < k1[q]; k += 32) my[col[k]] += al[k];
            } else {
               if (k1[q] == k0[q]) continue;
               double d = 0.0;
               for (int64_t k = k0[q] + lane; k < k1[q]; k += 32) d += al[k] * th[col[k]];
               d = warp_sum(d);
               if (d == 0) { zero = 1; continue; }
               const double r = (double)ne[q] / d;
               for (int64_t k = k0[q] + lane; k < k1[q]; k += 32) {
                  const int cc = col[k];
                  my[cc] += al[k] * th[cc] * r;
               }
            }
            __syncwarp();
         }
      }
      __syncwarp();
   }
}

__global__ void __launch_bounds__(GT_NT, 1)
em_grid_kernel(DevParams p, const int32_t* __restrict__ list, int n_list, GridScratch gs) {
   cg::grid_group grid = cg::this_grid();
   extern __shared__ double smem[];
   __shared__ double red[GT_NT / 32];
   __shared__ int s_rows[2];
   const int tid = threadIdx.x;
   const int nb = gridDim.x, b = blockIdx.x;

   for (int item = 0; item < n_list; ++item) {
      const int l = list[item];
      const int64_t r0 = p.loc_row_off[l];
      const int R = (int)(p.loc_row_off[l + 1] - r0);
      const int64_t t0 = p.loc_iso_off[l];
      const int T = (int)(p.loc_iso_off[l + 1] - t0);
      const int W = grid_tier_warps(T);
      double* th = smem;
      double* cur = th + T;
      double* sdiv = cur + T;
      double* acc = sdiv + T;   // [W][T]
      const int64_t* __restrict__ rp = p.row_ptr + r0;
      int32_t* neff = p.neff + r0;
      const int32_t* cnt = p.count + r0;
      double* my_partial = gs.partial + (size_t)b * gs.tstride;

      grid_row_range(rp, R, 1, b, nb, s_rows);
      for (int x = tid; x < W * T; x += GT_NT) acc[x] = 0.0;
      __syncthreads();
      const int ra = s_rows[0], rb = s_rows[1];

      // ---- setup
      long long tot = 0, kept = 0;
      int zero = 0;
      grid_row_pass<true>(p, rp, neff, cnt, ra, rb, W, th, acc, T, tot, kept, zero);
      grid_publish_counts(gs, item, tot, kept);
      __syncthreads();
      for (int j = tid; j < T; j += GT_NT) {
         double sj = 0.0;
         for (int w = 0; w < W; ++w) { sj += acc[(size_t)w * T + j]; acc[(size_t)w * T + j] = 0.0; }
         my_partial[j] = sj;
      }
      grid_owner_reduce<GT_NT>(grid, gs, T);
      const double total = (double)__ldcg(gs.ctr + 2 * item);
      const long long kept_all = __ldcg(gs.ctr + 2 * item + 1);
      const double theta0 = total / (double)T;
      for (int j = tid; j < T; j += GT_NT) {
         sdiv[j] = __ldcg(gs.theta_next + j);
         cur[j] = theta0;
         th[j] = theta0;
      }
      grid.sync();   // theta_next is rewritten in iteration 0 only after everyone copied s_j out

      int status = LOCUS_ITER_CAP, iters = 0;
      if (kept_all == 0) {
         status = LOCUS_NO_ROWS;
      } else {
         for (int it = 0; it < p.max_iter; ++it) {
            iters = it + 1;
            zero = 0;
            long long dummy0 = 0, dummy1 = 0;
            grid_row_pass<false>(p, rp, neff, cnt, ra, rb, W, th, acc, T, dummy0, dummy1, zero);
            zero = __syncthreads_or(zero);
            if (zero && tid == 0) atomicOr(&gs.zero_flag[item], 1);
            for (int j = tid; j < T; j += GT_NT) {
               double sj = 0.0;
               for (int w = 0; w < W; ++w) { sj += acc[(size_t)w * T + j]; acc[(size_t)w * T + j] = 0.0; }
               my_partial[j] = sj;
            }
            grid_owner_reduce<GT_NT>(grid, gs, T);
            const int zf = *(volatile int*)&gs.zero_flag[item];
            const double d2 = grid_read_next<GT_NT>(gs, cur, th, T, red);
            if (zf) { status = LOCUS_ZERO_DENOM; break; }
            // (the TMA and two-slot kernels test d2 < tol^2: the two tests can disagree in the last bit, so unifying them could
            // change an iteration count)
            if (sqrt(d2) < p.tol) { status = LOCUS_OK; break; }
            for (int j = tid; j < T; j += GT_NT) {
               const double nj = th[j];
               cur[j] = nj;
               const double sj = sdiv[j];
               th[j] = (sj != 0) ? nj / sj : 0.0;
            }
            __syncthreads();
         }
      }

      // ---- outputs + epilogue by CTA 0 (src/estimate.cpp:310-356)
      if (b == 0) {
         locus_epilogue_block<GT_NT>(p, l, t0, T, status, iters, theta0, cur, th, red);
      }
      grid.sync();   // scratch (partial, theta_next) is reused by the next locus
   }
}

// ---- host side

// Device buffer that grows on demand (it allocates 1/8 more than asked).
struct DevBuf {
   void* p = nullptr;
   size_t cap = 0;
   bool reserve(size_t bytes) {
      if (bytes <= cap) return true;
      if (p) cudaFree(p);
      p = nullptr;
      cap = 0;
      size_t want = bytes + bytes / 8 + 4096;
      if (cudaMalloc(&p, want) != cudaSuccess) return false;
      cap = want;
      return true;
   }
   void release() {
      if (p) cudaFree(p);
      p = nullptr;
      cap = 0;
   }
};

// Global scratch of one giant-tier launch, carved out of buf (grown if needed): partial[nb][tstride], then (cur_glob != nullptr)
// the per-CTA theta copies [nb][tstride], theta_next[tstride] and the per-entry counters, which are cleared on st.
// Returns 0 or an sbq_error code (<0).
inline int grid_scratch(DevBuf& buf, int nb, int tstride, int n_list, double** cur_glob, cudaStream_t st, GridScratch* gs) {
   const size_t arr = (size_t)nb * tstride * sizeof(double);
   const size_t ctr_bytes = (size_t)n_list * (2 * sizeof(long long) + sizeof(int));
   if (!buf.reserve(arr * (cur_glob ? 2 : 1) + (size_t)tstride * sizeof(double) + ctr_bytes + 1024)) return -4;
   char* q = (char*)buf.p;
   gs->partial = (double*)q; q += arr;
   if (cur_glob) { *cur_glob = (double*)q; q += arr; }
   gs->theta_next = (double*)q; q += (size_t)tstride * sizeof(double);
   gs->ctr = (long long*)q; q += (size_t)n_list * 2 * sizeof(long long);
   gs->zero_flag = (int*)q;
   gs->tstride = tstride;
   return cudaMemsetAsync(gs->ctr, 0, ctr_bytes, st) == cudaSuccess ? 0 : -3;
}

// Calls launch(i0, i1, nc, max_iso) for every run [i0, i1) of list entries with the same warp count nc = nc_of(T) (the planner
// sorts the list by it; max_iso: the largest T of the run), one cooperative launch each. Returns the first non-zero result.
template <typename NcOf, typename Launch>
inline int grid_for_each_run(const int* h_iso, int n_list, NcOf nc_of, Launch launch) {
   for (int i0 = 0; i0 < n_list;) {
      const int nc = nc_of(h_iso[i0]);
      int i1 = i0, mx = 1;
      while (i1 < n_list && nc_of(h_iso[i1]) == nc) { mx = mx > h_iso[i1] ? mx : h_iso[i1]; ++i1; }
      if (const int rc = launch(i0, i1, nc, mx)) return rc;
      i0 = i1;
   }
   return 0;
}

// Host launcher. Returns 0 or an sbq_error code (<0). scratch: a device buffer the caller owns and this function may grow.
inline int grid_tier_launch(const DevParams& dp, const int32_t* d_list, int n_list, const cudaDeviceProp& prop, DevBuf& scratch, cudaStream_t st,
                            int* n_launch) {
   *n_launch = 0;
   if (n_list == 0) return 0;
   const size_t smem = GT_SMEM_CAP;
   if (cudaFuncSetAttribute(em_grid_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess) return -3;
   int per_sm = 0;
   if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, em_grid_kernel, GT_NT, smem) != cudaSuccess || per_sm < 1) return -3;
   const int nb = prop.multiProcessorCount;   // one CTA per SM
   GridScratch gs;
   // tstride 4096: >= T for every locus grid_tier_supports() accepts
   if (const int rc = grid_scratch(scratch, nb, 4096, n_list, nullptr, st, &gs)) return rc;
   DevParams dpc = dp;
   void* args[] = {(void*)&dpc, (void*)&d_list, (void*)&n_list, (void*)&gs};
   if (cudaLaunchCooperativeKernel((void*)em_grid_kernel, dim3(nb), dim3(GT_NT), args, smem, st) != cudaSuccess) return -3;
   *n_launch = 1;
   return 0;
}

}  // namespace sbq

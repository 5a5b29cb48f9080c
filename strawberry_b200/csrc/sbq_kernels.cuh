// sbq_kernels.cuh - sm_100a EM kernels for the per-locus Latent-Class-Model quantification.
//
// What is computed (semantics of EmSolver::init + run, reference src/estimate.cpp:366-488, and of the
// FPKM/frac/filter tail of LocusContext::estimate_abundances, src/estimate.cpp:310-356):
//
//   total   = sum_i n_i over ALL rows;            theta_j = total / T                      (:374-375)
//   keep_i  = any_j alpha_ij > row_eps;           no kept row -> NO_ROWS                   (:377-391)
//   it = 0..max_iter-1:                                                                    (:444)
//       d_i      = sum_j F_ij theta_j  (kept rows);   any d_i == 0 -> ZERO_DENOM, theta := total/T (:449-453)
//       theta'_j = sum_i n_i F_ij theta_j / d_i                                           (:455-464)
//       F_ij    <- F_ij / s_j,  s_j = sum_i F_ij  (columns with s_j == 0 untouched)        (:466-478)
//       ||theta' - theta||_2 < tol -> stop, theta is NOT advanced                          (:479-480)
//       theta <- theta'                                                                    (:481)
//
// Design notes shared by the three tiers:
//  * The matrix is never rewritten. Column normalisation is idempotent after the first pass, so
//    F^(it>=1)_ij theta_j == alpha_ij * (theta_j / s_j): the kernels keep a scaled copy
//    th_j = theta_j / s_j in shared memory (th_j = theta_j during iteration 0) and stream raw alpha.
//  * One division per ROW (r_i = n_i / d_i), then u_ij = alpha_ij * th_j * r_i.
//  * No floating-point atomics anywhere. theta' is accumulated into accumulators that are PRIVATE to
//    the lane group that owns the row (a row's columns are distinct, so the lanes of one group never
//    collide) and then reduced over groups / CTAs in a fixed order -> results are bit-reproducible
//    run to run for a given plan.
//  * fp64 throughout.
#pragma once
#include <cooperative_groups.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace sbq {
namespace cg = cooperative_groups;

enum : int { LOCUS_OK = 0, LOCUS_ITER_CAP = 1, LOCUS_ZERO_DENOM = 2, LOCUS_NO_ROWS = 3 };

struct DevParams {
   // flat batch (see include/sbq.h, sbq_submit_flat)
   const int64_t* loc_row_off;
   const int64_t* loc_iso_off;
   const int64_t* row_ptr;
   const int32_t* col;
   const double* alpha;
   const int32_t* count;
   const int32_t* iso_len;
   // scratch: per-row effective count, -1 = row dropped by the row filter
   int32_t* neff;
   // scratch: per-non-zero transposed index (CSR position | local row << 16) for cluster-tier slices whose CSR
   // fits shared memory but whose CSC index does not
   unsigned* csc;
   // per-isoform outputs
   double* theta;
   double* fpkm;
   double* frac;
   int32_t* keep;
   // per-locus outputs
   int32_t* iters;
   int32_t* status;
   double* locus_fpkm;   // sum of FPKM over the isoforms the locus keeps
   // configuration
   int max_iter;
   double tol;
   double row_eps;
   double min_frac;
   int eff_len_norm;
   double insert_mean;
   double rpm;           // 1e6 / total_mapped_reads   (src/estimate.cpp:328)
};

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
   for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
   return v;
}
__device__ __forceinline__ long long warp_sum_ll(long long v) {
#pragma unroll
   for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
   return v;
}
template <int W>
__device__ __forceinline__ double group_sum(double v) {
#pragma unroll
   for (int o = W / 2; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
   return v;
}

// FPKM of one isoform (src/estimate.cpp:314-331). na = the effective_len_norm "NA" case.
__device__ __forceinline__ double iso_fpkm(const DevParams& p, double theta, int len, bool& na) {
   double kb;
   na = false;
   if (p.eff_len_norm) {
      kb = (double)len - p.insert_mean;
      if (kb < 0) { na = true; return 0.0; }
      kb = 1e3 / kb;
   } else {
      kb = 1e3 / (double)len;
   }
   return theta * p.rpm * kb;
}

template <int NT>
__device__ __forceinline__ double block_sum(double v, double* red) {
   // fixed shape: warp butterfly, then every thread adds the warp totals in warp order
   v = warp_sum(v);
   if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
   __syncthreads();
   double t = 0.0;
#pragma unroll
   for (int w = 0; w < NT / 32; ++w) t += red[w];
   __syncthreads();
   return t;
}

// FPKM / frac / keep tail of one locus (src/estimate.cpp:310-356), written by the NT threads of one CTA. cur: theta of the
// locus (ignored when the status resets it to theta0); na_scratch: T doubles of shared memory; red: block_sum's NT / 32 doubles.
template <int NT>
__device__ __forceinline__ void locus_epilogue_block(const DevParams& p, int l, int64_t t0, int T, int status, int iters, double theta0,
                                                     const double* cur, double* na_scratch, double* red) {
   const bool uniform = status == LOCUS_ZERO_DENOM || status == LOCUS_NO_ROWS;
   double fsum = 0.0;
   for (int j = threadIdx.x; j < T; j += NT) {
      const double tj = uniform ? theta0 : cur[j];
      bool na = false;
      double f = 0.0;
      if (status != LOCUS_NO_ROWS) f = iso_fpkm(p, tj, p.iso_len[t0 + j], na);
      p.theta[t0 + j] = tj;
      p.fpkm[t0 + j] = f;
      na_scratch[j] = na ? -1.0 : 0.0;   // remember NA
      fsum += f;
   }
   fsum = block_sum<NT>(fsum, red);
   double ksum = 0.0;
   for (int j = threadIdx.x; j < T; j += NT) {
      const bool na = na_scratch[j] < 0;
      const double f = p.fpkm[t0 + j];
      double fr = 0.0;
      int kp = 0;
      if (status != LOCUS_NO_ROWS) {
         if (!na) fr = f / fsum;
         kp = !(fr < p.min_frac) ? (na ? -1 : 1) : 0;
      }
      p.frac[t0 + j] = fr;
      p.keep[t0 + j] = kp;
      if (kp != 0) ksum += f;
   }
   ksum = block_sum<NT>(ksum, red);
   if (threadIdx.x == 0) {
      p.iters[l] = iters;
      p.status[l] = status;
      p.locus_fpkm[l] = ksum;
   }
}

// The same tail for a locus whose T <= 32 isoforms are owned one per lane of a warp; cur: this lane's theta.
__device__ __forceinline__ void locus_epilogue_warp(const DevParams& p, int l, int64_t t0, int T, int lane, int status, int iters, double theta0,
                                                    double cur) {
   const double theta_out = (status == LOCUS_ZERO_DENOM || status == LOCUS_NO_ROWS) ? theta0 : cur;
   bool na = false;
   double f = 0.0;
   if (lane < T && status != LOCUS_NO_ROWS) f = iso_fpkm(p, theta_out, p.iso_len[t0 + lane], na);
   const double sum = warp_sum(f);
   double fr = 0.0;
   int kp = 0;
   if (lane < T && status != LOCUS_NO_ROWS) {
      if (!na) fr = f / sum;
      kp = !(fr < p.min_frac) ? (na ? -1 : 1) : 0;
   }
   const double kept_sum = warp_sum(kp != 0 ? f : 0.0);
   if (lane < T) {
      p.theta[t0 + lane] = theta_out;
      p.fpkm[t0 + lane] = f;
      p.frac[t0 + lane] = fr;
      p.keep[t0 + lane] = kp;
   }
   if (lane == 0) {
      p.iters[l] = iters;
      p.status[l] = status;
      p.locus_fpkm[l] = kept_sum;
   }
}

// --------------------------------------------------------------------------------------------
// Tier 1: one warp per small locus (T <= 32). Lane i owns rows i, i+32, ...; lane j owns theta_j.
// Accumulators acc[j][lane] are lane-private (stride 33 doubles per column: conflict-free both for
// the lane-private updates and for the per-column fixed-order sum over lanes).
// --------------------------------------------------------------------------------------------
#ifdef SBQ_TRACE
// -DSBQ_TRACE build: every CTA leaves one record (class, threads, locus, rank, SM, start, end, iterations) in a device array
// that sbq_debug_trace() copies out - no printf, so the timeline is not distorted (tools/trace_timeline.py).
constexpr unsigned TRACE_CAP = 1u << 18;
__device__ unsigned long long g_trace[TRACE_CAP * 4];
__device__ unsigned g_trace_n;
__device__ __forceinline__ unsigned long long trace_now() { unsigned long long t; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t)); return t; }
__device__ __forceinline__ unsigned trace_smid() { unsigned s; asm volatile("mov.u32 %0, %%smid;" : "=r"(s)); return s; }
__device__ __forceinline__ void trace_emit(unsigned cs, unsigned nt, int locus, unsigned rank, unsigned long long t0, int iters) {
   const unsigned i = atomicAdd(&g_trace_n, 1u);
   if (i < TRACE_CAP) {
      g_trace[4 * i] = ((unsigned long long)cs << 48) | ((unsigned long long)nt << 32) | (unsigned)locus;
      g_trace[4 * i + 1] = ((unsigned long long)rank << 48) | ((unsigned long long)trace_smid() << 32) | (unsigned)iters;
      g_trace[4 * i + 2] = t0;
      g_trace[4 * i + 3] = trace_now();
   }
}
#endif
constexpr int WT_WARPS = 8;
constexpr int WT_MAX_ISO = 32;
constexpr int WT_MAX_ROWS = 64;    // planner: loci a warp still takes (a lane then walks two rows per iteration); measured: with 256 rows /
constexpr int WT_MAX_NNZ = 256;    // 1024 non-zeros the warp tier's longest locus takes 3.1 ms (8 rows per lane from L1/L2 every iteration)
constexpr int WT_STRIDE = 33;

__host__ __device__ inline size_t warp_tier_smem_bytes(int max_iso) {
   return (size_t)WT_WARPS * ((size_t)max_iso * WT_STRIDE + WT_MAX_ISO) * sizeof(double);
}

constexpr int WT_REG = 4;   // non-zeros per row a lane keeps in registers on the single-row fast path

// Persistent warps: every warp pulls the next locus from a global queue (list is sorted by descending
// non-zeros), so a long-running locus never holds back the other warps of its CTA.
__global__ void __launch_bounds__(WT_WARPS * 32)
em_warp_kernel(DevParams p, const int32_t* __restrict__ list, int n_list, int max_iso, int* queue) {
   extern __shared__ double smem[];
   const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
   double* acc = smem + (size_t)warp * ((size_t)max_iso * WT_STRIDE + WT_MAX_ISO);
   double* th = acc + (size_t)max_iso * WT_STRIDE;
   const int32_t* __restrict__ col = p.col;
   const double* __restrict__ al = p.alpha;
   const double tol2 = p.tol * p.tol;
#ifdef SBQ_TRACE
   const unsigned long long trace_t0 = trace_now();
#endif

   for (;;) {
      int w = 0;
      if (lane == 0) w = atomicAdd(queue, 1);
      w = __shfl_sync(0xffffffffu, w, 0);
      if (w >= n_list) {
#ifdef SBQ_TRACE
         if (threadIdx.x == 0) trace_emit(0, WT_WARPS * 32, -1, 0, trace_t0, 0);
#endif
         break;
      }
      const int l = list[w];
      const int64_t r0 = p.loc_row_off[l];
      const int R = (int)(p.loc_row_off[l + 1] - r0);
      const int64_t t0 = p.loc_iso_off[l];
      const int T = (int)(p.loc_iso_off[l + 1] - t0);
      const int64_t* __restrict__ rp = p.row_ptr + r0;
      int32_t* neff = p.neff + r0;

      for (int x = lane; x < T * WT_STRIDE; x += 32) acc[x] = 0.0;
      __syncwarp();

      // ---- setup: total, row filter, column sums over kept rows
      long long tot = 0;
      int kept = 0;
      int64_t my_k0 = 0;
      int my_cnt = 0, my_ne = -1;
      for (int i = lane; i < R; i += 32) {
         const int64_t k0 = rp[i], k1 = rp[i + 1];
         const int n = p.count[r0 + i];
         tot += n;
         bool keep = false;
         for (int64_t k = k0; k < k1; ++k) keep |= al[k] > p.row_eps;
         neff[i] = keep ? n : -1;
         if (keep) {
            ++kept;
            for (int64_t k = k0; k < k1; ++k) acc[col[k] * WT_STRIDE + lane] += al[k];
         }
         if (i == lane) { my_k0 = k0; my_cnt = (int)(k1 - k0); my_ne = keep ? n : -1; }
      }
      tot = warp_sum_ll(tot);
      kept = (int)warp_sum_ll(kept);
      __syncwarp();
      const int nl = R < 32 ? R : 32;   // lanes that own at least one row
      double s = 0.0;
      if (lane < T) {
         for (int x = 0; x < nl; ++x) { s += acc[lane * WT_STRIDE + x]; acc[lane * WT_STRIDE + x] = 0.0; }
      }
      // single-row fast path: one row per lane, at most WT_REG non-zeros each, held in registers
      const bool fast = R <= 32 && __all_sync(0xffffffffu, my_cnt <= WT_REG);
      double ra[WT_REG];
      int rc[WT_REG];
#pragma unroll
      for (int e = 0; e < WT_REG; ++e) {
         const bool v = fast && my_ne >= 0 && e < my_cnt;
         ra[e] = v ? al[my_k0 + e] : 0.0;
         rc[e] = v ? col[my_k0 + e] : 0;
      }
      const double theta0 = (double)tot / (double)T;
      double cur = theta0;
      int status = LOCUS_ITER_CAP, iters = 0;
      if (kept == 0) {
         status = LOCUS_NO_ROWS;
      } else {
         if (lane < T) th[lane] = cur;   // iteration 0 runs on raw alpha
         __syncwarp();
         for (int it = 0; it < p.max_iter; ++it) {
            iters = it + 1;
            bool zero = false;
            if (fast) {
               double t[WT_REG], d = 0.0;
#pragma unroll
               for (int e = 0; e < WT_REG; ++e) { t[e] = th[rc[e]]; d += ra[e] * t[e]; }
               if (my_ne >= 0) {
                  if (d == 0) {
                     zero = true;
                  } else {
                     const double r = (double)my_ne / d;
#pragma unroll
                     for (int e = 0; e < WT_REG; ++e)
                        if (ra[e] != 0.0) acc[rc[e] * WT_STRIDE + lane] += ra[e] * t[e] * r;
                  }
               }
            } else {
               for (int i = lane; i < R; i += 32) {
                  const int ne = neff[i];
                  if (ne < 0) continue;
                  const int64_t k0 = rp[i], k1 = rp[i + 1];
                  double d = 0.0;
                  for (int64_t k = k0; k < k1; ++k) d += al[k] * th[col[k]];
                  if (d == 0) {
                     zero = true;
                  } else {
                     const double r = (double)ne / d;
                     for (int64_t k = k0; k < k1; ++k) {
                        const int c = col[k];
                        acc[c * WT_STRIDE + lane] += al[k] * th[c] * r;
                     }
                  }
               }
            }
            if (__any_sync(0xffffffffu, zero)) { status = LOCUS_ZERO_DENOM; break; }
            __syncwarp();
            double nw = 0.0;
            if (lane < T) {
               double n0 = 0.0, n1 = 0.0;   // fixed two-way split of the sum over lanes (order does not depend on data)
               int x = 0;
               for (; x + 1 < nl; x += 2) {
                  n0 += acc[lane * WT_STRIDE + x];
                  n1 += acc[lane * WT_STRIDE + x + 1];
                  acc[lane * WT_STRIDE + x] = 0.0;
                  acc[lane * WT_STRIDE + x + 1] = 0.0;
               }
               if (x < nl) { n0 += acc[lane * WT_STRIDE + x]; acc[lane * WT_STRIDE + x] = 0.0; }
               nw = n0 + n1;
            }
            const double diff = lane < T ? nw - cur : 0.0;
            const double d2 = warp_sum(diff * diff);
            if (d2 < tol2) { status = LOCUS_OK; break; }   // ||theta' - theta||_2 < tol  (src/estimate.cpp:479-480)
            cur = nw;
            __syncwarp();
            if (lane < T) th[lane] = (s != 0) ? cur / s : 0.0;
            __syncwarp();
         }
      }

      // ---- outputs + epilogue (src/estimate.cpp:310-356)
      locus_epilogue_warp(p, l, t0, T, lane, status, iters, theta0, cur);
      __syncwarp();
   }
}

// --------------------------------------------------------------------------------------------
// Tier 2: one thread-block CLUSTER per locus (cluster size 1, 2, 4, 8 or 16 chosen by nnz).
// Rows are split over the CTAs of the cluster by non-zero count; inside a CTA, groups of LPR lanes
// own one row at a time and a private accumulator row acc[g][T] in shared memory. Per iteration:
// row pass -> fixed-order sum over groups -> partial theta' exchanged through distributed shared
// memory (one cluster barrier, double-buffered) -> every CTA forms the same theta' and norm.
// --------------------------------------------------------------------------------------------
constexpr int CL_NT = 512;           // threads per CTA of the cluster tier (small single-CTA loci use 64 or 128, see BUCKET_NT in sbq.cu)
constexpr int CL_LPR_STREAM = 32;    // lanes per row of the streaming fallback

// Exchange of the partial theta' inside a cluster, two forms. All-to-all: every CTA broadcasts its row of T partials to all peers and
// every CTA adds the CS rows itself - ONE blocking cluster barrier per iteration, but an exchange area of CS x T doubles. Owner form:
// column j is reduced by CTA j / B, which pushes the result back - two barriers, 3T remote stores, 2T doubles. A locus gets the
// all-to-all form when the CS x T partials are at most CL_A2A_MAX doubles AND its estimated slice, transposed index included, still
// fits next to them (the index of the largest loci spills to L2 as it is: they keep the small exchange area). A function of the
// locus alone (T, rows, non-zeros, CS), evaluated identically by the planner and the kernel.
constexpr int CL_A2A_MAX = 4096;
constexpr size_t CL_SMEM_CAP = 220 * 1024;   // dynamic shared memory a CTA asks for at most (227 KB usable, ~5.3 KB of them static)
__host__ __device__ inline int cluster_a2a_stride(int T) { return (T + 1) & ~1; }                 // rows of the exchange area are 16-byte aligned
__host__ __device__ inline bool cluster_a2a(int T, int cs, size_t slice_bytes) {
   if (cs <= 1 || (long long)cs * cluster_a2a_stride(T) > CL_A2A_MAX) return false;
   return ((size_t)4 * T + (size_t)cs * cluster_a2a_stride(T) + 64) * sizeof(double) + slice_bytes + 256 <= CL_SMEM_CAP;
}
// th, theta x2, s_j, exchange area ([CS][T] + 64 all-to-all, [2T+64] otherwise)
__host__ __device__ inline size_t cluster_fixed_doubles(int T, int cs, size_t slice_bytes) {
   return (size_t)4 * T + (cluster_a2a(T, cs, slice_bytes) ? (size_t)cs * cluster_a2a_stride(T) + 64 : (size_t)2 * T + 64);
}

// groups of the streaming fallback that fit next to the fixed arrays
__host__ __device__ inline int cluster_stream_groups(int T, size_t smem_bytes, int nt, int cs, size_t slice_bytes) {
   const long long budget = (long long)(smem_bytes / sizeof(double)) - (long long)cluster_fixed_doubles(T, cs, slice_bytes);
   long long G = budget / (T > 0 ? T : 1);
   if (G > nt / CL_LPR_STREAM) G = nt / CL_LPR_STREAM;
   return (int)G;   // 0 => does not fit
}
// bytes of one CTA's resident slice: row part (alpha, col, diagonal offsets, row lengths, counts, r) and the CSC index (pos, row)
__host__ __device__ inline int cluster_diag_slots(int T) { return (T + 7) & ~3; }   // diagonal offsets, read four at a time
__host__ __device__ inline size_t cluster_resident_csr_bytes(size_t nnz_c, size_t nrows, int T) {
   const size_t npos = nnz_c + (size_t)T;   // every diagonal may carry one padding slot (odd stride, see the kernel)
   return (npos + 1) * 8 + (nrows + 2) * 8 + (size_t)cluster_diag_slots(T) * 4 + nrows * 4 + ((size_t)T + 1) * 4 + nrows * 2 + npos * 2 + 64;
}
__host__ __device__ inline size_t cluster_resident_bytes(size_t nnz_c, size_t nrows, int T) {
   return cluster_resident_csr_bytes(nnz_c, nrows, T) + nnz_c * 4 + 4;
}

// Shared memory a cluster-tier CTA asks for, as a function of the LOCUS alone (T, estimated per-CTA slice, thread count):
// fixed arrays + the larger of (estimated largest resident slice, a full set of streaming accumulators). Host planner and
// kernel evaluate the same expression, so what a locus keeps resident - and with it the order of every sum - does not
// depend on which other loci share its launch: results are invariant under any partition of the loci over devices.
__host__ __device__ inline size_t cluster_class_smem(int max_iso, size_t slice_bytes, int nt, int cs) {
   const size_t fixed = cluster_fixed_doubles(max_iso, cs, slice_bytes) * sizeof(double);
   const size_t stream = (size_t)(nt / CL_LPR_STREAM) * max_iso * sizeof(double);
   const size_t want = fixed + (slice_bytes > stream ? slice_bytes : stream) + 256;
   return want < CL_SMEM_CAP ? want : CL_SMEM_CAP;
}
// per-CTA resident slice estimate with 12 % slack for the row-granular split
__host__ __device__ inline size_t cluster_slice_estimate(long long nnz, long long R, int T, int cs) {
   return (size_t)(1.12 * (double)cluster_resident_bytes((size_t)(nnz / cs + 1), (size_t)(R / cs + 1), T)) + 512;
}

// The path one CTA of em_cluster_kernel takes, from the locus (T, cluster size, slice estimate), the launch (threads, dynamic
// shared memory) and the CTA's own share of the rows (nrows, non-zeros nnz_c, whether a row is longer than T).
struct ClusterCtaPath {
   bool resident;       // the slice sits in shared memory (else it streams from L2 with G accumulator groups)
   bool csc_in_smem;    // ... with all of its CSC index; otherwise the first n_ent_s entries of the index, the rest in L2
   unsigned n_ent_s;
   int G;
   bool row_slots;      // balanced E-step (nrows <= NT), else four rows per thread
   bool col_slots;      // balanced M-step (T <= NT), else one thread per column
   bool a2a;            // all-to-all exchange, else the owner form with B columns per CTA
   int B;
};
__host__ __device__ inline ClusterCtaPath cluster_cta_path(int T, int cs, int nt, int nrows, unsigned nnz_c, bool too_long, size_t slice_est,
                                                           unsigned smem_launch) {
   ClusterCtaPath c;
   // this locus' own shared-memory budget (<= what the launch provides: the class maximum of the same expression)
   const size_t cls = cluster_class_smem(T, slice_est, nt, cs), smem_bytes = smem_launch < cls ? smem_launch : cls;
   const size_t used = cluster_fixed_doubles(T, cs, slice_est) * sizeof(double);
   const size_t csr = cluster_resident_csr_bytes(nnz_c, (size_t)nrows, T);
   // 16-bit positions and rows; the diagonal table has room for rows of up to T entries (a valid row has no more)
   const bool small_idx = (uint64_t)nnz_c + (uint64_t)T <= 65535u && nrows <= 65535 && !too_long;
   c.csc_in_smem = small_idx && used + cluster_resident_bytes(nnz_c, (size_t)nrows, T) <= smem_bytes;
   c.resident = small_idx && used + csr <= smem_bytes;
   c.n_ent_s = 0;
   if (c.csc_in_smem) c.n_ent_s = nnz_c;
   else if (c.resident) c.n_ent_s = (unsigned)(nnz_c < (smem_bytes - used - csr) / 4 ? nnz_c : (smem_bytes - used - csr) / 4);
   c.G = c.resident ? 0 : cluster_stream_groups(T, smem_bytes, nt, cs, slice_est);
   c.row_slots = c.resident && nrows <= nt;
   c.col_slots = c.resident && T <= nt;
   c.a2a = cluster_a2a(T, cs, slice_est);
   c.B = c.a2a ? cluster_a2a_stride(T) : (T + cs - 1) / cs;
   return c;
}

// Row accessor of one CTA's slice streamed from global/L2 (fallback when the slice does not fit shared memory).
struct GlobalRows {
   const int64_t* rp;      // row_ptr of the slice's first row
   const double* al;       // alpha + k_a
   const int32_t* col;     // col + k_a
   int32_t* ne;            // neff of the slice's first row
   int64_t k_a;
   __device__ __forceinline__ unsigned start(int i) const { return (unsigned)(rp[i] - k_a); }
   __device__ __forceinline__ double a(unsigned k) const { return al[k]; }
   __device__ __forceinline__ int c(unsigned k) const { return col[k]; }
   __device__ __forceinline__ int get_ne(int i) const { return ne[i]; }
   __device__ __forceinline__ void set_ne(int i, int v) const { ne[i] = v; }
};

// streaming fallback, setup pass: total count, row filter (-> ne), column sums of the kept rows
template <int LPR, typename Rows>
__device__ __forceinline__ void cluster_setup_pass(const Rows& rows, const int32_t* __restrict__ cnt, int nrows, int G, int g, int lg,
                                                   double row_eps, double* my_acc, long long& tot, int& kept) {
   for (int base = 0; base < nrows; base += G) {
      const int i = base + g;
      const bool valid = i < nrows;
      unsigned k0 = 0, k1 = 0;
      int n = 0;
      if (valid) { k0 = rows.start(i); k1 = rows.start(i + 1); n = cnt[i]; }
      bool keep = false;
      for (unsigned k = k0 + lg; k < k1; k += LPR) keep |= rows.a(k) > row_eps;
#pragma unroll
      for (int o = LPR / 2; o > 0; o >>= 1) keep |= (bool)__shfl_xor_sync(0xffffffffu, (int)keep, o);
      if (valid && lg == 0) { rows.set_ne(i, keep ? n : -1); tot += n; kept += keep; }
      if (keep)
         for (unsigned k = k0 + lg; k < k1; k += LPR) my_acc[rows.c(k)] += rows.a(k);
      __syncwarp();   // the next row of this group may touch the same accumulator column from another lane
   }
}

// streaming fallback, one E/M pass with the scaled theta in th[]; two rows per group in flight
template <int LPR, typename Rows>
__device__ __forceinline__ void cluster_em_pass(const Rows& rows, int nrows, int G, int g, int lg, const double* th, double* my_acc, int& zero) {
   for (int base = 0; base < nrows; base += 2 * G) {
      const int i0 = base + g, i1 = base + G + g;
      int ne0 = -1, ne1 = -1;
      unsigned a0 = 0, b0 = 0, a1 = 0, b1 = 0;
      if (i0 < nrows) { ne0 = rows.get_ne(i0); if (ne0 >= 0) { a0 = rows.start(i0); b0 = rows.start(i0 + 1); } }
      if (i1 < nrows) { ne1 = rows.get_ne(i1); if (ne1 >= 0) { a1 = rows.start(i1); b1 = rows.start(i1 + 1); } }
      double d0 = 0.0, d1 = 0.0;
      for (unsigned k = a0 + lg; k < b0; k += LPR) d0 += rows.a(k) * th[rows.c(k)];
      for (unsigned k = a1 + lg; k < b1; k += LPR) d1 += rows.a(k) * th[rows.c(k)];
#pragma unroll
      for (int o = LPR / 2; o > 0; o >>= 1) {
         d0 += __shfl_xor_sync(0xffffffffu, d0, o);
         d1 += __shfl_xor_sync(0xffffffffu, d1, o);
      }
      if (ne0 >= 0) {
         if (d0 == 0) zero = 1;
         else {
            const double r = (double)ne0 / d0;
            for (unsigned k = a0 + lg; k < b0; k += LPR) { const int c = rows.c(k); my_acc[c] += rows.a(k) * th[c] * r; }
         }
      }
      __syncwarp();   // row i1 of the same group may share columns with row i0
      if (ne1 >= 0) {
         if (d1 == 0) zero = 1;
         else {
            const double r = (double)ne1 / d1;
            for (unsigned k = a1 + lg; k < b1; k += LPR) { const int c = rows.c(k); my_acc[c] += rows.a(k) * th[c] * r; }
         }
      }
      __syncwarp();   // the next rows of this group may touch the same accumulator columns from other lanes
   }
}

// Resident slice of one CTA in shared memory. Rows are sorted by descending length and stored in jagged-diagonal
// order: element k of sorted row s lives at jd[k] + s, so that consecutive lanes (consecutive rows) read consecutive
// addresses - no padding and no bank conflicts for a thread-per-row E-step. A per-CTA transposed (CSC) index
// lists every column's entries for the M-step.
struct ResidentSlice {
   double* al;             // [npos+1]  alpha, jagged-diagonal order; al[npos] = 0 (padding target of the M-step)
   double* r;              // [nrows+1] per sorted row r_s = n_s / d_s of the current iteration (0 for dropped rows); r[nrows] = 0
   unsigned* jd;           // [jdn]     diagonal offsets (16-byte aligned, read four at a time)
   int* ne;                // [nrows]   n_s, or -1 for a dropped row
   unsigned* cp;           // [T+1]     column pointers into ent
   unsigned short* rlen;   // [nrows]   row lengths, descending
   unsigned short* col;    // [npos+1]  column of every entry, jagged-diagonal order; col[npos] = 0
   unsigned* ent;          // [n_ent_s] CSC order, sorted rows ascending within a column: position in al | sorted row << 16
   unsigned* ent_g;        //           entries n_ent_s.. of the index live in global scratch (L2) when shared memory is full
   unsigned n_ent_s;
   __device__ __forceinline__ unsigned get_ent(unsigned x) const { return x < n_ent_s ? ent[x] : ent_g[x]; }
   __device__ __forceinline__ void put_ent(unsigned x, unsigned v) const { if (x < n_ent_s) ent[x] = v; else ent_g[x] = v; }
   int nrows, T;
   unsigned nnz, npos;     // entries, and positions of al/col (entries + one padding slot per diagonal at most)
};

// E-step on the resident slice: d_s = sum_k alpha_k th[col_k]  ->  r_s = n_s / d_s   (one division per row).
// Generic form for slices with more rows than threads, one lane per row: four rows per thread at a time
// (rows tid, tid + NT, ... are sorted by descending length, so the first of the four is the longest).
template <int NT>
__device__ __forceinline__ void resident_e_pass_rows4(const ResidentSlice& S, const double* th, int& zero) {
   const int tid = threadIdx.x;
   for (int base = 0; base < S.nrows; base += 4 * NT) {
      int sv[4], ne[4], len[4];
      double d[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) {
         sv[u] = base + u * NT + tid;
         ne[u] = -1; len[u] = 0; d[u] = 0.0;
         if (sv[u] < S.nrows) {
            ne[u] = S.ne[sv[u]];
            if (ne[u] >= 0) len[u] = S.rlen[sv[u]];
         }
      }
      const int maxlen = max(max(len[0], len[1]), max(len[2], len[3]));
      for (int k = 0; k < maxlen; k += 4) {
         const uint4 o = *reinterpret_cast<const uint4*>(S.jd + k);
         const unsigned ov[4] = {o.x, o.y, o.z, o.w};
         double a[4][4];
         int c[4][4];
         // entries past the end of a row read the padding slot (alpha 0, column 0): plain loads, no divergence
#pragma unroll
         for (int u = 0; u < 4; ++u)
#pragma unroll
            for (int e = 0; e < 4; ++e) {
               const unsigned pos = k + e < len[u] ? ov[e] + (unsigned)sv[u] : S.npos;
               a[u][e] = S.al[pos];
               c[u][e] = (int)S.col[pos];
            }
#pragma unroll
         for (int u = 0; u < 4; ++u)
#pragma unroll
            for (int e = 0; e < 4; ++e) {
               const double t = a[u][e] * th[c[u][e]];
               d[u] += k + e < len[u] ? t : 0.0;
            }
      }
#pragma unroll
      for (int u = 0; u < 4; ++u) {
         if (sv[u] < S.nrows) {
            double r = 0.0;
            if (ne[u] >= 0) {
               if (d[u] == 0) zero = 1; else r = (double)ne[u] / d[u];
            }
            S.r[sv[u]] = r;
         }
      }
   }
}

// M-step on the resident slice through the CSC index: out_j = scale_j * sum_{k in column j} alpha_k r_row(k).
// Fixed lane assignment and summation order -> deterministic, no accumulators, no atomics.
// Generic form (any T): one thread per column, index entries read from memory eight at a time.
template <int NT, typename Emit>
__device__ __forceinline__ void resident_col_pass(const ResidentSlice& S, const double* scale, const Emit& emit) {
   const unsigned pad = ((unsigned)S.nrows << 16) | S.npos;
   for (int j = threadIdx.x; j < S.T; j += NT) {
      double sum = 0.0;
      const unsigned x1 = S.cp[j + 1];
      for (unsigned x = S.cp[j]; x < x1; x += 8) {
         unsigned e[8];
#pragma unroll
         for (int u = 0; u < 8; ++u) e[u] = (x + u < x1) ? S.get_ent(x + u) : pad;
#pragma unroll
         for (int u = 0; u < 8; ++u) sum += S.al[e[u] & 0xffffu] * S.r[e[u] >> 16];
      }
      *emit.ptr(j) = scale ? scale[j] * sum : sum;
   }
}

// Balanced form (items <= threads): every thread owns one (item, lane) slot for the whole solve. Rows and columns get
// a power-of-two number of lanes in proportion to their length, so that every lane walks about the same number of entries.
struct ColSlot {
   int j;                      // column, or -1 for an idle thread
   int q, lanes, wl;           // this thread is lane q of `lanes`; wl = largest group of the warp
   unsigned x0, x1;            // index entries of this lane: x0, x0 + lanes, ... < x1
   double* out;                // where lane 0 of the column stores the result
};
struct RowSlot {
   int s;                      // sorted row, or -1 for an idle thread
   int q, lanes, n;            // this thread is lane q of `lanes`; the lanes of a row are n threads apart (see assign_row_slots)
   int len;                    // entries of the row (0 for a dropped row)
   int ne;                     // n_s, or -1 for a dropped row
};

// Slots for n_items <= NT items of the given lengths: lanes_i = ceil(len_i / E) (1..32) with E the smallest target
// (in steps of 1/8) for which all lanes fit the CTA; the lanes of an item are consecutive threads of one warp.
// Returns this thread's slot: item | lane << 16 | lanes << 24, or 0xffffffff for an idle thread.
template <int NT>
__device__ __forceinline__ unsigned assign_slots(int n_items, int my_len, unsigned total_work, unsigned* s_slot, int* s_lanes, int* s_total) {
   const int tid = threadIdx.x;
   // sum_i ceil(len_i / E) ~ total / E + n_items / 2, and a little is lost at warp boundaries
   const int budget = max(NT / 4, NT - n_items / 2 - 16);
   int E = max(8, (int)((total_work + budget - 1) / budget));        // at least eight entries per lane: short reductions
   for (;;) {
      if (tid < n_items) s_lanes[tid] = min(32, max(1, (my_len + E - 1) / E));
      __syncthreads();
      if (tid == 0) {                         // greedy packing in item order; a group never straddles a warp
         int off = 0;
         for (int i0 = 0; i0 < n_items; i0 += 8) {
            int L[8];
#pragma unroll
            for (int u = 0; u < 8; ++u) L[u] = i0 + u < n_items ? s_lanes[i0 + u] : 0;
#pragma unroll
            for (int u = 0; u < 8; ++u) {
               if ((off & 31) + L[u] > 32) off = (off + 31) & ~31;
               const int o = off;
               off += L[u];
               L[u] = o | (L[u] << 16);
            }
#pragma unroll
            for (int u = 0; u < 8; ++u)
               if (i0 + u < n_items) s_lanes[i0 + u] = L[u];
         }
         *s_total = off;
      }
      __syncthreads();
      const int total = *s_total;
      if (total <= NT) break;
      __syncthreads();
      E += max(1, E >> 3);
   }
   s_slot[tid] = 0xffffffffu;
   __syncthreads();
   if (tid < n_items) {
      const int off = s_lanes[tid] & 0xffff, L = s_lanes[tid] >> 16;
      for (int q = 0; q < L; ++q) s_slot[off + q] = (unsigned)tid | ((unsigned)q << 16) | ((unsigned)L << 24);
   }
   __syncthreads();
   const unsigned sl = s_slot[tid];
   __syncthreads();
   return sl;
}

// Row slots (rows sorted by descending length, nrows <= NT): every warp serves n = 32 / L consecutive rows with L lanes
// each, L = the lanes its first (longest) row needs for the target E. Lane l of the warp is lane q = l / n of row
// first + l % n, so lanes with equal q read consecutive rows of one diagonal - consecutive shared-memory addresses.
// Returns first | n << 16 | L << 24 of this thread's warp (0xffffffff for an idle warp).
template <int NT>
__device__ __forceinline__ unsigned assign_row_slots(const unsigned short* rlen, int nrows, unsigned total_work, unsigned* s_winfo) {
   const int tid = threadIdx.x;
   if (tid < 32) {
      // lane c of warp 0 tries the target E0 * (1 + c / 8); the smallest target whose packing fits wins
      const int E0 = max(8, (int)((total_work + NT - 1) / NT));            // at least eight entries per lane: short reductions
      const int longest = nrows > 0 ? (int)rlen[0] : 1;
      int E = E0 + (E0 * tid + 7) / 8;
      if (tid == 31) E = max(E, longest);                   // one lane per row always fits (nrows <= NT)
      int first = 0;
      for (int w = 0; w < NT / 32 && first < nrows; ++w) first += 32 / min(32, max(1, ((int)rlen[first] + E - 1) / E));
      const unsigned fits = __ballot_sync(0xffffffffu, first >= nrows);
      if (tid == __ffs(fits) - 1) {
         int f = 0, w = 0;
         for (; w < NT / 32 && f < nrows; ++w) {
            const int L = min(32, max(1, ((int)rlen[f] + E - 1) / E));
            const int n = 32 / L;
            s_winfo[w] = (unsigned)f | ((unsigned)n << 16) | ((unsigned)L << 24);
            f += n;
         }
         for (; w < NT / 32; ++w) s_winfo[w] = 0xffffffffu;
      }
   }
   __syncthreads();
   const unsigned info = s_winfo[tid >> 5];
   __syncthreads();
   return info;
}

// fixed-shape sum over the lanes of a row (n threads apart, lane 0 of the row holds the result)
__device__ __forceinline__ double row_sum(double v, int q, int lanes, int n) {
   for (int o = 1; o < lanes; o <<= 1) {        // lanes is warp-uniform
      const double u = __shfl_down_sync(0xffffffffu, v, o * n);
      if (q + o < lanes) v += u;
   }
   return v;
}

// fixed-shape sum over the lanes of a slot group (consecutive lanes of one warp); lane 0 of the group holds the result.
// wl = the largest group of this warp (warp-uniform), so warps of single-lane groups do not shuffle at all
__device__ __forceinline__ double group_sum(double v, int q, int lanes, int wl) {
   for (int o = 1; o < wl; o <<= 1) {
      const double u = __shfl_down_sync(0xffffffffu, v, o);
      if (q + o < lanes) v += u;
   }
   return v;
}

// E-step, balanced form: the lanes of a row take its entries in interleaved groups of four.
__device__ __forceinline__ void slot_e_pass(const ResidentSlice& S, const RowSlot& rs, const double* th, int& zero) {
   const unsigned s = (unsigned)max(rs.s, 0);
   const int len = rs.len, step = 4 * rs.lanes;
   double d0 = 0.0, d1 = 0.0;
   int k = 4 * rs.q;
   // eight entries per trip while two full groups of four remain (sixteen loads in flight per lane)
   for (; k + step + 4 <= len; k += 2 * step) {
      const uint4 o = *reinterpret_cast<const uint4*>(S.jd + k);
      const uint4 q = *reinterpret_cast<const uint4*>(S.jd + k + step);
      const unsigned p0 = o.x + s, p1 = o.y + s, p2 = o.z + s, p3 = o.w + s;
      const unsigned p4 = q.x + s, p5 = q.y + s, p6 = q.z + s, p7 = q.w + s;
      const int c0 = S.col[p0], c1 = S.col[p1], c2 = S.col[p2], c3 = S.col[p3];
      const int c4 = S.col[p4], c5 = S.col[p5], c6 = S.col[p6], c7 = S.col[p7];
      const double a0 = S.al[p0], a1 = S.al[p1], a2 = S.al[p2], a3 = S.al[p3];
      const double a4 = S.al[p4], a5 = S.al[p5], a6 = S.al[p6], a7 = S.al[p7];
      const double t0 = th[c0], t1 = th[c1], t2 = th[c2], t3 = th[c3];
      const double t4 = th[c4], t5 = th[c5], t6 = th[c6], t7 = th[c7];
      d0 += a0 * t0;
      d1 += a1 * t1;
      d0 += a2 * t2;
      d1 += a3 * t3;
      d0 += a4 * t4;
      d1 += a5 * t5;
      d0 += a6 * t6;
      d1 += a7 * t7;
   }
   for (; k < len; k += step) {                       // last groups: entries past the end read the padding slot
      const uint4 o = *reinterpret_cast<const uint4*>(S.jd + k);
      const bool v1 = k + 1 < len, v2 = k + 2 < len, v3 = k + 3 < len;
      const unsigned p0 = o.x + s, p1 = v1 ? o.y + s : S.npos, p2 = v2 ? o.z + s : S.npos, p3 = v3 ? o.w + s : S.npos;
      const double a0 = S.al[p0], a1 = S.al[p1], a2 = S.al[p2], a3 = S.al[p3];
      const int c0 = S.col[p0], c1 = S.col[p1], c2 = S.col[p2], c3 = S.col[p3];
      const double t0 = a0 * th[c0], t1 = a1 * th[c1], t2 = a2 * th[c2], t3 = a3 * th[c3];
      d0 += t0;
      d1 += v1 ? t1 : 0.0;
      d0 += v2 ? t2 : 0.0;
      d1 += v3 ? t3 : 0.0;
   }
   const double d = row_sum(d0 + d1, rs.q, rs.lanes, rs.n);
   if (rs.s >= 0 && rs.q == 0) {
      double r = 0.0;
      if (rs.ne >= 0) {
         if (d == 0) zero = 1; else r = (double)rs.ne / d;
      }
      S.r[s] = r;
   }
}

__device__ __forceinline__ void slot_col_pass(const ResidentSlice& S, const ColSlot& cs, const double* scale) {
   double s0 = 0.0, s1 = 0.0;
   const unsigned pad = ((unsigned)S.nrows << 16) | S.npos;
   for (unsigned x = cs.x0; x < cs.x1; x += 8 * cs.lanes) {
      unsigned e[8];
#pragma unroll
      for (int u = 0; u < 8; ++u) e[u] = (x + u * cs.lanes < cs.x1) ? S.get_ent(x + u * cs.lanes) : pad;
      double a[8], r[8];
#pragma unroll
      for (int u = 0; u < 8; ++u) { a[u] = S.al[e[u] & 0xffffu]; r[u] = S.r[e[u] >> 16]; }
#pragma unroll
      for (int u = 0; u < 8; u += 2) {
         s0 += a[u] * r[u];
         s1 += a[u + 1] * r[u + 1];
      }
   }
   const double sum = group_sum(s0 + s1, cs.q, cs.lanes, cs.wl);
   if (cs.j >= 0 && cs.q == 0) *cs.out = scale ? scale[cs.j] * sum : sum;
}

// split cluster barrier (all threads of every CTA execute them, convergently)
__device__ __forceinline__ void cluster_arrive_release() { asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory"); }
__device__ __forceinline__ void cluster_arrive_relaxed() { asm volatile("barrier.cluster.arrive.relaxed.aligned;" ::: "memory"); }
__device__ __forceinline__ void cluster_wait() { asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory"); }

// Where the partial theta'_j of this CTA goes: column j is owned by CTA j / B of the cluster, which keeps one
// row of B partials per peer in its exchange area (written through distributed shared memory).
struct OwnerMap {
   cg::cluster_group* cluster;
   double* stage;     // [CS][B] in every CTA
   int B;
   unsigned rank, CS;
   __device__ __forceinline__ double* ptr(int j) const {
      const int o = j / B;
      double* base = CS > 1 ? cluster->map_shared_rank(stage, (unsigned)o) : stage;
      return base + (size_t)rank * B + (j - o * B);
   }
};
struct LocalOut {
   double* out;
   __device__ __forceinline__ double* ptr(int j) const { return out + j; }
};

// NT = 64 / 128 / 512 threads: eight / four / one CTA per SM (the register cap follows from it)
template <int NT>
__global__ void __launch_bounds__(NT, CL_NT / NT)
em_cluster_kernel(DevParams p, const int32_t* __restrict__ list, int n_list, unsigned smem_launch) {
   cg::cluster_group cluster = cg::this_cluster();
   const unsigned CS = cluster.num_blocks();
   const unsigned rank = cluster.block_rank();
   const int item = blockIdx.x / CS;
   const int l = list[item];
   const int tid = threadIdx.x, lane = tid & 31;
#ifdef SBQ_TRACE
   const unsigned long long trace_t0 = trace_now();
#endif

   const int64_t r0 = p.loc_row_off[l];
   const int R = (int)(p.loc_row_off[l + 1] - r0);
   const int64_t t0 = p.loc_iso_off[l];
   const int T = (int)(p.loc_iso_off[l + 1] - t0);

   extern __shared__ double smem[];
   double* th = smem;                  // [T] scaled theta used by the passes
   double* bufA = th + T;              // [T] theta (current / next, swapped by pointer)
   double* bufB = bufA + T;            // [T]
   double* sdiv = bufB + T;            // [T] column sums s_j of the kept rows
   double* part = sdiv + T;            // exchange area: stage [CS][B] of partial theta', dsq [B], flags [16], d2p [16] - or [CS][T] + 64 (all-to-all)
   const int64_t* __restrict__ rp = p.row_ptr + r0;
   const size_t slice_est = cluster_slice_estimate((long long)(rp[R] - rp[0]), R, T, (int)CS);
   double* dyn = smem + cluster_fixed_doubles(T, (int)CS, slice_est);    // resident slice, or the streaming accumulators
   __shared__ double red[NT / 32];
   __shared__ int s_rows[2];
   double* cur = bufA;
   double* nxt = bufB;

   // rows of this CTA: split by non-zeros (lower_bound on row_ptr)
   if (tid < 2) {
      const int64_t base = rp[0], nnz = rp[R] - base;
      const int64_t target = base + (nnz * (int64_t)(rank + tid)) / CS;
      int lo = 0, hi = R;
      if (rank + tid >= CS) lo = R;
      else if (rank + tid == 0) hi = 0;
      while (lo < hi) {
         const int mid = (lo + hi) >> 1;
         if (rp[mid] < target) lo = mid + 1; else hi = mid;
      }
      s_rows[tid] = lo;
   }
   __syncthreads();
   const int ra = s_rows[0], rb = s_rows[1], nrows = rb - ra;
   const int64_t k_a = rp[ra];
   const unsigned nnz_c = (unsigned)(rp[rb] - k_a);

   // longest row of the slice: the diagonal table has room for rows of up to T entries (a valid row has no more)
   int too_long = 0;
   for (int i = tid; i < nrows; i += NT) too_long |= (rp[ra + i + 1] - rp[ra + i]) > (int64_t)T;
   too_long = __syncthreads_or(too_long);
   const ClusterCtaPath path = cluster_cta_path(T, (int)CS, NT, nrows, nnz_c, too_long != 0, slice_est, smem_launch);
   const unsigned npos = nnz_c + (unsigned)T;
   const int jdn = cluster_diag_slots(T);
   ResidentSlice S;
   S.al = dyn;
   S.r = S.al + npos + 1;
   S.jd = (unsigned*)(S.r + nrows + 1 + ((npos + nrows) & 1u));                             // 16-byte aligned
   S.ne = (int*)(S.jd + jdn);
   S.cp = (unsigned*)(S.ne + nrows);
   S.rlen = (unsigned short*)(S.cp + T + 1);
   S.col = S.rlen + nrows;
   S.ent = (unsigned*)(S.col + npos + 1 + ((npos + 1 + nrows) & 1u));                        // 4-byte aligned
   S.ent_g = p.csc + (size_t)k_a;      // the part of the CSC index that does not fit shared memory lives in global scratch (L2)
   S.n_ent_s = path.n_ent_s;
   S.nrows = nrows; S.T = T; S.nnz = nnz_c; S.npos = npos;
   GlobalRows grows{rp + ra, p.alpha + k_a, p.col + k_a, p.neff + r0 + ra, k_a};
   const int G = path.G;
   double* acc = dyn;                                           // [G][T] (streaming only)
   const int g32 = tid / CL_LPR_STREAM, lg32 = tid % CL_LPR_STREAM;
   double* my_acc = acc + (size_t)(g32 < G ? g32 : 0) * T;
   ColSlot slot;
   slot.j = -1; slot.q = 0; slot.lanes = 1; slot.wl = 1; slot.x0 = slot.x1 = 0; slot.out = part;
   RowSlot rslot;
   rslot.s = -1; rslot.q = 0; rslot.lanes = 1; rslot.n = 1; rslot.len = 0; rslot.ne = -1;

#ifdef SBQ_PHASE_TIMING
   long long ph[8] = {0, 0, 0, 0, 0, 0, 0, 0};
#define SBQ_TICK(k) { const long long t_ = clock64(); ph[k] += t_ - t_prev; t_prev = t_; }
#define SBQ_STICK(k) { const long long t_ = clock64(); st[k] += t_ - t_prev; t_prev = t_; }
   long long st[8] = {0, 0, 0, 0, 0, 0, 0, 0};
   long long t_prev = clock64();
   const long long t_start = t_prev;
#else
#define SBQ_TICK(k)
#define SBQ_STICK(k)
#endif
   long long tot = 0;
   int kept = 0;
   if (path.resident) {
      // ---- rows sorted by descending length (ties by row index): bitonic sort of (65535 - len) << 16 | row
      unsigned* keys = (unsigned*)S.al;                                    // scratch: alpha is loaded afterwards
      int P = 1;
      while (P < nrows) P <<= 1;
      for (int i = tid; i < P; i += NT)
         keys[i] = i < nrows ? ((65535u - (unsigned)(rp[ra + i + 1] - rp[ra + i])) << 16) | (unsigned)i : 0xffffffffu;
      __syncthreads();
      for (int kk = 2; kk <= P; kk <<= 1) {
         for (int jj = kk >> 1; jj > 0; jj >>= 1) {
            for (int i = tid; i < P; i += NT) {
               const int x = i ^ jj;
               if (x > i) {
                  const unsigned a = keys[i], b = keys[x];
                  if (((i & kk) == 0) ? (a > b) : (a < b)) { keys[i] = b; keys[x] = a; }
               }
            }
            __syncthreads();
         }
      }
      SBQ_STICK(0)
      for (int i = tid; i < nrows; i += NT) {
         const unsigned key = keys[i];
         S.rlen[i] = (unsigned short)(65535u - (key >> 16));
         S.ne[i] = (int)(key & 0xffffu);                                   // original row, until the fill replaces it by n_s
      }
      for (int j = tid; j <= T; j += NT) S.cp[j] = 0;
      __syncthreads();
      // ---- diagonal offsets: diagonal k holds the rows longer than k (a prefix of the sorted rows)
      for (int k = tid; k < jdn; k += NT) {
         unsigned v = 0;
         if (k > 0) {
            int lo = 0, hi = nrows;                                        // first sorted row with rlen <= k - 1
            while (lo < hi) {
               const int mid = (lo + hi) >> 1;
               if ((int)S.rlen[mid] > k - 1) lo = mid + 1; else hi = mid;
            }
            v = (unsigned)lo | (lo > 0 ? 1u : 0u);                         // odd stride: neighbouring diagonals fall into different banks
         }
         S.jd[k] = v;
      }
      __syncthreads();
      if (tid < 32) {                                                      // inclusive scan over jdn (warp 0)
         const int chunk = (jdn + 31) / 32, k0 = lane * chunk, k1 = min(jdn, k0 + chunk);
         unsigned sum = 0;
         for (int k = k0; k < k1; ++k) sum += S.jd[k];
         unsigned incl = sum;
         for (int o = 1; o < 32; o <<= 1) {
            const unsigned v = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl += v;
         }
         unsigned run = incl - sum;
         for (int k = k0; k < k1; ++k) { run += S.jd[k]; S.jd[k] = run; }
      }
      __syncthreads();
      SBQ_STICK(1)
      // ---- load the slice, row filter, column counts: lf lanes per row
      {
         const int32_t* __restrict__ cnt = p.count + r0 + ra;
         int lf = 1;
         while (lf < 32 && (long long)lf * nrows < (long long)nnz_c) lf <<= 1;      // ~ mean row length
         const int g = tid / lf, lg = tid % lf, par = NT / lf;
         // two rows per trip, the first four chunks of each fetched before anything is stored (eight loads in flight)
         for (int base = 0; base < nrows; base += 2 * par) {
            int sv[2], iv[2], lenv[2], keepv[2];
            unsigned g0v[2];
            double a[2][4];
            int c[2][4];
#pragma unroll
            for (int r = 0; r < 2; ++r) {
               sv[r] = base + r * par + g;
               iv[r] = 0; lenv[r] = 0; g0v[r] = 0; keepv[r] = 0;
               if (sv[r] < nrows) {
                  iv[r] = S.ne[sv[r]];
                  lenv[r] = S.rlen[sv[r]];
               }
            }
#pragma unroll
            for (int r = 0; r < 2; ++r)
               if (sv[r] < nrows) g0v[r] = (unsigned)(rp[ra + iv[r]] - k_a);
#pragma unroll
            for (int r = 0; r < 2; ++r)
#pragma unroll
               for (int u = 0; u < 4; ++u) {
                  const int k = lg + u * lf;
                  a[r][u] = 0.0; c[r][u] = 0;
                  if (k < lenv[r]) { a[r][u] = grows.al[g0v[r] + k]; c[r][u] = grows.col[g0v[r] + k]; }
               }
#pragma unroll
            for (int r = 0; r < 2; ++r) {
#pragma unroll
               for (int u = 0; u < 4; ++u) {
                  const int k = lg + u * lf;
                  if (k < lenv[r]) {
                     const unsigned pos = S.jd[k] + sv[r];
                     S.al[pos] = a[r][u];
                     S.col[pos] = (unsigned short)c[r][u];
                     keepv[r] |= a[r][u] > p.row_eps;
                     atomicAdd(&S.cp[c[r][u] + 1], 1u);                               // column counts (integers: exact)
                  }
               }
               for (int k = lg + 4 * lf; k < lenv[r]; k += lf) {
                  const double av = grows.al[g0v[r] + k];
                  const int cv = grows.col[g0v[r] + k];
                  const unsigned pos = S.jd[k] + sv[r];
                  S.al[pos] = av;
                  S.col[pos] = (unsigned short)cv;
                  keepv[r] |= av > p.row_eps;
                  atomicAdd(&S.cp[cv + 1], 1u);
               }
            }
            __syncwarp();   // every lane of a group has read the row's original index before lane 0 replaces it by n_s
#pragma unroll
            for (int r = 0; r < 2; ++r) {
               int keep = keepv[r];
               for (int o = lf >> 1; o > 0; o >>= 1) keep |= __shfl_xor_sync(0xffffffffu, keep, o);
               if (sv[r] < nrows && lg == 0) {
                  const int n = cnt[iv[r]];
                  S.ne[sv[r]] = keep ? n : -1;
                  S.r[sv[r]] = keep ? 1.0 : 0.0;
                  tot += n;
                  kept += keep;
               }
            }
         }
         if (tid == 0) { S.al[npos] = 0.0; S.col[npos] = 0; S.r[nrows] = 0.0; }
      }
      __syncthreads();
      if (tid < 32) {                                                                        // exclusive scan over T (warp 0)
         const int chunk = (T + 31) / 32, j0 = lane * chunk, j1 = min(T, j0 + chunk);
         unsigned sum = 0;
         for (int j = j0; j < j1; ++j) sum += S.cp[j + 1];
         unsigned incl = sum;
         for (int o = 1; o < 32; o <<= 1) {
            const unsigned v = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl += v;
         }
         unsigned run = incl - sum;
         for (int j = j0; j < j1; ++j) { const unsigned c = S.cp[j + 1]; S.cp[j + 1] = run + c; run += c; }
      }
      __syncthreads();
      SBQ_STICK(2)
      // ordered fill: a warp owns a chunk of up to 32 neighbouring columns (lane i keeps the write pointer of column
      // jlo + i) and walks the sorted rows 32 at a time, every lane with a cursor into its own row (columns ascend
      // within a row). Every column lists its entries by ascending sorted row; no atomics, fixed order.
      {
         const int nw = NT / 32, w = tid >> 5;
         const int C = min(32, (T + nw - 1) / nw);
         const int nchunks = (T + C - 1) / C;
         const unsigned lt = (1u << lane) - 1u;
         for (int ch = w; ch < nchunks; ch += nw) {
            const int jlo = ch * C, jn = min(C, T - jlo);
            unsigned wp = lane < jn ? S.cp[jlo + lane] : 0u;
            for (int base = 0; base < nrows; base += 32) {
               const int s = base + lane;
               int len = 0, cur = 0;
               if (s < nrows) {
                  len = S.rlen[s];
                  int lo = 0, hi = len;                       // first entry of the row with column >= jlo
                  while (lo < hi) {
                     const int mid = (lo + hi) >> 1;
                     if ((int)S.col[S.jd[mid] + s] < jlo) lo = mid + 1; else hi = mid;
                  }
                  cur = lo;
               }
               unsigned pos = 0;
               int nextc = -1;
               if (cur < len) { pos = S.jd[cur] + s; nextc = S.col[pos]; }
               if (__ballot_sync(0xffffffffu, nextc >= 0 && nextc < jlo + jn) == 0u) continue;
               for (int jj = 0; jj < jn; ++jj) {
                  const bool hit = nextc == jlo + jj;
                  const unsigned m = __ballot_sync(0xffffffffu, hit);
                  const unsigned basep = __shfl_sync(0xffffffffu, wp, jj);
                  if (hit) {
                     S.put_ent(basep + __popc(m & lt), pos | ((unsigned)s << 16));
                     ++cur;
                     nextc = -1;
                     if (cur < len) { pos = S.jd[cur] + s; nextc = S.col[pos]; }
                  }
                  if (lane == jj) wp += __popc(m);
               }
            }
         }
      }
      __syncthreads();
      SBQ_STICK(3)
      // ---- balanced slots (rows for the E-step, columns for the M-step)
      __shared__ unsigned s_slot[NT];
      __shared__ int s_lanes[NT];
      __shared__ int s_total;
      if (path.row_slots) {
         const unsigned info = assign_row_slots<NT>(S.rlen, nrows, nnz_c, s_slot);
         if (info != 0xffffffffu) {
            const int first = (int)(info & 0xffffu), n = (int)((info >> 16) & 0xffu), L = (int)(info >> 24);
            rslot.lanes = L;
            rslot.n = n;
            rslot.q = lane / n;
            const int row = first + lane % n;
            if (rslot.q < L && row < nrows) {
               rslot.s = row;
               rslot.ne = S.ne[row];
               rslot.len = rslot.ne >= 0 ? (int)S.rlen[row] : 0;
            } else {
               rslot.q = L;                    // idle lane: never adds, never stores
            }
         }
      }
      SBQ_STICK(4)
      if (path.col_slots) {
         const int len_j = tid < T ? (int)(S.cp[tid + 1] - S.cp[tid]) : 0;
         const unsigned sl = assign_slots<NT>(T, len_j, nnz_c, s_slot, s_lanes, &s_total);
         if (sl != 0xffffffffu) {
            slot.j = (int)(sl & 0xffffu);
            slot.lanes = (int)(sl >> 24);
            slot.q = (int)((sl >> 16) & 0xffu);
            slot.x0 = S.cp[slot.j] + (unsigned)slot.q;
            slot.x1 = S.cp[slot.j + 1];
            slot.out = part + slot.j;
         }
         slot.wl = __reduce_max_sync(0xffffffffu, slot.lanes);
         SBQ_STICK(5)
         slot_col_pass(S, slot, nullptr);                                                     // s_j partial (r = keep flag)
      } else {
         resident_col_pass<NT>(S, nullptr, LocalOut{part});
      }
   } else {
      for (int x = tid; x < G * T; x += NT) acc[x] = 0.0;
      __syncthreads();
      if (g32 < G) cluster_setup_pass<CL_LPR_STREAM>(grows, p.count + r0 + ra, nrows, G, g32, lg32, p.row_eps, my_acc, tot, kept);
      __syncthreads();
      for (int j = tid; j < T; j += NT) {
         double sj = 0.0;
         for (int gg = 0; gg < G; ++gg) { sj += acc[(size_t)gg * T + j]; acc[(size_t)gg * T + j] = 0.0; }
         part[j] = sj;
      }
   }
   {
      const double tot_b = block_sum<NT>((double)tot, red);
      const double kept_b = block_sum<NT>((double)kept, red);
      if (tid == 0) { part[T + 1] = tot_b; part[T + 2] = kept_b; }
   }
   cluster.sync();
   double total = 0.0, kept_all = 0.0;
   for (unsigned r = 0; r < CS; ++r) {
      const double* rp_part = CS > 1 ? cluster.map_shared_rank(part, r) : part;
      total += rp_part[T + 1];
      kept_all += rp_part[T + 2];
   }
   for (int j = tid; j < T; j += NT) {
      double sj = 0.0;
      for (unsigned r = 0; r < CS; ++r) {
         const double* rp_part = CS > 1 ? cluster.map_shared_rank(part, r) : part;
         sj += rp_part[j];
      }
      sdiv[j] = sj;
   }
   const double theta0 = total / (double)T;
   for (int j = tid; j < T; j += NT) { cur[j] = theta0; th[j] = theta0; }
   cluster.sync();   // everyone has read part[0] before it is reused; th/cur visible CTA-wide

   const double tol2 = p.tol * p.tol;
   int status = LOCUS_ITER_CAP, iters = 0;
#ifdef SBQ_PHASE_TIMING
   const long long t_setup = clock64() - t_start;
   t_prev = clock64();
#endif
   // ---- exchange area: column j belongs to CTA j / B; every CTA pushes its partial theta'_j to the owner, the owner
   //      adds the CS partials in a fixed shape and pushes theta'_j and theta'_j / s_j back to everyone
   const bool a2a = path.a2a;
   const int Tp = cluster_a2a_stride(T);
   const int B = path.B;
   double* stage = part;                       // [CS][B]; all-to-all: [CS][Tp], row r = the partials of CTA r
   double* dsq = a2a ? part + (size_t)CS * Tp : part + T + 16;            // [B] squared changes of the owned columns ([NT / 32] per-warp sums)
   double* flags = a2a ? dsq + 16 : part + 2 * T + 32;                    // [CS] zero-denominator flag of every CTA
   double* d2p = flags + 16;                   // [CS] partial ||theta' - theta||^2 of every owner
   // all-to-all: the passes write this CTA's own row; owner form: column j goes to CTA j / B
   const OwnerMap own{&cluster, a2a ? stage + (size_t)rank * Tp : stage, a2a ? T : B, a2a ? 0u : rank, a2a ? 1u : CS};
   if (slot.j >= 0) slot.out = own.ptr(slot.j);
   const int nb = max(0, min(B, T - (int)rank * B));      // columns this CTA owns
   bool pend_b = false;                        // all-to-all: arrived at the "stage has been read" barrier, not yet waited
   if (kept_all == 0) {
      status = LOCUS_NO_ROWS;
   } else {
      for (int it = 0; it < p.max_iter; ++it) {
         iters = it + 1;
         int zero = 0;
         if (path.resident) {
            if (path.row_slots) slot_e_pass(S, rslot, th, zero);
            else resident_e_pass_rows4<NT>(S, th, zero);
            SBQ_TICK(0)
            zero = __syncthreads_or(zero);
            SBQ_TICK(1)
            if (path.col_slots) slot_col_pass(S, slot, th);
            else resident_col_pass<NT>(S, th, own);
            SBQ_TICK(2)
         } else {
            if (g32 < G) cluster_em_pass<CL_LPR_STREAM>(grows, nrows, G, g32, lg32, th, my_acc, zero);
            zero = __syncthreads_or(zero);
            for (int j = tid; j < T; j += NT) {
               double sj = 0.0;
               for (int gg = 0; gg < G; ++gg) { sj += acc[(size_t)gg * T + j]; acc[(size_t)gg * T + j] = 0.0; }
               *own.ptr(j) = sj;
            }
         }
         double d2 = 0.0;
         if (CS == 1) {
            // single CTA: theta' is the stage row itself; one division per column, ||theta' - theta||^2 by warp
            __syncthreads();
            SBQ_TICK(3)
            if (zero) { status = LOCUS_ZERO_DENOM; break; }
            double dd = 0.0;
            for (int j = tid; j < T; j += NT) {
               const double v = stage[j], sj = sdiv[j];
               nxt[j] = v;
               th[j] = (sj != 0) ? v / sj : 0.0;
               const double diff = v - cur[j];
               dd += diff * diff;
            }
            if ((tid & ~31) < T) dd = warp_sum(dd);            // warps without columns hold 0 already
            if (lane == 0) dsq[tid >> 5] = dd;
            SBQ_TICK(4)
            __syncthreads();
            SBQ_TICK(6)
#pragma unroll
            for (int w = 0; w < NT / 32; ++w) d2 += dsq[w];      // same order in every thread
         } else if (a2a) {
            __syncthreads();                                     // this CTA's row of partials is complete
            if (pend_b) { cluster_wait(); pend_b = false; }      // every peer has finished reading the previous iteration's rows
            {
               // broadcast the row (and the zero-denominator flag) to the CS - 1 peers: coalesced 16-byte remote stores
               const int half = Tp >> 1, items = ((int)CS - 1) * half;
               const double2* mine = reinterpret_cast<const double2*>(stage + (size_t)rank * Tp);
               for (int x = tid; x < items; x += NT) {
                  const int pr = x / half, jj = x - pr * half;
                  const unsigned peer = (rank + 1u + (unsigned)pr) & (CS - 1u);
                  reinterpret_cast<double2*>(cluster.map_shared_rank(stage, peer) + (size_t)rank * Tp)[jj] = mine[jj];
               }
               if (tid < (int)CS) cluster.map_shared_rank(flags, (unsigned)tid)[rank] = (double)zero;
            }
            SBQ_TICK(3)
            cluster_arrive_release();
            cluster_wait();
            SBQ_TICK(4)
            double zf = 0.0;
            for (unsigned r = 0; r < CS; ++r) zf += flags[r];
            if (zf != 0.0) { status = LOCUS_ZERO_DENOM; break; }
            // every CTA adds the CS rows itself, in the shape of a butterfly over CS lanes (the association of the owner form)
            double dd = 0.0;
            for (int j = tid; j < T; j += NT) {
               double a[16];
#pragma unroll
               for (int r = 0; r < 16; ++r) a[r] = r < (int)CS ? stage[(size_t)r * Tp + j] : 0.0;
#pragma unroll
               for (int o = 8; o > 0; o >>= 1)
#pragma unroll
                  for (int r = 0; r < o; ++r) a[r] += a[r + o];
               const double v = a[0], sj = sdiv[j];
               nxt[j] = v;
               th[j] = (sj != 0) ? v / sj : 0.0;
               const double diff = v - cur[j];
               dd += diff * diff;
            }
            if ((tid & ~31) < T) dd = warp_sum(dd);              // warps without columns hold 0 already
            if (lane == 0) dsq[tid >> 5] = dd;
            SBQ_TICK(5)
            __syncthreads();
            cluster_arrive_relaxed();                            // done reading the rows and the flags (waited for before the next broadcast)
            pend_b = true;
            SBQ_TICK(6)
#pragma unroll
            for (int w = 0; w < NT / 32; ++w) d2 += dsq[w];      // same order in every thread of every CTA
         } else {
            if (tid < (int)CS) cluster.map_shared_rank(flags, (unsigned)tid)[rank] = (double)zero;
            cluster.sync();
            SBQ_TICK(3)
            double zf = 0.0;
            for (unsigned r = 0; r < CS; ++r) zf += flags[r];
            if (zf != 0.0) { status = LOCUS_ZERO_DENOM; break; }
            // owner: CS lanes per owned column, fixed butterfly; lane r pushes the result to peer r
            {
               const int items = nb * (int)CS;
               const unsigned r = (unsigned)tid % CS;
               double* peer_nxt = cluster.map_shared_rank(nxt, r);
               double* peer_th = cluster.map_shared_rank(th, r);
               for (int base = 0; base < items; base += NT) {
                  const int x = base + tid, jj = x / (int)CS;
                  double v = x < items ? stage[(size_t)r * B + jj] : 0.0;
                  for (unsigned o = CS >> 1; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
                  if (x < items) {
                     const int j = (int)rank * B + jj;
                     const double sj = sdiv[j];
                     peer_nxt[j] = v;
                     peer_th[j] = (sj != 0) ? v / sj : 0.0;
                     if (r == 0) { const double diff = v - cur[j]; dsq[jj] = diff * diff; }
                  }
               }
            }
            SBQ_TICK(4)
            __syncthreads();
            if (tid < 32) {
               double d = 0.0;
               for (int jj = lane; jj < nb; jj += 32) d += dsq[jj];
               d = warp_sum(d);
               if (lane < (int)CS) cluster.map_shared_rank(d2p, (unsigned)lane)[rank] = d;
            }
            SBQ_TICK(5)
            cluster.sync();
            SBQ_TICK(6)
            for (unsigned r = 0; r < CS; ++r) d2 += d2p[r];      // same order in every thread of every CTA
         }
         if (d2 < tol2) { status = LOCUS_OK; break; }           // ||theta' - theta||_2 < tol; theta is NOT advanced
         { double* t_ = cur; cur = nxt; nxt = t_; }
         SBQ_TICK(7)
      }
   }
#ifdef SBQ_PHASE_TIMING
   if (rank == 0 && (tid == 0 || tid == NT - 32))
      printf("setup: sort %lld jd %lld fill %lld csc %lld rowslots %lld colslots %lld\n", st[0], st[1], st[2], st[3], st[4], st[5]);
   if (rank == 0 && (tid == 0 || tid == NT - 32))
      printf("locus %d tid %d iters %d resident %d csc_smem %d slots %d/%d lanes %d/%d nrows %d nnz %u setup %lld | E %lld or %lld col %lld csync1 %lld own %lld d2 %lld csync2 %lld chk %lld (cycles/iter)\n", l, tid, iters,
             (int)path.resident, (int)path.csc_in_smem, (int)path.row_slots, (int)path.col_slots, rslot.lanes, slot.lanes, nrows, nnz_c, t_setup, ph[0] / iters, ph[1] / iters, ph[2] / iters, ph[3] / iters, ph[4] / iters, ph[5] / iters, ph[6] / iters, ph[7] / iters);
#endif
   if (pend_b) cluster_wait();
   cluster.sync();   // no CTA may exit while a peer can still read its shared memory
#ifdef SBQ_TRACE
   if (tid == 0) trace_emit(CS, NT, l, rank, trace_t0, iters);
#endif

   if (rank != 0) return;
   // ---- outputs + epilogue (src/estimate.cpp:310-356), CTA 0 of the cluster
   locus_epilogue_block<NT>(p, l, t0, T, status, iters, theta0, cur, th, red);
}

// --------------------------------------------------------------------------------------------
// TPM denominator and TPM (src/alignments.cpp:1821-1829)
// --------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(1024) fpkm_sum_kernel(const double* __restrict__ locus_fpkm, int64_t n, double* out) {
   __shared__ double red[32];
   double v = 0.0;
   for (int64_t i = threadIdx.x; i < n; i += 1024) v += locus_fpkm[i];
   v = block_sum<1024>(v, red);
   if (threadIdx.x == 0) *out = v;
}

__global__ void tpm_kernel(const double* __restrict__ fpkm, double* __restrict__ tpm, int64_t n, double total) {
   const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
   if (i < n) tpm[i] = 1e6 * fpkm[i] / total;
}

// fragment total of every locus (sum of its class counts): one warp per locus. Only the benchmark metric needs it.
__global__ void __launch_bounds__(256) locus_frags_kernel(const int64_t* __restrict__ loc_row_off, const int32_t* __restrict__ count, int64_t n_loci, long long* __restrict__ out) {
   const int lane = threadIdx.x & 31;
   const int64_t nw = ((int64_t)gridDim.x * blockDim.x) >> 5;
   for (int64_t l = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; l < n_loci; l += nw) {
      long long v = 0;
      for (int64_t i = loc_row_off[l] + lane; i < loc_row_off[l + 1]; i += 32) v += count[i];
      v = warp_sum_ll(v);
      if (lane == 0) out[l] = v;
   }
}

// same, with the denominator read from device memory (multi-GPU: the all-reduced sum never visits the host)
__global__ void tpm_dev_kernel(const double* __restrict__ fpkm, double* __restrict__ tpm, int64_t n, const double* __restrict__ total) {
   const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
   const double tot = *total;
   if (i < n) tpm[i] = 1e6 * fpkm[i] / tot;
}

}  // namespace sbq

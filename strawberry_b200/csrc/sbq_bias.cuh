// sbq_bias.cuh - bias-corrected EM (bias_mode = 1): theta-EM, bias-weight update and both convergence tests fused
// in one persistent kernel, one thread-block CLUSTER per locus (1, 2, 4, 8 or 16 CTAs by non-zeros; the rows are split
// over the CTAs by non-zero count and every partial sum is exchanged through distributed shared memory in rank order).
//
// THE REFERENCE HAS NO BIAS IMPLEMENTATION (src/bias.cpp is entirely commented out, EmSolver's bias members and the
// 4-argument init() are never defined or read; SURVEY section 0.2). What runs here is OUR definition, documented in
// DESIGN.md section 7 and restated on the CPU by the test oracle (orc_em_bias_csr) - parity is against that
// restatement only ("parity unpinned" with respect to the reference). It reuses the constants the reference declares
// for the purpose (include/estimate.hpp:237-242): <= 100 outer rounds, <= 5000 theta iterations, <= 10 bias
// iterations, bias change limit 1e-2.
//
//   row weight   w_i = exp(clamp(beta . x_i, +-30)),  x_i = the row's covariates (gc, gc^2, gc^3, log len, ...)
//   model        F_ij = alpha_ij w_i, column-normalised over the kept rows: s_j = sum_i alpha_ij w_i
//   outer round  (1) theta-EM with beta fixed until ||theta' - theta||_2 < theta_tol (theta advanced);
//                (2) Newton steps of the Poisson log-linear fit n_i ~ w_i d_i, d_i = sum_j alpha_ij theta_j / s_j fixed:
//                    g = sum_i (n_i - mu_i) x_i,  H = sum_i mu_i x_i x_i^T (+ ridge),  beta += H^-1 g,
//                    until ||delta beta||_2 < bias_tol;
//                (3) stop when beta moved less than bias_tol in this round.
#pragma once
#include "sbq_kernels.cuh"

namespace sbq {

constexpr int BI_NT = 256;
constexpr int BI_W = BI_NT / 32;
constexpr int BI_MAX_COV = 6;
constexpr int BI_NGH = BI_MAX_COV + BI_MAX_COV * (BI_MAX_COV + 1) / 2;   // gradient + upper triangle of the Hessian

struct BiasParams {
   const double* x;      // [n_row][n_cov] covariates, row-major over the whole batch
   double* w;            // [n_row] scratch: row weights
   double* d;            // [n_row] scratch: row normalisers of the last theta
   double* beta;         // [n_loci][n_cov] out
   int32_t* outer;       // [n_loci] out: outer rounds executed
   int n_cov, max_out_it, max_theta_it, max_bias_it;
   double bias_tol;
};

// th, theta x2, s_j, this CTA's partial sums [T + 8], warp-private accumulators [BI_W][T]
__host__ __device__ inline size_t bias_smem_bytes(int T) { return ((size_t)5 * T + 8 + (size_t)BI_W * T) * sizeof(double); }
// CTAs per locus: a function of the locus alone (so is every summation order)
inline int bias_cluster_size(int64_t nnz) { return nnz <= 6000 ? 1 : nnz <= 16000 ? 2 : nnz <= 40000 ? 4 : nnz <= 100000 ? 8 : 16; }

// warp-per-row pass over the rows [ra, rb) of this CTA;
//    MODE 0: acc[col] += alpha * w_i (column sums of the biased model)
//    MODE 1: E/M step with th[] (acc[col] += alpha th r_i), flags zero denominators
//    MODE 2: d_i = sum alpha th  -> dbuf[i]
template <int MODE>
__device__ __forceinline__ void bias_row_pass(const DevParams& p, const int64_t* __restrict__ rp, const int32_t* neff, int ra, int rb, const double* th,
                                              double* my_acc, const double* wbuf, double* dbuf, int& zero) {
   const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
   for (int i = ra + warp; i < rb; i += BI_W) {
      const int ne = neff[i];
      if (ne < 0) { if (MODE == 2 && lane == 0) dbuf[i] = 0.0; continue; }
      const int64_t k0 = rp[i], k1 = rp[i + 1];
      if (MODE == 0) {
         const double wi = wbuf[i];
         for (int64_t k = k0 + lane; k < k1; k += 32) my_acc[p.col[k]] += p.alpha[k] * wi;
      } else {
         double d = 0.0;
         for (int64_t k = k0 + lane; k < k1; k += 32) d += p.alpha[k] * th[p.col[k]];
         d = warp_sum(d);
         if (MODE == 2) {
            if (lane == 0) dbuf[i] = d;
         } else {
            if (d == 0) { zero = 1; continue; }
            const double r = (double)ne / d;
            for (int64_t k = k0 + lane; k < k1; k += 32) { const int c = p.col[k]; my_acc[c] += p.alpha[k] * th[c] * r; }
         }
      }
      __syncwarp();   // the warp's next row may touch the same accumulator column from another lane
   }
}

__global__ void __launch_bounds__(BI_NT)
em_bias_kernel(DevParams p, BiasParams bp, const int32_t* __restrict__ list, int n_list) {
   (void)n_list;
   cg::cluster_group cluster = cg::this_cluster();
   const unsigned CS = cluster.num_blocks(), rank = cluster.block_rank();
   const int l = list[blockIdx.x / CS];
   const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
   const int K = bp.n_cov;
   const int64_t r0 = p.loc_row_off[l];
   const int R = (int)(p.loc_row_off[l + 1] - r0);
   const int64_t t0 = p.loc_iso_off[l];
   const int T = (int)(p.loc_iso_off[l + 1] - t0);
   extern __shared__ double smem[];
   double* th = smem;
   double* cur = th + T;
   double* nxt = cur + T;
   double* sdiv = nxt + T;
   double* part = sdiv + T;  // [T + 8] this CTA's partial sums, read by the peers; part[T] = one scalar summed alongside
   double* acc = part + T + 8;   // [BI_W][T]
   __shared__ double red[BI_NT / 32];
   __shared__ double s_beta[BI_MAX_COV], s_gh[BI_MAX_COV + BI_MAX_COV * BI_MAX_COV];
   __shared__ double s_x[BI_NGH + 5];   // this CTA's scalars, read by the peers
   __shared__ double s_n2;
   __shared__ int s_rows[2];
   const int64_t* __restrict__ rp = p.row_ptr + r0;
   int32_t* neff = p.neff + r0;
   double* wbuf = bp.w + r0;
   double* dbuf = bp.d + r0;
   const double* __restrict__ X = bp.x + (size_t)r0 * K;
   double* my_acc = acc + (size_t)warp * T;

   // rows of this CTA: split by non-zeros (lower_bound on row_ptr), as in the cluster tier
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
   const int ra = s_rows[0], rb = s_rows[1];

   // Fixed-order sum over the warp-private accumulators of this CTA, then over the CTAs of the cluster in rank order: every CTA
   // ends up with the same out[]. One scalar per CTA (extra) is summed alongside; returns its cluster-wide sum.
   auto reduce_acc = [&](double* out, double extra) -> double {
      for (int j = tid; j < T; j += BI_NT) {
         double s = 0.0;
         for (int w = 0; w < BI_W; ++w) { s += acc[(size_t)w * T + j]; acc[(size_t)w * T + j] = 0.0; }
         if (CS > 1) part[j] = s; else out[j] = s;
      }
      if (CS == 1) { __syncthreads(); return extra; }
      if (tid == 0) part[T] = extra;
      cluster.sync();
      for (int j = tid; j < T; j += BI_NT) {
         double s = 0.0;
         for (unsigned r = 0; r < CS; ++r) s += cluster.map_shared_rank(part, r)[j];
         out[j] = s;
      }
      double ex = 0.0;
      for (unsigned r = 0; r < CS; ++r) ex += cluster.map_shared_rank(part, r)[T];
      cluster.sync();   // the peers have read part[]; out[] is visible CTA-wide
      return ex;
   };
   // n scalars held by thread 0 in s_x[0..n): cluster-wide sums, in rank order, left in s_x of every CTA
   auto cluster_scalars = [&](int n) {
      if (CS == 1) { __syncthreads(); return; }
      cluster.sync();
      double v = 0.0;
      if (tid < n)
         for (unsigned r = 0; r < CS; ++r) v += cluster.map_shared_rank(s_x, r)[tid];
      cluster.sync();
      if (tid < n) s_x[tid] = v;
      __syncthreads();
   };

   // ---- setup: total, row filter, unit weights
   long long tot = 0;
   int kept = 0;
   for (int x = tid; x < BI_W * T; x += BI_NT) acc[x] = 0.0;
   for (int i = ra + warp; i < rb; i += BI_W) {
      const int64_t k0 = rp[i], k1 = rp[i + 1];
      bool keep = false;
      for (int64_t k = k0 + lane; k < k1; k += 32) keep |= p.alpha[k] > p.row_eps;
      keep = __any_sync(0xffffffffu, keep);
      if (lane == 0) {
         const int n = p.count[r0 + i];
         neff[i] = keep ? n : -1;
         wbuf[i] = 1.0;
         tot += n;
         kept += keep;
      }
   }
   if (tid < BI_MAX_COV) s_beta[tid] = 0.0;
   {
      const double tb = block_sum<BI_NT>((double)tot, red);
      const double kb = block_sum<BI_NT>((double)kept, red);
      if (tid == 0) { s_x[0] = tb; s_x[1] = kb; }
      cluster_scalars(2);
   }
   const double total = s_x[0], kept_all = s_x[1];
   const double theta0 = total / (double)T;
   for (int j = tid; j < T; j += BI_NT) cur[j] = theta0;
   __syncthreads();

   int status = LOCUS_ITER_CAP, iters = 0, outer = 0;
   if (kept_all == 0) {
      status = LOCUS_NO_ROWS;
   } else {
      for (int out = 0; out < bp.max_out_it && status == LOCUS_ITER_CAP; ++out) {
         outer = out + 1;
         int zero = 0;
         bias_row_pass<0>(p, rp, neff, ra, rb, th, my_acc, wbuf, dbuf, zero);
         __syncthreads();
         reduce_acc(sdiv, 0.0);
         // (1) theta-EM with the current bias
         for (int it = 0; it < bp.max_theta_it; ++it) {
            ++iters;
            for (int j = tid; j < T; j += BI_NT) th[j] = sdiv[j] != 0 ? cur[j] / sdiv[j] : 0.0;
            __syncthreads();
            bias_row_pass<1>(p, rp, neff, ra, rb, th, my_acc, wbuf, dbuf, zero);
            zero = __syncthreads_or(zero);
            const double zf = reduce_acc(nxt, (double)zero);
            double d2 = 0.0;
            for (int j = tid; j < T; j += BI_NT) { const double df = nxt[j] - cur[j]; d2 += df * df; }
            d2 = block_sum<BI_NT>(d2, red);      // the same value in every CTA: nxt and cur are
            if (zf != 0.0) { status = LOCUS_ZERO_DENOM; break; }
            for (int j = tid; j < T; j += BI_NT) cur[j] = nxt[j];
            __syncthreads();
            if (sqrt(d2) < p.tol) break;
         }
         if (status == LOCUS_ZERO_DENOM) break;
         if (K == 0) { status = LOCUS_OK; break; }
         // (2) bias-weight update: Newton steps on beta with d_i fixed
         for (int j = tid; j < T; j += BI_NT) th[j] = sdiv[j] != 0 ? cur[j] / sdiv[j] : 0.0;
         __syncthreads();
         bias_row_pass<2>(p, rp, neff, ra, rb, th, my_acc, wbuf, dbuf, zero);
         double bprev[BI_MAX_COV];
         for (int a = 0; a < BI_MAX_COV; ++a) bprev[a] = a < K ? s_beta[a] : 0.0;
         __syncthreads();
         for (int nb = 0; nb < bp.max_bias_it; ++nb) {
            double g[BI_MAX_COV], H[BI_MAX_COV * (BI_MAX_COV + 1) / 2];
#pragma unroll
            for (int a = 0; a < BI_MAX_COV; ++a) g[a] = 0.0;
#pragma unroll
            for (int a = 0; a < BI_MAX_COV * (BI_MAX_COV + 1) / 2; ++a) H[a] = 0.0;
            for (int i = ra + tid; i < rb; i += BI_NT) {
               const int ne = neff[i];
               if (ne < 0) continue;
               const double mu = wbuf[i] * dbuf[i];
               const double res = (double)ne - mu;
               int h = 0;
#pragma unroll
               for (int a = 0; a < BI_MAX_COV; ++a) {
                  const double xa = a < K ? X[(size_t)i * K + a] : 0.0;
                  g[a] += res * xa;
#pragma unroll
                  for (int b = a; b < BI_MAX_COV; ++b) {
                     const double xb = b < K ? X[(size_t)i * K + b] : 0.0;
                     H[h++] += mu * xa * xb;
                  }
               }
            }
            {
               int h = 0;
#pragma unroll
               for (int a = 0; a < BI_MAX_COV; ++a) {
                  const double ga = block_sum<BI_NT>(g[a], red);
                  if (tid == 0) s_x[a] = ga;
#pragma unroll
                  for (int b = a; b < BI_MAX_COV; ++b) {
                     const double hab = block_sum<BI_NT>(H[h], red);
                     if (tid == 0) s_x[BI_MAX_COV + h] = hab;
                     ++h;
                  }
               }
               cluster_scalars(BI_NGH);
               if (tid == 0) {
                  h = 0;
                  for (int a = 0; a < BI_MAX_COV; ++a) {
                     s_gh[a] = s_x[a];
                     for (int b = a; b < BI_MAX_COV; ++b) {
                        const double hab = s_x[BI_MAX_COV + h++];
                        s_gh[BI_MAX_COV + a * BI_MAX_COV + b] = hab;
                        s_gh[BI_MAX_COV + b * BI_MAX_COV + a] = hab;
                     }
                  }
               }
            }
            if (tid == 0) {
               // K x K solve with a small ridge (Gaussian elimination with partial pivoting, like the restatement); every CTA of the
               // cluster solves the same system
               double A[BI_MAX_COV * BI_MAX_COV], v[BI_MAX_COV];
               double tr = 0.0;
               for (int a = 0; a < K; ++a) tr += s_gh[BI_MAX_COV + a * BI_MAX_COV + a];
               for (int a = 0; a < K; ++a) {
                  v[a] = s_gh[a];
                  for (int b = 0; b < K; ++b) A[a * K + b] = s_gh[BI_MAX_COV + a * BI_MAX_COV + b] + (a == b ? 1e-9 * tr + 1e-12 : 0.0);
               }
               bool ok = true;
               for (int c = 0; c < K && ok; ++c) {
                  int piv = c;
                  for (int r = c + 1; r < K; ++r)
                     if (fabs(A[r * K + c]) > fabs(A[piv * K + c])) piv = r;
                  if (A[piv * K + c] == 0.0) { ok = false; break; }
                  if (piv != c) {
                     for (int k = 0; k < K; ++k) { const double t = A[c * K + k]; A[c * K + k] = A[piv * K + k]; A[piv * K + k] = t; }
                     const double t = v[c]; v[c] = v[piv]; v[piv] = t;
                  }
                  for (int r = c + 1; r < K; ++r) {
                     const double f = A[r * K + c] / A[c * K + c];
                     for (int k = c; k < K; ++k) A[r * K + k] -= f * A[c * K + k];
                     v[r] -= f * v[c];
                  }
               }
               double n2 = -1.0;
               if (ok) {
                  for (int c = K - 1; c >= 0; --c) {
                     double s = v[c];
                     for (int k = c + 1; k < K; ++k) s -= A[c * K + k] * v[k];
                     v[c] = s / A[c * K + c];
                  }
                  n2 = 0.0;
                  for (int a = 0; a < K; ++a) { s_beta[a] += v[a]; n2 += v[a] * v[a]; }
               }
               s_n2 = n2;
            }
            __syncthreads();
            const double n2 = s_n2;
            if (n2 < 0) break;   // singular system: keep beta
            for (int i = ra + tid; i < rb; i += BI_NT) {
               double e = 0.0;
               for (int a = 0; a < K; ++a) e += s_beta[a] * X[(size_t)i * K + a];
               e = e > 30.0 ? 30.0 : (e < -30.0 ? -30.0 : e);
               wbuf[i] = exp(e);
            }
            __syncthreads();
            if (sqrt(n2) < bp.bias_tol) break;
         }
         // (3) outer convergence on beta
         double m2 = 0.0;
         for (int a = 0; a < K; ++a) m2 += (s_beta[a] - bprev[a]) * (s_beta[a] - bprev[a]);
         __syncthreads();
         if (sqrt(m2) < bp.bias_tol) status = LOCUS_OK;
      }
   }
   if (CS > 1) {
      cluster.sync();   // no CTA may exit while a peer can still read its shared memory
      if (rank != 0) return;
   }

   // ---- outputs + epilogue (same tail as the other tiers, src/estimate.cpp:310-356)
   locus_epilogue_block<BI_NT>(p, l, t0, T, status, iters, theta0, cur, th, red);
   if (tid == 0) {
      bp.outer[l] = outer;
      for (int a = 0; a < K; ++a) bp.beta[(size_t)l * K + a] = s_beta[a];
   }
}


// --------------------------------------------------------------------------------------------
// Small loci (T <= 32, R <= 64, <= 256 non-zeros: the shapes of the EM warp tier, 92 % of a human-shaped sample): ONE WARP per
// locus, persistent warps pulling loci from a queue. Lane i owns rows i and i + 32 - their counts, weights w_i, normalisers d_i and
// covariates live in registers - and lane j owns theta_j / s_j. Accumulators are lane-private (stride 33), column sums are taken
// over the lanes in a fixed order, the 27 Newton sums by warp butterflies; lane 0 solves the K x K system. No block barriers:
// an iteration of the theta-EM costs what it costs in the EM warp tier instead of the ~3.5 us of a 256-thread CTA (the bias
// leg of the benchmark was bound by ONE 15-row locus that needs 77 573 theta iterations).
// --------------------------------------------------------------------------------------------
constexpr int BW_WARPS = 4;
constexpr int BW_REG = 8;    // non-zeros per row a lane keeps in registers on the single-row fast path
__host__ __device__ inline size_t bias_warp_smem_bytes() { return (size_t)BW_WARPS * ((size_t)WT_MAX_ISO * WT_STRIDE + WT_MAX_ISO) * sizeof(double); }
__host__ __device__ inline bool bias_warp_tier(int64_t nnz, int R, int T) { return T <= WT_MAX_ISO && R <= WT_MAX_ROWS && nnz <= WT_MAX_NNZ; }

__global__ void __launch_bounds__(BW_WARPS * 32)
em_bias_warp_kernel(DevParams p, BiasParams bp, const int32_t* __restrict__ list, int n_list, int* queue) {
   extern __shared__ double smem[];
   const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
   double* acc = smem + (size_t)warp * ((size_t)WT_MAX_ISO * WT_STRIDE + WT_MAX_ISO);
   double* th = acc + (size_t)WT_MAX_ISO * WT_STRIDE;
   const int32_t* __restrict__ col = p.col;
   const double* __restrict__ al = p.alpha;
   const int K = bp.n_cov;

   for (;;) {
      int wq = 0;
      if (lane == 0) wq = atomicAdd(queue, 1);
      wq = __shfl_sync(0xffffffffu, wq, 0);
      if (wq >= n_list) break;
      const int l = list[wq];
      const int64_t r0 = p.loc_row_off[l];
      const int R = (int)(p.loc_row_off[l + 1] - r0);
      const int64_t t0 = p.loc_iso_off[l];
      const int T = (int)(p.loc_iso_off[l + 1] - t0);
      const int64_t* __restrict__ rp = p.row_ptr + r0;
      const int nl = R < 32 ? R : 32;   // lanes that own at least one row

      for (int x = lane; x < T * WT_STRIDE; x += 32) acc[x] = 0.0;
      // ---- this lane's rows: extent, count, row filter, covariates
      int64_t k0[2], k1[2];
      int ne[2];
      double w[2], d[2], xr[2][BI_MAX_COV];
      long long tot = 0;
      int kept = 0;
#pragma unroll
      for (int q = 0; q < 2; ++q) {
         const int i = lane + 32 * q;
         k0[q] = k1[q] = 0; ne[q] = -1; w[q] = 1.0; d[q] = 0.0;
#pragma unroll
         for (int a = 0; a < BI_MAX_COV; ++a) xr[q][a] = 0.0;
         if (i < R) {
            k0[q] = rp[i]; k1[q] = rp[i + 1];
            const int n = p.count[r0 + i];
            tot += n;
            bool keep = false;
            for (int64_t k = k0[q]; k < k1[q]; ++k) keep |= al[k] > p.row_eps;
            if (keep) { ne[q] = n; ++kept; }
#pragma unroll
            for (int a = 0; a < BI_MAX_COV; ++a)
               if (a < K) xr[q][a] = bp.x[(size_t)(r0 + i) * K + a];
         }
      }
      tot = warp_sum_ll(tot);
      kept = (int)warp_sum_ll(kept);
      __syncwarp();
      // fast path: one row per lane, at most BW_REG non-zeros each, held in registers for the whole solve (same order of every sum
      // as the general path: padding entries carry alpha = 0). The locus that bounds the benchmark's bias leg - 15 rows, 41
      // non-zeros, 77 573 theta iterations - runs here.
      const bool fast = R <= 32 && __all_sync(0xffffffffu, (int)(k1[0] - k0[0]) <= BW_REG);
      double ra[BW_REG];
      int rc[BW_REG];
#pragma unroll
      for (int e = 0; e < BW_REG; ++e) {
         const bool v = fast && ne[0] >= 0 && k0[0] + e < k1[0];
         ra[e] = v ? al[k0[0] + e] : 0.0;
         rc[e] = v ? col[k0[0] + e] : 0;
      }
      // column sum over the lanes, fixed order (lane j: column j); clears the accumulators
      auto col_sum = [&]() -> double {
         double s0 = 0.0;
         if (lane < T)
            for (int x = 0; x < nl; ++x) { s0 += acc[lane * WT_STRIDE + x]; acc[lane * WT_STRIDE + x] = 0.0; }
         return s0;
      };
      double beta[BI_MAX_COV];
#pragma unroll
      for (int a = 0; a < BI_MAX_COV; ++a) beta[a] = 0.0;
      const double theta0 = (double)tot / (double)T;
      double cur = theta0;
      int status = LOCUS_ITER_CAP, iters = 0, outer = 0;
      if (kept == 0) {
         status = LOCUS_NO_ROWS;
      } else {
         for (int out = 0; out < bp.max_out_it && status == LOCUS_ITER_CAP; ++out) {
            outer = out + 1;
            // s_j = sum_i alpha_ij w_i over the kept rows
            if (fast) {
#pragma unroll
               for (int e = 0; e < BW_REG; ++e)
                  if (ra[e] != 0.0) acc[rc[e] * WT_STRIDE + lane] += ra[e] * w[0];
            } else {
#pragma unroll
               for (int q = 0; q < 2; ++q)
                  if (ne[q] >= 0)
                     for (int64_t k = k0[q]; k < k1[q]; ++k) acc[col[k] * WT_STRIDE + lane] += al[k] * w[q];
            }
            __syncwarp();
            const double s = col_sum();
            __syncwarp();
            // (1) theta-EM with the current bias (theta is advanced before the convergence test, as in the restatement)
            bool zero = false;
            for (int it = 0; it < bp.max_theta_it; ++it) {
               ++iters;
               if (lane < T) th[lane] = (s != 0) ? cur / s : 0.0;
               __syncwarp();
               if (fast) {
                  double t[BW_REG], dd = 0.0;
#pragma unroll
                  for (int e = 0; e < BW_REG; ++e) { t[e] = th[rc[e]]; dd += ra[e] * t[e]; }
                  if (ne[0] >= 0) {
                     if (dd == 0) {
                        zero = true;
                     } else {
                        const double r = (double)ne[0] / dd;
#pragma unroll
                        for (int e = 0; e < BW_REG; ++e)
                           if (ra[e] != 0.0) acc[rc[e] * WT_STRIDE + lane] += ra[e] * t[e] * r;
                     }
                  }
               } else {
#pragma unroll
                  for (int q = 0; q < 2; ++q) {
                     if (ne[q] < 0) continue;
                     double dd = 0.0;
                     for (int64_t k = k0[q]; k < k1[q]; ++k) dd += al[k] * th[col[k]];
                     if (dd == 0) { zero = true; continue; }
                     const double r = (double)ne[q] / dd;
                     for (int64_t k = k0[q]; k < k1[q]; ++k) { const int c = col[k]; acc[c * WT_STRIDE + lane] += al[k] * th[c] * r; }
                  }
               }
               zero = __any_sync(0xffffffffu, zero);
               __syncwarp();
               const double nw = col_sum();
               const double diff = lane < T ? nw - cur : 0.0;
               const double d2 = warp_sum(diff * diff);
               if (zero) { status = LOCUS_ZERO_DENOM; break; }
               cur = nw;
               __syncwarp();
               if (sqrt(d2) < p.tol) break;
            }
            if (status == LOCUS_ZERO_DENOM) break;
            if (K == 0) { status = LOCUS_OK; break; }
            // (2) bias-weight update: Newton steps on beta with d_i fixed
            if (lane < T) th[lane] = (s != 0) ? cur / s : 0.0;
            __syncwarp();
            if (fast) {
               d[0] = 0.0;
               d[1] = 0.0;
#pragma unroll
               for (int e = 0; e < BW_REG; ++e) d[0] += ra[e] * th[rc[e]];
            } else {
#pragma unroll
               for (int q = 0; q < 2; ++q) {
                  d[q] = 0.0;
                  if (ne[q] >= 0)
                     for (int64_t k = k0[q]; k < k1[q]; ++k) d[q] += al[k] * th[col[k]];
               }
            }
            __syncwarp();
            double bprev[BI_MAX_COV];
#pragma unroll
            for (int a = 0; a < BI_MAX_COV; ++a) bprev[a] = beta[a];
            for (int nb = 0; nb < bp.max_bias_it; ++nb) {
               double g[BI_MAX_COV], H[BI_MAX_COV * (BI_MAX_COV + 1) / 2];
#pragma unroll
               for (int a = 0; a < BI_MAX_COV; ++a) g[a] = 0.0;
#pragma unroll
               for (int a = 0; a < BI_MAX_COV * (BI_MAX_COV + 1) / 2; ++a) H[a] = 0.0;
#pragma unroll
               for (int q = 0; q < 2; ++q) {
                  if (ne[q] < 0) continue;
                  const double mu = w[q] * d[q];
                  const double res = (double)ne[q] - mu;
                  int h = 0;
#pragma unroll
                  for (int a = 0; a < BI_MAX_COV; ++a) {
                     g[a] += res * xr[q][a];
#pragma unroll
                     for (int b = a; b < BI_MAX_COV; ++b) H[h++] += mu * xr[q][a] * xr[q][b];
                  }
               }
#pragma unroll
               for (int a = 0; a < BI_MAX_COV; ++a) g[a] = warp_sum(g[a]);
#pragma unroll
               for (int a = 0; a < BI_MAX_COV * (BI_MAX_COV + 1) / 2; ++a) H[a] = warp_sum(H[a]);
               double v[BI_MAX_COV], n2 = -1.0;
#pragma unroll
               for (int a = 0; a < BI_MAX_COV; ++a) v[a] = 0.0;
               if (lane == 0) {
                  // K x K solve with a small ridge (Gaussian elimination with partial pivoting, like the restatement)
                  double A[BI_MAX_COV * BI_MAX_COV], y[BI_MAX_COV];
                  double tr = 0.0;
                  {
                     int h = 0;
                     for (int a = 0; a < BI_MAX_COV; ++a)
                        for (int b = a; b < BI_MAX_COV; ++b) {
                           const double hab = H[h++];
                           if (a < K && b < K) { A[a * K + b] = hab; A[b * K + a] = hab; }
                        }
                  }
                  for (int a = 0; a < K; ++a) tr += A[a * K + a];
                  for (int a = 0; a < K; ++a) { y[a] = g[a]; A[a * K + a] += 1e-9 * tr + 1e-12; }
                  bool ok = true;
                  for (int c = 0; c < K && ok; ++c) {
                     int piv = c;
                     for (int r = c + 1; r < K; ++r)
                        if (fabs(A[r * K + c]) > fabs(A[piv * K + c])) piv = r;
                     if (A[piv * K + c] == 0.0) { ok = false; break; }
                     if (piv != c) {
                        for (int k = 0; k < K; ++k) { const double t = A[c * K + k]; A[c * K + k] = A[piv * K + k]; A[piv * K + k] = t; }
                        const double t = y[c]; y[c] = y[piv]; y[piv] = t;
                     }
                     for (int r = c + 1; r < K; ++r) {
                        const double f = A[r * K + c] / A[c * K + c];
                        for (int k = c; k < K; ++k) A[r * K + k] -= f * A[c * K + k];
                        y[r] -= f * y[c];
                     }
                  }
                  if (ok) {
                     for (int c = K - 1; c >= 0; --c) {
                        double sacc = y[c];
                        for (int k = c + 1; k < K; ++k) sacc -= A[c * K + k] * y[k];
                        y[c] = sacc / A[c * K + c];
                     }
                     n2 = 0.0;
                     for (int a = 0; a < K; ++a) n2 += y[a] * y[a];
#pragma unroll
                     for (int a = 0; a < BI_MAX_COV; ++a) v[a] = a < K ? y[a] : 0.0;
                  }
               }
               n2 = __shfl_sync(0xffffffffu, n2, 0);
               if (n2 < 0) break;   // singular system: keep beta
#pragma unroll
               for (int a = 0; a < BI_MAX_COV; ++a) beta[a] += __shfl_sync(0xffffffffu, v[a], 0);
#pragma unroll
               for (int q = 0; q < 2; ++q) {
                  double e = 0.0;
#pragma unroll
                  for (int a = 0; a < BI_MAX_COV; ++a) e += beta[a] * xr[q][a];     // covariates beyond K are 0
                  e = e > 30.0 ? 30.0 : (e < -30.0 ? -30.0 : e);
                  w[q] = exp(e);
               }
               if (sqrt(n2) < bp.bias_tol) break;
            }
            // (3) outer convergence on beta
            double m2 = 0.0;
#pragma unroll
            for (int a = 0; a < BI_MAX_COV; ++a) m2 += (beta[a] - bprev[a]) * (beta[a] - bprev[a]);
            if (sqrt(m2) < bp.bias_tol) status = LOCUS_OK;
         }
      }

      // ---- outputs + epilogue (same tail as the EM warp tier, src/estimate.cpp:310-356)
      locus_epilogue_warp(p, l, t0, T, lane, status, iters, theta0, cur);
      if (lane == 0) bp.outer[l] = outer;
#pragma unroll
      for (int a = 0; a < BI_MAX_COV; ++a)
         if (lane == 0 && a < K) bp.beta[(size_t)l * K + a] = beta[a];
      __syncwarp();
   }
}

}  // namespace sbq

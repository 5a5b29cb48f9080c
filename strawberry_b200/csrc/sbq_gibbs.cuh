// sbq_gibbs.cuh - Gibbs posterior samples of a resident, solved batch (sbq_gibbs, DESIGN.md §8c "Gibbs posterior samples"; our
// definition, the reference has none).
//
// An uncollapsed data-augmentation sampler for the model the EM maximises: per locus, with F_ij = alpha_ij / s_j, the likelihood
// prod_i (sum_j F_ij pi_j)^{n_i} and a symmetric Dirichlet(prior) prior on pi. The state is phi_j = pi_j / s_j. A round
//   assignment  every fragment of a kept row picks an entry of its row with probability alpha_ij phi_j / sum_k alpha_ik phi_k,
//               by inverse CDF over the row's running sums in CSR order; c_j = fragments that landed on isoform j
//   Dirichlet   g_j ~ Gamma(c_j + prior) (Marsaglia-Tsang, polar normals, our own log / exp), pi = g / sum g, phi = pi / s
// Every operation below is a correctly rounded IEEE fp64 operation (the g_* helpers: __dadd_rn etc. on the device, nothing the
// compiler may contract into an FMA), so tests/gibbs_ref.py restates a sample bit for bit. The constants are those of §8c.
#pragma once
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>
#include <string.h>

#include "sbq_bootstrap.cuh"
#include "sbq_grid_dual.cuh"
#include "sbq_kernels.cuh"
#include "sbq_synth.cuh"

namespace sbq {

constexpr uint64_t GIBBS_SALT = 0x9FB21C651E98DF25ull;   // round key: sm64(sm64(sm64(seed ^ GIBBS_SALT) + r) + l)
constexpr uint64_t GAMMA_SALT = 0xC2B2AE3D27D4EB4Full;   // gamma stream of isoform j: sm64(sm64(gk ^ GAMMA_SALT) + j)
constexpr int GIBBS_NT = 256;                            // threads of gibbs_theta_kernel (block_sum shape of the restatement)
constexpr int GIBBS_LIGHT = 8;                           // rows of at most this many fragments draw in the row pass

// ---- correctly rounded arithmetic, never contracted ----------------------------------------------------------------------------
__host__ __device__ __forceinline__ double g_add(double a, double b) {
#ifdef __CUDA_ARCH__
   return __dadd_rn(a, b);
#else
   return a + b;
#endif
}
__host__ __device__ __forceinline__ double g_sub(double a, double b) { return g_add(a, -b); }
__host__ __device__ __forceinline__ double g_mul(double a, double b) {
#ifdef __CUDA_ARCH__
   return __dmul_rn(a, b);
#else
   return a * b;
#endif
}
__host__ __device__ __forceinline__ double g_div(double a, double b) {
#ifdef __CUDA_ARCH__
   return __ddiv_rn(a, b);
#else
   return a / b;
#endif
}
__host__ __device__ __forceinline__ double g_sqrt(double a) {
#ifdef __CUDA_ARCH__
   return __dsqrt_rn(a);
#else
   return sqrt(a);
#endif
}
__host__ __device__ __forceinline__ double g_pow2(int n) {   // 2^n, -1022 <= n <= 1023, from its bits
   const uint64_t b = (uint64_t)(n + 1023) << 52;
   double d;
   memcpy(&d, &b, 8);
   return d;
}

// uniform in (0, 1): (2 (h >> 12) + 1) 2^-53, exact
__host__ __device__ __forceinline__ double g_u(uint64_t h) { return (double)(((h >> 12) << 1) | 1ull) * 0x1p-53; }

// natural log of a finite x > 0 (subnormals included): frexp reduction to m in [sqrt(1/2), sqrt 2), then the fdlibm e_log.c
// polynomial (public domain, Sun Microsystems 1993) in s = f / (2 + f), f = m - 1
__host__ __device__ __forceinline__ double g_log(double x) {
   int e;
   double m = frexp(x, &e);
   if (m < 0.70710678118654752440) { m = g_mul(m, 2.0); --e; }
   const double f = g_sub(m, 1.0);
   const double s = g_div(f, g_add(2.0, f));
   const double dk = (double)e;
   const double z = g_mul(s, s), w = g_mul(z, z);
   const double t1 = g_mul(w, g_add(3.999999999940941908e-01, g_mul(w, g_add(2.222219843214978396e-01, g_mul(w, 1.531383769920937332e-01)))));
   const double t2 = g_mul(z, g_add(6.666666666666735130e-01, g_mul(w, g_add(2.857142874366239149e-01, g_mul(w, g_add(1.818357216161805012e-01,
                                                                                                                 g_mul(w, 1.479819860511658591e-01)))))));
   const double R = g_add(t2, t1);
   const double hfsq = g_mul(g_mul(0.5, f), f);
   return g_sub(g_mul(dk, 6.93147180369123816490e-01), g_sub(g_sub(hfsq, g_add(g_mul(s, g_add(hfsq, R)), g_mul(dk, 1.90821492927058770002e-10))), f));
}

// e^x: k = floor(x / ln 2 + 1/2), r = x - k ln 2 (two-part ln 2), the fdlibm e_exp.c polynomial, then y 2^k in two exact-or-one-
// rounding multiplies (so a subnormal result is rounded once, as IEEE multiplication rounds it)
__host__ __device__ __forceinline__ double g_exp(double x) {
   if (x > 709.782712893383973096) return INFINITY;
   if (x < -745.133219101941108420) return 0.0;
   const double kd = floor(g_add(g_mul(x, 1.44269504088896338700e+00), 0.5));
   const int k = (int)kd;
   const double hi = g_sub(x, g_mul(kd, 6.93147180369123816490e-01));
   const double lo = g_mul(kd, 1.90821492927058770002e-10);
   const double r = g_sub(hi, lo);
   const double t = g_mul(r, r);
   const double c = g_sub(r, g_mul(t, g_add(1.66666666666666019037e-01, g_mul(t, g_add(-2.77777777770155933842e-03, g_mul(t, g_add(6.61375632143793436117e-05,
                                                       g_mul(t, g_add(-1.65339022054652515390e-06, g_mul(t, 4.13813679705723846039e-08))))))))));
   const double y = g_sub(1.0, g_sub(g_sub(lo, g_div(g_mul(r, c), g_sub(2.0, c))), hi));
   if (k > 1000) return g_mul(g_mul(y, g_pow2(k - 1000)), g_pow2(1000));
   if (k < -1000) return g_mul(g_mul(y, g_pow2(k + 1000)), g_pow2(-1000));
   return g_mul(y, g_pow2(k));
}

// the uniforms t = 0, 1, ... of one gamma draw: g_u(sm64(key + t))
struct GibbsStream {
   uint64_t key, t;
   __host__ __device__ __forceinline__ double next() { return g_u(sm64(key + t++)); }
};

// standard normal, Marsaglia's polar method: x = 2 u_t - 1, y = 2 u_{t+1} - 1 until 0 < q = x^2 + y^2 < 1; returns
// x sqrt(-2 log q / q) (y's twin is not kept)
__host__ __device__ __forceinline__ double gibbs_normal(GibbsStream& s) {
   for (;;) {
      const double x = g_sub(g_mul(2.0, s.next()), 1.0);
      const double y = g_sub(g_mul(2.0, s.next()), 1.0);
      const double q = g_add(g_mul(x, x), g_mul(y, y));
      if (q < 1.0 && q > 0.0) return g_mul(x, g_sqrt(g_div(g_mul(-2.0, g_log(q)), q)));
   }
}

// Gamma(a, 1) for a >= 1: Marsaglia-Tsang with the squeeze. d = a - 1/3, c = 1 / sqrt(9 d); per try a normal x (redrawn while
// v = 1 + c x <= 0), v = v^3, then one uniform u: accept d v if u < 1 - 0.0331 x^4 or log u < x^2 / 2 + d (1 - v + log v)
__host__ __device__ __forceinline__ double gibbs_gamma_ge1(double a, GibbsStream& s) {
   const double d = g_sub(a, 1.0 / 3.0), c = g_div(1.0, g_sqrt(g_mul(9.0, d)));
   for (;;) {
      double x, v;
      do {
         x = gibbs_normal(s);
         v = g_add(1.0, g_mul(c, x));
      } while (v <= 0.0);
      v = g_mul(g_mul(v, v), v);
      const double u = s.next(), x2 = g_mul(x, x);
      if (u < g_sub(1.0, g_mul(0.0331, g_mul(x2, x2)))) return g_mul(d, v);
      if (g_log(u) < g_add(g_mul(0.5, x2), g_mul(d, g_add(g_sub(1.0, v), g_log(v))))) return g_mul(d, v);
   }
}

// Gamma(a, 1), a > 0: a < 1 draws Gamma(a + 1) first, then one uniform U, and returns Gamma(a + 1) exp(log U / a)
__host__ __device__ __forceinline__ double gibbs_gamma(double a, uint64_t key) {
   GibbsStream s{key, 0};
   if (a >= 1.0) return gibbs_gamma_ge1(a, s);
   const double g = gibbs_gamma_ge1(g_add(a, 1.0), s);
   return g_mul(g, g_exp(g_div(g_log(s.next()), a)));
}

// ---- kernels ---------------------------------------------------------------------------------------------------------------------

// The giant tier's one-off layout passes reorder the weights inside rows of at most G6_MAXROW entries IN PLACE and keep the
// column of every weight in the 16-bit slot array (dual: slot << 3, slot B decoded back to its column; TMA ring: the column).
// This pass writes every weight of the listed loci back to its submitted CSR position in ga (which holds a copy of alpha): the
// sampler's running sums are defined in submitted order. One warp per row; a row's columns are distinct.
__global__ void __launch_bounds__(256) gibbs_unpermute_kernel(DevParams p, const int32_t* __restrict__ list, int n_list,
                                                              const unsigned short* __restrict__ col16, int dual, double* __restrict__ ga) {
   const int lane = threadIdx.x & 31;
   const int64_t wid = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5, nw = ((int64_t)gridDim.x * blockDim.x) >> 5;
   for (int item = 0; item < n_list; ++item) {
      const int l = list[item];
      const int64_t r0 = p.loc_row_off[l], r1 = p.loc_row_off[l + 1];
      const int Tp = g6_tp((int)(p.loc_iso_off[l + 1] - p.loc_iso_off[l]));
      for (int64_t row = r0 + wid; row < r1; row += nw) {
         const int64_t k0 = p.row_ptr[row];
         const int len = (int)(p.row_ptr[row + 1] - k0);
         if (len > G6_MAXROW) continue;   // longer rows are never reordered
         for (int idx = lane; idx < len; idx += 32) {
            const unsigned v = col16[k0 + idx];
            int cc = (int)v;
            if (dual) {
               const int slot = (int)(v >> 3);
               if (slot < Tp) cc = slot;
               else {
                  const int sb = slot - Tp, blk = sb & ~15;
                  cc = blk + (((sb & 15) - (blk >> 4)) & 15);
               }
            }
            int m = 0;
            while (m < len && p.col[k0 + m] != cc) ++m;
            if (m < len) ga[k0 + m] = p.alpha[k0 + idx];
         }
      }
   }
}

// Once per call, one warp per locus walking its rows in order: the row filter of the EM (a row is kept when one of its weights
// exceeds row_eps), s_j = sum of alpha_ij over kept rows ADDED IN ASCENDING ROW ORDER (the lanes of one row hold distinct
// columns), N_kept, the locus of every row, gn[i] = n_i for kept rows of sampled loci (else -1) and hv[i] = n_i for the rows whose
// draws go to gibbs_heavy_kernel (else 0). Loci whose point status is NO_ROWS or ZERO_DENOM are not sampled. s must be zero.
__global__ void __launch_bounds__(256) gibbs_colsum_kernel(DevParams p, const double* __restrict__ ga, int64_t n_loci, double* __restrict__ s,
                                                           int32_t* __restrict__ gn, int32_t* __restrict__ hv, int32_t* __restrict__ row_loc,
                                                           double* __restrict__ nkept) {
   const int lane = threadIdx.x & 31;
   const int64_t nw = ((int64_t)gridDim.x * blockDim.x) >> 5;
   for (int64_t l = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; l < n_loci; l += nw) {
      const int st = p.status[l];
      const bool sampled = st != LOCUS_NO_ROWS && st != LOCUS_ZERO_DENOM;
      const int64_t t0 = p.loc_iso_off[l];
      double* sl = s + t0;
      long long nk = 0;
      for (int64_t i = p.loc_row_off[l]; i < p.loc_row_off[l + 1]; ++i) {
         const int64_t k0 = p.row_ptr[i], k1 = p.row_ptr[i + 1];
         bool keep = false;
         for (int64_t k = k0 + lane; k < k1; k += 32) keep |= ga[k] > p.row_eps;
         keep = __any_sync(0xffffffffu, keep) && sampled;
         const int n = p.count[i];
         if (lane == 0) {
            row_loc[i] = (int32_t)l;
            gn[i] = keep ? n : -1;
            hv[i] = keep && n > GIBBS_LIGHT ? n : 0;
         }
         if (keep) {
            nk += n;
            for (int64_t k = k0 + lane; k < k1; k += 32) sl[p.col[k]] = g_add(sl[p.col[k]], ga[k]);
         }
         __syncwarp();
      }
      if (lane == 0) nkept[l] = (double)nk;
   }
}

// phi^0_j = theta_hat_j / s_j (0 where s_j = 0)
__global__ void __launch_bounds__(256) gibbs_init_kernel(const double* __restrict__ theta_hat, const double* __restrict__ s, int64_t n, double* __restrict__ phi) {
   const int64_t stride = (int64_t)gridDim.x * blockDim.x;
   for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < n; t += stride) phi[t] = s[t] != 0.0 ? g_div(theta_hat[t], s[t]) : 0.0;
}

// The first k of row [k0, k1) whose running sum exceeds thr, else the last entry; the running sum is recomputed in CSR order.
__device__ __forceinline__ int64_t gibbs_pick_walk(const double* __restrict__ ga, const int32_t* __restrict__ col, const double* __restrict__ ph,
                                                   int64_t k0, int64_t k1, double thr) {
   double run = 0.0;
   int64_t k = k0;
   for (; k < k1 - 1; ++k) {
      run = g_add(run, g_mul(ga[k], ph[col[k]]));
      if (run > thr) break;
   }
   return k;
}

// Assignment, row pass: one thread per row (grid-stride). A kept row with 0 < n_i <= GIBBS_LIGHT forms its total, then every
// draw d = (C_i - C_first) + m walks the row again; a row with more fragments writes its running sums to cum for
// gibbs_heavy_kernel. rkey = sm64(sm64(seed ^ GIBBS_SALT) + r); locus_id as in boot_resample_kernel.
__global__ void __launch_bounds__(256) gibbs_assign_kernel(DevParams p, const double* __restrict__ ga, const int32_t* __restrict__ gn,
                                                           const int32_t* __restrict__ row_loc, const int64_t* __restrict__ draw_off,
                                                           const int64_t* __restrict__ loc_draw_off, const int32_t* __restrict__ locus_id,
                                                           const double* __restrict__ phi, uint64_t rkey, int64_t n_row,
                                                           double* __restrict__ cum, int32_t* __restrict__ cnt) {
   const int64_t stride = (int64_t)gridDim.x * blockDim.x;
   for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_row; i += stride) {
      const int n = gn[i];
      if (n <= 0) continue;
      const int l = row_loc[i];
      const int64_t t0 = p.loc_iso_off[l], k0 = p.row_ptr[i], k1 = p.row_ptr[i + 1];
      const double* ph = phi + t0;
      double acc = 0.0;
      if (n > GIBBS_LIGHT) {
         for (int64_t k = k0; k < k1; ++k) {
            acc = g_add(acc, g_mul(ga[k], ph[p.col[k]]));
            cum[k] = acc;
         }
         continue;
      }
      for (int64_t k = k0; k < k1; ++k) acc = g_add(acc, g_mul(ga[k], ph[p.col[k]]));
      const uint64_t gk = sm64(rkey + (uint64_t)(locus_id ? locus_id[l] : l));
      const uint64_t d0 = (uint64_t)(draw_off[i] - loc_draw_off[l]);
      for (int m = 0; m < n; ++m) {
         const double thr = g_mul(g_u(sm64(gk + d0 + (uint64_t)m)), acc);
         atomicAdd(cnt + t0 + p.col[gibbs_pick_walk(ga, p.col, ph, k0, k1, thr)], 1);
      }
   }
}

// Assignment, heavy rows: one thread per draw of the rows with hv[i] > 0 (hoff = exclusive prefix of hv), binary search for the
// first running sum in cum that exceeds the threshold. Lanes that pick the same isoform add once.
__global__ void __launch_bounds__(256) gibbs_heavy_kernel(DevParams p, const int64_t* __restrict__ hoff, int64_t n_row, const int32_t* __restrict__ row_loc,
                                                          const int64_t* __restrict__ draw_off, const int64_t* __restrict__ loc_draw_off,
                                                          const int32_t* __restrict__ locus_id, uint64_t rkey, const double* __restrict__ cum,
                                                          int32_t* __restrict__ cnt) {
   const int64_t total = hoff[n_row];
   const int lane = threadIdx.x & 31;
   const int64_t stride = (int64_t)gridDim.x * blockDim.x;
   for (int64_t g0 = (int64_t)blockIdx.x * blockDim.x + (threadIdx.x & ~31); g0 < total; g0 += stride) {   // warp-uniform bound
      const int64_t g = g0 + lane;
      int64_t iso = -1;
      if (g < total) {
         const int64_t i = boot_last_le(hoff, 0, n_row, g);
         const int l = row_loc[i];
         const uint64_t gk = sm64(rkey + (uint64_t)(locus_id ? locus_id[l] : l));
         const uint64_t d = (uint64_t)(draw_off[i] - loc_draw_off[l] + (g - hoff[i]));
         int64_t lo = p.row_ptr[i], hi = p.row_ptr[i + 1] - 1;
         const double thr = g_mul(g_u(sm64(gk + d)), cum[hi]);
         while (lo < hi) {
            const int64_t mid = lo + ((hi - lo) >> 1);
            if (cum[mid] > thr) hi = mid; else lo = mid + 1;
         }
         iso = p.loc_iso_off[l] + p.col[lo];
      }
      const unsigned peers = __match_any_sync(0xffffffffu, (unsigned long long)iso);
      if (iso >= 0 && lane == __ffs(peers) - 1) atomicAdd(cnt + iso, __popc(peers));
   }
}

// Dirichlet step, one CTA of GIBBS_NT threads per locus: g_j ~ Gamma(c_j + prior) (thread j mod NT, isoforms in ascending order),
// G = block_sum of the per-thread partials, pi_j = g_j / G (1 / T if G = 0), phi_j = pi_j / s_j; c is zeroed. sample: p points at
// the sample's slots, theta_j = N_kept pi_j and the locus epilogue runs. Loci that are not sampled only get their epilogue (on the
// point estimate's uniform theta).
__global__ void __launch_bounds__(GIBBS_NT) gibbs_theta_kernel(DevParams p, int64_t n_loci, const double* __restrict__ theta_hat,
                                                               const int32_t* __restrict__ pstatus, const double* __restrict__ s,
                                                               const double* __restrict__ nkept, const int32_t* __restrict__ locus_id,
                                                               uint64_t rkey, double prior, int sample, int32_t* __restrict__ cnt,
                                                               double* __restrict__ phi, double* __restrict__ gbuf, double* __restrict__ nabuf) {
   __shared__ double red[GIBBS_NT / 32];
   for (int64_t l = blockIdx.x; l < n_loci; l += gridDim.x) {
      const int64_t t0 = p.loc_iso_off[l];
      const int T = (int)(p.loc_iso_off[l + 1] - t0);
      const int st = pstatus[l];
      if (st == LOCUS_NO_ROWS || st == LOCUS_ZERO_DENOM) {
         if (sample) locus_epilogue_block<GIBBS_NT>(p, (int)l, t0, T, st, 0, theta_hat[t0], theta_hat + t0, nabuf + t0, red);
         continue;
      }
      const uint64_t gkey = sm64(sm64(rkey + (uint64_t)(locus_id ? locus_id[l] : l)) ^ GAMMA_SALT);
      double part = 0.0;
      for (int j = threadIdx.x; j < T; j += GIBBS_NT) {
         const double g = gibbs_gamma(g_add((double)cnt[t0 + j], prior), sm64(gkey + (uint64_t)j));
         cnt[t0 + j] = 0;
         gbuf[t0 + j] = g;
         part = g_add(part, g);
      }
      const double G = block_sum<GIBBS_NT>(part, red);
      const double nk = nkept[l];
      for (int j = threadIdx.x; j < T; j += GIBBS_NT) {
         const double pi = G != 0.0 ? g_div(gbuf[t0 + j], G) : g_div(1.0, (double)T);
         const double sj = s[t0 + j];
         phi[t0 + j] = sj != 0.0 ? g_div(pi, sj) : 0.0;
         if (sample) gbuf[t0 + j] = g_mul(nk, pi);
      }
      if (sample) locus_epilogue_block<GIBBS_NT>(p, (int)l, t0, T, st, 0, 0.0, gbuf + t0, nabuf + t0, red);
   }
}

}  // namespace sbq

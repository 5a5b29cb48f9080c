// sbq_grid_tma.cuh - Tier 3, main path: multi-CTA streaming EM for giant loci with a TMA bulk-copy pipeline.
//
// Same algorithm and reduction structure as em_grid_kernel (sbq_grid.cuh), different data movement:
//  * one persistent CTA per SM = 16 consumer warps + 1 producer warp;
//  * the CTA's contiguous row range is cut into chunks of C::ROWS rows; the producer lane streams every chunk
//    into a C::NS-deep shared-memory ring with 1-D bulk copies (cp.async.bulk ... mbarrier::complete_tx::bytes,
//    SASS UBLKCP): alpha slab (8 B/nz), 16-bit column slab (2 B/nz), row-pointer slab, count slab. The rows of a
//    CTA are contiguous in CSR, so each slab is one contiguous, 16-byte aligned piece of HBM;
//  * full/empty mbarriers per stage; consumers wait (try_wait.parity), take two rows of the chunk per warp,
//    and release the stage. HBM latency is covered by the ring depth instead of by registers;
//  * columns are pre-narrowed to u16 by grid_prepare_kernel once per upload (10 B of HBM traffic per non-zero and
//    iteration instead of 12; the algorithmic-byte accounting of SURVEY 8d stays 12).
// Reductions (warp-private accumulators -> per-CTA partial -> column owners -> theta') are unchanged and
// deterministic. Chunks whose non-zeros exceed the stage capacity are processed straight from global memory
// by the consumers (both sides skip the ring for them).
#pragma once
#include "sbq_grid.cuh"

namespace sbq {

constexpr int G4_EPL = 2;                    // elements per lane per row on the register path (rows up to 64 non-zeros)
constexpr int G4_MAX_CHUNKS = 2048;          // chunk table entries per CTA
constexpr int G4_CHUNK_BYTES = (((G4_MAX_CHUNKS + 1) * 4 + 127) / 128) * 128;

// Geometry of one kernel instantiation: NC consumer warps (one warp-private accumulator row each) and a ring of
// NS stages. More consumer warps hide more shared-memory / shuffle latency but cost NC * T * 8 B of accumulators,
// so every locus takes the largest NC whose shared memory fits its own T (grid_tma_nc).
template <int NC, int NSTAGE>
struct G4Cfg {
   static constexpr int CONSUMERS = NC;
   static constexpr int ACC = NC;                              // accumulator rows
   static constexpr int ROWS = 2 * NC;                         // rows per chunk (two per consumer warp)
   static constexpr int CAP = 64 * ROWS;                       // non-zeros a stage can hold
   static constexpr int NS = NSTAGE;                           // ring depth
   static constexpr int NT = (NC + 1) * 32;                    // + one producer warp
   // stage layout (bytes): alpha | col16 | row pointers | counts
   static constexpr int A_BYTES = (CAP + 2) * 8;
   static constexpr int C_OFF = A_BYTES;
   static constexpr int C_BYTES = (CAP + 8) * 2 + 16;
   static constexpr int R_OFF = C_OFF + C_BYTES;
   static constexpr int R_BYTES = (ROWS + 4) * 8;
   static constexpr int N_OFF = R_OFF + R_BYTES;
   static constexpr int N_BYTES = (ROWS + 8) * 4;
   static constexpr int STAGE_BYTES = ((N_OFF + N_BYTES + 127) / 128) * 128;
   static_assert(A_BYTES % 16 == 0 && C_OFF % 16 == 0 && R_OFF % 16 == 0 && N_OFF % 16 == 0, "bulk copies need 16-byte alignment");
   static size_t smem_bytes(int T) {   // th[T] | acc[NC][T] | chunk table | ring
      return ((size_t)T * (1 + ACC)) * sizeof(double) + (size_t)G4_CHUNK_BYTES + (size_t)NS * STAGE_BYTES;
   }
};

// consumer warps for a locus of T isoforms: the most whose shared memory fits, 0 if none does. A function of the LOCUS alone
// (the launcher groups loci by it), so that neither the speed nor the summation order of a locus depends on which other loci
// share its batch
inline int grid_tma_nc(int T) {
   const size_t cap = 225 * 1024;
   if (G4Cfg<24, 3>::smem_bytes(T) <= cap) return 24;
   if (G4Cfg<20, 3>::smem_bytes(T) <= cap) return 20;
   if (G4Cfg<16, 4>::smem_bytes(T) <= cap) return 16;
   if (G4Cfg<12, 4>::smem_bytes(T) <= cap) return 12;
   if (G4Cfg<8, 4>::smem_bytes(T) <= cap) return 8;
   return 0;
}

inline bool grid_tma_supports(int T, long long rows, int n_cta) {
   return grid_tma_nc(T) > 0 && T <= 65535 && rows / n_cta + 64 < (long long)G4_MAX_CHUNKS * 16;
}

// One-off prepare pass for giant loci (run once per upload): reorder the non-zeros INSIDE every row (<= 64 entries) so
// that each run of 16 consecutive entries - the unit one half-warp touches in a 64-bit shared-memory access - spreads
// over the 16 eight-byte banks as evenly as the row allows. The EM is invariant to the order of a row's entries; the
// theta gather and the accumulator read-modify-write are indexed by column, bank = column mod 16, and random columns
// cost ~3.1 wavefronts per half-warp instead of 1. Entries are ranked bank-major and dealt round-robin over the row's
// 16-entry groups (closed form below), which gives every bank at most ceil(h_b / groups) entries per group.
// alpha is permuted in place, the u16 column copy is written permuted. One warp per row.
__global__ void __launch_bounds__(256)
grid_prepare_kernel(DevParams p, const int32_t* __restrict__ list, int n_list, unsigned short* __restrict__ col16) {
   const int lane = threadIdx.x & 31;
   const int64_t wid = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5, nw = ((int64_t)gridDim.x * blockDim.x) >> 5;
   double* alpha = const_cast<double*>(p.alpha);
   for (int item = 0; item < n_list; ++item) {
      const int l = list[item];
      const int64_t r0 = p.loc_row_off[l], r1 = p.loc_row_off[l + 1];
      for (int64_t row = r0 + wid; row < r1; row += nw) {
         const int64_t k0 = p.row_ptr[row], k1 = p.row_ptr[row + 1];
         const int len = (int)(k1 - k0);
         if (len > 64 || len <= 16) {   // long rows keep their order; one group cannot be improved
            for (int64_t k = k0 + lane; k < k1; k += 32) col16[k] = (unsigned short)p.col[k];
            continue;
         }
         const bool v0 = lane < len, v1 = lane + 32 < len;
         const double a0 = v0 ? alpha[k0 + lane] : 0.0, a1 = v1 ? alpha[k0 + lane + 32] : 0.0;
         const int c0 = v0 ? p.col[k0 + lane] : 0, c1 = v1 ? p.col[k0 + lane + 32] : 0;
         const unsigned lt = (1u << lane) - 1u;
         int seq0 = 0, seq1 = 0, base = 0;
#pragma unroll
         for (int b = 0; b < 16; ++b) {
            const unsigned m0 = __ballot_sync(0xffffffffu, v0 && (c0 & 15) == b);
            const unsigned m1 = __ballot_sync(0xffffffffu, v1 && (c1 & 15) == b);
            if (v0 && (c0 & 15) == b) seq0 = base + __popc(m0 & lt);
            if (v1 && (c1 & 15) == b) seq1 = base + __popc(m0) + __popc(m1 & lt);
            base += __popc(m0) + __popc(m1);
         }
         // deal the bank-major sequence over G groups of 16 (the last one holds rem entries)
         const int G = (len + 15) >> 4, rem = len - 16 * (G - 1);
         auto place = [&](int seq) {
            if (seq < rem * G) return 16 * (seq % G) + seq / G;
            const int s2 = seq - rem * G;
            return 16 * (s2 % (G - 1)) + rem + s2 / (G - 1);
         };
         __syncwarp();   // every lane has read its entries before anything is overwritten
         if (v0) { const int q = place(seq0); alpha[k0 + q] = a0; col16[k0 + q] = (unsigned short)c0; }
         if (v1) { const int q = place(seq1); alpha[k0 + q] = a1; col16[k0 + q] = (unsigned short)c1; }
      }
   }
}

// n / d for d > 0 finite: hardware reciprocal seed (MUFU.RCP64H), two Newton steps, one residual correction of the
// quotient. Straight-line (no special-case branches); the result is within 1 ulp of the correctly rounded quotient.
__device__ __forceinline__ double fast_div_pos(double n, double d) {
   double y;
   asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(d));
   y = fma(y, fma(-d, y, 1.0), y);
   y = fma(y, fma(-d, y, 1.0), y);
   double q = n * y;
   return fma(y, fma(-d, q, n), q);
}

__device__ __forceinline__ unsigned smem_u32(const void* p) { return (unsigned)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, unsigned count) {
   asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, unsigned bytes) {
   asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
   asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, unsigned parity) {
   asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "WAIT_%=:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
      "@p bra DONE_%=;\n"
      "bra WAIT_%=;\n"
      "DONE_%=:\n"
      "}\n" ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}
__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, unsigned bytes, uint64_t* bar) {
   asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst)), "l"(src),
                "r"(bytes), "r"(smem_u32(bar))
                : "memory");
}

struct G4Ring {
   char* stage;          // NS * STAGE_BYTES
   uint64_t* full;       // [NS]
   uint64_t* empty;      // [NS]
};

// Producer: stream the chunks [0, n_chunk) of this CTA's rows into the ring. `use` counts ring uses across
// passes so that the mbarrier parities stay in step with the consumers.
template <typename C>
__device__ __forceinline__ void g4_produce(const DevParams& p, const unsigned short* __restrict__ col16, const int32_t* __restrict__ cnt_or_neff,
                                           int64_t row_base /* absolute row of local row 0 */, int64_t kb, const unsigned* s_chunk, int ra, int rb,
                                           int n_chunk, const G4Ring& ring, unsigned& use) {
   asm volatile("fence.proxy.async;" ::: "memory");   // neff written with ordinary stores in the setup pass is read by bulk copies
   for (int c = 0; c < n_chunk; ++c) {
      const unsigned ck0 = s_chunk[c], ck1 = s_chunk[c + 1];
      if (ck1 - ck0 > (unsigned)C::CAP) continue;          // oversize chunk: consumers read it from global memory
      const int s = use % C::NS;
      const unsigned n_use = use / C::NS;
      mbar_wait(&ring.empty[s], (n_use & 1u) ^ 1u);
      char* st = ring.stage + (size_t)s * C::STAGE_BYTES;
      const int i0 = ra + c * C::ROWS, i1 = min(i0 + C::ROWS, rb);
      const int64_t k0 = kb + ck0, k1 = kb + ck1;
      const int64_t ka = k0 & ~(int64_t)1, kc = k0 & ~(int64_t)7;
      const unsigned a_bytes = (unsigned)(((k1 - ka + 1) & ~(int64_t)1) * 8);
      const unsigned c_bytes = (unsigned)(((k1 - kc + 7) & ~(int64_t)7) * 2);
      const int64_t g0 = row_base + i0, g1 = row_base + i1;   // absolute rows; need row_ptr[g0 .. g1]
      const int64_t gr = g0 & ~(int64_t)1, gn = g0 & ~(int64_t)3;
      const unsigned r_bytes = (unsigned)(((g1 + 1 - gr + 1) & ~(int64_t)1) * 8);
      const unsigned n_bytes = (unsigned)(((g1 - gn + 3) & ~(int64_t)3) * 4);
      mbar_expect_tx(&ring.full[s], a_bytes + c_bytes + r_bytes + n_bytes);
      if (a_bytes) bulk_g2s(st, p.alpha + ka, a_bytes, &ring.full[s]);
      if (c_bytes) bulk_g2s(st + C::C_OFF, col16 + kc, c_bytes, &ring.full[s]);
      bulk_g2s(st + C::R_OFF, p.row_ptr + gr, r_bytes, &ring.full[s]);
      if (n_bytes) bulk_g2s(st + C::N_OFF, cnt_or_neff + gn, n_bytes, &ring.full[s]);
      ++use;
   }
}

// Consumer side of one pass over the CTA's rows. SETUP: row filter + column sums (+ total / kept counts, neff
// written to global). !SETUP: one E/M pass with the scaled theta in th[].
template <typename C, bool SETUP>
__device__ __forceinline__ void g4_consume(const DevParams& p, const unsigned short* __restrict__ col16, int32_t* neff_glob /* local row 0 */,
                                           const int32_t* __restrict__ cnt_glob, const int64_t* __restrict__ rp_loc, int64_t row_base, int64_t kb,
                                           const unsigned* s_chunk, int ra, int rb, int n_chunk, const G4Ring& ring, unsigned& use,
                                           const double* th, double* my_half /* this half-warp's accumulator row */, int acc_stride,
                                           long long& tot, long long& kept, int& zero) {
   const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
   for (int c = 0; c < n_chunk; ++c) {
      const unsigned ck0 = s_chunk[c], ck1 = s_chunk[c + 1];
      const int i0 = ra + c * C::ROWS, i1 = min(i0 + C::ROWS, rb);
      if (ck1 - ck0 > (unsigned)C::CAP) {
         // oversize chunk, generic path straight from global memory (whole warp per row, half-0 accumulator row)
         double* my = my_half;
         for (int q = warp; i0 + q < i1; q += C::CONSUMERS) {
            const int i = i0 + q;
            const int64_t a = rp_loc[i], b = rp_loc[i + 1];
            if (SETUP) {
               const int n = cnt_glob[i];
               bool keep = false;
               for (int64_t k = a + lane; k < b; k += 32) keep |= p.alpha[k] > p.row_eps;
               keep = __any_sync(0xffffffffu, keep);
               if (lane == 0) { neff_glob[i] = keep ? n : -1; tot += n; kept += keep; }
               if (keep)
                  for (int64_t k = a + lane; k < b; k += 32) my[col16[k]] += p.alpha[k];
            } else {
               const int ne = neff_glob[i];
               if (ne < 0) continue;
               double d = 0.0;
               for (int64_t k = a + lane; k < b; k += 32) d += p.alpha[k] * th[col16[k]];
               d = warp_sum(d);
               if (d == 0) { zero = 1; continue; }
               const double rr = (double)ne / d;
               for (int64_t k = a + lane; k < b; k += 32) { const int cc = col16[k]; my[cc] += p.alpha[k] * th[cc] * rr; }
            }
         }
         continue;
      }
      double* my = my_half;
      const int s = use % C::NS;
      const unsigned n_use = use / C::NS;
      mbar_wait(&ring.full[s], n_use & 1u);
      const char* st = ring.stage + (size_t)s * C::STAGE_BYTES;
      const int64_t k0 = kb + ck0;
      const double* a_s = (const double*)st + (k0 & 1);
      const unsigned short* c_s = (const unsigned short*)(st + C::C_OFF) + (k0 & 7);
      const int64_t g0 = row_base + i0;
      const int64_t* r_s = (const int64_t*)(st + C::R_OFF) + (g0 & 1);
      const int* n_s = (const int*)(st + C::N_OFF) + (g0 & 3);
      const int nrow = i1 - i0;
      // Two rows per warp (rows warp and warp + 16 of the chunk), each spread over all 32 lanes with up to G4_EPL
      // elements per lane held in registers between the normaliser and the accumulation. A row's columns are
      // distinct, so the 32 lanes never collide in the warp-private accumulator row.
      double a[2][G4_EPL];
      int cc[2][G4_EPL], ne[2];
      unsigned rs[2], re[2];
      bool longrow = false;
#pragma unroll
      for (int q = 0; q < 2; ++q) {
         const int rq = warp + q * C::CONSUMERS;
         const bool vr = rq < nrow;
         rs[q] = vr ? (unsigned)(r_s[rq] - k0) : 0u;
         re[q] = vr ? (unsigned)(r_s[rq + 1] - k0) : 0u;
         ne[q] = vr ? n_s[rq] : -1;
         if (!SETUP && ne[q] < 0) re[q] = rs[q];
         longrow |= re[q] - rs[q] > 32u * G4_EPL;
#pragma unroll
         for (int e = 0; e < G4_EPL; ++e) {
            const unsigned k = rs[q] + lane + 32 * e;
            const bool v = k < re[q];
            a[q][e] = v ? a_s[k] : 0.0;
            cc[q][e] = v ? (int)c_s[k] : 0;
         }
      }
      if (!longrow) {
         if (SETUP) {
#pragma unroll
            for (int q = 0; q < 2; ++q) {
               const bool keep = __any_sync(0xffffffffu, a[q][0] > p.row_eps || a[q][1] > p.row_eps);
               const int rq = warp + q * C::CONSUMERS;
               if (rq < nrow) {
                  if (lane == 0) { neff_glob[i0 + rq] = keep ? ne[q] : -1; tot += ne[q]; kept += keep; }
                  if (keep) {
                     if (a[q][0] != 0.0) my[cc[q][0]] += a[q][0];
                     if (a[q][1] != 0.0) my[cc[q][1]] += a[q][1];
                  }
               }
               __syncwarp();   // the second row of the pair may touch the same accumulator column from another lane
            }
         } else {
            double t[2][G4_EPL], d[2];
#pragma unroll
            for (int q = 0; q < 2; ++q) {
               t[q][0] = th[cc[q][0]];
               t[q][1] = th[cc[q][1]];
               d[q] = a[q][0] * t[q][0] + a[q][1] * t[q][1];
            }
            // both normalisers in five shuffles: swap halves (lanes 0-15 collect row 0, lanes 16-31 row 1), then a
            // 4-step butterfly inside each half; lanes 0 and 16 divide; two shuffles broadcast r_0 and r_1
            const bool hi = lane >= 16;
            double v = (hi ? d[1] : d[0]) + __shfl_xor_sync(0xffffffffu, hi ? d[0] : d[1], 16);
#pragma unroll
            for (int o = 8; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
            double rmine = 0.0;
            if ((lane & 15) == 0) {
               const int q = lane >> 4;
               if (re[q] > rs[q]) {
                  if (v == 0) zero = 1; else rmine = (v > 1e-290 && v < 1e290) ? fast_div_pos((double)ne[q], v) : (double)ne[q] / v;
               }
            }
#pragma unroll
            for (int q = 0; q < 2; ++q) {
               const double rr = __shfl_sync(0xffffffffu, rmine, 16 * q);
               if (a[q][0] != 0.0) my[cc[q][0]] += a[q][0] * t[q][0] * rr;
               if (a[q][1] != 0.0) my[cc[q][1]] += a[q][1] * t[q][1] * rr;
               __syncwarp();   // row 1 of the pair may touch the same accumulator column from another lane
            }
         }
      } else {
         // a row longer than 64 non-zeros inside a staged chunk: loop over it in shared memory
         for (int q = 0; q < 2; ++q) {
            const int rq = warp + q * C::CONSUMERS;
            if (rq >= nrow) break;
            if (SETUP) {
               bool keep = false;
               for (unsigned k = rs[q] + lane; k < re[q]; k += 32) keep |= a_s[k] > p.row_eps;
               keep = __any_sync(0xffffffffu, keep);
               if (lane == 0) { neff_glob[i0 + rq] = keep ? ne[q] : -1; tot += ne[q]; kept += keep; }
               if (keep)
                  for (unsigned k = rs[q] + lane; k < re[q]; k += 32) my[c_s[k]] += a_s[k];
            } else {
               if (re[q] == rs[q]) continue;
               double d = 0.0;
               for (unsigned k = rs[q] + lane; k < re[q]; k += 32) d += a_s[k] * th[c_s[k]];
               d = warp_sum(d);
               if (d == 0) { zero = 1; continue; }
               const double rr = (double)ne[q] / d;
               for (unsigned k = rs[q] + lane; k < re[q]; k += 32) { const int c2 = c_s[k]; my[c2] += a_s[k] * th[c2] * rr; }
            }
            __syncwarp();
         }
      }
      __syncwarp();
      if (lane == 0) mbar_arrive(&ring.empty[s]);
      ++use;
   }
}

template <typename C>
__global__ void __launch_bounds__(C::NT, 1)
em_grid_tma_kernel(DevParams p, const unsigned short* __restrict__ col16, const int32_t* __restrict__ list, int n_list, GridScratch gs,
                   double* cur_glob /* [n_cta][tstride] */) {
   cg::grid_group grid = cg::this_grid();
   extern __shared__ __align__(128) unsigned char g4_smem[];
   __shared__ double red[C::NT / 32];
   __shared__ int s_rows[2];
   __shared__ __align__(8) uint64_t s_bar[2 * C::NS];
   const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
   const int nb = gridDim.x, b = blockIdx.x;
   const bool producer = warp == C::CONSUMERS;

   G4Ring ring;
   ring.stage = (char*)g4_smem;
   ring.full = s_bar;
   ring.empty = s_bar + C::NS;
   if (tid == 0) {
      for (int s = 0; s < C::NS; ++s) { mbar_init(&ring.full[s], 1); mbar_init(&ring.empty[s], C::CONSUMERS); }
      asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
   }
   __syncthreads();
   unsigned use = 0;   // ring uses so far (same sequence on the producer and on every consumer warp)
   double* my_cur = cur_glob + (size_t)b * gs.tstride;   // this CTA's copy of theta (L2-resident, touched once per iteration)

   for (int item = 0; item < n_list; ++item) {
      const int l = list[item];
      const int64_t r0 = p.loc_row_off[l];
      const int R = (int)(p.loc_row_off[l + 1] - r0);
      const int64_t t0 = p.loc_iso_off[l];
      const int T = (int)(p.loc_iso_off[l + 1] - t0);
      unsigned* s_chunk = (unsigned*)(g4_smem + (size_t)C::NS * C::STAGE_BYTES);
      double* th = (double*)(g4_smem + (size_t)C::NS * C::STAGE_BYTES + G4_CHUNK_BYTES);
      double* acc = th + T;   // [C::ACC][T]
      const int64_t* __restrict__ rp = p.row_ptr + r0;
      int32_t* neff = p.neff + r0;
      const int32_t* cnt = p.count + r0;
      double* my_partial = gs.partial + (size_t)b * gs.tstride;

      grid_row_range(rp, R, 1, b, nb, s_rows);
      for (int x = tid; x < C::ACC * T; x += C::NT) acc[x] = 0.0;
      __syncthreads();
      const int ra = s_rows[0], rb = s_rows[1];
      const int n_chunk = (rb - ra + C::ROWS - 1) / C::ROWS;
      const int64_t kb = rp[ra];
      for (int c = tid; c <= n_chunk; c += C::NT) s_chunk[c] = (unsigned)(rp[min(ra + c * C::ROWS, rb)] - kb);
      __syncthreads();
      double* my_acc = acc + (size_t)(producer ? 0 : warp) * T;

      // ---- setup pass
      long long tot = 0, kept = 0;
      int zero = 0;
      if (producer) {
         if (lane == 0) g4_produce<C>(p, col16, p.count, r0, kb, s_chunk, ra, rb, n_chunk, ring, use);
         use = __shfl_sync(0xffffffffu, use, 0);
      } else {
         g4_consume<C, true>(p, col16, neff, cnt, rp, r0, kb, s_chunk, ra, rb, n_chunk, ring, use, th, my_acc, T, tot, kept, zero);
      }
      grid_publish_counts(gs, item, tot, kept);
      __threadfence();
      asm volatile("fence.proxy.async;" ::: "memory");
      __syncthreads();
      for (int j = tid; j < T; j += C::NT) {
         double sj = 0.0;
         for (int w = 0; w < C::ACC; ++w) { sj += acc[(size_t)w * T + j]; acc[(size_t)w * T + j] = 0.0; }
         my_partial[j] = sj;
      }
      grid_owner_reduce<C::NT>(grid, gs, T);
      const double total = (double)__ldcg(gs.ctr + 2 * item);
      const long long kept_all = __ldcg(gs.ctr + 2 * item + 1);
      const double theta0 = total / (double)T;
      // s_j is kept in the upper half of this CTA's theta copy: my_cur[j] = theta_j, my_cur[tstride/2 + j] = s_j
      double* my_sdiv = my_cur + gs.tstride / 2;
      for (int j = tid; j < T; j += C::NT) {
         my_sdiv[j] = __ldcg(gs.theta_next + j);
         my_cur[j] = theta0;
         th[j] = theta0;
      }
      grid.sync();   // theta_next is rewritten in iteration 0 only after everyone copied s_j out

      const double tol2 = p.tol * p.tol;
      int status = LOCUS_ITER_CAP, iters = 0;
      if (kept_all == 0) {
         status = LOCUS_NO_ROWS;
      } else {
         for (int it = 0; it < p.max_iter; ++it) {
            iters = it + 1;
            zero = 0;
            long long d0 = 0, d1 = 0;
            if (producer) {
               if (lane == 0) g4_produce<C>(p, col16, p.neff, r0, kb, s_chunk, ra, rb, n_chunk, ring, use);
               use = __shfl_sync(0xffffffffu, use, 0);
            } else {
               g4_consume<C, false>(p, col16, neff, cnt, rp, r0, kb, s_chunk, ra, rb, n_chunk, ring, use, th, my_acc, T, d0, d1, zero);
            }
            zero = __syncthreads_or(zero);
            if (zero && tid == 0) atomicOr(&gs.zero_flag[item], 1);
            for (int j = tid; j < T; j += C::NT) {
               double sj = 0.0;
               for (int w = 0; w < C::ACC; ++w) { sj += acc[(size_t)w * T + j]; acc[(size_t)w * T + j] = 0.0; }
               my_partial[j] = sj;
            }
            grid_owner_reduce<C::NT>(grid, gs, T);
            const int zf = *(volatile int*)&gs.zero_flag[item];
            const double d2 = grid_read_next<C::NT>(gs, my_cur, th, T, red);
            if (zf) { status = LOCUS_ZERO_DENOM; break; }
            if (d2 < tol2) { status = LOCUS_OK; break; }
            for (int j = tid; j < T; j += C::NT) {
               const double nj = th[j];
               my_cur[j] = nj;
               const double sj = my_sdiv[j];
               th[j] = (sj != 0) ? nj / sj : 0.0;
            }
            __syncthreads();
         }
      }

      // ---- outputs + epilogue by CTA 0 (src/estimate.cpp:310-356)
      if (b == 0) {
         locus_epilogue_block<C::NT>(p, l, t0, T, status, iters, theta0, my_cur, th, red);
      }
      grid.sync();   // scratch (partial, theta_next) is reused by the next locus
   }
}

// One cooperative launch of the TMA path for loci of up to max_iso isoforms (the u16 columns are in place).
template <typename C>
inline int grid_tma_launch_cfg(const DevParams& dp, const int32_t* d_list, int n_list, int max_iso, const cudaDeviceProp& prop, DevBuf& scratch,
                               const unsigned short* c16, cudaStream_t st, int* n_launch) {
   const size_t smem = C::smem_bytes(max_iso);
   auto kernel = em_grid_tma_kernel<C>;
   if (cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess) return -3;
   int per_sm = 0;
   if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, C::NT, smem) != cudaSuccess || per_sm < 1) return -3;
   const int nb = prop.multiProcessorCount;
   GridScratch gs;
   double* cur_glob = nullptr;
   // tstride 8192: theta copy in the lower half, s_j in the upper half
   if (const int rc = grid_scratch(scratch, nb, 8192, n_list, &cur_glob, st, &gs)) return rc;
   DevParams dpc = dp;
   void* args[] = {(void*)&dpc, (void*)&c16, (void*)&d_list, (void*)&n_list, (void*)&gs, (void*)&cur_glob};
   if (cudaLaunchCooperativeKernel((void*)kernel, dim3(nb), dim3(C::NT), args, smem, st) != cudaSuccess) return -3;
   ++*n_launch;
   return 0;
}

// Host launcher of the TMA path. h_iso: T of every list entry (host); the planner sorts the list by grid_tma_nc. c16: the u16
// columns of the whole batch (the caller sizes the buffer); cols_ready: the prepare pass of this upload already filled it.
inline int grid_tma_launch(const DevParams& dp, const int32_t* d_list, int n_list, const int* h_iso, const cudaDeviceProp& prop, DevBuf& scratch,
                           unsigned short* c16, bool cols_ready, cudaStream_t st, int* n_launch) {
   *n_launch = 0;
   if (n_list == 0) return 0;
   if (!cols_ready) {
      grid_prepare_kernel<<<prop.multiProcessorCount * 8, 256, 0, st>>>(dp, d_list, n_list, c16);
      ++*n_launch;
   }
   return grid_for_each_run(h_iso, n_list, grid_tma_nc, [&](int i0, int i1, int nc, int mx) {
      const int32_t* li = d_list + i0;
      switch (nc) {
         case 24: return grid_tma_launch_cfg<G4Cfg<24, 3>>(dp, li, i1 - i0, mx, prop, scratch, c16, st, n_launch);
         case 20: return grid_tma_launch_cfg<G4Cfg<20, 3>>(dp, li, i1 - i0, mx, prop, scratch, c16, st, n_launch);
         case 16: return grid_tma_launch_cfg<G4Cfg<16, 4>>(dp, li, i1 - i0, mx, prop, scratch, c16, st, n_launch);
         case 12: return grid_tma_launch_cfg<G4Cfg<12, 4>>(dp, li, i1 - i0, mx, prop, scratch, c16, st, n_launch);
         case 8: return grid_tma_launch_cfg<G4Cfg<8, 4>>(dp, li, i1 - i0, mx, prop, scratch, c16, st, n_launch);
         default: return -6;
      }
   });
}

}  // namespace sbq

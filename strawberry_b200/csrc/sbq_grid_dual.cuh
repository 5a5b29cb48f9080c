// sbq_grid_dual.cuh - Tier 3, fast path: multi-CTA streaming EM for giant loci over a BANK-ALIGNED, TWO-CHOICE row layout.
//
// The TMA ring kernel of sbq_grid_tma.cuh is bound by the shared-memory pipe, not by HBM: the theta gather and the
// accumulator read-modify-write are 64-bit accesses indexed by column, and the 16 lanes of a half-warp that work on
// one row hit the 16 eight-byte banks unevenly - the fullest bank of a 48-entry row holds ~7 entries where 3 would be
// ideal, so every such access costs ~7 wavefronts instead of 3. This kernel removes the conflicts by construction:
//
//  * TWO SLOTS PER COLUMN. theta and the warp-private accumulators are kept twice: slot A(j) = j (bank j mod 16) and
//    slot B(j) = Tp + 16*(j/16) + ((j + j/16) mod 16) (the column's 16-block rotated by the block index: a different
//    bank). Every non-zero may use either slot of its column, which turns "48 balls into 16 bins" into a two-choice
//    allocation: the fullest bank drops from ~7 to ~3.85 entries.
//  * dual_prepare_kernel (once per upload; a warp stages 32 rows, every lane allocates one row, the warp permutes) picks the
//    slot of every non-zero (greedy least-loaded bank + two improvement sweeps) and re-sorts the row IN PLACE inside its
//    CSR range into a jagged-diagonal order: step-major, within a step one entry per bank, banks ranked by load. Lane x
//    of a half-warp then only ever touches bank rank x: the alpha / column reads are contiguous and the theta gather and
//    the accumulator update are conflict-free. Rows r and r + 4 of every 8-row group - the rows the two half-warps of a
//    warp work on at the same time - get DISJOINT slot sets (a column both hold takes slot A in one and slot B in the
//    other), so both half-warps update the accumulators in the same instructions. The u16 column copy holds the slot as a
//    byte offset (slot * 8); a 16-byte record per row holds the per-step entry counts, the effective count, the row's
//    offset and a summary byte of its 8-row group (it replaces row pointer + count in the stream: same bytes).
//  * em_grid_dual_kernel: persistent cooperative kernel, one CTA of NC warps per SM, no producer warp: warp w takes the
//    8-row chunks w, w + NC, ... of the CTA's rows and owns a private shared-memory stage that it refills itself
//    (alpha slab, u16 slab, record slab - three 1-D TMA bulk copies issued by lane 0, one mbarrier per stage) AS SOON AS
//    the chunk sits in registers, so the copy overlaps the E- and M-phase of the same chunk. Eight rows per warp are in
//    flight (four per half-warp): loads (step-major: independent rows adjacent in the instruction stream), theta gather
//    and products, a transposing four-row shuffle reduction, one normaliser division per lane, then the accumulator
//    update - four dependent load-add-store blocks per turn. A lane without an entry in a step works on a dummy slot of
//    its own (theta = 0), so the steps are branch-free; straight-line bodies exist for 4, 5 and 6 steps.
//  * reductions (warp-private accumulators -> per-CTA partial -> column owners -> theta') are those of the other grid
//    kernels: fixed order, no floating-point atomics. Both slots of a column are summed there.
//
// Rows with more than 96 non-zeros, with columns that are not strictly ascending, or whose fullest bank still holds more
// than 6 entries keep their CSR order (flag in the record) and are walked by a whole warp from global memory, as are the
// rows of a chunk fuller than a stage. Eligibility (host planner, per locus): T <= 4048 and shared memory for at least
// 8 warps (T <~ 1300), locus non-zeros < 2^32, on average <= 56 non-zeros per row. Anything else runs on
// em_grid_tma_kernel / em_grid_kernel.
#pragma once
#include "sbq_grid_tma.cuh"

namespace sbq {

constexpr int G6_LMAX = 6;                       // steps of the register path (fullest bank of a row)
constexpr int G6_MAXROW = 96;                    // longest row the sorted layout takes
constexpr unsigned char G6_FLAG = 255;           // cnt[0] of a row left in CSR order

struct __align__(16) RowRec {
   unsigned char cnt[8];     // cnt[e], e < 6: entries of step e (<= 16, descending); cnt[7]: number of steps;
                             // cnt[6]: summary of the row's 8-row group: most steps of its rows | 0x80 if a row of it is left in CSR order
   int32_t neff;             // effective count (-1: dropped by the row filter)
   uint32_t koff;            // first non-zero of the row, relative to the locus' first non-zero
};
static_assert(sizeof(RowRec) == 16, "one 16-byte unit per row");

constexpr int G6_NR = 4;                         // rows a half-warp keeps in flight
constexpr int G6_MAX_SPW = 4;                    // ring stages per warp (at most)
constexpr int G6_MAX_WARPS = 16;
constexpr int G6_MAX_ISO = 4048;                 // slot * 8 must fit the u16 stream: (2 Tp + 64) * 8 <= 65535

// Packed chunk stream (written once per upload by dual_pack_kernel): everything a warp turn needs - the chunk's 8 + 1 row records,
// its weights and its u16 slots - lies back to back at a fixed stride, so a stage is refilled by ONE bulk copy instead of three
// (issuing the three copies plus the proxy fence took ~590 of the ~3 650 cycles of a turn on the thread that issues them).
//   chunk g of a locus:  [ 9 records, 144 B | alpha, n x 8 B rounded up to 16 B | slots, n x 2 B rounded up to 16 B ]   at g * G6_PK_STRIDE
// A chunk with more than G6_PK_CAP non-zeros only carries its records (its rows are walked from the CSR arrays).
constexpr int G6_PK_ROWS = 2 * G6_NR;                                    // rows per chunk
constexpr int G6_PK_CAP = G6_PK_ROWS * 56;                               // non-zeros a staged chunk holds at most
constexpr int G6_PK_RECS = (G6_PK_ROWS + 1) * (int)sizeof(RowRec);       // 144 B
constexpr int G6_PK_STRIDE = ((G6_PK_RECS + ((G6_PK_CAP + 1) & ~1) * 8 + ((G6_PK_CAP + 7) & ~7) * 2 + 127) / 128) * 128;   // 4 736 B
__host__ __device__ __forceinline__ unsigned g6_pk_abytes(unsigned n) { return ((n + 1u) & ~1u) * 8u; }
__host__ __device__ __forceinline__ unsigned g6_pk_cbytes(unsigned n) { return ((n + 7u) & ~7u) * 2u; }

__host__ __device__ __forceinline__ int g6_tp(int T) { return (T + 15) & ~15; }
__host__ __device__ __forceinline__ int g6_slot_b(int j, int Tp) { return Tp + (j & ~15) + ((j + (j >> 4)) & 15); }

// Geometry: NC warps per CTA, every one a consumer that also streams its own chunks: warp w takes the chunks
// w, w + NC, ... of the CTA (8 rows each) and owns SPW private ring stages. After a chunk is done its stage is refilled
// with the warp's chunk SPW turns ahead (three 1-D bulk copies issued by lane 0) - no producer warp, no "empty"
// barriers. (A dedicated producer thread tops out at one 8-row chunk per ~860 cycles - 90 cycles per try_wait plus the
// copies - which caps the kernel at 0.37 ms per pass; measured.)
template <int NC>
struct G6Cfg {
   static constexpr int CONSUMERS = NC;
   static constexpr int NT = NC * 32;
   static constexpr int CROWS = G6_PK_ROWS;               // rows per chunk (four per half-warp)
   static constexpr int CAP = G6_PK_CAP;                  // non-zeros a stage holds; fuller chunks are read from global memory
   // stage layout (bytes) = the packed chunk: records | alpha | slots. Lanes past a step's last entry still read (and discard)
   // up to 18 weights and 16 slots behind the chunk's own: the stage leaves room for that (those bytes are older weights or
   // slots - finite as doubles for every T this kernel takes - never NaN, so "alpha x theta[dummy] = 0" holds).
   static constexpr int A_OFF = G6_PK_RECS;
   static constexpr int STAGE_BYTES = G6_PK_STRIDE;
   static_assert(G6_PK_RECS + ((G6_PK_CAP + 1) & ~1) * 8 + (G6_PK_CAP + 16 + 8) * 2 <= STAGE_BYTES, "room for the slot over-read behind the fullest chunk");
   static size_t fixed_bytes(int T) { return (size_t)(2 * g6_tp(T) + 64) * (1 + NC) * sizeof(double); }   // th2[2Tp+64] | acc[NC][2Tp+64]
   static int stages_per_warp(int T) {   // ring depth per warp that fits beside the accumulators
      // 227 KB usable per CTA (232 448 B) minus the kernel's static shared memory (640 B) and a little slack: T = 800 still gets
      // twelve warps (173 056 B of theta + accumulators + 12 x 4 864 B of stages)
      const long long room = 231680LL - (long long)fixed_bytes(T);
      long long spw = room / ((long long)STAGE_BYTES * NC);
      if (spw > G6_MAX_SPW) spw = G6_MAX_SPW;
      return (int)spw;
   }
   static bool fits(int T, int spw_min = 2) { return stages_per_warp(T) >= spw_min; }
};

// ------------------------------------------------------------------------------------------------------------------
// prepare: a warp takes 32 consecutive rows. The rows' bank pairs are staged in shared memory by the whole warp, then
// every LANE runs the (sequential) two-choice allocation of one row, then the whole warp permutes the rows in place.
// ------------------------------------------------------------------------------------------------------------------
constexpr int G6_PREP_WARPS = 8;
constexpr int G6_PSTRIDE = G6_MAXROW + 1;   // odd byte stride between the rows of a tile

struct G6PrepTile {
   unsigned char bank_a[32][G6_PSTRIDE];   // bit 0-3: bank of slot A, bit 7: the entry uses slot B; finally (destination | slot choice << 7)
   unsigned char bank_b[32][G6_PSTRIDE];   // bank of slot B
   unsigned char col_hi[32][G6_PSTRIDE];   // column >> 4 (column = col_hi << 4 | bank of slot A)
   unsigned char load[16][32], fill[16][32], pos[16][32];   // per-lane scratch, [bank][lane]: conflict-free
   unsigned char pre[G6_LMAX + 1][32];
   unsigned char cnt[32][8];               // record bytes of the 32 rows
   unsigned char cand[32];                 // row takes part in the sorted layout so far
};

// Rows r and r + 4 of an 8-row group are updated TOGETHER by the two half-warps of a warp (em_grid_dual_kernel, M-phase),
// so their slot sets must be disjoint: a column both rows hold gets slot A in one row and slot B in the other.
__global__ void __launch_bounds__(G6_PREP_WARPS * 32)
dual_prepare_kernel(DevParams p, const int32_t* __restrict__ list, int n_list, const int64_t* __restrict__ rec_off, RowRec* __restrict__ recs,
                    unsigned short* __restrict__ col16) {
   extern __shared__ __align__(16) unsigned char g6_prep_smem[];
   const int lane = threadIdx.x & 31;
   G6PrepTile& tl = reinterpret_cast<G6PrepTile*>(g6_prep_smem)[threadIdx.x >> 5];
   const int64_t wid = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5, nw = ((int64_t)gridDim.x * blockDim.x) >> 5;
   double* alpha = const_cast<double*>(p.alpha);
   for (int item = 0; item < n_list; ++item) {
      const int l = list[item];
      const int64_t r0 = p.loc_row_off[l];
      const int64_t R = p.loc_row_off[l + 1] - r0;
      const int T = (int)(p.loc_iso_off[l + 1] - p.loc_iso_off[l]);
      const int Tp = g6_tp(T);
      const int64_t* __restrict__ rp = p.row_ptr + r0;
      const int64_t kbase = rp[0];
      RowRec* rec_l = recs + rec_off[item];
      if (wid == 0 && lane < 8) {   // sentinel record R: its offset closes the last chunk
         rec_l[R].cnt[lane] = 0;
         if (lane == 0) { rec_l[R].neff = -1; rec_l[R].koff = (uint32_t)(rp[R] - kbase); }
      }
      for (int64_t tile0 = wid * 32; tile0 < R; tile0 += nw * 32) {   // tiles start at multiples of 32 rows: whole 8-row groups
         const int nrow = (int)min((int64_t)32, R - tile0);
         const int64_t my_k0 = lane < nrow ? rp[tile0 + lane] : 0, my_k1 = lane < nrow ? rp[tile0 + lane + 1] : 0;
         const int my_n = (int)min((int64_t)(G6_MAXROW + 1), my_k1 - my_k0);
         tl.cand[lane] = lane < nrow && my_n <= G6_MAXROW;
         __syncwarp();
         // phase A (whole warp): stage bank pairs and column high bits of the 32 rows; a row whose columns are not strictly
         // ascending (the pairing below merges two rows' column lists) stays in CSR order
         for (int r = 0; r < nrow; ++r) {
            const int64_t k0 = __shfl_sync(0xffffffffu, my_k0, r);
            const int n = __shfl_sync(0xffffffffu, my_n, r);
            if (n > G6_MAXROW) continue;
            bool bad = false;
            for (int idx = lane; idx < n; idx += 32) {
               const int c = p.col[k0 + idx];
               if (idx > 0 && p.col[k0 + idx - 1] >= c) bad = true;
               tl.bank_a[r][idx] = (unsigned char)(c & 15);
               tl.bank_b[r][idx] = (unsigned char)((c + (c >> 4)) & 15);
               tl.col_hi[r][idx] = (unsigned char)(c >> 4);
            }
            if (__any_sync(0xffffffffu, bad) && lane == 0) tl.cand[r] = 0;
         }
         __syncwarp();
         // phase B1 (lane = row): two-choice allocation - greedy least-loaded bank, then two sweeps that move an entry to its
         // other bank when that lowers the larger of the two loads
         const bool cand = tl.cand[lane];
         if (cand) {
            const int n = my_n;
#pragma unroll
            for (int b = 0; b < 16; ++b) tl.load[b][lane] = 0;
            for (int e = 0; e < n; ++e) {
               const int ba = tl.bank_a[lane][e], bb = tl.bank_b[lane][e];
               const bool pk = tl.load[bb][lane] < tl.load[ba][lane];
               if (pk) tl.bank_a[lane][e] = (unsigned char)(ba | 0x80);
               ++tl.load[pk ? bb : ba][lane];
            }
            for (int sweep = 0; sweep < 2; ++sweep) {
               for (int e = 0; e < n; ++e) {
                  const int va = tl.bank_a[lane][e], ba = va & 15, bb = tl.bank_b[lane][e];
                  const bool pk = va & 0x80;
                  const int cur = pk ? bb : ba, alt = pk ? ba : bb;
                  if (tl.load[cur][lane] > tl.load[alt][lane] + 1) {
                     --tl.load[cur][lane];
                     ++tl.load[alt][lane];
                     tl.bank_a[lane][e] = (unsigned char)(va ^ 0x80);
                  }
               }
            }
         }
         __syncwarp();
         // phase B2 (one lane per pair of rows r, r + 4): a column held by both rows must use different slots
         const int n_partner = __shfl_sync(0xffffffffu, my_n, lane ^ 4);
         if ((lane & 4) == 0 && cand && tl.cand[lane + 4]) {
            const int r1 = lane, r2 = lane + 4, n1 = my_n, n2 = n_partner;
            int e1 = 0, e2 = 0;
            while (e1 < n1 && e2 < n2) {
               const int v1 = tl.bank_a[r1][e1], v2 = tl.bank_a[r2][e2];
               const int c1 = (tl.col_hi[r1][e1] << 4) | (v1 & 15), c2 = (tl.col_hi[r2][e2] << 4) | (v2 & 15);
               if (c1 < c2) { ++e1; continue; }
               if (c2 < c1) { ++e2; continue; }
               if ((v1 & 0x80) == (v2 & 0x80)) {
                  // same slot in both rows: flip the entry whose other bank is the emptier one
                  const int ba = v1 & 15, bb = tl.bank_b[r1][e1];   // same column: same bank pair in both rows
                  const bool pk = v1 & 0x80;
                  const int cur = pk ? bb : ba, alt = pk ? ba : bb;
                  const int rr = tl.load[alt][r1] <= tl.load[alt][r2] ? r1 : r2;
                  --tl.load[cur][rr];
                  ++tl.load[alt][rr];
                  if (rr == r1) tl.bank_a[r1][e1] = (unsigned char)(v1 ^ 0x80);
                  else tl.bank_a[r2][e2] = (unsigned char)(v2 ^ 0x80);
               }
               ++e1;
               ++e2;
            }
         }
         __syncwarp();
         // phase B3 (lane = row): step layout
         bool sorted = cand;
         if (sorted) {
            const int n = my_n;
            int L = 0;
#pragma unroll
            for (int b = 0; b < 16; ++b) L = max(L, (int)tl.load[b][lane]);
            sorted = L <= G6_LMAX;
            if (sorted) {
               // banks ranked by (load desc, bank asc) -> lane position; per-step entry counts and their prefix
               for (int b = 0; b < 16; ++b) {
                  const int lb = tl.load[b][lane];
                  int ps = 0;
#pragma unroll
                  for (int y = 0; y < 16; ++y) { const int ly = tl.load[y][lane]; ps += (ly > lb) || (ly == lb && y < b); }
                  tl.pos[b][lane] = (unsigned char)ps;
                  tl.fill[b][lane] = 0;
               }
               int acc = 0, steps = 0;
               for (int s = 0; s <= G6_LMAX; ++s) {
                  tl.pre[s][lane] = (unsigned char)acc;
                  int cn = 0;
#pragma unroll
                  for (int b = 0; b < 16; ++b) cn += tl.load[b][lane] > s;
                  if (s < G6_LMAX) { tl.cnt[lane][s] = (unsigned char)cn; steps += cn > 0; }
                  acc += cn;
               }
               tl.cnt[lane][7] = (unsigned char)steps;
               for (int e = 0; e < n; ++e) {
                  const int va = tl.bank_a[lane][e];
                  const bool pk = va & 0x80;
                  const int bk = pk ? tl.bank_b[lane][e] : (va & 15);
                  const int sq = tl.fill[bk][lane]++;
                  tl.bank_a[lane][e] = (unsigned char)((tl.pre[sq][lane] + tl.pos[bk][lane]) | (pk ? 0x80 : 0));
               }
            }
         }
         if (lane < nrow && !sorted) {
#pragma unroll
            for (int s = 0; s < 8; ++s) tl.cnt[lane][s] = s == 0 ? G6_FLAG : 0;
         }
         {  // summary of every 8-row group (8 consecutive lanes): most steps, any row left in CSR order
            int gs = (lane < nrow && sorted) ? (int)tl.cnt[lane][7] : 0;
            int gf = (lane < nrow && !sorted) ? 1 : 0;
#pragma unroll
            for (int o = 1; o < 8; o <<= 1) {
               gs = max(gs, __shfl_xor_sync(0xffffffffu, gs, o));
               gf |= __shfl_xor_sync(0xffffffffu, gf, o);
            }
            if (lane < nrow) tl.cnt[lane][6] = (unsigned char)(gs | (gf ? 0x80 : 0));
         }
         __syncwarp();
         // phase C (whole warp): permute the rows in place (alpha) and write slots and records
         for (int r = 0; r < nrow; ++r) {
            const int64_t k0 = __shfl_sync(0xffffffffu, my_k0, r), k1 = __shfl_sync(0xffffffffu, my_k1, r);
            const bool srt = __shfl_sync(0xffffffffu, (int)sorted, r);
            RowRec* rec = rec_l + tile0 + r;
            if (lane < 8) rec->cnt[lane] = tl.cnt[r][lane];
            if (lane == 0) { rec->neff = -1; rec->koff = (uint32_t)(k0 - kbase); }
            if (!srt) {   // left in CSR order with plain (slot A) columns; the EM kernel walks it from global memory
               for (int64_t k = k0 + lane; k < k1; k += 32) col16[k] = (unsigned short)(p.col[k] << 3);
               continue;
            }
            const int n = (int)(k1 - k0);
            double a[3];
            int c[3];
#pragma unroll
            for (int m = 0; m < 3; ++m) {
               const int idx = lane + 32 * m;
               a[m] = idx < n ? alpha[k0 + idx] : 0.0;
               c[m] = idx < n ? p.col[k0 + idx] : 0;
            }
            __syncwarp();   // the row is in registers before any of it is overwritten
#pragma unroll
            for (int m = 0; m < 3; ++m) {
               const int idx = lane + 32 * m;
               if (idx < n) {
                  const unsigned d = tl.bank_a[r][idx];
                  alpha[k0 + (d & 0x7fu)] = a[m];
                  col16[k0 + (d & 0x7fu)] = (unsigned short)(((d & 0x80u) ? g6_slot_b(c[m], Tp) : c[m]) << 3);
               }
            }
         }
         __syncwarp();
      }
   }
}

// Debug check of the prepared layout (SBQ_DUAL_VERIFY=1; used by the tests): one warp per 8-row group counts (a) steps whose
// entries do not sit in 16 distinct banks, (b) slots held by both rows r and r + 4 of the group, (c) slots repeated in a row.
__global__ void __launch_bounds__(256)
dual_verify_kernel(DevParams p, const int32_t* __restrict__ list, int n_list, const int64_t* __restrict__ rec_off, const RowRec* __restrict__ recs,
                   const unsigned short* __restrict__ col16, int* __restrict__ violations) {
   const int lane = threadIdx.x & 31;
   const int64_t wid = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5, nw = ((int64_t)gridDim.x * blockDim.x) >> 5;
   for (int item = 0; item < n_list; ++item) {
      const int l = list[item];
      const int64_t r0 = p.loc_row_off[l];
      const int64_t R = p.loc_row_off[l + 1] - r0;
      const int64_t kbase = p.row_ptr[r0];
      const RowRec* rec_l = recs + rec_off[item];
      for (int64_t g = wid; g * 8 < R; g += nw) {
         int bad = 0;
         for (int q = 0; q < 8; ++q) {
            const int64_t row = g * 8 + q;
            if (row >= R || rec_l[row].cnt[0] == G6_FLAG) continue;
            const int64_t k0 = kbase + rec_l[row].koff, k1 = kbase + rec_l[row + 1].koff;
            // (a) banks inside every step
            int64_t k = k0;
            int total = 0;
            for (int e = 0; e < G6_LMAX; ++e) {
               const int ce = rec_l[row].cnt[e];
               const int bank = lane < ce ? (col16[k + lane] >> 3) & 15 : -1 - lane;
               for (int y = 0; y < 16; ++y) {
                  const int by = __shfl_sync(0xffffffffu, bank, y);
                  if (lane < ce && y != lane && by == bank) bad = 1;
               }
               if (ce > 16) bad = 1;
               k += ce;
               total += ce;
            }
            if (total != (int)(k1 - k0)) bad = 1;
            // (c) slots inside the row, (b) against the partner row
            const int64_t prow = row + 4;
            const bool pair = (q & 4) == 0 && prow < R && rec_l[prow].cnt[0] != G6_FLAG;
            const int64_t pk0 = pair ? kbase + rec_l[prow].koff : 0, pk1 = pair ? kbase + rec_l[prow + 1].koff : 0;
            for (int64_t x = k0 + lane; x < k1; x += 32) {
               const unsigned short sx = col16[x];
               for (int64_t y = k0; y < k1; ++y)
                  if (y != x && col16[y] == sx) bad = 1;
               for (int64_t y = pk0; y < pk1; ++y)
                  if (col16[y] == sx) bad = 1;
            }
         }
         if (__any_sync(0xffffffffu, bad) && lane == 0) atomicAdd(violations, 1);
      }
   }
}

// One warp per chunk: copy the chunk's records, weights and slots (all final after dual_prepare_kernel) into the packed stream.
__global__ void __launch_bounds__(256)
dual_pack_kernel(DevParams p, const int32_t* __restrict__ list, int n_list, const int64_t* __restrict__ rec_off, const RowRec* __restrict__ recs,
                 const unsigned short* __restrict__ col16, const int64_t* __restrict__ pk_off, unsigned char* __restrict__ pk) {
   const int lane = threadIdx.x & 31;
   const int64_t wid = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5, nw = ((int64_t)gridDim.x * blockDim.x) >> 5;
   for (int item = 0; item < n_list; ++item) {
      const int l = list[item];
      const int64_t r0 = p.loc_row_off[l];
      const int64_t R = p.loc_row_off[l + 1] - r0;
      const int64_t kbase = p.row_ptr[r0];
      const RowRec* rec_l = recs + rec_off[item];
      const int64_t n_chunk = (R + G6_PK_ROWS - 1) / G6_PK_ROWS;
      for (int64_t g = wid; g < n_chunk; g += nw) {
         const int64_t i0 = g * G6_PK_ROWS, i1 = min(i0 + (int64_t)G6_PK_ROWS, R);
         unsigned char* dst = pk + (size_t)(pk_off[item] + g) * G6_PK_STRIDE;
         const uint32_t ck0 = rec_l[i0].koff, ck1 = rec_l[i1].koff;
         if (lane <= G6_PK_ROWS) {
            uint4 v = make_uint4(0u, 0u, 0xffffffffu, ck1);      // rows the chunk does not have: no entries, dropped, offset = end
            if (i0 + lane <= i1) v = *reinterpret_cast<const uint4*>(rec_l + i0 + lane);
            *reinterpret_cast<uint4*>(dst + lane * 16) = v;
         }
         const unsigned n = ck1 - ck0;
         if (n <= (unsigned)G6_PK_CAP) {
            double* da = reinterpret_cast<double*>(dst + G6_PK_RECS);
            unsigned short* dc = reinterpret_cast<unsigned short*>(dst + G6_PK_RECS + g6_pk_abytes(n));
            const int64_t k0 = kbase + ck0;
            for (unsigned x = lane; x < ((n + 1u) & ~1u); x += 32) da[x] = x < n ? p.alpha[k0 + x] : 0.0;
            for (unsigned x = lane; x < ((n + 7u) & ~7u); x += 32) dc[x] = x < n ? col16[k0 + x] : (unsigned short)0;
         }
      }
   }
}

// ------------------------------------------------------------------------------------------------------------------
// consumer side
// ------------------------------------------------------------------------------------------------------------------
#ifdef SBQ_G6_PHASES
// debug build: clock cycles a warp spends per phase of its turns (printed by lane 0 of warp 0 of CTA 0 per locus)
struct G6Phases { long long wait, decode, load, refill, ephase, mphase, other, turns; };
__device__ G6Phases g6_ph;
#define G6_TICK(field) { const long long now_ = clock64(); if ((threadIdx.x & 31) == 0 && threadIdx.x < 32 && blockIdx.x == 0) g6_ph.field += now_ - g6_t_; g6_t_ = now_; }
#define G6_TICK_DECL long long g6_t_ = clock64();
#else
#define G6_TICK(field)
#define G6_TICK_DECL
#endif

struct G6Ring {      // the private ring of one warp
   char* stage;      // spw stages
   uint64_t* full;   // [spw]
   int spw;
   int next;         // stage of the next chunk this warp consumes
   unsigned phase;   // bit s: parity the next wait on stage s expects
};

__device__ __forceinline__ double g6_half_sum(double v) {   // sum over the 16 lanes of a half-warp
#pragma unroll
   for (int o = 8; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
   return v;
}

// A row walked by the whole warp straight from global memory (any entry order; columns are slots).
template <bool SETUP>
__device__ __forceinline__ void g6_walk_row(const DevParams& p, const unsigned short* __restrict__ col16, RowRec* rec_g, int64_t a, int64_t b, int n_i,
                                            int32_t* neff_row, const double* th2, double* my, long long& tot, long long& kept, int& zero) {
   const int lane = threadIdx.x & 31;
   if (SETUP) {
      bool keep = false;
      for (int64_t k = a + lane; k < b; k += 32) keep |= p.alpha[k] > p.row_eps;
      keep = __any_sync(0xffffffffu, keep);
      if (lane == 0) { rec_g->neff = keep ? n_i : -1; *neff_row = keep ? n_i : -1; tot += n_i; kept += keep; }
      if (keep)
         for (int64_t k = a + lane; k < b; k += 32) my[col16[k] >> 3] += p.alpha[k];
   } else {
      const int ne = rec_g->neff;
      if (ne >= 0) {
         double d = 0.0;
         for (int64_t k = a + lane; k < b; k += 32) d += p.alpha[k] * th2[col16[k] >> 3];
         d = warp_sum(d);
         if (d == 0) {
            zero = 1;
         } else {
            const double rr = (double)ne / d;
            for (int64_t k = a + lane; k < b; k += 32) { const int cc = col16[k] >> 3; my[cc] += p.alpha[k] * th2[cc] * rr; }
         }
      }
   }
   __syncwarp();
}

// One warp turn on a staged chunk: G6_NR rows per half-warp, all in flight. rec0: record of the half-warp's first row in
// the stage; n_here: how many of its G6_NR rows exist. a_s / c_s: entry 0 of the chunk in the stage. Returns the mask of
// rows (bit q, this half-warp) that must be walked instead (flagged).
//
// Branch-free inner steps: a lane that holds no entry in a step works on its DUMMY slot instead - slot 2 Tp + (bank of
// the lane's step-0 entry), which lies in the lane's own bank (no conflict with the other lanes), reads theta = 0 and
// accumulates zeros. Lanes without any entry in the row (fewer than 16 banks used) sit the row out.
template <bool SETUP, int LS, typename Refill>
__device__ __forceinline__ void g6_turn_steps(const DevParams& p, const double* __restrict__ a_s, const unsigned short* __restrict__ c_s, const unsigned (&cw0)[G6_NR],
                                              const unsigned (&cw1)[G6_NR], unsigned (&kk)[G6_NR], const int (&ne)[G6_NR], unsigned flagged, RowRec* rec_g0,
                                              const int32_t* cnt_g0, int32_t* neff_g0, int n_here, int dummy0, const double* th2, double* my, long long& tot,
                                              long long& kept, int& zero, Refill& refill, long long& g6_t_) {
   const int lane = threadIdx.x & 31, x = lane & 15;
   double pr[G6_NR][LS];          // alpha (SETUP) or alpha * theta
   unsigned so[G6_NR][LS];        // slot * 8 (as stored in the u16 stream): byte offset into theta (th2) and into the accumulator row (my)
   // (step-major loops: consecutive instructions belong to different rows, i.e. to independent dependency chains)
   // Dummy slots: 64 behind the two slot ranges - per half-warp 16 by bank (lanes that hold a step-0 entry: distinct banks,
   // so distinct slots) and 16 by lane (lanes without any entry): no two lanes of a warp ever share a dummy slot.
   const int dbase = dummy0 + (lane & 16) * 16;
   int dummy[G6_NR];
#pragma unroll
   for (int e = 0; e < LS; ++e) {
#pragma unroll
      for (int q = 0; q < G6_NR; ++q) {
         const unsigned ce = ((e < 4 ? cw0[q] : cw1[q]) >> (8 * (e & 3))) & 0xffu;
         const bool valid = (unsigned)x < ce;
         const double a = a_s[kk[q]];
         const int c = (int)c_s[kk[q]];
         if (e == 0) dummy[q] = dbase + (valid ? (c & 0x78) : 128 + 8 * x);   // a lane without any entry in the row: a slot of its own (rare extra wavefront)
         pr[q][e] = (SETUP && !valid) ? 0.0 : a;   // EM: a lane without an entry reads a finite stale alpha and multiplies it by theta[dummy] = 0
         so[q][e] = (unsigned)(valid ? c : dummy[q]);
         kk[q] += ce;
      }
   }
   // everything this turn needs from the stage now sits in registers: the stage can be refilled while the turn computes
   __syncwarp();
   G6_TICK(load)
   refill();
   G6_TICK(refill)
   const char* th2b = reinterpret_cast<const char*>(th2);
   char* myb = reinterpret_cast<char*>(my);
   // E-phase
   double r[G6_NR];
   if (SETUP) {
#pragma unroll
      for (int q = 0; q < G6_NR; ++q) {
         bool big = false;
#pragma unroll
         for (int e = 0; e < LS; ++e) big |= pr[q][e] > p.row_eps;
         const unsigned bal = __ballot_sync(0xffffffffu, big);
         const bool keep = ((bal >> (lane & 16)) & 0xffffu) != 0;
         r[q] = keep ? 1.0 : 0.0;
         if (x == 0 && q < n_here && !((flagged >> q) & 1u)) {
            const int n = cnt_g0[q];
            rec_g0[q].neff = keep ? n : -1;
            neff_g0[q] = keep ? n : -1;
            tot += n;
            kept += keep;
         }
      }
   } else {
      double d[G6_NR];
#pragma unroll
      for (int q = 0; q < G6_NR; ++q) d[q] = 0.0;
#pragma unroll
      for (int e = 0; e < LS; ++e) {
#pragma unroll
         for (int q = 0; q < G6_NR; ++q) {
            pr[q][e] *= *reinterpret_cast<const double*>(th2b + so[q][e]);
            d[q] += pr[q][e];
         }
      }
      // the four row sums of a half-warp in five shuffles (transposing butterfly): afterwards every lane holds the total of
      // row 2 * bit3 + bit2 of its lane id; it forms that row's r = n / d (one division per lane instead of four) and the
      // four ratios are broadcast from lanes 0, 4, 8, 12 of the half-warp
      static_assert(G6_NR == 4, "the transposing reduction is written for four rows per half-warp");
      const bool b3 = lane & 8, b2 = lane & 4;
      double s0 = b3 ? d[2] : d[0], s1 = b3 ? d[3] : d[1];
      const double o0 = b3 ? d[0] : d[2], o1 = b3 ? d[1] : d[3];
      s0 += __shfl_xor_sync(0xffffffffu, o0, 8);
      s1 += __shfl_xor_sync(0xffffffffu, o1, 8);
      double u = b2 ? s1 : s0;
      const double ox = b2 ? s0 : s1;
      u += __shfl_xor_sync(0xffffffffu, ox, 4);
      u += __shfl_xor_sync(0xffffffffu, u, 2);
      u += __shfl_xor_sync(0xffffffffu, u, 1);
      const int n_mine = b3 ? (b2 ? ne[3] : ne[2]) : (b2 ? ne[1] : ne[0]);
      const bool live = n_mine >= 0;
      const bool safe = u > 1e-290 && u < 1e290;   // the straight-line division's range; anything else (never seen on real data) divides in IEEE
      if (live && u == 0) zero = 1;
      double rm = fast_div_pos((double)max(n_mine, 0), safe ? u : 1.0);
      if (live && u != 0 && !safe) rm = (double)n_mine / u;
      rm = (live && u != 0) ? rm : 0.0;
      const int hb = lane & 16;
#pragma unroll
      for (int q = 0; q < G6_NR; ++q) r[q] = __shfl_sync(0xffffffffu, rm, hb + 4 * q);
   }
   G6_TICK(ephase)
   // M-phase: the rows of a half-warp one after the other (they may share a slot); the two half-warps update their q-th rows
   // TOGETHER - the prepare pass made the slot sets of rows r and r + 4 of every 8-row group disjoint, and a row's own slots
   // are distinct, so the loads of a step group are issued together, then the stores.
#pragma unroll
   for (int q = 0; q < G6_NR; ++q) {
      double o[LS];
#pragma unroll
      for (int e = 0; e < LS; ++e) o[e] = *reinterpret_cast<double*>(myb + so[q][e]);
#pragma unroll
      for (int e = 0; e < LS; ++e) *reinterpret_cast<double*>(myb + so[q][e]) = fma(pr[q][e], r[q], o[e]);
      __syncwarp();
   }
   G6_TICK(mphase)
}

template <bool SETUP, typename Refill>
__device__ __forceinline__ unsigned g6_turn(const DevParams& p, const double* __restrict__ a_s, const unsigned short* __restrict__ c_s, const RowRec* rec0,
                                            RowRec* rec_g0, const int32_t* cnt_g0, int32_t* neff_g0, int n_here, bool complete, uint32_t ck0, int dummy0,
                                            const double* th2, double* my, long long& tot, long long& kept, int& zero, Refill refill, long long& g6_t_) {
   const int x = threadIdx.x & 15;
   int ne[G6_NR];
   unsigned flagged = 0;
   int L = 0;
   unsigned cw0[G6_NR], cw1[G6_NR], kk[G6_NR];
   const unsigned gsum = (complete && n_here > 0) ? rec0[0].cnt[6] : 0x80u;   // the same byte for both half-warps (same 8-row group)
   if (!(gsum & 0x80u)) {
      // whole chunk, every row in the sorted layout: nothing to check, the step count comes with the records
#pragma unroll
      for (int q = 0; q < G6_NR; ++q) {
         const uint4 rc = *reinterpret_cast<const uint4*>(&rec0[q]);
         cw0[q] = rc.x;
         cw1[q] = rc.y;
         ne[q] = (int)rc.z;
         kk[q] = rc.w - ck0 + x;
      }
      L = (int)(gsum & 7u);
   } else {
#pragma unroll
      for (int q = 0; q < G6_NR; ++q) {
         const bool ex = q < n_here;
         const uint2 cw = ex ? *reinterpret_cast<const uint2*>(rec0[q].cnt) : make_uint2(0u, 0u);
         const uint2 nk = ex ? *reinterpret_cast<const uint2*>(&rec0[q].neff) : make_uint2(0xffffffffu, ck0);
         const bool fl = (cw.x & 0xffu) == G6_FLAG;
         if (fl) flagged |= 1u << q;
         ne[q] = fl ? -1 : (int)nk.x;
         cw0[q] = fl ? 0u : cw.x;
         cw1[q] = fl ? 0u : cw.y;
         L = max(L, (int)(cw1[q] >> 24));
         kk[q] = nk.y - ck0 + x;
      }
      L = max(L, __shfl_xor_sync(0xffffffffu, L, 16));   // steps of the longest of the warp's eight rows
   }
   G6_TICK(decode)
   // straight-line bodies for 4, 5 and 6 steps (a row's fullest bank holds 4 entries in ~70 % of the rows, 5 in most others)
   if (SETUP || L > 5) g6_turn_steps<SETUP, 6>(p, a_s, c_s, cw0, cw1, kk, ne, flagged, rec_g0, cnt_g0, neff_g0, n_here, dummy0, th2, my, tot, kept, zero, refill, g6_t_);
   else if (L == 5) g6_turn_steps<SETUP, 5>(p, a_s, c_s, cw0, cw1, kk, ne, flagged, rec_g0, cnt_g0, neff_g0, n_here, dummy0, th2, my, tot, kept, zero, refill, g6_t_);
   else g6_turn_steps<SETUP, 4>(p, a_s, c_s, cw0, cw1, kk, ne, flagged, rec_g0, cnt_g0, neff_g0, n_here, dummy0, th2, my, tot, kept, zero, refill, g6_t_);
   return flagged;
}

// Lane 0: start the bulk copy of CTA-local chunk c of the packed stream into stage `st` (k0, k1: its non-zero range).
template <typename C>
__device__ __forceinline__ void g6_issue(const unsigned char* __restrict__ pk_cta, int c, int64_t k0, int64_t k1, char* st, uint64_t* full) {
   const unsigned n = (unsigned)(k1 - k0);
   const unsigned bytes = (unsigned)G6_PK_RECS + (n <= (unsigned)C::CAP ? g6_pk_abytes(n) + g6_pk_cbytes(n) : 0u);   // a fuller chunk only brings its records
   asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // the stage was last read with ordinary shared-memory loads
   mbar_expect_tx(full, bytes);
   bulk_g2s(st, pk_cta + (size_t)c * G6_PK_STRIDE, bytes, full);
}

// One pass of this warp over its chunks (w, w + NC, ...) of the CTA's rows.
template <typename C, bool SETUP>
__device__ __forceinline__ void g6_pass(const DevParams& p, const unsigned short* __restrict__ col16, unsigned char* __restrict__ pk_cta /* packed chunk 0 of this CTA */,
                                        RowRec* __restrict__ rec_cta /* row 0 of this CTA in the record array (rows walked from the CSR arrays) */,
                                        const int64_t* __restrict__ rp_cta /* row pointer of the CTA's row 0 */, const int64_t kbase /* first non-zero of the locus */,
                                        int64_t row_abs0 /* absolute row of the CTA's row 0 */, int n_rows, int n_chunk, G6Ring& ring,
                                        int dummy0 /* byte offset of the first dummy slot = 8 * 2 Tp */, const double* th2, double* my, long long& tot, long long& kept, int& zero) {
   const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
   const int n_mine = warp < n_chunk ? (n_chunk - warp + C::CONSUMERS - 1) / C::CONSUMERS : 0;
   // prologue: fill the ring (records written with ordinary global stores in the setup pass are read by bulk copies)
   asm volatile("fence.proxy.async;" ::: "memory");
   if (lane == 0) {
      int sx = ring.next;
      for (int i = 0; i < min(ring.spw, n_mine); ++i) {
         const int c = warp + i * C::CONSUMERS;
         g6_issue<C>(pk_cta, c, rp_cta[min(c * C::CROWS, n_rows)], rp_cta[min((c + 1) * C::CROWS, n_rows)],
                     ring.stage + (size_t)sx * C::STAGE_BYTES, &ring.full[sx]);
         sx = sx + 1 == ring.spw ? 0 : sx + 1;
      }
   }
   __syncwarp();
   long long g6_t_ = clock64();
   for (int i = 0; i < n_mine; ++i) {
      G6_TICK(other)
      const int c = warp + i * C::CONSUMERS;
      const int sidx = ring.next;
      // boundaries of the chunk that will refill this stage, fetched now so that the loads overlap the turn
      const int cn = c + ring.spw * C::CONSUMERS;
      int64_t kn0 = 0, kn1 = 0;
      if (lane == 0 && cn < n_chunk) { kn0 = rp_cta[min(cn * C::CROWS, n_rows)]; kn1 = rp_cta[min((cn + 1) * C::CROWS, n_rows)]; }
      const int i0 = c * C::CROWS, i1 = min(i0 + C::CROWS, n_rows);       // rows of the chunk (CTA-local)
      mbar_wait(&ring.full[sidx], (ring.phase >> sidx) & 1u);
      G6_TICK(wait)
#ifdef SBQ_G6_PHASES
      if (threadIdx.x == 0 && blockIdx.x == 0) ++g6_ph.turns;
#endif
      ring.phase ^= 1u << sidx;
      ring.next = sidx + 1 == ring.spw ? 0 : sidx + 1;
      char* st = ring.stage + (size_t)sidx * C::STAGE_BYTES;
      const RowRec* rec_s = (const RowRec*)st;
      const uint32_t ck0 = rec_s[0].koff;
      const uint32_t ck1 = rec_s[i1 - i0].koff;
      const bool staged = ck1 - ck0 <= (uint32_t)C::CAP;   // same decision as g6_issue
      const int h0 = i0 + (lane >> 4) * G6_NR;             // first row of this half-warp
      unsigned walk = 0;                                   // bit i: row i0 + i is walked from global memory
      auto refill = [&]() {
         if (lane == 0 && cn < n_chunk) g6_issue<C>(pk_cta, cn, kn0, kn1, st, &ring.full[sidx]);
      };
      if (staged) {
         // setup pass: the effective counts go into the PACKED records (what the EM passes stage); walked rows keep theirs in the record array
         RowRec* rec_pk = reinterpret_cast<RowRec*>(pk_cta + (size_t)c * G6_PK_STRIDE) + (h0 - i0);
         const unsigned fl = g6_turn<SETUP>(p, (const double*)(st + C::A_OFF), (const unsigned short*)(st + C::A_OFF + g6_pk_abytes(ck1 - ck0)), rec_s + (min(h0, i1 - 1) - i0),
                                            rec_pk, p.count + row_abs0 + h0, p.neff + row_abs0 + h0, max(0, min(G6_NR, i1 - h0)), i1 - i0 == C::CROWS, ck0, dummy0, th2, my,
                                            tot, kept, zero, refill, g6_t_);
         walk = __shfl_sync(0xffffffffu, fl, 0) | (__shfl_sync(0xffffffffu, fl, 16) << G6_NR);
      } else {
         walk = (1u << C::CROWS) - 1u;
         __syncwarp();
         refill();
      }
      while (walk) {
         const int r = __ffs(walk) - 1;
         walk &= walk - 1;
         const int row = i0 + r;
         if (row < i1)
            g6_walk_row<SETUP>(p, col16, rec_cta + row, rp_cta[row], rp_cta[row + 1], SETUP ? p.count[row_abs0 + row] : 0, p.neff + row_abs0 + row, th2, my,
                               tot, kept, zero);
      }
   }
}

template <typename C>
__global__ void __launch_bounds__(C::NT, 1)
em_grid_dual_kernel(DevParams p, const unsigned short* __restrict__ col16, RowRec* __restrict__ recs, const int64_t* __restrict__ rec_off,
                    const int32_t* __restrict__ list, int n_list, GridScratch gs, double* cur_glob /* [n_cta][tstride] */, int spw,
                    unsigned char* __restrict__ pk, const int64_t* __restrict__ pk_off) {
   cg::grid_group grid = cg::this_grid();
   extern __shared__ __align__(128) unsigned char g6_smem[];
   __shared__ double red[C::NT / 32];
   __shared__ int s_rows[2];
   __shared__ __align__(8) uint64_t s_bar[G6_MAX_WARPS * G6_MAX_SPW];
   const int tid = threadIdx.x, warp = tid >> 5;
   const int nb = gridDim.x, b = blockIdx.x;
   const int ns = spw * C::CONSUMERS;   // stages of the CTA

   G6Ring ring;
   ring.stage = (char*)g6_smem + (size_t)warp * spw * C::STAGE_BYTES;
   ring.full = s_bar + warp * G6_MAX_SPW;
   ring.spw = spw;
   ring.next = 0;
   ring.phase = 0;
   for (int x = tid; x < ns * C::STAGE_BYTES / 8; x += C::NT) ((double*)g6_smem)[x] = 0.0;   // stale alpha reads must be finite
   if (tid == 0) {
      for (int s = 0; s < G6_MAX_WARPS * G6_MAX_SPW; ++s) mbar_init(&s_bar[s], 1);
      asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
   }
   __syncthreads();
   double* my_cur = cur_glob + (size_t)b * gs.tstride;

   for (int item = 0; item < n_list; ++item) {
      const int l = list[item];
      const int64_t r0 = p.loc_row_off[l];
      const int R = (int)(p.loc_row_off[l + 1] - r0);
      const int64_t t0 = p.loc_iso_off[l];
      const int T = (int)(p.loc_iso_off[l + 1] - t0);
      const int Tp = g6_tp(T), T2 = 2 * Tp + 64;   // two slots per column + 64 dummy slots
      double* th2 = (double*)(g6_smem + (size_t)ns * C::STAGE_BYTES);   // [2 Tp]: slot A | slot B
      double* acc = th2 + T2;                                           // [NC][2 Tp]
      const int64_t* __restrict__ rp = p.row_ptr + r0;
      double* my_partial = gs.partial + (size_t)b * gs.tstride;
      RowRec* rec_l = recs + rec_off[item];

      grid_row_range(rp, R, C::CROWS, b, nb, s_rows);
      for (int x = tid; x < C::CONSUMERS * T2; x += C::NT) acc[x] = 0.0;
      if (tid < 64) th2[2 * Tp + tid] = 0.0;   // dummy slots read as theta = 0
      __syncthreads();
      const int ra = s_rows[0], rb = s_rows[1];
      const int n_chunk = (rb - ra + C::CROWS - 1) / C::CROWS;
      const int64_t kbase = rp[0];
      RowRec* rec_cta = rec_l + ra;
      unsigned char* pk_cta = pk + (size_t)(pk_off[item] + ra / C::CROWS) * G6_PK_STRIDE;   // ra is a multiple of the chunk size
      double* my_acc = acc + (size_t)warp * T2;
      // sum of a column's two slots over the warp-private accumulators (fixed order), accumulators cleared
      auto fold = [&](int j) {
         const int sb = g6_slot_b(j, Tp);
         double sj = 0.0;
         for (int w = 0; w < C::CONSUMERS; ++w) {
            double* aw = acc + (size_t)w * T2;
            sj += aw[j] + aw[sb];
            aw[j] = 0.0;
            aw[sb] = 0.0;
         }
         return sj;
      };

      // ---- setup pass
      long long tot = 0, kept = 0;
      int zero = 0;
      g6_pass<C, true>(p, col16, pk_cta, rec_cta, rp + ra, kbase, r0 + ra, rb - ra, n_chunk, ring, 16 * Tp, th2, my_acc, tot, kept, zero);
      grid_publish_counts(gs, item, tot, kept);
      __threadfence();
      asm volatile("fence.proxy.async;" ::: "memory");
      __syncthreads();
      for (int j = tid; j < T; j += C::NT) my_partial[j] = fold(j);
      grid_owner_reduce<C::NT>(grid, gs, T);
      const double total = (double)__ldcg(gs.ctr + 2 * item);
      const long long kept_all = __ldcg(gs.ctr + 2 * item + 1);
      const double theta0 = total / (double)T;
      double* my_sdiv = my_cur + gs.tstride / 2;   // s_j in the upper half of this CTA's theta copy
      for (int j = tid; j < T; j += C::NT) {
         my_sdiv[j] = __ldcg(gs.theta_next + j);
         my_cur[j] = theta0;
         th2[j] = theta0;
         th2[g6_slot_b(j, Tp)] = theta0;
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
            g6_pass<C, false>(p, col16, pk_cta, rec_cta, rp + ra, kbase, r0 + ra, rb - ra, n_chunk, ring, 16 * Tp, th2, my_acc, d0, d1, zero);
            zero = __syncthreads_or(zero);
            if (zero && tid == 0) atomicOr(&gs.zero_flag[item], 1);
            for (int j = tid; j < T; j += C::NT) my_partial[j] = fold(j);
            grid_owner_reduce<C::NT>(grid, gs, T);
            const int zf = *(volatile int*)&gs.zero_flag[item];
            const double d2 = grid_read_next<C::NT>(gs, my_cur, th2, T, red);
            if (zf) { status = LOCUS_ZERO_DENOM; break; }
            if (d2 < tol2) { status = LOCUS_OK; break; }
            for (int j = tid; j < T; j += C::NT) {
               const double nj = th2[j];
               my_cur[j] = nj;
               const double sj = my_sdiv[j];
               const double sc = (sj != 0) ? nj / sj : 0.0;
               th2[j] = sc;
               th2[g6_slot_b(j, Tp)] = sc;
            }
            __syncthreads();
         }
      }

      // ---- outputs + epilogue by CTA 0 (src/estimate.cpp:310-356)
      if (b == 0) {
         locus_epilogue_block<C::NT>(p, l, t0, T, status, iters, theta0, my_cur, th2, red);
      }
      grid.sync();   // scratch (partial, theta_next) is reused by the next locus
   }
#ifdef SBQ_G6_PHASES
   if (b == 0 && tid == 0 && g6_ph.turns)
      printf("G6PHASES turns %lld per-turn cycles: wait %lld decode %lld load %lld refill %lld E %lld M %lld other %lld\n", g6_ph.turns, g6_ph.wait / g6_ph.turns,
             g6_ph.decode / g6_ph.turns, g6_ph.load / g6_ph.turns, g6_ph.refill / g6_ph.turns, g6_ph.ephase / g6_ph.turns, g6_ph.mphase / g6_ph.turns,
             g6_ph.other / g6_ph.turns);
#endif
}

// ------------------------------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------------------------------
// The kernel is bound by instruction latency, so it lives on warps per SM: 0.143 / 0.160 / 0.172 / 0.217 ms per pass with
// 12 / 10 / 8 / 6 warps on the configs[3] shape, against 0.2045 ms for the TMA ring kernel. It is used where at least 8
// warps fit (T <= ~1300; 12 warps up to T ~ 800).
// default wherever the kernel can run: measured on 1 M rows x 48 non-zeros, even its 4-warp configuration (T = 2000: 0.32 of the HBM
// peak, T = 1400 with 6 warps: 0.43) beats the TMA ring kernel (0.27 / 0.37), which remains for T > G6_MAX_ISO and dense rows
inline bool grid_dual_supports_iso(int T) { return T <= G6_MAX_ISO && G6Cfg<4>::fits(T, 1); }

// warps per CTA for a locus of T isoforms: a function of the LOCUS alone (the launcher groups loci by it), so that neither the
// speed nor the summation order of a locus depends on which other loci share its batch
inline int grid_dual_nc(int T) {
#define SBQ_NC6(NC) if (G6Cfg<NC>::fits(T, 1)) return NC;
   // (14 warps fit up to T = 624 but force 128 registers per thread: measured 0.1427 ms per pass against 0.1433 with 12 - not worth a variant)
   SBQ_NC6(12) SBQ_NC6(10) SBQ_NC6(8) SBQ_NC6(6) SBQ_NC6(4)
#undef SBQ_NC6
   return 0;
}

template <typename C>
inline int grid_dual_launch_cfg(const DevParams& dp, const int32_t* d_list, int n_list, int max_iso, const cudaDeviceProp& prop, DevBuf& scratch,
                                const unsigned short* c16, const int64_t* d_rec_off, RowRec* d_recs, unsigned char* pk, const int64_t* d_pk_off,
                                cudaStream_t st, int* n_launch) {
   const int spw = C::stages_per_warp(max_iso);
   const size_t smem = (size_t)spw * C::CONSUMERS * C::STAGE_BYTES + C::fixed_bytes(max_iso);
   auto kernel = em_grid_dual_kernel<C>;
   if (cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess) return -3;
   int per_sm = 0;
   if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, C::NT, smem) != cudaSuccess || per_sm < 1) return -3;
   const int nb = prop.multiProcessorCount;
   GridScratch gs;
   double* cur_glob = nullptr;
   // theta copy in the lower half of tstride, s_j in the upper half
   if (const int rc = grid_scratch(scratch, nb, 2 * (((max_iso + 255) / 256) * 256), n_list, &cur_glob, st, &gs)) return rc;
   DevParams dpc = dp;
   int ns_arg = spw;
   void* args[] = {(void*)&dpc, (void*)&c16, (void*)&d_recs, (void*)&d_rec_off, (void*)&d_list, (void*)&n_list, (void*)&gs, (void*)&cur_glob, (void*)&ns_arg,
                   (void*)&pk, (void*)&d_pk_off};
   if (cudaLaunchCooperativeKernel((void*)kernel, dim3(nb), dim3(C::NT), args, smem, st) != cudaSuccess) return -3;
   ++*n_launch;
   return 0;
}

// h_rec_off: n_list + 1 record offsets (host; a locus of R rows owns R + 1 records). c16: the u16 slots of the whole batch (the
// caller sizes the buffer). recs: per-locus record offsets and first packed chunks (int64 each, at the front) + row records of
// the giant loci; pk: their packed chunk stream (G6_PK_STRIDE bytes per 8-row chunk). prepared: the sorted layout of this upload
// is already in place.
inline int grid_dual_launch(const DevParams& dp, const int32_t* d_list, int n_list, const int* h_iso /* T of every list entry */, const int64_t* h_rec_off,
                            const cudaDeviceProp& prop, DevBuf& scratch, unsigned short* c16, DevBuf& recs, DevBuf& pk, bool prepared, cudaStream_t st,
                            int* n_launch) {
   *n_launch = 0;
   if (n_list == 0) return 0;
   const size_t off_bytes = (((size_t)(n_list + 1) * 2 * sizeof(int64_t) + 255) / 256) * 256;   // record offsets | first packed chunks
   const size_t need_rec = off_bytes + (size_t)(h_rec_off[n_list] + 64) * sizeof(RowRec);
   std::vector<int64_t> h_off(2 * (size_t)(n_list + 1));
   for (int i = 0; i <= n_list; ++i) h_off[i] = h_rec_off[i];
   h_off[n_list + 1] = 0;
   for (int i = 0; i < n_list; ++i) {
      const int64_t R = h_rec_off[i + 1] - h_rec_off[i] - 1;   // a locus of R rows owns R + 1 records
      h_off[n_list + 1 + i + 1] = h_off[n_list + 1 + i] + (R + G6_PK_ROWS - 1) / G6_PK_ROWS;
   }
   const size_t need_pk = (size_t)h_off[2 * n_list + 1] * G6_PK_STRIDE + 256;
   if (need_pk > pk.cap || need_rec > recs.cap) {
      if (!pk.reserve(need_pk) || !recs.reserve(need_rec)) return -4;
      prepared = false;
   }
   const int64_t* d_rec_off = (const int64_t*)recs.p;
   const int64_t* d_pk_off = d_rec_off + (n_list + 1);
   RowRec* d_recs = (RowRec*)((char*)recs.p + off_bytes);
   if (!prepared) {
      // (pageable host vector: the copy is staged by the runtime before the call returns)
      if (cudaMemcpyAsync(recs.p, h_off.data(), h_off.size() * sizeof(int64_t), cudaMemcpyHostToDevice, st) != cudaSuccess) return -3;
      const size_t psmem = (size_t)G6_PREP_WARPS * sizeof(G6PrepTile);
      if (cudaFuncSetAttribute(dual_prepare_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)psmem) != cudaSuccess) return -3;
      dual_prepare_kernel<<<prop.multiProcessorCount * 2, G6_PREP_WARPS * 32, psmem, st>>>(dp, d_list, n_list, d_rec_off, d_recs, c16);
      ++*n_launch;
      if (getenv("SBQ_DUAL_VERIFY")) {   // tests: the prepared layout must satisfy the kernel's conflict-freedom assumptions
         int* d_viol = nullptr;
         int h_viol = -1;
         if (cudaMalloc(&d_viol, sizeof(int)) != cudaSuccess) return -4;
         cudaMemsetAsync(d_viol, 0, sizeof(int), st);
         dual_verify_kernel<<<prop.multiProcessorCount * 4, 256, 0, st>>>(dp, d_list, n_list, d_rec_off, d_recs, c16, d_viol);
         cudaMemcpyAsync(&h_viol, d_viol, sizeof(int), cudaMemcpyDeviceToHost, st);
         cudaStreamSynchronize(st);
         cudaFree(d_viol);
         if (h_viol != 0) { fprintf(stderr, "sbq: two-slot layout check failed: %d groups violate it\n", h_viol); return -7; }
      }
      dual_pack_kernel<<<prop.multiProcessorCount * 8, 256, 0, st>>>(dp, d_list, n_list, d_rec_off, d_recs, c16, d_pk_off, (unsigned char*)pk.p);
      ++*n_launch;
   }
   return grid_for_each_run(h_iso, n_list, grid_dual_nc, [&](int i0, int i1, int nc, int mx) {
      const int32_t* li = d_list + i0;
      unsigned char* pkp = (unsigned char*)pk.p;
      switch (nc) {
         case 12: return grid_dual_launch_cfg<G6Cfg<12>>(dp, li, i1 - i0, mx, prop, scratch, c16, d_rec_off + i0, d_recs, pkp, d_pk_off + i0, st, n_launch);
         case 10: return grid_dual_launch_cfg<G6Cfg<10>>(dp, li, i1 - i0, mx, prop, scratch, c16, d_rec_off + i0, d_recs, pkp, d_pk_off + i0, st, n_launch);
         case 8: return grid_dual_launch_cfg<G6Cfg<8>>(dp, li, i1 - i0, mx, prop, scratch, c16, d_rec_off + i0, d_recs, pkp, d_pk_off + i0, st, n_launch);
         case 6: return grid_dual_launch_cfg<G6Cfg<6>>(dp, li, i1 - i0, mx, prop, scratch, c16, d_rec_off + i0, d_recs, pkp, d_pk_off + i0, st, n_launch);
         case 4: return grid_dual_launch_cfg<G6Cfg<4>>(dp, li, i1 - i0, mx, prop, scratch, c16, d_rec_off + i0, d_recs, pkp, d_pk_off + i0, st, n_launch);
         default: return -6;
      }
   });
}

}  // namespace sbq

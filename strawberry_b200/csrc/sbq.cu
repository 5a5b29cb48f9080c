// sbq.cu - runtime + C ABI (include/sbq.h) of the B200-native quantification engine.
//
// Host side of the hot path: stages submitted loci into one flat, pinned CSR batch, plans the
// kernel tiers (warp / cluster / grid) by locus size, moves the batch to HBM, launches the EM
// kernels of sbq_kernels.cuh on concurrent streams and brings the per-isoform results back.
// Replaces, for everything numeric, the loop body of Sample::procSample -> quantifyCluster ->
// LocusContext::estimate_abundances -> EmSolver (reference src/alignments.cpp:1756-1829,
// src/estimate.cpp:279-488). There is no CPU fallback in this file by design.
#include <algorithm>
#include <chrono>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <dlfcn.h>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include <nccl.h>   // types and prototypes only: the library itself is dlopen'ed by multi-GPU contexts (NcclApi below)

#include "../../include/sbq.h"
#include "../../include/sbq_builder.h"
#include "sbq_kernels.cuh"
#include "sbq_grid.cuh"
#include "sbq_grid_tma.cuh"
#include "sbq_grid_dual.cuh"
#include "sbq_bias.cuh"
#include "sbq_weights.cuh"
#include "sbq_synth.cuh"
#include "sbq_rawbuild.cuh"
#include "sbq_bootstrap.cuh"
#include "sbq_gibbs.cuh"

using namespace sbq;

namespace {

constexpr size_t SMEM_CAP = CL_SMEM_CAP;   // dynamic shared memory we ask for at most (227 KB usable)
constexpr int N_SIDE_STREAMS = 12;

// ---- pinned host array with geometric growth -------------------------------------------------
template <typename T>
struct PinnedVec {
   T* p = nullptr;
   size_t n = 0, cap = 0;
   bool reserve(size_t want) {
      if (want <= cap) return true;
      size_t ncap = std::max(want, cap + cap / 2 + 1024);
      T* q = nullptr;
      if (cudaMallocHost((void**)&q, ncap * sizeof(T)) != cudaSuccess) return false;
      if (n) memcpy(q, p, n * sizeof(T));
      if (p) cudaFreeHost(p);
      p = q;
      cap = ncap;
      return true;
   }
   bool append(const T* src, size_t k) {
      if (!reserve(n + k)) return false;
      if (k) memcpy(p + n, src, k * sizeof(T));
      n += k;
      return true;
   }
   void clear() { n = 0; }
   void release() {
      if (p) cudaFreeHost(p);
      p = nullptr;
      n = cap = 0;
   }
};

struct LaunchClass {      // one kernel launch of the cluster tier
   int cs, nt;            // cluster size, threads per CTA
   std::vector<int32_t> loci;
   int max_iso = 0;
   size_t max_slice = 0;  // estimated bytes of the largest per-CTA resident CSR slice
   size_t list_off = 0;   // offset into the device list buffer
   size_t smem = 0;
};

struct BiasClass {        // one launch of the bias kernel: the loci of one cluster size
   int cs = 1, max_iso = 1;
   size_t off = 0, n = 0;
};

struct LaunchTimer {      // CUDA events around one kernel launch, on the stream it is launched on
   cudaEvent_t e0 = nullptr, e1 = nullptr;
   bool used = false;
};

// One class of giant-tier loci: 0 = the full grid on the main stream, 1 = the "small giants" (below SGRID_MAX_NNZ non-zeros, a
// few thousand rows) on a SUB-GRID of SGRID_CTAS CTAs, on a stream of its own, so that the cluster and warp tiers keep the other
// SMs (the full-grid launch of a 400 k-non-zero locus idles most of the GPU for milliseconds: its iterations are barrier latency,
// not bandwidth). The same kernels run both classes.
struct GridClass {
   std::vector<int32_t> list;       // two-slot loci, then TMA ring loci, then register-staged loci (plan() sorts it)
   std::vector<int64_t> rec_off;    // row-record offset of every two-slot locus (+ total), list order
   size_t list_off = 0;             // offset into the device list buffer
   size_t n_dual = 0, n_tma = 0;    // sizes of the two-slot and TMA ring parts of the list
   int n_cta = 0;
   int variant = 0;                 // the first kernel the last solve launched (sbq_launch_stat.variant)
   DevBuf scratch, rowrec, pk;
   cudaStream_t st = nullptr;
   LaunchTimer lt;
};

}  // namespace

struct MultiState;   // n_gpus > 1: one child context per device + the NCCL communicators (defined further down)

struct sbq_ctx {
   sbq_config cfg;
   MultiState* multi = nullptr;
   int device = 0;
   cudaDeviceProp prop;
   cudaStream_t stream = nullptr;
   cudaStream_t copy_st = nullptr;                      // host -> device copies of sbq_upload*, in the order the solve needs them
   cudaEvent_t ev_class_ready[N_SIDE_STREAMS] = {};     // weights of cluster launch i are on the device
   cudaEvent_t ev_grid_ready = nullptr;
   bool class_ready[N_SIDE_STREAMS] = {};               // the event above was recorded by the last upload (else: wait for ev[1], everything)
   bool grid_ready = false;
   bool upload_pending = false;                         // upload_begin's copies have not been waited for yet
   cudaStream_t side[N_SIDE_STREAMS] = {};
   cudaEvent_t ev[9] = {};
   cudaEvent_t ev_fork = nullptr, ev_join[N_SIDE_STREAMS] = {};
   LaunchTimer lt[1 + N_SIDE_STREAMS];          // [0] warp tier, [1+i] cluster class i
   std::vector<sbq_launch_stat> launch_stats;   // filled by sbq_solve (+ bytes by sbq_download)
   std::vector<int32_t> locus_launch;           // locus -> index into launch_stats
   std::mutex mu;
   std::string err;

   // staged batch (host, pinned)
   PinnedVec<int64_t> h_loc_row_off, h_loc_iso_off, h_row_ptr;
   PinnedVec<int32_t> h_col, h_count, h_iso_len;
   PinnedVec<double> h_alpha;
   // borrowed flat batch (caller-pinned arrays used in place)
   bool borrowed = false;
   const int64_t *b_loc_row_off = nullptr, *b_loc_iso_off = nullptr, *b_row_ptr = nullptr;
   const int32_t *b_col = nullptr, *b_count = nullptr, *b_iso_len = nullptr;
   const double* b_alpha = nullptr;
   int64_t n_loci = 0, n_row = 0, n_iso = 0, nnz = 0;
   bool host_released = false;   // a borrowed batch was uploaded: the caller may have freed its arrays, nothing on the host side may be re-read
   // per-locus shape and fragment total, captured by plan() while the host arrays are still valid (metric accounting)
   struct LocusMeta { int64_t nnz, frags; int32_t R, T; };
   std::vector<LocusMeta> meta;

   // bias mode
   PinnedVec<double> h_cov;
   int n_cov = 0;
   bool have_cov = false;
   DevBuf d_bias;
   int32_t* d_bias_list = nullptr;          // loci grouped by the cluster size of the bias kernel (inside d_bias)
   std::vector<int32_t> bias_list;
   BiasClass bias_cls[6];                   // cluster sizes 16, 8, 4, 2, 1 and the warp tier
   int* d_bias_queue = nullptr;             // work queue of the persistent warps of em_bias_warp_kernel
   BiasParams bpar{};
   PinnedVec<double> r_beta;
   PinnedVec<int32_t> r_outer;
   int max_iso_all = 1;

   // deferred (GPU) weights
   int deferred = 0;                 // 0 = nothing queued yet, 1 = every queued locus is deferred, 2 = host-weighted batch
   PinnedVec<int64_t> h_wseg, h_wpool_off;   // h_wpool_off[l]: first pool element of deferred locus l (multi-GPU gather)
   PinnedVec<uint8_t> h_wn;
   PinnedVec<uint32_t> h_wmask, h_wpool;
   PinnedVec<int32_t> h_wlen;
   std::vector<double> model_emp;
   sbq_insert_model model{};
   int model_read_len = 0;
   bool have_model = false;
   DevBuf d_weights;
   double weights_ms = 0.0;

   // raw loci (class assignment on the device, sbq_rawbuild.cuh): flattened feature lists of hits and isoforms + the static
   // per-locus tables (segments, isoform segment lists) staged on the host until sbq_upload
   struct RawStage {
      std::vector<int32_t> hit_locus, hit_ref, iso_seg;
      std::vector<int64_t> hit_feat_ptr{0}, iso_feat_ptr{0}, loc_hit_off{0}, loc_seg_off{0}, iso_seg_ptr{0};
      std::vector<uint32_t> hf_off, hf_len, if_off, if_len, seg_left, seg_right;
      std::vector<uint8_t> hf_code, if_code;
      std::vector<float> hit_mass;
      int long_read = 0;
      void clear() { *this = RawStage(); }
   } raw;
   bool raw_mode = false;
   int32_t raw_mass_mode = SBQ_RAW_MASS_HALVES;   // sbq_set_raw_mass_mode
   DevBuf d_raw, d_raw2;
   RawBatch rb{};                    // device view of the last raw upload (tests fetch the class table through it)

   // plan
   int force_tier = 0, force_cluster = 0;
   std::vector<int32_t> warp_list;
   std::vector<LaunchClass> classes;
   GridClass grid[2];                           // [0] full grid on the main stream, [1] sub-grid on its own stream
   int warp_max_iso = 1;
   PinnedVec<int32_t> h_lists;
   size_t warp_list_off = 0;

   // device
   DevBuf d_in, d_out, d_lists, d_col16, d_csc, d_synth;
   bool col16_ready = false;
   DevParams dp{};
   double* d_tpm = nullptr;
   double* d_fpkm_sum = nullptr;
   int32_t* d_lists_p = nullptr;
   bool resident = false, solved = false, downloaded = false;

   // results (host, pinned)
   PinnedVec<double> r_theta, r_fpkm, r_frac, r_tpm, r_locus_fpkm;
   PinnedVec<int32_t> r_keep, r_iters, r_status;
   PinnedVec<long long> r_frags;   // fragment total per locus (device sum, metric accounting)
   DevBuf d_frags;
   double r_fpkm_sum = 0.0;

   sbq_stats stats{};
   bool stats_stale = false;

   // bootstrap replicates (sbq_bootstrap): draw offsets of the resident batch (built once per upload), per-replicate scratch and the
   // replicate matrices of the last call
   struct Boot {
      DevBuf prefix, scratch, out, sums;
      bool prefix_ready = false;
      int64_t* draw_off = nullptr;       // [n_row + 1] exclusive prefix of the counts
      int64_t* loc_draw_off = nullptr;   // [n_loci + 1] the same at the locus boundaries
      int32_t* d_lid = nullptr;          // [n_loci] hash position of every locus (multi-GPU children)
      std::vector<int32_t> lid;          // multi-GPU children: the parent's submit position of each locus; empty = own index
      bool done = false;                 // the replicate matrices in `out` belong to the resident batch
      sbq_bootstrap_stat stat{};
      std::vector<cudaEvent_t> ev;
   } boot;

   // Gibbs posterior samples (sbq_gibbs): setup + per-round scratch and the sample matrices of the last call
   struct Gibbs {
      DevBuf scratch, out, sums;
      bool done = false;                 // the sample matrices in `out` belong to the resident batch
      sbq_gibbs_stat stat{};
      std::vector<cudaEvent_t> ev;       // start, setup end, end, then a ring of (round start, assigned, done) triples
   } gibbs;
};

namespace {

int fail(sbq_ctx* c, int code, const char* fmt, ...) {
   if (c) {
      char buf[512];
      va_list ap;
      va_start(ap, fmt);
      vsnprintf(buf, sizeof buf, fmt, ap);
      va_end(ap);
      c->err = buf;
   }
   return code;
}

#define CU(call)                                                                                   \
   do {                                                                                            \
      cudaError_t e_ = (call);                                                                     \
      if (e_ != cudaSuccess)                                                                       \
         return fail(c, SBQ_ERR_CUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, __LINE__); \
   } while (0)

const int64_t* loc_row_off(const sbq_ctx* c) { return c->borrowed ? c->b_loc_row_off : c->h_loc_row_off.p; }
const int64_t* loc_iso_off(const sbq_ctx* c) { return c->borrowed ? c->b_loc_iso_off : c->h_loc_iso_off.p; }
const int64_t* row_ptr(const sbq_ctx* c) { return c->borrowed ? c->b_row_ptr : c->h_row_ptr.p; }
const int32_t* colp(const sbq_ctx* c) { return c->borrowed ? c->b_col : c->h_col.p; }
const int32_t* countp(const sbq_ctx* c) { return c->borrowed ? c->b_count : c->h_count.p; }
const int32_t* iso_lenp(const sbq_ctx* c) { return c->borrowed ? c->b_iso_len : c->h_iso_len.p; }
const double* alphap(const sbq_ctx* c) { return c->borrowed ? c->b_alpha : c->h_alpha.p; }

bool is_pinned(const void* p) {
   cudaPointerAttributes a;
   if (cudaPointerGetAttributes(&a, p) != cudaSuccess) {
      cudaGetLastError();
      return false;
   }
   return a.type == cudaMemoryTypeHost;
}

// copy a borrowed batch into our own staging (needed before anything else is appended)
int materialise(sbq_ctx* c) {
   if (!c->borrowed) return SBQ_SUCCESS;
   if (c->host_released) return fail(c, SBQ_ERR_STATE, "the borrowed batch was released by sbq_upload: sbq_clear and submit again");
   bool ok = true;
   c->h_loc_row_off.clear(); c->h_loc_iso_off.clear(); c->h_row_ptr.clear();
   c->h_col.clear(); c->h_count.clear(); c->h_iso_len.clear(); c->h_alpha.clear();
   ok &= c->h_loc_row_off.append(c->b_loc_row_off, c->n_loci + 1);
   ok &= c->h_loc_iso_off.append(c->b_loc_iso_off, c->n_loci + 1);
   ok &= c->h_row_ptr.append(c->b_row_ptr, c->n_row + 1);
   ok &= c->h_col.append(c->b_col, c->nnz);
   ok &= c->h_alpha.append(c->b_alpha, c->nnz);
   ok &= c->h_count.append(c->b_count, c->n_row);
   ok &= c->h_iso_len.append(c->b_iso_len, c->n_iso);
   c->borrowed = false;
   return ok ? SBQ_SUCCESS : fail(c, SBQ_ERR_NOMEM, "pinned staging allocation failed");
}

void reset_batch(sbq_ctx* c) {
   c->borrowed = false;
   c->host_released = false;
   c->meta.clear();
   c->h_loc_row_off.clear(); c->h_loc_iso_off.clear(); c->h_row_ptr.clear();
   c->h_col.clear(); c->h_count.clear(); c->h_iso_len.clear(); c->h_alpha.clear();
   c->n_loci = c->n_row = c->n_iso = c->nnz = 0;
   c->have_cov = false;
   c->h_cov.clear();
   c->deferred = 0;
   c->raw.clear();
   c->raw_mode = false;
   c->h_wseg.clear(); c->h_wn.clear(); c->h_wmask.clear(); c->h_wpool.clear(); c->h_wlen.clear(); c->h_wpool_off.clear();
   c->resident = c->solved = c->downloaded = false;
   c->boot.prefix_ready = c->boot.done = c->gibbs.done = false;
}

int ensure_origin(sbq_ctx* c) {
   if (c->h_loc_row_off.n == 0) {
      int64_t z = 0;
      if (!c->h_loc_row_off.append(&z, 1) || !c->h_loc_iso_off.append(&z, 1) || !c->h_row_ptr.append(&z, 1))
         return fail(c, SBQ_ERR_NOMEM, "pinned staging allocation failed");
   }
   return SBQ_SUCCESS;
}

// Single-CTA loci are bucketed by shared-memory need, and for the two smallest buckets the bucket also sets the THREADS of
// the CTA: the EM of a small locus is a chain of short barrier-separated phases, i.e. latency-bound, so its cost in SM time is
// (time per iteration) x (share of the SM it holds); small CTAs let several loci share an SM (registers: 125 per thread).
// Larger single-CTA loci keep 512 threads: measured, fewer threads lengthen their iterations (159 loci of <= 54 KB: 3.1 ms
// with 512 threads, 3.95 ms with 128) and the step is as long as its slowest locus.
//   bucket 0  <=  12 KB   64 threads  8 per SM        bucket 2  <=  56 KB  512 threads  1 per SM (registers)
//   bucket 1  <=  24 KB  128 threads  4 per SM        bucket 3  <= 112 KB, bucket 4: rest, 512 threads
constexpr int N_BUCKETS = 5;
const int BUCKET_NT[N_BUCKETS] = {64, 128, 512, 512, 512};
int smem_bucket(size_t bytes) { return bytes <= 12 * 1024 ? 0 : bytes <= 24 * 1024 ? 1 : bytes <= 56 * 1024 ? 2 : bytes <= 112 * 1024 ? 3 : 4; }

constexpr int64_t GRID_MIN_NNZ = 300 * 1000;         // loci of at least this many non-zeros go to the grid tier
constexpr int64_t SGRID_MAX_NNZ = 1000 * 1000;       // grid-tier loci below this run on a sub-grid (their passes are barrier latency; above, bandwidth starts to count) ...
constexpr int SGRID_CTAS = 32;                       // ... of this many CTAs (one per SM), beside the other tiers

int cluster_size_for(int64_t nnz) {
   // ~14 B of shared memory per non-zero (row part + CSC index): a CTA's slice stays under ~14k non-zeros, which still
   // fits with its CSC index. Smaller clusters cost latency per iteration (fewer SMs per locus) but less SM time in
   // total; these thresholds were the best of a sweep on the human-shaped workload (profiles/r01_cluster_thresholds.txt).
   if (nnz <= 16 * 1024) return 1;
   if (nnz <= 32 * 1024) return 2;
   if (nnz <= 64 * 1024) return 4;
   if (nnz <= 150 * 1024) return 8;
   return 16;
}

// ---- planner: tier per locus, launch classes, work lists sorted by descending size -------------
// per-locus shape and fragment total from the staged host arrays (while they are still valid)
// (the fragment totals, an O(rows) sum, are taken on the device by locus_frags_kernel and filled in by upload_wait)
void capture_meta_host(sbq_ctx* c) {
   const int64_t *lro = loc_row_off(c), *lio = loc_iso_off(c), *rp = row_ptr(c);
   c->meta.resize((size_t)c->n_loci);
   for (int64_t l = 0; l < c->n_loci; ++l)
      c->meta[l] = {rp[lro[l + 1]] - rp[lro[l]], 0, (int32_t)(lro[l + 1] - lro[l]), (int32_t)(lio[l + 1] - lio[l])};
}

// works from c->meta only, so that batches that exist only on the device (sbq_synth_giant) are planned the same way
int plan(sbq_ctx* c) {
   c->warp_list.clear();
   for (auto& g : c->grid) g.list.clear();
   c->classes.clear();
   c->warp_max_iso = 1;
   c->max_iso_all = 1;
   enum { DUAL, TMA, REG };
   std::vector<char> grid_kernel(c->n_loci, 0);   // giant loci: which of the three grid kernels solves the locus
   std::vector<int64_t> nnz_of(c->n_loci);
   LaunchClass* slot[5][N_BUCKETS] = {};
   std::vector<LaunchClass> tmp;
   tmp.reserve(20);
   for (int64_t l = 0; l < c->n_loci; ++l) {
      const int64_t R = c->meta[l].R, T = c->meta[l].T, nnz = c->meta[l].nnz;
      nnz_of[l] = nnz;
      c->max_iso_all = std::max(c->max_iso_all, (int)T);
      if (T > SBQ_MAX_ISO) return fail(c, SBQ_ERR_UNSUPPORTED, "locus %lld has %lld isoforms (> SBQ_MAX_ISO)", (long long)l, (long long)T);
      int tier;
      if (c->force_tier) tier = c->force_tier;
      // warp tier: one warp per locus, no block barriers, ~1/24 of an SM. Loci of up to 32 isoforms and a few hundred rows belong
      // here even though a lane then walks several rows: they are latency-bound either way, and a CTA of the cluster tier would
      // hold 4 - 30 times more of the SM per iteration (plus its one-off sort / transposed-index setup)
      else if (T <= WT_MAX_ISO && R <= WT_MAX_ROWS && nnz <= WT_MAX_NNZ) tier = 1;
      else if (nnz >= GRID_MIN_NNZ) tier = 3;
      else tier = 2;
      if (tier == 1 && T > WT_MAX_ISO) tier = 2;
      // every T <= SBQ_MAX_ISO fits both the cluster tier (streaming accumulators) and the register-staged grid kernel;
      // the checks stay so that a future change of either limit degrades to the other tier instead of failing the upload
      if (tier == 3 && !grid_tier_supports((int)T)) tier = 2;
      if (tier == 2 && cluster_stream_groups((int)T, SMEM_CAP, CL_NT, 1, 0) <= 0) {
         if (!grid_tier_supports((int)T)) return fail(c, SBQ_ERR_UNSUPPORTED, "locus %lld: %lld isoforms fit no tier", (long long)l, (long long)T);
         tier = 3;
      }
      if (tier == 1) {
         c->warp_list.push_back((int32_t)l);
         c->warp_max_iso = std::max(c->warp_max_iso, (int)T);
      } else if (tier == 3) {
         // class and kernel are functions of the locus alone (a forced tier - tests, tools - keeps the full grid): the bank-aligned
         // two-slot layout (16-bit slot offsets, 32-bit offsets inside the locus, rows short enough on average), else the TMA ring,
         // else the register-staged kernel
         GridClass& g = c->grid[!c->force_tier && nnz < SGRID_MAX_NNZ];
         g.list.push_back((int32_t)l);
         grid_kernel[l] = grid_dual_supports_iso((int)T) && nnz < (1LL << 32) && nnz <= 56 * R ? DUAL :
                          grid_tma_supports((int)T, (long long)R, g.n_cta) ? TMA : REG;
      } else {
         int cs = c->force_cluster ? c->force_cluster : cluster_size_for(nnz);
         int csi = cs == 1 ? 0 : cs == 2 ? 1 : cs == 4 ? 2 : cs == 8 ? 3 : 4;
         const size_t slice = cluster_slice_estimate(nnz, R, (int)T, cs);
         const int bucket = cs == 1 ? smem_bucket(cluster_fixed_doubles((int)T, 1, slice) * sizeof(double) + slice + 256) : N_BUCKETS - 1;
         if (!slot[csi][bucket]) {
            tmp.push_back(LaunchClass{cs, BUCKET_NT[bucket], {}, 0, 0, 0, 0});
            slot[csi][bucket] = &tmp.back();
         }
         LaunchClass* lc = slot[csi][bucket];
         lc->loci.push_back((int32_t)l);
         lc->max_iso = std::max(lc->max_iso, (int)T);
         lc->max_slice = std::max(lc->max_slice, slice);
         // shared memory of the launch = the largest need of its loci (the need is not monotone in T: the exchange area of a
         // narrow locus in a big cluster, CS x T, can exceed that of a wide one, 2T)
         lc->smem = std::max(lc->smem, cluster_class_smem((int)T, slice, lc->nt, cs));
      }
   }
   auto by_size = [&](int32_t a, int32_t b) { return nnz_of[a] != nnz_of[b] ? nnz_of[a] > nnz_of[b] : a < b; };
   {
      // warp-tier work list by descending non-zeros (ties by index): a counting sort - the keys are <= WT_MAX_NNZ unless the
      // tier was forced, and a comparison sort of ~18 k indirect keys costs more host time than the rest of the plan together
      bool small_keys = true;
      for (int32_t l : c->warp_list) small_keys &= nnz_of[l] <= WT_MAX_NNZ;
      if (small_keys) {
         std::vector<int32_t> first(WT_MAX_NNZ + 2, 0), sorted(c->warp_list.size());
         for (int32_t l : c->warp_list) ++first[WT_MAX_NNZ - (int)nnz_of[l] + 1];
         for (int k = 1; k <= WT_MAX_NNZ + 1; ++k) first[k] += first[k - 1];
         for (int32_t l : c->warp_list) sorted[first[WT_MAX_NNZ - (int)nnz_of[l]]++] = l;   // the list is in ascending index order: stable
         c->warp_list.swap(sorted);
      } else {
         std::sort(c->warp_list.begin(), c->warp_list.end(), by_size);
      }
   }
   // two-slot loci, then TMA ring loci, then register-staged loci; inside the first two parts by the warp count the locus' own T
   // selects, so that every launch is homogeneous; then by descending size
   auto warps = [&](int32_t l) { return grid_kernel[l] == DUAL ? grid_dual_nc(c->meta[l].T) : grid_kernel[l] == TMA ? grid_tma_nc(c->meta[l].T) : 0; };
   for (auto& g : c->grid) {
      std::sort(g.list.begin(), g.list.end(), [&](int32_t a, int32_t b) {
         if (grid_kernel[a] != grid_kernel[b]) return grid_kernel[a] < grid_kernel[b];
         const int na = warps(a), nb_ = warps(b);
         if (na != nb_) return na > nb_;
         return by_size(a, b);
      });
      g.n_dual = g.n_tma = 0;
      for (int32_t l : g.list) {
         g.n_dual += grid_kernel[l] == DUAL;
         g.n_tma += grid_kernel[l] == TMA;
      }
      g.rec_off.assign(g.n_dual + 1, 0);
      for (size_t i = 0; i < g.n_dual; ++i) g.rec_off[i + 1] = g.rec_off[i] + c->meta[g.list[i]].R + 1;
   }
   for (auto& lc : tmp) {
      std::sort(lc.loci.begin(), lc.loci.end(), by_size);
      if (cluster_stream_groups(lc.max_iso, SMEM_CAP, lc.nt, 1, 0) <= 0)
         return fail(c, SBQ_ERR_UNSUPPORTED, "locus with %d isoforms does not fit the cluster tier", lc.max_iso);
      c->classes.push_back(std::move(lc));
   }
   // biggest clusters first: they sit on the critical path
   std::sort(c->classes.begin(), c->classes.end(), [](const LaunchClass& a, const LaunchClass& b) { return a.cs != b.cs ? a.cs > b.cs : a.max_slice > b.max_slice; });

   c->h_lists.clear();
   c->warp_list_off = 0;
   if (!c->h_lists.append(c->warp_list.data(), c->warp_list.size())) return fail(c, SBQ_ERR_NOMEM, "list staging");
   for (auto& g : c->grid) {
      g.list_off = c->h_lists.n;
      if (!c->h_lists.append(g.list.data(), g.list.size())) return fail(c, SBQ_ERR_NOMEM, "list staging");
   }
   for (auto& lc : c->classes) {
      lc.list_off = c->h_lists.n;
      if (!c->h_lists.append(lc.loci.data(), lc.loci.size())) return fail(c, SBQ_ERR_NOMEM, "list staging");
   }
   c->stats.loci_warp = (int64_t)c->warp_list.size();
   c->stats.loci_grid = (int64_t)(c->grid[0].list.size() + c->grid[1].list.size());
   c->stats.loci_cta = c->n_loci - c->stats.loci_warp - c->stats.loci_grid;
   return SBQ_SUCCESS;
}

size_t align_up(size_t x, size_t a = 256) { return (x + a - 1) / a * a; }

// device arrays of the batch (sizes from c->n_loci / n_row / n_iso / nnz) and of its results; fills c->dp
int alloc_device(sbq_ctx* c) {
   // +64 B of slack per array: the giant-locus kernel's 16-byte-granular bulk copies may read a few elements past the end
   const size_t sz_lro = align_up((c->n_loci + 1) * sizeof(int64_t)), sz_rp = align_up((c->n_row + 1) * sizeof(int64_t) + 64);
   const size_t sz_col = align_up(c->nnz * sizeof(int32_t) + 64), sz_al = align_up(c->nnz * sizeof(double) + 64);
   const size_t sz_cnt = align_up(c->n_row * sizeof(int32_t) + 64), sz_il = align_up(c->n_iso * sizeof(int32_t));
   const size_t in_bytes = 2 * sz_lro + sz_rp + sz_col + sz_al + 2 * sz_cnt + sz_il;
   const size_t sz_iso_d = align_up(c->n_iso * sizeof(double)), sz_iso_i = align_up(c->n_iso * sizeof(int32_t));
   const size_t sz_loc_i = align_up(c->n_loci * sizeof(int32_t)), sz_loc_d = align_up(c->n_loci * sizeof(double));
   const size_t out_bytes = 4 * sz_iso_d + sz_iso_i + 2 * sz_loc_i + sz_loc_d + 256;
   if (!c->d_in.reserve(in_bytes) || !c->d_out.reserve(out_bytes) || !c->d_lists.reserve(align_up((size_t)c->n_loci * sizeof(int32_t)) + 256))
      return fail(c, SBQ_ERR_NOMEM, "device allocation failed (%zu MB)", (in_bytes + out_bytes) >> 20);

   char* p = (char*)c->d_in.p;
   DevParams& dp = c->dp;
   auto carve = [&](size_t bytes) { char* q = p; p += bytes; return q; };
   int64_t* d_lro = (int64_t*)carve(sz_lro);
   int64_t* d_lio = (int64_t*)carve(sz_lro);
   int64_t* d_rp = (int64_t*)carve(sz_rp);
   int32_t* d_col = (int32_t*)carve(sz_col);
   double* d_al = (double*)carve(sz_al);
   int32_t* d_cnt = (int32_t*)carve(sz_cnt);
   dp.neff = (int32_t*)carve(sz_cnt);
   int32_t* d_il = (int32_t*)carve(sz_il);
   dp.csc = nullptr;   // allocated after the plan, only when the cluster tier has loci
   dp.loc_row_off = d_lro; dp.loc_iso_off = d_lio; dp.row_ptr = d_rp; dp.col = d_col; dp.alpha = d_al;
   dp.count = d_cnt; dp.iso_len = d_il;
   p = (char*)c->d_out.p;
   dp.theta = (double*)carve(sz_iso_d);
   dp.fpkm = (double*)carve(sz_iso_d);
   dp.frac = (double*)carve(sz_iso_d);
   c->d_tpm = (double*)carve(sz_iso_d);
   dp.keep = (int32_t*)carve(sz_iso_i);
   dp.iters = (int32_t*)carve(sz_loc_i);
   dp.status = (int32_t*)carve(sz_loc_i);
   dp.locus_fpkm = (double*)carve(sz_loc_d);
   c->d_fpkm_sum = (double*)carve(256);
   c->d_lists_p = (int32_t*)c->d_lists.p;
   return SBQ_SUCCESS;
}

template <typename K>
int set_kernel_attrs(sbq_ctx* c, K kernel, size_t smem, bool nonportable) {
   CU(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
   if (nonportable) CU(cudaFuncSetAttribute(kernel, cudaFuncAttributeNonPortableClusterSizeAllowed, 1));
   return SBQ_SUCCESS;
}

template <int NT>
int launch_cluster_class_nt(sbq_ctx* c, const LaunchClass& lc, cudaStream_t st) {
   auto kernel = em_cluster_kernel<NT>;
   int rc = set_kernel_attrs(c, kernel, lc.smem, lc.cs > 8);
   if (rc) return rc;
   cudaLaunchConfig_t cfg{};
   cfg.gridDim = dim3((unsigned)(lc.loci.size() * lc.cs));
   cfg.blockDim = dim3(NT);
   cfg.dynamicSmemBytes = lc.smem;
   cfg.stream = st;
   cudaLaunchAttribute attr[1];
   attr[0].id = cudaLaunchAttributeClusterDimension;
   attr[0].val.clusterDim.x = (unsigned)lc.cs;
   attr[0].val.clusterDim.y = 1;
   attr[0].val.clusterDim.z = 1;
   cfg.attrs = attr;
   cfg.numAttrs = 1;
   const int32_t* list = c->d_lists_p + lc.list_off;
   CU(cudaLaunchKernelEx(&cfg, kernel, c->dp, list, (int)lc.loci.size(), (unsigned)lc.smem));
   return SBQ_SUCCESS;
}

// The kernels of one giant-tier class on its stream, each on its part of the list (two-slot, TMA ring, register-staged); the
// one-off layout passes run on the first solve of an upload. Returns 0 or the launchers' negative code.
int launch_grid_class(sbq_ctx* c, GridClass& g, int& n_launch) {
   cudaDeviceProp prop = c->prop;
   prop.multiProcessorCount = g.n_cta;   // the launchers size their grids by it
   const int32_t* d_list = c->d_lists_p + g.list_off;
   const int n_dual = (int)g.n_dual, n_tma = (int)g.n_tma, n_reg = (int)(g.list.size() - g.n_dual - g.n_tma);
   std::vector<int> h_iso(g.list.size());
   for (size_t i = 0; i < g.list.size(); ++i) h_iso[i] = c->meta[g.list[i]].T;
   g.variant = n_dual ? 3 : n_tma ? 2 : 1;
   int rc = 0, nl = 0;
   unsigned short* c16 = (unsigned short*)c->d_col16.p;   // sized by sbq_solve before any giant class launches
   if (n_dual) {
      rc = grid_dual_launch(c->dp, d_list, n_dual, h_iso.data(), g.rec_off.data(), prop, g.scratch, c16, g.rowrec, g.pk, c->col16_ready, g.st, &nl);
      n_launch += nl;
   }
   if (rc == 0 && n_tma) {
      rc = grid_tma_launch(c->dp, d_list + n_dual, n_tma, h_iso.data() + n_dual, prop, g.scratch, c16, c->col16_ready, g.st, &nl);
      n_launch += nl;
   }
   if (rc == 0 && n_reg) {
      rc = grid_tier_launch(c->dp, d_list + n_dual + n_tma, n_reg, prop, g.scratch, g.st, &nl);
      n_launch += nl;
   }
   return rc;
}

// Snapshot of the staging sizes, restored when a submit fails half-way (a failed call leaves the queue unchanged).
struct StagingMark {
   size_t lro, lio, rp, col, al, cnt, il, wseg, wn, wmask, wlen, wpool, wpoff;
   int64_t n_loci, n_row, n_iso, nnz;
   explicit StagingMark(const sbq_ctx* c)
       : lro(c->h_loc_row_off.n), lio(c->h_loc_iso_off.n), rp(c->h_row_ptr.n), col(c->h_col.n), al(c->h_alpha.n), cnt(c->h_count.n), il(c->h_iso_len.n),
         wseg(c->h_wseg.n), wn(c->h_wn.n), wmask(c->h_wmask.n), wlen(c->h_wlen.n), wpool(c->h_wpool.n), wpoff(c->h_wpool_off.n),
         n_loci(c->n_loci), n_row(c->n_row), n_iso(c->n_iso), nnz(c->nnz) {}
   void restore(sbq_ctx* c) const {
      c->h_loc_row_off.n = lro; c->h_loc_iso_off.n = lio; c->h_row_ptr.n = rp; c->h_col.n = col; c->h_alpha.n = al; c->h_count.n = cnt; c->h_iso_len.n = il;
      c->h_wseg.n = wseg; c->h_wn.n = wn; c->h_wmask.n = wmask; c->h_wlen.n = wlen; c->h_wpool.n = wpool; c->h_wpool_off.n = wpoff;
      c->n_loci = n_loci; c->n_row = n_row; c->n_iso = n_iso; c->nnz = nnz;
   }
};

// Append loci to the staged batch; the caller holds c->mu. Every locus is validated (shape, pointers, monotone row_ptr)
// BEFORE anything is appended, and a failed allocation rolls the staging back: an error return leaves the queue as it was.
int submit_locked(sbq_ctx* c, const sbq_locus* loci, int64_t n_loci) {
   if (c->host_released) return fail(c, SBQ_ERR_STATE, "the borrowed batch was released by sbq_upload: sbq_clear and submit again");
   for (int64_t l = 0; l < n_loci; ++l) {
      const sbq_locus& L = loci[l];
      if (L.n_iso < 1 || L.n_row < 0 || !L.row_ptr || !L.iso_len || (L.n_row > 0 && !L.count))
         return fail(c, SBQ_ERR_INVALID, "locus %lld: bad shape or null pointer", (long long)l);
      if (L.n_iso > SBQ_MAX_ISO) return fail(c, SBQ_ERR_UNSUPPORTED, "locus %lld: %d isoforms > SBQ_MAX_ISO", (long long)l, L.n_iso);
      for (int32_t i = 1; i <= L.n_row; ++i)
         if (L.row_ptr[i] < L.row_ptr[i - 1]) return fail(c, SBQ_ERR_INVALID, "locus %lld: row_ptr not monotone", (long long)l);
      if (L.row_ptr[L.n_row] > L.row_ptr[0] && (!L.col || !L.alpha)) return fail(c, SBQ_ERR_INVALID, "locus %lld: null col / alpha", (long long)l);
   }
   cudaSetDevice(c->device);
   int rc = materialise(c);
   if (rc) return rc;
   if ((rc = ensure_origin(c))) return rc;
   const StagingMark mark(c);
   for (int64_t l = 0; l < n_loci; ++l) {
      const sbq_locus& L = loci[l];
      const int64_t k0 = L.row_ptr[0], k1 = L.row_ptr[L.n_row];
      const int64_t base = c->nnz - k0;
      bool ok = c->h_row_ptr.reserve(c->h_row_ptr.n + L.n_row);
      if (ok) {
         for (int32_t i = 1; i <= L.n_row; ++i) c->h_row_ptr.p[c->h_row_ptr.n++] = L.row_ptr[i] + base;
         ok = c->h_col.append(L.col + k0, k1 - k0) && c->h_alpha.append(L.alpha + k0, k1 - k0) &&
              c->h_count.append(L.count, L.n_row) && c->h_iso_len.append(L.iso_len, L.n_iso);
      }
      c->nnz += k1 - k0;
      c->n_row += L.n_row;
      c->n_iso += L.n_iso;
      c->n_loci += 1;
      ok = ok && c->h_loc_row_off.append(&c->n_row, 1) && c->h_loc_iso_off.append(&c->n_iso, 1);
      if (!ok) {
         mark.restore(c);
         return fail(c, SBQ_ERR_NOMEM, "pinned staging");
      }
   }
   c->resident = c->solved = c->downloaded = false;
   return SBQ_SUCCESS;
}

// bootstrap replicates on one device (defined with sbq_bootstrap at the end of this file); the caller holds c->mu
int boot_em_locked(sbq_ctx* c, uint64_t seed, int64_t first, int32_t n);
int boot_finish_locked(sbq_ctx* c);
int boot_counts_locked(sbq_ctx* c, uint64_t seed, int64_t rep, int32_t* count);
int boot_results_locked(sbq_ctx* c, double* theta, double* tpm, int32_t* iters, int32_t* status);
// Gibbs samples on one device (defined with sbq_gibbs at the end of this file); the caller holds c->mu
int gibbs_run_locked(sbq_ctx* c, uint64_t seed, int32_t n, int32_t thin, int32_t burn_in, double prior);
int gibbs_finish_locked(sbq_ctx* c);
int gibbs_results_locked(sbq_ctx* c, double* theta, double* tpm, int32_t* status);

}  // namespace

#include "sbq_multi.cuh"

// ================================================================================================
extern "C" {

int sbq_abi_version(void) { return SBQ_ABI_VERSION; }

const char* sbq_error_string(int err) {
   switch (err) {
      case SBQ_SUCCESS: return "success";
      case SBQ_ERR_INVALID: return "invalid argument";
      case SBQ_ERR_NO_DEVICE: return "no CUDA device (libsbq has no CPU path)";
      case SBQ_ERR_CUDA: return "CUDA runtime error";
      case SBQ_ERR_NOMEM: return "out of memory";
      case SBQ_ERR_STATE: return "invalid call sequence";
      case SBQ_ERR_UNSUPPORTED: return "shape outside supported limits";
      default: return "unknown error";
   }
}

const char* sbq_last_error(const sbq_ctx* c) { return c ? c->err.c_str() : ""; }

void sbq_config_default(sbq_config* cfg) {
   if (!cfg) return;
   memset(cfg, 0, sizeof *cfg);
   cfg->device = -1;
   cfg->max_iter = 1000;
   cfg->theta_tol = 1e-2;
   cfg->row_eps = 1e-5;
   cfg->min_iso_frac = 0.0;
   cfg->effective_len_norm = 0;
   cfg->insert_mean = 0.0;
   cfg->bias_mode = 0;
   cfg->max_out_it = 100;
   cfg->max_theta_it = 5000;
   cfg->max_bias_it = 10;
   cfg->bias_tol = 1e-2;
   cfg->n_gpus = 1;
}

int sbq_create(const sbq_config* cfg, sbq_ctx** out) {
   if (!cfg || !out) return SBQ_ERR_INVALID;
   *out = nullptr;
   if (cfg->max_iter < 1 || !(cfg->theta_tol >= 0) || cfg->bias_mode < 0 || cfg->bias_mode > 1) return SBQ_ERR_INVALID;
   if (cfg->bias_mode == 1 && (cfg->max_out_it < 1 || cfg->max_theta_it < 1 || cfg->max_bias_it < 1 || !(cfg->bias_tol >= 0))) return SBQ_ERR_INVALID;
   if (cfg->n_gpus < 0 || cfg->n_gpus > 64) return SBQ_ERR_INVALID;
   // A solve runs up to ~12 kernels concurrently, one stream each. The default of 8 hardware work queues makes streams share a
   // queue, and a launch then waits behind an unrelated kernel (measured: the warp tier started 2.1 ms late behind the 8-CTA
   // cluster launch). Only effective if the process has not created its CUDA context yet; callers that initialise CUDA first
   // (bench.py, the tests) export the variable themselves.
   setenv("CUDA_DEVICE_MAX_CONNECTIONS", "32", 0);
   int ndev = 0;
   if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
      cudaGetLastError();
      return SBQ_ERR_NO_DEVICE;
   }
   int dev = cfg->device;
   if (dev < 0) {
      if (cfg->n_gpus > 1) dev = 0;   // a multi-GPU context counts its devices from 0 unless told otherwise
      else if (cudaGetDevice(&dev) != cudaSuccess) return SBQ_ERR_NO_DEVICE;
   }
   if (dev >= ndev) return SBQ_ERR_INVALID;
   if (cfg->n_gpus > 1 && dev + cfg->n_gpus > ndev) return SBQ_ERR_NO_DEVICE;
   sbq_ctx* c = new sbq_ctx();
   c->cfg = *cfg;
   c->device = dev;
   auto bail = [&](int code) { sbq_destroy(c); return code; };
   if (cudaSetDevice(dev) != cudaSuccess) return bail(SBQ_ERR_CUDA);
   if (cudaGetDeviceProperties(&c->prop, dev) != cudaSuccess) return bail(SBQ_ERR_CUDA);
   if (c->prop.major < 10) return bail(SBQ_ERR_NO_DEVICE);   // sm_100a code only
   if (cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking) != cudaSuccess) return bail(SBQ_ERR_CUDA);
   if (cudaStreamCreateWithFlags(&c->copy_st, cudaStreamNonBlocking) != cudaSuccess) return bail(SBQ_ERR_CUDA);
   if (cudaEventCreateWithFlags(&c->ev_grid_ready, cudaEventDisableTiming) != cudaSuccess) return bail(SBQ_ERR_CUDA);
   for (auto& e : c->ev_class_ready)
      if (cudaEventCreateWithFlags(&e, cudaEventDisableTiming) != cudaSuccess) return bail(SBQ_ERR_CUDA);
   for (auto& s : c->side)
      if (cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking) != cudaSuccess) return bail(SBQ_ERR_CUDA);
   for (auto& e : c->ev)
      if (cudaEventCreate(&e) != cudaSuccess) return bail(SBQ_ERR_CUDA);
   if (cudaEventCreateWithFlags(&c->ev_fork, cudaEventDisableTiming) != cudaSuccess) return bail(SBQ_ERR_CUDA);
   for (auto& e : c->ev_join)
      if (cudaEventCreateWithFlags(&e, cudaEventDisableTiming) != cudaSuccess) return bail(SBQ_ERR_CUDA);
   for (auto& t : c->lt)
      if (cudaEventCreate(&t.e0) != cudaSuccess || cudaEventCreate(&t.e1) != cudaSuccess) return bail(SBQ_ERR_CUDA);
   c->grid[0].st = c->stream;
   c->grid[0].n_cta = c->prop.multiProcessorCount;
   if (cudaStreamCreateWithFlags(&c->grid[1].st, cudaStreamNonBlocking) != cudaSuccess) return bail(SBQ_ERR_CUDA);
   c->grid[1].n_cta = std::min(SGRID_CTAS, c->prop.multiProcessorCount);
   for (auto& g : c->grid)
      if (cudaEventCreate(&g.lt.e0) != cudaSuccess || cudaEventCreate(&g.lt.e1) != cudaSuccess) return bail(SBQ_ERR_CUDA);
   if (cfg->n_gpus > 1) {
      const int rc = multi_create(c, ndev);
      if (rc) {
         fprintf(stderr, "libsbq: %s\n", c->err.c_str());
         return bail(rc);
      }
   }
   *out = c;
   return SBQ_SUCCESS;
}

void sbq_destroy(sbq_ctx* c) {
   if (!c) return;
   multi_destroy(c);
   cudaSetDevice(c->device);
   if (c->copy_st) cudaStreamSynchronize(c->copy_st);
   if (c->stream) cudaStreamSynchronize(c->stream);
   c->h_loc_row_off.release(); c->h_loc_iso_off.release(); c->h_row_ptr.release();
   c->h_col.release(); c->h_count.release(); c->h_iso_len.release(); c->h_alpha.release();
   c->h_lists.release();
   c->r_theta.release(); c->r_fpkm.release(); c->r_frac.release(); c->r_tpm.release();
   c->r_locus_fpkm.release(); c->r_keep.release(); c->r_iters.release(); c->r_status.release(); c->r_frags.release(); c->d_frags.release();
   c->d_in.release(); c->d_out.release(); c->d_lists.release(); c->d_col16.release(); c->d_csc.release(); c->d_synth.release(); c->d_raw.release(); c->d_raw2.release(); c->d_bias.release();
   for (auto& g : c->grid) {
      g.scratch.release(); g.rowrec.release(); g.pk.release();
      if (g.lt.e0) cudaEventDestroy(g.lt.e0);
      if (g.lt.e1) cudaEventDestroy(g.lt.e1);
   }
   if (c->grid[1].st) cudaStreamSynchronize(c->grid[1].st), cudaStreamDestroy(c->grid[1].st);   // grid[0] runs on c->stream
   c->h_cov.release(); c->r_beta.release(); c->r_outer.release();
   c->h_wseg.release(); c->h_wn.release(); c->h_wmask.release(); c->h_wpool.release(); c->h_wlen.release(); c->h_wpool_off.release(); c->d_weights.release();
   c->boot.prefix.release(); c->boot.scratch.release(); c->boot.out.release(); c->boot.sums.release();
   for (auto& e : c->boot.ev) cudaEventDestroy(e);
   c->gibbs.scratch.release(); c->gibbs.out.release(); c->gibbs.sums.release();
   for (auto& e : c->gibbs.ev) cudaEventDestroy(e);
   for (auto& e : c->ev) if (e) cudaEventDestroy(e);
   if (c->ev_fork) cudaEventDestroy(c->ev_fork);
   for (auto& e : c->ev_join) if (e) cudaEventDestroy(e);
   for (auto& t : c->lt) { if (t.e0) cudaEventDestroy(t.e0); if (t.e1) cudaEventDestroy(t.e1); }
   for (auto& s : c->side) if (s) cudaStreamDestroy(s);
   if (c->ev_grid_ready) cudaEventDestroy(c->ev_grid_ready);
   for (auto& e : c->ev_class_ready) if (e) cudaEventDestroy(e);
   if (c->copy_st) cudaStreamDestroy(c->copy_st);
   if (c->stream) cudaStreamDestroy(c->stream);
   delete c;
}

int sbq_set_plan(sbq_ctx* c, int force_tier, int force_cluster) {
   if (!c) return SBQ_ERR_INVALID;
   if (force_tier < 0 || force_tier > 3) return fail(c, SBQ_ERR_INVALID, "force_tier must be 0..3");
   if (force_cluster != 0 && force_cluster != 1 && force_cluster != 2 && force_cluster != 4 && force_cluster != 8 && force_cluster != 16)
      return fail(c, SBQ_ERR_INVALID, "force_cluster must be 0, 1, 2, 4, 8 or 16");
   if (c->force_tier != force_tier || c->force_cluster != force_cluster) c->resident = c->solved = c->downloaded = false;
   c->force_tier = force_tier;
   c->force_cluster = force_cluster;
   return SBQ_SUCCESS;
}

int sbq_clear(sbq_ctx* c) {
   if (!c) return SBQ_ERR_INVALID;
   std::lock_guard<std::mutex> lk(c->mu);
   if (c->upload_pending) {   // copies of an asynchronous upload still read the host arrays
      cudaSetDevice(c->device);
      cudaStreamSynchronize(c->copy_st);
      c->upload_pending = false;
   }
   if (c->multi && c->raw_mode)
      for (sbq_ctx* ch : c->multi->child) sbq_clear(ch);   // raw loci are staged in the children
   reset_batch(c);
   return SBQ_SUCCESS;
}

int sbq_submit(sbq_ctx* c, const sbq_locus* loci, int64_t n_loci) {
   if (!c || (!loci && n_loci > 0) || n_loci < 0) return SBQ_ERR_INVALID;
   std::lock_guard<std::mutex> lk(c->mu);
   if (c->deferred == 1) return fail(c, SBQ_ERR_STATE, "a batch is either all deferred-weight or all host-weighted");
   const int rc = submit_locked(c, loci, n_loci);
   if (rc == SBQ_SUCCESS && n_loci > 0) c->deferred = 2;
   return rc;
}

int sbq_submit_flat(sbq_ctx* c, int64_t n_loci, const int64_t* lro, const int64_t* lio, const int64_t* rp,
                    const int32_t* col, const double* alpha, const int32_t* count, const int32_t* iso_len) {
   if (!c || n_loci < 0) return SBQ_ERR_INVALID;
   if (n_loci == 0) return SBQ_SUCCESS;
   if (!lro || !lio || !rp || !iso_len) return fail(c, SBQ_ERR_INVALID, "null offset array");
   std::lock_guard<std::mutex> lk(c->mu);
   cudaSetDevice(c->device);
   if (c->deferred == 1) return fail(c, SBQ_ERR_STATE, "a batch is either all deferred-weight or all host-weighted");
   const int64_t rows = lro[n_loci] - lro[0], isos = lio[n_loci] - lio[0];
   if (rows < 0 || isos < n_loci) return fail(c, SBQ_ERR_INVALID, "bad locus offsets");
   const int64_t k0 = rp[lro[0]], k1 = rp[lro[n_loci]];
   if (k1 < k0 || (k1 > k0 && (!col || !alpha)) || (rows > 0 && !count)) return fail(c, SBQ_ERR_INVALID, "bad CSR arrays");
   for (int64_t l = 0; l < n_loci; ++l) {
      const int64_t T = lio[l + 1] - lio[l];
      if (lro[l + 1] < lro[l] || T < 1) return fail(c, SBQ_ERR_INVALID, "locus %lld: bad shape", (long long)l);
      if (T > SBQ_MAX_ISO) return fail(c, SBQ_ERR_UNSUPPORTED, "locus %lld: %lld isoforms > SBQ_MAX_ISO", (long long)l, (long long)T);
   }
   // zero-copy: a first, origin-based submission whose arrays are already page-locked is used in place
   if (c->n_loci == 0 && lro[0] == 0 && lio[0] == 0 && k0 == 0 && is_pinned(lro) && is_pinned(lio) && is_pinned(rp) &&
       is_pinned(iso_len) && (rows == 0 || is_pinned(count)) && (k1 == 0 || (is_pinned(col) && is_pinned(alpha)))) {
      c->borrowed = true;
      c->b_loc_row_off = lro; c->b_loc_iso_off = lio; c->b_row_ptr = rp;
      c->b_col = col; c->b_alpha = alpha; c->b_count = count; c->b_iso_len = iso_len;
      c->n_loci = n_loci; c->n_row = rows; c->n_iso = isos; c->nnz = k1;
      c->deferred = 2;
      c->resident = c->solved = c->downloaded = false;
      return SBQ_SUCCESS;
   }
   if (c->host_released) return fail(c, SBQ_ERR_STATE, "the borrowed batch was released by sbq_upload: sbq_clear and submit again");
   for (int64_t i = lro[0]; i < lro[n_loci]; ++i)
      if (rp[i + 1] < rp[i]) return fail(c, SBQ_ERR_INVALID, "row %lld: row_ptr not monotone", (long long)i);
   int rc = materialise(c);
   if (rc) return rc;
   if ((rc = ensure_origin(c))) return rc;
   // reserve everything first: nothing is appended unless all of it fits (a failed call leaves the queue unchanged)
   const bool ok = c->h_loc_row_off.reserve(c->h_loc_row_off.n + n_loci) && c->h_loc_iso_off.reserve(c->h_loc_iso_off.n + n_loci) &&
                   c->h_row_ptr.reserve(c->h_row_ptr.n + rows) && c->h_col.reserve(c->h_col.n + (k1 - k0)) && c->h_alpha.reserve(c->h_alpha.n + (k1 - k0)) &&
                   c->h_count.reserve(c->h_count.n + rows) && c->h_iso_len.reserve(c->h_iso_len.n + isos);
   if (!ok) return fail(c, SBQ_ERR_NOMEM, "pinned staging");
   for (int64_t l = 1; l <= n_loci; ++l) {
      c->h_loc_row_off.p[c->h_loc_row_off.n++] = c->n_row + (lro[l] - lro[0]);
      c->h_loc_iso_off.p[c->h_loc_iso_off.n++] = c->n_iso + (lio[l] - lio[0]);
   }
   const int64_t base = c->nnz - k0;
   for (int64_t i = 1; i <= rows; ++i) c->h_row_ptr.p[c->h_row_ptr.n++] = rp[lro[0] + i] + base;
   c->h_col.append(col + k0, k1 - k0);
   c->h_alpha.append(alpha + k0, k1 - k0);
   c->h_count.append(count + lro[0], rows);
   c->h_iso_len.append(iso_len + lio[0], isos);
   c->n_loci += n_loci; c->n_row += rows; c->n_iso += isos; c->nnz += k1 - k0;
   c->deferred = 2;
   c->resident = c->solved = c->downloaded = false;
   return SBQ_SUCCESS;
}

int sbq_validate(sbq_ctx* c) {
   if (!c) return SBQ_ERR_INVALID;
   std::lock_guard<std::mutex> lk(c->mu);
   if (c->host_released) return fail(c, SBQ_ERR_STATE, "the borrowed batch was released by sbq_upload");
   const int64_t *lro = loc_row_off(c), *lio = loc_iso_off(c), *rp = row_ptr(c);
   const int32_t* col = colp(c);
   for (int64_t l = 0; l < c->n_loci; ++l) {
      const int64_t T = lio[l + 1] - lio[l];
      for (int64_t i = lro[l]; i < lro[l + 1]; ++i) {
         if (rp[i + 1] < rp[i]) return fail(c, SBQ_ERR_INVALID, "locus %lld row %lld: row_ptr not monotone", (long long)l, (long long)(i - lro[l]));
         for (int64_t k = rp[i]; k < rp[i + 1]; ++k) {
            if (col[k] < 0 || col[k] >= T) return fail(c, SBQ_ERR_INVALID, "locus %lld: column %d out of range", (long long)l, col[k]);
            if (k > rp[i] && col[k] <= col[k - 1]) return fail(c, SBQ_ERR_INVALID, "locus %lld row %lld: columns not strictly ascending", (long long)l, (long long)(i - lro[l]));
         }
      }
   }
   return SBQ_SUCCESS;
}

} // extern "C" (reopened below)

// Host -> device copies of the staged batch, ENQUEUED in the order the solve needs them (caller holds c->mu):
//   1. offsets, row pointers, counts, lengths and ALL columns in bulk - while they move, the host plans the tiers;
//   2. the weights (two thirds of the bytes) locus by locus for the launches on the critical path: giant loci, then the
//      cluster-tier launches of 8 and 16 CTAs per locus (a few dozen large loci), one "ready" event per launch;
//   3. the weights of everything else (the gaps between the ranges of step 2).
// sbq_solve makes every launch wait for its own event only, so the largest loci start iterating while the rest of the batch
// is still crossing PCIe. Nothing is synchronised here: the host arrays must stay valid until upload_finish / the solve.
static int raw_upload(sbq_ctx* c);   // raw loci: class assignment on the device (defined further down)

static int upload_begin(sbq_ctx* c) {
   CU(cudaSetDevice(c->device));
   if (c->upload_pending) {
      CU(cudaStreamSynchronize(c->copy_st));
      c->upload_pending = false;
   }
   if (c->n_loci == 0) return fail(c, SBQ_ERR_STATE, "nothing submitted");
   if (c->host_released) return fail(c, SBQ_ERR_STATE, "the borrowed batch was released by the previous sbq_upload: sbq_clear and submit again");
   {
      const int rc = alloc_device(c);
      if (rc) return rc;
   }
   DevParams& dp = c->dp;
   int64_t *d_lro = const_cast<int64_t*>(dp.loc_row_off), *d_lio = const_cast<int64_t*>(dp.loc_iso_off), *d_rp = const_cast<int64_t*>(dp.row_ptr);
   int32_t *d_col = const_cast<int32_t*>(dp.col), *d_cnt = const_cast<int32_t*>(dp.count), *d_il = const_cast<int32_t*>(dp.iso_len);
   double* d_al = const_cast<double*>(dp.alpha);

   cudaStream_t st = c->copy_st;
   c->upload_pending = true;
   c->resident = c->solved = c->downloaded = false;
   c->boot.prefix_ready = c->boot.done = c->gibbs.done = false;
   CU(cudaEventRecord(c->ev[0], st));
   CU(cudaMemcpyAsync(d_lro, loc_row_off(c), (c->n_loci + 1) * sizeof(int64_t), cudaMemcpyHostToDevice, st));
   CU(cudaMemcpyAsync(d_lio, loc_iso_off(c), (c->n_loci + 1) * sizeof(int64_t), cudaMemcpyHostToDevice, st));
   CU(cudaMemcpyAsync(d_rp, row_ptr(c), (c->n_row + 1) * sizeof(int64_t), cudaMemcpyHostToDevice, st));
   if (c->n_row) CU(cudaMemcpyAsync(d_cnt, countp(c), c->n_row * sizeof(int32_t), cudaMemcpyHostToDevice, st));
   CU(cudaMemcpyAsync(d_il, iso_lenp(c), c->n_iso * sizeof(int32_t), cudaMemcpyHostToDevice, st));
   // fragment total of every locus (metric accounting only), summed on the device from the counts that just arrived
   if (!c->r_frags.reserve((size_t)c->n_loci) || !c->d_frags.reserve(align_up((size_t)c->n_loci * 8))) return fail(c, SBQ_ERR_NOMEM, "fragment-total buffers");
   locus_frags_kernel<<<std::max(1, std::min<int>((int)((c->n_loci + 7) / 8), c->prop.multiProcessorCount * 8)), 256, 0, st>>>(d_lro, d_cnt, c->n_loci, (long long*)c->d_frags.p);
   CU(cudaGetLastError());
   CU(cudaMemcpyAsync(c->r_frags.p, c->d_frags.p, (size_t)c->n_loci * 8, cudaMemcpyDeviceToHost, st));
   if (c->nnz) CU(cudaMemcpyAsync(d_col, colp(c), c->nnz * sizeof(int32_t), cudaMemcpyHostToDevice, st));
   const bool timing = getenv("SBQ_TIMING") != nullptr;
   const auto t_plan0 = std::chrono::steady_clock::now();
   // the tier plan (O(loci + rows) on the host) is made while the DMA engine moves the first ~40 % of the bytes
   {
      capture_meta_host(c);
      const int rc = plan(c);
      if (rc) {
         cudaStreamSynchronize(st);
         c->upload_pending = false;
         return rc;
      }
   }
   if (timing) fprintf(stderr, "SBQ_TIMING plan_ms %.3f\n", std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_plan0).count());
   if (c->h_lists.n) CU(cudaMemcpyAsync(c->d_lists_p, c->h_lists.p, c->h_lists.n * sizeof(int32_t), cudaMemcpyHostToDevice, st));
   // weights in priority order
   const int64_t* lro = loc_row_off(c);
   const int64_t* rp = row_ptr(c);
   const double* al = alphap(c);
   std::vector<std::pair<int64_t, int64_t>> done;   // [k0, k1) ranges already enqueued
   auto copy_loci = [&](const std::vector<int32_t>& loci) -> int {
      for (int32_t l : loci) {
         const int64_t k0 = rp[lro[l]], k1 = rp[lro[l + 1]];
         if (k1 > k0) {
            CU(cudaMemcpyAsync(d_al + k0, al + k0, (size_t)(k1 - k0) * sizeof(double), cudaMemcpyHostToDevice, st));
            done.emplace_back(k0, k1);
         }
      }
      return SBQ_SUCCESS;
   };
   for (auto& r : c->class_ready) r = false;
   c->grid_ready = false;
   const size_t n_giant = c->grid[0].list.size() + c->grid[1].list.size();
   if (n_giant > 0 && n_giant <= 16) {
      for (auto& g : c->grid) {
         const int rc = copy_loci(g.list);
         if (rc) return rc;
      }
      CU(cudaEventRecord(c->ev_grid_ready, st));
      c->grid_ready = true;
   }
   // Only launches of a few LARGE loci are worth their own copies: a copy costs ~6 us of DMA set-up whatever its size (measured:
   // 1150 per-locus copies took 7.3 ms for the 66 MB that seven bulk copies move in 1.5 ms).
   size_t n_prio = 0;
   for (size_t i = 0; i < c->classes.size() && i < (size_t)N_SIDE_STREAMS; ++i) {
      if (c->classes[i].cs < 8 || n_prio + c->classes[i].loci.size() > 48) continue;   // the rest goes with the bulk of step 3
      n_prio += c->classes[i].loci.size();
      const int rc = copy_loci(c->classes[i].loci);
      if (rc) return rc;
      CU(cudaEventRecord(c->ev_class_ready[i], st));
      c->class_ready[i] = true;
   }
   std::sort(done.begin(), done.end());
   int64_t pos = 0;
   for (size_t i = 0; i <= done.size(); ++i) {
      const int64_t end = i < done.size() ? done[i].first : c->nnz;
      if (end > pos) CU(cudaMemcpyAsync(d_al + pos, al + pos, (size_t)(end - pos) * sizeof(double), cudaMemcpyHostToDevice, st));
      if (i < done.size()) pos = std::max(pos, done[i].second);
   }
   CU(cudaEventRecord(c->ev[1], st));   // everything is on the device when this fires
   if (!c->classes.empty()) {
      // L2-resident overflow of the cluster tier's transposed index (4 B per non-zero, indexed like col/alpha)
      if (!c->d_csc.reserve(align_up(c->nnz * 4 + 16))) return fail(c, SBQ_ERR_NOMEM, "device allocation failed (transposed-index scratch)");
      dp.csc = (unsigned*)c->d_csc.p;
   }
   c->stats.h2d_bytes = 2 * (c->n_loci + 1) * 8 + (c->n_row + 1) * 8 + c->nnz * 12 + c->n_row * 4 + c->n_iso * 4 + (int64_t)c->h_lists.n * 4;
   c->stats.n_loci = c->n_loci; c->stats.n_row = c->n_row; c->stats.n_iso = c->n_iso; c->stats.nnz = c->nnz;
   c->stats.weights_ms = 0.0;
   c->col16_ready = false;
   c->resident = true;                  // the solve may be enqueued: its launches wait for the "ready" events
   return SBQ_SUCCESS;
}

// wait for the copies of upload_begin (the caller's arrays may be released afterwards) and record the upload time
static int upload_wait(sbq_ctx* c) {
   if (!c->upload_pending) return SBQ_SUCCESS;
   CU(cudaSetDevice(c->device));
   CU(cudaStreamSynchronize(c->copy_st));
   c->upload_pending = false;
   if (c->borrowed) c->host_released = true;   // from here on nothing reads the caller's arrays (metric accounting uses c->meta)
   for (size_t l = 0; l < c->meta.size(); ++l) c->meta[l].frags = c->r_frags.p[l];
   float ms = 0;
   CU(cudaEventElapsedTime(&ms, c->ev[0], c->ev[1]));
   c->stats.upload_ms = ms;
   return SBQ_SUCCESS;
}

// The EM launches of one solve of the resident batch, into the outputs c->dp points at: grid tier, cluster classes and warp tier
// forked from c->stream and joined back onto it. sbq_solve runs it once, sbq_bootstrap once per replicate with dp.count pointing at
// the replicate's counts. pending: the launches wait for the copies of an asynchronous upload.
static int launch_em(sbq_ctx* c, bool pending, int64_t& launches) {
   cudaStream_t st = c->stream;
   CU(cudaEventRecord(c->ev_fork, st));
   for (auto& t : c->lt) t.used = false;
   if (!(c->grid[0].list.empty() && c->grid[1].list.empty())) {
      // the 16-bit slot array is shared by both classes (indexed by non-zero): sized here, so that neither launch re-allocates it
      // under the other
      const size_t need16 = (size_t)c->nnz * 2 + 256;
      if (need16 > c->d_col16.cap) {
         if (!c->d_col16.reserve(need16)) return fail(c, SBQ_ERR_NOMEM, "device allocation failed (16-bit slots)");
         c->col16_ready = false;
      }
   }
   // grid tier first: the full grid on the main stream (it owns the whole GPU while it runs), then the sub-grid on its own stream,
   // launched before the cluster classes so that it is resident when they fill the other SMs
   for (int k = 0; k < 2; ++k) {
      GridClass& g = c->grid[k];
      g.lt.used = false;
      if (g.list.empty()) continue;
      CU(cudaStreamWaitEvent(g.st, c->ev_fork, 0));
      if (k == 1 && c->grid[0].lt.used) CU(cudaStreamWaitEvent(g.st, c->grid[0].lt.e1, 0));   // the full-grid class owns the GPU first
      if (pending) CU(cudaStreamWaitEvent(g.st, c->grid_ready ? c->ev_grid_ready : c->ev[1], 0));
      CU(cudaEventRecord(g.lt.e0, g.st));
      int n_launch = 0;
      const int rc = launch_grid_class(c, g, n_launch);
      if (rc != 0) {
         // the one-off layout passes permute alpha inside each giant row IN PLACE: after a failure the resident copy can no
         // longer be trusted to match the column arrays, so the batch has to be uploaded again
         c->resident = false;
         c->col16_ready = false;
         return fail(c, rc < -6 ? SBQ_ERR_CUDA : rc, "grid tier launch failed: %s", cudaGetErrorString(cudaGetLastError()));
      }
      launches += n_launch;
      CU(cudaEventRecord(g.lt.e1, g.st));
      g.lt.used = true;
   }
   if (!(c->grid[0].list.empty() && c->grid[1].list.empty())) c->col16_ready = true;
   // Launch order: the cluster classes (biggest clusters first, see plan()), then the warp tier. The work distributor serves
   // kernels roughly in launch order, 16- and 8-CTA clusters strand a few SMs per GPC that only single CTAs can use, and the
   // many small loci have critical paths of their own (~1 ms): see DESIGN.md section 5 for the measured timelines.
   const int ncls = (int)c->classes.size();
   for (int i = 0; i < ncls; ++i) {
      const LaunchClass& lc = c->classes[i];
      cudaStream_t ss = c->side[i % N_SIDE_STREAMS];
      if (i < N_SIDE_STREAMS) CU(cudaStreamWaitEvent(ss, c->ev_fork, 0));
      if (pending) CU(cudaStreamWaitEvent(ss, (i < N_SIDE_STREAMS && c->class_ready[i]) ? c->ev_class_ready[i] : c->ev[1], 0));
      LaunchTimer& t = c->lt[1 + i % N_SIDE_STREAMS];
      CU(cudaEventRecord(t.e0, ss));
      // one arm per thread count of BUCKET_NT
      int rc = lc.nt == 64 ? launch_cluster_class_nt<64>(c, lc, ss) : lc.nt == 128 ? launch_cluster_class_nt<128>(c, lc, ss) :
               launch_cluster_class_nt<512>(c, lc, ss);
      if (rc) return rc;
      CU(cudaEventRecord(t.e1, ss));
      t.used = true;
      ++launches;
   }
   if (!c->warp_list.empty()) {
      const size_t smem = warp_tier_smem_bytes(c->warp_max_iso);
      CU(cudaFuncSetAttribute(em_warp_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
      const int n = (int)c->warp_list.size();
      int per_sm = 1;
      CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, em_warp_kernel, WT_WARPS * 32, smem));
      const int grid = std::max(1, std::min((n + WT_WARPS - 1) / WT_WARPS, per_sm * c->prop.multiProcessorCount));   // persistent warps: the grid only sets the parallelism
      int* queue = (int*)((char*)c->d_fpkm_sum + 64);
      if (pending) CU(cudaStreamWaitEvent(st, c->ev[1], 0));   // many small loci all over the batch: they need everything
      CU(cudaMemsetAsync(queue, 0, sizeof(int), st));
      CU(cudaEventRecord(c->lt[0].e0, st));
      em_warp_kernel<<<grid, WT_WARPS * 32, smem, st>>>(c->dp, c->d_lists_p + c->warp_list_off, n, c->warp_max_iso, queue);
      CU(cudaGetLastError());
      CU(cudaEventRecord(c->lt[0].e1, st));
      c->lt[0].used = true;
      ++launches;
   }
   for (int i = 0; i < std::min(ncls, N_SIDE_STREAMS); ++i) {
      CU(cudaEventRecord(c->ev_join[i], c->side[i]));
      CU(cudaStreamWaitEvent(st, c->ev_join[i], 0));
   }
   if (c->grid[1].lt.used) CU(cudaStreamWaitEvent(st, c->grid[1].lt.e1, 0));
   return SBQ_SUCCESS;
}

extern "C" {

int sbq_upload_begin(sbq_ctx* c) {
   if (!c) return SBQ_ERR_INVALID;
   if (c->multi || c->deferred == 1 || c->raw_mode || c->cfg.bias_mode == 1) return sbq_upload(c);   // these paths have extra stages: synchronous upload
   std::lock_guard<std::mutex> lk(c->mu);
   return upload_begin(c);
}

int sbq_upload(sbq_ctx* c) {
   if (!c) return SBQ_ERR_INVALID;
   if (c->multi) return multi_upload(c);
   std::lock_guard<std::mutex> lk(c->mu);
   if (c->raw_mode) {
      if (c->n_loci == 0) return fail(c, SBQ_ERR_STATE, "nothing submitted");
      return raw_upload(c);
   }
   {
      int rc = upload_begin(c);
      if (!rc) rc = upload_wait(c);   // borrowed host arrays may be released after this returns
      if (rc) return rc;
   }
   if (c->deferred == 1) {
      // alpha on the GPU: upload the per-entry descriptors and the insert model, one warp per CSR entry
      if (!c->have_model) return fail(c, SBQ_ERR_STATE, "deferred weights need sbq_set_insert_model()");
      if ((int64_t)c->h_wseg.n != c->nnz) return fail(c, SBQ_ERR_STATE, "deferred-weight descriptors do not cover the batch");
      const size_t b_seg = align_up(c->nnz * 8 + 8), b_n = align_up(c->nnz + 8), b_m = align_up(c->nnz * 4 + 8), b_l = align_up(c->nnz * 4 + 8);
      const size_t b_pool = align_up(c->h_wpool.n * 4 + 8), b_emp = align_up(c->model_emp.size() * 8 + 8);
      if (!c->d_weights.reserve(b_seg + b_n + b_m + b_l + b_pool + b_emp)) return fail(c, SBQ_ERR_NOMEM, "device allocation failed (weight descriptors)");
      char* q = (char*)c->d_weights.p;
      int64_t* d_seg = (int64_t*)q; q += b_seg;
      uint8_t* d_n = (uint8_t*)q; q += b_n;
      uint32_t* d_m = (uint32_t*)q; q += b_m;
      int32_t* d_l = (int32_t*)q; q += b_l;
      uint32_t* d_pool = (uint32_t*)q; q += b_pool;
      double* d_emp = (double*)q;
      cudaStream_t st = c->stream;
      CU(cudaEventRecord(c->ev[5], st));
      CU(cudaMemcpyAsync(d_seg, c->h_wseg.p, c->nnz * 8, cudaMemcpyHostToDevice, st));
      CU(cudaMemcpyAsync(d_n, c->h_wn.p, c->nnz, cudaMemcpyHostToDevice, st));
      CU(cudaMemcpyAsync(d_m, c->h_wmask.p, c->nnz * 4, cudaMemcpyHostToDevice, st));
      CU(cudaMemcpyAsync(d_l, c->h_wlen.p, c->nnz * 4, cudaMemcpyHostToDevice, st));
      if (c->h_wpool.n) CU(cudaMemcpyAsync(d_pool, c->h_wpool.p, c->h_wpool.n * 4, cudaMemcpyHostToDevice, st));
      if (!c->model_emp.empty()) CU(cudaMemcpyAsync(d_emp, c->model_emp.data(), c->model_emp.size() * 8, cudaMemcpyHostToDevice, st));
      WeightModel wm{c->model.use_emp, c->model.start_offset, c->model.end_offset, c->model.total_reads, d_emp, c->model.mean, c->model.sd, c->model_read_len};
      const int blocks = std::max(1, std::min<int>((int)((c->nnz + 7) / 8), c->prop.multiProcessorCount * 16));
      weights_kernel<uint8_t><<<blocks, 256, 0, st>>>(c->nnz, d_seg, d_n, d_m, d_l, d_pool, wm, const_cast<double*>(c->dp.alpha));
      CU(cudaGetLastError());
      CU(cudaEventRecord(c->ev[6], st));
      CU(cudaStreamSynchronize(st));
      float wms = 0;
      CU(cudaEventElapsedTime(&wms, c->ev[5], c->ev[6]));
      c->weights_ms = wms;
      c->stats.weights_ms = wms;
      c->stats.h2d_bytes += (int64_t)(c->nnz * 17 + c->h_wpool.n * 4 + c->model_emp.size() * 8);
   }
   if (c->cfg.bias_mode == 1) {
      if (!c->have_cov) return fail(c, SBQ_ERR_STATE, "bias_mode = 1 needs sbq_set_covariates() after the last submit");
      const size_t K = (size_t)c->n_cov;
      const size_t bx = align_up(c->n_row * K * 8 + 8), bw = align_up(c->n_row * 8 + 8), bb = align_up(c->n_loci * K * 8 + 8), bo = align_up(c->n_loci * 4 + 8);
      if (!c->d_bias.reserve(bx + 2 * bw + bb + 2 * bo + 64)) return fail(c, SBQ_ERR_NOMEM, "device allocation failed (bias scratch)");
      char* q = (char*)c->d_bias.p;
      c->bpar.x = (const double*)q; q += bx;
      c->bpar.w = (double*)q; q += bw;
      c->bpar.d = (double*)q; q += bw;
      c->bpar.beta = (double*)q; q += bb;
      c->bpar.outer = (int32_t*)q; q += bo;
      c->d_bias_list = (int32_t*)q; q += bo;
      c->d_bias_queue = (int*)q;
      c->bpar.n_cov = c->n_cov;
      // launch classes of the bias kernel: cluster size by non-zeros (a function of the locus alone), biggest loci first
      {
         c->bias_list.clear();
         std::vector<int32_t> cls[6];
         for (int k = 0; k < 6; ++k) c->bias_cls[k] = BiasClass{};
         for (int64_t l = 0; l < c->n_loci; ++l) {
            const int cs = bias_cluster_size(c->meta[l].nnz);
            // class 5: small loci, one warp each (em_bias_warp_kernel)
            const int k = bias_warp_tier(c->meta[l].nnz, c->meta[l].R, c->meta[l].T) ? 5 : cs == 16 ? 0 : cs == 8 ? 1 : cs == 4 ? 2 : cs == 2 ? 3 : 4;
            cls[k].push_back((int32_t)l);
            c->bias_cls[k].cs = cs;
            c->bias_cls[k].max_iso = std::max(c->bias_cls[k].max_iso, (int)c->meta[l].T);
         }
         for (int k = 0; k < 6; ++k) {
            std::sort(cls[k].begin(), cls[k].end(), [&](int32_t a, int32_t b) { return c->meta[a].nnz != c->meta[b].nnz ? c->meta[a].nnz > c->meta[b].nnz : a < b; });
            c->bias_cls[k].off = c->bias_list.size();
            c->bias_cls[k].n = cls[k].size();
            c->bias_list.insert(c->bias_list.end(), cls[k].begin(), cls[k].end());
         }
         if (c->n_loci) CU(cudaMemcpyAsync(c->d_bias_list, c->bias_list.data(), c->n_loci * 4, cudaMemcpyHostToDevice, c->stream));
      }
      if (K) CU(cudaMemcpyAsync((void*)c->bpar.x, c->h_cov.p, c->n_row * K * 8, cudaMemcpyHostToDevice, c->stream));
      CU(cudaStreamSynchronize(c->stream));
      c->stats.h2d_bytes += (int64_t)(c->n_row * K * 8);
   }
   c->resident = true;
   c->col16_ready = false;
   c->solved = c->downloaded = false;
   return SBQ_SUCCESS;
}

int sbq_solve(sbq_ctx* c, int64_t total_mapped_reads) {
   if (!c) return SBQ_ERR_INVALID;
   if (c->multi) return multi_solve(c, total_mapped_reads);
   std::lock_guard<std::mutex> lk(c->mu);
   CU(cudaSetDevice(c->device));
   if (!c->resident) return fail(c, SBQ_ERR_STATE, "sbq_solve before sbq_upload");

   DevParams& dp = c->dp;
   dp.max_iter = c->cfg.max_iter;
   dp.tol = c->cfg.theta_tol;
   dp.row_eps = c->cfg.row_eps;
   dp.min_frac = c->cfg.min_iso_frac;
   dp.eff_len_norm = c->cfg.effective_len_norm;
   dp.insert_mean = c->cfg.insert_mean;
   dp.rpm = 1e6 / (double)(int)total_mapped_reads;   // total_mapped_reads() returns int (src/estimate.cpp:328)

   cudaStream_t st = c->stream;
   int64_t launches = 0;
   if (c->cfg.bias_mode == 1) {
      // bias-corrected EM: one fused kernel (theta-EM + bias-weight update + both convergence tests), one cluster of 1 - 16 CTAs
      // per locus; one launch per cluster size, concurrently on the side streams, the biggest clusters first
      const size_t smem = bias_smem_bytes(c->max_iso_all);
      if (smem > SMEM_CAP) return fail(c, SBQ_ERR_UNSUPPORTED, "bias mode supports up to %d isoforms per locus", (int)((SMEM_CAP / 8 - 8) / (5 + BI_W)));
      c->bpar.max_out_it = c->cfg.max_out_it;
      c->bpar.max_theta_it = c->cfg.max_theta_it;
      c->bpar.max_bias_it = c->cfg.max_bias_it;
      c->bpar.bias_tol = c->cfg.bias_tol;
      int rc_attr = set_kernel_attrs(c, em_bias_kernel, smem, c->bias_cls[0].n > 0);
      if (rc_attr) return rc_attr;
      CU(cudaEventRecord(c->ev[2], st));
      CU(cudaEventRecord(c->ev_fork, st));
      int n_side = 0;
      if (c->bias_cls[5].n) {
         // small loci: persistent warps, one locus per warp at a time (longest first); runs beside the cluster launches
         const BiasClass& bc = c->bias_cls[5];
         cudaStream_t ss = c->side[n_side];
         CU(cudaStreamWaitEvent(ss, c->ev_fork, 0));
         ++n_side;
         const size_t wsmem = bias_warp_smem_bytes();
         CU(cudaFuncSetAttribute(em_bias_warp_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)wsmem));
         int occ = 1;
         CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, em_bias_warp_kernel, BW_WARPS * 32, wsmem));
         const long long want = ((long long)bc.n + BW_WARPS - 1) / BW_WARPS;
         const unsigned grid = (unsigned)std::max(1LL, std::min(want, (long long)c->prop.multiProcessorCount * std::max(1, occ)));
         CU(cudaMemsetAsync(c->d_bias_queue, 0, sizeof(int), ss));
         em_bias_warp_kernel<<<grid, BW_WARPS * 32, wsmem, ss>>>(c->dp, c->bpar, (const int32_t*)(c->d_bias_list + bc.off), (int)bc.n, c->d_bias_queue);
         CU(cudaGetLastError());
         ++launches;
      }
      for (int k = 0; k < 5; ++k) {
         const BiasClass& bc = c->bias_cls[k];
         if (!bc.n) continue;
         cudaStream_t ss = c->side[n_side % N_SIDE_STREAMS];
         if (n_side < N_SIDE_STREAMS) CU(cudaStreamWaitEvent(ss, c->ev_fork, 0));
         ++n_side;
         cudaLaunchConfig_t cfg{};
         cfg.gridDim = dim3((unsigned)(bc.n * bc.cs));
         cfg.blockDim = dim3(BI_NT);
         cfg.dynamicSmemBytes = bias_smem_bytes(bc.max_iso);
         cfg.stream = ss;
         cudaLaunchAttribute attr[1];
         attr[0].id = cudaLaunchAttributeClusterDimension;
         attr[0].val.clusterDim.x = (unsigned)bc.cs;
         attr[0].val.clusterDim.y = 1;
         attr[0].val.clusterDim.z = 1;
         cfg.attrs = attr;
         cfg.numAttrs = 1;
         CU(cudaLaunchKernelEx(&cfg, em_bias_kernel, c->dp, c->bpar, (const int32_t*)(c->d_bias_list + bc.off), (int)bc.n));
         ++launches;
      }
      for (int i = 0; i < std::min(n_side, N_SIDE_STREAMS); ++i) {
         CU(cudaEventRecord(c->ev_join[i], c->side[i]));
         CU(cudaStreamWaitEvent(st, c->ev_join[i], 0));
      }
      CU(cudaEventRecord(c->ev[3], st));
      fpkm_sum_kernel<<<1, 1024, 0, st>>>(dp.locus_fpkm, c->n_loci, c->d_fpkm_sum);
      CU(cudaGetLastError());
      CU(cudaEventRecord(c->ev[4], st));
      CU(cudaStreamSynchronize(st));
      float ms_ = 0;
      CU(cudaEventElapsedTime(&ms_, c->ev[2], c->ev[4]));
      c->stats.solve_ms = ms_;
      CU(cudaEventElapsedTime(&ms_, c->ev[2], c->ev[3]));
      c->stats.em_ms = ms_;
      c->stats.grid_em_ms = 0;
      c->stats.kernel_launches = launches + 1;
      c->launch_stats.clear();
      c->locus_launch.assign(c->n_loci, -1);
      c->solved = true;
      c->downloaded = false;
      return SBQ_SUCCESS;
   }
   CU(cudaEventRecord(c->ev[2], st));
   c->stats.grid_em_ms = 0;
   const bool pending = c->upload_pending;   // asynchronous upload in flight: every launch waits for the copies it needs only
   {
      const int rc = launch_em(c, pending, launches);
      if (rc) return rc;
   }
   CU(cudaEventRecord(c->ev[3], st));
   fpkm_sum_kernel<<<1, 1024, 0, st>>>(dp.locus_fpkm, c->n_loci, c->d_fpkm_sum);
   CU(cudaGetLastError());
   ++launches;
   CU(cudaEventRecord(c->ev[4], st));
   CU(cudaStreamSynchronize(st));
   if (pending) {
      const int rcw = upload_wait(c);   // complete by now (the last launches waited for it): records the upload time, releases the host arrays
      if (rcw) return rcw;
   }
   float ms = 0;
   CU(cudaEventElapsedTime(&ms, c->ev[2], c->ev[4]));
   c->stats.solve_ms = ms;
   CU(cudaEventElapsedTime(&ms, c->ev[2], c->ev[3]));
   c->stats.em_ms = ms;
   // per-launch records: [warp] [grid classes...] [cluster classes...]
   c->launch_stats.clear();
   c->locus_launch.assign(c->n_loci, -1);
   auto add_stat = [&](int kind, int cs, int lpr, const std::vector<int32_t>& loci, double ms_, cudaEvent_t e0 = nullptr) {
      sbq_launch_stat ls{};
      ls.kind = kind; ls.cluster_size = cs; ls.lanes_per_row = lpr; ls.n_loci = (int64_t)loci.size(); ls.ms = ms_;
      float st_ms = 0;
      if (e0 && cudaEventElapsedTime(&st_ms, c->ev[2], e0) == cudaSuccess) ls.start_ms = st_ms;
      for (int32_t l : loci) c->locus_launch[l] = (int32_t)c->launch_stats.size();
      c->launch_stats.push_back(ls);
   };
   if (c->lt[0].used) { CU(cudaEventElapsedTime(&ms, c->lt[0].e0, c->lt[0].e1)); add_stat(1, 1, 1, c->warp_list, ms, c->lt[0].e0); }
   for (int k = 0; k < 2; ++k) {
      const GridClass& g = c->grid[k];
      if (!g.lt.used) continue;
      CU(cudaEventElapsedTime(&ms, g.lt.e0, g.lt.e1));
      if (k == 0) c->stats.grid_em_ms = ms;                        // grid_em_ms: the full grid only
      add_stat(3, k == 0 ? 0 : g.n_cta, 32, g.list, ms, g.lt.e0);   // cluster_size: 0 for the full grid, the CTA count of the sub-grid
      c->launch_stats.back().variant = g.variant;
   }
   for (size_t i = 0; i < c->classes.size(); ++i) {
      LaunchTimer& t = c->lt[1 + i % N_SIDE_STREAMS];
      CU(cudaEventElapsedTime(&ms, t.e0, t.e1));
      add_stat(2, c->classes[i].cs, c->classes[i].nt, c->classes[i].loci, ms, t.e0);
   }
   c->stats.kernel_launches = launches;
   c->solved = true;
   c->downloaded = false;
   return SBQ_SUCCESS;
}

int sbq_fpkm_sum(sbq_ctx* c, double* local_sum) {
   if (!c || !local_sum) return SBQ_ERR_INVALID;
   if (c->multi) {   // the sum over ALL devices of the context (all-reduced on the devices)
      std::lock_guard<std::mutex> lk(c->mu);
      if (!c->solved) return fail(c, SBQ_ERR_STATE, "sbq_fpkm_sum before sbq_solve");
      const int rc = multi_allreduce_locked(c);
      if (!rc) *local_sum = c->multi->global_sum;
      return rc;
   }
   std::lock_guard<std::mutex> lk(c->mu);
   CU(cudaSetDevice(c->device));
   if (!c->solved) return fail(c, SBQ_ERR_STATE, "sbq_fpkm_sum before sbq_solve");
   CU(cudaMemcpyAsync(local_sum, c->d_fpkm_sum, sizeof(double), cudaMemcpyDeviceToHost, c->stream));
   CU(cudaStreamSynchronize(c->stream));
   return SBQ_SUCCESS;
}

int sbq_fpkm_sum_to_device(sbq_ctx* c, void* dev_double) {
   if (!c || !dev_double) return SBQ_ERR_INVALID;
   if (c->multi) {
      std::lock_guard<std::mutex> lk(c->mu);
      if (!c->solved) return fail(c, SBQ_ERR_STATE, "sbq_fpkm_sum_to_device before sbq_solve");
      const int rc = multi_allreduce_locked(c);
      if (rc) return rc;
      CU(cudaMemcpy(dev_double, c->multi->d_sum[0] + 1, sizeof(double), cudaMemcpyDefault));
      return SBQ_SUCCESS;
   }
   std::lock_guard<std::mutex> lk(c->mu);
   CU(cudaSetDevice(c->device));
   if (!c->solved) return fail(c, SBQ_ERR_STATE, "sbq_fpkm_sum_to_device before sbq_solve");
   CU(cudaMemcpyAsync(dev_double, c->d_fpkm_sum, sizeof(double), cudaMemcpyDeviceToDevice, c->stream));
   CU(cudaStreamSynchronize(c->stream));
   return SBQ_SUCCESS;
}

int sbq_finalize_tpm(sbq_ctx* c, double global_fpkm_sum) {
   if (!c) return SBQ_ERR_INVALID;
   if (c->multi) return multi_finalize_tpm(c, global_fpkm_sum);
   std::lock_guard<std::mutex> lk(c->mu);
   CU(cudaSetDevice(c->device));
   if (!c->solved) return fail(c, SBQ_ERR_STATE, "sbq_finalize_tpm before sbq_solve");
   const int64_t n = c->n_iso;
   tpm_kernel<<<(unsigned)((n + 255) / 256), 256, 0, c->stream>>>(c->dp.fpkm, c->d_tpm, n, global_fpkm_sum);
   CU(cudaGetLastError());
   c->stats.kernel_launches += 1;
   c->downloaded = false;
   return SBQ_SUCCESS;
}

int sbq_download(sbq_ctx* c) {
   if (!c) return SBQ_ERR_INVALID;
   if (c->multi) return multi_download(c);
   std::lock_guard<std::mutex> lk(c->mu);
   CU(cudaSetDevice(c->device));
   if (!c->solved) return fail(c, SBQ_ERR_STATE, "sbq_download before sbq_solve");
   const size_t ni = c->n_iso, nl = c->n_loci;
   bool ok = c->r_theta.reserve(ni) && c->r_fpkm.reserve(ni) && c->r_frac.reserve(ni) && c->r_tpm.reserve(ni) &&
             c->r_keep.reserve(ni) && c->r_iters.reserve(nl) && c->r_status.reserve(nl) && c->r_locus_fpkm.reserve(nl);
   if (!ok) return fail(c, SBQ_ERR_NOMEM, "pinned result buffers");
   cudaStream_t st = c->stream;
   CU(cudaEventRecord(c->ev[7], st));
   CU(cudaMemcpyAsync(c->r_theta.p, c->dp.theta, ni * 8, cudaMemcpyDeviceToHost, st));
   CU(cudaMemcpyAsync(c->r_fpkm.p, c->dp.fpkm, ni * 8, cudaMemcpyDeviceToHost, st));
   CU(cudaMemcpyAsync(c->r_frac.p, c->dp.frac, ni * 8, cudaMemcpyDeviceToHost, st));
   CU(cudaMemcpyAsync(c->r_tpm.p, c->d_tpm, ni * 8, cudaMemcpyDeviceToHost, st));
   CU(cudaMemcpyAsync(c->r_keep.p, c->dp.keep, ni * 4, cudaMemcpyDeviceToHost, st));
   CU(cudaMemcpyAsync(c->r_iters.p, c->dp.iters, nl * 4, cudaMemcpyDeviceToHost, st));
   CU(cudaMemcpyAsync(c->r_status.p, c->dp.status, nl * 4, cudaMemcpyDeviceToHost, st));
   CU(cudaMemcpyAsync(&c->r_fpkm_sum, c->d_fpkm_sum, 8, cudaMemcpyDeviceToHost, st));
   CU(cudaEventRecord(c->ev[8], st));
   CU(cudaStreamSynchronize(st));
   float ms = 0;
   CU(cudaEventElapsedTime(&ms, c->ev[7], c->ev[8]));
   c->stats.download_ms = ms;
   c->stats.d2h_bytes = (int64_t)ni * 36 + (int64_t)nl * 8 + 8;

   c->stats_stale = true;   // metric accounting (O(rows) on the host) is done lazily by sbq_get_stats
   c->downloaded = true;
   return SBQ_SUCCESS;
}

int sbq_run(sbq_ctx* c, int64_t total_mapped_reads) {
   int rc = sbq_upload_begin(c);   // the solve overlaps the tail of the copies (synchronous for multi-GPU / deferred / bias batches)
   if (rc) return rc;
   if ((rc = sbq_solve(c, total_mapped_reads))) return rc;
   if (c->multi) {   // N devices: one ncclAllReduce of the FPKM sums, TPM from the device copy of the result
      if ((rc = multi_tpm(c))) return rc;
      return sbq_download(c);
   }
   double s = 0.0;
   if ((rc = sbq_fpkm_sum(c, &s))) return rc;
   if ((rc = sbq_finalize_tpm(c, s))) return rc;
   return sbq_download(c);
}

} // extern "C" (reopened below)

// Accounting for the benchmark metric: fragments*EM-iters and algorithmic bytes (SURVEY section 8d). O(rows) on the
// host, so it is evaluated lazily by sbq_get_stats / sbq_get_launch_stats rather than inside sbq_download.
static void account(sbq_ctx* c) {
   if (!c->stats_stale || !c->downloaded) return;
   const size_t nl = (size_t)c->n_loci;
   std::vector<char> is_grid(nl, 0);
   for (int32_t l : c->grid[0].list) is_grid[l] = 1;   // grid_alg_bytes goes with grid_em_ms: the full grid only
   int64_t it_total = 0, frag_iters = 0, alg = 0, galg = 0;
   for (auto& ls : c->launch_stats) ls.nnz = ls.alg_bytes = ls.frag_iters = ls.max_iters = 0;
   for (size_t l = 0; l < nl && l < c->meta.size(); ++l) {   // shapes captured at upload: the host arrays may be gone by now
      const int64_t it = c->r_iters.p[l];
      const sbq_ctx::LocusMeta& m = c->meta[l];
      it_total += it;
      frag_iters += m.frags * it;
      const int64_t b = (12 * m.nnz + 12 * (int64_t)m.R + 16 * (int64_t)m.T) * it;
      alg += b;
      if (is_grid[l]) galg += b;
      const int32_t li = l < c->locus_launch.size() ? c->locus_launch[l] : -1;
      if (li >= 0) {
         c->launch_stats[li].nnz += m.nnz;
         c->launch_stats[li].alg_bytes += b;
         c->launch_stats[li].frag_iters += m.frags * it;
         c->launch_stats[li].max_iters = std::max<int64_t>(c->launch_stats[li].max_iters, it);
      }
   }
   c->stats.em_iters_total = it_total;
   c->stats.frag_iters = frag_iters;
   c->stats.alg_bytes = alg;
   c->stats.grid_alg_bytes = galg;
   c->stats_stale = false;
}

extern "C" {

int sbq_results(sbq_ctx* c, double* theta, double* fpkm, double* frac, double* tpm, int32_t* keep, int32_t* iters, int32_t* status) {
   if (!c) return SBQ_ERR_INVALID;
   std::lock_guard<std::mutex> lk(c->mu);
   if (!c->downloaded) return fail(c, SBQ_ERR_STATE, "sbq_results before sbq_download / sbq_run");
   const size_t ni = c->n_iso, nl = c->n_loci;
   if (theta) memcpy(theta, c->r_theta.p, ni * 8);
   if (fpkm) memcpy(fpkm, c->r_fpkm.p, ni * 8);
   if (frac) memcpy(frac, c->r_frac.p, ni * 8);
   if (tpm) memcpy(tpm, c->r_tpm.p, ni * 8);
   if (keep) memcpy(keep, c->r_keep.p, ni * 4);
   if (iters) memcpy(iters, c->r_iters.p, nl * 4);
   if (status) memcpy(status, c->r_status.p, nl * 4);
   return SBQ_SUCCESS;
}

int sbq_get_stats(const sbq_ctx* cc, sbq_stats* out) {
   if (!cc || !out) return SBQ_ERR_INVALID;
   sbq_ctx* c = const_cast<sbq_ctx*>(cc);
   std::lock_guard<std::mutex> lk(c->mu);
   if (c->multi) {
      multi_stats(c, out);
      return SBQ_SUCCESS;
   }
   account(c);
   *out = c->stats;
   return SBQ_SUCCESS;
}

int sbq_set_insert_model(sbq_ctx* c, const sbq_insert_model* model, int32_t read_len) {
   if (!c || !model || read_len < 1) return SBQ_ERR_INVALID;
   std::lock_guard<std::mutex> lk(c->mu);
   c->model = *model;
   c->model_emp.clear();
   if (model->use_emp) {
      if (!model->emp_dist || model->end_offset < model->start_offset) return fail(c, SBQ_ERR_INVALID, "bad empirical insert model");
      c->model_emp.assign(model->emp_dist, model->emp_dist + (model->end_offset - model->start_offset + 1));
   }
   c->model.emp_dist = nullptr;
   c->model_read_len = read_len;
   c->have_model = true;
   c->resident = c->solved = c->downloaded = false;
   return SBQ_SUCCESS;
}

int sbq_set_raw_mass_mode(sbq_ctx* c, int32_t mode) {
   if (!c || (mode != SBQ_RAW_MASS_HALVES && mode != SBQ_RAW_MASS_ANY)) return SBQ_ERR_INVALID;
   std::lock_guard<std::mutex> lk(c->mu);
   c->raw_mass_mode = mode;
   c->resident = c->solved = c->downloaded = false;
   return SBQ_SUCCESS;
}

int sbq_submit_deferred(sbq_ctx* c, const sbq_table* const* tables, int64_t n_tables) {
   if (!c || (!tables && n_tables > 0) || n_tables < 0) return SBQ_ERR_INVALID;
   for (int64_t t = 0; t < n_tables; ++t) {
      sbq_locus L;
      sbq_weight_desc d;
      if (!tables[t] || sbq_table_locus(tables[t], &L) || sbq_table_weight_desc(tables[t], &d)) return SBQ_ERR_INVALID;
      const int64_t nnz = L.row_ptr[L.n_row] - L.row_ptr[0];
      // descriptors and CSR of one table are appended under ONE lock, so concurrent submits cannot interleave them
      std::lock_guard<std::mutex> lk(c->mu);
      if (d.n_entry != nnz) return fail(c, SBQ_ERR_INVALID, "table %lld was not built with defer_weights = 1", (long long)t);
      if (c->deferred == 2) return fail(c, SBQ_ERR_STATE, "a batch is either all deferred-weight or all host-weighted");
      cudaSetDevice(c->device);
      const StagingMark mark(c);
      const int64_t pool_base = (int64_t)c->h_wpool.n;
      const bool ok = c->h_wseg.reserve(c->h_wseg.n + nnz) && c->h_wn.append(d.n_seg, nnz) && c->h_wmask.append(d.implicit_mask, nnz) &&
                      c->h_wlen.append(d.iso_len, nnz) && c->h_wpool.append(d.pool, d.n_pool) && c->h_wpool_off.append(&pool_base, 1);
      if (!ok) {
         mark.restore(c);
         return fail(c, SBQ_ERR_NOMEM, "pinned staging");
      }
      for (int64_t k = 0; k < nnz; ++k) c->h_wseg.p[c->h_wseg.n++] = d.seg_ptr[k] < 0 ? -1 : d.seg_ptr[k] + pool_base;
      const int rc = submit_locked(c, &L, 1);
      if (rc) {
         mark.restore(c);   // the descriptors go with the locus that was refused
         return rc;
      }
      c->deferred = 1;
   }
   return SBQ_SUCCESS;
}

// ---- raw loci: fragment-class assignment on the device (sbq_rawbuild.cuh) ---------------------------------------------
int sbq_submit_raw(sbq_ctx* c, const sbq_locus_input* in, int64_t* locus_index) {
   if (!c || !in || in->n_iso < 1 || in->n_hit < 0 || !in->iso_feat_ptr || (in->n_hit > 0 && (!in->hit_feat_ptr || !in->hit_mass))) return SBQ_ERR_INVALID;
   if (c->cfg.bias_mode) return fail(c, SBQ_ERR_UNSUPPORTED, "raw loci carry no covariates");
   if (c->multi) return multi_submit_raw(c, in, locus_index);
   if (in->n_iso > SBQ_MAX_ISO) return fail(c, SBQ_ERR_UNSUPPORTED, "%d isoforms > SBQ_MAX_ISO", in->n_iso);
   // static part of the class table on the host (cheap, O(exons + T S)): disjoint exon segments, isoform segment lists, lengths
   sbq_locus_input st = *in;
   st.n_hit = 0;
   st.defer_weights = 1;
   sbq_table* tb = nullptr;
   sbq_insert_model dummy{0, 0, 0, nullptr, 0, 200.0, 20.0};
   int rc = sbq_build_locus(&st, &dummy, &tb);
   if (rc) return fail(c, rc, "sbq_build_locus (static part) failed");
   sbq_table_dims d;
   sbq_table_get_dims(tb, &d);
   sbq_locus L;
   sbq_table_locus(tb, &L);
   std::lock_guard<std::mutex> lk(c->mu);
   if (c->host_released || (c->n_loci > 0 && !c->raw_mode)) { sbq_table_free(tb); return fail(c, SBQ_ERR_STATE, "a batch is either all raw loci or none"); }
   if (c->n_loci > 0 && c->raw.long_read != (in->long_read ? 1 : 0)) { sbq_table_free(tb); return fail(c, SBQ_ERR_STATE, "long_read must be the same for every raw locus of a batch"); }
   if (d.n_seg > 65535) { sbq_table_free(tb); return fail(c, SBQ_ERR_UNSUPPORTED, "more than 65535 exon segments in one locus"); }
   auto& r = c->raw;
   r.long_read = in->long_read ? 1 : 0;
   const int32_t locus = (int32_t)c->n_loci;
   std::vector<uint32_t> sl(d.n_seg), sr(d.n_seg);
   std::vector<int32_t> isp(d.n_iso + 1), isg;
   sbq_table_segments(tb, sl.data(), sr.data());
   sbq_table_iso_segments(tb, isp.data(), nullptr);
   isg.resize(isp[d.n_iso]);
   sbq_table_iso_segments(tb, nullptr, isg.data());
   r.seg_left.insert(r.seg_left.end(), sl.begin(), sl.end());
   r.seg_right.insert(r.seg_right.end(), sr.begin(), sr.end());
   r.loc_seg_off.push_back((int64_t)r.seg_left.size());
   const int64_t seg_base = (int64_t)r.iso_seg.size();
   r.iso_seg.insert(r.iso_seg.end(), isg.begin(), isg.end());
   for (int t = 1; t <= d.n_iso; ++t) r.iso_seg_ptr.push_back(seg_base + isp[t]);
   const int64_t if_base = (int64_t)r.if_off.size();
   const int nif = in->iso_feat_ptr[in->n_iso];
   r.if_off.insert(r.if_off.end(), in->iso_feat_off, in->iso_feat_off + nif);
   r.if_len.insert(r.if_len.end(), in->iso_feat_len, in->iso_feat_len + nif);
   r.if_code.insert(r.if_code.end(), in->iso_feat_code, in->iso_feat_code + nif);
   for (int t = 1; t <= in->n_iso; ++t) r.iso_feat_ptr.push_back(if_base + in->iso_feat_ptr[t]);
   const int64_t hf_base = (int64_t)r.hf_off.size();
   const int nhf = in->n_hit > 0 ? in->hit_feat_ptr[in->n_hit] : 0;
   if (nhf) {
      r.hf_off.insert(r.hf_off.end(), in->hit_feat_off, in->hit_feat_off + nhf);
      r.hf_len.insert(r.hf_len.end(), in->hit_feat_len, in->hit_feat_len + nhf);
      r.hf_code.insert(r.hf_code.end(), in->hit_feat_code, in->hit_feat_code + nhf);
   }
   for (int h = 0; h < in->n_hit; ++h) {
      r.hit_feat_ptr.push_back(hf_base + in->hit_feat_ptr[h + 1]);
      r.hit_locus.push_back(locus);
      r.hit_mass.push_back((float)in->hit_mass[h]);
      r.hit_ref.push_back(in->hit_ref_id ? in->hit_ref_id[h] : 0);
   }
   r.loc_hit_off.push_back((int64_t)r.hit_locus.size());
   cudaSetDevice(c->device);
   if ((rc = ensure_origin(c))) { sbq_table_free(tb); return rc; }
   c->n_iso += d.n_iso;
   c->n_loci += 1;
   bool ok = c->h_loc_iso_off.append(&c->n_iso, 1) && c->h_iso_len.append(L.iso_len, d.n_iso);
   sbq_table_free(tb);
   if (!ok) return fail(c, SBQ_ERR_NOMEM, "pinned staging");
   c->raw_mode = true;
   c->deferred = 1;
   c->resident = c->solved = c->downloaded = false;
   if (locus_index) *locus_index = locus;
   return SBQ_SUCCESS;
}

} // extern "C" (reopened below)

namespace {
int rb_scan(cudaStream_t st, const int32_t* v, int64_t n, long long* block_tmp, int64_t* out) {
   const int nb = (int)((n + RB_SCAN_BLOCK - 1) / RB_SCAN_BLOCK);
   if (n == 0) return cudaMemsetAsync(out, 0, 8, st) == cudaSuccess ? 0 : -3;
   rb_scan_sums_kernel<<<nb, 1024, 0, st>>>(v, n, block_tmp);
   synth_scan_blocks_kernel<<<1, 1024, 0, st>>>(block_tmp, nb);
   rb_scan_fill_kernel<<<nb, 1024, 0, st>>>(v, n, block_tmp, out);
   return cudaGetLastError() == cudaSuccess ? 0 : -3;
}
}  // namespace

// Upload of a raw batch: feature lists to the device, class assignment there, CSR + weight descriptors + alpha on the device.
static int raw_upload(sbq_ctx* c) {
   CU(cudaSetDevice(c->device));
   if (!c->have_model && !c->raw.long_read) return fail(c, SBQ_ERR_STATE, "raw loci need sbq_set_insert_model()");
   c->boot.prefix_ready = c->boot.done = c->gibbs.done = false;
   auto& r = c->raw;
   const int64_t L = c->n_loci, H = (int64_t)r.hit_locus.size(), T = c->n_iso, S = (int64_t)r.seg_left.size();
   const int64_t* lio = c->h_loc_iso_off.p;
   std::vector<int64_t> cm_off(L + 1, 0), tab_off(L + 1, 0);
   for (int64_t l = 0; l < L; ++l) {
      const int64_t Hl = r.loc_hit_off[l + 1] - r.loc_hit_off[l], W = (lio[l + 1] - lio[l] + 31) / 32;
      cm_off[l + 1] = cm_off[l] + Hl * W;
      int64_t cap = 8;
      while (cap < 2 * Hl) cap <<= 1;
      tab_off[l + 1] = tab_off[l] + cap;
   }
   const int64_t CM = cm_off[L], TAB = tab_off[L];
   const int n_scan = (int)((std::max<int64_t>(H, 1) + RB_SCAN_BLOCK - 1) / RB_SCAN_BLOCK);
   // ---- carve inputs + workspace
   size_t need = 0;
   auto sz = [&](size_t bytes) { const size_t o = need; need += align_up(bytes + 16); return o; };
   const size_t o_hl = sz(H * 4), o_hfp = sz((H + 1) * 8), o_hfo = sz(r.hf_off.size() * 4), o_hfl = sz(r.hf_len.size() * 4), o_hfc = sz(r.hf_code.size());
   const size_t o_hm = sz(H * 4), o_hr = sz(H * 4), o_lho = sz((L + 1) * 8), o_lio = sz((L + 1) * 8), o_lso = sz((L + 1) * 8);
   const size_t o_ifp = sz((T + 1) * 8), o_ifo = sz(r.if_off.size() * 4), o_ifl = sz(r.if_len.size() * 4), o_ifc = sz(r.if_code.size());
   const size_t o_sl = sz(S * 4), o_sr = sz(S * 4), o_isp = sz((T + 1) * 8), o_isg = sz(r.iso_seg.size() * 4), o_il = sz(T * 4);
   const size_t o_nc = sz(H * 4), o_co = sz((H + 1) * 8), o_va = sz(H), o_ch = sz(H * 8), o_fh = sz(H * 8), o_cmo = sz((L + 1) * 8), o_cm = sz(CM * 4);
   const size_t o_to = sz((L + 1) * 8), o_k1 = sz(TAB * 8), o_m1 = sz(TAB * 4), o_s1 = sz(H * 4), o_k2 = sz(TAB * 8), o_m2 = sz(TAB * 4), o_s2 = sz(H * 4);
   const size_t o_ir = sz(H * 4), o_cp = sz((H + 1) * 8), o_hc = sz(H * 4), o_fl = sz(64), o_bs = sz((size_t)n_scan * 8 + 8), o_g = sz((L + 1) * 8);
   if (!c->d_raw.reserve(need)) return fail(c, SBQ_ERR_NOMEM, "device allocation failed (raw batch, %zu MB)", need >> 20);
   char* base = (char*)c->d_raw.p;
   cudaStream_t st = c->stream;
   CU(cudaEventRecord(c->ev[0], st));
   auto up = [&](size_t off, const void* src, size_t bytes) -> int {
      if (bytes) CU(cudaMemcpyAsync(base + off, src, bytes, cudaMemcpyHostToDevice, st));
      return 0;
   };
   int rc = 0;
   rc |= up(o_hl, r.hit_locus.data(), H * 4); rc |= up(o_hfp, r.hit_feat_ptr.data(), (H + 1) * 8); rc |= up(o_hfo, r.hf_off.data(), r.hf_off.size() * 4);
   rc |= up(o_hfl, r.hf_len.data(), r.hf_len.size() * 4); rc |= up(o_hfc, r.hf_code.data(), r.hf_code.size()); rc |= up(o_hm, r.hit_mass.data(), H * 4);
   rc |= up(o_hr, r.hit_ref.data(), H * 4); rc |= up(o_lho, r.loc_hit_off.data(), (L + 1) * 8); rc |= up(o_lio, lio, (L + 1) * 8);
   rc |= up(o_lso, r.loc_seg_off.data(), (L + 1) * 8); rc |= up(o_ifp, r.iso_feat_ptr.data(), (T + 1) * 8); rc |= up(o_ifo, r.if_off.data(), r.if_off.size() * 4);
   rc |= up(o_ifl, r.if_len.data(), r.if_len.size() * 4); rc |= up(o_ifc, r.if_code.data(), r.if_code.size()); rc |= up(o_sl, r.seg_left.data(), S * 4);
   rc |= up(o_sr, r.seg_right.data(), S * 4); rc |= up(o_isp, r.iso_seg_ptr.data(), (T + 1) * 8); rc |= up(o_isg, r.iso_seg.data(), r.iso_seg.size() * 4);
   rc |= up(o_il, c->h_iso_len.p, T * 4); rc |= up(o_cmo, cm_off.data(), (L + 1) * 8); rc |= up(o_to, tab_off.data(), (L + 1) * 8);
   if (rc) return SBQ_ERR_CUDA;
   RawBatch& b = c->rb;
   b = RawBatch{};
   b.n_hit = H; b.n_loci = (int32_t)L; b.long_read = r.long_read;
   const bool ordered = c->raw_mass_mode == SBQ_RAW_MASS_ANY;
   b.mass_mode = ordered ? RB_MASS_ANY : RB_MASS_HALVES;
   b.hit_locus = (const int32_t*)(base + o_hl); b.hit_feat_ptr = (const int64_t*)(base + o_hfp); b.hf_off = (const uint32_t*)(base + o_hfo);
   b.hf_len = (const uint32_t*)(base + o_hfl); b.hf_code = (const uint8_t*)(base + o_hfc); b.hit_mass = (const float*)(base + o_hm);
   b.hit_ref = (const int32_t*)(base + o_hr); b.loc_hit_off = (const int64_t*)(base + o_lho); b.loc_iso_off = (const int64_t*)(base + o_lio);
   b.loc_seg_off = (const int64_t*)(base + o_lso); b.iso_feat_ptr = (const int64_t*)(base + o_ifp); b.if_off = (const uint32_t*)(base + o_ifo);
   b.if_len = (const uint32_t*)(base + o_ifl); b.if_code = (const uint8_t*)(base + o_ifc); b.seg_left = (const uint32_t*)(base + o_sl);
   b.seg_right = (const uint32_t*)(base + o_sr); b.iso_seg_ptr = (const int64_t*)(base + o_isp); b.iso_seg = (const int32_t*)(base + o_isg);
   b.iso_len = (const int32_t*)(base + o_il);
   b.ncoord = (int32_t*)(base + o_nc); b.coord_off = (int64_t*)(base + o_co); b.valid = (uint8_t*)(base + o_va); b.chash = (unsigned long long*)(base + o_ch);
   b.fhash = (unsigned long long*)(base + o_fh); b.loc_cm_off = (const int64_t*)(base + o_cmo); b.cm = (uint32_t*)(base + o_cm);
   b.loc_tab_off = (const int64_t*)(base + o_to); b.keys1 = (unsigned long long*)(base + o_k1); b.min1 = (uint32_t*)(base + o_m1); b.slot1 = (uint32_t*)(base + o_s1);
   b.keys2 = (unsigned long long*)(base + o_k2); b.min2 = (uint32_t*)(base + o_m2); b.slot2 = (uint32_t*)(base + o_s2);
   b.is_rep = (int32_t*)(base + o_ir); b.cls_prefix = (int64_t*)(base + o_cp); b.hit_class = (int32_t*)(base + o_hc); b.flags = (int*)(base + o_fl);
   long long* d_bs = (long long*)(base + o_bs);
   int64_t* d_gather = (int64_t*)(base + o_g);
   CU(cudaMemsetAsync(base + o_k1, 0xff, TAB * 8, st));
   CU(cudaMemsetAsync(base + o_m1, 0xff, TAB * 4, st));
   CU(cudaMemsetAsync(base + o_k2, 0xff, TAB * 8, st));
   CU(cudaMemsetAsync(base + o_m2, 0xff, TAB * 4, st));
   CU(cudaMemsetAsync(b.flags, 0, 64, st));
   const int nbk = std::max(1, std::min<int>((int)((H + 127) / 128), c->prop.multiProcessorCount * 16));
   auto check_flags = [&](const char* where) -> int {
      int f = 0;
      CU(cudaMemcpyAsync(&f, b.flags, sizeof f, cudaMemcpyDeviceToHost, st));
      CU(cudaStreamSynchronize(st));
      if (f) return fail(c, SBQ_ERR_UNSUPPORTED, "device class assignment refused the batch (%s, mass mode %s):%s%s%s - use the host builder (sbq_build_locus) for it", where,
                         ordered ? "SBQ_RAW_MASS_ANY" : "SBQ_RAW_MASS_HALVES", f & RB_FLAG_COLLISION ? " 64-bit hash collision;" : "",
                         !(f & RB_FLAG_MASS) ? ""
                         : ordered ? " a fragment mass is NaN, infinite or negative (or a class holds >= 2^31, where (int) is undefined);"
                                   : " fragment masses are not multiples of 1/2 (or a class holds >= 2^23): the float sum would depend on the set order (SBQ_RAW_MASS_ANY sums in set order);",
                         f & RB_FLAG_NSEG ? " a class coordinate lies outside the isoform's segments (the reference asserts);" : "");
      return 0;
   };
   if (H) {
      raw_hit_kernel<<<nbk, 128, 0, st>>>(b);
      raw_class_insert_kernel<<<nbk, 256, 0, st>>>(b);
      raw_class_rep_kernel<<<nbk, 256, 0, st>>>(b);
      CU(cudaGetLastError());
   }
   if (rb_scan(st, b.is_rep, H, d_bs, b.cls_prefix)) return fail(c, SBQ_ERR_CUDA, "scan failed");
   if (rb_scan(st, b.ncoord, H, d_bs, b.coord_off)) return fail(c, SBQ_ERR_CUDA, "scan failed");
   // ---- round trip 1: classes per locus, length of the coordinate pool
   rb_gather_kernel<<<(unsigned)((L + 1 + 255) / 256), 256, 0, st>>>(b.cls_prefix, b.loc_hit_off, L + 1, d_gather);
   std::vector<int64_t> cls_off(L + 1);
   CU(cudaMemcpyAsync(cls_off.data(), d_gather, (L + 1) * 8, cudaMemcpyDeviceToHost, st));
   CU(cudaMemcpyAsync(&b.n_coord, b.coord_off + H, 8, cudaMemcpyDeviceToHost, st));
   if ((rc = check_flags("hits"))) return rc;
   const int64_t R = cls_off[L];
   std::vector<int64_t> cmask_off(L + 1, 0);
   std::vector<int32_t> class_locus((size_t)R);
   for (int64_t l = 0; l < L; ++l) {
      const int64_t W = (lio[l + 1] - lio[l] + 31) / 32;
      cmask_off[l + 1] = cmask_off[l] + (cls_off[l + 1] - cls_off[l]) * W;
      for (int64_t x = cls_off[l]; x < cls_off[l + 1]; ++x) class_locus[x] = (int32_t)l;
   }
   size_t need2 = 0;
   auto sz2 = [&](size_t bytes) { const size_t o = need2; need2 += align_up(bytes + 16); return o; };
   const int n_scan2 = (int)((std::max<int64_t>(R, 1) + RB_SCAN_BLOCK - 1) / RB_SCAN_BLOCK);
   const size_t p_co = sz2((L + 1) * 8), p_mo = sz2((L + 1) * 8), p_cl = sz2(R * 4), p_rep = sz2(R * 8), p_ms = sz2(R * 4), p_nf = sz2(R * 4), p_cmk = sz2(cmask_off[L] * 4),
                p_nz = sz2(R * 4), p_rp = sz2((R + 1) * 8), p_bs = sz2((size_t)n_scan2 * 8 + 8), p_g = sz2((L + 1) * 8), p_hc = sz2(b.n_coord * 2),
                p_ns = sz2(R * 4), p_po = sz2((R + 1) * 8);
   // set-order mass sum: member offsets, per-class cursors, the survivors (at most H) as (class, prefix, hit) twice (merge ping-pong)
   const int64_t HM = ordered ? H : 0;
   const size_t p_mof = sz2(ordered ? (R + 1) * 8 : 0), p_cur = sz2(ordered ? R * 4 : 0), p_sk0 = sz2(HM * 8), p_sk1 = sz2(HM * 8), p_sh = sz2(HM * 8),
                p_tk0 = sz2(HM * 8), p_tk1 = sz2(HM * 8), p_th = sz2(HM * 8);
   if (!c->d_raw2.reserve(need2)) return fail(c, SBQ_ERR_NOMEM, "device allocation failed (class arrays)");
   char* base2 = (char*)c->d_raw2.p;
   CU(cudaMemcpyAsync(base2 + p_co, cls_off.data(), (L + 1) * 8, cudaMemcpyHostToDevice, st));
   CU(cudaMemcpyAsync(base2 + p_mo, cmask_off.data(), (L + 1) * 8, cudaMemcpyHostToDevice, st));
   if (R) CU(cudaMemcpyAsync(base2 + p_cl, class_locus.data(), R * 4, cudaMemcpyHostToDevice, st));
   CU(cudaMemsetAsync(base2 + p_ms, 0, align_up(R * 4 + 16), st));
   CU(cudaMemsetAsync(base2 + p_nf, 0, align_up(R * 4 + 16), st));
   CU(cudaMemsetAsync(base2 + p_cmk, 0, align_up(cmask_off[L] * 4 + 16), st));
   b.loc_cls_off = (const int64_t*)(base2 + p_co); b.loc_cmask_off = (const int64_t*)(base2 + p_mo); b.class_rep = (int64_t*)(base2 + p_rep);
   b.class_mass = (float*)(base2 + p_ms); b.class_nfrag = (int32_t*)(base2 + p_nf); b.cmask = (uint32_t*)(base2 + p_cmk); b.class_nnz = (int32_t*)(base2 + p_nz);
   b.coords = (uint16_t*)(base2 + p_hc); b.class_nseg = (int32_t*)(base2 + p_ns);
   int64_t* d_pool_off = (int64_t*)(base2 + p_po);
   const int32_t* d_class_locus = (const int32_t*)(base2 + p_cl);
   int64_t* d_rp_tmp = (int64_t*)(base2 + p_rp);
   const int nbc = std::max(1, std::min<int>((int)((R + 127) / 128), c->prop.multiProcessorCount * 16));
   if (H) {
      raw_coord_kernel<<<nbk, 128, 0, st>>>(b);
      raw_member_kernel<<<nbk, 256, 0, st>>>(b);
      raw_mass_kernel<<<nbk, 256, 0, st>>>(b);
   }
   if (ordered && R) {   // class masses in set order (SBQ_RAW_MASS_ANY); the number of survivors stays on the device (member_off[R])
      int64_t* d_mof = (int64_t*)(base2 + p_mof);
      unsigned long long *k0 = (unsigned long long*)(base2 + p_sk0), *k1 = (unsigned long long*)(base2 + p_sk1);
      unsigned long long *t0 = (unsigned long long*)(base2 + p_tk0), *t1 = (unsigned long long*)(base2 + p_tk1);
      int64_t *hh = (int64_t*)(base2 + p_sh), *th = (int64_t*)(base2 + p_th);
      if (rb_scan(st, b.class_nfrag, R, (long long*)(base2 + p_bs), d_mof)) return fail(c, SBQ_ERR_CUDA, "scan failed");
      CU(cudaMemsetAsync(base2 + p_cur, 0, R * 4, st));
      raw_member_scatter_kernel<<<nbk, 256, 0, st>>>(b, d_mof, (int32_t*)(base2 + p_cur), k0, k1, hh);
      raw_member_tile_sort_kernel<<<(unsigned)((H + RB_SORT_TILE - 1) / RB_SORT_TILE), RB_SORT_TILE / 2, 0, st>>>(b, d_mof + R, k0, k1, hh);
      const int nbm = std::max(1, std::min<int>((int)((H + 256 * RB_MERGE_PER_THREAD - 1) / (256 * RB_MERGE_PER_THREAD)), c->prop.multiProcessorCount * 16));
      for (int64_t w = RB_SORT_TILE; w < H; w *= 2) {   // H bounds the survivors: a pass whose runs already cover them all is a copy
         raw_member_merge_kernel<<<nbm, 256, 0, st>>>(b, d_mof + R, w, k0, k1, hh, t0, t1, th);
         std::swap(k0, t0); std::swap(k1, t1); std::swap(hh, th);
      }
      raw_member_sum_kernel<<<nbc, 256, 0, st>>>(b, R, d_mof, hh);
   }
   if (R) raw_nnz_kernel<<<nbc, 256, 0, st>>>(b, R, d_class_locus);
   CU(cudaGetLastError());
   if (rb_scan(st, b.class_nnz, R, (long long*)(base2 + p_bs), d_rp_tmp)) return fail(c, SBQ_ERR_CUDA, "scan failed");
   if (rb_scan(st, b.class_nseg, R, (long long*)(base2 + p_bs), d_pool_off)) return fail(c, SBQ_ERR_CUDA, "scan failed");
   // ---- round trip 2: non-zeros per locus, length of the descriptor pool
   rb_gather_kernel<<<(unsigned)((L + 1 + 255) / 256), 256, 0, st>>>(d_rp_tmp, b.loc_cls_off, L + 1, (int64_t*)(base2 + p_g));
   std::vector<int64_t> nz_off(L + 1);
   int64_t n_pool = 0;
   CU(cudaMemcpyAsync(nz_off.data(), base2 + p_g, (L + 1) * 8, cudaMemcpyDeviceToHost, st));
   CU(cudaMemcpyAsync(&n_pool, d_pool_off + R, 8, cudaMemcpyDeviceToHost, st));
   if ((rc = check_flags("classes"))) return rc;
   c->n_row = R;
   c->nnz = nz_off[L];
   if ((rc = alloc_device(c))) return rc;
   DevParams& dp = c->dp;
   CU(cudaMemcpyAsync(const_cast<int64_t*>(dp.loc_row_off), cls_off.data(), (L + 1) * 8, cudaMemcpyHostToDevice, st));
   CU(cudaMemcpyAsync(const_cast<int64_t*>(dp.loc_iso_off), lio, (L + 1) * 8, cudaMemcpyHostToDevice, st));
   CU(cudaMemcpyAsync(const_cast<int64_t*>(dp.row_ptr), d_rp_tmp, (R + 1) * 8, cudaMemcpyDeviceToDevice, st));
   CU(cudaMemcpyAsync(const_cast<int32_t*>(dp.iso_len), c->h_iso_len.p, T * 4, cudaMemcpyHostToDevice, st));
   // ---- CSR rows, counts, weight descriptors; alpha by weights_kernel (the same kernel the deferred host tables use)
   const int64_t nnz = c->nnz;
   const size_t b_seg = align_up(nnz * 8 + 8), b_n = align_up(nnz * 2 + 8), b_m = align_up(nnz * 4 + 8), b_l = align_up(nnz * 4 + 8), b_pool = align_up((size_t)n_pool * 4 + 8),
                b_emp = align_up(c->model_emp.size() * 8 + 8);
   if (!c->d_weights.reserve(b_seg + b_n + b_m + b_l + b_pool + b_emp)) return fail(c, SBQ_ERR_NOMEM, "device allocation failed (weight descriptors)");
   char* q = (char*)c->d_weights.p;
   int64_t* d_seg = (int64_t*)q; q += b_seg;
   uint16_t* d_n = (uint16_t*)q; q += b_n;
   uint32_t* d_m = (uint32_t*)q; q += b_m;
   int32_t* d_l = (int32_t*)q; q += b_l;
   uint32_t* d_pool = (uint32_t*)q; q += b_pool;
   double* d_emp = (double*)q;
   if (R) raw_fill_kernel<<<nbc, 128, 0, st>>>(b, R, d_class_locus, dp.row_ptr, d_pool_off, const_cast<int32_t*>(dp.col), const_cast<double*>(dp.alpha),
                                               const_cast<int32_t*>(dp.count), d_seg, d_n, d_m, d_l, d_pool);
   CU(cudaGetLastError());
   if ((rc = check_flags("weights"))) return rc;
   CU(cudaEventRecord(c->ev[5], st));
   if (!r.long_read && nnz) {
      if (!c->model_emp.empty()) CU(cudaMemcpyAsync(d_emp, c->model_emp.data(), c->model_emp.size() * 8, cudaMemcpyHostToDevice, st));
      WeightModel wm{c->model.use_emp, c->model.start_offset, c->model.end_offset, c->model.total_reads, d_emp, c->model.mean, c->model.sd, c->model_read_len};
      const int blocks = std::max(1, std::min<int>((int)((nnz + 7) / 8), c->prop.multiProcessorCount * 16));
      weights_kernel<uint16_t><<<blocks, 256, 0, st>>>(nnz, d_seg, d_n, d_m, d_l, d_pool, wm, const_cast<double*>(dp.alpha));
      CU(cudaGetLastError());
   }
   CU(cudaEventRecord(c->ev[6], st));
   // fragment totals, plan, work lists
   if (!c->r_frags.reserve((size_t)L) || !c->d_frags.reserve(align_up((size_t)L * 8))) return fail(c, SBQ_ERR_NOMEM, "fragment-total buffers");
   locus_frags_kernel<<<std::max(1, std::min<int>((int)((L + 7) / 8), c->prop.multiProcessorCount * 8)), 256, 0, st>>>(dp.loc_row_off, dp.count, L, (long long*)c->d_frags.p);
   CU(cudaMemcpyAsync(c->r_frags.p, c->d_frags.p, (size_t)L * 8, cudaMemcpyDeviceToHost, st));
   CU(cudaStreamSynchronize(st));
   c->meta.resize((size_t)L);
   for (int64_t l = 0; l < L; ++l) c->meta[l] = {nz_off[l + 1] - nz_off[l], c->r_frags.p[l], (int32_t)(cls_off[l + 1] - cls_off[l]), (int32_t)(lio[l + 1] - lio[l])};
   if ((rc = plan(c))) return rc;
   if (c->h_lists.n) CU(cudaMemcpyAsync(c->d_lists_p, c->h_lists.p, c->h_lists.n * sizeof(int32_t), cudaMemcpyHostToDevice, st));
   if (!c->classes.empty()) {
      if (!c->d_csc.reserve(align_up(c->nnz * 4 + 16))) return fail(c, SBQ_ERR_NOMEM, "device allocation failed (transposed-index scratch)");
      dp.csc = (unsigned*)c->d_csc.p;
   }
   CU(cudaEventRecord(c->ev[1], st));
   CU(cudaStreamSynchronize(st));
   float ms = 0;
   CU(cudaEventElapsedTime(&ms, c->ev[0], c->ev[1]));
   c->stats.upload_ms = ms;
   CU(cudaEventElapsedTime(&ms, c->ev[5], c->ev[6]));
   c->stats.weights_ms = ms;
   c->weights_ms = ms;
   c->stats.h2d_bytes = (int64_t)(H * 20 + r.hf_off.size() * 9 + r.if_off.size() * 9 + S * 8 + r.iso_seg.size() * 4 + T * 20 + L * 40);
   c->stats.n_loci = c->n_loci; c->stats.n_row = c->n_row; c->stats.n_iso = c->n_iso; c->stats.nnz = c->nnz;
   c->resident = true;
   c->col16_ready = false;
   c->solved = c->downloaded = false;
   return SBQ_SUCCESS;
}

extern "C" {

// Tests: the device-built class table of the last raw upload. hit_class[n_hit] (local class id or -1), hit_ncoord[n_hit] and
// hit_coords[n_hit][16] (segment indices a hit touches: the first 16 of them, zeros after the last; the count saturates at 255 -
// sbq_fetch_raw_coords has the full lists), class_rep[n_row] (representative hit, batch-wide index), class_mass[n_row],
// class_nfrag[n_row]; the CSR itself comes from sbq_fetch_batch. Any pointer may be NULL.
int sbq_fetch_raw_classes(sbq_ctx* c, int32_t* hit_class, uint8_t* hit_ncoord, uint16_t* hit_coords, int64_t* class_rep, float* class_mass, int32_t* class_nfrag) {
   if (!c) return SBQ_ERR_INVALID;
   std::lock_guard<std::mutex> lk(c->mu);
   if (c->multi) return fail(c, SBQ_ERR_UNSUPPORTED, "sbq_fetch_raw_classes is single-device (a test aid)");
   CU(cudaSetDevice(c->device));
   if (!c->resident || !c->raw_mode) return fail(c, SBQ_ERR_STATE, "sbq_fetch_raw_classes needs an uploaded raw batch");
   const RawBatch& b = c->rb;
   cudaStream_t st = c->stream;
   std::vector<int64_t> off;
   std::vector<uint16_t> pool;
   if ((hit_ncoord || hit_coords) && b.n_hit) {
      off.resize(b.n_hit + 1);
      pool.resize(b.n_coord);
      CU(cudaMemcpyAsync(off.data(), b.coord_off, (b.n_hit + 1) * 8, cudaMemcpyDeviceToHost, st));
      if (b.n_coord) CU(cudaMemcpyAsync(pool.data(), b.coords, b.n_coord * 2, cudaMemcpyDeviceToHost, st));
   }
   if (hit_class && b.n_hit) CU(cudaMemcpyAsync(hit_class, b.hit_class, b.n_hit * 4, cudaMemcpyDeviceToHost, st));
   if (class_rep && c->n_row) CU(cudaMemcpyAsync(class_rep, b.class_rep, c->n_row * 8, cudaMemcpyDeviceToHost, st));
   if (class_mass && c->n_row) CU(cudaMemcpyAsync(class_mass, b.class_mass, c->n_row * 4, cudaMemcpyDeviceToHost, st));
   if (class_nfrag && c->n_row) CU(cudaMemcpyAsync(class_nfrag, b.class_nfrag, c->n_row * 4, cudaMemcpyDeviceToHost, st));
   CU(cudaStreamSynchronize(st));
   for (int64_t h = 0; h < (int64_t)off.size() - 1; ++h) {
      const int64_t n = off[h + 1] - off[h];
      if (hit_ncoord) hit_ncoord[h] = (uint8_t)std::min<int64_t>(n, 255);
      if (hit_coords)
         for (int64_t i = 0; i < 16; ++i) hit_coords[h * 16 + i] = i < n ? pool[off[h] + i] : 0;
   }
   return SBQ_SUCCESS;
}

// Tests: the full coordinate lists of the last raw upload. Hit h touches segments hit_coords[hit_coord_off[h] .. hit_coord_off[h + 1]);
// hit_coord_off[n_hit] is the length of hit_coords. Either pointer may be NULL.
int sbq_fetch_raw_coords(sbq_ctx* c, int64_t* hit_coord_off, uint16_t* hit_coords) {
   if (!c) return SBQ_ERR_INVALID;
   std::lock_guard<std::mutex> lk(c->mu);
   if (c->multi) return fail(c, SBQ_ERR_UNSUPPORTED, "sbq_fetch_raw_coords is single-device (a test aid)");
   CU(cudaSetDevice(c->device));
   if (!c->resident || !c->raw_mode) return fail(c, SBQ_ERR_STATE, "sbq_fetch_raw_coords needs an uploaded raw batch");
   const RawBatch& b = c->rb;
   cudaStream_t st = c->stream;
   if (hit_coord_off) CU(cudaMemcpyAsync(hit_coord_off, b.coord_off, (b.n_hit + 1) * 8, cudaMemcpyDeviceToHost, st));
   if (hit_coords && b.n_coord) CU(cudaMemcpyAsync(hit_coords, b.coords, b.n_coord * 2, cudaMemcpyDeviceToHost, st));
   CU(cudaStreamSynchronize(st));
   return SBQ_SUCCESS;
}

int sbq_synth_giant(sbq_ctx* c, const sbq_synth_giant_spec* sp) {
   if (!c || !sp || sp->n_loci < 1 || sp->rows_per_locus < 1 || sp->iso_lo < 1 || sp->iso_hi < sp->iso_lo || sp->iso_hi > SBQ_MAX_ISO ||
       !(sp->mean_extra >= 0) || sp->mean_extra > 200.0)
      return SBQ_ERR_INVALID;
   if (c->multi) return fail(c, SBQ_ERR_UNSUPPORTED, "sbq_synth_giant is per device: give every device of a partition its own locus ids");
   if (c->cfg.bias_mode) return fail(c, SBQ_ERR_UNSUPPORTED, "sbq_synth_giant generates no covariates");
   std::lock_guard<std::mutex> lk(c->mu);
   CU(cudaSetDevice(c->device));
   reset_batch(c);
   const int L = sp->n_loci;
   const int64_t rows = sp->rows_per_locus, n_row = (int64_t)L * rows;
   // per-locus keys and T on the host (same hash as the device code), Poisson CDF by the exactly reproducible recurrence
   std::vector<SynthLocus> hl((size_t)L);
   std::vector<int64_t> h_lro((size_t)L + 1), h_lio((size_t)L + 1, 0);
   for (int l = 0; l < L; ++l) {
      const uint64_t id = sp->locus_ids ? (uint64_t)(uint32_t)sp->locus_ids[l] : (uint64_t)l;
      hl[l].key_deg = synth_key(sp->seed, id, 1);
      hl[l].key_ent = synth_key(sp->seed, id, 2);
      hl[l].key_len = synth_key(sp->seed, id, 3);
      hl[l].T = sp->iso_lo + (int32_t)(sm64(synth_key(sp->seed, id, 0)) % (uint64_t)(sp->iso_hi - sp->iso_lo + 1));
      hl[l].pad = 0;
      h_lro[l] = (int64_t)l * rows;
      h_lio[l + 1] = h_lio[l] + hl[l].T;
   }
   h_lro[L] = n_row;
   double cdf[SYN_CDF];
   {
      double pk = std::exp(-sp->mean_extra);
      cdf[0] = pk;
      for (int k = 1; k < SYN_CDF; ++k) {
         pk = pk * (sp->mean_extra / (double)k);
         cdf[k] = cdf[k - 1] + pk;
      }
   }
   const int n_scan = (int)((n_row + SYN_SCAN_BLOCK - 1) / SYN_SCAN_BLOCK);
   const size_t b_loci = align_up(L * sizeof(SynthLocus)), b_cdf = align_up(sizeof cdf), b_deg = align_up((size_t)n_row), b_sum = align_up((size_t)n_scan * 8 + 8);
   if (!c->d_synth.reserve(b_loci + b_cdf + b_deg + b_sum + 256)) return fail(c, SBQ_ERR_NOMEM, "device allocation failed (generator scratch)");
   char* q = (char*)c->d_synth.p;
   SynthLocus* d_loci = (SynthLocus*)q; q += b_loci;
   double* d_cdf = (double*)q; q += b_cdf;
   unsigned char* d_deg = (unsigned char*)q; q += b_deg;
   long long* d_bsum = (long long*)q; q += b_sum;
   unsigned long long* d_total = (unsigned long long*)q;
   cudaStream_t st = c->stream;
   CU(cudaEventRecord(c->ev[0], st));
   CU(cudaMemcpyAsync(d_loci, hl.data(), L * sizeof(SynthLocus), cudaMemcpyHostToDevice, st));
   CU(cudaMemcpyAsync(d_cdf, cdf, sizeof cdf, cudaMemcpyHostToDevice, st));
   CU(cudaMemsetAsync(d_total, 0, 8, st));
   const int nb = c->prop.multiProcessorCount * 8;
   synth_degree_kernel<<<nb, 256, 0, st>>>(d_loci, L, rows, d_cdf, d_deg, d_total);
   CU(cudaGetLastError());
   unsigned long long total = 0;
   CU(cudaMemcpyAsync(&total, d_total, 8, cudaMemcpyDeviceToHost, st));
   CU(cudaStreamSynchronize(st));
   c->n_loci = L; c->n_row = n_row; c->n_iso = h_lio[L]; c->nnz = (int64_t)total;
   {
      const int rc = alloc_device(c);
      if (rc) { reset_batch(c); return rc; }
   }
   DevParams& dp = c->dp;
   CU(cudaMemcpyAsync(const_cast<int64_t*>(dp.loc_row_off), h_lro.data(), (L + 1) * 8, cudaMemcpyHostToDevice, st));
   CU(cudaMemcpyAsync(const_cast<int64_t*>(dp.loc_iso_off), h_lio.data(), (L + 1) * 8, cudaMemcpyHostToDevice, st));
   synth_scan_sums_kernel<<<n_scan, 1024, 0, st>>>(d_deg, n_row, d_bsum);
   synth_scan_blocks_kernel<<<1, 1024, 0, st>>>(d_bsum, n_scan);
   synth_scan_fill_kernel<<<n_scan, 1024, 0, st>>>(d_deg, n_row, d_bsum, const_cast<int64_t*>(dp.row_ptr), const_cast<int32_t*>(dp.count));
   synth_fill_kernel<<<nb, 256, 0, st>>>(d_loci, L, rows, dp.row_ptr, const_cast<int32_t*>(dp.col), const_cast<double*>(dp.alpha));
   synth_len_kernel<<<std::min(L, 1024), 256, 0, st>>>(d_loci, L, dp.loc_iso_off, const_cast<int32_t*>(dp.iso_len));
   CU(cudaGetLastError());
   // per-locus non-zeros for the planner: row_ptr at the locus boundaries (one strided copy)
   std::vector<int64_t> bound((size_t)L + 1);
   CU(cudaMemcpy2DAsync(bound.data(), 8, dp.row_ptr, (size_t)rows * 8, 8, (size_t)L + 1, cudaMemcpyDeviceToHost, st));
   CU(cudaStreamSynchronize(st));
   c->meta.resize((size_t)L);
   for (int l = 0; l < L; ++l) c->meta[l] = {bound[l + 1] - bound[l], rows, (int32_t)rows, hl[l].T};
   if (rows > INT32_MAX) return fail(c, SBQ_ERR_INVALID, "rows_per_locus too large");
   {
      const int rc = plan(c);
      if (rc) { reset_batch(c); return rc; }
   }
   if (c->h_lists.n) CU(cudaMemcpyAsync(c->d_lists_p, c->h_lists.p, c->h_lists.n * sizeof(int32_t), cudaMemcpyHostToDevice, st));
   if (!c->classes.empty()) {
      if (!c->d_csc.reserve(align_up(c->nnz * 4 + 16))) return fail(c, SBQ_ERR_NOMEM, "device allocation failed (transposed-index scratch)");
      dp.csc = (unsigned*)c->d_csc.p;
   }
   CU(cudaEventRecord(c->ev[1], st));
   CU(cudaStreamSynchronize(st));
   float ms = 0;
   CU(cudaEventElapsedTime(&ms, c->ev[0], c->ev[1]));
   c->stats.upload_ms = ms;   // generation time stands in for the upload
   c->stats.h2d_bytes = 0;
   c->stats.n_loci = c->n_loci; c->stats.n_row = c->n_row; c->stats.n_iso = c->n_iso; c->stats.nnz = c->nnz;
   c->stats.weights_ms = 0.0;
   c->deferred = 2;
   c->host_released = true;   // the batch exists on the device only
   c->resident = true;
   c->col16_ready = false;
   c->solved = c->downloaded = false;
   return SBQ_SUCCESS;
}

int sbq_fetch_batch(sbq_ctx* c, int64_t* loc_row_off_, int64_t* loc_iso_off_, int64_t* row_ptr_, int32_t* col, double* alpha, int32_t* count, int32_t* iso_len) {
   if (!c) return SBQ_ERR_INVALID;
   if (c->multi) return fail(c, SBQ_ERR_UNSUPPORTED, "sbq_fetch_batch is single-device");
   std::lock_guard<std::mutex> lk(c->mu);
   CU(cudaSetDevice(c->device));
   if (!c->resident) return fail(c, SBQ_ERR_STATE, "sbq_fetch_batch before sbq_upload / sbq_synth_giant");
   { const int rcw = upload_wait(c); if (rcw) return rcw; }
   cudaStream_t st = c->stream;
   if (loc_row_off_) CU(cudaMemcpyAsync(loc_row_off_, c->dp.loc_row_off, (c->n_loci + 1) * 8, cudaMemcpyDeviceToHost, st));
   if (loc_iso_off_) CU(cudaMemcpyAsync(loc_iso_off_, c->dp.loc_iso_off, (c->n_loci + 1) * 8, cudaMemcpyDeviceToHost, st));
   if (row_ptr_) CU(cudaMemcpyAsync(row_ptr_, c->dp.row_ptr, (c->n_row + 1) * 8, cudaMemcpyDeviceToHost, st));
   if (col) CU(cudaMemcpyAsync(col, c->dp.col, c->nnz * 4, cudaMemcpyDeviceToHost, st));
   if (alpha) CU(cudaMemcpyAsync(alpha, c->dp.alpha, c->nnz * 8, cudaMemcpyDeviceToHost, st));
   if (count) CU(cudaMemcpyAsync(count, c->dp.count, c->n_row * 4, cudaMemcpyDeviceToHost, st));
   if (iso_len) CU(cudaMemcpyAsync(iso_len, c->dp.iso_len, c->n_iso * 4, cudaMemcpyDeviceToHost, st));
   CU(cudaStreamSynchronize(st));
   return SBQ_SUCCESS;
}

int sbq_fetch_alpha(sbq_ctx* c, double* alpha) {
   if (!c || !alpha) return SBQ_ERR_INVALID;
   if (c->multi) return fail(c, SBQ_ERR_UNSUPPORTED, "sbq_fetch_alpha is single-device");
   std::lock_guard<std::mutex> lk(c->mu);
   CU(cudaSetDevice(c->device));
   if (!c->resident) return fail(c, SBQ_ERR_STATE, "sbq_fetch_alpha before sbq_upload");
   { const int rcw = upload_wait(c); if (rcw) return rcw; }
   CU(cudaMemcpyAsync(alpha, c->dp.alpha, c->nnz * 8, cudaMemcpyDeviceToHost, c->stream));
   CU(cudaStreamSynchronize(c->stream));
   return SBQ_SUCCESS;
}

int sbq_set_covariates(sbq_ctx* c, const double* x, int64_t n_row, int32_t n_cov) {
   if (!c || n_cov < 0 || n_cov > BI_MAX_COV || (n_cov > 0 && !x)) return SBQ_ERR_INVALID;
   std::lock_guard<std::mutex> lk(c->mu);
   if (n_row != c->n_row) return fail(c, SBQ_ERR_INVALID, "covariates for %lld rows, %lld rows queued", (long long)n_row, (long long)c->n_row);
   cudaSetDevice(c->device);
   c->h_cov.clear();
   if (!c->h_cov.append(x, (size_t)n_row * n_cov)) return fail(c, SBQ_ERR_NOMEM, "pinned staging");
   c->n_cov = n_cov;
   c->have_cov = true;
   c->resident = c->solved = c->downloaded = false;
   return SBQ_SUCCESS;
}

int sbq_bias_results(sbq_ctx* c, double* beta, int32_t* outer_iters) {
   if (!c) return SBQ_ERR_INVALID;
   std::lock_guard<std::mutex> lk(c->mu);
   CU(cudaSetDevice(c->device));
   if (c->cfg.bias_mode != 1 || !c->solved) return fail(c, SBQ_ERR_STATE, "sbq_bias_results needs a solved bias-mode batch");
   if (c->multi) {   // per-device results scattered back into submit order
      MultiState& m = *c->multi;
      const size_t K = (size_t)c->n_cov;
      for (size_t i = 0; i < m.child.size(); ++i) {
         const size_t n = m.loci_of[i].size();
         if (!n) continue;
         std::vector<double> b(n * K + 1);
         std::vector<int32_t> o(n);
         const int rc = sbq_bias_results(m.child[i], b.data(), o.data());
         if (rc) return fail(c, rc, "device %d: %s", m.devices[i], m.child[i]->err.c_str());
         for (size_t x = 0; x < n; ++x) {
            const int32_t l = m.loci_of[i][x];
            if (beta && K) memcpy(beta + (size_t)l * K, b.data() + x * K, K * 8);
            if (outer_iters) outer_iters[l] = o[x];
         }
      }
      return SBQ_SUCCESS;
   }
   const size_t K = (size_t)c->n_cov, nl = (size_t)c->n_loci;
   if (!c->r_beta.reserve(nl * K + 1) || !c->r_outer.reserve(nl)) return fail(c, SBQ_ERR_NOMEM, "pinned result buffers");
   if (K) CU(cudaMemcpyAsync(c->r_beta.p, c->bpar.beta, nl * K * 8, cudaMemcpyDeviceToHost, c->stream));
   CU(cudaMemcpyAsync(c->r_outer.p, c->bpar.outer, nl * 4, cudaMemcpyDeviceToHost, c->stream));
   CU(cudaStreamSynchronize(c->stream));
   if (beta && K) memcpy(beta, c->r_beta.p, nl * K * 8);
   if (outer_iters) memcpy(outer_iters, c->r_outer.p, nl * 4);
   return SBQ_SUCCESS;
}

int sbq_get_launch_stats(const sbq_ctx* cc, sbq_launch_stat* out, int cap) {
   if (!cc || (!out && cap > 0)) return SBQ_ERR_INVALID;
   sbq_ctx* c = const_cast<sbq_ctx*>(cc);
   std::lock_guard<std::mutex> lk(c->mu);
   if (c->multi) {   // the children's records, device after device
      int n = 0;
      for (sbq_ctx* ch : c->multi->child) {
         const int k = sbq_get_launch_stats(ch, out && n < cap ? out + n : nullptr, n < cap ? cap - n : 0);
         if (k > 0) n += k;
      }
      return n;
   }
   account(c);
   const int n = (int)c->launch_stats.size();
   for (int i = 0; i < n && i < cap; ++i) out[i] = c->launch_stats[i];
   return n;
}

int sbq_partition_lpt(const int64_t* cost, int64_t n, int32_t n_parts, int32_t* owner) {
   if (n < 0 || n_parts < 1 || (n > 0 && (!cost || !owner))) return SBQ_ERR_INVALID;
   std::vector<int64_t> order((size_t)n);
   for (int64_t i = 0; i < n; ++i) order[i] = i;
   std::sort(order.begin(), order.end(), [&](int64_t a, int64_t b) { return cost[a] != cost[b] ? cost[a] > cost[b] : a < b; });
   std::vector<int64_t> load((size_t)n_parts, 0);
   for (int64_t l : order) {
      int32_t best = 0;
      for (int32_t q = 1; q < n_parts; ++q)
         if (load[q] < load[best]) best = q;
      owner[l] = best;
      load[best] += cost[l];
   }
   return SBQ_SUCCESS;
}

int sbq_locus_devices(sbq_ctx* c, int32_t* device_of_locus) {
   if (!c || !device_of_locus) return SBQ_ERR_INVALID;
   std::lock_guard<std::mutex> lk(c->mu);
   if (!c->resident) return fail(c, SBQ_ERR_STATE, "sbq_locus_devices before sbq_upload");
   for (int64_t l = 0; l < c->n_loci; ++l) device_of_locus[l] = c->multi ? c->multi->devices[c->multi->owner[l]] : c->device;
   return SBQ_SUCCESS;
}

int sbq_em_solve(sbq_ctx* c, const sbq_locus* locus, double* theta, int32_t* iters) {
   if (!c || !locus || !theta) return SBQ_ERR_INVALID;
   int rc = sbq_clear(c);
   if (rc) return rc;
   if ((rc = sbq_submit(c, locus, 1))) return rc;
   if ((rc = sbq_run(c, 1000000))) return rc;
   int32_t it = 0, st = 0;
   if ((rc = sbq_results(c, theta, nullptr, nullptr, nullptr, nullptr, &it, &st))) return rc;
   if (iters) *iters = it;
   return st;
}

#ifdef SBQ_TRACE
// debug builds only (not part of the ABI header): copy out and reset the CTA timeline; 4 words per record, returns the count
int sbq_debug_trace(unsigned long long* out, int cap) {
   unsigned n = 0;
   cudaDeviceSynchronize();
   cudaMemcpyFromSymbol(&n, sbq::g_trace_n, sizeof n);
   if (n > sbq::TRACE_CAP) n = sbq::TRACE_CAP;
   if ((int)n > cap) n = (unsigned)cap;
   if (n) cudaMemcpyFromSymbol(out, sbq::g_trace, (size_t)n * 32);
   const unsigned zero = 0;
   cudaMemcpyToSymbol(sbq::g_trace_n, &zero, sizeof zero);
   return (int)n;
}
#endif

// page-locked host memory for callers that want sbq_submit_flat to use their arrays in place
void* sbq_host_alloc(size_t bytes) {
   void* p = nullptr;
   if (cudaMallocHost(&p, bytes ? bytes : 1) != cudaSuccess) {
      cudaGetLastError();
      return nullptr;
   }
   return p;
}
void sbq_host_free(void* p) {
   if (p) cudaFreeHost(p);
}

}  // extern "C"

// ================================================================================================
// Bootstrap replicates (sbq_bootstrap.cuh; DESIGN.md "Bootstrap replicates")
namespace {

struct BootOut {
   double *theta, *tpm;
   int32_t *iters, *status;
};

size_t boot_out_bytes(const sbq_ctx* c, int64_t n) { return 2 * align_up((size_t)n * c->n_iso * 8) + 2 * align_up((size_t)n * c->n_loci * 4); }

BootOut boot_out(const sbq_ctx* c, int64_t n) {
   char* q = (char*)c->boot.out.p;
   BootOut o;
   o.theta = (double*)q; q += align_up((size_t)n * c->n_iso * 8);
   o.tpm = (double*)q; q += align_up((size_t)n * c->n_iso * 8);
   o.iters = (int32_t*)q; q += align_up((size_t)n * c->n_loci * 4);
   o.status = (int32_t*)q;
   return o;
}

// draw offsets of the resident batch (once per upload: the counts do not change) and the loci's hash positions (every call: a
// multi-GPU parent sets them before it calls)
int boot_prefix(sbq_ctx* c) {
   sbq_ctx::Boot& B = c->boot;
   cudaStream_t st = c->stream;
   const int64_t L = c->n_loci, R = c->n_row;
   if (!B.prefix_ready) {
      for (int64_t l = 0; l < L && l < (int64_t)c->meta.size(); ++l)
         if (c->meta[l].frags > INT32_MAX)
            return fail(c, SBQ_ERR_UNSUPPORTED, "locus %lld holds %lld fragments: a resampled class count must fit int32", (long long)l, (long long)c->meta[l].frags);
      const int64_t nb = (R + RB_SCAN_BLOCK - 1) / RB_SCAN_BLOCK;
      const size_t b_row = align_up((R + 1) * 8), b_loc = align_up((L + 1) * 8), b_lid = align_up(L * 4 + 4), b_tmp = align_up((nb + 1) * 8);
      if (!B.prefix.reserve(b_row + b_loc + b_lid + b_tmp)) {
         cudaGetLastError();   // a failed allocation is not an error of the context
         return fail(c, SBQ_ERR_NOMEM, "device allocation failed (bootstrap draw offsets)");
      }
      char* q = (char*)B.prefix.p;
      B.draw_off = (int64_t*)q; q += b_row;
      B.loc_draw_off = (int64_t*)q; q += b_loc;
      B.d_lid = (int32_t*)q; q += b_lid;
      if (rb_scan(st, c->dp.count, R, (long long*)q, B.draw_off)) return fail(c, SBQ_ERR_CUDA, "bootstrap count prefix: %s", cudaGetErrorString(cudaGetLastError()));
      rb_gather_kernel<<<(unsigned)((L + 1 + 255) / 256), 256, 0, st>>>(B.draw_off, c->dp.loc_row_off, L + 1, B.loc_draw_off);
      CU(cudaGetLastError());
      B.prefix_ready = true;
   }
   if (!B.lid.empty()) CU(cudaMemcpyAsync(B.d_lid, B.lid.data(), (size_t)L * 4, cudaMemcpyHostToDevice, st));
   return SBQ_SUCCESS;
}

// the counts of replicate `rep` into out[n_row], on c->stream
int boot_resample(sbq_ctx* c, uint64_t seed, uint64_t rep, int32_t* out) {
   const sbq_ctx::Boot& B = c->boot;
   cudaStream_t st = c->stream;
   if (c->n_row) CU(cudaMemsetAsync(out, 0, (size_t)c->n_row * 4, st));
   boot_resample_kernel<<<c->prop.multiProcessorCount * 8, 256, 0, st>>>(B.draw_off, B.loc_draw_off, c->dp.loc_row_off, c->n_loci,
                                                                        B.lid.empty() ? nullptr : B.d_lid, seed, rep, out);
   CU(cudaGetLastError());
   return SBQ_SUCCESS;
}

// replicate scratch: counts [n_row], frac [n_iso], keep [n_iso], locus FPKM [n_loci]
size_t boot_scratch_bytes(const sbq_ctx* c) { return align_up(c->n_row * 4 + 4) + align_up(c->n_iso * 8 + 8) + align_up(c->n_iso * 4 + 4) + align_up(c->n_loci * 8 + 8); }

// resample + EM + FPKM sum of every replicate; dp points at replicate j's slots while its launches are enqueued (c->dp is
// restored by the caller)
int boot_replicates(sbq_ctx* c, uint64_t seed, int64_t first, int32_t n) {
   sbq_ctx::Boot& B = c->boot;
   DevParams& dp = c->dp;
   cudaStream_t st = c->stream;
   const size_t ni = c->n_iso, nl = c->n_loci;
   char* q = (char*)B.scratch.p;
   int32_t* cnt = (int32_t*)q; q += align_up(c->n_row * 4 + 4);
   dp.frac = (double*)q; q += align_up(ni * 8 + 8);
   dp.keep = (int32_t*)q; q += align_up(ni * 4 + 4);
   dp.locus_fpkm = (double*)q;
   dp.count = cnt;
   const BootOut o = boot_out(c, n);
   double* sums = (double*)B.sums.p;
   int64_t launches = 0;
   for (int32_t j = 0; j < n; ++j) {
      CU(cudaEventRecord(B.ev[2 * j], st));
      int rc = boot_resample(c, seed, (uint64_t)first + (uint64_t)j, cnt);
      if (rc) return rc;
      CU(cudaEventRecord(B.ev[2 * j + 1], st));
      dp.theta = o.theta + j * ni;
      dp.fpkm = o.tpm + j * ni;   // FPKM now, TPM after the last replicate (boot_finish_locked)
      dp.iters = o.iters + j * nl;
      dp.status = o.status + j * nl;
      if ((rc = launch_em(c, false, launches))) return rc;
      fpkm_sum_kernel<<<1, 1024, 0, st>>>(dp.locus_fpkm, c->n_loci, sums + j);
      CU(cudaGetLastError());
   }
   CU(cudaEventRecord(B.ev[2 * n], st));
   return SBQ_SUCCESS;
}

}  // namespace

namespace {

int boot_em_locked(sbq_ctx* c, uint64_t seed, int64_t first, int32_t n) {
   CU(cudaSetDevice(c->device));
   if (!c->resident || !c->solved) return fail(c, SBQ_ERR_STATE, "sbq_bootstrap before sbq_solve");
   sbq_ctx::Boot& B = c->boot;
   B.done = false;
   int rc = boot_prefix(c);
   if (rc) return rc;
   if (!B.scratch.reserve(boot_scratch_bytes(c)) || !B.sums.reserve((size_t)n * 8) || !B.out.reserve(boot_out_bytes(c, n))) {
      cudaGetLastError();
      return fail(c, SBQ_ERR_NOMEM, "device allocation failed (%d bootstrap replicates: %zu MB)", n, (boot_out_bytes(c, n) + boot_scratch_bytes(c)) >> 20);
   }
   while (B.ev.size() < 2 * (size_t)n + 2) {
      cudaEvent_t e = nullptr;
      CU(cudaEventCreate(&e));
      B.ev.push_back(e);
   }
   B.stat = sbq_bootstrap_stat{first, n, 0.0, 0.0, 0.0};
   const DevParams point = c->dp;
   rc = boot_replicates(c, seed, first, n);
   c->dp = point;
   return rc;
}

// TPM of every replicate from its FPKM sum in B.sums (multi-GPU: all-reduced), then the timing
int boot_finish_locked(sbq_ctx* c) {
   sbq_ctx::Boot& B = c->boot;
   CU(cudaSetDevice(c->device));
   cudaStream_t st = c->stream;
   const int64_t n = B.stat.n, tot = n * c->n_iso;
   if (tot) {
      const int blocks = (int)std::min<int64_t>((tot + 255) / 256, (int64_t)c->prop.multiProcessorCount * 16);
      boot_tpm_kernel<<<blocks, 256, 0, st>>>(boot_out(c, n).tpm, c->n_iso, n, (const double*)B.sums.p);
      CU(cudaGetLastError());
   }
   CU(cudaEventRecord(B.ev[2 * n + 1], st));
   CU(cudaStreamSynchronize(st));
   float ms = 0;
   for (int64_t j = 0; j < n; ++j) {
      CU(cudaEventElapsedTime(&ms, B.ev[2 * j], B.ev[2 * j + 1]));
      B.stat.resample_ms += ms;
      CU(cudaEventElapsedTime(&ms, B.ev[2 * j + 1], B.ev[2 * j + 2]));
      B.stat.em_ms += ms;
   }
   CU(cudaEventElapsedTime(&ms, B.ev[0], B.ev[2 * n + 1]));
   B.stat.total_ms = ms;
   B.done = true;
   return SBQ_SUCCESS;
}

int boot_counts_locked(sbq_ctx* c, uint64_t seed, int64_t rep, int32_t* count) {
   CU(cudaSetDevice(c->device));
   if (!c->resident) return fail(c, SBQ_ERR_STATE, "sbq_bootstrap_counts before sbq_upload");
   int rc = upload_wait(c);
   if (!rc) rc = boot_prefix(c);
   if (rc) return rc;
   if (!c->boot.scratch.reserve(boot_scratch_bytes(c))) {
      cudaGetLastError();
      return fail(c, SBQ_ERR_NOMEM, "device allocation failed (bootstrap counts)");
   }
   int32_t* d = (int32_t*)c->boot.scratch.p;
   if ((rc = boot_resample(c, seed, (uint64_t)rep, d))) return rc;
   if (c->n_row) CU(cudaMemcpyAsync(count, d, (size_t)c->n_row * 4, cudaMemcpyDeviceToHost, c->stream));
   CU(cudaStreamSynchronize(c->stream));
   return SBQ_SUCCESS;
}

int boot_results_locked(sbq_ctx* c, double* theta, double* tpm, int32_t* iters, int32_t* status) {
   CU(cudaSetDevice(c->device));
   if (!c->boot.done) return fail(c, SBQ_ERR_STATE, "sbq_bootstrap_results before sbq_bootstrap");
   const int64_t n = c->boot.stat.n;
   const BootOut o = boot_out(c, n);
   cudaStream_t st = c->stream;
   const size_t bi = (size_t)n * c->n_iso, bl = (size_t)n * c->n_loci;
   if (theta && bi) CU(cudaMemcpyAsync(theta, o.theta, bi * 8, cudaMemcpyDeviceToHost, st));
   if (tpm && bi) CU(cudaMemcpyAsync(tpm, o.tpm, bi * 8, cudaMemcpyDeviceToHost, st));
   if (iters && bl) CU(cudaMemcpyAsync(iters, o.iters, bl * 4, cudaMemcpyDeviceToHost, st));
   if (status && bl) CU(cudaMemcpyAsync(status, o.status, bl * 4, cudaMemcpyDeviceToHost, st));
   CU(cudaStreamSynchronize(st));
   return SBQ_SUCCESS;
}

}  // namespace

extern "C" {

int sbq_bootstrap(sbq_ctx* c, uint64_t seed, int64_t first, int32_t n) {
   if (!c) return SBQ_ERR_INVALID;
   if (c->cfg.bias_mode == 1) return fail(c, SBQ_ERR_UNSUPPORTED, "bootstrap replicates are defined for the reference EM only (bias_mode = 0)");
   if (n < 1 || first < 0) return fail(c, SBQ_ERR_INVALID, "sbq_bootstrap: n = %d, first = %lld", n, (long long)first);
   if (c->multi) return multi_bootstrap(c, seed, first, n);
   std::lock_guard<std::mutex> lk(c->mu);
   int rc = boot_em_locked(c, seed, first, n);
   if (!rc) rc = boot_finish_locked(c);
   return rc;
}

int sbq_bootstrap_results(sbq_ctx* c, double* theta, double* tpm, int32_t* iters, int32_t* status) {
   if (!c) return SBQ_ERR_INVALID;
   if (c->multi) return multi_bootstrap_results(c, theta, tpm, iters, status);
   std::lock_guard<std::mutex> lk(c->mu);
   return boot_results_locked(c, theta, tpm, iters, status);
}

int sbq_bootstrap_counts(sbq_ctx* c, uint64_t seed, int64_t replicate, int32_t* count) {
   if (!c) return SBQ_ERR_INVALID;
   if (!count || replicate < 0) return fail(c, SBQ_ERR_INVALID, "sbq_bootstrap_counts: null output or replicate < 0");
   if (c->multi) return multi_bootstrap_counts(c, seed, replicate, count);
   std::lock_guard<std::mutex> lk(c->mu);
   return boot_counts_locked(c, seed, replicate, count);
}

int sbq_bootstrap_stats(const sbq_ctx* cc, sbq_bootstrap_stat* out) {
   if (!cc || !out) return SBQ_ERR_INVALID;
   sbq_ctx* c = const_cast<sbq_ctx*>(cc);
   std::lock_guard<std::mutex> lk(c->mu);
   if (!c->boot.done) return fail(c, SBQ_ERR_STATE, "sbq_bootstrap_stats before sbq_bootstrap");
   *out = c->boot.stat;
   return SBQ_SUCCESS;
}

}  // extern "C"

// ================================================================================================
// Gibbs posterior samples (sbq_gibbs.cuh; DESIGN.md "Gibbs posterior samples")
namespace {

constexpr int GIBBS_RING = 256;   // rounds whose events are in flight before the oldest is read back

struct GibbsOut {
   double *theta, *tpm;
   int32_t* status;
};

size_t gibbs_out_bytes(const sbq_ctx* c, int64_t n) { return 2 * align_up((size_t)n * c->n_iso * 8) + align_up((size_t)n * c->n_loci * 4); }

GibbsOut gibbs_out(const sbq_ctx* c, int64_t n) {
   char* q = (char*)c->gibbs.out.p;
   GibbsOut o;
   o.theta = (double*)q; q += align_up((size_t)n * c->n_iso * 8);
   o.tpm = (double*)q; q += align_up((size_t)n * c->n_iso * 8);
   o.status = (int32_t*)q;
   return o;
}

// scratch of one call: weights in submitted order and running sums [nnz]; s, phi, gammas / sample theta, NA flags, frac [n_iso];
// counts, keep [n_iso]; gn, hv, row -> locus [n_row]; heavy-draw offsets [n_row + 1]; scan blocks; N_kept, locus FPKM [n_loci];
// iters [n_loci]
struct GibbsScratch {
   double *ga, *cum, *s, *phi, *gbuf, *nabuf, *frac, *nkept, *lfpkm;
   int32_t *cnt, *keep, *gn, *hv, *row_loc, *iters;
   int64_t* hoff;
   long long* scan_tmp;
};

size_t gibbs_scratch_layout(const sbq_ctx* c, GibbsScratch* g) {
   const size_t nz = align_up(c->nnz * 8 + 8), di = align_up(c->n_iso * 8 + 8), ii = align_up(c->n_iso * 4 + 4);
   const size_t ri = align_up(c->n_row * 4 + 4), ro = align_up((c->n_row + 1) * 8);
   const size_t nb = align_up(((c->n_row + RB_SCAN_BLOCK - 1) / RB_SCAN_BLOCK + 1) * 8);
   const size_t ld = align_up(c->n_loci * 8 + 8), li = align_up(c->n_loci * 4 + 4);
   const size_t total = 2 * nz + 5 * di + 2 * ii + 3 * ri + ro + nb + 2 * ld + li;
   if (!g) return total;
   char* q = (char*)c->gibbs.scratch.p;
   auto take = [&](size_t b) { char* r = q; q += b; return r; };
   g->ga = (double*)take(nz); g->cum = (double*)take(nz);
   g->s = (double*)take(di); g->phi = (double*)take(di); g->gbuf = (double*)take(di); g->nabuf = (double*)take(di); g->frac = (double*)take(di);
   g->cnt = (int32_t*)take(ii); g->keep = (int32_t*)take(ii);
   g->gn = (int32_t*)take(ri); g->hv = (int32_t*)take(ri); g->row_loc = (int32_t*)take(ri);
   g->hoff = (int64_t*)take(ro);
   g->scan_tmp = (long long*)take(nb);
   g->nkept = (double*)take(ld); g->lfpkm = (double*)take(ld);
   g->iters = (int32_t*)take(li);
   return total;
}

// The one-off setup of a call on c->stream: ga = alpha in submitted CSR order (the giant tier's layout passes reorder rows in
// place), column sums, row filter, heavy-draw offsets, phi^0 = theta_hat / s.
int gibbs_setup(sbq_ctx* c, const GibbsScratch& g) {
   cudaStream_t st = c->stream;
   const DevParams& dp = c->dp;
   const int sms = c->prop.multiProcessorCount;
   if (c->nnz) CU(cudaMemcpyAsync(g.ga, dp.alpha, (size_t)c->nnz * 8, cudaMemcpyDeviceToDevice, st));
   if (c->col16_ready) {
      for (const GridClass& gc : c->grid) {
         const int32_t* list = c->d_lists_p + gc.list_off;
         const unsigned short* c16 = (const unsigned short*)c->d_col16.p;
         if (gc.n_dual) gibbs_unpermute_kernel<<<sms * 8, 256, 0, st>>>(dp, list, (int)gc.n_dual, c16, 1, g.ga);
         if (gc.n_tma) gibbs_unpermute_kernel<<<sms * 8, 256, 0, st>>>(dp, list + gc.n_dual, (int)gc.n_tma, c16, 0, g.ga);
         CU(cudaGetLastError());
      }
   }
   if (c->n_iso) CU(cudaMemsetAsync(g.s, 0, (size_t)c->n_iso * 8, st));
   if (c->n_iso) CU(cudaMemsetAsync(g.cnt, 0, (size_t)c->n_iso * 4, st));
   if (c->n_loci) {
      gibbs_colsum_kernel<<<(unsigned)std::min<int64_t>((c->n_loci + 7) / 8, (int64_t)sms * 16), 256, 0, st>>>(dp, g.ga, c->n_loci, g.s, g.gn, g.hv, g.row_loc, g.nkept);
      CU(cudaGetLastError());
   }
   if (rb_scan(st, g.hv, c->n_row, g.scan_tmp, g.hoff)) return fail(c, SBQ_ERR_CUDA, "gibbs heavy-draw prefix: %s", cudaGetErrorString(cudaGetLastError()));
   if (c->n_iso) {
      gibbs_init_kernel<<<(unsigned)std::min<int64_t>((c->n_iso + 255) / 256, (int64_t)sms * 16), 256, 0, st>>>(dp.theta, g.s, c->n_iso, g.phi);
      CU(cudaGetLastError());
   }
   return SBQ_SUCCESS;
}

// elapsed times of ring slot `slot` into the stat
int gibbs_read_slot(sbq_ctx* c, int slot) {
   cudaEvent_t* e = c->gibbs.ev.data() + 3 + 3 * slot;
   float a = 0, t = 0;
   CU(cudaEventSynchronize(e[2]));
   CU(cudaEventElapsedTime(&a, e[0], e[1]));
   CU(cudaEventElapsedTime(&t, e[1], e[2]));
   c->gibbs.stat.assign_ms += a;
   c->gibbs.stat.theta_ms += t;
   return SBQ_SUCCESS;
}

int gibbs_run_locked(sbq_ctx* c, uint64_t seed, int32_t n, int32_t thin, int32_t burn_in, double prior) {
   CU(cudaSetDevice(c->device));
   if (!c->resident || !c->solved) return fail(c, SBQ_ERR_STATE, "sbq_gibbs before sbq_solve");
   sbq_ctx::Gibbs& G = c->gibbs;
   G.done = false;
   int rc = boot_prefix(c);   // draw offsets (and the 2^31-fragment refusal) and the loci's hash positions
   if (rc) return rc;
   const size_t sb = gibbs_scratch_layout(c, nullptr);
   if (!G.scratch.reserve(sb) || !G.sums.reserve((size_t)n * 8) || !G.out.reserve(gibbs_out_bytes(c, n))) {
      cudaGetLastError();   // a failed allocation is not an error of the context
      return fail(c, SBQ_ERR_NOMEM, "device allocation failed (%d Gibbs samples: %zu MB)", n, (gibbs_out_bytes(c, n) + sb) >> 20);
   }
   while (G.ev.size() < 3 + 3 * (size_t)GIBBS_RING) {
      cudaEvent_t e = nullptr;
      CU(cudaEventCreate(&e));
      G.ev.push_back(e);
   }
   GibbsScratch g;
   gibbs_scratch_layout(c, &g);
   const int64_t rounds = (int64_t)burn_in + (int64_t)n * thin;
   G.stat = sbq_gibbs_stat{n, rounds, 0.0, 0.0, 0.0, 0.0};
   cudaStream_t st = c->stream;
   const sbq_ctx::Boot& B = c->boot;
   const int32_t* lid = B.lid.empty() ? nullptr : B.d_lid;
   const int sms = c->prop.multiProcessorCount;
   CU(cudaEventRecord(G.ev[0], st));
   if ((rc = gibbs_setup(c, g))) return rc;
   CU(cudaEventRecord(G.ev[1], st));
   const GibbsOut o = gibbs_out(c, n);
   const uint64_t skey = sm64(seed ^ GIBBS_SALT);
   const unsigned row_blocks = (unsigned)std::max<int64_t>(1, std::min<int64_t>((c->n_row + 255) / 256, (int64_t)sms * 16));
   const unsigned loc_blocks = (unsigned)std::max<int64_t>(1, std::min<int64_t>(c->n_loci, (int64_t)sms * 8));
   DevParams sp = c->dp;   // the sample's slots: theta / FPKM / status of the output matrices, the rest scratch
   sp.frac = g.frac;
   sp.keep = g.keep;
   sp.iters = g.iters;
   sp.locus_fpkm = g.lfpkm;
   for (int64_t r = 1; r <= rounds; ++r) {
      const int slot = (int)((r - 1) % GIBBS_RING);
      if (r > GIBBS_RING && (rc = gibbs_read_slot(c, slot))) return rc;
      cudaEvent_t* e = G.ev.data() + 3 + 3 * slot;
      const uint64_t rkey = sm64(skey + (uint64_t)r);
      CU(cudaEventRecord(e[0], st));
      if (c->n_row) {
         gibbs_assign_kernel<<<row_blocks, 256, 0, st>>>(c->dp, g.ga, g.gn, g.row_loc, B.draw_off, B.loc_draw_off, lid, g.phi, rkey, c->n_row, g.cum, g.cnt);
         gibbs_heavy_kernel<<<sms * 8, 256, 0, st>>>(c->dp, g.hoff, c->n_row, g.row_loc, B.draw_off, B.loc_draw_off, lid, rkey, g.cum, g.cnt);
         CU(cudaGetLastError());
      }
      CU(cudaEventRecord(e[1], st));
      const int64_t sr = r - burn_in;
      const int sample = sr > 0 && sr % thin == 0;
      const int64_t s = sample ? sr / thin - 1 : 0;
      if (sample) {
         sp.theta = o.theta + s * c->n_iso;
         sp.fpkm = o.tpm + s * c->n_iso;   // FPKM now, TPM after the last round (gibbs_finish_locked)
         sp.status = o.status + s * c->n_loci;
      }
      if (c->n_loci) {
         gibbs_theta_kernel<<<loc_blocks, GIBBS_NT, 0, st>>>(sp, c->n_loci, c->dp.theta, c->dp.status, g.s, g.nkept, lid, rkey, prior, sample, g.cnt, g.phi, g.gbuf, g.nabuf);
         CU(cudaGetLastError());
      }
      if (sample) {
         fpkm_sum_kernel<<<1, 1024, 0, st>>>(g.lfpkm, c->n_loci, (double*)G.sums.p + s);
         CU(cudaGetLastError());
      }
      CU(cudaEventRecord(e[2], st));
   }
   return SBQ_SUCCESS;
}

// TPM of every sample from its FPKM sum in G.sums (multi-GPU: all-reduced), then the timing
int gibbs_finish_locked(sbq_ctx* c) {
   sbq_ctx::Gibbs& G = c->gibbs;
   CU(cudaSetDevice(c->device));
   cudaStream_t st = c->stream;
   const int64_t n = G.stat.n, tot = n * c->n_iso;
   if (tot) {
      const int blocks = (int)std::min<int64_t>((tot + 255) / 256, (int64_t)c->prop.multiProcessorCount * 16);
      boot_tpm_kernel<<<blocks, 256, 0, st>>>(gibbs_out(c, n).tpm, c->n_iso, n, (const double*)G.sums.p);
      CU(cudaGetLastError());
   }
   CU(cudaEventRecord(G.ev[2], st));
   CU(cudaStreamSynchronize(st));
   const int64_t rounds = G.stat.rounds;
   for (int64_t r = std::max<int64_t>(1, rounds - GIBBS_RING + 1); r <= rounds; ++r) {
      const int rc = gibbs_read_slot(c, (int)((r - 1) % GIBBS_RING));
      if (rc) return rc;
   }
   float ms = 0;
   CU(cudaEventElapsedTime(&ms, G.ev[0], G.ev[1]));
   G.stat.colsum_ms = ms;
   CU(cudaEventElapsedTime(&ms, G.ev[0], G.ev[2]));
   G.stat.total_ms = ms;
   G.done = true;
   return SBQ_SUCCESS;
}

int gibbs_results_locked(sbq_ctx* c, double* theta, double* tpm, int32_t* status) {
   CU(cudaSetDevice(c->device));
   if (!c->gibbs.done) return fail(c, SBQ_ERR_STATE, "sbq_gibbs_results before sbq_gibbs");
   const int64_t n = c->gibbs.stat.n;
   const GibbsOut o = gibbs_out(c, n);
   cudaStream_t st = c->stream;
   const size_t bi = (size_t)n * c->n_iso, bl = (size_t)n * c->n_loci;
   if (theta && bi) CU(cudaMemcpyAsync(theta, o.theta, bi * 8, cudaMemcpyDeviceToHost, st));
   if (tpm && bi) CU(cudaMemcpyAsync(tpm, o.tpm, bi * 8, cudaMemcpyDeviceToHost, st));
   if (status && bl) CU(cudaMemcpyAsync(status, o.status, bl * 4, cudaMemcpyDeviceToHost, st));
   CU(cudaStreamSynchronize(st));
   return SBQ_SUCCESS;
}

}  // namespace

extern "C" {

int sbq_gibbs(sbq_ctx* c, uint64_t seed, int32_t n, int32_t thin, int32_t burn_in, double prior) {
   if (!c) return SBQ_ERR_INVALID;
   if (c->cfg.bias_mode == 1) return fail(c, SBQ_ERR_UNSUPPORTED, "Gibbs samples are defined for the reference EM only (bias_mode = 0)");
   if (n < 1 || thin < 1 || burn_in < 0 || !(prior > 0.0 && prior < INFINITY))
      return fail(c, SBQ_ERR_INVALID, "sbq_gibbs: n = %d, thin = %d, burn_in = %d, prior = %g", n, thin, burn_in, prior);
   if (c->multi) return multi_gibbs(c, seed, n, thin, burn_in, prior);
   std::lock_guard<std::mutex> lk(c->mu);
   int rc = gibbs_run_locked(c, seed, n, thin, burn_in, prior);
   if (!rc) rc = gibbs_finish_locked(c);
   return rc;
}

int sbq_gibbs_results(sbq_ctx* c, double* theta, double* tpm, int32_t* status) {
   if (!c) return SBQ_ERR_INVALID;
   if (c->multi) return multi_gibbs_results(c, theta, tpm, status);
   std::lock_guard<std::mutex> lk(c->mu);
   return gibbs_results_locked(c, theta, tpm, status);
}

int sbq_gibbs_stats(const sbq_ctx* cc, sbq_gibbs_stat* out) {
   if (!cc || !out) return SBQ_ERR_INVALID;
   sbq_ctx* c = const_cast<sbq_ctx*>(cc);
   std::lock_guard<std::mutex> lk(c->mu);
   if (!c->gibbs.done) return fail(c, SBQ_ERR_STATE, "sbq_gibbs_stats before sbq_gibbs");
   *out = c->gibbs.stat;
   return SBQ_SUCCESS;
}

}  // extern "C"

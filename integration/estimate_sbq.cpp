// estimate_sbq.cpp - link-seam replacement for the reference's src/estimate.cpp.
//
// Compiled against the UNMODIFIED reference headers and linked with the reference's other objects in place of
// estimate.o (integration/Makefile). It keeps exactly the symbols alignments.o imports from estimate.o
// (LocusContext::assign_exon_bin / overlap_exons / set_theory_bin_weight / set_bin_weight_without_frag_dist /
// estimate_abundances, LocusContext::_kMinFrac) and forwards the work to libsbq:
//   class table + weights  -> sbq_build_locus   (host builder, include/sbq_builder.h)
//   EM + FPKM/frac/filter  -> sbq_submit / sbq_run / sbq_results on the GPU (include/sbq.h)
// Everything else (BAM/GTF I/O, clustering, TPM loop, GTF printing) is the reference's own code.
#include <atomic>
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <memory>
#include <mutex>
#include <unordered_map>
#include <vector>

#include "estimate.hpp"
#include "sbq.h"
#include "sbq_builder.h"

using namespace std;

const double LocusContext::_kMinFrac = kMinIsoformFrac;

namespace {

struct TableDeleter {
   void operator()(sbq_table* t) const { sbq_table_free(t); }
};
// The constructor (header-inline, include/estimate.hpp:61-109) calls assign_exon_bin and then one of the two
// weight setters on the same thread: the table built by the first call is handed to the second through this slot.
thread_local unique_ptr<sbq_table, TableDeleter> tl_table;
thread_local bool tl_deferred = false;      // the table of this thread's current locus was built with defer_weights = 1
thread_local bool tl_raw = false;           // this thread's current locus was queued raw (class table built on the device)
atomic<bool> g_model_set{false};

mutex g_ctx_mu;
sbq_ctx* g_ctx = nullptr;
double g_insert_mean = 0.0;   // set from the Sample of the first locus, before the context is created

// ---- batched mode (integration/procsample_sbq.cpp): estimate_abundances() is called twice per locus. The first call
// ("stage") queues the locus' class table with sbq_submit and returns; after ONE sbq_run for the whole sample the second
// call ("finish") performs the reference's per-locus tail (theta log line, FPKM / frac strings, low-fraction erase) from
// the results of that locus. Per-locus mode (the default, used when the reference's own procSample drives) does both at once.
enum { MODE_PER_LOCUS = 0, MODE_STAGE = 1, MODE_FINISH = 2 };
int g_mode = MODE_PER_LOCUS;
struct Staged { int64_t locus, iso_off; };   // iso_off < 0: not known yet (raw loci submitted concurrently; filled by sbq_batch_run)
unordered_map<const LocusContext*, Staged> g_staged;
int64_t g_n_loci = 0, g_n_iso = 0;
vector<int32_t> g_raw_niso;                    // isoforms of every raw locus by batch position
vector<double> g_theta, g_fpkm, g_frac, g_tpm;
vector<int32_t> g_keep, g_status;

struct Timers {   // SBQ_TIMING=1: where quantification time goes (printed at exit)
   atomic<long long> table_ns{0}, stage_ns{0}, run_ns{0}, finish_ns{0};
   atomic<long long> loci{0}, device_class_loci{0};
   bool on = getenv("SBQ_TIMING") != nullptr;
   ~Timers() {
      if (!on) return;
      sbq_stats st{};
      if (g_ctx) sbq_get_stats(g_ctx, &st);
      fprintf(stderr, "SBQ_TIMING sbq loci %lld class_table_ms %.3f stage_ms %.3f run_ms %.3f (upload %.3f solve %.3f download %.3f) finish_ms %.3f device_class_loci %lld\n",
              loci.load(), table_ns / 1e6, stage_ns / 1e6, run_ns / 1e6, st.upload_ms, st.solve_ms, st.download_ms, finish_ns / 1e6, device_class_loci.load());
   }
} g_tm;
long long now_ns() { return chrono::duration_cast<chrono::nanoseconds>(chrono::steady_clock::now().time_since_epoch()).count(); }

sbq_ctx* context() {   // caller holds g_ctx_mu
   if (!g_ctx) {
      sbq_config cfg;
      sbq_config_default(&cfg);
      cfg.min_iso_frac = kMinIsoformFrac;                 // -m / forced 0 with -r (src/Strawberry.cpp:158-162)
      cfg.effective_len_norm = effective_len_norm ? 1 : 0;
      cfg.insert_mean = g_insert_mean;                    // kb = _length - _insert_size_dist->_mean (src/estimate.cpp:318)
      if (const char* e = getenv("SBQ_N_GPUS")) cfg.n_gpus = atoi(e) > 1 ? atoi(e) : 1;   // loci partitioned over N devices inside libsbq
      const int rc = sbq_create(&cfg, &g_ctx);
      if (rc != SBQ_SUCCESS) {
         fprintf(stderr, "libsbq: %s\n", sbq_error_string(rc));
         exit(1);
      }
   }
   return g_ctx;
}

void flatten(const vector<GenomicFeature>& feats, vector<uint32_t>& off, vector<uint32_t>& len, vector<uint8_t>& code) {
   for (auto const& f : feats) {
      off.push_back(f._genomic_offset);
      len.push_back(f._match_op._len);
      code.push_back((uint8_t)f._match_op._code);
   }
}

}  // namespace

set<pair<uint, uint>> LocusContext::overlap_exons(const vector<GenomicFeature>& exons, const Contig& read) const {
   // segments that any aligned block of the read touches (closed intervals); still needed by the header-inline
   // get_frag_info() for the -f fragment-context output
   set<pair<uint, uint>> coords;
   for (auto const& seg : exons) {
      if (seg._match_op._code != Match_t::S_MATCH) continue;
      for (auto const& f : read._genomic_feats)
         if (f._match_op._code == Match_t::S_MATCH && f.left() <= seg.right() && seg.left() <= f.right()) {
            coords.insert(make_pair(seg.left(), seg.right()));
            break;
         }
   }
   return coords;
}

void LocusContext::assign_exon_bin(const vector<Contig>& hits, const vector<GenomicFeature>& exon_segs) {
   // flatten the locus and let the libsbq host builder make the class table and the weights
   vector<int32_t> iso_ptr(1, 0), hit_ptr(1, 0), ref_ids;
   vector<uint32_t> ioff, ilen, hoff, hlen;
   vector<uint8_t> icode, hcode;
   vector<double> mass;
   for (auto const& iso : _transcripts) {
      flatten(iso._contig._genomic_feats, ioff, ilen, icode);
      iso_ptr.push_back((int32_t)ioff.size());
   }
   for (auto const& h : hits) {
      flatten(h._genomic_feats, hoff, hlen, hcode);
      hit_ptr.push_back((int32_t)hoff.size());
      mass.push_back((double)h.mass());
      ref_ids.push_back(h.ref_id());
   }
   const InsertSize& ins = *_sample._insert_size_dist;
   sbq_insert_model model{ins._use_emp ? 1 : 0, ins._use_emp ? ins._start_offset : 0, ins._use_emp ? ins._end_offset : 0,
                          ins._use_emp ? ins._emp_dist.data() : nullptr, ins._use_emp ? ins._total_reads : 0, ins._mean, ins._sd};
   // batched mode: the alpha sums (set_theory_bin_weight, ~80 % of the reference's quantification time) are evaluated on the GPU
   // during sbq_upload; only -f needs the alpha rows in ExonBin::_bin_weight_map on the host
   const int defer = (g_mode == MODE_STAGE && !print_frag_context && !getenv("SBQ_HOST_WEIGHTS")) ? 1 : 0;
   sbq_locus_input in{(int32_t)_transcripts.size(), iso_ptr.data(), ioff.data(), ilen.data(), icode.data(),
                      (int32_t)hits.size(), hit_ptr.data(), hoff.data(), hlen.data(), hcode.data(), mass.data(), ref_ids.data(),
                      _read_len, long_read_sample ? 1 : 0, defer};
   tl_deferred = defer != 0;
   // Class assignment on the device as well (sbq_submit_raw): the locus is queued as it is - flattened hits and isoforms - and
   // the whole class table of the sample is built by CUDA kernels during sbq_upload. With --allow-multimapped-hits the masses
   // are 1/NH fractions, so the device adds them in the reference's set order (SBQ_RAW_MASS_ANY). -f needs the table on the
   // host; SBQ_HOST_CLASSES=1 keeps the host builder.
   tl_raw = defer && !getenv("SBQ_HOST_CLASSES");   // (on N GPUs libsbq deals every raw locus to a device at submit time)
   if (defer && !g_model_set.load()) {      // the context's insert model, read length and mass mode (once per sample)
      lock_guard<mutex> lk(g_ctx_mu);
      if (!g_model_set.load()) {
         if (!g_ctx) g_insert_mean = ins._mean;
         const int rcm = sbq_set_insert_model(context(), &model, _read_len);
         if (rcm != SBQ_SUCCESS) { fprintf(stderr, "libsbq: sbq_set_insert_model: %s\n", sbq_error_string(rcm)); exit(1); }
         if (!use_only_unique_hits) {
            const int rcx = sbq_set_raw_mass_mode(context(), SBQ_RAW_MASS_ANY);
            if (rcx != SBQ_SUCCESS) { fprintf(stderr, "libsbq: sbq_set_raw_mass_mode: %s\n", sbq_error_string(rcx)); exit(1); }
         }
         g_model_set = true;
      }
   }
   if (tl_raw) {
      const long long t_raw = now_ns();
      sbq_ctx* ctx;
      {
         lock_guard<mutex> lk(g_ctx_mu);
         ctx = context();
      }
      int64_t idx = -1;
      const int rcr = sbq_submit_raw(ctx, &in, &idx);          // thread-safe; the static part of the table is built outside libsbq's lock
      if (rcr != SBQ_SUCCESS) { fprintf(stderr, "libsbq: sbq_submit_raw: %s (%s)\n", sbq_error_string(rcr), sbq_last_error(ctx)); exit(1); }
      {
         lock_guard<mutex> lk(g_ctx_mu);
         g_staged[this] = Staged{idx, -1};
         if ((int64_t)g_raw_niso.size() <= idx) g_raw_niso.resize(idx + 1, 0);
         g_raw_niso[idx] = (int32_t)_transcripts.size();
         g_n_loci += 1;
         g_n_iso += (int64_t)_transcripts.size();
      }
      g_tm.table_ns += now_ns() - t_raw;
      g_tm.loci += 1;
      g_tm.device_class_loci += 1;
      return;                                  // exon_bins stay empty: nothing on the host needs them without -f
   }
   sbq_table* tb = nullptr;
   const long long t_build = now_ns();
   const int rc = sbq_build_locus(&in, &model, &tb);
   g_tm.table_ns += now_ns() - t_build;
   if (rc != SBQ_SUCCESS) {
      fprintf(stderr, "libsbq: sbq_build_locus: %s\n", sbq_error_string(rc));
      exit(1);
   }
   tl_table.reset(tb);

   sbq_table_dims d;
   sbq_table_get_dims(tb, &d);
   assert((size_t)d.n_seg == exon_segs.size());
   vector<int32_t> cptr(d.n_class + 1), coord(max<int64_t>(1, d.n_coord)), hclass(max<size_t>(1, hits.size()));
   sbq_table_classes(tb, cptr.data(), coord.data(), nullptr, nullptr, nullptr);
   sbq_table_hit_classes(tb, hclass.data());
   exon_bins.clear();
   for (int c = 0; c < d.n_class; ++c) {
      set<pair<uint, uint>> coords;
      for (int k = cptr[c]; k < cptr[c + 1]; ++k) coords.insert(make_pair(exon_segs[coord[k]].left(), exon_segs[coord[k]].right()));
      ExonBin eb(coords);
      eb.id() = c;
      exon_bins.push_back(eb);
   }
   for (size_t h = 0; h < hits.size(); ++h)
      if (hclass[h] >= 0) exon_bins[hclass[h]].add_frag(hits[h]);   // keeps read_count() / get_frag_info() working
   sbq_locus L;
   sbq_table_locus(tb, &L);
   for (int c = 0; c < L.n_row; ++c)
      for (int64_t k = L.row_ptr[c]; k < L.row_ptr[c + 1]; ++k) iso_2_bins_map[L.col[k]].insert(c);
}

static void weights_from_table(vector<ExonBin>& bins) {
   if (tl_raw) return;                         // raw locus: there is no host table
   sbq_locus L;
   sbq_table_locus(tl_table.get(), &L);
   for (int c = 0; c < L.n_row; ++c)
      for (int64_t k = L.row_ptr[c]; k < L.row_ptr[c + 1]; ++k) bins[c]._bin_weight_map[L.col[k]] = L.alpha[k];   // 0 placeholders when deferred
   if (!tl_deferred) tl_table.reset();      // a deferred table is queued as it is by estimate_abundances() (stage mode)
}

void LocusContext::set_theory_bin_weight() { weights_from_table(exon_bins); }
void LocusContext::set_bin_weight_without_frag_dist() { weights_from_table(exon_bins); }

bool LocusContext::estimate_abundances() {
   const size_t nrow = exon_bins.size(), niso = _transcripts.size();
   vector<double> theta(niso), fpkm(niso), frac(niso);
   vector<int32_t> keep(niso);
   int32_t status = 0;
   if (g_mode == MODE_STAGE && tl_raw) {       // already queued by assign_exon_bin (sbq_submit_raw)
      tl_raw = false;
      return true;
   }
   if (g_mode != MODE_FINISH) {
      const long long t0 = now_ns();
      vector<int64_t> row_ptr(1, 0);
      vector<int32_t> col, count, iso_len;
      vector<double> alpha;
      for (auto const& bin : exon_bins) {
         count.push_back((int)bin.read_count());
         for (auto const& w : bin._bin_weight_map) { col.push_back(w.first); alpha.push_back(w.second); }
         row_ptr.push_back((int64_t)col.size());
      }
      for (auto const& t : _transcripts) iso_len.push_back(t._length);
      sbq_locus L{(int32_t)niso, (int32_t)nrow, row_ptr.data(), col.data(), alpha.data(), count.data(), iso_len.data()};
      lock_guard<mutex> lk(g_ctx_mu);
      if (!g_ctx) g_insert_mean = _sample._insert_size_dist ? _sample._insert_size_dist->_mean : 0.0;
      sbq_ctx* c = context();
      int rc = 0;
      if (g_mode == MODE_STAGE) {
         if (tl_deferred && tl_table) {                   // class table as built, alpha evaluated on the GPU at upload
            const sbq_table* tb = tl_table.get();
            rc = sbq_submit_deferred(c, &tb, 1);
         } else {
            rc = sbq_submit(c, &L, 1);                    // queued; solved by sbq_batch_run() together with every other locus
         }
         g_staged[this] = Staged{g_n_loci, g_n_iso};
         g_n_loci += 1;
         g_n_iso += (int64_t)niso;
      } else {
         int32_t iters = 0;
         rc = sbq_clear(c);
         if (!rc) rc = sbq_submit(c, &L, 1);
         if (!rc) rc = sbq_run(c, _sample.total_mapped_reads());
         if (!rc) rc = sbq_results(c, theta.data(), fpkm.data(), frac.data(), nullptr, keep.data(), &iters, &status);
      }
      if (rc) {
         fprintf(stderr, "libsbq: %s (%s)\n", sbq_error_string(rc), sbq_last_error(c));
         exit(1);
      }
      g_tm.stage_ns += now_ns() - t0;
      g_tm.loci += 1;
      tl_table.reset();
      tl_deferred = false;
      if (g_mode == MODE_STAGE) return true;
   } else {
      const auto it = g_staged.find(this);
      if (it == g_staged.end()) { fprintf(stderr, "libsbq integration: locus was not staged\n"); exit(1); }
      const Staged sg = it->second;
      for (size_t i = 0; i < niso; ++i) {
         theta[i] = g_theta[sg.iso_off + i]; fpkm[i] = g_fpkm[sg.iso_off + i]; frac[i] = g_frac[sg.iso_off + i]; keep[i] = g_keep[sg.iso_off + i];
      }
      status = g_status[sg.locus];
   }
   const long long t1 = now_ns();
   const bool success = status != SBQ_LOCUS_NO_ROWS;
   if (!success) return false;
   for (size_t i = 0; i < niso; ++i) fprintf(_p_log_file, "isoform %d has %f raw read count.\n", (int)i + 1, theta[i]);
   for (size_t i = 0; i < niso; ++i) {
      if (keep[i] < 0) {                       // effective_len_norm "NA" case
         _transcripts[i]._FPKM_s = "NA";
         _transcripts[i]._frac_s = "NA";
         continue;
      }
      _transcripts[i]._FPKM = fpkm[i];
      _transcripts[i]._FPKM_s = to_string(fpkm[i]);
      _transcripts[i]._frac = frac[i];
      _transcripts[i]._frac_s = to_string(frac[i]);
      if (g_mode == MODE_FINISH) {             // batched mode: TPM comes from the device too (all-reduced over the GPUs of the context)
         const int64_t off = g_staged[this].iso_off;
         _transcripts[i]._TPM = g_tpm[off + i];
         _transcripts[i]._TPM_s = to_string(g_tpm[off + i]);
      }
   }
   if (filter_by_expression) {
      size_t i = 0;
      for (auto it = _transcripts.begin(); it != _transcripts.end(); ++i) {
         if (keep[i] == 0) it = _transcripts.erase(it); else ++it;
      }
   }
   g_tm.finish_ns += now_ns() - t1;
   return true;
}

// ---- batched drop-in hooks, called by the batched Sample::procSample (integration/procsample_sbq.cpp)
void sbq_batch_begin() {
   lock_guard<mutex> lk(g_ctx_mu);
   g_mode = MODE_STAGE;
   g_staged.clear();
   g_raw_niso.clear();
   g_n_loci = g_n_iso = 0;
   if (g_ctx) sbq_clear(g_ctx);
}

// one sbq_run for every staged locus: EM + FPKM / frac / filter + TPM on the GPU(s); afterwards estimate_abundances() finishes loci
void sbq_batch_run(int total_mapped_reads) {
   lock_guard<mutex> lk(g_ctx_mu);
   g_mode = MODE_FINISH;
   if (g_n_loci == 0) return;
   if (!g_raw_niso.empty()) {                  // raw loci: isoform offsets from the batch positions libsbq assigned
      vector<int64_t> off(g_raw_niso.size() + 1, 0);
      for (size_t i = 0; i < g_raw_niso.size(); ++i) off[i + 1] = off[i] + g_raw_niso[i];
      for (auto& kv : g_staged) kv.second.iso_off = off[kv.second.locus];
   }
   const long long t0 = now_ns();
   sbq_ctx* c = context();
   g_theta.resize(g_n_iso); g_fpkm.resize(g_n_iso); g_frac.resize(g_n_iso); g_tpm.resize(g_n_iso); g_keep.resize(g_n_iso); g_status.resize(g_n_loci);
   int rc = sbq_run(c, total_mapped_reads);
   if (!rc) rc = sbq_results(c, g_theta.data(), g_fpkm.data(), g_frac.data(), g_tpm.data(), g_keep.data(), nullptr, g_status.data());
   if (rc) {
      fprintf(stderr, "libsbq: %s (%s)\n", sbq_error_string(rc), sbq_last_error(c));
      exit(1);
   }
   g_tm.run_ns += now_ns() - t0;
}

void sbq_batch_end() {
   lock_guard<mutex> lk(g_ctx_mu);
   g_mode = MODE_PER_LOCUS;
   g_staged.clear();
}

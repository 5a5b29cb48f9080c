// sbq_multi.cuh - multi-GPU inside the C ABI (sbq_config.n_gpus > 1), included by sbq.cu.
//
// Loci are independent (SURVEY section 8e), so the parent context partitions the queued loci over one child context
// per device - greedy LPT by non-zeros, a locus is never split - and every child solves its share with the
// single-device runtime of sbq.cu on its own streams, driven from one host thread per device. The path's only
// exchange step is the TPM denominator, sum of FPKM over the surviving isoforms of ALL loci (reference
// src/alignments.cpp:1821-1824): one ncclAllReduce(ncclDouble, count 1, ncclSum) over the devices, enqueued on each
// child's stream between its EM kernels and its TPM kernel. NCCL is dlopen'ed on first use (libsbq.so carries no
// DT_NEEDED on it, so single-device users and processes that already hold torch's NCCL are unaffected).
#pragma once

namespace {

struct NcclApi {
   void* handle = nullptr;
   ncclResult_t (*CommInitAll)(ncclComm_t*, int, const int*) = nullptr;
   ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
   ncclResult_t (*AllReduce)(const void*, void*, size_t, ncclDataType_t, ncclRedOp_t, ncclComm_t, cudaStream_t) = nullptr;
   ncclResult_t (*GroupStart)() = nullptr;
   ncclResult_t (*GroupEnd)() = nullptr;
   const char* (*GetErrorString)(ncclResult_t) = nullptr;

   bool load(std::string& err) {
      if (handle) return true;
      // a copy the process already holds (e.g. the one bundled with torch) wins, then the system library
      const char* names[] = {"libnccl.so.2", "libnccl.so"};
      for (const char* n : names)
         if ((handle = dlopen(n, RTLD_NOW | RTLD_NOLOAD | RTLD_LOCAL))) break;
      if (!handle)
         for (const char* n : names)
            if ((handle = dlopen(n, RTLD_NOW | RTLD_LOCAL))) break;
      if (!handle) {
         err = std::string("cannot load NCCL (libnccl.so.2): ") + (dlerror() ? dlerror() : "not found");
         return false;
      }
      bool ok = true;
      auto sym = [&](const char* name) {
         void* p = dlsym(handle, name);
         if (!p) { ok = false; err = std::string("NCCL symbol missing: ") + name; }
         return p;
      };
      CommInitAll = (decltype(CommInitAll))sym("ncclCommInitAll");
      CommDestroy = (decltype(CommDestroy))sym("ncclCommDestroy");
      AllReduce = (decltype(AllReduce))sym("ncclAllReduce");
      GroupStart = (decltype(GroupStart))sym("ncclGroupStart");
      GroupEnd = (decltype(GroupEnd))sym("ncclGroupEnd");
      GetErrorString = (decltype(GetErrorString))sym("ncclGetErrorString");
      return ok;
   }
};

NcclApi g_nccl;
std::mutex g_nccl_mu;

}  // namespace

struct MultiState {
   std::vector<sbq_ctx*> child;                  // one single-device context per GPU
   std::vector<int> devices;
   std::vector<ncclComm_t> comm;
   std::vector<double*> d_sum;                   // per device: [0] local FPKM sum (input), [1] all-reduced sum (output)
   std::vector<int32_t> owner;                   // locus -> child (valid after sbq_upload)
   std::vector<std::vector<int32_t>> loci_of;    // child -> its loci, ascending submit order
   std::vector<int64_t> raw_load;                // raw batches: work dealt to every child so far (hits x isoforms)
   bool reduced = false;                         // the all-reduce of the current solve has been enqueued
   double global_sum = 0.0;
};

namespace {

// run f(child index) on one host thread per child that owns loci; returns the first error (and copies its message)
template <typename F>
int multi_for_each(sbq_ctx* c, const F& f) {
   MultiState& m = *c->multi;
   const size_t n = m.child.size();
   std::vector<int> rc(n, 0);
   std::vector<std::thread> th;
   for (size_t i = 0; i < n; ++i) {
      if (m.loci_of[i].empty()) continue;
      th.emplace_back([&, i] { rc[i] = f((int)i); });
   }
   for (auto& t : th) t.join();
   for (size_t i = 0; i < n; ++i)
      if (rc[i]) return fail(c, rc[i], "device %d: %s", m.devices[i], m.child[i]->err.c_str());
   return SBQ_SUCCESS;
}

void multi_destroy(sbq_ctx* c) {
   MultiState* m = c->multi;
   if (!m) return;
   for (size_t i = 0; i < m->comm.size(); ++i)
      if (m->comm[i] && g_nccl.CommDestroy) g_nccl.CommDestroy(m->comm[i]);
   for (size_t i = 0; i < m->d_sum.size(); ++i)
      if (m->d_sum[i]) { cudaSetDevice(m->devices[i]); cudaFree(m->d_sum[i]); }
   for (sbq_ctx* ch : m->child) sbq_destroy(ch);
   delete m;
   c->multi = nullptr;
}

// called by sbq_create for cfg.n_gpus > 1 (c is already a valid single-device context on the first device)
int multi_create(sbq_ctx* c, int n_dev_visible) {
   const int n = c->cfg.n_gpus, base = c->device;
   if (base + n > n_dev_visible) return fail(c, SBQ_ERR_NO_DEVICE, "n_gpus = %d from device %d, but only %d devices are visible", n, base, n_dev_visible);
   {
      std::lock_guard<std::mutex> lk(g_nccl_mu);
      if (!g_nccl.load(c->err)) return SBQ_ERR_NO_DEVICE;
   }
   MultiState* m = new MultiState();
   c->multi = m;
   m->child.assign(n, nullptr);
   m->comm.assign(n, nullptr);
   m->d_sum.assign(n, nullptr);
   m->loci_of.resize(n);
   for (int i = 0; i < n; ++i) m->devices.push_back(base + i);
   for (int i = 0; i < n; ++i) {
      sbq_config cc = c->cfg;
      cc.device = base + i;
      cc.n_gpus = 1;
      const int rc = sbq_create(&cc, &m->child[i]);
      if (rc) return fail(c, rc, "cannot create the context of device %d", base + i);
      if (cudaSetDevice(base + i) != cudaSuccess || cudaMalloc((void**)&m->d_sum[i], 2 * sizeof(double)) != cudaSuccess)
         return fail(c, SBQ_ERR_CUDA, "device %d: allocation failed", base + i);
      cudaMemset(m->d_sum[i], 0, 2 * sizeof(double));
   }
   const ncclResult_t r = g_nccl.CommInitAll(m->comm.data(), n, m->devices.data());
   if (r != ncclSuccess) return fail(c, SBQ_ERR_CUDA, "ncclCommInitAll over %d devices failed: %s", n, g_nccl.GetErrorString(r));
   cudaSetDevice(base);
   return SBQ_SUCCESS;
}

// copy the loci `list` (ascending) of the parent's staged batch into the child's own staging, back to back
int multi_gather(sbq_ctx* par, sbq_ctx* ch, const std::vector<int32_t>& list) {
   const int64_t *lro = loc_row_off(par), *lio = loc_iso_off(par), *rp = row_ptr(par);
   const int32_t *col = colp(par), *cnt = countp(par), *il = iso_lenp(par);
   const double* al = alphap(par);
   int64_t rows = 0, isos = 0, nnz = 0;
   for (int32_t l : list) { rows += lro[l + 1] - lro[l]; isos += lio[l + 1] - lio[l]; nnz += rp[lro[l + 1]] - rp[lro[l]]; }
   std::lock_guard<std::mutex> lk(ch->mu);
   cudaSetDevice(ch->device);
   reset_batch(ch);
   int rc = ensure_origin(ch);
   if (rc) return rc;
   const bool ok = ch->h_loc_row_off.reserve(1 + list.size()) && ch->h_loc_iso_off.reserve(1 + list.size()) && ch->h_row_ptr.reserve(1 + rows) &&
                   ch->h_col.reserve(nnz) && ch->h_alpha.reserve(nnz) && ch->h_count.reserve(rows) && ch->h_iso_len.reserve(isos) &&
                   (!par->have_cov || ch->h_cov.reserve((size_t)rows * par->n_cov));
   if (!ok) return fail(ch, SBQ_ERR_NOMEM, "pinned staging");
   for (size_t x = 0; x < list.size();) {
      // a run of consecutive loci is one contiguous range in every array
      size_t y = x + 1;
      while (y < list.size() && list[y] == list[y - 1] + 1) ++y;
      const int64_t l0 = list[x], l1 = (int64_t)list[y - 1] + 1;
      const int64_t r0 = lro[l0], r1 = lro[l1], k0 = rp[r0], k1 = rp[r1];
      for (int64_t l = l0 + 1; l <= l1; ++l) {
         ch->h_loc_row_off.p[ch->h_loc_row_off.n++] = ch->n_row + (lro[l] - r0);
         ch->h_loc_iso_off.p[ch->h_loc_iso_off.n++] = ch->n_iso + (lio[l] - lio[l0]);
      }
      const int64_t base = ch->nnz - k0;
      for (int64_t i = r0 + 1; i <= r1; ++i) ch->h_row_ptr.p[ch->h_row_ptr.n++] = rp[i] + base;
      ch->h_col.append(col + k0, k1 - k0);
      ch->h_alpha.append(al + k0, k1 - k0);
      ch->h_count.append(cnt + r0, r1 - r0);
      ch->h_iso_len.append(il + lio[l0], lio[l1] - lio[l0]);
      if (par->have_cov) ch->h_cov.append(par->h_cov.p + (size_t)r0 * par->n_cov, (size_t)(r1 - r0) * par->n_cov);
      ch->n_loci += l1 - l0; ch->n_row += r1 - r0; ch->n_iso += lio[l1] - lio[l0]; ch->nnz += k1 - k0;
      x = y;
   }
   if (par->have_cov) { ch->n_cov = par->n_cov; ch->have_cov = true; }
   ch->deferred = 2;
   if (par->deferred == 1) {
      // deferred (GPU) weights: the per-entry descriptors travel with their loci, segment pointers re-based into the child's pool
      if (!ch->h_wseg.reserve(nnz) || !ch->h_wn.reserve(nnz) || !ch->h_wmask.reserve(nnz) || !ch->h_wlen.reserve(nnz)) return fail(ch, SBQ_ERR_NOMEM, "pinned staging");
      for (int32_t l : list) {
         const int64_t k0 = rp[lro[l]], k1 = rp[lro[l + 1]];
         const int64_t p0 = par->h_wpool_off.p[l], p1 = (size_t)l + 1 < par->h_wpool_off.n ? par->h_wpool_off.p[l + 1] : (int64_t)par->h_wpool.n;
         const int64_t shift = (int64_t)ch->h_wpool.n - p0;
         if (!ch->h_wpool.append(par->h_wpool.p + p0, (size_t)(p1 - p0))) return fail(ch, SBQ_ERR_NOMEM, "pinned staging");
         for (int64_t k = k0; k < k1; ++k) ch->h_wseg.p[ch->h_wseg.n++] = par->h_wseg.p[k] < 0 ? -1 : par->h_wseg.p[k] + shift;
         ch->h_wn.append(par->h_wn.p + k0, (size_t)(k1 - k0));
         ch->h_wmask.append(par->h_wmask.p + k0, (size_t)(k1 - k0));
         ch->h_wlen.append(par->h_wlen.p + k0, (size_t)(k1 - k0));
      }
      ch->model = par->model;
      ch->model_emp = par->model_emp;
      ch->model_read_len = par->model_read_len;
      ch->have_model = par->have_model;
      ch->deferred = 1;
   }
   return SBQ_SUCCESS;
}

// Raw loci (class assignment on the device, sbq_submit_raw) on N devices. The non-zeros of a raw locus are not known before its
// device has built the class table, so the locus is dealt at SUBMIT time: to the device with the least work so far, work = hits x
// isoforms (what the compatibility pass and, through the classes, the EM scale with). A function of the submit sequence only.
// The locus is staged directly in that device's context; sbq_upload then builds every device's class tables concurrently.
int multi_submit_raw(sbq_ctx* c, const sbq_locus_input* in, int64_t* locus_index) {
   MultiState& m = *c->multi;
   std::lock_guard<std::mutex> lk(c->mu);
   if (c->host_released || (c->n_loci > 0 && !c->raw_mode)) return fail(c, SBQ_ERR_STATE, "a batch is either all raw loci or none");
   const size_t n = m.child.size();
   if (c->n_loci == 0) {
      for (sbq_ctx* ch : m.child) sbq_clear(ch);
      m.owner.clear();
      for (auto& v : m.loci_of) v.clear();
      m.raw_load.assign(n, 0);
   }
   size_t k = 0;
   for (size_t i = 1; i < n; ++i)
      if (m.raw_load[i] < m.raw_load[k]) k = i;
   const int rc = sbq_submit_raw(m.child[k], in, nullptr);
   if (rc) return fail(c, rc, "device %d: %s", m.devices[k], m.child[k]->err.c_str());
   m.raw_load[k] += (int64_t)in->n_hit * in->n_iso + in->n_hit + in->n_iso;
   m.owner.push_back((int32_t)k);
   m.loci_of[k].push_back((int32_t)c->n_loci);
   if (locus_index) *locus_index = c->n_loci;
   c->n_loci += 1;
   c->n_iso += in->n_iso;
   c->raw_mode = true;
   c->deferred = 1;
   c->resident = c->solved = c->downloaded = false;
   return SBQ_SUCCESS;
}

int multi_upload(sbq_ctx* c) {
   MultiState& m = *c->multi;
   std::lock_guard<std::mutex> lk(c->mu);
   if (c->n_loci == 0) return fail(c, SBQ_ERR_STATE, "nothing submitted");
   c->boot.done = c->gibbs.done = false;
   if (c->raw_mode) {   // the loci already sit in their devices' contexts
      for (sbq_ctx* ch : m.child) {
         sbq_set_plan(ch, c->force_tier, c->force_cluster);
         ch->model = c->model;
         ch->model_emp = c->model_emp;
         ch->model_read_len = c->model_read_len;
         ch->have_model = c->have_model;
         ch->raw_mass_mode = c->raw_mass_mode;
      }
      const int rcr = multi_for_each(c, [&](int i) { return sbq_upload(m.child[i]); });
      if (rcr) return rcr;
      m.reduced = false;
      c->resident = true;
      c->solved = c->downloaded = false;
      return SBQ_SUCCESS;
   }
   if (c->host_released) return fail(c, SBQ_ERR_STATE, "the borrowed batch was released by the previous sbq_upload: sbq_clear and submit again");
   if (c->deferred == 1 && !c->have_model) return fail(c, SBQ_ERR_STATE, "deferred weights need sbq_set_insert_model()");
   if (c->cfg.bias_mode == 1 && !c->have_cov) return fail(c, SBQ_ERR_STATE, "bias_mode = 1 needs sbq_set_covariates() after the last submit");
   const int n = (int)m.child.size();
   const int64_t *lro = loc_row_off(c), *lio = loc_iso_off(c), *rp = row_ptr(c);
   std::vector<int64_t> cost((size_t)c->n_loci);
   for (int64_t l = 0; l < c->n_loci; ++l) cost[l] = (rp[lro[l + 1]] - rp[lro[l]]) + (lro[l + 1] - lro[l]) + (lio[l + 1] - lio[l]);
   m.owner.assign((size_t)c->n_loci, 0);
   sbq_partition_lpt(cost.data(), c->n_loci, n, m.owner.data());
   for (auto& v : m.loci_of) v.clear();
   for (int64_t l = 0; l < c->n_loci; ++l) m.loci_of[m.owner[l]].push_back((int32_t)l);
   for (int i = 0; i < n; ++i) {
      sbq_set_plan(m.child[i], c->force_tier, c->force_cluster);
      if (m.loci_of[i].empty()) sbq_clear(m.child[i]);
   }
   const int rc = multi_for_each(c, [&](int i) {
      int r = multi_gather(c, m.child[i], m.loci_of[i]);
      if (!r) r = sbq_upload(m.child[i]);
      return r;
   });
   if (rc) return rc;
   if (c->borrowed) c->host_released = true;
   m.reduced = false;
   c->resident = true;
   c->solved = c->downloaded = false;
   return SBQ_SUCCESS;
}

int multi_solve(sbq_ctx* c, int64_t total_mapped_reads) {
   MultiState& m = *c->multi;
   std::lock_guard<std::mutex> lk(c->mu);
   if (!c->resident) return fail(c, SBQ_ERR_STATE, "sbq_solve before sbq_upload");
   const int rc = multi_for_each(c, [&](int i) { return sbq_solve(m.child[i], total_mapped_reads); });
   if (rc) return rc;
   m.reduced = false;
   c->solved = true;
   c->downloaded = false;
   return SBQ_SUCCESS;
}

// The path's one collective: all-reduce the per-device FPKM sums (one double), caller holds c->mu.
int multi_allreduce_locked(sbq_ctx* c) {
   MultiState& m = *c->multi;
   if (m.reduced) return SBQ_SUCCESS;
   const int n = (int)m.child.size();
   for (int i = 0; i < n; ++i) {
      sbq_ctx* ch = m.child[i];
      CU(cudaSetDevice(m.devices[i]));
      if (m.loci_of[i].empty()) CU(cudaMemsetAsync(m.d_sum[i], 0, sizeof(double), ch->stream));
      else CU(cudaMemcpyAsync(m.d_sum[i], ch->d_fpkm_sum, sizeof(double), cudaMemcpyDeviceToDevice, ch->stream));
   }
   ncclResult_t r = g_nccl.GroupStart();
   for (int i = 0; i < n && r == ncclSuccess; ++i)
      r = g_nccl.AllReduce(m.d_sum[i], m.d_sum[i] + 1, 1, ncclDouble, ncclSum, m.comm[i], m.child[i]->stream);
   const ncclResult_t r2 = g_nccl.GroupEnd();
   if (r != ncclSuccess || r2 != ncclSuccess) return fail(c, SBQ_ERR_CUDA, "ncclAllReduce failed: %s", g_nccl.GetErrorString(r != ncclSuccess ? r : r2));
   CU(cudaSetDevice(m.devices[0]));
   CU(cudaMemcpyAsync(&m.global_sum, m.d_sum[0] + 1, sizeof(double), cudaMemcpyDeviceToHost, m.child[0]->stream));
   CU(cudaStreamSynchronize(m.child[0]->stream));
   m.reduced = true;
   return SBQ_SUCCESS;
}

// all-reduce + TPM on every device from the DEVICE copy of the reduced sum (no host round trip per device)
int multi_tpm(sbq_ctx* c) {
   MultiState& m = *c->multi;
   std::lock_guard<std::mutex> lk(c->mu);
   if (!c->solved) return fail(c, SBQ_ERR_STATE, "TPM before sbq_solve");
   int rc = multi_allreduce_locked(c);
   if (rc) return rc;
   for (size_t i = 0; i < m.child.size(); ++i) {
      sbq_ctx* ch = m.child[i];
      if (m.loci_of[i].empty()) continue;
      CU(cudaSetDevice(m.devices[i]));
      const int64_t n = ch->n_iso;
      sbq::tpm_dev_kernel<<<(unsigned)((n + 255) / 256), 256, 0, ch->stream>>>(ch->dp.fpkm, ch->d_tpm, n, m.d_sum[i] + 1);
      CU(cudaGetLastError());
      ch->stats.kernel_launches += 1;
      ch->downloaded = false;
   }
   c->downloaded = false;
   return SBQ_SUCCESS;
}

int multi_finalize_tpm(sbq_ctx* c, double global_fpkm_sum) {
   MultiState& m = *c->multi;
   std::lock_guard<std::mutex> lk(c->mu);
   if (!c->solved) return fail(c, SBQ_ERR_STATE, "sbq_finalize_tpm before sbq_solve");
   for (size_t i = 0; i < m.child.size(); ++i) {
      if (m.loci_of[i].empty()) continue;
      const int rc = sbq_finalize_tpm(m.child[i], global_fpkm_sum);
      if (rc) return fail(c, rc, "device %d: %s", m.devices[i], m.child[i]->err.c_str());
   }
   c->downloaded = false;
   return SBQ_SUCCESS;
}

int multi_download(sbq_ctx* c) {
   MultiState& m = *c->multi;
   std::lock_guard<std::mutex> lk(c->mu);
   if (!c->solved) return fail(c, SBQ_ERR_STATE, "sbq_download before sbq_solve");
   const size_t ni = c->n_iso, nl = c->n_loci;
   cudaSetDevice(c->device);
   const bool ok = c->r_theta.reserve(ni) && c->r_fpkm.reserve(ni) && c->r_frac.reserve(ni) && c->r_tpm.reserve(ni) &&
                   c->r_keep.reserve(ni) && c->r_iters.reserve(nl) && c->r_status.reserve(nl);
   if (!ok) return fail(c, SBQ_ERR_NOMEM, "pinned result buffers");
   const int64_t* lio = nullptr;
   // isoform offsets of the parent batch: the host arrays may be gone (borrowed batch), so they are rebuilt from the children
   std::vector<int64_t> iso_off(nl + 1, 0);
   for (size_t i = 0; i < m.child.size(); ++i) {
      const sbq_ctx* ch = m.child[i];
      for (size_t x = 0; x < m.loci_of[i].size(); ++x) iso_off[m.loci_of[i][x] + 1] = ch->meta[x].T;
   }
   for (size_t l = 0; l < nl; ++l) iso_off[l + 1] += iso_off[l];
   lio = iso_off.data();
   const int rc = multi_for_each(c, [&](int i) {
      sbq_ctx* ch = m.child[i];
      const int r = sbq_download(ch);
      if (r) return r;
      int64_t o = 0;
      for (size_t x = 0; x < m.loci_of[i].size(); ++x) {   // scatter back into submit order
         const int32_t l = m.loci_of[i][x];
         const int64_t T = lio[l + 1] - lio[l], d = lio[l];
         memcpy(c->r_theta.p + d, ch->r_theta.p + o, T * 8);
         memcpy(c->r_fpkm.p + d, ch->r_fpkm.p + o, T * 8);
         memcpy(c->r_frac.p + d, ch->r_frac.p + o, T * 8);
         memcpy(c->r_tpm.p + d, ch->r_tpm.p + o, T * 8);
         memcpy(c->r_keep.p + d, ch->r_keep.p + o, T * 4);
         c->r_iters.p[l] = ch->r_iters.p[x];
         c->r_status.p[l] = ch->r_status.p[x];
         o += T;
      }
      return 0;
   });
   if (rc) return rc;
   c->r_fpkm_sum = m.global_sum;
   c->downloaded = true;
   return SBQ_SUCCESS;
}

// Offsets of the parent batch's rows (what = 0) or isoforms (what = 1) in submit order, rebuilt from the children (the parent's host
// arrays may be gone: borrowed batch; raw loci never had them)
std::vector<int64_t> multi_offsets(sbq_ctx* c, int what) {
   MultiState& m = *c->multi;
   std::vector<int64_t> off((size_t)c->n_loci + 1, 0);
   for (size_t i = 0; i < m.child.size(); ++i)
      for (size_t x = 0; x < m.loci_of[i].size(); ++x) off[m.loci_of[i][x] + 1] = what ? m.child[i]->meta[x].T : m.child[i]->meta[x].R;
   for (size_t l = 0; l < (size_t)c->n_loci; ++l) off[l + 1] += off[l];
   return off;
}

// Bootstrap replicates on N devices. Every child resamples its loci under their PARENT submit positions, so a replicate does not
// depend on the partition; the n replicate FPKM sums then meet in ONE ncclAllReduce (count n) before every device's TPM pass.
int multi_bootstrap(sbq_ctx* c, uint64_t seed, int64_t first, int32_t n) {
   MultiState& m = *c->multi;
   std::lock_guard<std::mutex> lk(c->mu);
   if (!c->resident || !c->solved) return fail(c, SBQ_ERR_STATE, "sbq_bootstrap before sbq_solve");
   c->boot.done = false;
   const int nd = (int)m.child.size();
   for (int i = 0; i < nd; ++i) m.child[i]->boot.lid = m.loci_of[i];
   int rc = multi_for_each(c, [&](int i) {
      std::lock_guard<std::mutex> lk2(m.child[i]->mu);
      return boot_em_locked(m.child[i], seed, first, n);
   });
   if (rc) return rc;
   for (int i = 0; i < nd; ++i) {   // devices without loci join the all-reduce with zeros
      if (!m.loci_of[i].empty()) continue;
      sbq_ctx* ch = m.child[i];
      CU(cudaSetDevice(m.devices[i]));
      if (!ch->boot.sums.reserve((size_t)n * 8)) {
         cudaGetLastError();
         return fail(c, SBQ_ERR_NOMEM, "device %d: allocation failed (bootstrap sums)", m.devices[i]);
      }
      CU(cudaMemsetAsync(ch->boot.sums.p, 0, (size_t)n * 8, ch->stream));
   }
   ncclResult_t r = g_nccl.GroupStart();
   for (int i = 0; i < nd && r == ncclSuccess; ++i)
      r = g_nccl.AllReduce(m.child[i]->boot.sums.p, m.child[i]->boot.sums.p, (size_t)n, ncclDouble, ncclSum, m.comm[i], m.child[i]->stream);
   const ncclResult_t r2 = g_nccl.GroupEnd();
   if (r != ncclSuccess || r2 != ncclSuccess) return fail(c, SBQ_ERR_CUDA, "ncclAllReduce failed: %s", g_nccl.GetErrorString(r != ncclSuccess ? r : r2));
   rc = multi_for_each(c, [&](int i) {
      std::lock_guard<std::mutex> lk2(m.child[i]->mu);
      return boot_finish_locked(m.child[i]);
   });
   if (rc) return rc;
   sbq_bootstrap_stat s{first, n, 0.0, 0.0, 0.0};   // device times: the slowest device's
   for (int i = 0; i < nd; ++i) {
      if (m.loci_of[i].empty()) continue;
      const sbq_bootstrap_stat& t = m.child[i]->boot.stat;
      s.resample_ms = std::max(s.resample_ms, t.resample_ms);
      s.em_ms = std::max(s.em_ms, t.em_ms);
      s.total_ms = std::max(s.total_ms, t.total_ms);
   }
   c->boot.stat = s;
   c->boot.done = true;
   return SBQ_SUCCESS;
}

// the children's replicate matrices, scattered back into submit order like multi_download
int multi_bootstrap_results(sbq_ctx* c, double* theta, double* tpm, int32_t* iters, int32_t* status) {
   MultiState& m = *c->multi;
   std::lock_guard<std::mutex> lk(c->mu);
   if (!c->boot.done) return fail(c, SBQ_ERR_STATE, "sbq_bootstrap_results before sbq_bootstrap");
   const int64_t n = c->boot.stat.n, NI = c->n_iso, NL = c->n_loci;
   const std::vector<int64_t> lio = multi_offsets(c, 1);
   return multi_for_each(c, [&](int i) {
      sbq_ctx* ch = m.child[i];
      const int64_t ni = ch->n_iso, nl = ch->n_loci;
      std::vector<double> th(theta ? n * ni : 0), tp(tpm ? n * ni : 0);
      std::vector<int32_t> it(iters ? n * nl : 0), stt(status ? n * nl : 0);
      {
         std::lock_guard<std::mutex> lk2(ch->mu);
         const int r = boot_results_locked(ch, theta ? th.data() : nullptr, tpm ? tp.data() : nullptr, iters ? it.data() : nullptr, status ? stt.data() : nullptr);
         if (r) return r;
      }
      for (int64_t b = 0; b < n; ++b) {
         int64_t o = 0;
         for (size_t x = 0; x < m.loci_of[i].size(); ++x) {
            const int32_t l = m.loci_of[i][x];
            const int64_t T = lio[l + 1] - lio[l], d = b * NI + lio[l], s = b * ni + o;
            if (theta) memcpy(theta + d, th.data() + s, T * 8);
            if (tpm) memcpy(tpm + d, tp.data() + s, T * 8);
            if (iters) iters[b * NL + l] = it[b * nl + x];
            if (status) status[b * NL + l] = stt[b * nl + x];
            o += T;
         }
      }
      return 0;
   });
}

int multi_bootstrap_counts(sbq_ctx* c, uint64_t seed, int64_t rep, int32_t* count) {
   MultiState& m = *c->multi;
   std::lock_guard<std::mutex> lk(c->mu);
   if (!c->resident) return fail(c, SBQ_ERR_STATE, "sbq_bootstrap_counts before sbq_upload");
   for (size_t i = 0; i < m.child.size(); ++i) m.child[i]->boot.lid = m.loci_of[i];
   const std::vector<int64_t> lro = multi_offsets(c, 0);
   return multi_for_each(c, [&](int i) {
      sbq_ctx* ch = m.child[i];
      std::vector<int32_t> h((size_t)ch->n_row);
      {
         std::lock_guard<std::mutex> lk2(ch->mu);
         const int r = boot_counts_locked(ch, seed, rep, h.data());
         if (r) return r;
      }
      int64_t o = 0;
      for (size_t x = 0; x < m.loci_of[i].size(); ++x) {
         const int32_t l = m.loci_of[i][x];
         const int64_t R = lro[l + 1] - lro[l];
         memcpy(count + lro[l], h.data() + o, R * 4);
         o += R;
      }
      return 0;
   });
}

// Gibbs samples on N devices, as multi_bootstrap: every child samples its loci under their PARENT submit positions, the n sample
// FPKM sums meet in ONE ncclAllReduce before every device's TPM pass.
int multi_gibbs(sbq_ctx* c, uint64_t seed, int32_t n, int32_t thin, int32_t burn_in, double prior) {
   MultiState& m = *c->multi;
   std::lock_guard<std::mutex> lk(c->mu);
   if (!c->resident || !c->solved) return fail(c, SBQ_ERR_STATE, "sbq_gibbs before sbq_solve");
   c->gibbs.done = false;
   const int nd = (int)m.child.size();
   for (int i = 0; i < nd; ++i) m.child[i]->boot.lid = m.loci_of[i];
   int rc = multi_for_each(c, [&](int i) {
      std::lock_guard<std::mutex> lk2(m.child[i]->mu);
      return gibbs_run_locked(m.child[i], seed, n, thin, burn_in, prior);
   });
   if (rc) return rc;
   for (int i = 0; i < nd; ++i) {   // devices without loci join the all-reduce with zeros
      if (!m.loci_of[i].empty()) continue;
      sbq_ctx* ch = m.child[i];
      CU(cudaSetDevice(m.devices[i]));
      if (!ch->gibbs.sums.reserve((size_t)n * 8)) {
         cudaGetLastError();
         return fail(c, SBQ_ERR_NOMEM, "device %d: allocation failed (Gibbs sums)", m.devices[i]);
      }
      CU(cudaMemsetAsync(ch->gibbs.sums.p, 0, (size_t)n * 8, ch->stream));
   }
   ncclResult_t r = g_nccl.GroupStart();
   for (int i = 0; i < nd && r == ncclSuccess; ++i)
      r = g_nccl.AllReduce(m.child[i]->gibbs.sums.p, m.child[i]->gibbs.sums.p, (size_t)n, ncclDouble, ncclSum, m.comm[i], m.child[i]->stream);
   const ncclResult_t r2 = g_nccl.GroupEnd();
   if (r != ncclSuccess || r2 != ncclSuccess) return fail(c, SBQ_ERR_CUDA, "ncclAllReduce failed: %s", g_nccl.GetErrorString(r != ncclSuccess ? r : r2));
   rc = multi_for_each(c, [&](int i) {
      std::lock_guard<std::mutex> lk2(m.child[i]->mu);
      return gibbs_finish_locked(m.child[i]);
   });
   if (rc) return rc;
   sbq_gibbs_stat s{n, (int64_t)burn_in + (int64_t)n * thin, 0.0, 0.0, 0.0, 0.0};   // device times: the slowest device's
   for (int i = 0; i < nd; ++i) {
      if (m.loci_of[i].empty()) continue;
      const sbq_gibbs_stat& t = m.child[i]->gibbs.stat;
      s.colsum_ms = std::max(s.colsum_ms, t.colsum_ms);
      s.assign_ms = std::max(s.assign_ms, t.assign_ms);
      s.theta_ms = std::max(s.theta_ms, t.theta_ms);
      s.total_ms = std::max(s.total_ms, t.total_ms);
   }
   c->gibbs.stat = s;
   c->gibbs.done = true;
   return SBQ_SUCCESS;
}

// the children's sample matrices, scattered back into submit order like multi_bootstrap_results
int multi_gibbs_results(sbq_ctx* c, double* theta, double* tpm, int32_t* status) {
   MultiState& m = *c->multi;
   std::lock_guard<std::mutex> lk(c->mu);
   if (!c->gibbs.done) return fail(c, SBQ_ERR_STATE, "sbq_gibbs_results before sbq_gibbs");
   const int64_t n = c->gibbs.stat.n, NI = c->n_iso, NL = c->n_loci;
   const std::vector<int64_t> lio = multi_offsets(c, 1);
   return multi_for_each(c, [&](int i) {
      sbq_ctx* ch = m.child[i];
      const int64_t ni = ch->n_iso, nl = ch->n_loci;
      std::vector<double> th(theta ? n * ni : 0), tp(tpm ? n * ni : 0);
      std::vector<int32_t> stt(status ? n * nl : 0);
      {
         std::lock_guard<std::mutex> lk2(ch->mu);
         const int r = gibbs_results_locked(ch, theta ? th.data() : nullptr, tpm ? tp.data() : nullptr, status ? stt.data() : nullptr);
         if (r) return r;
      }
      for (int64_t b = 0; b < n; ++b) {
         int64_t o = 0;
         for (size_t x = 0; x < m.loci_of[i].size(); ++x) {
            const int32_t l = m.loci_of[i][x];
            const int64_t T = lio[l + 1] - lio[l], d = b * NI + lio[l], s = b * ni + o;
            if (theta) memcpy(theta + d, th.data() + s, T * 8);
            if (tpm) memcpy(tpm + d, tp.data() + s, T * 8);
            if (status) status[b * NL + l] = stt[b * nl + x];
            o += T;
         }
      }
      return 0;
   });
}

// aggregate: counts and bytes add up, device times are the slowest device's (the devices run concurrently)
void multi_stats(sbq_ctx* c, sbq_stats* out) {
   MultiState& m = *c->multi;
   sbq_stats a{};
   for (size_t i = 0; i < m.child.size(); ++i) {
      if (m.loci_of[i].empty()) continue;
      sbq_stats s{};
      sbq_get_stats(m.child[i], &s);
      a.n_loci += s.n_loci; a.n_row += s.n_row; a.n_iso += s.n_iso; a.nnz += s.nnz;
      a.loci_warp += s.loci_warp; a.loci_cta += s.loci_cta; a.loci_grid += s.loci_grid;
      a.kernel_launches += s.kernel_launches; a.h2d_bytes += s.h2d_bytes; a.d2h_bytes += s.d2h_bytes;
      a.upload_ms = std::max(a.upload_ms, s.upload_ms); a.solve_ms = std::max(a.solve_ms, s.solve_ms);
      a.download_ms = std::max(a.download_ms, s.download_ms); a.em_ms = std::max(a.em_ms, s.em_ms);
      a.grid_em_ms = std::max(a.grid_em_ms, s.grid_em_ms); a.weights_ms = std::max(a.weights_ms, s.weights_ms);
      a.em_iters_total += s.em_iters_total; a.frag_iters += s.frag_iters; a.alg_bytes += s.alg_bytes; a.grid_alg_bytes += s.grid_alg_bytes;
   }
   *out = a;
}

}  // namespace

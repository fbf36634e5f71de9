// api.cu -- the C ABI of include/maxdecoy.h on top of the CUDA subsystems (digest / index / decoy / score).
#include <algorithm>
#include <cctype>
#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>

#include "cubx.cuh"

namespace {

thread_local std::string g_err;

int fail(md_ctx* ctx, int code, const std::string& msg) {
  if (ctx) ctx->err = msg;
  g_err = msg;
  return code;
}

// run `body`, translating MdError / std exceptions into status codes
template <class F>
int guarded(md_ctx* ctx, F body) {
  try {
    if (ctx) MD_CUDA(cudaSetDevice(ctx->device));
    body();
    return MD_OK;
  } catch (const MdError& e) {
    return fail(ctx, e.code, e.msg);
  } catch (const std::bad_alloc&) {
    return fail(ctx, MD_ERR_NOMEM, "out of host memory");
  } catch (const std::exception& e) {
    return fail(ctx, MD_ERR_INVALID, e.what());
  }
}

// Rust's `as i64` (mass/mod.rs:6-8): saturating, NaN -> 0 (a plain C++ cast would be undefined there)
int64_t sat_i64(double x) {
  if (std::isnan(x)) return 0;
  if (x >= 9223372036854775807.0) return INT64_MAX;
  if (x <= -9223372036854775808.0) return INT64_MIN;
  return (int64_t)x;
}

void host_precursor_window(double mz, uint32_t z, int64_t lppm, int64_t uppm, int64_t* P, int64_t* lo, int64_t* hi) {
  // tasks/identification.rs:203-211; every product/sum rounded on its own (volatile blocks contraction)
  const double H = 1.007276;
  volatile double zc = (double)(uint8_t)z;
  volatile double q = mz / 1000000.0;
  volatile double tl = q * (double)lppm;
  volatile double tu = q * (double)uppm;
  volatile double b = H * zc;
  volatile double a = mz * zc;
  volatile double d0 = a - b;
  *P = sat_i64(d0 * 1000000.0);
  volatile double ml = mz - tl; volatile double al = ml * zc; volatile double dl = al - b;
  *lo = sat_i64(dl * 1000000.0);
  volatile double mu = mz + tu; volatile double au = mu * zc; volatile double du = au - b;
  *hi = sat_i64(du * 1000000.0);
}

template <class T>
T* host_copy(md_ctx* ctx, const T* dev, size_t n) {
  T* h = (T*)malloc((n ? n : 1) * sizeof(T));
  MD_REQUIRE(h != nullptr, MD_ERR_NOMEM, "out of host memory");
  if (n) MD_CUDA(cudaMemcpyAsync(h, dev, n * sizeof(T), cudaMemcpyDeviceToHost, ctx->stream));
  return h;
}

void validate_params(const md_search_params* p) {
  MD_REQUIRE(p->decoy_mode >= 0 && p->decoy_mode <= 2, MD_ERR_INVALID, "md_identify: unknown decoy mode");
  const int64_t w = (int64_t)llround(p->fragment_tolerance * 1000000.0);
  MD_REQUIRE(w >= 100 && w <= 2000000, MD_ERR_INVALID, "md_identify: fragment_tolerance must be in [0.0001, 2] Da");
  MD_REQUIRE(p->top_k <= 128, MD_ERR_INVALID, "md_identify: top_k > 128");
}

float elapsed(cudaEvent_t a, cudaEvent_t b) { float ms = 0; cudaEventElapsedTime(&ms, a, b); return ms; }

// the identification of one batch of spectra that already sits in device memory
void identify_batch(md_ctx* ctx, const SpectraDev& S, uint64_t n_peaks, const md_search_params& p, md_psm* psm_dev, md_identify_stats* st,
                    uint32_t id_base, bool want_all) {
  cudaStream_t s = ctx->stream;
  ctx->marks.clear(); ctx->mark("begin");
  MD_CUDA(cudaEventRecord(ctx->ev[0], s));
  precursors_dev(ctx, S, p, id_base);
  ctx->mark("precursors");
  score_prepare_dev(ctx, S, n_peaks, p);        // (side stream)
  const uint64_t n_targets = index_candidates_dev(ctx, S.n);
  ctx->mark("candidates");
  MD_CUDA(cudaEventRecord(ctx->ev[1], s));
  decoys_generate_dev(ctx, S.n, p.n_decoys, p.decoy_mode, p.seed);
  ctx->mark("decoys");
  MD_CUDA(cudaEventRecord(ctx->ev[2], s));
  score_run_dev(ctx, S, p, p.n_decoys, psm_dev, want_all);
  MD_CUDA(cudaEventRecord(ctx->ev[3], s));
  MD_CUDA(cudaStreamSynchronize(s));
  ctx->mark("score");
  ctx->dump_marks("identify_batch");
  if (st) {
    st->n_spectra += S.n; st->n_targets += n_targets;
    if (p.n_decoys && S.n) {
      std::vector<uint32_t> cnt(S.n);
      MD_CUDA(cudaMemcpy(cnt.data(), ctx->ws.dec_count.p, S.n * sizeof(uint32_t), cudaMemcpyDeviceToHost));
      for (uint32_t c : cnt) { st->n_decoys += c; if (c < p.n_decoys) st->n_less_decoys++; }
    }
    st->ms_lookup += elapsed(ctx->ev[0], ctx->ev[1]); st->ms_decoys += elapsed(ctx->ev[1], ctx->ev[2]);
    st->ms_score += elapsed(ctx->ev[2], ctx->ev[3]); st->ms_total += elapsed(ctx->ev[0], ctx->ev[3]);
  }
}


// Splits a batch into passes the workspaces can hold: the flattened candidate windows of one pass stay below 2^29 index
// entries and its decoy slots below 2^26 (open searches with ~1M candidates per spectrum, or 100k-spectrum files, run
// as several passes; results do not depend on the split).  MD_MAX_PASS_SPECTRA caps the spectra per pass (tests).
std::vector<uint32_t> plan_passes(md_ctx* ctx, const SpectraDev& S, const md_search_params& p) {
  const uint32_t n = S.n;
  IdentifyWorkspace& W = ctx->ws;
  precursors_dev(ctx, S, p, 0);
  W.rbegin.need(n + 1); W.rend.need(n + 1);
  index_window_search_dev(ctx, W.prec.p, n, W.rbegin.p, W.rend.p);
  std::vector<uint64_t> b(n), e(n);
  MD_CUDA(cudaMemcpyAsync(b.data(), W.rbegin.p, n * sizeof(uint64_t), cudaMemcpyDeviceToHost, ctx->stream));
  MD_CUDA(cudaMemcpyAsync(e.data(), W.rend.p, n * sizeof(uint64_t), cudaMemcpyDeviceToHost, ctx->stream));
  MD_CUDA(cudaStreamSynchronize(ctx->stream));
  const uint64_t max_entries = 1ull << 29, max_slots = 1ull << 26;
  uint64_t max_spectra = 0xFFFFFFFFull;
  if (const char* env = getenv("MD_MAX_PASS_SPECTRA")) max_spectra = std::max<long long>(1, atoll(env));
  std::vector<uint32_t> cut{0};
  uint64_t entries = 0, count = 0;
  for (uint32_t s = 0; s < n; s++) {
    const uint64_t sz = e[s] - b[s];
    MD_REQUIRE(sz < max_entries, MD_ERR_UNSUPPORTED, "one spectrum's precursor window spans more than 2^29 index entries");
    if (count && (entries + sz > max_entries || (count + 1) * (uint64_t)p.n_decoys > max_slots || count + 1 > max_spectra)) { cut.push_back(s); entries = 0; count = 0; }
    entries += sz; count++;
  }
  cut.push_back(n);
  return cut;
}

SpectraDev pass_view(const SpectraDev& S, uint32_t a, uint32_t b) {
  return SpectraDev{b - a, S.pmz + a, S.charge + a, S.sid ? S.sid + a : nullptr, S.peak_off + a, S.peak_mz, S.peak_int};
}

}  // namespace
void md_ctx::mark(const char* what) {
  if (!trace) return;
  cudaStreamSynchronize(stream);
  marks.push_back({what, std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count()});
}
void md_ctx::dump_marks(const char* call) {
  if (!trace || marks.empty()) return;
  fprintf(stderr, "[md_trace] %s:", call);
  for (size_t i = 1; i < marks.size(); i++) fprintf(stderr, " %s=%.2fms", marks[i].first, marks[i].second - marks[i - 1].second);
  fprintf(stderr, " total=%.2fms\n", marks.back().second - marks.front().second);
  marks.clear();
}
namespace {
void fill_kernel_stats(md_ctx* ctx, md_identify_stats* st) {
  st->n_kernel_launches = ctx->launches;
  st->ms_kernel_score = ctx->acc_ms_kscore; st->ms_kernel_decoy = ctx->acc_ms_kdecoy;
  st->n_attempts = ctx->acc_attempts; st->n_pairs = ctx->acc_pairs; st->score_bytes = ctx->acc_score_bytes;
  st->ms_score_prepare = ctx->acc_ms_prepare; st->n_score_left = ctx->acc_left; st->score_pipelined = ctx->acc_pipelined;
}

}  // namespace

extern "C" {

const char* md_backend_name(void) { return "cuda-sm100a"; }
void* md_stream_handle(md_ctx* ctx) { return ctx ? (void*)ctx->stream : nullptr; }

int md_create(const md_config* cfg, md_ctx** out) {
  if (!out) return fail(nullptr, MD_ERR_INVALID, "md_create: out is NULL");
  *out = nullptr;
  md_ctx* c = nullptr;
  try {
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0)
      return fail(nullptr, MD_ERR_DEVICE, std::string("md_create: no CUDA device (") + cudaGetErrorString(e) + "); this library has no CPU fallback");
    c = new md_ctx();
    c->device = cfg ? cfg->device : 0;
    MD_REQUIRE(c->device >= 0 && c->device < ndev, MD_ERR_INVALID, "md_create: device ordinal out of range");
    MD_CUDA(cudaSetDevice(c->device));
    cudaDeviceProp prop;
    MD_CUDA(cudaGetDeviceProperties(&prop, c->device));
    MD_REQUIRE(prop.major >= 10, MD_ERR_DEVICE, "md_create: this library is built for sm_100a (Blackwell B200) only");
    c->n_sm = prop.multiProcessorCount;
    c->trace = getenv("MD_TRACE") != nullptr;
    MD_CUDA(cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking));
    MD_CUDA(cudaStreamCreateWithFlags(&c->stream2, cudaStreamNonBlocking));
    MD_CUDA(cudaEventCreateWithFlags(&c->ev_fork, cudaEventDisableTiming));
    MD_CUDA(cudaEventCreateWithFlags(&c->ev_prep, cudaEventDisableTiming));
    MD_CUDA(cudaEventCreate(&c->ev_side0)); MD_CUDA(cudaEventCreate(&c->ev_side1));
    for (auto& ev : c->ev) MD_CUDA(cudaEventCreate(&ev));
    if (c->trace) for (auto& ev : c->ev_trace) MD_CUDA(cudaEventCreate(&ev));
    *out = c;
    return MD_OK;
  } catch (const MdError& e) {
    delete c;
    return fail(nullptr, e.code, e.msg);
  }
}

void md_destroy(md_ctx* ctx) {
  if (!ctx) return;
  cudaSetDevice(ctx->device);
  if (ctx->stream) { cudaStreamSynchronize(ctx->stream); }
  if (ctx->stream2) { cudaStreamSynchronize(ctx->stream2); cudaStreamDestroy(ctx->stream2); }
  if (ctx->ev_fork) cudaEventDestroy(ctx->ev_fork);
  if (ctx->ev_prep) cudaEventDestroy(ctx->ev_prep);
  if (ctx->ev_side0) cudaEventDestroy(ctx->ev_side0);
  if (ctx->ev_side1) cudaEventDestroy(ctx->ev_side1);
  comm_release(ctx);
  for (auto& ev : ctx->ev) if (ev) cudaEventDestroy(ev);
  for (auto& ev : ctx->ev_trace) if (ev) cudaEventDestroy(ev);
  cudaStream_t s = ctx->stream;
  delete ctx;  // frees the device buffers
  if (s) cudaStreamDestroy(s);
}

const char* md_last_error(const md_ctx* ctx) { return ctx ? ctx->err.c_str() : g_err.c_str(); }
void md_free(void* p) { free(p); }
int md_sync(md_ctx* ctx) {
  if (!ctx) return fail(ctx, MD_ERR_INVALID, "md_sync: null ctx");
  return guarded(ctx, [&] { MD_CUDA(cudaStreamSynchronize(ctx->stream)); comm_sync(ctx); });
}

int64_t md_residue_mass(uint8_t c) { return kResidueMassByCode[md_code_of(c)]; }
int64_t md_sequence_weight(const uint8_t* seq, uint32_t len) {
  int64_t w = MD_WATER_UDA;
  for (uint32_t i = 0; i < len; i++) w += kResidueMassByCode[md_code_of(seq[i])];
  return w;
}
int md_precursor_window(double mz, uint32_t charge, int64_t lppm, int64_t uppm, int64_t* P, int64_t* lo, int64_t* hi) {
  if (!P || !lo || !hi || charge == 0 || charge > 255) return fail(nullptr, MD_ERR_INVALID, "md_precursor_window: bad argument");
  host_precursor_window(mz, charge, lppm, uppm, P, lo, hi);
  return MD_OK;
}

int md_set_modifications(md_ctx* ctx, const md_modification* mods, uint32_t n, uint32_t max_var) {
  if (!ctx || (n && !mods)) return fail(ctx, MD_ERR_INVALID, "md_set_modifications: null argument");
  return guarded(ctx, [&] {
    MD_REQUIRE(max_var <= 255, MD_ERR_INVALID, "md_set_modifications: max_variable_mods > 255 (u8 in the reference)");
    ModTables M;
    memset(&M, 0, sizeof(M));
    for (int c = 0; c < MD_NCODES; c++) M.mass[c] = kResidueMassByCode[c];
    M.nvar = max_var; M.var_simple_code = -1;
    for (uint32_t i = 0; i < n; i++) {
      uint8_t pos = (uint8_t)toupper(mods[i].position);
      MD_REQUIRE(pos == 'A' || pos == 'N' || pos == 'C', MD_ERR_INVALID, "modification position must be A, N or C");
      const uint8_t pcode = pos == 'A' ? MD_POS_A : pos == 'N' ? MD_POS_N : MD_POS_C;
      uint8_t aa = (uint8_t)toupper(mods[i].amino_acid);
      uint32_t code = md_code_of(aa);
      MD_REQUIRE(md_alpha_of_code(code) >= 0, MD_ERR_INVALID, "modification on a letter without a <x>_count column (alphabet " MD_ALPHABET ")");
      if (mods[i].is_fix) { M.has_fix[code] = 1; M.fix[code] = mods[i].mono_mass; M.fix_pos[code] = pcode; }
      else { M.has_var[code] = 1; M.var[code] = mods[i].mono_mass; M.var_pos[code] = pcode; }
    }
    for (int c = 0; c < MD_NCODES; c++)
      if ((M.has_fix[c] && M.fix_pos[c] != MD_POS_A) || (M.has_var[c] && M.var_pos[c] != MD_POS_A)) M.has_terminal = 1;
    // sorted modifiable letters (identification.rs:173-178): ascending by character
    int n_var_letters = 0, var_code = -1;
    for (int ch = 'A'; ch <= 'Z'; ch++) {
      uint32_t code = md_code_of((uint8_t)ch);
      if (!M.has_fix[code] && !M.has_var[code]) continue;
      int64_t merged = M.has_var[code] ? M.var[code] : M.fix[code];
      MD_REQUIRE(M.mass[code] + merged > 0, MD_ERR_INVALID, "modified residue mass must be positive");
      MD_REQUIRE(M.mass[code] + (M.has_fix[code] ? M.fix[code] : 0) > 0, MD_ERR_INVALID, "modified residue mass must be positive");
      MD_REQUIRE(M.mass[code] + M.fix[code] + M.var[code] < (1ll << 40), MD_ERR_INVALID, "modification mass too large");
      int k = M.n_letters++;
      M.letter_alpha[k] = md_alpha_of_code(code); M.letter_delta[k] = merged; M.letter_mass[k] = M.mass[code] + merged;
      if (M.has_var[code]) { n_var_letters++; var_code = (int)code; }
    }
    if (n_var_letters == 1 && !M.has_fix[var_code] && !M.has_terminal) M.var_simple_code = var_code;
    ctx->mods = M; ctx->mods_set = true; ctx->index.ready = false; ctx->dindex.ready = false;
  });
}

int md_set_variable_mode(md_ctx* ctx, int mode) {
  if (!ctx) return fail(ctx, MD_ERR_INVALID, "md_set_variable_mode: null ctx");
  if (mode != MD_VARMOD_REFERENCE && mode != MD_VARMOD_EXPANDED) return fail(ctx, MD_ERR_INVALID, "md_set_variable_mode: unknown mode");
  if (mode != ctx->var_mode) { ctx->var_mode = mode; ctx->index.ready = false; ctx->dindex.ready = false; }
  return MD_OK;
}

int md_substitution_map(md_ctx* ctx, int64_t* out) {
  if (!ctx || !out) return fail(ctx, MD_ERR_INVALID, "md_substitution_map: null argument");
  ModTables M = ctx->mods;
  if (!ctx->mods_set) { memset(&M, 0, sizeof(M)); for (int c = 0; c < MD_NCODES; c++) M.mass[c] = kResidueMassByCode[c]; }
  const char* alpha = MD_ALPHABET;
  int64_t mp[MD_ALPHABET_SIZE];
  for (int a = 0; a < MD_ALPHABET_SIZE; a++) { uint32_t c = md_code_of((uint8_t)alpha[a]); mp[a] = M.mass[c] + (M.has_fix[c] ? M.fix[c] : 0); }
  for (int a = 0; a < MD_ALPHABET_SIZE; a++) for (int b = 0; b < MD_ALPHABET_SIZE; b++) out[a * MD_ALPHABET_SIZE + b] = mp[b] - mp[a];
  return MD_OK;
}

int md_digest(md_ctx* ctx, const uint8_t* residues, const uint64_t* off, uint32_t n_prot, const md_digest_params* p, uint64_t* n_out) {
  if (!ctx || !p || (n_prot && (!residues || !off))) return fail(ctx, MD_ERR_INVALID, "md_digest: null argument");
  return guarded(ctx, [&] {
    ctx->reset_counters();
    digest_run(ctx, residues, off, n_prot, *p);
    if (n_out) *n_out = ctx->peps.n;
  });
}

int md_peptides_export(md_ctx* ctx, md_peptide_table* out) {
  if (!ctx || !out) return fail(ctx, MD_ERR_INVALID, "md_peptides_export: null argument");
  return guarded(ctx, [&] { digest_export(ctx, out); });
}
void md_peptide_table_free(md_peptide_table* t) {
  if (!t) return;
  free(t->seq); free(t->seq_off); free(t->missed_cleavages); free(t->weight); free(t->counts); free(t->assoc_off); free(t->assoc_protein);
  memset(t, 0, sizeof(*t));
}

int md_index_build(md_ctx* ctx) {
  if (!ctx) return fail(ctx, MD_ERR_INVALID, "md_index_build: null ctx");
  return guarded(ctx, [&] { ctx->reset_counters(); index_build_run(ctx); });
}

int md_index_stats_get(md_ctx* ctx, md_index_stats* out) {
  if (!ctx || !out) return fail(ctx, MD_ERR_INVALID, "md_index_stats_get: null argument");
  if (!ctx->index.ready) return fail(ctx, MD_ERR_STATE, "md_index_stats_get: md_index_build first");
  memset(out, 0, sizeof(*out));
  const MassIndex& X = ctx->index; const PeptideStore& P = ctx->peps;
  out->n_peptides = X.n; out->seq_bytes = P.seq_bytes; out->min_key = X.min_key; out->max_key = X.max_key;
  out->device_bytes = X.key.bytes() + X.pep.bytes() + X.wfix.bytes() + X.varpos.bytes() + X.desc.bytes() + X.rows.bytes() + P.seq.bytes() + P.seq_off.bytes() +
                      P.len.bytes() + P.mc.bytes() + P.weight.bytes() + P.counts.bytes() + P.hash.bytes() + P.assoc_off.bytes() + P.assoc_protein.bytes() +
                      P.ht_key.bytes() + P.ht_val.bytes();
  return MD_OK;
}

int md_window_search(md_ctx* ctx, const int64_t* lo, const int64_t* hi, uint32_t n, uint64_t* begin, uint64_t* end) {
  if (!ctx || (n && (!lo || !hi || !begin || !end))) return fail(ctx, MD_ERR_INVALID, "md_window_search: null argument");
  if (!ctx->index.ready) return fail(ctx, MD_ERR_STATE, "md_window_search: md_index_build first");
  return guarded(ctx, [&] {
    if (!n) return;
    std::vector<md_precursor> pr(n);
    for (uint32_t i = 0; i < n; i++) { pr[i].mass = 0; pr[i].lo = lo[i]; pr[i].hi = hi[i]; pr[i].charge = 1; pr[i].spectrum_id = i; }
    IdentifyWorkspace& W = ctx->ws;
    W.prec.need(n); W.rbegin.need(n); W.rend.need(n);
    MD_CUDA(cudaMemcpyAsync(W.prec.p, pr.data(), n * sizeof(md_precursor), cudaMemcpyHostToDevice, ctx->stream));
    index_window_search_dev(ctx, W.prec.p, n, W.rbegin.p, W.rend.p);
    MD_CUDA(cudaMemcpyAsync(begin, W.rbegin.p, n * sizeof(uint64_t), cudaMemcpyDeviceToHost, ctx->stream));
    MD_CUDA(cudaMemcpyAsync(end, W.rend.p, n * sizeof(uint64_t), cudaMemcpyDeviceToHost, ctx->stream));
    MD_CUDA(cudaStreamSynchronize(ctx->stream));
  });
}

int md_index_export(md_ctx* ctx, uint64_t begin, uint64_t count, uint64_t* pid, int64_t* key) {
  if (!ctx) return fail(ctx, MD_ERR_INVALID, "md_index_export: null ctx");
  if (!ctx->index.ready) return fail(ctx, MD_ERR_STATE, "md_index_export: md_index_build first");
  if (begin + count > ctx->index.n) return fail(ctx, MD_ERR_INVALID, "md_index_export: range out of bounds");
  return guarded(ctx, [&] {
    if (!count) return;
    if (key) MD_CUDA(cudaMemcpyAsync(key, ctx->index.key.p + begin, count * sizeof(int64_t), cudaMemcpyDeviceToHost, ctx->stream));
    std::vector<uint32_t> pep(count);
    MD_CUDA(cudaMemcpyAsync(pep.data(), ctx->index.pep.p + begin, count * sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx->stream));
    MD_CUDA(cudaStreamSynchronize(ctx->stream));
    if (pid) for (uint64_t i = 0; i < count; i++) pid[i] = (uint64_t)pep[i] + 1;
  });
}

int md_candidates(md_ctx* ctx, const md_precursor* pr, uint32_t n, md_candidate_table* out) {
  if (!ctx || !out || (n && !pr)) return fail(ctx, MD_ERR_INVALID, "md_candidates: null argument");
  if (!ctx->index.ready) return fail(ctx, MD_ERR_STATE, "md_candidates: md_index_build first");
  return guarded(ctx, [&] {
    memset(out, 0, sizeof(*out));
    IdentifyWorkspace& W = ctx->ws;
    W.prec.need(n + 1);
    if (n) MD_CUDA(cudaMemcpyAsync(W.prec.p, pr, n * sizeof(md_precursor), cudaMemcpyHostToDevice, ctx->stream));
    const uint64_t total = index_candidates_dev(ctx, n);
    out->n_spectra = n; out->n = total;
    if (n) out->off = host_copy(ctx, W.cand_off.p, n + 1);
    else { out->off = (uint64_t*)calloc(1, sizeof(uint64_t)); }
    out->var_mask = host_copy(ctx, W.cand_mask.p, total);
    out->mod_weight = host_copy(ctx, W.cand_w.p, total);
    uint32_t* pep = host_copy(ctx, W.cand_pep.p, total);
    MD_CUDA(cudaStreamSynchronize(ctx->stream));
    out->peptide_id = (uint64_t*)malloc((total + 1) * sizeof(uint64_t));
    for (uint64_t i = 0; i < total; i++) out->peptide_id[i] = (uint64_t)pep[i] + 1;
    free(pep);
  });
}
void md_candidate_table_free(md_candidate_table* t) {
  if (!t) return;
  free(t->off); free(t->peptide_id); free(t->var_mask); free(t->mod_weight);
  memset(t, 0, sizeof(*t));
}

// Stored decoys (the `decoys` table): validated, deduplicated and put into canonical order (weight, sequence hash, sequence)
// on the host -- a one-time upload, not on the hot path -- then laid out like the peptide store so that the same index
// build, window search and filter kernels serve it.
int md_decoy_store_set(md_ctx* ctx, const uint8_t* seq, const uint64_t* off, uint64_t n) {
  if (!ctx || (n && (!seq || !off))) return fail(ctx, MD_ERR_INVALID, "md_decoy_store_set: null argument");
  return guarded(ctx, [&] {
    struct E { int64_t w; uint64_t h; uint64_t o; uint32_t len; };
    std::vector<E> v; v.reserve(n);
    for (uint64_t i = 0; i < n; i++) {
      MD_REQUIRE(off[i + 1] >= off[i], MD_ERR_INVALID, "md_decoy_store_set: offsets not monotone");
      const uint64_t L = off[i + 1] - off[i];
      MD_REQUIRE(L >= 1 && L <= MD_MAX_PEPTIDE_LEN, MD_ERR_INVALID, "md_decoy_store_set: sequence length must be 1..60");
      int64_t w = MD_WATER_UDA; uint64_t h = md_hash_init();
      for (uint64_t k = 0; k < L; k++) {
        const uint8_t c = seq[off[i] + k];
        MD_REQUIRE(md_alpha_of_code(md_code_of(c)) >= 0, MD_ERR_INVALID, "md_decoy_store_set: letter outside the decoy alphabet " MD_ALPHABET);
        w += kResidueMassByCode[md_code_of(c)]; h = md_hash_step(h, c);
      }
      v.push_back({w, md_hash_fin(h, (uint32_t)L), off[i], (uint32_t)L});
    }
    auto cmp_seq = [&](const E& a, const E& b) {
      const int c = memcmp(seq + a.o, seq + b.o, std::min(a.len, b.len));
      return c != 0 ? c : (int)a.len - (int)b.len;
    };
    std::sort(v.begin(), v.end(), [&](const E& a, const E& b) { return a.w != b.w ? a.w < b.w : a.h != b.h ? a.h < b.h : cmp_seq(a, b) < 0; });
    std::vector<uint8_t> h_seq, h_len; std::vector<uint32_t> h_off{0}; std::vector<int64_t> h_w; std::vector<int16_t> h_cnt; std::vector<uint64_t> h_hash;
    for (size_t i = 0; i < v.size(); i++) {
      if (i && v[i].len == v[i - 1].len && memcmp(seq + v[i].o, seq + v[i - 1].o, v[i].len) == 0) continue;   // UNIQUE (aa_sequence, weight)
      int16_t cnt[MD_ALPHABET_SIZE] = {};
      for (uint32_t k = 0; k < v[i].len; k++) { const uint8_t c = seq[v[i].o + k]; h_seq.push_back(c); cnt[md_alpha_of_code(md_code_of(c))]++; }
      h_off.push_back((uint32_t)h_seq.size()); h_len.push_back((uint8_t)v[i].len); h_w.push_back(v[i].w); h_hash.push_back(v[i].h);
      h_cnt.insert(h_cnt.end(), cnt, cnt + MD_ALPHABET_SIZE);
    }
    PeptideStore& D = ctx->dstore;
    D.ready = false; ctx->dindex.ready = false;
    const size_t m = h_len.size();
    D.n = m; D.seq_bytes = h_seq.size(); D.n_assoc = 0;
    if (m) {
      D.seq.need(h_seq.size() + 1); D.seq_off.need(m + 1); D.len.need(m); D.mc.need(m); D.weight.need(m); D.counts.need(m * MD_ALPHABET_SIZE); D.hash.need(m);
      MD_CUDA(cudaMemcpyAsync(D.seq.p, h_seq.data(), h_seq.size(), cudaMemcpyHostToDevice, ctx->stream));
      MD_CUDA(cudaMemcpyAsync(D.seq_off.p, h_off.data(), (m + 1) * sizeof(uint32_t), cudaMemcpyHostToDevice, ctx->stream));
      MD_CUDA(cudaMemcpyAsync(D.len.p, h_len.data(), m, cudaMemcpyHostToDevice, ctx->stream));
      MD_CUDA(cudaMemsetAsync(D.mc.p, 0, m, ctx->stream));
      MD_CUDA(cudaMemcpyAsync(D.weight.p, h_w.data(), m * sizeof(int64_t), cudaMemcpyHostToDevice, ctx->stream));
      MD_CUDA(cudaMemcpyAsync(D.counts.p, h_cnt.data(), m * MD_ALPHABET_SIZE * sizeof(int16_t), cudaMemcpyHostToDevice, ctx->stream));
      MD_CUDA(cudaMemcpyAsync(D.hash.p, h_hash.data(), m * sizeof(uint64_t), cudaMemcpyHostToDevice, ctx->stream));
      MD_CUDA(cudaStreamSynchronize(ctx->stream));
      D.ready = true;
    }
    if (ctx->index.ready) index_build_store(ctx);
  });
}

int md_generate_decoys(md_ctx* ctx, const md_precursor* pr, uint32_t n_spec, uint32_t n_per, int mode, uint64_t seed, md_decoy_table* out) {
  if (!ctx || !out || (n_spec && !pr)) return fail(ctx, MD_ERR_INVALID, "md_generate_decoys: null argument");
  if (!ctx->index.ready) return fail(ctx, MD_ERR_STATE, "md_generate_decoys: md_index_build first");
  if (mode < 0 || mode > 2) return fail(ctx, MD_ERR_INVALID, "md_generate_decoys: unknown mode");
  return guarded(ctx, [&] {
    IdentifyWorkspace& W = ctx->ws;
    ctx->reset_counters();
    W.prec.need(n_spec + 1);
    if (n_spec) MD_CUDA(cudaMemcpyAsync(W.prec.p, pr, n_spec * sizeof(md_precursor), cudaMemcpyHostToDevice, ctx->stream));
    if (mode == MD_DECOY_PERMUTE_TARGET) index_candidates_dev(ctx, n_spec);
    decoys_generate_dev(ctx, n_spec, n_per, mode, seed);
    decoys_export(ctx, n_spec, n_per, out);
  });
}
void md_decoy_table_free(md_decoy_table* t) {
  if (!t) return;
  free(t->off); free(t->seq); free(t->seq_off); free(t->var_mask); free(t->weight); free(t->mod_weight); free(t->attempt);
  memset(t, 0, sizeof(*t));
}

int md_identify_device(md_ctx* ctx, const md_spectra* S, const md_search_params* p, md_psm* psms_dev, md_identify_stats* stats) {
  if (!ctx || !S || !p || (S->n && p->top_k && !psms_dev)) return fail(ctx, MD_ERR_INVALID, "md_identify_device: null argument");
  if (!ctx->index.ready) return fail(ctx, MD_ERR_STATE, "md_identify_device: md_index_build first");
  if (S->n && (!S->precursor_mz || !S->charge || !S->peak_off)) return fail(ctx, MD_ERR_INVALID, "spectra: null array");
  return guarded(ctx, [&] {
    validate_params(p);
    if (stats) memset(stats, 0, sizeof(*stats));
    ctx->reset_counters(); ctx->last.have = false;
    if (!S->n) return;
    comm_wait_for_buffer(ctx, psms_dev);
    // (the caller's buffers must be complete when the call is made: work on other streams is the caller's to wait for)
    uint64_t n_peaks = 0;
    MD_CUDA(cudaMemcpyAsync(&n_peaks, (const uint64_t*)S->peak_off + S->n, sizeof(uint64_t), cudaMemcpyDeviceToHost, ctx->stream));
    MD_CUDA(cudaStreamSynchronize(ctx->stream));
    MD_REQUIRE(S->n == 0 || n_peaks < (1ull << 40), MD_ERR_INVALID, "spectra: peak_off[n] is not a plausible peak count");
    SpectraDev D{S->n, S->precursor_mz, S->charge, S->spectrum_id, S->peak_off, S->peak_mz, S->peak_intensity};
    const std::vector<uint32_t> cut = plan_passes(ctx, D, *p);
    MD_REQUIRE(cut.size() == 2 || !p->keep_decoys, MD_ERR_UNSUPPORTED, "keep_decoys needs a batch that fits one pass");
    for (size_t k = 0; k + 1 < cut.size(); k++)
      identify_batch(ctx, pass_view(D, cut[k], cut[k + 1]), n_peaks, *p, psms_dev + (size_t)cut[k] * p->top_k, stats, cut[k], false);
    if (stats) fill_kernel_stats(ctx, stats);
  });
}

int md_identify(md_ctx* ctx, const md_spectra* S, const md_search_params* p, md_psm* psms, md_identify_stats* stats, int64_t** all_scores, uint64_t** all_off) {
  if (!ctx || !S || !p || (S->n && p->top_k && !psms)) return fail(ctx, MD_ERR_INVALID, "md_identify: null argument");
  if (!ctx->index.ready) return fail(ctx, MD_ERR_STATE, "md_identify: md_index_build first");
  if (S->n && (!S->precursor_mz || !S->charge || !S->peak_off)) return fail(ctx, MD_ERR_INVALID, "spectra: null array");
  return guarded(ctx, [&] {
    validate_params(p);
    if (stats) memset(stats, 0, sizeof(*stats));
    if (all_scores) *all_scores = nullptr;
    if (all_off) *all_off = nullptr;
    ctx->reset_counters(); ctx->last.have = false;
    const uint32_t n = S->n;
    for (uint32_t s = 0; s < n; s++) {
      MD_REQUIRE(S->peak_off[s + 1] >= S->peak_off[s], MD_ERR_INVALID, "spectra: peak_off not monotone");
      MD_REQUIRE(S->charge[s] != 0, MD_ERR_INVALID, "spectra: charge 0");
      MD_REQUIRE(std::isfinite(S->precursor_mz[s]) && S->precursor_mz[s] > 0.0 && S->precursor_mz[s] < 1.0e7, MD_ERR_INVALID, "spectra: precursor m/z must be finite and in (0, 1e7)");
    }
    if (!n) { if (all_scores && all_off) { *all_scores = (int64_t*)calloc(1, 8); *all_off = (uint64_t*)calloc(1, 8); } return; }
    IdentifyWorkspace& W = ctx->ws;
    cudaStream_t st = ctx->stream;
    const uint64_t np = S->peak_off[n] - S->peak_off[0];
    MD_REQUIRE(S->peak_off[0] == 0, MD_ERR_INVALID, "spectra: peak_off[0] must be 0");
    W.pmz.need(n); W.charge.need(n); W.sid.need(n); W.peak_off.need(n + 1); W.peak_mz.need(np + 1); W.peak_int.need(np + 1);
    W.psm.need((size_t)n * p->top_k + 1);
    MD_CUDA(cudaMemcpyAsync(W.pmz.p, S->precursor_mz, n * sizeof(double), cudaMemcpyHostToDevice, st));
    MD_CUDA(cudaMemcpyAsync(W.charge.p, S->charge, n, cudaMemcpyHostToDevice, st));
    if (S->spectrum_id) MD_CUDA(cudaMemcpyAsync(W.sid.p, S->spectrum_id, n * sizeof(uint32_t), cudaMemcpyHostToDevice, st));
    MD_CUDA(cudaMemcpyAsync(W.peak_off.p, S->peak_off, (n + 1) * sizeof(uint64_t), cudaMemcpyHostToDevice, st));
    if (np) {
      MD_CUDA(cudaMemcpyAsync(W.peak_mz.p, S->peak_mz, np * sizeof(double), cudaMemcpyHostToDevice, st));
      MD_CUDA(cudaMemcpyAsync(W.peak_int.p, S->peak_intensity, np * sizeof(float), cudaMemcpyHostToDevice, st));
    }
    SpectraDev D{n, W.pmz.p, W.charge.p, S->spectrum_id ? W.sid.p : nullptr, W.peak_off.p, W.peak_mz.p, W.peak_int.p};
    const bool want_all = all_scores && all_off;
    const std::vector<uint32_t> cut = plan_passes(ctx, D, *p);
    MD_REQUIRE(cut.size() == 2 || !p->keep_decoys, MD_ERR_UNSUPPORTED, "keep_decoys needs a batch that fits one pass");
    std::vector<int64_t> flat; std::vector<uint64_t> foff(1, 0);
    for (size_t k = 0; k + 1 < cut.size(); k++) {
      const uint32_t a = cut[k], m = cut[k + 1] - cut[k];
      identify_batch(ctx, pass_view(D, a, a + m), np, *p, W.psm.p + (size_t)a * p->top_k, stats, a, want_all);
      if (want_all) {  // raw scores of this pass: targets in index order, then decoys
        std::vector<uint64_t> coff(m + 1); std::vector<uint32_t> dcnt(m, 0);
        MD_CUDA(cudaMemcpy(coff.data(), W.cand_off.p, (m + 1) * sizeof(uint64_t), cudaMemcpyDeviceToHost));
        if (p->n_decoys) MD_CUDA(cudaMemcpy(dcnt.data(), W.dec_count.p, m * sizeof(uint32_t), cudaMemcpyDeviceToHost));
        std::vector<int64_t> ts(coff[m] + 1), ds((size_t)m * p->n_decoys + 1);
        if (coff[m]) MD_CUDA(cudaMemcpy(ts.data(), W.tscore.p, coff[m] * sizeof(int64_t), cudaMemcpyDeviceToHost));
        if ((size_t)m * p->n_decoys) MD_CUDA(cudaMemcpy(ds.data(), W.dscore.p, (size_t)m * p->n_decoys * sizeof(int64_t), cudaMemcpyDeviceToHost));
        for (uint32_t s = 0; s < m; s++) {
          for (uint64_t c = coff[s]; c < coff[s + 1]; c++) flat.push_back(ts[c]);
          for (uint32_t j = 0; j < dcnt[s]; j++) flat.push_back(ds[(size_t)s * p->n_decoys + j]);
          foff.push_back(flat.size());
        }
      }
    }
    if (p->top_k) MD_CUDA(cudaMemcpyAsync(psms, W.psm.p, (size_t)n * p->top_k * sizeof(md_psm), cudaMemcpyDeviceToHost, st));
    MD_CUDA(cudaStreamSynchronize(st));
    if (stats) fill_kernel_stats(ctx, stats);
    if (want_all) {
      int64_t* out_scores = (int64_t*)malloc((flat.size() + 1) * sizeof(int64_t)); uint64_t* out_off = (uint64_t*)malloc((n + 1) * sizeof(uint64_t));
      MD_REQUIRE(out_scores && out_off, MD_ERR_NOMEM, "out of host memory");
      if (!flat.empty()) memcpy(out_scores, flat.data(), flat.size() * sizeof(int64_t));
      memcpy(out_off, foff.data(), (n + 1) * sizeof(uint64_t));
      *all_scores = out_scores; *all_off = out_off;
    }
    if (p->keep_decoys) {
      LastDecoys& L = ctx->last;
      L.n_spectra = n; L.n_per = p->n_decoys; L.have = true;
    }
  });
}

int md_last_decoys_export(md_ctx* ctx, md_decoy_table* out) {
  if (!ctx || !out) return fail(ctx, MD_ERR_INVALID, "md_last_decoys_export: null argument");
  if (!ctx->last.have) return fail(ctx, MD_ERR_STATE, "md_last_decoys_export: no identify call with keep_decoys");
  return guarded(ctx, [&] { decoys_export(ctx, ctx->last.n_spectra, ctx->last.n_per, out); });
}

}  // extern "C"

// index.cu -- K2: the mass-sorted in-HBM peptide index and the candidate lookup.
//
// Replaces the per-spectrum SQL fan-out of identification_task (tasks/identification.rs:24,180-188,
// 214-241,374-403; models/persistable.rs:251-267): every enumerated query
//   weight BETWEEN lo - sum k_a d_a AND hi - sum k_a d_a AND a_count = k_a ...
// retrieves exactly the peptides with lo <= W* <= hi, W* = weight + sum_a count_a * d_a, so one radix
// sort by W* and one window search per spectrum serve all of them.  The ModifiedPeptide filter
// (identification.rs:242-257) then runs on the window's entries, one thread per entry.
#include "cubx.cuh"
#include "modpep.cuh"
#include "decoyutil.cuh"

namespace {

inline uint32_t blocks(uint64_t n, uint32_t bs = 256) { return (uint32_t)((n + bs - 1) / bs); }

__global__ void k_index_keys(const int64_t* __restrict__ weight, const int16_t* __restrict__ counts, uint32_t n, const __grid_constant__ ModTables M,
                             int64_t* __restrict__ key, uint32_t* __restrict__ ord) {
  uint32_t p = blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= n) return;
  int64_t k = weight[p];
  for (int i = 0; i < M.n_letters; i++) k += (int64_t)counts[(size_t)p * MD_ALPHABET_SIZE + M.letter_alpha[i]] * M.letter_delta[i];
  key[p] = k;
  ord[p] = p;
}

// per index entry: weight with fixed mods, mask of variable-modifiable positions, padded row length
__global__ void k_index_entries(const uint32_t* __restrict__ pep, uint32_t n, const uint8_t* __restrict__ seq, const uint32_t* __restrict__ seq_off,
                                const uint8_t* __restrict__ len, const int64_t* __restrict__ weight, const __grid_constant__ ModTables M, int64_t* __restrict__ wfix,
                                uint64_t* __restrict__ varpos, uint32_t* __restrict__ row16) {
  uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i > n) return;
  if (i == n) { row16[i] = 0; return; }
  uint32_t p = pep[i];
  const uint8_t* s = seq + seq_off[p];
  uint32_t L = len[p];
  int64_t w = weight[p];
  uint64_t vp = 0;
  for (uint32_t k = 0; k < L; k++) {
    uint32_t c = md_code_of(s[k]);
    if (md_fix_applies(M, c, k, L)) w += M.fix[c];
    if (M.has_var[c]) vp |= 1ULL << k;
  }
  wfix[i] = w; varpos[i] = vp;
  row16[i] = (L + 15) >> 4;
}

__global__ void k_index_rows(const uint32_t* __restrict__ pep, uint32_t n, const uint8_t* __restrict__ seq, const uint32_t* __restrict__ seq_off,
                             const uint8_t* __restrict__ len, const uint32_t* __restrict__ row_off16, uint8_t* __restrict__ rows, uint64_t* __restrict__ desc) {
  uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  uint32_t p = pep[i];
  const uint8_t* s = seq + seq_off[p];
  uint32_t L = len[p];
  uint8_t* d = rows + (size_t)row_off16[i] * 16;
  uint32_t padded = ((L + 15) >> 4) << 4;
  for (uint32_t k = 0; k < padded; k++) d[k] = k < L ? (uint8_t)md_code_of(s[k]) : (uint8_t)MD_CODE_OTHER;
  desc[i] = (uint64_t)row_off16[i] | ((uint64_t)L << 40);
}

// Warp-cooperative 32-ary search: first index in [0,n) whose key is >= target (UPPER: > target).
template <bool UPPER>
__device__ uint64_t warp_bound(const int64_t* __restrict__ key, uint64_t n, int64_t target, uint32_t lane) {
  uint64_t lo = 0, hi = n;  // answer in [lo, hi]; everything below lo is "false", hi (if < n) is "true"
  while (hi - lo > 32) {
    uint64_t stride = (hi - lo + 31) / 32;
    uint64_t pos = lo + (uint64_t)(lane + 1) * stride - 1;
    bool valid = pos < hi;
    int64_t v = valid ? key[pos] : 0;
    bool t = valid ? (UPPER ? v > target : v >= target) : true;
    uint32_t b = __ballot_sync(0xffffffffu, t);
    if (b == 0) return hi;                           // every probe is "false": the answer is the upper end
    uint32_t f = __ffs(b) - 1;
    uint64_t new_lo = lo + (uint64_t)f * stride;
    uint64_t new_hi = lo + (uint64_t)(f + 1) * stride - 1;
    lo = new_lo;
    hi = new_hi < hi ? new_hi : hi;
  }
  uint64_t pos = lo + lane;
  bool valid = pos < hi;
  int64_t v = valid ? key[pos] : 0;
  bool t = valid ? (UPPER ? v > target : v >= target) : true;
  uint32_t b = __ballot_sync(0xffffffffu, t);
  if (b == 0) return hi;
  uint32_t f = __ffs(b) - 1;
  uint64_t ans = lo + f;
  return ans < hi ? ans : hi;
}

// one warp per precursor: [begin, end) = { i : lo <= W*[i] <= hi }
// per index entry: the peptide's counts of the modifiable letters (what the filter's fan-out test reads), in index order
__global__ void k_index_letter_counts(const uint32_t* __restrict__ pep, uint32_t n, const int16_t* __restrict__ counts, const __grid_constant__ ModTables M,
                                      int16_t* __restrict__ lcnt) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const uint32_t p = pep[i];
  for (int k = 0; k < M.n_letters; k++) lcnt[(uint64_t)i * M.n_letters + k] = counts[(size_t)p * MD_ALPHABET_SIZE + M.letter_alpha[k]];
}

__global__ void k_window_search(const int64_t* __restrict__ key, uint64_t n, const md_precursor* __restrict__ prec, uint32_t n_prec,
                                uint64_t* __restrict__ begin, uint64_t* __restrict__ end) {
  uint32_t warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (warp >= n_prec) return;
  int64_t lo = prec[warp].lo, hi = prec[warp].hi;
  uint64_t b = warp_bound<false>(key, n, lo, lane);
  uint64_t e = warp_bound<true>(key, n, hi, lane);
  if (e < b) e = b;
  if (lane == 0) { begin[warp] = b; end[warp] = e; }
}

__global__ void k_range_sizes(const uint64_t* __restrict__ b, const uint64_t* __restrict__ e, uint32_t n, uint64_t* __restrict__ size) {
  uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i > n) return;
  size[i] = i < n ? e[i] - b[i] : 0;
}

// identification.rs:214-222: K_a = (P / (m_a + d_a)) as i16, one per (spectrum, modifiable letter)
__global__ void k_spectrum_limits(const md_precursor* __restrict__ prec, uint32_t n, const __grid_constant__ ModTables M, int16_t* __restrict__ K) {
  uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n * (uint32_t)MD_ALPHABET_SIZE) return;
  uint32_t s = t / MD_ALPHABET_SIZE, i = t % MD_ALPHABET_SIZE;
  int16_t k = 0;
  if ((int)i < M.n_letters) k = (int16_t)(prec[s].mass / M.letter_mass[i]);
  K[t] = k;
}

struct RowSeq {
  const uint8_t* r;
  __device__ __forceinline__ uint32_t operator()(uint32_t i) const { return r[i]; }
};

// The ModifiedPeptide filter for every entry of every window (identification.rs:231-257,374-403).
__global__ void k_filter(const uint64_t* __restrict__ flat_off, const uint64_t* __restrict__ rbegin, const md_precursor* __restrict__ prec, uint32_t n_spec,
                         uint64_t n_entries, const uint32_t* __restrict__ idx_pep, const int64_t* __restrict__ idx_wfix, const uint64_t* __restrict__ idx_varpos,
                         const uint64_t* __restrict__ idx_desc, const uint8_t* __restrict__ rows, const int16_t* __restrict__ lcnt,
                         const int16_t* __restrict__ specK, const __grid_constant__ ModTables M, uint32_t* __restrict__ flag, uint64_t* __restrict__ emask,
                         int64_t* __restrict__ ew, int* __restrict__ overflow) {
  uint64_t e = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= n_entries) return;
  // spectrum of this entry: last s with flat_off[s] <= e
  uint32_t lo = 0, hi = n_spec;
  while (hi - lo > 1) { uint32_t mid = (lo + hi) >> 1; if (flat_off[mid] <= e) lo = mid; else hi = mid; }
  const uint32_t s = lo;
  const uint64_t i = rbegin[s] + (e - flat_off[s]);
  const md_precursor pr = prec[s];
  (void)idx_pep;
  bool ok = M.n_letters > 0;  // no modifiable letter -> the recursion emits no query (identification.rs:375-379)
  int64_t cur_lo = pr.lo;
  for (int k = 0; k < M.n_letters && ok; k++) {
    int16_t c = lcnt[i * (uint64_t)M.n_letters + k];         // the peptide's count of the k-th modifiable letter, in index order (k_index_letter_counts)
    if (!(c < specK[s * MD_ALPHABET_SIZE + k])) ok = false;   // 0..max_modification_count (exclusive, :381)
    if (!(cur_lo > 0)) ok = false;                           // :387
    cur_lo -= (int64_t)c * M.letter_delta[k];
  }
  int64_t w = idx_wfix[i];
  uint64_t mask = 0;
  if (ok) {
    if (!md_in_window(w, pr.lo, pr.hi)) {                    // :246-249
      uint64_t d = idx_desc[i];
      RowSeq seq{rows + (d & 0xFFFFFFFFFFull) * 16};
      (void)idx_varpos;
      ok = md_try_variable(M, seq, (uint32_t)(d >> 40) & 0xFF, w, mask, pr.lo, pr.hi, overflow);
    }
  }
  flag[e] = ok ? 1u : 0u;
  if (emask) { emask[e] = mask; ew[e] = w; }     // (NULL: no variable modification is configured, an accepted entry is (0, wfix))
}

__global__ void k_scatter_candidates(const uint64_t* __restrict__ flat_off, const uint64_t* __restrict__ rbegin, uint32_t n_spec, uint64_t n_entries,
                                     const uint32_t* __restrict__ flag, const uint32_t* __restrict__ pos, const uint64_t* __restrict__ emask,
                                     const int64_t* __restrict__ ew, const uint32_t* __restrict__ idx_pep, const uint64_t* __restrict__ idx_desc,
                                     const int64_t* __restrict__ idx_wfix, uint64_t* __restrict__ cand_desc, uint64_t* __restrict__ cand_mask,
                                     int64_t* __restrict__ cand_w, uint32_t* __restrict__ cand_pep) {
  uint64_t e = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= n_entries || !flag[e]) return;
  uint32_t lo = 0, hi = n_spec;
  while (hi - lo > 1) { uint32_t mid = (lo + hi) >> 1; if (flat_off[mid] <= e) lo = mid; else hi = mid; }
  const uint64_t i = rbegin[lo] + (e - flat_off[lo]);
  uint32_t o = pos[e];
  cand_desc[o] = idx_desc[i]; cand_mask[o] = emask ? emask[e] : 0ull; cand_w[o] = emask ? ew[e] : idx_wfix[i]; cand_pep[o] = idx_pep[i];
}

// accepted window entries of the decoy store -> the first decoy slots of their spectrum (rank within the spectrum < n_per)
__global__ void k_scatter_stored_decoys(const uint64_t* __restrict__ flat_off, const uint64_t* __restrict__ rbegin, uint32_t n_spec, uint64_t n_entries,
                                        const uint32_t* __restrict__ flag, const uint32_t* __restrict__ pos, const uint64_t* __restrict__ emask,
                                        const int64_t* __restrict__ ew, const uint32_t* __restrict__ idx_pep, const uint64_t* __restrict__ idx_desc,
                                        const uint8_t* __restrict__ rows, const uint64_t* __restrict__ store_hash, uint32_t n_per, DecoyOut D) {
  uint64_t e = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= n_entries || !flag[e]) return;
  uint32_t lo = 0, hi = n_spec;
  while (hi - lo > 1) { uint32_t mid = (lo + hi) >> 1; if (flat_off[mid] <= e) lo = mid; else hi = mid; }
  const uint32_t s = lo;
  const uint32_t rank = pos[e] - pos[flat_off[s]];
  if (rank >= n_per) return;
  const uint64_t i = rbegin[s] + (e - flat_off[s]);
  const uint64_t d = idx_desc[i];
  const uint8_t* src = rows + (d & 0xFFFFFFFFFFull) * 16;
  const uint32_t L = (uint32_t)(d >> 40) & 0xFF;
  const uint64_t slot = (uint64_t)s * n_per + rank;
  for (uint32_t k = 0; k < MD_DECOY_ROW; k++) D.rows[md_dec_byte(D.n_slots, slot, k)] = k < L ? src[k] : (uint8_t)MD_CODE_OTHER;
  D.len[slot] = (uint8_t)L; D.mask[slot] = emask[e]; D.w[slot] = ew[e]; D.hash[slot] = store_hash[idx_pep[i]];
  D.attempt[slot] = MD_DECOY_STORED;
}

__global__ void k_stored_counts(const uint64_t* __restrict__ flat_off, const uint32_t* __restrict__ pos, uint32_t n_spec, uint32_t n_per,
                                uint32_t* __restrict__ dec_count) {
  uint32_t s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= n_spec) return;
  dec_count[s] = min(n_per, pos[flat_off[s + 1]] - pos[flat_off[s]]);
}

// ------------------------------------------------------------------------------------------------
// MD_VARMOD_EXPANDED: every placement of up to nvar variable modifications is a candidate of its own
// ------------------------------------------------------------------------------------------------
constexpr int kMaxVarLetters = 6, kMaxVarCombos = 96;
struct VarCombos {
  int n_letters, n_combos;
  uint8_t code[kMaxVarLetters];              // residue codes of the variable-modifiable letters, ascending
  uint8_t pos[kMaxVarLetters];               // where the letter's variable modification can sit (MD_POS_A / _N / _C)
  int64_t delta[kMaxVarLetters];
  uint8_t k[kMaxVarCombos][kMaxVarLetters];  // count vectors, sum <= nvar
  int64_t shift[kMaxVarCombos];              // sum k_a * delta_a
};

__global__ void k_iota(uint32_t* __restrict__ v, uint32_t n) { uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; if (i < n) v[i] = i; }

// window (s, q) on the fixed-modification weight: [lo - shift_q, hi - shift_q]
__global__ void k_shifted_windows(const md_precursor* __restrict__ prec, uint32_t n, const __grid_constant__ VarCombos V, md_precursor* __restrict__ out) {
  uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n * (uint32_t)V.n_combos) return;
  const uint32_t s = t / V.n_combos, q = t % V.n_combos;
  md_precursor p = prec[s];
  p.lo -= V.shift[q]; p.hi -= V.shift[q];
  out[t] = p;
}

__device__ __forceinline__ uint64_t binom_capped(uint32_t n, uint32_t k) {   // C(n, k), n <= 60; capped at 2^32
  if (k > n) return 0;
  uint64_t r = 1;
  for (uint32_t i = 1; i <= k; i++) { r = r * (n - k + i) / i; if (r > 0xFFFFFFFFull) return 0x100000000ull; }
  return r;
}

// placements of window entry e: prod_a C(count_a, k_a)
__global__ void k_expand_count(const uint64_t* __restrict__ flat_off, const uint64_t* __restrict__ rbegin, uint32_t n_win, uint64_t n_entries,
                               const uint32_t* __restrict__ fent, const uint64_t* __restrict__ idx_desc, const uint8_t* __restrict__ rows,
                               const __grid_constant__ VarCombos V, uint32_t* __restrict__ count, int* __restrict__ overflow) {
  uint64_t e = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= n_entries) return;
  uint32_t lo = 0, hi = n_win;
  while (hi - lo > 1) { uint32_t mid = (lo + hi) >> 1; if (flat_off[mid] <= e) lo = mid; else hi = mid; }
  const uint32_t q = lo % V.n_combos;
  const uint32_t ent = fent[rbegin[lo] + (e - flat_off[lo])];
  const uint64_t d = idx_desc[ent];
  const uint8_t* r = rows + (d & 0xFFFFFFFFFFull) * 16;
  const uint32_t L = (uint32_t)(d >> 40) & 0xFF;
  uint64_t total = 1;
  for (int a = 0; a < V.n_letters; a++) {
    uint32_t c = 0;
    for (uint32_t i = 0; i < L; i++) c += r[i] == V.code[a] && md_pos_at(V.pos[a], i, L);
    total *= binom_capped(c, V.k[q][a]);
    if (total > 0xFFFFFull) { *overflow = 1; total = 0; break; }   // more than 2^20 placements of one peptide
  }
  count[e] = (uint32_t)total;
}

// the count-th .. placements of entry e, odometer over the letters (last letter fastest), each letter's subsets in NChooseK order
__global__ void k_expand_scatter(const uint64_t* __restrict__ flat_off, const uint64_t* __restrict__ rbegin, uint32_t n_win, uint64_t n_entries,
                                 const uint32_t* __restrict__ count, const uint32_t* __restrict__ pos, const uint32_t* __restrict__ fent,
                                 const int64_t* __restrict__ fkey, const uint32_t* __restrict__ idx_pep, const uint64_t* __restrict__ idx_desc,
                                 const uint8_t* __restrict__ rows, const __grid_constant__ VarCombos V, uint64_t* __restrict__ cand_desc,
                                 uint64_t* __restrict__ cand_mask, int64_t* __restrict__ cand_w, uint32_t* __restrict__ cand_pep) {
  uint64_t e = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= n_entries || !count[e]) return;
  uint32_t lo = 0, hi = n_win;
  while (hi - lo > 1) { uint32_t mid = (lo + hi) >> 1; if (flat_off[mid] <= e) lo = mid; else hi = mid; }
  const uint32_t q = lo % V.n_combos;
  const uint64_t fi = rbegin[lo] + (e - flat_off[lo]);
  const uint32_t ent = fent[fi];
  const uint64_t d = idx_desc[ent];
  const uint8_t* r = rows + (d & 0xFFFFFFFFFFull) * 16;
  const uint32_t L = (uint32_t)(d >> 40) & 0xFF;
  const int64_t w = fkey[fi] + V.shift[q];
  const uint32_t pep = idx_pep[ent];
  uint64_t allpos[kMaxVarLetters], cm[kMaxVarLetters], first[kMaxVarLetters];
  uint32_t dcount[kMaxVarLetters];
  for (int a = 0; a < V.n_letters; a++) {
    uint64_t m = 0;
    for (uint32_t i = 0; i < L; i++) if (r[i] == V.code[a] && md_pos_at(V.pos[a], i, L)) m |= 1ULL << i;
    allpos[a] = m; dcount[a] = (uint32_t)__popcll(m);
    const uint32_t k = V.k[q][a];
    first[a] = k == 0 ? 0ULL : (((1ULL << dcount[a]) - 1) ^ ((1ULL << (dcount[a] - k)) - 1));   // 2^d - 2^(d-k)
    cm[a] = first[a];
  }
  uint32_t o = pos[e];
  for (uint32_t j = 0; j < count[e]; j++, o++) {
    uint64_t mask = 0;
    for (int a = 0; a < V.n_letters; a++) {
      // compressed bit (d-1-b) <-> b-th position (ascending) of allpos
      uint64_t rest = allpos[a];
      for (uint32_t b = 0; b < dcount[a]; b++) {
        const uint64_t bit = rest & (~rest + 1); rest &= rest - 1;
        if ((cm[a] >> (dcount[a] - 1 - b)) & 1) mask |= bit;
      }
    }
    cand_desc[o] = d; cand_mask[o] = mask; cand_w[o] = w; cand_pep[o] = pep;
    // next placement
    for (int a = V.n_letters - 1; a >= 0; a--) {
      if (V.k[q][a] == 0) continue;
      const uint64_t nx = md_prev_combination(cm[a]);
      if (nx) { cm[a] = nx; break; }
      cm[a] = first[a];
    }
  }
}

__global__ void k_cand_offsets_expanded(const uint64_t* __restrict__ flat_off, const uint32_t* __restrict__ pos, uint32_t n_spec, uint32_t n_combos,
                                        uint64_t* __restrict__ cand_off) {
  uint32_t s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s > n_spec) return;
  cand_off[s] = pos[flat_off[(uint64_t)s * n_combos]];
}

__global__ void k_cand_offsets(const uint64_t* __restrict__ flat_off, const uint32_t* __restrict__ pos, uint32_t n_spec, uint64_t* __restrict__ cand_off) {
  uint32_t s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s > n_spec) return;
  cand_off[s] = pos[flat_off[s]];  // pos has n_entries+1 elements (exclusive scan incl. the total)
}

}  // namespace

static void index_build_for(md_ctx* ctx, PeptideStore& P, MassIndex& X) {
  X.ready = false;
  const uint32_t n = (uint32_t)P.n;
  X.n = n; X.row_bytes = 0; X.min_key = X.max_key = 0;
  if (n == 0) { X.key.need(1); X.ready = true; return; }
  DevBuf<int64_t> d_key; DevBuf<uint32_t> d_ord, d_row16, d_rowoff;
  d_key.need(n); d_ord.need(n); d_row16.need(n + 1); d_rowoff.need(n + 1);
  X.key.need(n); X.pep.need(n); X.wfix.need(n); X.varpos.need(n); X.desc.need(n);
  MD_LAUNCH(ctx, k_index_keys, blocks(n), 256, 0, P.weight.p, P.counts.p, n, ctx->mods, d_key.p, d_ord.p);
  cubx_sort_pairs(ctx, d_key.p, X.key.p, d_ord.p, X.pep.p, n);  // stable: ties keep canonical peptide order
  MD_LAUNCH(ctx, k_index_entries, blocks(n + 1), 256, 0, X.pep.p, n, P.seq.p, P.seq_off.p, P.len.p, P.weight.p, ctx->mods, X.wfix.p, X.varpos.p, d_row16.p);
  cubx_exclusive_sum(ctx, d_row16.p, d_rowoff.p, n + 1);
  const uint32_t total16 = d2h_scalar(ctx, d_rowoff.p + n);
  X.row_bytes = (uint64_t)total16 * 16;
  X.rows.need(X.row_bytes + 64);
  MD_LAUNCH(ctx, k_index_rows, blocks(n), 256, 0, X.pep.p, n, P.seq.p, P.seq_off.p, P.len.p, d_rowoff.p, X.rows.p, X.desc.p);
  X.lcnt.need((size_t)n * std::max(1, ctx->mods.n_letters));
  MD_LAUNCH(ctx, k_index_letter_counts, blocks(n), 256, 0, X.pep.p, n, P.counts.p, ctx->mods, X.lcnt.p);
  int64_t mm[2];
  MD_CUDA(cudaMemcpyAsync(&mm[0], X.key.p, sizeof(int64_t), cudaMemcpyDeviceToHost, ctx->stream));
  MD_CUDA(cudaMemcpyAsync(&mm[1], X.key.p + (n - 1), sizeof(int64_t), cudaMemcpyDeviceToHost, ctx->stream));
  MD_CUDA(cudaStreamSynchronize(ctx->stream));
  X.min_key = mm[0]; X.max_key = mm[1];
  if (ctx->var_mode == MD_VARMOD_EXPANDED && &X == &ctx->index) {   // second order of the same entries: by fixed-modification weight
    DevBuf<uint32_t> d_iota; d_iota.need(n);
    X.fkey.need(n); X.fent.need(n);
    MD_LAUNCH(ctx, k_iota, blocks(n), 256, 0, d_iota.p, n);
    cubx_sort_pairs(ctx, X.wfix.p, X.fkey.p, d_iota.p, X.fent.p, n);  // stable: ties keep index order
    MD_CUDA(cudaStreamSynchronize(ctx->stream));
  }
  X.ready = true;
}

void index_build_run(md_ctx* ctx) {
  MD_REQUIRE(ctx->peps.ready, MD_ERR_STATE, "md_index_build: md_digest first");
  MD_REQUIRE(ctx->mods_set, MD_ERR_STATE, "md_index_build: md_set_modifications first");
  index_build_for(ctx, ctx->peps, ctx->index);
  index_build_store(ctx);
}

void index_build_store(md_ctx* ctx) {
  ctx->dindex.ready = false;
  if (!ctx->dstore.ready || !ctx->mods_set) return;
  index_build_for(ctx, ctx->dstore, ctx->dindex);
}

void index_window_search_dev(md_ctx* ctx, const md_precursor* prec_dev, uint32_t n, uint64_t* begin_dev, uint64_t* end_dev) {
  if (!n) return;
  MD_LAUNCH(ctx, k_window_search, blocks((uint64_t)n * 32, 128), 128, 0, ctx->index.key.p, ctx->index.n, prec_dev, n, begin_dev, end_dev);
}

// Window search + ModifiedPeptide filter of the n precursors in ws.prec against one index: leaves the flattened windows
// (ws.rbegin, ws.flat_off), the per-entry results (t_flag, emask, ew) and the exclusive scan of the flags (t_pos, E+1
// entries) in the workspace; returns the number of window entries E and the number of accepted ones.
static uint64_t filter_windows(md_ctx* ctx, const MassIndex& X, uint32_t n, uint32_t* total_out, bool* lean_io = nullptr) {
  IdentifyWorkspace& W = ctx->ws;
  W.rbegin.need(n + 1); W.rend.need(n + 1); W.flat_off.need(n + 2);
  MD_LAUNCH(ctx, k_window_search, blocks((uint64_t)n * 32, 128), 128, 0, X.key.p, X.n, W.prec.p, n, W.rbegin.p, W.rend.p);
  ctx->mark("  window_search");
  DevBuf<uint64_t>& d_size = W.t_size; d_size.need(n + 1);
  MD_LAUNCH(ctx, k_range_sizes, blocks(n + 1), 256, 0, W.rbegin.p, W.rend.p, n, d_size.p);
  cubx_exclusive_sum(ctx, d_size.p, W.flat_off.p, n + 1);
  const uint64_t E = d2h_scalar(ctx, W.flat_off.p + n);
  MD_REQUIRE(E < 0x7FFFFF00ull, MD_ERR_UNSUPPORTED, "candidate windows of one batch exceed 2^31 index entries; use smaller batches");
  DevBuf<int16_t>& d_K = W.t_K; d_K.need((size_t)n * MD_ALPHABET_SIZE);
  MD_LAUNCH(ctx, k_spectrum_limits, blocks((uint64_t)n * MD_ALPHABET_SIZE), 256, 0, W.prec.p, n, ctx->mods, d_K.p);
  DevBuf<uint32_t>& d_flag = W.t_flag; DevBuf<uint32_t>& d_pos = W.t_pos; DevBuf<int>& d_ovf = W.t_ovf;
  d_flag.need(E + 1); d_pos.need(E + 1); d_ovf.need(1);
  // lean: the caller takes (0, wfix) for an accepted entry when no variable modification can apply (md_try_variable then never
  // changes an entry), and the per-entry mask / weight are neither written nor read
  bool any_var = false;
  for (int c = 0; c < MD_NCODES; c++) any_var |= ctx->mods.has_var[c] != 0;
  const bool lean = lean_io && *lean_io && (ctx->mods.nvar == 0 || !any_var);
  if (lean_io) *lean_io = lean;
  if (!lean) { W.emask.need(E + 1); W.ew.need(E + 1); }
  MD_CUDA(cudaMemsetAsync(d_ovf.p, 0, sizeof(int), ctx->stream));
  MD_CUDA(cudaMemsetAsync(d_flag.p + E, 0, sizeof(uint32_t), ctx->stream));
  ctx->mark("  alloc");
  if (E) {
    MD_LAUNCH(ctx, k_filter, blocks(E), 256, 0, W.flat_off.p, W.rbegin.p, W.prec.p, n, E, X.pep.p, X.wfix.p, X.varpos.p, X.desc.p, X.rows.p,
              X.lcnt.p, d_K.p, ctx->mods, d_flag.p, lean ? nullptr : W.emask.p, lean ? nullptr : W.ew.p, d_ovf.p);
  }
  ctx->mark("  filter");
  cubx_exclusive_sum(ctx, d_flag.p, d_pos.p, E + 1);
  *total_out = d2h_scalar(ctx, d_pos.p + E);
  const int ovf = d2h_scalar(ctx, d_ovf.p);
  MD_REQUIRE(!ovf, MD_ERR_UNSUPPORTED, "variable-modification placement enumeration exceeds 2^22 subsets for one peptide");
  return E;
}

// MD_VARMOD_EXPANDED: for every count vector (k_a) over the variable letters, the window [lo - sum k_a d_a, hi - sum k_a d_a]
// on the fixed-modification weight; every entry with count_a >= k_a contributes prod_a C(count_a, k_a) placements.
static uint64_t candidates_expanded_dev(md_ctx* ctx, uint32_t n) {
  IdentifyWorkspace& W = ctx->ws; MassIndex& X = ctx->index; const ModTables& M = ctx->mods;
  VarCombos V;
  memset(&V, 0, sizeof(V));
  for (int ch = 'A'; ch <= 'Z'; ch++) {
    const uint32_t code = md_code_of((uint8_t)ch);
    if (!M.has_var[code] || (M.has_fix[code] && M.fix_pos[code] == M.var_pos[code])) continue;   // (its slot holds the fixed modification)
    MD_REQUIRE(V.n_letters < kMaxVarLetters, MD_ERR_UNSUPPORTED, "expanded variable-modification mode: more than 6 variable letters");
    V.code[V.n_letters] = (uint8_t)code; V.pos[V.n_letters] = M.var_pos[code]; V.delta[V.n_letters] = M.var[code]; V.n_letters++;
  }
  {  // count vectors in ascending mixed-radix order, last letter fastest
    std::vector<uint8_t> k(kMaxVarLetters, 0);
    for (;;) {
      uint32_t sum = 0; int64_t sh = 0;
      for (int a = 0; a < V.n_letters; a++) { sum += k[a]; sh += (int64_t)k[a] * V.delta[a]; }
      if (sum <= M.nvar) {
        MD_REQUIRE(V.n_combos < kMaxVarCombos, MD_ERR_UNSUPPORTED, "expanded variable-modification mode: more than 96 count vectors");
        for (int a = 0; a < V.n_letters; a++) V.k[V.n_combos][a] = k[a];
        V.shift[V.n_combos++] = sh;
      }
      int a = V.n_letters - 1;
      while (a >= 0 && k[a] >= M.nvar) { k[a] = 0; a--; }
      if (a < 0) break;
      k[a]++;
    }
  }
  const uint32_t Q = (uint32_t)V.n_combos, nw = n * Q;
  MD_REQUIRE((uint64_t)n * Q < 0x7FFFFFFFull, MD_ERR_UNSUPPORTED, "expanded variable-modification mode: too many windows in one batch");
  W.rbegin.need(nw + 1); W.rend.need(nw + 1); W.flat_off.need(nw + 2); W.cand_off.need(n + 2);
  DevBuf<md_precursor>& d_win = W.t_win; d_win.need(nw + 1);
  MD_LAUNCH(ctx, k_shifted_windows, blocks(nw), 256, 0, W.prec.p, n, V, d_win.p);
  MD_LAUNCH(ctx, k_window_search, blocks((uint64_t)nw * 32, 128), 128, 0, X.fkey.p, X.n, d_win.p, nw, W.rbegin.p, W.rend.p);
  DevBuf<uint64_t>& d_size = W.t_size; d_size.need(nw + 1);
  MD_LAUNCH(ctx, k_range_sizes, blocks(nw + 1), 256, 0, W.rbegin.p, W.rend.p, nw, d_size.p);
  cubx_exclusive_sum(ctx, d_size.p, W.flat_off.p, nw + 1);
  const uint64_t E = d2h_scalar(ctx, W.flat_off.p + nw);
  MD_REQUIRE(E < 0x7FFFFF00ull, MD_ERR_UNSUPPORTED, "candidate windows of one batch exceed 2^31 index entries; use smaller batches");
  DevBuf<uint32_t>& d_cnt = W.t_flag; DevBuf<uint32_t>& d_pos = W.t_pos; DevBuf<int>& d_ovf = W.t_ovf;
  d_cnt.need(E + 1); d_pos.need(E + 1); d_ovf.need(1);
  MD_CUDA(cudaMemsetAsync(d_ovf.p, 0, sizeof(int), ctx->stream));
  MD_CUDA(cudaMemsetAsync(d_cnt.p + E, 0, sizeof(uint32_t), ctx->stream));
  if (E) MD_LAUNCH(ctx, k_expand_count, blocks(E), 256, 0, W.flat_off.p, W.rbegin.p, nw, E, X.fent.p, X.desc.p, X.rows.p, V, d_cnt.p, d_ovf.p);
  cubx_exclusive_sum(ctx, d_cnt.p, d_pos.p, E + 1);
  const uint32_t total = d2h_scalar(ctx, d_pos.p + E);
  const int ovf = d2h_scalar(ctx, d_ovf.p);
  MD_REQUIRE(!ovf, MD_ERR_UNSUPPORTED, "expanded variable-modification mode: more than 2^20 placements for one peptide");
  MD_REQUIRE(total < 0x7FFFFF00u, MD_ERR_UNSUPPORTED, "expanded variable-modification mode: more than 2^31 candidates in one batch");
  W.cand_desc.need(total + 1); W.cand_mask.need(total + 1); W.cand_w.need(total + 1); W.cand_pep.need(total + 1);
  if (E) MD_LAUNCH(ctx, k_expand_scatter, blocks(E), 256, 0, W.flat_off.p, W.rbegin.p, nw, E, d_cnt.p, d_pos.p, X.fent.p, X.fkey.p, X.pep.p, X.desc.p, X.rows.p, V,
                   W.cand_desc.p, W.cand_mask.p, W.cand_w.p, W.cand_pep.p);
  MD_LAUNCH(ctx, k_cand_offsets_expanded, blocks(n + 1), 256, 0, W.flat_off.p, d_pos.p, n, Q, W.cand_off.p);
  ctx->mark("  expanded");
  return total;
}

uint64_t index_candidates_dev(md_ctx* ctx, uint32_t n) {
  IdentifyWorkspace& W = ctx->ws; MassIndex& X = ctx->index;
  W.rbegin.need(n + 1); W.rend.need(n + 1); W.flat_off.need(n + 2); W.cand_off.need(n + 2);
  if (!n) return 0;
  if (ctx->var_mode == MD_VARMOD_EXPANDED) return candidates_expanded_dev(ctx, n);
  uint32_t total = 0;
  bool lean = true;
  const uint64_t E = filter_windows(ctx, X, n, &total, &lean);
  W.cand_desc.need(total + 1); W.cand_mask.need(total + 1); W.cand_w.need(total + 1); W.cand_pep.need(total + 1);
  if (E) {
    MD_LAUNCH(ctx, k_scatter_candidates, blocks(E), 256, 0, W.flat_off.p, W.rbegin.p, n, E, W.t_flag.p, W.t_pos.p, lean ? nullptr : W.emask.p, lean ? nullptr : W.ew.p,
              X.pep.p, X.desc.p, X.wfix.p, W.cand_desc.p, W.cand_mask.p, W.cand_w.p, W.cand_pep.p);
  }
  MD_LAUNCH(ctx, k_cand_offsets, blocks(n + 1), 256, 0, W.flat_off.p, W.t_pos.p, n, W.cand_off.p);
  ctx->mark("  scatter");
  return total;
}

// Decoy reuse (tasks/identification.rs:259-283): the stored decoys of each precursor's window that pass the filter, in
// store-index order, become the first decoys of the spectrum.
void decoys_reuse_dev(md_ctx* ctx, uint32_t n, uint32_t n_per) {
  IdentifyWorkspace& W = ctx->ws; MassIndex& X = ctx->dindex;
  if (!n || !n_per || !X.ready || X.n == 0) return;
  uint32_t total = 0;
  const uint64_t E = filter_windows(ctx, X, n, &total);
  if (E) {
    const DecoyOut D{W.dec_rows.p, W.dec_len.p, W.dec_mask.p, W.dec_w.p, W.dec_hash.p, W.dec_attempt.p, W.dec_count.p, (uint64_t)n * n_per};
    MD_LAUNCH(ctx, k_scatter_stored_decoys, blocks(E), 256, 0, W.flat_off.p, W.rbegin.p, n, E, W.t_flag.p, W.t_pos.p, W.emask.p, W.ew.p, X.pep.p, X.desc.p,
              X.rows.p, ctx->dstore.hash.p, n_per, D);
  }
  MD_LAUNCH(ctx, k_stored_counts, blocks(n), 256, 0, W.flat_off.p, W.t_pos.p, n, n_per, W.dec_count.p);
  ctx->mark("  reuse");
}

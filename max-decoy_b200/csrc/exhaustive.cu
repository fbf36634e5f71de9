// exhaustive.cu -- MD_DECOY_EXHAUSTIVE: every sequence whose (fixed-modification) weight lies in the precursor window, in a
// canonical order, until n_per decoys are found.  Builder-defined mode named by the north star ("decoys in
// exhaustive-enumeration mode, bit-exact"); the definition is the oracle's (oracle/maxdecoy_oracle.cpp, decoys_exhaustive):
//   compositions = count vectors (c_A, c_R, ..., c_Y) over MD_ALPHABET with H2O + sum c_a * (mass_a + fixed_a) in [lo, hi]
//   and 1 <= length <= 60, in ascending lexicographic order; per composition its distinct permutations in ascending
//   lexicographic order of alphabet indices; sequences that are peptides of the index are skipped (Decoy::is_peptide,
//   models/peptides/decoy.rs:49-60) but counted in the ordinal that is reported as `attempt`.
// One thread walks one spectrum: a depth-first search over the count vector (the last letter's count follows from the
// remainder by one division) and std::next_permutation's algorithm inside each composition.  The order is inherently
// sequential per spectrum; spectra are independent, so a batch fills the GPU.  The walk is bounded by kMaxSteps search
// steps per spectrum (reported as MD_ERR_UNSUPPORTED, never silently truncated).
#include "cubx.cuh"
#include "decoyutil.cuh"

namespace {

constexpr unsigned long long kMaxSteps = 1ull << 28;

struct ExTables {
  int64_t m[MD_ALPHABET_SIZE];        // mass + fixed delta by alphabet index
  uint8_t code_of_a[MD_ALPHABET_SIZE];
};

__global__ void __launch_bounds__(64) k_decoy_exhaustive(const md_precursor* __restrict__ prec, uint32_t n_spec, uint32_t n_per,
                                                         const __grid_constant__ ExTables T, PeptideView PV, DecoyOut O, int* __restrict__ too_large) {
  const uint32_t s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= n_spec) return;
  const md_precursor pr = prec[s];
  const uint64_t dbase = (uint64_t)s * n_per;
  uint32_t found = 0, ordinal = 0;
  unsigned long long steps = 0;
  const int64_t LO = pr.lo - MD_WATER_UDA, HI = pr.hi - MD_WATER_UDA;   // window for the residue sum
  constexpr int NL = MD_ALPHABET_SIZE, LAST = MD_ALPHABET_SIZE - 1;
  uint8_t cnt[NL]; int64_t psum[NL]; uint32_t plen[NL];                  // psum/plen = sums over the letters before a
  uint8_t cur[MD_MAX_PEPTIDE_LEN]; uint8_t ascii[MD_MAX_PEPTIDE_LEN];
  for (int a = 0; a < NL; a++) { cnt[a] = 0; psum[a] = 0; plen[a] = 0; }
  if (n_per == 0 || HI < 0) { O.count[s] = 0; return; }
  int a = 0;
  bool done = false;
  while (!done) {
    if (++steps > kMaxSteps) { *too_large = 1; break; }
    if (a < LAST) {
      const int64_t used = (int64_t)cnt[a] * T.m[a];
      if (plen[a] + cnt[a] > MD_MAX_PEPTIDE_LEN || psum[a] + used > HI) {
        // level a is exhausted: back to the previous letter, next count
        cnt[a] = 0;
        if (a == 0) break;
        a--; cnt[a]++;
        continue;
      }
      psum[a + 1] = psum[a] + used; plen[a + 1] = plen[a] + cnt[a];
      a++; cnt[a] = 0;
      continue;
    }
    // last letter: its count follows from the remainder
    {
      const int64_t rlo = LO - psum[LAST], rhi = HI - psum[LAST], ma = T.m[LAST];
      const int64_t kmin = rlo <= 0 ? 0 : (rlo + ma - 1) / ma, kmax = rhi / ma;
      for (int64_t k = kmin; k <= kmax && plen[LAST] + k <= MD_MAX_PEPTIDE_LEN && !done; k++) {
        const uint32_t L = plen[LAST] + (uint32_t)k;
        if (L == 0) continue;
        cnt[LAST] = (uint8_t)k;
        // first permutation: the multiset in ascending order
        uint32_t q = 0; int64_t w = MD_WATER_UDA;
        for (int b = 0; b < NL; b++) for (uint32_t c = 0; c < cnt[b]; c++) { cur[q++] = (uint8_t)b; w += T.m[b]; }
        for (;;) {
          if (++steps > kMaxSteps) { *too_large = 1; done = true; break; }
          uint64_t h = md_hash_init();
          for (uint32_t i = 0; i < L; i++) { ascii[i] = md_letter_of(T.code_of_a[cur[i]]); h = md_hash_step(h, ascii[i]); }
          h = md_hash_fin(h, L);
          const uint32_t ord = ordinal++;
          if (!is_peptide(ascii, L, h, PV.ht_key, PV.ht_val, PV.ht_mask, PV.seq, PV.off, PV.len)) {
            const uint64_t slot = dbase + found;
            for (uint32_t i = 0; i < MD_DECOY_ROW; i++) O.rows[md_dec_byte(O.n_slots, slot, i)] = i < L ? T.code_of_a[cur[i]] : (uint8_t)MD_CODE_OTHER;
            O.len[slot] = (uint8_t)L; O.mask[slot] = 0; O.w[slot] = w; O.hash[slot] = h; O.attempt[slot] = ord;
            if (++found >= n_per) { done = true; break; }
          }
          // std::next_permutation
          int i = (int)L - 2;
          while (i >= 0 && cur[i] >= cur[i + 1]) i--;
          if (i < 0) break;
          int j = (int)L - 1;
          while (cur[j] <= cur[i]) j--;
          uint8_t t = cur[i]; cur[i] = cur[j]; cur[j] = t;
          for (int x = i + 1, y = (int)L - 1; x < y; x++, y--) { t = cur[x]; cur[x] = cur[y]; cur[y] = t; }
        }
      }
      cnt[LAST] = 0;
      if (done) break;
      // back to the previous letter, next count
      a = LAST - 1; cnt[a]++;
    }
  }
  O.count[s] = found;
}

}  // namespace

void decoys_exhaustive_dev(md_ctx* ctx, uint32_t n, uint32_t n_per) {
  IdentifyWorkspace& W = ctx->ws; PeptideStore& P = ctx->peps;
  ExTables T;
  const char* alpha = MD_ALPHABET;
  for (int a = 0; a < MD_ALPHABET_SIZE; a++) {
    const uint32_t code = md_code_of((uint8_t)alpha[a]);
    T.code_of_a[a] = (uint8_t)code;
    T.m[a] = ctx->mods.mass[code] + (ctx->mods.has_fix[code] ? ctx->mods.fix[code] : 0);
    MD_REQUIRE(T.m[a] > 0, MD_ERR_INVALID, "exhaustive decoys need positive residue masses");
  }
  PeptideView PV{(const unsigned long long*)P.ht_key.p, P.ht_val.p, P.ht_mask, P.seq.p, P.seq_off.p, P.len.p};
  DecoyOut O{W.dec_rows.p, W.dec_len.p, W.dec_mask.p, W.dec_w.p, W.dec_hash.p, W.dec_attempt.p, W.dec_count.p, (uint64_t)n * n_per};
  DevBuf<int>& flag = W.t_ovf; flag.need(1);
  MD_CUDA(cudaMemsetAsync(flag.p, 0, sizeof(int), ctx->stream));
  MD_CUDA(cudaEventRecord(ctx->ev[4], ctx->stream));
  MD_LAUNCH(ctx, k_decoy_exhaustive, (n + 63) / 64, 64, 0, W.prec.p, n, n_per, T, PV, O, flag.p);
  MD_CUDA(cudaEventRecord(ctx->ev[5], ctx->stream));
  const int too_large = d2h_scalar(ctx, flag.p);
  { float ms = 0; cudaEventElapsedTime(&ms, ctx->ev[4], ctx->ev[5]); ctx->acc_ms_kdecoy += ms; }
  MD_REQUIRE(!too_large, MD_ERR_UNSUPPORTED, "exhaustive decoy enumeration exceeds 2^28 search steps for one spectrum");
}

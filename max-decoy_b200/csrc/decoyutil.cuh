// decoyutil.cuh -- device helpers shared by the decoy kernels (decoy.cu, exhaustive.cu).
#pragma once
#include "common.cuh"

#include <type_traits>

struct PeptideView {
  const unsigned long long* ht_key; const uint32_t* ht_val; uint32_t ht_mask;
  const uint8_t* seq; const uint32_t* off; const uint8_t* len;
};

// Decoy::is_peptide (decoy.rs:49-60): exact membership in the peptide table; `ascii` = the letters, or a function i -> letter i
template <class Ascii>
__device__ inline bool is_peptide(Ascii ascii, uint32_t len, uint64_t h, const unsigned long long* __restrict__ ht_key,
                           const uint32_t* __restrict__ ht_val, uint32_t ht_mask, const uint8_t* __restrict__ pep_seq,
                           const uint32_t* __restrict__ pep_off, const uint8_t* __restrict__ pep_len) {
  auto letter = [&](uint32_t i) -> uint8_t { if constexpr (std::is_pointer<Ascii>::value) return ascii[i]; else return ascii(i); };
  if (h == 0) h = 1;
  uint32_t slot = (uint32_t)h & ht_mask;
  for (;;) {
    unsigned long long k = ht_key[slot];
    if (k == 0ULL) return false;
    if (k == h) {
      uint32_t p = ht_val[slot];
      if (pep_len[p] == len) {
        const uint8_t* s = pep_seq + pep_off[p];
        bool eq = true;
        for (uint32_t i = 0; i < len; i++) if (s[i] != letter(i)) { eq = false; break; }
        if (eq) return true;
      }
    }
    slot = (slot + 1) & ht_mask;
  }
}


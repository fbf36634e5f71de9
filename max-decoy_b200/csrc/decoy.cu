// decoy.cu -- K3: mass-constrained decoy generation on the GPU.
//
// REFERENCE_RANDOM restates DecoyGenerator::generate_decoys' worker loop (utility/decoy_generator.rs:127-188)
// and ModifiedPeptide::swap_amino_acids_to_hit_mass_tolerance (models/peptides/modified_peptide.rs:451-508):
// grow a random sequence until its weight exceeds the upper limit, then repair it by greedy single-residue
// substitutions (<= 100 passes, one random kick per pass), testing the window / variable modifications after
// every applied substitution.  One GPU lane runs one attempt at a time and fetches the next attempt from a
// global queue the moment it finishes, so lanes never idle behind a slow neighbour.  Attempts are keyed by
// (seed, spectrum_id, attempt) through a Philox counter RNG, so the decoys of a spectrum are the first n distinct
// non-peptide successes in attempt order, independent of scheduling, batching and sharding.
// PERMUTE_TARGET restates DecoyGenerator::vary_targets (decoy_generator.rs:265-296).
#include "cubx.cuh"
#include "modpep.cuh"
#include "decoyutil.cuh"

#include <algorithm>

namespace {

inline uint32_t blocks(uint64_t n, uint32_t bs = 256) { return (uint32_t)((n + bs - 1) / bs); }

constexpr int kThreads = 128;          // lanes per CTA of the attempt kernels
// MD_ROUND_ATTEMPTS and MD_SELECT_SMEM_MAX (test builds only) shrink the list entries and the hash selection's shared-memory
// budget, so that small inputs run several levels per round and reach k_decoy_select's exact route
#ifndef MD_ROUND_ATTEMPTS
#define MD_ROUND_ATTEMPTS 4096
#endif
#ifndef MD_SELECT_SMEM_MAX
#define MD_SELECT_SMEM_MAX (220 * 1024)
#endif
constexpr int kMaxRoundAttempts = MD_ROUND_ATTEMPTS;  // per list entry (bounds the selection kernel's shared memory)
static_assert(kMaxRoundAttempts >= 1 && kMaxRoundAttempts <= 8192, "k_decoy_select keeps one thread's share of an entry in a 32-bit mask");
constexpr int kRoundLevels = 4;          // list entries one spectrum can have in a round: its attempts in consecutive chunks, selected one after the other

// letter tables in alphabet-index space, built once per call on the host
constexpr uint32_t kGapTab = 512, kNnTab = 1024;
struct DecoyTables {
  int64_t mprime[32];      // residue mass + fixed delta, by alphabet index (0..20)
  uint8_t code_of_a[32];   // residue code of alphabet index
  int64_t var_a[32];
  // improving-substitution filter: letter a has a substitution that strictly reduces |d| iff its gap to the next lighter
  // (d > 0) / heavier (d < 0) distinct mass is < 2|d|.  Gaps sorted ascending + the letter set of every prefix.
  uint32_t gapb_sorted[32], gapa_sorted[32];   // padded with 0xFFFFFFFF
  uint32_t maskb_prefix[33], maska_prefix[33];
  // bucket tables that replace the binary searches of the repair loop (a short residual scan finishes each lookup):
  // gap_tab[sign][min(x >> gap_shift, kGapTab-1)] = number of sorted gaps below the bucket's first x
  uint8_t gap_tab[2][kGapTab];
  uint32_t gap_shift;
  // nearest (mass + fixed delta) to a target t: distinct masses u[0..n), letter of each (lowest alphabet index of an
  // equal-mass run), thresholds in doubled space thr2[j] between u[j] and u[j+1] (ties to the lower alphabet index):
  // nearest = #{j : 2t > thr2[j]}; nn_tab[(clamp(t) - nn_lo) >> nn_shift] = that count at the bucket's first t
  uint8_t nn_tab[kNnTab];
  int32_t nn_thr2[32];        // padded with INT32_MAX
  uint8_t nn_letter[32];
  int32_t nn_lo, nn_hi;
  uint32_t nn_shift;
};

struct TSeq {  // a lane's working sequence in shared memory (alphabet indices), transposed for conflict-free access
  uint8_t* base;
  __device__ __forceinline__ uint8_t& at(uint32_t i) const { return base[i * kThreads]; }
  __device__ __forceinline__ uint32_t get(uint32_t i) const { return base[i * kThreads]; }
};
// k_decoy_random's sequences, word-interleaved: one 32-bit word holds four consecutive positions of one lane, position i of
// lane l at byte ((i >> 2) * kThreads + l) * 4 + (i & 3).  Lanes never share a bank whatever position each accesses (the
// transposed byte layout put lanes 4k..4k+3 in one bank), and the sequence moves to and from its row (alphabet indices,
// four positions per little-endian word) in whole words.  Accessed through an explicit 32-bit shared-memory address `a` =
// array + 4 * lane; the byte offset of position i is IMAD + LOP3: i * 129 = (i << 7) | i for i < 128, and the mask keeps
// (i >> 2) << 9 and i & 3; it is added to `a`, not OR-ed, as the array's shared address need not be a multiple of its size.
// All accesses are volatile asm: ordered among themselves, invisible to the compiler's alias analysis -- the array must not
// be touched through C++ pointers as well.
constexpr uint32_t kSeqWordStride = kThreads * 4u;     // bytes between the words of one lane
static_assert(kSeqWordStride == 512u, "SSeq::addr builds (i >> 2) * kSeqWordStride by masking i * 129");
struct SSeq {
  uint32_t a;
  __device__ __forceinline__ uint32_t addr(uint32_t i) const { return ((i * 129u) & ~0x1FCu) + a; }
  __device__ __forceinline__ uint32_t get(uint32_t i) const {
    uint32_t v; asm volatile("ld.shared.u8 %0, [%1];" : "=r"(v) : "r"(addr(i))); return v;
  }
  __device__ __forceinline__ void set(uint32_t i, uint32_t v) const { asm volatile("st.shared.u8 [%0], %1;" ::"r"(addr(i)), "r"(v)); }
  __device__ __forceinline__ uint32_t get_word(uint32_t k) const {   // positions 4k .. 4k+3
    uint32_t v; asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(a + k * kSeqWordStride)); return v;
  }
  __device__ __forceinline__ void set_word(uint32_t k, uint32_t v) const { asm volatile("st.shared.u32 [%0], %1;" ::"r"(a + k * kSeqWordStride), "r"(v)); }
};
template <class SeqT>
struct SeqCode {  // view as residue codes for md_try_variable
  SeqT s; const uint8_t* code_of_a;
  __device__ __forceinline__ uint32_t operator()(uint32_t i) const { return code_of_a[s.get(i)]; }
};

struct AttemptOut {
  uint8_t* rows; uint8_t* len; uint64_t* mask; int64_t* w; uint64_t* hash;
};

// write one finished attempt (len == 0 -> failure)
template <class SeqT>
__device__ void store_attempt(const AttemptOut& O, uint64_t slot, const SeqT& seq, uint32_t L, uint64_t mask, int64_t w, const DecoyTables& T,
                              const PeptideView& PV) {
  if (L == 0) { O.len[slot] = 0; return; }
  uint8_t ascii[MD_MAX_PEPTIDE_LEN];
  uint64_t h = md_hash_init();
  uint8_t* row = O.rows + slot * MD_DECOY_ROW;
  for (uint32_t i = 0; i < L; i++) {
    uint8_t code = T.code_of_a[seq.get(i)];
    uint8_t ch = md_letter_of(code);
    ascii[i] = ch; row[i] = code;
    h = md_hash_step(h, ch);
  }
  for (uint32_t i = L; i < ((L + 15u) & ~15u); i++) row[i] = MD_CODE_OTHER;   // pad the last 16-byte chunk
  { const uint32_t pad = MD_CODE_OTHER * 0x01010101u;
    for (uint32_t c = (L + 15u) >> 4; c < MD_DECOY_ROW / 16; c++) reinterpret_cast<uint4*>(row)[c] = make_uint4(pad, pad, pad, pad); }
  h = md_hash_fin(h, L);
  if (is_peptide(ascii, L, h, PV.ht_key, PV.ht_val, PV.ht_mask, PV.seq, PV.off, PV.len)) { O.len[slot] = 0; return; }
  O.len[slot] = (uint8_t)L; O.mask[slot] = mask; O.w[slot] = w; O.hash[slot] = h;
}

// work item -> (list entry, attempt ordinal) by binary search on the round's prefix of attempt counts, narrowed by a coarse
// table: blk[b] = entry of work item b << kBlkLog (the search runs between two neighbouring table values)
constexpr uint32_t kBlkLog = 10;
__device__ __forceinline__ uint32_t find_entry_coarse(const uint32_t* __restrict__ att_off, const uint32_t* __restrict__ blk, uint32_t w) {
  uint32_t lo = blk[w >> kBlkLog], hi = blk[(w >> kBlkLog) + 1] + 1u;   // att_off[lo] <= w < att_off[hi]
  while (hi - lo > 1) { uint32_t mid = (lo + hi) >> 1; if (att_off[mid] <= w) lo = mid; else hi = mid; }
  return lo;
}

// One Philox4x32-10 block of the decoy stream (Philox4::refill with c3 = MD_TAG_RANDOM).  Each product is one mul.wide.u32:
// written as a 64-bit C++ multiply, the compiler added a zero high word (VIADD ..., URZ) behind every IMAD.WIDE.U32.
__device__ __forceinline__ uint4 philox_block(uint32_t a, uint32_t b, uint32_t c, uint32_t x, uint32_t y) {
  uint32_t d = MD_TAG_RANDOM;
#pragma unroll
  for (int r = 0; r < 10; r++) {
    uint32_t lo0, hi0, lo1, hi1;
    asm("{ .reg .b64 t; mul.wide.u32 t, %2, %3; mov.b64 {%0, %1}, t; }" : "=r"(lo0), "=r"(hi0) : "r"(a), "n"(0xD2511F53u));
    asm("{ .reg .b64 t; mul.wide.u32 t, %2, %3; mov.b64 {%0, %1}, t; }" : "=r"(lo1), "=r"(hi1) : "r"(c), "n"(0xCD9E8D57u));
    a = hi1 ^ b ^ x; b = lo1; c = hi0 ^ d ^ y; d = lo0;
    x += 0x9E3779B9u; y += 0xBB67AE85u;
  }
  return make_uint4(a, b, c, d);
}

// Philox4x32-10 output stream of one attempt, buffered in a per-lane shared-memory ring so that the block function runs
// for the whole warp at once (every kRngPeriod steps of the kernel loop) instead of as a divergent tail behind whichever
// lane happens to run dry.  The stream is exactly Philox4::next()'s: blocks c0 = 0, 1, 2, ... in order, four words each.
#ifndef MD_RNG_RING
#define MD_RNG_RING 8
#endif
constexpr uint32_t kRing = MD_RNG_RING;   // words per lane (power of two)
struct RngRing {
  uint32_t addr;                 // shared-memory address of the lane's kRing words, stride kThreads (accessed through volatile asm only)
  uint32_t k0, k1, c0, c1, c2;   // key, next block, attempt, spectrum
  uint32_t head, count;
  // continue the stream of (seed, spectrum_id, attempt) at word w, given block w / 4 (its first w % 4 words are skipped)
  __device__ __forceinline__ void resume(uint64_t seed, uint32_t spectrum_id, uint32_t attempt, uint32_t w, uint4 block) {
    k0 = (uint32_t)seed; k1 = (uint32_t)(seed >> 32); c0 = (w >> 2) + 1u; c1 = attempt; c2 = spectrum_id;
    put(0, block.x); put(1, block.y); put(2, block.z); put(3, block.w);
    head = w & 3u; count = 4u - (w & 3u);
  }
  __device__ __forceinline__ void put(uint32_t t, uint32_t v) const { asm volatile("st.shared.u32 [%0], %1;" ::"r"(addr + (t & (kRing - 1)) * (kThreads * 4u)), "r"(v)); }
  __device__ __forceinline__ void produce() {   // one block -> 4 words into the ring (needs count <= kRing - 4)
    const uint4 o = philox_block(c0, c1, c2, k0, k1);
    const uint32_t t = head + count;
    put(t + 0, o.x); put(t + 1, o.y); put(t + 2, o.z); put(t + 3, o.w);
    c0++; count += 4;
  }
  __device__ __forceinline__ uint32_t next() {
    if (count == 0) produce();
    uint32_t v; asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(addr + (head & (kRing - 1)) * (kThreads * 4u)));
    head++; count--;
    return v;
  }
};
#ifndef MD_RNG_PERIOD
#define MD_RNG_PERIOD 8
#endif
constexpr uint32_t kRngPeriod = MD_RNG_PERIOD;
#ifndef MD_REFILL_MIN
#define MD_REFILL_MIN 3
#endif
constexpr int kRefillMin = MD_REFILL_MIN;   // free lanes of a warp that trigger a refill

// position masks are 32 bits wide in the narrow pass (sequences of <= 32 residues: nearly all of them) and 64 in the wide one
template <class MaskT> struct MaskOps;
template <> struct MaskOps<uint32_t> {
  static constexpr uint32_t bits = 32;
  static __device__ __forceinline__ uint32_t ffs(uint32_t v) { return (uint32_t)__ffs((int)v); }
  static __device__ __forceinline__ uint32_t popc(uint32_t v) { return (uint32_t)__popc(v); }
  static __device__ __forceinline__ uint32_t ld(uint32_t addr) { uint32_t v; asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(addr)); return v; }
  static __device__ __forceinline__ void st(uint32_t addr, uint32_t v) { asm volatile("st.shared.u32 [%0], %1;" ::"r"(addr), "r"(v)); }
};
template <> struct MaskOps<uint64_t> {
  static constexpr uint32_t bits = 64;
  static __device__ __forceinline__ uint32_t ffs(uint64_t v) { return (uint32_t)__ffsll((long long)v); }
  static __device__ __forceinline__ uint32_t popc(uint64_t v) { return (uint32_t)__popcll(v); }
  static __device__ __forceinline__ uint64_t ld(uint32_t addr) { uint64_t v; asm volatile("ld.shared.u64 %0, [%1];" : "=l"(v) : "r"(addr)); return v; }
  static __device__ __forceinline__ void st(uint32_t addr, uint64_t v) { asm volatile("st.shared.u64 [%0], %1;" ::"r"(addr), "l"(v)); }
};

// try_variable_modifications (modified_peptide.rs:512-543) for one variable letter without a fixed modification, on the
// residual d = weight - precursor: the weight depends on the subset size only, and the first subset of size n in NChooseK
// order is the first n positions (same contract as md_try_variable_simple: on failure the last subset stays applied).
template <class MaskT>
__device__ __forceinline__ bool try_variable_simple_d(uint32_t nvar, int32_t delta, MaskT allpos, int32_t& d, MaskT& mask, int32_t dlo, uint32_t span) {
  using MO = MaskOps<MaskT>;
  const uint32_t cnt = MO::popc(allpos);
  const uint32_t nmax = nvar < cnt ? nvar : cnt;
  const int32_t base = d - (int32_t)MO::popc(mask) * delta;
  // The subset sizes are walked with nothing but the residual: base + n * delta, n = 1..nmax, first one inside the window.
  // Every lane that holds the letter runs these few instructions together.  (A "cannot hit" test in front of a loop that
  // also built the subsets was slower: after a failure the reference leaves the nmax modifications applied, the repair
  // loop then steers THAT weight towards the precursor, so base sits nmax * delta away from the window and the test
  // passes for most of the lanes that get here -- they then ran the loop two or three at a time.)
  uint32_t nhit = 0;
  int32_t dn = base;
  if (nvar <= 4u) {      // (the usual -n: four predicated steps, no loop whose trip count differs from lane to lane)
#pragma unroll
    for (uint32_t n = 1; n <= 4u; n++) {
      dn += delta;
      if (n <= nmax && nhit == 0u && (uint32_t)dn - (uint32_t)dlo <= span) nhit = n;
    }
    dn = base + (int32_t)nmax * delta;
  } else {
#pragma unroll 1
    for (uint32_t n = 1; n <= nmax; n++) {
      dn += delta;
      if (nhit == 0u && (uint32_t)dn - (uint32_t)dlo <= span) nhit = n;
    }
  }
  if (nhit) {                                 // the first nhit positions (NChooseK order: the first subset of that size)
    MaskT first = 0, rest = allpos;
    for (uint32_t n = 0; n < nhit; n++) { first |= rest & ((MaskT)0 - rest); rest &= rest - 1; }
    d = base + (int32_t)nhit * delta; mask = first;
    return true;
  }
  MaskT last = allpos;                        // on failure the last subset tried stays applied: the nmax last positions
#pragma unroll 1
  for (uint32_t k = cnt; k > nmax; k--) last &= last - 1;
  d = dn; mask = last;
  return false;
}

// The kernel's small lookup tables live in ONE shared-memory block and are read through ld.shared with the table's offset as
// an immediate: address = (block's shared address + index), one LEA + LDS per lookup.  (Declared as separate __shared__ arrays
// the compiler rebuilt every table's window address -- S2R CgaCtaId, MOV, VIADD, LEA -- in front of every lookup, under the
// 48-register cap that buys 10 CTAs per SM: about 20 of the ~290 instructions of a loop pass.)
namespace tabs {
constexpr uint32_t kAboveOfs = 40;                                  // offset of the d < 0 tables inside gap / gmask
constexpr uint32_t mprime = 0;                                       // int32[32], by alphabet index
constexpr uint32_t var = mprime + 32 * 4;                            // int32[32]
constexpr uint32_t gap = var + 32 * 4;                               // uint32[kAboveOfs + 32]: d > 0 tables at [0..], d < 0 tables at [kAboveOfs..]
constexpr uint32_t gmask = gap + (kAboveOfs + 32) * 4;               // uint32[kAboveOfs + 33]
constexpr uint32_t thr2 = gmask + (kAboveOfs + 33) * 4;              // int32[32]
constexpr uint32_t nnletter = thr2 + 32 * 4;                         // uint8[32]
constexpr uint32_t gtab = nnletter + 32;                             // uint8[2 * kGapTab]
constexpr uint32_t nntab = gtab + 2 * kGapTab;                       // uint8[kNnTab]
constexpr uint32_t bytes = (nntab + kNnTab + 15u) & ~15u;
}  // namespace tabs
template <uint32_t OFF> __device__ __forceinline__ uint32_t tab_u32(uint32_t addr) {
  uint32_t v; asm("ld.shared.u32 %0, [%1+%2];" : "=r"(v) : "r"(addr), "n"(OFF)); return v;
}
template <uint32_t OFF> __device__ __forceinline__ uint32_t tab_u8(uint32_t addr) {
  uint32_t v; asm("ld.shared.u8 %0, [%1+%2];" : "=r"(v) : "r"(addr), "n"(OFF)); return v;
}

struct RandomArgs {   // the work items of a round: list entries (spectrum, attempt ordinals) and their prefix of attempt counts
  const md_precursor* prec; const uint32_t* list; const uint32_t* att_off; const uint32_t* att_base;
  const uint32_t* att_blk;              // coarse index into att_off (find_entry_coarse)
  uint32_t total;
  uint64_t seed; int* overflow;
};

// A grown attempt, from k_decoy_grow to k_decoy_random and k_decoy_finish: its residual d = weight - precursor and the
// window [dlo, dlo + span] in 32-bit residual space, its length, its RNG counter and the precursor mass.  The alphabet-index
// sequence is in the attempt's row of AttemptOut::rows.  k_decoy_random writes the final residual of a hit back into d.
struct __align__(16) GrownAttempt {
  int32_t d, dlo; uint32_t span, L;
  uint32_t spectrum_id, attempt; int64_t P;
};
// The rest of a grown attempt's start state in k_decoy_random, also written by k_decoy_grow, so that a lane's refill is
// word copies and straight-line logic instead of a walk over the sequence and a Philox block: the alphabet indices as five
// bit planes of the position masks (bit i of plane k = bit k of the letter at position i; low halves first, so that the
// narrow pass reads the first 48 bytes only), the letter set, and Philox block L / 4 of the attempt's stream, where the
// repair continues at word L.  Written and read as four uint4.
struct __align__(16) StartState {
  uint32_t plane_lo[5], present, block[4];
  uint32_t plane_hi[5], pad;
};
static_assert(sizeof(StartState) == 64, "four uint4");

// Grow phase of REFERENCE_RANDOM (decoy_generator.rs:142-159), one thread per work item of the round: uniform letters until the
// weight exceeds the upper limit.  A sequence longer than 60 residues (VARCHAR(60) would reject it) is a failure (len = 0) here;
// every other attempt is flagged for the repair pass of its length -- 32-bit position masks up to `narrow_max` residues, 64-bit
// ones above -- and k_decoy_random continues its RNG stream at word L.  The sequence goes to the row as alphabet indices in
// 16-byte stores (the finished words of a chunk wait in registers), not byte by byte; its bit planes, letter set and the
// Philox block the repair resumes with go to the attempt's StartState.
constexpr int kGrowThreads = 256;
__global__ void __launch_bounds__(kGrowThreads) k_decoy_grow(const RandomArgs A, const __grid_constant__ DecoyTables T, AttemptOut O,
                                                             GrownAttempt* __restrict__ grown, StartState* __restrict__ start,
                                                             uint8_t* __restrict__ to_narrow, uint8_t* __restrict__ to_wide, uint32_t narrow_max) {
  __shared__ int32_t s_m[32];
  if (threadIdx.x < 32) s_m[threadIdx.x] = (int32_t)T.mprime[threadIdx.x];
  __syncthreads();
  const uint32_t wi = blockIdx.x * blockDim.x + threadIdx.x;
  if (wi >= A.total) return;
  const uint32_t li = find_entry_coarse(A.att_off, A.att_blk, wi);
  const md_precursor pr = A.prec[A.list[li]];
  const uint32_t attempt = A.att_base[li] + (wi - A.att_off[li]);
  uint4* row = reinterpret_cast<uint4*>(O.rows + (size_t)wi * MD_DECOY_ROW);
  int64_t w = MD_WATER_UDA;
  uint32_t L = 0, b = 0, word = 0;
  uint32_t w0 = 0, w1 = 0, w2 = 0;   // the finished words of the current 16-byte chunk, the newest in w2
  uint64_t plane[5] = {0, 0, 0, 0, 0};
  uint32_t present = 0;
  uint4 r;
  bool dead = false;
  for (;; b++) {   // Philox block b = words 4b .. 4b+3 = residues 4b .. 4b+3 = the b-th 32-bit word of the row
    r = philox_block(b, attempt, pr.spectrum_id, (uint32_t)A.seed, (uint32_t)(A.seed >> 32));
    const uint32_t rw[4] = {r.x, r.y, r.z, r.w};
    bool done = false;
    word = 0;
#pragma unroll
    for (int j = 0; j < 4; j++) {
      if (!done) {
        const uint32_t a = (uint32_t)(((uint64_t)rw[j] * MD_ALPHABET_SIZE) >> 32);
        if (L >= MD_MAX_PEPTIDE_LEN) { dead = true; done = true; }
        else {
          word |= a << (8 * j); L++;
          present |= 1u << a;
          w += s_m[a];
          done = w > pr.hi;
        }
      }
    }
    // bit k of the word's four letters -> bits 4b .. 4b+3 of plane k (the multiply gathers bit 0 of each byte into bits 24..27)
#pragma unroll
    for (int k = 0; k < 5; k++) plane[k] |= (uint64_t)((((word >> k) & 0x01010101u) * 0x01020408u) >> 24) << (4u * b);
    if (done) break;
    if ((b & 3u) == 3u) row[b >> 2] = make_uint4(w0, w1, w2, word);
    else { w0 = w1; w1 = w2; w2 = word; }
  }
  const int64_t dd = w - pr.mass, dl = pr.lo - pr.mass, sp = pr.hi - pr.lo;
  if (!dead && (dd > 0x3FFFFFFF || dd < -0x3FFFFFFF || dl > 0x3FFFFFFF || dl < -0x3FFFFFFF || sp < 0 || sp > 0x7FFFFFFF)) { atomicMax(A.overflow, 2); dead = true; }
  to_narrow[wi] = !dead && L <= narrow_max;
  to_wide[wi] = !dead && L > narrow_max;
  if (dead) { O.len[wi] = 0; return; }
  for (uint32_t k = b & 3u; k < 3u; k++) { w0 = w1; w1 = w2; w2 = word; word = 0; }   // the last chunk: its words in front
  row[b >> 2] = make_uint4(w0, w1, w2, word);
  grown[wi] = GrownAttempt{(int32_t)dd, (int32_t)dl, (uint32_t)sp, L, pr.spectrum_id, attempt, pr.mass};
  // the repair continues at word L: block b unless the last letter took its last word (L == 4b + 4)
  if ((L >> 2) != b) r = philox_block(L >> 2, attempt, pr.spectrum_id, (uint32_t)A.seed, (uint32_t)(A.seed >> 32));
  uint4* st = reinterpret_cast<uint4*>(start + wi);
  st[0] = make_uint4((uint32_t)plane[0], (uint32_t)plane[1], (uint32_t)plane[2], (uint32_t)plane[3]);
  st[1] = make_uint4((uint32_t)plane[4], present, r.x, r.y);
  st[2] = make_uint4(r.z, r.w, (uint32_t)(plane[0] >> 32), (uint32_t)(plane[1] >> 32));
  st[3] = make_uint4((uint32_t)(plane[2] >> 32), (uint32_t)(plane[3] >> 32), (uint32_t)(plane[4] >> 32), 0u);
}

struct RepairArgs {
  const uint32_t* items; const uint32_t* n_items;   // the attempts of this pass (k_decoy_grow's narrow or wide list) and their count
  uint32_t* queue;                                   // work counter of this launch
  GrownAttempt* grown; const StartState* start;
  uint64_t seed; int* overflow;
};

// Repair phase (modified_peptide.rs:451-508) of the attempts k_decoy_grow left to one pass.
// One lane = one attempt at a time, run as a flat state machine: every pass of the kernel loop does ONE step for every
// lane that has an attempt -- the first improving substitution at or behind the pass position, or, when the pass is
// over, the random kick -- and both kinds of step end in the same "put letter c at position p" code, so the lanes of a
// warp stay together although their attempts are at different tries / positions / lengths (nested try/position loops
// would make 31 finished lanes wait for the one that runs all 100 tries).  Lanes whose attempt ends (hit, or 100 tries
// without one) park until kRefillMin lanes of the warp are free, then write their results and load new grown attempts
// together.  Inside the loop an attempt is its residual d = weight - precursor in 32 bits (|d| stays far below 2^30 uDa
// after the grow phase; checked, reported via `overflow`) and the window is [dlo, dlo + span] in the same space.  A hit
// leaves its alphabet-index sequence in the row, its mask, its length and its final d; k_decoy_finish does the rest.
// VMODE: 0 = no variable modification can apply, 1 = one variable letter without a fixed modification (its positions are
// tracked, try_variable_modifications needs no walk over the sequence), 2 = anything else (generic enumeration).
// (The wide pass is bounded to 6 CTAs/SM, all that its shared memory allows: unbounded, its 64-bit refill took 88 registers.)
template <int VMODE, class MaskT>
__global__ void __launch_bounds__(kThreads, sizeof(MaskT) == 4 ? (VMODE < 2 ? 10 : 8) : 6) k_decoy_random(const RepairArgs A, const __grid_constant__ ModTables M, const __grid_constant__ DecoyTables T,
                                                           AttemptOut O) {
  using MO = MaskOps<MaskT>;
  constexpr uint32_t kBits = MO::bits;
  constexpr bool kNarrow = kBits < MD_MAX_PEPTIDE_LEN;
  constexpr uint32_t kRows = kNarrow ? kBits : MD_MAX_PEPTIDE_LEN;
  constexpr uint32_t kAbove = tabs::kAboveOfs;       // offset of the d < 0 tables
  constexpr uint32_t kSeqWords = (kRows + 15u) / 16u * 4u;   // whole 16-byte chunks of the row per lane (the refill copies chunks)
  __shared__ __align__(16) uint8_t sseq[kSeqWords * kSeqWordStride];
  __shared__ uint32_t s_rng[kRing * kThreads];
  __shared__ MaskT s_pm[MD_ALPHABET_SIZE * kThreads];   // per lane and letter: the positions holding that letter
  __shared__ __align__(16) uint8_t s_tab[tabs::bytes];   // the lookup tables (namespace tabs)
  {
    int32_t* s_mprime = reinterpret_cast<int32_t*>(s_tab + tabs::mprime); int32_t* s_var = reinterpret_cast<int32_t*>(s_tab + tabs::var);
    uint32_t* s_gap = reinterpret_cast<uint32_t*>(s_tab + tabs::gap); uint32_t* s_gmask = reinterpret_cast<uint32_t*>(s_tab + tabs::gmask);
    int32_t* s_thr2 = reinterpret_cast<int32_t*>(s_tab + tabs::thr2);
    uint8_t* s_nnletter = s_tab + tabs::nnletter; uint8_t* s_gtab = s_tab + tabs::gtab; uint8_t* s_nntab = s_tab + tabs::nntab;
    for (uint32_t i = threadIdx.x; i < 2 * kGapTab; i += kThreads) s_gtab[i] = T.gap_tab[i / kGapTab][i % kGapTab];
    for (uint32_t i = threadIdx.x; i < kNnTab; i += kThreads) s_nntab[i] = T.nn_tab[i];
    if (threadIdx.x < 33) { s_gmask[threadIdx.x] = T.maskb_prefix[threadIdx.x]; s_gmask[kAbove + threadIdx.x] = T.maska_prefix[threadIdx.x]; }
    if (threadIdx.x < 32) {
      s_gap[threadIdx.x] = T.gapb_sorted[threadIdx.x]; s_gap[kAbove + threadIdx.x] = T.gapa_sorted[threadIdx.x];
      s_mprime[threadIdx.x] = (int32_t)T.mprime[threadIdx.x]; s_var[threadIdx.x] = (int32_t)T.var_a[threadIdx.x];
      s_thr2[threadIdx.x] = T.nn_thr2[threadIdx.x]; s_nnletter[threadIdx.x] = T.nn_letter[threadIdx.x];
    }
  }
  __syncthreads();
  uint32_t tb;    // the block's shared-memory address (made opaque: it is to stay in a register, not to be rebuilt per lookup)
  asm volatile("mov.u32 %0, %1;" : "=r"(tb) : "r"((uint32_t)__cvta_generic_to_shared(s_tab)) : "memory");   // (the tables' stores above stay in front of it)
  SSeq seq;
  asm volatile("mov.u32 %0, %1;" : "=r"(seq.a) : "r"((uint32_t)__cvta_generic_to_shared(sseq) + 4u * threadIdx.x));
  const uint32_t gap_shift = T.gap_shift, nn_shift = T.nn_shift;
  const int32_t nn_lo = T.nn_lo, nn_hi = T.nn_hi;
  const int va = VMODE == 1 ? md_alpha_of_code((uint32_t)M.var_simple_code) : -1;
  const int32_t vdelta = VMODE == 1 ? (int32_t)M.var[M.var_simple_code] : 0;
  const uint32_t total = *A.n_items;

  bool busy = false, drained = false;
  uint32_t pending = 0;           // 1 = hit, 2 = gave up: the result is written when the free lanes refill together
  uint32_t present = 0;           // letters in the sequence
  // (the position masks, like the sequence and the ring, through explicit shared addresses and volatile asm only)
  constexpr uint32_t kPmStride = kThreads * (uint32_t)sizeof(MaskT);
  uint32_t pm_a;
  asm volatile("mov.u32 %0, %1;" : "=r"(pm_a) : "r"((uint32_t)__cvta_generic_to_shared(s_pm) + (uint32_t)sizeof(MaskT) * threadIdx.x));
  auto add_letter = [&](uint32_t a, uint32_t i) { const uint32_t ad = pm_a + a * kPmStride; MO::st(ad, MO::ld(ad) | (MaskT)1 << i); present |= 1u << a; };
  auto del_letter = [&](uint32_t a, uint32_t i) { const uint32_t ad = pm_a + a * kPmStride; const MaskT v = MO::ld(ad) & ~((MaskT)1 << i); MO::st(ad, v); if (v == 0) present &= ~(1u << a); };
  uint32_t wi = 0, L = 0, pos = 0, tries = 0, span = 0, flags = 0;
  int64_t P = 0;                  // (VMODE 2 only: md_try_variable works on weights)
  int32_t d = 0, dlo = 0;
  MaskT mask = 0, vpos = 0, lmask = 0;
  RngRing rng;
  asm volatile("mov.u32 %0, %1;" : "=r"(rng.addr) : "r"((uint32_t)__cvta_generic_to_shared(s_rng) + 4u * threadIdx.x));

  uint32_t rng_timer = 1;
  for (;;) {
    // ---- refill: when at least kRefillMin lanes are free (or nobody works), they write their results and load new attempts together
    uint32_t busy_m = __ballot_sync(0xffffffffu, busy);
    uint32_t free_m = 0;
    if (__popc(busy_m) <= 32 - kRefillMin) free_m = __ballot_sync(0xffffffffu, !busy && (!drained || pending));
    if (free_m && (__popc(free_m) >= kRefillMin || busy_m == 0)) {
      if (!busy && pending) {
        if (pending == 1) {   // the final sequence (alphabet indices) back into the row, 16 bytes at a time (k_decoy_finish
                              // reads the positions < L only)
          uint4* row = reinterpret_cast<uint4*>(O.rows + (size_t)wi * MD_DECOY_ROW);
#pragma unroll
          for (uint32_t c = 0; c < kSeqWords / 4u; c++)
            if (16u * c < L) row[c] = make_uint4(seq.get_word(4u * c), seq.get_word(4u * c + 1u), seq.get_word(4u * c + 2u), seq.get_word(4u * c + 3u));
          O.mask[wi] = (uint64_t)mask; A.grown[wi].d = d;
        }
        O.len[wi] = pending == 1 ? (uint8_t)L : 0;
        pending = 0;
      }
      if (!busy && !drained) {
        const uint32_t q = atomicAdd(A.queue, 1u);
        if (q >= total) drained = true;
        else {
          wi = A.items[q];
          const GrownAttempt* g = A.grown + wi;
          const uint4* st = reinterpret_cast<const uint4*>(A.start + wi);
          const uint4* row = reinterpret_cast<const uint4*>(O.rows + (size_t)wi * MD_DECOY_ROW);
          L = g->L; d = g->d; dlo = g->dlo; span = g->span;
          if (VMODE == 2) P = g->P;
          const uint4 s0 = st[0], s1 = st[1], s2 = st[2];
          MaskT pl[5] = {s0.x, s0.y, s0.z, s0.w, s1.x};   // the bit planes (StartState)
          if (!kNarrow) {
            const uint4 s3 = st[3];
            const uint32_t hi[5] = {s2.z, s2.w, s3.x, s3.y, s3.z};
#pragma unroll
            for (int k = 0; k < 5; k++) pl[k] |= (MaskT)hi[k] << (kBits / 2);
          }
          present = s1.y;
          rng.resume(A.seed, g->spectrum_id, g->attempt, L, make_uint4(s1.z, s1.w, s2.x, s2.y));   // the grow phase drew L words
          lmask = L >= kBits ? ~(MaskT)0 : (((MaskT)1 << L) - 1);
          // the per-letter position masks: the positions whose letter has the bits of a, from the planes (a is a constant of
          // the unrolled loop; positions >= L have all planes 0, so only letter 0 needs lmask)
#pragma unroll
          for (uint32_t a = 0; a < MD_ALPHABET_SIZE; a++) {
            const MaskT m = ((a & 1u) ? pl[0] : ~pl[0]) & ((a & 2u) ? pl[1] : ~pl[1]) & ((a & 4u) ? pl[2] : ~pl[2]) &
                            ((a & 8u) ? pl[3] : ~pl[3]) & ((a & 16u) ? pl[4] : ~pl[4]);
            MO::st(pm_a + a * kPmStride, a == 0 ? m & lmask : m);
          }
          mask = 0;
          if (VMODE == 1) vpos = MO::ld(pm_a + (uint32_t)va * kPmStride);
          // the sequence, whole 16-byte chunks of the row (positions >= L are never read)
#pragma unroll
          for (uint32_t c = 0; c < kSeqWords / 4u; c++)
            if (16u * c < L) {
              const uint4 v = row[c];
              seq.set_word(4u * c, v.x); seq.set_word(4u * c + 1u, v.y); seq.set_word(4u * c + 2u, v.z); seq.set_word(4u * c + 3u, v.w);
            }
          busy = true; tries = 0; pos = 0;
        }
      }
      busy_m = __ballot_sync(0xffffffffu, busy);
    }
    if (busy_m == 0) {
      if (__ballot_sync(0xffffffffu, !drained || pending) == 0) break;
      continue;
    }
    // ---- keep the random-number rings topped up, all lanes together
    if (--rng_timer == 0) { rng_timer = kRngPeriod; if (busy && rng.count <= kRing - 4) rng.produce(); }
    if (busy) {
      // ---- which LETTERS have a substitution that strictly reduces |d| follows from d alone (see DecoyTables) ...
      uint32_t fm;
      {
        const uint32_t ad = (uint32_t)(d < 0 ? -d : d), x = 2u * ad;
        const uint32_t gofs = d > 0 ? 0u : kAbove;
        const uint32_t k0 = tab_u8<tabs::gtab>(tb + (d > 0 ? 0u : kGapTab) + min(x >> gap_shift, kGapTab - 1u));
        uint32_t ga = tb + 4u * (gofs + k0);                             // walks gap[gofs + k] and, at the same index, gmask
        for (uint32_t gk = tab_u32<tabs::gap>(ga); gk < x; gk = tab_u32<tabs::gap>(ga)) ga += 4u;   // number of gaps below x (padding: 0xFFFFFFFF)
        fm = tab_u32<tabs::gmask>(ga);                                   // d == 0: x == 0, k == 0, empty prefix
      }
      // ---- ... and the per-letter position masks give the first position of the pass that can improve: OR of the masks of
      //      the qualifying letters -- or, when most letters qualify (right after a kick), the complement of the OR over
      //      the few that do not (every position holds exactly one of the present letters).
      MaskT cand;
      {
        const uint32_t m0 = fm & present, n0 = present & ~fm;
        const bool inv = __popc(n0) < __popc(m0);
        MaskT acc = 0;
        for (uint32_t m = inv ? n0 : m0; m;) {     // from the top bit: one FLO (bfind) per letter instead of BREV + FLO for __ffs
          uint32_t h;
          asm("bfind.u32 %0, %1;" : "=r"(h) : "r"(m));
          acc |= MO::ld(pm_a + h * kPmStride);
          m &= ~(1u << h);
        }
        cand = inv ? ~acc & lmask : acc;
        cand = pos < L ? cand & (~(MaskT)0 << pos) : (MaskT)0;           // pos == L: the pass ended with a substitution
      }
      // ---- the step: substitution at the first improving position (modified_peptide.rs:454-487), else the kick (:489-505)
      const bool sub = cand != 0;
      uint32_t p;
      // the kick takes ONE word r of the attempt's stream: position = high half of r*L, letter = high half of low32(r*L)*21
      uint32_t kick_lo = 0;
      if (sub) p = MO::ffs(cand) - 1u;
      else { const uint64_t rl = (uint64_t)rng.next() * L; p = (uint32_t)(rl >> 32); kick_lo = (uint32_t)rl; }
      const uint32_t old = seq.get(p);
      const int32_t m_old = (int32_t)tab_u32<tabs::mprime>(tb + 4u * old);
      uint32_t c;
      if (sub) {
        // best single substitution = letter whose (mass+fixed) is closest to mprime[old] - d; strict improvement,
        // ties by alphabet order (the reference follows HashMap order there)
        const int32_t target = min(max(m_old - d, nn_lo), nn_hi);
        const int32_t t2 = 2 * target;
        uint32_t k = tab_u8<tabs::nntab>(tb + ((uint32_t)(target - nn_lo) >> nn_shift));
        for (int32_t th = (int32_t)tab_u32<tabs::thr2>(tb + 4u * k); t2 > th; th = (int32_t)tab_u32<tabs::thr2>(tb + 4u * k)) k++;   // nearest distinct mass (padding: INT32_MAX)
        c = tab_u8<tabs::nnletter>(tb + k);
#ifdef MD_DECOY_CHECK   // (debug builds) the letter filter and the nearest-mass search must agree
        const int32_t nd = d + (int32_t)tab_u32<tabs::mprime>(tb + 4u * c) - m_old;
        if (!((uint32_t)(nd < 0 ? -nd : nd) < (uint32_t)(d < 0 ? -d : d) && c != old)) { flags |= 4u; c = old; }
#endif
      } else {
        c = (uint32_t)(((uint64_t)kick_lo * MD_ALPHABET_SIZE) >> 32);
      }
      // ---- put letter c at position p: remove_modification_at + swap + fixed modification of the new letter (:470-482)
      {
        const MaskT bit = (MaskT)1 << p;
        if (VMODE != 0) { if (mask & bit) { d -= (int32_t)tab_u32<tabs::var>(tb + 4u * old); mask &= ~bit; } }
        d += (int32_t)tab_u32<tabs::mprime>(tb + 4u * c) - m_old;
        seq.set(p, c); del_letter(old, p); add_letter(c, p);
        if (VMODE == 1) vpos = (vpos & ~bit) | ((int)c == va ? bit : (MaskT)0);
      }
      bool hit = false;
      if (sub) {
        hit = (uint32_t)d - (uint32_t)dlo <= span;
        if (VMODE == 1) {
          if (!hit && vpos) hit = try_variable_simple_d<MaskT>(M.nvar, vdelta, vpos, d, mask, dlo, span);
        } else if (VMODE == 2) {
          if (!hit) {
            SeqCode<SSeq> sc{seq, T.code_of_a};
            int64_t w = P + d; uint64_t m64 = (uint64_t)mask;
            const int64_t lo = P + dlo;
            if (md_try_variable(M, sc, L, w, m64, lo, lo + (int64_t)span, A.overflow)) hit = true;
            const int64_t dd = w - P;
            if (dd > 0x3FFFFFFF || dd < -0x3FFFFFFF) flags |= 2u;
            d = (int32_t)dd; mask = (MaskT)m64;
          }
        }
        pos = p + 1;
      } else {
        pos = 0; tries++;
      }
      if ((uint32_t)d + 0x3FFFFFFFu > 0x7FFFFFFEu) flags |= 2u;
      if (hit) { pending = 1; busy = false; }
      else if (!sub && tries == 100) { pending = 2; busy = false; }
    }
  }
  if (flags) atomicMax(A.overflow, (flags & 4u) ? 3 : 2);
}

// Finish phase, one thread per work item of the round: every hit k_decoy_random left (alphabet indices in the row, final d in
// GrownAttempt) becomes what store_attempt writes -- residue codes padded with MD_CODE_OTHER to the whole row, the sequence
// hash, the weight P + d -- unless it is a peptide of the index (len = 0).
__global__ void __launch_bounds__(256) k_decoy_finish(uint32_t total, const __grid_constant__ DecoyTables T, AttemptOut O,
                                                      const GrownAttempt* __restrict__ grown, PeptideView PV) {
  __shared__ uint8_t s_code[32];
  if (threadIdx.x < 32) s_code[threadIdx.x] = T.code_of_a[threadIdx.x];
  __syncthreads();
  const uint32_t wi = blockIdx.x * blockDim.x + threadIdx.x;
  if (wi >= total) return;
  const uint32_t L = O.len[wi];
  if (L == 0) return;
  uint8_t* rowb = O.rows + (size_t)wi * MD_DECOY_ROW;
  uint4* row = reinterpret_cast<uint4*>(rowb);
  const uint32_t pad = MD_CODE_OTHER * 0x01010101u;
  uint64_t h = md_hash_init();
#pragma unroll
  for (uint32_t c = 0; c < MD_DECOY_ROW / 16; c++) {
    uint32_t wd[4] = {pad, pad, pad, pad};
    if (16u * c < L) {
      const uint4 v = row[c];
      const uint32_t in[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
      for (uint32_t j = 0; j < 16; j++) {
        const uint32_t i = 16u * c + j;
        if (i < L) {
          const uint32_t code = s_code[(in[j >> 2] >> (8 * (j & 3))) & 0xFFu];
          h = md_hash_step(h, md_letter_of(code));
          wd[j >> 2] = (wd[j >> 2] & ~(0xFFu << (8 * (j & 3)))) | code << (8 * (j & 3));
        }
      }
    }
    row[c] = make_uint4(wd[0], wd[1], wd[2], wd[3]);
  }
  h = md_hash_fin(h, L);
  if (is_peptide([rowb](uint32_t i) { return md_letter_of(rowb[i]); }, L, h, PV.ht_key, PV.ht_val, PV.ht_mask, PV.seq, PV.off, PV.len)) { O.len[wi] = 0; return; }
  const GrownAttempt& g = grown[wi];
  O.w[wi] = g.P + g.d; O.hash[wi] = h;
}

// Terminal modifications (position N / C): the attempt restated literally, one lane per attempt -- the weight of a residue
// depends on where it stands (md_fix_applies), so neither the letter filter nor the per-letter position masks of
// k_decoy_random hold.  As in the reference the repair loop rates a substitution with the position-blind substitution map
// (get_one_amino_acid_substitute_map, decoy_generator.rs:301-324: every letter with its fixed delta) and then applies it
// with add_modification_at's position rules (modified_peptide.rs:421-447).  Same RNG stream, same output rows as
// k_decoy_random; a correctness path, not a tuned one.
__global__ void __launch_bounds__(kThreads) k_decoy_random_terminal(const RandomArgs A, const __grid_constant__ ModTables M, const __grid_constant__ DecoyTables T,
                                                                    AttemptOut O, PeptideView PV) {
  __shared__ uint8_t sseq[MD_MAX_PEPTIDE_LEN * kThreads];
  TSeq seq{sseq + threadIdx.x};
  auto fixd = [&](uint32_t a, uint32_t i, uint32_t L) -> int64_t { const uint32_t c = T.code_of_a[a]; return md_fix_applies(M, c, i, L) ? M.fix[c] : 0; };
  for (uint32_t wi = blockIdx.x * blockDim.x + threadIdx.x; wi < A.total; wi += gridDim.x * blockDim.x) {
    const uint32_t li = find_entry_coarse(A.att_off, A.att_blk, wi);
    const md_precursor pr = A.prec[A.list[li]];
    Philox4 rng; rng.init(A.seed, pr.spectrum_id, A.att_base[li] + (wi - A.att_off[li]), MD_TAG_RANDOM);
    // grow (decoy_generator.rs:142-159; push_modification, modified_peptide.rs:182-208: the residue that was last loses its
    // C-terminus modification, the new one takes its letter's fixed modification where its position allows)
    int64_t w = MD_WATER_UDA;
    uint32_t L = 0; bool dead = false;
    for (;;) {
      const uint32_t a = rng.below(MD_ALPHABET_SIZE);
      if (L >= MD_MAX_PEPTIDE_LEN) { dead = true; break; }
      if (L > 0) { const uint32_t pc = T.code_of_a[seq.get(L - 1)]; if (M.has_fix[pc] && M.fix_pos[pc] == MD_POS_C) w -= M.fix[pc]; }
      seq.at(L) = (uint8_t)a; L++;
      w += M.mass[T.code_of_a[a]] + fixd(a, L - 1, L);
      if (w > pr.hi) break;
    }
    uint64_t mask = 0;
    bool hit = false;
    // put letter c at position p: remove_modification_at + swap + add_modification_at (:470-482, :493-505)
    auto replace_at = [&](uint32_t p, uint32_t c) {
      const uint32_t old = seq.get(p);
      w -= M.mass[T.code_of_a[old]] + fixd(old, p, L);
      if ((mask >> p) & 1) { w -= M.var[T.code_of_a[old]]; mask &= ~(1ull << p); }
      seq.at(p) = (uint8_t)c;
      w += M.mass[T.code_of_a[c]] + fixd(c, p, L);
    };
    for (uint32_t t = 0; t < 100 && !dead && !hit; t++) {                    // 'tries (:453)
      for (uint32_t i = 0; i < L && !hit; i++) {                             // 'sequence (:454)
        const uint32_t cur = seq.get(i);
        int64_t best = pr.mass - w; if (best < 0) best = -best;
        uint32_t bestc = cur;
        for (uint32_t c = 0; c < MD_ALPHABET_SIZE; c++) {                    // 'swaps (:459-468), alphabet order
          if (c == cur) continue;
          int64_t d = pr.mass - (w + T.mprime[c] - T.mprime[cur]); if (d < 0) d = -d;
          if (d < best) { best = d; bestc = c; }
        }
        if (bestc != cur) {
          replace_at(i, bestc);
          if (md_in_window(w, pr.lo, pr.hi)) hit = true;                     // :483
          else { SeqCode<TSeq> sc{seq, T.code_of_a}; if (md_try_variable(M, sc, L, w, mask, pr.lo, pr.hi, A.overflow)) hit = true; }   // :484
        }
      }
      if (hit) break;
      const uint64_t rl = (uint64_t)rng.next() * L;                           // the kick (:489-505), one word as in k_decoy_random
      replace_at((uint32_t)(rl >> 32), (uint32_t)(((uint64_t)(uint32_t)rl * MD_ALPHABET_SIZE) >> 32));
    }
    store_attempt(O, wi, seq, hit ? L : 0, mask, w, T, PV);
  }
}

// vary_targets (decoy_generator.rs:265-296), counter-based: attempt a shuffles target (a mod T) of the spectrum
__global__ void __launch_bounds__(kThreads) k_decoy_permute(const RandomArgs A, const __grid_constant__ DecoyTables T,
                                                            const uint64_t* __restrict__ cand_off, const uint64_t* __restrict__ cand_desc,
                                                            const uint64_t* __restrict__ cand_mask, const int64_t* __restrict__ cand_w,
                                                            const uint8_t* __restrict__ idx_rows, AttemptOut O, PeptideView PV,
                                                            const __grid_constant__ ModTables M) {
  __shared__ uint8_t sseq[MD_MAX_PEPTIDE_LEN * kThreads];
  TSeq seq{sseq + threadIdx.x};
  const uint32_t wi = blockIdx.x * blockDim.x + threadIdx.x;
  if (wi >= A.total) return;
  const uint32_t li = find_entry_coarse(A.att_off, A.att_blk, wi);
  const uint32_t s = A.list[li];
  const md_precursor pr = A.prec[s];
  const uint32_t attempt = A.att_base[li] + (wi - A.att_off[li]);
  const uint64_t t0 = cand_off[s], nt = cand_off[s + 1] - t0;
  if (nt == 0) { O.len[wi] = 0; return; }
  const uint64_t c = t0 + attempt % nt;
  const uint64_t d = cand_desc[c];
  const uint8_t* row = idx_rows + (d & 0xFFFFFFFFFFull) * 16;
  const uint32_t L = (uint32_t)(d >> 40) & 0xFF;
  // the reference tests the shuffled sequence with fixed modifications only (:278-279): the candidate's weight without
  // the variable modifications it was found with (a permutation keeps the weight)
  int64_t wfix = cand_w[c];
  for (uint64_t m = cand_mask[c]; m; m &= m - 1) {
    const int a = md_alpha_of_code(row[__ffsll((long long)m) - 1]);
    if (a >= 0) wfix -= T.var_a[a];
  }
  if (!M.has_terminal && !md_in_window(wfix, pr.lo, pr.hi)) { O.len[wi] = 0; return; }   // (a permutation keeps this weight)
  bool ok = true;
  for (uint32_t i = 0; i < L; i++) {
    int a = md_alpha_of_code(row[i]);
    if (a < 0) ok = false;  // letters outside the decoy alphabet cannot be written back as a decoy row
    seq.at(i) = (uint8_t)(a < 0 ? 0 : a);
  }
  if (!ok) { O.len[wi] = 0; return; }
  Philox4 rng; rng.init(A.seed, pr.spectrum_id, attempt, MD_TAG_PERMUTE);
  for (uint32_t i = L; i > 1; i--) {
    uint32_t j = rng.below(i);
    uint8_t a = seq.at(i - 1); seq.at(i - 1) = seq.at(j); seq.at(j) = a;
  }
  if (M.has_terminal) {   // terminal modifications: the weight depends on which residues end up first and last (from_string, modified_peptide.rs:118-139)
    wfix = MD_WATER_UDA;
    for (uint32_t i = 0; i < L; i++) { const uint32_t cc = T.code_of_a[seq.get(i)]; wfix += M.mass[cc] + (md_fix_applies(M, cc, i, L) ? M.fix[cc] : 0); }
    if (!md_in_window(wfix, pr.lo, pr.hi)) { O.len[wi] = 0; return; }
  }
  store_attempt(O, wi, seq, L, 0, wfix, T, PV);
}

// One CTA per listed spectrum: keep the successes of this round that are new (not equal to an accepted decoy or to an
// earlier success), in attempt order, until the spectrum has n_per decoys (HashSet<Decoy>, decoy_generator.rs:40,164).
// Two routes to the keep decision; the host takes the hash set when it fits shared memory (slots > 0), else the exact scan:
// - Hash set, linear time: accepted decoys and successes go into a shared-memory hash set keyed by the 64-bit sequence hash,
//   each entry remembering the lowest ordinal (accepted decoys first, then attempts in order) that carried the key; a success
//   is kept iff it is that first carrier.  A success that is NOT the first carrier of its hash is compared with that carrier
//   byte for byte: equal = a duplicate (the usual case); different = two sequences share a 64-bit hash, and the CTA redoes
//   the spectrum with the exact scan.
// - Exact scan, quadratic: a success is kept iff no accepted decoy and no earlier success is the same sequence (HashSet<Decoy>
//   compares strings).  Attempts are strided across the threads: a chunk per thread would leave the last chunk's owner
//   comparing against nearly every success.
// The attempt hashes are read from HBM once (staged in shared memory); the kept rows are copied by the whole CTA, four lanes
// per 64-byte row.
__global__ void __launch_bounds__(256) k_decoy_select(const uint32_t* __restrict__ list, const uint32_t* __restrict__ att_off,
                                                      const uint32_t* __restrict__ att_base, uint32_t n_per, uint32_t slots, uint32_t max_na, AttemptOut A,
                                                      DecoyOut D) {
  extern __shared__ __align__(16) unsigned long long s_key[];     // slots (0 = empty)
  unsigned long long* s_hash = s_key + slots;                     // max_na: hash of a success (0 -> 1), 0 = failed attempt
  uint32_t* s_ord = reinterpret_cast<uint32_t*>(s_hash + max_na); // slots
  uint16_t* s_list = reinterpret_cast<uint16_t*>(s_ord + slots);  // max_na: kept attempts, in order (before that: the exact scan's keep flags)
  __shared__ uint32_t s_wsum[8];
  __shared__ uint32_t s_collision;
  const uint32_t li = blockIdx.x, s = list[li];
  const uint32_t a0 = att_off[li], na = att_off[li + 1] - a0;
  const uint32_t have = D.count[s];
  const uint64_t dbase = (uint64_t)s * n_per;
  const uint32_t smask = slots - 1;
  const uint32_t tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  if (tid == 0) s_collision = 0;
  // success `a` of this round against carrier `rep` (an accepted decoy if rep < have, else success rep - have): same sequence?
  auto same_sequence = [&](uint32_t a, uint32_t rep) -> bool {
    const uint32_t L = A.len[a0 + a];
    const uint8_t* mine = A.rows + (uint64_t)(a0 + a) * MD_DECOY_ROW;
    if (rep < have) {
      if (D.len[dbase + rep] != L) return false;
      for (uint32_t i = 0; i < L; i++) if (D.rows[md_dec_byte(D.n_slots, dbase + rep, i)] != mine[i]) return false;
    } else {
      if (A.len[a0 + rep - have] != L) return false;
      const uint8_t* o = A.rows + (uint64_t)(a0 + rep - have) * MD_DECOY_ROW;
      for (uint32_t i = 0; i < L; i++) if (o[i] != mine[i]) return false;
    }
    return true;
  };
  for (uint32_t i = tid; i < slots; i += 256) { s_key[i] = 0ULL; s_ord[i] = 0xFFFFFFFFu; }
  // MD_SELECT_HASH_MASK (test builds only) keeps a few bits of the hashes, so that colliding sequences are common
#ifndef MD_SELECT_HASH_MASK
#define MD_SELECT_HASH_MASK 0xFFFFFFFFFFFFFFFFull
#endif
#pragma unroll 4
  for (uint32_t a = tid; a < na; a += 256) {
    const uint32_t L = A.len[a0 + a];
    unsigned long long h = __ldg(reinterpret_cast<const unsigned long long*>(A.hash) + a0 + a) & MD_SELECT_HASH_MASK;
    s_hash[a] = L ? (h ? h : 1ULL) : 0ULL;
  }
  __syncthreads();
  // keep flags + ordered compaction: thread t owns the contiguous chunk [t*per, (t+1)*per), per <= 16
  const uint32_t per = (na + 255u) / 256u;
  const uint32_t cb = tid * per, ce = min(cb + per, na);
  uint32_t keepbits = 0, c = 0;
  if (slots) {
    auto insert = [&](unsigned long long h, uint32_t ord) {
      uint32_t slot = (uint32_t)h & smask;
      for (;;) {
        const unsigned long long prev = atomicCAS(&s_key[slot], 0ULL, h);
        if (prev == 0ULL || prev == h) { atomicMin(&s_ord[slot], ord); return; }
        slot = (slot + 1) & smask;
      }
    };
    for (uint32_t j = tid; j < have; j += 256) { const unsigned long long h = D.hash[dbase + j] & MD_SELECT_HASH_MASK; insert(h ? h : 1ULL, j); }
    for (uint32_t a = tid; a < na; a += 256) { const unsigned long long h = s_hash[a]; if (h) insert(h, have + a); }
    __syncthreads();
    for (uint32_t a = cb; a < ce; a++) {
      const unsigned long long h = s_hash[a];
      bool keep = h != 0ULL;
      if (keep) {
        uint32_t slot = (uint32_t)h & smask;
        while (s_key[slot] != h) slot = (slot + 1) & smask;
        keep = s_ord[slot] == have + a;
        if (!keep && !same_sequence(a, s_ord[slot])) s_collision = 1;    // not a duplicate after all
      }
      if (keep) { keepbits |= 1u << (a - cb); c++; }
    }
    __syncthreads();
  }
  if (!slots || s_collision) {   // (after a collision: two sequences with one 64-bit hash, practically never)
    uint8_t* s_keep = reinterpret_cast<uint8_t*>(s_list);
    for (uint32_t a = tid; a < na; a += 256) {
      const unsigned long long h = s_hash[a];
      bool keep = h != 0ULL;
      // (against the accepted decoys: their hashes as stored, without the hash set's 0 -> 1)
      const unsigned long long hr = keep ? A.hash[a0 + a] & MD_SELECT_HASH_MASK : 0ULL;
      for (uint32_t j = 0; j < have && keep; j++) if ((D.hash[dbase + j] & MD_SELECT_HASH_MASK) == hr && same_sequence(a, j)) keep = false;
      for (uint32_t b = 0; b < a && keep; b++) if (s_hash[b] == h && same_sequence(a, have + b)) keep = false;
      s_keep[a] = keep;
    }
    __syncthreads();
    keepbits = 0; c = 0;
    for (uint32_t a = cb; a < ce; a++) if (s_keep[a]) { keepbits |= 1u << (a - cb); c++; }
  }
  uint32_t incl = c;
  for (int o = 1; o < 32; o <<= 1) { const uint32_t t = __shfl_up_sync(0xffffffffu, incl, o); if ((int)lane >= o) incl += t; }
  if (lane == 31) s_wsum[warp] = incl;
  __syncthreads();   // (also: every keep flag is read before s_list is written)
  uint32_t before = incl - c, total = 0;
  for (uint32_t w = 0; w < 8; w++) { const uint32_t v = s_wsum[w]; if (w < warp) before += v; total += v; }
  const uint32_t room = n_per > have ? n_per - have : 0u;
  const uint32_t nk = min(total, room);
  {
    uint32_t o = before;
    for (uint32_t m = keepbits; m; m &= m - 1) { if (o < nk) s_list[o] = (uint16_t)(cb + (uint32_t)__ffs(m) - 1u); o++; }
  }
  __syncthreads();
  // copy the kept rows (four lanes per row) and their scalars; loads are issued four at a time before their stores (the
  // compiler may not move a load above a store through these pointers, and one row per round trip to HBM is what made
  // this phase two thirds of the kernel)
  for (uint32_t t0 = tid; t0 < nk * 4u; t0 += 4u * 256u) {
    uint4 v[4];
#pragma unroll
    for (int j = 0; j < 4; j++) {
      const uint32_t t = t0 + (uint32_t)j * 256u;
      if (t < nk * 4u) v[j] = __ldg(reinterpret_cast<const uint4*>(A.rows + (uint64_t)(a0 + s_list[t >> 2]) * MD_DECOY_ROW) + (t & 3u));
    }
#pragma unroll
    for (int j = 0; j < 4; j++) {
      const uint32_t t = t0 + (uint32_t)j * 256u;
      if (t < nk * 4u) *reinterpret_cast<uint4*>(D.rows + md_dec_byte(D.n_slots, dbase + have + (t >> 2), (t & 3u) * 16u)) = v[j];
    }
  }
  for (uint32_t r0 = tid; r0 < nk; r0 += 2u * 256u) {
    uint8_t ln[2]; uint64_t mk[2], hs[2]; int64_t wt[2];
#pragma unroll
    for (int j = 0; j < 2; j++) {
      const uint32_t r = r0 + (uint32_t)j * 256u;
      if (r < nk) { const uint64_t src = a0 + s_list[r]; ln[j] = A.len[src]; mk[j] = A.mask[src]; wt[j] = A.w[src]; hs[j] = A.hash[src]; }
    }
#pragma unroll
    for (int j = 0; j < 2; j++) {
      const uint32_t r = r0 + (uint32_t)j * 256u;
      if (r < nk) {
        const uint64_t dst = dbase + have + r;
        D.len[dst] = ln[j]; D.mask[dst] = mk[j]; D.w[dst] = wt[j]; D.hash[dst] = hs[j];
        D.attempt[dst] = att_base[li] + s_list[r];
      }
    }
  }
  if (tid == 0) D.count[s] = have + nk;
}

// the repair kernel of a vmode (see k_decoy_random)
template <class MaskT>
auto random_kernel(int vmode) { return vmode == 0 ? k_decoy_random<0, MaskT> : vmode == 1 ? k_decoy_random<1, MaskT> : k_decoy_random<2, MaskT>; }
template <class MaskT>
int random_occupancy(int vmode) {
  static int cached[3] = {0, 0, 0};     // (a property of the kernel image: queried once per process)
  if (!cached[vmode]) {
    int occ = 0;
    MD_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, random_kernel<MaskT>(vmode), kThreads, 0));
    cached[vmode] = occ > 0 ? occ : 1;
  }
  return cached[vmode];
}

DecoyTables make_tables(const ModTables& M) {
  DecoyTables T;
  memset(&T, 0, sizeof(T));
  const char* alpha = MD_ALPHABET;
  struct E { int64_t m; int a; };
  std::vector<E> v;   // the letters by mprime ascending, ties by alphabet index
  for (int a = 0; a < MD_ALPHABET_SIZE; a++) {
    uint32_t code = md_code_of((uint8_t)alpha[a]);
    T.code_of_a[a] = (uint8_t)code;
    T.var_a[a] = M.var[code];
    T.mprime[a] = M.mass[code] + (M.has_fix[code] ? M.fix[code] : 0);
    v.push_back({T.mprime[a], a});
  }
  std::sort(v.begin(), v.end(), [](const E& x, const E& y) { return x.m != y.m ? x.m < y.m : x.a < y.a; });
  uint8_t run_min[MD_ALPHABET_SIZE];   // lowest alphabet index among the letters of equal mass, at each sorted position
  for (int k = 0; k < MD_ALPHABET_SIZE; k++) {
    int j = k; while (j > 0 && v[j - 1].m == v[k].m) j--;  // first of the equal-mass run has the lowest alphabet index
    run_min[k] = (uint8_t)v[j].a;
  }
  // gap tables
  {
    struct G { uint32_t g; int a; };
    std::vector<G> gb, ga;
    for (int a = 0; a < MD_ALPHABET_SIZE; a++) {
      int64_t below = -1, above = -1;
      for (int c = 0; c < MD_ALPHABET_SIZE; c++) {
        if (T.mprime[c] < T.mprime[a] && (below < 0 || T.mprime[c] > below)) below = T.mprime[c];
        if (T.mprime[c] > T.mprime[a] && (above < 0 || T.mprime[c] < above)) above = T.mprime[c];
      }
      gb.push_back({below < 0 ? 0xFFFFFFFFu : (uint32_t)std::min<int64_t>(T.mprime[a] - below, 0xFFFFFFFEll), a});
      ga.push_back({above < 0 ? 0xFFFFFFFFu : (uint32_t)std::min<int64_t>(above - T.mprime[a], 0xFFFFFFFEll), a});
    }
    auto by_gap = [](const G& x, const G& y) { return x.g != y.g ? x.g < y.g : x.a < y.a; };
    std::sort(gb.begin(), gb.end(), by_gap); std::sort(ga.begin(), ga.end(), by_gap);
    for (int k = 0; k < 32; k++) { T.gapb_sorted[k] = 0xFFFFFFFFu; T.gapa_sorted[k] = 0xFFFFFFFFu; }
    T.maskb_prefix[0] = 0; T.maska_prefix[0] = 0;
    for (int k = 0; k < MD_ALPHABET_SIZE; k++) {
      T.gapb_sorted[k] = gb[k].g; T.maskb_prefix[k + 1] = T.maskb_prefix[k] | (gb[k].g == 0xFFFFFFFFu ? 0u : 1u << gb[k].a);
      T.gapa_sorted[k] = ga[k].g; T.maska_prefix[k + 1] = T.maska_prefix[k] | (ga[k].g == 0xFFFFFFFFu ? 0u : 1u << ga[k].a);
    }
    for (int k = MD_ALPHABET_SIZE + 1; k < 33; k++) { T.maskb_prefix[k] = T.maskb_prefix[MD_ALPHABET_SIZE]; T.maska_prefix[k] = T.maska_prefix[MD_ALPHABET_SIZE]; }
    // bucket table over x = 2|d|: the last bucket takes every larger x (the residual scan finishes the count)
    uint32_t gmax = 1;
    for (int k = 0; k < MD_ALPHABET_SIZE; k++) { if (gb[k].g != 0xFFFFFFFFu) gmax = std::max(gmax, gb[k].g); if (ga[k].g != 0xFFFFFFFFu) gmax = std::max(gmax, ga[k].g); }
    T.gap_shift = 0;
    while (((uint64_t)gmax >> T.gap_shift) >= kGapTab - 1) T.gap_shift++;
    for (int sgn = 0; sgn < 2; sgn++) {
      const uint32_t* g = sgn == 0 ? T.gapb_sorted : T.gapa_sorted;
      for (uint32_t b = 0; b < kGapTab; b++) {
        const uint64_t x0 = (uint64_t)b << T.gap_shift;   // first x of the bucket: gaps < x0 are below every x of the bucket
        uint32_t c = 0;
        while (c < MD_ALPHABET_SIZE && (uint64_t)g[c] < x0) c++;
        T.gap_tab[sgn][b] = (uint8_t)c;
      }
    }
  }
  // nearest-mass tables
  {
    int n = 0; int64_t u[32]; uint8_t rep[32];
    for (int k = 0; k < MD_ALPHABET_SIZE; k++)
      if (n == 0 || v[k].m != u[n - 1]) { u[n] = v[k].m; rep[n] = run_min[k]; n++; }
    for (int j = 0; j < 32; j++) { T.nn_thr2[j] = INT32_MAX; T.nn_letter[j] = j < n ? rep[j] : rep[n - 1]; }
    for (int j = 0; j + 1 < n; j++) T.nn_thr2[j] = (int32_t)(u[j] + u[j + 1] - (rep[j] < rep[j + 1] ? 0 : 1));
    T.nn_lo = (int32_t)(u[0] - 1); T.nn_hi = (int32_t)(u[n - 1] + 1);
    T.nn_shift = 0;
    while ((((uint64_t)(T.nn_hi - T.nn_lo)) >> T.nn_shift) >= kNnTab) T.nn_shift++;
    for (uint32_t b = 0; b < kNnTab; b++) {
      const int64_t t0 = (int64_t)T.nn_lo + ((int64_t)b << T.nn_shift);   // first t of the bucket
      uint32_t c = 0;
      while (c + 1 < (uint32_t)n && 2 * t0 > (int64_t)T.nn_thr2[c]) c++;
      T.nn_tab[b] = (uint8_t)c;
    }
  }
  return T;
}

// Spectra in (roughly) ascending precursor mass: neighbouring attempts grow sequences of similar length (lockstep passes).
// (The order only steers which attempts run side by side, not the results: a counting sort into 4096 mass buckets is
// as good as an exact sort and costs microseconds instead of half a millisecond of host time per call.)
std::vector<uint32_t> mass_order(const std::vector<md_precursor>& prec) {
  const uint32_t n = (uint32_t)prec.size();
  int64_t mlo = INT64_MAX, mhi = INT64_MIN;
  for (uint32_t s = 0; s < n; s++) { mlo = std::min(mlo, prec[s].mass); mhi = std::max(mhi, prec[s].mass); }
  constexpr uint32_t kBuckets = 4096;
  const double scale = mhi > mlo ? (double)(kBuckets - 1) / (double)(mhi - mlo) : 0.0;
  std::vector<uint32_t> head(kBuckets + 1, 0), bucket(n), order(n);
  for (uint32_t s = 0; s < n; s++) { bucket[s] = (uint32_t)((double)(prec[s].mass - mlo) * scale); head[bucket[s] + 1]++; }
  for (uint32_t b = 0; b < kBuckets; b++) head[b + 1] += head[b];
  for (uint32_t s = 0; s < n; s++) order[head[bucket[s]]++] = s;
  return order;
}

// The work items of one round: list entries of (spectrum, consecutive attempt ordinals), level by level.
struct RoundPlan {
  std::vector<uint32_t> list, off, base;   // per entry: spectrum, prefix of attempt counts (one more), first attempt ordinal
  std::vector<uint32_t> blk;               // coarse index into off (find_entry_coarse)
  uint32_t level_begin[kRoundLevels + 1] = {};
};

// How many attempts each unfinished spectrum gets in this round (count: its decoys so far; used: its attempts so far, of at
// most cap; visited in `order`).  A spectrum's decoys are its first n distinct successes in attempt order, so asking for too
// many only wastes work; asking for too few costs another round, and a round never takes less than one 100-try attempt
// (~0.3 ms) however small it is.  Round 0 asks for want0_pct % of the n still missing + 32; later rounds use the spectrum's
// own yield with later_factor head room (their attempts are the expensive ones: hard spectra), and rounds too small to fill
// the GPU ask for up to 4x that.  No entries: every spectrum has its decoys or has used up its attempts.
RoundPlan plan_round(const std::vector<uint32_t>& count, const std::vector<uint32_t>& used, const std::vector<uint32_t>& cap,
                     const std::vector<uint32_t>& order, uint32_t n_per, int round, uint32_t want0_pct, double later_factor) {
  std::vector<uint32_t> wants, todo;
  uint64_t sum = 0;
  for (const uint32_t s : order) {
    if (count[s] >= n_per || used[s] >= cap[s]) continue;
    uint32_t want;
    if (used[s] == 0) { const uint32_t rem = n_per - count[s]; want = (uint32_t)((uint64_t)rem * want0_pct / 100u) + 32; }
    else {
      double yield = std::max(0.02, (double)count[s] / (double)used[s]);
      want = (uint32_t)((double)(n_per - count[s]) / yield * later_factor) + 48;
    }
    want = std::min<uint32_t>({want, (uint32_t)(kMaxRoundAttempts * kRoundLevels), cap[s] - used[s]});
    todo.push_back(s); wants.push_back(want); sum += want;
  }
  const double boost = round == 0 || sum == 0 ? 1.0 : std::min(4.0, std::max(1.0, 300000.0 / (double)sum));
  // A list entry is at most kMaxRoundAttempts attempts of one spectrum (the selection kernel's table); a spectrum that gets
  // more this round -- the hard ones, which would otherwise need a round per 4096 attempts, each round as long as its slowest
  // attempt however few attempts it has -- has several entries with consecutive attempt ordinals.  The list holds every
  // spectrum's first entry, then the second entries, ...: k_decoy_select runs once per level, in that order.
  struct Entry { uint32_t s, n, base; };
  std::vector<Entry> level[kRoundLevels];
  uint64_t planned = 0;
  for (size_t i = 0; i < todo.size(); i++) {
    const uint32_t s = todo[i];
    const uint32_t want = std::min<uint32_t>({(uint32_t)((double)wants[i] * boost), (uint32_t)(kMaxRoundAttempts * kRoundLevels), cap[s] - used[s]});
    if (planned + want > 0x7FFFFFFFull) break;  // the rest waits for the next round
    planned += want;
    for (uint32_t c = 0, done = 0; done < want; c++) {
      const uint32_t chunk = std::min<uint32_t>(want - done, (uint32_t)kMaxRoundAttempts);
      level[c].push_back(Entry{s, chunk, used[s] + done});
      done += chunk;
    }
  }
  RoundPlan R;
  R.off.assign(1, 0);
  for (int c = 0; c < kRoundLevels; c++) {
    R.level_begin[c] = (uint32_t)R.list.size();
    for (const Entry& e : level[c]) { R.list.push_back(e.s); R.base.push_back(e.base); R.off.push_back(R.off.back() + e.n); }
  }
  R.level_begin[kRoundLevels] = (uint32_t)R.list.size();
  if (R.list.empty()) return R;
  // coarse index: entry of every 1024th work item (+ one past the end)
  const uint32_t n_list = (uint32_t)R.list.size(), total = R.off.back(), nb = (total >> kBlkLog) + 2;
  R.blk.resize(nb);
  for (uint32_t b = 0, e = 0; b < nb; b++) {
    const uint64_t w0 = std::min<uint64_t>((uint64_t)b << kBlkLog, total - 1);
    while (e + 1 < n_list && R.off[e + 1] <= w0) e++;
    R.blk[b] = e;
  }
  return R;
}

// The attempt kernels of one round: every work item of RA becomes one row of O (len 0: no decoy).  Returns whether
// ctx->ev_trace holds the round's per-kernel times.
bool launch_attempts(md_ctx* ctx, int mode, int vmode, bool wide_only, const RandomArgs& RA, const DecoyTables& T, const AttemptOut& O,
                     const PeptideView& PV) {
  IdentifyWorkspace& W = ctx->ws;
  const uint32_t total = RA.total;
  if (mode == MD_DECOY_PERMUTE_TARGET) {
    MD_LAUNCH(ctx, k_decoy_permute, blocks(total, kThreads), kThreads, 0, RA, T, W.cand_off.p, W.cand_desc.p, W.cand_mask.p, W.cand_w.p, ctx->index.rows.p,
              O, PV, ctx->mods);
    return false;
  }
  if (ctx->mods.has_terminal) {
    MD_LAUNCH(ctx, k_decoy_random_terminal, std::min<uint32_t>((total + kThreads - 1) / kThreads, (uint32_t)ctx->n_sm * 8u), kThreads, 0, RA, ctx->mods, T, O, PV);
    return false;
  }
  // grow every attempt; repair those up to 32 residues with 32-bit position masks, then the longer ones with 64-bit
  // masks; finish the hits.  The two lists keep the work-item order (spectra by mass: neighbouring lanes repair
  // sequences of similar length).
  const size_t tpad = ((size_t)total + 15) & ~(size_t)15;
  W.t_grown.need(2 * (size_t)total + 2); W.t_start.need(4 * (size_t)total + 4); W.t_route.need(2 * tpad); W.t_narrow.need((size_t)total + 1);
  W.t_wide.need((size_t)total + 1);
  GrownAttempt* grown = reinterpret_cast<GrownAttempt*>(W.t_grown.p);
  StartState* start = reinterpret_cast<StartState*>(W.t_start.p);
  uint8_t* to_narrow = W.t_route.p; uint8_t* to_wide = W.t_route.p + tpad;
  uint32_t* queue = W.t_queue.p;
  // (MD_TRACE: an event behind each step, printed with the round's line)
  auto trace_ev = [&](int i) { if (ctx->trace) MD_CUDA(cudaEventRecord(ctx->ev_trace[i], ctx->stream)); };
  MD_CUDA(cudaMemsetAsync(queue, 0, 4 * sizeof(uint32_t), ctx->stream));
  trace_ev(0);
  MD_LAUNCH(ctx, k_decoy_grow, blocks(total, kGrowThreads), kGrowThreads, 0, RA, T, O, grown, start, to_narrow, to_wide, wide_only ? 0u : 32u);
  trace_ev(1);
  cubx_select_flagged_index(ctx, to_narrow, W.t_narrow.p, queue + 1, total);
  cubx_select_flagged_index(ctx, to_wide, W.t_wide.p, queue + 3, total);
  trace_ev(2);
  const auto narrow = random_kernel<uint32_t>(vmode), wide = random_kernel<uint64_t>(vmode);
  const uint32_t grid = (total + kThreads - 1) / kThreads;
  if (!wide_only)
    MD_LAUNCH(ctx, narrow, std::min<uint32_t>(grid, (uint32_t)ctx->n_sm * (uint32_t)random_occupancy<uint32_t>(vmode)), kThreads, 0,
              (RepairArgs{W.t_narrow.p, queue + 1, queue, grown, start, RA.seed, RA.overflow}), ctx->mods, T, O);
  trace_ev(3);
  MD_LAUNCH(ctx, wide, std::min<uint32_t>(grid, (uint32_t)ctx->n_sm * (uint32_t)random_occupancy<uint64_t>(vmode)), kThreads, 0,
            (RepairArgs{W.t_wide.p, queue + 3, queue + 2, grown, start, RA.seed, RA.overflow}), ctx->mods, T, O);
  trace_ev(4);
  MD_LAUNCH(ctx, k_decoy_finish, blocks(total, 256), 256, 0, total, T, O, grown, PV);
  trace_ev(5);
  return ctx->trace;
}

// k_decoy_select once per level of the round, in level order (a spectrum's later entries see what its earlier ones kept),
// through the hash set when it fits shared memory, else the exact scan.
void launch_selects(md_ctx* ctx, const RoundPlan& R, const std::vector<uint32_t>& count, int round, uint32_t n, uint32_t n_per, const AttemptOut& O) {
  IdentifyWorkspace& W = ctx->ws;
  const DecoyOut D{W.dec_rows.p, W.dec_len.p, W.dec_mask.p, W.dec_w.p, W.dec_hash.p, W.dec_attempt.p, W.dec_count.p, (uint64_t)n * n_per};
  for (int c = 0; c < kRoundLevels; c++) {
    const uint32_t lb = R.level_begin[c], le = R.level_begin[c + 1];
    if (lb == le) continue;
    uint32_t need = 1, max_na = 1;                        // most (accepted + attempted) / attempted of one entry of this level
    for (uint32_t i = lb; i < le; i++) {
      const uint32_t na = R.off[i + 1] - R.off[i];
      need = std::max(need, std::min(n_per, count[R.list[i]] + c * (uint32_t)kMaxRoundAttempts) + na); max_na = std::max(max_na, na);
    }
    uint32_t slots = 1024; while ((uint64_t)slots * 3 < (uint64_t)need * 4) slots <<= 1;   // load factor <= 0.75 even if every attempt succeeded
    max_na = (max_na + 7u) & ~7u;
    const bool hashed = (size_t)slots * 12 + (size_t)max_na * 10 <= (size_t)(MD_SELECT_SMEM_MAX);
    if (!hashed) slots = 0;                                // the exact scan: hashes and kept list only
    const size_t smem = (size_t)slots * 12 + (size_t)max_na * 10;
    if (ctx->trace) fprintf(stderr, "[md_trace]   decoy select round %d level %d: entries=%u kernel=%s\n", round, c, le - lb, hashed ? "hash" : "n2");
    MD_CUDA(cudaFuncSetAttribute(k_decoy_select, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    MD_LAUNCH(ctx, k_decoy_select, le - lb, 256, smem, W.t_list.p + lb, W.t_off.p + lb, W.t_base.p + lb, n_per, slots, max_na, O, D);
  }
}

}  // namespace

void decoys_exhaustive_dev(md_ctx* ctx, uint32_t n, uint32_t n_per);  // exhaustive.cu

void decoys_generate_dev(md_ctx* ctx, uint32_t n, uint32_t n_per, int mode, uint64_t seed) {
  IdentifyWorkspace& W = ctx->ws; PeptideStore& P = ctx->peps;
  const size_t slots = (size_t)n * n_per;
  W.dec_rows.need(slots * MD_DECOY_ROW + 64); W.dec_len.need(slots + 1); W.dec_mask.need(slots + 1); W.dec_w.need(slots + 1);
  W.dec_hash.need(slots + 1); W.dec_attempt.need(slots + 1); W.dec_count.need(n + 1);
  MD_CUDA(cudaMemsetAsync(W.dec_count.p, 0, (n + 1) * sizeof(uint32_t), ctx->stream));
  if (!n || !n_per) return;
  if (mode == MD_DECOY_EXHAUSTIVE) {
    MD_REQUIRE(!ctx->mods.has_terminal, MD_ERR_UNSUPPORTED, "exhaustive decoys enumerate compositions: not defined with terminal modifications (the weight depends on the order)");
    decoys_exhaustive_dev(ctx, n, n_per); return;
  }
  MD_REQUIRE(mode == MD_DECOY_REFERENCE_RANDOM || mode == MD_DECOY_PERMUTE_TARGET, MD_ERR_INVALID, "unknown decoy mode");

  const DecoyTables T = make_tables(ctx->mods);
  if (mode == MD_DECOY_REFERENCE_RANDOM)
    for (int a = 0; a < MD_ALPHABET_SIZE; a++)
      MD_REQUIRE(T.mprime[a] > 0 && T.mprime[a] < (1 << 29) && T.var_a[a] > -(1 << 29) && T.var_a[a] < (1 << 29), MD_ERR_UNSUPPORTED,
                 "decoy generation works in 32-bit residuals: residue and modification masses must stay below 536 Da");
  PeptideView PV{(const unsigned long long*)P.ht_key.p, P.ht_val.p, P.ht_mask, P.seq.p, P.seq_off.p, P.len.p};
  // stored decoys come first (tasks/identification.rs:259-283); only the remainder is generated
  const bool stored = mode == MD_DECOY_REFERENCE_RANDOM && ctx->dindex.ready && ctx->dindex.n > 0;
  if (stored) decoys_reuse_dev(ctx, n, n_per);
  // per spectrum bookkeeping on the host: decoys so far, attempts used, attempt cap
  std::vector<uint32_t> count(n, 0), used(n, 0), cap(n);
  std::vector<md_precursor> hp(n);
  std::vector<uint64_t> h_cand_off(mode == MD_DECOY_PERMUTE_TARGET ? n + 1 : 0);
  MD_CUDA(cudaMemcpyAsync(hp.data(), W.prec.p, n * sizeof(md_precursor), cudaMemcpyDeviceToHost, ctx->stream));
  if (stored) MD_CUDA(cudaMemcpyAsync(count.data(), W.dec_count.p, n * sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx->stream));
  if (!h_cand_off.empty()) MD_CUDA(cudaMemcpyAsync(h_cand_off.data(), W.cand_off.p, (n + 1) * sizeof(uint64_t), cudaMemcpyDeviceToHost, ctx->stream));
  MD_CUDA(cudaStreamSynchronize(ctx->stream));
  const std::vector<uint32_t> by_mass = mass_order(hp);
  for (uint32_t s = 0; s < n; s++) {
    uint64_t c = md_attempt_cap(n_per);
    if (mode == MD_DECOY_PERMUTE_TARGET) c = std::min<uint64_t>(c, (h_cand_off[s + 1] - h_cand_off[s]) * 1000ull);
    cap[s] = (uint32_t)c;
  }
  // how try_variable_modifications runs inside the repair loop (see k_decoy_random)
  int vmode = 0;
  bool any_var_letter = false;
  for (int a = 0; a < MD_ALPHABET_SIZE; a++) any_var_letter |= ctx->mods.has_var[T.code_of_a[a]] != 0;
  if (ctx->mods.nvar > 0 && any_var_letter)
    vmode = (ctx->mods.var_simple_code >= 0 && md_alpha_of_code((uint32_t)ctx->mods.var_simple_code) >= 0) ? 1 : 2;
  const bool wide_only = getenv("MD_DECOY_WIDE_ONLY") != nullptr;   // debugging: skip the 32-bit pass
  const double later_factor = getenv("MD_DECOY_LATER_PCT") ? std::max(100, atoi(getenv("MD_DECOY_LATER_PCT"))) / 100.0 : 1.05;   // head room of the later rounds (swept on C2: 100..180 %)
  const uint32_t want0_pct = getenv("MD_DECOY_WANT0_PCT") ? (uint32_t)std::max(100, atoi(getenv("MD_DECOY_WANT0_PCT"))) : 110u;   // round 0 asks for n * 1.10 + 32 attempts (swept on C2: 100..160 %)
  W.t_list.need((size_t)n * kRoundLevels + 1); W.t_off.need((size_t)n * kRoundLevels + 2); W.t_base.need((size_t)n * kRoundLevels + 1); W.t_queue.need(4); W.t_ovf.need(1);
  MD_CUDA(cudaMemsetAsync(W.t_ovf.p, 0, sizeof(int), ctx->stream));
  for (int round = 0;; round++) {   // until every spectrum has its decoys or has used up its attempts (every round makes progress)
    const RoundPlan R = plan_round(count, used, cap, by_mass, n_per, round, want0_pct, later_factor);
    if (R.list.empty()) break;
    const uint32_t n_list = (uint32_t)R.list.size(), total = R.off.back(), nb = (uint32_t)R.blk.size();
    W.att_rows.need((size_t)total * MD_DECOY_ROW + 64); W.att_len.need(total + 1); W.att_mask.need(total + 1); W.att_w.need(total + 1); W.att_hash.need(total + 1);
    W.t_blk.need(nb);
    const AttemptOut O{W.att_rows.p, W.att_len.p, W.att_mask.p, W.att_w.p, W.att_hash.p};
    MD_CUDA(cudaMemcpyAsync(W.t_list.p, R.list.data(), n_list * sizeof(uint32_t), cudaMemcpyHostToDevice, ctx->stream));
    MD_CUDA(cudaMemcpyAsync(W.t_off.p, R.off.data(), (n_list + 1) * sizeof(uint32_t), cudaMemcpyHostToDevice, ctx->stream));
    MD_CUDA(cudaMemcpyAsync(W.t_base.p, R.base.data(), n_list * sizeof(uint32_t), cudaMemcpyHostToDevice, ctx->stream));
    MD_CUDA(cudaMemcpyAsync(W.t_blk.p, R.blk.data(), nb * sizeof(uint32_t), cudaMemcpyHostToDevice, ctx->stream));
    MD_CUDA(cudaEventRecord(ctx->ev[4], ctx->stream));
    const RandomArgs RA{W.prec.p, W.t_list.p, W.t_off.p, W.t_base.p, W.t_blk.p, total, seed, W.t_ovf.p};
    const bool split = launch_attempts(ctx, mode, vmode, wide_only, RA, T, O, PV);
    MD_CUDA(cudaEventRecord(ctx->ev[5], ctx->stream));
    ctx->mark("  attempts");
    launch_selects(ctx, R, count, round, n, n_per, O);
    MD_CUDA(cudaMemcpyAsync(count.data(), W.dec_count.p, n * sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx->stream));
    MD_CUDA(cudaStreamSynchronize(ctx->stream));
    ctx->mark("  select");
    for (uint32_t i = 0; i < n_list; i++) used[R.list[i]] += R.off[i + 1] - R.off[i];
    float ms = 0; cudaEventElapsedTime(&ms, ctx->ev[4], ctx->ev[5]); ctx->acc_ms_kdecoy += ms; ctx->acc_attempts += total;
    if (ctx->trace) fprintf(stderr, "[md_trace]   decoy round %d: spectra=%u attempts=%u kernel=%.3f ms\n", round, n_list, total, ms);
    if (split) {
      float t[5];
      for (int i = 0; i < 5; i++) MD_CUDA(cudaEventElapsedTime(&t[i], ctx->ev_trace[i], ctx->ev_trace[i + 1]));
      fprintf(stderr, "[md_trace]   decoy round %d kernels: grow=%.3f lists=%.3f narrow=%.3f wide=%.3f finish=%.3f ms\n", round, t[0], t[1], t[2], t[3], t[4]);
    }
  }
  const int ovf = d2h_scalar(ctx, W.t_ovf.p);
  MD_REQUIRE(ovf != 3, MD_ERR_DEVICE, "decoy generation: internal error (substitution filter disagrees with the mass search)");
  MD_REQUIRE(ovf != 2, MD_ERR_UNSUPPORTED, "decoy generation: |weight - precursor| left the 32-bit range (residue or modification masses above ~1000 Da?)");
  MD_REQUIRE(!ovf, MD_ERR_UNSUPPORTED, "variable-modification placement enumeration exceeds 2^22 subsets for one decoy");
}

void decoys_export(md_ctx* ctx, uint32_t n, uint32_t n_per, md_decoy_table* out) {
  IdentifyWorkspace& W = ctx->ws;
  memset(out, 0, sizeof(*out));
  const size_t slots = (size_t)n * n_per;
  std::vector<uint8_t> rows(slots * MD_DECOY_ROW + 1), len(slots + 1);
  std::vector<uint64_t> mask(slots + 1); std::vector<int64_t> w(slots + 1); std::vector<uint32_t> att(slots + 1), count(n + 1);
  if (slots) {
    MD_CUDA(cudaMemcpyAsync(rows.data(), W.dec_rows.p, slots * MD_DECOY_ROW, cudaMemcpyDeviceToHost, ctx->stream));
    MD_CUDA(cudaMemcpyAsync(len.data(), W.dec_len.p, slots, cudaMemcpyDeviceToHost, ctx->stream));
    MD_CUDA(cudaMemcpyAsync(mask.data(), W.dec_mask.p, slots * 8, cudaMemcpyDeviceToHost, ctx->stream));
    MD_CUDA(cudaMemcpyAsync(w.data(), W.dec_w.p, slots * 8, cudaMemcpyDeviceToHost, ctx->stream));
    MD_CUDA(cudaMemcpyAsync(att.data(), W.dec_attempt.p, slots * 4, cudaMemcpyDeviceToHost, ctx->stream));
  }
  if (n) MD_CUDA(cudaMemcpyAsync(count.data(), W.dec_count.p, n * 4, cudaMemcpyDeviceToHost, ctx->stream));
  MD_CUDA(cudaStreamSynchronize(ctx->stream));
  uint64_t total = 0, bytes = 0;
  for (uint32_t s = 0; s < n; s++) for (uint32_t j = 0; j < count[s]; j++) { total++; bytes += len[(size_t)s * n_per + j]; }
  out->n_spectra = n; out->n = total; out->seq_bytes = bytes;
  out->off = (uint64_t*)malloc((n + 1) * 8); out->seq = (uint8_t*)malloc(bytes + 1); out->seq_off = (uint64_t*)malloc((total + 1) * 8);
  out->var_mask = (uint64_t*)malloc((total + 1) * 8); out->weight = (int64_t*)malloc((total + 1) * 8); out->mod_weight = (int64_t*)malloc((total + 1) * 8);
  out->attempt = (uint32_t*)malloc((total + 1) * 4);
  uint64_t k = 0, b = 0;
  out->off[0] = 0; out->seq_off[0] = 0;
  for (uint32_t s = 0; s < n; s++) {
    for (uint32_t j = 0; j < count[s]; j++) {
      size_t slot = (size_t)s * n_per + j;
      uint32_t L = len[slot];
      int64_t wu = MD_WATER_UDA;
      for (uint32_t i = 0; i < L; i++) { uint8_t code = rows[md_dec_byte(slots, slot, i)]; out->seq[b + i] = md_letter_of(code); wu += kResidueMassByCode[code]; }
      b += L;
      out->seq_off[k + 1] = b; out->var_mask[k] = mask[slot]; out->weight[k] = wu; out->mod_weight[k] = w[slot]; out->attempt[k] = att[slot];
      k++;
    }
    out->off[s + 1] = k;
  }
}

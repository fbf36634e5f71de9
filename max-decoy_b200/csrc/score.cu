// score.cu -- K4: spectrum binning + the fused fragment-and-score kernel + per-spectrum top-k.
//
// The reference has no scorer: identification_task writes <spectrum>.fasta / .comet.params and an external Comet
// binary computes b/y cross-correlation (tasks/identification.rs:323-368; utility/comet_parameter.rs:6-124;
// run_splitup_and_identification.sh:47-60).  This file does that step in place, with a Comet-style fast xcorr
// consistent with the emitted parameters (b/y ions, monoisotopic fragments, fragment_bin_tol = tolerance,
// fragment_bin_offset = 0, theoretical_fragment_ions = 1 (no flanking), max_fragment_charge = 3) but defined in
// exact integers so that it is reproducible bit for bit (see oracle/maxdecoy_oracle.cpp, same definition):
//   bin(m/z)   = floor(m/z[uDa] / w) + 1,  w = fragment tolerance in uDa
//   y[bin]     = max over peaks of sqrt(I), scaled to 50 per tenth of the m/z range, peaks <= 5 % of the base peak dropped,
//                quantised to Q16
//   T[b]       = 151*y[b] - sum_{j=b-75..b+75} y[j]          (= 150 * 2^16 * fast_xcorr[b])
//   raw score  = sum over b/y fragments and fragment charges of T[bin];   score = 0.005 * raw / (150 * 2^16)
//
// Kernel design (B200): one persistent CTA of 768 threads per SM (spectra from a global queue).  T[b] is non-zero only
// within 75 bins of a peak, i.e. on a few hundred 64-bin blocks of the 100k+ bins a 0.02-Da table spans, so the CTA keeps
// a BLOCK-COMPRESSED table in shared memory: a 16-bit block map (bin >> 6 -> compressed block << 6 | 63, 0 = the all-zero block)
// plus up to 719 dense 64-bin blocks (180 KiB of int32).  A centroided MS2 spectrum (~100-400 peaks above the 5 %
// threshold) fits whole, so every candidate is walked ONCE; denser spectra fall back to several tiles of compressed
// blocks.  Build: peaks mark their blocks in a bitmap (shared-memory atomicOr), a warp scan numbers the blocks, the
// occupied blocks are zeroed with vectorised stores, every peak drops its window as a difference pair (+y at bin-75, -y
// at bin+76) and its spike as (-151y, +151y) with shared-memory atomics, and one block-wide inclusive scan straight over
// the compressed blocks turns the differences into -T (the running sum is 0 at the end of every run of occupied blocks,
// so the scan needs no notion of where the runs are).  Scoring: the
// candidates are counting-sorted by length into 32-candidate units that warps pull from a shared counter; a thread
// scores one candidate: 128-bit row loads, the per-letter (q, r) mass table in registers read by warp shuffle, a
// division-free running (Q, R) prefix, two shared-memory loads per fragment (block map, then table), a stop offset at
// the last residue instead of a per-residue length predicate, IMAD.WIDE accumulation.  Partial scores of a candidate
// chunk stay in shared memory across tiles; top-k packs (score, ordinal) into one 64-bit key, warp-local REDUX max,
// merged by warp 0 while the other warps already stage the next spectrum.  Only PSM rows go to HBM unless the
// caller asks for all scores.
#include "cubx.cuh"

#include <algorithm>

namespace {

inline uint32_t blocks(uint64_t n, uint32_t bs = 256) { return (uint32_t)((n + bs - 1) / bs); }

constexpr int kXcorrOffset = 75;
#ifndef MD_SCORE_THREADS
#define MD_SCORE_THREADS 768
#endif
constexpr int kScoreThreads = MD_SCORE_THREADS;
constexpr uint32_t kBlkShift = 6, kBlk = 1u << kBlkShift;      // table block = 64 bins
constexpr uint32_t kTileBins = 46080;      // 180 KiB of int32 per CTA = 720 blocks, block 0 is the all-zero block
constexpr uint32_t kTileBlocks = kTileBins / kBlk - 1;          // usable blocks per tile
static_assert(kTileBlocks < (1u << (16 - kBlkShift)), "a block-map entry holds the compressed block in its upper 10 bits");
constexpr uint32_t kMapCap = 6144;         // block-map entries staged in shared memory (393k bins; larger tables use an HBM map)
constexpr uint32_t kCandChunk = 1536;      // candidates whose partial scores stay in shared memory across tiles
constexpr uint32_t kPeakCap = 512;         // binned peaks staged in shared memory, double-buffered (larger spectra read them from HBM)
constexpr uint32_t kMaxBins = 1u << 26;    // table bins per spectrum (bins must stay far below kStop)
constexpr uint32_t kMaxTopK = 128;
constexpr uint32_t kFastTopK = 8;
constexpr uint32_t kMaxParts = 16;         // most work items a spectrum is split into (merge_parts)

// ------------------------------------------------------------------------------------------------
// precursor windows: tasks/identification.rs:203-211 (utility/mod.rs:9-11; models/mass/mod.rs:6-8,14-16)
// every operation rounded separately (no FMA), truncating conversion
// ------------------------------------------------------------------------------------------------
__global__ void k_precursors(const double* __restrict__ pmz, const uint8_t* __restrict__ charge, const uint32_t* __restrict__ sid, uint32_t n,
                             int64_t lppm, int64_t uppm, int64_t abs_lo, int64_t abs_hi, uint32_t id_base, md_precursor* __restrict__ out) {
  uint32_t s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= n) return;
  const double mz = pmz[s], zc = (double)charge[s], H = 1.007276;
  const double tl = __dmul_rn(__ddiv_rn(mz, 1000000.0), (double)lppm);
  const double tu = __dmul_rn(__ddiv_rn(mz, 1000000.0), (double)uppm);
  const double b = __dmul_rn(H, zc);
  int64_t P = (int64_t)__dmul_rn(__dsub_rn(__dmul_rn(mz, zc), b), 1000000.0);
  int64_t lo = (int64_t)__dmul_rn(__dsub_rn(__dmul_rn(__dsub_rn(mz, tl), zc), b), 1000000.0);
  int64_t hi = (int64_t)__dmul_rn(__dsub_rn(__dmul_rn(__dadd_rn(mz, tu), zc), b), 1000000.0);
  if (abs_lo != 0 || abs_hi != 0) { lo = P - abs_lo; hi = P + abs_hi; }
  md_precursor pr;
  pr.mass = P; pr.lo = lo; pr.hi = hi; pr.charge = charge[s]; pr.spectrum_id = sid ? sid[s] : id_base + s;
  out[s] = pr;
}

// ------------------------------------------------------------------------------------------------
// K4a: bin one spectrum per warp -> sorted unique (bin, yq) list
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ double warp_max_d(double v) {
  for (int o = 16; o; o >>= 1) { double t = __shfl_xor_sync(0xffffffffu, v, o); v = t > v ? t : v; }
  return v;
}
__device__ __forceinline__ int warp_max_i(int v) {
  for (int o = 16; o; o >>= 1) { int t = __shfl_xor_sync(0xffffffffu, v, o); v = t > v ? t : v; }
  return v;
}

struct PeakEval { bool valid; int32_t bin; double raw; };
__device__ __forceinline__ PeakEval eval_peak(double mz, float I, int64_t P, int64_t w) {
  PeakEval r; r.valid = false; r.bin = 0; r.raw = 0.0;
  if (!(I > 0.0f) || !(mz > 0.0) || !(mz < 1.0e7)) return r;
  int64_t mzint = (int64_t)__dmul_rn(mz, 1000000.0);
  if (!(mzint > 0) || !(mzint < P + 50000000LL)) return r;
  r.valid = true; r.bin = (int32_t)(mzint / w) + 1; r.raw = sqrt((double)I);
  return r;
}

__global__ void k_bin_spectra(const uint64_t* __restrict__ peak_off, const double* __restrict__ peak_mz, const float* __restrict__ peak_int,
                              const md_precursor* __restrict__ prec, uint32_t n, int64_t w, uint32_t min_peaks, int32_t* __restrict__ pk_bin,
                              int32_t* __restrict__ pk_yq, uint32_t* __restrict__ pk_count, int32_t* __restrict__ pk_hbin, int* __restrict__ unsorted) {
  const uint32_t s = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (s >= n) return;
  const uint64_t p0 = peak_off[s], p1 = peak_off[s + 1];
  const int64_t P = prec[s].mass;
  // pass A: base peak, highest bin, number of usable peaks, sortedness
  double gmax = 0.0; int hbin = 0; uint32_t nvalid = 0; bool bad = false;
  for (uint64_t i = p0 + lane; i < p1; i += 32) {
    double mz = peak_mz[i];
    if (i > p0 && mz < peak_mz[i - 1]) bad = true;
    PeakEval e = eval_peak(mz, peak_int[i], P, w);
    if (e.valid) { nvalid++; if (e.raw > gmax) gmax = e.raw; if (e.bin > hbin) hbin = e.bin; }
  }
  gmax = warp_max_d(gmax); hbin = warp_max_i(hbin);
  for (int o = 16; o; o >>= 1) nvalid += __shfl_xor_sync(0xffffffffu, nvalid, o);
  if (__any_sync(0xffffffffu, bad)) { if (lane == 0) *unsorted = 1; }
  if (nvalid < min_peaks || nvalid == 0) {
    if (lane == 0) { pk_count[s] = 0; pk_hbin[s] = -1; }  // not scored (Comet minimum_peaks, comet_parameter.rs:62)
    return;
  }
  // pass B: maximum per tenth of the bin range
  const int wsize = hbin / 10 + 1;
  double winmax[10];
#pragma unroll
  for (int k = 0; k < 10; k++) winmax[k] = 0.0;
  for (uint64_t i = p0 + lane; i < p1; i += 32) {
    PeakEval e = eval_peak(peak_mz[i], peak_int[i], P, w);
    if (e.valid) {
      int k = e.bin / wsize;
#pragma unroll
      for (int q = 0; q < 10; q++) if (q == k && e.raw > winmax[q]) winmax[q] = e.raw;
    }
  }
#pragma unroll
  for (int k = 0; k < 10; k++) winmax[k] = warp_max_d(winmax[k]);
  // pass C: emit runs of equal bins (peaks are sorted by m/z, so bins are non-decreasing)
  const double thr = __dmul_rn(0.05, gmax);
  int carry_bin = 0; uint32_t carry_cnt = 0;
  for (uint64_t base = p0; base < p1; base += 32) {
    uint64_t i = base + lane;
    PeakEval e; e.valid = false; e.bin = 0; e.raw = 0.0;
    if (i < p1) e = eval_peak(peak_mz[i], peak_int[i], P, w);
    const bool kept = e.valid && e.raw > thr;
    int32_t yq = 0;
    if (kept) {
      int k = e.bin / wsize; double wm = 0.0;
#pragma unroll
      for (int q = 0; q < 10; q++) if (q == k) wm = winmax[q];
      double y = __dmul_rn(e.raw, __ddiv_rn(50.0, wm));
      yq = (int32_t)__dadd_rn(__dmul_rn(y, 65536.0), 0.5);
    }
    // bin of the previous kept peak = exclusive prefix max over kept bins (0 = none)
    int v = kept ? e.bin : 0, incl = v;
    for (int o = 1; o < 32; o <<= 1) { int t = __shfl_up_sync(0xffffffffu, incl, o); if ((int)lane >= o && t > incl) incl = t; }
    int prev = __shfl_up_sync(0xffffffffu, incl, 1);
    if (lane == 0) prev = 0;
    if (carry_bin > prev) prev = carry_bin;
    const bool head = kept && e.bin != prev;
    const uint32_t hb = __ballot_sync(0xffffffffu, head);
    const uint32_t rank = __popc(hb & ((2u << lane) - 1));  // heads at or before this lane
    if (kept) {
      uint64_t o = p0 + carry_cnt + rank - 1;
      if (head) pk_bin[o] = e.bin;
      atomicMax(&pk_yq[o], yq);
    }
    carry_cnt += __popc(hb);
    int last = __shfl_sync(0xffffffffu, incl, 31);
    if (last > carry_bin) carry_bin = last;
  }
  if (lane == 0) { pk_count[s] = carry_cnt; pk_hbin[s] = hbin; }
}

// ------------------------------------------------------------------------------------------------
// K4: score
// ------------------------------------------------------------------------------------------------
struct ScoreConst {
  uint32_t w;                 // bin width, uDa
  float rcp_w;                // ~ 1/w
  uint32_t qp, rp;            // proton  = qp*w + rp
  uint32_t q2p, r2p;          // 2*proton
  uint32_t tq[32], tr[32];    // per residue code: (mass + fixed delta) = q*w + r
  uint32_t vq[32], vr[32];    // per residue code: (mass + fixed + variable delta)
  // per residue code: its letter's fixed N-terminus modification as floor-split (q, r) (q may be "negative", i.e. wrapped), added
  // to the b-ion prefix when the code is the first residue -- k_score only; with such a modification nothing runs through
  // k_score_pipe.  (C-terminus modifications need nothing here: no b ion holds the last residue, and the y ions come from
  // the candidate's modified weight; a variable terminal modification is a mask bit on the end residue like any other.)
  uint32_t nq[32], nr[32];
  uint32_t max_frag_charge;
  uint32_t top_k, n_per;
};

struct ScoreArgs {
  const md_precursor* prec; uint32_t n_spec;
  const uint64_t* peak_off; const int32_t* pk_bin; const int32_t* pk_yq; const uint32_t* pk_count; const int32_t* pk_hbin;
  const uint64_t* cand_off; const uint64_t* cand_desc; const uint64_t* cand_mask; const int64_t* cand_w; const uint32_t* cand_pep;
  const uint8_t* idx_rows;
  uint64_t dec_slots;   // decoy slots of the batch: the second halves of the decoy rows start dec_slots * 32 bytes in (md_dec_byte)
  const uint8_t* dec_rows; const uint8_t* dec_len; const uint64_t* dec_mask; const int64_t* dec_w; const uint32_t* dec_count;
  int64_t* tscore; int64_t* dscore;   // raw score of every candidate, or NULL (PSM rows only)
  md_psm* psm;
  uint32_t* work;
  unsigned long long* stat64;  // [0] pairs scored, [1] algorithmic bytes (14 + len per pair)
  int* error;                  // set when a spectrum needs more table bins than kMaxBins
  // spectra with very many candidates (open searches) are split into `parts` work items, one contiguous range of candidate
  // chunks each; a part leaves its K best keys in part_top and the last part to finish (parts_done) writes the PSM rows
  uint32_t parts; unsigned long long* part_top; uint32_t* parts_done;
  uint16_t* gmap; uint32_t* gbits; uint32_t gmap_stride;   // per-CTA block map / block bitmap in HBM for tables beyond kMapCap blocks
  // k_score's spectra: n_work of them, spectrum remap[i] (or i itself without a list) -- the whole batch, or the spectra
  // k_build_tables left to k_score
  uint32_t n_work; const uint32_t* remap;
};

__device__ __forceinline__ uint32_t div3(uint32_t x) { return __umulhi(x, 0xAAAAAAABu) >> 1; }

// (not volatile: the table does not change while candidates are scored against it, and the scheduler must be free to issue
// the independent loads of a residue's fragments back to back instead of one dependent map -> table pair after the other;
// the addresses derive from candidate rows loaded behind the barrier that publishes the table, so no load can move above it)
__device__ __forceinline__ int32_t lds_s32(uint32_t addr) {
  int32_t v;
  asm("ld.shared.s32 %0, [%1];" : "=r"(v) : "r"(addr));
  return v;
}
__device__ __forceinline__ uint32_t lds_u16(uint32_t addr) {
  uint32_t v;
  asm("ld.shared.u16 %0, [%1];" : "=r"(v) : "r"(addr));
  return v;
}
__device__ __forceinline__ void acc_wide(int64_t& acc, int32_t v) {  // acc += v as one IMAD.WIDE
  asm("mad.wide.s32 %0, %1, 1, %0;" : "+l"(acc) : "r"(v));
}
// The table as the scoring loop sees it: block map (shared memory address, or an HBM pointer when MAPG) + dense blocks.
struct TableView { uint32_t tab_s, map_s, nblk; const uint16_t* gmap; };
// one fragment: bin -> block (clamped onto the map's zero entry) -> compressed block -> table entry; branch-free
template <bool MAPG>
__device__ __forceinline__ int32_t gather(uint32_t bin, const TableView& V) {
  const uint32_t blk = min(bin >> kBlkShift, V.nblk);
  const uint32_t e = MAPG ? (uint32_t)V.gmap[blk] : lds_u16(V.map_s + 2u * blk);
  // e = (compressed block << 6) | 63, or 0: one AND yields the table index, and every fragment that misses reads the
  // same word (entry 0 of the all-zero block), which the shared-memory pipe serves as one broadcast instead of a
  // bank-conflicting random access
  const uint32_t t = e & (bin | ~(kBlk - 1u));
  return lds_s32(V.tab_s + (t << 2));
}
// the two halves of a gather: fragment bin -> table index (block map), table index -> entry
template <bool MAPG>
__device__ __forceinline__ uint32_t gather_index(uint32_t bin, const TableView& V) {
  const uint32_t blk = min(bin >> kBlkShift, V.nblk);
  const uint32_t e = MAPG ? (uint32_t)V.gmap[blk] : lds_u16(V.map_s + 2u * blk);
  return e & (bin | ~(kBlk - 1u));
}
__device__ __forceinline__ int32_t gather_entry(uint32_t t, const TableView& V) { return lds_s32(V.tab_s + (t << 2)); }
struct LaneTab { uint32_t q, r, vq, vr; };      // lane = residue code
constexpr uint32_t kStop = 1u << 30;            // added to the running bin at the last residue: every later bin misses

struct CandRef { const uint4* row; const uint4* row_hi; uint32_t len; uint64_t mask; int64_t modw; };   // row: bytes 0..31, row_hi: bytes 32..63

// Raw score of one candidate against the (tile of the) block-compressed table.
//   b ion of split k, charge c: floor((B_k + c*proton) / (c*w)) + 1;  y ion: floor((modw - B_k + c*proton) / (c*w)) + 1
// with X = B_k + proton kept as (Q, R), X = Q*w + R, R < w, so no fragment needs a division.  QB = Q + 1 is the charge-1
// b bin itself; bins past the table, and the wrapped "negative" ones, are clamped onto the map's zero entry by one
// unsigned min.  The last residue is never a prefix: at position len-1 kStop is added to QB, which throws every later
// b and y bin of every charge out of the table -- no per-residue length predicate.  The loop runs in 4-residue words up
// to the longest candidate of the warp.
template <int NCH, bool HASVAR, bool MAPG, bool TERM = false>
__device__ __forceinline__ int64_t score_one(const CandRef& cr, uint32_t maxlen, const TableView& V, const ScoreConst& C, const LaneTab& L) {
  const uint32_t w = C.w;
  const uint32_t K2 = C.qp - 1u, K3 = C.q2p - 1u;
  const uint32_t nword = maxlen > 1 ? (maxlen - 1 + 3) >> 2 : 0;  // warp-uniform
  // T_c = modw + (c+1)*proton  ->  (Qt, Rt)
  const uint64_t T1 = (uint64_t)cr.modw + 2ull * MD_PROTON_UDA;
  // T1 = Qt1*w + Rt1 without the 64-bit division routine (~100 instructions per candidate): float estimate of the
  // quotient (T1 < 2^34, so it is off by a few units at most), exact remainder, stepwise correction
  uint32_t Qt1 = (uint32_t)__fmul_rz((float)T1, C.rcp_w);
  int64_t rem = (int64_t)T1 - (int64_t)((uint64_t)Qt1 * w);
  while (rem < 0) { Qt1--; rem += w; }
  while (rem >= (int64_t)w) { Qt1++; rem -= w; }
  const uint32_t Rt1 = (uint32_t)rem;
  uint32_t Qt2 = Qt1 + C.qp, Rt2 = Rt1 + C.rp; if (Rt2 >= w) { Rt2 -= w; Qt2++; }
  uint32_t Qt3 = Qt2 + C.qp, Rt3 = Rt2 + C.rp; if (Rt3 >= w) { Rt3 -= w; Qt3++; }
  const uint32_t Y1 = Qt1 + 2u;               // y1 bin = Y1 - QB - borrow
  const uint32_t Y2 = Qt2 + 1u, Y3 = Qt3 + 1u;  // Qt_c - Q - borrow = Y_c - QB - borrow, then halved / divided by 3, + 1
  uint32_t QB = C.qp + 1u, R1 = C.rp;         // X = B_k + proton
  const uint32_t nsplit = cr.len > 0 ? cr.len - 1 : 0;   // residues 0..len-2 are followed by a split
  if (nsplit == 0) QB += kStop;
  int64_t acc = 0;
  // (the first two 16-residue chunks are requested together: one round trip to L2 / HBM instead of two for the usual 17..32-residue candidate)
  const uint4 v0 = __ldg(cr.row);
  uint4 v1 = make_uint4(0u, 0u, 0u, 0u);
  if (nword > 4) v1 = __ldg(cr.row + 1);
  if (TERM) {   // a fixed N-terminus modification of the first residue's letter is part of every b ion
    const uint32_t code0 = v0.x & 31u;
    QB += C.nq[code0]; R1 += C.nr[code0];
    if (R1 >= w) { R1 -= w; QB++; }
  }
  for (uint32_t c = 0; c * 4 < nword; c++) {
    const uint4 v = c == 0 ? v0 : (c == 1 ? v1 : __ldg(cr.row_hi + (c - 2)));
    const uint32_t words[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
    for (int k = 0; k < 4; k++) {
      if (c * 4 + k >= nword) break;
#pragma unroll
      for (int j = 0; j < 4; j++) {
        const uint32_t pos = c * 16 + k * 4 + j;
        const uint32_t code = words[k] >> (8 * j);            // (shfl takes the source lane modulo 32; codes are < 32)
        uint32_t q = __shfl_sync(0xffffffffu, L.q, code), r = __shfl_sync(0xffffffffu, L.r, code);
        if (HASVAR) {
          const uint32_t qv = __shfl_sync(0xffffffffu, L.vq, code), rv = __shfl_sync(0xffffffffu, L.vr, code);
          if ((cr.mask >> pos) & 1) { q = qv; r = rv; }
        }
        QB += q; R1 += r;
        if (R1 >= w) { R1 -= w; QB++; }
        // |T| <= 151 * 50 * 2^16 < 2^29: up to four entries add up in 32 bits, then one IMAD.WIDE into the 64-bit score
        // all block-map loads of the residue first, then all table loads: the fragments are independent of one another
        const uint32_t ib1 = gather_index<MAPG>(QB, V), iy1 = gather_index<MAPG>(Y1 - QB - (Rt1 < R1 ? 1u : 0u), V);     // fragment charge 1
        uint32_t ib2 = 0, iy2 = 0, ib3 = 0, iy3 = 0;
        if (NCH >= 2) {
          ib2 = gather_index<MAPG>(((QB + K2 + (R1 + C.rp >= w ? 1u : 0u)) >> 1) + 1u, V);
          iy2 = gather_index<MAPG>(((Y2 - QB - (Rt2 < R1 ? 1u : 0u)) >> 1) + 1u, V);
        }
        if (NCH >= 3) {
          ib3 = gather_index<MAPG>(div3(QB + K3 + (R1 + C.r2p >= w ? 1u : 0u)) + 1u, V);
          iy3 = gather_index<MAPG>(div3(Y3 - QB - (Rt3 < R1 ? 1u : 0u)) + 1u, V);
        }
        int32_t s4 = gather_entry(ib1, V) + gather_entry(iy1, V);
        if (NCH >= 2) s4 += gather_entry(ib2, V) + gather_entry(iy2, V);
        acc_wide(acc, s4);
        if (NCH >= 3) acc_wide(acc, gather_entry(ib3, V) + gather_entry(iy3, V));
        if (pos + 1 == nsplit) QB += kStop;   // the next residue is the last one
      }
    }
  }
  return acc;
}

// (without variable modifications every mask is 0: not read)
template <bool HASVAR>
__device__ __forceinline__ CandRef cand_ref(const ScoreArgs& A, uint32_t s, uint32_t v, uint32_t nt, uint64_t t0c, uint32_t n_per) {
  CandRef r;
  if (v < nt) {
    const uint64_t c = t0c + v, d = A.cand_desc[c];
    r.row = reinterpret_cast<const uint4*>(A.idx_rows + (d & 0xFFFFFFFFFFull) * 16); r.row_hi = r.row + 2;
    r.len = (uint32_t)(d >> 40) & 0xFF; r.mask = HASVAR ? A.cand_mask[c] : 0ull; r.modw = A.cand_w[c];
  } else {
    const uint64_t j = (uint64_t)s * n_per + (v - nt);
    r.row = reinterpret_cast<const uint4*>(A.dec_rows + j * MD_DECOY_HALF); r.row_hi = reinterpret_cast<const uint4*>(A.dec_rows + (A.dec_slots + j) * MD_DECOY_HALF);
    r.len = A.dec_len[j]; r.mask = HASVAR ? A.dec_mask[j] : 0ull; r.modw = A.dec_w[j];
  }
  return r;
}

// PSM order: raw score descending, candidate ordinal ascending  <=>  key descending
constexpr int64_t kKeyBias = 1ll << 39;
__device__ __forceinline__ unsigned long long psm_key(int64_t score, uint32_t v) {
  return ((unsigned long long)(score + kKeyBias) << 24) | (unsigned long long)(0xFFFFFFu - v);
}
__device__ __forceinline__ unsigned long long warp_max_u64(unsigned long long k) {
  const uint32_t hi = (uint32_t)(k >> 32);
  const uint32_t mh = __reduce_max_sync(0xffffffffu, hi);
  const uint32_t ml = __reduce_max_sync(0xffffffffu, hi == mh ? (uint32_t)k : 0u);
  return ((unsigned long long)mh << 32) | ml;
}

__device__ __forceinline__ void write_psm_row(const ScoreArgs& A, const ScoreConst& C, const md_precursor& pr, uint32_t s, uint32_t r, unsigned long long k,
                                              uint32_t nt, uint32_t nd, uint64_t t0c) {
  md_psm row;
  row.spectrum_id = pr.spectrum_id; row.rank = 0; row.is_decoy = 0; row.charge = (uint8_t)pr.charge; row.candidate = 0; row.var_mask = 0;
  row.mod_weight = 0; row.raw_score = 0; row.score = 0.0f; row.n_targets = nt; row.n_decoys = nd; row._pad = 0;
  if (k != 0ull) {
    const uint32_t bv = 0xFFFFFFu - (uint32_t)(k & 0xFFFFFFull);
    const int64_t bs = (int64_t)(k >> 24) - kKeyBias;
    row.rank = (uint16_t)(r + 1); row.raw_score = bs;
    row.score = (float)(0.005 * (double)bs / (150.0 * 65536.0));
    if (bv < nt) { row.is_decoy = 0; row.candidate = (uint64_t)A.cand_pep[t0c + bv] + 1; row.var_mask = A.cand_mask[t0c + bv]; row.mod_weight = A.cand_w[t0c + bv]; }
    else { const uint64_t j = (uint64_t)s * C.n_per + (bv - nt); row.is_decoy = 1; row.candidate = bv - nt; row.var_mask = A.dec_mask[j]; row.mod_weight = A.dec_w[j]; }
  }
  A.psm[(uint64_t)s * C.top_k + r] = row;
}


// One warp's share of a tile pass: units of 32 candidates in length-descending order (s_order), fetched from a
// shared counter, so that warps stay busy until the chunk is done and every warp runs candidates of one length.
template <int NCH, bool HASVAR, bool MAPG>
__device__ __forceinline__ void score_units(const ScoreArgs& A, const ScoreConst& C, uint32_t s, uint32_t c0, uint32_t cn, uint32_t nt, uint64_t t0c,
                                            const TableView& V, const LaneTab& L, int64_t* s_score, const uint16_t* s_order, uint32_t* s_unit) {
  const uint32_t lane = threadIdx.x & 31, units = (cn + 31) >> 5;
  for (;;) {
    uint32_t u = 0;
    if (lane == 0) u = atomicAdd(s_unit, 1u);
    u = __shfl_sync(0xffffffffu, u, 0);
    if (u >= units) break;
    const uint32_t slot = u * 32 + lane;
    CandRef cr;
    cr.row = reinterpret_cast<const uint4*>(A.idx_rows); cr.row_hi = cr.row; cr.len = 0; cr.mask = 0; cr.modw = 0;
    uint32_t v = 0;
    if (slot < cn) {
      v = s_order[slot];
      cr = cand_ref<HASVAR>(A, s, c0 + v, nt, t0c, C.n_per);
    }
    const uint32_t maxlen = __reduce_max_sync(0xffffffffu, cr.len);
    const int64_t part = score_one<NCH, HASVAR, MAPG, true>(cr, maxlen, V, C, L);
    if (slot < cn) s_score[v] += part;
  }
}

// What the prefetch warp leaves for the next spectrum of the CTA (double-buffered with the staged peaks, the block bitmap
// and the sorted candidate order).
struct SpecMeta {
  md_precursor pr;
  uint64_t t0c, pk0;
  uint32_t s, nt, nd, npk, nact;
  uint32_t part, c_lo, c_hi;         // this work item's part of the spectrum: candidates [c_lo, c_hi)
  int32_t hbin;
  uint32_t pre_blocks;               // peaks, bitmap and block numbering are already in shared memory
};

struct FinRecord { md_precursor pr; uint64_t t0c; uint32_t s, nt, nd, pending, ranked, part; };

struct SpecShared {
  SpecMeta meta[2];
  unsigned long long wkey[2][kScoreThreads / 32];
  unsigned long long top[kMaxTopK];
  unsigned long long wtop[2][kScoreThreads / 32][kFastTopK];  // per-warp best keys of a spectrum, descending
  FinRecord fin[2];         // what the finish warp needs to write that spectrum's PSM rows
  uint32_t hist[64];        // candidates per length (counting sort of a chunk by the whole CTA)
  uint32_t unit;            // next unit of the current tile pass
  uint32_t nact;            // occupied table blocks of the spectrum
  uint32_t x0; int32_t cin; // first bin of the current tile, running sum in front of it
  uint32_t wsum[kScoreThreads / 32];
  uint32_t bits[2][kMapCap / 32], bpre[2][kMapCap / 32];   // occupied-block bitmap and its exclusive popcount prefix
};

__device__ __forceinline__ void cp_async4(void* smem_dst, const void* gsrc) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"((uint32_t)__cvta_generic_to_shared(smem_dst)), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.commit_group;\n\tcp.async.wait_group 0;" ::: "memory"); }

__device__ __forceinline__ uint32_t cand_len(const ScoreArgs& A, uint32_t s, uint32_t u, uint32_t nt, uint64_t t0c, uint32_t n_per) {
  return u < nt ? (uint32_t)(A.cand_desc[t0c + u] >> 40) & 0xFF : A.dec_len[(uint64_t)s * n_per + (u - nt)];
}

// One warp: the exclusive popcount prefix of the occupied-block bitmap bits[0, nwords) into pre[] (the compressed block of
// the first occupied block of each word); returns the number of occupied blocks to every lane.
__device__ __forceinline__ uint32_t warp_bitmap_prefix(const uint32_t* bits, uint32_t* pre, uint32_t nwords) {
  const uint32_t lane = threadIdx.x & 31;
  uint32_t run = 0;
  for (uint32_t base = 0; base < nwords; base += 32) {
    const uint32_t i = base + lane;
    const uint32_t c = i < nwords ? (uint32_t)__popc(bits[i]) : 0u;
    uint32_t incl = c;
    for (int o = 1; o < 32; o <<= 1) { const uint32_t t = __shfl_up_sync(0xffffffffu, incl, o); if ((int)lane >= o) incl += t; }
    if (i < nwords) pre[i] = run + incl - c;
    run += __shfl_sync(0xffffffffu, incl, 31);
  }
  return run;
}

// One warp: the 64-bucket length histogram of a counting sort, in place, into its exclusive prefix (each bucket's first slot).
__device__ __forceinline__ void warp_hist64_prefix(uint32_t* hist) {
  const uint32_t lane = threadIdx.x & 31;
  const uint32_t h0 = hist[2 * lane], h1 = hist[2 * lane + 1];
  uint32_t incl = h0 + h1;
  for (int o = 1; o < 32; o <<= 1) { const uint32_t t = __shfl_up_sync(0xffffffffu, incl, o); if ((int)lane >= o) incl += t; }
  hist[2 * lane] = incl - h0 - h1; hist[2 * lane + 1] = incl - h1;
}

// A spectrum split into parts: the work item leaves its K best keys (lane r: its r-th best).  The last part of the spectrum to
// arrive merges them all (lane r gets the spectrum's r-th best key) and its warp writes the rows; the others get last = false.
// (The key comes back by value: an out-parameter would keep the caller's key in local memory.)
struct PartMerge { bool last; unsigned long long best; };
__device__ __noinline__ PartMerge merge_parts(const ScoreArgs& A, uint32_t s, uint32_t part, uint32_t parts, uint32_t K, unsigned long long best) {
  const uint32_t lane = threadIdx.x & 31;
  unsigned long long* pt = A.part_top + (size_t)s * parts * kFastTopK;
  if (lane < kFastTopK) pt[part * kFastTopK + lane] = lane < K ? best : 0ull;
  __threadfence();
  __syncwarp();
  uint32_t arrived = 0;
  if (lane == 0) arrived = atomicAdd(&A.parts_done[s], 1u);
  arrived = __shfl_sync(0xffffffffu, arrived, 0);
  if (arrived + 1 != parts) return PartMerge{false, 0ull};
  __threadfence();
  static_assert(kMaxParts * kFastTopK <= 128, "a lane merges at most four keys of the parts' lists");
  unsigned long long k[4];
#pragma unroll
  for (int j = 0; j < 4; j++) k[j] = lane + 32u * j < parts * kFastTopK ? __ldcg(pt + lane + 32u * j) : 0ull;
  best = 0ull;
  for (uint32_t r = 0; r < K; r++) {
    unsigned long long m = k[0];
#pragma unroll
    for (int j = 1; j < 4; j++) m = k[j] > m ? k[j] : m;
    const unsigned long long wm = warp_max_u64(m);
    if (wm != 0ull) {
      bool gone = false;     // (keys are unique: at most one of the lane's four matches)
#pragma unroll
      for (int j = 0; j < 4; j++) if (!gone && k[j] == wm) { k[j] = 0ull; gone = true; }
    }
    if (lane == r) best = wm;
  }
  return PartMerge{true, best};
}

// Run by ONE warp while the others score: take the CTA's next spectrum from the queue and leave in shared memory what
// its iteration would otherwise wait for -- the precursor and candidate ranges, the binned peaks (cp.async) and the
// occupied-block bitmap with its numbering.
__device__ __noinline__ void prefetch_spectrum(const ScoreArgs& A, SpecShared& sh, uint32_t slot, int32_t* s_bin, int32_t* s_yq) {
  const uint32_t lane = threadIdx.x & 31;
  uint32_t vn = 0;
  if (lane == 0) vn = atomicAdd(A.work, 1u);
  vn = __shfl_sync(0xffffffffu, vn, 0);
  const uint32_t wn = vn / A.parts;          // work item -> (spectrum, part); sn >= n_spec ends the CTA
  const uint32_t sn = wn < A.n_work ? (A.remap ? A.remap[wn] : wn) : A.n_spec;
  SpecMeta m;
  m.part = vn % A.parts; m.c_lo = 0; m.c_hi = 0;
  m.s = sn; m.pre_blocks = 0; m.nact = 0; m.nt = 0; m.nd = 0; m.npk = 0; m.hbin = -1; m.t0c = 0; m.pk0 = 0;
  m.pr.mass = 0; m.pr.lo = 0; m.pr.hi = 0; m.pr.charge = 0; m.pr.spectrum_id = 0;
  if (sn < A.n_spec) {
    m.pr = A.prec[sn];
    m.t0c = A.cand_off[sn];
    m.nt = (uint32_t)(A.cand_off[sn + 1] - m.t0c);
    m.nd = A.dec_count ? A.dec_count[sn] : 0;
    m.hbin = A.pk_hbin[sn]; m.npk = A.pk_count[sn]; m.pk0 = A.peak_off[sn];
    const uint32_t NB = m.hbin >= 0 ? (uint32_t)m.hbin + kXcorrOffset + 1 : 0;
    const uint32_t nblk = (NB + kBlk - 1) >> kBlkShift, nwords = (nblk + 31) >> 5;
    const uint32_t ncand = m.nt + m.nd;
    {   // this part's contiguous range of candidate chunks
      const uint32_t nchunks = (ncand + kCandChunk - 1) / kCandChunk, per = (nchunks + A.parts - 1) / A.parts;
      m.c_lo = min(m.part * per * kCandChunk, ncand); m.c_hi = min((m.part + 1) * per * kCandChunk, ncand);
    }
    const bool scored = m.hbin >= 0 && NB <= kMaxBins && ncand <= 0xFFFFFFu;
    if (scored && m.npk <= kPeakCap && nblk <= kMapCap) {
      const int32_t* gb = A.pk_bin + m.pk0; const int32_t* gy = A.pk_yq + m.pk0;
      int32_t* sb = s_bin + slot * kPeakCap; int32_t* sy = s_yq + slot * kPeakCap;
      for (uint32_t i = lane; i < m.npk; i += 32) { cp_async4(sb + i, gb + i); cp_async4(sy + i, gy + i); }
      uint32_t* bits = sh.bits[slot]; uint32_t* bpre = sh.bpre[slot];
      for (uint32_t i = lane; i < nwords; i += 32) bits[i] = 0;
      cp_async_wait_all();
      __syncwarp();
      for (uint32_t p = lane; p < m.npk; p += 32) {     // every bin within 75 of a peak, and the bin behind
        const int32_t b = sb[p];
        const uint32_t b0 = (uint32_t)max(b - kXcorrOffset, 0) >> kBlkShift, b1 = min((uint32_t)(b + kXcorrOffset + 1), NB - 1) >> kBlkShift;
        for (uint32_t k = b0; k <= b1; k++) atomicOr(&bits[k >> 5], 1u << (k & 31));
      }
      __syncwarp();
      m.nact = warp_bitmap_prefix(bits, bpre, nwords); m.pre_blocks = 1;
    }
  }
  __syncwarp();
  if (lane == 0) sh.meta[slot] = m;
}

// Run by ONE warp while the others score the next spectrum: merge the per-warp top-k lists of spectrum fin[slot] (lane r
// ends up with its r-th best key) and write its PSM rows.
__device__ __noinline__ void finish_spectrum(const ScoreArgs& A, const ScoreConst& C, SpecShared& sh, uint32_t slot) {
  const FinRecord f = sh.fin[slot];
  if (!f.pending) return;
  const uint32_t lane = threadIdx.x & 31, K = C.top_k;
  constexpr uint32_t NW = kScoreThreads / 32;
  unsigned long long mine = 0ull;
  if (f.ranked) {
    uint32_t idx = 0;
    for (uint32_t r = 0; r < K; r++) {
      const unsigned long long head = (lane < NW && idx < K) ? sh.wtop[slot][lane][idx] : 0ull;
      const unsigned long long wm = warp_max_u64(head);
      if (wm != 0ull && head == wm) idx++;
      if (lane == r) mine = wm;
    }
  }
  if (A.parts > 1) {
    const PartMerge pm = merge_parts(A, f.s, f.part, A.parts, K, mine);
    if (!pm.last) return;
    mine = pm.best;
  }
  if (lane < K) write_psm_row(A, C, f.pr, f.s, lane, mine, f.nt, f.nd, f.t0c);
}

// MODE 0: no spectrum of the batch has more candidates than one chunk (the usual 10-ppm search: the chunk loop runs once,
// known at compile time); 1: general; 2: general, and spectra are divided into parts (ScoreArgs::parts > 1)
template <bool HASVAR, int MODE>
__global__ void __launch_bounds__(kScoreThreads, 1) k_score(const __grid_constant__ ScoreArgs A, const __grid_constant__ ScoreConst C) {
  extern __shared__ __align__(16) int32_t tab[];                     // kTileBins
  int64_t* s_score = reinterpret_cast<int64_t*>(tab + kTileBins);    // kCandChunk
  int32_t* s_bin = reinterpret_cast<int32_t*>(s_score + kCandChunk); // 2 x kPeakCap
  int32_t* s_yq = s_bin + 2 * kPeakCap;                              // 2 x kPeakCap
  uint16_t* s_order = reinterpret_cast<uint16_t*>(s_yq + 2 * kPeakCap);   // kCandChunk: chunk slots in length-descending order
  uint16_t* s_map = s_order + kCandChunk;                            // kMapCap + 2
  __shared__ SpecShared sh;
  const uint32_t tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  constexpr uint32_t NW = kScoreThreads / 32;
  // two warps start every scoring phase with a side job: one fetches the CTA's next spectrum, the other merges the
  // per-warp top-k lists of the previous spectrum and writes its PSM rows -- both off the critical path
  constexpr uint32_t kPrefetchWarp = NW - 1, kFinishWarp = NW - 2;
  const LaneTab L{C.tq[lane], C.tr[lane], C.vq[lane], C.vr[lane]};   // per-letter (q, r) tables in registers: lane = residue code
  uint32_t my_pairs = 0, my_bytes = 0;   // per thread, summed at the end

  if (warp == kPrefetchWarp) prefetch_spectrum(A, sh, 0, s_bin, s_yq);
  if (tid < 2) sh.fin[tid].pending = 0;
  for (uint32_t it = 0;; it++) {
    const uint32_t slot = it & 1;
    __syncthreads();                  // this spectrum's prefetch is visible; the other slot's buffers are free again
    const SpecMeta mt = sh.meta[slot];
    const uint32_t s = mt.s;
    if (s >= A.n_spec) {
      if (warp == kFinishWarp && it > 0) finish_spectrum(A, C, sh, slot ^ 1u);     // the CTA's last spectrum
      break;
    }
    bool side_done = false;           // (helper warps) this iteration's side job is done
    const md_precursor pr = mt.pr;
    const uint64_t t0c = mt.t0c;
    const uint32_t nt = mt.nt, nd = mt.nd;
    const uint32_t ncand = nt + nd;
    const int32_t hbin = mt.hbin;
    const uint32_t npk = mt.npk;
    const uint64_t pk0 = mt.pk0;
    const uint32_t K = C.top_k;
    uint32_t nch = pr.charge > 1 ? pr.charge - 1 : 1;
    if (nch > C.max_frag_charge) nch = C.max_frag_charge;
    if (nch < 1) nch = 1;
    const uint32_t NB = hbin >= 0 ? (uint32_t)hbin + kXcorrOffset + 1 : 0;  // table bins [0, NB)
    const uint32_t nblk = (NB + kBlk - 1) >> kBlkShift;
    bool scored = hbin >= 0;
    const bool mapg = nblk > kMapCap;
    if (NB > kMaxBins || ncand > 0xFFFFFFu || (mapg && (!A.gmap || nblk + 1 > A.gmap_stride))) { if (tid == 0) *A.error = 1; scored = false; }
    uint16_t* map = mapg ? A.gmap + (size_t)blockIdx.x * A.gmap_stride : s_map;
    uint32_t* bits = mapg ? A.gbits + (size_t)blockIdx.x * 2 * (A.gmap_stride / 32 + 1) : sh.bits[slot];
    uint32_t* bpre = mapg ? bits + (A.gmap_stride / 32 + 1) : sh.bpre[slot];
    const uint32_t nwords = (nblk + 31) >> 5;
    const int32_t* pbin = A.pk_bin + pk0; const int32_t* pyq = A.pk_yq + pk0;
    if (npk <= kPeakCap && mt.pre_blocks) { pbin = s_bin + slot * kPeakCap; pyq = s_yq + slot * kPeakCap; }
    for (uint32_t r = tid; r < K; r += kScoreThreads) sh.top[r] = 0ull;

    if (scored && !mt.pre_blocks) {
      // ---- (spectra the prefetch warp left alone: more peaks or table blocks than the shared-memory staging holds)
      for (uint32_t i = tid; i < nwords; i += kScoreThreads) bits[i] = 0;
      __syncthreads();
      for (uint32_t p = tid; p < npk; p += kScoreThreads) {   // every bin within 75 of a peak, and the bin behind
        const int32_t b = pbin[p];
        const uint32_t b0 = (uint32_t)max(b - kXcorrOffset, 0) >> kBlkShift, b1 = min((uint32_t)(b + kXcorrOffset + 1), NB - 1) >> kBlkShift;
        for (uint32_t k = b0; k <= b1; k++) atomicOr(&bits[k >> 5], 1u << (k & 31));
      }
      __syncthreads();
      if (warp == 0) {
        const uint32_t run = warp_bitmap_prefix(bits, bpre, nwords);
        if (lane == 0) sh.nact = run;
      }
      __syncthreads();
    }
    const uint32_t nact = scored ? (mt.pre_blocks ? mt.nact : sh.nact) : 0;

    const bool fast = K <= kFastTopK;   // per-warp running top-k lists, merged by the finish warp while the CTA scores the next spectrum
    // the table of one tile of occupied blocks [cb0, cb0 + cbn) (block-uniform: every thread calls it)
    auto build_tile = [&](const uint32_t cb0, const uint32_t cbn) {
      // (1) block map of the tile (0 = the all-zero block), zero the occupied blocks
      for (uint32_t k = tid; k <= nblk; k += kScoreThreads) {
        uint32_t m = 0;
        if (k < nblk) {
          const uint32_t wd = bits[k >> 5];
          if ((wd >> (k & 31)) & 1u) {
            const uint32_t c = bpre[k >> 5] + (uint32_t)__popc(wd & ((1u << (k & 31)) - 1u));
            if (c >= cb0 && c < cb0 + cbn) m = c - cb0 + 1u;
          }
        }
        map[k] = (uint16_t)(m ? (m << kBlkShift) | (kBlk - 1u) : 0u);
        if (m == 1u) sh.x0 = k << kBlkShift;                              // first bin of the tile
      }
      {
        uint4* z = reinterpret_cast<uint4*>(tab);
        const uint32_t n4 = (cbn + 1u) * (kBlk / 4);
        for (uint32_t i = tid; i < n4; i += kScoreThreads) z[i] = make_uint4(0, 0, 0, 0);
        if (tid == 0) { sh.unit = 0; sh.cin = 0; }
      }
      __syncthreads();
      // (2) T as a difference array: every peak adds +y at the first bin of its window (bin-75), -y behind its last
      //     (bin+76), and its own 151*y spike as -151*y at bin / +151*y at bin+1, so that the running sum over the
      //     bins is R[b] = S[b] - 151*y[b] = -T[b].  All four bins lie in occupied blocks (the marking covers
      //     [bin-75, bin+76]), R is 0 at the end of every run of occupied blocks, and the compressed blocks are in
      //     bin order: one inclusive scan straight over the compressed table yields -T.  Integer adds commute, so
      //     the shared-memory atomics keep the table exact.  A later tile starts from the sum of the differences
      //     at the bins in front of it (sh.cin).
      {
        const uint32_t X0 = sh.x0;
        int32_t cin = 0;
        for (uint32_t p = tid; p < npk; p += kScoreThreads) {
          const int32_t bp = pbin[p], y = pyq[p];
          const uint32_t xa = (uint32_t)max(bp - kXcorrOffset, 0), xe = (uint32_t)(bp + kXcorrOffset + 1), xs = (uint32_t)bp;
          const int32_t spike = 151 * y;
          uint32_t m;
          m = (uint32_t)map[xa >> kBlkShift] >> kBlkShift; if (m) atomicAdd(&tab[(m << kBlkShift) + (xa & (kBlk - 1u))], y);
          // (xe == NB for the last peak: the bins of the last block behind the table's end must read 0 too)
          if (xe < (nblk << kBlkShift)) { m = (uint32_t)map[xe >> kBlkShift] >> kBlkShift; if (m) atomicAdd(&tab[(m << kBlkShift) + (xe & (kBlk - 1u))], -y); }
          m = (uint32_t)map[xs >> kBlkShift] >> kBlkShift; if (m) atomicAdd(&tab[(m << kBlkShift) + (xs & (kBlk - 1u))], -spike);
          m = (uint32_t)map[(xs + 1u) >> kBlkShift] >> kBlkShift; if (m) atomicAdd(&tab[(m << kBlkShift) + ((xs + 1u) & (kBlk - 1u))], spike);
          if (cb0 > 0) cin += (xa < X0 ? y : 0) - (xe < X0 ? y : 0) - (xs < X0 ? spike : 0) + (xs + 1u < X0 ? spike : 0);
        }
        if (cb0 > 0 && cin != 0) atomicAdd(&sh.cin, cin);
      }
      __syncthreads();
      // (3) the scan, in place, negated: every thread owns a contiguous range of 16-byte words (an odd number of them:
      //     the 128-bit accesses of a quarter warp then fall into distinct banks); pass A adds up the ranges, a warp scan
      //     and the per-warp sums give every thread its start value, pass B rescans the range
      {
        uint4* t4 = reinterpret_cast<uint4*>(tab) + kBlk / 4;            // entry 0 = first occupied block
        const uint32_t N4 = cbn * (kBlk / 4);
        const uint32_t c4 = ((N4 + kScoreThreads - 1) / kScoreThreads) | 1u;
        const uint32_t s0 = min(tid * c4, N4), s1 = min(s0 + c4, N4);
        uint32_t part = 0;
        for (uint32_t i = s0; i < s1; i++) { const uint4 v = t4[i]; part += v.x + v.y + v.z + v.w; }
        uint32_t incl = part;
        for (int o = 1; o < 32; o <<= 1) { const uint32_t t = __shfl_up_sync(0xffffffffu, incl, o); if ((int)lane >= o) incl += t; }
        if (lane == 31) sh.wsum[warp] = incl;
        __syncthreads();
        uint32_t run = __reduce_add_sync(0xffffffffu, lane < warp ? sh.wsum[lane] : 0u) + (uint32_t)sh.cin + incl - part;
        for (uint32_t i = s0; i < s1; i++) {
          uint4 v = t4[i];
          v.x += run; v.y += v.x; v.z += v.y; v.w += v.z; run = v.w;
          t4[i] = make_uint4(0u - v.x, 0u - v.y, 0u - v.z, 0u - v.w);
        }
      }
      __syncthreads();
    };
    const bool one_tile = nact <= kTileBlocks;   // the usual case: the table is built once and serves every chunk of candidates
    const uint32_t c_lo = MODE == 2 ? mt.c_lo : 0u, c_hi = MODE == 2 ? mt.c_hi : ncand;     // this work item's candidates (the whole spectrum unless it was split)
    for (uint32_t c0 = c_lo; MODE == 0 ? c0 == 0 : (c0 < c_hi || c0 == c_lo); c0 += kCandChunk) {
      const uint32_t cn = c0 < c_hi ? min(kCandChunk, c_hi - c0) : 0u;
      for (uint32_t v = tid; v < cn; v += kScoreThreads) s_score[v] = 0;
      // counting sort of the chunk by peptide length, longest first
      {
        if (tid < 64) sh.hist[tid] = 0;
        __syncthreads();
        static_assert(kCandChunk <= 2 * kScoreThreads, "a thread sorts at most two candidates of a chunk");
        uint32_t len2[2] = {0, 0};
        if (scored) {
#pragma unroll
          for (int h = 0; h < 2; h++) {
            const uint32_t v = tid + h * kScoreThreads;
            if (v < cn) {
              const uint32_t len = cand_len(A, s, c0 + v, nt, t0c, C.n_per);
              len2[h] = len;
              atomicAdd(&sh.hist[63u - min(len, 63u)], 1u);
              my_pairs++; my_bytes += 14 + len;
            }
          }
        }
        __syncthreads();
        if (warp == 0) warp_hist64_prefix(sh.hist);
        __syncthreads();
        if (scored) {
#pragma unroll
          for (int h = 0; h < 2; h++) {
            const uint32_t v = tid + h * kScoreThreads;
            if (v < cn) s_order[atomicAdd(&sh.hist[63u - min(len2[h], 63u)], 1u)] = (uint16_t)v;
          }
        }
      }
      // (visible to the scoring warps after the table-build barriers)
      if (scored && cn) {
        for (uint32_t cb0 = 0; cb0 < nact; cb0 += kTileBlocks) {       // tiles of occupied blocks (usually one)
          const uint32_t cbn = min(kTileBlocks, nact - cb0);
          if (!one_tile || c0 == c_lo) build_tile(cb0, cbn);
          else { if (tid == 0) sh.unit = 0; __syncthreads(); }               // same table; the chunk's order and zeroed scores are visible
          // (4) score the chunk against the tile; one warp first fetches the CTA's next spectrum
          if (!side_done) {
            if (warp == kPrefetchWarp) prefetch_spectrum(A, sh, slot ^ 1u, s_bin, s_yq);
            if (warp == kFinishWarp && it > 0) finish_spectrum(A, C, sh, slot ^ 1u);
            side_done = true;
          }
          {
            TableView V;
            V.tab_s = (uint32_t)__cvta_generic_to_shared(tab); V.map_s = (uint32_t)__cvta_generic_to_shared(s_map); V.nblk = nblk; V.gmap = map;
            switch (nch * 2 + (mapg ? 1 : 0)) {
              case 2: score_units<1, HASVAR, false>(A, C, s, c0, cn, nt, t0c, V, L, s_score, s_order, &sh.unit); break;
              case 3: score_units<1, HASVAR, true>(A, C, s, c0, cn, nt, t0c, V, L, s_score, s_order, &sh.unit); break;
              case 4: score_units<2, HASVAR, false>(A, C, s, c0, cn, nt, t0c, V, L, s_score, s_order, &sh.unit); break;
              case 5: score_units<2, HASVAR, true>(A, C, s, c0, cn, nt, t0c, V, L, s_score, s_order, &sh.unit); break;
              case 6: score_units<3, HASVAR, false>(A, C, s, c0, cn, nt, t0c, V, L, s_score, s_order, &sh.unit); break;
              default: score_units<3, HASVAR, true>(A, C, s, c0, cn, nt, t0c, V, L, s_score, s_order, &sh.unit); break;
            }
          }
          __syncthreads();
        }
      }
      // ---- raw scores of every candidate (on request)
      if (A.tscore) {
        for (uint32_t v = tid; v < cn; v += kScoreThreads) {
          const uint32_t u = c0 + v;
          if (u < nt) A.tscore[t0c + u] = s_score[v]; else A.dscore[(uint64_t)s * C.n_per + (u - nt)] = s_score[v];
        }
      }
      // ---- top-k, K <= 8: every warp keeps the K best keys it has seen so far (lane r holds its r-th best across chunks)
      if (fast && scored && K) {   // (also without a candidate: the lists must not keep an earlier spectrum's keys)
        unsigned long long k0 = tid < cn ? psm_key(s_score[tid], c0 + tid) : 0ull;
        unsigned long long k1 = tid + kScoreThreads < cn ? psm_key(s_score[tid + kScoreThreads], c0 + tid + kScoreThreads) : 0ull;
        if (MODE == 0 || c_hi - c_lo <= kCandChunk) {      // one chunk (the usual case): nothing to carry over
          for (uint32_t r = 0; r < K; r++) {
            const unsigned long long wm = warp_max_u64(k0 > k1 ? k0 : k1);
            if (wm != 0ull) { if (k0 == wm) k0 = 0ull; else if (k1 == wm) k1 = 0ull; }
            if (lane == 0) sh.wtop[slot][warp][r] = wm;
          }
        } else {
          unsigned long long carry = (c0 > c_lo && lane < K) ? sh.wtop[slot][warp][lane] : 0ull, mine = 0ull;
          for (uint32_t r = 0; r < K; r++) {
            const unsigned long long b01 = k0 > k1 ? k0 : k1;
            const unsigned long long wm = warp_max_u64(b01 > carry ? b01 : carry);
            if (wm != 0ull) { if (k0 == wm) k0 = 0ull; else if (k1 == wm) k1 = 0ull; else if (carry == wm) carry = 0ull; }
            if (lane == r) mine = wm;
          }
          __syncwarp();
          if (lane < K) sh.wtop[slot][warp][lane] = mine;
        }
      }
      // ---- top-k of (this chunk's candidates) U (best of the earlier chunks), K > 8: K rounds of block-wide max
      if (!fast && scored && cn && K) {
        // scores -> keys, in place; slots cn..cn+K-1 (conceptually) hold the running list, owned by threads < K
        for (uint32_t v = tid; v < cn; v += kScoreThreads) s_score[v] = (int64_t)psm_key(s_score[v], c0 + v);
        unsigned long long carry = tid < K ? sh.top[tid] : 0ull;   // this thread's entry of the running list
        __syncthreads();
        unsigned long long prev = ~0ull;
        for (uint32_t r = 0; r < K; r++) {
          unsigned long long best = (carry < prev) ? carry : 0ull;
          for (uint32_t v = tid; v < cn; v += kScoreThreads) {
            const unsigned long long k = (unsigned long long)s_score[v];
            if (k < prev && k > best) best = k;
          }
          best = warp_max_u64(best);
          if (lane == 0) sh.wkey[r & 1][warp] = best;
          __syncthreads();
          unsigned long long m = lane < NW ? sh.wkey[r & 1][lane] : 0ull;
          m = warp_max_u64(m);
          if (tid == 0) sh.top[r] = m;
          prev = m;
          if (m == 0ull) break;   // fewer candidates than rows (uniform: every thread sees the same m)
        }
        __syncthreads();
      }
    }
    if (!side_done) {   // (nothing was scored)
      if (warp == kPrefetchWarp) prefetch_spectrum(A, sh, slot ^ 1u, s_bin, s_yq);
      if (warp == kFinishWarp && it > 0) finish_spectrum(A, C, sh, slot ^ 1u);
    }
    // ---- PSM rows
    if (fast) {
      // the per-warp top-k lists are complete; the finish warp merges them and writes the rows during the next scoring phase
      if (tid == 0) {
        FinRecord f; f.pr = pr; f.t0c = t0c; f.s = s; f.nt = nt; f.nd = nd; f.pending = 1; f.ranked = (scored && K) ? 1u : 0u; f.part = mt.part;
        sh.fin[slot] = f;
      }
    } else {
      for (uint32_t r = tid; r < K; r += kScoreThreads) write_psm_row(A, C, pr, s, r, scored ? sh.top[r] : 0ull, nt, nd, t0c);
      if (tid == 0) sh.fin[slot].pending = 0;
      __syncthreads();
    }
  }
  unsigned long long wp = my_pairs, wb = my_bytes;
  for (int o = 16; o; o >>= 1) { wp += __shfl_xor_sync(0xffffffffu, wp, o); wb += __shfl_xor_sync(0xffffffffu, wb, o); }
  if (lane == 0 && wp) { atomicAdd(&A.stat64[0], wp); atomicAdd(&A.stat64[1], wb); }
}

// ------------------------------------------------------------------------------------------------
// K4, pipelined: tables are built ahead by their own kernel, a loader warp streams them into shared memory with bulk
// asynchronous copies, and the scorer warps never meet at a barrier
// ------------------------------------------------------------------------------------------------
// k_score above runs a spectrum's phases one after the other behind block-wide barriers (stage, sort, build, score,
// top-k), so the shared-memory pipe and the issue slots idle through every phase change and behind the slowest warp of
// the scoring phase.  Here the phases are taken apart:
//   k_build_tables  one CTA per spectrum, the whole GPU at once: number the occupied 64-bin blocks, write the block map
//                   and fill the table DIRECTLY -- T[b] = 151*y[b] - sum of y over the peaks within 75 bins, evaluated per
//                   bin from the few peaks that reach it: no zero fill, no difference array, no scan -- into one
//                   contiguous record per spectrum in HBM: [block map][all-zero block][occupied blocks].  It depends on
//                   the spectra only.
//   k_cand_order    one CTA per spectrum: the candidates counting-sorted by length, longest first (units of 32 then hold
//                   candidates of one length).
//   k_score_pipe    one persistent CTA per SM.  A LOADER warp takes the next spectrum from the queue, finds room for its
//                   table in a RING of shared-memory blocks (two spectra are resident whenever their tables fit side by
//                   side) and issues cp.async.bulk copies of map, table and candidate order that complete on the slot's
//                   mbarrier.  The other warps (19 at 640 threads) SCORE: each pulls 32-candidate units of the current
//                   spectrum, keeps its K best keys in registers, and when the units run out leaves them in shared memory
//                   and walks on to the next spectrum if its table has landed; the last warp to leave a spectrum merges
//                   the lists, releases the slot (empty mbarrier) and then writes the PSM rows -- for a spectrum split
//                   into parts, only the last part to finish does, after merging the parts' lists (merge_parts).
// Same arithmetic as k_score (score_one): bit-identical rows.  Batches this path does not take (top_k > 8, a fixed
// N-terminus modification, MD_SCORE_CLASSIC, split batches under MD_SCORE_SPLIT_CLASSIC) use k_score; a spectrum it cannot
// hold (more than 1024 binned peaks, a block map beyond 4096 entries, a table record beyond the ring) goes onto the list
// that k_build_tables leaves, and k_score works that list off on the side stream beside this kernel.
#ifndef MD_PIPE_THREADS
#define MD_PIPE_THREADS 640     // swept on C2 / C3: 448 .. 1024 threads; 640 (19 scorer warps at up to 102 registers) is the fastest
#endif
constexpr uint32_t kPipeThreads = MD_PIPE_THREADS, kPipeWarps = kPipeThreads / 32;
constexpr uint32_t kScoreWarps = kPipeWarps - 1, kLoaderWarp = kPipeWarps - 1;
constexpr uint32_t kPMapCap = 4096;        // block-map entries per slot (262k bins)
constexpr uint32_t kPOrder = 2048;         // candidates that are sorted by length (spectra with more are walked in their natural order)
constexpr uint32_t kPPeaks = 1024;         // binned peaks k_build_tables stages
constexpr uint32_t kPoolBlocks = 856;      // most 64-bin blocks (the all-zero block included) of a table the pipelined kernel takes
constexpr uint32_t kRingBytes = 214 * 1024; // shared-memory ring that holds the table records (block map + table) of two spectra
constexpr uint32_t kPipeEnd = 0xFFFFFFFFu, kTabLeft = 0xFFFFFFFFu;
constexpr uint32_t kTabThreads = 256;

// where a spectrum's table record lies in the pool.  nblk == 0: the spectrum is not scored (too few peaks); nact == kTabLeft: k_score takes it
struct TabDesc { unsigned long long off; uint32_t nact, nblk; };
__host__ __device__ inline uint32_t tab_map_bytes(uint32_t nblk) { return ((nblk + 1u) * 2u + 15u) & ~15u; }
constexpr size_t kTabMaxBytes = (((size_t)kPMapCap + 1) * 2 + 15) / 16 * 16 + (size_t)kPoolBlocks * kBlk * 4;

__global__ void __launch_bounds__(kTabThreads) k_build_tables(const uint64_t* __restrict__ peak_off, const int32_t* __restrict__ pk_bin, const int32_t* __restrict__ pk_yq,
                                                              const uint32_t* __restrict__ pk_count, const int32_t* __restrict__ pk_hbin, uint8_t* __restrict__ pool,
                                                              unsigned long long* __restrict__ pool_top, TabDesc* __restrict__ desc,
                                                              uint32_t* __restrict__ left_list, uint32_t* __restrict__ n_left) {
  __shared__ int32_t s_bin[kPPeaks], s_yq[kPPeaks];
  __shared__ uint32_t s_bits[kPMapCap / 32], s_pre[kPMapCap / 32];
  __shared__ uint16_t s_blk[kPoolBlocks];
  __shared__ uint32_t s_nact;
  __shared__ unsigned long long s_base;
  const uint32_t s = blockIdx.x, tid = threadIdx.x, lane = tid & 31;
  const int32_t hbin = pk_hbin[s];
  const uint32_t npk = pk_count[s];
  const uint64_t pk0 = peak_off[s];
  const uint32_t NB = hbin >= 0 ? (uint32_t)hbin + kXcorrOffset + 1 : 0u;       // table bins [0, NB)
  const uint32_t nblk = (NB + kBlk - 1) >> kBlkShift, nwords = (nblk + 31) >> 5;
  if (hbin < 0 || NB > kMaxBins) { if (tid == 0) desc[s] = TabDesc{0ull, 0u, 0u}; return; }
  if (npk > kPPeaks || nblk > kPMapCap) { if (tid == 0) { desc[s] = TabDesc{0ull, kTabLeft, nblk}; left_list[atomicAdd(n_left, 1u)] = s; } return; }
  for (uint32_t i = tid; i < npk; i += kTabThreads) { s_bin[i] = pk_bin[pk0 + i]; s_yq[i] = pk_yq[pk0 + i]; }
  for (uint32_t i = tid; i < nwords; i += kTabThreads) s_bits[i] = 0;
  __syncthreads();
  for (uint32_t p = tid; p < npk; p += kTabThreads) {     // every bin within 75 of a peak
    const int32_t bp = s_bin[p];
    const uint32_t b0 = (uint32_t)max(bp - kXcorrOffset, 0) >> kBlkShift, b1 = min((uint32_t)(bp + kXcorrOffset), NB - 1) >> kBlkShift;
    for (uint32_t k = b0; k <= b1; k++) atomicOr(&s_bits[k >> 5], 1u << (k & 31));
  }
  __syncthreads();
  if (tid < 32) {
    const uint32_t run = warp_bitmap_prefix(s_bits, s_pre, nwords);
    if (lane == 0) {
      s_nact = run;
      if (run + 1u <= kPoolBlocks && tab_map_bytes(nblk) + (run + 1u) * kBlk * 4u <= kRingBytes) s_base = atomicAdd(pool_top, (unsigned long long)tab_map_bytes(nblk) + (unsigned long long)(run + 1u) * kBlk * 4u);
    }
  }
  __syncthreads();
  const uint32_t nact = s_nact;
  if (nact + 1u > kPoolBlocks || tab_map_bytes(nblk) + (nact + 1u) * kBlk * 4u > kRingBytes) { if (tid == 0) { desc[s] = TabDesc{0ull, kTabLeft, nblk}; left_list[atomicAdd(n_left, 1u)] = s; } return; }
  const unsigned long long base = s_base;
  if (tid == 0) desc[s] = TabDesc{base, nact, nblk};
  // ---- block map: entry = (block of the record << 6) | 63, block 0 of the record = the all-zero block every miss reads
  uint16_t* gmap = reinterpret_cast<uint16_t*>(pool + base);
  const uint32_t map_entries = tab_map_bytes(nblk) / 2u;
  for (uint32_t k = tid; k < map_entries; k += kTabThreads) {
    uint32_t m = 0;
    if (k < nblk) {
      const uint32_t wd = s_bits[k >> 5];
      if ((wd >> (k & 31)) & 1u) {
        const uint32_t c = s_pre[k >> 5] + (uint32_t)__popc(wd & ((1u << (k & 31)) - 1u));
        m = c + 1u; s_blk[c] = (uint16_t)k;
      }
    }
    gmap[k] = (uint16_t)(m ? (m << kBlkShift) | (kBlk - 1u) : 0u);
  }
  int4* gtab = reinterpret_cast<int4*>(pool + base + tab_map_bytes(nblk));
  if (tid < kBlk / 4) gtab[tid] = make_int4(0, 0, 0, 0);
  __syncthreads();
  // ---- the table: eight threads per block, eight bins per thread; the peaks are sorted and unique by bin, those within 75
  //      bins of the thread's bins are consecutive
  for (uint32_t wk = tid; wk < nact * 8u; wk += kTabThreads) {
    const uint32_t c = wk >> 3, sub = wk & 7u;
    const int32_t x0 = (int32_t)((uint32_t)s_blk[c] << kBlkShift) + (int32_t)(sub * 8u);
    uint32_t lo = 0, hi = npk;                          // first peak with bin >= x0 - 75
    while (lo < hi) { const uint32_t mid = (lo + hi) >> 1; if (s_bin[mid] < x0 - kXcorrOffset) lo = mid + 1; else hi = mid; }
    int32_t t[8];
#pragma unroll
    for (int j = 0; j < 8; j++) t[j] = 0;
    for (uint32_t p = lo; p < npk; p++) {
      const int32_t bp = s_bin[p];
      if (bp > x0 + 7 + kXcorrOffset) break;
      const int32_t y = s_yq[p];
#pragma unroll
      for (int j = 0; j < 8; j++) {
        const int32_t d = bp - (x0 + j);
        t[j] -= (d <= kXcorrOffset && d >= -kXcorrOffset) ? y : 0;
        t[j] += d == 0 ? 151 * y : 0;
      }
    }
    int4* dst = gtab + (size_t)(c + 1u) * (kBlk / 4) + sub * 2u;
    dst[0] = make_int4(t[0], t[1], t[2], t[3]); dst[1] = make_int4(t[4], t[5], t[6], t[7]);
  }
}

// The order in which the persistent CTAs take the spectra: pairs of (large record, small record) -- the p-th largest with the
// p-th smallest -- so that two consecutive spectra of a CTA nearly always fit the ring side by side and every pair is about
// the same amount of work.  k_table_keys: record size per spectrum (the sort key); k_pair_schedule: sorted order -> pairs.
// A split batch (parts > 1) is scheduled by work instead: the spectra with the most candidates first.
__global__ void k_table_keys(const TabDesc* __restrict__ desc, uint32_t n, const uint64_t* __restrict__ cand_off, const uint32_t* __restrict__ dec_count, bool by_work,
                             uint32_t* __restrict__ key, uint32_t* __restrict__ val) {
  const uint32_t s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= n) return;
  const TabDesc d = desc[s];
  const bool scored = d.nblk != 0u && d.nact != kTabLeft;
  if (by_work) key[s] = scored ? (uint32_t)min(cand_off[s + 1] - cand_off[s] + (dec_count ? dec_count[s] : 0u), (uint64_t)0xFFFFFFFFu) : 0u;
  else key[s] = scored ? tab_map_bytes(d.nblk) + (d.nact + 1u) * kBlk * 4u : 0u;
  val[s] = s;
}
__global__ void k_pair_schedule(const uint32_t* __restrict__ asc, uint32_t n, bool descending, uint32_t* __restrict__ sched) {
  const uint32_t p = blockIdx.x * blockDim.x + threadIdx.x;   // pair
  if (2 * p >= n) return;
  if (descending) { sched[2 * p] = asc[n - 1 - 2 * p]; if (2 * p + 1 < n) sched[2 * p + 1] = asc[n - 2 - 2 * p]; return; }
  sched[2 * p] = asc[n - 1 - p];
  if (2 * p + 1 < n) sched[2 * p + 1] = asc[p];
}

// candidates of every spectrum with at most kPOrder of them, counting-sorted by length (longest first) -> order[s * kPOrder + i]
__global__ void __launch_bounds__(256) k_cand_order(const ScoreArgs A, uint32_t n_per, uint16_t* __restrict__ order) {
  __shared__ uint32_t hist[64];
  const uint32_t s = blockIdx.x, tid = threadIdx.x;
  const uint64_t t0c = A.cand_off[s];
  const uint32_t nt = (uint32_t)(A.cand_off[s + 1] - t0c), nd = A.dec_count ? A.dec_count[s] : 0u, ncand = nt + nd;
  if (ncand > kPOrder || A.pk_hbin[s] < 0) return;
  if (tid < 64) hist[tid] = 0;
  __syncthreads();
  uint8_t lens[kPOrder / 256];
#pragma unroll
  for (uint32_t h = 0; h < kPOrder / 256; h++) {
    const uint32_t v = tid + h * 256;
    lens[h] = v < ncand ? (uint8_t)cand_len(A, s, v, nt, t0c, n_per) : (uint8_t)0;
  }
#pragma unroll
  for (uint32_t h = 0; h < kPOrder / 256; h++) if (tid + h * 256 < ncand) atomicAdd(&hist[63u - min((uint32_t)lens[h], 63u)], 1u);
  __syncthreads();
  if (tid < 32) warp_hist64_prefix(hist);
  __syncthreads();
  uint16_t* out = order + (size_t)s * kPOrder;
#pragma unroll
  for (uint32_t h = 0; h < kPOrder / 256; h++) {
    const uint32_t v = tid + h * 256;
    if (v < ncand) out[atomicAdd(&hist[63u - min((uint32_t)lens[h], 63u)], 1u)] = (uint16_t)v;
  }
}

struct PipeSlot {
  md_precursor pr;
  uint64_t t0c;
  uint32_t s, nt, nd, ncand, nunits, nblk, scored, sorted, left, base;
  uint32_t part, u_hi; // the work item's part of the spectrum, and where its units end (the whole spectrum unless the batch is split)
  uint32_t unit;      // next unit of the spectrum (scorers)
  uint32_t done;      // scorer warps that have left the spectrum
};
struct PipeShared {
  PipeSlot slot[2];
  unsigned long long ready[2], empty[2];                       // mbarriers
  unsigned long long wtop[2][kScoreWarps][kFastTopK];
};

__device__ __forceinline__ void prefetch_l2(const void* p) { asm volatile("prefetch.global.L2 [%0];" ::"l"(p)); }
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(unsigned long long* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_arrive(unsigned long long* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(unsigned long long* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
// global -> shared bulk asynchronous copy (the TMA engine moves the bytes; they count towards the mbarrier's transaction)
__device__ __forceinline__ void bulk_g2s(void* smem_dst, const void* gsrc, uint32_t bytes, unsigned long long* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(smem_dst)), "l"(gsrc), "r"(bytes),
               "r"(smem_u32(bar)) : "memory");
}
// try_wait with a suspend-time hint: the hardware parks the thread until the phase completes (or the hint runs out), so a
// waiting warp takes no issue slots from the warps it is waiting for
__device__ __forceinline__ bool mbar_try_wait(unsigned long long* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n"
      ".reg .pred P1;\n"
      "mbarrier.try_wait.parity.shared::cta.b64 P1, [%1], %2, %3;\n"
      "selp.u32 %0, 1, 0, P1;\n"
      "}" : "=r"(ok) : "r"(smem_u32(bar)), "r"(parity), "r"(1000000u) : "memory");
  return ok != 0;
}
// (a wait that lasts seconds is a protocol error: stop the kernel with a launch failure instead of hanging the device)
__device__ __forceinline__ void mbar_wait(unsigned long long* bar, uint32_t parity) {
  uint32_t spins = 0;
  while (!mbar_try_wait(bar, parity)) { if (++spins > 4000u) __trap(); }
}
// one lane polls for its warp (32 pollers per warp would take the issue slots of the warps that are being waited for)
__device__ __forceinline__ void mbar_wait_warp(unsigned long long* bar, uint32_t parity) {
  if ((threadIdx.x & 31u) == 0u) mbar_wait(bar, parity);
  __syncwarp();
}

constexpr size_t kPipeSmem = (size_t)kRingBytes + 2 * (size_t)kPOrder * 2;

struct PipeArgs { const TabDesc* desc; const uint8_t* pool; const uint16_t* order; const uint32_t* sched; uint32_t parts; };

template <bool HASVAR>
__global__ void __launch_bounds__(kPipeThreads, 1) k_score_pipe(const __grid_constant__ ScoreArgs A, const __grid_constant__ ScoreConst C, const PipeArgs T) {
  extern __shared__ __align__(128) uint8_t ring[];                                      // kRingBytes: table records [block map][all-zero block][occupied blocks]
  uint16_t* s_order0 = reinterpret_cast<uint16_t*>(ring + kRingBytes);                  // 2 x kPOrder
  __shared__ PipeShared sh;
  const uint32_t tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  if (tid == 0) {
    for (int b = 0; b < 2; b++) { mbar_init(&sh.ready[b], 1); mbar_init(&sh.empty[b], 1); sh.slot[b].done = 0; sh.slot[b].unit = 0; }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();

  if (warp == kLoaderWarp) {
    // =============================================================================== loader (one lane works; the warp keeps it company)
    if (lane == 0) {
      uint32_t prev_need = 0;                          // ring bytes of the previous spectrum's record (it lies at the other end of the ring)
      uint32_t pend = kPipeEnd;                        // second spectrum of the pair that was drawn last
      for (uint32_t q = 0;; q++) {
        const uint32_t b = q & 1, use = q >> 1;
        PipeSlot& S = sh.slot[b];
        // work items are PAIRS of the schedule (large record, then small record)
        // (a split batch -- few spectra, very many candidates each -- has parts x spectra items instead: consecutive tickets are
        //  the parts of one spectrum, which different CTAs then score at the same time)
        uint32_t s = pend, part = 0;
        pend = kPipeEnd;
        if (s == kPipeEnd) {
          const uint32_t t = atomicAdd(A.work, 1u);
          if (T.parts > 1) { if (t < (unsigned long long)A.n_spec * T.parts) { s = T.sched[t / T.parts]; part = t % T.parts; } }
          else if (2ull * t < A.n_spec) { s = T.sched[2 * t]; if (2 * t + 1 < A.n_spec) pend = T.sched[2 * t + 1]; }
        }
        const bool end = s == kPipeEnd;
        // (what the spectrum needs is fetched before the slot is waited for)
        md_precursor pr; pr.mass = 0; pr.lo = 0; pr.hi = 0; pr.charge = 0; pr.spectrum_id = 0;
        uint64_t t0c = 0; uint32_t nt = 0, nd = 0;
        TabDesc d{0ull, 0u, 0u};
        if (!end) { pr = A.prec[s]; t0c = A.cand_off[s]; nt = (uint32_t)(A.cand_off[s + 1] - t0c); nd = A.dec_count ? A.dec_count[s] : 0u; d = T.desc[s]; }
        const uint32_t ncand = nt + nd;
        if (use > 0) mbar_wait(&sh.empty[b], (use - 1) & 1);   // the slot's previous spectrum has left
        if (end) { S.s = kPipeEnd; __threadfence_block(); mbar_arrive(&sh.ready[b]); break; }
        bool scored = d.nblk != 0u, left = false;
        if (scored && ncand > 0xFFFFFFu) { *A.error = 1; scored = false; }
        if (scored && d.nact == kTabLeft) { left = true; scored = false; }
        const bool sorted = scored && ncand <= kPOrder;
        uint32_t base = 0, need = 0;
        if (scored) {
          // ---- room for the record in the ring: records alternate between its two ends, so two spectra are resident whenever
          //      their records fit side by side; if they do not, the previous spectrum has to leave first
          need = tab_map_bytes(d.nblk) + (d.nact + 1u) * kBlk * 4u;
          if (prev_need + need > kRingBytes && q > 0) mbar_wait(&sh.empty[b ^ 1u], ((q - 1) >> 1) & 1);
          base = b ? kRingBytes - need : 0u;
        }
        S.pr = pr; S.t0c = t0c; S.s = s; S.nt = nt; S.nd = nd; S.ncand = ncand; S.nunits = (ncand + 31) >> 5; S.nblk = d.nblk;
        S.scored = scored ? 1u : 0u; S.sorted = sorted ? 1u : 0u; S.left = left ? 1u : 0u; S.base = base;
        {
          const uint32_t nunits = (ncand + 31) >> 5, per = (nunits + T.parts - 1) / T.parts;
          const uint32_t u_lo = min(nunits, part * per);
          S.part = part; S.unit = u_lo; S.u_hi = min(nunits, u_lo + per);
        }
        __threadfence_block();
        if (scored) {
          const uint32_t obytes = sorted ? ((ncand * 2u + 15u) & ~15u) : 0u;
          mbar_arrive_expect_tx(&sh.ready[b], need + obytes);
          const uint8_t* src = T.pool + d.off;
          uint8_t* dst = ring + base;
          for (uint32_t left_b = need; left_b;) {      // (pieces of at most 64 KB)
            const uint32_t piece = min(left_b, 65536u);
            bulk_g2s(dst, src, piece, &sh.ready[b]);
            dst += piece; src += piece; left_b -= piece;
          }
          if (sorted) bulk_g2s(s_order0 + b * kPOrder, T.order + (size_t)s * kPOrder, obytes, &sh.ready[b]);
          prev_need = need;
        } else {
          mbar_arrive(&sh.ready[b]);
          prev_need = 0;
        }
      }
    }
    return;
  }

  // ================================================================================= scorers
  const LaneTab L{C.tq[lane], C.tr[lane], C.vq[lane], C.vr[lane]};   // per-letter (q, r) tables in registers: lane = residue code
  uint32_t my_pairs = 0, my_bytes = 0;
  const uint32_t K = C.top_k;
  for (uint32_t q = 0;; q++) {
    const uint32_t b = q & 1, use = q >> 1;
    mbar_wait_warp(&sh.ready[b], use & 1);
    PipeSlot& S = sh.slot[b];
    const uint32_t s = S.s;
    if (s == kPipeEnd) break;
    const md_precursor pr = S.pr;
    const uint64_t t0c = S.t0c;
    const uint32_t nt = S.nt, nd = S.nd, ncand = S.ncand, nunits = S.u_hi;
    const bool scored = S.scored != 0, sorted = S.sorted != 0, left_out = S.left != 0;
    const uint32_t S_part = S.part;
    const uint16_t* order = s_order0 + b * kPOrder;
    uint32_t nch = pr.charge > 1 ? pr.charge - 1 : 1;
    if (nch > C.max_frag_charge) nch = C.max_frag_charge;
    if (nch < 1) nch = 1;
    TableView V;
    V.map_s = smem_u32(ring + S.base); V.tab_s = V.map_s + tab_map_bytes(S.nblk); V.nblk = S.nblk; V.gmap = nullptr;
    unsigned long long mine = 0ull;     // lane r: this warp's r-th best key of the spectrum
    if (scored || (A.tscore && !left_out)) {
      uint32_t u = 0;
      if (lane == 0) u = atomicAdd(&S.unit, 1u);
      u = __shfl_sync(0xffffffffu, u, 0);
      while (u < nunits) {
        // the warp's next unit is drawn one ahead, and what it will read first is requested into L2 while this unit is scored
        uint32_t un = 0;
        if (lane == 0) un = atomicAdd(&S.unit, 1u);
        un = __shfl_sync(0xffffffffu, un, 0);
        if (scored && un < nunits) {
          const uint32_t i2 = un * 32 + lane;
          if (i2 < ncand) {
            const uint32_t v2 = sorted ? (uint32_t)order[i2] : i2;
            if (v2 < nt) { prefetch_l2(A.cand_desc + t0c + v2); prefetch_l2(A.cand_w + t0c + v2); }
            else { const uint64_t j = (uint64_t)s * C.n_per + (v2 - nt); prefetch_l2(A.dec_rows + j * MD_DECOY_HALF); prefetch_l2(A.dec_len + j); prefetch_l2(A.dec_w + j); }
          }
        }
        const uint32_t i = u * 32 + lane;
        CandRef cr;
        cr.row = reinterpret_cast<const uint4*>(A.idx_rows); cr.row_hi = cr.row; cr.len = 0; cr.mask = 0; cr.modw = 0;
        uint32_t v = 0;
        const bool valid = i < ncand;
        if (valid) {
          v = sorted ? (uint32_t)order[i] : i;
          if (scored) { cr = cand_ref<HASVAR>(A, s, v, nt, t0c, C.n_per); my_pairs++; my_bytes += 14 + cr.len; }
        }
        int64_t score = 0;
        if (scored) {
          const uint32_t maxlen = __reduce_max_sync(0xffffffffu, cr.len);
          switch (nch) {
            case 1: score = score_one<1, HASVAR, false>(cr, maxlen, V, C, L); break;
            case 2: score = score_one<2, HASVAR, false>(cr, maxlen, V, C, L); break;
            default: score = score_one<3, HASVAR, false>(cr, maxlen, V, C, L); break;
          }
        }
        if (A.tscore && valid) { if (v < nt) A.tscore[t0c + v] = score; else A.dscore[(uint64_t)s * C.n_per + (v - nt)] = score; }
        if (scored && K) {
          // the unit's keys against the warp's running list: nothing to do unless the best new key beats the K-th best kept
          unsigned long long nk = valid ? psm_key(score, v) : 0ull;
          const unsigned long long kth = __shfl_sync(0xffffffffu, mine, (int)K - 1);
          if (warp_max_u64(nk) > kth) {
            unsigned long long carry = lane < K ? mine : 0ull, out = 0ull;
            for (uint32_t r = 0; r < K; r++) {
              const unsigned long long wm = warp_max_u64(nk > carry ? nk : carry);
              if (wm != 0ull) { if (nk == wm) nk = 0ull; else if (carry == wm) carry = 0ull; }
              if (lane == r) out = wm;
            }
            mine = out;
          }
        }
        u = un;
      }
    }
    // ---- leave the spectrum: the warp's list goes to shared memory; the last warp merges all lists and writes the PSM rows
    if (lane < kFastTopK) sh.wtop[b][warp][lane] = lane < K ? mine : 0ull;
    __threadfence_block();
    __syncwarp();
    uint32_t left = 0;
    if (lane == 0) left = atomicAdd(&S.done, 1u);
    left = __shfl_sync(0xffffffffu, left, 0);
    if (left == kScoreWarps - 1) {
      __threadfence_block();
      unsigned long long best = 0ull;
      if (scored && K) {
        uint32_t idx = 0;
        for (uint32_t r = 0; r < K; r++) {
          const unsigned long long head = (lane < kScoreWarps && idx < K) ? sh.wtop[b][lane][idx] : 0ull;
          const unsigned long long wm = warp_max_u64(head);
          if (wm != 0ull && head == wm) idx++;
          if (lane == r) best = wm;
        }
      }
      // the slot is free as soon as the lists are merged: the rows (an FP64 division each, thousands of cycles on this part)
      // are written from registers while the loader already brings the slot's next spectrum
      __syncwarp();
      if (lane == 0) { S.done = 0; __threadfence_block(); mbar_arrive(&sh.empty[b]); }
      if (T.parts > 1 && !left_out) {
        const PartMerge pm = merge_parts(A, s, S_part, T.parts, K, best);
        if (!pm.last) continue;
        best = pm.best;
      }
      if (lane < K && !left_out) write_psm_row(A, C, pr, s, lane, best, nt, nd, t0c);
    }
  }
  unsigned long long wp = my_pairs, wb = my_bytes;
  for (int o = 16; o; o >>= 1) { wp += __shfl_xor_sync(0xffffffffu, wp, o); wb += __shfl_xor_sync(0xffffffffu, wb, o); }
  if (lane == 0 && wp) { atomicAdd(&A.stat64[0], wp); atomicAdd(&A.stat64[1], wb); }
}

__global__ void k_max_i32(const int32_t* __restrict__ v, uint32_t n, int32_t* __restrict__ out) {
  int32_t m = INT32_MIN;
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) m = max(m, v[i]);
  m = __reduce_max_sync(0xffffffffu, m);
  if ((threadIdx.x & 31) == 0) atomicMax(out, m);
}

// most candidates (targets + decoys) of one spectrum of the batch
__global__ void k_max_candidates(const uint64_t* __restrict__ cand_off, const uint32_t* __restrict__ dec_count, uint32_t n, int32_t* __restrict__ out) {
  int32_t m = 0;
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const uint64_t c = cand_off[i + 1] - cand_off[i] + (dec_count ? dec_count[i] : 0u);
    m = max(m, (int32_t)min(c, (uint64_t)0x7FFFFFFF));
  }
  m = __reduce_max_sync(0xffffffffu, m);
  if ((threadIdx.x & 31) == 0) atomicMax(out, m);
}

void split_qr(int64_t m, uint32_t w, uint32_t* q, uint32_t* r) {
  if (m < 0) m = 0;
  *q = (uint32_t)(m / w); *r = (uint32_t)(m % w);
}

// k_score_pipe scores with position-independent residue masses; a fixed N-terminus modification needs k_score (ScoreConst::nq)
bool classic_only(const md_ctx* ctx) {
  if (getenv("MD_SCORE_CLASSIC") != nullptr) return true;
  for (int c = 0; c < MD_NCODES; c++) if (ctx->mods.has_fix[c] && ctx->mods.fix_pos[c] == MD_POS_N) return true;
  return false;
}

constexpr size_t kScoreSmem = (size_t)kTileBins * sizeof(int32_t) + (size_t)kCandChunk * sizeof(int64_t) + 2 * (size_t)kPeakCap * 8 + (size_t)kCandChunk * 2 +
                              ((size_t)kMapCap + 2) * 2;

// k_score over the work items of A on `stream`, instantiated for the batch: HASVAR = any variable modification, MODE from
// A.parts and `single` (every spectrum of the batch fits one chunk of candidates)
void launch_k_score(md_ctx* ctx, cudaStream_t stream, uint32_t grid, const ScoreArgs& A, const ScoreConst& C, bool has_var, bool single) {
  auto go = [&](auto kernel) {
    MD_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kScoreSmem));
    kernel<<<grid, kScoreThreads, kScoreSmem, stream>>>(A, C);
    ctx->launches++;
    MD_CUDA(cudaGetLastError());
  };
  const int mode = A.parts > 1 ? 2 : (single ? 0 : 1);
  if (has_var) { if (mode == 2) go(k_score<true, 2>); else if (mode == 0) go(k_score<true, 0>); else go(k_score<true, 1>); }
  else { if (mode == 2) go(k_score<false, 2>); else if (mode == 0) go(k_score<false, 0>); else go(k_score<false, 1>); }
}

}  // namespace

void precursors_dev(md_ctx* ctx, const SpectraDev& S, const md_search_params& p, uint32_t id_base) {
  ctx->ws.prec.need(S.n + 1);
  if (!S.n) return;
  MD_LAUNCH(ctx, k_precursors, blocks(S.n), 256, 0, S.pmz, S.charge, S.sid, S.n, p.lower_ppm, p.upper_ppm, p.abs_lower_uda, p.abs_upper_uda, id_base, ctx->ws.prec.p);
}

// What the scoring needs from the spectra alone -- binned peaks (K4a) and, for the pipelined kernel, the table records -- runs on
// the ctx's side stream from the moment the precursors are known, i.e. beside the candidate lookup and the decoy generation
// (which keep the SMs' issue slots busy but leave HBM idle); score_run_dev waits for it.
void score_prepare_dev(md_ctx* ctx, const SpectraDev& S, uint64_t n_peaks, const md_search_params& p) {
  IdentifyWorkspace& W = ctx->ws;
  const uint32_t n = S.n;
  if (!n) return;
  const int64_t w = (int64_t)llround(p.fragment_tolerance * 1000000.0);
  W.pk_bin.need(n_peaks + 1); W.pk_yq.need(n_peaks + 1); W.pk_count.need(n + 1); W.pk_hbin.need(n + 1);
  DevBuf<int>& d_flag = W.t_unsorted; d_flag.need(4);
  W.stat64.need(5);
  const bool tables = p.top_k <= kFastTopK && !classic_only(ctx);
  W.tables_built = tables;
  if (tables) { W.tab_pool.need((size_t)n * kTabMaxBytes + 256); W.tab_desc.need((size_t)n * sizeof(TabDesc) + 16); W.left_list.need(n + 2); }
  cudaStream_t main = ctx->stream, side = ctx->stream2;
  MD_CUDA(cudaEventRecord(ctx->ev_fork, main));
  MD_CUDA(cudaStreamWaitEvent(side, ctx->ev_fork, 0));
  ctx->stream = side;     // (MD_LAUNCH launches on ctx->stream)
  try {
    MD_CUDA(cudaEventRecord(ctx->ev_side0, side));
    MD_CUDA(cudaMemsetAsync(d_flag.p, 0, 4 * sizeof(int), side));
    MD_CUDA(cudaMemsetAsync(W.pk_yq.p, 0, (n_peaks + 1) * sizeof(int32_t), side));
    MD_LAUNCH(ctx, k_bin_spectra, blocks((uint64_t)n * 32, 128), 128, 0, S.peak_off, S.peak_mz, S.peak_int, W.prec.p, n, w, p.min_peaks, W.pk_bin.p, W.pk_yq.p,
              W.pk_count.p, W.pk_hbin.p, d_flag.p);
    // the largest table of the batch decides whether the block maps fit shared memory
    MD_LAUNCH(ctx, k_max_i32, std::min<uint32_t>(blocks(n), 64), 256, 0, W.pk_hbin.p, n, d_flag.p + 2);
    if (tables) {
      MD_CUDA(cudaMemsetAsync(W.stat64.p + 4, 0, sizeof(unsigned long long), side));
      MD_CUDA(cudaMemsetAsync(W.left_list.p + n, 0, sizeof(uint32_t), side));                  // [n] = how many spectra k_build_tables leaves to k_score
      MD_LAUNCH(ctx, k_build_tables, n, kTabThreads, 0, S.peak_off, W.pk_bin.p, W.pk_yq.p, W.pk_count.p, W.pk_hbin.p, W.tab_pool.p, W.stat64.p + 4, reinterpret_cast<TabDesc*>(W.tab_desc.p),
                W.left_list.p, W.left_list.p + n);
    }
    MD_CUDA(cudaEventRecord(ctx->ev_side1, side));
    MD_CUDA(cudaEventRecord(ctx->ev_prep, side));
  } catch (...) { ctx->stream = main; throw; }
  ctx->stream = main;
}

void score_run_dev(md_ctx* ctx, const SpectraDev& S, const md_search_params& p, uint32_t n_per, md_psm* psm_dev, bool want_all) {
  IdentifyWorkspace& W = ctx->ws;
  const uint32_t n = S.n;
  if (!n) return;
  const int64_t w = (int64_t)llround(p.fragment_tolerance * 1000000.0);
  const uint32_t mfc = p.max_fragment_charge ? p.max_fragment_charge : 3;
  MD_REQUIRE(mfc <= 3, MD_ERR_UNSUPPORTED, "max_fragment_charge > 3 (the reference fixes it to 3: comet_parameter.rs:55)");
  MD_REQUIRE(p.top_k <= kMaxTopK, MD_ERR_UNSUPPORTED, "top_k > 128");
  DevBuf<int>& d_flag = W.t_unsorted;
  MD_CUDA(cudaStreamWaitEvent(ctx->stream, ctx->ev_prep, 0));      // K4a and the table records (score_prepare_dev)
  MD_LAUNCH(ctx, k_max_candidates, std::min<uint32_t>(blocks(n), 64), 256, 0, W.cand_off.p, n_per ? W.dec_count.p : nullptr, n, d_flag.p + 3);
  int h_pre[4] = {0, 0, 0, 0};
  uint32_t n_left = 0;           // spectra k_build_tables found too dense for the pipelined kernel
  MD_CUDA(cudaMemcpyAsync(h_pre, d_flag.p, sizeof(h_pre), cudaMemcpyDeviceToHost, ctx->stream));
  if (W.tables_built) MD_CUDA(cudaMemcpyAsync(&n_left, W.left_list.p + n, sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx->stream));
  // ---- K4
  ScoreConst C;
  memset(&C, 0, sizeof(C));
  C.w = (uint32_t)w; C.rcp_w = 1.0f / (float)w; C.max_frag_charge = mfc; C.top_k = p.top_k; C.n_per = n_per;
  split_qr(MD_PROTON_UDA, C.w, &C.qp, &C.rp);
  split_qr(2 * MD_PROTON_UDA, C.w, &C.q2p, &C.r2p);
  bool has_var = false;
  for (int c = 0; c < 32; c++) {
    int64_t m = c < MD_NCODES ? ctx->mods.mass[c] : 0;
    int64_t f = (c < MD_NCODES && ctx->mods.has_fix[c] && ctx->mods.fix_pos[c] == MD_POS_A) ? ctx->mods.fix[c] : 0;
    int64_t v = (c < MD_NCODES && ctx->mods.has_var[c]) ? ctx->mods.var[c] : 0;
    if (c < MD_NCODES && ctx->mods.has_fix[c] && ctx->mods.fix_pos[c] == MD_POS_N) {   // floor split: the remainder stays in [0, w)
      const int64_t d = ctx->mods.fix[c], wq = (int64_t)C.w;
      int64_t q = d / wq, r = d % wq;
      if (r < 0) { r += wq; q--; }
      C.nq[c] = (uint32_t)q; C.nr[c] = (uint32_t)r;
    }
    split_qr(m + f, C.w, &C.tq[c], &C.tr[c]);
    split_qr(m + f + v, C.w, &C.vq[c], &C.vr[c]);
    MD_REQUIRE(C.tq[c] < (1u << 22) && C.vq[c] < (1u << 22), MD_ERR_UNSUPPORTED, "fragment_tolerance too small for this residue mass");
    if (c < MD_NCODES && ctx->mods.has_var[c]) has_var = true;
  }
  uint64_t n_targets = 0;
  MD_CUDA(cudaMemcpyAsync(&n_targets, W.cand_off.p + n, sizeof(uint64_t), cudaMemcpyDeviceToHost, ctx->stream));
  MD_CUDA(cudaStreamSynchronize(ctx->stream));
  MD_REQUIRE(!h_pre[0], MD_ERR_INVALID, "spectra: peaks of a spectrum must be sorted by m/z");
  // a table beyond kMaxBins is refused on every path: k_build_tables would leave such a spectrum unscored, k_score flags it
  MD_REQUIRE(h_pre[2] < 0 || (uint64_t)h_pre[2] + kXcorrOffset + 1 <= kMaxBins, MD_ERR_UNSUPPORTED,
             "a spectrum needs more than 2^26 fragment bins or has more than 2^24 candidates");
  if (want_all) { W.tscore.need(n_targets + 1); W.dscore.need((size_t)n * n_per + 1); }
  // Few spectra with very many candidates each (open searches) would leave SMs idle and make one CTA walk hundreds of
  // chunks: split every spectrum into `parts` work items (contiguous ranges of candidate chunks; each builds the table
  // itself, which is cheap beside the chunks), about two items per SM.  MD_SCORE_SPLIT_MIN = candidates per spectrum
  // (batch average) from which that is done (tests lower it).  Only the per-warp top-k lists (top_k <= 8) merge across parts.
  const bool split_classic = getenv("MD_SCORE_SPLIT_CLASSIC") != nullptr;   // (tests: a split batch goes through k_score)
  uint32_t parts = 1;
  if (p.top_k <= kFastTopK) {
    const uint64_t n_cand = (uint64_t)n * n_per + n_targets;
    uint64_t split_min = 16ull * kCandChunk;
    if (const char* env = getenv("MD_SCORE_SPLIT_MIN")) split_min = std::max<long long>(1, atoll(env));
    if (n < (uint32_t)ctx->n_sm && n_cand / n >= split_min)
      parts = std::min<uint32_t>(std::min<uint32_t>(8u, (2u * (uint32_t)ctx->n_sm + n - 1) / n), (uint32_t)((n_cand / n + kCandChunk - 1) / kCandChunk));
    parts = std::max(parts, 1u);
    // the pipelined kernel: of the part counts that leave every scorer warp a few units, the one whose items fill whole rounds
    // of the persistent CTAs best
    if (parts > 1 && W.tables_built && !split_classic) {
      const uint64_t units = (n_cand / n + 31) / 32;
      double best_fill = 0;
      for (uint32_t k = parts; k <= kMaxParts && units / k >= 8ull * kScoreWarps; k++) {
        const double rounds = (double)n * k / ctx->n_sm, fill = rounds / std::ceil(rounds);
        if (fill > best_fill + 0.02) { best_fill = fill; parts = k; }
      }
    }
    if (const char* env = getenv("MD_SCORE_PARTS")) parts = std::min<uint32_t>(std::max(1, atoi(env)), kMaxParts);   // (tests)
  }
  // the pipelined kernel (builders + scorers) takes every batch whose table records were built, unless a split batch is sent to k_score
  const bool pipe = W.tables_built && (parts == 1 || !split_classic);
  const uint32_t grid = std::min<uint32_t>(n * parts, (uint32_t)ctx->n_sm);
  const uint32_t max_nblk = h_pre[2] >= 0 ? ((uint32_t)h_pre[2] + kXcorrOffset + 1 + kBlk - 1) / kBlk : 0;
  uint32_t gstride = 0;
  if (max_nblk > kMapCap && max_nblk <= (kMaxBins >> kBlkShift)) {   // block maps of this batch do not fit shared memory
    gstride = (max_nblk + 64) & ~31u;
    W.gmap.need((size_t)grid * gstride); W.gbits.need((size_t)grid * 2 * (gstride / 32 + 1));
  }
  DevBuf<uint32_t>& work = W.counters; work.need(4);
  MD_CUDA(cudaMemsetAsync(work.p, 0, 4 * sizeof(uint32_t), ctx->stream));
  MD_CUDA(cudaMemsetAsync(W.stat64.p, 0, 4 * sizeof(unsigned long long), ctx->stream));                    // [0..1] statistics; [4] = the table pool's fill (score_prepare_dev)
  ScoreArgs A;
  A.prec = W.prec.p; A.n_spec = n; A.peak_off = S.peak_off; A.pk_bin = W.pk_bin.p; A.pk_yq = W.pk_yq.p; A.pk_count = W.pk_count.p; A.pk_hbin = W.pk_hbin.p;
  A.cand_off = W.cand_off.p; A.cand_desc = W.cand_desc.p; A.cand_mask = W.cand_mask.p; A.cand_w = W.cand_w.p; A.cand_pep = W.cand_pep.p;
  A.idx_rows = ctx->index.rows.p;
  A.dec_slots = (uint64_t)n * n_per; A.dec_rows = W.dec_rows.p; A.dec_len = W.dec_len.p; A.dec_mask = W.dec_mask.p; A.dec_w = W.dec_w.p; A.dec_count = n_per ? W.dec_count.p : nullptr;
  A.tscore = want_all ? W.tscore.p : nullptr; A.dscore = want_all ? W.dscore.p : nullptr; A.psm = psm_dev; A.work = work.p; A.stat64 = W.stat64.p;
  A.error = d_flag.p + 1;
  A.gmap = gstride ? W.gmap.p : nullptr; A.gbits = gstride ? W.gbits.p : nullptr; A.gmap_stride = gstride;
  A.parts = parts; A.part_top = nullptr; A.parts_done = nullptr;
  A.n_work = n; A.remap = nullptr;
  if (parts > 1) {
    W.part_top.need((size_t)n * parts * kFastTopK); W.parts_done.need(n);
    MD_CUDA(cudaMemsetAsync(W.parts_done.p, 0, n * sizeof(uint32_t), ctx->stream));
    A.part_top = W.part_top.p; A.parts_done = W.parts_done.p;
  }
  const bool single = parts == 1 && h_pre[3] <= (int)kCandChunk;     // every spectrum fits one chunk of candidates
  MD_CUDA(cudaEventRecord(ctx->ev[6], ctx->stream));
  if (pipe) {
    // the table records are there (score_prepare_dev); the length-sorted candidate order and the schedule, each by the whole GPU at once
    W.cand_order.need((size_t)n * kPOrder + 16);
    MD_LAUNCH(ctx, k_cand_order, n, 256, 0, A, n_per, W.cand_order.p);
    W.sched_key.need(2 * (size_t)n + 2); W.sched_val.need(2 * (size_t)n + 2); W.sched.need(n + 2);
    MD_LAUNCH(ctx, k_table_keys, blocks(n), 256, 0, reinterpret_cast<const TabDesc*>(W.tab_desc.p), n, W.cand_off.p, n_per ? W.dec_count.p : nullptr, parts > 1, W.sched_key.p,
              W.sched_val.p);
    cubx_sort_pairs<uint32_t, uint32_t>(ctx, W.sched_key.p, W.sched_key.p + n, W.sched_val.p, W.sched_val.p + n, n);
    MD_LAUNCH(ctx, k_pair_schedule, blocks((n + 1) / 2), 256, 0, W.sched_val.p + n, n, parts > 1, W.sched.p);
    MD_CUDA(cudaEventRecord(ctx->ev[6], ctx->stream));
    // spectra too dense for the pipelined kernel (more binned peaks / a larger block map / a larger table record than it stages):
    // k_score works them off on the side stream, beside the pipelined kernel, whose persistent CTAs leave it g2 SMs (its CTAs
    // would otherwise wait for the first of them to end)
    const uint32_t g2 = n_left ? std::min<uint32_t>(std::min<uint32_t>(n_left, grid), std::max<uint32_t>(1u, grid / 8)) : 0u;
    if (n_left) {
      MD_CUDA(cudaStreamWaitEvent(ctx->stream2, ctx->ev[6], 0));
      ScoreArgs A2 = A;
      A2.n_work = n_left; A2.remap = W.left_list.p; A2.work = work.p + 2; A2.parts = 1;
      launch_k_score(ctx, ctx->stream2, g2, A2, C, has_var, single);
      MD_CUDA(cudaEventRecord(ctx->ev_prep, ctx->stream2));
      if (ctx->trace) fprintf(stderr, "[md_trace]   score: %u of %u spectra left to k_score\n", n_left, n);
    }
    const PipeArgs PA{reinterpret_cast<const TabDesc*>(W.tab_desc.p), W.tab_pool.p, W.cand_order.p, W.sched.p, parts};
    auto launch_pipe = [&](auto kernel) {
      MD_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kPipeSmem));
      MD_LAUNCH(ctx, kernel, grid > g2 ? grid - g2 : grid, kPipeThreads, kPipeSmem, A, C, PA);
    };
    if (has_var) launch_pipe(k_score_pipe<true>); else launch_pipe(k_score_pipe<false>);
    if (n_left) MD_CUDA(cudaStreamWaitEvent(ctx->stream, ctx->ev_prep, 0));
    MD_CUDA(cudaEventRecord(ctx->ev[7], ctx->stream));
    if (ctx->trace) {
      unsigned long long top = 0;
      MD_CUDA(cudaMemcpy(&top, W.stat64.p + 4, sizeof(top), cudaMemcpyDeviceToHost));

      std::vector<TabDesc> hd(n);
      MD_CUDA(cudaMemcpy(hd.data(), W.tab_desc.p, n * sizeof(TabDesc), cudaMemcpyDeviceToHost));
      std::vector<uint32_t> na; for (auto& d : hd) if (d.nblk && d.nact != kTabLeft) na.push_back(d.nact);
      std::sort(na.begin(), na.end());
      if (!na.empty()) fprintf(stderr, "[md_trace]   score tables: %.1f KB per spectrum; occupied blocks p10=%u p50=%u p90=%u p99=%u max=%u\n", (double)top / n / 1024.0,
                               na[na.size() / 10], na[na.size() / 2], na[na.size() * 9 / 10], na[na.size() * 99 / 100], na.back());
    }
  } else {
    launch_k_score(ctx, ctx->stream, grid, A, C, has_var, single);
    MD_CUDA(cudaEventRecord(ctx->ev[7], ctx->stream));
  }
  unsigned long long h_stat[2] = {0, 0};
  int h_flag[2] = {0, 0};
  MD_CUDA(cudaMemcpyAsync(h_stat, W.stat64.p, sizeof(h_stat), cudaMemcpyDeviceToHost, ctx->stream));
  MD_CUDA(cudaMemcpyAsync(h_flag, d_flag.p, sizeof(h_flag), cudaMemcpyDeviceToHost, ctx->stream));
  MD_CUDA(cudaStreamSynchronize(ctx->stream));
  { float ms = 0; cudaEventElapsedTime(&ms, ctx->ev[6], ctx->ev[7]); ctx->acc_ms_kscore += ms; ctx->acc_pairs += h_stat[0]; ctx->acc_score_bytes += h_stat[1]; }
  { float ms = 0; if (cudaEventElapsedTime(&ms, ctx->ev_side0, ctx->ev_side1) == cudaSuccess) ctx->acc_ms_prepare += ms; else cudaGetLastError(); }
  ctx->acc_left += pipe ? n_left : 0u; ctx->acc_pipelined = pipe ? 1u : 0u;
  MD_REQUIRE(!h_flag[1], MD_ERR_UNSUPPORTED, "a spectrum needs more than 2^26 fragment bins or has more than 2^24 candidates");
}

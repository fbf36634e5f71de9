// ctx.h -- the per-device context: everything that stays resident in HBM between calls.
#pragma once
#include "common.cuh"

// Resident peptide table (rows of `peptides`, db/schema.sql:14-43), canonical order.
struct PeptideStore {
  bool ready = false;
  uint64_t n = 0;          // unique peptides
  uint64_t seq_bytes = 0;
  uint64_t n_assoc = 0;
  DevBuf<uint8_t> seq;     // generalized ASCII sequences, concatenated
  DevBuf<uint32_t> seq_off;// n+1
  DevBuf<uint8_t> len;     // n
  DevBuf<uint8_t> mc;      // n, min over occurrences
  DevBuf<int64_t> weight;  // n
  DevBuf<int16_t> counts;  // n*21
  DevBuf<uint64_t> hash;   // n
  DevBuf<uint32_t> assoc_off;     // n+1
  DevBuf<uint32_t> assoc_protein; // n_assoc
  // membership table for Decoy::is_peptide (decoy.rs:49-60): open addressing on hash64
  DevBuf<uint64_t> ht_key; // 0 = empty
  DevBuf<uint32_t> ht_val; // peptide ordinal
  uint32_t ht_mask = 0;
};

// Mass-sorted index (replaces `weight BETWEEN ... AND x_count = ...`, identification.rs:24,180-188)
struct MassIndex {
  bool ready = false;
  uint64_t n = 0;
  DevBuf<int64_t> key;      // W*, ascending
  DevBuf<uint32_t> pep;     // peptide ordinal
  DevBuf<int64_t> wfix;     // weight incl. fixed mods
  DevBuf<uint64_t> varpos;  // positions whose letter has a variable modification
  DevBuf<uint64_t> desc;    // score-row descriptor: row offset/16 | len << 40
  DevBuf<uint8_t> rows;     // residue codes, 16-byte padded rows, index order
  DevBuf<int16_t> lcnt;     // per entry: the peptide's counts of the modifiable letters (ModTables::letter_alpha order)
  // MD_VARMOD_EXPANDED: the same entries ordered by wfix (stable over index order)
  DevBuf<int64_t> fkey;     // wfix, ascending
  DevBuf<uint32_t> fent;    // index entry of that key
  uint64_t row_bytes = 0;
  int64_t min_key = 0, max_key = 0;
};

struct IdentifyWorkspace {
  // spectra staged on device by the host-buffer entry point
  DevBuf<double> pmz; DevBuf<uint8_t> charge; DevBuf<uint32_t> sid; DevBuf<uint64_t> peak_off;
  DevBuf<double> peak_mz; DevBuf<float> peak_int;
  DevBuf<md_psm> psm;
  // per spectrum
  DevBuf<md_precursor> prec;
  DevBuf<uint64_t> rbegin, rend;     // index range
  DevBuf<uint64_t> flat_off;         // prefix of range sizes (n+1)
  DevBuf<uint64_t> cand_off;         // CSR of accepted targets (n+1)
  // per index entry in the flattened ranges
  DevBuf<uint64_t> emask; DevBuf<int64_t> ew;
  // accepted targets
  DevBuf<uint64_t> cand_desc; DevBuf<uint64_t> cand_mask; DevBuf<int64_t> cand_w; DevBuf<uint32_t> cand_pep;
  // decoy attempts (one slot per attempt of the current round) and accepted decoys (n_per slots per spectrum)
  DevBuf<uint8_t> att_rows; DevBuf<uint8_t> att_len; DevBuf<uint64_t> att_mask; DevBuf<int64_t> att_w; DevBuf<uint64_t> att_hash;
  DevBuf<uint8_t> dec_rows; DevBuf<uint8_t> dec_len; DevBuf<uint64_t> dec_mask; DevBuf<int64_t> dec_w; DevBuf<uint64_t> dec_hash;
  DevBuf<uint32_t> dec_attempt; DevBuf<uint32_t> dec_count;
  DevBuf<uint32_t> counters; DevBuf<unsigned long long> stat64;
  // binned spectra
  DevBuf<uint16_t> gmap; DevBuf<uint32_t> gbits;   // per-CTA block maps in HBM (tables beyond the shared-memory map)
  DevBuf<int32_t> pk_bin; DevBuf<int32_t> pk_yq; DevBuf<uint32_t> pk_count; DevBuf<int32_t> pk_hbin;
  // scores
  DevBuf<int64_t> tscore; DevBuf<int64_t> dscore;
  DevBuf<uint32_t> left_list;        // spectra the pipelined score kernel left to k_score
  DevBuf<uint8_t> tab_pool, tab_desc; DevBuf<uint16_t> cand_order;   // k_build_tables / k_cand_order -> k_score_pipe
  bool tables_built = false;         // score_prepare_dev built the current batch's table records: score_run_dev may use k_score_pipe
  DevBuf<uint32_t> sched_key, sched_val, sched;                      // the order in which k_score_pipe takes the spectra
  DevBuf<unsigned long long> part_top; DevBuf<uint32_t> parts_done;   // spectra split into parts (open searches): per-part top-k keys, arrival counters
  DevBuf<uint8_t> cub_tmp;
  // per-call temporaries kept between calls (cudaMalloc/cudaFree inside a call would serialise the device)
  DevBuf<uint64_t> t_size; DevBuf<int16_t> t_K; DevBuf<uint32_t> t_flag, t_pos; DevBuf<int> t_ovf, t_unsorted;
  DevBuf<uint32_t> t_list, t_off, t_base, t_queue, t_blk;
  DevBuf<uint4> t_grown; DevBuf<uint8_t> t_route; DevBuf<uint32_t> t_narrow, t_wide;   // decoy rounds: grown attempts (32 B each), repair-pass flags and lists
  DevBuf<uint4> t_start;             // decoy rounds: the repair passes' start state of each grown attempt (64 B each)
  DevBuf<md_precursor> t_win;        // MD_VARMOD_EXPANDED: shifted windows, one per (spectrum, count vector)
};

struct LastDecoys {   // the batch of the last identify call with keep_decoys: its decoys stay in ws.dec_*
  bool have = false;
  uint32_t n_spectra = 0, n_per = 0;
};

struct md_ctx {
  std::string err;
  int device = 0;
  int n_sm = MD_NSM_FALLBACK;
  cudaStream_t stream = nullptr;
  cudaStream_t stream2 = nullptr;          // side stream: work that depends on the spectra alone runs beside the decoy generation
  cudaEvent_t ev_fork = nullptr, ev_prep = nullptr, ev_side0 = nullptr, ev_side1 = nullptr;   // (ev_side*: timing of the side stream's work)
  cudaEvent_t ev[8] = {};
  cudaEvent_t ev_trace[6] = {};   // MD_TRACE only: per-kernel times of a decoy round
  // modifications
  bool mods_set = false;
  ModTables mods;          // host copy (passed to kernels by value)
  int var_mode = 0;        // md_varmod_mode
  // stores
  PeptideStore peps;
  MassIndex index;
  // stored decoys (the `decoys` table): same layout and index as the peptides, no protein associations / hash table
  PeptideStore dstore;
  MassIndex dindex;
  IdentifyWorkspace ws;
  LastDecoys last;
  // multi-GPU (comm.cu): NCCL communicator of this rank, staging buffers of md_gather_psms for host pointers
  void* comm = nullptr;
  int rank = 0, nranks = 1;
  DevBuf<md_psm> gat_send, gat_recv;
  // device-to-device gathers run on their own stream behind the rows they send, so that the next batch is searched
  // meanwhile; the last two are remembered: md_identify_device waits (on the device) before it overwrites a buffer
  // whose gather may still be in flight
  cudaStream_t comm_stream = nullptr;
  cudaEvent_t ev_rows = nullptr;
  struct PendingGather { const void* local = nullptr; cudaEvent_t done = nullptr; } pending[2];
  uint32_t n_gathers = 0;
  uint64_t launches = 0;   // hand-written kernels launched by the current call
  uint64_t cub_calls = 0;  // CUB primitive invocations (scan/select/sort), counted separately
  // per-call accumulators reported through md_identify_stats
  double acc_ms_kscore = 0, acc_ms_kdecoy = 0, acc_ms_prepare = 0;
  uint64_t acc_left = 0; uint32_t acc_pipelined = 0;
  uint64_t acc_attempts = 0, acc_pairs = 0, acc_score_bytes = 0;
  // MD_TRACE=1: host wall-clock marks of the current call, dumped to stderr at its end
  bool trace = false;
  std::vector<std::pair<const char*, double>> marks;
  void mark(const char* what);
  void dump_marks(const char* call);
  void reset_counters() { launches = 0; cub_calls = 0; acc_ms_kscore = acc_ms_kdecoy = acc_ms_prepare = 0; acc_attempts = acc_pairs = acc_score_bytes = 0; acc_left = 0; acc_pipelined = 0; }
};

// per-call helper: count our own kernel launches (bench.py reports it as gpu_launches)
#define MD_LAUNCH(ctx, kernel, grid, block, smem, ...)                         \
  do {                                                                         \
    kernel<<<(grid), (block), (smem), (ctx)->stream>>>(__VA_ARGS__);           \
    (ctx)->launches++;                                                         \
    MD_CUDA(cudaGetLastError());                                               \
  } while (0)

// stage entry points (each file implements one subsystem)
void digest_run(md_ctx* ctx, const uint8_t* residues, const uint64_t* off, uint32_t n_prot, const md_digest_params& p);
void digest_export(md_ctx* ctx, md_peptide_table* out);
void index_build_run(md_ctx* ctx);
// (re)index the stored decoys with the current modifications (no-op without a store)
void index_build_store(md_ctx* ctx);
// stored decoys that pass the ModifiedPeptide filter, in store-index order, into the first decoy slots of each of the n
// precursors in ws.prec (ws.dec_* must be allocated); sets ws.dec_count
void decoys_reuse_dev(md_ctx* ctx, uint32_t n, uint32_t n_per);
void index_window_search_dev(md_ctx* ctx, const md_precursor* prec_dev, uint32_t n, uint64_t* begin_dev, uint64_t* end_dev);
// fills ws.cand_* and ws.cand_off for the n precursors in ws.prec; returns total accepted
uint64_t index_candidates_dev(md_ctx* ctx, uint32_t n);
// fills ws.dec_* for n precursors in ws.prec
void decoys_generate_dev(md_ctx* ctx, uint32_t n, uint32_t n_per, int mode, uint64_t seed);
void decoys_export(md_ctx* ctx, uint32_t n, uint32_t n_per, md_decoy_table* out);
// bins the n spectra (device SoA), scores targets+decoys, writes PSM rows
struct SpectraDev { uint32_t n; const double* pmz; const uint8_t* charge; const uint32_t* sid; const uint64_t* peak_off; const double* peak_mz; const float* peak_int; };
void score_prepare_dev(md_ctx* ctx, const SpectraDev& S, uint64_t n_peaks, const md_search_params& p);
void score_run_dev(md_ctx* ctx, const SpectraDev& S, const md_search_params& p, uint32_t n_per, md_psm* psm_dev, bool want_all);
void precursors_dev(md_ctx* ctx, const SpectraDev& S, const md_search_params& p, uint32_t id_base);

size_t cub_temp_bytes_max(size_t n);
void comm_release(md_ctx* ctx);   // comm.cu: ncclCommDestroy if a communicator exists
void comm_wait_for_buffer(md_ctx* ctx, const void* buf);   // comm.cu: the ctx stream waits for a gather still reading `buf`
void comm_sync(md_ctx* ctx);

/*
 * maxdecoy.h -- C ABI of the B200-native MaxDecoy identification hot path.
 *
 * One header, two implementations with identical symbols:
 *   - max-decoy_b200/csrc/libmaxdecoy_cuda.so   hand-written sm_100a CUDA (the product)
 *   - oracle/libmaxdecoy_oracle.so              CPU restatement (test infrastructure only)
 *
 * The reference (mpc-bioinformatics/max-decoy, Rust) has no FFI of its own; every entry
 * point below names the reference function (file:line under /root/reference/src/proteomic
 * unless stated otherwise) whose work it takes over, so a Rust host can bind it 1:1 with
 * `extern "C"` + `#[repr(C)]` (see INTEGRATION.md).
 *
 * Conventions
 *   - every function returns md_status (0 = ok, negative = error); nothing throws or
 *     aborts across the boundary (the reference panics instead: e.g. tasks/identification.rs:240);
 *   - md_last_error(ctx) gives the message of the last failing call on that ctx;
 *   - inputs are borrowed for the duration of the call; tables the library allocates
 *     (md_*_table) are released with the matching md_*_table_free;
 *   - one md_ctx per device; calls on one ctx are serialised by the caller; ctxs on
 *     different devices are independent;
 *   - all masses are int64 micro-dalton ("uDa"), the reference's integer mass unit
 *     (models/mass/mod.rs:3-8, truncating conversion);
 *   - residues are ASCII one-letter codes.  Peptide sequences inside the library are
 *     "generalized" (I,L -> J; models/amino_acids/amino_acid.rs:139-141).
 */
#ifndef MAXDECOY_H
#define MAXDECOY_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MD_API __attribute__((visibility("default")))

/* The 21 letters used for decoy generation and for the <x>_count columns
 * (models/amino_acids/amino_acid.rs:4-5; db/schema.sql:20-40). Index = column order. */
#define MD_ALPHABET "ARNDCEQGHJKMFPOSTUVWY"
#define MD_ALPHABET_SIZE 21
#define MD_MAX_PEPTIDE_LEN 60 /* VARCHAR(60): db/schema.sql:16,165; digestion.rs:74,101 */
#define MD_WATER_UDA 18010565LL /* models/mass/neutral_loss.rs:3 */
#define MD_PROTON_UDA 1007276LL /* models/mass/mod.rs:4 (1.007276 * 1e6, exact) */

typedef enum md_status {
  MD_OK = 0,
  MD_ERR_INVALID = -1,     /* bad argument / malformed input */
  MD_ERR_STATE = -2,       /* call order violated (e.g. index before digest) */
  MD_ERR_DEVICE = -3,      /* CUDA error (message in md_last_error) */
  MD_ERR_NOMEM = -4,
  MD_ERR_UNSUPPORTED = -5  /* feature outside the hot path (see DESIGN.md) */
} md_status;

typedef struct md_ctx md_ctx;

typedef struct md_config {
  int32_t device;     /* CUDA ordinal; ignored by the oracle */
  uint32_t n_threads; /* oracle only: host threads for the spectrum loop (0 = 1) */
} md_config;

MD_API int md_create(const md_config* cfg, md_ctx** out);
MD_API void md_destroy(md_ctx* ctx);
MD_API const char* md_last_error(const md_ctx* ctx);
/* "cuda-sm100a" or "cpu-oracle" */
MD_API const char* md_backend_name(void);

/* ------------------------------------------------------------------ masses (pure) */

/* AminoAcid::get(c).get_mono_mass()  (amino_acid.rs:7-35,87-117; unknown letter -> X -> 0) */
MD_API int64_t md_residue_mass(uint8_t one_letter_code);
/* AminoAcid::get_sequence_weight  (amino_acid.rs:130-136): H2O + sum of residue masses.
 * `sequence-mass` subcommand: tasks/sequence_mass.rs:24-27. */
MD_API int64_t md_sequence_weight(const uint8_t* seq, uint32_t len);
/* Precursor mass and tolerance window of one spectrum, tasks/identification.rs:203-211
 * (utility/mod.rs:9-11, models/mass/mod.rs:6-8,14-16); all f64, no FMA, truncation. */
MD_API int md_precursor_window(double mz, uint32_t charge, int64_t lower_ppm, int64_t upper_ppm,
                               int64_t* precursor, int64_t* lo, int64_t* hi);

/* ------------------------------------------------------------------ modifications */

/* One row of the modification CSV (models/amino_acids/modification.rs:36-76). */
typedef struct md_modification {
  char accession[24];  /* lower-cased by the library (modification.rs:48) */
  char name[40];
  uint8_t position;    /* 'A' anywhere, 'N' / 'C' terminus (modification.rs:24-33): a terminal modification sits on the first / last residue
                        * only, and only when that residue is `amino_acid` (add_modification_at, modified_peptide.rs:421-447;
                        * set_variable_modification_at, :339-367).  MD_DECOY_EXHAUSTIVE returns MD_ERR_UNSUPPORTED
                        * with terminal modifications (compositions: the weight would depend on the order). */
  uint8_t is_fix;      /* != 0 -> fixed */
  uint8_t amino_acid;  /* one letter code, upper-cased */
  uint8_t _pad[5];
  int64_t mono_mass;   /* uDa, convert_mass_to_int of the CSV value */
} md_modification;

/* Replaces the fixed/variable maps of identification_task (tasks/identification.rs:163-196).
 * `max_variable_mods` is `-n` (max_number_of_variable_modification_per_decoy). */
MD_API int md_set_modifications(md_ctx* ctx, const md_modification* mods, uint32_t n_mods,
                                uint32_t max_variable_mods);
/* DecoyGenerator::get_one_amino_acid_substitute_map (utility/decoy_generator.rs:301-324):
 * out[from*21+to] = (m[to]+fix[to]) - (m[from]+fix[from]); `amino-acid-substitution` subcommand. */
MD_API int md_substitution_map(md_ctx* ctx, int64_t* out441);

/* ------------------------------------------------------------------ digest (K1) */

typedef struct md_digest_params {
  uint32_t max_missed_cleavages; /* -c */
  uint32_t min_len;              /* -l */
  uint32_t max_len;              /* -h, <= 60 */
} md_digest_params;

/* Trypsin digest of `n_proteins` proteins given as one concatenated residue buffer and
 * n_proteins+1 offsets.  Replaces FastaDigester -> DigestEnzym::digest -> Peptide::new
 * (utility/input_file_digester/fasta_digester.rs:69-140; models/enzyms/digest_enzym.rs:61-86;
 * models/enzyms/trypsin.rs:29; models/peptides/peptide.rs:27-37).  The result -- unique
 * generalized sequences (UNIQUE(aa_sequence, weight), db/schema.sql:41), in canonical order
 * (weight, hash64(sequence), first occurrence) -- stays resident in the ctx (HBM). */
MD_API int md_digest(md_ctx* ctx, const uint8_t* residues, const uint64_t* protein_offsets,
                     uint32_t n_proteins, const md_digest_params* params, uint64_t* n_peptides);

/* Host copy of the resident peptide table: rows of table `peptides` (db/schema.sql:14-43)
 * plus the `peptides_proteins` links as CSR.  peptide id = row index + 1. */
typedef struct md_peptide_table {
  uint64_t n;
  uint64_t seq_bytes;
  uint64_t n_assoc;
  uint8_t* seq;             /* concatenated generalized sequences */
  uint64_t* seq_off;        /* n+1 */
  uint8_t* missed_cleavages;/* min over occurrences */
  int64_t* weight;          /* unmodified, H2O included */
  int16_t* counts;          /* n*21, MD_ALPHABET order (peptide_interface.rs:22-28) */
  uint64_t* assoc_off;      /* n+1 */
  uint32_t* assoc_protein;  /* protein ordinals, ascending, unique per peptide */
} md_peptide_table;
MD_API int md_peptides_export(md_ctx* ctx, md_peptide_table* out);
MD_API void md_peptide_table_free(md_peptide_table* t);

/* ------------------------------------------------------------------ index + lookup (K2) */

/* Sort the resident peptides by W* = weight + sum_a count_a * delta_a (a over the modifiable
 * letters; variable overrides fixed): the single window the reference's SQL fan-out
 * (tasks/identification.rs:24,180-188,214-241,374-403) is equivalent to.  Needs md_digest
 * and md_set_modifications. */
MD_API int md_index_build(md_ctx* ctx);

typedef struct md_index_stats {
  uint64_t n_peptides;
  uint64_t seq_bytes;
  uint64_t device_bytes;
  int64_t min_key;
  int64_t max_key;
} md_index_stats;
MD_API int md_index_stats_get(md_ctx* ctx, md_index_stats* out);

/* For each [lo,hi]: begin = first index position with W* >= lo, end = first with W* > hi. */
MD_API int md_window_search(md_ctx* ctx, const int64_t* lo, const int64_t* hi, uint32_t n,
                            uint64_t* begin, uint64_t* end);
/* Index rows [begin, begin+count): peptide id (1-based) and W*; parity helper. */
MD_API int md_index_export(md_ctx* ctx, uint64_t begin, uint64_t count, uint64_t* peptide_id,
                           int64_t* key);

/* How a target peptide's variable modifications are placed (md_candidates / md_identify*; decoys always follow the
 * reference's repair loop).
 *  MD_VARMOD_REFERENCE: the reference's procedure (tasks/identification.rs:242-257 +
 *    ModifiedPeptide::try_variable_modifications, models/peptides/modified_peptide.rs:512-543): the SQL fan-out only
 *    retrieves peptides whose FULLY modified weight W* lies in the window, and the first placement that hits wins, so a
 *    peptide is found with all of its variable-modifiable residues modified or not at all (SURVEY A.4).
 *  MD_VARMOD_EXPANDED (SURVEY 8(f) row 4; not in the reference): every (peptide, set S of variable-modifiable residues,
 *    |S| <= max_variable_mods) whose weight incl. fixed modifications + the deltas of S lies in the window is a candidate
 *    of its own -- partial occupancy is found, and every placement is scored.  A residue whose letter also has a fixed
 *    modification is not variable-modifiable (modified_peptide.rs:355,532).  Candidate order per spectrum: count
 *    vectors (k_a over the variable letters in alphabetical order, sum <= max_variable_mods, ascending as mixed-radix
 *    numbers with the last letter fastest), then ascending fixed-modification weight (ties: index order), then
 *    placements with the last letter fastest, each letter's subsets in NChooseK order (utility/combinations/n_choose_k.rs:12-49).
 * Changing the mode invalidates the index (md_index_build again).
 * Limits of the CUDA lookup; each returns MD_ERR_UNSUPPORTED from md_candidates / md_identify*, the oracle has none:
 *  MD_VARMOD_REFERENCE: 2^22 subsets tried for one (spectrum, peptide): sum over n <= max_variable_mods of
 *    C(d, n), d = the peptide's residues of variable letters, when no smaller placement lands in the window.
 *  MD_VARMOD_EXPANDED: at most 6 variable letters (a letter whose fixed modification holds the variable slot does not
 *    count), at most 96 count vectors (C(max_variable_mods + letters, letters)), and at most 2^20 - 1 placements
 *    (prod_a C(count_a, k_a)) of one peptide for one count vector. */
typedef enum md_varmod_mode { MD_VARMOD_REFERENCE = 0, MD_VARMOD_EXPANDED = 1 } md_varmod_mode;
MD_API int md_set_variable_mode(md_ctx* ctx, int mode);

typedef struct md_precursor {
  int64_t mass;         /* P  */
  int64_t lo;           /* lower tolerance limit */
  int64_t hi;           /* upper tolerance limit */
  uint32_t charge;
  uint32_t spectrum_id; /* global id; keys the decoy RNG so results do not depend on sharding */
} md_precursor;

/* Targets of each precursor after the ModifiedPeptide filter (tasks/identification.rs:231-257;
 * models/peptides/modified_peptide.rs:118-159,512-543): index order, CSR by spectrum.
 * var_mask bit i = residue i carries its variable modification (first hit of
 * try_variable_modifications); mod_weight = weight incl. all applied modifications. */
typedef struct md_candidate_table {
  uint32_t n_spectra;
  uint64_t n;
  uint64_t* off;        /* n_spectra+1 */
  uint64_t* peptide_id; /* 1-based */
  uint64_t* var_mask;
  int64_t* mod_weight;
} md_candidate_table;
MD_API int md_candidates(md_ctx* ctx, const md_precursor* precursors, uint32_t n_spectra,
                         md_candidate_table* out);
MD_API void md_candidate_table_free(md_candidate_table* t);

/* ------------------------------------------------------------------ decoys (K3) */

typedef enum md_decoy_mode {
  /* DecoyGenerator::generate_decoys + swap_amino_acids_to_hit_mass_tolerance
   * (utility/decoy_generator.rs:127-188; modified_peptide.rs:451-508) with a counter-based
   * RNG keyed by (seed, spectrum_id, attempt); the reference's RNG is unseeded.  The repair loop works in 32-bit
   * residuals: md_generate_decoys returns MD_ERR_UNSUPPORTED when a residue with its fixed modification (or a variable
   * modification) reaches 2^29 uDa (536.87 Da), or when a precursor window reaches further than 2^30 - 1 uDa
   * (1073.74 Da) from its mass; the reference has neither limit. */
  MD_DECOY_REFERENCE_RANDOM = 0,
  /* every sequence whose fixed-modification weight lies in the window: compositions (count vectors over MD_ALPHABET)
   * in ascending lexicographic order, per composition its distinct permutations in ascending lexicographic order;
   * peptides of the index are skipped; `attempt` = ordinal in that enumeration */
  MD_DECOY_EXHAUSTIVE = 1,
  /* DecoyGenerator::vary_targets (utility/decoy_generator.rs:265-296): shuffled targets */
  MD_DECOY_PERMUTE_TARGET = 2
} md_decoy_mode;

typedef struct md_decoy_table {
  uint32_t n_spectra;
  uint64_t n;
  uint64_t seq_bytes;
  uint64_t* off;        /* n_spectra+1; off[s+1]-off[s] < requested  <=>  `.less_decoys` */
  uint8_t* seq;
  uint64_t* seq_off;    /* n+1 */
  uint64_t* var_mask;
  int64_t* weight;      /* Decoy::new: unmodified weight (models/peptides/decoy.rs:25-36) */
  int64_t* mod_weight;  /* weight incl. modifications; lo <= mod_weight <= hi */
  uint32_t* attempt;    /* attempt / enumeration ordinal that produced it */
} md_decoy_table;
/* Stored decoys: the `decoys` table (db/schema.sql:163-192; Decoy::find_where, models/peptides/decoy.rs:118-153).
 * identification_task looks persisted decoys up with the same window/count queries as the targets, passes them
 * through the same ModifiedPeptide filter and reuses them before it generates new ones
 * (tasks/identification.rs:259-283).  md_decoy_store_set replaces the ctx's store with `n` sequences over MD_ALPHABET
 * (length 1..60; duplicates are dropped; n = 0 clears it); the store is indexed by W* by md_index_build, or at once if
 * an index is already built.  With a non-empty store, MD_DECOY_REFERENCE_RANDOM first takes, per spectrum, the stored
 * decoys that pass the filter in store-index order (W*, then (weight, sequence hash, sequence)) up to the requested
 * number -- reported with `attempt` = MD_DECOY_STORED -- and generates only the remainder (the reference's order is
 * the database's row order, i.e. unspecified).  The other modes ignore the store. */
#define MD_DECOY_STORED 0xFFFFFFFFu
MD_API int md_decoy_store_set(md_ctx* ctx, const uint8_t* seq, const uint64_t* seq_off, uint64_t n);

MD_API int md_generate_decoys(md_ctx* ctx, const md_precursor* precursors, uint32_t n_spectra,
                              uint32_t n_per_spectrum, int mode, uint64_t seed,
                              md_decoy_table* out);
MD_API void md_decoy_table_free(md_decoy_table* t);

/* ------------------------------------------------------------------ identify = lookup + decoys + score (K4) */

/* MS2 spectra, structure of arrays.  Peaks of one spectrum must be sorted by m/z. */
typedef struct md_spectra {
  uint32_t n;
  const double* precursor_mz;   /* `selected ion m/z`  (utility/mz_ml/spectrum.rs:33-103) */
  const uint8_t* charge;        /* `charge state` */
  const uint32_t* spectrum_id;  /* may be NULL -> 0..n-1 */
  const uint64_t* peak_off;     /* n+1 */
  const double* peak_mz;
  const float* peak_intensity;
} md_spectra;

typedef struct md_search_params {
  int64_t lower_ppm;            /* -l */
  int64_t upper_ppm;            /* -u */
  int64_t abs_lower_uda;        /* if abs_lower_uda|abs_upper_uda != 0: window = [P-abs_lower, P+abs_upper] (open search) */
  int64_t abs_upper_uda;
  double fragment_tolerance;    /* --fragmentation-tolerance, Comet fragment_bin_tol (comet_parameter.rs:103); 0.0001..2 Da,
                                 * rounded to whole uDa (w).  The CUDA library refuses with MD_ERR_UNSUPPORTED (the oracle
                                 * accepts): a scored spectrum whose table needs more than 2^26 bins, i.e. a usable peak at
                                 * m/z >= (2^26 - 76) * w (6.71 kDa at 0.0001 Da); a residue whose mass with its fixed and
                                 * variable modifications reaches 2^22 * w (419 Da at 0.0001 Da). */
  uint32_t n_decoys;            /* -d */
  int32_t decoy_mode;           /* md_decoy_mode */
  uint64_t seed;
  uint32_t top_k;               /* PSM rows per spectrum (<= 128) */
  uint32_t min_peaks;           /* Comet minimum_peaks (comet_parameter.rs:62) */
  uint32_t max_fragment_charge; /* Comet max_fragment_charge (comet_parameter.rs:55) */
  uint32_t keep_decoys;         /* != 0: keep the generated decoys for md_last_decoys_export */
} md_search_params;

/* One row of the (new) psms table; fixed width so that per-rank tables can be gathered
 * with one collective.  56 bytes. */
typedef struct md_psm {
  uint32_t spectrum_id;
  uint16_t rank;        /* 1..top_k; 0 = empty row */
  uint8_t is_decoy;
  uint8_t charge;
  uint64_t candidate;   /* target: peptide id (1-based); decoy: ordinal within the spectrum's decoys */
  uint64_t var_mask;
  int64_t mod_weight;
  int64_t raw_score;    /* exact integer: 150 * 2^16 * sum of fast-xcorr bins */
  float score;          /* 0.005 * raw_score / (150 * 65536) */
  uint32_t n_targets;   /* candidates scored for this spectrum */
  uint32_t n_decoys;
  uint32_t _pad;
} md_psm;

typedef struct md_identify_stats {
  uint64_t n_spectra;
  uint64_t n_targets;       /* target candidates scored */
  uint64_t n_decoys;        /* decoys generated and scored */
  uint64_t n_less_decoys;   /* spectra that got fewer decoys than requested */
  uint64_t n_kernel_launches; /* hand-written kernels launched by the call (CUB primitives not counted) */
  double ms_lookup, ms_decoys, ms_score, ms_total; /* device time (CUDA events) / host time (oracle) */
  /* per-kernel device time, CUDA events on the ctx stream (0 in the oracle) */
  double ms_kernel_score;     /* the fused fragment-and-score kernel alone */
  double ms_kernel_decoy;     /* the decoy attempt kernels (all rounds) */
  uint64_t n_attempts;        /* decoy attempts run */
  uint64_t n_pairs;           /* (spectrum, candidate) pairs scored */
  uint64_t score_bytes;       /* algorithmic bytes of the score kernel: sum over pairs of (14 + len) */
  /* the pipelined score path (DESIGN.md section 4): device time of what runs beside the decoy generation on the side
   * stream (spectrum binning + table records), spectra the pipelined kernel left to the classic one, and which kernel ran */
  double ms_score_prepare;
  uint64_t n_score_left;
  uint32_t score_pipelined;   /* 1: k_score_pipe scored the batch; 0: k_score */
  uint32_t _pad;
} md_identify_stats;

/* identification_task for a batch of spectra (tasks/identification.rs:201-368), with the
 * b/y fragment scoring the reference delegates to Comet (utility/comet_parameter.rs:6-124;
 * run_splitup_and_identification.sh:47-60) done in place.  Host buffers in, host PSM rows out
 * (n * top_k rows, spectrum-major).  `all_scores`, if not NULL, receives the raw score of every
 * candidate (targets in index order, then decoys) and `all_off` (n+1) their CSR offsets; both
 * are malloc'ed by the library and released with md_free. */
MD_API int md_identify(md_ctx* ctx, const md_spectra* spectra, const md_search_params* params,
                       md_psm* psms, md_identify_stats* stats, int64_t** all_scores,
                       uint64_t** all_off);
/* Same, with every pointer inside `spectra` and `psms` being a device pointer on the ctx's
 * device (e.g. `psms` = the NCCL send buffer of the PSM gather).  The work runs on the ctx
 * stream; the call returns when the PSM rows are in `psms`.  CUDA implementation only. */
MD_API int md_identify_device(md_ctx* ctx, const md_spectra* spectra_dev,
                              const md_search_params* params, md_psm* psms_dev,
                              md_identify_stats* stats);
/* ------------------------------------------------------------------ multi-GPU: spectra sharded, index replicated */

/* The reference walks the spectra one after the other (the `for spectrum in spectra` loop of identification_task,
 * tasks/identification.rs:201) and no iteration reads what another one wrote, so the loop is the unit of parallelism:
 * one process and one md_ctx per GPU, every rank digests the same FASTA (the index is replicated), identifies its own
 * share of the spectra (global spectrum ids key the decoy RNG, so the result does not depend on the number of ranks)
 * and the only exchange is the gather of the fixed-width PSM tables -- NCCL over NVLink.
 *
 * md_comm_unique_id: rank 0 draws the communicator id (ncclGetUniqueId) and hands the bytes to the other ranks by
 *   whatever channel the host has (a file, an environment variable, MPI, a torch.distributed store).
 * md_comm_init: collective over all ranks (ncclCommInitRank on the ctx's device).  nranks == 1 needs no NCCL at all.
 * md_gather_psms: all-gather of `rows_per_rank` PSM rows from every rank into `all` (nranks * rows_per_rank rows, rank
 *   major) on the ctx stream.  `local` and `all` may each be a device pointer (used in place: `local` can be the
 *   buffer md_identify_device wrote) or a host pointer (staged through the ctx); every rank passes the same
 *   rows_per_rank (pad short shards with rows whose rank field is 0).  Returns after the rows are in `all` unless both
 *   pointers are device pointers, in which case the gather is asynchronous on the ctx stream until md_sync.
 *   Without md_comm_init (or with nranks == 1) it is a copy.
 * md_comm_destroy: releases the communicator (md_destroy does it too). */
#define MD_COMM_ID_BYTES 128
MD_API int md_comm_unique_id(uint8_t id[MD_COMM_ID_BYTES]);
MD_API int md_comm_init(md_ctx* ctx, int32_t rank, int32_t nranks, const uint8_t id[MD_COMM_ID_BYTES]);
MD_API int md_gather_psms(md_ctx* ctx, const md_psm* local, uint64_t rows_per_rank, md_psm* all);
MD_API int md_comm_destroy(md_ctx* ctx);

MD_API int md_sync(md_ctx* ctx);
/* The cudaStream_t the ctx launches on (NULL in the oracle), for callers that bracket calls
 * with their own CUDA events. */
MD_API void* md_stream_handle(md_ctx* ctx);
/* The decoys of the last md_identify* call with keep_decoys != 0. */
MD_API int md_last_decoys_export(md_ctx* ctx, md_decoy_table* out);
MD_API void md_free(void* p);

#ifdef __cplusplus
}
#endif
#endif /* MAXDECOY_H */

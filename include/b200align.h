/*
 * b200align.h -- C ABI of libb200align.so: the drop-in boundary for the
 * `bio::alignment::pairwise` hot path of rust-bio 4.0.1, rebuilt B200-native.
 *
 * The reference has no FFI for this path: its boundary is the Rust method
 * surface (reference src/alignment/pairwise/mod.rs):
 *     Scoring<F>                       mod.rs:238-429
 *     Aligner::with_capacity / ...     mod.rs:495-583
 *     Aligner::custom                  mod.rs:591-922
 *     Aligner::global                  mod.rs:925-951
 *     Aligner::semiglobal              mod.rs:954-983
 *     Aligner::local                   mod.rs:986-1015
 *     banded::Aligner::*               banded.rs:150-401, 872-1004
 * A per-pair call cannot feed a GPU, so every entry point here is the BATCH
 * form of one of those methods; a single-pair call is a batch of one.  The
 * Rust shim (rust_bio_b200/rust/src/lib.rs) and the Python mirror
 * (rust_bio_b200/pairwise.py) bind exactly these symbols.
 *
 * Conventions
 *   - plain C, no exceptions / unwinding across the boundary;
 *   - every function returns 0 on success or a negative B2A_E_* code;
 *     b2a_last_error() gives the text for the calling engine;
 *   - an engine handle is bound to ONE CUDA device and may be used by one
 *     host thread at a time (the reference's `&mut self` contract,
 *     mod.rs:591,925,954,986);
 *   - there is NO CPU fallback: every align call fails with
 *     B2A_E_NO_DEVICE if the CUDA device cannot be used.
 */
#ifndef B200ALIGN_H_
#define B200ALIGN_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* pairwise::MIN_SCORE (mod.rs:174) */
#define B2A_MIN_SCORE (-858993459)

/* banded::MAX_CELLS (banded.rs:104) */
#define B2A_BANDED_MAX_CELLS 5000000ull

/* AlignmentMode, in bio-types variant order (used at mod.rs:920,942,971,1003) */
enum {
  B2A_MODE_CUSTOM = 0,     /* Aligner::custom      mod.rs:591 */
  B2A_MODE_GLOBAL = 1,     /* Aligner::global      mod.rs:925 */
  B2A_MODE_SEMIGLOBAL = 2, /* Aligner::semiglobal  mod.rs:954 */
  B2A_MODE_LOCAL = 3       /* Aligner::local       mod.rs:986 */
};

/* AlignmentOperation codes (bio-types variant order; pushed at mod.rs:860-900) */
enum {
  B2A_OP_MATCH = 0,
  B2A_OP_SUBST = 1,
  B2A_OP_DEL = 2,
  B2A_OP_INS = 3,
  B2A_OP_XCLIP = 4, /* length is in clip_len, in order of appearance */
  B2A_OP_YCLIP = 5
};

/* error codes */
enum {
  B2A_OK = 0,
  B2A_E_INVALID = -1,     /* bad argument (the reference would panic: mod.rs:517-518,554-571) */
  B2A_E_NO_DEVICE = -2,   /* CUDA device / driver unusable: no CPU fallback exists */
  B2A_E_CUDA = -3,        /* a CUDA runtime call failed; see b2a_last_error */
  B2A_E_RANGE = -4,       /* scores/lengths would overflow i32 in the reference recurrence */
  B2A_E_CAPACITY = -5,    /* caller's ops buffer too small */
  B2A_E_STATE = -6,       /* stage/run/fetch called out of order */
  B2A_E_UNSUPPORTED = -7  /* sequence too long for this build's on-chip staging */
};

/* Scoring<F> (mod.rs:238-247).  `table`, when non-NULL, is the host-tabulated
 * MatchFunc: 256x256 row-major, table[a*256+b] = match_fn.score(a, b)
 * (mod.rs:177-228); only entries for symbols present in the batch are read.
 * When NULL, MatchParams semantics apply (mod.rs:208-217).
 * has_match_scores/match_score mirror `match_scores: Option<(i32,i32)>`
 * (mod.rs:242), which only banded::Band::create consults (banded.rs:1315-1318). */
typedef struct b2a_scoring {
  int32_t gap_open;
  int32_t gap_extend;
  int32_t xclip_prefix;
  int32_t xclip_suffix;
  int32_t yclip_prefix;
  int32_t yclip_suffix;
  int32_t match_score;
  int32_t mismatch_score;
  int32_t has_match_scores;
  const int32_t* table;
  /* Symbols for which `table` is valid (e.g. "A-Z*" for bio::scores matrices).
   * NULL with a non-NULL table: the engine scans the batch for the symbols
   * present (slower).  A sequence byte outside the alphabet is B2A_E_INVALID
   * (bio::scores::lookup would index out of bounds, scores/mod.rs:22-35). */
  const uint8_t* alphabet;
  uint32_t alphabet_len;
} b2a_scoring;

/* A batch of (x, y) pairs: TextSlice arguments of the align methods. */
typedef struct b2a_pairs {
  const uint8_t* seq_blob;  /* all sequences, any layout */
  const uint64_t* x_off;    /* [n_pairs] byte offset of x in seq_blob */
  const uint32_t* x_len;    /* [n_pairs] m */
  const uint64_t* y_off;    /* [n_pairs] */
  const uint32_t* y_len;    /* [n_pairs] n */
  uint64_t blob_bytes;
  uint64_t n_pairs;
} b2a_pairs;

/* Caller-allocated host outputs == the fields of bio_types Alignment
 * (built at mod.rs:911-921); xlen/ylen/mode are known to the caller. */
typedef struct b2a_results {
  int32_t* score;      /* [n_pairs] */
  uint32_t* xstart;    /* [n_pairs] */
  uint32_t* xend;      /* [n_pairs] */
  uint32_t* ystart;    /* [n_pairs] */
  uint32_t* yend;      /* [n_pairs] */
  uint64_t* ops_off;   /* [n_pairs+1] prefix offsets into ops */
  uint8_t* ops;        /* [ops_capacity] B2A_OP_* codes, alignment order */
  uint64_t ops_capacity;
  uint32_t* clip_len;  /* [4*n_pairs] lengths of the Xclip/Yclip ops of a pair, in order of appearance */
  /* [n_pairs] B2A_PAIR_* per pair, or NULL.  The reference fails per CALL: a pair on which it would panic
   * (mod.rs:905 "Dint expect this!", banded.rs walk on a corrupt cell, an asserting caller-supplied match list)
   * or never return takes only that pair down.  With status == NULL such a pair fails the whole batch
   * (B2A_E_RANGE / B2A_E_INVALID / B2A_E_CAPACITY); with a status array the batch succeeds, the pair's status is
   * non-zero and its other outputs are score = B2A_MIN_SCORE, no ops. */
  uint32_t* status;
} b2a_results;

enum {
  B2A_PAIR_OK = 0,
  B2A_PAIR_PANIC = 1,        /* the reference panics (or loops forever) on this pair */
  B2A_PAIR_CAPACITY = 2,     /* banded: more k-mer matches than the engine's per-pair limit (2^22) */
  B2A_PAIR_INVALID_HINT = 4  /* banded: caller-supplied matches/path the reference asserts on */
};

typedef struct b2a_stats {
  uint64_t cells;          /* sum of DP cells (m*n, or Band::num_cells for banded) */
  uint64_t h2d_bytes;
  uint64_t d2h_bytes;
  uint64_t traceback_bytes; /* traceback bit-vector bytes the fill kernel stores */
  float pack_ms;           /* K0 */
  float fill_ms;           /* K1 (or K3) */
  float walk_ms;           /* K2 epilogue + traceback walk (+ ops compaction) */
  float band_ms;           /* K4 (banded only) */
  uint32_t kernel_launches;
  uint32_t waves;          /* sub-batches the traceback budget forced */
  uint32_t fill_lanes_per_pair; /* G of the fill kernel variant used */
  uint32_t fill_rows_per_lane;  /* R */
} b2a_stats;

typedef struct b2a_engine b2a_engine;

/* lifecycle */
int32_t b2a_engine_create(b2a_engine** out, int32_t device_id);
int32_t b2a_engine_destroy(b2a_engine* e);
const char* b2a_last_error(const b2a_engine* e);
const char* b2a_version(void);

/* Run all engine work on this cudaStream_t (default: an engine-owned stream). */
int32_t b2a_engine_set_stream(b2a_engine* e, void* cuda_stream);
/* Upper bound (bytes) on device scratch for traceback bit-vectors; larger
 * batches are processed in waves. 0 = default (60% of free HBM). */
int32_t b2a_engine_set_traceback_budget(b2a_engine* e, uint64_t bytes);
/* Force the fill-kernel shape (lanes per pair G in {1,2,4,8,32}, rows per
 * lane R in {8,16,20}: the built pairs are 1x8 1x16 1x20 2x16 2x20 4x16 8x16 8x20 32x8 32x16); 0,0 = automatic. */
int32_t b2a_engine_set_tuning(b2a_engine* e, int32_t lanes_per_pair, int32_t rows_per_lane);

/* The alphabet the last stage used: the caller's, or the byte values the engine found in the batch when
 * b2a_scoring.alphabet was NULL (symbols[256], ascending).  A caller that cuts one batch into pieces can hand the
 * first piece's alphabet to the others (b2a_scoring.alphabet) and spare them the discovery pass and its
 * synchronisation; a piece holding a byte outside it fails with B2A_E_INVALID and is redone without. */
int32_t b2a_engine_last_alphabet(const b2a_engine* e, uint8_t* symbols, uint32_t* n_symbols);

/* K2 (row m, last-column fix-ups, traceback walk) runs one lane per pair (1) or one warp per pair (2);
 * 0 = automatic: warp per pair for waves of up to 16,384 pairs.  Results are identical either way. */
int32_t b2a_engine_set_walk(b2a_engine* e, int32_t mode);

/* b2a_align_batch cuts batches of >= 262,144 pairs into `chunks` pieces that alternate between two
 * internal engines, so one chunk's copies and host planning overlap the other's kernels.
 * chunks < 2 disables the pipeline (default 5, relative sizes 1,3,6,6,3). Results are identical either way. */
int32_t b2a_engine_set_pipeline(b2a_engine* e, int32_t chunks);

/* One-call form: Aligner::{custom,global,semiglobal,local} over a batch with
 * HOST inputs and HOST outputs (copies inside). mode = B2A_MODE_*. */
int32_t b2a_align_batch(b2a_engine* e, int32_t mode, const b2a_scoring* scoring,
                        const b2a_pairs* pairs, b2a_results* results, b2a_stats* stats);

/* Score-only outputs: the score, xend and yend of the Alignment b2a_align_batch would return (caller-allocated
 * host arrays; any of them may be NULL). */
typedef struct b2a_score_results {
  int32_t* score;   /* [n_pairs] */
  uint32_t* xend;   /* [n_pairs] */
  uint32_t* yend;   /* [n_pairs] */
  uint32_t* status; /* [n_pairs] B2A_PAIR_* or NULL, same contract as b2a_results.status */
} b2a_score_results;

/* Score-only form of b2a_align_batch, for callers that rank or filter candidates and never read the path: the
 * fill keeps no traceback (stats.traceback_bytes == 0, one wave whatever the traceback budget), and K2 computes
 * row m and the last-column fix-ups, then walks only row m and column n -- the only cells whose moves change xend
 * and yend.  score, xend and yend are bit-identical to b2a_align_batch's for every pair that call reports as
 * B2A_PAIR_OK; xstart, ystart and ops are not produced.  Validation, errors, shape choice and the chunk pipeline of
 * batches >= 262,144 pairs are b2a_align_batch's.  A reference panic is seen only where that walk meets it: a pair
 * whose corrupt move lies deeper inside the matrix keeps its score with status B2A_PAIR_OK here. */
int32_t b2a_score_batch(b2a_engine* e, int32_t mode, const b2a_scoring* scoring, const b2a_pairs* pairs,
                        b2a_score_results* results, b2a_stats* stats);

/* Packed input (SURVEY 8f rank 2): the sequences as bio::data_structures::bitenc::BitEnc storage
 * (src/data_structures/bitenc.rs:50-56: 32-bit blocks, `width` bits per symbol, 32 - 32 % width usable bits per
 * block; symbol i sits at bit (i*width) % usable of block (i*width) / usable, bitenc.rs:319-338), holding the ranks
 * alphabets::RankTransform::transform yields (src/alphabets/mod.rs:220-283).  x_block / y_block are block indices
 * into `blocks`.  The packed blocks are what crosses PCIe (width 2: a quarter of the bytes); scores are those of
 * `scoring` applied to the RANKS: MatchParams by equality, `table[a*256+b]` indexed by rank. */
typedef struct b2a_packed_pairs {
  const uint32_t* blocks;   /* all BitEnc storages, concatenated */
  const uint64_t* x_block;  /* [n_pairs] first block of x */
  const uint32_t* x_len;    /* [n_pairs] symbols (BitEnc::nr_symbols) */
  const uint64_t* y_block;
  const uint32_t* y_len;
  uint64_t n_blocks;
  uint64_t n_pairs;
  uint32_t width;           /* BitEnc::new(width), 1..8 */
} b2a_packed_pairs;
int32_t b2a_align_batch_packed(b2a_engine* e, int32_t mode, const b2a_scoring* scoring,
                               const b2a_packed_pairs* pairs, b2a_results* results, b2a_stats* stats);
int32_t b2a_align_batch_banded_packed(b2a_engine* e, int32_t mode, const b2a_scoring* scoring, uint32_t k, uint32_t w,
                                      const b2a_packed_pairs* pairs, b2a_results* results, b2a_stats* stats);

/* banded::Aligner::{custom,global,semiglobal,local} (banded.rs:282,872,901,942)
 * with k-mer length k and band half-width w (banded.rs:150-180). */
int32_t b2a_align_batch_banded(b2a_engine* e, int32_t mode, const b2a_scoring* scoring,
                               uint32_t k, uint32_t w, const b2a_pairs* pairs,
                               b2a_results* results, b2a_stats* stats);

/* The banded::Aligner entry points that take the band's inputs from the caller (banded.rs:294-401, 938-975):
 *   custom_with_prehash / semiglobal_with_prehash   the k-mer hash of y only speeds the reference's match search
 *                                                   up; the matches, hence the results, are those of custom /
 *                                                   semiglobal: call b2a_align_batch_banded
 *   custom_with_matches(x, y, matches)              match_off + match_xy
 *   custom_with_expanded_matches(.., allowed_mismatches, use_lcskpp_union)
 *                                                   match_off + match_xy, allowed_mismatches (-1 = None),
 *                                                   use_lcskpp_union
 *   custom_with_match_path(x, y, matches, path)     match_off + match_xy + path_off + path_idx
 * Pair p's matches are (match_xy[2i], match_xy[2i+1]) = (xpos, ypos) for i in [match_off[p], match_off[p+1]),
 * its path the indices path_idx[path_off[p] .. path_off[p+1]) into those matches.  Where the reference panics
 * (matches not strictly ascending, a path index out of range, an empty path, positions outside the matrix) the
 * batch is refused with B2A_E_INVALID. */
typedef struct b2a_band_hints {
  const uint64_t* match_off; /* n_pairs + 1 */
  const uint32_t* match_xy;
  const uint64_t* path_off;  /* n_pairs + 1, or NULL */
  const uint32_t* path_idx;
  int32_t allowed_mismatches; /* -1: matches are used as given */
  int32_t use_lcskpp_union;
} b2a_band_hints;
int32_t b2a_align_batch_banded_hinted(b2a_engine* e, int32_t mode, const b2a_scoring* scoring,
                                      uint32_t k, uint32_t w, const b2a_pairs* pairs,
                                      const b2a_band_hints* hints, b2a_results* results, b2a_stats* stats);

/* Band::ranges of one pair of the last banded call (what banded::Aligner::visualize draws, banded.rs:1007-1030):
 * y_len + 1 half-open row ranges as (start, end) u32 pairs; an empty column is (x_len + 1, 0) (banded.rs:1065).
 * Kept on the device for the pairs of the call's last wave (every pair, unless the batch needed several waves). */
int32_t b2a_banded_band_ranges(b2a_engine* e, uint64_t pair, uint32_t* ranges, uint64_t capacity_pairs);

/* How many pairs of the last banded call K4 marked for the strip-wavefront fill (the packed-cell kernel for bands
 * whose starts and ends never decrease; the rest -- and the rare marked pair that path hands back -- ran the literal /
 * register-resident column loops of banded.rs:511-681).  A measurement aid: results do not depend on the path. */
int32_t b2a_banded_strip_pairs(b2a_engine* e, uint64_t* n_pairs);

/* Staged form of b2a_align_batch, so a caller can keep a batch resident in HBM:
 *   stage: validate, plan, host->device copy of the batch (async on the stream);
 *   run:   launch K0..K2 on the stream (async; may be called repeatedly);
 *   fetch: device->host copy of the results, stream-synchronised. */
int32_t b2a_batch_stage(b2a_engine* e, int32_t mode, const b2a_scoring* scoring,
                        const b2a_pairs* pairs);
int32_t b2a_batch_run(b2a_engine* e);
int32_t b2a_batch_fetch(b2a_engine* e, b2a_results* results, b2a_stats* stats);

/* Fixed-stride per-pair result records of the staged batch in DEVICE memory,
 * the unit that is all-gathered across GPUs (one ncclAllGather, SURVEY 8e):
 *   record = { int32 score; uint32 xstart, xend, ystart, yend, n_ops;
 *              uint32 clip_len[4]; uint8 ops[stride - 40] }.
 * Valid after b2a_batch_run until the next stage. */
int32_t b2a_batch_records(b2a_engine* e, void** dev_records, uint32_t* stride_bytes,
                          uint64_t* n_records);
/* Same records, but written into caller-provided DEVICE memory (e.g. a torch
 * tensor that is then handed to torch.distributed.all_gather_into_tensor). */
int32_t b2a_batch_records_into(b2a_engine* e, void* dev_dst, uint64_t dst_bytes,
                               uint32_t* stride_bytes);
uint32_t b2a_record_stride(uint32_t max_m, uint32_t max_n);

/* Decode host copies of gathered records into b2a_results (pure host code). */
int32_t b2a_records_decode(const void* host_records, uint32_t stride_bytes, uint64_t n_records,
                           b2a_results* results);

/* Compact form of the same results for the all-gather (what `bench.py --gpus N` and
 * rust_bio_b200/dist.py exchange): one segment per rank,
 *   { uint64 n_pairs; uint64 ops_bytes; uint8 pad[48]; }                       64 bytes
 *   int32 score[n]; uint32 xstart[n], xend[n], ystart[n], yend[n], n_ops[n]; uint32 clip_len[4n];
 *   uint8 ops[ops_bytes]                      (pair p's ops follow pair p-1's, b2a_results order)
 * i.e. 64 + 40 n + ops_bytes bytes instead of n * b2a_record_stride(): short alignments (local mode on
 * reads) travel at their real length.  b2a_batch_compact_bytes waits for the batch to finish and returns the
 * segment size; ranks agree on the largest one (a MAX all-reduce of one integer), each writes its segment
 * into a buffer of that size and a single all-gather moves them. */
int32_t b2a_batch_compact_bytes(b2a_engine* e, uint64_t* segment_bytes);
int32_t b2a_batch_compact_into(b2a_engine* e, void* dev_dst, uint64_t dst_bytes);
/* The same segment with a capacity the CALLER fixes (e.g. from the previous batch, or the bound
 * 64 + 40 n + sum(m + n + 4)): nothing here waits for the batch or reads a size back, so ranks need no size
 * agreement before the all-gather and the exchange of batch k can overlap the kernels of batch k + 1.  The header
 * is written on the device: { n_pairs, ops_bytes produced, ops_bytes kept (<= capacity), 0... }; a segment whose
 * ops did not fit is cut and says so (kept < produced) -- b2a_gathered_fetch refuses it (B2A_E_CAPACITY). */
int32_t b2a_batch_compact_fixed(b2a_engine* e, void* dev_dst, uint64_t capacity_bytes);
/* Reassembly on the rank that returns the results (SURVEY 8e: "rank 0's copy is what the shim returns"):
 * `dev_gathered` = n_segments segments of segment_bytes each, as all-gathered in DEVICE memory, in rank order.
 * Copies every field straight into `results` (host memory, pinned for speed) in that order and builds ops_off. */
int32_t b2a_gathered_fetch(b2a_engine* e, const void* dev_gathered, uint64_t segment_bytes, uint32_t n_segments,
                           b2a_results* results, uint64_t* n_pairs_total, uint64_t* d2h_bytes);
/* Decode one gathered segment (host memory) into `results` starting at pair index `pair_base` and ops offset
 * `ops_base`; returns the segment's pair count and ops bytes.  ops_off[pair_base + i] is written for every
 * pair of the segment (the caller writes the final ops_off[n_total]). */
int32_t b2a_compact_decode(const void* host_segment, uint64_t segment_bytes, uint64_t pair_base,
                           uint64_t ops_base, b2a_results* results, uint64_t* n_pairs, uint64_t* ops_bytes);

/* ---- every visible GPU from ONE process (SURVEY 8b / 8e; what a Rust caller of the shim uses on an 8 x B200 box)
 * b2a_multi_create: one engine + one stream per device (device_ids == NULL / n_devices <= 0: all visible devices)
 * and an NCCL communicator over them (ncclCommInitAll, libnccl.so.2 bound at run time).
 * b2a_multi_align_batch: Aligner::{custom,global,semiglobal,local} over a batch with HOST inputs and outputs -- the
 * pair list is split contiguously into equal shares, every device stages and runs its share side by side, ONE
 * ncclAllGather of the compact result segments reassembles the per-pair results on every device, and device 0's copy
 * is decoded into `results`.  Bit-identical to b2a_align_batch on one device.  Without libnccl the segments are
 * gathered onto device 0 with peer copies instead; b2a_multi_exchange_kind() names what is in use. */
typedef struct b2a_multi b2a_multi;
int32_t b2a_multi_create(b2a_multi** out, const int32_t* device_ids, int32_t n_devices);
int32_t b2a_multi_destroy(b2a_multi* m);
int32_t b2a_multi_device_count(const b2a_multi* m);
const char* b2a_multi_last_error(const b2a_multi* m);
const char* b2a_multi_exchange_kind(const b2a_multi* m);
int32_t b2a_multi_align_batch(b2a_multi* m, int32_t mode, const b2a_scoring* scoring, const b2a_pairs* pairs,
                              b2a_results* results, b2a_stats* stats);

/* Measurement utility for the int32-ALU roofline (SURVEY 8d): tera lane-ops/s of
 * independent add / min-max / add+max register chains over all SMs of the device. */
int32_t b2a_util_int32_peak(int32_t device_id, float* tops_add, float* tops_minmax, float* tops_mixed);

#ifdef __cplusplus
}
#endif
#endif /* B200ALIGN_H_ */

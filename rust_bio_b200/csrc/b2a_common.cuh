// Shared definitions of the B200 pairwise engine: device-side scoring, the
// per-block plan, scratch layouts and the closed-form DP boundaries.
//
// Reference being re-implemented: rust-bio 4.0.1 src/alignment/pairwise/mod.rs
//   Aligner::custom   591-922   (cell rule 729-805, fix-ups 809-843, walk 845-908)
// Nothing here is a translation of that loop nest: the fill is a row-strip
// wavefront (b2a_fill.cuh), rows 1..m-1 only; row m, the last-column fix-ups and
// the traceback walk run thread-per-pair in b2a_walk.cuh.
#pragma once
#include <stdint.h>

#if defined(__CUDACC__)
#define B2A_HD __host__ __device__ __forceinline__
#else
#define B2A_HD inline
// plain-C++ stand-ins for the CUDA vector types (CPU simulation harness only)
struct int4 { int x, y, z, w; };
struct int2 { int x, y; };
struct uint4 { unsigned x, y, z, w; };
inline int4 make_int4(int x, int y, int z, int w) { return int4{x, y, z, w}; }
#endif

namespace b2a {

#if defined(B2A_HOST_WARP) && !defined(__CUDACC__)
// Test-only (tests/sim): a 32-lane warp emulated on the host so that the not-gpu suite runs the W = 32
// instantiations too.  The lanes are 32 cooperatively scheduled contexts of one thread; a warp barrier hands
// control to the next lane (round robin, so a lane resumes after every other lane reached the barrier), and
// shuffles / votes go through an exchange buffer between two barriers.
struct HostWarp {
  long long x[32];
  void (*next_lane)(void*);  // provided by the harness: switch to the next unfinished lane
  void* harness;
  void (*other_warp)(void*);  // or null: let another emulated warp run (a lane is polling a progress word)
};
inline HostWarp* host_warp = nullptr;
inline int host_lane = 0;
inline void host_warp_sync() { host_warp->next_lane(host_warp->harness); }
inline void host_spin_yield() {
  if (host_warp && host_warp->other_warp) host_warp->other_warp(host_warp->harness);
}
template <class Pick>
inline long long host_warp_exchange(long long mine, Pick pick) {
  host_warp->x[host_lane] = mine;
  host_warp_sync();
  const long long r = pick(host_warp->x);
  host_warp_sync();
  return r;
}
#endif

constexpr int32_t MIN_SCORE = -858993459;  // mod.rs:174
// A clip penalty at or below this can never win against a real path given the
// range check in the engine (|any S| <= 2^27): treated as "dead" (SURVEY 3.2).
constexpr int32_t DEAD_CLIP = MIN_SCORE / 2;

// Traceback move codes, mod.rs:1036-1045
enum : uint32_t {
  TB_START = 0, TB_INS = 1, TB_DEL = 2, TB_SUBST = 3, TB_MATCH = 4,
  TB_XCLIP_PREFIX = 5, TB_XCLIP_SUFFIX = 6, TB_YCLIP_PREFIX = 7, TB_YCLIP_SUFFIX = 8
};

// Compressed interior traceback nibble (rows 1..m-1, columns 1..n):
//   bits 1:0  S source = the priority code the fill's packed max carries:
//             3 diagonal (Match/Subst by byte equality), 2 Ins, 1 Del,
//             0 x-prefix clip (the only other move that can win there, see DESIGN.md)
//   bit  2    I came from extension (else from S of the cell above)
//   bit  3    D came from extension (else from S of the cell to the left)
enum : uint32_t { NB_DIAG = 3, NB_INS = 2, NB_DEL = 1, NB_CLIP = 0, NB_IEXT = 4, NB_DEXT = 8 };

// Kernel specialisation flags
enum : int {
  F_TRACK_ROWS = 1,  // yclip_suffix live: per-row (Sn, Ly) arg-max over columns (mod.rs:799-802)
  F_TRACK_COLS = 2,  // xclip_suffix live: per-column (S[curr][m], Lx) arg-max over rows (mod.rs:793-796)
  F_CLIPX = 4,       // xclip_prefix and yclip_prefix live: xclip_score term (mod.rs:724-728,775-778)
  F_LUT = 8,         // substitution scores from a compact LUT in shared memory (else MatchParams)
  F_PACKTRK = 16,    // trackers as packed keys 4096*value + (4095-index): needs m,n <= 4095, |S| < 2^17
  F_RELU = 32,       // with F_CLIPX: xclip_score(j) == 0 for every column (x/y prefix clips both 0): one fused max3-relu
  // 64 is F_CLIPY of the banded strip fill (b2a_banded_strip.cuh)
  F_PACKREL = 128,   // long sequences (m or n > 4095, |S| < 2^18): the same packed keys with RELATIVE indices -- the row
                     // tracker's column inside a chunk of 2^KREL_BITS columns (flushed to the rows arena at each chunk
                     // end), the column tracker's row inside the strip (made absolute where the strip hands it on)
  F_NOTB = 256,      // score-only batch (b2a_score_batch): no interior traceback -- no nibble accumulators, no stores to
                     // the traceback arena; the boundary row, rows arena and row m-1 stay word for word the same
};
#ifndef B2A_KREL_BITS
#define B2A_KREL_BITS 12  // (a test build shortens the chunks to exercise the flushes on small inputs)
#endif
constexpr int32_t KREL_BITS = B2A_KREL_BITS, KREL_MASK = (1 << KREL_BITS) - 1;

struct DevScoring {
  int32_t gap_open, gap_extend;
  int32_t xclip_prefix, xclip_suffix, yclip_prefix, yclip_suffix;
  int32_t match_score, mismatch_score;
  int32_t alpha;  // LUT alphabet size (0 = MatchParams)
};

// One block = up to 32 pairs of the (sorted) batch; the walk kernel gives one
// lane to each pair of a block, the fill kernel gives G lanes to each pair, so a
// block is G warp-tasks of 32/G pairs.  All per-pair scratch is laid out
// [index][pair-in-block] so that a warp touching index k for its 32 pairs makes
// one contiguous access.
struct Block {
  uint32_t first;    // first sorted pair
  uint32_t npairs;   // <= 32
  uint32_t maxm, maxn;
  uint32_t uniform;  // every pair of the block has m == maxm and n == maxn
  uint32_t nstrips;  // row strips of G*R rows covering rows 1..maxm-1
  uint32_t xwords;   // staged 32-bit words per x (multiple of 4; 16-byte TMA granules)
  uint32_t ywords;
  uint32_t K;        // 8-column traceback groups per strip: ceil((maxn + G - 1) / 8)
  uint32_t rows_pad; // row slots in the rows arena: nstrips*G*R + 2
  uint64_t seq_off;  // bytes into the staged-sequence arena (x tasks, then y tasks)
  uint64_t bnd_off;  // bytes into the boundary arena: (maxn+1) * 32 * 16
  uint64_t rows_off; // bytes into the rows arena: 5 arrays of rows_pad*32 int32
  uint64_t rowm_off; // bytes into the row-m arena: (maxn+1)*32 bytes
  uint64_t tb_off;   // bytes into the traceback arena: G * nstrips * K * TBW * 512
  uint64_t ops_off;  // bytes into the ops scratch: 32 * (maxm+maxn+4)
  uint64_t strip_task_base;  // strip-pipelined fill (G == 32): tasks (pair, strip) of earlier blocks of the wave
};

// rows arena sub-arrays (each rows_pad*32 int32, index [row][pair])
enum { ROWS_SN = 0, ROWS_LY = 1, ROWS_SL = 2, ROWS_IL = 3, ROWS_NL = 4, ROWS_ARRAYS = 5 };

B2A_HD int32_t imax(int32_t a, int32_t b) { return a > b ? a : b; }

// ---- closed-form boundaries (SURVEY Appendix A; reference mod.rs:597-717) ----

// I(i,0), i >= 1 (mod.rs:625-639)
B2A_HD int32_t col0_I(const DevScoring& sc, int32_t i) {
  if (i == 1) return sc.gap_open;
  return imax(sc.gap_open + sc.gap_extend * (i - 1), sc.xclip_prefix + sc.gap_open);
}
// i_bits(i,0), i >= 1
B2A_HD uint32_t col0_ibits(const DevScoring& sc, int32_t i) {
  if (i == 1) return TB_START;
  return (sc.gap_open + sc.gap_extend * (i - 1) > sc.xclip_prefix + sc.gap_open) ? TB_INS
                                                                                   : TB_XCLIP_PREFIX;
}
// S(i,0) for 1 <= i < m (mod.rs:641-655 with S starting at MIN_SCORE)
B2A_HD int32_t col0_S(const DevScoring& sc, int32_t i) {
  return imax(col0_I(sc, i), sc.xclip_prefix);
}
B2A_HD uint32_t col0_sbits(const DevScoring& sc, int32_t i) {
  return sc.xclip_prefix > col0_I(sc, i) ? TB_XCLIP_PREFIX : TB_INS;
}
// D(0,j), j >= 1 (mod.rs:683-697)
B2A_HD int32_t row0_D(const DevScoring& sc, int32_t j) {
  if (j == 1) return sc.gap_open;
  return imax(sc.gap_open + sc.gap_extend * (j - 1), sc.yclip_prefix + sc.gap_open);
}
B2A_HD uint32_t row0_dbits(const DevScoring& sc, int32_t j) {
  if (j == 1) return TB_START;
  return (sc.gap_open + sc.gap_extend * (j - 1) > sc.yclip_prefix + sc.gap_open) ? TB_DEL
                                                                                   : TB_YCLIP_PREFIX;
}
// S(0,j), j >= 1, including the j == n suffix-clip override (mod.rs:698-714).
// Sn[0] stays at yclip_suffix for the whole fill because S(0,j) <= 0 (mod.rs:711).
B2A_HD int32_t row0_S(const DevScoring& sc, int32_t j, int32_t n) {
  int32_t s = imax(row0_D(sc, j), sc.yclip_prefix);
  if (j == n && sc.yclip_suffix > s) s = sc.yclip_suffix;
  return s;
}
B2A_HD uint32_t row0_sbits(const DevScoring& sc, int32_t j, int32_t n) {
  if (j == 0) return TB_START;
  const int32_t d = row0_D(sc, j);
  uint32_t b = d > sc.yclip_prefix ? TB_DEL : TB_YCLIP_PREFIX;
  if (j == n && sc.yclip_suffix > imax(d, sc.yclip_prefix)) b = TB_YCLIP_SUFFIX;
  return b;
}
// xclip_score of column j (mod.rs:724-728)
B2A_HD int32_t xclip_score(const DevScoring& sc, int32_t j) {
  return sc.xclip_prefix + imax(sc.yclip_prefix, sc.gap_open + sc.gap_extend * (j - 1));
}

// Boundary-row index of (column j, pair pi) inside a block.  Fills with several pairs per warp (G < 32)
// want [column][pair] (the warp's pairs touch one line per column); the warp-per-pair fill (G == 32)
// reads/writes one pair's row column after column from a single lane, so [pair][column] keeps those
// accesses inside cache lines (measured on C5: 408 -> 325 ms; the same layout for G = 8 cost C3 8 %).
B2A_HD int64_t bnd_index(int32_t G, int32_t j, int32_t pi, int32_t maxn) {
  return G < 32 ? (int64_t)j * 32 + pi : (int64_t)pi * (maxn + 1) + j;
}

// K1's scaled LUT: alpha real rows of alpha entries, then one poison row (the substitution "score" gap_open for
// every y symbol, i.e. the entry 4*go + 3 - (4*go + 1) = 2) that the padded rows of a masked strip read
#if defined(__CUDACC__)
__host__ __device__
#endif
constexpr int lut_entries(int alpha) { return (alpha + 1) * alpha; }
#if defined(__CUDACC__)
__host__ __device__
#endif
constexpr uint32_t lut_smem_bytes(int alpha) { return ((uint32_t)lut_entries(alpha) * 4u + 127u) & ~127u; }
constexpr int32_t LUT_POISON = 2;

// Warps per CTA of the K1 fill kernel (a build knob for the 8x20 shape; registers are allocated to a CTA in
// units of four warps, so 3-warp CTAs do not buy a ninth resident warp at 224 registers).
#ifndef B2A_W_8_20
#define B2A_W_8_20 4
#endif
#if defined(__CUDACC__)
__host__ __device__
#endif
constexpr int fill_warps_of(int G, int R) { return (G == 8 && R == 20) ? B2A_W_8_20 : 4; }
// strips whose capture row is dispatched at compile time (see column_step): the shapes that run small batches
#if defined(__CUDACC__)
__host__ __device__
#endif
constexpr bool cap_dispatch_of(int G) { return G == 8; }

// Traceback words per lane per 8-column group: rows are grouped by four so the
// fill stores whole 128-bit vectors.
#if defined(__CUDACC__)
__host__ __device__
#endif
constexpr int tbw_of(int R) { return (R + 3) / 4; }

}  // namespace b2a

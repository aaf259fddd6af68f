// K1: DP fill of rows 1..m-1 as a row-strip wavefront.
//
// What it computes (reference rust-bio 4.0.1 src/alignment/pairwise/mod.rs):
//   the per-cell rule of Aligner::custom, mod.rs:729-805, for rows i < m:
//     M = S(i-1,j-1) + score          733
//     I = max(I(i-1,j)+ge, S(i-1,j)+go), ties -> open      735-744
//     D = max(D(i,j-1)+ge, S(i,j-1)+go), ties -> open      746-755
//     S = first strict maximum in the order M, I, D, xclip_score   757-778
//       (for i < m the running value starts at MIN_SCORE and the y-prefix clip
//        can never beat I -- DESIGN.md "dead terms" -- so S has 4 sources)
//     column tracker (S[curr][m], Lx[j]) and row tracker (Sn[i], Ly[i])  793-802
// How: G lanes own one pair; lane l owns R consecutive rows held in registers
// (S and D of the previous column, row trackers, traceback accumulators); at
// step t lane l is at column t-l+1 (anti-diagonal wavefront), handing
// (S, I, column tracker) of its bottom row to lane l+1 by warp shuffle.  Rows
// beyond G*R are done in further strips; the strip boundary row lives in HBM
// ([column][pair] so a warp's access is one line) and is also what the walk
// kernel needs to finish row m.  Traceback is 4 bits per cell, eight columns
// per 32-bit register, flushed with 128-bit stores that are contiguous across
// the warp.  Sequences arrive in shared memory by cp.async.bulk (TMA bulk copy)
// completing on an mbarrier; substitution scores come from MatchParams
// compare/select or from a compact LUT in shared memory.
#pragma once
#include "b2a_common.cuh"

namespace b2a {

struct FillParams {
  const Block* blocks;
  uint32_t nblocks;
  const uint32_t* pm;  // [sorted pair] m
  const uint32_t* pn;  // [sorted pair] n
  const uint8_t* seq;  // staged sequences
  uint8_t* bnd;
  uint8_t* rows;
  uint8_t* tb;
  const int32_t* lut;  // scaled LUT 4*score + 3 - (4*gap_open + 1), alpha*alpha (global) or null
  uint32_t* task_counter;
  uint32_t smem_seq_bytes;  // per-warp staging bytes
  int32_t one;              // must be 1 (opaque to the compiler, see fmad())
  int32_t ge4;              // must be 4 * sc.gap_extend
  uint32_t* progress;       // strip-pipelined mode (G == 32): columns published per (pair, strip) task, else null
  uint32_t n_strip_tasks;   // strip-pipelined mode: number of (pair, strip) tasks of this launch
  uint32_t task_limit;      // 0: persistent (a warp pulls tasks until none is left); k: a warp retires after k tasks, so
                            // CTAs turn over and a higher-priority kernel's CTAs get onto the SMs (chunk pipeline)
  DevScoring sc;
};

// Per-lane view of one warp-task (32/G pairs of one block).
template <int G>
struct LaneCtx {
  DevScoring sc;
  const int32_t* lut;    // LUT in shared memory (device) / host memory (sim)
  const uint32_t* xs;    // staged x words of the task: [w][P]
  const uint32_t* ys;    // staged y words of the task: [w][P]
  int32_t m, n;          // this lane's pair
  int32_t maxn;          // block maximum (loop bound shared by the warp)
  int32_t maxm;          // block maximum of m (uniform blocks: every valid pair's m)
  int32_t g;             // pair slot inside the task (lane / G)
  int32_t l;             // lane inside the group (lane % G)
  int32_t lane;          // 0..31
  int32_t pi;            // pair index inside the block
  int32_t nstrips;
  int32_t K;
  int32_t rows_pad;
  bool uniform;
  int4* bnd;             // block base, [column][32]
  int32_t* rows;         // block base, ROWS_ARRAYS arrays of [rows_pad][32]
  uint4* tb;             // task base: [strip][k][q][32]
  uint32_t lut_base;     // device: shared-space byte address of the LUT; host sim: 0
  uint32_t* prog_mine;   // strip-pipelined: where this strip publishes its boundary progress (else null)
  uint32_t* prog_prev;   // strip-pipelined: progress of the strip above (null for strip 0)
  int32_t only_strip;    // strip-pipelined: the one strip this task fills (-1: all strips in order)
  int32_t one;           // an opaque 1 (kernel parameter): lets adds be issued as IMAD on the FMA pipe
  int32_t ge4;           // 4 * gap_extend, opaque as well (kept out of constant folding)
};

#if defined(__CUDA_ARCH__)
#define B2A_SHFL_UP(v, G) __shfl_up_sync(0xffffffffu, (v), 1, (G))
#elif defined(B2A_HOST_WARP) && !defined(__CUDACC__)
// tests/sim: the value of the lane below inside a group of G lanes (own value for the group's first lane)
inline int32_t host_shfl_up_group(int32_t v, int G) {
  if (!host_warp) return v;
  const int me = host_lane;
  return (int32_t)host_warp_exchange(v, [&](const long long* x) { return (me % G) ? x[me - 1] : x[me]; });
}
#define B2A_SHFL_UP(v, G) host_shfl_up_group((v), (G))
#define B2A_SPIN_YIELD() host_spin_yield()
#else
#define B2A_SHFL_UP(v, G) (v)
#endif
#ifndef B2A_SPIN_YIELD
#define B2A_SPIN_YIELD() ((void)0)
#endif

// ---- scaled/packed score domain of the fill ------------------------------------------------
// Inside K1 every score is carried as 4*value + a 2-bit priority code in the low bits:
//   S4 = 4*S (clean), M4 = 4*M + 3, I4 = 4*I + 2, D4 = 4*D + 1, X4 = 4*xclip_score + 0.
// One 3-way integer max of (M4, I4, D4) [then max with X4] yields the new S *and* which source won,
// with exactly the reference's tie order M > I > D > x-prefix-clip (mod.rs:757-778: each later
// candidate must be strictly greater).  The I/D "came from extension" flags are min(I4 - open, 4):
// 0 when the open candidate won or tied (mod.rs:738-744, 749-755), 4 otherwise.
// The engine only uses K1 when every real score fits in +-2^27, so 4x fits in i32.
constexpr int32_t NEG4 = -(1 << 30);  // "-infinity" in the scaled domain

B2A_HD int32_t max3(int32_t a, int32_t b, int32_t c) {
#if defined(__CUDA_ARCH__)
  return __vimax3_s32(a, b, c);
#else
  return imax(a, imax(b, c));
#endif
}
B2A_HD int32_t max3_relu(int32_t a, int32_t b, int32_t c) {  // max(a, b, c, 0): one VIMNMX3.RELU
#if defined(__CUDA_ARCH__)
  return __vimax3_s32_relu(a, b, c);
#else
  return imax(imax(a, imax(b, c)), 0);
#endif
}
B2A_HD int32_t imin(int32_t a, int32_t b) { return a < b ? a : b; }
// fused add+max / add+min (DPX: one VIADDMNMX on the ALU pipe)
B2A_HD int32_t addmax(int32_t a, int32_t b, int32_t c) {
#if defined(__CUDA_ARCH__)
  return __viaddmax_s32(a, b, c);
#else
  return imax(a + b, c);
#endif
}
B2A_HD int32_t addmin(int32_t a, int32_t b, int32_t c) {
#if defined(__CUDA_ARCH__)
  return __viaddmin_s32(a, b, c);
#else
  return imin(a + b, c);
#endif
}
// 4*v, except that dead (MIN_SCORE-like) penalties map to NEG4 instead of overflowing
B2A_HD int32_t scale4(int32_t v) { return v <= DEAD_CLIP ? NEG4 : 4 * v; }

// The fill is bound by the integer ALU pipe (VIMNMX/LOP3/...), while the FMA pipe (IMAD) idles.
// Plain adds are therefore written as a*k+b with k an opaque kernel parameter, which ptxas must
// issue as IMAD: the max/min/select work stays on the ALU pipe, the additions move to the FMA pipe.
B2A_HD int32_t fmad(int32_t a, int32_t k, int32_t b) {
#if defined(__CUDA_ARCH__)
  int32_t d;
  asm("mad.lo.s32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(k), "r"(b));
  return d;
#else
  return a * k + b;
#endif
}
B2A_HD int32_t lut_at(const void* host_base, uint32_t byte_addr) {
#if defined(__CUDA_ARCH__)
  int32_t v;
  asm("ld.shared.s32 %0, [%1];" : "=r"(v) : "r"(byte_addr));
  return v;
#else
  return *reinterpret_cast<const int32_t*>(reinterpret_cast<const char*>(host_base) + byte_addr);
#endif
}

// strip-pipelined mode: strips of one pair run concurrently in different warps; the boundary row is
// handed over through HBM/L2 with a per-strip progress word (release: fence + volatile store,
// acquire: volatile poll + fence, boundary loads bypass L1).
B2A_HD uint32_t ld_progress(const uint32_t* p) {
#if defined(__CUDA_ARCH__)
  return *reinterpret_cast<const volatile uint32_t*>(p);
#else
  return *p;
#endif
}
B2A_HD int4 ld_boundary(const int4* p, bool bypass_l1) {
#if defined(__CUDA_ARCH__)
  return bypass_l1 ? __ldcg(p) : *p;
#else
  (void)bypass_l1;
  return *p;
#endif
}
B2A_HD void fence_device() {
#if defined(__CUDA_ARCH__)
  __threadfence();
#endif
}

// packed arg-max keys (F_PACKTRK): 4096*value + (4095 - index): max() keeps the first index on ties
constexpr int32_t KEY_NONE = (int32_t)0x80000000;

// MASKED strips (rows beyond m-1 inside the strip):
//  * with a LUT the padded rows read a poison LUT row (score = gap_open for every y symbol, see lut_entries()):
//    by induction over the columns S(pad_k, j) <= S(pad_k-1, j) <= ... <= S(m-1, j) and D likewise
//    (M(pad) = S(above, j-1) + go <= D(above, j) <= S(above, j); I(pad) <= S(above); D(pad, j) from the
//    smaller S/D of column j-1; column 0 is non-increasing in i), and they sit at higher row indices, so they can
//    never win the column tracker's first-maximum: no per-row mask is needed there;
//  * the writer needs (S, I) of row m-1 = the partial lane's row rv-1.  CAPQ >= 0: uniform block, that row is
//    known to lie in row-quad CAPQ (compile time), so only four rows carry the capture compare; CAPQ == R/4: no
//    lane of the strip is partial; CAPQ == -1: ragged block, every row compares.
template <int G, int R, int FLAGS, bool MASKED, bool LAST, int CAPQ>
B2A_HD void column_step(const LaneCtx<G>& c, const int32_t j, const int32_t tstep, const int32_t q, const int32_t rowbase,
                        const int32_t rv, int32_t (&Sp)[R], int32_t (&Dp)[R], int32_t (&SnR)[R],
                        int32_t (&LyR)[R], uint32_t (&tbacc)[R], const int32_t (&xc)[R],
                        int32_t sdiag, int32_t& sup, int32_t& iup, int32_t& Tv, int32_t& Ti,
                        int32_t& cap_s, int32_t& cap_i) {
  constexpr bool TR = (FLAGS & F_TRACK_ROWS) != 0;
  constexpr bool TC = (FLAGS & F_TRACK_COLS) != 0;
  constexpr bool CX = (FLAGS & F_CLIPX) != 0;
  constexpr bool LUT = (FLAGS & F_LUT) != 0;
  constexpr bool PR = (FLAGS & F_PACKREL) != 0;  // packed keys with relative indices (see F_PACKREL): here like PK,
  constexpr bool PK = (FLAGS & F_PACKTRK) != 0 || PR;  // the caller passes chunk- / strip-relative cj and rowbase
  constexpr bool RELU = (FLAGS & F_RELU) != 0;
  constexpr bool NOTB = (FLAGS & F_NOTB) != 0;
  constexpr bool TMASK = MASKED && !LUT;  // the column tracker has to skip the padded rows explicitly
  // S travels between cells as "S + open": So_d = S4 + go4d feeds the D chain of the next column and (as
  // the diagonal input) M of the next column, whose LUT/compare scores are pre-biased by -go4d; the I chain
  // of the row below wants go4i = go4d + 1.  One IMAD per consumer instead of two, and the chains
  // themselves are single fused add-max instructions (ge4 is an opaque kernel parameter for that reason).
  const int32_t go4i = 4 * c.sc.gap_open + 2, go4d = 4 * c.sc.gap_open + 1, ge4 = c.ge4;
  const int32_t ma4 = 4 * c.sc.match_score + 3 - go4d, mi4 = 4 * c.sc.mismatch_score + 3 - go4d;
  const int32_t x4 = CX ? scale4(xclip_score(c.sc, j)) : 0;
  const int32_t xs4 = scale4(c.sc.xclip_suffix), ys4 = scale4(c.sc.yclip_suffix);
  // packed row-tracker index field: the column, or (PR) the STEP inside its chunk of 2^KREL_BITS steps -- the lanes
  // of a pair sit at different columns in one step, but they all reach a chunk's end together, so the flush of the
  // row trackers to the rows arena happens between two runs of the column loop, not inside it
  const int32_t cj = 4095 - (PR ? (tstep & KREL_MASK) : j);
  const int32_t one = c.one, k2 = one + one, k16 = k2 * 8, k1024 = k16 * 64;
  const int32_t q4 = q * 4;
  int32_t Tl = KEY_NONE;        // packed column tracker of this lane's rows (local row index)
  int32_t key_even = KEY_NONE;
  int32_t sdo = fmad(sdiag, one, go4d);  // diagonal S, open-biased
  int32_t iop = fmad(sup, one, go4i);    // S of the row above + I open
  int32_t s4 = sup;
#pragma unroll
  for (int r = 0; r < R; ++r) {
    int32_t sub4;
    if (LUT) {
      sub4 = lut_at(c.lut, (uint32_t)fmad(q4, one, xc[r]));  // 4*score + 3 - go4d
    } else {
      sub4 = (xc[r] == q) ? ma4 : mi4;
    }
    const int32_t m4 = fmad(sdo, one, sub4);
    const int32_t i4 = addmax(iup, ge4, iop);
    const int32_t dop = Sp[r];  // S4 of this row in the previous column + go4d
    const int32_t d4 = addmax(Dp[r], ge4, dop);
    int32_t sP;
    if (CX && RELU) {
      sP = max3_relu(m4, i4, d4);  // x4 == 0 (code 0 in the low bits) for every column
    } else {
      sP = max3(m4, i4, d4);
      if (CX) sP = imax(sP, x4);
    }
    s4 = sP & ~3;
    // nibble = code | iext << 2 | dext << 3 = (sP - s4) + min(i4 - iop, 4) + 2 * min(d4 - dop, 4),
    // accumulated as tbacc*16 + nibble (the oldest nibble falls off the top); score-only: column n's nibble only
    int32_t nib = 0;
    if (!NOTB || LAST) {
      const int32_t fi = addmin(i4, -iop, 4), fd = addmin(d4, -dop, 4);
      nib = fmad(fd, k2, fi) + sP - s4;
      if (!NOTB) tbacc[r] = (uint32_t)(fmad((int32_t)tbacc[r], k16, fmad(fd, k2, fi)) + sP - s4);
    }
    if (TC) {
      if (PK) {
        if (TMASK) {
          if (r < rv) Tl = imax(Tl, fmad(s4, k1024, 4095 - r));
        } else {  // two rows per 3-input max
          const int32_t key = fmad(s4, k1024, 4095 - r);
          if (r & 1) Tl = max3(Tl, key_even, key);
          else key_even = key;
        }
      } else {
        const int32_t v = s4 + xs4;
        if ((!TMASK || r < rv) && v > Tv) {
          Tv = v;
          Ti = rowbase + 1 + r;
        }
      }
    }
    if (TR) {
      if (PK) {
        SnR[r] = imax(SnR[r], fmad(s4, k1024, cj));
      } else {
        const int32_t v = s4 + ys4;
        if (v > SnR[r]) {
          SnR[r] = v;
          LyR[r] = j;
        }
      }
    }
    if (LAST) {
      const int32_t slot = (rowbase + 1 + r) * 32 + c.pi;
      c.rows[ROWS_SL * c.rows_pad * 32 + slot] = s4 >> 2;
      c.rows[ROWS_IL * c.rows_pad * 32 + slot] = i4 >> 2;
      c.rows[ROWS_NL * c.rows_pad * 32 + slot] = nib;
    }
    if (MASKED && (CAPQ < 0 || (r >> 2) == CAPQ)) {
      if (r == rv - 1) {
        cap_s = s4;
        cap_i = i4;
      }
    }
    sdo = dop;
    Sp[r] = fmad(s4, one, go4d);
    iop = fmad(s4, one, go4i);
    Dp[r] = d4;
    iup = i4;
  }
  sup = s4;
  if (TC && PK) {
    // local row index -> global (PR: inside the strip): (4095 - r) - (rowbase + 1) = 4095 - i ; Tv carries the packed key
    if (Tl != KEY_NONE) Tv = imax(Tv, Tl - ((PR ? c.l * R : rowbase) + 1));
  }
}

// One strip (rows s*G*R+1 .. (s+1)*G*R) of one lane's pair.
template <int G, int R, int FLAGS, bool MASKED, int CAPQ>
B2A_HD void run_strip(const LaneCtx<G>& c, const int32_t s) {
  constexpr bool TR = (FLAGS & F_TRACK_ROWS) != 0;
  constexpr bool TC = (FLAGS & F_TRACK_COLS) != 0;
  constexpr bool LUT = (FLAGS & F_LUT) != 0;
  constexpr bool PR = (FLAGS & F_PACKREL) != 0;
  constexpr bool PK = (FLAGS & F_PACKTRK) != 0 || PR;  // packed keys in the lanes (PR: relative indices)
  constexpr bool NOTB = (FLAGS & F_NOTB) != 0;
  constexpr int P = 32 / G;
  constexpr int TBW = tbw_of(R);
  const int32_t m = c.m, n = c.n;
  const int32_t rowbase = s * (G * R) + c.l * R;  // row above this lane's first row
  // valid rows of this lane: rows <= m-1
  int32_t rv = m - 1 - rowbase;
  rv = rv < 0 ? 0 : (rv > R ? R : rv);
  const int32_t ys = c.sc.yclip_suffix;

  int32_t Sp[R], Dp[R], SnR[R], LyR[R], xc[R];
  uint32_t tbacc[R];
  // x symbols of my rows: rows rowbase+1.. are x[rowbase..], R % 4 == 0 so word aligned
#pragma unroll
  for (int w = 0; w < R / 4; ++w) {
    const uint32_t xw = c.xs[(rowbase / 4 + w) * P + c.g];
#pragma unroll
    for (int b = 0; b < 4; ++b) {
      const int32_t sym = (int32_t)((xw >> (8 * b)) & 0xffu);
      // LUT mode: byte address of the symbol's LUT row (shared-space on the device)
      xc[w * 4 + b] = LUT ? (int32_t)(c.lut_base + (uint32_t)(sym * c.sc.alpha * 4)) : sym;
      // padded rows: the poison row that follows the alpha real rows of the LUT
      if (MASKED && LUT && w * 4 + b >= rv) xc[w * 4 + b] = (int32_t)(c.lut_base + (uint32_t)(c.sc.alpha * c.sc.alpha * 4));
    }
  }
#pragma unroll
  for (int r = 0; r < R; ++r) {
    const int32_t i = rowbase + 1 + r;
    const int32_t s0 = col0_S(c.sc, i);
    Sp[r] = 4 * s0 + (4 * c.sc.gap_open + 1);  // open-biased, see column_step
    Dp[r] = NEG4;
    tbacc[r] = 0;
    LyR[r] = 0;
    if (TR) {  // mod.rs:667-670 (column 0 is index 0)
      if (PK) {
        SnR[r] = s0 * 4096 + 4095;
      } else {
        const int32_t v = s0 + ys;
        SnR[r] = (ys > DEAD_CLIP && v > MIN_SCORE) ? 4 * v : NEG4;
      }
    } else {
      SnR[r] = 0;
    }
  }
  // S of the row above my first row, in column 0 (the first diagonal input), scaled
  int32_t sup_prev = rowbase == 0 ? 0 : 4 * col0_S(c.sc, rowbase);
  // values arriving from above for my next column (scaled domain; tracker as key or as (4*T, index))
  const int32_t t_none = PK ? KEY_NONE : NEG4;
  int32_t in_s = 0, in_i = NEG4, in_tv = t_none, in_ti = m;
  // PR: the column tracker of the strips above (value 4*(S + xs), absolute row), carried beside this strip's packed
  // key down the lanes; where the strip hands the boundary on the two are merged (the strip above wins ties: it holds
  // the lower rows)
  int32_t up_tv = NEG4, up_ti = m;
  const int32_t xs4_pr = scale4(c.sc.xclip_suffix);
  // PR: the row trackers are flushed to the rows arena (seeded with column 0's value, below) at the end of every chunk
  // of steps and kept only if strictly better, so the earlier column wins ties
  auto flush_rows = [&](const int32_t chunk, int32_t (&SnRr)[R]) {
#pragma unroll
    for (int r = 0; r < R; ++r) {
      const int32_t slot = (rowbase + 1 + r) * 32 + c.pi;
      if (SnRr[r] != KEY_NONE) {
        const int32_t sn = (SnRr[r] >> 12) + ys;
        const int32_t step = (chunk << KREL_BITS) + (4095 - (SnRr[r] & 4095));
        if (sn > c.rows[ROWS_SN * c.rows_pad * 32 + slot]) {
          c.rows[ROWS_SN * c.rows_pad * 32 + slot] = sn;
          c.rows[ROWS_LY * c.rows_pad * 32 + slot] = step - c.l + 1;  // the lane's column at that step
        }
      }
      SnRr[r] = KEY_NONE;
    }
  };
  int4 pre = make_int4(0, 0, 0, 0);
  const bool top_from_mem = (c.l == 0) && (s > 0);
  const bool top_from_row0 = (c.l == 0) && (s == 0);
  // strip-pipelined: number of columns the strip above has published so far
  uint32_t avail = 0;
  const bool piped = c.prog_mine != nullptr;
  auto wait_col = [&](int32_t col) {
    if (piped && c.prog_prev && (int32_t)avail < col) {
      do {
        avail = ld_progress(c.prog_prev);
        B2A_SPIN_YIELD();  // nothing on the device (tests/sim: let the producer's emulated warp run)
      } while ((int32_t)avail < col);
      fence_device();
    }
  };
  const bool top_valid = top_from_mem && rv >= 1;  // a strip without valid rows needs no boundary (ragged blocks)
  if (top_valid && n >= 1) {
    wait_col(1);
    pre = ld_boundary(&c.bnd[bnd_index(G, 1, c.pi, c.maxn)], piped);
  }
  const bool writer =
      MASKED ? (rv >= 1 && (c.l == G - 1 || rowbase + R >= m - 1)) : (c.l == G - 1);
  int32_t cap_s = 0, cap_i = 0;
  uint32_t yw = 0;
  uint4* tbs = c.tb + (size_t)s * c.K * TBW * 32;
  const int32_t nsteps = c.K * 8;

  if (PR && TR) {
#pragma unroll
    for (int r = 0; r < R; ++r) {
      const int32_t slot = (rowbase + 1 + r) * 32 + c.pi;
      c.rows[ROWS_SN * c.rows_pad * 32 + slot] = col0_S(c.sc, rowbase + 1 + r) + ys;  // column 0 (mod.rs:667-670)
      c.rows[ROWS_LY * c.rows_pad * 32 + slot] = 0;
      SnR[r] = KEY_NONE;
    }
  }
  for (int32_t t0 = 0; t0 < nsteps; t0 += (PR ? (1 << KREL_BITS) : nsteps)) {
  const int32_t t1 = PR ? ((t0 + (1 << KREL_BITS) < nsteps) ? t0 + (1 << KREL_BITS) : nsteps) : nsteps;
  for (int32_t t = t0; t < t1; ++t) {
    const int32_t j = t - c.l + 1;
    const bool active = (j >= 1) && (j <= n);
    if (active) {
      // y symbol of column j
      int32_t q;
      if (G == 1) {
        if ((t & 3) == 0) yw = c.ys[(t >> 2) * P + c.g];
        q = (int32_t)(yw & 0xffu);
        yw >>= 8;
      } else {
        const int32_t jb = j - 1;
        q = (int32_t)((c.ys[(jb >> 2) * P + c.g] >> (8 * (jb & 3))) & 0xffu);
      }
      if (top_from_row0) {
        in_s = 4 * row0_S(c.sc, j, n);
        in_i = NEG4;
        in_tv = t_none;
        in_ti = m;
        if (PR) {
          up_tv = NEG4;
          up_ti = m;
        }
      } else if (top_from_mem) {  // the boundary row is kept in the fill's own scaled domain
        in_s = pre.x;
        in_i = pre.y;
        if (TC) {
          if (PR) {  // unpacked (value, row) of the strips above; this strip's own key starts empty
            up_tv = pre.z;
            up_ti = pre.w;
            in_tv = KEY_NONE;
          } else {
            in_tv = pre.z;
            in_ti = pre.w;
          }
        }
        if (j < n && top_valid) {  // prefetch next column's boundary
          wait_col(j + 1);
          pre = ld_boundary(&c.bnd[bnd_index(G, j + 1, c.pi, c.maxn)], piped);
        }
      }
      int32_t sup = in_s, iup = in_i, Tv = in_tv, Ti = in_ti;
      if (j == n) {
        column_step<G, R, FLAGS, MASKED, true, CAPQ>(c, j, t, q, rowbase, rv, Sp, Dp, SnR, LyR, tbacc, xc,
                                               sup_prev, sup, iup, Tv, Ti, cap_s, cap_i);
      } else {
        column_step<G, R, FLAGS, MASKED, false, CAPQ>(c, j, t, q, rowbase, rv, Sp, Dp, SnR, LyR, tbacc, xc,
                                                sup_prev, sup, iup, Tv, Ti, cap_s, cap_i);
      }
      sup_prev = in_s;
      if (writer) {
        int4 o;  // decoded by decode_boundary() in b2a_walk.cuh
        o.x = (MASKED && rv < R) ? cap_s : sup;  // a full lane's row m-1 is its bottom row
        o.y = (MASKED && rv < R) ? cap_i : iup;
        o.z = TC ? Tv : t_none;
        o.w = TC ? Ti : m;
        if (PR) {  // the boundary row leaves the strip unpacked, as K2 and the strip below read it
          o.z = NEG4;
          o.w = m;
          if (TC) {
            o.z = up_tv;
            o.w = up_ti;
            if (Tv != KEY_NONE) {
              const int32_t loc_v = ((Tv >> 12) << 2) + xs4_pr;  // 4 * (S + xs)
              if (loc_v > up_tv) {
                o.z = loc_v;
                o.w = s * (G * R) + (4095 - (Tv & 4095));
              }
            }
          }
        }
        c.bnd[bnd_index(G, j, c.pi, c.maxn)] = o;
        if (piped && ((j & 15) == 0 || j == n)) {  // publish (release) every 16 columns and at the end
          fence_device();
          *reinterpret_cast<volatile uint32_t*>(c.prog_mine) = (uint32_t)j;
          B2A_SPIN_YIELD();  // nothing on the device (tests/sim: the consumer's emulated warp gets a turn)
        }
      }
      in_s = sup;
      in_i = iup;
      in_tv = Tv;
      in_ti = Ti;
    } else if (!NOTB) {
#pragma unroll
      for (int r = 0; r < R; ++r) tbacc[r] <<= 4;
    }
    if (G > 1) {  // hand my bottom row to the lane below (it is one column behind me)
      in_s = B2A_SHFL_UP(in_s, G);
      in_i = B2A_SHFL_UP(in_i, G);
      if (TC) {
        in_tv = B2A_SHFL_UP(in_tv, G);
        if (!PK) in_ti = B2A_SHFL_UP(in_ti, G);
        if (PR) {
          up_tv = B2A_SHFL_UP(up_tv, G);
          up_ti = B2A_SHFL_UP(up_ti, G);
        }
      }
    }
    if (!NOTB && (t & 7) == 7) {
      uint4* dst = tbs + (size_t)(t >> 3) * TBW * 32 + c.lane;
#pragma unroll
      for (int qd = 0; qd < TBW; ++qd) {
        uint4 v;
        v.x = tbacc[qd * 4 + 0];
        v.y = (qd * 4 + 1 < R) ? tbacc[qd * 4 + 1] : 0u;
        v.z = (qd * 4 + 2 < R) ? tbacc[qd * 4 + 2] : 0u;
        v.w = (qd * 4 + 3 < R) ? tbacc[qd * 4 + 3] : 0u;
        dst[qd * 32] = v;
      }
    }
  }
  if (PR && TR) flush_rows(t0 >> KREL_BITS, SnR);
  }  // chunks of steps
  if (TR && !PR) {
#pragma unroll
    for (int r = 0; r < R; ++r) {
      const int32_t slot = (rowbase + 1 + r) * 32 + c.pi;
      int32_t sn, ly;
      if (PK) {
        sn = (SnR[r] >> 12) + ys;
        ly = 4095 - (SnR[r] & 4095);
      } else {
        sn = (SnR[r] <= NEG4 / 2) ? MIN_SCORE : (SnR[r] >> 2);
        ly = LyR[r];
      }
      c.rows[ROWS_SN * c.rows_pad * 32 + slot] = sn;
      c.rows[ROWS_LY * c.rows_pad * 32 + slot] = ly;
    }
  }
}

template <int G, int R, int FLAGS>
B2A_HD void fill_lane(const LaneCtx<G>& c) {
  const int32_t s_lo = c.only_strip >= 0 ? c.only_strip : 0;
  const int32_t s_hi = c.only_strip >= 0 ? c.only_strip + 1 : c.nstrips;
  for (int32_t s = s_lo; s < s_hi; ++s) {
    // a strip is "full" when every lane of every pair of the task owns R valid rows
    // decided from the block maximum so that the whole warp takes the same branch (the padding lanes of a
    // last, partly filled task have m = 0 and simply never become active)
    const bool full = c.uniform && ((s + 1) * (G * R) <= c.maxm - 1);
    if (full) {
      run_strip<G, R, FLAGS, false, -1>(c, s);
    } else if (cap_dispatch_of(G) && c.uniform) {
      // uniform block: the one partial lane of the strip (if any) has the same valid-row count for every pair
      const int32_t left = c.maxm - 1 - s * (G * R);  // valid rows from the strip's first row on
      const int32_t part = (left > 0 && left < G * R) ? left % R : 0;
      switch (part ? (part - 1) >> 2 : R / 4) {
        case 0: run_strip<G, R, FLAGS, true, 0>(c, s); break;
        case 1: run_strip<G, R, FLAGS, true, (1 <= R / 4 ? 1 : -1)>(c, s); break;
        case 2: run_strip<G, R, FLAGS, true, (2 <= R / 4 ? 2 : -1)>(c, s); break;
        case 3: run_strip<G, R, FLAGS, true, (3 <= R / 4 ? 3 : -1)>(c, s); break;
        case 4: run_strip<G, R, FLAGS, true, (4 <= R / 4 ? 4 : -1)>(c, s); break;
        case 5: run_strip<G, R, FLAGS, true, (5 <= R / 4 ? 5 : -1)>(c, s); break;
        default: run_strip<G, R, FLAGS, true, -1>(c, s); break;
      }
    } else {
      run_strip<G, R, FLAGS, true, -1>(c, s);
    }
  }
}

#if defined(__CUDACC__)

// ---- TMA bulk copy + mbarrier helpers (sm_90+ PTX; UBLKCP / SYNCS in SASS) ----
__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return (uint32_t)__cvta_generic_to_shared(p);
}
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)),
               "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void tma_bulk_g2s(void* dst_smem, const void* src_gmem, uint32_t bytes,
                                             uint64_t* bar) {
  asm volatile(
      "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
          smem_u32(dst_smem)),
      "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar))
      : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t done;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.b32 %0, 1, 0, p;\n\t}"
      : "=r"(done)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return done != 0;
}

#ifndef B2A_MINB
#define B2A_MINB 1  // minimum resident CTAs per SM requested from ptxas (set per shape by build.py)
#endif

// Persistent kernel: every warp pulls warp-tasks (32/G pairs) from a global
// counter, stages their sequences with two bulk copies and fills them.
template <int G, int R, int FLAGS>
__global__ void __launch_bounds__(fill_warps_of(G, R) * 32, B2A_MINB) fill_kernel(const FillParams prm) {
  extern __shared__ __align__(128) uint8_t smem[];
  constexpr int P = 32 / G;
  constexpr int FILL_WARPS = fill_warps_of(G, R);
  constexpr bool LUT = (FLAGS & F_LUT) != 0;
  constexpr int TBW = tbw_of(R);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  // smem: [FILL_WARPS mbarriers (64 bytes)][LUT][per-warp staging]
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem);
  int32_t* lut_s = reinterpret_cast<int32_t*>(smem + 64);
  const uint32_t lut_bytes = LUT ? lut_smem_bytes(prm.sc.alpha) : 0u;
  uint8_t* stage = smem + 64 + lut_bytes + (size_t)warp * prm.smem_seq_bytes;
  uint64_t* bar = &bars[warp];
  if (threadIdx.x < FILL_WARPS) mbar_init(&bars[threadIdx.x], 1);
  if (LUT) {
    for (int k = threadIdx.x; k < lut_entries(prm.sc.alpha); k += blockDim.x) lut_s[k] = prm.lut[k];  // 4*score + 3 - (4*gap_open + 1)
  }
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  __syncthreads();

  const bool strip_tasks = (G == 32) && prm.progress != nullptr;
  const uint32_t ntasks = strip_tasks ? prm.n_strip_tasks : prm.nblocks * G;
  uint32_t parity = 0;

  for (uint32_t done = 0; prm.task_limit == 0 || done < prm.task_limit; ++done) {
    uint32_t task = 0;
    if (lane == 0) task = atomicAdd(prm.task_counter, 1u);
    task = __shfl_sync(0xffffffffu, task, 0);
    if (task >= ntasks) break;
    uint32_t b, sub;
    int32_t only_strip = -1;
    if (strip_tasks) {
      // (pair, strip) tasks in pair-major order: find the block by its task base (blocks are few)
      uint32_t lo = 0, hi = prm.nblocks;
      while (hi - lo > 1) {
        const uint32_t mid = (lo + hi) / 2;
        if (prm.blocks[mid].strip_task_base <= task) lo = mid;
        else hi = mid;
      }
      b = lo;
      const uint32_t rel = task - (uint32_t)prm.blocks[b].strip_task_base;
      const uint32_t ns = prm.blocks[b].nstrips;
      sub = rel / ns;
      only_strip = (int32_t)(rel % ns);
    } else {
      b = task / G;
      sub = task % G;
    }
    const Block blk = prm.blocks[b];
    if (strip_tasks && sub >= blk.npairs) continue;  // padding pair of the last block: nothing to do
    const uint32_t xbytes = blk.xwords * P * 4, ybytes = blk.ywords * P * 4;
    // a strip task stages only the G*R x symbols of its own rows (P == 1 there); y is needed whole
    const uint32_t xoff = strip_tasks ? (uint32_t)only_strip * G * R : 0u;
    const uint32_t xstage = strip_tasks ? (uint32_t)(G * R) : xbytes;
    if (lane == 0) {
      // the previous task's generic-proxy reads of the staging buffer are done (syncwarp below)
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
      mbar_expect_tx(bar, xstage + ybytes);
      const uint8_t* src = prm.seq + blk.seq_off;
      tma_bulk_g2s(stage, src + (size_t)sub * xbytes + xoff, xstage, bar);
      tma_bulk_g2s(stage + xstage, src + (size_t)G * xbytes + (size_t)sub * ybytes, ybytes, bar);
    }
    LaneCtx<G> c;
    c.sc = prm.sc;
    c.lut = lut_s;
    c.lut_base = smem_u32(lut_s);
    c.one = prm.one;
    c.ge4 = prm.ge4;
    c.only_strip = only_strip;
    c.prog_mine = strip_tasks ? prm.progress + task : nullptr;
    c.prog_prev = (strip_tasks && only_strip > 0) ? prm.progress + task - 1 : nullptr;
    c.xs = reinterpret_cast<const uint32_t*>(stage) - xoff / 4;  // indexed by absolute row word
    c.ys = reinterpret_cast<const uint32_t*>(stage + xstage);
    c.g = lane / G;
    c.l = lane % G;
    c.lane = lane;
    c.pi = (int32_t)(sub * P) + c.g;
    const bool valid = (uint32_t)c.pi < blk.npairs;
    c.m = valid ? (int32_t)prm.pm[blk.first + c.pi] : 0;
    c.n = valid ? (int32_t)prm.pn[blk.first + c.pi] : 0;
    c.maxn = (int32_t)blk.maxn;
    c.maxm = (int32_t)blk.maxm;
    c.nstrips = (int32_t)blk.nstrips;
    c.K = (int32_t)blk.K;
    c.rows_pad = (int32_t)blk.rows_pad;
    c.uniform = blk.uniform != 0;
    c.bnd = reinterpret_cast<int4*>(prm.bnd + blk.bnd_off);
    c.rows = reinterpret_cast<int32_t*>(prm.rows + blk.rows_off);
    c.tb = reinterpret_cast<uint4*>(prm.tb + blk.tb_off) +
           (size_t)sub * blk.nstrips * blk.K * TBW * 32;
    while (!mbar_try_wait(bar, parity)) {
    }
    parity ^= 1u;
    fill_lane<G, R, FLAGS>(c);
    __syncwarp();
  }
}

#endif  // __CUDACC__

}  // namespace b2a

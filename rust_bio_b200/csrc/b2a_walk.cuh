// K2: row m, last-column fix-ups and the traceback walk -- one lane per pair.
//
// Reference rust-bio 4.0.1 src/alignment/pairwise/mod.rs, Aligner::custom:
//   row m of the fill (the only row whose S starts from the column tracker
//     S[curr][m] instead of MIN_SCORE)                      641-645, 757-758
//   "Handle suffix clipping in the j=n case"                809-821
//   "recompute the last column of I"                        825-843
//   the traceback state machine                             845-908
//   Alignment construction / clip filtering                 910-921, 974, 1006
// These parts are sequential per pair and O(m+n); they are replayed literally
// here on top of what K1 left in HBM: the boundary row m-1 (S, I, column
// tracker), the row trackers, the last column and the 4-bit traceback.
#pragma once
#include "b2a_common.cuh"
#include "b2a_coop.cuh"

namespace b2a {

struct WalkParams {
  const Block* blocks;
  uint32_t nblocks;
  const uint32_t* pm;
  const uint32_t* pn;
  const uint32_t* order;  // sorted pair -> caller's pair index
  const uint8_t* seq;
  const uint8_t* bnd;
  uint8_t* rows;
  uint8_t* rowm;
  const uint8_t* tb;
  uint8_t* ops_scratch;
  const int32_t* lut;
  DevScoring sc;
  int32_t G, R;
  int32_t filter_clips;  // semiglobal / local: Alignment::filter_clip_operations
  int32_t packtrk;       // K1 ran with F_PACKTRK (how the column tracker in the boundary row is encoded)
  uint32_t seq_smem_per_warp;  // warp-per-pair K2: bytes of shared memory per warp for the pair's x and y (0: none)
  // outputs, indexed by the caller's pair index
  int32_t* score;
  uint32_t* xstart;
  uint32_t* xend;
  uint32_t* ystart;
  uint32_t* yend;
  uint32_t* n_ops;
  uint64_t* ops_src;   // where the pair's ops start inside ops_scratch
  uint32_t* clip_len;  // 4 per pair
  uint32_t* status;    // 0 ok, 1 = corrupt traceback (reference would panic, mod.rs:905)
  uint32_t* err_flag;  // set to 1 if any pair's status is non-zero
};

constexpr uint32_t LAZY = 15;  // "came from S of the neighbour": resolved when the walk needs it

struct PairView {
  DevScoring sc;
  const int32_t* lut;
  const uint32_t* xw;  // staged x words of this pair's task; word w at xw[w*P]
  const uint32_t* yw;
  int32_t P;
  int32_t m, n, pi;
  int32_t G, R, TBW, nstrips, K;
  const int4* bnd;     // [column][32]
  int32_t* rows;       // arrays of [rows_pad][32]
  int32_t rows_pad;
  uint16_t* rowm;      // [column][32]
  const uint32_t* tb;  // block base
  int32_t sub, g;      // task inside the block, slot inside the task
  int32_t packtrk;
  int32_t maxn;        // block maximum of n
  int64_t bnd_base;    // boundary row of this pair: bnd[bnd_base + j * bnd_stride] (see bnd_index)
  int32_t bnd_stride;
  const uint8_t* xs8 = nullptr;  // warp-per-pair K2: the pair's staged x / y copied into shared memory (or null)
  const uint8_t* ys8 = nullptr;
  // exact division by R and by G*R without a divide: q = (x * mul) >> 40 with mul = ceil(2^40 / d) is floor(x / d)
  // for x < 2^24 and d <= 2^10 (the walk computes a traceback address per move; sequence lengths are < 2^24)
  uint64_t mulR = 0, mulGR = 0;
  B2A_HD void set_shape(int32_t G_, int32_t R_) {
    G = G_;
    R = R_;
    TBW = (R_ + 3) / 4;
    mulR = ((1ull << 40) + (uint64_t)R_ - 1) / (uint64_t)R_;
    mulGR = ((1ull << 40) + (uint64_t)(G_ * R_) - 1) / (uint64_t)(G_ * R_);
  }

  B2A_HD int32_t xsym(int32_t i) const {  // x[i-1]
    const int32_t b = i - 1;
    if (xs8) return (int32_t)xs8[b];
    return (int32_t)((xw[(b >> 2) * P] >> (8 * (b & 3))) & 0xffu);
  }
  B2A_HD int32_t ysym(int32_t j) const {
    const int32_t b = j - 1;
    if (ys8) return (int32_t)ys8[b];
    return (int32_t)((yw[(b >> 2) * P] >> (8 * (b & 3))) & 0xffu);
  }
  B2A_HD int32_t score(int32_t p, int32_t q) const {
    if (sc.alpha) return lut[p * sc.alpha + q];
    return p == q ? sc.match_score : sc.mismatch_score;
  }
  B2A_HD int32_t& row(int arr, int32_t i) const { return rows[(arr * rows_pad + i) * 32 + pi]; }
  B2A_HD int4 load_bnd(int32_t j) const {
#if defined(__CUDA_ARCH__)
    return __ldg(&bnd[bnd_base + (int64_t)j * bnd_stride]);  // read-only path: K1 wrote it in an earlier launch
#else
    return bnd[bnd_base + (int64_t)j * bnd_stride];
#endif
  }
  // compressed traceback nibble of an interior cell 1 <= i <= m-1, 1 <= j <= n
  B2A_HD uint32_t nib(int32_t i, int32_t j) const {
    const int32_t GR = G * R;
    const int32_t s = (int32_t)(((uint64_t)(uint32_t)(i - 1) * mulGR) >> 40), rem = (i - 1) - s * GR;
    const int32_t l = (int32_t)(((uint64_t)(uint32_t)rem * mulR) >> 40), r = rem - l * R;
    const int32_t lane = g * G + l;
    const int32_t t = (j - 1) + l;
    const size_t word =
        ((((size_t)(sub * nstrips + s) * K + (t >> 3)) * TBW + (r >> 2)) * 32 + lane) * 4 + (r & 3);
    return (tb[word] >> (4 * (7 - (t & 7)))) & 15u;
  }
  B2A_HD uint32_t nib_scode(uint32_t nb, int32_t i, int32_t j) const {
    switch (nb & 3u) {
      case NB_DIAG: return xsym(i) == ysym(j) ? TB_MATCH : TB_SUBST;
      case NB_INS: return TB_INS;
      case NB_DEL: return TB_DEL;
      default: return TB_XCLIP_PREFIX;
    }
  }
};

// Boundary row m-1 as K1 leaves it (scaled domain, b2a_fill.cuh): x = 4*S, y = 4*I + 2,
// z/w = column tracker: packed key 4096*(max S) + (4095 - first row) [F_PACKTRK] or (4*(T), row).
struct Boundary {
  int32_t S, I, Tv, Ti;
};
B2A_HD Boundary decode_boundary(const int4 b, const bool packtrk, const int32_t xs, const int32_t m) {
  Boundary o;
  o.S = b.x >> 2;
  o.I = b.y >> 2;
  o.Tv = MIN_SCORE;
  o.Ti = m;
  if (packtrk) {
    if (b.z != (int32_t)0x80000000) {
      o.Tv = (b.z >> 12) + xs;
      o.Ti = 4095 - (b.z & 4095);
    }
  } else if (b.z > -(1 << 29)) {
    o.Tv = b.z >> 2;
    o.Ti = b.w;
  }
  return o;
}

// cells kept as the reference's u16: i | d << 4 | s << 8 (mod.rs:1031-1033)
B2A_HD uint32_t cell_make(uint32_t i, uint32_t d, uint32_t s) { return i | (d << 4) | (s << 8); }
B2A_HD uint32_t cell_i(uint32_t c) { return c & 15u; }
B2A_HD uint32_t cell_d(uint32_t c) { return (c >> 4) & 15u; }
B2A_HD uint32_t cell_s(uint32_t c) { return (c >> 8) & 15u; }
B2A_HD uint32_t cell_set_s(uint32_t c, uint32_t s) { return (c & ~0xF00u) | (s << 8); }
B2A_HD uint32_t cell_set_i(uint32_t c, uint32_t i) { return (c & ~0x00Fu) | i; }

struct WalkOut {
  int32_t score;
  uint32_t xstart, xend, ystart, yend, n_ops, status;
  uint32_t clip[4];
};

// What row m and the last-column fix-ups leave for the walk: the far-corner cell and the clip jumps that are
// not stored per cell.
struct EndState {
  int32_t SmN, ImN;   // S(m,n), I(m,n)
  uint32_t cmN;       // cell (m,n)
  int32_t Snm, Lym;   // Sn[m], Ly[m]
  int32_t Lx0, LxN;   // Lx[0], Lx[n]
};

// Row m (mod.rs:641-645, 729-805 at i == m), the two last-column fix-up passes (809-843): one lane, literally.
B2A_HD void finish_matrix_seq(const PairView& v, EndState& es) {
  const DevScoring& sc = v.sc;
  const int32_t m = v.m, n = v.n;
  const int32_t go = sc.gap_open, ge = sc.gap_extend;
  const int32_t xp = sc.xclip_prefix, xs = sc.xclip_suffix, yp = sc.yclip_prefix,
                ys = sc.yclip_suffix;

  // ------------------------------------------------------------------ row m
  int32_t SmN = 0, ImN = MIN_SCORE;   // S(m,n), I(m,n)
  uint32_t cmN = 0;                   // cell (m,n)
  int32_t Snm = MIN_SCORE, Lym = 0;   // Sn[m], Ly[m]
  int32_t Lx0 = 0, LxN = 0;           // Lx[0], Lx[n]
  if (m >= 1) {
    // column 0 (mod.rs:622-671 at i == m); the tracker over rows 1..m-1 first
    int32_t T = MIN_SCORE;
    for (int32_t i = 1; i < m; ++i) {
      const int32_t val = col0_S(sc, i) + xs;
      if (val > T) {
        T = val;
        Lx0 = m - i;
      }
    }
    int32_t Im = col0_I(sc, m);
    uint32_t ib = col0_ibits(sc, m);
    int32_t Sm = T;
    uint32_t sb = TB_XCLIP_SUFFIX;
    if (Im > Sm) {
      Sm = Im;
      sb = TB_INS;
    }
    if (xp > Sm) {
      Sm = xp;
      sb = TB_XCLIP_PREFIX;
    }
    if (Sm + ys > Snm) {
      Snm = Sm + ys;
      Lym = n;
    }
    int32_t Dm = MIN_SCORE;
    uint32_t cell = cell_make(ib, TB_START, sb);
    v.rowm[0 * 32 + v.pi] = (uint16_t)cell;
    LxN = Lx0;
    const int32_t p = v.xsym(m);
    const int32_t yclip_score = yp + go + ge * (m - 1);
    int32_t sdiag = (m == 1) ? 0 : col0_S(sc, m - 1);
    // columns are walked four at a time: the boundary row and y symbols of a group are loaded up front
    // (independent loads in flight), then the recurrence runs over them in order
    constexpr int UB = 4;
    for (int32_t j0 = 1; j0 <= n; j0 += UB) {
      int4 braw[UB];
      int32_t qv[UB];
#pragma unroll
      for (int u = 0; u < UB; ++u) {
        const int32_t jj = j0 + u;
        braw[u] = make_int4(0, 0, 0, 0);
        qv[u] = 0;
        if (jj <= n) {
          if (m != 1) braw[u] = v.load_bnd(jj);
          qv[u] = v.ysym(jj);
        }
      }
#pragma unroll
      for (int u = 0; u < UB; ++u) {
      const int32_t j = j0 + u;
      if (j > n) break;
      int32_t sup, iup, Tv, Ti;
      if (m == 1) {
        sup = row0_S(sc, j, n);
        iup = MIN_SCORE;
        Tv = MIN_SCORE;
        Ti = m;
      } else {
        const Boundary b = decode_boundary(braw[u], v.packtrk != 0, xs, m);
        sup = b.S;
        iup = b.I;
        Tv = b.Tv;
        Ti = b.Ti;
      }
      const int32_t q = qv[u];
      const int32_t m_score = sdiag + v.score(p, q);
      int32_t best_i, best_d;
      {
        const int32_t i_score = iup + ge, s_score = sup + go;
        if (i_score > s_score) {
          best_i = i_score;
          ib = TB_INS;
        } else {
          best_i = s_score;
          ib = LAZY;
        }
      }
      uint32_t db;
      {
        const int32_t d_score = Dm + ge, s_score = Sm + go;
        if (d_score > s_score) {
          best_d = d_score;
          db = TB_DEL;
        } else {
          best_d = s_score;
          db = sb;  // s_bits of (m, j-1), final for j-1 < n
        }
      }
      int32_t best = Tv;
      sb = TB_XCLIP_SUFFIX;
      if (m_score > best) {
        best = m_score;
        sb = (p == q) ? TB_MATCH : TB_SUBST;
      }
      if (best_i > best) {
        best = best_i;
        sb = TB_INS;
      }
      if (best_d > best) {
        best = best_d;
        sb = TB_DEL;
      }
      const int32_t xcs = xclip_score(sc, j);
      if (xcs > best) {
        best = xcs;
        sb = TB_XCLIP_PREFIX;
      }
      if (yclip_score > best) {
        best = yclip_score;
        sb = TB_YCLIP_PREFIX;
      }
      Sm = best;
      Im = best_i;
      Dm = best_d;
      if (Sm + ys > Snm) {
        Snm = Sm + ys;
        Lym = n - j;
      }
      if (j == n) {
        LxN = m - Ti;
        if (ib == LAZY) {  // i_bits captured before the fix-ups touch (m-1, n)
          ib = (m == 1) ? row0_sbits(sc, n, n)
                        : v.nib_scode((uint32_t)v.row(ROWS_NL, m - 1), m - 1, n);
        }
      }
      cell = cell_make(ib, db, sb);
      v.rowm[j * 32 + v.pi] = (uint16_t)cell;
      sdiag = sup;
          }
    }
    SmN = Sm;
    ImN = Im;
    cmN = cell;
  }

  // ------------------------------- column n: materialise the cells K1 left as nibbles and run fix-up 1
  // (mod.rs:809-821) in the same pass over the rows; rows 0..m-1 keep S in ROWS_SL, I in ROWS_IL, the
  // literal cell in ROWS_NL.  i_bits are captured from the PRE-fix-up s_bits of the row above (743),
  // exactly as the reference's fill did before its fix-up loops ran.
  // K1 only keeps the row trackers when yclip_suffix is live; a dead one can never win (Sn <= MIN/2 + S)
  const bool ys_live = ys > DEAD_CLIP;
  {
    int32_t s0, c0;
    if (n == 0) {
      s0 = 0;
      c0 = (int32_t)cell_make(TB_START, TB_START, TB_START);
    } else {
      s0 = row0_S(sc, n, n);
      c0 = (int32_t)cell_make(TB_START, row0_dbits(sc, n), row0_sbits(sc, n, n));
    }
    if (m == 0) {
      SmN = s0;
      cmN = (uint32_t)c0;
      Snm = ys;
      Lym = n;
    } else {
      uint32_t s_above = cell_s((uint32_t)c0);  // pre fix-up s_bits(i-1, n)
      {  // row 0: Sn[0] = yclip_suffix (mod.rs:618, 711)
        int32_t S = s0;
        uint32_t cell = (uint32_t)c0;
        if (ys > S) {
          S = ys;
          cell = cell_set_s(cell, TB_YCLIP_SUFFIX);
        }
        v.row(ROWS_SL, 0) = S;
        v.row(ROWS_IL, 0) = MIN_SCORE;
        v.row(ROWS_NL, 0) = (int32_t)cell;
        if (S + xs > SmN) {
          SmN = S + xs;
          LxN = m;
          cmN = cell_set_s(cmN, TB_XCLIP_SUFFIX);
        }
      }
      constexpr int UB = 4;
      for (int32_t i0 = 1; i0 < m; i0 += UB) {
        int32_t nbv[UB], Sv[UB], Snv[UB];
#pragma unroll
        for (int u = 0; u < UB; ++u) {
          const int32_t i = i0 + u;
          nbv[u] = Sv[u] = 0;
          Snv[u] = MIN_SCORE;
          if (i < m && n != 0) {
            nbv[u] = v.row(ROWS_NL, i);
            Sv[u] = v.row(ROWS_SL, i);
            if (ys_live) Snv[u] = v.row(ROWS_SN, i);
          }
        }
#pragma unroll
        for (int u = 0; u < UB; ++u) {
          const int32_t i = i0 + u;
          if (i >= m) break;
          uint32_t cell;
          int32_t S, Sn;
          if (n == 0) {  // column n is column 0: closed forms (mod.rs:622-671)
            S = col0_S(sc, i);
            v.row(ROWS_IL, i) = col0_I(sc, i);
            cell = cell_make(col0_ibits(sc, i), TB_START, col0_sbits(sc, i));
            const int32_t val = S + ys;
            Sn = val > MIN_SCORE ? val : MIN_SCORE;
            if (!ys_live) Sn = MIN_SCORE;
            v.row(ROWS_LY, i) = 0;
          } else {
            const uint32_t nb = (uint32_t)nbv[u];
            cell = cell_make((nb & NB_IEXT) ? (uint32_t)TB_INS : s_above, (nb & NB_DEXT) ? (uint32_t)TB_DEL : LAZY,
                             v.nib_scode(nb, i, n));
            S = Sv[u];
            Sn = Snv[u];
          }
          s_above = cell_s(cell);
          if (Sn > S) {  // fix-up 1
            S = Sn;
            cell = cell_set_s(cell, TB_YCLIP_SUFFIX);
          }
          v.row(ROWS_SL, i) = S;
          v.row(ROWS_NL, i) = (int32_t)cell;
          if (S + xs > SmN) {
            SmN = S + xs;
            LxN = m - i;
            cmN = cell_set_s(cmN, TB_XCLIP_SUFFIX);
          }
        }
      }
      if (Snm > SmN) {  // i == m
        SmN = Snm;
        cmN = cell_set_s(cmN, TB_YCLIP_SUFFIX);
      }
      // ---------------------------------------------- fix-up 2, mod.rs:825-843
      int32_t S_prev = v.row(ROWS_SL, 0);
      uint32_t cell_prev = (uint32_t)v.row(ROWS_NL, 0);
      for (int32_t i0 = 1; i0 <= m; i0 += UB) {
        int32_t Iv[UB], Sv[UB], Cv[UB];
#pragma unroll
        for (int u = 0; u < UB; ++u) {
          const int32_t i = i0 + u;
          Iv[u] = Sv[u] = Cv[u] = 0;
          if (i < m) {
            Iv[u] = v.row(ROWS_IL, i);
            Sv[u] = v.row(ROWS_SL, i);
            Cv[u] = v.row(ROWS_NL, i);
          }
        }
#pragma unroll
        for (int u = 0; u < UB; ++u) {
          const int32_t i = i0 + u;
          if (i > m) break;
          const int32_t s_score = S_prev + go;
          int32_t I = (i == m) ? ImN : Iv[u];
          int32_t S = (i == m) ? SmN : Sv[u];
          uint32_t cell = (i == m) ? cmN : (uint32_t)Cv[u];
          bool dirty = false;
          if (s_score > I) {
            I = s_score;
            cell = cell_set_i(cell, cell_s(cell_prev));
            dirty = true;
          }
          if (s_score > S) {
            S = s_score;
            cell = cell_set_s(cell, TB_INS);
            dirty = true;
            if (i != m && S + xs > SmN) {
              SmN = S + xs;
              LxN = m - i;
              cmN = cell_set_s(cmN, TB_XCLIP_SUFFIX);
            }
          }
          if (i == m) {
            ImN = I;
            SmN = S;
            cmN = cell;
          } else if (dirty) {
            v.row(ROWS_IL, i) = I;
            v.row(ROWS_SL, i) = S;
            v.row(ROWS_NL, i) = (int32_t)cell;
          }
          S_prev = S;
          cell_prev = cell;
        }
      }
    }
  }

  es.SmN = SmN;
  es.ImN = ImN;
  es.cmN = cmN;
  es.Snm = Snm;
  es.Lym = Lym;
  es.Lx0 = Lx0;
  es.LxN = LxN;
}

// The traceback state machine (mod.rs:845-908) as a resumable loop: walk_run() advances at most `max_steps`
// moves, so a warp can interleave lane 0's walk with prefetches issued by the other lanes.
struct WalkState {
  int32_t i, j;
  uint32_t layer;
  uint32_t xstart, ystart, xend, yend;
  uint32_t nops, nclip, status;
  uint32_t clips[4];
  int32_t guard;
  uint8_t* ops_end;  // ops are written backwards into ops_end[-1], ops_end[-2], ...
};

B2A_HD void walk_begin(const PairView& v, const EndState& es, uint8_t* ops_end, WalkState& w) {
  w.i = v.m;
  w.j = v.n;
  w.layer = cell_s(es.cmN);
  w.xstart = w.ystart = 0;
  w.xend = (uint32_t)v.m;
  w.yend = (uint32_t)v.n;
  w.nops = w.nclip = w.status = 0;
  w.clips[0] = w.clips[1] = w.clips[2] = w.clips[3] = 0;
  w.guard = v.m + v.n + 8;
  w.ops_end = ops_end;
}

// returns true when the walk has ended (TB_START reached, or a panic path of the reference)
B2A_HD bool walk_run(const PairView& v, const EndState& es, const bool filter_clips, WalkState& w, int32_t max_steps) {
  const DevScoring& sc = v.sc;
  const int32_t m = v.m, n = v.n;
  const int32_t xs = sc.xclip_suffix;
  const uint32_t cmN = es.cmN;
  const int32_t LxN = es.LxN, Lx0 = es.Lx0, Lym = es.Lym;
  auto get_cell_n = [&](int32_t i) -> uint32_t {  // column n, after the fix-ups
    return (i == m) ? cmN : (uint32_t)v.row(ROWS_NL, i);
  };
  auto get_s = [&](int32_t i, int32_t j) -> uint32_t {
    if (j == n) return cell_s(get_cell_n(i));
    if (i == 0) return row0_sbits(sc, j, n);
    if (i == m) return cell_s((uint32_t)v.rowm[j * 32 + v.pi]);
    if (j == 0) return col0_sbits(sc, i);
    return v.nib_scode(v.nib(i, j), i, j);
  };
  int32_t i = w.i, j = w.j;
  uint32_t xstart = w.xstart, ystart = w.ystart, xend = w.xend, yend = w.yend;
  uint32_t nops = w.nops, nclip = w.nclip, status = w.status;
  uint32_t clips[4] = {w.clips[0], w.clips[1], w.clips[2], w.clips[3]};
  uint32_t layer = w.layer;
  int32_t guard = w.guard;
  uint8_t* ops_end = w.ops_end;
  while (layer != TB_START && status == 0) {
    if (max_steps-- <= 0) break;
    if (--guard < 0) {
      status = 1;
      break;
    }
    uint32_t next;
    if (layer == TB_INS) {
      *(--ops_end) = 3;
      ++nops;
      uint32_t c;
      if (j == n) {
        c = cell_i(get_cell_n(i));
      } else if (i == m) {
        c = cell_i((uint32_t)v.rowm[j * 32 + v.pi]);
        if (c == LAZY) c = get_s(m - 1, j);
      } else if (j == 0) {
        c = col0_ibits(sc, i);
      } else {
        c = (v.nib(i, j) & NB_IEXT) ? (uint32_t)TB_INS : get_s(i - 1, j);
      }
      next = c;
      i -= 1;
    } else if (layer == TB_DEL) {
      *(--ops_end) = 2;
      ++nops;
      uint32_t c;
      if (i == 0) {
        c = row0_dbits(sc, j);
      } else if (i == m) {
        c = cell_d((uint32_t)v.rowm[j * 32 + v.pi]);
      } else if (j == n) {
        c = cell_d(get_cell_n(i));
        if (c == LAZY) c = get_s(i, n - 1);
      } else {
        c = (v.nib(i, j) & NB_DEXT) ? (uint32_t)TB_DEL : get_s(i, j - 1);
      }
      next = c;
      j -= 1;
    } else if (layer == TB_MATCH || layer == TB_SUBST) {
      *(--ops_end) = (layer == TB_MATCH) ? 0 : 1;
      ++nops;
      next = get_s(i - 1, j - 1);
      i -= 1;
      j -= 1;
    } else if (layer == TB_XCLIP_PREFIX) {
      if (!filter_clips) {
        *(--ops_end) = 4;
        ++nops;
        if (nclip < 4) clips[nclip] = (uint32_t)i;
        ++nclip;
      }
      xstart = (uint32_t)i;
      i = 0;
      next = get_s(0, j);
    } else if (layer == TB_XCLIP_SUFFIX) {
      int32_t lx;
      if (j == n) lx = LxN;
      else if (j == 0) lx = Lx0;
      else lx = (m >= 2) ? m - decode_boundary(v.load_bnd(j), v.packtrk != 0, xs, m).Ti : 0;
      if (!filter_clips) {
        *(--ops_end) = 4;
        ++nops;
        if (nclip < 4) clips[nclip] = (uint32_t)lx;
        ++nclip;
      }
      i -= lx;
      xend = (uint32_t)i;
      next = get_s(i, j);
    } else if (layer == TB_YCLIP_PREFIX) {
      if (!filter_clips) {
        *(--ops_end) = 5;
        ++nops;
        if (nclip < 4) clips[nclip] = (uint32_t)j;
        ++nclip;
      }
      ystart = (uint32_t)j;
      j = 0;
      next = get_s(i, 0);
    } else if (layer == TB_YCLIP_SUFFIX) {
      int32_t ly;
      if (i == m) ly = Lym;
      else if (i == 0 || n == 0) ly = n;
      else ly = n - v.row(ROWS_LY, i);
      if (!filter_clips) {
        *(--ops_end) = 5;
        ++nops;
        if (nclip < 4) clips[nclip] = (uint32_t)ly;
        ++nclip;
      }
      j -= ly;
      yend = (uint32_t)j;
      next = get_s(i, j);
    } else {
      status = 1;  // panic!("Dint expect this!") mod.rs:905
      break;
    }
    if (i < 0 || j < 0) {
      status = 1;
      break;
    }
    layer = next;
  }
  w.i = i;
  w.j = j;
  w.layer = layer;
  w.xstart = xstart;
  w.ystart = ystart;
  w.xend = xend;
  w.yend = yend;
  w.nops = nops;
  w.nclip = nclip;
  w.status = status;
  for (int k = 0; k < 4; ++k) w.clips[k] = clips[k];
  w.guard = guard;
  w.ops_end = ops_end;
  return layer == TB_START || status != 0;
}

B2A_HD void walk_finish(const EndState& es, const WalkState& w, WalkOut& out) {
  out.score = es.SmN;
  out.xstart = w.xstart;
  out.xend = w.xend;
  out.ystart = w.ystart;
  out.yend = w.yend;
  out.n_ops = w.nops;
  out.status = (w.nclip > 4) ? 1u : w.status;
  // clips were met end-to-start; report them in alignment order
  const uint32_t nc = w.nclip > 4 ? 4 : w.nclip;
  for (uint32_t k = 0; k < 4; ++k) out.clip[k] = (k < nc) ? w.clips[nc - 1 - k] : 0u;
}

// K2 for one pair by one lane: ops are written backwards into ops_end[-1], ops_end[-2], ...
B2A_HD void walk_pair(const PairView& v, const bool filter_clips, uint8_t* ops_end, WalkOut& out) {
  EndState es;
  finish_matrix_seq(v, es);
  WalkState w;
  walk_begin(v, es, ops_end, w);
  walk_run(v, es, filter_clips, w, 0x7fffffff);
  walk_finish(es, w, out);
}

// ---------------------------------------------------------------------------------------------------------
// Warp-per-pair K2 (small and medium batches, long sequences): the three O(m + n) passes of
// finish_matrix_seq are sequential only through one max-plus chain each, which W lanes resolve with a prefix
// maximum, 32 columns / rows at a time; every strict comparison of the reference is then re-evaluated
// literally per element from its neighbours' final values (the same device as K3's column chunks):
//   row m      D(m,j) = max(D(m,j-1)+ge, S(m,j-1)+go) with S = max(A, D), A = the best non-D candidate
//              => D(m,j) = max(D(m,j-1) + gs, A(j-1) + go), gs = max(ge, go): D(m,j) - gs*j is a running maximum;
//   fix-up 1   element-wise; the re-maximisation of S(m,n) is an arg-max with the lowest row winning ties;
//   fix-up 2   S'(i) = max(S(i), S'(i-1)+go): S'(i) - go*i is a running maximum of S(k) - go*k.
// All arithmetic is exact (the engine's range guard keeps every real score within +-2^27).  The walk itself
// stays on lane 0 (each move depends on the cell the previous one read); the other lanes pull the traceback
// words along the diagonal ahead of it into the cache.
B2A_HD int32_t imin32(int32_t a, int32_t b) { return a < b ? a : b; }

template <int W>
B2A_HD int32_t coop_scan_max(int lane, int32_t v) {  // inclusive prefix maximum over the lanes
  using C = Coop<W>;
  for (int d = 1; d < W; d <<= 1) {
    const int32_t t = C::up(v, d);
    if (lane >= d) v = imax(v, t);
  }
  return v;
}

// first lane (lowest index) holding the maximum of `val` over the lanes with `has`; returns false if none has.
// Callers pass has = (candidate beats the running value): the running value is the same on every lane, so a
// candidate that does not beat it cannot be the arg-max that does, and most chunks skip the reduction after one
// ballot.  `packed`: values within +-2^17 and indices <= 4095 (K1's F_PACKTRK condition): one 32-bit REDUX on the
// key 4096*value + (4095 - index) instead of five 64-bit shuffle rounds.
template <int W>
B2A_HD bool coop_argmax_first(int lane, bool has, int32_t val, int32_t idx, int32_t& best_val, int32_t& best_idx,
                              bool packed = false) {
  using C = Coop<W>;
  (void)lane;
  if (C::ballot(has) == 0u) return false;
  if (packed) {
    const int32_t key = C::all_max32(has ? val * 4096 + (4095 - idx) : (int32_t)0x80000000);
    best_val = key >> 12;
    best_idx = 4095 - (key & 4095);
    return true;
  }
  // key: value high, (0x7fffffff - idx) low: the largest key is the largest value at the smallest index
  const long long none = (long long)0x8000000000000000ull;
  long long key = has ? (long long)(((unsigned long long)(long long)val << 32) | (unsigned long long)(uint32_t)(0x7fffffff - idx))
                      : none;
  key = C::all_max(key);
  best_val = (int32_t)(key >> 32);
  best_idx = 0x7fffffff - (int32_t)(uint32_t)(key & 0xffffffffll);
  return true;
}

template <int W>
B2A_HD void finish_matrix_coop(const int lane, const PairView& v, EndState& es) {
  using C = Coop<W>;
  const DevScoring& sc = v.sc;
  const int32_t m = v.m, n = v.n;
  if (m < 2 || n < 1) {  // degenerate shapes: closed forms only, nothing to share out
    if (lane == 0) finish_matrix_seq(v, es);
    C::sync();
    es.SmN = C::from(es.SmN, 0);
    es.ImN = C::from(es.ImN, 0);
    es.cmN = (uint32_t)C::from((int32_t)es.cmN, 0);
    es.Snm = C::from(es.Snm, 0);
    es.Lym = C::from(es.Lym, 0);
    es.Lx0 = C::from(es.Lx0, 0);
    es.LxN = C::from(es.LxN, 0);
    return;
  }
  const int32_t go = sc.gap_open, ge = sc.gap_extend;
  const int32_t xp = sc.xclip_prefix, xs = sc.xclip_suffix, yp = sc.yclip_prefix, ys = sc.yclip_suffix;
  const int32_t gs = imax(ge, go);
  const bool pk = v.packtrk != 0;

  // ------------------------------------------------------------------ row m, column 0 (mod.rs:622-671 at i == m)
  // column 0's tracker over rows 1..m-1 (mod.rs:657-661): col0_S(i) never increases with i (go + ge*(i-1) falls,
  // the clip terms are constants, and col0_S(1) = max(go, xp) bounds both), so the first maximum is row 1
  int32_t T = MIN_SCORE, Lx0 = 0;
  if (col0_S(sc, 1) + xs > MIN_SCORE) {  // m >= 2 here
    T = col0_S(sc, 1) + xs;
    Lx0 = m - 1;
  }
  int32_t Im0 = col0_I(sc, m);
  const uint32_t ib0 = col0_ibits(sc, m);
  int32_t Sm0 = T;
  uint32_t sb0 = TB_XCLIP_SUFFIX;
  if (Im0 > Sm0) {
    Sm0 = Im0;
    sb0 = TB_INS;
  }
  if (xp > Sm0) {
    Sm0 = xp;
    sb0 = TB_XCLIP_PREFIX;
  }
  int32_t Snm = MIN_SCORE, Lym = 0;
  if (Sm0 + ys > Snm) {
    Snm = Sm0 + ys;
    Lym = n;
  }
  if (lane == 0) v.rowm[0 * 32 + v.pi] = (uint16_t)cell_make(ib0, TB_START, sb0);
  int32_t LxN = Lx0;
  const int32_t p = v.xsym(m);
  const int32_t yclip_score = yp + go + ge * (m - 1);
  // ------------------------------------------------------------------ row m, columns 1..n in chunks of W
  // carries = the last column done so far (every lane holds the same values)
  int32_t cSup = col0_S(sc, m - 1);  // S(m-1, j-1) for the chunk's first column
  int32_t cD = MIN_SCORE, cS = Sm0;  // D(m, j-1), S(m, j-1)
  uint32_t csb = sb0;                // s_bits(m, j-1)
  int32_t SmN = 0, ImN = MIN_SCORE;
  uint32_t cmN = 0;
  // the boundary row of the NEXT chunk is requested before this chunk's chain is resolved (the loads do not
  // depend on the carries), so every chunk after the first finds its operands already on the way
  int4 braw_next = v.load_bnd(imin32(1 + lane, n));
  for (int32_t base = 1; base <= n; base += W) {
    const int32_t j = base + lane;
    const bool act = j <= n;
    const int32_t jc = act ? j : n;  // idle lanes repeat the last column: loads stay in bounds, nothing is stored
    const int4 braw = braw_next;
    if (base + W <= n) braw_next = v.load_bnd(imin32(base + W + lane, n));
    const Boundary b = decode_boundary(braw, pk, xs, m);
    const int32_t q = v.ysym(jc);
    int32_t sdiag = C::up(b.S, 1);
    if (lane == 0) sdiag = cSup;
    const int32_t m_score = sdiag + v.score(p, q);
    uint32_t ib;
    int32_t best_i;
    {
      const int32_t i_score = b.I + ge, s_score = b.S + go;
      if (i_score > s_score) {
        best_i = i_score;
        ib = TB_INS;
      } else {
        best_i = s_score;
        ib = LAZY;
      }
    }
    const int32_t xcs = xclip_score(sc, jc);
    const int32_t A = imax(imax(imax(b.Tv, m_score), imax(best_i, xcs)), yclip_score);
    // D(m,j) - gs*j as a running maximum
    int32_t t;
    {
      const int32_t aprev = C::up(A, 1);
      if (lane == 0) t = imax(cD + ge, cS + go) - gs * jc;
      else t = aprev + go - gs * jc;
    }
    const int32_t best_d = coop_scan_max<W>(lane, t) + gs * jc;
    // the cell, literally (mod.rs:757-786 with the running best starting from the column tracker)
    int32_t best = b.Tv;
    uint32_t sb = TB_XCLIP_SUFFIX;
    if (m_score > best) {
      best = m_score;
      sb = (p == q) ? TB_MATCH : TB_SUBST;
    }
    if (best_i > best) {
      best = best_i;
      sb = TB_INS;
    }
    if (best_d > best) {
      best = best_d;
      sb = TB_DEL;
    }
    if (xcs > best) {
      best = xcs;
      sb = TB_XCLIP_PREFIX;
    }
    if (yclip_score > best) {
      best = yclip_score;
      sb = TB_YCLIP_PREFIX;
    }
    // d_bits from the final values of column j-1
    int32_t pD = C::up(best_d, 1), pS = C::up(best, 1);
    uint32_t psb = (uint32_t)C::up((int32_t)sb, 1);
    if (lane == 0) {
      pD = cD;
      pS = cS;
      psb = csb;
    }
    const uint32_t db = (pD + ge > pS + go) ? (uint32_t)TB_DEL : psb;
    // row tracker of row m (mod.rs:799-802): first column with the highest S + ys, if above the running value
    {
      int32_t gv, gj;  // arg-max over the real scores (every `best` of row m is one); the clip is added afterwards
      if (coop_argmax_first<W>(lane, act && best + ys > Snm, best, j, gv, gj, pk)) {
        Snm = gv + ys;
        Lym = n - gj;
      }
    }
    if (act && j == n) {
      if (ib == LAZY) ib = v.nib_scode((uint32_t)v.row(ROWS_NL, m - 1), m - 1, n);  // captured before the fix-ups
    }
    const uint32_t cell = cell_make(ib, db, sb);
    if (act) v.rowm[j * 32 + v.pi] = (uint16_t)cell;
    const int32_t left = n - base;
    const int src = left < W - 1 ? left : W - 1;
    cSup = C::from(b.S, src);
    cD = C::from(best_d, src);
    cS = C::from(best, src);
    csb = (uint32_t)C::from((int32_t)sb, src);
    if (base + W > n) {  // the chunk holding column n
      SmN = cS;
      ImN = C::from(best_i, src);
      cmN = (uint32_t)C::from((int32_t)cell, src);
      LxN = m - C::from(b.Ti, src);
    }
  }

  C::sync();  // row m read the cell (m-1, n) that fix-up 1 is about to rewrite

  // ------------------------------------------------------------------ column n + fix-up 1 (mod.rs:809-821)
  const bool ys_live = ys > DEAD_CLIP;
  const int32_t s0 = row0_S(sc, n, n);
  const uint32_t c0 = cell_make(TB_START, row0_dbits(sc, n), row0_sbits(sc, n, n));
  {  // row 0
    int32_t S = s0;
    uint32_t cell = c0;
    if (ys > S) {
      S = ys;
      cell = cell_set_s(cell, TB_YCLIP_SUFFIX);
    }
    if (lane == 0) {
      v.row(ROWS_SL, 0) = S;
      v.row(ROWS_IL, 0) = MIN_SCORE;
      v.row(ROWS_NL, 0) = (int32_t)cell;
    }
    if (S + xs > SmN) {
      SmN = S + xs;
      LxN = m;
      cmN = cell_set_s(cmN, TB_XCLIP_SUFFIX);
    }
  }
  {
    uint32_t c_above = cell_s(c0);  // pre-fix-up s_bits of the row above the chunk
    const int32_t yn = v.ysym(n);
    int32_t nb_next, S_next, Sn_next = MIN_SCORE;
    {
      const int32_t i0 = imin32(1 + lane, m - 1);
      nb_next = v.row(ROWS_NL, i0);
      S_next = v.row(ROWS_SL, i0);
      if (ys_live) Sn_next = v.row(ROWS_SN, i0);
    }
    for (int32_t base = 1; base < m; base += W) {
      const int32_t i = base + lane;
      const bool act = i < m;
      const int32_t ic = act ? i : m - 1;
      const uint32_t nb = (uint32_t)nb_next;
      int32_t S = S_next;
      const int32_t Sn = Sn_next;
      if (base + W < m) {  // next chunk's operands
        const int32_t i1 = imin32(base + W + lane, m - 1);
        nb_next = v.row(ROWS_NL, i1);
        S_next = v.row(ROWS_SL, i1);
        if (ys_live) Sn_next = v.row(ROWS_SN, i1);
      }
      uint32_t sbi;
      switch (nb & 3u) {
        case NB_DIAG: sbi = v.xsym(ic) == yn ? TB_MATCH : TB_SUBST; break;
        case NB_INS: sbi = TB_INS; break;
        case NB_DEL: sbi = TB_DEL; break;
        default: sbi = TB_XCLIP_PREFIX; break;
      }
      uint32_t s_above = (uint32_t)C::up((int32_t)sbi, 1);
      if (lane == 0) s_above = c_above;
      uint32_t cell = cell_make((nb & NB_IEXT) ? (uint32_t)TB_INS : s_above, (nb & NB_DEXT) ? (uint32_t)TB_DEL : LAZY, sbi);
      if (Sn > S) {  // fix-up 1
        S = Sn;
        cell = cell_set_s(cell, TB_YCLIP_SUFFIX);
      }
      if (act) {
        v.row(ROWS_SL, i) = S;
        v.row(ROWS_NL, i) = (int32_t)cell;
      }
      int32_t gv, gi;
      if (coop_argmax_first<W>(lane, act && S + xs > SmN, S, i, gv, gi, pk)) {  // S(i, n) is a real score
        SmN = gv + xs;
        LxN = m - gi;
        cmN = cell_set_s(cmN, TB_XCLIP_SUFFIX);
      }
      const int32_t left = m - 1 - base;
      c_above = (uint32_t)C::from((int32_t)sbi, left < W - 1 ? left : W - 1);
    }
  }
  if (Snm > SmN) {  // i == m
    SmN = Snm;
    cmN = cell_set_s(cmN, TB_YCLIP_SUFFIX);
  }
  C::sync();  // the rows arena as fix-up 1 left it is what fix-up 2 reads

  // ------------------------------------------------------------------ fix-up 2 (mod.rs:825-843), rows 1..m-1
  int32_t cSp;     // S'(i-1) for the chunk's first row
  uint32_t ccell;  // cell (i-1, n) after its own fix-up 2
  {
    int32_t S = s0;
    uint32_t cell = c0;
    if (ys > S) {
      S = ys;
      cell = cell_set_s(cell, TB_YCLIP_SUFFIX);
    }
    cSp = S;
    ccell = cell;
  }
  int32_t I_next, S2_next, c_next;
  {
    const int32_t i0 = imin32(1 + lane, m - 1);
    I_next = v.row(ROWS_IL, i0);
    S2_next = v.row(ROWS_SL, i0);
    c_next = v.row(ROWS_NL, i0);
  }
  for (int32_t base = 1; base < m; base += W) {
    const int32_t i = base + lane;
    const bool act = i < m;
    const int32_t ic = act ? i : m - 1;
    int32_t I = I_next, S = S2_next;
    uint32_t cell = (uint32_t)c_next;
    if (base + W < m) {
      const int32_t i1 = imin32(base + W + lane, m - 1);
      I_next = v.row(ROWS_IL, i1);
      S2_next = v.row(ROWS_SL, i1);
      c_next = v.row(ROWS_NL, i1);
    }
    // S'(i) - go*i = max(S'(i-1) - go*(i-1) ... ) : inclusive running maximum of S(k) - go*k, seeded by the carry
    // The first row a pass raises has an unraised row above it, so S(i-1) + go > S(i) holds there with the values
    // as loaded (the carry for the chunk's first row): when no lane sees that, the pass changes no S of the chunk
    // and the scan is skipped.
    int32_t Sprev = C::up(S, 1);
    if (lane == 0) Sprev = cSp;
    if (C::ballot(Sprev + go > S) != 0u) {
      int32_t t = S - go * ic;
      if (lane == 0) t = imax(t, cSp + go - go * ic);
      const int32_t Snew = coop_scan_max<W>(lane, t) + go * ic;  // S'(i)
      Sprev = C::up(Snew, 1);
      if (lane == 0) Sprev = cSp;
    }
    const int32_t s_score = Sprev + go;
    // cell (i-1) after its own pass: only its s_bits can have changed, to TB_INS
    const bool raised = s_score > S;
    uint32_t my_s_after = raised ? (uint32_t)TB_INS : cell_s(cell);
    uint32_t prev_s_after = (uint32_t)C::up((int32_t)my_s_after, 1);
    if (lane == 0) prev_s_after = cell_s(ccell);
    bool dirty = false;
    if (s_score > I) {
      I = s_score;
      cell = cell_set_i(cell, prev_s_after);
      dirty = true;
    }
    if (raised) {
      S = s_score;
      cell = cell_set_s(cell, TB_INS);
      dirty = true;
    }
    if (act && dirty) {
      v.row(ROWS_IL, i) = I;
      v.row(ROWS_SL, i) = S;
      v.row(ROWS_NL, i) = (int32_t)cell;
    }
    int32_t gv, gi;
    if (coop_argmax_first<W>(lane, act && raised && S + xs > SmN, S, i, gv, gi, pk)) {
      SmN = gv + xs;
      LxN = m - gi;
      cmN = cell_set_s(cmN, TB_XCLIP_SUFFIX);
    }
    const int32_t left = m - 1 - base;
    const int src = left < W - 1 ? left : W - 1;
    cSp = C::from(S, src);  // == S'(i) of the chunk's last row
    ccell = (uint32_t)C::from((int32_t)cell, src);
  }
  {  // i == m
    const int32_t s_score = cSp + go;
    if (s_score > ImN) {
      ImN = s_score;
      cmN = cell_set_i(cmN, cell_s(ccell));
    }
    if (s_score > SmN) {
      SmN = s_score;
      cmN = cell_set_s(cmN, TB_INS);
    }
  }
  C::sync();
  es.SmN = SmN;
  es.ImN = ImN;
  es.cmN = cmN;
  es.Snm = Snm;
  es.Lym = Lym;
  es.Lx0 = Lx0;
  es.LxN = LxN;
}

// touch the traceback words the walk is likely to read next (the diagonal below the current cell)
B2A_HD void prefetch_tb(const PairView& v, int32_t i, int32_t j) {
#if defined(__CUDA_ARCH__)
  if (i >= 1 && i <= v.m - 1 && j >= 1 && j <= v.n) {
    const int32_t GR = v.G * v.R;
    const int32_t s = (int32_t)(((uint64_t)(uint32_t)(i - 1) * v.mulGR) >> 40), rem = (i - 1) - s * GR;
    const int32_t l = (int32_t)(((uint64_t)(uint32_t)rem * v.mulR) >> 40), r = rem - l * v.R;
    const int32_t ln = v.g * v.G + l;
    const int32_t t = (j - 1) + l;
    const size_t word =
        ((((size_t)(v.sub * v.nstrips + s) * v.K + (t >> 3)) * v.TBW + (r >> 2)) * 32 + ln) * 4 + (r & 3);
    asm volatile("prefetch.global.L1 [%0];" ::"l"(v.tb + word));
  }
#else
  (void)v;
  (void)i;
  (void)j;
#endif
}

// K2 for one pair by W cooperating lanes; `out` is complete on lane 0
template <int W>
B2A_HD void walk_pair_coop(const int lane, const PairView& v, const bool filter_clips, uint8_t* ops_end, WalkOut& out) {
  using C = Coop<W>;
  EndState es;
  finish_matrix_coop<W>(lane, v, es);
  WalkState w;
  walk_begin(v, es, ops_end, w);
  constexpr int32_t kBurst = 24;  // moves of lane 0 between two rounds of prefetches
  for (;;) {
    // every lane looks a different distance down the diagonal from where lane 0 stands
    const int32_t ci = C::from(w.i, 0), cj = C::from(w.j, 0);
    prefetch_tb(v, ci - 1 - lane, cj - 1 - lane);
    int32_t done = 0;
    if (lane == 0) done = walk_run(v, es, filter_clips, w, kBurst) ? 1 : 0;
    if (C::from(done, 0)) break;
  }
  walk_finish(es, w, out);
}

// ---------------------------------------------------------------------------------------------------------
// Score-only K2 (b2a_score_batch): score, xend and yend without the interior traceback (K1 ran with F_NOTB).
// score is S(m, n) after the fix-ups, which finish_matrix_* compute from what K1 leaves without the traceback.
// xend / yend change only on TB_XCLIP_SUFFIX / TB_YCLIP_SUFFIX, and those codes live only in row m and column n;
// the walk's (i, j) never increases, so once it stands on a cell with i < m and j < n neither can change again.
// end_walk() is walk_run's state machine restricted to row m and column n: it stops at the first move that leaves
// them (a prefix clip included), BEFORE it resolves the next layer -- the two LAZY resolutions that read an interior
// nibble, INS out of row m and DEL out of column n, are such moves.  It flags the pair (status 1) on walk_run's
// conditions met on that stretch; a reference panic deeper inside the matrix is not seen (the pair keeps the
// fill's score and status 0).
struct EndOut {
  int32_t score;
  uint32_t xend, yend, status;
};

B2A_HD void end_walk(const PairView& v, const EndState& es, const bool filter_clips, EndOut& out) {
  const DevScoring& sc = v.sc;
  const int32_t m = v.m, n = v.n;
  const uint32_t cmN = es.cmN;
  auto get_cell_n = [&](int32_t i) -> uint32_t { return (i == m) ? cmN : (uint32_t)v.row(ROWS_NL, i); };
  auto get_s = [&](int32_t i, int32_t j) -> uint32_t {  // (i, j) in row m or column n (walk_run's order of cases)
    if (j == n) return cell_s(get_cell_n(i));
    if (i == 0) return row0_sbits(sc, j, n);  // m == 0: K2 keeps no row-m cells
    return cell_s((uint32_t)v.rowm[j * 32 + v.pi]);
  };
  int32_t i = m, j = n, guard = m + n + 8;
  uint32_t layer = cell_s(cmN), xend = (uint32_t)m, yend = (uint32_t)n, status = 0, nclip = 0;
  while (layer != TB_START) {
    if (--guard < 0) {
      status = 1;
      break;
    }
    uint32_t next = 0;
    bool lazy = true;  // the next layer is S of the cell the move lands on
    if (layer == TB_INS) {
      if (j == n) {
        next = cell_i(get_cell_n(i));
        lazy = false;
      } else {
        next = cell_i((uint32_t)v.rowm[j * 32 + v.pi]);  // i == m
        lazy = next == LAZY;
      }
      i -= 1;
    } else if (layer == TB_DEL) {
      if (i == 0 || i == m) {
        next = (i == 0) ? row0_dbits(sc, j) : cell_d((uint32_t)v.rowm[j * 32 + v.pi]);
        lazy = false;
      } else {
        next = cell_d(get_cell_n(i));  // j == n
        lazy = next == LAZY;
      }
      j -= 1;
    } else if (layer == TB_MATCH || layer == TB_SUBST) {
      i -= 1;
      j -= 1;
    } else if (layer == TB_XCLIP_PREFIX) {
      if (!filter_clips) ++nclip;
      i = 0;
    } else if (layer == TB_XCLIP_SUFFIX) {
      int32_t lx;
      if (j == n) lx = es.LxN;
      else if (j == 0) lx = es.Lx0;
      else lx = (m >= 2) ? m - decode_boundary(v.load_bnd(j), v.packtrk != 0, sc.xclip_suffix, m).Ti : 0;
      if (!filter_clips) ++nclip;
      i -= lx;
      xend = (uint32_t)i;
    } else if (layer == TB_YCLIP_PREFIX) {
      if (!filter_clips) ++nclip;
      j = 0;
    } else if (layer == TB_YCLIP_SUFFIX) {
      int32_t ly;
      if (i == m) ly = es.Lym;
      else if (i == 0 || n == 0) ly = n;
      else ly = n - v.row(ROWS_LY, i);
      if (!filter_clips) ++nclip;
      j -= ly;
      yend = (uint32_t)j;
    } else {
      status = 1;  // panic!("Dint expect this!") mod.rs:905
      break;
    }
    if (i < 0 || j < 0) {
      status = 1;
      break;
    }
    if (i != m && j != n) break;  // left row m and column n: xend and yend are final
    layer = lazy ? get_s(i, j) : next;
  }
  if (nclip > 4) status = 1;  // walk_finish: a lower bound of the full walk's clip count
  out.score = es.SmN;
  out.xend = xend;
  out.yend = yend;
  out.status = status;
  if (status) {  // as walk_lane reports a pair the reference panics on
    out.score = MIN_SCORE;
    out.xend = out.yend = 0;
  }
}

#if defined(__CUDACC__)

// the view K2 has of pair `pi` of a block
__device__ __forceinline__ PairView pair_view(const WalkParams& prm, const Block& blk, const int pi) {
  const uint32_t sp = blk.first + pi;
  const int32_t P = 32 / prm.G;
  PairView v;
  v.sc = prm.sc;
  v.lut = prm.lut;
  v.P = P;
  v.m = (int32_t)prm.pm[sp];
  v.n = (int32_t)prm.pn[sp];
  v.pi = pi;
  v.set_shape(prm.G, prm.R);
  v.nstrips = (int32_t)blk.nstrips;
  v.K = (int32_t)blk.K;
  v.sub = pi / P;
  v.g = pi % P;
  v.packtrk = prm.packtrk;
  v.maxn = (int32_t)blk.maxn;
  v.bnd_base = bnd_index(prm.G, 0, pi, v.maxn);
  v.bnd_stride = (int32_t)(bnd_index(prm.G, 1, pi, v.maxn) - v.bnd_base);
  const uint32_t* seqw = reinterpret_cast<const uint32_t*>(prm.seq + blk.seq_off);
  v.xw = seqw + (size_t)v.sub * blk.xwords * P + v.g;
  v.yw = seqw + (size_t)prm.G * blk.xwords * P + (size_t)v.sub * blk.ywords * P + v.g;
  v.bnd = reinterpret_cast<const int4*>(prm.bnd + blk.bnd_off);
  v.rows = reinterpret_cast<int32_t*>(prm.rows + blk.rows_off);
  v.rows_pad = (int32_t)blk.rows_pad;
  v.rowm = reinterpret_cast<uint16_t*>(prm.rowm + blk.rowm_off);
  v.tb = reinterpret_cast<const uint32_t*>(prm.tb + blk.tb_off);
  return v;
}

// K2 for one pair (lane) of a block
__device__ __forceinline__ void walk_lane(const WalkParams& prm, const Block& blk, const int lane) {
  if ((uint32_t)lane >= blk.npairs) return;
  const uint32_t sp = blk.first + lane;
  const PairView v = pair_view(prm, blk, lane);
  const uint32_t cap = blk.maxm + blk.maxn + 4;
  uint8_t* ops_end = prm.ops_scratch + blk.ops_off + (size_t)(lane + 1) * cap;
  WalkOut o;
  walk_pair(v, prm.filter_clips != 0, ops_end, o);
  if (o.status) {  // the reference panics on this pair (mod.rs:905): no alignment is reported for it
    o.score = MIN_SCORE;
    o.n_ops = 0;
    o.xstart = o.xend = o.ystart = o.yend = 0;
    o.clip[0] = o.clip[1] = o.clip[2] = o.clip[3] = 0;
  }
  const uint32_t dst = prm.order[sp];
  prm.score[dst] = o.score;
  prm.xstart[dst] = o.xstart;
  prm.xend[dst] = o.xend;
  prm.ystart[dst] = o.ystart;
  prm.yend[dst] = o.yend;
  prm.n_ops[dst] = o.n_ops;
  prm.ops_src[dst] = blk.ops_off + (uint64_t)(lane + 1) * cap - o.n_ops;
  prm.status[dst] = o.status;
  if (o.status) atomicOr(prm.err_flag, 1u);
#pragma unroll
  for (int k = 0; k < 4; ++k) prm.clip_len[4 * (size_t)dst + k] = o.clip[k];
}

// K2, one warp per pair
// the pair's x and y copied into this warp's slice of the CTA's dynamic shared memory (x bytes, then y bytes)
__device__ __forceinline__ void stage_pair_seqs(PairView& v, const Block& blk, const int lane, uint8_t* seq_smem) {
  const int32_t P = v.P;
  const int32_t xwn = (v.m + 3) >> 2, ywn = (v.n + 3) >> 2;
  uint32_t* xs = reinterpret_cast<uint32_t*>(seq_smem);
  uint32_t* ys = xs + ((blk.maxm + 3) >> 2);
  for (int32_t w = lane; w < xwn; w += 32) xs[w] = v.xw[(size_t)w * P];
  for (int32_t w = lane; w < ywn; w += 32) ys[w] = v.yw[(size_t)w * P];
  __syncwarp();
  v.xs8 = reinterpret_cast<const uint8_t*>(xs);
  v.ys8 = reinterpret_cast<const uint8_t*>(ys);
}

__device__ __forceinline__ void walk_warp(const WalkParams& prm, const Block& blk, const int pi, const int lane,
                                          uint8_t* seq_smem) {
  const uint32_t sp = blk.first + pi;
  PairView v = pair_view(prm, blk, pi);
  if (seq_smem) stage_pair_seqs(v, blk, lane, seq_smem);
  const uint32_t cap = blk.maxm + blk.maxn + 4;
  uint8_t* ops_end = prm.ops_scratch + blk.ops_off + (size_t)(pi + 1) * cap;
  WalkOut o;
  walk_pair_coop<32>(lane, v, prm.filter_clips != 0, ops_end, o);
  if (lane != 0) return;
  if (o.status) {  // the reference panics on this pair (mod.rs:905): no alignment is reported for it
    o.score = MIN_SCORE;
    o.n_ops = 0;
    o.xstart = o.xend = o.ystart = o.yend = 0;
    o.clip[0] = o.clip[1] = o.clip[2] = o.clip[3] = 0;
  }
  const uint32_t dst = prm.order[sp];
  prm.score[dst] = o.score;
  prm.xstart[dst] = o.xstart;
  prm.xend[dst] = o.xend;
  prm.ystart[dst] = o.ystart;
  prm.yend[dst] = o.yend;
  prm.n_ops[dst] = o.n_ops;
  prm.ops_src[dst] = blk.ops_off + (uint64_t)(pi + 1) * cap - o.n_ops;
  prm.status[dst] = o.status;
  if (o.status) atomicOr(prm.err_flag, 1u);
#pragma unroll
  for (int k = 0; k < 4; ++k) prm.clip_len[4 * (size_t)dst + k] = o.clip[k];
}

__device__ __forceinline__ void score_store(const WalkParams& prm, const uint32_t sp, const EndOut& o) {
  const uint32_t dst = prm.order[sp];
  prm.score[dst] = o.score;
  prm.xend[dst] = o.xend;
  prm.yend[dst] = o.yend;
  prm.status[dst] = o.status;
  if (o.status) atomicOr(prm.err_flag, 1u);
}

// score-only K2 for one pair (lane) of a block: row m and the fix-ups, then the end walk
__device__ __forceinline__ void score_lane(const WalkParams& prm, const Block& blk, const int lane) {
  if ((uint32_t)lane >= blk.npairs) return;
  const PairView v = pair_view(prm, blk, lane);
  EndState es;
  finish_matrix_seq(v, es);
  EndOut o;
  end_walk(v, es, prm.filter_clips != 0, o);
  score_store(prm, blk.first + lane, o);
}

// score-only K2, one warp per pair: the cooperative row m and fix-ups, then lane 0's end walk
__device__ __forceinline__ void score_warp(const WalkParams& prm, const Block& blk, const int pi, const int lane,
                                           uint8_t* seq_smem) {
  PairView v = pair_view(prm, blk, pi);
  if (seq_smem) stage_pair_seqs(v, blk, lane, seq_smem);
  EndState es;
  finish_matrix_coop<32>(lane, v, es);
  if (lane != 0) return;
  EndOut o;
  end_walk(v, es, prm.filter_clips != 0, o);
  score_store(prm, blk.first + pi, o);
}

#if defined(B2A_DEFINE_WALK_KERNEL)  // one translation unit (b2a_engine.cu) owns the stand-alone kernel
__global__ void __launch_bounds__(1024, 1) walk_warp_kernel(const WalkParams prm) {  // 64 registers; CTAs of 1..32 warps
  extern __shared__ __align__(16) uint8_t walk_smem[];  // seq_smem_per_warp bytes per warp, or none
  const uint32_t gw = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;  // one warp per (block, pair)
  const int lane = threadIdx.x & 31;
  const uint32_t b = gw >> 5, pi = gw & 31u;
  if (b >= prm.nblocks) return;
  const Block blk = prm.blocks[b];
  if (pi >= blk.npairs) return;
  uint8_t* mine = prm.seq_smem_per_warp ? walk_smem + (size_t)(threadIdx.x >> 5) * prm.seq_smem_per_warp : nullptr;
  walk_warp(prm, blk, (int)pi, lane, mine);
}

__global__ void __launch_bounds__(128, 8) walk_kernel(const WalkParams prm) {
  const uint32_t gw = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (gw >= prm.nblocks) return;
  const Block blk = prm.blocks[gw];
  walk_lane(prm, blk, lane);
}

// score-only K2 in the two forms of walk_warp_kernel / walk_kernel
__global__ void __launch_bounds__(1024, 1) score_warp_kernel(const WalkParams prm) {
  extern __shared__ __align__(16) uint8_t walk_smem[];
  const uint32_t gw = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  const uint32_t b = gw >> 5, pi = gw & 31u;
  if (b >= prm.nblocks) return;
  const Block blk = prm.blocks[b];
  if (pi >= blk.npairs) return;
  uint8_t* mine = prm.seq_smem_per_warp ? walk_smem + (size_t)(threadIdx.x >> 5) * prm.seq_smem_per_warp : nullptr;
  score_warp(prm, blk, (int)pi, lane, mine);
}

__global__ void __launch_bounds__(128, 8) score_kernel(const WalkParams prm) {
  const uint32_t gw = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (gw >= prm.nblocks) return;
  const Block blk = prm.blocks[gw];
  score_lane(prm, blk, lane);
}
#endif

#endif

}  // namespace b2a

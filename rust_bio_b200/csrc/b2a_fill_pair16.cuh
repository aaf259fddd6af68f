// K1, pair-packed: the thread-per-pair local fill (shape 1x16, flags F_LUT | F_TRACK_ROWS | F_TRACK_COLS |
// F_CLIPX | F_PACKTRK | F_RELU) with every register holding TWO pairs as int16x2.
//
// Lane t of a warp-task owns pair t of 32-pair block A (low halves) and pair t of block B (high halves), so one
// 16x2 DPX instruction (VIADDMNMX.S16x2, VIMNMX3.S16x2, VIMNMX.U16x2, ...) does the work of two int32 cells.  The
// cell is column_step's cell (b2a_fill.cuh) in the same packed score domain (4*value + 2-bit priority, same tie
// order), moved by a bias so that every live value is a small non-negative 16-bit number:
//   stored = 4*value + code + bias,   bias = 4*max(-gap_open, -min substitution score, 0)
// The engine takes this path only when the whole wave is one shape with m <= 256, n <= 255, at most 7 symbols and
// a best score of at most 255 (b2a_engine.cu pair16_eligible): then every stored value lies in [0, 16384).
//
// Two kinds of arithmetic are exact per half:
//  * DPX 16x2 instructions (no carry crosses bit 16 by construction);
//  * plain 32-bit IADD/IMAD on registers whose halves are non-negative, provided the low half's TRUE result lies in
//    [0, 65536): a register with halves (h, l) is the integer h*65536 + l, a ring expression of such integers is
//    (expr of the h's)*65536 + (expr of the l's), so the low half is exact and the high half is exact mod 2^16.
//    Constants are added as c*0x10001 (c*65536 + c) for that reason.
// The substitution comes from a JOINT LUT in shared memory: one 32-bit word per (x_A, x_B, y_A, y_B) holds both
// pairs' scaled scores, so one LDS serves two cells; row x's offset is kept in xc[r] as in the int32 kernel, the
// column adds (y_A * alpha + y_B) * 4.  Its last (alpha+1)^2 - alpha^2 rows are the poison rows of padded rows.
//
// What leaves the kernel is exactly what fill_kernel<1,16,63> writes, for both blocks: the 4-bit traceback words
// (two 16-bit accumulators per row, 4 columns each, joined by one PRMT per pair at each 8-column flush), the rows
// arena (row trackers, row-m inputs) and the int32 boundary row m-1 that K2 decodes.  Between strips the boundary
// row travels as one 16-byte word per column for BOTH pairs {S, I, column-tracker key} (16x2 each), written in place
// into block A's boundary arena: half the bytes of the int32 form.  The last strip reads column j+1 of it before it
// writes the int32 column j over it, so the two forms never collide.
#pragma once
#include "b2a_fill.cuh"

namespace b2a {

// ---- 16x2 helpers: one DPX / integer instruction on the device, exact per-half arithmetic on the host ----------
B2A_HD int32_t p16_lo(uint32_t v) { return (int32_t)(int16_t)(uint16_t)(v & 0xffffu); }
B2A_HD int32_t p16_hi(uint32_t v) { return (int32_t)(int16_t)(uint16_t)(v >> 16); }
B2A_HD uint32_t p16_pack(int32_t lo, int32_t hi) { return ((uint32_t)hi << 16) | ((uint32_t)lo & 0xffffu); }
B2A_HD uint32_t p16_splat(int32_t v) { return p16_pack(v, v); }

// max(a + b, c) per signed half
B2A_HD uint32_t p16_addmax(uint32_t a, uint32_t b, uint32_t c) {
#if defined(__CUDA_ARCH__)
  return __viaddmax_s16x2(a, b, c);
#else
  return p16_pack(imax(p16_lo(a) + p16_lo(b), p16_lo(c)), imax(p16_hi(a) + p16_hi(b), p16_hi(c)));
#endif
}
// min(a + b, c) per signed half
B2A_HD uint32_t p16_addmin(uint32_t a, uint32_t b, uint32_t c) {
#if defined(__CUDA_ARCH__)
  return __viaddmin_s16x2(a, b, c);
#else
  const int32_t l = p16_lo(a) + p16_lo(b), h = p16_hi(a) + p16_hi(b);
  return p16_pack(l < p16_lo(c) ? l : p16_lo(c), h < p16_hi(c) ? h : p16_hi(c));
#endif
}
// max(a, b, c) per signed half
B2A_HD uint32_t p16_max3(uint32_t a, uint32_t b, uint32_t c) {
#if defined(__CUDA_ARCH__)
  return __vimax3_s16x2(a, b, c);
#else
  return p16_pack(imax(p16_lo(a), imax(p16_lo(b), p16_lo(c))), imax(p16_hi(a), imax(p16_hi(b), p16_hi(c))));
#endif
}
// max(a, b) / max(a, b, c) per unsigned half (the tracker keys)
B2A_HD uint32_t p16_umax(uint32_t a, uint32_t b) {
#if defined(__CUDA_ARCH__)
  return __vmaxu2(a, b);
#else
  const uint32_t l = (a & 0xffffu) > (b & 0xffffu) ? (a & 0xffffu) : (b & 0xffffu);
  const uint32_t h = (a >> 16) > (b >> 16) ? (a >> 16) : (b >> 16);
  return (h << 16) | l;
#endif
}
B2A_HD uint32_t p16_umax3(uint32_t a, uint32_t b, uint32_t c) {
#if defined(__CUDA_ARCH__)
  return __vimax3_u16x2(a, b, c);
#else
  return p16_umax(a, p16_umax(b, c));
#endif
}
B2A_HD uint32_t byte_perm(uint32_t x, uint32_t y, uint32_t s) {
#if defined(__CUDA_ARCH__)
  return __byte_perm(x, y, s);
#else
  const uint64_t v = ((uint64_t)y << 32) | x;
  uint32_t r = 0;
  for (int k = 0; k < 4; ++k) r |= (uint32_t)((v >> (8 * ((s >> (4 * k)) & 7))) & 0xffu) << (8 * k);
  return r;
#endif
}
B2A_HD uint32_t ld_global_u32(const uint32_t* p) {
#if defined(__CUDA_ARCH__)
  return __ldg(p);
#else
  return *p;
#endif
}

// The flags the packed fill implements (C1/C2: local alignment with a compact alphabet)
constexpr int P16_FLAGS = F_LUT | F_TRACK_ROWS | F_TRACK_COLS | F_CLIPX | F_PACKTRK | F_RELU;
constexpr int P16_MAX_ALPHA = 7;

// joint LUT: ((alpha+1)^2 rows of (x_A, x_B)) x (alpha^2 columns of (y_A, y_B)) 32-bit words
#if defined(__CUDACC__)
__host__ __device__
#endif
constexpr int p16_lut_entries(int alpha) { return (alpha + 1) * (alpha + 1) * alpha * alpha; }
#if defined(__CUDACC__)
__host__ __device__
#endif
constexpr uint32_t p16_lut_smem_bytes(int alpha) { return ((uint32_t)p16_lut_entries(alpha) * 4u + 127u) & ~127u; }

// Joint LUT from K1's scaled int32 LUT (alpha rows of alpha entries, then the poison row): the word of
// (x_A, x_B, y_A, y_B) holds entry (x_A, y_A) in the low half and (x_B, y_B) in the high half.
inline void p16_build_lut(const int32_t* scaled, int alpha, int32_t* out) {
  const int a1 = alpha + 1, aa = alpha * alpha;
  for (int xa = 0; xa < a1; ++xa)
    for (int xb = 0; xb < a1; ++xb)
      for (int ya = 0; ya < alpha; ++ya)
        for (int yb = 0; yb < alpha; ++yb)
          out[(xa * a1 + xb) * aa + ya * alpha + yb] =
              (int32_t)p16_pack(scaled[xa * alpha + ya], scaled[xb * alpha + yb]);
}

// Per-lane view of one task: pair `lane` of block A and of block B.
struct P16Ctx {
  DevScoring sc;
  const int32_t* lut;     // joint LUT in shared memory (device) / host memory (sim)
  uint32_t lut_base;      // device: shared-space byte address of the LUT; host sim: 0
  const uint32_t* xa;     // x words [w][32] of block A (global memory: read once per strip)
  const uint32_t* xb;
  const uint32_t* ya;     // staged y words [w][32] of block A / B
  const uint32_t* yb;
  int32_t m, n;           // the wave's one shape
  int32_t nstrips, K, rows_pad, lane;
  bool has_b;             // false: the last block of an odd count; the high half repeats A and stores nothing
  int4* bnd_a;            // block bases (bnd_index(1, j, lane) = j*32 + lane)
  int4* bnd_b;
  int32_t* rows_a;
  int32_t* rows_b;
  uint4* tb_a;            // task bases: [strip][k][q][32]
  uint4* tb_b;
  int32_t one, mone;      // opaque 1 and -1 (kernel parameters): adds issue as IMAD on the FMA pipe
  int32_t k16;            // opaque 16
  int32_t ge4;            // 4 * gap_extend
  int32_t bias;
};

// one column of this lane's R rows (see column_step in b2a_fill.cuh for the cell it mirrors); NOTB: score-only
// (F_NOTB), no nibble accumulators -- column n's nibbles (the rows arena) are still computed
template <int R, bool MASKED, bool LAST, bool NOTB>
B2A_HD void p16_column(const P16Ctx& c, const int32_t j, const int32_t q4, const int32_t rowbase, const int32_t rv,
                       uint32_t (&Sp)[R], uint32_t (&Dp)[R], uint32_t (&SnR)[R], uint32_t (&acc)[R],
                       const int32_t (&xc)[R], const int32_t (&kcol)[R], const int32_t kmul, const uint32_t sdiag,
                       uint32_t& sup, uint32_t& iup, uint32_t& Tv, uint32_t& cap_s, uint32_t& cap_i) {
  const int32_t one = c.one, mone = c.mone, k2 = one + one, k64 = c.k16 * 4;
  const int32_t B = c.bias;
  const int32_t go4d = 4 * c.sc.gap_open + 1, go4i = 4 * c.sc.gap_open + 2;
  const uint32_t GE2 = p16_splat(c.ge4), FLOOR2 = p16_splat(B), FOUR2 = p16_splat(4);
  const int32_t GO4D2 = go4d * 0x10001, GO4I2 = go4i * 0x10001;  // plain adds: the results stay >= 1
  // row-tracker key 256*S + (255 - j) = 64*s4 + (255 - j) - 64*bias (s4 = 4*S + bias)
  const int32_t kj = (255 - j - 64 * B) * 0x10001;
  uint32_t Tl = 0, key_even = 0;  // 0: no key (real keys of rows <= 255 are > 0 or lose every tie)
  uint32_t sdo = (uint32_t)fmad((int32_t)sdiag, one, GO4D2);  // diagonal S, open-biased
  uint32_t iop = (uint32_t)fmad((int32_t)sup, one, GO4I2);
#pragma unroll
  for (int r = 0; r < R; ++r) {
    const uint32_t sub = (uint32_t)lut_at(c.lut, (uint32_t)fmad(q4, one, xc[r]));
    const uint32_t dop = Sp[r];  // S of this row in the previous column + open, biased
    const uint32_t i4 = p16_addmax(iup, GE2, iop);
    const uint32_t d4 = p16_addmax(Dp[r], GE2, dop);
    // S = first strict maximum of M, I, D, the zero floor (code 0); M = diagonal + substitution, fused
    const uint32_t sP = p16_addmax(sdo, sub, p16_max3(i4, d4, FLOOR2));
    const uint32_t s4 = sP & 0xfffcfffcu;
    // ext flags: min(I4 - open, 4), min(D4 - open, 4) as min(open + 4, X4) - open; nibble =
    // code + iext*4 + dext*8 = (sP - s4) + (fi - iop) + 2*(fd - dop), exact per half (see the header)
    int32_t fsum = 0, osum = 0, code = 0;
    if (!NOTB || LAST) {
      const uint32_t fi = p16_addmin(iop, FOUR2, i4), fd = p16_addmin(dop, FOUR2, d4);
      fsum = fmad((int32_t)fd, k2, (int32_t)fi);
      osum = fmad((int32_t)dop, k2, (int32_t)iop);
      code = fmad((int32_t)s4, mone, (int32_t)sP);
    }
    if (!NOTB) {
      int32_t a = fmad((int32_t)acc[r], kmul, fsum);
      a = fmad(osum, mone, a);
      acc[r] = (uint32_t)fmad(code, one, a);
    }
    // column tracker: local key 256*S + (255 - r), two rows per 3-input max
    const uint32_t key = (uint32_t)fmad((int32_t)s4, k64, kcol[r]);
    if (r & 1) Tl = p16_umax3(Tl, key_even, key);
    else key_even = key;
    if (R & 1) {
      if (r == R - 1) Tl = p16_umax(Tl, key);
    }
    SnR[r] = p16_umax(SnR[r], (uint32_t)fmad((int32_t)s4, k64, kj));
    if (LAST) {  // row-m inputs of K2 (column n): S, I and the nibble of every row, both pairs
      const int32_t nib = fmad(osum, mone, fmad(code, one, fsum));
      const int32_t slot = (rowbase + 1 + r) * 32 + c.lane;
      c.rows_a[ROWS_SL * c.rows_pad * 32 + slot] = (p16_lo(s4) - B) >> 2;
      c.rows_a[ROWS_IL * c.rows_pad * 32 + slot] = (p16_lo(i4) - B) >> 2;
      c.rows_a[ROWS_NL * c.rows_pad * 32 + slot] = p16_lo((uint32_t)nib);
      if (c.has_b) {
        c.rows_b[ROWS_SL * c.rows_pad * 32 + slot] = (p16_hi(s4) - B) >> 2;
        c.rows_b[ROWS_IL * c.rows_pad * 32 + slot] = (p16_hi(i4) - B) >> 2;
        c.rows_b[ROWS_NL * c.rows_pad * 32 + slot] = p16_hi((uint32_t)nib);
      }
    }
    if (MASKED) {
      if (r == rv - 1) {
        cap_s = s4;
        cap_i = i4;
      }
    }
    sdo = dop;
    Sp[r] = (uint32_t)fmad((int32_t)s4, one, GO4D2);
    iop = (uint32_t)fmad((int32_t)s4, one, GO4I2);
    Dp[r] = d4;
    iup = i4;
    sup = s4;
  }
  // local row index -> global: (255 - r) - rowbase = 256 - i
  Tv = p16_umax(Tv, (uint32_t)fmad(rowbase, mone * 0x10001, (int32_t)Tl));
}

// 16-bit column-tracker key (256*S + 256 - i) -> K1's int32 key (4096*S + 4095 - i)
B2A_HD int32_t p16_key32(uint32_t k16) { return (int32_t)((k16 >> 8) << 12) + 3839 + (int32_t)(k16 & 255u); }

// One strip (rows s*R+1 .. (s+1)*R) of this lane's two pairs.
template <int R, bool MASKED, bool NOTB>
B2A_HD void p16_strip(const P16Ctx& c, const int32_t s) {
  constexpr int TBW = tbw_of(R);
  const int32_t m = c.m, n = c.n, alpha = c.sc.alpha, B = c.bias;
  const int32_t rowbase = s * R;
  int32_t rv = m - 1 - rowbase;
  rv = rv < 0 ? 0 : (rv > R ? R : rv);
  const bool final_strip = s == c.nstrips - 1;
  const int32_t go4d = 4 * c.sc.gap_open + 1;
  const int32_t row_words = alpha * alpha * 4;  // bytes per joint LUT row

  uint32_t Sp[R], Dp[R], SnR[R], acc[R], acc_hi[R];
  int32_t xc[R], kcol[R];
#pragma unroll
  for (int w = 0; w < R / 4; ++w) {
    const uint32_t wa = ld_global_u32(c.xa + (size_t)(rowbase / 4 + w) * 32);
    const uint32_t wb = c.has_b ? ld_global_u32(c.xb + (size_t)(rowbase / 4 + w) * 32) : wa;
#pragma unroll
    for (int b = 0; b < 4; ++b) {
      uint32_t sa = (wa >> (8 * b)) & 0xffu, sb = (wb >> (8 * b)) & 0xffu;
      sa = sa < (uint32_t)alpha ? sa : (uint32_t)alpha - 1;  // K0 has flagged any symbol outside the alphabet
      sb = sb < (uint32_t)alpha ? sb : (uint32_t)alpha - 1;
      int32_t rx = (int32_t)(sa * (alpha + 1) + sb);
      if (MASKED && w * 4 + b >= rv) rx = alpha * (alpha + 1) + alpha;  // padded rows: poison for both pairs
      xc[w * 4 + b] = (int32_t)c.lut_base + rx * row_words;
    }
  }
#pragma unroll
  for (int r = 0; r < R; ++r) {
    const int32_t s0 = col0_S(c.sc, rowbase + 1 + r);  // >= 0 with the local clips
    Sp[r] = p16_splat(4 * s0 + go4d + B);
    Dp[r] = 0;  // "no D yet": below every real D (>= 1 stored)
    SnR[r] = p16_splat(256 * s0 + 255);  // column 0 (mod.rs:667-670)
    acc[r] = 0;
    acc_hi[r] = 0;
    kcol[r] = (255 - r - 64 * B) * 0x10001;
  }
  uint32_t sup_prev = p16_splat(4 * (rowbase == 0 ? 0 : col0_S(c.sc, rowbase)) + B);
  uint32_t in_s = 0, in_i = 0, in_t = 0;
  uint4 pre = {0u, 0u, 0u, 0u};
  uint4* bnd16 = reinterpret_cast<uint4*>(c.bnd_a);
  if (s > 0 && n >= 1) pre = bnd16[1 * 32 + c.lane];
  uint32_t cap_s = 0, cap_i = 0, ywa = 0, ywb = 0;
  const int32_t nsteps = c.K * 8;
  const int32_t k16 = c.k16;
  for (int32_t t = 0; t < nsteps; ++t) {
    const int32_t j = t + 1;
    const int32_t kmul = (t & 3) ? k16 : 0;  // a fresh accumulator every four columns
    if (j <= n) {
      if ((t & 3) == 0) {
        ywa = c.ya[(t >> 2) * 32 + c.lane];
        ywb = c.has_b ? c.yb[(t >> 2) * 32 + c.lane] : ywa;
      }
      uint32_t qa = ywa & 0xffu, qb = ywb & 0xffu;
      ywa >>= 8;
      ywb >>= 8;
      qa = qa < (uint32_t)alpha ? qa : (uint32_t)alpha - 1;
      qb = qb < (uint32_t)alpha ? qb : (uint32_t)alpha - 1;
      const int32_t q4 = (int32_t)(qa * alpha + qb) * 4;
      if (s == 0) {
        in_s = p16_splat(4 * row0_S(c.sc, j, n) + B);
        in_i = 0;
        in_t = 0;
      } else {
        in_s = pre.x;
        in_i = pre.y;
        in_t = pre.z;
        if (j < n) pre = bnd16[(j + 1) * 32 + c.lane];  // read before column j is overwritten below
      }
      uint32_t sup = in_s, iup = in_i, Tv = in_t;
      if (j == n) {
        p16_column<R, MASKED, true, NOTB>(c, j, q4, rowbase, rv, Sp, Dp, SnR, acc, xc, kcol, kmul, sup_prev, sup, iup, Tv,
                                    cap_s, cap_i);
      } else {
        p16_column<R, MASKED, false, NOTB>(c, j, q4, rowbase, rv, Sp, Dp, SnR, acc, xc, kcol, kmul, sup_prev, sup, iup, Tv,
                                     cap_s, cap_i);
      }
      sup_prev = in_s;
      if (rv >= 1) {
        const uint32_t os = (MASKED && rv < R) ? cap_s : sup;  // row m-1 (a full strip: its bottom row)
        const uint32_t oi = (MASKED && rv < R) ? cap_i : iup;
        if (final_strip) {  // K2's int32 boundary row (decode_boundary), both blocks
          c.bnd_a[j * 32 + c.lane] = make_int4(p16_lo(os) - B, p16_lo(oi) - B, p16_key32(Tv & 0xffffu), m);
          if (c.has_b) c.bnd_b[j * 32 + c.lane] = make_int4(p16_hi(os) - B, p16_hi(oi) - B, p16_key32(Tv >> 16), m);
        } else {
          uint4 o;
          o.x = os;
          o.y = oi;
          o.z = Tv;
          o.w = 0;
          bnd16[j * 32 + c.lane] = o;
        }
      }
      in_s = sup;
      in_i = iup;
      in_t = Tv;
    } else if (!NOTB) {
#pragma unroll
      for (int r = 0; r < R; ++r) acc[r] = (uint32_t)fmad((int32_t)acc[r], kmul, 0);
    }
    if (!NOTB && (t & 7) == 3) {
#pragma unroll
      for (int r = 0; r < R; ++r) acc_hi[r] = acc[r];  // columns 0-3 of the group: the word's top 16 bits
    } else if (!NOTB && (t & 7) == 7) {
      uint4* da = c.tb_a + (size_t)s * c.K * TBW * 32 + (size_t)(t >> 3) * TBW * 32 + c.lane;
      uint4* db = c.tb_b + (size_t)s * c.K * TBW * 32 + (size_t)(t >> 3) * TBW * 32 + c.lane;
#pragma unroll
      for (int qd = 0; qd < TBW; ++qd) {
        uint32_t wa[4], wb[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          const int r = qd * 4 + k;
          wa[k] = r < R ? byte_perm(acc[r], acc_hi[r], 0x5410) : 0u;
          wb[k] = r < R ? byte_perm(acc[r], acc_hi[r], 0x7632) : 0u;
        }
        da[qd * 32] = uint4{wa[0], wa[1], wa[2], wa[3]};
        if (c.has_b) db[qd * 32] = uint4{wb[0], wb[1], wb[2], wb[3]};
      }
    }
  }
  // row trackers: 256*S + (255 - j) -> (S + yclip_suffix, j), as the int32 kernel writes them
  const int32_t ys = c.sc.yclip_suffix;
#pragma unroll
  for (int r = 0; r < R; ++r) {
    const int32_t slot = (rowbase + 1 + r) * 32 + c.lane;
    const uint32_t ka = SnR[r] & 0xffffu, kb = SnR[r] >> 16;
    c.rows_a[ROWS_SN * c.rows_pad * 32 + slot] = (int32_t)(ka >> 8) + ys;
    c.rows_a[ROWS_LY * c.rows_pad * 32 + slot] = 255 - (int32_t)(ka & 255u);
    if (c.has_b) {
      c.rows_b[ROWS_SN * c.rows_pad * 32 + slot] = (int32_t)(kb >> 8) + ys;
      c.rows_b[ROWS_LY * c.rows_pad * 32 + slot] = 255 - (int32_t)(kb & 255u);
    }
  }
}

template <int R, bool NOTB = false>
B2A_HD void p16_fill_lane(const P16Ctx& c) {
  for (int32_t s = 0; s < c.nstrips; ++s) {
    if ((s + 1) * R <= c.m - 1) p16_strip<R, false, NOTB>(c, s);
    else p16_strip<R, true, NOTB>(c, s);
  }
}

#if defined(__CUDACC__)

// Persistent kernel: a warp-task is a pair of blocks (2k, 2k+1) of the wave; y of both is staged by bulk copy,
// x is read from global memory once per strip.
template <int R, bool NOTB>
__global__ void __launch_bounds__(128, B2A_MINB) fill_pair16_kernel(const FillParams prm, const int32_t bias) {
  extern __shared__ __align__(128) uint8_t smem[];
  constexpr int WARPS = 4;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem);
  int32_t* lut_s = reinterpret_cast<int32_t*>(smem + 64);
  const uint32_t lut_bytes = p16_lut_smem_bytes(prm.sc.alpha);
  uint8_t* stage = smem + 64 + lut_bytes + (size_t)warp * prm.smem_seq_bytes;
  uint64_t* bar = &bars[warp];
  if (threadIdx.x < WARPS) mbar_init(&bars[threadIdx.x], 1);
  for (int k = threadIdx.x; k < p16_lut_entries(prm.sc.alpha); k += blockDim.x) lut_s[k] = prm.lut[k];
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  __syncthreads();

  const uint32_t ntasks = (prm.nblocks + 1) / 2;
  uint32_t parity = 0;
  for (uint32_t done = 0; prm.task_limit == 0 || done < prm.task_limit; ++done) {
    uint32_t task = 0;
    if (lane == 0) task = atomicAdd(prm.task_counter, 1u);
    task = __shfl_sync(0xffffffffu, task, 0);
    if (task >= ntasks) break;
    const uint32_t ba = 2 * task;
    const bool has_b = ba + 1 < prm.nblocks;
    const Block blk = prm.blocks[ba];
    const Block blkb = prm.blocks[has_b ? ba + 1 : ba];
    const uint32_t xbytes = blk.xwords * 32 * 4, ybytes = blk.ywords * 32 * 4;
    if (lane == 0) {
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
      mbar_expect_tx(bar, 2 * ybytes);
      tma_bulk_g2s(stage, prm.seq + blk.seq_off + xbytes, ybytes, bar);
      tma_bulk_g2s(stage + ybytes, prm.seq + blkb.seq_off + xbytes, ybytes, bar);
    }
    P16Ctx c;
    c.sc = prm.sc;
    c.lut = lut_s;
    c.lut_base = smem_u32(lut_s);
    c.xa = reinterpret_cast<const uint32_t*>(prm.seq + blk.seq_off) + lane;
    c.xb = reinterpret_cast<const uint32_t*>(prm.seq + blkb.seq_off) + lane;
    c.ya = reinterpret_cast<const uint32_t*>(stage);
    c.yb = reinterpret_cast<const uint32_t*>(stage + ybytes);
    c.m = (int32_t)blk.maxm;
    c.n = (int32_t)blk.maxn;
    c.nstrips = (int32_t)blk.nstrips;
    c.K = (int32_t)blk.K;
    c.rows_pad = (int32_t)blk.rows_pad;
    c.lane = lane;
    c.has_b = has_b;
    c.bnd_a = reinterpret_cast<int4*>(prm.bnd + blk.bnd_off);
    c.bnd_b = reinterpret_cast<int4*>(prm.bnd + blkb.bnd_off);
    c.rows_a = reinterpret_cast<int32_t*>(prm.rows + blk.rows_off);
    c.rows_b = reinterpret_cast<int32_t*>(prm.rows + blkb.rows_off);
    c.tb_a = reinterpret_cast<uint4*>(prm.tb + blk.tb_off);
    c.tb_b = reinterpret_cast<uint4*>(prm.tb + blkb.tb_off);
    c.one = prm.one;
    c.mone = -prm.one;
    c.k16 = 16 * prm.one;
    c.ge4 = prm.ge4;
    c.bias = bias;
    while (!mbar_try_wait(bar, parity)) {
    }
    parity ^= 1u;
    p16_fill_lane<R, NOTB>(c);
    __syncwarp();
  }
}

#endif  // __CUDACC__

}  // namespace b2a

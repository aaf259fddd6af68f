// CPU harness for the score-only path (b2a_score_batch): the K1 fill with F_NOTB and the score-only K2 epilogue
// (finish_matrix_* + end_walk, b2a_walk.cuh) compiled for the host.  It stages a batch as K0 does, fills it twice --
// with the traceback and score-only, from the same scratch garbage -- and counts the bytes of the boundary and
// rows arenas that differ (none may).  It then runs the score-only epilogue on the score-only fill's scratch (the
// traceback arena is never given to it), in the lane-per-pair or the warp-per-pair form.
#include "b2a_sim.cpp"

namespace {

template <int G, int R, bool PIPED>
void fill_dispatch_notb(int flags, const Plan& p, const Block& blk, const DevScoring& sc, const int32_t* lut,
                        std::vector<uint8_t>& seq, std::vector<uint8_t>& bnd, std::vector<uint8_t>& rows,
                        std::vector<uint8_t>& tb) {
  constexpr int ALL = F_TRACK_ROWS | F_TRACK_COLS | F_CLIPX;
#define SIM_NOTB_CASE(F)                                                                              \
  case (F):                                                                                           \
    if constexpr (PIPED) fill_block_piped<R, (F) | F_NOTB>(p, blk, sc, lut, seq, bnd, rows, tb);      \
    else fill_block<G, R, (F) | F_NOTB>(p, blk, sc, lut, seq, bnd, rows, tb);                         \
    break;
  switch (flags) {
    SIM_NOTB_CASE(0)
    SIM_NOTB_CASE(F_TRACK_ROWS)
    SIM_NOTB_CASE(F_TRACK_ROWS | F_PACKTRK)
    SIM_NOTB_CASE(ALL)
    SIM_NOTB_CASE(ALL | F_PACKTRK)
    SIM_NOTB_CASE(F_LUT)
    SIM_NOTB_CASE(F_LUT | F_TRACK_ROWS)
    SIM_NOTB_CASE(F_LUT | F_TRACK_ROWS | F_PACKTRK)
    SIM_NOTB_CASE(F_LUT | ALL)
    SIM_NOTB_CASE(F_LUT | ALL | F_PACKTRK)
    SIM_NOTB_CASE(ALL | F_RELU)
    SIM_NOTB_CASE(ALL | F_PACKTRK | F_RELU)
    SIM_NOTB_CASE(F_LUT | ALL | F_RELU)
    SIM_NOTB_CASE(F_LUT | ALL | F_PACKTRK | F_RELU)
    SIM_NOTB_CASE(F_TRACK_ROWS | F_PACKREL)
    SIM_NOTB_CASE(ALL | F_PACKREL)
    SIM_NOTB_CASE(ALL | F_PACKREL | F_RELU)
    SIM_NOTB_CASE(F_LUT | F_TRACK_ROWS | F_PACKREL)
    SIM_NOTB_CASE(F_LUT | ALL | F_PACKREL)
    SIM_NOTB_CASE(F_LUT | ALL | F_PACKREL | F_RELU)
    default: std::abort();
  }
#undef SIM_NOTB_CASE
}

}  // namespace

extern "C" {

// Returns -1 for an unsupported shape, else the number of boundary / rows arena bytes in which the score-only fill
// differs from the traceback fill.  Outputs per pair (caller order): score, xend, yend, status of the score-only
// epilogue; gap_clip = 1 where the full walk (walk_run, one move at a time on the traceback fill's scratch), still
// inside row m and column n, takes a suffix clip after a gap move along them -- the case the end walk must follow.
// Gsel / modebits as in sim_align_batch_g (modebits & 8: the warp-per-pair epilogue).
int sim_scores_batch(int mode, const sim_scoring* s, const uint8_t* blob, const uint64_t* x_off, const uint32_t* x_len,
                     const uint64_t* y_off, const uint32_t* y_len, uint64_t n_pairs, int Gsel, int R, int modebits,
                     int garbage, int32_t* score, uint32_t* xend, uint32_t* yend, uint32_t* status,
                     uint32_t* gap_clip) {
  DevScoring sc{};
  sc.gap_open = s->gap_open;
  sc.gap_extend = s->gap_extend;
  sc.xclip_prefix = s->xclip_prefix;
  sc.xclip_suffix = s->xclip_suffix;
  sc.yclip_prefix = s->yclip_prefix;
  sc.yclip_suffix = s->yclip_suffix;
  if (mode == 1) sc.xclip_prefix = sc.xclip_suffix = sc.yclip_prefix = sc.yclip_suffix = MIN_SCORE;
  if (mode == 2) { sc.xclip_prefix = sc.xclip_suffix = MIN_SCORE; sc.yclip_prefix = sc.yclip_suffix = 0; }
  if (mode == 3) sc.xclip_prefix = sc.xclip_suffix = sc.yclip_prefix = sc.yclip_suffix = 0;
  sc.match_score = s->match_score;
  sc.mismatch_score = s->mismatch_score;
  uint8_t codemap[256];
  for (int k = 0; k < 256; ++k) codemap[k] = (uint8_t)k;
  std::vector<int32_t> lut;
  int64_t maxabs = std::max<int64_t>(std::llabs((long long)s->match_score), std::llabs((long long)s->mismatch_score));
  {
    bool present[256] = {false};
    for (uint64_t p = 0; p < n_pairs; ++p) {
      for (uint32_t k = 0; k < x_len[p]; ++k) present[blob[x_off[p] + k]] = true;
      for (uint32_t k = 0; k < y_len[p]; ++k) present[blob[y_off[p] + k]] = true;
    }
    std::vector<int> syms;
    for (int k = 0; k < 256; ++k)
      if (present[k]) syms.push_back(k);
    if (syms.empty()) syms.push_back(0);
    const bool use_lut = s->table || !(modebits & 4);
    if (use_lut && syms.size() <= 64) {
      for (size_t a = 0; a < syms.size(); ++a) codemap[syms[a]] = (uint8_t)a;
      sc.alpha = (int32_t)syms.size();
      const size_t aa = (size_t)sc.alpha * sc.alpha;
      lut.resize(aa + (size_t)lut_entries(sc.alpha));
      if (s->table) maxabs = 0;
      for (int a = 0; a < sc.alpha; ++a)
        for (int b = 0; b < sc.alpha; ++b) {
          const int32_t v = s->table ? s->table[syms[a] * 256 + syms[b]] : (a == b ? s->match_score : s->mismatch_score);
          lut[(size_t)a * sc.alpha + b] = v;
          maxabs = std::max<int64_t>(maxabs, std::llabs((long long)v));
        }
      for (size_t k = 0; k < aa; ++k) lut[aa + k] = 4 * lut[k] + 3 - (4 * sc.gap_open + 1);
      for (size_t k = aa; k < (size_t)lut_entries(sc.alpha); ++k) lut[aa + k] = LUT_POISON;
    }
  }
  const bool piped = Gsel == 132;
  const int G = piped ? 32 : Gsel;
  Plan p, ps;
  build_plan(p, x_len, y_len, n_pairs, G, R, ~0ull);
  build_plan(ps, x_len, y_len, n_pairs, G, R, 1, true);  // a 1-byte budget: only the traceback arena could close a wave
  if (ps.total_tb != 0 || ps.waves.size() > 1 || ps.max_bnd != p.max_bnd || ps.max_rows != p.max_rows) return -2;
  const int P = 32 / G;
  const int64_t unit = std::max<int64_t>(maxabs, std::max<int64_t>(-(int64_t)sc.gap_open, -(int64_t)sc.gap_extend));
  const int64_t bound = ((int64_t)p.maxm + p.maxn + 2) * unit - (int64_t)sc.gap_open;
  int flags = scoring_flags(sc, bound, p.maxm, p.maxn);
  if (modebits & 2) flags &= ~(F_PACKTRK | F_PACKREL);
  if ((modebits & 16) && (flags & (F_TRACK_ROWS | F_TRACK_COLS))) {
    flags &= ~F_PACKTRK;
    flags |= F_PACKREL;
  }
  const int32_t* lut_plain = lut.data();
  const int32_t* lut_scaled = lut.data() + (size_t)sc.alpha * sc.alpha;
  const uint8_t gb = (uint8_t)garbage;
  std::vector<uint8_t> seq(p.seq_bytes, 0), bnd(p.max_bnd, gb), rows(p.max_rows, gb), tb(p.max_tb, gb),
      bnd2(p.max_bnd, gb), rows2(p.max_rows, gb), tb2(16, gb), rowm(p.max_rowm, gb);
  for (const Block& blk : p.blocks) {
    uint32_t* seqw = reinterpret_cast<uint32_t*>(seq.data() + blk.seq_off);
    for (uint32_t q = 0; q < blk.npairs; ++q) {
      const uint32_t orig = p.order[blk.first + q];
      const uint32_t sub = q / P, slot = q % P;
      uint32_t* xw = seqw + (size_t)sub * blk.xwords * P;
      for (uint32_t k = 0; k < x_len[orig]; ++k)
        reinterpret_cast<uint8_t*>(&xw[(k >> 2) * P + slot])[k & 3] = codemap[blob[x_off[orig] + k]];
      uint32_t* yw = seqw + (size_t)G * blk.xwords * P + (size_t)sub * blk.ywords * P;
      for (uint32_t k = 0; k < y_len[orig]; ++k)
        reinterpret_cast<uint8_t*>(&yw[(k >> 2) * P + slot])[k & 3] = codemap[blob[y_off[orig] + k]];
    }
  }
  for (size_t b = 0; b < p.blocks.size(); ++b) {
    const Block& blk = p.blocks[b];
    Block blk0 = ps.blocks[b];  // the score-only plan's block: no traceback offset
    switch ((piped ? 10000 : 0) + G * 100 + R) {
      case 116:
        fill_dispatch<1, 16>(flags, p, blk, sc, lut_scaled, seq, bnd, rows, tb);
        fill_dispatch_notb<1, 16, false>(flags, ps, blk0, sc, lut_scaled, seq, bnd2, rows2, tb2);
        break;
      case 808:
        fill_dispatch<8, 8>(flags, p, blk, sc, lut_scaled, seq, bnd, rows, tb);
        fill_dispatch_notb<8, 8, false>(flags, ps, blk0, sc, lut_scaled, seq, bnd2, rows2, tb2);
        break;
      case 820:
        fill_dispatch<8, 20>(flags, p, blk, sc, lut_scaled, seq, bnd, rows, tb);
        fill_dispatch_notb<8, 20, false>(flags, ps, blk0, sc, lut_scaled, seq, bnd2, rows2, tb2);
        break;
      case 3208:
        fill_dispatch<32, 8>(flags, p, blk, sc, lut_scaled, seq, bnd, rows, tb);
        fill_dispatch_notb<32, 8, false>(flags, ps, blk0, sc, lut_scaled, seq, bnd2, rows2, tb2);
        break;
      case 13208:
        fill_dispatch<32, 8, true>(flags, p, blk, sc, lut_scaled, seq, bnd, rows, tb);
        fill_dispatch_notb<32, 8, true>(flags, ps, blk0, sc, lut_scaled, seq, bnd2, rows2, tb2);
        break;
      default: return -1;
    }
  }
  int diff = 0;
  for (size_t k = 0; k < bnd.size(); ++k) diff += bnd[k] != bnd2[k];
  for (size_t k = 0; k < rows.size(); ++k) diff += rows[k] != rows2[k];
  if (tb2 != std::vector<uint8_t>(16, gb)) ++diff;  // the score-only fill stores no traceback
  for (const Block& blk : ps.blocks) {
    for (uint32_t lane = 0; lane < blk.npairs; ++lane) {
      const uint32_t sp = blk.first + lane;
      PairView v;
      v.sc = sc;
      v.lut = lut_plain;
      v.P = P;
      v.m = (int32_t)ps.pm[sp];
      v.n = (int32_t)ps.pn[sp];
      v.pi = (int32_t)lane;
      v.set_shape(G, R);
      v.nstrips = (int32_t)blk.nstrips;
      v.K = (int32_t)blk.K;
      v.sub = (int32_t)lane / P;
      v.g = (int32_t)lane % P;
      v.packtrk = (flags & F_PACKTRK) ? 1 : 0;
      v.maxn = (int32_t)blk.maxn;
      v.bnd_base = bnd_index(G, 0, (int32_t)lane, v.maxn);
      v.bnd_stride = (int32_t)(bnd_index(G, 1, (int32_t)lane, v.maxn) - v.bnd_base);
      const uint32_t* seqw = reinterpret_cast<const uint32_t*>(seq.data() + blk.seq_off);
      v.xw = seqw + (size_t)v.sub * blk.xwords * P + v.g;
      v.yw = seqw + (size_t)G * blk.xwords * P + (size_t)v.sub * blk.ywords * P + v.g;
      v.bnd = reinterpret_cast<const int4*>(bnd2.data() + blk.bnd_off);
      v.rows = reinterpret_cast<int32_t*>(rows2.data() + blk.rows_off);
      v.rows_pad = (int32_t)blk.rows_pad;
      v.rowm = reinterpret_cast<uint16_t*>(rowm.data() + blk.rowm_off);
      v.tb = nullptr;  // the epilogue must not read a traceback
      const bool filter = mode == 2 || mode == 3;
      EndOut o;
      if (modebits & 8) {  // the warp-per-pair form: cooperative finish on 32 emulated lanes, lane 0's end walk
        LaneFibers::run([&](int l) {
          EndState es;
          finish_matrix_coop<32>(l, v, es);
          if (l == 0) end_walk(v, es, filter, o);
        });
      } else {
        EndState es;
        finish_matrix_seq(v, es);
        end_walk(v, es, filter, o);
      }
      const uint32_t dst = ps.order[sp];
      {  // the full walk on the traceback fill's scratch, move by move
        PairView vf = v;
        const Block& bf = p.blocks[&blk - ps.blocks.data()];
        vf.bnd = reinterpret_cast<const int4*>(bnd.data() + bf.bnd_off);
        vf.rows = reinterpret_cast<int32_t*>(rows.data() + bf.rows_off);
        vf.tb = reinterpret_cast<const uint32_t*>(tb.data() + bf.tb_off);
        std::vector<uint8_t> rowm_f(rowm.size(), gb), ops_f((size_t)v.m + v.n + 8);
        vf.rowm = reinterpret_cast<uint16_t*>(rowm_f.data() + blk.rowm_off);
        EndState es;
        finish_matrix_seq(vf, es);
        WalkState w;
        walk_begin(vf, es, ops_f.data() + ops_f.size(), w);
        bool gap = false, done = false;
        gap_clip[dst] = 0;
        while (!done && (w.i == v.m || w.j == v.n)) {
          const uint32_t layer = w.layer;
          if ((layer == TB_INS && w.j == v.n) || (layer == TB_DEL && w.i == v.m)) gap = true;
          if ((layer == TB_XCLIP_SUFFIX || layer == TB_YCLIP_SUFFIX) && gap) gap_clip[dst] = 1;
          done = walk_run(vf, es, filter, w, 1);
        }
      }
      score[dst] = o.score;
      xend[dst] = o.xend;
      yend[dst] = o.yend;
      status[dst] = o.status;
    }
  }
  return diff;
}
}

// CPU harness for the pair-packed K1 fill (b2a_fill_pair16.cuh): the kernel's per-lane code compiled for the host.
// It stages a batch as K0 does, fills it twice -- with fill_lane<1,16,63> (the int32 kernel) and with the packed
// fill over pairs of blocks -- and compares everything K2 reads (traceback words, rows arena, the final boundary row)
// on the valid pairs.  It then runs K2's walk on the packed fill's scratch, so the tests can diff the alignments
// against the oracle as well.
#include "b2a_sim.cpp"

#include "../../rust_bio_b200/csrc/b2a_fill_pair16.cuh"

namespace {

// byte arenas of one fill of the whole batch
struct Arenas {
  std::vector<uint8_t> bnd, rows, tb;
};

}  // namespace

extern "C" {

// Returns -1 if the batch is not a pair-packed batch (caller error), else the number of 32-bit scratch words that
// differ between the two fills.  Outputs as in sim_align_batch_g, from the packed fill.
int sim_pair16_batch(const sim_scoring* s, const uint8_t* blob, const uint64_t* x_off, const uint32_t* x_len,
                     const uint64_t* y_off, const uint32_t* y_len, uint64_t n_pairs, int garbage, int32_t* score,
                     uint32_t* xstart, uint32_t* xend, uint32_t* ystart, uint32_t* yend, uint32_t* n_ops,
                     uint32_t* clip_len, uint32_t* status, uint8_t* ops, const uint64_t* ops_off) {
  constexpr int G = 1, R = 16, P = 32, TBW = tbw_of(R);
  DevScoring sc{};
  sc.gap_open = s->gap_open;
  sc.gap_extend = s->gap_extend;
  sc.xclip_prefix = sc.xclip_suffix = sc.yclip_prefix = sc.yclip_suffix = 0;  // local
  sc.match_score = s->match_score;
  sc.mismatch_score = s->mismatch_score;
  uint8_t codemap[256];
  bool present[256] = {false};
  for (uint64_t p = 0; p < n_pairs; ++p) {
    for (uint32_t k = 0; k < x_len[p]; ++k) present[blob[x_off[p] + k]] = true;
    for (uint32_t k = 0; k < y_len[p]; ++k) present[blob[y_off[p] + k]] = true;
  }
  if (s->alphabet)
    for (uint32_t k = 0; k < s->alphabet_len; ++k) present[s->alphabet[k]] = true;
  std::vector<int> syms;
  for (int k = 0; k < 256; ++k)
    if (present[k]) syms.push_back(k);
  if (syms.empty() || syms.size() > (size_t)P16_MAX_ALPHA) return -1;
  for (int k = 0; k < 256; ++k) codemap[k] = 0xFF;
  for (size_t a = 0; a < syms.size(); ++a) codemap[syms[a]] = (uint8_t)a;
  sc.alpha = (int32_t)syms.size();
  const size_t aa = (size_t)sc.alpha * sc.alpha;
  std::vector<int32_t> lut(aa + (size_t)lut_entries(sc.alpha));
  int32_t lo = 0, hi = 0;
  for (int a = 0; a < sc.alpha; ++a)
    for (int b = 0; b < sc.alpha; ++b) {
      const int32_t v = s->table ? s->table[syms[a] * 256 + syms[b]] : (a == b ? s->match_score : s->mismatch_score);
      lut[(size_t)a * sc.alpha + b] = v;
      lo = (a || b) ? std::min(lo, v) : v;
      hi = (a || b) ? std::max(hi, v) : v;
    }
  for (size_t k = 0; k < aa; ++k) lut[aa + k] = 4 * lut[k] + 3 - (4 * sc.gap_open + 1);
  for (size_t k = aa; k < (size_t)lut_entries(sc.alpha); ++k) lut[aa + k] = LUT_POISON;
  std::vector<int32_t> lut16((size_t)p16_lut_entries(sc.alpha));
  p16_build_lut(lut.data() + aa, sc.alpha, lut16.data());

  Plan p;
  build_plan(p, x_len, y_len, n_pairs, G, R, ~0ull);
  for (uint64_t i = 0; i < n_pairs; ++i)
    if (p.pm[i] != p.maxm || p.pn[i] != p.maxn) return -1;
  if (p.maxm > 256 || p.maxn > 255 || (int64_t)std::min(p.maxm, p.maxn) * std::max(hi, 0) > 255) return -1;
  const int32_t bias = 4 * std::max(std::max(-sc.gap_open, -lo), 0);

  std::vector<uint8_t> seq(p.seq_bytes, 0);
  for (const Block& blk : p.blocks) {
    uint32_t* seqw = reinterpret_cast<uint32_t*>(seq.data() + blk.seq_off);
    for (uint32_t q = 0; q < blk.npairs; ++q) {
      const uint32_t orig = p.order[blk.first + q];
      for (uint32_t k = 0; k < x_len[orig]; ++k)
        reinterpret_cast<uint8_t*>(&seqw[(k >> 2) * P + q])[k & 3] = codemap[blob[x_off[orig] + k]];
      uint32_t* yw = seqw + (size_t)blk.xwords * P;
      for (uint32_t k = 0; k < y_len[orig]; ++k)
        reinterpret_cast<uint8_t*>(&yw[(k >> 2) * P + q])[k & 3] = codemap[blob[y_off[orig] + k]];
    }
  }
  const uint8_t gb = (uint8_t)garbage;
  Arenas ref{std::vector<uint8_t>(p.max_bnd, gb), std::vector<uint8_t>(p.max_rows, gb), std::vector<uint8_t>(p.max_tb, gb)};
  Arenas pk{std::vector<uint8_t>(p.max_bnd, (uint8_t)~gb), std::vector<uint8_t>(p.max_rows, (uint8_t)~gb),
            std::vector<uint8_t>(p.max_tb, (uint8_t)~gb)};
  for (const Block& blk : p.blocks)
    fill_block<G, R, P16_FLAGS>(p, blk, sc, lut.data() + aa, seq, ref.bnd, ref.rows, ref.tb);
  // the packed fill: block pairs (2k, 2k+1), lane after lane
  const uint32_t nb = (uint32_t)p.blocks.size();
  for (uint32_t ba = 0; ba < nb; ba += 2) {
    const bool has_b = ba + 1 < nb;
    const Block& A = p.blocks[ba];
    const Block& Bk = p.blocks[has_b ? ba + 1 : ba];
    for (int lane = 0; lane < 32; ++lane) {
      P16Ctx c;
      c.sc = sc;
      c.lut = lut16.data();
      c.lut_base = 0;
      c.xa = reinterpret_cast<const uint32_t*>(seq.data() + A.seq_off) + lane;
      c.xb = reinterpret_cast<const uint32_t*>(seq.data() + Bk.seq_off) + lane;
      c.ya = reinterpret_cast<const uint32_t*>(seq.data() + A.seq_off) + (size_t)A.xwords * P;
      c.yb = reinterpret_cast<const uint32_t*>(seq.data() + Bk.seq_off) + (size_t)Bk.xwords * P;
      c.m = (int32_t)A.maxm;
      c.n = (int32_t)A.maxn;
      c.nstrips = (int32_t)A.nstrips;
      c.K = (int32_t)A.K;
      c.rows_pad = (int32_t)A.rows_pad;
      c.lane = lane;
      c.has_b = has_b;
      c.bnd_a = reinterpret_cast<int4*>(pk.bnd.data() + A.bnd_off);
      c.bnd_b = reinterpret_cast<int4*>(pk.bnd.data() + Bk.bnd_off);
      c.rows_a = reinterpret_cast<int32_t*>(pk.rows.data() + A.rows_off);
      c.rows_b = reinterpret_cast<int32_t*>(pk.rows.data() + Bk.rows_off);
      c.tb_a = reinterpret_cast<uint4*>(pk.tb.data() + A.tb_off);
      c.tb_b = reinterpret_cast<uint4*>(pk.tb.data() + Bk.tb_off);
      c.one = 1;
      c.mone = -1;
      c.k16 = 16;
      c.ge4 = 4 * sc.gap_extend;
      c.bias = bias;
      p16_fill_lane<R>(c);
    }
  }
  // compare what K2 reads, valid pairs only (slot = word index % 32 in every [index][32] layout)
  int diff = 0;
  for (const Block& blk : p.blocks) {
    const size_t nbnd = (size_t)(blk.maxn + 1) * 32 * 4, nrows = (size_t)ROWS_ARRAYS * blk.rows_pad * 32,
                 ntb = (size_t)blk.nstrips * blk.K * TBW * 32 * 4;
    auto cmp = [&](const std::vector<uint8_t>& a, const std::vector<uint8_t>& b, uint64_t off, size_t words,
                   size_t skip_lo, size_t per_slot) {
      const uint32_t* wa = reinterpret_cast<const uint32_t*>(a.data() + off);
      const uint32_t* wb = reinterpret_cast<const uint32_t*>(b.data() + off);
      for (size_t k = skip_lo; k < words; ++k)
        if ((k / per_slot) % 32 < blk.npairs && wa[k] != wb[k]) ++diff;
    };
    cmp(ref.bnd, pk.bnd, blk.bnd_off, nbnd, 32 * 4, 4);  // columns 1..n (column 0 is never written)
    // rows arena: rows 1 .. nstrips*R of every array
    for (int arr = 0; arr < ROWS_ARRAYS; ++arr) {
      const size_t base = (size_t)arr * blk.rows_pad * 32;
      const uint32_t* wa = reinterpret_cast<const uint32_t*>(ref.rows.data() + blk.rows_off) + base;
      const uint32_t* wb = reinterpret_cast<const uint32_t*>(pk.rows.data() + blk.rows_off) + base;
      for (size_t k = 32; k < (size_t)(blk.nstrips * R + 1) * 32; ++k)
        if (k % 32 < blk.npairs && wa[k] != wb[k]) ++diff;
    }
    (void)nrows;
    cmp(ref.tb, pk.tb, blk.tb_off, ntb, 0, 4);
  }
  // K2 on the packed fill's scratch
  std::vector<uint8_t> rowm(p.max_rowm, gb), opsb(p.ops_bytes, 0);
  for (const Block& blk : p.blocks) {
    for (uint32_t lane = 0; lane < blk.npairs; ++lane) {
      const uint32_t sp = blk.first + lane;
      PairView v;
      v.sc = sc;
      v.lut = lut.data();
      v.P = P;
      v.m = (int32_t)p.pm[sp];
      v.n = (int32_t)p.pn[sp];
      v.pi = (int32_t)lane;
      v.set_shape(G, R);
      v.nstrips = (int32_t)blk.nstrips;
      v.K = (int32_t)blk.K;
      v.sub = 0;
      v.g = (int32_t)lane;
      v.packtrk = 1;
      v.maxn = (int32_t)blk.maxn;
      v.bnd_base = bnd_index(G, 0, (int32_t)lane, v.maxn);
      v.bnd_stride = (int32_t)(bnd_index(G, 1, (int32_t)lane, v.maxn) - v.bnd_base);
      const uint32_t* seqw = reinterpret_cast<const uint32_t*>(seq.data() + blk.seq_off);
      v.xw = seqw + lane;
      v.yw = seqw + (size_t)blk.xwords * P + lane;
      v.bnd = reinterpret_cast<const int4*>(pk.bnd.data() + blk.bnd_off);
      v.rows = reinterpret_cast<int32_t*>(pk.rows.data() + blk.rows_off);
      v.rows_pad = (int32_t)blk.rows_pad;
      v.rowm = reinterpret_cast<uint16_t*>(rowm.data() + blk.rowm_off);
      v.tb = reinterpret_cast<const uint32_t*>(pk.tb.data() + blk.tb_off);
      const uint32_t cap = blk.maxm + blk.maxn + 4;
      uint8_t* ops_end = opsb.data() + blk.ops_off + (size_t)(lane + 1) * cap;
      WalkOut o;
      walk_pair(v, true, ops_end, o);
      const uint32_t dst = p.order[sp];
      score[dst] = o.score;
      xstart[dst] = o.xstart;
      xend[dst] = o.xend;
      ystart[dst] = o.ystart;
      yend[dst] = o.yend;
      n_ops[dst] = o.n_ops;
      status[dst] = o.status;
      for (int k = 0; k < 4; ++k) clip_len[4 * (size_t)dst + k] = o.clip[k];
      std::memcpy(ops + ops_off[dst], ops_end - o.n_ops, o.n_ops);
    }
  }
  return diff;
}
}

// Host-side batch plan: sort pairs by shape, cut them into blocks of 32, size
// the HBM arenas and the traceback waves.  Pure C++ (used by the engine and by
// the CPU simulation harness in tests/sim/).
#pragma once
#include <algorithm>
#include <cstdint>
#include <numeric>
#include <vector>

#include "b2a_common.cuh"

namespace b2a {

struct Wave {
  uint32_t block_lo, block_hi;  // [lo, hi)
  uint64_t bnd_bytes, rows_bytes, rowm_bytes, tb_bytes;
  uint64_t strip_tasks;  // sum over the wave's blocks of 32 * nstrips
};

struct Plan {
  int G = 1, R = 16;
  uint64_t n_pairs = 0;
  std::vector<uint32_t> order;  // sorted index -> caller index
  std::vector<uint32_t> pm, pn; // sorted
  std::vector<Block> blocks;
  std::vector<Wave> waves;
  uint64_t seq_bytes = 0, ops_bytes = 0;
  uint64_t max_bnd = 0, max_rows = 0, max_rowm = 0, max_tb = 0;  // per-wave maxima
  uint64_t max_strip_tasks = 0;
  uint64_t total_tb = 0;   // traceback bytes the fill stores over the whole batch
  uint64_t cells = 0;
  uint32_t smem_seq_bytes = 0;  // per-warp staging
  uint32_t maxm = 0, maxn = 0;
};

inline uint64_t align_up(uint64_t v, uint64_t a) { return (v + a - 1) / a * a; }

// score_only: the plan of a score-only batch (K1 with F_NOTB): no traceback arena, so the budget never closes a
// wave -- the batch is one wave
inline void build_plan(Plan& p, const uint32_t* x_len, const uint32_t* y_len, uint64_t n_pairs, int G,
                       int R, uint64_t tb_budget, bool score_only = false) {
  p.G = G;
  p.R = R;
  p.n_pairs = n_pairs;
  p.order.resize(n_pairs);
  std::iota(p.order.begin(), p.order.end(), 0u);
  bool uniform_all = true;
  for (uint64_t i = 1; i < n_pairs && uniform_all; ++i)
    uniform_all = (x_len[i] == x_len[0]) && (y_len[i] == y_len[0]);
  if (!uniform_all) {
    std::stable_sort(p.order.begin(), p.order.end(), [&](uint32_t a, uint32_t b) {
      if (x_len[a] != x_len[b]) return x_len[a] > x_len[b];
      return y_len[a] > y_len[b];
    });
  }
  p.pm.resize(n_pairs);
  p.pn.resize(n_pairs);
  p.cells = 0;
  for (uint64_t i = 0; i < n_pairs; ++i) {
    p.pm[i] = x_len[p.order[i]];
    p.pn[i] = y_len[p.order[i]];
    p.cells += (uint64_t)p.pm[i] * p.pn[i];
  }
  const uint32_t nblocks = (uint32_t)((n_pairs + 31) / 32);
  const int P = 32 / G, TBW = tbw_of(R);
  p.blocks.assign(nblocks, Block{});
  p.waves.clear();
  p.seq_bytes = p.ops_bytes = 0;
  p.max_bnd = p.max_rows = p.max_rowm = p.max_tb = 0;
  p.max_strip_tasks = 0;
  p.total_tb = 0;
  p.smem_seq_bytes = 0;
  p.maxm = p.maxn = 0;
  Wave w{0, 0, 0, 0, 0, 0, 0};
  for (uint32_t b = 0; b < nblocks; ++b) {
    Block& k = p.blocks[b];
    k.first = b * 32;
    k.npairs = (uint32_t)std::min<uint64_t>(32, n_pairs - (uint64_t)b * 32);
    k.maxm = k.maxn = 0;
    for (uint32_t q = 0; q < k.npairs; ++q) {
      k.maxm = std::max(k.maxm, p.pm[k.first + q]);
      k.maxn = std::max(k.maxn, p.pn[k.first + q]);
    }
    k.uniform = 1;
    for (uint32_t q = 0; q < k.npairs; ++q)
      if (p.pm[k.first + q] != k.maxm || p.pn[k.first + q] != k.maxn) k.uniform = 0;
    k.nstrips = k.maxm >= 2 ? (k.maxm - 1 + G * R - 1) / (G * R) : 0;
    const uint32_t xw = std::max<uint32_t>((k.maxm + 3) / 4, k.nstrips * G * R / 4);
    k.xwords = (uint32_t)align_up(std::max<uint32_t>(xw, 4), 4);
    k.ywords = (uint32_t)align_up(std::max<uint32_t>((k.maxn + 3) / 4, 4), 4);
    k.K = k.maxn ? (k.maxn + G - 1 + 7) / 8 : 0;
    k.rows_pad = k.nstrips * G * R + 2;
    p.maxm = std::max(p.maxm, k.maxm);
    p.maxn = std::max(p.maxn, k.maxn);
    // the warp-per-pair shape runs (pair, strip) tasks that stage one strip of x (b2a_fill.cuh)
    const uint32_t stage_x = G == 32 ? (uint32_t)(G * R) : k.xwords * P * 4;
    p.smem_seq_bytes = std::max<uint32_t>(p.smem_seq_bytes, stage_x + k.ywords * P * 4);
    const uint64_t bnd = align_up((uint64_t)(k.maxn + 1) * 32 * 16, 256);
    const uint64_t rows = align_up((uint64_t)ROWS_ARRAYS * k.rows_pad * 32 * 4, 256);
    const uint64_t rowm = align_up((uint64_t)(k.maxn + 1) * 32 * 2, 256);
    const uint64_t tb_raw = score_only ? 0 : (uint64_t)G * k.nstrips * k.K * TBW * 512;
    const uint64_t tb = align_up(tb_raw, 256);
    if (b > w.block_lo && w.tb_bytes + tb > tb_budget) {  // close the wave
      w.block_hi = b;
      p.waves.push_back(w);
      w = Wave{b, b, 0, 0, 0, 0, 0};
    }
    k.seq_off = p.seq_bytes;
    p.seq_bytes += align_up((uint64_t)32 * (k.xwords + k.ywords) * 4, 256);
    k.ops_off = p.ops_bytes;
    p.ops_bytes += align_up((uint64_t)32 * (k.maxm + k.maxn + 4), 256);
    k.strip_task_base = w.strip_tasks;
    w.strip_tasks += (uint64_t)32 * k.nstrips;
    k.bnd_off = w.bnd_bytes;
    k.rows_off = w.rows_bytes;
    k.rowm_off = w.rowm_bytes;
    k.tb_off = w.tb_bytes;
    w.bnd_bytes += bnd;
    w.rows_bytes += rows;
    w.rowm_bytes += rowm;
    w.tb_bytes += tb;
    p.total_tb += tb_raw;
  }
  if (nblocks) {
    w.block_hi = nblocks;
    p.waves.push_back(w);
  }
  for (const Wave& v : p.waves) {
    p.max_bnd = std::max(p.max_bnd, v.bnd_bytes);
    p.max_rows = std::max(p.max_rows, v.rows_bytes);
    p.max_rowm = std::max(p.max_rowm, v.rowm_bytes);
    p.max_tb = std::max(p.max_tb, v.tb_bytes);
    p.max_strip_tasks = std::max(p.max_strip_tasks, v.strip_tasks);
  }
}

// Kernel flags for a scoring (SURVEY 3.2 "derived mode specialisations").
// `score_bound` = (maxm+maxn+2)*max|score, go, ge| + |go|: every real S/I/D lies within +-score_bound.
inline int scoring_flags(const DevScoring& sc, int64_t score_bound = (1ll << 40), uint32_t maxm = ~0u,
                         uint32_t maxn = ~0u) {
  const bool xp = sc.xclip_prefix > DEAD_CLIP, xs = sc.xclip_suffix > DEAD_CLIP;
  const bool yp = sc.yclip_prefix > DEAD_CLIP, ys = sc.yclip_suffix > DEAD_CLIP;
  int f = 0;
  if (xs || (xp && yp)) {
    f = F_TRACK_ROWS | F_TRACK_COLS | F_CLIPX;  // general variant
  } else if (ys) {
    f = F_TRACK_ROWS;
  }
  if (sc.alpha) f |= F_LUT;
  // local-style clips: xclip_score(j) = xp + max(yp, go + ge (j-1)) == 0 for every j (go, ge <= 0)
  if ((f & F_CLIPX) && sc.xclip_prefix == 0 && sc.yclip_prefix == 0) f |= F_RELU;
  if ((f & (F_TRACK_ROWS | F_TRACK_COLS)) && score_bound < (1ll << 17) && maxm <= 4095 && maxn <= 4095)
    f |= F_PACKTRK;
  else if ((f & (F_TRACK_ROWS | F_TRACK_COLS)) && score_bound < (1ll << 18))
    f |= F_PACKREL;  // longer sequences: the packed keys with chunk- / strip-relative indices
  return f;
}

}  // namespace b2a

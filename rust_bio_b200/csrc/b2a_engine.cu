// libb200align.so: engine + C ABI (include/b200align.h).
//
// Host side of the B200 pairwise path: validates a batch the way the reference's
// constructors do (mod.rs:517-518, 554-571), plans it (b2a_plan.h), moves it to
// HBM and launches K0 (pack) -> K1 (fill) -> K2 (row m, fix-ups, walk) ->
// ops compaction on one CUDA stream.  There is no CPU implementation of the
// alignment in this library: without a usable CUDA device every call fails.
#include <cuda_runtime.h>

#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <cub/device/device_scan.cuh>
#include <string>
#include <vector>

#define B2A_DEFINE_WALK_KERNEL
#include "../../include/b200align.h"
#include "b2a_fill_launch.h"
#include "b2a_fill_pair16.cuh"
#include "b2a_kernels.cuh"
#include "b2a_plan.h"
#include "b2a_walk.cuh"
#include "b2a_banded.cuh"
#include "b2a_banded_strip.cuh"

using namespace b2a;

namespace {

struct DevBuf {
  void* p = nullptr;
  size_t cap = 0;
  cudaError_t reserve(size_t n) {
    if (n <= cap) return cudaSuccess;
    if (p) cudaFree(p);
    p = nullptr;
    cap = 0;
    size_t want = n + n / 8 + 256;
    cudaError_t e = cudaMalloc(&p, want);
    if (e != cudaSuccess) {
      want = n;
      e = cudaMalloc(&p, want);
    }
    if (e == cudaSuccess) cap = want;
    return e;
  }
  void release() {
    if (p) cudaFree(p);
    p = nullptr;
    cap = 0;
  }
  template <class T>
  T* as() const {
    return reinterpret_cast<T*>(p);
  }
};

const FillLaunch kFillShapes[] = {
    {1, 16, launch_fill_1_16}, {1, 8, launch_fill_1_8},   {1, 20, launch_fill_1_20},
    {2, 16, launch_fill_2_16}, {2, 20, launch_fill_2_20}, {4, 16, launch_fill_4_16},
    {8, 16, launch_fill_8_16}, {8, 20, launch_fill_8_20}, {32, 8, launch_fill_32_8}, {32, 16, launch_fill_32_16},
};

const FillLaunch* find_shape(int G, int R) {
  for (const FillLaunch& f : kFillShapes)
    if (f.G == G && f.R == R) return &f;
  return nullptr;
}

constexpr uint32_t kMaxStageSmem = 200 * 1024;  // of the 227 KB a CTA may use
constexpr uint64_t kWarpWalkMaxPairs = 16384;  // waves up to this many pairs use the warp-per-pair K2
constexpr int kMaxAlpha = 64;        // MatchParams: LUT up to this many symbols, compare/select beyond
constexpr int kMaxAlphaTable = 128;  // tabulated MatchFunc: a 128 x 128 LUT (64 KB of shared memory) covers 7-bit alphabets

}  // namespace

struct b2a_engine {
  int device = 0;
  int num_sms = 0;
  cudaStream_t stream = nullptr, own_stream = nullptr;
  // pipeline slots only: K2 + ops compaction + result copies run on this high-priority stream, so that an
  // older chunk's short, latency-bound tail is scheduled ahead of the next chunk's fill CTAs
  cudaStream_t tail_stream = nullptr;
  cudaStream_t aux_stream = nullptr;   // second fill stream of the small-batch overlap (b2a_batch_run)
  std::vector<cudaEvent_t> sub_ev;
  bool overlap_small = true;
  bool overlap_big = false;
  bool no_packrel = false;         // B2A_NO_PACKREL=1: long sequences keep explicit (value, index) trackers (test knob)
  bool tail_split = true;          // small batches: the fill's thin last round of tasks runs under K2 of the rest
  bool split_timing = false;       // B2A_SPLIT_TIMING=1: print where the split step's time goes (dev aid)
  cudaEvent_t split_ev[5] = {nullptr, nullptr, nullptr, nullptr, nullptr};
  bool split_ran = false;
  uint32_t walk_cta_warps = 0;     // warps (pairs) per CTA of the warp-per-pair K2: 1, 2, 4, 8, 16, 32 or 0 = automatic
  cudaEvent_t ev_fill = nullptr;
  bool tail_used = false;          // the last run put K2 and the compaction on tail_stream
  bool is_slot = false;            // this engine is a slot of another engine's chunk pipeline
  bool stage_nosync = false;       // pipeline slots: the caller's arrays outlive the call, no sync at the end of stage
  uint32_t fill_task_limit = 0;    // pipeline slots: fill CTAs retire after this many tasks per warp (CTA turnover)
  uint8_t* h_plan = nullptr;       // pinned staging of the plan vectors (async H2D)
  size_t h_plan_cap = 0;
  cudaStream_t res_stream() const { return tail_used ? tail_stream : stream; }  // where the results become ready
  uint64_t compact_hdr[8] = {~0ull, 0, 0, 0, 0, 0, 0, 0};  // header of the compact result segment
  // the band of the last banded call's last wave (Band::ranges), for b2a_banded_band_ranges
  uint64_t band_wave_lo = 0;
  std::vector<uint64_t> band_roff;
  std::vector<uint32_t> band_ylen;
  std::string err;
  int tune_G = 0, tune_R = 0;
  int walk_mode = 0;  // 0 automatic, 1 one lane per pair, 2 one warp per pair
  bool banded_fast = true;  // K3: register-resident column loop for the pairs K4 marks (B2A_BANDED_LITERAL=1: never)
  bool banded_strip = true;  // K3s: strip-wavefront fill for the pairs K4 marks (B2A_BANDED_STRIP=0: never)
  bool banded_strip_lastcol = true;  // ... also for bands reaching column n (B2A_BANDED_STRIP_LASTCOL=0: those stay with K3)
  uint64_t strip_pairs = 0;  // pairs the strip path finished in the last banded call (the rest ran the K3 loops)
  // packed input (b2a_align_batch_packed): the caller's "blob" is BitEnc storage of this width (0 = bytes); the
  // engine unpacks it on the device and uses its own byte offsets (eff_xoff / eff_yoff) from then on
  uint32_t packed_width = 0;
  std::vector<uint64_t> eff_xoff, eff_yoff;
  bool last_walk_warp = false;
  uint64_t tb_budget = 0;
  bool pairpack = true;            // B2A_PAIRPACK=0: never the pair-packed 1x16 fill (development knob: compare both)
  bool p16 = false;                // the staged batch runs the pair-packed fill (pair16_eligible)
  int32_t p16_bias = 0;
  uint32_t p16_stage = 0;          // its per-warp staging: y of both blocks

  // batch state
  bool staged = false, ran = false;
  bool score_only = false;         // the staged batch is a score-only one (b2a_score_batch): F_NOTB fill, score-only K2
  Plan plan;
  DevScoring sc{};
  int flags = 0, mode = 0;
  const FillLaunch* shape = nullptr;
  uint64_t n_pairs = 0, blob_bytes = 0;
  uint64_t h2d_bytes = 0;
  std::vector<int32_t> lut_host;
  std::vector<uint8_t> last_syms;  // alphabet used by the last stage (given or discovered)
  uint8_t codemap_host[256];

  DevBuf d_blob, d_xoff, d_xlen, d_yoff, d_ylen, d_order, d_pm, d_pn, d_blocks, d_seq, d_bnd, d_rows,
      d_rowm, d_tb, d_opsscratch, d_lut, d_codemap, d_ctl, d_score, d_xs, d_xe, d_ys, d_ye, d_nops,
      d_opssrc, d_clip, d_status, d_nops64, d_opsoff, d_opsdense, d_scan, d_records, d_prog, d_bcells, d_bstatus,
      d_bopsend, d_bslab, d_branges, d_broff, d_bfill, d_bfoff, d_hmoff, d_hmxy, d_hpoff, d_hpidx, d_raw, d_gnops,
      d_gnops64, d_goff, d_bcols, d_bstrip, d_bsoff, d_belig, d_lut16;
  uint32_t* h_nops = nullptr;  // pinned staging of b2a_gathered_fetch
  uint64_t h_nops_cap = 0;
  cudaEvent_t ev[6] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
  std::vector<cudaEvent_t> wave_ev;  // 3 per wave: fill start, fill stop / walk start, walk stop
  uint32_t launches = 0;
  int last_grid = 0;

  // software pipeline of b2a_align_batch: the batch is cut into chunks that alternate between two
  // child engines (own streams and buffers) so chunk c+1's H2D and host planning overlap chunk c's kernels
  int pipe_chunks = 5;
  struct PipeSlot {
    b2a_engine* eng = nullptr;
    uint64_t* h_opsoff = nullptr;  // pinned
    uint32_t* h_ctl = nullptr;     // pinned
    size_t h_cap = 0;
    std::vector<uint64_t> xoff, yoff;
    std::vector<uint8_t> packed;  // the chunk's sequences gathered from a scattered caller blob
    uint64_t lo = 0, n = 0;
    bool busy = false;
  } slots[3];
  static constexpr int kSlots = 3;

  int fail(int code, const std::string& what) {
    err = what;
    return code;
  }
  int cuda_fail(const char* what, cudaError_t e) {
    err = std::string(what) + ": " + cudaGetErrorString(e);
    return B2A_E_CUDA;
  }
};

#define CK(expr)                                              \
  do {                                                        \
    cudaError_t _e = (expr);                                  \
    if (_e != cudaSuccess) return e->cuda_fail(#expr, _e);    \
  } while (0)

namespace {

// 32-bit blocks a BitEnc of `len` symbols of `width` bits occupies (bitenc.rs:332-338: 32 - 32 % width usable
// bits per block)
inline uint64_t bitenc_blocks(uint64_t len, uint32_t width) {
  const uint64_t usable = 32 - 32 % width;
  return (len * width + usable - 1) / usable;
}

// BitEnc storage -> one byte per symbol (ranks), one warp per sequence (x and y of every pair)
__global__ void __launch_bounds__(128) unpack_bitenc_kernel(const uint32_t* __restrict__ blocks,
                                                             const uint64_t* __restrict__ x_block,
                                                             const uint64_t* __restrict__ y_block,
                                                             const uint64_t* __restrict__ x_off,
                                                             const uint64_t* __restrict__ y_off,
                                                             const uint32_t* __restrict__ x_len,
                                                             const uint32_t* __restrict__ y_len, uint64_t n_pairs,
                                                             uint32_t width, uint8_t* __restrict__ out) {
  const uint32_t usable = 32 - 32 % width, per_block = usable / width, mask = (1u << width) - 1u;
  const uint32_t lane = threadIdx.x & 31u;
  const uint64_t nwarps = ((uint64_t)gridDim.x * blockDim.x) >> 5;
  for (uint64_t t = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; t < 2 * n_pairs; t += nwarps) {
    const uint64_t p = t >> 1;
    const bool isy = t & 1;
    const uint32_t* src = blocks + (isy ? y_block[p] : x_block[p]);
    uint8_t* dst = out + (isy ? y_off[p] : x_off[p]);
    const uint32_t len = isy ? y_len[p] : x_len[p];
    for (uint32_t i = lane; i < len; i += 32) {
      const uint32_t blk = i / per_block, bit = (i % per_block) * width;  // bitenc.rs:319-321, 332-338
      dst[i] = (uint8_t)((src[blk] >> bit) & mask);
    }
  }
}

// pick the fill shape for a batch (measured crossover: see DESIGN.md "shape selection")
void choose_shape(const b2a_engine* e, uint32_t maxm, uint32_t maxn, uint64_t n_pairs, int* G, int* R) {
  if (e->tune_G && e->tune_R) {
    *G = e->tune_G;
    *R = e->tune_R;
    return;
  }
  const uint64_t stage1 = (uint64_t)((maxm + 15) / 16 * 16 + 64 + (maxn + 15) / 16 * 16 + 64) * 32 * fill_warps_of(1, 16);
  if (n_pairs >= 49152 && stage1 <= kMaxStageSmem && maxm <= 2048) {  // measured: 8x20 wins below ~50k reads of 150
    *G = 1;
    *R = 16;
  } else if ((n_pairs >= 4096 && maxm <= 4096) || maxm <= 161) {
    // four pairs to a warp: enough warps to fill the GPU (or a single strip anyway).  128-row or 160-row
    // strips, whichever pads the rows less: 10k reads of 150 run as one strip of 8x20 (7 % padding) at
    // 0.34 ms against 0.46 (2x16), 0.52 (8x16: two strips) and 0.68 (32x8) -- profiles/r02_small_batch_shapes.txt
    const uint64_t rows = maxm > 1 ? maxm - 1 : 1;
    const uint64_t pad16 = (rows + 127) / 128 * 128, pad20 = (rows + 159) / 160 * 160;
    *G = 8;
    *R = pad20 < pad16 ? 20 : 16;
  } else {
    // warp per pair, (pair, strip) tasks pipelined through the boundary row: fills the GPU from a few long
    // pairs.  16 rows per lane is ~15% faster per cell than 8 unless the 512-row strips pad m much more.
    *G = 32;
    const uint64_t rows = maxm > 1 ? maxm - 1 : 1;
    const uint64_t pad16 = (rows + 511) / 512 * 512, pad8 = (rows + 255) / 256 * 256;
    *R = (pad16 * 100 <= pad8 * 112) ? 16 : 8;
  }
}

int validate_scoring(b2a_engine* e, const b2a_scoring* s) {
  // the reference's constructor asserts (mod.rs:517-518, 554-571)
  if (s->gap_open > 0) return e->fail(B2A_E_INVALID, "gap_open can't be positive");
  if (s->gap_extend > 0) return e->fail(B2A_E_INVALID, "gap_extend can't be positive");
  if (s->xclip_prefix > 0) return e->fail(B2A_E_INVALID, "Clipping penalty (x prefix) can't be positive");
  if (s->xclip_suffix > 0) return e->fail(B2A_E_INVALID, "Clipping penalty (x suffix) can't be positive");
  if (s->yclip_prefix > 0) return e->fail(B2A_E_INVALID, "Clipping penalty (y prefix) can't be positive");
  if (s->yclip_suffix > 0) return e->fail(B2A_E_INVALID, "Clipping penalty (y suffix) can't be positive");
  const int32_t clips[4] = {s->xclip_prefix, s->xclip_suffix, s->yclip_prefix, s->yclip_suffix};
  for (int32_t c : clips)
    if (c < B2A_MIN_SCORE) return e->fail(B2A_E_RANGE, "clip penalty below MIN_SCORE");
  return B2A_OK;
}

}  // namespace

extern "C" {

const char* b2a_version(void) { return "b200align 0.1 (sm_100a)"; }

const char* b2a_last_error(const b2a_engine* e) { return e ? e->err.c_str() : "null engine"; }

int32_t b2a_engine_create(b2a_engine** out, int32_t device_id) {
  if (!out) return B2A_E_INVALID;
  *out = nullptr;
  int count = 0;
  cudaError_t ce = cudaGetDeviceCount(&count);
  if (ce != cudaSuccess || count <= 0 || device_id < 0 || device_id >= count) return B2A_E_NO_DEVICE;
  if (cudaSetDevice(device_id) != cudaSuccess) return B2A_E_NO_DEVICE;
  cudaDeviceProp prop;
  if (cudaGetDeviceProperties(&prop, device_id) != cudaSuccess) return B2A_E_NO_DEVICE;
  if (prop.major < 10) return B2A_E_NO_DEVICE;  // kernels are built for sm_100a only
  b2a_engine* e = new b2a_engine();
  e->device = device_id;
  e->num_sms = prop.multiProcessorCount;
  // (measured on 10k reads: K1 at 67 % issue and K2 at 36 % are both instruction-bound, and K2's CTAs displace K1's
  //  register-heavy ones: 0.571 ms overlapped against 0.558 ms back to back -- off unless asked for)
  e->overlap_small = false;
  if (const char* env = getenv("B2A_BANDED_LITERAL")) e->banded_fast = atoi(env) == 0;
  if (const char* env = getenv("B2A_BANDED_STRIP")) e->banded_strip = atoi(env) != 0;
  if (const char* env = getenv("B2A_BANDED_STRIP_LASTCOL")) e->banded_strip_lastcol = atoi(env) != 0;
  if (const char* env = getenv("B2A_OVERLAP")) e->overlap_small = atoi(env) != 0;
  if (const char* env = getenv("B2A_OVERLAP_BIG")) e->overlap_big = atoi(env) != 0;
  if (const char* env = getenv("B2A_TAIL_SPLIT")) e->tail_split = atoi(env) != 0;
  if (const char* env = getenv("B2A_NO_PACKREL")) e->no_packrel = atoi(env) != 0;
  if (const char* env = getenv("B2A_SPLIT_TIMING")) e->split_timing = atoi(env) != 0;
  if (const char* env = getenv("B2A_PAIRPACK")) e->pairpack = atoi(env) != 0;
  if (const char* env = getenv("B2A_WALK_CTA_WARPS")) {
    const int v = atoi(env);
    if (v == 1 || v == 2 || v == 4 || v == 8 || v == 16 || v == 32) e->walk_cta_warps = (uint32_t)v;
  }
  if (cudaStreamCreateWithFlags(&e->own_stream, cudaStreamNonBlocking) != cudaSuccess) {
    delete e;
    return B2A_E_CUDA;
  }
  e->stream = e->own_stream;
  for (auto& v : e->ev) cudaEventCreate(&v);
  *out = e;
  return B2A_OK;
}

int32_t b2a_engine_destroy(b2a_engine* e) {
  if (!e) return B2A_OK;
  cudaSetDevice(e->device);
  for (auto& sl : e->slots) {
    if (sl.h_opsoff) cudaFreeHost(sl.h_opsoff);
    if (sl.h_ctl) cudaFreeHost(sl.h_ctl);
    if (sl.eng) b2a_engine_destroy(sl.eng);
    sl.eng = nullptr;
  }
  cudaStreamSynchronize(e->stream);
  if (e->tail_stream) {
    cudaStreamSynchronize(e->tail_stream);
    cudaStreamDestroy(e->tail_stream);
  }
  if (e->ev_fill) cudaEventDestroy(e->ev_fill);
  if (e->aux_stream) {
    cudaStreamSynchronize(e->aux_stream);
    cudaStreamDestroy(e->aux_stream);
  }
  for (auto& v : e->sub_ev) cudaEventDestroy(v);
  if (e->h_plan) cudaFreeHost(e->h_plan);
  if (e->h_nops) cudaFreeHost(e->h_nops);
  DevBuf* bufs[] = {&e->d_blob, &e->d_xoff, &e->d_xlen, &e->d_yoff, &e->d_ylen, &e->d_order, &e->d_pm,
                    &e->d_pn, &e->d_blocks, &e->d_seq, &e->d_bnd, &e->d_rows, &e->d_rowm, &e->d_tb,
                    &e->d_opsscratch, &e->d_lut, &e->d_codemap, &e->d_ctl, &e->d_score, &e->d_xs,
                    &e->d_xe, &e->d_ys, &e->d_ye, &e->d_nops, &e->d_opssrc, &e->d_clip, &e->d_status,
                    &e->d_nops64, &e->d_opsoff, &e->d_opsdense, &e->d_scan, &e->d_records, &e->d_prog, &e->d_bcells,
                    &e->d_bstatus, &e->d_bopsend, &e->d_bslab, &e->d_branges, &e->d_broff, &e->d_bfill, &e->d_hmoff, &e->d_hmxy,
                    &e->d_hpoff, &e->d_hpidx, &e->d_raw, &e->d_gnops, &e->d_gnops64, &e->d_goff,
                    &e->d_bfoff, &e->d_bcols, &e->d_bstrip, &e->d_bsoff, &e->d_belig, &e->d_lut16};
  for (DevBuf* b : bufs) b->release();
  for (auto& v : e->ev)
    if (v) cudaEventDestroy(v);
  for (auto& v : e->wave_ev) cudaEventDestroy(v);
  if (e->own_stream) cudaStreamDestroy(e->own_stream);
  delete e;
  return B2A_OK;
}

int32_t b2a_engine_set_stream(b2a_engine* e, void* cuda_stream) {
  if (!e) return B2A_E_INVALID;
  e->stream = cuda_stream ? reinterpret_cast<cudaStream_t>(cuda_stream) : e->own_stream;
  return B2A_OK;
}

int32_t b2a_engine_set_traceback_budget(b2a_engine* e, uint64_t bytes) {
  if (!e) return B2A_E_INVALID;
  e->tb_budget = bytes;
  return B2A_OK;
}

int32_t b2a_engine_set_pipeline(b2a_engine* e, int32_t chunks) {
  if (!e) return B2A_E_INVALID;
  e->pipe_chunks = chunks < 2 ? 0 : (chunks > 64 ? 64 : chunks);
  return B2A_OK;
}

int32_t b2a_engine_last_alphabet(const b2a_engine* e, uint8_t* symbols, uint32_t* n_symbols) {
  if (!e || !symbols || !n_symbols) return B2A_E_INVALID;
  *n_symbols = (uint32_t)e->last_syms.size();
  for (size_t k = 0; k < e->last_syms.size() && k < 256; ++k) symbols[k] = e->last_syms[k];
  return B2A_OK;
}

int32_t b2a_engine_set_walk(b2a_engine* e, int32_t mode) {
  if (!e) return B2A_E_INVALID;
  if (mode < 0 || mode > 2) return e->fail(B2A_E_INVALID, "walk mode must be 0 (automatic), 1 (lane per pair) or 2 (warp per pair)");
  e->walk_mode = mode;
  return B2A_OK;
}

int32_t b2a_engine_set_tuning(b2a_engine* e, int32_t G, int32_t R) {
  if (!e) return B2A_E_INVALID;
  if (G == 0 && R == 0) {
    e->tune_G = e->tune_R = 0;
    return B2A_OK;
  }
  if (!find_shape(G, R)) return e->fail(B2A_E_INVALID, "fill shape (G,R) not built into this library");
  e->tune_G = G;
  e->tune_R = R;
  return B2A_OK;
}

}  // extern "C"

// Shared front half of a batch: validation (the reference's constructor asserts), clip presets, the
// i32 range guard, alphabet discovery + LUT, and the upload of the caller's blob.
static int32_t stage_front(b2a_engine* e, int32_t mode, const b2a_scoring* s, const b2a_pairs* pairs,
                           uint32_t& maxm, uint32_t& maxn, int64_t& score_bound) {
  if (!e || !s || !pairs) return B2A_E_INVALID;
  e->staged = e->ran = false;
  e->score_only = false;
  if (mode < 0 || mode > 3) return e->fail(B2A_E_INVALID, "mode must be B2A_MODE_*");
  int rc = validate_scoring(e, s);
  if (rc) return rc;
  if (cudaSetDevice(e->device) != cudaSuccess) return e->fail(B2A_E_NO_DEVICE, "cudaSetDevice failed");
  if (e->stage_nosync) {  // a previous stage's copies out of the pinned plan arena must have landed
    if (cudaStreamSynchronize(e->stream) != cudaSuccess) return e->fail(B2A_E_CUDA, "cudaStreamSynchronize failed");
  }
  const uint64_t n = pairs->n_pairs;
  if (n > 0x7ffffffeull) return e->fail(B2A_E_INVALID, "more than 2^31 - 2 pairs in one batch");
  e->n_pairs = n;
  e->mode = mode;

  // scoring with the mode's clip preset (mod.rs:935-938, 964-967, 996-999)
  DevScoring sc{};
  sc.gap_open = s->gap_open;
  sc.gap_extend = s->gap_extend;
  sc.xclip_prefix = s->xclip_prefix;
  sc.xclip_suffix = s->xclip_suffix;
  sc.yclip_prefix = s->yclip_prefix;
  sc.yclip_suffix = s->yclip_suffix;
  if (mode == B2A_MODE_GLOBAL) sc.xclip_prefix = sc.xclip_suffix = sc.yclip_prefix = sc.yclip_suffix = MIN_SCORE;
  if (mode == B2A_MODE_SEMIGLOBAL) {
    sc.xclip_prefix = sc.xclip_suffix = MIN_SCORE;
    sc.yclip_prefix = sc.yclip_suffix = 0;
  }
  if (mode == B2A_MODE_LOCAL) sc.xclip_prefix = sc.xclip_suffix = sc.yclip_prefix = sc.yclip_suffix = 0;
  sc.match_score = s->match_score;
  sc.mismatch_score = s->mismatch_score;
  sc.alpha = 0;

  // lengths / offsets sanity
  maxm = 0;
  maxn = 0;
  const uint32_t pw = e->packed_width;  // 0: bytes; else offsets and blob size are in 32-bit BitEnc blocks
  const uint64_t unit_total = pw ? pairs->blob_bytes / 4 : pairs->blob_bytes;
  for (uint64_t p = 0; p < n; ++p) {
    // offset + length may not wrap: compare each against what is left of the blob
    const uint64_t bb = unit_total, xo = pairs->x_off[p], yo = pairs->y_off[p];
    const uint64_t xu = pw ? bitenc_blocks(pairs->x_len[p], pw) : pairs->x_len[p];
    const uint64_t yu = pw ? bitenc_blocks(pairs->y_len[p], pw) : pairs->y_len[p];
    if (xo > bb || xu > bb - xo || yo > bb || yu > bb - yo)
      return e->fail(B2A_E_INVALID, "sequence offset/length outside seq_blob");
    maxm = std::max(maxm, pairs->x_len[p]);
    maxn = std::max(maxn, pairs->y_len[p]);
  }
  if (maxm > (1u << 24) || maxn > (1u << 24)) return e->fail(B2A_E_RANGE, "sequence longer than 2^24");

  // The alphabet: given by the caller, else found on the device (one flat pass over the blob).
  // Both MatchParams and tabulated MatchFuncs then run from a compact LUT in shared memory;
  // MatchParams over more than 64 distinct bytes falls back to compare/select in the kernel.
  cudaStream_t st = e->stream;
  e->blob_bytes = pairs->blob_bytes;
  e->h2d_bytes = 0;
  auto up = [&](DevBuf& bf, const void* src, size_t bytes) -> cudaError_t {
    e->h2d_bytes += bytes;
    return bytes ? cudaMemcpyAsync(bf.p, src, bytes, cudaMemcpyHostToDevice, st) : cudaSuccess;
  };
  CK(e->d_ctl.reserve(2048));
  bool present[256] = {false};
  if (pw) {
    // BitEnc storage in, one byte per symbol on the device: the packed blocks are what crosses PCIe (4x fewer
    // bytes at width 2), an unpack pass writes the byte blob K0 / K4 read, at 16-byte aligned offsets of our own
    e->eff_xoff.resize(n);
    e->eff_yoff.resize(n);
    uint64_t pos = 0;
    for (uint64_t p = 0; p < n; ++p) {
      e->eff_xoff[p] = pos;
      pos += ((uint64_t)pairs->x_len[p] + 15) & ~15ull;
      e->eff_yoff[p] = pos;
      pos += ((uint64_t)pairs->y_len[p] + 15) & ~15ull;
    }
    e->blob_bytes = pos;
    CK(e->d_raw.reserve(pairs->blob_bytes + 16));
    CK(e->d_blob.reserve(pos + 16));
    CK(e->d_xoff.reserve(n * 8 + 8));
    CK(e->d_yoff.reserve(n * 8 + 8));
    CK(e->d_xlen.reserve(n * 4 + 4));
    CK(e->d_ylen.reserve(n * 4 + 4));
    CK(e->d_opssrc.reserve(n * 8 + 8));
    CK(e->d_nops64.reserve((n + 1) * 8));
    CK(up(e->d_raw, pairs->seq_blob, pairs->blob_bytes));
    // block indices ride in two scratch arrays that are not in use yet (d_opssrc, d_nops64)
    CK(up(e->d_opssrc, pairs->x_off, n * 8));
    CK(up(e->d_nops64, pairs->y_off, n * 8));
    CK(up(e->d_xoff, e->eff_xoff.data(), n * 8));
    CK(up(e->d_yoff, e->eff_yoff.data(), n * 8));
    CK(up(e->d_xlen, pairs->x_len, n * 4));
    CK(up(e->d_ylen, pairs->y_len, n * 4));
    if (n) {
      unpack_bitenc_kernel<<<(unsigned)std::min<uint64_t>((2 * n + 3) / 4, 1u << 20), 128, 0, st>>>(
          e->d_raw.as<uint32_t>(), e->d_opssrc.as<uint64_t>(), e->d_nops64.as<uint64_t>(), e->d_xoff.as<uint64_t>(),
          e->d_yoff.as<uint64_t>(), e->d_xlen.as<uint32_t>(), e->d_ylen.as<uint32_t>(), n, pw, e->d_blob.as<uint8_t>());
      CK(cudaGetLastError());
    }
    CK(cudaStreamSynchronize(st));  // eff_xoff / eff_yoff are pageable vectors reused by the next call
    if (!(s->alphabet && s->alphabet_len))
      for (uint32_t k = 0; k < (1u << pw); ++k) present[k] = true;  // the ranks a BitEnc of this width can hold
  } else {
    CK(e->d_blob.reserve(pairs->blob_bytes + 16));
    CK(up(e->d_blob, pairs->seq_blob, pairs->blob_bytes));
  }
  if (s->alphabet && s->alphabet_len) {  // caller-supplied alphabet (tabulated MatchFunc or MatchParams alike)
    for (uint32_t k = 0; k < s->alphabet_len; ++k) present[s->alphabet[k]] = true;
  } else if (!pw) {
    uint32_t* flags = e->d_ctl.as<uint32_t>() + 256;  // 256 words
    CK(cudaMemsetAsync(flags, 0, 1024, st));
    if (pairs->blob_bytes) {
      symbols_kernel<<<e->num_sms * 8, 256, 0, st>>>(e->d_blob.as<uint8_t>(), pairs->blob_bytes, flags);
      CK(cudaGetLastError());
    }
    uint32_t hflags[256];
    CK(cudaMemcpyAsync(hflags, flags, 1024, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    for (int k = 0; k < 256; ++k) present[k] = hflags[k] != 0;
  }
  std::vector<int> syms;
  for (int k = 0; k < 256; ++k)
    if (present[k]) syms.push_back(k);
  if (syms.empty()) syms.push_back(0);
  e->last_syms.assign(syms.begin(), syms.end());
  int64_t maxabs = std::max<int64_t>(std::llabs((long long)s->match_score), std::llabs((long long)s->mismatch_score));
  for (int k = 0; k < 256; ++k) e->codemap_host[k] = (uint8_t)k;
  e->lut_host.clear();
  if (s->table && (int)syms.size() > kMaxAlphaTable)
    return e->fail(B2A_E_UNSUPPORTED, "MatchFunc table over more than 128 distinct symbols");
  if ((int)syms.size() <= (s->table ? kMaxAlphaTable : kMaxAlpha)) {
    sc.alpha = (int32_t)syms.size();
    for (int k = 0; k < 256; ++k) e->codemap_host[k] = 0xFF;
    for (int a = 0; a < sc.alpha; ++a) e->codemap_host[syms[a]] = (uint8_t)a;
    const size_t aa = (size_t)sc.alpha * sc.alpha;
    e->lut_host.resize(aa + (size_t)lut_entries(sc.alpha));  // [plain | 4*v+3 for K1's packed domain + its poison row]
    if (s->table) maxabs = 0;
    for (int a = 0; a < sc.alpha; ++a)
      for (int b = 0; b < sc.alpha; ++b) {
        const int32_t v = s->table ? s->table[syms[a] * 256 + syms[b]]
                                   : (a == b ? s->match_score : s->mismatch_score);
        e->lut_host[(size_t)a * sc.alpha + b] = v;
        maxabs = std::max<int64_t>(maxabs, std::llabs((long long)v));
      }
    if (maxabs > (1ll << 27)) return e->fail(B2A_E_RANGE, "substitution score magnitude above 2^27");
    // K1's copy: packed domain (4*v + 3 = "diagonal" priority) minus the open bias S carries there
    for (size_t k = 0; k < aa; ++k) e->lut_host[aa + k] = 4 * e->lut_host[k] + 3 - (4 * sc.gap_open + 1);
    for (size_t k = aa; k < (size_t)lut_entries(sc.alpha); ++k) e->lut_host[aa + k] = LUT_POISON;
  }
  score_bound = 0;
  // i32 range guard: every S/I/D of a real path stays within +-2^27, so MIN_SCORE-based
  // sentinels can neither win nor overflow (the reference would silently wrap)
  {
    const int64_t unit = std::max<int64_t>(maxabs, std::max<int64_t>(-(int64_t)sc.gap_open, -(int64_t)sc.gap_extend));
    const int64_t bound = ((int64_t)maxm + maxn + 2) * unit - (int64_t)sc.gap_open;
    score_bound = bound;
    if (bound > (1ll << 27)) return e->fail(B2A_E_RANGE, "scores x lengths exceed the i32-safe range (2^27)");
    const int32_t clips[4] = {sc.xclip_prefix, sc.xclip_suffix, sc.yclip_prefix, sc.yclip_suffix};
    for (int32_t c : clips)
      if (c > DEAD_CLIP && -(int64_t)c > (1ll << 27))
        return e->fail(B2A_E_RANGE, "clip penalty between -2^27 and MIN_SCORE/2 is not supported");
  }
  e->sc = sc;
  e->flags = scoring_flags(sc, score_bound, maxm, maxn);
  if (e->no_packrel) e->flags &= ~F_PACKREL;  // (test knob: the explicit (value, index) trackers for long sequences)

  return B2A_OK;
}

// ops compaction shared by the full and the banded path: widen -> exclusive scan -> gather
static int32_t compact_ops(b2a_engine* e, uint64_t scratch_bytes, cudaStream_t st) {
  const uint64_t n = e->n_pairs;
  if (n) {
    if (n <= 65536) {  // small batches: one single-CTA launch for the offsets
      scan_small_kernel<<<1, 1024, 0, st>>>(e->d_nops.as<uint32_t>(), e->d_opsoff.as<uint64_t>(), (uint32_t)n);
      CK(cudaGetLastError());
    } else {
    const unsigned g1 = (unsigned)((n + 1 + 255) / 256);
    widen_kernel<<<g1, 256, 0, st>>>(e->d_nops.as<uint32_t>(), e->d_nops64.as<uint64_t>(), n);
    CK(cudaGetLastError());
    size_t tmp = 0;
    CK(cub::DeviceScan::ExclusiveSum(nullptr, tmp, e->d_nops64.as<uint64_t>(), e->d_opsoff.as<uint64_t>(),
                                     (int64_t)(n + 1), st));
    CK(e->d_scan.reserve(tmp + 16));
    CK(cub::DeviceScan::ExclusiveSum(e->d_scan.p, tmp, e->d_nops64.as<uint64_t>(),
                                     e->d_opsoff.as<uint64_t>(), (int64_t)(n + 1), st));
    }
    // worst case every pair emits m+n+4 ops; size the dense buffer by the scratch size
    CK(e->d_opsdense.reserve(scratch_bytes + 16));
    const unsigned g2 = (unsigned)((n * 32 + 255) / 256);
    gather_ops_kernel<<<g2, 256, 0, st>>>(e->d_opsscratch.as<uint8_t>(), e->d_opssrc.as<uint64_t>(),
                                          e->d_opsoff.as<uint64_t>(), e->d_opsdense.as<uint8_t>(), n);
    CK(cudaGetLastError());
    e->launches += n <= 65536 ? 2 : 4;
  }
  return B2A_OK;
}

// The pair-packed fill (b2a_fill_pair16.cuh) carries every value in 16 bits: it runs a wave of the 1x16 local
// fill only when the wave is one shape small enough for that.  Returns the bias of its score domain, or -1.
static int32_t pair16_eligible(const b2a_engine* e, const Plan& pl, int G, int R) {
  const DevScoring& sc = e->sc;
  if (!e->pairpack || G != 1 || R != 16 || e->flags != P16_FLAGS) return -1;
  if (sc.alpha < 1 || sc.alpha > P16_MAX_ALPHA || pl.maxm > 256 || pl.maxn > 255 || pl.blocks.empty()) return -1;
  for (uint64_t i = 0; i < pl.n_pairs; ++i)  // one shape: the two blocks of a task share their loop bounds
    if (pl.pm[i] != pl.maxm || pl.pn[i] != pl.maxn) return -1;
  int32_t lo = e->lut_host[0], hi = e->lut_host[0];
  for (int k = 0; k < sc.alpha * sc.alpha; ++k) {
    lo = std::min(lo, e->lut_host[k]);
    hi = std::max(hi, e->lut_host[k]);
  }
  // a local score never exceeds min(m, n) substitutions at the best score: the tracker keys hold it in 8 bits
  if ((int64_t)std::min(pl.maxm, pl.maxn) * std::max(hi, 0) > 255) return -1;
  if (sc.gap_open < -2048 || sc.gap_extend < -2048 || lo < -2048) return -1;  // stored values stay below 2^14
  return 4 * std::max(std::max(-sc.gap_open, -lo), 0);
}

// K1 of a wave (or a part of one): the pair-packed fill when the batch was staged for it, else the int32 shape
static cudaError_t launch_fill(b2a_engine* e, const FillParams& fp, uint32_t ntasks, cudaStream_t st, int* grid_out,
                               int dry) {
  if (e->p16) {
    FillParams f = fp;
    f.lut = e->d_lut16.as<int32_t>();
    f.smem_seq_bytes = e->p16_stage;
    return launch_fill_pair16(f, e->p16_bias, e->score_only, e->num_sms, st, grid_out, dry);
  }
  return e->shape->launch(e->flags | (e->score_only ? F_NOTB : 0), fp, ntasks, e->num_sms, st, grid_out, dry);
}

// Stage a batch for b2a_batch_run: the full batch, or (score_only) the score-only one of b2a_score_batch, which
// fills without the traceback (one wave, no traceback arena) and runs the score-only K2 without ops.
static int32_t batch_stage(b2a_engine* e, int32_t mode, const b2a_scoring* s, const b2a_pairs* pairs, bool score_only) {
  if (!e || !s || !pairs) return B2A_E_INVALID;
  uint32_t maxm = 0, maxn = 0;
  int64_t score_bound = 0;
  int rc = stage_front(e, mode, s, pairs, maxm, maxn, score_bound);
  if (rc) return rc;
  e->score_only = score_only;
  const uint64_t n = e->n_pairs;
  const DevScoring sc = e->sc;
  cudaStream_t st = e->stream;
  auto up = [&](DevBuf& bf, const void* src, size_t bytes) -> cudaError_t {
    e->h2d_bytes += bytes;
    return bytes ? cudaMemcpyAsync(bf.p, src, bytes, cudaMemcpyHostToDevice, st) : cudaSuccess;
  };
  // shape + plan
  int G = 1, R = 16;
  choose_shape(e, maxm, maxn, n, &G, &R);
  uint64_t budget = e->tb_budget;
  if (!budget) {
    size_t fr = 0, tot = 0;
    CK(cudaMemGetInfo(&fr, &tot));
    budget = (uint64_t)((double)fr * 0.6);
  }
  const uint32_t lut_bytes = sc.alpha ? lut_smem_bytes(sc.alpha) : 0u;
  for (int attempt = 0;; ++attempt) {
    e->shape = find_shape(G, R);
    if (!e->shape) return e->fail(B2A_E_INVALID, "no fill kernel for the requested shape");
    build_plan(e->plan, pairs->x_len, pairs->y_len, n, G, R, budget, score_only);
    if (64 + lut_bytes + (uint64_t)fill_warps_of(G, R) * e->plan.smem_seq_bytes <= kMaxStageSmem) break;
    // Shapes with several pairs per warp stage 32/G whole (x, y) per warp; long sequences (a read against a
    // 15 kb reference ...) only fit the warp-per-pair shape, which stages one strip of x and one y per warp
    // (n up to ~50,000 symbols: 4 warps x (n + G*R + padding) bytes <= 200 KB).  Forced shapes are not replaced.
    if ((e->tune_G && e->tune_R) || G == 32 || attempt > 0)
      return e->fail(B2A_E_UNSUPPORTED, "sequences too long for on-chip staging with this fill shape");
    G = 32;
    const uint64_t rows = maxm > 1 ? maxm - 1 : 1;
    const uint64_t pad16 = (rows + 511) / 512 * 512, pad8 = (rows + 255) / 256 * 256;
    R = (pad16 * 100 <= pad8 * 112) ? 16 : 8;
  }
  const Plan& pl = e->plan;
  const int32_t p16_bias = pair16_eligible(e, pl, G, R);
  e->p16 = p16_bias >= 0;
  e->p16_bias = e->p16 ? p16_bias : 0;
  e->p16_stage = e->p16 ? 2 * pl.blocks[0].ywords * 32 * 4 : 0;
  std::vector<int32_t> lut16;
  if (e->p16) {
    lut16.resize((size_t)p16_lut_entries(sc.alpha));
    p16_build_lut(e->lut_host.data() + (size_t)sc.alpha * sc.alpha, sc.alpha, lut16.data());
    CK(e->d_lut16.reserve(lut16.size() * 4 + 16));
  }

  // device memory
  CK(e->d_xoff.reserve(n * 8 + 8));
  CK(e->d_yoff.reserve(n * 8 + 8));
  CK(e->d_xlen.reserve(n * 4 + 4));
  CK(e->d_ylen.reserve(n * 4 + 4));
  CK(e->d_order.reserve(n * 4 + 4));
  CK(e->d_pm.reserve(n * 4 + 4));
  CK(e->d_pn.reserve(n * 4 + 4));
  CK(e->d_blocks.reserve(pl.blocks.size() * sizeof(Block) + 8));
  CK(e->d_seq.reserve(pl.seq_bytes + 16));
  CK(e->d_bnd.reserve(pl.max_bnd + 16));
  CK(e->d_rows.reserve(pl.max_rows + 16));
  CK(e->d_rowm.reserve(pl.max_rowm + 16));
  CK(e->d_tb.reserve(pl.max_tb + 16));
  CK(e->d_prog.reserve(pl.max_strip_tasks * 4 + 16));
  CK(e->d_lut.reserve(e->lut_host.size() * 4 + 16));
  CK(e->d_codemap.reserve(256));
  CK(e->d_score.reserve(n * 4 + 4));
  CK(e->d_xe.reserve(n * 4 + 4));
  CK(e->d_ye.reserve(n * 4 + 4));
  CK(e->d_status.reserve(n * 4 + 4));
  if (!score_only) {  // the ops and the start coordinates of the full path
    CK(e->d_opsscratch.reserve(pl.ops_bytes + 16));
    CK(e->d_xs.reserve(n * 4 + 4));
    CK(e->d_ys.reserve(n * 4 + 4));
    CK(e->d_nops.reserve(n * 4 + 4));
    CK(e->d_opssrc.reserve(n * 8 + 8));
    CK(e->d_clip.reserve(n * 16 + 16));
    CK(e->d_nops64.reserve((n + 1) * 8));
    CK(e->d_opsoff.reserve((n + 1) * 8));
  }

  // host -> device.  The plan vectors go through a pinned staging arena so that their copies are truly
  // asynchronous (a copy from pageable memory first waits for the stream: it would serialise the host with the
  // blob's H2D in the chunk pipeline).
  if (!e->packed_width) {  // (packed input: stage_front already placed offsets and lengths)
    CK(up(e->d_xoff, pairs->x_off, n * 8));
    CK(up(e->d_yoff, pairs->y_off, n * 8));
    CK(up(e->d_xlen, pairs->x_len, n * 4));
    CK(up(e->d_ylen, pairs->y_len, n * 4));
  }
  {
    const size_t blocks_bytes = pl.blocks.size() * sizeof(Block), lut_b = e->lut_host.size() * 4;
    const size_t need = 3 * n * 4 + blocks_bytes + 256 + lut_b + lut16.size() * 4 + 80;
    if (e->h_plan_cap < need) {
      if (e->h_plan) cudaFreeHost(e->h_plan);
      e->h_plan = nullptr;
      e->h_plan_cap = 0;
      CK(cudaMallocHost(&e->h_plan, need + need / 4));
      e->h_plan_cap = need + need / 4;
    }
    size_t pos = 0;
    auto up_staged = [&](DevBuf& bf, const void* src, size_t bytes) -> cudaError_t {
      if (!bytes) return cudaSuccess;
      std::memcpy(e->h_plan + pos, src, bytes);
      const cudaError_t ce = up(bf, e->h_plan + pos, bytes);
      pos += (bytes + 15) & ~(size_t)15;
      return ce;
    };
    CK(up_staged(e->d_order, pl.order.data(), n * 4));
    CK(up_staged(e->d_pm, pl.pm.data(), n * 4));
    CK(up_staged(e->d_pn, pl.pn.data(), n * 4));
    CK(up_staged(e->d_blocks, pl.blocks.data(), blocks_bytes));
    CK(up_staged(e->d_codemap, e->codemap_host, 256));
    if (lut_b) CK(up_staged(e->d_lut, e->lut_host.data(), lut_b));
    if (!lut16.empty()) CK(up_staged(e->d_lut16, lut16.data(), lut16.size() * 4));
  }
  // the caller's arrays are read by the copies above: wait for them unless the caller (the chunk pipeline of
  // b2a_align_batch) keeps them alive itself
  if (!e->stage_nosync) CK(cudaStreamSynchronize(st));
  e->staged = true;
  return B2A_OK;
}

extern "C" {

int32_t b2a_batch_stage(b2a_engine* e, int32_t mode, const b2a_scoring* s, const b2a_pairs* pairs) {
  return batch_stage(e, mode, s, pairs, false);
}

int32_t b2a_batch_run(b2a_engine* e) {
  if (!e) return B2A_E_INVALID;
  if (!e->staged) return e->fail(B2A_E_STATE, "b2a_batch_run before b2a_batch_stage");
  if (cudaSetDevice(e->device) != cudaSuccess) return e->fail(B2A_E_NO_DEVICE, "cudaSetDevice failed");
  const Plan& pl = e->plan;
  cudaStream_t st = e->stream;
  // pipeline slots put K2 and what follows on their high-priority stream (several waves share scratch: one stream)
  const bool use_tail = e->is_slot && e->tail_stream != nullptr && pl.waves.size() == 1;
  e->tail_used = use_tail;
  e->launches = 0;
  uint32_t* ctl = e->d_ctl.as<uint32_t>();  // [0] bad symbol, [1] walk error, [2..] per-wave task counters
  CK(cudaMemsetAsync(ctl, 0, 256, st));
  CK(cudaEventRecord(e->ev[0], st));
  if (!pl.blocks.empty()) {
    PackParams pk{};
    pk.blocks = e->d_blocks.as<Block>();
    pk.order = e->d_order.as<uint32_t>();
    pk.blob = e->d_blob.as<uint8_t>();
    pk.x_off = e->d_xoff.as<uint64_t>();
    pk.x_len = e->d_xlen.as<uint32_t>();
    pk.y_off = e->d_yoff.as<uint64_t>();
    pk.y_len = e->d_ylen.as<uint32_t>();
    pk.codemap = e->d_codemap.as<uint8_t>();
    pk.seq = e->d_seq.as<uint8_t>();
    pk.bad_symbol = ctl;
    pk.G = pl.G;
    pack_kernel<<<(unsigned)pl.blocks.size(), 256, 0, st>>>(pk);
    CK(cudaGetLastError());
    ++e->launches;
  }
  CK(cudaEventRecord(e->ev[1], st));
  size_t wi = 0;
  for (const Wave& w : pl.waves) {
    const uint32_t nb = w.block_hi - w.block_lo;
    if (wi >= 60) return e->fail(B2A_E_UNSUPPORTED, "more than 60 traceback waves; raise the budget");
    FillParams fp{};
    fp.blocks = e->d_blocks.as<Block>() + w.block_lo;
    fp.nblocks = nb;
    fp.pm = e->d_pm.as<uint32_t>();
    fp.pn = e->d_pn.as<uint32_t>();
    fp.seq = e->d_seq.as<uint8_t>();
    fp.bnd = e->d_bnd.as<uint8_t>();
    fp.rows = e->d_rows.as<uint8_t>();
    fp.tb = e->d_tb.as<uint8_t>();
    fp.lut = e->d_lut.as<int32_t>() + (size_t)e->sc.alpha * e->sc.alpha;  // the scaled copy
    fp.task_counter = ctl + 2 + wi;
    fp.smem_seq_bytes = pl.smem_seq_bytes;
    fp.one = 1;
    fp.ge4 = 4 * e->sc.gap_extend;
    uint32_t fill_tasks = nb * (uint32_t)pl.G;
    if (pl.G == 32 && w.strip_tasks >= 0x7fffffffull) return e->fail(B2A_E_RANGE, "too many strip tasks in one wave");
    if (pl.G == 32 && w.strip_tasks > 0) {
      // warp-per-pair shape: the strips of a pair are separate tasks that pipeline through the boundary row
      // (b2a_fill.cuh "strip-pipelined mode"), so a few long pairs still fill the GPU
      fp.progress = e->d_prog.as<uint32_t>();
      fp.n_strip_tasks = (uint32_t)w.strip_tasks;
      fill_tasks = fp.n_strip_tasks;
      CK(cudaMemsetAsync(fp.progress, 0, (size_t)w.strip_tasks * 4, st));
    }
    fp.sc = e->sc;
    while (e->wave_ev.size() < 3 * (wi + 1)) {
      cudaEvent_t v;
      CK(cudaEventCreate(&v));
      e->wave_ev.push_back(v);
    }
    WalkParams wp{};
    wp.blocks = fp.blocks;
    wp.nblocks = nb;
    wp.pm = fp.pm;
    wp.pn = fp.pn;
    wp.order = e->d_order.as<uint32_t>();
    wp.seq = fp.seq;
    wp.bnd = fp.bnd;
    wp.rows = fp.rows;
    wp.rowm = e->d_rowm.as<uint8_t>();
    wp.tb = fp.tb;
    wp.ops_scratch = e->d_opsscratch.as<uint8_t>();
    wp.lut = e->d_lut.as<int32_t>();  // the unscaled copy
    wp.sc = e->sc;
    wp.G = pl.G;
    wp.R = pl.R;
    wp.packtrk = (e->flags & F_PACKTRK) ? 1 : 0;
    wp.filter_clips = (e->mode == B2A_MODE_SEMIGLOBAL || e->mode == B2A_MODE_LOCAL) ? 1 : 0;
    wp.score = e->d_score.as<int32_t>();
    wp.xstart = e->d_xs.as<uint32_t>();
    wp.xend = e->d_xe.as<uint32_t>();
    wp.ystart = e->d_ys.as<uint32_t>();
    wp.yend = e->d_ye.as<uint32_t>();
    wp.n_ops = e->d_nops.as<uint32_t>();
    wp.ops_src = e->d_opssrc.as<uint64_t>();
    wp.clip_len = e->d_clip.as<uint32_t>();
    wp.status = e->d_status.as<uint32_t>();
    wp.err_flag = ctl + 1;
    // (running K2 inside K1's warps was measured: 28.4 ms vs 22.4 + 3.2 ms separately -- the latency-bound
    //  walk holds one of only 12 resident warps per SM; K2 stays its own launch)
    const bool fuse = false;
    // K2 in its two forms: the walk, or the score-only epilogue (row m, fix-ups, end walk) of a score-only batch
    void (*const k2_warp)(const WalkParams) = e->score_only ? score_warp_kernel : walk_warp_kernel;
    void (*const k2_lane)(const WalkParams) = e->score_only ? score_kernel : walk_kernel;
    fp.task_limit = (pl.G == 32) ? 0u : e->fill_task_limit;  // strip-pipelined tasks need the persistent grid
    const uint64_t wave_pairs = (uint64_t)nb * 32;
    const bool warp_walk = e->walk_mode == 2 || (e->walk_mode == 0 && wave_pairs <= kWarpWalkMaxPairs);
    uint32_t per_warp_smem = 0;
    // warps (pairs of one 32-pair block) per CTA of the warp-per-pair K2: the block's scratch is laid out
    // [index][pair], so the pairs of a CTA share the sectors they read through L1
    // (10k reads: 8 warps 0.134 ms, 4 warps 0.159, 16 warps 0.142, 32 warps 0.155 -- profiles/r02_10k_target.txt)
    uint32_t wcta_warps = e->walk_cta_warps;
    if (warp_walk) {
      // the pair's x and y are copied into shared memory when the CTA's pairs' worth fits its budget
      const uint32_t per_warp = ((pl.maxm + 3) / 4 + (pl.maxn + 3) / 4) * 4 + 16;
      if (!wcta_warps) wcta_warps = (uint64_t)per_warp * 8 <= 96 * 1024 ? 8u : 4u;
      per_warp_smem = (uint64_t)per_warp * wcta_warps <= 96 * 1024 ? per_warp : 0u;
      if ((size_t)per_warp_smem * wcta_warps > 48 * 1024)
        CK(cudaFuncSetAttribute(k2_warp, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(per_warp_smem * wcta_warps)));
    }
    if (!wcta_warps) wcta_warps = 4;
    wp.seq_smem_per_warp = per_warp_smem;
    // Small batches (a few thousand pairs: neither kernel fills the GPU): the wave is cut into sub-ranges of
    // blocks whose fills alternate between two streams (they overlap: the next fill's CTAs take the SM slots the
    // previous one's leave) and whose walks run on a high-priority stream as soon as their own fill is done --
    // K2 of sub-range s overlaps K1 of sub-range s+1, and only the last sub-range's K2 is exposed.
    // The same cut pays for LARGE batches with the lane-per-pair K2 (B2A_OVERLAP_BIG): K2 is latency/bandwidth-bound
    // (12 % of the 1M-pair step) and hides under the next sub-range's fill.
    const bool overlap_big = e->overlap_big && pl.waves.size() == 1 && !warp_walk && pl.G != 32 && nb >= 4096 && !use_tail;
    const bool overlap = overlap_big || (e->overlap_small && pl.waves.size() == 1 && warp_walk && pl.G != 32 && nb >= 64 &&
                                         !use_tail && e->walk_mode != 1);
    // Tail-aware split (small batches of equal tasks): the persistent fill runs whole rounds of one task per
    // resident warp; what is left over is a thin last round (10k reads on 8x20: 2,500 tasks on 1,184 warps = two
    // rounds + 132 tasks that take 0.07 ms with the SMs 7/8 idle).  The pairs of the whole rounds (A) and the
    // remainder (B) are filled back to back, and K2 of A runs beside the fill of B: B's few CTAs go out on the
    // high-priority stream first, A's walk takes the rest of the GPU.
    uint32_t split_b = 0;  // blocks of part A (0: no split)
    if (e->tail_split && !e->p16 && !overlap && pl.waves.size() == 1 && warp_walk && pl.G != 32 && !use_tail && e->walk_mode != 1 &&
        fp.task_limit == 0) {
      int resident = 0;
      CK(launch_fill(e, fp, fill_tasks, st, &resident, 1));
      const uint32_t slots = (uint32_t)resident, tasks = fill_tasks;
      if (slots > 0 && tasks > slots) {
        const uint32_t rounds = tasks / slots, rem = tasks % slots;
        const uint32_t a_blocks = (uint32_t)((uint64_t)rounds * slots / (uint32_t)pl.G);
        // (measured: 10k reads, a remainder of 0.11 rounds: 0.506 -> 0.464 ms; 7k reads, 0.48 rounds: 0.391 -> 0.411)
        if (rem > 0 && rounds <= 6 && rem * 4 <= slots && a_blocks > 0 && a_blocks < nb) split_b = a_blocks;
      }
    }
    if (split_b) {
      if (!e->tail_stream) {
        int lo_pri = 0, hi_pri = 0;
        cudaDeviceGetStreamPriorityRange(&lo_pri, &hi_pri);
        CK(cudaStreamCreateWithPriority(&e->tail_stream, cudaStreamNonBlocking, hi_pri));
        CK(cudaEventCreateWithFlags(&e->ev_fill, cudaEventDisableTiming));
      }
      if (!e->aux_stream) CK(cudaStreamCreateWithFlags(&e->aux_stream, cudaStreamNonBlocking));
      while (e->sub_ev.size() < 6) {
        cudaEvent_t v;
        CK(cudaEventCreateWithFlags(&v, cudaEventDisableTiming));
        e->sub_ev.push_back(v);
      }
      CK(cudaEventRecord(e->wave_ev[3 * wi + 0], st));
      FillParams fa = fp, fb = fp;
      fa.nblocks = split_b;
      fb.blocks = fp.blocks + split_b;
      fb.nblocks = nb - split_b;
      fb.task_counter = ctl + 8;
      WalkParams wa = wp, wb = wp;
      wa.nblocks = split_b;
      wb.blocks = wp.blocks + split_b;
      wb.nblocks = nb - split_b;
      if (e->split_timing && !e->split_ev[0])
        for (auto& v : e->split_ev) CK(cudaEventCreate(&v));
      if (e->split_timing) CK(cudaEventRecord(e->split_ev[0], st));
      CK(launch_fill(e, fa, fa.nblocks * (uint32_t)pl.G, st, &e->last_grid, 0));
      if (e->split_timing) CK(cudaEventRecord(e->split_ev[1], st));
      CK(cudaEventRecord(e->sub_ev[0], st));  // fill A done
      // fill B + walk B on the high-priority stream, walk A on the auxiliary one
      // (measured, profiles/r02_10k_target.txt: beside walk A the fill of B takes 144 us instead of 86 -- walk A's 64
      //  resident warps per SM crowd it -- so B's chain, +186 us, ends the step; walk A at a quarter of its occupancy
      //  frees B (+100 us) but then takes +246 us itself; swapping the stream priorities changes nothing)
      cudaStream_t sB = e->tail_stream, sA = e->aux_stream;
      CK(cudaStreamWaitEvent(sB, e->sub_ev[0], 0));
      CK(cudaStreamWaitEvent(sA, e->sub_ev[0], 0));
      CK(launch_fill(e, fb, fb.nblocks * (uint32_t)pl.G, sB, nullptr, 0));
      CK(cudaEventRecord(e->wave_ev[3 * wi + 1], sB));  // every fill has finished
      if (e->split_timing) CK(cudaEventRecord(e->split_ev[2], sB));
      k2_warp<<<wa.nblocks * 32 / wcta_warps, wcta_warps * 32, (size_t)per_warp_smem * wcta_warps, sA>>>(wa);
      CK(cudaGetLastError());
      if (e->split_timing) CK(cudaEventRecord(e->split_ev[3], sA));
      k2_warp<<<wb.nblocks * 32 / wcta_warps, wcta_warps * 32, (size_t)per_warp_smem * wcta_warps, sB>>>(wb);
      CK(cudaGetLastError());
      if (e->split_timing) CK(cudaEventRecord(e->split_ev[4], sB));
      e->split_ran = true;
      e->launches += 4;
      CK(cudaEventRecord(e->sub_ev[1], e->aux_stream));
      CK(cudaEventRecord(e->sub_ev[2], e->tail_stream));
      CK(cudaStreamWaitEvent(st, e->sub_ev[1], 0));  // everything rejoins the engine's stream
      CK(cudaStreamWaitEvent(st, e->sub_ev[2], 0));
      e->last_walk_warp = true;
      CK(cudaEventRecord(e->wave_ev[3 * wi + 2], st));
      ++wi;
      continue;
    }
    if (overlap) {
      constexpr int kSub = 4;
      if (!e->tail_stream) {
        int lo_pri = 0, hi_pri = 0;
        cudaDeviceGetStreamPriorityRange(&lo_pri, &hi_pri);
        CK(cudaStreamCreateWithPriority(&e->tail_stream, cudaStreamNonBlocking, hi_pri));
        CK(cudaEventCreateWithFlags(&e->ev_fill, cudaEventDisableTiming));
      }
      if (!e->aux_stream) CK(cudaStreamCreateWithFlags(&e->aux_stream, cudaStreamNonBlocking));
      while (e->sub_ev.size() < kSub + 2) {
        cudaEvent_t v;
        CK(cudaEventCreateWithFlags(&v, cudaEventDisableTiming));
        e->sub_ev.push_back(v);
      }
      CK(cudaEventRecord(e->wave_ev[3 * wi + 0], st));
      CK(cudaEventRecord(e->sub_ev[kSub], st));  // K0 and the counters' memset are done
      CK(cudaStreamWaitEvent(e->aux_stream, e->sub_ev[kSub], 0));
      CK(cudaStreamWaitEvent(e->tail_stream, e->sub_ev[kSub], 0));
      for (int sidx = 0; sidx < kSub; ++sidx) {
        const uint32_t lo_b = (uint32_t)((uint64_t)nb * sidx / kSub), hi_b = (uint32_t)((uint64_t)nb * (sidx + 1) / kSub);
        if (hi_b <= lo_b) continue;
        cudaStream_t fs = (sidx & 1) ? e->aux_stream : st;
        FillParams f2 = fp;
        f2.blocks = fp.blocks + lo_b;
        f2.nblocks = hi_b - lo_b;
        f2.task_counter = ctl + 8 + sidx;
        f2.task_limit = 1;  // CTAs retire after one task per warp: the walks' CTAs get onto the SMs in between
        CK(launch_fill(e, f2, f2.nblocks * (uint32_t)pl.G, fs, &e->last_grid, 0));
        ++e->launches;
        CK(cudaEventRecord(e->sub_ev[sidx], fs));
        CK(cudaStreamWaitEvent(e->tail_stream, e->sub_ev[sidx], 0));
        if (sidx == kSub - 1) CK(cudaEventRecord(e->wave_ev[3 * wi + 1], e->tail_stream));  // every fill has finished
        WalkParams w2 = wp;
        w2.blocks = wp.blocks + lo_b;
        w2.nblocks = hi_b - lo_b;
        if (warp_walk) k2_warp<<<w2.nblocks * 32 / wcta_warps, wcta_warps * 32, (size_t)per_warp_smem * wcta_warps, e->tail_stream>>>(w2);
        else k2_lane<<<(w2.nblocks * 32 + 127) / 128, 128, 0, e->tail_stream>>>(w2);
        CK(cudaGetLastError());
        ++e->launches;
      }
      CK(cudaEventRecord(e->sub_ev[kSub + 1], e->tail_stream));
      CK(cudaStreamWaitEvent(st, e->sub_ev[kSub + 1], 0));  // everything rejoins the engine's stream
      e->last_walk_warp = warp_walk;
      CK(cudaEventRecord(e->wave_ev[3 * wi + 2], st));
      ++wi;
      continue;
    }
    CK(cudaEventRecord(e->wave_ev[3 * wi + 0], st));
    CK(launch_fill(e, fp, fill_tasks, st, &e->last_grid, 0));
    ++e->launches;
    CK(cudaEventRecord(e->wave_ev[3 * wi + 1], st));
    if (use_tail) {  // K2 and everything after it on the high-priority stream
      CK(cudaEventRecord(e->ev_fill, st));
      CK(cudaStreamWaitEvent(e->tail_stream, e->ev_fill, 0));
      st = e->tail_stream;
    }
    if (!fuse) {
      // K2 shape: one lane per pair is the bandwidth-efficient form for large batches of reads (a warp's 32
      // pairs share every cache line); one WARP per pair cuts the per-pair latency chain (prefix-maximum passes,
      // prefetched walk) and is what small / medium batches and long sequences need (b2a_walk.cuh).
      if (warp_walk) {
        k2_warp<<<nb * 32 / wcta_warps, wcta_warps * 32, (size_t)per_warp_smem * wcta_warps, st>>>(wp);  // 32 warps (pairs) per block of the plan
      } else {
        const unsigned wgrid = (nb * 32 + 127) / 128;
        k2_lane<<<wgrid, 128, 0, st>>>(wp);
      }
      CK(cudaGetLastError());
      ++e->launches;
      e->last_walk_warp = warp_walk;
    }
    CK(cudaEventRecord(e->wave_ev[3 * wi + 2], st));
    ++wi;
  }
  CK(cudaEventRecord(e->ev[4], st));
  if (!e->score_only) {
    int rc2 = compact_ops(e, pl.ops_bytes, st);
    if (rc2) return rc2;
  }
  CK(cudaEventRecord(e->ev[5], st));
  e->ran = true;
  return B2A_OK;
}

int32_t b2a_batch_fetch(b2a_engine* e, b2a_results* r, b2a_stats* stats) {
  if (!e) return B2A_E_INVALID;
  if (!e->ran) return e->fail(B2A_E_STATE, "b2a_batch_fetch before b2a_batch_run");
  if (cudaSetDevice(e->device) != cudaSuccess) return e->fail(B2A_E_NO_DEVICE, "cudaSetDevice failed");
  cudaStream_t st = e->res_stream();
  const uint64_t n = e->n_pairs;
  uint64_t d2h = 0;
  uint32_t ctl[2] = {0, 0};
  CK(cudaMemcpyAsync(ctl, e->d_ctl.p, 8, cudaMemcpyDeviceToHost, st));
  if (r && n) {
    auto down = [&](void* dst, const DevBuf& b, size_t bytes) -> cudaError_t {
      if (!dst || !bytes) return cudaSuccess;
      d2h += bytes;
      return cudaMemcpyAsync(dst, b.p, bytes, cudaMemcpyDeviceToHost, st);
    };
    CK(down(r->score, e->d_score, n * 4));
    CK(down(r->xstart, e->d_xs, n * 4));
    CK(down(r->xend, e->d_xe, n * 4));
    CK(down(r->ystart, e->d_ys, n * 4));
    CK(down(r->yend, e->d_ye, n * 4));
    CK(down(r->clip_len, e->d_clip, n * 16));
    CK(down(r->status, e->d_status, n * 4));
    uint64_t total = 0;
    if (r->ops_off) {
      CK(down(r->ops_off, e->d_opsoff, (n + 1) * 8));
      CK(cudaStreamSynchronize(st));
      total = r->ops_off[n];
    } else {
      CK(cudaMemcpyAsync(&total, e->d_opsoff.as<uint64_t>() + n, 8, cudaMemcpyDeviceToHost, st));
      CK(cudaStreamSynchronize(st));
    }
    if (r->ops) {
      if (total > r->ops_capacity) return e->fail(B2A_E_CAPACITY, "ops buffer too small for this batch");
      CK(down(r->ops, e->d_opsdense, total));
    }
  }
  CK(cudaStreamSynchronize(st));
  if (ctl[0]) return e->fail(B2A_E_INVALID, "a sequence byte is outside the scoring alphabet");
  if (ctl[1] & 4u) return e->fail(B2A_E_INVALID, "a sequence byte is outside the scoring alphabet");
  // per-pair failures: reported per pair when the caller gave a status array, else they fail the batch
  if (!(r && r->status)) {
    if (ctl[1] & 2u) return e->fail(B2A_E_CAPACITY, "banded: more k-mer matches than the per-pair capacity");
    if (ctl[1] & 8u)
      return e->fail(B2A_E_INVALID, "banded: the reference panics on these caller-supplied matches/path (not strictly ascending, index out of range, or outside the matrix)");
    if (ctl[1]) return e->fail(B2A_E_RANGE, "traceback walk met an impossible move or never terminates (the reference panics / hangs here: mod.rs:905, banded.rs:777-831)");
  }
  if (e->split_timing && e->split_ran) {
    float a = 0, b = 0, c = 0, d = 0;
    cudaEventElapsedTime(&a, e->split_ev[0], e->split_ev[1]);
    cudaEventElapsedTime(&b, e->split_ev[1], e->split_ev[2]);
    cudaEventElapsedTime(&c, e->split_ev[1], e->split_ev[3]);
    cudaEventElapsedTime(&d, e->split_ev[1], e->split_ev[4]);
    fprintf(stderr, "[split] fill A %.1f us; after it: fill B done +%.1f, walk A done +%.1f, walk B done +%.1f us\n", a * 1e3,
            b * 1e3, c * 1e3, d * 1e3);
    e->split_ran = false;
  }
  if (stats) {
    std::memset(stats, 0, sizeof(*stats));
    stats->cells = e->plan.cells;
    stats->h2d_bytes = e->h2d_bytes;
    stats->d2h_bytes = d2h;
    stats->traceback_bytes = e->plan.total_tb;
    cudaEventElapsedTime(&stats->pack_ms, e->ev[0], e->ev[1]);
    for (size_t wv = 0; wv < e->plan.waves.size(); ++wv) {
      float a = 0.f, b = 0.f;
      cudaEventElapsedTime(&a, e->wave_ev[3 * wv + 0], e->wave_ev[3 * wv + 1]);
      cudaEventElapsedTime(&b, e->wave_ev[3 * wv + 1], e->wave_ev[3 * wv + 2]);
      stats->fill_ms += a;
      stats->walk_ms += b;
    }
    float tail = 0.f;
    cudaEventElapsedTime(&tail, e->ev[4], e->ev[5]);  // ops compaction
    stats->walk_ms += tail;
    stats->kernel_launches = e->launches;
    stats->waves = (uint32_t)e->plan.waves.size();
    stats->fill_lanes_per_pair = (uint32_t)e->plan.G;
    stats->fill_rows_per_lane = (uint32_t)e->plan.R;
  }
  return B2A_OK;
}

// kernel-time part of the stats of an engine whose batch has completed
static void collect_stats(b2a_engine* e, b2a_stats* stats) {
  stats->cells += e->plan.cells;
  stats->h2d_bytes += e->h2d_bytes;
  stats->traceback_bytes += e->plan.total_tb;
  float v = 0.f;
  cudaEventElapsedTime(&v, e->ev[0], e->ev[1]);
  stats->pack_ms += v;
  for (size_t wv = 0; wv < e->plan.waves.size(); ++wv) {
    float a = 0.f, b = 0.f;
    cudaEventElapsedTime(&a, e->wave_ev[3 * wv + 0], e->wave_ev[3 * wv + 1]);
    cudaEventElapsedTime(&b, e->wave_ev[3 * wv + 1], e->wave_ev[3 * wv + 2]);
    stats->fill_ms += a;
    stats->walk_ms += b;
  }
  cudaEventElapsedTime(&v, e->ev[4], e->ev[5]);
  stats->walk_ms += v;
  stats->kernel_launches += e->launches;
  stats->waves += (uint32_t)e->plan.waves.size();
  stats->fill_lanes_per_pair = (uint32_t)e->plan.G;
  stats->fill_rows_per_lane = (uint32_t)e->plan.R;
}

// finish one pipeline slot: its chunk's results are complete on the device; place its ops after `base`
// (r == null: a score-only chunk, `status` is its caller's status array)
static int32_t slot_finish(b2a_engine* e, b2a_engine::PipeSlot& sl, b2a_results* r, const uint32_t* status,
                           uint64_t& base, b2a_stats* agg) {
  b2a_engine* c = sl.eng;
  sl.busy = false;
  cudaError_t ce = cudaStreamSynchronize(c->res_stream());
  if (ce != cudaSuccess) return e->cuda_fail("pipeline: cudaStreamSynchronize", ce);
  if (sl.h_ctl[0]) return e->fail(B2A_E_INVALID, "a sequence byte is outside the scoring alphabet");
  if (sl.h_ctl[1] && !status) return e->fail(B2A_E_RANGE, "traceback walk met an impossible move (reference panics at mod.rs:905)");
  if (!r) {
    collect_stats(c, agg);
    return B2A_OK;
  }
  const uint64_t total = sl.h_opsoff[sl.n];
  if (r->ops) {
    if (base + total > r->ops_capacity) return e->fail(B2A_E_CAPACITY, "ops buffer too small for this batch");
    if (total) {
      ce = cudaMemcpyAsync(r->ops + base, c->d_opsdense.p, total, cudaMemcpyDeviceToHost, c->res_stream());
      if (ce != cudaSuccess) return e->cuda_fail("pipeline: ops D2H", ce);
      agg->d2h_bytes += total;
    }
  }
  if (r->ops_off)
    for (uint64_t i = 0; i < sl.n; ++i) r->ops_off[sl.lo + i] = base + sl.h_opsoff[i];
  base += total;
  ce = cudaStreamSynchronize(c->res_stream());
  if (ce != cudaSuccess) return e->cuda_fail("pipeline: cudaStreamSynchronize", ce);
  collect_stats(c, agg);
  return B2A_OK;
}

static int32_t score_fetch(b2a_engine* e, b2a_score_results* r, b2a_stats* stats);

// The chunk pipeline of a large batch: full results into r, or (r == null) score-only results into sr
static int32_t align_batch_pipelined(b2a_engine* e, int32_t mode, const b2a_scoring* scoring,
                                     const b2a_pairs* pairs, b2a_results* r, b2a_score_results* sr, b2a_stats* stats) {
  const uint64_t n = pairs->n_pairs;
  const bool score_only = r == nullptr;
  const uint32_t* status = score_only ? sr->status : r->status;
  // chunk boundaries: K chunks, the first and the last half as large as the middle ones (the GPU idles
  // while the first chunk is staged and the host idles while the last one drains)
  uint64_t K = (uint64_t)e->pipe_chunks;
  // A small first chunk (its H2D is exposed), then growing ones (each chunk costs a fill tail of about half
  // a warp-task), and a smaller last one (its walk and D2H are exposed).  Measured on 1M x 150x150:
  // 1,3,6,6,3 -> 28.4-29.5 ms against 31.7 ms for 1,2,2,2,1 (profiles/r01_e2e_chunk_schedules.txt).
  std::vector<double> wts(K, 6.0);
  wts[0] = 1.0;
  if (K >= 3) wts[1] = 3.0;
  wts[K - 1] = K >= 4 ? 3.0 : 2.0;
  // three slots (round 2): the last chunk's walk and copies hide under nothing, but its fill no longer waits for
  // a slot, so equal late chunks measure best: 1,3,5,5,5 -> 26.9 ms per 1M-pair call against 27.3 for 1,3,6,6,3
  // (profiles/r02_e2e_chunk_schedules.txt)
  if (K == 5) wts = {1.0, 3.0, 5.0, 5.0, 5.0};
  if (const char* env = getenv("B2A_PIPE_WEIGHTS")) {  // development knob: comma-separated chunk weights
    std::vector<double> w2;
    for (const char* q = env; *q;) {
      char* end = nullptr;
      const double v = strtod(q, &end);
      if (end == q) break;
      if (v > 0) w2.push_back(v);
      q = *end ? end + 1 : end;
    }
    if (w2.size() >= 2) {
      wts = w2;
      K = wts.size();
    }
  }
  std::vector<uint64_t> cut(K + 1, 0);
  {
    double tot = 0, acc = 0;
    for (double w : wts) tot += w;
    for (uint64_t c = 0; c < K; ++c) {
      acc += wts[c] / tot * (double)n;
      cut[c + 1] = std::min<uint64_t>(n, ((uint64_t)acc + 31) / 32 * 32);
    }
    cut[K] = n;
  }
  b2a_stats agg;
  std::memset(&agg, 0, sizeof(agg));
  uint64_t base = 0;
  int32_t rc = B2A_OK;
  std::vector<uint8_t> inferred;
  const bool dbg = getenv("B2A_DEBUG_TIMING") != nullptr;
  auto now = []() { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count(); };
  const double t00 = now();
  for (uint64_t c = 0; c < K && rc == B2A_OK; ++c) {
    const double tc0 = now();
    if (cut[c + 1] <= cut[c]) continue;
    const uint64_t lo = cut[c], hi = cut[c + 1], nc = hi - lo;
    b2a_engine::PipeSlot& sl = e->slots[c % b2a_engine::kSlots];
    if (sl.busy) {
      rc = slot_finish(e, sl, r, status, base, &agg);
      if (rc) break;
    }
    if (!sl.eng) {
      rc = b2a_engine_create(&sl.eng, e->device);
      if (rc) {
        e->fail(rc, "pipeline: cannot create a slot engine");
        break;
      }
    }
    if (!sl.eng->tail_stream) {
      int lo_pri = 0, hi_pri = 0;
      cudaDeviceGetStreamPriorityRange(&lo_pri, &hi_pri);
      if (cudaStreamCreateWithPriority(&sl.eng->tail_stream, cudaStreamNonBlocking, hi_pri) != cudaSuccess ||
          cudaEventCreateWithFlags(&sl.eng->ev_fill, cudaEventDisableTiming) != cudaSuccess) {
        rc = e->fail(B2A_E_CUDA, "pipeline: cannot create the slot's tail stream");
        break;
      }
    }
    sl.eng->is_slot = true;
    sl.eng->stage_nosync = true;
    sl.eng->fill_task_limit = 1;
    sl.eng->packed_width = e->packed_width;
    sl.eng->tune_G = e->tune_G;
    sl.eng->tune_R = e->tune_R;
    sl.eng->walk_mode = e->walk_mode;
    sl.eng->tb_budget = e->tb_budget;
    sl.eng->pipe_chunks = 0;
    if (sl.h_cap < nc + 1) {
      if (sl.h_opsoff) cudaFreeHost(sl.h_opsoff);
      sl.h_opsoff = nullptr;
      if (cudaMallocHost(&sl.h_opsoff, (nc + 1) * 8) != cudaSuccess) {
        rc = e->fail(B2A_E_CUDA, "pipeline: cudaMallocHost failed");
        break;
      }
      sl.h_cap = nc + 1;
    }
    if (!sl.h_ctl && cudaMallocHost(&sl.h_ctl, 64) != cudaSuccess) {
      rc = e->fail(B2A_E_CUDA, "pipeline: cudaMallocHost failed");
      break;
    }
    // the chunk's slice of the caller's blob, offsets rebased
    // offsets and extents are bytes, or 32-bit BitEnc blocks for packed input
    const uint32_t pw = e->packed_width;
    const uint64_t unit = pw ? 4 : 1;
    uint64_t bmin = ~0ull, bmax = 0, seq_sum = 0;
    bool inside = true;
    for (uint64_t p = lo; p < hi; ++p) {
      const uint64_t bb = pairs->blob_bytes / unit, xo = pairs->x_off[p], yo = pairs->y_off[p];
      const uint64_t xu = pw ? bitenc_blocks(pairs->x_len[p], pw) : pairs->x_len[p];
      const uint64_t yu = pw ? bitenc_blocks(pairs->y_len[p], pw) : pairs->y_len[p];
      if (xo > bb || xu > bb - xo || yo > bb || yu > bb - yo) {
        inside = false;
        break;
      }
      bmin = std::min(bmin, std::min(xo, yo));
      bmax = std::max(bmax, std::max(xo + xu, yo + yu));
      seq_sum += xu + yu;
    }
    if (!inside) {
      rc = e->fail(B2A_E_INVALID, "sequence offset/length outside seq_blob");
      break;
    }
    if (bmin > bmax) bmin = bmax = 0;
    sl.xoff.resize(nc);
    sl.yoff.resize(nc);
    const uint8_t* chunk_blob = pairs->seq_blob + bmin * unit;
    uint64_t chunk_bytes = (bmax - bmin) * unit;
    if (!pw && chunk_bytes > 2 * seq_sum + (1ull << 20)) {
      // the chunk's sequences are scattered over a much larger span of the caller's blob (e.g. all x, then all
      // y): uploading the span would move most of the blob once per chunk, so gather them into a compact blob
      uint64_t pos = 0;
      sl.packed.resize(seq_sum + 32 * nc + 16);
      for (uint64_t i = 0; i < nc; ++i) {
        sl.xoff[i] = pos;
        std::memcpy(sl.packed.data() + pos, pairs->seq_blob + pairs->x_off[lo + i], pairs->x_len[lo + i]);
        pos += ((uint64_t)pairs->x_len[lo + i] + 15) & ~15ull;
        sl.yoff[i] = pos;
        std::memcpy(sl.packed.data() + pos, pairs->seq_blob + pairs->y_off[lo + i], pairs->y_len[lo + i]);
        pos += ((uint64_t)pairs->y_len[lo + i] + 15) & ~15ull;
      }
      chunk_blob = sl.packed.data();
      chunk_bytes = pos;
    } else {
      for (uint64_t i = 0; i < nc; ++i) {
        sl.xoff[i] = pairs->x_off[lo + i] - bmin;
        sl.yoff[i] = pairs->y_off[lo + i] - bmin;
      }
    }
    b2a_pairs sub{chunk_blob, sl.xoff.data(), pairs->x_len + lo, sl.yoff.data(), pairs->y_len + lo, chunk_bytes, nc};
    b2a_engine* ch = sl.eng;
    const double tc1 = now();
    // Alphabet: chunk 0 discovers it on the (then idle) device; later chunks reuse it optimistically so
    // that their stage does not have to wait behind the other slot's persistent fill kernel.  A byte
    // outside it is caught by K0 (bad-symbol flag) and the whole batch is then redone in one shot.
    b2a_scoring sc_chunk = *scoring;
    if (!(scoring->alphabet && scoring->alphabet_len) && c > 0 && !inferred.empty()) {
      sc_chunk.alphabet = inferred.data();
      sc_chunk.alphabet_len = (uint32_t)inferred.size();
    }
    rc = batch_stage(ch, mode, &sc_chunk, &sub, score_only);
    if (rc == B2A_OK && c == 0 && !(scoring->alphabet && scoring->alphabet_len)) inferred = ch->last_syms;
    const double tc2 = now();
    if (rc == B2A_OK) rc = b2a_batch_run(ch);
    const double tc3 = now();
    if (dbg)
      fprintf(stderr, "[b2a pipe] chunk %llu: t=%.2f finish+prep %.2f ms, stage %.2f ms, run(launch) %.2f ms\n",
              (unsigned long long)c, tc0 - t00, tc1 - tc0, tc2 - tc1, tc3 - tc2);
    if (rc) {
      e->fail(rc, ch->err);
      break;
    }
    cudaStream_t st = ch->res_stream();
    auto down = [&](void* dst, const DevBuf& bf, size_t bytes) -> cudaError_t {
      if (!dst || !bytes) return cudaSuccess;
      agg.d2h_bytes += bytes;
      return cudaMemcpyAsync(dst, bf.p, bytes, cudaMemcpyDeviceToHost, st);
    };
    cudaError_t ce = cudaMemcpyAsync(sl.h_ctl, ch->d_ctl.p, 8, cudaMemcpyDeviceToHost, st);
    if (score_only) {
      if (ce == cudaSuccess) ce = down(sr->score ? sr->score + lo : nullptr, ch->d_score, nc * 4);
      if (ce == cudaSuccess) ce = down(sr->xend ? sr->xend + lo : nullptr, ch->d_xe, nc * 4);
      if (ce == cudaSuccess) ce = down(sr->yend ? sr->yend + lo : nullptr, ch->d_ye, nc * 4);
      if (ce == cudaSuccess) ce = down(sr->status ? sr->status + lo : nullptr, ch->d_status, nc * 4);
      if (ce != cudaSuccess) {
        rc = e->cuda_fail("pipeline: result D2H", ce);
        break;
      }
      sl.lo = lo;
      sl.n = nc;
      sl.busy = true;
      continue;
    }
    if (ce == cudaSuccess) ce = down(r->score ? r->score + lo : nullptr, ch->d_score, nc * 4);
    if (ce == cudaSuccess) ce = down(r->xstart ? r->xstart + lo : nullptr, ch->d_xs, nc * 4);
    if (ce == cudaSuccess) ce = down(r->xend ? r->xend + lo : nullptr, ch->d_xe, nc * 4);
    if (ce == cudaSuccess) ce = down(r->ystart ? r->ystart + lo : nullptr, ch->d_ys, nc * 4);
    if (ce == cudaSuccess) ce = down(r->yend ? r->yend + lo : nullptr, ch->d_ye, nc * 4);
    if (ce == cudaSuccess) ce = down(r->clip_len ? r->clip_len + 4 * lo : nullptr, ch->d_clip, nc * 16);
    if (ce == cudaSuccess) ce = down(r->status ? r->status + lo : nullptr, ch->d_status, nc * 4);
    if (ce == cudaSuccess) ce = down(sl.h_opsoff, ch->d_opsoff, (nc + 1) * 8);
    if (ce != cudaSuccess) {
      rc = e->cuda_fail("pipeline: result D2H", ce);
      break;
    }
    sl.lo = lo;
    sl.n = nc;
    sl.busy = true;
  }
  // drain in chunk order: the older chunk lives in the slot the next chunk would use
  // (slots hold chunks in alternation; the one with the smaller `lo` is the older)
  for (int pass = 0; pass < b2a_engine::kSlots; ++pass) {
    b2a_engine::PipeSlot* pick = nullptr;
    for (auto& cand : e->slots)
      if (cand.busy && (!pick || cand.lo < pick->lo)) pick = &cand;
    if (!pick) break;
    b2a_engine::PipeSlot& sl = *pick;
    if (rc == B2A_OK) {
      rc = slot_finish(e, sl, r, status, base, &agg);
    } else {
      cudaStreamSynchronize(sl.eng->stream);
      cudaStreamSynchronize(sl.eng->res_stream());
      sl.busy = false;
    }
  }
  if (rc == B2A_E_INVALID && !inferred.empty() && e->err.find("alphabet") != std::string::npos) {
    // a later chunk held a byte the first chunk did not: redo the batch without the optimistic reuse
    int32_t r2 = batch_stage(e, mode, scoring, pairs, score_only);
    if (r2 == B2A_OK) r2 = b2a_batch_run(e);
    if (r2 == B2A_OK) r2 = score_only ? score_fetch(e, sr, stats) : b2a_batch_fetch(e, r, stats);
    return r2;
  }
  if (rc) return rc;
  if (!score_only && r->ops_off) r->ops_off[n] = base;
  if (stats) *stats = agg;
  return B2A_OK;
}

int32_t b2a_align_batch(b2a_engine* e, int32_t mode, const b2a_scoring* scoring, const b2a_pairs* pairs,
                        b2a_results* results, b2a_stats* stats) {
  if (!e || !scoring || !pairs) return B2A_E_INVALID;
  // large batches with host outputs: pipeline chunks so copies and planning overlap the kernels
  if (e->pipe_chunks >= 2 && results && pairs->n_pairs >= 262144) {
    e->staged = e->ran = false;
    if (cudaSetDevice(e->device) != cudaSuccess) return e->fail(B2A_E_NO_DEVICE, "cudaSetDevice failed");
    return align_batch_pipelined(e, mode, scoring, pairs, results, nullptr, stats);
  }
  int rc = b2a_batch_stage(e, mode, scoring, pairs);
  if (rc) return rc;
  rc = b2a_batch_run(e);
  if (rc) return rc;
  return b2a_batch_fetch(e, results, stats);
}

}  // extern "C"

// results of a score-only batch that b2a_batch_run has run
static int32_t score_fetch(b2a_engine* e, b2a_score_results* r, b2a_stats* stats) {
  cudaStream_t st = e->res_stream();
  const uint64_t n = e->n_pairs;
  uint64_t d2h = 0;
  uint32_t ctl[2] = {0, 0};
  CK(cudaMemcpyAsync(ctl, e->d_ctl.p, 8, cudaMemcpyDeviceToHost, st));
  if (r && n) {
    auto down = [&](void* dst, const DevBuf& b, size_t bytes) -> cudaError_t {
      if (!dst || !bytes) return cudaSuccess;
      d2h += bytes;
      return cudaMemcpyAsync(dst, b.p, bytes, cudaMemcpyDeviceToHost, st);
    };
    CK(down(r->score, e->d_score, n * 4));
    CK(down(r->xend, e->d_xe, n * 4));
    CK(down(r->yend, e->d_ye, n * 4));
    CK(down(r->status, e->d_status, n * 4));
  }
  CK(cudaStreamSynchronize(st));
  if (ctl[0]) return e->fail(B2A_E_INVALID, "a sequence byte is outside the scoring alphabet");
  if (ctl[1] && !(r && r->status))
    return e->fail(B2A_E_RANGE, "traceback walk met an impossible move (the reference panics here: mod.rs:905)");
  if (stats) {
    std::memset(stats, 0, sizeof(*stats));
    collect_stats(e, stats);
    stats->d2h_bytes = d2h;
  }
  return B2A_OK;
}

extern "C" {

int32_t b2a_score_batch(b2a_engine* e, int32_t mode, const b2a_scoring* scoring, const b2a_pairs* pairs,
                        b2a_score_results* results, b2a_stats* stats) {
  if (!e || !scoring || !pairs) return B2A_E_INVALID;
  int32_t rc;
  if (e->pipe_chunks >= 2 && results && pairs->n_pairs >= 262144) {  // as b2a_align_batch
    e->staged = e->ran = false;
    if (cudaSetDevice(e->device) != cudaSuccess) return e->fail(B2A_E_NO_DEVICE, "cudaSetDevice failed");
    rc = align_batch_pipelined(e, mode, scoring, pairs, nullptr, results, stats);
  } else {
    rc = batch_stage(e, mode, scoring, pairs, true);
    if (rc == B2A_OK) rc = b2a_batch_run(e);
    if (rc == B2A_OK) rc = score_fetch(e, results, stats);
  }
  // the scratch now holds no traceback and no ops: nothing for b2a_batch_fetch / the record and compact calls
  e->staged = e->ran = false;
  return rc;
}

static int32_t banded_impl(b2a_engine* e, int32_t mode, const b2a_scoring* s, uint32_t k, uint32_t w,
                           const b2a_pairs* pairs, const b2a_band_hints* hints, b2a_results* results,
                           b2a_stats* stats);

// BitEnc storage as the input of Aligner::{custom,global,semiglobal,local} (and of the banded aligner when k > 0)
static int32_t packed_view(b2a_engine* e, const b2a_packed_pairs* pp, b2a_pairs* view) {
  if (!e || !pp) return B2A_E_INVALID;
  if (pp->width < 1 || pp->width > 8) return e->fail(B2A_E_INVALID, "BitEnc width must be 1..8 (bitenc.rs:75)");
  view->seq_blob = reinterpret_cast<const uint8_t*>(pp->blocks);
  view->x_off = pp->x_block;
  view->x_len = pp->x_len;
  view->y_off = pp->y_block;
  view->y_len = pp->y_len;
  view->blob_bytes = pp->n_blocks * 4;
  view->n_pairs = pp->n_pairs;
  return B2A_OK;
}

int32_t b2a_align_batch_packed(b2a_engine* e, int32_t mode, const b2a_scoring* scoring, const b2a_packed_pairs* pp,
                               b2a_results* results, b2a_stats* stats) {
  b2a_pairs view;
  int rc = packed_view(e, pp, &view);
  if (rc) return rc;
  e->packed_width = pp->width;
  rc = b2a_align_batch(e, mode, scoring, &view, results, stats);
  e->packed_width = 0;
  return rc;
}

int32_t b2a_align_batch_banded_packed(b2a_engine* e, int32_t mode, const b2a_scoring* scoring, uint32_t k, uint32_t w,
                                      const b2a_packed_pairs* pp, b2a_results* results, b2a_stats* stats) {
  b2a_pairs view;
  int rc = packed_view(e, pp, &view);
  if (rc) return rc;
  e->packed_width = pp->width;
  rc = banded_impl(e, mode, scoring, k, w, &view, nullptr, results, stats);
  e->packed_width = 0;
  return rc;
}

int32_t b2a_align_batch_banded(b2a_engine* e, int32_t mode, const b2a_scoring* s, uint32_t k, uint32_t w,
                               const b2a_pairs* pairs, b2a_results* results, b2a_stats* stats) {
  return banded_impl(e, mode, s, k, w, pairs, nullptr, results, stats);
}

int32_t b2a_align_batch_banded_hinted(b2a_engine* e, int32_t mode, const b2a_scoring* s, uint32_t k, uint32_t w,
                                      const b2a_pairs* pairs, const b2a_band_hints* hints, b2a_results* results,
                                      b2a_stats* stats) {
  if (!e || !hints) return B2A_E_INVALID;
  if (!hints->match_off || (!hints->match_xy && pairs && pairs->n_pairs && hints->match_off[pairs->n_pairs]))
    return e->fail(B2A_E_INVALID, "banded hints: match_off / match_xy missing");
  if (hints->path_off && (hints->allowed_mismatches >= 0 || hints->use_lcskpp_union))
    return e->fail(B2A_E_INVALID, "banded hints: a match path excludes allowed_mismatches / use_lcskpp_union");
  return banded_impl(e, mode, s, k, w, pairs, hints, results, stats);
}

static int32_t banded_impl(b2a_engine* e, int32_t mode, const b2a_scoring* s, uint32_t k, uint32_t w,
                           const b2a_pairs* pairs, const b2a_band_hints* hints, b2a_results* results,
                           b2a_stats* stats) {
  if (!e || !s || !pairs) return B2A_E_INVALID;
  if (k == 0) return e->fail(B2A_E_INVALID, "banded: k-mer length must be >= 1");
  uint32_t maxm = 0, maxn = 0;
  int64_t score_bound = 0;
  int rc = stage_front(e, mode, s, pairs, maxm, maxn, score_bound);
  if (rc) return rc;
  const uint64_t n = e->n_pairs;
  cudaStream_t st = e->stream;
  auto up = [&](DevBuf& bf, const void* src, size_t bytes) -> cudaError_t {
    e->h2d_bytes += bytes;
    return bytes ? cudaMemcpyAsync(bf.p, src, bytes, cudaMemcpyHostToDevice, st) : cudaSuccess;
  };
  // per-pair ops regions (written backwards from their end) and output arrays
  std::vector<uint64_t> ops_end(n);
  uint64_t ops_total = 0;
  for (uint64_t p = 0; p < n; ++p) {
    ops_total += (uint64_t)pairs->x_len[p] + pairs->y_len[p] + 8;
    ops_end[p] = ops_total;
  }
  CK(e->d_xoff.reserve(n * 8 + 8));
  CK(e->d_yoff.reserve(n * 8 + 8));
  CK(e->d_xlen.reserve(n * 4 + 4));
  CK(e->d_ylen.reserve(n * 4 + 4));
  CK(e->d_codemap.reserve(256));
  CK(e->d_lut.reserve(e->lut_host.size() * 4 + 16));
  CK(e->d_score.reserve(n * 4 + 4));
  CK(e->d_xs.reserve(n * 4 + 4));
  CK(e->d_xe.reserve(n * 4 + 4));
  CK(e->d_ys.reserve(n * 4 + 4));
  CK(e->d_ye.reserve(n * 4 + 4));
  CK(e->d_nops.reserve(n * 4 + 4));
  CK(e->d_opssrc.reserve(n * 8 + 8));
  CK(e->d_clip.reserve(n * 16 + 16));
  CK(e->d_status.reserve(n * 4 + 4));
  CK(e->d_nops64.reserve((n + 1) * 8));
  CK(e->d_opsoff.reserve((n + 1) * 8));
  CK(e->d_opsscratch.reserve(ops_total + 16));
  CK(e->d_bcells.reserve(n * 8 + 8));
  CK(e->d_bstatus.reserve(n * 4 + 4));
  CK(e->d_bcols.reserve(n * 12 + 16));
  CK(e->d_bopsend.reserve(n * 8 + 8));
  if (!e->packed_width) {
    CK(up(e->d_xoff, pairs->x_off, n * 8));
    CK(up(e->d_yoff, pairs->y_off, n * 8));
    CK(up(e->d_xlen, pairs->x_len, n * 4));
    CK(up(e->d_ylen, pairs->y_len, n * 4));
  }
  CK(up(e->d_codemap, e->codemap_host, 256));
  if (!e->lut_host.empty()) CK(up(e->d_lut, e->lut_host.data(), e->lut_host.size() * 4));
  CK(up(e->d_bopsend, ops_end.data(), n * 8));
  uint32_t* ctl = e->d_ctl.as<uint32_t>();
  CK(cudaMemsetAsync(ctl, 0, 256, st));

  const uint32_t short_max = std::min(maxm, maxn);
  uint64_t cap64 = 4ull * short_max + 1024;
  if (hints) {  // the caller's matches (and what expanding them can add) must fit the per-pair slab
    uint64_t most = 0, most_path = 0;
    for (uint64_t p = 0; p < n; ++p) {
      if (hints->match_off[p + 1] < hints->match_off[p]) return e->fail(B2A_E_INVALID, "banded hints: match_off not ascending");
      most = std::max(most, hints->match_off[p + 1] - hints->match_off[p]);
      if (hints->path_off) {
        if (hints->path_off[p + 1] < hints->path_off[p]) return e->fail(B2A_E_INVALID, "banded hints: path_off not ascending");
        most_path = std::max(most_path, hints->path_off[p + 1] - hints->path_off[p]);
      }
    }
    cap64 = std::max(cap64, most + 16);
    cap64 = std::max(cap64, (most_path + 1) / 2 + 16);
    if (hints->allowed_mismatches >= 0) cap64 = std::max<uint64_t>(cap64, 8 * most + 4ull * short_max + 1024);
    const uint64_t tm = hints->match_off[n], tp = hints->path_off ? hints->path_off[n] : 0;
    CK(e->d_hmoff.reserve((n + 1) * 8));
    CK(e->d_hmxy.reserve(tm * 8 + 16));
    CK(up(e->d_hmoff, hints->match_off, (n + 1) * 8));
    CK(up(e->d_hmxy, hints->match_xy, tm * 8));
    if (hints->path_off) {
      CK(e->d_hpoff.reserve((n + 1) * 8));
      CK(e->d_hpidx.reserve(tp * 4 + 16));
      CK(up(e->d_hpoff, hints->path_off, (n + 1) * 8));
      CK(up(e->d_hpidx, hints->path_idx, tp * 4));
    }
  }
  // Per-pair capacity of the k-mer match list.  The reference's find_kmer_matches has no limit (low-complexity
  // sequences give up to O(m n) matches: a 60-nt homopolymer in both reads is 53 x 53 8-mer matches), so the
  // capacity starts at a size that covers ordinary batches and a wave whose pairs overflow it is redone with
  // eight times the capacity, up to kCapMax per pair (beyond that the pair reports B2A_PAIR_CAPACITY).
  constexpr uint32_t kCapMax = 1u << 22;
  uint32_t cap = (uint32_t)std::min<uint64_t>(cap64, kCapMax);
  if (const char* env = getenv("B2A_BANDED_CAP")) {  // test knob: start from a tiny capacity
    const long v = atol(env);
    if (v > 0) cap = (uint32_t)std::min<long>(v, (long)kCapMax);
  }
  uint64_t k4_bytes = k4_slab_bytes(cap, short_max);
  uint64_t budget = e->tb_budget;
  if (!budget) {
    size_t fr = 0, tot = 0;
    CK(cudaMemGetInfo(&fr, &tot));
    budget = (uint64_t)((double)fr * 0.5);
  }
  auto wave_for = [&](uint64_t slab_bytes) {
    const uint64_t per_pair_k4 = slab_bytes + ((uint64_t)maxn + 1) * 8 + 64;
    uint64_t wv = std::max<uint64_t>(1, (budget / 2) / per_pair_k4);
    wv = std::min<uint64_t>(wv, std::max<uint64_t>(n, 1));
    return std::min<uint64_t>(wv, 1u << 20);
  };
  uint64_t wave = wave_for(k4_bytes);

  BandedParams bp{};
  bp.blob = e->d_blob.as<uint8_t>();
  bp.x_off = e->d_xoff.as<uint64_t>();
  bp.x_len = e->d_xlen.as<uint32_t>();
  bp.y_off = e->d_yoff.as<uint64_t>();
  bp.y_len = e->d_ylen.as<uint32_t>();
  bp.codemap = e->d_codemap.as<uint8_t>();
  bp.lut = e->d_lut.as<int32_t>();
  bp.sc = e->sc;
  // MatchParams keeps its compare/select form here (scores are read per cell from the blob bytes)
  if (!s->table) bp.sc.alpha = 0;
  bp.has_match_scores = s->has_match_scores;
  bp.allowed_mismatches = -1;
  if (hints) {
    bp.hint_match_off = e->d_hmoff.as<uint64_t>();
    bp.hint_match_xy = e->d_hmxy.as<uint32_t>();
    if (hints->path_off) {
      bp.hint_path_off = e->d_hpoff.as<uint64_t>();
      bp.hint_path_idx = e->d_hpidx.as<uint32_t>();
    }
    bp.allowed_mismatches = hints->allowed_mismatches;
    bp.use_lcskpp_union = hints->use_lcskpp_union;
  }
  bp.k = k;
  bp.w = w;
  bp.cap_matches = cap;
  bp.n_pairs = n;
  bp.slab_stride = k4_bytes;
  bp.num_cells = e->d_bcells.as<uint64_t>();
  bp.k4_status = e->d_bstatus.as<uint32_t>();
  bp.band_cols = e->d_bcols.as<uint32_t>();
  // The strip-wavefront fill (b2a_banded_strip.cuh) covers every real score within +-2^26 (its sentinel
  // arithmetic); row / column trackers only as packed keys (below).
  {
    const bool xs_dead = e->sc.xclip_suffix <= DEAD_CLIP, ys_dead = e->sc.yclip_suffix <= DEAD_CLIP;
    const bool yp_live = e->sc.yclip_prefix > DEAD_CLIP;
    // trackers are packed keys: every band cell's S has to be real (a live y-prefix clip guarantees it: S >=
    // yclip_score(i)) and below 2^17; the column tracker's key also holds the row (x no longer than 4,095)
    const bool trackers_ok = (xs_dead && ys_dead) || (yp_live && score_bound < (1ll << 17) && (xs_dead || maxm <= 4095));
    bp.strip_ok = (e->banded_strip && e->banded_fast && score_bound < (1ll << 26) && trackers_ok) ? 1 : 0;
    if (bp.strip_ok && e->banded_strip_lastcol) bp.strip_ok |= 2;  // bands that hold cells of column n as well
  }
  e->strip_pairs = 0;
  bp.filter_clips = (mode == B2A_MODE_SEMIGLOBAL || mode == B2A_MODE_LOCAL) ? 1 : 0;
  bp.score = e->d_score.as<int32_t>();
  bp.xstart = e->d_xs.as<uint32_t>();
  bp.xend = e->d_xe.as<uint32_t>();
  bp.ystart = e->d_ys.as<uint32_t>();
  bp.yend = e->d_ye.as<uint32_t>();
  bp.n_ops = e->d_nops.as<uint32_t>();
  bp.ops_src = e->d_opssrc.as<uint64_t>();
  bp.clip_len = e->d_clip.as<uint32_t>();
  bp.status = e->d_status.as<uint32_t>();
  bp.err_flag = ctl + 1;
  bp.ops_scratch = e->d_opsscratch.as<uint8_t>();
  bp.ops_off = e->d_bopsend.as<uint64_t>();

  e->launches = 0;
  float band_ms = 0.f, fill_ms = 0.f;
  uint64_t total_cells = 0;
  std::vector<uint64_t> h_cells, roff, foff, soff;
  std::vector<uint32_t> h_k4, h_cols, elig;
  cudaEvent_t ev0 = e->ev[0], ev1 = e->ev[1], ev2 = e->ev[2];
  for (uint64_t lo = 0; lo < n;) {
    const uint32_t nw = (uint32_t)std::min<uint64_t>(wave, n - lo);
    bp.cap_matches = cap;
    bp.slab_stride = k4_bytes;
    roff.resize(nw);
    uint64_t rbytes = 0;
    for (uint32_t t = 0; t < nw; ++t) {
      roff[t] = rbytes;
      rbytes += (((uint64_t)pairs->y_len[lo + t] + 1) * 8 + 15) & ~15ull;
    }
    CK(e->d_bslab.reserve((uint64_t)nw * k4_bytes + 16));
    CK(e->d_branges.reserve(rbytes + 16));
    CK(e->d_broff.reserve((uint64_t)nw * 8 + 8));
    CK(up(e->d_broff, roff.data(), (size_t)nw * 8));
    e->band_wave_lo = lo;
    e->band_roff = roff;
    e->band_ylen.assign(pairs->y_len + lo, pairs->y_len + lo + nw);
    bp.pair_lo = (uint32_t)lo;
    bp.slab = e->d_bslab.as<uint8_t>();
    bp.ranges = e->d_branges.as<uint32_t>();
    bp.ranges_off = e->d_broff.as<uint64_t>();
    CK(cudaEventRecord(ev0, st));
    band_kernel<<<(nw + 3) / 4, 128, 0, st>>>(bp, nw);  // one warp per pair
    CK(cudaGetLastError());
    ++e->launches;
    CK(cudaEventRecord(ev1, st));
    h_cells.resize(nw);
    h_k4.resize(nw);
    CK(cudaMemcpyAsync(h_cells.data(), e->d_bcells.as<uint64_t>() + lo, (size_t)nw * 8, cudaMemcpyDeviceToHost, st));
    CK(cudaMemcpyAsync(h_k4.data(), e->d_bstatus.as<uint32_t>() + lo, (size_t)nw * 4, cudaMemcpyDeviceToHost, st));
    h_cols.resize((size_t)nw * 3);
    if (bp.strip_ok)
      CK(cudaMemcpyAsync(h_cols.data(), e->d_bcols.as<uint32_t>() + 3 * lo, (size_t)nw * 12, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    {
      float ms = 0.f;
      cudaEventElapsedTime(&ms, ev0, ev1);
      band_ms += ms;
    }
    bool overflowed = false;
    for (uint32_t& v : h_k4) {
      overflowed |= (v & 0xFFu) == 1u;
      if (!e->banded_fast) v &= 0xFFu;
      if (!bp.strip_ok) v &= ~0x200u;
    }
    if (!e->banded_fast)  // the literal loop for every pair: clear K4's marks on the device as well
      CK(cudaMemcpyAsync(e->d_bstatus.as<uint32_t>() + lo, h_k4.data(), (size_t)nw * 4, cudaMemcpyHostToDevice, st));
    if (cap < kCapMax && overflowed) {
      // a pair of this wave has more matches than the slab holds: redo the wave (K4 is idempotent) with a
      // larger capacity, in as many pairs as then fit the budget
      cap = (uint32_t)std::min<uint64_t>((uint64_t)cap * 8, kCapMax);
      k4_bytes = k4_slab_bytes(cap, short_max);
      wave = wave_for(k4_bytes);
      continue;
    }
    // K3 in sub-waves sized by the exact slab bytes
    uint32_t s0 = 0;
    while (s0 < nw) {
      foff.clear();
      soff.clear();
      elig.clear();
      uint64_t fbytes = 0, sbytes = 0;
      uint32_t s1 = s0;
      auto strip_need = [&](uint32_t t) -> uint64_t {  // bytes of the pair's strip area (0: not a strip pair)
        if (!(h_k4[t] & 0x200u)) return 0;
        const uint64_t mm = pairs->x_len[lo + t], nn = pairs->y_len[lo + t];
        const uint64_t c0 = std::max<uint64_t>(h_cols[3 * (size_t)t], 1), c1 = std::min<uint64_t>(h_cols[3 * (size_t)t + 1], nn - 1);
        return ks_layout(mm, c1 >= c0 ? c1 - c0 + 1 : 0, h_cols[3 * (size_t)t + 2]).total;
      };
      while (s1 < nw) {
        const uint64_t need = k3_slab_bytes(pairs->x_len[lo + s1], pairs->y_len[lo + s1], h_cells[s1]);
        const uint64_t sneed = strip_need(s1);
        if (s1 > s0 && fbytes + sbytes + need + sneed > budget / 2) break;
        foff.push_back(fbytes);
        soff.push_back(sbytes);
        if (sneed) elig.push_back(s1 - s0);
        fbytes += need;
        sbytes += sneed;
        total_cells += h_cells[s1];
        ++s1;
      }
      const uint32_t ns = s1 - s0;
      CK(e->d_bfill.reserve(fbytes + 16));
      CK(e->d_bfoff.reserve((uint64_t)ns * 8 + 8));
      CK(up(e->d_bfoff, foff.data(), (size_t)ns * 8));
      BandedParams b3 = bp;
      b3.pair_lo = (uint32_t)(lo + s0);
      b3.ranges_off = e->d_broff.as<uint64_t>() + s0;
      b3.fill = e->d_bfill.as<uint8_t>();
      b3.fill_off = e->d_bfoff.as<uint64_t>();
      CK(cudaEventRecord(ev1, st));
      if (!elig.empty()) {
        // K3s: the strip-wavefront fill (four pairs to a warp) and its finish pass (one warp per pair) for the pairs
        // K4 marked; a pair the path turns out not to cover is handed back (bit 10) to the two loops below
        CK(e->d_bstrip.reserve(sbytes + 16));
        CK(e->d_bsoff.reserve((uint64_t)ns * 8 + 8));
        CK(e->d_belig.reserve(elig.size() * 4 + 16));
        CK(up(e->d_bsoff, soff.data(), (size_t)ns * 8));
        CK(up(e->d_belig, elig.data(), elig.size() * 4));
        StripParams sp{};
        sp.blob = bp.blob;
        sp.x_off = bp.x_off;
        sp.x_len = bp.x_len;
        sp.y_off = bp.y_off;
        sp.y_len = bp.y_len;
        sp.pair_lo = b3.pair_lo;
        sp.elig = e->d_belig.as<uint32_t>();
        sp.n_elig = (uint32_t)elig.size();
        sp.task_counter = ctl + 32;
        sp.ranges = bp.ranges;
        sp.ranges_off = b3.ranges_off;
        sp.fill = b3.fill;
        sp.fill_off = b3.fill_off;
        sp.strip = e->d_bstrip.as<uint8_t>();
        sp.strip_off = e->d_bsoff.as<uint64_t>();
        sp.num_cells = bp.num_cells;
        sp.band_cols = bp.band_cols;
        sp.k4_status = bp.k4_status;
        sp.sc = e->sc;
        sp.lut = s->table ? e->d_lut.as<int32_t>() + (size_t)e->sc.alpha * e->sc.alpha : nullptr;  // K1's scaled copy
        sp.codemap = bp.codemap;
        sp.err_flag = ctl + 1;
        sp.one = 1;
        sp.ge4 = 4 * e->sc.gap_extend;
        const int fl = (e->sc.yclip_suffix > DEAD_CLIP ? (int)F_TRACK_ROWS : 0) | (e->sc.xclip_suffix > DEAD_CLIP ? (int)F_TRACK_COLS : 0) |
                       (e->sc.xclip_prefix > DEAD_CLIP ? (int)F_CLIPX : 0) | (e->sc.yclip_prefix > DEAD_CLIP ? (int)F_CLIPY : 0) |
                       (s->table ? (int)F_LUT : 0);
        sp.flags = fl;
        CK(cudaMemsetAsync(sp.task_counter, 0, 4, st));
        const uint32_t ntasks = (sp.n_elig + 3) / 4;
        const unsigned sgrid = (unsigned)std::min<uint32_t>((ntasks + KS_WARPS - 1) / KS_WARPS, (uint32_t)e->num_sms * (uint32_t)B2A_KS_MINB);
        const size_t ks_smem = ks_smem_bytes(fl, e->sc.alpha);
        switch (fl) {
#define B2A_KS_CASE1(F)                                                                                                   \
  case (F):                                                                                                               \
    if (ks_smem > 48 * 1024)                                                                                              \
      CK(cudaFuncSetAttribute(banded_strip_fill_kernel<(F)>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ks_smem)); \
    banded_strip_fill_kernel<(F)><<<sgrid, KS_WARPS * 32, ks_smem, st>>>(sp);                                             \
    break;
#define B2A_KS_CASE(F) B2A_KS_CASE1(F) B2A_KS_CASE1((F) | F_LUT)
          B2A_KS_CASE(0)
          B2A_KS_CASE(F_TRACK_ROWS)
          B2A_KS_CASE(F_CLIPX)
          B2A_KS_CASE(F_CLIPY)
          B2A_KS_CASE(F_TRACK_ROWS | F_CLIPX)
          B2A_KS_CASE(F_TRACK_ROWS | F_CLIPY)
          B2A_KS_CASE(F_CLIPX | F_CLIPY)
          B2A_KS_CASE(F_TRACK_ROWS | F_CLIPX | F_CLIPY)
          B2A_KS_CASE(F_TRACK_COLS)
          B2A_KS_CASE(F_TRACK_COLS | F_TRACK_ROWS)
          B2A_KS_CASE(F_TRACK_COLS | F_CLIPX)
          B2A_KS_CASE(F_TRACK_COLS | F_CLIPY)
          B2A_KS_CASE(F_TRACK_COLS | F_TRACK_ROWS | F_CLIPX)
          B2A_KS_CASE(F_TRACK_COLS | F_TRACK_ROWS | F_CLIPY)
          B2A_KS_CASE(F_TRACK_COLS | F_CLIPX | F_CLIPY)
          B2A_KS_CASE(F_TRACK_COLS | F_TRACK_ROWS | F_CLIPX | F_CLIPY)
#undef B2A_KS_CASE
#undef B2A_KS_CASE1
          default: return e->fail(B2A_E_INVALID, "banded strip fill: unexpected flag set");
        }
        CK(cudaGetLastError());
        b3.strip = sp.strip;
        b3.strip_off = sp.strip_off;
        banded_strip_finish_kernel<<<(ns + 3) / 4, 128, 0, st>>>(b3, ns);
        CK(cudaGetLastError());
        banded_strip_walk_kernel<<<(ns + 127) / 128, 128, 0, st>>>(b3, ns);  // one pair per thread
        CK(cudaGetLastError());
        e->launches += 3;
        e->strip_pairs += elig.size();
      }
      // The column loops, one warp per pair, for the pairs K4 did not mark for the strip path (K4 marked those whose
      // band suits the register-resident loop; each kernel skips the other's pairs).  With strip pairs in the
      // sub-wave they run beside the strip kernels on a stream of their own -- a lone unmarked pair takes ~2 ms on
      // its single warp -- and a second, normally empty pass afterwards takes what the strip path handed back.
      const bool side = !elig.empty() && elig.size() < ns;
      cudaStream_t cs = st;
      if (side) {
        if (!e->aux_stream) CK(cudaStreamCreateWithFlags(&e->aux_stream, cudaStreamNonBlocking));
        while (e->sub_ev.size() < 6) {
          cudaEvent_t v;
          CK(cudaEventCreateWithFlags(&v, cudaEventDisableTiming));
          e->sub_ev.push_back(v);
        }
        cs = e->aux_stream;
        CK(cudaStreamWaitEvent(cs, ev1, 0));  // K4's results and the sub-wave's uploads
      }
      for (int pass = 0; pass < (elig.empty() ? 1 : 2); ++pass) {
        if (pass == 0 && elig.size() == ns) continue;  // every pair is a strip pair
        BandedParams bc = b3;
        bc.redo_pass = pass;
        cudaStream_t ks = pass == 0 ? cs : st;
        if (pass == 1 && side) {  // the first pass is done before the hand-backs run (same slabs, same outputs)
          CK(cudaEventRecord(e->sub_ev[3], cs));
          CK(cudaStreamWaitEvent(st, e->sub_ev[3], 0));
        }
        if (e->banded_fast) {
          banded_fill_fast_kernel<<<(ns + 3) / 4, 128, 0, ks>>>(bc, ns);
          CK(cudaGetLastError());
          ++e->launches;
        }
        banded_fill_kernel<<<(ns + 3) / 4, 128, 0, ks>>>(bc, ns);
        CK(cudaGetLastError());
        ++e->launches;
      }
      CK(cudaEventRecord(ev2, st));
      CK(cudaStreamSynchronize(st));  // foff (host vector) is reused by the next sub-wave
      float ms = 0.f;
      cudaEventElapsedTime(&ms, ev1, ev2);
      fill_ms += ms;
      s0 = s1;
    }
    lo += nw;
  }
  CK(cudaEventRecord(e->ev[4], st));
  rc = compact_ops(e, ops_total, st);
  if (rc) return rc;
  CK(cudaEventRecord(e->ev[5], st));
  e->plan = Plan{};
  e->plan.cells = total_cells;
  e->ran = true;
  rc = b2a_batch_fetch(e, results, stats);
  if (stats) {
    stats->cells = total_cells;
    stats->band_ms = band_ms;
    stats->fill_ms = fill_ms;
    float tail = 0.f;
    cudaEventElapsedTime(&tail, e->ev[4], e->ev[5]);
    stats->walk_ms = tail;
    // the path most pairs took: the strip-wavefront fill (8 lanes x 16 rows) or one warp per pair
    stats->fill_lanes_per_pair = e->strip_pairs * 2 > n ? (uint32_t)KS_G : 1u;
    stats->fill_rows_per_lane = e->strip_pairs * 2 > n ? (uint32_t)KS_R : 0u;
  }
  e->ran = false;
  return rc;
}

int32_t b2a_banded_band_ranges(b2a_engine* e, uint64_t pair, uint32_t* ranges, uint64_t capacity_pairs) {
  if (!e || !ranges) return B2A_E_INVALID;
  if (cudaSetDevice(e->device) != cudaSuccess) return e->fail(B2A_E_NO_DEVICE, "cudaSetDevice failed");
  if (pair < e->band_wave_lo || pair - e->band_wave_lo >= e->band_roff.size())
    return e->fail(B2A_E_STATE, "band ranges are kept for the pairs of the last banded call's last wave only");
  const uint64_t t = pair - e->band_wave_lo, cols = (uint64_t)e->band_ylen[t] + 1;
  if (capacity_pairs < cols) return e->fail(B2A_E_CAPACITY, "ranges buffer too small (needs y_len + 1 pairs)");
  CK(cudaMemcpyAsync(ranges, e->d_branges.as<uint8_t>() + e->band_roff[t], cols * 8, cudaMemcpyDeviceToHost, e->stream));
  CK(cudaStreamSynchronize(e->stream));
  return B2A_OK;
}

int32_t b2a_banded_strip_pairs(b2a_engine* e, uint64_t* n_pairs) {
  if (!e || !n_pairs) return B2A_E_INVALID;
  *n_pairs = e->strip_pairs;
  return B2A_OK;
}

uint32_t b2a_record_stride(uint32_t max_m, uint32_t max_n) {
  return 40u + ((max_m + max_n + 4u + 15u) & ~15u);
}

int32_t b2a_batch_records_into(b2a_engine* e, void* dev_dst, uint64_t dst_bytes, uint32_t* stride_bytes) {
  if (!e) return B2A_E_INVALID;
  if (!e->ran) return e->fail(B2A_E_STATE, "records requested before b2a_batch_run");
  if (cudaSetDevice(e->device) != cudaSuccess) return e->fail(B2A_E_NO_DEVICE, "cudaSetDevice failed");
  const uint32_t stride = b2a_record_stride(e->plan.maxm, e->plan.maxn);
  if (stride_bytes) *stride_bytes = stride;
  const uint64_t n = e->n_pairs;
  if (dst_bytes < n * stride) return e->fail(B2A_E_CAPACITY, "record buffer too small");
  if (n) {
    const unsigned g = (unsigned)((n * 32 + 255) / 256);
    records_kernel<<<g, 256, 0, e->stream>>>(
        e->d_score.as<int32_t>(), e->d_xs.as<uint32_t>(), e->d_xe.as<uint32_t>(), e->d_ys.as<uint32_t>(),
        e->d_ye.as<uint32_t>(), e->d_nops.as<uint32_t>(), e->d_clip.as<uint32_t>(),
        e->d_opsscratch.as<uint8_t>(), e->d_opssrc.as<uint64_t>(), reinterpret_cast<uint8_t*>(dev_dst),
        stride, n);
    CK(cudaGetLastError());
  }
  return B2A_OK;
}

int32_t b2a_batch_records(b2a_engine* e, void** dev_records, uint32_t* stride_bytes, uint64_t* n_records) {
  if (!e || !dev_records) return B2A_E_INVALID;
  if (!e->ran) return e->fail(B2A_E_STATE, "records requested before b2a_batch_run");
  const uint32_t stride = b2a_record_stride(e->plan.maxm, e->plan.maxn);
  CK(e->d_records.reserve(e->n_pairs * (uint64_t)stride + 16));
  int rc = b2a_batch_records_into(e, e->d_records.p, e->n_pairs * (uint64_t)stride, stride_bytes);
  if (rc) return rc;
  *dev_records = e->d_records.p;
  if (n_records) *n_records = e->n_pairs;
  return B2A_OK;
}

int32_t b2a_batch_compact_bytes(b2a_engine* e, uint64_t* segment_bytes) {
  if (!e || !segment_bytes) return B2A_E_INVALID;
  if (!e->ran) return e->fail(B2A_E_STATE, "compact results requested before b2a_batch_run");
  if (cudaSetDevice(e->device) != cudaSuccess) return e->fail(B2A_E_NO_DEVICE, "cudaSetDevice failed");
  const uint64_t n = e->n_pairs;
  uint64_t total = 0;
  if (n) CK(cudaMemcpyAsync(&total, e->d_opsoff.as<uint64_t>() + n, 8, cudaMemcpyDeviceToHost, e->stream));
  CK(cudaStreamSynchronize(e->stream));
  e->compact_hdr[0] = n;
  e->compact_hdr[1] = total;
  *segment_bytes = 64 + 40 * n + total;
  return B2A_OK;
}

int32_t b2a_batch_compact_into(b2a_engine* e, void* dev_dst, uint64_t dst_bytes) {
  if (!e || !dev_dst) return B2A_E_INVALID;
  if (!e->ran) return e->fail(B2A_E_STATE, "compact results requested before b2a_batch_run");
  if (cudaSetDevice(e->device) != cudaSuccess) return e->fail(B2A_E_NO_DEVICE, "cudaSetDevice failed");
  const uint64_t n = e->n_pairs;
  if (e->compact_hdr[0] != n) return e->fail(B2A_E_STATE, "b2a_batch_compact_bytes must be called first");
  const uint64_t total = e->compact_hdr[1];
  if (dst_bytes < 64 + 40 * n + total) return e->fail(B2A_E_CAPACITY, "compact buffer too small");
  uint8_t* dst = reinterpret_cast<uint8_t*>(dev_dst);
  cudaStream_t st = e->stream;
  CK(cudaMemcpyAsync(dst, e->compact_hdr, 64, cudaMemcpyHostToDevice, st));
  const DevBuf* arrays[6] = {&e->d_score, &e->d_xs, &e->d_xe, &e->d_ys, &e->d_ye, &e->d_nops};
  uint64_t off = 64;
  for (const DevBuf* a : arrays) {
    if (n) CK(cudaMemcpyAsync(dst + off, a->p, 4 * n, cudaMemcpyDeviceToDevice, st));
    off += 4 * n;
  }
  if (n) CK(cudaMemcpyAsync(dst + off, e->d_clip.p, 16 * n, cudaMemcpyDeviceToDevice, st));
  off += 16 * n;
  if (total) CK(cudaMemcpyAsync(dst + off, e->d_opsdense.p, total, cudaMemcpyDeviceToDevice, st));
  return B2A_OK;
}

// header of a fixed-capacity segment, written on the device: {n_pairs, ops_bytes (as produced), ops_bytes_kept}
__global__ void compact_header_kernel(uint64_t* hdr, const uint64_t* ops_off, uint64_t n, uint64_t cap_ops) {
  if (threadIdx.x == 0 && blockIdx.x == 0) {
    const uint64_t total = n ? ops_off[n] : 0;
    hdr[0] = n;
    hdr[1] = total;
    hdr[2] = total < cap_ops ? total : cap_ops;
    for (int k = 3; k < 8; ++k) hdr[k] = 0;
  }
}

int32_t b2a_batch_compact_fixed(b2a_engine* e, void* dev_dst, uint64_t capacity_bytes) {
  if (!e || !dev_dst) return B2A_E_INVALID;
  if (!e->ran) return e->fail(B2A_E_STATE, "compact results requested before b2a_batch_run");
  if (cudaSetDevice(e->device) != cudaSuccess) return e->fail(B2A_E_NO_DEVICE, "cudaSetDevice failed");
  const uint64_t n = e->n_pairs;
  if (capacity_bytes < 64 + 40 * n) return e->fail(B2A_E_CAPACITY, "compact segment capacity below 64 + 40 n_pairs");
  // never read past the dense ops buffer: the kept part is also bounded by what the buffer holds
  const uint64_t cap_ops = std::min<uint64_t>(capacity_bytes - 64 - 40 * n, e->d_opsdense.cap);
  uint8_t* dst = reinterpret_cast<uint8_t*>(dev_dst);
  cudaStream_t st = e->stream;
  compact_header_kernel<<<1, 32, 0, st>>>(reinterpret_cast<uint64_t*>(dst), e->d_opsoff.as<uint64_t>(), n, cap_ops);
  CK(cudaGetLastError());
  const DevBuf* arrays[6] = {&e->d_score, &e->d_xs, &e->d_xe, &e->d_ys, &e->d_ye, &e->d_nops};
  uint64_t off = 64;
  for (const DevBuf* a : arrays) {
    if (n) CK(cudaMemcpyAsync(dst + off, a->p, 4 * n, cudaMemcpyDeviceToDevice, st));
    off += 4 * n;
  }
  if (n) CK(cudaMemcpyAsync(dst + off, e->d_clip.p, 16 * n, cudaMemcpyDeviceToDevice, st));
  off += 16 * n;
  if (cap_ops && n) CK(cudaMemcpyAsync(dst + off, e->d_opsdense.p, cap_ops, cudaMemcpyDeviceToDevice, st));
  return B2A_OK;
}

int32_t b2a_gathered_fetch(b2a_engine* e, const void* dev_gathered, uint64_t segment_bytes, uint32_t n_segments,
                           b2a_results* r, uint64_t* n_pairs_total, uint64_t* d2h_bytes) {
  if (!e || !dev_gathered || !r || segment_bytes < 64) return B2A_E_INVALID;
  if (cudaSetDevice(e->device) != cudaSuccess) return e->fail(B2A_E_NO_DEVICE, "cudaSetDevice failed");
  cudaStream_t st = e->stream;
  const uint8_t* base = reinterpret_cast<const uint8_t*>(dev_gathered);
  std::vector<uint64_t> hdr((size_t)n_segments * 8);
  CK(cudaMemcpy2DAsync(hdr.data(), 64, base, segment_bytes, 64, n_segments, cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  uint64_t pairs = 0, ops = 0, moved = (uint64_t)n_segments * 64;
  for (uint32_t g = 0; g < n_segments; ++g) {
    const uint64_t n = hdr[8 * g], total = hdr[8 * g + 1];
    const uint64_t kept = hdr[8 * g + 2] ? hdr[8 * g + 2] : total;  // segments of b2a_batch_compact_into carry 0 there
    if (n > (segment_bytes - 64) / 40 || kept > segment_bytes - 64 - 40 * n)
      return e->fail(B2A_E_INVALID, "gathered segment header does not fit its segment");
    if (kept < total) return e->fail(B2A_E_CAPACITY, "a gathered segment was cut: its capacity was below its ops bytes");
    pairs += n;
    ops += total;
  }
  if (r->ops && ops > r->ops_capacity) return e->fail(B2A_E_CAPACITY, "ops buffer too small for the gathered batch");
  // ops_off of the whole batch = exclusive scan of every segment's n_ops in segment order, done on the device
  // (widen + cub scan over the concatenated counts) and copied straight into the caller's array; everything else
  // goes straight to its place in the caller's arrays as well
  if (r->ops_off && pairs) {
    CK(e->d_gnops.reserve((pairs + 1) * 4));
    CK(e->d_gnops64.reserve((pairs + 1) * 8));
    CK(e->d_goff.reserve((pairs + 1) * 8));
    uint64_t pb0 = 0;
    for (uint32_t g = 0; g < n_segments; ++g) {
      const uint64_t n = hdr[8 * g];
      if (n) CK(cudaMemcpyAsync(e->d_gnops.as<uint32_t>() + pb0, base + (uint64_t)g * segment_bytes + 64 + 20 * n, 4 * n,
                                cudaMemcpyDeviceToDevice, st));
      pb0 += n;
    }
    widen_kernel<<<(unsigned)((pairs + 1 + 255) / 256), 256, 0, st>>>(e->d_gnops.as<uint32_t>(), e->d_gnops64.as<uint64_t>(), pairs);
    CK(cudaGetLastError());
    size_t tmp = 0;
    CK(cub::DeviceScan::ExclusiveSum(nullptr, tmp, e->d_gnops64.as<uint64_t>(), e->d_goff.as<uint64_t>(), (int64_t)(pairs + 1), st));
    CK(e->d_scan.reserve(tmp + 16));
    CK(cub::DeviceScan::ExclusiveSum(e->d_scan.p, tmp, e->d_gnops64.as<uint64_t>(), e->d_goff.as<uint64_t>(), (int64_t)(pairs + 1), st));
    CK(cudaMemcpyAsync(r->ops_off, e->d_goff.p, (pairs + 1) * 8, cudaMemcpyDeviceToHost, st));
    moved += (pairs + 1) * 8;
  }
  uint64_t pb = 0, ob = 0;
  for (uint32_t g = 0; g < n_segments; ++g) {
    const uint64_t n = hdr[8 * g], total = hdr[8 * g + 1];
    const uint8_t* seg = base + (uint64_t)g * segment_bytes + 64;
    auto down = [&](void* dst, uint64_t off, uint64_t bytes) -> cudaError_t {
      if (!dst || !bytes) return cudaSuccess;
      moved += bytes;
      return cudaMemcpyAsync(dst, seg + off, bytes, cudaMemcpyDeviceToHost, st);
    };
    CK(down(r->score ? r->score + pb : nullptr, 0, 4 * n));
    CK(down(r->xstart ? r->xstart + pb : nullptr, 4 * n, 4 * n));
    CK(down(r->xend ? r->xend + pb : nullptr, 8 * n, 4 * n));
    CK(down(r->ystart ? r->ystart + pb : nullptr, 12 * n, 4 * n));
    CK(down(r->yend ? r->yend + pb : nullptr, 16 * n, 4 * n));
    CK(down(r->clip_len ? r->clip_len + 4 * pb : nullptr, 24 * n, 16 * n));
    CK(down(r->ops ? r->ops + ob : nullptr, 40 * n, total));
    pb += n;
    ob += total;
  }
  CK(cudaStreamSynchronize(st));
  if (r->ops_off) {
    if (!pairs) r->ops_off[0] = 0;
    if (r->ops_off[pairs] != ops) return e->fail(B2A_E_INVALID, "gathered segments: n_ops do not add up to the ops bytes");
  }
  if (r->status) std::memset(r->status, 0, pairs * 4);  // segments only carry completed batches
  if (n_pairs_total) *n_pairs_total = pairs;
  if (d2h_bytes) *d2h_bytes = moved;
  return B2A_OK;
}

int32_t b2a_compact_decode(const void* host_segment, uint64_t segment_bytes, uint64_t pair_base,
                           uint64_t ops_base, b2a_results* r, uint64_t* n_pairs, uint64_t* ops_bytes) {
  if (!host_segment || !r || segment_bytes < 64) return B2A_E_INVALID;
  const uint8_t* base = reinterpret_cast<const uint8_t*>(host_segment);
  uint64_t hdr[2];
  std::memcpy(hdr, base, 16);
  const uint64_t n = hdr[0], total = hdr[1];
  if (n > (segment_bytes - 64) / 40 || total > segment_bytes - 64 - 40 * n) return B2A_E_INVALID;
  const uint32_t* a = reinterpret_cast<const uint32_t*>(base + 64);
  if (r->score) std::memcpy(r->score + pair_base, a, 4 * n);
  if (r->xstart) std::memcpy(r->xstart + pair_base, a + n, 4 * n);
  if (r->xend) std::memcpy(r->xend + pair_base, a + 2 * n, 4 * n);
  if (r->ystart) std::memcpy(r->ystart + pair_base, a + 3 * n, 4 * n);
  if (r->yend) std::memcpy(r->yend + pair_base, a + 4 * n, 4 * n);
  const uint32_t* nops = a + 5 * n;
  if (r->clip_len) std::memcpy(r->clip_len + 4 * pair_base, a + 6 * n, 16 * n);
  uint64_t acc = 0;
  for (uint64_t p = 0; p < n; ++p) {
    if (r->ops_off) r->ops_off[pair_base + p] = ops_base + acc;
    acc += nops[p];
  }
  if (acc != total) return B2A_E_INVALID;
  if (r->ops) {
    if (ops_base + total > r->ops_capacity) return B2A_E_CAPACITY;
    std::memcpy(r->ops + ops_base, base + 64 + 40 * n, total);
  }
  if (n_pairs) *n_pairs = n;
  if (ops_bytes) *ops_bytes = total;
  return B2A_OK;
}

int32_t b2a_records_decode(const void* host_records, uint32_t stride, uint64_t n, b2a_results* r) {
  if (!host_records || !r || stride < 40) return B2A_E_INVALID;
  const uint8_t* base = reinterpret_cast<const uint8_t*>(host_records);
  uint64_t off = 0;
  for (uint64_t p = 0; p < n; ++p) {
    const uint32_t* h = reinterpret_cast<const uint32_t*>(base + p * stride);
    if (r->score) r->score[p] = (int32_t)h[0];
    if (r->xstart) r->xstart[p] = h[1];
    if (r->xend) r->xend[p] = h[2];
    if (r->ystart) r->ystart[p] = h[3];
    if (r->yend) r->yend[p] = h[4];
    const uint32_t nops = h[5];
    if (nops > stride - 40) return B2A_E_INVALID;
    if (r->clip_len)
      for (int k = 0; k < 4; ++k) r->clip_len[4 * p + k] = h[6 + k];
    if (r->ops_off) r->ops_off[p] = off;
    if (r->ops) {
      if (off + nops > r->ops_capacity) return B2A_E_CAPACITY;
      std::memcpy(r->ops + off, base + p * stride + 40, nops);
    }
    off += nops;
  }
  if (r->ops_off) r->ops_off[n] = off;
  return B2A_OK;
}

}  // extern "C"

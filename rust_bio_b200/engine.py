"""Engine: one CUDA device, batches in / Alignment fields out (thin wrapper over the C ABI)."""
from __future__ import annotations

import ctypes as C
from typing import Dict, Optional, Tuple

import numpy as np

from . import _lib
from ._lib import B2AError, CPairs, CResults, CScoreResults, CScoring, CStats

Batch = Tuple[np.ndarray, np.ndarray, np.ndarray, np.ndarray, np.ndarray]


def pack_pairs(pairs) -> Batch:
    """[(x_bytes, y_bytes), ...] -> (blob, x_off, x_len, y_off, y_len), 16-byte aligned sequences."""
    n = len(pairs)
    x_len = np.fromiter((len(p[0]) for p in pairs), dtype=np.uint32, count=n)
    y_len = np.fromiter((len(p[1]) for p in pairs), dtype=np.uint32, count=n)
    pad = lambda v: (v.astype(np.uint64) + np.uint64(15)) // np.uint64(16) * np.uint64(16)
    sizes = np.stack([pad(x_len), pad(y_len)], axis=1).reshape(-1)
    offs = np.concatenate([[0], np.cumsum(sizes)]).astype(np.uint64)
    blob = np.zeros(int(offs[-1]) + 16, dtype=np.uint8)
    x_off, y_off = offs[0:-1:2].copy(), offs[1::2].copy()
    for i, (x, y) in enumerate(pairs):
        blob[int(x_off[i]):int(x_off[i]) + len(x)] = np.frombuffer(bytes(x), dtype=np.uint8)
        blob[int(y_off[i]):int(y_off[i]) + len(y)] = np.frombuffer(bytes(y), dtype=np.uint8)
    return blob, x_off, x_len, y_off, y_len


class Results:
    """Host outputs of one batch (numpy arrays; pass pinned arrays via `out=` for speed)."""

    def __init__(self, n_pairs: int, ops_capacity: int, out: Optional[Dict[str, np.ndarray]] = None,
                 pair_status: bool = False):
        mk = lambda name, shape, dt: (out[name] if out and name in out else np.zeros(shape, dtype=dt))
        self.n_pairs = n_pairs
        self.score = mk("score", n_pairs, np.int32)
        self.xstart = mk("xstart", n_pairs, np.uint32)
        self.xend = mk("xend", n_pairs, np.uint32)
        self.ystart = mk("ystart", n_pairs, np.uint32)
        self.yend = mk("yend", n_pairs, np.uint32)
        self.ops_off = mk("ops_off", n_pairs + 1, np.uint64)
        self.ops = mk("ops", max(1, ops_capacity), np.uint8)
        self.clip_len = mk("clip_len", 4 * max(1, n_pairs), np.uint32)
        # per-pair B2A_PAIR_* codes: requested with pair_status=True (else a pair on which the reference would
        # panic fails the whole batch, include/b200align.h)
        self.status = mk("status", max(1, n_pairs), np.uint32) if pair_status else None
        p = lambda a: a.ctypes.data_as(C.c_void_p)
        self.c = CResults(p(self.score), p(self.xstart), p(self.xend), p(self.ystart), p(self.yend),
                          p(self.ops_off), p(self.ops), len(self.ops), p(self.clip_len),
                          p(self.status) if pair_status else None)

    def ops_of(self, i: int):
        """[(code, clip_len)] of pair i in alignment order."""
        lo, hi = int(self.ops_off[i]), int(self.ops_off[i + 1])
        res, k = [], 0
        for c in self.ops[lo:hi]:
            c = int(c)
            if c >= 4:
                res.append((c, int(self.clip_len[4 * i + k])))
                k += 1
            else:
                res.append((c, 0))
        return res

    def as_dict(self):
        return {k: getattr(self, k) for k in ("score", "xstart", "xend", "ystart", "yend")}


class ScoreResults:
    """Host outputs of one score-only batch: score, xend, yend (numpy arrays), and per-pair B2A_PAIR_* codes when
    requested with pair_status=True (else a pair on which the reference would panic fails the whole batch)."""

    def __init__(self, n_pairs: int, pair_status: bool = False):
        self.n_pairs = n_pairs
        self.score = np.zeros(n_pairs, dtype=np.int32)
        self.xend = np.zeros(n_pairs, dtype=np.uint32)
        self.yend = np.zeros(n_pairs, dtype=np.uint32)
        self.status = np.zeros(max(1, n_pairs), dtype=np.uint32) if pair_status else None
        p = lambda a: a.ctypes.data_as(C.c_void_p)
        self.c = CScoreResults(p(self.score), p(self.xend), p(self.yend), p(self.status) if pair_status else None)

    def as_dict(self):
        return {k: getattr(self, k) for k in ("score", "xend", "yend")}


class Engine:
    def __init__(self, device: int = 0):
        self._L = _lib.load()
        h = C.c_void_p()
        rc = self._L.b2a_engine_create(C.byref(h), int(device))
        if rc != 0:
            raise B2AError(rc, f"cannot create engine on cuda:{device} (no CPU fallback exists)")
        self._h = h
        self.device = device
        self.stats = CStats()
        self._keep = None

    def close(self):
        if getattr(self, "_h", None):
            self._L.b2a_engine_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc):
        if rc != 0:
            raise B2AError(rc, self._L.b2a_last_error(self._h).decode())

    def set_stream(self, cuda_stream: int):
        self._check(self._L.b2a_engine_set_stream(self._h, C.c_void_p(cuda_stream)))

    def set_tuning(self, lanes_per_pair: int, rows_per_lane: int):
        self._check(self._L.b2a_engine_set_tuning(self._h, lanes_per_pair, rows_per_lane))

    def last_alphabet(self) -> np.ndarray:
        """The alphabet the last stage used (given by the caller or found in the batch), ascending byte values."""
        buf = np.zeros(256, dtype=np.uint8)
        n = C.c_uint32()
        self._check(self._L.b2a_engine_last_alphabet(self._h, buf.ctypes.data_as(C.c_void_p), C.byref(n)))
        return buf[:n.value].copy()

    def set_walk(self, mode: int):
        """K2 shape: 0 automatic, 1 one lane per pair, 2 one warp per pair (b2a_engine_set_walk)."""
        self._check(self._L.b2a_engine_set_walk(self._h, int(mode)))

    def set_pipeline(self, chunks: int):
        self._check(self._L.b2a_engine_set_pipeline(self._h, int(chunks)))

    def set_traceback_budget(self, nbytes: int):
        self._check(self._L.b2a_engine_set_traceback_budget(self._h, int(nbytes)))

    @staticmethod
    def _cpairs(batch: Batch):
        blob, x_off, x_len, y_off, y_len = batch
        assert blob.dtype == np.uint8 and x_off.dtype == np.uint64 and y_off.dtype == np.uint64
        assert x_len.dtype == np.uint32 and y_len.dtype == np.uint32
        p = lambda a: a.ctypes.data_as(C.c_void_p)
        return CPairs(p(blob), p(x_off), p(x_len), p(y_off), p(y_len), blob.nbytes, len(x_len))

    @staticmethod
    def default_ops_capacity(batch: Batch) -> int:
        return int(batch[2].astype(np.uint64).sum() + batch[4].astype(np.uint64).sum() + 4 * len(batch[2]))

    def align_batch(self, mode: int, cscoring: CScoring, batch: Batch, results: Optional[Results] = None,
                    ops_capacity: Optional[int] = None) -> Results:
        """b2a_align_batch: host buffers in, host buffers out."""
        if results is None:
            results = Results(len(batch[2]), ops_capacity if ops_capacity is not None
                              else self.default_ops_capacity(batch))
        cp = self._cpairs(batch)
        self._check(self._L.b2a_align_batch(self._h, int(mode), C.byref(cscoring), C.byref(cp),
                                            C.byref(results.c), C.byref(self.stats)))
        return results

    def score_batch(self, mode: int, cscoring: CScoring, batch: Batch,
                    results: Optional[ScoreResults] = None) -> ScoreResults:
        """b2a_score_batch: score, xend and yend of every pair without the traceback (host buffers in and out)."""
        if results is None:
            results = ScoreResults(len(batch[2]))
        cp = self._cpairs(batch)
        self._check(self._L.b2a_score_batch(self._h, int(mode), C.byref(cscoring), C.byref(cp), C.byref(results.c),
                                            C.byref(self.stats)))
        return results

    def align_batch_banded(self, mode: int, cscoring: CScoring, k: int, w: int, batch: Batch,
                           results: Optional[Results] = None) -> Results:
        if results is None:
            results = Results(len(batch[2]), self.default_ops_capacity(batch))
        cp = self._cpairs(batch)
        self._check(self._L.b2a_align_batch_banded(self._h, int(mode), C.byref(cscoring), int(k), int(w),
                                                   C.byref(cp), C.byref(results.c), C.byref(self.stats)))
        return results

    @staticmethod
    def pack_bitenc_pairs(pairs):
        """[(BitEnc x, BitEnc y), ...] -> (blocks, x_block, x_len, y_block, y_len, width): the storages of all
        sequences concatenated (what b2a_packed_pairs points at)."""
        width = pairs[0][0].width if pairs else 2
        chunks, xb, xl, yb, yl, pos = [], [], [], [], [], 0
        for x, y in pairs:
            assert x.width == width and y.width == width, "one width per batch"
            xb.append(pos)
            xl.append(x.nr_symbols())
            chunks.append(x.storage)
            pos += x.nr_blocks()
            yb.append(pos)
            yl.append(y.nr_symbols())
            chunks.append(y.storage)
            pos += y.nr_blocks()
        blocks = np.concatenate(chunks + [np.zeros(4, dtype=np.uint32)]).astype(np.uint32)
        return (blocks, np.array(xb, dtype=np.uint64), np.array(xl, dtype=np.uint32), np.array(yb, dtype=np.uint64),
                np.array(yl, dtype=np.uint32), width)

    def align_batch_packed(self, mode: int, cscoring: CScoring, packed, results: Optional[Results] = None,
                           banded=None) -> Results:
        """b2a_align_batch_packed / b2a_align_batch_banded_packed: `packed` = pack_bitenc_pairs(...) (numpy arrays;
        pinned arrays give the fastest copies).  `banded` = (k, w) for the banded aligner."""
        from ._lib import CPackedPairs
        blocks, xb, xl, yb, yl, width = packed
        n = len(xl)
        if results is None:
            results = Results(n, int(xl.astype(np.uint64).sum() + yl.astype(np.uint64).sum() + 4 * n))
        p = lambda a: a.ctypes.data_as(C.c_void_p)
        pp = CPackedPairs(p(blocks), p(xb), p(xl), p(yb), p(yl), len(blocks), n, int(width))
        if banded is None:
            self._check(self._L.b2a_align_batch_packed(self._h, int(mode), C.byref(cscoring), C.byref(pp),
                                                       C.byref(results.c), C.byref(self.stats)))
        else:
            self._check(self._L.b2a_align_batch_banded_packed(self._h, int(mode), C.byref(cscoring), int(banded[0]),
                                                              int(banded[1]), C.byref(pp), C.byref(results.c),
                                                              C.byref(self.stats)))
        return results

    def align_batch_banded_hinted(self, mode: int, cscoring: CScoring, k: int, w: int, batch: Batch,
                                  matches, paths=None, allowed_mismatches: Optional[int] = None,
                                  use_lcskpp_union: bool = False, results: Optional[Results] = None) -> Results:
        """banded::Aligner::custom_with_{matches, expanded_matches, match_path} over a batch
        (b2a_align_batch_banded_hinted): matches[p] = [(xpos, ypos), ...] per pair, paths[p] = [index, ...]."""
        from ._lib import CBandHints
        n = len(batch[2])
        if len(matches) != n or (paths is not None and len(paths) != n):
            raise ValueError("one match list (and path) per pair")
        moff = np.zeros(n + 1, dtype=np.uint64)
        moff[1:] = np.cumsum([len(m) for m in matches])
        mxy = np.array([v for m in matches for mt in m for v in mt], dtype=np.uint32).reshape(-1)
        if mxy.size == 0:
            mxy = np.zeros(2, dtype=np.uint32)
        h = CBandHints(moff.ctypes.data, mxy.ctypes.data, None, None,
                       -1 if allowed_mismatches is None else int(allowed_mismatches), 1 if use_lcskpp_union else 0)
        if paths is not None:
            poff = np.zeros(n + 1, dtype=np.uint64)
            poff[1:] = np.cumsum([len(p) for p in paths])
            pidx = np.array([v for p in paths for v in p] or [0], dtype=np.uint32)
            h.path_off, h.path_idx = poff.ctypes.data, pidx.ctypes.data
        if results is None:
            results = Results(n, self.default_ops_capacity(batch))
        cp = self._cpairs(batch)
        self._check(self._L.b2a_align_batch_banded_hinted(self._h, int(mode), C.byref(cscoring), int(k), int(w),
                                                          C.byref(cp), C.byref(h), C.byref(results.c),
                                                          C.byref(self.stats)))
        return results

    def banded_band_ranges(self, pair: int, y_len: int) -> np.ndarray:
        """Band::ranges of `pair` of the last banded call: array [y_len + 1, 2] of (start, end) row ranges."""
        out = np.zeros((int(y_len) + 1, 2), dtype=np.uint32)
        self._check(self._L.b2a_banded_band_ranges(self._h, int(pair), out.ctypes.data_as(C.c_void_p), int(y_len) + 1))
        return out

    # staged form

    def banded_strip_pairs(self) -> int:
        """Pairs of the last banded call that ran the strip-wavefront fill (b2a_banded_strip_pairs)."""
        v = C.c_uint64(0)
        self._check(self._L.b2a_banded_strip_pairs(self._h, C.byref(v)))
        return int(v.value)

    def stage(self, mode: int, cscoring: CScoring, batch: Batch):
        self._keep = (batch, cscoring)
        cp = self._cpairs(batch)
        self._check(self._L.b2a_batch_stage(self._h, int(mode), C.byref(cscoring), C.byref(cp)))

    def run(self):
        self._check(self._L.b2a_batch_run(self._h))

    def fetch(self, results: Optional[Results]) -> Optional[Results]:
        self._check(self._L.b2a_batch_fetch(self._h, C.byref(results.c) if results else None,
                                            C.byref(self.stats)))
        return results

    def records_into(self, dev_ptr: int, nbytes: int) -> int:
        stride = C.c_uint32()
        self._check(self._L.b2a_batch_records_into(self._h, C.c_void_p(dev_ptr), int(nbytes), C.byref(stride)))
        return stride.value

    def compact_bytes(self) -> int:
        """Size of this batch's compact result segment (waits for the batch; see include/b200align.h)."""
        nb = C.c_uint64()
        self._check(self._L.b2a_batch_compact_bytes(self._h, C.byref(nb)))
        return int(nb.value)

    def compact_into(self, dev_ptr: int, nbytes: int) -> None:
        self._check(self._L.b2a_batch_compact_into(self._h, C.c_void_p(dev_ptr), int(nbytes)))

    def compact_fixed(self, dev_ptr: int, capacity_bytes: int) -> None:
        """b2a_batch_compact_fixed: the segment with a caller-fixed capacity; no wait, no size read-back."""
        self._check(self._L.b2a_batch_compact_fixed(self._h, C.c_void_p(dev_ptr), int(capacity_bytes)))

    def gathered_fetch(self, dev_ptr: int, segment_bytes: int, n_segments: int, results: Results):
        """b2a_gathered_fetch: gathered device segments -> host `results`; returns (pairs, d2h bytes)."""
        n, b = C.c_uint64(), C.c_uint64()
        self._check(self._L.b2a_gathered_fetch(self._h, C.c_void_p(dev_ptr), int(segment_bytes), int(n_segments),
                                               C.byref(results.c), C.byref(n), C.byref(b)))
        return int(n.value), int(b.value)

    def decode_compact(self, host_segments: np.ndarray, segment_bytes: int, n_segments: int, n_total: int,
                       ops_capacity: int) -> Results:
        """Decode `n_segments` gathered compact segments (each padded to segment_bytes) in rank order."""
        res = Results(n_total, ops_capacity)
        pair_base = ops_base = 0
        for r in range(n_segments):
            seg = host_segments[r * segment_bytes:(r + 1) * segment_bytes]
            n, nb = C.c_uint64(), C.c_uint64()
            rc = self._L.b2a_compact_decode(seg.ctypes.data_as(C.c_void_p), segment_bytes, pair_base, ops_base,
                                            C.byref(res.c), C.byref(n), C.byref(nb))
            if rc != 0:
                raise B2AError(rc, "b2a_compact_decode")
            pair_base += n.value
            ops_base += nb.value
        if pair_base != n_total:
            raise B2AError(-2, "compact segments hold %d pairs, expected %d" % (pair_base, n_total))
        res.ops_off[n_total] = ops_base
        return res

    def record_stride(self, max_m: int, max_n: int) -> int:
        return int(self._L.b2a_record_stride(max_m, max_n))

    def decode_records(self, host_records: np.ndarray, stride: int, n: int, ops_capacity: int) -> Results:
        res = Results(n, ops_capacity)
        rc = self._L.b2a_records_decode(host_records.ctypes.data_as(C.c_void_p), stride, n, C.byref(res.c))
        if rc != 0:
            raise B2AError(rc, "b2a_records_decode")
        return res


_default: Dict[int, Engine] = {}


def default_engine(device: int = 0) -> Engine:
    if device not in _default:
        _default[device] = Engine(device)
    return _default[device]


class MultiEngine:
    """Every visible GPU from one process (b2a_multi_*): the batch is split over the devices, one ncclAllGather
    reassembles the results, device 0's copy is returned.  Same results as Engine.align_batch."""

    def __init__(self, device_ids=None):
        self._L = _lib.load()
        h = C.c_void_p()
        if device_ids is None:
            rc = self._L.b2a_multi_create(C.byref(h), None, 0)
        else:
            ids = (C.c_int32 * len(device_ids))(*device_ids)
            rc = self._L.b2a_multi_create(C.byref(h), ids, len(device_ids))
        if rc != 0:
            raise B2AError(rc, "cannot create the multi-GPU engine (no CPU fallback exists)")
        self._h = h
        self.stats = CStats()

    @property
    def n_devices(self) -> int:
        return int(self._L.b2a_multi_device_count(self._h))

    @property
    def exchange_kind(self) -> str:
        return self._L.b2a_multi_exchange_kind(self._h).decode()

    def align_batch(self, mode: int, cscoring: CScoring, batch: Batch, results: Optional[Results] = None) -> Results:
        if results is None:
            results = Results(len(batch[2]), Engine.default_ops_capacity(batch))
        cp = Engine._cpairs(batch)
        rc = self._L.b2a_multi_align_batch(self._h, int(mode), C.byref(cscoring), C.byref(cp), C.byref(results.c),
                                           C.byref(self.stats))
        if rc != 0:
            raise B2AError(rc, self._L.b2a_multi_last_error(self._h).decode())
        return results

    def close(self):
        if getattr(self, "_h", None):
            self._L.b2a_multi_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

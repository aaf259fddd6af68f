"""Mirror of `bio::alignment::pairwise` (reference src/alignment/pairwise/mod.rs) on the B200 engine.

Same names, argument meaning and error behaviour as the reference:
  MIN_SCORE (mod.rs:174), MatchParams (186-217), Scoring (238-429), Aligner (472-1015).
`Aligner.global` is spelled `global_` (Python keyword).  Every per-pair method is a batch of one;
`*_batch` methods take [(x, y), ...] and are the form the GPU is built for.  The reference panics on
bad parameters (assert!); this mirror raises AssertionError with the same message.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass, replace
from typing import Callable, List, Optional, Sequence, Tuple, Union

import numpy as np

from . import scores as _scores
from ._lib import (CScoring, MIN_SCORE, MODE_CUSTOM, MODE_GLOBAL, MODE_LOCAL, MODE_SEMIGLOBAL)
from .alignment import Alignment, AlignmentMode, AlignmentOperation
from .engine import Engine, Results, ScoreResults, default_engine, pack_pairs

__all__ = ["MIN_SCORE", "MatchParams", "Scoring", "Aligner", "MatchFunc"]

MatchFunc = Union["MatchParams", Callable[[int, int], int]]
DEFAULT_ALIGNER_CAPACITY = 200  # mod.rs:483
_MATRIX_ALPHABET = bytes(range(65, 91)) + b"*"


@dataclass(frozen=True)
class MatchParams:
    """mod.rs:186-217"""
    match_score: int
    mismatch_score: int

    @staticmethod
    def new(match_score: int, mismatch_score: int) -> "MatchParams":
        assert match_score >= 0, "match_score can't be negative"
        assert mismatch_score <= 0, "mismatch_score can't be positive"
        return MatchParams(match_score, mismatch_score)

    def score(self, a: int, b: int) -> int:
        return self.match_score if a == b else self.mismatch_score

    def __call__(self, a: int, b: int) -> int:
        return self.score(a, b)


@dataclass
class Scoring:
    """mod.rs:238-429. Builders return a modified copy (the reference's `mut self -> Self`)."""
    gap_open: int
    gap_extend: int
    match_fn: MatchFunc
    match_scores: Optional[Tuple[int, int]] = None
    xclip_prefix: int = MIN_SCORE
    xclip_suffix: int = MIN_SCORE
    yclip_prefix: int = MIN_SCORE
    yclip_suffix: int = MIN_SCORE

    @staticmethod
    def from_scores(gap_open: int, gap_extend: int, match_score: int, mismatch_score: int) -> "Scoring":
        assert gap_open <= 0, "gap_open can't be positive"
        assert gap_extend <= 0, "gap_extend can't be positive"
        return Scoring(gap_open, gap_extend, MatchParams.new(match_score, mismatch_score),
                       (match_score, mismatch_score))

    @staticmethod
    def new(gap_open: int, gap_extend: int, match_fn: MatchFunc) -> "Scoring":
        assert gap_open <= 0, "gap_open can't be positive"
        assert gap_extend <= 0, "gap_extend can't be positive"
        return Scoring(gap_open, gap_extend, match_fn, None)

    def _clip(self, **kw) -> "Scoring":
        for v in kw.values():
            assert v <= 0, "Clipping penalty can't be positive"
        return replace(self, **kw)

    def xclip(self, penalty: int) -> "Scoring":
        return self._clip(xclip_prefix=penalty, xclip_suffix=penalty)

    def xclip_prefix_(self, penalty: int) -> "Scoring":
        return self._clip(xclip_prefix=penalty)

    def xclip_suffix_(self, penalty: int) -> "Scoring":
        return self._clip(xclip_suffix=penalty)

    def yclip(self, penalty: int) -> "Scoring":
        return self._clip(yclip_prefix=penalty, yclip_suffix=penalty)

    def yclip_prefix_(self, penalty: int) -> "Scoring":
        return self._clip(yclip_prefix=penalty)

    def yclip_suffix_(self, penalty: int) -> "Scoring":
        return self._clip(yclip_suffix=penalty)

    # -- C ABI view --------------------------------------------------------------------------
    def to_c(self, batch=None):
        """-> (CScoring, keepalive).  `batch` = (blob, x_off, x_len, y_off, y_len) (or a bare array of sequence
        bytes).  Closures are tabulated over the symbols present in the SEQUENCES (mod.rs:221-228: the
        reference only ever calls match_fn on sequence bytes) -- not over the blob's padding bytes."""
        keep = []
        cs = CScoring(self.gap_open, self.gap_extend, self.xclip_prefix, self.xclip_suffix,
                      self.yclip_prefix, self.yclip_suffix, 0, 0, 0, None, None, 0)
        if self.match_scores is not None:
            cs.has_match_scores = 1
        fn = self.match_fn
        if isinstance(fn, MatchParams):
            cs.match_score, cs.mismatch_score = fn.match_score, fn.mismatch_score
            if self.match_scores is not None:
                assert tuple(self.match_scores) == (fn.match_score, fn.mismatch_score)
        else:
            if getattr(fn, "matrix_name", None):
                table = _scores.matrix_table256(fn.matrix_name)
                alpha = np.frombuffer(_MATRIX_ALPHABET, dtype=np.uint8).copy()
            else:
                syms = _symbols_present(batch)
                table = _scores.tabulate(fn, syms.tolist())
                alpha = syms.astype(np.uint8)
            table = np.ascontiguousarray(table, dtype=np.int32)
            keep += [table, alpha]
            cs.table = table.ctypes.data_as(C.c_void_p)
            cs.alphabet = alpha.ctypes.data_as(C.c_void_p)
            cs.alphabet_len = len(alpha)
            if self.match_scores is not None:
                cs.match_score, cs.mismatch_score = self.match_scores
        return cs, keep


def _symbols_present(batch) -> np.ndarray:
    """Sorted distinct bytes of the sequences of a batch (padding between sequences is not looked at)."""
    if batch is None:
        return np.zeros(0, np.uint8)
    if isinstance(batch, np.ndarray):
        return np.unique(batch)
    blob, x_off, x_len, y_off, y_len = batch
    if len(x_len) == 0 or len(blob) == 0:
        return np.zeros(0, np.uint8)
    starts = np.concatenate([x_off, y_off]).astype(np.int64)
    lens = np.concatenate([x_len, y_len]).astype(np.int64)
    delta = np.zeros(len(blob) + 1, dtype=np.int32)
    np.add.at(delta, starts, 1)
    np.add.at(delta, starts + lens, -1)
    inside = np.cumsum(delta[:-1]) > 0
    return np.nonzero(np.bincount(blob[inside], minlength=256))[0].astype(np.uint8)


_PAIR_STATUS_TEXT = {1: "the reference panics (or never returns) on this pair: mod.rs:905 / banded.rs:777-831",
                     2: "banded: more k-mer matches than the engine's per-pair limit",
                     4: "banded: the reference panics on these caller-supplied matches/path"}


def _alignments(res: Results, pairs, mode: int, on_panic: str, banded: bool = False, result_mode=None) -> list:
    """Results -> [Alignment]; per-pair failures (Results.status) raise or become None."""
    from ._lib import B2AError
    out = []
    for i, (x, y) in enumerate(pairs):
        st = int(res.status[i]) if res.status is not None else 0
        if st:
            if on_panic == "raise":
                raise B2AError(-4 if st == 1 else (-5 if st == 2 else -1), f"pair {i}: " + _PAIR_STATUS_TEXT.get(st, str(st)))
            out.append(None)
            continue
        ops = [AlignmentOperation(c, l) for c, l in res.ops_of(i)]
        # banded.rs:407-420: a band above MAX_CELLS returns the empty alignment with xlen = ylen = 0
        refused = banded and int(res.score[i]) == MIN_SCORE and not ops
        out.append(Alignment(int(res.score[i]), int(res.ystart[i]), int(res.xstart[i]), int(res.yend[i]),
                             int(res.xend[i]), 0 if refused else len(y), 0 if refused else len(x), ops,
                             mode if result_mode is None else result_mode))
    return out


def _check_scoring(s: Scoring):
    """Aligner::with_capacity_and_scoring asserts, mod.rs:554-571"""
    assert s.gap_open <= 0, "gap_open can't be positive"
    assert s.gap_extend <= 0, "gap_extend can't be positive"
    assert s.xclip_prefix <= 0, "Clipping penalty (x prefix) can't be positive"
    assert s.xclip_suffix <= 0, "Clipping penalty (x suffix) can't be positive"
    assert s.yclip_prefix <= 0, "Clipping penalty (y prefix) can't be positive"
    assert s.yclip_suffix <= 0, "Clipping penalty (y suffix) can't be positive"


class Aligner:
    """mod.rs:472-1015. Holds a Scoring and an engine handle instead of host scratch vectors."""

    def __init__(self, scoring: Scoring, engine: Optional[Engine] = None):
        self.scoring = scoring
        self._engine = engine

    # constructors, mod.rs:495-583 (capacities are hints there; here they are ignored)
    @staticmethod
    def new(gap_open: int, gap_extend: int, match_fn: MatchFunc, engine: Optional[Engine] = None) -> "Aligner":
        return Aligner.with_capacity(DEFAULT_ALIGNER_CAPACITY, DEFAULT_ALIGNER_CAPACITY, gap_open,
                                     gap_extend, match_fn, engine)

    @staticmethod
    def with_capacity(m: int, n: int, gap_open: int, gap_extend: int, match_fn: MatchFunc,
                      engine: Optional[Engine] = None) -> "Aligner":
        assert gap_open <= 0, "gap_open can't be positive"
        assert gap_extend <= 0, "gap_extend can't be positive"
        return Aligner(Scoring.new(gap_open, gap_extend, match_fn), engine)

    @staticmethod
    def with_scoring(scoring: Scoring, engine: Optional[Engine] = None) -> "Aligner":
        return Aligner.with_capacity_and_scoring(DEFAULT_ALIGNER_CAPACITY, DEFAULT_ALIGNER_CAPACITY,
                                                 scoring, engine)

    @staticmethod
    def with_capacity_and_scoring(m: int, n: int, scoring: Scoring, engine: Optional[Engine] = None) -> "Aligner":
        _check_scoring(scoring)
        return Aligner(scoring, engine)

    @property
    def engine(self) -> Engine:
        if self._engine is None:
            self._engine = default_engine(0)
        return self._engine

    # batch forms ------------------------------------------------------------------------------
    def _batch(self, mode: int, pairs: Sequence[Tuple[bytes, bytes]], on_panic: str = "raise") -> List[Alignment]:
        """on_panic: the reference panics per CALL (mod.rs:905); a batch either raises for the first such pair
        ("raise", what a loop over the reference's per-pair calls does) or returns None in its place ("none")."""
        batch = pack_pairs(pairs)
        cs, keep = self.scoring.to_c(batch)
        res = self.engine.align_batch(mode, cs, batch, results=Results(len(pairs), Engine.default_ops_capacity(batch),
                                                                       pair_status=True))
        return _alignments(res, pairs, mode, on_panic)

    def batch_bitenc(self, mode: int, pairs, on_panic: str = "raise") -> List[Alignment]:
        """Aligner::{custom,global,semiglobal,local} over [(BitEnc x, BitEnc y), ...] (bio::data_structures::bitenc,
        holding alphabets::RankTransform ranks): the packed storage goes to the GPU as it is.  `match_fn` scores
        RANKS (MatchParams: equality of ranks == equality of symbols)."""
        packed = Engine.pack_bitenc_pairs(pairs)
        ranks = np.arange(1 << packed[5], dtype=np.uint8)
        cs, keep = self.scoring.to_c(ranks)
        lens = [(x.nr_symbols(), y.nr_symbols()) for x, y in pairs]
        res = Results(len(pairs), sum(a + b + 4 for a, b in lens), pair_status=True)
        self.engine.align_batch_packed(mode, cs, packed, results=res)
        fake = [(b"\0" * a, b"\0" * b) for a, b in lens]  # _alignments only needs the lengths
        return _alignments(res, fake, mode, on_panic)

    def custom_batch(self, pairs, on_panic: str = "raise"):
        return self._batch(MODE_CUSTOM, pairs, on_panic)

    def global_batch(self, pairs, on_panic: str = "raise"):
        return self._batch(MODE_GLOBAL, pairs, on_panic)

    def semiglobal_batch(self, pairs, on_panic: str = "raise"):
        return self._batch(MODE_SEMIGLOBAL, pairs, on_panic)

    def local_batch(self, pairs, on_panic: str = "raise"):
        return self._batch(MODE_LOCAL, pairs, on_panic)

    # score-only batch forms: (score, xend, yend) of the Alignment the batch forms above return, without the
    # traceback (b2a_score_batch) -- for callers that rank or filter candidates and never read the path
    def _scores_batch(self, mode: int, pairs: Sequence[Tuple[bytes, bytes]],
                      on_panic: str = "raise") -> List[Optional[Tuple[int, int, int]]]:
        """on_panic as in the batch forms.  A pair is flagged only where the reference's panic lies on the part
        of the walk the score-only call replays (row m and column n, include/b200align.h)."""
        from ._lib import B2AError
        batch = pack_pairs(pairs)
        cs, keep = self.scoring.to_c(batch)
        res = self.engine.score_batch(mode, cs, batch, results=ScoreResults(len(pairs), pair_status=True))
        out = []
        for i in range(len(pairs)):
            st = int(res.status[i])
            if st:
                if on_panic == "raise":
                    raise B2AError(-4, f"pair {i}: " + _PAIR_STATUS_TEXT.get(st, str(st)))
                out.append(None)
                continue
            out.append((int(res.score[i]), int(res.xend[i]), int(res.yend[i])))
        return out

    def custom_scores_batch(self, pairs, on_panic: str = "raise"):
        return self._scores_batch(MODE_CUSTOM, pairs, on_panic)

    def global_scores_batch(self, pairs, on_panic: str = "raise"):
        return self._scores_batch(MODE_GLOBAL, pairs, on_panic)

    def semiglobal_scores_batch(self, pairs, on_panic: str = "raise"):
        return self._scores_batch(MODE_SEMIGLOBAL, pairs, on_panic)

    def local_scores_batch(self, pairs, on_panic: str = "raise"):
        return self._scores_batch(MODE_LOCAL, pairs, on_panic)

    def custom_score(self, x: bytes, y: bytes) -> Tuple[int, int, int]:
        return self._scores_batch(MODE_CUSTOM, [(x, y)])[0]

    def global_score(self, x: bytes, y: bytes) -> Tuple[int, int, int]:
        return self._scores_batch(MODE_GLOBAL, [(x, y)])[0]

    def semiglobal_score(self, x: bytes, y: bytes) -> Tuple[int, int, int]:
        return self._scores_batch(MODE_SEMIGLOBAL, [(x, y)])[0]

    def local_score(self, x: bytes, y: bytes) -> Tuple[int, int, int]:
        return self._scores_batch(MODE_LOCAL, [(x, y)])[0]

    # per-pair forms, mod.rs:591, 925, 954, 986
    def custom(self, x: bytes, y: bytes) -> Alignment:
        return self._batch(MODE_CUSTOM, [(x, y)])[0]

    def global_(self, x: bytes, y: bytes) -> Alignment:
        return self._batch(MODE_GLOBAL, [(x, y)])[0]

    def semiglobal(self, x: bytes, y: bytes) -> Alignment:
        return self._batch(MODE_SEMIGLOBAL, [(x, y)])[0]

    def local(self, x: bytes, y: bytes) -> Alignment:
        return self._batch(MODE_LOCAL, [(x, y)])[0]


setattr(Aligner, "global", Aligner.global_)  # reachable as getattr(aligner, "global")


class TracebackCell:
    """`pairwise::TracebackCell` (mod.rs:1026-1114): the packed u16 of one traceback cell -- bits 0-3 the I
    layer's move, 4-7 the D layer's, 8-11 the S layer's.  The engine's own traceback is a 4-bit re-encoding
    (DESIGN.md section 2); this public type is kept for callers that used it."""
    TB_START, TB_INS, TB_DEL, TB_SUBST, TB_MATCH = 0, 1, 2, 3, 4
    TB_XCLIP_PREFIX, TB_XCLIP_SUFFIX, TB_YCLIP_PREFIX, TB_YCLIP_SUFFIX = 5, 6, 7, 8
    TB_MAX = 8
    _I_POS, _D_POS, _S_POS = 0, 4, 8
    __slots__ = ("v",)

    def __init__(self, v: int = 0):
        self.v = int(v) & 0xFFFF

    @staticmethod
    def new() -> "TracebackCell":
        return TracebackCell()

    def _set_bits(self, pos: int, value: int) -> None:
        assert value <= TracebackCell.TB_MAX, "Expected a value <= TB_MAX while setting traceback bits"
        self.v = (self.v & ~(0b1111 << pos) & 0xFFFF) | (value << pos)

    def set_i_bits(self, value: int) -> None:
        self._set_bits(self._I_POS, value)

    def set_d_bits(self, value: int) -> None:
        self._set_bits(self._D_POS, value)

    def set_s_bits(self, value: int) -> None:
        self._set_bits(self._S_POS, value)

    def get_i_bits(self) -> int:
        return (self.v >> self._I_POS) & 0b1111

    def get_d_bits(self) -> int:
        return (self.v >> self._D_POS) & 0b1111

    def get_s_bits(self) -> int:
        return (self.v >> self._S_POS) & 0b1111

    def set_all(self, value: int) -> None:
        self.set_i_bits(value)
        self.set_d_bits(value)
        self.set_s_bits(value)

    def __eq__(self, other) -> bool:
        return isinstance(other, TracebackCell) and self.v == other.v

    def __hash__(self) -> int:
        return hash(self.v)

    def __repr__(self) -> str:
        return "TracebackCell { v: %d }" % self.v

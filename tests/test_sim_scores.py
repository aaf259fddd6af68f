"""The score-only path (b2a_score_batch) compiled for the CPU: the F_NOTB fill must leave the boundary and rows
arenas word for word as the traceback fill does, and the score-only epilogue (row m, fix-ups, end walk) must give
the score, xend and yend of the full simulated walk and of the oracle."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import sim_util
from parity_util import MODES, oracle_batch
from rust_bio_b200 import engine, synth

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, "sim", "b2a_sim_scores.cpp")
DEPS = [SRC] + sim_util.DEPS
MIN = -858993459
FIELDS = ("score", "xend", "yend")

_libs = {}


def _sim(krel=None):
    """The harness library; krel: a build with chunks of 2^krel columns for the relative packed trackers."""
    if krel not in _libs:
        so = os.path.join(HERE, "sim", "libb2asim_scores%s.so" % (("_k%d" % krel) if krel else ""))
        if not os.path.exists(so) or any(os.path.getmtime(d) > os.path.getmtime(so) for d in DEPS):
            subprocess.check_call(["g++", "-O2", "-std=c++17", "-fwrapv", "-fPIC", "-shared", "-Wno-unknown-pragmas"] +
                                  ([f"-DB2A_KREL_BITS={krel}"] if krel else []) + ["-o", so, SRC])
        lib = C.CDLL(so)
        lib.sim_scores_batch.restype = C.c_int
        _libs[krel] = lib
    return _libs[krel]


def _scores(mode, s, batch, G=1, R=16, no_pack=0, no_lut=0, warp=0, rel_pack=0, krel=None):
    """Score-only results; two scratch fills must agree and neither may leave the arenas different."""
    blob, x_off, x_len, y_off, y_len = (np.ascontiguousarray(a) for a in batch)
    n = len(x_len)
    p = lambda a: a.ctypes.data_as(C.c_void_p)
    outs = []
    for garbage in (0x00, 0x7F):
        out = {k: np.zeros(n, dtype=np.uint32) for k in ("xend", "yend", "status", "gap_clip")}
        out["score"] = np.zeros(n, dtype=np.int32)
        bits = (2 if no_pack else 0) | (4 if no_lut else 0) | (8 if warp else 0) | (16 if rel_pack else 0)
        diff = _sim(krel).sim_scores_batch(int(mode), C.byref(sim_util.SimScoring.from_buffer_copy(bytes(s))), p(blob),
                                           p(x_off), p(x_len), p(y_off), p(y_len), C.c_uint64(n), int(G), int(R), bits,
                                           garbage, p(out["score"]), p(out["xend"]), p(out["yend"]), p(out["status"]),
                                           p(out["gap_clip"]))
        assert diff == 0, f"{diff} boundary / rows bytes differ from the traceback fill (or the plan is wrong)"
        outs.append(out)
    for k in outs[0]:
        assert np.array_equal(outs[0][k], outs[1][k]), ("scratch-dependent result", k)
    return outs[0]


def _check(oracle, mode, s, batch, what, full_kw=None, **kw):
    """Score-only fields == the full simulated walk's == the oracle's, for every pair; returns the number of pairs
    whose walk takes a suffix clip after a gap run along row m or column n."""
    ref, ref_ops = oracle_batch(oracle, mode, s, batch)
    got = _scores(MODES[mode], s, batch, **kw)
    full, _ = sim_util.align_batch(MODES[mode], s, *batch, **(full_kw if full_kw is not None else {
        k: v for k, v in kw.items() if k in ("G", "R", "no_pack", "no_lut", "rel_pack")}),
        warp_walk=kw.get("warp", 0))
    assert not np.any(full["status"]), what
    assert not np.any(got["status"]), what
    for f in FIELDS:
        bad = np.nonzero(got[f].astype(np.int64) != ref[f].astype(np.int64))[0]
        assert len(bad) == 0, f"{what}: {f} differs from the oracle for {len(bad)} pairs (first {bad[0]})"
        assert np.array_equal(got[f].astype(np.int64), full[f].astype(np.int64)), f"{what}: {f} vs the full walk"
    return int(got["gap_clip"].sum())


@pytest.mark.parametrize("mode", ["global", "semiglobal", "local", "custom"])
@pytest.mark.parametrize("G,R,warp", [(1, 16, 0), (8, 20, 1), (132, 8, 0), (32, 8, 1)])
def test_scores_ragged_modes_shapes(oracle, mode, G, R, warp):
    """Ragged, partly filled blocks; G = 1, 8 and 32 (132: strip-pipelined tasks); both epilogue forms."""
    L = 3 * (32 if G == 132 else G) * R // 2 + 19  # one and a half strips
    batch = synth.ragged_pairs(11 + G, 45, L, L)
    s, _ = oracle.make_scoring(-5, -1, 1, -1, None, -3, -2, 0, -4)  # custom: every clip live
    _check(oracle, mode, s, batch, f"{mode} {G}x{R}", G=G, R=R, warp=warp)


def test_scores_tiny_shapes(oracle):
    """m, n in {0, 1, 2} (and 3), every mode, dead and live clips."""
    xs, ys = [], []
    for m in range(0, 4):
        for n in range(0, 4):
            xs += [m] * 3
            ys += [n] * 3
    rng = np.random.default_rng(9)
    blob = np.frombuffer(b"ACGT", dtype=np.uint8)[rng.integers(0, 2, size=sum(xs) + sum(ys) + 1)]
    lens = np.array([v for pair in zip(xs, ys) for v in pair], dtype=np.uint64)
    offs = np.concatenate([[0], np.cumsum(lens)[:-1]]).astype(np.uint64)
    batch = (blob, offs[0::2].copy(), np.array(xs, dtype=np.uint32), offs[1::2].copy(), np.array(ys, dtype=np.uint32))
    for mode in ("custom", "local", "global", "semiglobal"):
        for clips in [(MIN, MIN, MIN, MIN), (0, 0, 0, 0), (-1, 0, MIN, -2), (0, MIN, MIN, 0), (MIN, 0, 0, MIN)]:
            s, _ = oracle.make_scoring(-2, -1, 2, -1, None, *clips)
            for warp in (0, 1):
                _check(oracle, mode, s, batch, f"tiny {mode} {clips} warp={warp}", R=16, warp=warp)


def test_scores_custom_clip_combinations(oracle):
    """Every live/dead combination of the four clip penalties, MatchParams by compare and by LUT, packed and
    explicit trackers; at least one path must end in a suffix clip followed by a gap run along row m or column n."""
    # gap_open above gap_extend: fix-up 2 can make S(m, n) an Ins out of a row whose y-suffix clip took all of y
    # (x = AA, y = CCC: Ins to (1, n), then Yclip)
    batch = synth.ragged_pairs(77, 160, 20, 40, alphabet=b"ACGT", min_len=1)
    tiny = synth.ragged_pairs(78, 96, 3, 6, alphabet=b"AC", min_len=1)
    hits = 0
    for combo in range(16):
        for go, ge, live, b in ((-1, -1, -1, batch), (-1, -5, 0, tiny)):
            clips = [(live if (combo >> k) & 1 else MIN) for k in range(4)]
            s, _ = oracle.make_scoring(go, ge, 1, -3, None, *clips)
            for no_pack, no_lut in ((0, 0), (1, 1)):
                hits += _check(oracle, "custom", s, b, f"clips {clips} go={go} ge={ge} no_pack={no_pack}", R=16,
                               no_pack=no_pack, no_lut=no_lut)
    assert hits > 0, "no case took a suffix clip after a gap run along row m or column n"


def test_scores_blosum62(oracle):
    from rust_bio_b200 import scores
    table = scores.matrix_table256("blosum62")
    batch = synth.ragged_pairs(3, 90, 60, 60, alphabet=synth.PROTEIN, min_len=1)
    for mode, go in (("local", -10), ("global", -5), ("semiglobal", -11), ("custom", -8)):
        s, keep = oracle.make_scoring(go, -1, 0, 0, table, -5, -5, -7, -7)
        _check(oracle, mode, s, batch, f"blosum62 {mode}", R=16)
        _check(oracle, mode, s, batch, f"blosum62 {mode} 8x20 warp", G=8, R=20, warp=1)


def test_scores_relative_trackers_short_chunks(oracle):
    """The long-sequence tracker form (F_PACKREL) with chunks of 2^3 columns, so that the row trackers are flushed
    many times inside each pair, on the thread-per-pair and the strip-pipelined warp-per-pair shapes."""
    batch = synth.ragged_pairs(5, 40, 30, 70)
    for mode, clips in (("local", None), ("custom", (-3, -2, MIN, -4)), ("custom", (MIN, -2, 0, MIN))):
        s, _ = oracle.make_scoring(-5, -1, 1, -1, None, *(clips or (MIN,) * 4))
        for G, R in ((1, 16), (132, 8)):
            _check(oracle, mode, s, batch, f"relpack {mode} {clips} {G}x{R}", full_kw={"G": G, "R": R, "rel_pack": 1},
                   G=G, R=R, rel_pack=1, krel=3)


def test_scores_uniform_c1_shape(oracle):
    """150 x 150 local (C1's shape): uniform blocks, an unpaired partly filled last block."""
    batch = synth.uniform_pairs(synth.BASES["C1"], 0, 70, 150, 150)
    s, _ = oracle.make_scoring(-5, -1, 1, -1)
    _check(oracle, "local", s, batch, "C1 shape", R=16)
    _check(oracle, "local", s, batch, "C1 shape 8x20 warp", G=8, R=20, warp=1)


def test_scores_engine_batch_pack_pairs(oracle):
    """Sequences given as Python pairs go through the same staging as the C-ABI layout."""
    pairs = [(b"ACGTACGT", b"ACGAACGT"), (b"", b"AC"), (b"GGG", b""), (b"A", b"A")]
    batch = engine.pack_pairs(pairs)
    s, _ = oracle.make_scoring(-5, -1, 1, -1, None, -1, -1, -1, -1)
    _check(oracle, "custom", s, batch, "pack_pairs", R=16)

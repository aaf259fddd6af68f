"""The pair-packed K1 fill (b2a_fill_pair16.cuh, int16x2 cells, two blocks per lane) compiled for the CPU: its
scratch must equal the int32 fill's word for word on every valid pair, and K2's walk on it must match the oracle."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import sim_util
from parity_util import assert_same, oracle_batch
from rust_bio_b200 import synth

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, "sim", "b2a_sim_pair16.cpp")
SO = os.path.join(HERE, "sim", "libb2asim_pair16.so")
DEPS = [SRC] + sim_util.DEPS + [os.path.join(sim_util.ROOT, "rust_bio_b200", "csrc", "b2a_fill_pair16.cuh")]

_lib = None


def _sim():
    global _lib
    if _lib is None:
        if not os.path.exists(SO) or any(os.path.getmtime(d) > os.path.getmtime(SO) for d in DEPS):
            subprocess.check_call(["g++", "-O2", "-std=c++17", "-fwrapv", "-fPIC", "-shared", "-Wno-unknown-pragmas",
                                   "-o", SO, SRC])
        _lib = C.CDLL(SO)
        _lib.sim_pair16_batch.restype = C.c_int
    return _lib


def _run(orc_scoring, batch, garbage=0x00):
    blob, x_off, x_len, y_off, y_len = batch
    s = sim_util.SimScoring.from_buffer_copy(bytes(orc_scoring))
    blob = np.ascontiguousarray(blob, dtype=np.uint8)
    x_off = np.ascontiguousarray(x_off, dtype=np.uint64)
    y_off = np.ascontiguousarray(y_off, dtype=np.uint64)
    x_len = np.ascontiguousarray(x_len, dtype=np.uint32)
    y_len = np.ascontiguousarray(y_len, dtype=np.uint32)
    n = len(x_len)
    cap = x_len.astype(np.uint64) + y_len.astype(np.uint64) + np.uint64(4)
    ops_off = np.concatenate([[0], np.cumsum(cap)]).astype(np.uint64)
    ops = np.zeros(int(ops_off[-1]), dtype=np.uint8)
    out = {k: np.zeros(n, dtype=np.uint32) for k in ("xstart", "xend", "ystart", "yend", "n_ops", "status")}
    out["score"] = np.zeros(n, dtype=np.int32)
    out["clip_len"] = np.zeros(4 * n, dtype=np.uint32)
    p = lambda a: a.ctypes.data_as(C.c_void_p)
    diff = _sim().sim_pair16_batch(C.byref(s), p(blob), p(x_off), p(x_len), p(y_off), p(y_len), C.c_uint64(n),
                                   int(garbage), p(out["score"]), p(out["xstart"]), p(out["xend"]), p(out["ystart"]),
                                   p(out["yend"]), p(out["n_ops"]), p(out["clip_len"]), p(out["status"]), p(ops),
                                   p(ops_off))
    oplists = []
    for i in range(n):
        codes = ops[int(ops_off[i]):int(ops_off[i]) + int(out["n_ops"][i])]
        oplists.append(sim_util.decode_ops(codes, out["clip_len"][4 * i:4 * i + 4]))
    return diff, out, oplists


def _check(oracle, scoring, batch, what):
    for garbage in (0x00, 0x7F):
        diff, got, ops = _run(scoring, batch, garbage)
        assert diff == 0, f"{what}: {diff} scratch words differ from the int32 fill"
    ref, ref_ops = oracle_batch(oracle, "local", scoring, batch)
    assert_same(got, ops, ref, ref_ops, batch, what)
    return got


def _same_pairs(x: bytes, y: bytes, count: int):
    blob = np.frombuffer((x + y) * count, dtype=np.uint8)
    step = len(x) + len(y)
    xo = np.arange(count, dtype=np.uint64) * np.uint64(step)
    return (blob, xo, np.full(count, len(x), dtype=np.uint32), xo + np.uint64(len(x)),
            np.full(count, len(y), dtype=np.uint32))


def _concat(a, b):
    """Two batches in the C-ABI layout as one."""
    shift = np.uint64(len(a[0]))
    return (np.concatenate([a[0], b[0]]), np.concatenate([a[1], b[1] + shift]), np.concatenate([a[2], b[2]]),
            np.concatenate([a[3], b[3] + shift]), np.concatenate([a[4], b[4]]))


@pytest.mark.parametrize("n_pairs", [64, 96, 70, 33])
def test_pairpack_uniform_150_local(oracle, n_pairs):
    """C1/C2's shape; 96 and 33 pairs leave the last block without a partner, 70 and 33 fill it partly."""
    batch = synth.uniform_pairs(synth.BASES["C2"], 0, n_pairs, 150, 150)
    s, _ = oracle.make_scoring(-5, -1, 1, -1)
    _check(oracle, s, batch, f"150x150 local, {n_pairs} pairs")


@pytest.mark.parametrize("m,n", [(161, 150), (17, 40), (2, 9), (100, 1)])
def test_pairpack_strip_edges(oracle, m, n):
    """m - 1 a multiple of 16 (no poison rows), one row, a single column."""
    batch = synth.uniform_pairs(synth.BASES["C1"], 7, 64, m, n)
    s, _ = oracle.make_scoring(-5, -1, 1, -1)
    _check(oracle, s, batch, f"{m}x{n} local")


def test_pairpack_score_bound_255(oracle):
    """m = 256, n = 255: the longest shape, and identical sequences reach the score bound 255 exactly."""
    rand = synth.uniform_pairs(synth.BASES["C2"], 100, 40, 256, 255)
    x = bytes(rand[0][int(rand[1][0]):int(rand[1][0]) + 256])
    batch = _concat(_same_pairs(x, x[:255], 30), rand)
    s, _ = oracle.make_scoring(-5, -1, 1, -1)
    got = _check(oracle, s, batch, "256x255 local")
    assert int(got["score"].max()) == 255


def test_pairpack_acgtn_and_wide_penalties(oracle):
    """Five symbols, a mismatch below the gap-open penalty (a larger bias), and a table-free MatchParams LUT."""
    batch = synth.uniform_pairs(synth.BASES["C1"], 3, 80, 120, 110, alphabet=b"ACGTN")
    s, _ = oracle.make_scoring(-3, -2, 2, -7)
    _check(oracle, s, batch, "ACGTN 120x110 local (2, -7, -3, -2)")


def test_pairpack_seven_symbols(oracle):
    batch = synth.uniform_pairs(synth.BASES["C3"], 0, 64, 90, 90, alphabet=b"ACGTNRY")
    s, _ = oracle.make_scoring(-4, -1, 1, -2)
    _check(oracle, s, batch, "7-symbol 90x90 local")

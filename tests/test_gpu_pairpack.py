"""GPU parity of the pair-packed 1x16 local fill (b2a_fill_pair16.cuh) and of the int32 fill it falls back to just
beyond each of its limits; and the two paths against each other on a C2-sized batch (B2A_PAIRPACK)."""
import numpy as np
import pytest

from parity_util import MODES, assert_same, oracle_batch

pytestmark = pytest.mark.gpu
MIN = -858993459


@pytest.fixture(scope="module")
def eng():
    from rust_bio_b200.engine import Engine
    e = Engine(0)
    yield e
    e.close()


def _cs(go, ge, ma, mi, mode):
    from rust_bio_b200._lib import CScoring
    clips = (0, 0, 0, 0) if mode == "local" else (MIN, MIN, MIN, MIN)
    return CScoring(go, ge, clips[0], clips[1], clips[2], clips[3], ma, mi, 0, None, None, 0)


def _run(eng, oracle, batch, mode="local", sc=(-5, -1, 1, -1), shape=(1, 16), what=""):
    s, _ = oracle.make_scoring(*sc)
    ref, ref_ops = oracle_batch(oracle, mode, s, batch, threads=8)
    if shape:
        eng.set_tuning(*shape)
    try:
        res = eng.align_batch(MODES[mode], _cs(*sc, mode), batch)
    finally:
        eng.set_tuning(0, 0)
    got = res.as_dict()
    assert_same(got, [res.ops_of(i) for i in range(res.n_pairs)], ref, ref_ops, batch, what)
    return got


def _concat(a, b):
    shift = np.uint64(len(a[0]))
    return (np.concatenate([a[0], b[0]]), np.concatenate([a[1], b[1] + shift]), np.concatenate([a[2], b[2]]),
            np.concatenate([a[3], b[3] + shift]), np.concatenate([a[4], b[4]]))


def _bound_batch(m, n, count, seed):
    """Random m x n pairs plus pairs whose y is a prefix of x: the local score is min(m, n) * match."""
    from rust_bio_b200 import engine, synth
    rand = synth.uniform_pairs(synth.BASES["C2"], seed, count, m, n)
    x = bytes(rand[0][int(rand[1][0]):int(rand[1][0]) + m])
    same = engine.pack_pairs([(x, x[:n])] * 40)
    return _concat(same, rand)


@pytest.mark.parametrize("n_pairs", [1000, 1024 + 33, 100_000])
def test_pairpack_c2_shape_every_field(eng, oracle, n_pairs):
    """150x150 local (1, -1, -5, -1); 1,057 pairs leave an unpaired, partly filled last block.  100k pairs pick
    the 1x16 shape without tuning."""
    from rust_bio_b200 import synth
    batch = synth.uniform_pairs(synth.BASES["C2"], 0, n_pairs, 150, 150)
    _run(eng, oracle, batch, shape=None if n_pairs >= 49152 else (1, 16), what=f"C2 shape {n_pairs} pairs")


def test_pairpack_score_bound_255(eng, oracle):
    got = _run(eng, oracle, _bound_batch(256, 255, 1000, 11), what="256x255, score 255")
    assert int(got["score"].max()) == 255


def test_pairpack_acgtn(eng, oracle):
    from rust_bio_b200 import synth
    batch = synth.uniform_pairs(synth.BASES["C1"], 5, 1000, 140, 130, alphabet=b"ACGTN")
    _run(eng, oracle, batch, sc=(-3, -2, 2, -7), what="ACGTN (2, -7, -3, -2)")


@pytest.mark.parametrize("case", ["m257", "score256", "eight_symbols", "ragged", "global"])
def test_int32_fill_just_beyond_each_limit(eng, oracle, case):
    """Each limit of the packed path exceeded by one: the int32 fill runs these, with the same results."""
    from rust_bio_b200 import synth
    mode, sc = "local", (-5, -1, 1, -1)
    if case == "m257":
        batch = synth.uniform_pairs(synth.BASES["C1"], 0, 1000, 257, 200)
    elif case == "score256":
        batch = _bound_batch(256, 128, 1000, 3)
        sc = (-5, -1, 2, -1)
    elif case == "eight_symbols":
        batch = synth.uniform_pairs(synth.BASES["C1"], 0, 1000, 150, 150, alphabet=b"ACGTNRYK")
    elif case == "ragged":
        a = synth.uniform_pairs(synth.BASES["C1"], 0, 500, 150, 150)
        b = synth.uniform_pairs(synth.BASES["C1"], 500, 500, 151, 150)
        batch = _concat(a, b)
    else:
        mode = "global"
        batch = synth.uniform_pairs(synth.BASES["C1"], 0, 1000, 150, 150)
    _run(eng, oracle, batch, mode=mode, sc=sc, what=case)


def test_pairpack_on_and_off_agree_200k(monkeypatch):
    """200k C2 pairs with B2A_PAIRPACK=0 (int32 fill) and =1 (pair-packed): identical results, fresh engines."""
    from rust_bio_b200 import synth
    from rust_bio_b200.engine import Engine
    batch = synth.uniform_pairs(synth.BASES["C2"], 0, 200_000, 150, 150)
    out = {}
    for knob in ("0", "1"):
        monkeypatch.setenv("B2A_PAIRPACK", knob)
        e = Engine(0)
        try:
            res = e.align_batch(MODES["local"], _cs(-5, -1, 1, -1, "local"), batch)
            out[knob] = (res.as_dict(), [res.ops_of(i) for i in range(0, res.n_pairs, 97)])
        finally:
            e.close()
    for k in out["0"][0]:
        assert np.array_equal(out["0"][0][k], out["1"][0][k]), k
    assert out["0"][1] == out["1"][1]

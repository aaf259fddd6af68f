"""GPU tests of the score-only batch (b2a_score_batch): score, xend and yend equal the full call's (and the
oracle's) for every pair it reports as OK, in every shape, mode, tracker form, wave count and through the chunk
pipeline; errors are the full call's."""
import os
import subprocess
import sys

import numpy as np
import pytest

from parity_util import MODES, oracle_batch

pytestmark = pytest.mark.gpu
MIN = -858993459
FIELDS = ("score", "xend", "yend")
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def eng():
    from rust_bio_b200.engine import Engine
    e = Engine(0)
    yield e
    e.close()


def _cs(go, ge, ma, mi, clips=(MIN, MIN, MIN, MIN), table=None):
    from rust_bio_b200._lib import CScoring
    import ctypes as C
    t = None if table is None else table.ctypes.data_as(C.c_void_p)
    return CScoring(go, ge, clips[0], clips[1], clips[2], clips[3], ma, mi, 0, t, None, 0)


def _both(eng, mode, cs, batch):
    """(full Results, ScoreResults), both with per-pair status"""
    from rust_bio_b200.engine import Engine, Results, ScoreResults
    n = len(batch[2])
    full = eng.align_batch(MODES[mode], cs, batch, results=Results(n, Engine.default_ops_capacity(batch), pair_status=True))
    full_stats = dict(eng.stats.as_dict())
    got = eng.score_batch(MODES[mode], cs, batch, results=ScoreResults(n, pair_status=True))
    return full, full_stats, got, dict(eng.stats.as_dict())


def _same_as_full(full, got, what):
    """Equal on every pair the full call reports OK; a pair only the full call flags must be an interior panic."""
    ok = full.status[:full.n_pairs] == 0
    for f in FIELDS:
        a, b = getattr(full, f)[ok].astype(np.int64), getattr(got, f)[ok].astype(np.int64)
        bad = np.nonzero(a != b)[0]
        assert len(bad) == 0, f"{what}: {f} differs on {len(bad)} pairs"
    both = (full.status[:full.n_pairs] != 0) & (got.status[:got.n_pairs] != 0)
    only_full = (full.status[:full.n_pairs] != 0) & (got.status[:got.n_pairs] == 0)
    assert not np.any((got.status[:got.n_pairs] != 0) & ok), f"{what}: score-only flags a pair the full call does not"
    if only_full.any():
        print(f"{what}: {int(only_full.sum())} pairs panic in the interior walk only (flagged by the full call)")
    return int(both.sum()), int(only_full.sum())


def test_c1_every_pair_equals_oracle(eng, oracle):
    from rust_bio_b200 import synth
    from rust_bio_b200.engine import ScoreResults
    batch = synth.uniform_pairs(synth.BASES["C1"], 0, 1000, 150, 150)
    s, _ = oracle.make_scoring(-5, -1, 1, -1, None, 0, 0, 0, 0)
    ref, _ = oracle_batch(oracle, "local", s, batch, threads=8)
    got = eng.score_batch(MODES["local"], _cs(-5, -1, 1, -1, (0, 0, 0, 0)), batch, results=ScoreResults(1000, True))
    assert not np.any(got.status)
    for f in FIELDS:
        assert np.array_equal(getattr(got, f).astype(np.int64), ref[f].astype(np.int64)), f
    assert eng.stats.traceback_bytes == 0


@pytest.mark.parametrize("pairpack", ["1", "0"])
def test_c2_200k_pairpack_on_off(pairpack):
    """200k C2 pairs, pair-packed fill on and off (B2A_PAIRPACK is read when the engine is created): identical to
    local_batch field for field.  A fresh process so that the knob takes effect."""
    code = (
        "import numpy as np\n"
        "from rust_bio_b200 import synth\n"
        "from rust_bio_b200.engine import Engine, Results, ScoreResults\n"
        "from rust_bio_b200._lib import CScoring\n"
        "b = synth.uniform_pairs(synth.BASES['C2'], 0, 200000, 150, 150)\n"
        "cs = CScoring(-5, -1, 0, 0, 0, 0, 1, -1, 0, None, None, 0)\n"
        "e = Engine(0)\n"
        "f = e.align_batch(3, cs, b)\n"
        "g = e.score_batch(3, cs, b, results=ScoreResults(200000, True))\n"
        "assert not g.status.any()\n"
        "assert e.stats.traceback_bytes == 0 and e.stats.fill_lanes_per_pair == 1\n"
        "for k in ('score', 'xend', 'yend'): assert np.array_equal(getattr(f, k), getattr(g, k)), k\n"
        "print('ok')\n")
    env = dict(os.environ, B2A_PAIRPACK=pairpack, PYTHONPATH=ROOT)
    r = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True, cwd=ROOT)
    assert r.returncode == 0 and "ok" in r.stdout, r.stdout + r.stderr


SHAPES = [(1, 16), (1, 8), (1, 20), (2, 16), (2, 20), (4, 16), (8, 16), (8, 20), (32, 8), (32, 16)]


@pytest.mark.parametrize("G,R", SHAPES)
def test_every_shape_ragged_mixed_modes(eng, G, R):
    from rust_bio_b200 import synth
    batch = synth.ragged_pairs(40 + G + R, 300, 700, 700)
    eng.set_tuning(G, R)
    try:
        for mode, clips in (("local", None), ("global", None), ("semiglobal", None), ("custom", (-3, -2, 0, -4)),
                            ("custom", (MIN, -1, MIN, -1))):
            for walk in (1, 2):
                eng.set_walk(walk)
                full, _, got, st = _both(eng, mode, _cs(-5, -1, 1, -1, clips or (MIN,) * 4), batch)
                _same_as_full(full, got, f"{G}x{R} {mode} {clips} walk={walk}")
                assert st["traceback_bytes"] == 0 and st["fill_lanes_per_pair"] == G
    finally:
        eng.set_walk(0)
        eng.set_tuning(0, 0)


@pytest.mark.parametrize("mode", ["global", "semiglobal", "local", "custom"])
@pytest.mark.parametrize("no_packrel", ["0", "1"])
def test_long_4200_all_modes(mode, no_packrel):
    """4,200 x 4,200: the relative packed trackers (F_PACKREL) and, with B2A_NO_PACKREL=1, the explicit ones."""
    code = (
        "import numpy as np\n"
        "from rust_bio_b200 import synth\n"
        "from rust_bio_b200.engine import Engine, Results, ScoreResults\n"
        "from rust_bio_b200._lib import CScoring\n"
        "MIN = -858993459\n"
        f"mode = {MODES[mode]}\n"
        "clips = {0: (-7, -3, -9, -2), 1: (MIN,) * 4, 2: (MIN, MIN, 0, 0), 3: (0, 0, 0, 0)}[mode]\n"
        "b = synth.uniform_pairs(synth.BASES['C4'], 0, 6, 4200, 4200)\n"
        "cs = CScoring(-5, -1, clips[0], clips[1], clips[2], clips[3], 1, -1, 0, None, None, 0)\n"
        "e = Engine(0)\n"
        "f = e.align_batch(mode, cs, b, results=Results(6, Engine.default_ops_capacity(b), pair_status=True))\n"
        "g = e.score_batch(mode, cs, b, results=ScoreResults(6, True))\n"
        "ok = f.status == 0\n"
        "assert not (g.status.astype(bool) & ok).any()\n"
        "for k in ('score', 'xend', 'yend'): assert np.array_equal(getattr(f, k)[ok], getattr(g, k)[ok]), k\n"
        "print('ok')\n")
    env = dict(os.environ, B2A_NO_PACKREL=no_packrel, PYTHONPATH=ROOT)
    r = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True, cwd=ROOT)
    assert r.returncode == 0 and "ok" in r.stdout, r.stdout + r.stderr


def test_10k_blosum62_local(eng):
    from rust_bio_b200 import scores, synth
    table = np.ascontiguousarray(scores.matrix_table256("blosum62"), dtype=np.int32).reshape(-1)
    batch = synth.uniform_pairs(synth.BASES["C5"], 0, 8, 10000, 10000, alphabet=synth.PROTEIN)
    full, _, got, st = _both(eng, "local", _cs(-11, -1, 0, 0, (0, 0, 0, 0), table), batch)
    assert not np.any(full.status)
    _same_as_full(full, got, "10k blosum62 local")
    assert st["traceback_bytes"] == 0


def test_small_budget_one_wave(eng):
    from rust_bio_b200 import synth
    batch = synth.ragged_pairs(8, 3000, 400, 400)
    eng.set_traceback_budget(8 << 20)
    try:
        full, fst, got, st = _both(eng, "local", _cs(-5, -1, 1, -1, (0, 0, 0, 0)), batch)
    finally:
        eng.set_traceback_budget(0)
    assert fst["waves"] > 2
    assert st["waves"] == 1 and st["traceback_bytes"] == 0
    _same_as_full(full, got, "small budget")


def test_pipelined_equals_unpipelined(eng):
    from rust_bio_b200 import synth
    from rust_bio_b200.engine import ScoreResults
    batch = synth.ragged_pairs(21, 300_000, 160, 160)
    cs = _cs(-5, -1, 1, -1, (-3, -2, 0, -4))
    a = eng.score_batch(MODES["custom"], cs, batch, results=ScoreResults(300_000, True))
    eng.set_pipeline(0)
    try:
        b = eng.score_batch(MODES["custom"], cs, batch, results=ScoreResults(300_000, True))
    finally:
        eng.set_pipeline(5)
    for f in FIELDS + ("status",):
        assert np.array_equal(getattr(a, f), getattr(b, f)), f
    full, _, got, _ = _both(eng, "custom", cs, batch)
    _same_as_full(full, got, "pipelined custom")


def test_error_parity(eng):
    from rust_bio_b200 import engine
    from rust_bio_b200._lib import B2AError
    from rust_bio_b200.engine import Results, ScoreResults

    def rc(fn):
        try:
            fn()
            return 0
        except B2AError as ex:
            return ex.code

    # scores x lengths beyond 2^27
    big = engine.pack_pairs([(b"A" * 3000, b"A" * 3000)])
    cs = _cs(-5, -1, 1 << 16, -1)
    r1 = rc(lambda: eng.align_batch(1, cs, big))
    r2 = rc(lambda: eng.score_batch(1, cs, big))
    assert r1 == r2 == -4
    # a byte outside the caller's alphabet
    alpha = np.frombuffer(b"ACGT", dtype=np.uint8).copy()
    from rust_bio_b200._lib import CScoring
    import ctypes as C
    csa = CScoring(-5, -1, MIN, MIN, MIN, MIN, 1, -1, 0, None, alpha.ctypes.data_as(C.c_void_p), 4)
    bad = engine.pack_pairs([(b"ACGT", b"ACGN")] * 3)
    r1 = rc(lambda: eng.align_batch(1, csa, bad))
    r2 = rc(lambda: eng.score_batch(1, csa, bad))
    assert r1 == r2 == -1
    # an empty batch
    empty = engine.pack_pairs([])
    r1 = rc(lambda: eng.align_batch(1, _cs(-5, -1, 1, -1), empty, results=Results(0, 1)))
    r2 = rc(lambda: eng.score_batch(1, _cs(-5, -1, 1, -1), empty, results=ScoreResults(0)))
    assert r1 == r2 == 0
    # a positive gap penalty
    r1 = rc(lambda: eng.align_batch(1, _cs(1, -1, 1, -1), bad))
    r2 = rc(lambda: eng.score_batch(1, _cs(1, -1, 1, -1), bad))
    assert r1 == r2 == -1


def test_status_parity_custom_clips(eng):
    """Random custom clip penalties with zero gap costs (the reference's panic paths live there): every pair the
    score-only call flags is flagged by the full call; the pairs only the full call flags are counted."""
    from rust_bio_b200 import synth
    rng = np.random.default_rng(4)
    total_both = total_interior = 0
    for k in range(12):
        pick = lambda: int(rng.choice([MIN, 0, 0, -1, -3]))
        cs = _cs(int(rng.choice([0, -1, -5])), int(rng.choice([0, -1])), 1, int(rng.choice([-1, 0, -3])),
                 (pick(), pick(), pick(), pick()))
        batch = synth.ragged_pairs(500 + k, 400, 60, 60, alphabet=b"AC")
        full, _, got, _ = _both(eng, "custom", cs, batch)
        b, i = _same_as_full(full, got, f"custom clips #{k}")
        total_both += b
        total_interior += i
    print(f"status parity: {total_both} pairs flagged by both calls, {total_interior} by the full call only")


def test_aligner_score_forms(eng):
    from rust_bio_b200.pairwise import Aligner, MatchParams
    al = Aligner.with_capacity(10, 10, -5, -1, MatchParams.new(1, -1), engine=eng)
    pairs = [(b"ACCGTGGAT", b"AAAAACCGTTGAT"), (b"ACGT", b"TTACGTTT"), (b"", b"AC")]
    for name in ("custom", "global_", "semiglobal", "local"):
        full = getattr(al, name.rstrip("_") + "_batch")(pairs)
        fn = name.rstrip("_") + "_scores_batch"
        sc = getattr(al, fn)(pairs)
        assert sc == [(a.score, a.xend, a.yend) for a in full], name
        one = getattr(al, name.rstrip("_") + "_score")(*pairs[0])
        assert one == sc[0]

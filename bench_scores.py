#!/usr/bin/env python
"""Full alignment vs score-only (b2a_score_batch) on the benchmark shapes, one GPU, one-call form (host inputs
and host outputs, copies included).

Configs (SURVEY 8d generators and BASE seeds): C2 (1M x 150x150 DNA local, 1 -1 -5 -1), C2_10k (10k of them),
C3 (100k x 1000x1000 DNA global, 1 -1 -5 -1) and C5's per-GPU share at 8 GPUs (1,250 x 10000x10000 protein,
BLOSUM62 go -10 ge -1, local).  Protocol: 3 warm-up calls per arm, then 10 timed calls per arm, the two arms
alternating; each call ends in the host copies, so a host clock around it times the whole step.  Reports median,
min and max per arm, the engine's fill / walk times, and checks that score, xend and yend of the score-only call
equal the full call's on every pair.  Writes one JSON file (--out) and prints it.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import subprocess
import time

import numpy as np

from rust_bio_b200 import scores, synth
from rust_bio_b200._lib import MIN_SCORE, MODE_GLOBAL, MODE_LOCAL, CScoring
from rust_bio_b200.engine import Engine, Results, ScoreResults


def configs(names):
    dna_local = CScoring(-5, -1, 0, 0, 0, 0, 1, -1, 1, None, None, 0)
    dna_global = CScoring(-5, -1, MIN_SCORE, MIN_SCORE, MIN_SCORE, MIN_SCORE, 1, -1, 1, None, None, 0)
    table = np.ascontiguousarray(scores.matrix_table256("blosum62"), dtype=np.int32)
    alpha = np.frombuffer(bytes(range(65, 91)) + b"*", dtype=np.uint8).copy()
    c5 = CScoring(-10, -1, 0, 0, 0, 0, 0, 0, 0, table.ctypes.data_as(C.c_void_p), alpha.ctypes.data_as(C.c_void_p),
                  len(alpha))
    make = {
        "C2": lambda: (synth.uniform_pairs(synth.BASES["C2"], 0, 1_000_000, 150, 150), MODE_LOCAL, dna_local),
        "C2_10k": lambda: (synth.uniform_pairs(synth.BASES["C2"], 0, 10_000, 150, 150), MODE_LOCAL, dna_local),
        "C3": lambda: (synth.uniform_pairs(synth.BASES["C3"], 0, 100_000, 1000, 1000), MODE_GLOBAL, dna_global),
        "C5": lambda: (synth.uniform_pairs(synth.BASES["C5"], 0, 1250, 10000, 10000, alphabet=synth.PROTEIN),
                       MODE_LOCAL, c5),
    }
    for n in names:
        yield (n,) + make[n]() + ((table, alpha),)


def stat(v):
    v = np.asarray(v, dtype=np.float64)
    return {"median": round(float(np.median(v)), 4), "min": round(float(v.min()), 4), "max": round(float(v.max()), 4)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--configs", default="C2,C2_10k,C3,C5")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--runs", type=int, default=10)
    ap.add_argument("--out", default=None, help="JSON output path")
    a = ap.parse_args()
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                         text=True).stdout.strip().splitlines()
    eng = Engine(0)
    out = {"gpu": gpu[0] if gpu else None, "protocol": f"{a.warmup} warm-up + {a.runs} timed one-call runs per arm, "
           "alternating; host clock around each call", "configs": []}
    for name, batch, mode, cs, _keep in configs([c for c in a.configs.split(",") if c]):
        n = len(batch[2])
        full = Results(n, Engine.default_ops_capacity(batch))
        so = ScoreResults(n)
        t = {"full": [], "score": []}
        k = {"full": {"fill_ms": [], "walk_ms": []}, "score": {"fill_ms": [], "walk_ms": []}}
        for it in range(a.warmup + a.runs):
            for arm in ("full", "score"):
                t0 = time.perf_counter()
                if arm == "full":
                    eng.align_batch(mode, cs, batch, results=full)
                else:
                    eng.score_batch(mode, cs, batch, results=so)
                dt = (time.perf_counter() - t0) * 1e3
                if it >= a.warmup:
                    t[arm].append(dt)
                    k[arm]["fill_ms"].append(eng.stats.fill_ms)
                    k[arm]["walk_ms"].append(eng.stats.walk_ms)
                if arm == "score":
                    tb = int(eng.stats.traceback_bytes)
        same = all(np.array_equal(getattr(full, f), getattr(so, f)) for f in ("score", "xend", "yend"))
        line = {"config": name, "pairs": n, "ms_full": stat(t["full"]), "ms_score": stat(t["score"]),
                "fill_ms_full": stat(k["full"]["fill_ms"]), "fill_ms_score": stat(k["score"]["fill_ms"]),
                "walk_ms_full": stat(k["full"]["walk_ms"]), "walk_ms_score": stat(k["score"]["walk_ms"]),
                "speedup": round(float(np.median(t["full"]) / np.median(t["score"])), 3),
                "score_traceback_bytes": tb, "fields_equal": bool(same)}
        out["configs"].append(line)
        print(json.dumps(line), flush=True)
    if a.out:
        with open(a.out, "w") as f:
            json.dump(out, f, indent=1)
    eng.close()
    if not all(c["fields_equal"] for c in out["configs"]):
        raise SystemExit("score-only fields differ from the full call")


if __name__ == "__main__":
    main()

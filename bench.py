#!/usr/bin/env python
"""bench.py -- GCUPS of the batched pairwise-alignment hot path on N B200s (BASELINE.json metric).

A step = one pass of the hot path (K0 pack -> K1 fill -> K2 row-m/fix-ups/walk -> ops compaction, plus the one
NCCL all-gather of result segments when N > 1) over one batch of synthetic pairs.
Headline workload at every N: BASELINE config 2 -- 1M pairs of 150x150 uniform random DNA per GPU, local affine
(match 1, mismatch -1, gap_open -5, gap_extend -1); weak scaling (the pair list is split by rank).

  value    : whole-job GCUPS with the batch resident in HBM (device-timed, CUDA events, max over ranks); at N > 1
             the all-gather of step k runs on a side stream under the kernels of step k+1 (fixed-capacity
             segments: no size agreement, no host sync inside the timed region)
  e2e      : the same metric from pinned HOST buffers to HOST results: b2a_align_batch at N = 1; at N > 1 every
             rank stages + runs its shard, the segments are all-gathered and rank 0 reassembles the whole batch in
             host memory (b2a_gathered_fetch) -- the gather and the reassembly are inside the timed region
  roofline : the K1 fill kernel against the int32-ALU roof (SURVEY 8d: 25 ops/cell local, 22 global/semiglobal/
             banded; peak = lane-ops/s measured in this run by b2a_util_int32_peak), with the HBM view beside it
             (roofline.hbm: SURVEY 8d algorithmic bytes, and the DRAM traffic ncu measured)
  configs  : the other BASELINE shapes on this GPU: C2 at 10k pairs (the north_star target), C3 (its 1/N share of
             100k pairs), C4 and C5 (the per-GPU share of the 8-GPU configuration), each with GCUPS, roofline
             fraction, fill shape and an oracle-checked sample
  verify   : (N > 1) the gathered segments decoded on rank 0 and compared with the oracle on a sample
  cpu_baseline / --impl reference : the oracle (C++ restatement of rust-bio 4.0.1: rust-bio itself cannot be
             built in this image) on the box's host cores, pinned threads, bounded sample
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

M, N_LEN = 150, 150
SCORING = dict(gap_open=-5, gap_extend=-1, match=1, mismatch=-1)
WORKLOAD = "C2: 1M pairs/GPU of 150x150 uniform random DNA, Aligner::local, match 1 mismatch -1 gap_open -5 gap_extend -1"
OPS_LOCAL, OPS_GLOBAL = 25, 22  # SURVEY 8d accounting convention (int32 ops per cell)
MODE_GLOBAL, MODE_SEMIGLOBAL, MODE_LOCAL = 1, 2, 3


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--pairs", type=int, default=1_000_000, help="pairs per GPU")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--configs", default="C2_10k,C3,C4,C5", help="extra configs to report ('' = none)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the results of the last timed step to DIR/<name>.npy (see dump_outputs)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs applies to --impl b200")
    return args


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            d = json.load(f)
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks/throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.tmp = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.proc = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={gpu_index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=self.tmp, stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        if self.proc is None:
            return out
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        self.tmp.flush()
        rows = [r.strip().split(",") for r in open(self.tmp.name) if r.strip()]
        os.unlink(self.tmp.name)
        sm, reasons, mx = [], set(), None
        for r in rows:
            try:
                r = [c.strip() for c in r]
                sm.append(float(r[1]))
                mx = float(r[2])
                for name, col in (("hw_slowdown", 5), ("hw_thermal_slowdown", 6),
                                  ("sw_thermal_slowdown", 7), ("sw_power_cap", 8)):
                    if r[col].lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                continue
        if sm:
            busy = sorted(sm)[len(sm) // 2:]  # upper half: samples taken under load
            out["sm_mhz"] = float(np.median(busy))
            out["sm_max_mhz"] = mx
            out["samples"] = len(sm)
        out["reasons"] = sorted(reasons)
        return out


def oracle_scoring(orc):
    s, _ = orc.make_scoring(SCORING["gap_open"], SCORING["gap_extend"], SCORING["match"], SCORING["mismatch"])
    return s


def cpu_sample(orc, threads: int, target_s: float):
    """Time the oracle on a bounded sample of the workload; returns (gcups, n_pairs, seconds)."""
    from rust_bio_b200 import synth
    s = oracle_scoring(orc)
    probe = synth.uniform_pairs(synth.BASES["C2"], 0, 64 * threads, M, N_LEN)
    _, _, _, t = orc.align_batch("local", s, *probe, threads=threads, want_ops=False)
    rate = 64 * threads / max(t, 1e-6)
    n = int(max(threads * 64, min(400_000, rate * target_s)))
    batch = synth.uniform_pairs(synth.BASES["C2"], 0, n, M, N_LEN)
    _, _, _, t = orc.align_batch("local", s, *batch, threads=threads, want_ops=False)
    return n * M * N_LEN / t / 1e9, n, t


def run_reference(args):
    """The reference arm: rust-bio's CPU path (oracle port) on all host threads, bounded sample per step."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import oracle as orc
    threads = orc.hardware_threads()
    vals, sample = [], None
    for it in range(args.warmup + args.steps):
        g, n, t = cpu_sample(orc, threads, target_s=4.0 if it >= args.warmup else 1.0)
        if it >= args.warmup:
            vals.append((g, n, t))
            sample = n
    cells = sum(v[1] for v in vals) * M * N_LEN
    secs = sum(v[2] for v in vals)
    value = cells / secs / 1e9
    g1, n1, t1 = cpu_sample(orc, 1, target_s=2.0)
    line = {
        "impl": "reference", "metric": "GCUPS", "value": round(value, 4), "unit": "GCUPS",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": round(secs / args.steps * 1e3, 3), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "int32", "data": "synthetic",
        "config": {"workload": WORKLOAD, "note": "rust-bio cannot be built here (no rustc); this is the C++ "
                   "restatement of rust-bio 4.0.1 pinned to the reference's known-answer vectors"},
        "cpu_baseline": {"value": round(value, 4), "unit": "GCUPS", "cores": threads, "kind": "port",
                         "sample": f"{sample} pairs of {M}x{N_LEN} per step, {threads} pinned threads",
                         "single_thread_value": round(g1, 4),
                         "parallel_efficiency": round(value / (threads * g1), 3),
                         "each_step": [round(v[0], 3) for v in vals]},
        "e2e": {"value": round(value, 4), "unit": "GCUPS", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------ helpers
def pinned_results(torch, Results, P, ops_cap):
    out_t = {"score": torch.empty(P, dtype=torch.int32).pin_memory(),
             "xstart": torch.empty(P, dtype=torch.int32).pin_memory(),
             "xend": torch.empty(P, dtype=torch.int32).pin_memory(),
             "ystart": torch.empty(P, dtype=torch.int32).pin_memory(),
             "yend": torch.empty(P, dtype=torch.int32).pin_memory(),
             "ops_off": torch.empty(P + 1, dtype=torch.int64).pin_memory(),
             "ops": torch.empty(ops_cap, dtype=torch.uint8).pin_memory(),
             "clip_len": torch.empty(4 * P, dtype=torch.int32).pin_memory()}
    views = {"score": out_t["score"].numpy(), "xstart": out_t["xstart"].numpy().view(np.uint32),
             "xend": out_t["xend"].numpy().view(np.uint32), "ystart": out_t["ystart"].numpy().view(np.uint32),
             "yend": out_t["yend"].numpy().view(np.uint32), "ops_off": out_t["ops_off"].numpy().view(np.uint64),
             "ops": out_t["ops"].numpy(), "clip_len": out_t["clip_len"].numpy().view(np.uint32)}
    return Results(P, ops_cap, out=views), out_t


DUMP_PAIRS, DUMP_OPS_PAIRS = 1 << 20, 4096  # 6 x 8 MB of per-pair fields + <= 10 MB of ops: < 64 MB in all


def dump_outputs(out_dir, res, n_pairs):
    """Write the results a caller of the timed path receives to out_dir/<name>.npy, so that two builds can be
    compared output for output: score, xstart, xend, ystart, yend of every pair (of a seeded sample of DUMP_PAIRS
    pairs when there are more; pair_index names them) and the operations of a seeded sample of DUMP_OPS_PAIRS pairs
    (ops: one (code, clip length) row per operation, ops_count rows per pair of ops_pair_index).  The fields are
    float64, which holds every int32 / uint32 exactly; op codes and clip lengths are small enough for float32."""
    os.makedirs(out_dir, exist_ok=True)
    rng = np.random.default_rng(0)
    idx = np.arange(n_pairs) if n_pairs <= DUMP_PAIRS else np.sort(rng.choice(n_pairs, DUMP_PAIRS, replace=False))
    arrays = {"pair_index": idx.astype(np.float64)}
    for f in ("score", "xstart", "xend", "ystart", "yend"):
        arrays[f] = getattr(res, f)[idx].astype(np.float64)
    oidx = np.sort(rng.choice(n_pairs, min(n_pairs, DUMP_OPS_PAIRS), replace=False))
    ops = [res.ops_of(int(p)) for p in oidx]
    arrays["ops_pair_index"] = oidx.astype(np.float64)
    arrays["ops_count"] = np.array([len(o) for o in ops], dtype=np.float64)
    arrays["ops"] = np.array([op for o in ops for op in o], dtype=np.float32).reshape(-1, 2)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def check_sample(orc, mode_name, oscoring, batch, idx, res, threads):
    """Oracle parity of the pairs `idx` of a fetched batch: every Alignment field and the ops."""
    blob, xo, xl, yo, yl = batch
    sub = (blob, xo[idx], xl[idx], yo[idx], yl[idx])
    ref, ops, off, _ = orc.align_batch(mode_name, oscoring, *sub, threads=threads)
    bad = 0
    for k, p in enumerate(idx):
        p = int(p)
        same = all(int(getattr(res, f)[p]) == int(ref[f][k]) for f in ("score", "xstart", "xend", "ystart", "yend"))
        want = [(int(v) & 7, int(v) >> 3) for v in ops[int(off[k]):int(off[k]) + int(ref["n_ops"][k])]]
        if not same or res.ops_of(p) != want:
            bad += 1
    return {"pairs_checked": int(len(idx)), "mismatches": bad, "ok": bad == 0,
            "what": "score, xstart, xend, ystart, yend and the operation vector vs the oracle"}


def main():
    args = parse_args()
    if args.impl == "reference":
        run_reference(args)
        return
    import torch
    import torch.distributed as dist
    from rust_bio_b200 import scores, synth
    from rust_bio_b200._lib import CScoring, MIN_SCORE, load
    from rust_bio_b200.engine import Engine, Results

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the product has no CPU path")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    P = args.pairs
    cells_rank = P * M * N_LEN
    steps, warm = args.steps, max(args.warmup, 0)

    # ---- synthetic inputs of the named shape, in PINNED host memory (this rank's shard of the pair list)
    blob, x_off, x_len, y_off, y_len = synth.uniform_pairs(synth.BASES["C2"], rank * P, P, M, N_LEN)

    def pin(a):
        t = torch.from_numpy(a).pin_memory()
        return t, t.numpy()

    keep = [pin(a) for a in (blob, x_off, x_len, y_off, y_len)]
    batch = tuple(k[1] for k in keep)
    ops_cap = 64 * P  # local alignments of random DNA are ~15 ops; capacity is checked by the ABI
    results, keep_out = pinned_results(torch, Results, P, ops_cap)

    eng = Engine(local)
    # a real (non-legacy-default) torch stream: the engine launches on it, torch.cuda.Event times it
    stream = torch.cuda.Stream()
    side = torch.cuda.Stream()  # the all-gather of step k runs here, under the kernels of step k+1
    torch.cuda.set_stream(stream)
    assert stream.cuda_stream != 0
    eng.set_stream(stream.cuda_stream)
    cs = CScoring(SCORING["gap_open"], SCORING["gap_extend"], MIN_SCORE, MIN_SCORE, MIN_SCORE, MIN_SCORE,
                  SCORING["match"], SCORING["mismatch"], 1, None, None, 0)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms: float) -> float:
        if world == 1:
            return ms
        t = torch.tensor([ms], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ---- device-resident arm: stage once, then time K passes of the hot path
    eng.stage(MODE_LOCAL, cs, batch)
    # N > 1: the one exchange of the path is the all-gather that reassembles the per-pair results on every rank.
    # Segment capacity is fixed ONCE, before the timed region (largest segment over the ranks + 12 %); inside the
    # timed region nothing is read back: b2a_batch_compact_fixed writes the segment (header on the device), the
    # all-gather of step k runs on `side` while step k+1's kernels run on `stream` (two segment buffers).
    seg = 0
    bufs = []
    gathered = {"bytes": 0}
    if world > 1:
        eng.run()
        size = torch.tensor([eng.compact_bytes()], dtype=torch.int64, device="cuda")
        dist.all_reduce(size, op=dist.ReduceOp.MAX)
        seg = (int(int(size.item()) * 1.12) + (1 << 20) - 1) >> 20 << 20
        for _ in range(2):
            bufs.append({"local": torch.empty(seg, dtype=torch.uint8, device="cuda"),
                         "all": torch.empty(world * seg, dtype=torch.uint8, device="cuda"),
                         "ready": torch.cuda.Event(), "done": torch.cuda.Event()})
            bufs[-1]["done"].record(side)
        gathered["bytes"] = world * seg
    step_no = {"k": 0}

    def step_resident():
        eng.run()
        if world > 1:
            b = bufs[step_no["k"] % 2]
            step_no["k"] += 1
            stream.wait_event(b["done"])       # the gather that last used this buffer pair has finished
            eng.compact_fixed(b["local"].data_ptr(), seg)
            b["ready"].record(stream)
            with torch.cuda.stream(side):
                side.wait_event(b["ready"])
                dist.all_gather_into_tensor(b["all"], b["local"])
                b["done"].record(side)

    def join_exchange():
        if world > 1:
            stream.wait_stream(side)

    for _ in range(warm):
        step_resident()
    join_exchange()
    barrier()
    sampler = ClockSampler(local) if rank == 0 else None
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record(stream)
    for _ in range(steps):
        step_resident()
    join_exchange()  # the last step's gather is inside the timed region
    ev1.record(stream)
    barrier()
    ms_total = ev0.elapsed_time(ev1)
    clocks = sampler.stop() if sampler else None
    ms_step = max_over_ranks(ms_total / steps)
    ms_ranks = [round(ms_total / steps, 4)]
    if world > 1:  # every rank's own step time: the slowest GPU sets `value`
        t = torch.zeros(world, dtype=torch.float64, device="cuda")
        t[rank] = ms_total / steps
        dist.all_reduce(t)
        ms_ranks = [round(float(v), 4) for v in t.tolist()]
    if args.dump_outputs and world == 1:
        eng.fetch(results)  # the last timed step's results; the passes below run the batch again
        dump_outputs(args.dump_outputs, results, P)
    else:
        eng.fetch(None)
    st = eng.stats
    launches_step = int(st.kernel_launches) + (1 if world > 1 else 0)  # + the segment-header kernel
    # kernel-level numbers over instrumented passes (engine CUDA events on the same stream)
    fills, walks, packs = [], [], []
    for _ in range(max(3, steps)):
        eng.run()
        eng.fetch(None)
        fills.append(eng.stats.fill_ms)
        walks.append(eng.stats.walk_ms)
        packs.append(eng.stats.pack_ms)
    fill_ms = float(np.mean(fills))
    value = world * cells_rank / (ms_step * 1e-3) / 1e9
    G, R = int(eng.stats.fill_lanes_per_pair), int(eng.stats.fill_rows_per_lane)

    # ---- N > 1: decode what was gathered and compare a sample of EVERY rank's share with the oracle
    verify = None
    if world > 1:
        b = bufs[(step_no["k"] - 1) % 2]
        torch.cuda.synchronize()
        if rank == 0:
            from oracle import oracle as orc
            total_pairs = world * P
            allres, keep_all = pinned_results(torch, Results, total_pairs, 64 * total_pairs)
            n_got, _ = eng.gathered_fetch(b["all"].data_ptr(), seg, world, allres)
            if args.dump_outputs:
                dump_outputs(args.dump_outputs, allres, total_pairs)
            rng = np.random.default_rng(7)
            bad, checked = 0, 0
            for r in range(world):
                # the first 128 pairs of the rank's shard and a random window of 128 (only those are generated)
                w0 = int(rng.integers(128, max(129, P - 128)))
                idx = np.concatenate([np.arange(min(128, P)), np.arange(w0, min(P, w0 + 128))])
                parts = [synth.uniform_pairs(synth.BASES["C2"], r * P + int(a), int(b - a), M, N_LEN)
                         for a, b in ((0, min(128, P)), (w0, min(P, w0 + 128)))]
                stride = len(parts[0][0]) // max(1, len(parts[0][2]))
                blob_s = np.concatenate([q[0] for q in parts])
                off0 = np.uint64(len(parts[0][0]))
                sub = (blob_s, np.concatenate([parts[0][1], parts[1][1] + off0]), np.concatenate([q[2] for q in parts]),
                       np.concatenate([parts[0][3], parts[1][3] + off0]), np.concatenate([q[4] for q in parts]))
                ref, ops, off, _ = orc.align_batch("local", oracle_scoring(orc), *sub, threads=min(16, orc.hardware_threads()))
                for k, p in enumerate(idx):
                    gp = r * P + int(p)
                    same = all(int(getattr(allres, f)[gp]) == int(ref[f][k]) for f in ("score", "xstart", "xend", "ystart", "yend"))
                    want = [(int(v) & 7, int(v) >> 3) for v in ops[int(off[k]):int(off[k]) + int(ref["n_ops"][k])]]
                    bad += 0 if (same and allres.ops_of(gp) == want) else 1
                    checked += 1
            verify = {"pairs_gathered": int(n_got), "pairs_expected": total_pairs, "pairs_checked": checked,
                      "mismatches": bad, "ok": bad == 0 and int(n_got) == total_pairs,
                      "what": "rank 0 decoded the all-gathered segments (b2a_gathered_fetch) and compared 256 pairs of every rank's shard with the oracle: all fields + ops"}
            del allres, keep_all

    # ---- end-to-end arm: pinned host buffers in, host results out, copies inside the timed region
    e2e_each = []
    if world == 1:
        for _ in range(max(warm, 3)):
            eng.align_batch(MODE_LOCAL, cs, batch, results=results)
        barrier()
        t0 = time.perf_counter()
        for _ in range(steps):
            t1 = time.perf_counter()
            eng.align_batch(MODE_LOCAL, cs, batch, results=results)  # returns with the results in host memory
            e2e_each.append(round((time.perf_counter() - t1) * 1e3, 2))
        torch.cuda.synchronize()
        e2e_ms = (time.perf_counter() - t0) / steps * 1e3
        h2d, d2h = int(eng.stats.h2d_bytes), int(eng.stats.d2h_bytes)
        e2e_note = "b2a_align_batch: pinned host inputs -> host results (chunked H2D / kernels / D2H pipeline inside)"
    else:
        from rust_bio_b200.dist import ShardedAligner
        total_pairs = world * P
        allres = None
        if rank == 0:
            allres, keep_all = pinned_results(torch, Results, total_pairs, 64 * total_pairs)
        sharded = ShardedAligner(local, chunks=3)
        d2h = 0

        def step_e2e():
            # the multi-process public call: pinned host shard in -> the whole batch in rank 0's host arrays
            sharded.align(MODE_LOCAL, cs, batch, allres)
        for _ in range(max(warm, 3)):
            step_e2e()
        barrier()
        t0 = time.perf_counter()
        for _ in range(steps):
            t1 = time.perf_counter()
            step_e2e()
            e2e_each.append(round((time.perf_counter() - t1) * 1e3, 2))
        torch.cuda.synchronize()
        e2e_ms = (time.perf_counter() - t0) / steps * 1e3
        h2d = 0
        for e in sharded.engs:
            e.fetch(None)
            h2d += int(e.stats.h2d_bytes)
        d2h = int(getattr(sharded, "d2h", 0))
        if rank == 0 and allres is not None:  # the e2e arm's own output, checked like the resident arm's
            from oracle import oracle as orc2
            idx = np.arange(0, P, max(1, P // 128))[:128]
            sub = (batch[0], batch[1][idx], batch[2][idx], batch[3][idx], batch[4][idx])
            ref, ops, off, _ = orc2.align_batch("local", oracle_scoring(orc2), *sub, threads=min(16, orc2.hardware_threads()))
            bad = 0
            for kk, p in enumerate(idx):
                same = all(int(getattr(allres, f)[int(p)]) == int(ref[f][kk]) for f in ("score", "xstart", "xend", "ystart", "yend"))
                want = [(int(v) & 7, int(v) >> 3) for v in ops[int(off[kk]):int(off[kk]) + int(ref["n_ops"][kk])]]
                bad += 0 if (same and allres.ops_of(int(p)) == want) else 1
            if verify is not None:
                verify["e2e_pairs_checked"] = int(len(idx))
                verify["e2e_mismatches"] = bad
                verify["ok"] = bool(verify["ok"] and bad == 0)
        sharded.close()
        e2e_note = ("rust_bio_b200.dist.ShardedAligner.align: per rank three pieces (own engine + stream each: the H2D of piece "
                    "c+1 under the kernels of piece c) -> fixed-capacity segments -> one NCCL all-gather -> rank 0 decodes all "
                    "%d pairs into pinned host arrays (b2a_gathered_fetch); h2d is per rank, d2h is rank 0's" % total_pairs)
    e2e_ms = max_over_ranks(e2e_ms)
    e2e_value = world * cells_rank / (e2e_ms * 1e-3) / 1e9
    tb_bytes = int(eng.stats.traceback_bytes)

    # ---- the other BASELINE configs on this GPU (device-timed per iteration, L2 flushed between iterations)
    cfg_lines = []
    L = load()
    fa, fb, fc = C.c_float(), C.c_float(), C.c_float()
    L.b2a_util_int32_peak(local, C.byref(fa), C.byref(fb), C.byref(fc))
    p_int = max(fa.value, fb.value, fc.value)  # tera lane-ops/s
    want_cfgs = [c for c in args.configs.split(",") if c]
    if want_cfgs:
        from oracle import oracle as orc
        othreads = min(32, orc.hardware_threads())
        flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")

        def timed_runs(fn, reps):
            out = []
            for _ in range(reps):
                flush.zero_()
                a, b2 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record(stream)
                fn()
                b2.record(stream)
                b2.synchronize()
                out.append(a.elapsed_time(b2))
            return out

        def full_config(name, desc, mode, mode_name, cscoring, oscoring, cbatch, ops_per_cell, sample_idx, scaling):
            res = Results(len(cbatch[2]), int(Engine.default_ops_capacity(cbatch)))
            eng.stage(mode, cscoring, cbatch)
            for _ in range(3):
                eng.run()
            ms = timed_runs(eng.run, max(3, min(steps, 10)))
            eng.fetch(res)
            s2 = eng.stats
            cells = int(s2.cells)
            step_ms = max_over_ranks(float(np.median(ms)))
            g = world * cells / (step_ms * 1e-3) / 1e9 if scaling == "weak" else None
            line = {"name": name, "workload": desc, "pairs_this_gpu": int(len(cbatch[2])), "scaling": scaling,
                    "ms_per_step": round(step_ms, 4), "ms_each": [round(v, 4) for v in ms],
                    "kernel_ms": {"pack": round(s2.pack_ms, 4), "fill": round(s2.fill_ms, 4), "walk_and_compact": round(s2.walk_ms, 4)},
                    "fill_shape": {"lanes_per_pair": int(s2.fill_lanes_per_pair), "rows_per_lane": int(s2.fill_rows_per_lane)},
                    "waves": int(s2.waves), "cells_this_gpu": cells, "ops_per_cell": ops_per_cell,
                    "gcups_this_gpu": round(cells / (step_ms * 1e-3) / 1e9, 2),
                    "fill_gcups_this_gpu": round(cells / (s2.fill_ms * 1e-3) / 1e9, 2),
                    "int32_frac_step": round(cells / (step_ms * 1e-3) / 1e9 * ops_per_cell / 1e3 / p_int, 4),
                    "int32_frac_fill": round(cells / (s2.fill_ms * 1e-3) / 1e9 * ops_per_cell / 1e3 / p_int, 4),
                    "l2": "flushed between timed iterations (256 MB write)"}
            if g is not None:
                line["gcups"] = round(g, 2)
            if rank == 0:
                line["parity_sample"] = check_sample(orc, mode_name, oscoring, cbatch, sample_idx, res, othreads)
            return line

        for cname in want_cfgs:
            if cname == "C2_10k":
                n10 = 10_000
                cb = synth.uniform_pairs(synth.BASES["C2"], rank * n10, n10, M, N_LEN)
                idx = np.arange(0, n10, 20)
                ln = full_config("C2_10k", "north_star target: 10k pairs of 150x150 random DNA, local affine (1,-1,-5,-1), per GPU",
                                 MODE_LOCAL, "local", cs, oracle_scoring(orc), cb, OPS_LOCAL, idx, "weak")
                ln["target"] = ">= 0.40 of the int32-ALU roofline (BASELINE north_star)"
                cfg_lines.append(ln)
            elif cname == "C3":
                tot = 100_000
                lo, hi = rank * tot // world, (rank + 1) * tot // world
                cb = synth.uniform_pairs(synth.BASES["C3"], lo, hi - lo, 1000, 1000)
                idx = np.arange(0, hi - lo, max(1, (hi - lo) // 64))[:64]
                ln = full_config("C3", "100k pairs of 1000x1000 random DNA, global affine, split over the ranks (strong scaling)",
                                 MODE_GLOBAL, "global", cs, oracle_scoring(orc), cb, OPS_GLOBAL, idx, "strong")
                ln["gcups"] = round(tot * 1e6 / (ln["ms_per_step"] * 1e-3) / 1e9, 2)  # whole job: 100k x 10^6 cells / slowest rank
                cfg_lines.append(ln)
            elif cname == "C5":
                n5 = 1250
                cb = synth.uniform_pairs(synth.BASES["C5"], rank * n5, n5, 10000, 10000, alphabet=synth.PROTEIN)
                table = np.ascontiguousarray(scores.matrix_table256("blosum62"), dtype=np.int32)
                alpha = np.frombuffer(bytes(range(65, 91)) + b"*", dtype=np.uint8).copy()
                c5 = CScoring(-10, -1, MIN_SCORE, MIN_SCORE, MIN_SCORE, MIN_SCORE, 0, 0, 0,
                              table.ctypes.data_as(C.c_void_p), alpha.ctypes.data_as(C.c_void_p), len(alpha))
                o5, keep5 = orc.make_scoring(-10, -1, 0, 0, table)
                ln = full_config("C5", "10k pairs of 10000x10000 protein, BLOSUM62 go -10 ge -1, local: the per-GPU share at 8 GPUs (1,250 pairs)",
                                 MODE_LOCAL, "local", c5, o5, cb, OPS_LOCAL, np.array([0, n5 - 1]), "weak")
                cfg_lines.append(ln)
            elif cname == "C4":
                n4 = 25_000
                cb = synth.mutated_window_pairs(synth.BASES["C4"], rank * n4, n4, 500, 10000)
                c4 = CScoring(-5, -1, MIN_SCORE, MIN_SCORE, MIN_SCORE, MIN_SCORE, 1, -1, 1, None, None, 0)
                res = Results(n4, int(Engine.default_ops_capacity(cb)))
                for _ in range(2):
                    eng.align_batch_banded(MODE_SEMIGLOBAL, c4, 32, 32, cb, results=res)
                ks = []
                for _ in range(3):
                    flush.zero_()
                    eng.align_batch_banded(MODE_SEMIGLOBAL, c4, 32, 32, cb, results=res)
                    s4 = eng.stats
                    ks.append((s4.band_ms + s4.fill_ms + s4.walk_ms, s4.band_ms, s4.fill_ms, s4.walk_ms))
                ks.sort()
                kms, band_ms, k3_ms, walk_ms = ks[len(ks) // 2]
                kms = max_over_ranks(float(kms))
                cells = int(eng.stats.cells)
                ln = {"name": "C4", "workload": "200k pairs of 500x10000 (x = mutated window of y), banded::Aligner::semiglobal k=32 w=32: "
                                                "the per-GPU share at 8 GPUs (25,000 pairs); named generator synth.mutated_window_pairs",
                      "pairs_this_gpu": n4, "scaling": "weak", "ms_per_step": round(kms, 3),
                      "kernel_ms": {"band_K4": round(band_ms, 3), "fill_walk_K3": round(k3_ms, 3), "compact": round(walk_ms, 3)},
                      "k3_path": {"strip_wavefront_pairs": int(eng.banded_strip_pairs()), "column_loop_pairs": n4 - int(eng.banded_strip_pairs()),
                                  "what": "K3s = strip-wavefront fill (8 lanes x 16 rows, four pairs to a warp, packed cell + band mask, 4-bit "
                                          "traceback) + finish pass + walk (one pair per thread); the pairs K4 does not mark (band reaching "
                                          "column n) run the K3 column loops on a side stream"},
                      "cells_this_gpu": cells, "cells_are": "Band::num_cells (banded.rs:1374-1380)", "ops_per_cell": OPS_GLOBAL,
                      "gcups_this_gpu": round(cells / (kms * 1e-3) / 1e9, 2), "gcups": round(world * cells / (kms * 1e-3) / 1e9, 2),
                      "mn_equivalent_gcups_this_gpu": round(n4 * 500 * 10000 / (kms * 1e-3) / 1e9, 1),
                      "pairs_per_s_this_gpu": round(n4 / (kms * 1e-3)),
                      "int32_frac_step": round(cells / (kms * 1e-3) / 1e9 * OPS_GLOBAL / 1e3 / p_int, 4),
                      "l2": "flushed between timed iterations (256 MB write)",
                      "timing": "engine CUDA events around K4, K3 and the ops compaction (host copies of the one-shot banded call excluded)"}
                if rank == 0:
                    idx = np.arange(0, n4, n4 // 100)[:100]
                    sub = (cb[0], cb[1][idx], cb[2][idx], cb[3][idx], cb[4][idx])
                    so, _ = orc.make_scoring(-5, -1, 1, -1, has_match_scores=1)
                    ref, rops, roff, _, _ = orc.banded_align_batch("semiglobal", so, 32, 32, *sub, threads=othreads)
                    bad = 0
                    for k, p in enumerate(idx):
                        p = int(p)
                        same = all(int(getattr(res, f)[p]) == int(ref[f][k]) for f in ("score", "xstart", "xend", "ystart", "yend"))
                        want = [(int(v) & 7, int(v) >> 3) for v in rops[int(roff[k]):int(roff[k]) + int(ref["n_ops"][k])]]
                        bad += 0 if (same and res.ops_of(p) == want) else 1
                    ln["parity_sample"] = {"pairs_checked": int(len(idx)), "mismatches": bad, "ok": bad == 0,
                                           "what": "score, xstart, xend, ystart, yend and the operation vector vs the banded oracle"}
                cfg_lines.append(ln)
        del flush

    if rank == 0:
        hbm_peak, peak_src = measured_peaks()
        fill_gcups = cells_rank / (fill_ms * 1e-3) / 1e9
        # SURVEY 8d algorithmic bytes of C2: sequences in (m + n), the 40-byte result record and <= m + n + 4 op
        # bytes out; the 4-bit traceback "fits on chip" in that accounting and is not counted
        algo_pair = (M + N_LEN) + 40 + (M + N_LEN + 4)
        algo_bytes = P * algo_pair
        traffic = None
        tsrc = None
        tpath = os.path.join(ROOT, "profiles", "fill_traffic.json")
        if os.path.exists(tpath):
            with open(tpath) as f:
                tj = json.load(f)
            if tuple(tj.get("shape", (1, 16))) == (G, R):
                traffic = int(tj["dram_bytes_per_pair"] * P)  # ncu dram read+write per pair x pairs of this launch
                tsrc = tj.get("source", "profiles/fill_traffic.json (ncu --set full capture, scaled per pair)")
        sm_max = (clocks or {}).get("sm_max_mhz") or 1965.0
        nominal = 148 * 128 * sm_max * 1e6 / 1e12
        k_all = float(np.mean(packs)) + fill_ms + float(np.mean(walks))
        roof = {"bound": "int32_alu", "kernel": f"fill_kernel<G={G},R={R},local> (K1: {100 * fill_ms / k_all:.0f}% of the step's kernel time)",
                "achieved": round(fill_gcups * OPS_LOCAL / 1e3, 3), "peak": round(p_int, 3), "unit": "tera int32 lane-ops/s",
                "frac": round(fill_gcups * OPS_LOCAL / 1e3 / p_int, 4),
                "frac_whole_step": round(value / world * OPS_LOCAL / 1e3 / p_int, 4),
                "ops_per_cell": OPS_LOCAL, "kernel_gcups": round(fill_gcups, 2), "kernel_ms": round(fill_ms, 4),
                "peak_source": "measured in this run by b2a_util_int32_peak: independent add / min-max / add+max register chains on all "
                               "SMs (tera lane-ops/s: add %.2f, minmax %.2f, mixed %.2f); the convention counts 25 plain ops per cell, the "
                               "kernel issues ~19 fused ones (DPX add-max, 3-way max)" % (fa.value, fb.value, fc.value),
                "peak_nominal": round(nominal, 2), "frac_of_nominal": round(fill_gcups * OPS_LOCAL / 1e3 / nominal, 4),
                "peak_nominal_source": "148 SMs x 128 int32 lanes x max SM clock",
                "traffic": traffic, "traffic_source": tsrc,
                "hbm": {"bound": "hbm", "achieved": round(algo_bytes / (fill_ms * 1e-3) / 1e9, 2), "peak": hbm_peak, "unit": "GB/s",
                        "frac": round(algo_bytes / (fill_ms * 1e-3) / 1e9 / hbm_peak, 5), "peak_source": peak_src,
                        "algorithmic_bytes_per_launch": int(algo_bytes),
                        "algorithmic_bytes_per_pair": algo_pair,
                        "traffic": traffic,
                        "traffic_frac_of_peak": round(traffic / (fill_ms * 1e-3) / 1e9 / hbm_peak, 4) if traffic else None,
                        "note": "SURVEY 8d bytes: (m+n) in + 40 B record + (m+n+4) op bytes out, traceback on chip; the kernel "
                                "itself streams its 4-bit traceback and strip-boundary rows through HBM (traffic)"}}
        cpu = None
        if world == 1 and not args.no_cpu_baseline:
            from oracle import oracle as orc
            threads = orc.hardware_threads()
            g, n, t = cpu_sample(orc, threads, target_s=12.0)
            g1, n1, t1 = cpu_sample(orc, 1, target_s=4.0)
            cpu = {"value": round(g, 4), "unit": "GCUPS", "cores": threads, "kind": "port",
                   "sample": f"{n} pairs of {M}x{N_LEN} ({t:.1f} s, {threads} pinned threads); 1 thread: {g1:.4f} GCUPS on {n1} pairs",
                   "single_thread_value": round(g1, 4), "parallel_efficiency": round(g / (threads * g1), 3)}
        line = {
            "metric": "GCUPS", "value": round(value, 2), "unit": "GCUPS", "n_gpus": world, "steps": steps,
            "warmup": warm, "ms_per_step": round(ms_step, 4), "ms_per_step_each_rank": ms_ranks,
            "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "int32", "data": "synthetic",
            "config": {"workload": WORKLOAD, "pairs_per_gpu": P, "m": M, "n": N_LEN,
                       "fill_shape": {"lanes_per_pair": G, "rows_per_lane": R},
                       "l2": "inputs larger than L2: 320 MB staged sequences + ~12 GB traceback stream per step (126 MB L2)",
                       "parallelism": (f"pair list sharded over {world} GPU(s); per step one NCCL all-gather of fixed-capacity result "
                                       f"segments ({gathered['bytes']} B received per rank) on a side stream, overlapping the next "
                                       f"step's kernels; no size agreement, no host sync in the timed region")
                       if world > 1 else "single GPU"},
            "e2e": {"value": round(e2e_value, 2), "unit": "GCUPS", "ms_per_step": round(e2e_ms, 3),
                    "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "ms_each_step": e2e_each,
                    "ms_median_step": float(np.median(e2e_each)),
                    "value_at_median_step": round(world * cells_rank / (float(np.median(e2e_each)) * 1e-3) / 1e9, 2),
                    "path": e2e_note},
            "gpu_launches": launches_step * steps,
            "kernel_ms": {"pack": round(float(np.mean(packs)), 4), "fill": round(fill_ms, 4),
                          "walk_and_compact": round(float(np.mean(walks)), 4)},
            "traceback_bytes_per_step": tb_bytes,
            "roofline": roof, "clocks": clocks,
        }
        if cfg_lines:
            line["configs"] = cfg_lines
        if verify:
            line["verify"] = verify
        if cpu:
            line["cpu_baseline"] = cpu
        print(json.dumps(line), flush=True)
    eng.close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()

#!/usr/bin/env python
"""bench.py -- headline benchmark of the B200 pairwise string-similarity hot path.

    python bench.py --gpus N --steps K --warmup W [--impl reference] [--dump-outputs DIR]

Workload (BASELINE.json configs[1]): char-trigram TF-IDF top-10, company-names self-match,
n = 100 000 -- on the reference's own data/company_names.json (shipped as a test fixture under
tests/golden/data/; seeded synthetic names calibrated to it, polyfuzz_b200/synth.py, when the fixture is
absent -- the `data` key says which).  One step = one pass of the whole hot path:
vectorise (K1) -> inverted index -> sparse cosine + top-10 (K2) [-> all-gather + merge for N > 1].

The same JSON line carries sub-records for the other BASELINE configs, each device-timed with its own clock
record and roofline: `c3` (Levenshtein / fuzz.ratio all-pairs on movie_titles, N = 1), `c4` (dense cosine
100k x 100k x 768 bf16 top-10, N = 1) and `c5` (TF-IDF top-10 on 1M x 1M uniform strings, to_list row-sharded
over the N GPUs: strong scaling).

N > 1 (torchrun, one rank per GPU, NCCL): weak scaling.  The to_list grows to N x 100 000 names and is
row-sharded (rank r owns block r); the from_list stays the first block (100 000 names), scored
against all shards with the global diagonal excluded -- i.e. one from-row-block of the N*100k
self-match.  Per-GPU work is fixed; one all-reduce (df) + one all-gather (top-k) per step.

--steps sets the number of timed steps of every leg and sub-record.  --dump-outputs DIR writes what the last timed step
of the headline leg returned (top-10 indices and scores per from-row) as DIR/<name>.npy in float64, so that the
outputs of two builds can be compared on identical inputs.

Prints ONE JSON line on rank 0 (see the repository README / DESIGN.md for the keys).
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "scored string pairs/sec (TF-IDF char-trigram top-10, top-k index bit-exact vs CPU ref)"
UNIT = "pairs/s"
N_PER_SHARD = 100_000
TOP_N = 10


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--n", type=int, default=N_PER_SHARD, help="rows per shard (default 100000)")
    ap.add_argument("--cpu-sample-rows", type=int, default=4096)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--skip", default="", help="comma list of sub-records to skip: c3,c4,c5,e2e")
    ap.add_argument("--c5-n", type=int, default=1_000_000, help="rows per list of the c5 sub-record")
    ap.add_argument("--synthetic", action="store_true", help="force the synthetic stand-in data")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's top-k indices / scores as DIR/<name>.npy")
    return ap.parse_args()


def config_dict(n, n_gpus, data_kind, extra=None):
    cfg = {"workload": "TF-IDF char-trigram top-10 self-match, company names (BASELINE configs[1]); data: " + data_kind,
           "n_from": n, "n_to": n * n_gpus, "top_n": TOP_N, "min_similarity": 0.0, "n_gram_range": [3, 3],
           "parallelism": "to_list row-sharded x%d, all-reduce(df) + all-gather(top-k)" % n_gpus if n_gpus > 1 else "single GPU",
           "l2": "flushed between steps (512 MiB write)"}
    if extra:
        cfg.update(extra)
    return cfg


# ------------------------------------------------------------------------------------------------
# CPU leg: the oracle port of the reference path (sklearn TfidfVectorizer with the restated
# analyzer + C restatement of awesome_cossim_topn + the reference's assembly tail), timed on a
# bounded sample and extrapolated to the whole job.
# ------------------------------------------------------------------------------------------------
def cpu_reference_step(names, sample_rows, threads):
    from oracle import native, tfidf
    from oracle.assemble import assemble
    n = len(names)
    t0 = time.perf_counter()
    a, _, _ = tfidf.fit_transform_sklearn(names)                 # whole list (fit + transform), 1 thread
    t1 = time.perf_counter()
    inv = native.InvertedIndex(a)                                # to_vector.T as awesome_cossim_topn takes it
    t2 = time.perf_counter()
    s = min(sample_rows, n)
    idx, val = native.spdot_topn(a[:s], inv, TOP_N, 0.0, self_match=True, n_threads=threads)
    t3 = time.perf_counter()
    assemble(names[:s], names, idx, val)
    t4 = time.perf_counter()
    t_vec, t_inv, t_cos, t_asm = t1 - t0, t2 - t1, t3 - t2, t4 - t3
    whole = t_vec + t_inv + (t_cos + t_asm) * (n / s)
    pairs = float(n) * n - n
    return {"pairs_per_s": pairs / whole, "t_step_measured_s": t4 - t0, "t_whole_job_extrapolated_s": whole,
            "t_vectorise_s": t_vec, "t_transpose_s": t_inv, "t_cos_sample_s": t_cos, "t_assemble_sample_s": t_asm,
            "sample_rows": s}


def cpu_threads():
    try:
        return len(os.sched_getaffinity(0))
    except AttributeError:
        return os.cpu_count() or 1


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import native
    native.build()
    names, _, _, _ = load_names(args, 0, 1)
    data_kind = data_kind_of(args, args.gpus)
    thr = cpu_threads()
    res = []
    for it in range(args.warmup + args.steps):
        r = cpu_reference_step(names, args.cpu_sample_rows, thr)
        if it >= args.warmup:
            res.append(r)
    v = float(np.mean([r["pairs_per_s"] for r in res]))
    ms = float(np.mean([r["t_step_measured_s"] for r in res])) * 1e3
    sample = ("per step: scikit-learn TfidfVectorizer (reference analyzer restated) on all %d names, 1 thread; "
              "C restatement of awesome_cossim_topn top-10 + reference assembly on the first %d from-rows x %d to-rows, "
              "%d OpenMP threads; value = n(n-1) / (t_vec + t_transpose + (t_cos + t_asm) * n / sample)"
              % (args.n, res[0]["sample_rows"], args.n, thr))
    line = {"impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f64", "data": data_kind, "config": config_dict(args.n, args.gpus, data_kind),
            "reference_block": "block 0 x block 0 (100k x 100k; CPU throughput is per pair)",
            "cpu_baseline": {"value": v, "unit": UNIT, "cores": thr, "kind": "port", "sample": sample,
                             "detail": {k: float(np.mean([r[k] for r in res])) for k in res[0] if k != "sample_rows"}},
            "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------
class ClockSampler:
    """SM clocks / throttle reasons DURING the timed region (B200_PROFILING.md).  Sampled in-process through NVML
    (nvidia_ml_py) every 50 ms: an external `nvidia-smi -lms` loop takes the driver lock for milliseconds per query and
    showed up as +4 ms outliers in 14 ms steps.  Falls back to nvidia-smi if NVML is unavailable."""
    REASONS = {"hw_slowdown": 0x8, "sw_power_cap": 0x4, "sw_thermal_slowdown": 0x20, "hw_thermal_slowdown": 0x40}

    def __init__(self, gpu_index, recording=True):
        # recording=False: the sampler thread (NVML init, first queries) starts during the warm-up and only records once
        # `recording` is set -- starting it right before the timed region cost rank 0 tens of ms in the first timed steps at N = 8
        self.recording = recording
        self.samples, self.maxs, self.reasons = [], [], set()
        self._stop = threading.Event()
        self.thread = None
        self.proc = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(gpu_index)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
            self.thread = threading.Thread(target=self._loop, daemon=True)
            self.thread.start()
        except Exception:
            self.nv = None
            self._start_smi(gpu_index)

    def _loop(self):
        nv = self.nv
        while not self._stop.is_set():
            try:
                mhz = float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                bits = int(nv.nvmlDeviceGetCurrentClocksEventReasons(self.h))
                if self.recording:
                    self.samples.append(mhz)
                    for name, bit in self.REASONS.items():
                        if bits & bit:
                            self.reasons.add(name)
            except Exception:
                pass
            self._stop.wait(0.05)

    def _start_smi(self, gpu_index):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(gpu_index), "--query-gpu=" + q, "--format=csv,noheader,nounits",
                                          "-lms", "250"], stdout=self.f, stderr=subprocess.DEVNULL)
        except OSError:
            self.proc = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0, "source": "nvml" if self.nv else "nvidia-smi"}
        if self.nv is not None:
            self._stop.set()
            self.thread.join(timeout=2)
            if self.samples:
                out.update(sm_mhz=float(np.median(self.samples)), sm_max_mhz=self.max_mhz, reasons=sorted(self.reasons),
                           samples=len(self.samples))
            return out
        if self.proc is None:
            return out
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        self.f.flush(); self.f.seek(0)
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.f.read().splitlines():
            parts = [x.strip() for x in ln.split(",")]
            if len(parts) < 8:
                continue
            try:
                sm.append(float(parts[0])); mx.append(float(parts[1]))
            except ValueError:
                continue
            for nm, val in zip(names, parts[4:8]):
                if val.lower().startswith("active"):
                    reasons.add(nm)
        self.f.close()
        try:
            os.unlink(self.f.name)
        except OSError:
            pass
        if sm:
            out.update(sm_mhz=float(np.median(sm)), sm_max_mhz=float(np.max(mx)), reasons=sorted(reasons), samples=len(sm))
        return out


def hbm_peak():
    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(peaks_path):
        pk = json.load(open(peaks_path))
        return pk, float(pk["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs, burst copy)"
    return {}, 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(out_dir, arrays):
    """Write each (rows x k) array as out_dir/<name>.npy in float64.  Above DUMP_LIMIT_BYTES in all, the same fixed,
    seeded sample of rows is written for every array, and the sampled row numbers as rows.npy."""
    arrays = {k: np.asarray(v, dtype=np.float64) for k, v in arrays.items()}
    n = len(next(iter(arrays.values())))
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_LIMIT_BYTES:
        keep = int(n * (DUMP_LIMIT_BYTES - (1 << 16)) // (total + 8 * n))      # 64 KiB left for the .npy headers
        rows = np.sort(np.random.default_rng(0).choice(n, keep, replace=False))
        arrays = {k: a[rows] for k, a in arrays.items()}
        arrays["rows"] = rows.astype(np.float64)
    os.makedirs(out_dir, exist_ok=True)
    for k, a in arrays.items():
        np.save(os.path.join(out_dir, k + ".npy"), a)


def timed(fn, warmup, steps, sync, flush=None):
    """Device time of fn() per call (CUDA events on the current stream), after `warmup` untimed calls."""
    import torch
    for _ in range(warmup):
        if flush is not None:
            flush.zero_()
        fn()
    sync()
    ms = []
    for _ in range(steps):
        if flush is not None:
            flush.zero_()
        sync()
        e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
        e0.record(); fn(); e1.record()
        sync()
        ms.append(e0.elapsed_time(e1))
    return ms


def data_kind_of(args, world):
    from polyfuzz_b200 import datasets
    kind = "synthetic" if args.synthetic else datasets.load_company_names(args.n, seed=0)[1]
    if world > 1:
        kind += " (block 0) + synthetic (blocks 1..%d)" % (world - 1)
    return kind


def load_names(args, rank, world):
    """Block 0 (the from-list, and rank 0's to-block) is the reference's company_names.json when the fixture is
    present; blocks 1..N-1 of the weak-scaling run are synthetic (the real list has 100 000 names)."""
    from polyfuzz_b200 import datasets, synth
    if args.synthetic:
        from_list, kind = synth.company_names(args.n, seed=0), "synthetic"
    else:
        from_list, kind = datasets.load_company_names(args.n, seed=0)
    shard = from_list if rank == 0 else synth.company_names(args.n, seed=rank)
    full_to = None
    if world > 1:
        full_to = from_list + [s for r in range(1, world) for s in synth.company_names(args.n, seed=r)]
    return from_list, shard, full_to, data_kind_of(args, world)


# ---- sub-records -------------------------------------------------------------------------------------
def sub_c3(dev, local_rank, sync, flush, steps):
    """BASELINE configs[2]: all-pairs edit distance on movie_titles (Netflix 6 172 x IMDB 80 852), per-row best match.
    Device-timed from staged blobs (EditQueries / EditTargets) to the arg-best arrays; integer-ALU roofline against the
    INT32 issue rate measured by pfz_int_alu_probe in this run."""
    import ctypes
    import torch
    from polyfuzz_b200 import _lib, datasets, editdist
    titles, kind = datasets.load_movie_titles()
    frm, to = titles["Netflix"], titles["IMDB"]
    Q = editdist.EditQueries(frm); T = editdist.EditTargets(to)
    fl = Q.lens.astype(np.float64); tl = T.lens.astype(np.float64)
    cells = float(fl.sum()) * float(tl.sum())
    pairs = float(len(frm)) * len(to)
    # 32-bit machine words per pattern (one 32-bit word up to 32 symbols, else 64-bit blocks)
    w32 = np.where(Q.lens <= 32, 1, 2 * np.ceil(Q.lens / 64.0)).astype(np.float64)
    word_steps32 = float(w32.sum()) * float(tl.sum())
    # probe: INT32 lane-ops/s of the ALU pipe (LOP3 + IADD chains)
    scratch = torch.empty(148 * 8 * 256 * 2, dtype=torch.int32, device=dev)
    nops = ctypes.c_int64(0)
    st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    probe_ms = timed(lambda: _lib.call("pfz_int_alu_probe", 4096, ctypes.c_void_p(scratch.data_ptr()), ctypes.byref(nops), st), 2, 5, sync)
    int_peak = float(nops.value) / (min(probe_ms) * 1e-3)
    sampler = ClockSampler(local_rank)
    out = {"workload": "all-pairs edit distance + per-row best, movie_titles Netflix x IMDB (BASELINE configs[2])", "data": kind,
           "n_from": len(frm), "n_to": len(to), "pairs": pairs, "dp_cells": cells,
           "int32_peak_lane_ops_per_s": int_peak, "int32_peak_source": "pfz_int_alu_probe (8 LOP3/IADD chains per thread), this run"}
    # algorithmic INT32 lane-ops per (text symbol x 32-bit pattern word): Myers/Hyyro column = 17 bit-ops, LCS column = 5
    for key, metric, ops in (("levenshtein", "norm_lev", 17.0), ("fuzz_ratio", "ratio", 5.0)):
        res = {}
        def run():
            res["r"] = editdist.edit_argbest_staged(Q, T, metric)
        ms = timed(run, 2, steps, sync, flush)
        t = float(np.median(ms)) * 1e-3
        alg_ops = word_steps32 * ops
        out[key] = {"ms": t * 1e3, "ms_each": [round(x, 3) for x in ms], "pairs_per_s": pairs / t, "gcups": cells / t / 1e9,
                    "word_steps32_per_s": word_steps32 / t,
                    "roofline": {"bound": "int-alu", "achieved": alg_ops / t, "peak": int_peak, "unit": "INT32 lane-ops/s",
                                 "frac": alg_ops / t / int_peak, "algorithmic_ops_per_word_step": ops}}
    out["ms"] = out["levenshtein"]["ms"]
    out["value"] = out["levenshtein"]["pairs_per_s"]; out["unit"] = UNIT
    out["roofline"] = out["levenshtein"]["roofline"]
    out["clocks"] = sampler.stop()
    return out


def sub_c4(dev, local_rank, sync, flush, peaks, steps):
    """BASELINE configs[3]: dense cosine top-10, 100k x 100k x 768 random unit vectors (bf16 in, fp32 accumulate)."""
    import torch
    from polyfuzz_b200 import dense
    n, d, k = 100_000, 768, 10
    torch.manual_seed(0); X = torch.randn(n, d, device=dev)
    torch.manual_seed(1); Y = torch.randn(n, d, device=dev)
    x, _ = dense.to_bf16_rows(X, True); y, _ = dense.to_bf16_rows(Y, True)
    del X, Y
    sampler = ClockSampler(local_rank)
    ms = timed(lambda: dense.dense_topk(x, y, k, 0.0), 3, steps, sync, flush)
    clocks = sampler.stop()
    t = float(np.median(ms)) * 1e-3
    flops = 2.0 * n * n * d
    burst = float(peaks.get("bf16_tflops", 1590.0)); sust = float(peaks.get("bf16_tflops_sustained", 1400.0))
    ach = flops / t / 1e12
    return {"workload": "dense cosine top-10, 100k x 100k x 768 random unit vectors, bf16 tcgen05 (BASELINE configs[3])", "data": "synthetic",
            "n_from": n, "n_to": n, "d": d, "top_n": k, "ms": t * 1e3, "ms_each": [round(v, 3) for v in ms],
            "value": float(n) * n / t, "unit": UNIT, "tflops": ach,
            "roofline": {"bound": "tensor", "achieved": ach, "peak": burst, "unit": "TFLOP/s", "frac": ach / burst,
                         "peak_sustained": sust, "frac_of_sustained": ach / sust,
                         "peak_source": "MEASURED_PEAKS.json bf16_tflops (cuBLAS burst) / bf16_tflops_sustained" if peaks else "fallback"},
            "clocks": clocks}


def sub_c5(args, dev, rank, local_rank, world, comm, barrier, flush, peak):
    """BASELINE configs[4]: TF-IDF char-trigram top-10 on n x n uniform 8..32-char strings (seed 0 = to, seed 1 = from),
    to_list row-sharded over the N GPUs (strong scaling: total work fixed).  Device-timed per step: K1 on the shard +
    all-reduce(df) + index + K2 (all from-rows x shard) + one all-gather(top-k) + merge."""
    import torch
    import torch.distributed as dist
    from polyfuzz_b200 import engine, synth
    from polyfuzz_b200.distributed import shard_bounds, tfidf_topk_sharded
    n = args.c5_n
    to = synth.uniform_strings(n, seed=0); frm = synth.uniform_strings(n, seed=1)
    lo, hi = shard_bounds(n, world, rank)
    vec0 = engine.NgramTfidf((3, 3), True, True)
    s_from = vec0.stage(frm); s_to = vec0.stage(to[lo:hi])
    del to, frm
    res = {}
    k2_events = []

    def step(rec):
        vec = engine.NgramTfidf((3, 3), True, True)
        idx, val, csr_to, index = tfidf_topk_sharded(vec, s_from, s_to, lo, TOP_N, 0.0, self_match=False, fit=True, fit_on_from=True,
                                                     comm=comm, timings=k2_events if rec else None, n_docs_total=2 * n)
        res.update(idx=idx, val=val, vec=vec, csr=csr_to, index=index)
    sampler = ClockSampler(local_rank, recording=False) if rank == 0 else None
    for _ in range(2):
        flush.zero_(); step(False)
    barrier()
    if sampler:
        sampler.recording = True
    ms = []
    for _ in range(args.steps):
        flush.zero_(); barrier()
        e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
        e0.record(); step(True); e1.record()
        barrier()
        ms.append(e0.elapsed_time(e1))
    clocks = sampler.stop() if sampler else None
    tot = torch.tensor([float(np.sum(ms))], dtype=torch.float64, device=dev)
    k2 = torch.tensor([float(np.mean([a.elapsed_time(b) for a, b in k2_events]))], dtype=torch.float64, device=dev)
    # postings visited by this rank: sum_t df_from(t) * df_to_shard(t)
    vec, csr = res["vec"], res["csr"]
    nnz = int(csr.indptr[-1].item())
    df_to = torch.bincount(csr.indices[:nnz].long(), minlength=vec.n_vocab).double()
    f_csr = vec.emit(vec.rows(s_from)); nf = int(f_csr.indptr[-1].item())
    df_from = torch.bincount(f_csr.indices[:nf].long(), minlength=vec.n_vocab).double()
    P = (df_from * df_to).sum().reshape(1)
    chk = torch.stack([res["idx"].long().sum().double(), res["val"].sum()])
    if world > 1:
        dist.all_reduce(tot, op=dist.ReduceOp.MAX); dist.all_reduce(k2, op=dist.ReduceOp.MAX); dist.all_reduce(P, op=dist.ReduceOp.SUM)
    t = float(tot.item()) / len(ms) * 1e-3
    P = float(P.item())
    s_bytes = 4 if res["index"].variant in ("dense32", "block", "hash") else 8     # stored weight: 32-bit fixed point / fp32, else fp64
    b_alg = P * (4 + s_bytes) + nf * 12.0 * world + float(n) * TOP_N * 12 * world
    k2_t = float(k2.item()) * 1e-3
    return {"workload": "TF-IDF char-trigram top-10, %d x %d uniform 8..32-char strings, to_list row-sharded x%d (BASELINE configs[4])" % (n, n, world),
            "data": "synthetic", "n_from": n, "n_to": n, "n_gpus": world, "scaling": "strong", "ms": t * 1e3, "ms_each": [round(v, 3) for v in ms],
            "value": float(n) * n / t, "unit": UNIT, "k2_variant": res["index"].variant, "tile": res["index"].tile, "V": vec.n_vocab,
            "k2_ms_max_over_ranks": k2_t * 1e3, "postings": P, "result_checksum": [float(chk[0].item()), float(chk[1].item())],
            "roofline": {"bound": "hbm", "kernel": "K2 (%s) on every rank" % res["index"].variant, "achieved": b_alg / k2_t / 1e9, "peak": peak * world,
                         "unit": "GB/s", "frac": b_alg / k2_t / 1e9 / (peak * world), "algorithmic_bytes": b_alg,
                         "weight_bytes_per_posting": s_bytes},
            "clocks": clocks}


def run_b200(args):
    import torch
    import torch.distributed as dist
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if world != args.gpus:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}; launch N>1 with torch.distributed.run")
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    skip = set(x for x in args.skip.split(",") if x)

    import polyfuzz_b200
    from polyfuzz_b200 import _lib, engine
    from polyfuzz_b200.distributed import get_comm, tfidf_topk_sharded
    comm = get_comm()
    n = args.n
    peaks, peak, peak_src = hbm_peak()

    # ---- data: rank r owns to-block r; the from-block is block 0 ----------------------------------
    from_list, shard, full_to, data_kind = load_names(args, rank, world)

    flush = torch.empty(512 << 20, dtype=torch.uint8, device=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- leg 1: device-resident inputs (value) -----------------------------------------------------
    vec0 = engine.NgramTfidf((3, 3), True, True)
    staged_from = vec0.stage(from_list)
    staged_to = staged_from if rank == 0 and world == 1 else vec0.stage(shard)
    if world > 1 and rank == 0:
        staged_to = vec0.stage(shard)                        # symmetric work on every rank
    k2_events = []
    k1_events = []
    result = {}

    def device_step(record_k2):
        vec = engine.NgramTfidf((3, 3), True, True)
        idx, val, csr_to, index = tfidf_topk_sharded(vec, staged_from, staged_to, rank * n, TOP_N, 0.0, self_match=True,
                                                     from_index_base=0, fit=True, fit_on_from=False, comm=comm,
                                                     timings=k2_events if record_k2 else None,
                                                     k1_timings=k1_events if record_k2 else None, n_docs_total=n * world)
        result["idx"], result["val"], result["vec"], result["csr"], result["index"] = idx, val, vec, csr_to, index

    import gc
    sampler = ClockSampler(local_rank, recording=False) if rank == 0 else None
    for _ in range(args.warmup + (2 if world > 1 else 0)):   # same code path as the timed steps (event creation included); N > 1 gets two
        flush.zero_(); barrier(); device_step(True)          # more untimed steps: the first collectives of a process are slow
    barrier()
    k2_events.clear(); k1_events.clear()
    gc.collect(); gc.disable()                               # no collector pauses inside the timed steps
    if sampler:
        sampler.recording = True
    launches0 = _lib.launch_count()
    step_ms = []
    for _ in range(args.steps):
        flush.zero_()
        barrier()
        e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
        e0.record(); device_step(True); e1.record()
        barrier()
        step_ms.append(e0.elapsed_time(e1))
    launches = _lib.launch_count() - launches0
    total_ms = torch.tensor([float(np.sum(step_ms))], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(total_ms, op=dist.ReduceOp.MAX)
    total_ms = float(total_ms.item())
    k2_ms = [a.elapsed_time(b) for a, b in k2_events]
    k1_ms = [a.elapsed_time(b) for a, b in k1_events]

    if args.dump_outputs and rank == 0:
        outputs = {"top_idx": result["idx"].cpu().numpy(), "top_val": result["val"].cpu().numpy()}
    keep = {k: result[k] for k in ("vec", "csr", "index")}
    result.clear(); result.update(keep)
    gc.enable(); gc.collect(); gc.disable()
    # ---- leg 2: end to end through the public matcher API with HOST lists (e2e) -------------------
    def e2e_step():
        m = polyfuzz_b200.TFIDF(n_gram_range=(3, 3), min_similarity=0.0, top_n=TOP_N, distributed=world > 1)
        if world > 1:
            # block 0 of the N*100k self-match: from-rows [0, n) against the full sharded list,
            # global diagonal excluded
            return m.match(full_to, from_block=(0, n))
        return m.match(from_list)

    e2e_ms = []
    e2e_steps = args.steps
    for it in range(2 + e2e_steps):
        flush.zero_()
        barrier()
        e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
        e0.record(); df = e2e_step(); e1.record()
        barrier()
        if it >= 2:
            e2e_ms.append(e0.elapsed_time(e1))
    e2e_total = torch.tensor([float(np.sum(e2e_ms))], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(e2e_total, op=dist.ReduceOp.MAX)
    e2e_ms_per_step = float(e2e_total.item()) / len(e2e_ms)
    gc.enable()
    del df
    clocks = sampler.stop() if sampler else None

    # ---- sub-records (other BASELINE configs), every one with its own clock record ----------------
    subs = {}
    if world == 1 and "c3" not in skip:
        subs["c3"] = sub_c3(dev, local_rank, torch.cuda.synchronize, flush, args.steps)
    if world == 1 and "c4" not in skip:
        subs["c4"] = sub_c4(dev, local_rank, torch.cuda.synchronize, flush, peaks, args.steps)
    if "c5" not in skip:
        keep_main = dict(result)
        subs["c5"] = sub_c5(args, dev, rank, local_rank, world, comm, barrier, flush, peak)
        result.clear(); result.update(keep_main)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- numbers ------------------------------------------------------------------------------------
    pairs = float(n) * (n * world) - n                       # from-block x all to-rows minus the diagonal
    ms_per_step = total_ms / args.steps
    value = pairs / (ms_per_step * 1e-3)
    vec, csr = result["vec"], result["csr"]
    nnz = int(csr.indptr[-1].item())
    # algorithmic bytes of the dominant kernel (SURVEY.md 8d): P*(4+s) + nnz_from*(4+s) + n_from*k*(4+8), s = bytes per
    # stored weight of the variant that ran (4 for the fp32 filter `dense32`, 8 for the fp64 kernels),
    # P = postings visited = sum_t df_from(t) * df_to_shard(t)
    cols = csr.indices[:nnz].cpu().numpy()
    df_to = np.bincount(cols, minlength=vec.n_vocab).astype(np.float64)
    if world == 1:
        df_from = df_to; nnz_from = nnz
    else:
        f_csr = vec.emit(vec.rows(staged_from)); nf = int(f_csr.indptr[-1].item())
        df_from = np.bincount(f_csr.indices[:nf].cpu().numpy(), minlength=vec.n_vocab).astype(np.float64); nnz_from = nf
    P = float((df_from * df_to).sum())
    variant = result["index"].variant
    s_bytes = 4 if variant in ("dense32", "block") else 8
    b_alg = P * (4 + s_bytes) + nnz_from * (4 + s_bytes) + n * TOP_N * 12
    b_alg_fp64 = P * 12 + nnz_from * 12 + n * TOP_N * 12
    k2_avg_ms = float(np.mean(k2_ms))
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "k2_ncu_summary.json")
    if os.path.exists(tpath):
        try:
            traffic = json.load(open(tpath)).get("dram_bytes_per_launch")
        except Exception:
            traffic = None
    achieved = b_alg / (k2_avg_ms * 1e-3) / 1e9
    roofline = {"bound": "hbm", "kernel": "K2 pfz_spcos_topk (variant %s)" % variant, "achieved": achieved, "peak": peak, "unit": "GB/s",
                "frac": achieved / peak, "traffic": traffic, "peak_source": peak_src,
                "weight_bytes_per_posting": s_bytes,
                "algorithmic_bytes_per_launch": b_alg, "postings_per_launch": P, "kernel_ms_avg": k2_avg_ms,
                "kernel_share_of_step": k2_avg_ms / ms_per_step,
                "frac_fp64_weight_model": b_alg_fp64 / (k2_avg_ms * 1e-3) / 1e9 / peak,
                "note": "frac uses the storage width of the variant that ran (SURVEY 8d: s = 4 for fp32 weights); frac_fp64_weight_model "
                        "is the same time against the reference's fp64 byte count (s = 8).  The index (~8-16 MB) is L2-resident: DRAM "
                        "traffic << algorithmic bytes by design (SURVEY 8d)"}

    from polyfuzz_b200.matchers._utils import LAST_TAIL
    h2d = staged_from.h2d_bytes * (1 if world == 1 else 2) + (n + 1) * 8            # packed strings + offsets + slot prefix, idf table
    d2h = LAST_TAIL["d2h_bytes"] + 3 * 8                                            # finished frame columns (K5) + the fit's three scalars
    e2e = {"value": pairs / (e2e_ms_per_step * 1e-3), "unit": UNIT, "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
           "ms_per_step": e2e_ms_per_step, "steps": len(e2e_ms), "ms_each": [round(x, 2) for x in e2e_ms],
           "frame_tail": "device (K5)" if LAST_TAIL["device"] else "host (Arrow)",
           "what": "TFIDF.match(list[str]) -> pandas.DataFrame: string packing, H2D, K1, index, K2, frame tail (rounding + string gathers"
                   " on the device), D2H of the finished columns, zero-copy Arrow/pandas wrap"}

    cpu = None
    if world == 1 and not args.no_cpu_baseline:
        from oracle import native
        native.build()
        thr = cpu_threads()
        r = cpu_reference_step(from_list, args.cpu_sample_rows, thr)
        cpu = {"value": r["pairs_per_s"], "unit": UNIT, "cores": thr, "kind": "port",
               "sample": "sklearn TfidfVectorizer (1 thread) on all %d names + C restatement of awesome_cossim_topn top-10 and the "
                         "reference assembly tail on the first %d from-rows x %d to-rows with %d OpenMP threads, extrapolated to the "
                         "whole job" % (n, r["sample_rows"], n, thr),
               "detail": {k: v for k, v in r.items() if k != "pairs_per_s"}}

    med = float(np.median(step_ms))
    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
            "data": data_kind, "config": config_dict(n, world, data_kind),
            "k2": {"tile": result["index"].tile, "variant": variant, "V": vec.n_vocab, "nnz": nnz,
                   "acc_bits": getattr(result["index"], "acc_bits", None), "block_rows": engine.BLOCK_ROWS if variant == "block" else None},
            "roofline": roofline, "cpu_baseline": cpu, "e2e": e2e, "gpu_launches": int(launches), "clocks": clocks,
            "step_ms_each": [round(x, 3) for x in step_ms], "step_ms_median": med,
            "step_outliers_over_5pct": int(sum(1 for x in step_ms if x > 1.05 * med)),
            "k1_ms_avg": float(np.mean(k1_ms)) if k1_ms else None, "k2_ms_avg": k2_avg_ms}
    line.update(subs)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, outputs)
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    args = parse()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()

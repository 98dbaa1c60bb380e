#!/usr/bin/env python
"""bench.py -- headline benchmark of the hot path (BASELINE.json `metric`):

    queries/sec, cosine top-10 @ 10 M x 384 fp32, single query per step; % of the HBM roofline; 1/2/4/8 GPUs.

A "step" is one pass of the hot path over the corpus for one query (BASELINE configs[1]).
    python bench.py --gpus 1 --steps K --warmup W
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N --steps K --warmup W
    python bench.py --impl reference ...      (the CPU restatement of the reference path on the host cores)

N > 1 is STRONG scaling: the same 10 M-row corpus row-sharded N ways (contiguous ranges), the query
replicated, the per-shard top-k lists exchanged over NVLink peer memory and merged inside the scan launch -- the only
exchange the path has (SURVEY.md section 8e).  Same measurement mode at every N: one query in flight.

Prints ONE JSON line (rank 0).  Keys follow the driver's contract; see DESIGN.md section "Measurement".
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

ROWS, DIMS, TOP_K = 10_000_000, 384, 10
CORPUS_SEED, QUERY_SEED = 2, 1002
SETTLE_STEPS = 20               # untimed searches before the W warm-ups + K timed steps (config.settle_steps)
METRIC_NAME = "queries/sec cosine top-10 @ 10Mx384 fp32"
FALLBACK_HBM_GBS = 6650.0       # /opt/skills/guides/B200_PROFILING.md fallback ("of fallback")


# ---------------------------------------------------------------------------------------------------------
def measured_peak():
    p = ROOT / "MEASURED_PEAKS.json"
    try:
        return float(json.loads(p.read_text())["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs, STREAM-style copy)"
    except Exception:
        return FALLBACK_HBM_GBS, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """nvidia-smi clocks + throttle reasons sampled DURING the timed region (B200_PROFILING.md recipe)."""
    FIELDS = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
              "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.rows, self.proc = index, [], None

    def __enter__(self):
        # NVML in-process first (a sample every 5 ms: the default timed region is only ~100 ms long), the
        # nvidia-smi loop of the recipe as the fallback.
        self.nvml = None
        self.stop = threading.Event()
        try:
            import pynvml
            pynvml.nvmlInit()
            handle = pynvml.nvmlDeviceGetHandleByIndex(self.index)
            pynvml.nvmlDeviceGetClockInfo(handle, pynvml.NVML_CLOCK_SM)
            self.nvml = (pynvml, handle)
            self.thread = threading.Thread(target=self._poll_nvml, daemon=True)
            self.thread.start()
            return self
        except Exception:
            self.nvml = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.FIELDS}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None
        return self

    def _poll_nvml(self):
        nv, h = self.nvml
        bits = (("hw_slowdown", 0x8), ("hw_thermal_slowdown", 0x40), ("sw_thermal_slowdown", 0x20), ("sw_power_cap", 0x4))
        try:
            mx = nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)
        except Exception:
            mx = 0
        get_reasons = getattr(nv, "nvmlDeviceGetCurrentClocksEventReasons", None) or \
            getattr(nv, "nvmlDeviceGetCurrentClocksThrottleReasons", None)
        while not self.stop.is_set():
            try:
                sm = nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)
                mask = int(get_reasons(h)) if get_reasons else 0
                self.rows.append([str(sm), str(mx)] + ["Active" if mask & b else "Not Active" for _, b in bits])
            except Exception:
                pass
            self.stop.wait(0.005)

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def __exit__(self, *exc):
        self.stop.set()
        if self.nvml:
            try:
                self.thread.join(timeout=1)
                self.nvml[0].nvmlShutdown()
            except Exception:
                pass
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()

    def summary(self):
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1]))
            except Exception:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[2:6]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons),
                "samples": len(sm), "source": "nvml" if getattr(self, "nvml", None) else "nvidia-smi"}


def host_queries(n: int) -> np.ndarray:
    """Seeded synthetic unit queries built on the host (uniform[-1,1] then L2-normalised, the reference
    benchmark embedder's distribution, RAGBenchmarkSupport.swift:130-156)."""
    rng = np.random.default_rng(QUERY_SEED)
    q = rng.uniform(-1.0, 1.0, size=(n, DIMS)).astype(np.float32)
    return (q / np.linalg.norm(q, axis=1, keepdims=True)).astype(np.float32)


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(out_dir, arrays: dict) -> None:
    """--dump-outputs: write what the timed calls returned in their last step as DIR/<name>.npy (ids as float64, exact
    below 2**53; scores as float32), so that two builds can be compared output for output on the same seeded inputs."""
    out = Path(out_dir)
    out.mkdir(parents=True, exist_ok=True)
    conv = {name: np.ascontiguousarray(a, dtype=np.float32 if np.asarray(a).dtype == np.float32 else np.float64)
            for name, a in arrays.items()}
    total = sum(a.nbytes for a in conv.values())
    assert total <= DUMP_LIMIT_BYTES, f"dump of {total} bytes exceeds {DUMP_LIMIT_BYTES}"
    for name, a in conv.items():
        np.save(out / f"{name}.npy", a)


def result_arrays(prefix: str, result) -> dict:
    """One search result (a list of (frame_id, score) pairs) as the arrays dump_outputs writes."""
    return {f"{prefix}_ids": np.array([r[0] for r in result], np.float64),
            f"{prefix}_scores": np.array([r[1] for r in result], np.float32)}


def host_mem_available_gb() -> float:
    try:
        for line in Path("/proc/meminfo").read_text().splitlines():
            if line.startswith("MemAvailable"):
                return int(line.split()[1]) / 1e6
    except Exception:
        pass
    return 0.0


# ---------------------------------------------------------------------------------------------------------
def cpu_reference_arm(rows: int, steps: int, warmup: int, budget_s: float = 25.0):
    """The reference's CPU path, restated (oracle ACC_F32_TREE, all host threads; `kind: port` because the
    Swift/USearch reference cannot be built in this image).  Bounded sample: as many corpus rows as fit the
    host and the time budget, materialised once; q/s is scaled to the full corpus by rows (the scan is linear)."""
    from oracle import oracle as o
    o.build()
    threads = o.host_threads()
    avail = host_mem_available_gb()
    sample_rows = rows
    max_rows_mem = int(max(avail - 8.0, 1.0) * 1e9 * 0.6 / (DIMS * 4))
    sample_rows = max(100_000, min(sample_rows, max_rows_mem, 10_000_000))
    t0 = time.perf_counter()
    corpus = o.synth_rows(CORPUS_SEED, 0, sample_rows, DIMS, normalize=True, threads=threads)
    gen_s = time.perf_counter() - t0
    qs = o.synth_rows(QUERY_SEED, 0, max(steps + warmup, 1), DIMS, normalize=True, threads=1)
    per = []
    t_start = time.perf_counter()
    for i in range(warmup + steps):
        t = time.perf_counter()
        o.search(o.COSINE, corpus, qs[i % len(qs)], TOP_K, mode=o.ACC_F32_TREE, threads=threads)
        dt = time.perf_counter() - t
        if i >= warmup:
            per.append(dt)
        if time.perf_counter() - t_start > budget_s and len(per) >= 3:
            break
    sec_per_query_full = float(np.mean(per)) * (rows / sample_rows)
    return {
        "value": 1.0 / sec_per_query_full, "unit": "queries/s", "cores": threads, "kind": "port",
        "sample": (f"{len(per)} queries x exact scan of {sample_rows} of {rows} rows x {DIMS} (oracle ACC_F32_TREE, "
                   f"{threads} threads, corpus materialised in {gen_s:.1f}s outside the timed region"
                   + (", time scaled by rows" if sample_rows != rows else "") + ")"),
        "ms_per_query_full_corpus": sec_per_query_full * 1e3, "steps_timed": len(per),
    }


def cpu_c1_single_thread(samples: int = 15, warmup: int = 2):
    """BASELINE configs[0]: 10 K x 384 fp32, 1 query, top-10 cosine on ONE host thread -- the reference's own
    CPU-runnable case, timed the way the reference times things (warm-up, then per-iteration samples:
    Tests/WaxIntegrationTests/RAGBenchmarkSupport.swift:285-308).  Both accumulation orders of the restatement:
    the scalar sequential loop (USearch's metric_cos / the in-test loop, the literal "reference order") and the
    SIMD-friendly tree order the kernels mirror."""
    from oracle import oracle as o
    o.build()
    corpus = o.synth_rows(1, 0, 10_000, DIMS, normalize=True, threads=1)
    q = o.synth_rows(QUERY_SEED, 0, 1, DIMS, normalize=True, threads=1)[0]
    out = {"workload": "10000 x 384 fp32 corpus (BASELINE configs[0]), 1 query, top-10 cosine, single host thread",
           "cores": 1, "kind": "port", "samples": samples, "warmup": warmup}
    for name, mode in (("f32_seq", o.ACC_F32_SEQ), ("f32_tree", o.ACC_F32_TREE)):
        for _ in range(warmup):
            o.search(o.COSINE, corpus, q, TOP_K, mode=mode, threads=1)
        ts = []
        for _ in range(samples):
            t = time.perf_counter()
            o.search(o.COSINE, corpus, q, TOP_K, mode=mode, threads=1)
            ts.append(time.perf_counter() - t)
        out[name] = {"ms_mean": float(np.mean(ts)) * 1e3, "ms_min": float(np.min(ts)) * 1e3,
                     "ms_median": float(np.median(ts)) * 1e3, "queries_per_s": 1.0 / float(np.mean(ts))}
    return out


def run_reference(args, rank: int):
    if rank != 0:
        return
    base = cpu_reference_arm(args.rows, args.steps, args.warmup)
    line = {
        "impl": "reference", "metric": METRIC_NAME, "value": base["value"], "unit": "queries/s",
        "n_gpus": args.gpus, "steps": base["steps_timed"], "warmup": args.warmup,
        "ms_per_step": base["ms_per_query_full_corpus"], "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args, max(args.gpus, 1)),
        "cpu_baseline": {k: base[k] for k in ("value", "unit", "cores", "kind", "sample")},
        "cpu_c1_single_thread": cpu_c1_single_thread(),
        "e2e": {"value": base["value"], "unit": "queries/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "note": "CPU restatement of the reference path (exact scan, USearch metric formulas); the shipped reference "
                "CPU engine is USearch HNSW (approximate) and cannot be built here (no Swift toolchain).",
    }
    print(json.dumps(line), flush=True)


def workload_config(args, world: int):
    return {
        "workload": f"{args.rows} x {DIMS} fp32 corpus (BASELINE configs[1]), 1 query per step, top-{TOP_K} cosine",
        "rows": args.rows, "dims": DIMS, "top_k": TOP_K,
        "sharding": f"{world} contiguous row shard(s), {args.rows // world} rows per GPU" if world > 1 else "single GPU",
        "l2": f"corpus {args.rows * DIMS * 4 / world / 1e9:.2f} GB per GPU vs 126 MB L2: inputs larger than L2, no flush"
              if args.rows * DIMS * 4 / world > 4 * 126e6 else "corpus per GPU not >> L2: L2 flushed between steps",
        "corpus_seed": CORPUS_SEED, "query_seed": QUERY_SEED, "settle_steps": SETTLE_STEPS,
    }


# ---------------------------------------------------------------------------------------------------------
def run_single(args):
    import torch
    from wax_b200 import CUDAVectorEngine, VectorMetric
    torch.cuda.set_device(0)
    eng = CUDAVectorEngine(VectorMetric.cosine, DIMS, device=0)
    eng.fill_synthetic(CORPUS_SEED, args.rows)
    for key, val in (kv.split("=") for kv in args.opt):
        eng.set_option(key, int(val))
    n_distinct = min(64, args.steps + args.warmup)

    small = args.rows * DIMS * 4 <= 4 * 126e6
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda") if small else None

    # ---- value: kernel-only, inputs resident in HBM, CUDA events on the launching stream (inside the library)
    torch.cuda.synchronize()
    with ClockSampler(0) as clk:
        if small:   # flush L2 between steps: time each step separately
            ms_total, launches = 0.0, 0
            eng.time_search(TOP_K, 1, warmup=max(args.warmup, 3), n_queries=n_distinct, seed=QUERY_SEED)
            for i in range(args.steps):
                flush.fill_(i & 0xFF); torch.cuda.synchronize()
                ms, ln = eng.time_search(TOP_K, 1, warmup=0, n_queries=1, seed=QUERY_SEED + i)
                ms_total += ms; launches += ln
        else:
            # an untimed settling pass first (the clocks / HBM of a GPU that has just been filled are still ramping: one
            # record had the first 100 ms 2 % slower than the e2e region that followed), then W warm-ups + K timed steps
            eng.time_search(TOP_K, SETTLE_STEPS, warmup=0, n_queries=n_distinct, seed=QUERY_SEED)
            ms_total, launches = eng.time_search(TOP_K, args.steps, warmup=max(args.warmup, 3),
                                                 n_queries=n_distinct, seed=QUERY_SEED)
        torch.cuda.synchronize()
        # ---- e2e: the public call a user makes (wax_vs_search through the mirror): HOST query in, HOST result out
        qs = host_queries(n_distinct)
        for i in range(max(args.warmup, 3)):
            eng.search(qs[i % n_distinct], TOP_K)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        last = None
        for i in range(args.steps):
            if small:
                flush.fill_(i & 0xFF)
            last = eng.search(qs[i % n_distinct], TOP_K)
        torch.cuda.synchronize()
        e2e_s = time.perf_counter() - t0
    clocks = clk.summary()
    ms_per_step = ms_total / args.steps
    value = args.steps / (ms_total / 1e3)

    peak, peak_src = measured_peak()
    read_ceiling = eng.stream_read_gbs(5)                # plain LDG.128 read of the same bytes, same box
    alg_bytes = args.rows * DIMS * 4                     # SURVEY 8d: N*D*4 algorithmic bytes per launch
    achieved = alg_bytes / (ms_per_step / 1e3) / 1e9
    traffic = None
    for tp in (ROOT / "profiles" / "traffic_r02.json", ROOT / "profiles" / "r01" / "traffic_r01.json"):
        if traffic is None and tp.exists():     # dram bytes per launch from the committed `ncu --set full` capture
            try:
                t = json.loads(tp.read_text())
                if t.get("rows") == args.rows:
                    traffic = t.get("dram_bytes_per_launch")
            except Exception:
                pass
    line = {
        "metric": METRIC_NAME, "value": value, "unit": "queries/s", "n_gpus": 1, "steps": args.steps,
        "warmup": max(args.warmup, 3), "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args, 1),
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                     "traffic": traffic, "peak_source": peak_src,
                     "stream_read_ceiling_gbs": read_ceiling, "frac_of_read_ceiling": achieved / read_ceiling if read_ceiling else None,
                     "nominal_hbm_gbs": 7700.0, "frac_of_nominal": achieved / 7700.0,
                     "kernel": "scan_tma_kernel<C=3,cosine> (fused scan+top-k, 1 launch per query)",
                     "algorithmic_bytes_per_launch": alg_bytes},
        "e2e": {"value": args.steps / e2e_s, "unit": "queries/s", "h2d_bytes_per_step": DIMS * 4,
                "d2h_bytes_per_step": TOP_K * 24, "ms_per_step": e2e_s / args.steps * 1e3,
                "api": "wax_vs_search (host query -> host ids/scores, synchronous)"},
        "gpu_launches": int(launches),
        "clocks": clocks,
        "check": {"top1_frame_id": last[0][0] if last else None, "top1_score": last[0][1] if last else None},
    }
    outputs = result_arrays("e2e", last) if last else {}
    if not args.no_shadow and not small:
        try:                        # an extra measurement must never cost the headline line
            line["shadow_filtered"] = shadow_filtered_arm(eng, args, qs, n_distinct, outputs)
        except Exception as ex:     # noqa: BLE001
            line["shadow_filtered"] = {"error": repr(ex)}
    if not args.no_shadow and not small:
        try:                        # BASELINE configs[2] on the same resident corpus: the tensor-bound companion number
            line["batched"] = batched_arm(eng, args, outputs=outputs)
        except Exception as ex:     # noqa: BLE001
            line["batched"] = {"error": repr(ex)}
    if not args.no_shadow and not small:
        eng.close()                 # free the 23 GB of configs[1]/[2] before the 46 GB of configs[4]
        try:
            line["batched_c5"] = batched_c5_arm(outputs=outputs)
        except Exception as ex:     # noqa: BLE001
            line["batched_c5"] = {"error": repr(ex)}
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, outputs)
    if not args.no_cpu_baseline:
        base = cpu_reference_arm(args.rows, steps=5, warmup=1, budget_s=20.0)
        line["cpu_baseline"] = {k: base[k] for k in ("value", "unit", "cores", "kind", "sample")}
        try:
            line["cpu_c1_single_thread"] = cpu_c1_single_thread()
            # the GPU side of configs[0] for context (launch-latency-bound: 15 MB is 2 us of HBM time)
        except Exception as ex:     # noqa: BLE001
            line["cpu_c1_single_thread"] = {"error": repr(ex)}
    print(json.dumps(line), flush=True)


def _tensor_peaks():
    try:
        return json.loads((ROOT / "MEASURED_PEAKS.json").read_text())
    except Exception:  # noqa: BLE001
        return {}


def _batched_line(eng, rows, dims, batch, top_k, metric_name, workload, steps, outputs=None, name=""):
    """Device-only time (CUDA events inside the library) + the same batch END TO END through wax_vs_search_batch with
    HOST buffers (queries H2D, ids/scores D2H inside the timed region) + which level answered.  The arrays of the last
    end-to-end step go into `outputs` (a dict) as <name>_ids / _scores / _counts when it is given."""
    import torch
    peaks = _tensor_peaks()
    ms, launches, unproven = eng.time_search_batch(batch, top_k, steps, warmup=4, seed=QUERY_SEED)
    per = ms / steps
    flops = 2.0 * batch * rows * dims
    tf = flops / (per * 1e-3) / 1e12
    bf16 = eng.counter("shadow_bytes") > 0
    peak = float(peaks.get("bf16_tflops", 2250.0)) if bf16 else 1100.0
    rng = np.random.default_rng(QUERY_SEED + batch)
    qs = rng.uniform(-1.0, 1.0, size=(batch, dims)).astype(np.float32)
    qs /= np.linalg.norm(qs, axis=1, keepdims=True)
    for _ in range(2):
        eng.search_batch_arrays(qs, top_k)
    t0q, f0q = eng.batch_stats()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(steps):
        ids, scores, ns = eng.search_batch_arrays(qs, top_k)
    torch.cuda.synchronize()
    e2e_s = (time.perf_counter() - t0) / steps
    if outputs is not None:
        outputs.update({f"{name}_ids": ids, f"{name}_scores": scores, f"{name}_counts": ns})
    t1q, f1q = eng.batch_stats()
    return {
        "workload": workload, "value": batch / per * 1e3, "unit": "queries/s", "ms_per_step": per, "steps": steps,
        "dtype": ("bf16" if bf16 else "tf32") + " nominations + f32 exact re-score",
        "roofline": {"bound": "tensor", "achieved": tf, "peak": peak, "unit": "TFLOP/s", "frac": tf / peak,
                     "peak_source": "measured cuBLAS bf16 burst (MEASURED_PEAKS.json bf16_tflops)" if bf16 and "bf16_tflops" in peaks
                     else ("nominal dense bf16" if bf16 else "nominal dense TF32"),
                     "frac_of_sustained": tf / float(peaks["bf16_tflops_sustained"]) if bf16 and "bf16_tflops_sustained" in peaks else None,
                     "useful_flops_per_launch": flops,
                     "hbm_floor_ms": rows * dims * (2 if bf16 else 4) / (float(peaks.get("hbm_gbs", FALLBACK_HBM_GBS)) * 1e9) * 1e3},
        "e2e": {"value": batch / e2e_s, "unit": "queries/s", "ms_per_step": e2e_s * 1e3,
                "h2d_bytes_per_step": batch * dims * 4, "d2h_bytes_per_step": batch * top_k * 24,
                "api": "wax_vs_search_batch (host queries -> host ids/scores, synchronous)"},
        "gpu_launches_per_step": launches / steps, "unproven_queries_last_step": unproven,
        "levels": {"tensor_proven_queries": t1q - t0q, "exact_scan_fallback_queries": f1q - f0q,
                   "shadow_unavailable_tf32_level": bool(eng.counter("shadow_unavailable")),
                   "shadow_gb": eng.counter("shadow_bytes") / 1e9},
        "metric": metric_name,
    }


def batched_arm(eng, args, batch: int = 1024, steps: int = 10, outputs=None):
    """NOT the headline: BASELINE configs[2] (batch of 1024 queries, top-10 cosine) on the corpus already resident for
    the headline -- tcgen05 nominations over the bf16 shadow + exact fp32 re-score + completeness proof (DESIGN 4.5.1),
    results identical to 1024 single-query scans (tests/test_gpu_fullsize.py checks that at this size)."""
    return _batched_line(eng, args.rows, DIMS, batch, TOP_K, "queries/sec cosine top-10, batch 1024 @ 10Mx384 fp32",
                         f"{args.rows} x {DIMS} fp32 corpus (BASELINE configs[2]), batch {batch}, top-{TOP_K} cosine", steps,
                         outputs, "batched")


def batched_c5_arm(rows: int = 10_000_000, dims: int = 768, batch: int = 256, top_k: int = 100, steps: int = 10,
                   outputs=None):
    """NOT the headline: BASELINE configs[4] -- 10 M x 768 fp32 rows that are NOT normalised, batch 256, top-100 under
    the dot metric (score = q.v - 1).  Its own engine (30.7 GB corpus + 15.4 GB bf16 shadow)."""
    from wax_b200 import CUDAVectorEngine, VectorMetric
    eng = CUDAVectorEngine(VectorMetric.dot, dims, device=0)
    try:
        eng.fill_synthetic(5, rows, normalize=False)
        return _batched_line(eng, rows, dims, batch, top_k, "queries/sec dot top-100, batch 256 @ 10Mx768 fp32",
                             f"{rows} x {dims} fp32 un-normalised corpus (BASELINE configs[4]), batch {batch}, top-{top_k} dot", steps,
                             outputs, "batched_c5")
    finally:
        eng.close()


def shadow_filtered_arm(eng, args, qs, n_distinct, outputs=None):
    """NOT the headline (`value` / `e2e` above are the fused fp32 scan north_star names): the same single-query
    workload with the opt-in `single_shadow` mode -- the query is first ranked against the bf16 shadow of the corpus
    (half the HBM bytes, DESIGN 4.5.1), the best nominees are re-scored exactly in fp32 and a completeness proof
    guards the result, so ids and score bits are identical to the fp32 scan (checked here on every step)."""
    import torch
    expect = [eng.search(qs[i % n_distinct], TOP_K) for i in range(min(args.steps, n_distinct))]
    eng.set_option("single_shadow", 1)
    try:
        ms, launches, unproven = eng.time_search_batch(1, TOP_K, args.steps, warmup=3, seed=QUERY_SEED)
        for i in range(3):
            eng.search(qs[i % n_distinct], TOP_K)
        f0 = eng.batch_stats()[1]
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        got = [eng.search(qs[i % n_distinct], TOP_K) for i in range(args.steps)]
        torch.cuda.synchronize()
        e2e_s = time.perf_counter() - t0
        same = all(got[i] == expect[i % len(expect)] for i in range(args.steps))
        if outputs is not None and got:
            outputs.update(result_arrays("shadow_filtered", got[-1]))
        return {
            "value": args.steps / (ms / 1e3), "unit": "queries/s", "ms_per_step": ms / args.steps,
            "e2e": {"value": args.steps / e2e_s, "unit": "queries/s", "ms_per_step": e2e_s / args.steps * 1e3},
            "gpu_launches_per_query": launches / args.steps, "identical_to_fp32_scan": bool(same),
            "exact_fallbacks": eng.batch_stats()[1] - f0, "shadow_gb": eng.counter("shadow_bytes") / 1e9,
            "hbm_bytes_per_query": args.rows * DIMS * 2,
            "achieved_gbs_on_shadow_bytes": args.rows * DIMS * 2 / (ms / args.steps / 1e3) / 1e9,
            "note": "opt-in mode (wax_vs_debug_set_option single_shadow=1); bf16 shadow nominates on the tensor path, "
                    "fp32 re-score + proof make the result identical; costs dims*2 B/row of extra HBM",
        }
    finally:
        eng.set_option("single_shadow", 0)


def run_sharded(args, rank: int, world: int, local_rank: int):
    """N > 1: the same 10 M-row corpus row-sharded N ways (STRONG scaling), measured in the SAME mode as N = 1:
    `value` = K collective searches strictly one at a time on one stream, CUDA events on that stream, max over ranks
    (N = 1 times K fused scans back to back on one stream the same way); `e2e` = K synchronous calls of the public
    sharded search with a HOST query and HOST results on every rank.  One kernel launch per query per rank: the
    exchange of the per-shard top-k lists and the merge run inside the scan launch over NVLink peer memory."""
    import torch
    import torch.distributed as dist
    from wax_b200 import VectorMetric, sharded
    torch.cuda.set_device(local_rank)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    eng = sharded.ShardedVectorEngine(VectorMetric.cosine, DIMS, total_rows=args.rows)
    eng.fill_synthetic(CORPUS_SEED)
    for key, val in (kv.split("=") for kv in args.opt):
        eng.engine.set_option(key, int(val))
    n_distinct = min(64, args.steps + args.warmup)
    qs_host = host_queries(n_distinct)
    warm = max(args.warmup, 3)
    shard_bytes = (eng.row_hi - eng.row_lo) * DIMS * 4
    fused = eng.transport == "p2p-fused"

    def max_over_ranks(x: float) -> float:
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def timed_value(e, steps):
        """K searches, one in flight, device-timed; returns (ms_total max over ranks, launches on this rank)."""
        dist.barrier(); torch.cuda.synchronize()
        if e.transport == "p2p-fused":
            ms, launches = e.time_search(TOP_K, steps, warmup=warm, n_queries=n_distinct, seed=QUERY_SEED)
        else:   # no peer mapping between the ranks: NCCL all-gather + host merge, still strictly one query at a time
            qs_dev = torch.from_numpy(qs_host).cuda()
            for i in range(warm):
                e.finish(e.search_async(qs_dev[i % n_distinct], TOP_K))
            torch.cuda.synchronize(); dist.barrier()
            ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            ev0.record()
            for i in range(steps):
                e.finish(e.search_async(qs_dev[i % n_distinct], TOP_K))
            ev1.record(); torch.cuda.synchronize()
            ms, launches = ev0.elapsed_time(ev1), steps
        torch.cuda.synchronize(); dist.barrier()
        return max_over_ranks(ms), launches

    def timed_e2e(e, steps):
        for i in range(warm):
            e.search(qs_host[i % n_distinct], TOP_K)
        dist.barrier(); torch.cuda.synchronize()
        t0 = time.perf_counter()
        last = None
        for i in range(steps):
            last = e.search(qs_host[i % n_distinct], TOP_K)      # host query in, merged host result out, synchronous
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        dist.barrier()
        return max_over_ranks(dt), last

    with ClockSampler(local_rank) as clk:
        timed_value(eng, SETTLE_STEPS)          # untimed settling pass (see run_single), collective on every rank
        ms_total, launches = timed_value(eng, args.steps)
        e2e_s, last = timed_e2e(eng, args.steps)
    clocks = clk.summary()
    # every rank must hold the same merged answer
    same = torch.tensor([last[0][0], int(np.float32(last[0][1]).view(np.uint32))], dtype=torch.int64, device="cuda")
    lo, hi = same.clone(), same.clone()
    dist.all_reduce(lo, op=dist.ReduceOp.MIN); dist.all_reduce(hi, op=dist.ReduceOp.MAX)
    ranks_agree = bool(torch.equal(lo, hi))

    transport, transport_note = eng.transport, eng.transport_note
    weak = None
    if not args.no_weak:
        try:
            weak = weak_arm(args, eng, world, timed_value, timed_e2e)
        except Exception as ex:     # noqa: BLE001
            weak = {"error": repr(ex)}
    eng.close()     # no-op for the engine the weak arm already closed
    if rank == 0:
        peak, peak_src = measured_peak()
        ms_per_step = ms_total / args.steps
        achieved = shard_bytes / (ms_per_step / 1e3) / 1e9
        line = {
            "metric": METRIC_NAME, "value": args.steps / (ms_total / 1e3), "unit": "queries/s", "n_gpus": world,
            "steps": args.steps, "warmup": warm, "ms_per_step": ms_per_step, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(args, world),
            "mode": "latency: strictly one query in flight, K launches back to back on one stream per rank (as N=1)",
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": None, "peak_source": peak_src,
                         "note": "per GPU: shard bytes / the step's single kernel launch (scan + NVLink exchange + merge "
                                 "in one launch; its duration includes waiting for the slowest rank)",
                         "algorithmic_bytes_per_launch": shard_bytes},
            "e2e": {"value": args.steps / e2e_s, "unit": "queries/s", "h2d_bytes_per_step": DIMS * 4,
                    "d2h_bytes_per_step": TOP_K * 24, "ms_per_step": e2e_s / args.steps * 1e3,
                    "api": "ShardedVectorEngine.search -> wax_vs_shard_search (host query -> merged host ids/scores on "
                           "every rank, synchronous)" if fused else "ShardedVectorEngine.search (all-gather transport)"},
            "gpu_launches": int(launches), "queries_in_flight": 1,
            "collective": ("none per query: the scan's last CTA writes its top-k (240 B) into every rank's mailbox over "
                           "NVLink peer memory and merges in-kernel; torch.distributed only passed the mailbox handles "
                           "at start-up") if fused else
                          f"1 all_gather_into_tensor of {TOP_K * 24} B per rank per step (nccl) + host merge",
            "transport": transport, "transport_note": transport_note,
            "clocks": clocks,
            "check": {"top1_frame_id": last[0][0], "top1_score": last[0][1], "ranks_agree": ranks_agree},
        }
        if weak is not None:
            line["weak"] = weak
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, result_arrays("e2e", last))
        print(json.dumps(line), flush=True)
    dist.destroy_process_group()


def weak_arm(args, strong_eng, world, timed_value, timed_e2e, rows_per_gpu: int = 12_500_000, steps: int = 10):
    """NOT the headline: WEAK scaling -- 12.5 M rows x 384 per GPU, generated on device (at 8 GPUs this is BASELINE
    configs[3]: 100 M x 384 row-sharded over 8 B200s, 19.2 GB per GPU, 1 query, top-10 cosine).  Same latency mode."""
    import torch
    import torch.distributed as dist
    from wax_b200 import VectorMetric, sharded
    strong_eng.close()
    total = rows_per_gpu * world
    eng = sharded.ShardedVectorEngine(VectorMetric.cosine, DIMS, total_rows=total)
    eng.fill_synthetic(4)
    ms_total, launches = timed_value(eng, steps)
    e2e_s, last = timed_e2e(eng, steps)
    per = ms_total / steps
    peak, _ = measured_peak()
    gbs = rows_per_gpu * DIMS * 4 / (per / 1e3) / 1e9
    out = {
        "workload": f"{total} x {DIMS} fp32 corpus row-sharded over {world} GPUs ({rows_per_gpu} rows = "
                    f"{rows_per_gpu * DIMS * 4 / 1e9:.1f} GB per GPU), 1 query per step, top-{TOP_K} cosine"
                    + (" (BASELINE configs[3])" if world == 8 else ""),
        "value": steps / (ms_total / 1e3), "unit": "queries/s", "ms_per_step": per, "steps": steps,
        "per_gpu_gbs": gbs, "per_gpu_frac_of_measured_peak": gbs / peak, "aggregate_gbs": gbs * world,
        "e2e": {"value": steps / e2e_s, "unit": "queries/s", "ms_per_step": e2e_s / steps * 1e3},
        "gpu_launches_per_step": launches / steps, "transport": eng.transport,
        "check": {"top1_frame_id": last[0][0], "top1_score": last[0][1]},
    }
    eng.close()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--rows", type=int, default=ROWS, help="override the corpus size (experiments only)")
    ap.add_argument("--opt", action="append", default=[], help="engine tuning option key=value (experiments)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-shadow", action="store_true", help="skip the extra `shadow_filtered` (opt-in mode) measurement")
    ap.add_argument("--no-weak", action="store_true", help="N>1: skip the extra weak-scaling (12.5 M rows per GPU) measurement")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the results of the last timed step of each search measured "
                         "(e2e_*: the public single-query search; batched_*, batched_c5_*, shadow_filtered_*: the extra "
                         "arms that ran) as DIR/<name>.npy; the inputs are seeded, so two builds compare output for output")
    args = ap.parse_args()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        return run_reference(args, rank)
    if world > 1:
        return run_sharded(args, rank, world, local_rank)
    return run_single(args)


if __name__ == "__main__":
    main()

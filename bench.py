#!/usr/bin/env python3
"""bench.py — queries/sec and GB/s of the VectorBase top-k lookup on B200.

One "step" = one pass of the hot path over one batch of synthetic queries:
the whole corpus is scored against B queries and the k best rows per query are returned.

Default workload (BASELINE.json `metric`: "top-k cosine on 10M x 768"): configs[2] =
10M x 768 bf16 corpus, batch 256, top-100, on one B200.  With --gpus N (launched by
torch.distributed.run, one rank per GPU) the SAME corpus is row-sharded over the N GPUs
(strong scaling): every rank searches its rows, per-rank candidates are exchanged and merged on
every rank.

Output: ONE JSON line (rank 0).
  value      queries/sec with inputs resident in HBM, CUDA events over exactly --steps steps
             (max over ranks);
  e2e        the same through the public host API (pinned host queries -> H2D -> search -> D2H
             results) inside the timed region;
  roofline   the dominant kernel's algorithmic bytes / its event-timed duration — events recorded
             by libtavec around that kernel INSIDE the timed region of `value` (same pass, so
             kernel_ms_per_step <= ms_per_step by construction) — against MEASURED_PEAKS.json;
             `sustained` repeats it over >= 2 s of back-to-back steps (the power-capped figure);
  cpu_baseline  the reference's own VectorBase (unmodified file, vendored under oracle/_ref by
             build(); else the numpy restatement) on this box's host cores over the FULL corpus;
  parity_checked  4 queries of the final step compared with the blocked numpy oracle over the
             device corpus at the contract tolerances;
  secondary  the other single-GPU BASELINE configs (c1, c2, c5; c4 at 8 GPUs), each with its own
             value / e2e / roofline / cpu_baseline.
`--impl reference` times the reference's CPU path alone (same metric / config strings, so the
driver can divide).

`--dump-outputs DIR` writes the hits of the last timed step of the main workload as
DIR/items.npy (float64 row ordinals), DIR/scores.npy (float32) and DIR/counts.npy (float64);
entries past a query's count are -1 / NaN.  Inputs are seeded, so two builds run with the same
arguments can be compared output for output.  Above 64 MB a fixed, seeded sample of the queries
is written, their indices in DIR/query_index.npy.  Apart from DIR the bench writes no files.
"""

from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True   # the tree may be read-only; keep the bench from writing __pycache__ into it

WORKLOADS = {
    # name: rows, dim, storage, batch, k, min_score
    "c1": dict(rows=10_000, dim=384, storage="float32", batch=1, k=10, min_score=0.0,
               desc="10k x 384 fp32, 1 query, top-10 (tools/benchmark_vectorbase.py)"),
    "c2": dict(rows=1_000_000, dim=768, storage="bfloat16", batch=64, k=32, min_score=0.0,
               desc="1M x 768 bf16, batch 64, top-32"),
    "c3": dict(rows=10_000_000, dim=768, storage="bfloat16", batch=256, k=100, min_score=0.0,
               desc="10M x 768 bf16, batch 256, top-100"),
    "c4": dict(rows=10_000_000, dim=1536, storage="float16", batch=1024, k=100, min_score=0.0,
               desc="10M x 1536 fp16 row-sharded, batch 1024, top-100"),
    "c5": dict(rows=50_000, dim=384, storage="bfloat16", batch=1000, k=5, min_score=0.0,
               desc="RelatedTerms 50k x 384, 1000 query terms, top-5"),
    "c5f32": dict(rows=50_000, dim=384, storage="float32", batch=1000, k=5, min_score=0.0,
                  desc="RelatedTerms 50k x 384 float32 (as the reference stores it), 1000 query terms, top-5"),
    "c2f32": dict(rows=1_000_000, dim=768, storage="float32", batch=64, k=32, min_score=0.0,
                  desc="1M x 768 float32, batch 64, top-32 (split-precision tensor path)"),
    "s1": dict(rows=10_000_000, dim=768, storage="float32", batch=1, k=10, min_score=0.0,
               desc="10M x 768 fp32, 1 query, top-10 (row-scan path at scale)"),
    "s8": dict(rows=10_000_000, dim=768, storage="float32", batch=8, k=10, min_score=0.0,
               desc="10M x 768 fp32, 8 queries, top-10 (row-scan path at scale)"),
}
ELEM = {"float32": 4, "bfloat16": 2, "float16": 2}
SEED = 20260922


def parse_args():
    p = argparse.ArgumentParser()
    p.add_argument("--gpus", type=int, default=1)
    p.add_argument("--steps", type=int, default=10)
    p.add_argument("--warmup", type=int, default=3)
    p.add_argument("--impl", choices=["b200", "reference"], default="b200")
    p.add_argument("--workload", choices=sorted(WORKLOADS), default="c3")
    p.add_argument("--rows", type=int, default=None, help="override corpus rows (experiments / tests)")
    p.add_argument("--batch", type=int, default=None)
    p.add_argument("--k", type=int, default=None)
    p.add_argument("--path", choices=["auto", "scan", "mma"], default="auto")
    p.add_argument("--no-cpu-baseline", action="store_true")
    p.add_argument("--no-secondary", action="store_true", help="skip the c1/c2/c5 (c4 at 8 GPUs) block")
    p.add_argument("--no-parity", action="store_true", help="skip the blocked-oracle check of the final step")
    p.add_argument("--sustain-seconds", type=float, default=2.0, help="0 disables the sustained roofline run")
    p.add_argument("--cpu-queries", type=int, default=8, help="timed single-query lookups of the cpu_baseline leg")
    p.add_argument("--dump-outputs", metavar="DIR", default=None,
                   help="write the hits of the last timed step as DIR/<name>.npy (see the module docstring)")
    args = p.parse_args()
    if args.steps < 1 or args.warmup < 0:
        p.error("--steps must be >= 1 and --warmup >= 0")
    if args.dump_outputs and args.impl != "b200":
        p.error("--dump-outputs writes the GPU path's hits; it needs --impl b200")
    return args


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(dump_dir, items, scores, counts):
    """Hits of one step (device tensors [B, k], [B, k], [B]) -> dump_dir/{items,scores,counts}.npy."""
    counts = counts.cpu().numpy().astype(np.int64)
    items = items.cpu().numpy().astype(np.float64)      # row ordinals < 2**53: exact
    scores = scores.cpu().numpy().astype(np.float32)
    past = np.arange(items.shape[1])[None, :] >= counts[:, None]
    items[past], scores[past] = -1.0, np.nan
    arrays = {"items": items, "scores": scores, "counts": counts.astype(np.float64)}
    per_query = sum(a[0].nbytes for a in arrays.values())
    if per_query * len(counts) > DUMP_LIMIT_BYTES:
        keep = np.sort(np.random.default_rng(SEED).choice(len(counts), DUMP_LIMIT_BYTES // per_query, replace=False))
        arrays = {name: a[keep] for name, a in arrays.items()}
        arrays["query_index"] = keep.astype(np.float64)
    os.makedirs(dump_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(dump_dir, name + ".npy"), a)


def metric_string(w):
    """The SAME string for the repo arm and the reference arm (the driver divides like by like)."""
    return ("queries/sec, top-k cosine (VectorBase.fuzzy_lookup_embedding) on "
            f"{w['rows']}x{w['dim']} {w['storage']}, batch {w['batch']}, top-{w['k']}")


def algorithmic_bytes(rows, dim, storage, batch, k):
    """SURVEY.md §8d: corpus read once per batch + queries + hits."""
    return rows * dim * ELEM[storage] + batch * dim * 4 + batch * k * 12


def load_ncu_traffic(workload, path, world, rows):
    """dram bytes per launch of the dominant kernel from the committed ncu capture, or None."""
    try:
        with open(os.path.join(ROOT, "profiles", "ncu_traffic.json")) as f:
            table = json.load(f)
    except Exception:
        return None
    key = f"{workload}/{path}/{world}"
    if rows != WORKLOADS[workload]["rows"]:
        key = f"{workload}-shard-{rows}/{path}/{world}"
    entry = table.get(key)
    return entry["bytes"] if entry else None


def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            p = json.load(f)
        return {"hbm_gbs": p["hbm_gbs"], "bf16_tflops": p.get("bf16_tflops"),
                "bf16_tflops_sustained": p.get("bf16_tflops_sustained"), "source": "measured"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "source": "fallback"}


def workload_config(w, n_gpus):
    return {
        "workload": w["desc"], "rows": w["rows"], "dim": w["dim"], "storage": w["storage"],
        "batch": w["batch"], "k": w["k"], "min_score": w["min_score"],
        "parallelism": f"row-sharded x{n_gpus}, candidate exchange + merge on every rank" if n_gpus > 1 else "single GPU",
        "l2": "corpus shard >> 126 MB L2, no flush needed" if w["rows"] * w["dim"] * ELEM[w["storage"]] / n_gpus > 4e8
              else "corpus fits L2: L2 flushed (256 MB write) between timed steps",
    }


# ----------------------------------------------------------------------------- CPU side
def host_threads():
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


def set_blas_threads(n):
    """Pin the BLAS pool to `n` threads whatever OMP_NUM_THREADS says (torch.distributed.run exports
    OMP_NUM_THREADS=1); returns (context manager or None, threads the pool reports)."""
    try:
        from threadpoolctl import threadpool_info, threadpool_limits

        ctl = threadpool_limits(limits=n, user_api="blas")
        got = [i.get("num_threads") for i in threadpool_info() if i.get("user_api") == "blas"]
        return ctl, (max(got) if got else n)
    except Exception:
        return None, n


def make_host_corpus(rows, dim, seed, threads):
    """Unit-norm float32 rows [rows, dim] on the host (what the reference stores), generated in
    1M-row blocks on a thread pool (numpy generators release the GIL): block b uses seed + b, as
    tools/benchmark_vectorbase.py:80-94 does for its single block."""
    from concurrent.futures import ThreadPoolExecutor

    out = np.empty((rows, dim), dtype=np.float32)
    block = 250_000

    def fill(b):
        lo, hi = b * block, min(rows, (b + 1) * block)
        rng = np.random.default_rng(seed + b)
        rng.standard_normal(out=out[lo:hi], dtype=np.float32)
        out[lo:hi] /= np.linalg.norm(out[lo:hi], axis=1, keepdims=True)

    n_blocks = -(-rows // block)
    with ThreadPoolExecutor(max_workers=max(1, min(threads, n_blocks))) as ex:
        list(ex.map(fill, range(n_blocks)))
    return out


class _NullModel:
    model_name = "bench-null"

    def add_embedding(self, key, embedding):
        return None


def make_cpu_lookup(vectors):
    """(callable(query, k, min_score) -> hits, kind): the UNMODIFIED reference VectorBase when its
    file is available (mounted, or vendored under oracle/_ref by build()), else the oracle port."""
    from oracle import ref_loader

    if ref_loader.reference_available():
        vb, _ = ref_loader.load_reference()
        base = vb.VectorBase(vb.TextEmbeddingIndexSettings(embedding_model=_NullModel()))
        base.deserialize(vectors)  # adopts the array, no copy (vectorbase.py:273-287)
        return (lambda q, k, ms: base.fuzzy_lookup_embedding(q, max_hits=k, min_score=ms)), "reference"
    from oracle import vectorbase_oracle as O

    return (lambda q, k, ms: O.lookup(vectors, q, k, ms)), "port"


def cpu_reference_leg(w, warmup, timed, want_batched=False):
    """The reference's CPU path on this box's host cores, FULL workload rows (no extrapolation):
    one VectorBase.fuzzy_lookup_embedding per query — np.dot sgemv over the whole float32 corpus ->
    score -> threshold -> argpartition — as every caller of the reference does
    (storage/memory/reltermsindex.py:326-331).  `warmup` + `timed` single-query lookups; the BLAS pool
    is set to the cores this process may run on.  Returns per-query seconds (list) and metadata."""
    threads = host_threads()
    ctl, blas_threads = set_blas_threads(threads)
    try:
        t0 = time.perf_counter()
        vectors = make_host_corpus(w["rows"], w["dim"], SEED + 1000, threads)
        gen_s = time.perf_counter() - t0
        rng = np.random.default_rng(7)
        n_q = warmup + timed
        q = rng.standard_normal((max(n_q, 1), w["dim"])).astype(np.float32)
        q /= np.linalg.norm(q, axis=1, keepdims=True)
        lookup, kind = make_cpu_lookup(vectors)
        times = []
        for i in range(n_q):
            t0 = time.perf_counter()
            hits = lookup(q[i], w["k"], w["min_score"])
            times.append(time.perf_counter() - t0)
            assert len(hits) == min(w["k"], w["rows"])
        batched = None
        if want_batched:
            # "strong" CPU baseline (SURVEY.md §8d-ii): ONE sgemm for a few queries, then the per-row
            # ranking — what a batched numpy caller could do; the reference itself never batches.
            from oracle import vectorbase_oracle as O

            nb = min(8, w["batch"])
            t0 = time.perf_counter()
            O.lookup_batch(vectors, q[:nb] if len(q) >= nb else np.repeat(q[:1], nb, 0), w["k"], w["min_score"],
                           one_gemm=True)
            batched = nb / (time.perf_counter() - t0)
    finally:
        if ctl is not None:
            ctl.restore_original_limits()
    steady = times[warmup:]
    med = statistics.median(steady)
    return {
        "per_query_s": steady, "median_s": med, "kind": kind, "cores": blas_threads,
        "gen_s": gen_s, "batched_sgemm_value": batched,
        "sample": (f"FULL corpus {w['rows']} x {w['dim']} float32 ({w['rows'] * w['dim'] * 4 / 1e9:.1f} GB) resident on "
                   f"the host; {timed} timed single-query lookups after {warmup} warm-up, median "
                   f"{med * 1e3:.2f} ms/query; {blas_threads} BLAS threads of {threads} usable cores; "
                   f"numpy {np.__version__}; " + ("unmodified reference VectorBase" if kind == "reference"
                                                 else "numpy restatement (oracle/)")),
        "gbs": w["rows"] * w["dim"] * 4 / med / 1e9,
    }


def cpu_baseline_block(leg):
    out = {"value": 1.0 / leg["median_s"], "unit": "queries/s", "cores": leg["cores"], "kind": leg["kind"],
           "sample": leg["sample"], "host_gb_per_s": leg["gbs"]}
    if leg.get("batched_sgemm_value"):
        out["batched_sgemm_value"] = leg["batched_sgemm_value"]
    return out


def run_reference_impl(args, w):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    # one step = ONE single-query lookup over the full corpus (a bounded sample of the batch's B
    # queries: the reference serves a batch as B such lookups); ms_per_step = B x median per query
    leg = cpu_reference_leg(w, warmup=args.warmup, timed=args.steps)
    qps = 1.0 / leg["median_s"]
    out = {
        "impl": "reference",
        "metric": metric_string(w),
        "value": qps, "unit": "queries/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": w["batch"] * leg["median_s"] * 1e3, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic (unit-norm gaussian rows; seeds in bench.py)",
        "config": workload_config(w, args.gpus),
        "cpu_baseline": cpu_baseline_block(leg),
        "e2e": {"value": qps, "unit": "queries/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "step_definition": "one step = one single-query lookup over the full corpus; ms_per_step = batch x "
                           "median per-query time (the reference runs a batch as B sequential lookups)",
    }
    print(json.dumps(out), file=_RESULT_OUT, flush=True)


# ----------------------------------------------------------------------------- GPU side
class ClockSampler:
    """SM clock / power / throttle reasons sampled every few ms DURING the timed region
    (NVML in a thread; falls back to polling nvidia-smi)."""

    def __init__(self, gpu_index: int, period_s: float = 0.004):
        self.samples = []  # (sm_mhz, power_w, reasons_bitmask)
        self.sm_max = None
        self.period = period_s
        self._stop = threading.Event()
        self.source = "nvml"
        try:
            import pynvml

            pynvml.nvmlInit()
            self.nv = pynvml
            # NVML enumerates physical order; honour CUDA_VISIBLE_DEVICES when it is a plain list
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = gpu_index
            if vis:
                try:
                    phys = int(vis.split(",")[gpu_index])
                except Exception:
                    phys = gpu_index
            self.h = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.sm_max = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
            self.thread = threading.Thread(target=self._loop_nvml, daemon=True)
        except Exception:
            self.nv = None
            self.source = "nvidia-smi"
            self.gpu_index = gpu_index
            self.thread = threading.Thread(target=self._loop_smi, daemon=True)
        self.thread.start()

    def _loop_nvml(self):
        nv = self.nv
        while not self._stop.is_set():
            try:
                sm = float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                pw = nv.nvmlDeviceGetPowerUsage(self.h) / 1000.0
                try:
                    rs = int(nv.nvmlDeviceGetCurrentClocksEventReasons(self.h))
                except Exception:
                    rs = int(nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h))
                self.samples.append((sm, pw, rs))
            except Exception:
                pass
            time.sleep(self.period)

    def _loop_smi(self):
        fields = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active"
        while not self._stop.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--id={self.gpu_index}", f"--query-gpu={fields}",
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5)
                parts = [p.strip() for p in out.stdout.strip().split(",")]
                self.sm_max = float(parts[1])
                self.samples.append((float(parts[0]), float(parts[2]), int(parts[3], 16)))
            except Exception:
                pass

    def mark(self):
        return len(self.samples)

    def summary(self, first=0):
        # NVML clocks-event reason bits
        names = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown",
                 0x4: "sw_power_cap", 0x80: "hw_power_brake_slowdown", 0x2: "applications_clocks_setting"}
        part = self.samples[first:]
        sm = [s for s, _, _ in part]
        pw = [p for _, p, _ in part]
        mask = 0
        for _, _, r in part:
            mask |= r
        reasons = sorted(n for bit, n in names.items() if mask & bit)
        # "under load": samples whose power is within 25% of the run's maximum
        pmax = max(pw) if pw else 0.0
        busy = [s for s, p in zip(sm, pw) if p >= 0.75 * pmax] or sm
        return {"sm_mhz": statistics.median(busy) if busy else None, "sm_min_mhz": min(busy) if busy else None,
                "sm_max_mhz": self.sm_max, "power_w_max": pmax if pw else None, "samples": len(sm),
                "source": self.source, "reasons": reasons}

    def stop(self):
        self._stop.set()
        self.thread.join(timeout=5)
        return self.summary()


def make_shard_on_device(torch, device, lo, hi, dim, storage, seed):
    """Synthetic unit-norm rows [lo, hi) generated on the GPU in 1M-row blocks (float32
    standard normal -> row-normalised in float32 -> rounded to the storage dtype), mirroring
    tools/benchmark_vectorbase.py:80-94.  Block b of the global corpus uses seed + b, so any
    sharding produces the same corpus."""
    tdt = {"float32": torch.float32, "bfloat16": torch.bfloat16, "float16": torch.float16}[storage]
    out = torch.empty((hi - lo, dim), dtype=tdt, device=device)
    block = 1_000_000
    gen = torch.Generator(device=device)
    pos = lo
    while pos < hi:
        b = pos // block
        gen.manual_seed(seed + b)
        x = torch.randn((block, dim), generator=gen, device=device, dtype=torch.float32)
        x /= x.norm(dim=1, keepdim=True)
        start = pos - b * block
        stop = min(hi - b * block, block)
        out[pos - lo: pos - lo + (stop - start)] = x[start:stop].to(tdt)
        pos += stop - start
        del x
    return out


class Bench:
    """Device-side state shared by the workloads of one run."""

    def __init__(self, args):
        import torch
        import torch.distributed as dist

        self.torch, self.dist, self.args = torch, dist, args
        self.rank = int(os.environ.get("RANK", "0"))
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.local_rank = int(os.environ.get("LOCAL_RANK", "0"))
        if self.world != args.gpus and self.world == 1 and args.gpus > 1:
            raise SystemExit("launch with torch.distributed.run --nproc-per-node N for --gpus N")
        torch.cuda.set_device(self.local_rank)
        self.device = torch.device("cuda", self.local_rank)
        if self.world > 1:
            os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
            dist.init_process_group("nccl", device_id=self.device)
        self.peaks = load_peaks()

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def max_over_ranks(self, ms):
        if self.world == 1:
            return ms
        t = self.torch.tensor([ms], dtype=self.torch.float64, device=self.device)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def close(self):
        if self.world > 1:
            self.dist.destroy_process_group()


def measure(bn: Bench, name, w, steps, warmup, *, force=None, sustain_s=0.0, parity=True, cpu=True, cpu_queries=8,
            dump_dir=None):
    """One workload on the GPUs of this run -> the result dict (rank 0) or None (other ranks)."""
    import typeagent_py_b200 as tab
    from typeagent_py_b200.sharded import ShardedVectorBase, shard_bounds

    torch, world, rank, device = bn.torch, bn.world, bn.rank, bn.device
    rows, dim, storage, batch, k = w["rows"], w["dim"], w["storage"], w["batch"], w["k"]
    lo, hi = shard_bounds(rows, world)[rank]
    corpus = make_shard_on_device(torch, device, lo, hi, dim, storage, seed=SEED)
    torch.cuda.synchronize()

    settings = tab.TextEmbeddingIndexSettings(embedding_model=_NullModel(), min_score=w["min_score"])
    if world == 1:
        base = tab.VectorBase.from_device_tensor(settings, corpus)
        sharded = None
    else:
        sharded = ShardedVectorBase(settings, device=bn.local_rank, storage_dtype=storage)
        sharded.load_local_shard(corpus, rows)
        base = sharded._engine.base
    base.force_path = force
    # events around the DOMINANT kernel (and the whole search) only, recorded inside the timed region; the
    # per-kind breakdown comes from a separate, untimed pass below (an event pair per kernel boundary is a
    # measurable share of a 0.1-0.4 ms search)
    base.enable_timing(main_only=True)

    rng = np.random.default_rng(7)
    q_host = torch.empty((batch, dim), dtype=torch.float32).pin_memory()
    qn = rng.standard_normal((batch, dim)).astype(np.float32)
    qn /= np.linalg.norm(qn, axis=1, keepdims=True)
    q_host.copy_(torch.from_numpy(qn))
    q_dev = q_host.to(device)
    out_items = torch.empty((batch, k), dtype=torch.int64).pin_memory()
    out_scores = torch.empty((batch, k), dtype=torch.float32).pin_memory()
    out_counts = torch.empty((batch,), dtype=torch.int32).pin_memory()

    shard_bytes = (hi - lo) * dim * ELEM[storage]
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=device) if shard_bytes < 4e8 else None
    res_out = (torch.empty((batch, k), dtype=torch.int64, device=device),
               torch.empty((batch, k), dtype=torch.float32, device=device),
               torch.empty((batch,), dtype=torch.int32, device=device))

    def step_resident():
        # fully asynchronous; the "did any query need the exact fallback" check of every step is
        # kept on the device and resolved by finish_resident() inside the timed region
        if sharded is None:
            return base.search_device(q_dev, k, w["min_score"], out=res_out, defer_check=True)
        return sharded.search_tensors(q_dev, k, w["min_score"], defer_check=True)

    fallbacks = [0]

    def finish_resident():
        # exact fallbacks are legitimate (probability ~1e-7 per query) and their cost stays in the
        # timed region; they are counted and reported
        fallbacks[0] += base.finish_search() if sharded is None else sharded.finish()

    q_one = q_host.numpy()[0]

    def step_e2e():
        # public host API: pinned host queries -> H2D -> search -> D2H of the hits
        if sharded is None and batch == 1:
            # the reference's own call shape (tools/benchmark_vectorbase.py:97-109): one embedding in,
            # list[ScoredInt] out
            return base.fuzzy_lookup_embedding(q_one, max_hits=k, min_score=w["min_score"])
        if sharded is None:
            return base.search_arrays(q_host.numpy(), k, w["min_score"],
                                      out=(out_items.numpy(), out_scores.numpy(), out_counts.numpy()))
        qd = q_host.to(device, non_blocking=True)
        items, scores, counts = sharded.search_tensors(qd, k, w["min_score"])
        out_items.copy_(items, non_blocking=True)
        out_scores.copy_(scores, non_blocking=True)
        out_counts.copy_(counts, non_blocking=True)
        torch.cuda.current_stream().synchronize()
        return out_items, out_scores, out_counts

    def history(n):
        """per-kernel times of the last n searches (events recorded by libtavec inside the region)"""
        import ctypes as C

        from typeagent_py_b200 import _capi

        cap = 64
        arr = [(C.c_float * cap)() for _ in range(4)]
        got = C.c_int(0)
        _capi.check(_capi.load().tav_timing_history(base._ix, min(cap, n), arr[0], arr[1], arr[2], arr[3], C.byref(got)))
        m = got.value
        return {"main": list(arr[0][:m]), "sample": list(arr[1][:m]), "aux": list(arr[2][:m]), "search_total": list(arr[3][:m])}

    last_hits = [None]   # (items, scores, counts) of the latest timed step

    def timed_resident(n_steps):
        """EXACTLY n_steps steps, CUDA events on the launching stream; returns total ms (this rank)."""
        total = 0.0
        if flush is None:
            bn.barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for i in range(n_steps):
                last_hits[0] = step_resident()
                if (i & 7) == 7:
                    finish_resident()      # at most 8 (sharded) / 64 searches may be outstanding
            finish_resident()
            e1.record()
            bn.barrier()
            return e0.elapsed_time(e1)
        for _ in range(n_steps):
            flush.fill_(1)
            bn.barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            last_hits[0] = step_resident()
            finish_resident()
            e1.record()
            bn.barrier()
            total += e0.elapsed_time(e1)
        return total

    # warm-up (both legs), then the timed regions
    for _ in range(warmup):
        step_resident()
        finish_resident()
        step_e2e()
    bn.barrier()

    sampler = ClockSampler(bn.local_rank) if rank == 0 else None
    ms_resident = bn.max_over_ranks(timed_resident(steps))
    # later steps reuse the output buffers: copy the last timed step's hits (stream-ordered, untimed)
    dumped = tuple(t.clone() for t in last_hits[0]) if dump_dir and rank == 0 else None
    hist = history(steps)                       # the SAME pass as ms_resident
    # rank-to-rank spread of the local search (a sharded step ends when the SLOWEST rank has published)
    per_rank = None
    if world > 1:
        mine = (statistics.fmean(hist["main"]) if hist["main"] else None,
                statistics.fmean(hist["search_total"]) if hist["search_total"] else None)
        gathered = [None] * world
        bn.dist.all_gather_object(gathered, mine)
        mains = [g[0] for g in gathered if g and g[0] is not None]
        totals = [g[1] for g in gathered if g and g[1] is not None]
        if mains and totals:
            per_rank = {"main_kernel_ms": {"min": min(mains), "max": max(mains)},
                        "local_search_ms": {"min": min(totals), "max": max(totals)}}
    lt = base.last_timing()
    launches_per_step = lt["launches"] + (2 if world > 1 else 0)
    path = lt["path"]
    # e2e: each step ends with a host synchronisation (the D2H result read).  Timed per step so that
    # the L2 flush of the small workloads stays outside the timed region, as in the resident leg.
    ms_e2e_local, wall_e2e = 0.0, 0.0
    for _ in range(steps):
        if flush is not None:
            flush.fill_(1)
        bn.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter()
        e0.record()
        step_e2e()
        e1.record()
        e1.synchronize()
        wall_e2e += time.perf_counter() - t0
        ms_e2e_local += e0.elapsed_time(e1)
    ms_e2e = bn.max_over_ranks(ms_e2e_local)
    lt_e2e = base.last_timing()                 # the last e2e step's device-side share (first launch -> last result byte)
    clocks = sampler.summary() if sampler else None

    # sustained: >= sustain_s seconds of back-to-back steps (the power cap engages after ~50 ms)
    sustained = None
    if sustain_s > 0 and flush is None:
        per_step_s = max(ms_resident / steps / 1e3, 1e-5)
        n_sus = int(min(max(sustain_s / per_step_s, 64), 200_000))
        mark = sampler.mark() if sampler else 0
        ms_sus = bn.max_over_ranks(timed_resident(n_sus))
        h = history(64)
        sus_clocks = sampler.summary(mark) if sampler else None
        sustained = {"steps": n_sus, "seconds": ms_sus / 1e3, "ms_per_step": ms_sus / n_sus,
                     "kernel_ms": statistics.fmean(h["main"]) if h["main"] else None,
                     "sm_mhz": sus_clocks["sm_mhz"] if sus_clocks else None,
                     "reasons": sus_clocks["reasons"] if sus_clocks else None}
    if sampler:
        sampler.stop()

    # per-kind breakdown (prep / sample / main / finalize): a few extra steps with an event pair per kernel
    base.enable_timing()
    for _ in range(5):
        if flush is not None:
            flush.fill_(1)
        step_resident()
        finish_resident()
    kinds = history(5)
    base.enable_timing(main_only=True)

    # the result of a last step: well-formed, and equal to the oracle's for sampled queries
    items, scores, counts = step_resident()
    finish_resident()
    torch.cuda.synchronize()
    assert int(counts.min()) == min(k, rows) and bool((scores[:, :-1] >= scores[:, 1:]).all())
    assert int(items.min()) >= 0 and int(items.max()) < rows
    parity_checked, parity_note = False, "skipped"
    if parity:
        parity_checked, parity_note = check_parity(bn, corpus, lo, qn, items, scores, counts, k, w["min_score"], storage)
    if dumped is not None:
        dump_outputs(dump_dir, *dumped)

    del corpus, base, sharded
    torch.cuda.empty_cache()
    if rank != 0:
        return None

    peaks = bn.peaks
    ms_step = ms_resident / steps
    qps = batch / (ms_step / 1e3)
    e2e_ms_step = ms_e2e / steps
    kernel_ms = statistics.fmean(hist["main"]) if hist["main"] else float("nan")
    breakdown = {name_: statistics.fmean(v) for name_, v in kinds.items() if v}
    # per-GPU dominant kernel: this rank's shard is read once per pass of the kernel
    passes = 1 if path in ("mma", "mma_split") else -(-batch // 8)
    algo_bytes = algorithmic_bytes(hi - lo, dim, storage, batch, k)
    algo_launch_bytes = (hi - lo) * dim * ELEM[storage] * passes + batch * dim * 4 + batch * k * 12
    achieved = algo_bytes / (kernel_ms / 1e3) / 1e9
    flops = 2.0 * batch * (hi - lo) * dim
    tensor_bound = path in ("mma", "mma_split") and flops / (peaks["bf16_tflops"] or 1.6e3) / 1e12 > \
        algo_bytes / peaks["hbm_gbs"] / 1e9 * 1.25
    out = {
        "metric": metric_string(w),
        "value": qps, "unit": "queries/s", "n_gpus": world, "steps": steps, "warmup": warmup,
        "ms_per_step": ms_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": {"float32": "f32", "bfloat16": "bf16", "float16": "f16"}[storage],
        "dtype_detail": "operands in the storage dtype, float32 accumulate, float32 scores (the reference: float32 throughout)",
        "data": "synthetic (unit-norm gaussian rows, generated on device; seeds in bench.py)",
        "config": workload_config(w, world),
        "path": path,
        "gb_per_s": algorithmic_bytes(rows, dim, storage, batch, k) / (ms_step / 1e3) / 1e9,
        "e2e": {"value": batch / (e2e_ms_step / 1e3), "unit": "queries/s",
                "h2d_bytes_per_step": batch * dim * 4, "d2h_bytes_per_step": batch * k * 12 + batch * 4,
                "ms_per_step": e2e_ms_step, "wall_ms_per_step": wall_e2e * 1e3 / steps,
                "device_search_ms_last_step": lt_e2e["total_ms"], "main_kernel_ms_last_step": lt_e2e["scan_ms"],
                "api": ("VectorBase.fuzzy_lookup_embedding(host float32 embedding) -> list[ScoredInt]" if batch == 1 and world == 1
                        else "VectorBase.search_arrays(host float32 queries) -> host int64/float32 hits")},
        "gpu_launches": launches_per_step * steps,
        "exact_fallback_queries": fallbacks[0],
        "parity_checked": parity_checked, "parity": parity_note,
        "roofline": {
            "bound": "hbm", "kernel": "scan_rows_kernel" if path == "scan" else "mma_topk_kernel (" + path + ")",
            "achieved": achieved, "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": achieved / peaks["hbm_gbs"],
            "of": peaks["source"], "traffic": load_ncu_traffic(name, path, world, rows),
            "kernel_ms_per_step": kernel_ms,
            "search_ms_per_step_same_pass": statistics.fmean(hist["search_total"]) if hist["search_total"] else None,
            "per_step_ms_by_kernel_kind": breakdown,
            "breakdown_note": "per_step_ms_by_kernel_kind: a separate pass of 5 steps with an event pair around every "
                              "kernel; kernel_ms_per_step / search_ms_per_step_same_pass: the timed pass itself",
            "algorithmic_bytes_per_step": algo_bytes,
            "bytes_actually_requested_per_step": algo_launch_bytes,
            "note": "achieved = algorithmic bytes (corpus shard read once per batch) / duration of the dominant "
                    "kernel (the MAIN launch of the tcgen05 kernel, or the row-scan kernel), CUDA events recorded by "
                    "libtavec around it inside the timed region of `value` (same pass)" + ("" if passes == 1 else
                    f"; the row-scan path re-reads the corpus once per 8 queries ({passes} passes)"),
        },
        "clocks": clocks,
    }
    if per_rank:
        per_rank["exchange_and_skew_ms"] = ms_step - per_rank["local_search_ms"]["max"]
        per_rank["note"] = ("a sharded step = the slowest rank's local search + candidate exchange (publish over NVLink, "
                            "flag wait, merge); exchange_and_skew = ms_per_step - the slowest rank's local search")
        out["per_rank"] = per_rank
    if peaks.get("bf16_tflops") and path in ("mma", "mma_split"):
        rf = out["roofline"]
        rf["tensor_tflops"] = flops / (kernel_ms / 1e3) / 1e12
        rf["tensor_frac_of_burst"] = rf["tensor_tflops"] / peaks["bf16_tflops"]
        if tensor_bound:
            # arithmetic intensity well above the ridge: the tensor pipe, not HBM, bounds this shape
            rf["hbm_gbs"], rf["hbm_frac"] = rf["achieved"], rf["frac"]
            rf.update({"bound": "tensor", "achieved": rf["tensor_tflops"], "peak": peaks["bf16_tflops"],
                       "unit": "TFLOP/s", "frac": rf["tensor_frac_of_burst"]})
    if sustained:
        s_ach = algo_bytes / (sustained["kernel_ms"] / 1e3) / 1e9 if sustained["kernel_ms"] else None
        out["roofline"]["sustained"] = {
            **sustained, "achieved": s_ach, "frac": s_ach / peaks["hbm_gbs"] if s_ach else None,
            "value": batch / (sustained["ms_per_step"] / 1e3),
            "note": "same measurement over >= 2 s of back-to-back steps (kernel_ms = mean of the last 64): the "
                    "figure under the 1 kW power cap"}
        if peaks.get("bf16_tflops_sustained") and sustained["kernel_ms"]:
            out["roofline"]["sustained"]["tensor_frac_of_sustained"] = \
                flops / (sustained["kernel_ms"] / 1e3) / 1e12 / peaks["bf16_tflops_sustained"]
    if cpu and world == 1:
        leg = cpu_reference_leg(w, warmup=3, timed=cpu_queries, want_batched=True)
        out["cpu_baseline"] = cpu_baseline_block(leg)
    return out


def check_parity(bn, corpus, lo, qn, items, scores, counts, k, min_score, storage):
    """4 queries of the final step vs the blocked numpy oracle over the DEVICE corpus (each rank its
    own shard, lists merged like shards), at the contract tolerances (scores 1e-4, ties 2e-6)."""
    from oracle import vectorbase_oracle as O
    from tests.parity import assert_hits_match, blocked_oracle_lookup

    torch = bn.torch
    b = len(qn)
    pick = sorted({0, b // 3, (2 * b) // 3, b - 1})
    q_pick = O.round_to_storage(qn[pick], storage)      # the device rounds queries to the storage dtype
    local = blocked_oracle_lookup(corpus, q_pick, k, min_score, row_offset=lo)
    if bn.world > 1:
        gathered = [None] * bn.world
        bn.dist.all_gather_object(gathered, [[(h.item, h.score) for h in hits] for hits in local])
        if bn.rank != 0:
            return True, "checked on rank 0"
        local = [O.merge_shard_hits([[O.Hit(i, s) for i, s in shard[j]] for shard in gathered], k)
                 for j in range(len(pick))]
    it, sc, ct = items.cpu().numpy(), scores.cpu().numpy(), counts.cpu().numpy()
    for j, qi in enumerate(pick):
        got = {"items": it[qi, : ct[qi]].tolist(), "scores": sc[qi, : ct[qi]].tolist()}
        assert_hits_match(got, local[j], score_tol=1e-4, tie_tol=2e-6, min_score=min_score,
                          what=f"bench parity q{qi}")
    return True, f"queries {pick} of the final step == blocked numpy oracle (scores 1e-4, ties 2e-6)"


def run_b200(args, w):
    bn = Bench(args)
    force = None if args.path == "auto" else args.path
    out = measure(bn, args.workload, w, args.steps, args.warmup, force=force, sustain_s=args.sustain_seconds,
                  parity=not args.no_parity, cpu=not args.no_cpu_baseline, cpu_queries=args.cpu_queries,
                  dump_dir=args.dump_outputs)
    # the other BASELINE configs ride along so that the driver's records carry them
    secondary = {}
    if not args.no_secondary and args.workload == "c3" and args.rows is None:
        names = ["c1", "c2", "c5"] if bn.world == 1 else (["c4"] if bn.world == 8 else [])
        for name in names:
            sw = dict(WORKLOADS[name])
            res = measure(bn, name, sw, steps=args.steps, warmup=args.warmup, sustain_s=0.0,
                          parity=not args.no_parity, cpu=not args.no_cpu_baseline, cpu_queries=args.cpu_queries)
            if res is not None:
                keep = ("metric", "value", "unit", "ms_per_step", "path", "e2e", "roofline", "cpu_baseline",
                        "parity_checked", "exact_fallback_queries", "gpu_launches", "config", "per_rank")
                secondary[name] = {kk: res[kk] for kk in keep if kk in res}
    if out is not None:
        if secondary:
            out["secondary"] = secondary
        print(json.dumps(out), file=_RESULT_OUT, flush=True)
    bn.close()


_RESULT_OUT = sys.stdout


def main():
    # Libraries (NCCL prints "NCCL version ..." to stdout) must not pollute the one-JSON-line
    # contract: route fd 1 to stderr for the whole run and keep a private handle for the result.
    global _RESULT_OUT
    _RESULT_OUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    args = parse_args()
    w = dict(WORKLOADS[args.workload])
    for name in ("rows", "batch", "k"):
        if getattr(args, name) is not None:
            w[name] = getattr(args, name)
            w["desc"] += f" [{name}={w[name]}]"
    if args.impl == "reference":
        run_reference_impl(args, w)
    else:
        run_b200(args, w)


if __name__ == "__main__":
    main()

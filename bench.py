#!/usr/bin/env python
"""bench.py -- tokens/s of the SCONE input-embedding lookup on B200, with roofline and CPU baseline.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload suite|config1..config5|config3s]

One "step" = one pass of the fused hot path (longest f-gram match + row gather + dequant + fallback) over
one [B, L] batch of synthetic token ids.  The headline workload is BASELINE.json configs[1]: GPT-2-medium
shape, 1 M f-grams, max_n = 4, INT8 cache, batch 64 x 1024, bf16 output.

Default (`--workload suite`) prints ONE JSON line (rank 0):
  * the headline fields are config 2 (at N > 1: one replica per GPU, weak scaling, no data-path collective):
    `value` = whole-job tokens/s with inputs resident in HBM (K steps replayed as one CUDA graph, CUDA events, max
    over ranks); `e2e` = the same metric through the drop-in class -- `EmbeddingCache.lookup()` /
    `EmbeddingCache.host_pipeline()` -- with the ids coming from pinned HOST memory and the match result read back to
    the host every step (`e2e.embeds_to_host`: the embeddings cross the host link as well); `roofline` = algorithmic
    bytes / kernel time against MEASURED_PEAKS.json; `cpu_baseline` = the oracle's port of the reference path timed on
    this box's cores.
  * N = 1 adds `configs`: config 1, config 3 (full size) and config 5 (offloaded tier, as many rows as the box's RAM
    allows), each measured by a child process of this script with its own clocks, hit rate and roofline.
  * N > 1 adds `configs.config3` (N replicas of config 3, the config BASELINE names "on 1 and 8xB200") and `sharded`: config 4 -- the table row-sharded over the N GPUs at 12.5 M rows per GPU (819 GB at N = 8) --
    through the peer-direct fused kernel and through the NCCL all-to-all variant, with NVLink and HBM fractions, a clock
    record, and an in-run bit-exact check of a sample of every rank's output against the oracle.

`--workload configX` measures that workload alone (what the child processes run).  `--impl reference` times the CPU
port of the reference path alone (all cores, fork pool over batch rows) -- the reference is pure Python and cannot
travel to the GPU box, so the port (oracle/py_oracle.py, pinned to fixtures generated from the unmodified reference)
stands in for it.

`--dump-outputs DIR` (the suite's headline and config1..config3) writes what the last timed step handed its caller,
so that two builds can be compared output for output on identical seeded inputs (rank 0's batch at N > 1):
  DIR/fgram_id.npy    float64 [B, L]
  DIR/match_len.npy   float32 [B, L]
  DIR/embeddings.npy  float32 [S, D]: the bf16 embeddings at S token positions (flat index b * L + l) drawn without
                      replacement by numpy.random.default_rng(0) and sorted, S = min(B * L, 32 MiB / (4 * D))
"""

from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: N f-grams, D, V, max_n, quant, B, L   (BASELINE.json configs; SURVEY.md section 8d)
    "config1": dict(N=100_000, D=768, V=50_257, max_n=3, quant="fp16", B=8, L=512,
                    desc="GPT-2 small, small-100k f-grams, max_n=3, FP16 cache, batch 8x512"),
    "config2": dict(N=1_000_000, D=1024, V=50_257, max_n=4, quant="int8", B=64, L=1024,
                    desc="GPT-2 medium, medium-1m f-grams, max_n=4, INT8 cache, batch 64x1024"),
    "config3": dict(N=10_000_000, D=4096, V=128_000, max_n=5, quant="int4", B=256, L=2048,
                    desc="hidden 4096, 10M f-grams, max_n=5, INT4 g128 cache, batch 256x2048"),
    # N here is PER GPU (12.5 M rows x 8 192 B = 102 GB per GPU; 100 M f-grams at 8 GPUs)
    "config4": dict(N=12_500_000, D=4096, V=128_000, max_n=5, quant="fp16", B=256, L=2048, tier="sharded",
                    desc="hidden 4096, 100M f-grams (12.5M per GPU), FP16 cache row-sharded by id % W, batch 256x2048 per GPU"),
    # config 3's table row-sharded instead of replicated (SURVEY 8d: "8-GPU run: replicas and sharded variant for comparison")
    "config3s": dict(N=1_250_000, D=4096, V=128_000, max_n=5, quant="int4", B=256, L=2048, tier="sharded",
                     desc="hidden 4096, 10M f-grams (1.25M per GPU), INT4 g128 cache row-sharded by id % W, batch 256x2048 per GPU"),
    # N is capped by the box's host RAM (pinned); 200 M rows need 416 GB
    "config5": dict(N=200_000_000, D=2048, V=128_000, max_n=5, quant="int8", B=256, L=2048, tier="host",
                    desc="hidden 2048, 200M f-grams, INT8 cache in pinned host RAM read zero-copy (TMA bulk over the host link), batch 256x2048"),
}
N_BATCHES = 8          # distinct id batches rotated through the timed steps (rows touched >> L2)
METRIC = "tokens/sec embedded"
NVLINK_PEAK_GBS = 770.0    # B200_PROFILING.md: measured peer copy, per direction per GPU
HOST_LINK_PEAK_GBS = 64.0  # nominal PCIe Gen5 x16 per direction


def row_bytes_algorithmic(quant: str, D: int, group: int = 128) -> int:
    return {"fp32": 4 * D, "fp16": 2 * D, "int8": D + 4, "int4": D // 2 + 2 * D // group}[quant]


def bytes_per_token(w, hit: float, probes: float, slot_bytes: int = 32) -> float:
    """SURVEY.md 8d: id in + probed slots + hit row / fallback row + output + (id, len) out.  `slot_bytes` is the slot
    format the index actually built (32, or 16 for the compact format; the survey's own figure is 16)."""
    D = w["D"]
    return 8 + slot_bytes * probes + hit * row_bytes_algorithmic(w["quant"], D) + (1 - hit) * 2 * D + 2 * D + 5


def measured_peak_hbm():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 100 ms while the timed region runs.  `wait_first()` blocks until
    the first sample has arrived, so that a short timed region still has a record."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu, self.f, self.p = gpu_index, None, None

    def __enter__(self):
        try:
            self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
            self.p = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                                       "-i", str(self.gpu)], stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None
        return self

    def _rows(self):
        try:
            return [r.split(",") for r in open(self.f.name).read().strip().splitlines() if r.count(",") >= 8]
        except Exception:
            return []

    def wait_first(self, timeout_s: float = 3.0):
        t0 = time.time()
        while self.p is not None and not self._rows() and time.time() - t0 < timeout_s:
            time.sleep(0.02)

    def __exit__(self, *a):
        if self.p is not None:
            self.p.terminate()
            try:
                self.p.wait(timeout=5)
            except Exception:
                self.p.kill()

    def summary(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.f is None:
            return out
        try:
            self.f.flush()
            rows = self._rows()
            os.unlink(self.f.name)
        except Exception:
            return out
        sm = sorted(float(r[1]) for r in rows if r[1].strip().replace(".", "").isdigit())
        if sm:
            out["sm_mhz"] = sm[len(sm) // 2]
            out["sm_max_mhz"] = float(rows[0][2])
        out["samples"] = len(rows)
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        out["reasons"] = [n for k, n in enumerate(names) if any("Active" in r[5 + k] and "Not" not in r[5 + k] for r in rows)]
        return out


# ------------------------------------------------------------------------------------------------------------
# CPU arms (the ONLY place bench.py touches oracle/, besides the in-run parity check of the sharded tier)
# ------------------------------------------------------------------------------------------------------------
_CPU = {}


def _cpu_rows(rows):
    """fork-pool worker: oracle port of the reference path on some batch rows."""
    from oracle import py_oracle as po
    s = _CPU
    out, fid, ml = po.embed_forward(s["g2i"], s["max_n"], s["table"], s["base_bits"], s["ids"][rows], "bf16")
    return int(out.shape[0] * out.shape[1]), int((fid >= 0).sum())


def cpu_setup(w, seed_rank=0):
    """Same construction as the GPU arm (same generators, run on the CPU device) at min(N, 2M) f-grams: Python
    dict probes are size-independent (SURVEY.md section 6) and the dict costs ~360 B / f-gram."""
    import numpy as np
    from oracle import py_oracle as po
    from scone_b200.utils import synthetic as S
    N = min(w["N"], 2_000_000)
    toks, lens, longest = S.make_vocab_device(N, w["max_n"], w["V"], seed=0, device="cpu", return_longest=True)
    ids = S.make_stream_device(toks, lens, w["B"], w["L"], w["V"], seed=100 + seed_rank, p_plant=1.0, pick_ids=longest).numpy()
    toks, lens = toks.numpy(), lens.numpy()
    g2i = {tuple(r[:n]): i for i, (r, n) in enumerate(zip(toks.tolist(), lens.tolist()))}
    rng = np.random.default_rng(2)
    # one quantised 65 536-row block tiled over the table: same footprint and gather pattern as N independent rows
    D = w["D"]
    blk = po.OracleTable.from_fp32(rng.standard_normal((min(N, 65536), D), dtype=np.float32) * np.float32(0.02), w["quant"])
    reps = (N + 65535) // 65536
    payload = np.tile(blk.payload, (reps, 1))[:N]
    scales = None if blk.scales is None else np.tile(blk.scales, (reps,) + (1,) * (blk.scales.ndim - 1))[:N]
    table = po.OracleTable(w["quant"], D, payload, scales)
    base_bits = po.cast_bits(rng.standard_normal((w["V"], D), dtype=np.float32) * np.float32(0.02), "bf16")
    _CPU.update(toks=toks, lens=lens)
    _CPU.update(g2i=g2i, max_n=w["max_n"], table=table, base_bits=base_bits, ids=ids, N=N)
    return N


def cpu_time_rows(rows_per_step, cores):
    """One CPU step over `rows_per_step` batch rows; returns (seconds, tokens)."""
    import numpy as np
    B = _CPU["ids"].shape[0]
    rows = np.arange(rows_per_step) % B
    t0 = time.perf_counter()
    if cores == 1:
        tok, _ = _cpu_rows(rows)
    else:
        parts = [p for p in np.array_split(rows, cores) if len(p)]
        tok = sum(t for t, _ in _CPU["pool"].map(_cpu_rows, parts))
    return time.perf_counter() - t0, tok


def run_reference(args, w, rank, world):
    """--impl reference: the CPU port, all host cores, bounded sample per step."""
    if rank != 0:
        return
    import multiprocessing as mp
    cores = os.cpu_count() or 1
    N = cpu_setup(w)
    _CPU["pool"] = mp.get_context("fork").Pool(cores) if cores > 1 else None
    B = w["B"]
    # size the per-step sample so the whole run stays within ~2 minutes
    dt, tok = cpu_time_rows(min(B, cores), cores)
    per_row = dt / max(1, min(B, cores))
    budget = 120.0 / max(1, args.steps + args.warmup)
    rows_per_step = int(max(1, min(B, budget / max(per_row, 1e-9))))
    for _ in range(args.warmup):
        cpu_time_rows(rows_per_step, cores)
    t_total, tok_total = 0.0, 0
    for _ in range(args.steps):
        dt, tok = cpu_time_rows(rows_per_step, cores)
        t_total += dt
        tok_total += tok
    if _CPU["pool"] is not None:
        _CPU["pool"].close()
    value = tok_total / t_total
    sample = f"{rows_per_step} of {B} batch rows x {w['L']} tokens per step; vocabulary {N} of {w['N']} f-grams (Python dict)"
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "tokens/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * t_total / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": f"{w['quant']}->bf16", "data": "synthetic",
        "config": {"workload": w["desc"], "f_grams": w["N"], "dim": w["D"], "max_n": w["max_n"], "quant": w["quant"],
                   "batch": [w["B"], w["L"]], "sample": sample},
        "cpu_baseline": {"value": value, "unit": "tokens/s", "cores": cores, "kind": "port", "sample": sample,
                         "what": "oracle/py_oracle.py embed_forward: dict probes n=max_n..1 + numpy gather/dequant/cast"},
        "e2e": {"value": value, "unit": "tokens/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------------------
# GPU arm, table resident on one GPU (configs 1-3; replicas at N > 1)
# ------------------------------------------------------------------------------------------------------------

def _fill_cache(cache, N, D, seed=2, std=0.02, chunk_bytes=1 << 30):
    """Random N(0, std^2) rows generated on the device and stored through the drop-in's own cache_embeddings (which
    quantises them on the GPU), one chunk at a time."""
    import torch
    gen = torch.Generator(device=cache.device)
    gen.manual_seed(seed)
    chunk = max(1, chunk_bytes // (4 * D))
    for s in range(0, N, chunk):
        k = min(chunk, N - s)
        rows = torch.randn((k, D), generator=gen, device=cache.device, dtype=torch.float32) * std
        cache.cache_embeddings(range(s, s + k), rows, verbose=False)


DUMP_EMBED_BYTES = 32 << 20     # float32 embeddings sample; the whole dump of config1..config3 stays under 64 MB


def _snapshot_outputs(out, out_id, out_len):
    """Device copies of a lookup's results, taken before the buffers are reused: fgram_id and match_len whole, the
    embeddings at the fixed, seeded sample of positions described in the module docstring."""
    import numpy as np
    import torch
    T, D = out_id.numel(), out.shape[-1]
    n = min(T, DUMP_EMBED_BYTES // (4 * D))
    pos = np.sort(np.random.default_rng(0).choice(T, size=n, replace=False))
    return {"embeddings": out.view(T, D)[torch.from_numpy(pos).to(out.device)],
            "fgram_id": out_id.clone(), "match_len": out_len.clone()}


def _dump_outputs(snap, out_dir):
    import numpy as np
    import torch
    os.makedirs(out_dir, exist_ok=True)
    for name, t in snap.items():
        a = t.cpu().to(torch.float64 if name == "fgram_id" else torch.float32)    # exact: bf16, int32 and uint8 values
        np.save(os.path.join(out_dir, name + ".npy"), a.numpy())


def run_ours(args, w, rank, local_rank, world, name, dump_dir=None):
    """Returns the JSON line (a dict) on rank 0, None elsewhere.  Leaves the process group alive.  With `dump_dir`, rank 0
    writes the results of the last timed step there (see the module docstring)."""
    import numpy as np
    import torch
    import torch.distributed as dist

    import scone_b200 as sb
    from scone_b200 import _lib
    from scone_b200.utils import synthetic as S

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- scone_b200 has no CPU path (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1 and not dist.is_initialized():
        dist.init_process_group("nccl", device_id=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        if world > 1:
            t = torch.tensor([x], device=dev, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            return float(t.item())
        return x

    B, L, D, N, V = w["B"], w["L"], w["D"], w["N"], w["V"]
    T = B * L
    steps = args.steps
    # ---- build (untimed): the drop-in objects -- extractor (vocabulary + device index), cache (table), fallback rows ----
    toks, lens, longest = S.make_vocab_device(N, w["max_n"], V, seed=0, device=dev, return_longest=True)
    ex = sb.NGramExtractor.from_arrays(toks.cpu().numpy(), lens.cpu().numpy(), device=dev)
    index = ex.device_index(dev)
    cache = sb.EmbeddingCache(ex, D, quant=w["quant"], out_dtype=torch.bfloat16, device=dev)
    _fill_cache(cache, N, D)
    table = cache.table
    base = S.make_base_device(V, D, torch.bfloat16, seed=3, device=dev)
    cache.set_base_embedding(base)
    if args.id_dist == "zipf":
        # secondary workload (SURVEY.md 8d): planted f-gram ids follow a Zipf-like law instead of being uniform over the
        # table, so hot rows hit L2 and the algorithmic GB/s exceeds the DRAM GB/s
        gen = torch.Generator(device=dev)
        gen.manual_seed(7)
        ranks = S.zipf_like_torch(gen, (8 * T,), longest.numel(), dev)
        longest = longest[ranks]
    batches = [S.make_stream_device(toks, lens, B, L, V, seed=100 + rank * N_BATCHES + k, p_plant=1.0, pick_ids=longest)
               for k in range(N_BATCHES)]
    del toks, lens
    out = torch.empty((B, L, D), dtype=torch.bfloat16, device=dev)
    out_id = torch.empty((B, L), dtype=torch.int32, device=dev)
    out_len = torch.empty((B, L), dtype=torch.uint8, device=dev)
    stable = not args.no_inputs_stable

    def step(k):
        # the id batches are static inputs and the table does not change: SCONE_EMBED_INPUTS_STABLE holds
        cache.lookup(batches[k % N_BATCHES], out=out, out_id=out_id, out_len=out_len, inputs_stable=stable)

    # hit rate / probe count of the workload (for the algorithmic byte count)
    hits = 0
    for k in range(N_BATCHES):
        step(k)
        hits += int((out_id >= 0).sum().item())
    hit = hits / (N_BATCHES * T)
    probes = bin(index.len_mask).count("1")

    # ---- device-resident timing: K steps captured into one CUDA graph, replayed once ---------------------------
    stream = torch.cuda.Stream(device=dev)
    with torch.cuda.stream(stream):
        for k in range(max(3, args.warmup)):
            step(k)
        stream.synchronize()
        launches0 = _lib.launch_count()
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph, stream=stream):
            for k in range(steps):
                step(k)
        gpu_launches = _lib.launch_count() - launches0
        graph.replay()                       # one untimed replay (graph upload)
        stream.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        graph.replay()
        e1.record(stream)
        stream.synchronize()
        reps = max(1, min(400, int(0.4 / max(1e-5, e0.elapsed_time(e1) * 1e-3))))   # keep the GPU busy ~0.4 s either side for the clock samples
        barrier()
        with ClockSampler(local_rank) as clocks:
            clocks.wait_first()
            for _ in range(reps):
                graph.replay()
            stream.synchronize()
            e0.record(stream)
            graph.replay()
            e1.record(stream)
            stream.synchronize()
            barrier()
            ms = e0.elapsed_time(e1)
            # the results of the timed replay's last step; the replays and e2e steps below overwrite the buffers
            snap = _snapshot_outputs(out, out_id, out_len) if dump_dir else None
            repeats = []
            for _ in range(4):                       # variance only; `value` is the ONE timed replay above
                r0, r1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                r0.record(stream)
                graph.replay()
                r1.record(stream)
                stream.synchronize()
                repeats.append(r0.elapsed_time(r1) / steps)
            for _ in range(reps):
                graph.replay()
            stream.synchronize()
        clk = clocks.summary()
        # one launch at a time (nothing before it on the stream to overlap with): what a lone lookup costs
        g1 = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g1, stream=stream):
            step(0)
        iso = []
        for _ in range(12):
            r0, r1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            stream.synchronize()
            r0.record(stream)
            g1.replay()
            r1.record(stream)
            stream.synchronize()
            iso.append(r0.elapsed_time(r1))
        isolated_ms = sorted(iso)[len(iso) // 2]
    ms = max_over_ranks(ms)
    assert cache.status() == 0
    value = world * T * steps / (ms * 1e-3)
    kernel_ms = ms / steps

    # ---- e2e: host ids -> the drop-in class -> match result back on the host, every step -----------------------------
    h_ids = [b.cpu().pin_memory() for b in batches]
    h_id = torch.empty((B, L), dtype=torch.int32).pin_memory()
    h_len = torch.empty((B, L), dtype=torch.uint8).pin_memory()
    d_ids = torch.empty((B, L), dtype=torch.int64, device=dev)

    def e2e_step(k, h_emb=None):
        d_ids.copy_(h_ids[k % N_BATCHES], non_blocking=True)
        cache.lookup(d_ids, out=out, out_id=out_id, out_len=out_len)          # EmbeddingCache.lookup(): the call a user makes
        h_id.copy_(out_id, non_blocking=True)
        h_len.copy_(out_len, non_blocking=True)
        if h_emb is not None:
            h_emb.copy_(out, non_blocking=True)
        torch.cuda.current_stream().synchronize()            # the caller has its results

    def time_e2e(n_steps, h_emb=None):
        for k in range(3):
            e2e_step(k, h_emb)
        barrier()
        t0 = time.perf_counter()
        for k in range(n_steps):
            e2e_step(k, h_emb)
        dt = time.perf_counter() - t0
        barrier()
        return world * T * n_steps / max_over_ranks(dt)

    sync_value = time_e2e(steps)

    # the throughput form of the same call: EmbeddingCache.host_pipeline() multi-buffers the batches, so the H2D copy of
    # batch k+1 and the D2H read of batch k-1 run under batch k's kernel.  Every step still copies its own ids from pinned
    # host memory and lands its own match result in pinned host memory inside the timed region.
    def time_pipelined():
        pipe = cache.host_pipeline((B, L))
        for k in range(max(3, args.warmup)):
            pipe.submit(h_ids[k % N_BATCHES])
        pipe.flush()
        barrier()
        t0 = time.perf_counter()
        n_done = 0
        for k in range(steps):
            if pipe.submit(h_ids[k % N_BATCHES]) is not None:
                n_done += 1
        n_done += len(pipe.flush())
        dt = time.perf_counter() - t0
        barrier()
        assert n_done == steps
        pipe.close()
        return world * T * steps / max_over_ranks(dt)

    pipe_value = time_pipelined()
    h_emb = torch.empty((B, L, D), dtype=torch.bfloat16).pin_memory()
    to_host_value = time_e2e(steps, h_emb)
    del h_emb
    e2e = {"value": max(pipe_value, sync_value), "unit": "tokens/s", "h2d_bytes_per_step": T * 8, "d2h_bytes_per_step": T * 5,
           "api": "EmbeddingCache.host_pipeline() (pipelined) / EmbeddingCache.lookup() (synchronous)",
           "mode": "pipelined (4 slots, up to 3 batches in flight)" if pipe_value >= sync_value else "synchronous call per step",
           "pipelined": pipe_value, "synchronous": sync_value,
           "embeds_to_host": {"value": to_host_value, "unit": "tokens/s", "d2h_bytes_per_step": T * 5 + T * D * 2, "steps": steps,
                              "note": "synchronous lookup() per step with the [B, L, D] embeddings ALSO copied to pinned host memory: "
                                      "host-link bound"},
           "note": "ids from pinned host memory; fgram_id + match_len read back to pinned host memory every step; the embeddings "
                   "stay in HBM for the transformer, as with the reference's get_embeddings(ids, device). `synchronous` = one "
                   "blocking lookup per step (copy in, kernel, copy out, stream sync)"}

    if rank != 0:
        return None
    if snap is not None:
        _dump_outputs(snap, dump_dir)

    # ---- in-run parity: two rows of batch 0 through the drop-in class against the oracle ---------------------------------
    parity = None
    if not args.no_parity:
        try:
            from oracle import py_oracle as po
            from oracle.c_oracle import COracleIndex
            t0 = time.perf_counter()
            o2, i2, l2 = cache.lookup(batches[0][:2].contiguous())
            q = batches[0][:2].cpu().numpy()
            wid, wlen = COracleIndex(*ex.vocab_arrays()).match(q, nthreads=min(16, os.cpu_count() or 1))
            hitm = wid >= 0
            rows = table.storage[torch.from_numpy(wid[hitm].astype(np.int64)).to(dev)].cpu().numpy()
            so = table.scale_offset
            tab = {"int8": lambda: po.OracleTable("int8", D, rows[:, :D].view(np.int8), rows[:, so:so + 4].copy().view(np.float32)[:, 0]),
                   "fp16": lambda: po.OracleTable("fp16", D, rows[:, :2 * D].view(np.float16)),
                   "fp32": lambda: po.OracleTable("fp32", D, rows[:, :4 * D].view(np.float32)),
                   "int4": lambda: po.OracleTable("int4", D, rows[:, :D // 2], rows[:, so:so + 2 * (D // table.group)].copy().view(np.float16), table.group)}[w["quant"]]()
            want = np.empty(q.shape + (D,), dtype=np.uint16)
            want[~hitm] = base.view(torch.int16).cpu().numpy().view(np.uint16)[q[~hitm]]
            want[hitm] = po.cast_bits(tab.rows_fp32(np.arange(rows.shape[0])), "bf16")
            ok = np.array_equal(wid, i2.cpu().numpy()) and np.array_equal(wlen, l2.cpu().numpy()) \
                and np.array_equal(o2.view(torch.int16).cpu().numpy().view(np.uint16), want)
            parity = {"result": "ok" if ok else "MISMATCH", "positions_checked": int(q.size), "seconds": time.perf_counter() - t0,
                      "what": "fgram_id / match_len against oracle/c_oracle.c over the whole vocabulary, embeddings bit for bit against "
                              "py_oracle's dequant + cast of the stored rows (or the fallback rows)"}
        except Exception as e:
            parity = {"result": "error: " + repr(e)}

    # ---- roofline ---------------------------------------------------------------------------------------------
    bpt = bytes_per_token(w, hit, probes, slot_bytes=index.slot_bytes)
    peak, peak_src = measured_peak_hbm()
    achieved = bpt * T / (kernel_ms * 1e-3) / 1e9
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": None, "peak_source": peak_src, "kernel": "embed_bulk_kernel (fused match+gather+dequant+fallback)", "slot_bytes": index.slot_bytes,
                "bytes_per_token": bpt, "hit_rate": hit, "probes_per_token": probes, "kernel_ms": kernel_ms,
                "isolated_kernel_ms": isolated_ms, "isolated_frac": bpt * T / (isolated_ms * 1e-3) / 1e9 / peak,
                "note": "kernel_ms = back-to-back launches (the K-step graph; consecutive launches overlap through programmatic dependent "
                        "launch" + (" + SCONE_EMBED_INPUTS_STABLE" if stable else "") + "); isolated_kernel_ms = one launch with an idle GPU before it"}
    prof = os.path.join(ROOT, "profiles", f"traffic_{name}.json")
    if os.path.exists(prof):
        try:
            roofline["traffic"] = json.load(open(prof))["dram_bytes_per_launch"]
        except Exception:
            pass

    # ---- CPU baseline (rank 0, N = 1 only): bounded sample of the same workload -----------------------------------
    cpu_baseline = None
    if world == 1 and not args.no_cpu_baseline:
        Ncpu = cpu_setup(w)
        cpu_time_rows(1, 1)
        dt, tok, passes = 0.0, 0, 0
        while dt < 10.0 and passes < 64:             # ~10 s of single-thread CPU work over whole batches
            d1, t1 = cpu_time_rows(B, 1)
            dt, tok, passes = dt + d1, tok + t1, passes + 1
        cpu_baseline = {"value": tok / dt, "unit": "tokens/s", "cores": 1, "kind": "port",
                        "sample": f"{passes} passes over the {B} x {L} batch ({dt:.1f} s); vocabulary {Ncpu} of {N} f-grams (Python dict)",
                        "what": "oracle/py_oracle.py embed_forward (Python port of the reference path), single thread"}
        try:
            from oracle.c_oracle import COracleIndex
            from scone_b200.utils.synthetic import pack_table_numpy
            tb = _CPU["table"]
            cix = COracleIndex(_CPU["toks"], _CPU["lens"])
            packed, stride, soff = pack_table_numpy(w["quant"], tb.payload, tb.scales)
            cores = os.cpu_count() or 1
            obuf = np.empty((B, L, D), np.uint16)
            cix.embed(w["quant"], D, 128, packed, stride, packed[:, soff:] if soff else None, stride, _CPU["base_bits"],
                      _CPU["ids"][:1], "bf16", nthreads=1)
            t0 = time.perf_counter()
            cix.embed(w["quant"], D, 128, packed, stride, packed[:, soff:] if soff else None, stride, _CPU["base_bits"],
                      _CPU["ids"], "bf16", nthreads=cores, out=obuf)
            dtc = time.perf_counter() - t0
            cpu_baseline["c_port"] = {"value": T / dtc, "unit": "tokens/s", "cores": cores,
                                      "what": f"oracle/c_oracle.c, {cores} pthreads, one full batch"}
        except Exception as e:  # the C number is informational
            cpu_baseline["c_port"] = {"error": repr(e)}

    line = {
        "metric": METRIC, "value": value, "unit": "tokens/s", "n_gpus": world, "steps": steps, "warmup": max(3, args.warmup),
        "ms_per_step": kernel_ms, "ms_per_step_repeats": repeats, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": f"{w['quant']}->bf16", "data": "synthetic",
        "config": {"workload": w["desc"], "f_grams": N, "dim": D, "max_n": w["max_n"], "quant": w["quant"], "batch": [B, L],
                   "per_gpu_batch": [B, L], "parallelism": f"replicas x{world} (table fits one GPU; no data-path collective)",
                   "hit_rate": hit, "id_dist": args.id_dist, "index_bytes": index.bytes, "index_slot_bytes": index.slot_bytes,
                   "index_filter_bytes": index.filter_bytes, "table_bytes": table.bytes, "inputs_stable": stable,
                   "quant_note": "INT8 / INT4 row formats are defined by this repo (the reference keeps fp32 rows): parity for them is "
                                 "against oracle/py_oracle.py's formulas" if w["quant"] in ("int8", "int4") else None,
                   "l2": f"inputs > L2: {N_BATCHES} rotating id batches gather rows uniformly from a {table.bytes / 1e9:.2f} GB "
                         f"table and each step writes {T * D * 2 / 1e6:.0f} MB of output; no explicit flush",
                   "timing": "K steps captured in one CUDA graph, CUDA events on the launching stream, max over ranks"},
        "e2e": e2e, "gpu_launches": int(gpu_launches), "clocks": clk, "roofline": roofline, "parity": parity,
    }
    if cpu_baseline is not None:
        line["cpu_baseline"] = cpu_baseline
    return line


def _tile_fill(table, block_rows=65536, seed=2, keep_block=False):
    """Fill a (possibly huge) table by tiling one quantised random block: same footprint / access pattern as N independent
    rows at a fraction of the generation time (benchmark data only; parity tests use real tables).  Row r = block row
    r % block_rows."""
    import torch
    import scone_b200 as sb
    from scone_b200.utils import synthetic as S
    blk = sb.CacheTable(min(block_rows, table.num_rows), table.dim, table.quant, table.group, device=table.device)
    S.fill_table_device(blk, seed=seed)
    src = blk.storage
    for s0 in range(0, table.num_rows, src.shape[0]):
        k = min(src.shape[0], table.num_rows - s0)
        table.storage[s0:s0 + k].copy_(src[:k], non_blocking=True)
    torch.cuda.synchronize()
    return blk if keep_block else None


def _timed_steps(step, steps, warmup, barrier, dev, world, clocks=None, min_busy_s=0.5):
    """Eager steps timed with CUDA events, max over ranks.  With a clock sampler the GPU is kept busy for `min_busy_s`
    either side of the timed region so that the record holds samples taken under load."""
    import torch
    import torch.distributed as dist
    for k in range(max(3, warmup)):
        step(k)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    step(0)
    torch.cuda.synchronize()
    one = max(1e-4, time.perf_counter() - t0)
    if world > 1:                                 # every rank must run the same number of (possibly collective) steps
        t = torch.tensor([one], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        one = float(t.item())
    pad = int(min(200, max(1, min_busy_s / one))) if clocks is not None else 0
    if clocks is not None:
        clocks.wait_first()
    for k in range(pad):
        step(k)
    barrier()
    e0.record()
    for k in range(steps):
        step(k)
    e1.record()
    torch.cuda.synchronize()
    barrier()
    for k in range(pad):
        step(k)
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    if world > 1:
        t = torch.tensor([ms], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    return ms


# ------------------------------------------------------------------------------------------------------------
# Row-sharded tier (config 4): one build, both exchange variants, in-run parity
# ------------------------------------------------------------------------------------------------------------

def run_sharded(args, w, rank, local_rank, world, modes=("peer", "nccl"), parity=True):
    """Table row-sharded over the ranks (id % W).  Returns a dict (rank 0) with one entry per exchange variant:
    `peer` = rows pulled from peer memory over NVLink inside the fused kernel; `nccl` = two NCCL all-to-alls per step."""
    import numpy as np
    import torch
    import torch.distributed as dist
    import scone_b200 as sb
    from scone_b200 import _lib, sharded
    from scone_b200.utils import synthetic as S
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if not dist.is_initialized():
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        os.environ.setdefault("MASTER_PORT", "29533")
        dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)

    def barrier():
        dist.barrier()
        torch.cuda.synchronize()

    B, L, D, V = w["B"], w["L"], w["D"], w["V"]
    T = B * L
    steps = args.steps
    rows_per_gpu = args.rows_per_gpu or w["N"]
    N = rows_per_gpu * world
    t_build = time.perf_counter()
    toks, lens, longest = S.make_vocab_device(N, w["max_n"], V, seed=0, device=dev, return_longest=True)
    index = sb.FGramIndex(toks, lens)
    # the shard lives in symmetric memory mapped by every rank; the NCCL variant serves from the same local shard
    ptab = sharded.PeerShardedTable(N, D, w["quant"], device=dev)
    table = ptab.local
    blk = _tile_fill(table, keep_block=True)
    base = S.make_base_device(V, D, torch.bfloat16, seed=3, device=dev)
    batches = [S.make_stream_device(toks, lens, B, L, V, seed=100 + rank * N_BATCHES + k, p_plant=1.0, pick_ids=longest) for k in range(4)]
    # the vocabulary goes to the host on rank 0 only (the oracle of the parity check); every rank frees its device copy
    h_vocab = (toks.cpu().numpy(), lens.cpu().numpy()) if (parity and rank == 0) else None
    del toks, lens, longest
    torch.cuda.empty_cache()
    out = torch.empty((B, L, D), dtype=torch.bfloat16, device=dev)
    out_id = torch.empty((B, L), dtype=torch.int32, device=dev)
    out_len = torch.empty((B, L), dtype=torch.uint8, device=dev)
    status = torch.zeros(1, dtype=torch.int32, device=dev)
    fid, _ = index.lookup(batches[0])
    hit = float((fid >= 0).float().mean().item())
    n_hits = int((fid >= 0).sum().item())
    remote = int(((fid >= 0) & (fid % world != rank)).sum().item())
    del fid
    ptab.publish()
    build_s = time.perf_counter() - t_build
    peak, peak_src = measured_peak_hbm()
    probes = bin(index.len_mask).count("1")
    result = {"workload": w["desc"], "f_grams": N, "rows_per_gpu": rows_per_gpu, "dim": D, "max_n": w["max_n"], "quant": w["quant"],
              "per_gpu_batch": [B, L], "table_bytes_total": table.row_stride * N, "table_bytes_per_gpu": table.bytes,
              "index_bytes_per_gpu": index.bytes, "hit_rate": hit, "remote_fraction": remote / max(1, n_hits), "steps": steps,
              "build_seconds": build_s, "partitioning": "row id % W -> owner, id // W -> local row; index replicated on every GPU",
              "timing": "eager steps, CUDA events, barrier both sides, max over ranks"}
    outs = {}
    for mode in modes:
        if mode == "peer":
            def step(k):
                sharded.embed_forward_sharded(index, ptab, base, batches[k % 4], out=out, status=status, out_id=out_id, out_len=out_len)
            launches_per_step = 1
        else:
            cache = sharded.ShardedEmbeddingCache(sharded.CudaOps(index, table, base), micro_batches=args.nccl_micro)
            l0 = _lib.launch_count()
            cache.lookup(batches[0], out=out)
            launches_per_step = _lib.launch_count() - l0

            def step(k):
                cache.lookup(batches[k % 4], out=out)
        with ClockSampler(local_rank) as clocks:
            ms = _timed_steps(step, steps, args.warmup, barrier, dev, world, clocks=clocks)
        clk = clocks.summary()
        # batch 0 again: rows 0-1 of its output (embeddings, f-gram ids, match lengths) are what the parity check looks at
        if mode == "peer":
            step(0)
            s_id, s_len = out_id[:2].clone(), out_len[:2].clone()
        else:
            _, s_id, s_len = cache.lookup(batches[0], out=out)
            s_id, s_len = s_id[:2].clone(), s_len[:2].clone()
        torch.cuda.synchronize()
        outs[mode] = (out[:2].clone(), s_id, s_len)
        step_s = ms * 1e-3 / steps
        nv_in = remote * (table.row_stride + (4 if mode == "nccl" else 0)) / step_s / 1e9
        bpt = bytes_per_token(w, hit, probes, slot_bytes=index.slot_bytes)
        if mode == "nccl":
            bpt += hit * 2 * table.row_stride                    # NCCL variant: the served copy is written and read once more
        result[mode] = {
            "value": world * T / step_s, "unit": "tokens/s", "tokens_per_s_per_gpu": T / step_s, "ms_per_step": ms / steps,
            "gpu_launches_per_step": int(launches_per_step), "clocks": clk,
            "exchange": ("rows pulled from peer memory over NVLink inside the fused kernel (TMA bulk, no collective call)" if mode == "peer"
                         else f"NCCL: all-to-all of int32 row numbers, owner-side packed gather, all-to-all of packed rows, local dequant"
                              + (f"; software-pipelined over {args.nccl_micro} micro-batches of batch rows" if args.nccl_micro > 1 else "")),
            "nvlink": {"achieved_in_GBps_per_gpu": nv_in, "peak": NVLINK_PEAK_GBS, "frac": nv_in / NVLINK_PEAK_GBS,
                       "peak_source": "B200_PROFILING.md measured peer copy, per direction per GPU",
                       "bytes_in_per_step_per_gpu": remote * table.row_stride},
            "roofline": {"bound": "nvlink" if world > 1 else "hbm", "achieved": bpt * T / step_s / 1e9, "peak": peak, "unit": "GB/s",
                         "frac": bpt * T / step_s / 1e9 / peak, "traffic": None, "peak_source": peak_src, "bytes_per_token": bpt,
                         "note": "HBM bytes per GPU against the HBM peak; the binding resource at W > 1 is NVLink, see nvlink.frac"},
        }
    assert int(status.item()) == 0
    # ---- in-run parity: rows 0-1 of every rank's batch 0 against the oracle ------------------------------------------
    if parity:
        sample_ids = batches[0][:2].contiguous()
        g_ids = [torch.empty_like(sample_ids) for _ in range(world)]
        dist.all_gather(g_ids, sample_ids)
        gathered = {}
        for mode in modes:
            per = []
            for t_ in outs[mode]:
                g = [torch.empty_like(t_) for _ in range(world)]
                dist.all_gather(g, t_.contiguous())
                per.append(g)
            gathered[mode] = per
        if rank == 0:
            try:
                from oracle import py_oracle as po
                from oracle.c_oracle import COracleIndex
                t0 = time.perf_counter()
                cix = COracleIndex(*h_vocab)
                blk_h = blk.storage.cpu().numpy()
                base_h = base.view(torch.int16).cpu().numpy().view(np.uint16)
                ok, checked, bad = True, 0, []
                for r in range(world):
                    q = g_ids[r].cpu().numpy()
                    wid, wlen = cix.match(q, nthreads=min(16, os.cpu_count() or 1))
                    # expected rows: global id g lives on rank g % W at local row g // W = block row (g // W) % block_rows
                    hitm = wid >= 0
                    want = np.empty(q.shape + (D,), dtype=np.uint16)
                    want[~hitm] = base_h[q[~hitm]]
                    rows = blk_h[(wid[hitm].astype(np.int64) // world) % blk_h.shape[0]]
                    if w["quant"] == "fp16":
                        tab = po.OracleTable("fp16", D, rows[:, :2 * D].view(np.float16))
                    elif w["quant"] == "int8":
                        tab = po.OracleTable("int8", D, rows[:, :D].view(np.int8), rows[:, table.scale_offset:table.scale_offset + 4].copy().view(np.float32)[:, 0])
                    elif w["quant"] == "int4":
                        ng = D // table.group
                        tab = po.OracleTable("int4", D, rows[:, :D // 2], rows[:, table.scale_offset:table.scale_offset + 2 * ng].copy().view(np.float16), table.group)
                    else:
                        tab = po.OracleTable("fp32", D, rows[:, :4 * D].view(np.float32))
                    want[hitm] = po.cast_bits(tab.rows_fp32(np.arange(rows.shape[0])), "bf16")
                    for mode in modes:
                        g_emb, g_fid, g_len = gathered[mode]
                        got = g_emb[r].view(torch.int16).cpu().numpy().view(np.uint16)
                        if not (np.array_equal(wid, g_fid[r].cpu().numpy()) and np.array_equal(wlen, g_len[r].cpu().numpy())
                                and np.array_equal(got, want)):
                            ok = False
                            bad.append(f"rank {r} {mode}")
                    checked += q.size
                result["parity"] = "ok" if ok else "MISMATCH: " + ", ".join(bad)
                result["parity_detail"] = {"positions_checked_per_variant": checked, "ranks": world, "seconds": time.perf_counter() - t0,
                                           "what": "fgram_id / match_len of rows 0-1 of every rank's batch 0 against oracle/c_oracle.c built over "
                                                   "the whole vocabulary; their embeddings bit for bit against py_oracle's dequant + cast of the "
                                                   "owner's stored row (or the fallback row)"}
            except Exception as e:
                result["parity"] = "error: " + repr(e)
    del ptab, table, blk
    return result if rank == 0 else None


def sharded_line(args, w, res, world):
    """Stand-alone JSON line for `--workload config4 / config3s` (the peer-direct variant is the headline)."""
    head = res["peer"] if "peer" in res else res["nccl"]
    return {
        "metric": METRIC, "value": head["value"], "unit": "tokens/s", "n_gpus": world, "steps": res["steps"], "warmup": max(3, args.warmup),
        "ms_per_step": head["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": f"{w['quant']}->bf16", "data": "synthetic",
        "config": {k: res[k] for k in ("workload", "f_grams", "rows_per_gpu", "dim", "max_n", "quant", "per_gpu_batch", "table_bytes_total",
                                       "hit_rate", "remote_fraction", "partitioning", "timing")},
        "e2e": {"value": head["value"], "unit": "tokens/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0,
                "note": "same call; ids resident on the device"},
        "gpu_launches": head["gpu_launches_per_step"] * res["steps"], "clocks": head["clocks"], "roofline": head["roofline"],
        "nvlink": head["nvlink"], "sharded": res,
    }


# ------------------------------------------------------------------------------------------------------------
# Offloaded tier (config 5)
# ------------------------------------------------------------------------------------------------------------

def run_host(args, w, rank, local_rank, world):
    """config 5: the table lives in pinned host RAM and is read zero-copy by the same kernels."""
    import torch
    import scone_b200 as sb
    from scone_b200 import _lib
    from scone_b200.utils import synthetic as S
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    B, L, D, V = w["B"], w["L"], w["D"], w["V"]
    T = B * L
    steps = args.steps
    stride, _ = sb.table_layout(w["quant"], D)
    total_ram = os.sysconf("SC_PAGE_SIZE") * os.sysconf("SC_PHYS_PAGES")
    avail = total_ram
    try:
        for ln in open("/proc/meminfo"):
            if ln.startswith("MemAvailable:"):
                avail = int(ln.split()[1]) * 1024
    except Exception:
        pass
    budget = int(min(total_ram * (args.host_fraction or 0.5), avail * 0.7))
    N = int(min(w["N"], args.rows_per_gpu or (budget // stride)))
    t0 = time.perf_counter()
    table = sb.CacheTable(N, D, w["quant"], device=dev, tier="host")
    pin_s = time.perf_counter() - t0
    blk = sb.CacheTable(min(1 << 20, N), D, w["quant"], device=dev)
    S.fill_table_device(blk, seed=2)
    for s0 in range(0, N, blk.num_rows):
        k = min(blk.num_rows, N - s0)
        table.storage[s0:s0 + k].copy_(blk.storage[:k], non_blocking=True)
    torch.cuda.synchronize()
    del blk
    toks, lens, longest = S.make_vocab_device(N, w["max_n"], V, seed=0, device=dev, return_longest=True)
    index = sb.FGramIndex(toks, lens)
    base = S.make_base_device(V, D, torch.bfloat16, seed=3, device=dev)
    batches = [S.make_stream_device(toks, lens, B, L, V, seed=100 + k, p_plant=1.0, pick_ids=longest) for k in range(4)]
    h_vocab = (toks.cpu().numpy(), lens.cpu().numpy()) if not args.no_parity else None
    del toks, lens, longest
    out = torch.empty((B, L, D), dtype=torch.bfloat16, device=dev)
    out_id = torch.empty((B, L), dtype=torch.int32, device=dev)
    out_len = torch.empty((B, L), dtype=torch.uint8, device=dev)

    def step(k):
        sb.embed_forward(index, table, base, batches[k % 4], out=out, out_id=out_id, out_len=out_len)

    step(0)
    hit = float((out_id >= 0).float().mean().item())
    # in-run parity: two batch rows of batch 0 against the oracle (ids / lengths from the C oracle over the whole vocabulary, rows
    # from py_oracle's dequant of the host-resident bytes the kernel read)
    parity = None
    if h_vocab is not None:
        try:
            import numpy as np
            from oracle import py_oracle as po
            from oracle.c_oracle import COracleIndex
            t0 = time.perf_counter()
            q = batches[0][:2].cpu().numpy()
            wid, wlen = COracleIndex(*h_vocab).match(q, nthreads=min(16, os.cpu_count() or 1))
            hitm = wid >= 0
            rows = table.storage[torch.from_numpy(wid[hitm].astype(np.int64))].numpy()
            so = table.scale_offset
            tab = {"int8": lambda: po.OracleTable("int8", D, rows[:, :D].view(np.int8), rows[:, so:so + 4].copy().view(np.float32)[:, 0]),
                   "fp16": lambda: po.OracleTable("fp16", D, rows[:, :2 * D].view(np.float16)),
                   "fp32": lambda: po.OracleTable("fp32", D, rows[:, :4 * D].view(np.float32)),
                   "int4": lambda: po.OracleTable("int4", D, rows[:, :D // 2], rows[:, so:so + 2 * (D // table.group)].copy().view(np.float16), table.group)}[w["quant"]]()
            want = np.empty(q.shape + (D,), dtype=np.uint16)
            want[~hitm] = base.view(torch.int16).cpu().numpy().view(np.uint16)[q[~hitm]]
            want[hitm] = po.cast_bits(tab.rows_fp32(np.arange(rows.shape[0])), "bf16")
            got = out[:2].view(torch.int16).cpu().numpy().view(np.uint16)
            ok = np.array_equal(wid, out_id[:2].cpu().numpy()) and np.array_equal(wlen, out_len[:2].cpu().numpy()) and np.array_equal(got, want)
            parity = {"result": "ok" if ok else "MISMATCH", "positions_checked": int(q.size), "seconds": time.perf_counter() - t0}
            del h_vocab
        except Exception as e:
            parity = {"result": "error: " + repr(e)}
    l0 = _lib.launch_count()
    with ClockSampler(local_rank) as clocks:
        ms = _timed_steps(step, steps, args.warmup, torch.cuda.synchronize, dev, 1, clocks=clocks, min_busy_s=0.3)
    clk = clocks.summary()
    launches = _lib.launch_count() - l0
    step_s = ms * 1e-3 / steps
    link = hit * T * stride / step_s / 1e9
    # the staged variant of the same tier: host threads gather rows into pinned staging, cudaMemcpyAsync on a side stream
    staged_info = None
    if not args.no_staged:
        from scone_b200.offload import StagedHostLookup
        staged = StagedHostLookup(index, table, base, micro_batches=8, max_positions=T)
        staged.lookup(batches[0], out=out)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for k in range(steps):
            staged.lookup(batches[k % 4], out=out)
        torch.cuda.synchronize()
        st_s = (time.perf_counter() - t0) / steps
        staged_info = {"value": T / st_s, "unit": "tokens/s", "host_link_GBps": hit * T * stride / st_s / 1e9, "micro_batches": 8,
                       "host_threads": staged.threads, "ms_per_step": st_s * 1e3,
                       "note": "match on the GPU, host threads gather the rows into pinned staging, cudaMemcpyAsync on a side stream, "
                               "dequantising gather; bounded by the host-side gather"}
    line = {
        "metric": METRIC, "value": T / step_s, "unit": "tokens/s", "n_gpus": 1, "steps": steps, "warmup": max(3, args.warmup),
        "ms_per_step": ms / steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": f"{w['quant']}->bf16", "data": "synthetic",
        "config": {"workload": w["desc"], "f_grams": N, "f_grams_named": w["N"], "dim": D, "max_n": w["max_n"], "quant": w["quant"],
                   "batch": [B, L], "hit_rate": hit, "host_ram_bytes": total_ram, "host_ram_available_bytes": avail,
                   "table_bytes_host": table.bytes, "pin_seconds": pin_s,
                   "scaled": (f"N scaled from {w['N']} to {N} rows ({table.bytes / 1e9:.1f} GB pinned): the box has {total_ram / 1e9:.0f} GB of "
                              f"host RAM ({avail / 1e9:.0f} GB available)") if N < w["N"] else None,
                   "tier": "zero-copy: cp.async.bulk straight from pinned host memory into shared memory",
                   "l2": "rows come over the host link, never cached", "timing": "eager steps, CUDA events"},
        "e2e": {"value": T / step_s, "unit": "tokens/s", "h2d_bytes_per_step": int(hit * T * stride), "d2h_bytes_per_step": 0,
                "note": "the row bytes cross the host link inside the kernel (zero-copy)"},
        "gpu_launches": int(launches), "clocks": clk,
        "roofline": {"bound": "host_link", "achieved": link, "peak": HOST_LINK_PEAK_GBS, "unit": "GB/s", "frac": link / HOST_LINK_PEAK_GBS,
                     "traffic": None, "peak_source": "nominal PCIe Gen5 x16 per direction (host-link bound, not HBM)",
                     "host_link_GBps": link, "bytes_per_token_over_link": hit * stride},
        "staged": staged_info, "parity": parity,
    }
    return line


# ------------------------------------------------------------------------------------------------------------
# The suite
# ------------------------------------------------------------------------------------------------------------

def _child(args, name, extra=(), timeout_s=600):
    """Run one workload in a child process of this script (its own CUDA context: a failure or a large footprint there cannot
    take the headline line down) and return its parsed JSON line reduced to what the parent reports."""
    cmd = [sys.executable, os.path.abspath(__file__), "--workload", name, "--steps", str(args.steps), "--warmup", str(args.warmup),
           "--no-cpu-baseline"] + list(extra)
    t0 = time.perf_counter()
    try:
        p = subprocess.run(cmd, capture_output=True, text=True, timeout=timeout_s)
    except subprocess.TimeoutExpired:
        return {"error": f"timed out after {timeout_s} s"}
    wall = time.perf_counter() - t0
    lines = [ln for ln in p.stdout.strip().splitlines() if ln.startswith("{")]
    if p.returncode != 0 or not lines:
        return {"error": f"rc={p.returncode}", "stderr_tail": p.stderr[-600:]}
    d = json.loads(lines[-1])
    keep = {k: d.get(k) for k in ("value", "unit", "ms_per_step", "steps", "dtype", "gpu_launches", "clocks", "roofline", "e2e", "staged", "parity")
            if d.get(k) is not None}
    keep["config"] = d.get("config")
    keep["wall_seconds"] = wall
    return keep


def run_suite(args, rank, local_rank, world):
    t_start = time.perf_counter()
    line = run_ours(args, WORKLOADS["config2"], rank, local_rank, world, "config2", dump_dir=args.dump_outputs)
    if world == 1:
        if not args.no_configs:
            import torch
            torch.cuda.empty_cache()
            # the whole default run must end within a few minutes: each child gets what is left of `--suite-seconds`
            left = lambda: max(30.0, args.suite_seconds - (time.perf_counter() - t_start))
            configs = {}
            configs["config1"] = _child(args, "config1", timeout_s=min(180.0, left()))
            configs["config3"] = _child(args, "config3", timeout_s=min(300.0, left()))
            configs["config5"] = _child(args, "config5", timeout_s=min(400.0, left()))
            line["configs"] = configs
            line["suite_seconds"] = time.perf_counter() - t_start
        print(json.dumps(line), flush=True)
        return
    # N > 1: config 4, row-sharded over the ranks.  A watchdog prints the headline line without it if it cannot finish.
    import torch
    import torch.distributed as dist
    done = threading.Event()

    def watchdog():
        if not done.wait(args.sharded_timeout):
            if rank == 0:
                line["sharded"] = {"error": f"did not finish within {args.sharded_timeout} s"}
                print(json.dumps(line), flush=True)
            os._exit(0)

    if not args.no_configs:
        # config 3 is named "on 1 and 8xB200": its 21 GB table fits every GPU, so at N > 1 it is N replicas with their own batches
        t0 = time.perf_counter()
        try:
            c3 = run_ours(args, WORKLOADS["config3"], rank, local_rank, world, "config3") or {}
            c3 = {k: c3.get(k) for k in ("value", "unit", "ms_per_step", "steps", "dtype", "gpu_launches", "clocks", "roofline", "e2e", "parity",
                                         "config") if c3.get(k) is not None}
        except Exception as e:
            c3 = {"error": repr(e)}
        c3["wall_seconds"] = time.perf_counter() - t0
        if rank == 0:
            line["configs"] = {"config3": c3}
        import gc
        gc.collect()
    if not args.no_sharded:
        threading.Thread(target=watchdog, daemon=True).start()
        torch.cuda.empty_cache()
        try:
            res = run_sharded(args, WORKLOADS["config4"], rank, local_rank, world)
        except Exception as e:                      # every rank raises or none does for deterministic failures (OOM, bad argument)
            res = {"error": repr(e)}
        if rank == 0:
            line["sharded"] = res
    done.set()
    if rank == 0:
        print(json.dumps(line), flush=True)
    try:
        dist.destroy_process_group()
    except Exception:
        pass


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50, help="timed steps of every measurement, child configs included")
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="suite", choices=["suite"] + sorted(WORKLOADS))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-configs", action="store_true", help="suite at N = 1: skip the config 1 / 3 / 5 child runs")
    ap.add_argument("--no-sharded", action="store_true", help="suite at N > 1: skip the row-sharded config 4 part")
    ap.add_argument("--no-staged", action="store_true", help="config5: skip the staged variant")
    ap.add_argument("--no-parity", action="store_true", help="config5: skip the in-run check against the oracle")
    ap.add_argument("--no-inputs-stable", action="store_true", help="do not pass SCONE_EMBED_INPUTS_STABLE in the device-timed steps")
    ap.add_argument("--sharded-timeout", type=float, default=600.0, help="suite at N > 1: seconds the config 4 part may take")
    ap.add_argument("--suite-seconds", type=float, default=660.0, help="suite at N = 1: wall-clock budget shared by the child runs")
    ap.add_argument("--id-dist", default="uniform", choices=["uniform", "zipf"],
                    help="distribution of the planted f-gram ids over the table: uniform (primary, worst case for caches) or Zipf-like")
    ap.add_argument("--rows-per-gpu", type=int, default=0, help="config4/5: table rows per GPU (default: the named size / what host RAM allows)")
    ap.add_argument("--sharded-mode", default="both", choices=["both", "peer", "nccl"], help="config4: which exchange variants to run")
    ap.add_argument("--nccl-micro", type=int, default=1, help="config4, NCCL variant: micro-batches the two all-to-alls are pipelined over")
    ap.add_argument("--host-fraction", type=float, default=0.0, help="config5: fraction of host RAM to pin (default 0.5)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the results of the last timed step to DIR/*.npy (suite headline and config1..config3)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or WORKLOADS.get(args.workload, {}).get("tier")):
        ap.error("--dump-outputs applies to the GPU suite and to config1..config3")
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if world == 1 and args.gpus > 1 and args.impl == "ours":
        # launched without torchrun: re-exec under it so that one process drives each GPU
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={args.gpus}",
               "--master-addr", "127.0.0.1", "--master-port", str(29500 + os.getpid() % 2000), os.path.abspath(__file__)] + sys.argv[1:]
        raise SystemExit(subprocess.call(cmd))
    if args.impl == "reference":
        run_reference(args, WORKLOADS["config2" if args.workload == "suite" else args.workload], rank, world)
        return
    if args.workload == "suite":
        run_suite(args, rank, local_rank, world)
        return
    w = WORKLOADS[args.workload]
    if w.get("tier") == "sharded":
        modes = ("peer", "nccl") if args.sharded_mode == "both" else (args.sharded_mode,)
        res = run_sharded(args, w, rank, local_rank, world, modes=modes)
        if rank == 0:
            print(json.dumps(sharded_line(args, w, res, world)), flush=True)
        import torch.distributed as dist
        dist.destroy_process_group()
    elif w.get("tier") == "host":
        print(json.dumps(run_host(args, w, rank, local_rank, world)), flush=True)
    else:
        line = run_ours(args, w, rank, local_rank, world, args.workload, dump_dir=args.dump_outputs)
        if rank == 0:
            print(json.dumps(line), flush=True)
        if world > 1:
            import torch.distributed as dist
            dist.destroy_process_group()


if __name__ == "__main__":
    sys.dont_write_bytecode = True      # the tree may be read-only: the benchmark writes nothing into it
    main()

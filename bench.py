#!/usr/bin/env python
"""bench.py — wake_up latency (s) and H2D GB/s of the sleep/wake weight-movement path on B200.

  python bench.py [--gpus N] [--steps K] [--warmup W]            this repo's engine (C-ABI libfma_b200.so)
  python bench.py --impl reference [--gpus N] ...                the reference data path: vLLM's OWN
                                                                 CuMemAllocator.sleep / wake_up (the code the
                                                                 reference launcher triggers with POST /sleep,
                                                                 /wake_up), same tables, same box
  N > 1:  python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 \
              --master-port P bench.py --gpus N --steps K --warmup W

A "step" is one level-1 sleep -> wake_up round trip of one rank's model shard (weights offloaded,
kv_cache discarded and remapped): BASELINE.json config[1] (Llama-3-8B, 1xB200, host-DRAM tier) at N=1,
config[2] (Llama-3-70B TP=8 per-rank shard, every rank concurrently, no collective) at N>1.

  value          aggregate wake H2D GB/s = N*W / max_ranks(mean device time of the wake pipeline, CUDA events)
  e2e.value      aggregate wake GB/s    = N*W / max_ranks(mean wall time of the public wake call: cuMemCreate/Map of
                 weights AND kv_cache + H2D from the pinned host store + K2 scatter + sync) — what /wake_up costs
  roofline       K2 (TMA page scatter) launches inside the timed region vs the measured HBM copy peak
  pcie           e2e per-GPU GB/s vs the 64 GB/s PCIe Gen5 x16 figure north_star names
  cpu_baseline   the reference data path (vLLM CuMemAllocator) timed in the same run on this box (N=1, rank 0)
  packed_image   (N=1, extra evidence, own process) the same table filled with bf16 dummy weights, slept and woken with the
                 PACKED host image (K4 / K5: 0.758 of the bytes cross PCIe), then four cycles with INCREMENTAL sleep
                 (packed_image.incremental_sleep: the sleeps after the first move nothing); never part of `value` / `e2e`

  --contents bf16   fill both arms with bf16 U(-1e-3, 1e-3) (vLLM's dummy weights) instead of incompressible bytes
  --pack 1          this arm sleeps / wakes with the PACKED image (e2e.link_bytes_per_step = bytes that crossed the link)
  --incremental 1   sleeps whose weights still match the image in the host store release the device side without a copy
  --extras packed,incremental   (any N, opt-in) after the main line, on the same engines: bf16 refill, PACKED cycles, then
                    INCREMENTAL cycles, aggregated like the main line (reported under `extras`)
  --dump-outputs DIR   after the timed steps, write what the last wake restored (every weight segment's digest and a fixed
                    sample of the weight bytes) as DIR/*.npy, so that two builds can be compared output for output

Synthetic data: counter-based splitmix64 bytes (seed 1234 + rank); the working set (>= 15 GiB per rank) is far
larger than the 126 MB L2, so no L2 flush is needed between iterations.
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

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

GiB = 1 << 30
PCIE_GEN5_X16_GBS = 64.0      # north_star's PCIe roofline, per direction per GPU
NVLINK5_GBS = 900.0           # north_star's NVLink roofline, per direction per GPU
HBM_FALLBACK_GBS = 6650.0     # /opt/skills/guides/B200_PROFILING.md fallback


def hbm_peak() -> tuple[float, str]:
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return HBM_FALLBACK_GBS, "fallback (B200_PROFILING.md)"


def workload_for(n_gpus: int, override: str | None) -> str:
    if override:
        return override
    return "llama-3-8b" if n_gpus == 1 else "llama-3-70b-tp8"


# --------------------------------------------------------------------------------------------------
# clocks: sample nvidia-smi DURING the timed region (B200_PROFILING.md recipe)
# --------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu_index = gpu_index
        self.lines: list[str] = []
        self.proc = None
        self.thread = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", os.environ.get("FMA_BENCH_CLOCKS_MS", "250"), "-i", str(self.gpu_index)],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None
            return
        self.thread = threading.Thread(target=self._pump, daemon=True)
        self.thread.start()

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self) -> dict:
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, power, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for l in self.lines:
            f = [x.strip() for x in l.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2])); power.append(float(f[3]))
            except ValueError:
                continue
            for name, v in zip(names, f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(power) if power else None, "samples": len(sm), "reasons": sorted(reasons),
                "note": "PCIe-bound path: SMs only run the short K1/K2 page copies, so SM clocks are not the limiter"}


# --------------------------------------------------------------------------------------------------
# this repo's arm
# --------------------------------------------------------------------------------------------------
def run_ours(args) -> None:
    import torch

    import fma_b200
    from fma_b200 import _lib as L
    from fma_b200 import workloads as W

    from fma_b200 import ranks

    rank, world, local_rank = ranks.rank_env()
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit(f"--gpus {args.gpus} needs torchrun (python -m torch.distributed.run --nproc-per-node {args.gpus} ...)")
        args.gpus = world
    torch.cuda.set_device(local_rank)
    group = ranks.RankGroup(backend="nccl" if world > 1 else None)   # plumbing only: barrier + max/sum of timings
    barrier, max_over_ranks, sum_over_ranks = group.barrier, group.max, group.sum

    tier = {"host": L.FMA_TIER_HOST, "peer": L.FMA_TIER_PEER, "local": L.FMA_TIER_LOCAL}[args.tier]
    mode = {"auto": L.FMA_MODE_AUTO, "direct": L.FMA_MODE_DIRECT, "staged": L.FMA_MODE_STAGED, "kernel": L.FMA_MODE_KERNEL}[args.mode]
    kernel = {"tma": L.FMA_KERNEL_TMA, "ldg": L.FMA_KERNEL_LDG}[args.kernel]
    cfg = fma_b200.EngineConfig(mode=mode, kernel=kernel, copy_streams=args.copy_streams,
                                chunk_bytes=args.chunk_mib << 20, ring_slots=args.ring_slots, map_threads=args.map_threads,
                                pack=args.pack)
    eng = fma_b200.Engine(local_rank, cfg)
    if args.incremental:
        eng.set_option("incremental", 1)
    workload = workload_for(args.gpus, args.workload)
    table = W.allocation_table(workload, kv_cache_bytes=int(args.kv_gib * GiB))
    for s in table:
        eng.alloc(s.bytes, s.tag)
    Wb = W.weight_bytes(table)
    fill_weights(eng, table, ranks.shard_seed(rank), args.contents, torch)
    before = eng.digest_all(["weights"])    # K3
    if tier == L.FMA_TIER_HOST:
        eng.host_reserve(Wb)                # pre-pin off the critical path (the engine's load-time hook does this)
    elif tier == L.FMA_TIER_PEER:
        eng.peer_reserve(ranks.parking_device(local_rank, world), Wb)
    pin_s = eng.stats()["host_store_pin_seconds"]

    timelines = {}
    phase_barrier = group.phase_barrier

    def cycle(capture: bool = False):
        # Executor semantics (vllm:v1/executor/abstract.py:327,347): sleep / wake_up are fanned out to every rank and return
        # when ALL ranks are done -> no rank starts waking while another still sleeps.  Host-side hand-shake, no GPU work.
        phase_barrier()
        eng.sleep(["weights"], tier=tier)
        s1 = eng.stats()
        if capture:
            timelines["sleep"] = eng.timeline()
        phase_barrier()
        eng.wake(None)
        s2 = eng.stats()
        if capture:
            timelines["wake"] = eng.timeline()
        return s1, s2

    for _ in range(max(args.warmup, 0)):
        cycle()
    launches0 = eng.stats()["total_kernel_launches"]
    sampler = ClockSampler(local_rank) if rank == 0 and os.environ.get("FMA_BENCH_NO_CLOCKS") != "1" else None
    barrier(); torch.cuda.synchronize()
    if sampler:
        sampler.start()
    rows = []
    t0 = time.perf_counter()
    for i in range(args.steps):
        rows.append(cycle(capture=bool(args.timeline) and i == args.steps - 1))   # reading the timeline happens after the step's stats
    torch.cuda.synchronize(); barrier()
    t1 = time.perf_counter()
    if args.timeline:      # per-rank phase timeline of the last timed step (fma_timeline): which phase bounds the wake
        os.makedirs(args.timeline, exist_ok=True)
        with open(os.path.join(args.timeline, f"n{world}_rank{rank}.csv"), "w") as f:
            f.write("op,kind,idx,t0_ms,t1_ms,bytes\n")
            for op in ("sleep", "wake"):
                for r in timelines.get(op, []):
                    f.write(f"{r['op']},{r['kind']},{r['idx']},{r['t0_ms']:.3f},{r['t1_ms']:.3f},{r['bytes']}\n")
    clocks = sampler.stop() if sampler else ({"sm_mhz": None, "sm_max_mhz": None, "reasons": ["sampling disabled (FMA_BENCH_NO_CLOCKS=1)"]} if rank == 0 else None)
    launches = eng.stats()["total_kernel_launches"] - launches0

    after = eng.digest_all(["weights"])
    bit_exact = after == before
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, eng, table, after, f"_rank{rank}" if world > 1 else "")

    mean = lambda xs: sum(xs) / len(xs)
    k2_s = sum(r[1]["kernel_seconds"] for r in rows); k2_b = sum(r[1]["kernel_bytes"] for r in rows)
    k2_n = sum(r[1]["kernel_launches"] for r in rows)
    k1_s = sum(r[0]["kernel_seconds"] for r in rows); k1_b = sum(r[0]["kernel_bytes"] for r in rows)
    k1_n = sum(r[0]["kernel_launches"] for r in rows)

    # job-level latency of step k = the slowest rank of step k (the executor returns when every rank is done)
    wake_dev_steps = group.max_vec([r[1]["wake_copy_seconds"] for r in rows])
    wake_wall_steps = group.max_vec([r[1]["wake_seconds"] for r in rows])
    sleep_dev_steps = group.max_vec([r[0]["sleep_copy_seconds"] for r in rows])
    sleep_wall_steps = group.max_vec([r[0]["sleep_seconds"] for r in rows])
    wake_dev_med, wake_wall_med = statistics.median(wake_dev_steps), statistics.median(wake_wall_steps)
    wake_dev_m, wake_wall_m = mean(wake_dev_steps), mean(wake_wall_steps)
    sleep_dev_m, sleep_wall_m = mean(sleep_dev_steps), mean(sleep_wall_steps)
    sleep_wall_med = statistics.median(sleep_wall_steps)
    total_s = max_over_ranks(t1 - t0)
    W_total = sum_over_ranks(float(Wb))
    launches_total = int(sum_over_ranks(float(launches)))
    all_exact = group.all_true(bit_exact)
    map_s = max_over_ranks(mean([r[1]["wake_map_seconds"] for r in rows]))
    unmap_s = max_over_ranks(mean([r[0]["sleep_unmap_seconds"] for r in rows]))
    st = eng.stats()
    sum_store = sum_over_ranks(float(rows[-1][0]["image_store_bytes"]))   # bytes that crossed PCIe per step (== W unless packed)

    # Plain pinned cudaMemcpyAsync on THIS box/slot (nothing of ours): boxes of the pool differ by several GB/s, so at
    # N=1 the fraction of this ceiling says more about the engine than the fraction of the nominal 64 GB/s.
    ceiling = None
    if tier == L.FMA_TIER_HOST:
        try:
            barrier()
            ceiling = max_over_ranks(-pcie_ceiling_gbs(torch))   # min over ranks, via max of the negation
            ceiling = -ceiling
        except Exception:
            ceiling = None

    peer = None
    if args.peer_extra and world > 1 and tier == L.FMA_TIER_HOST:
        peer = measure_peer(eng, L, Wb, local_rank, world, barrier, max_over_ranks, before, steps=3)

    extras = None
    if ("packed" in args.extras or "incremental" in args.extras) and tier == L.FMA_TIER_HOST:
        extras = measure_extras(args, eng, L, table, Wb, rank, world, barrier, max_over_ranks, sum_over_ranks, torch, group)

    roundrobin = None
    if "roundrobin" in args.extras and world >= 2 and tier == L.FMA_TIER_HOST:
        roundrobin = measure_roundrobin(args, L, W, local_rank, rank, world, group, torch)

    if rank == 0:
        peak, peak_src = hbm_peak()
        achieved = (k2_b / k2_s / 1e9) if k2_s > 0 else None
        bytes_per_launch = int(k2_b / k2_n) if k2_n else 0
        traffic, traffic_src = None, None
        tp = os.path.join(ROOT, "profiles", "k2_traffic.json")
        if os.path.exists(tp):      # NOT measured in this run: the ncu --set full capture of the same kernel, kept under profiles/
            try:
                tj = json.load(open(tp))
                if abs(tj.get("algorithmic_bytes_per_launch", 0) - bytes_per_launch) <= 0.02 * max(bytes_per_launch, 1):
                    traffic = tj.get("dram_bytes_per_launch")
                    traffic_src = "profiles/k2_traffic.json: dram__bytes_read+write of one launch of this size under ncu --set full (kept capture, profiles/k2_full_r2.md; a constant, not measured in this run)"
                else:
                    traffic_src = "no ncu capture for this launch size (profiles/k2_traffic.json is for 512 MiB slots)"
            except Exception:
                traffic = None
        e2e_gbs = W_total / wake_wall_med / 1e9
        e2e_mean_gbs = W_total / wake_wall_m / 1e9
        link_peak = PCIE_GEN5_X16_GBS if tier == L.FMA_TIER_HOST else NVLINK5_GBS
        out = {
            "metric": "wake_h2d_gbs", "value": round(W_total / wake_dev_med / 1e9, 3), "unit": "GB/s",
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": round(total_s / args.steps * 1e3, 3), "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "u8", "data": "synthetic",
            "config": bench_config(args, workload, Wb, len(table), world, ["auto", "direct", "staged", "kernel"][st["mode"]],
                                   bool(st["image_packed"]) if args.pack else False),
            "aggregation": "value / e2e = whole-job bytes / MEDIAN over the K timed steps of the per-step job latency (max over ranks of that "
                           "step); the mean-based figures are value_mean / e2e.mean_gbs / wake_latency_s_mean",
            "value_mean": round(W_total / wake_dev_m / 1e9, 3),
            "wake_latency_s": round(wake_wall_med, 5), "wake_latency_s_mean": round(wake_wall_m, 5),
            "wake_latency_s_min_max": [round(min(wake_wall_steps), 5), round(max(wake_wall_steps), 5)],
            "wake_latency_s_steps": [round(x, 4) for x in wake_wall_steps],
            "sleep_latency_s": round(sleep_wall_med, 5), "sleep_latency_s_mean": round(sleep_wall_m, 5),
            "sleep_d2h_gbs": round(W_total / sleep_dev_m / 1e9, 3) if sleep_dev_m > 0 else None,   # None: incremental sleeps moved nothing
            "sleep_copy_ops_last": rows[-1][0]["copy_ops"], "sleep_bytes_copied_last": rows[-1][0]["sleep_bytes_copied"],
            "wake_map_s": round(map_s, 5), "sleep_unmap_s": round(unmap_s, 5), "host_pin_s_untimed": round(pin_s, 3),
            "bit_exact": bool(all_exact),
            "e2e": {"value": round(e2e_gbs, 3), "unit": "GB/s", "h2d_bytes_per_step": int(W_total),
                    "d2h_bytes_per_step": int(W_total), "mean_gbs": round(e2e_mean_gbs, 3),
                    "link_bytes_per_step": int(sum_store),
                    "api": "fma_wake() through the C-ABI: VMM remap of weights+kv_cache, H2D from the pinned host store, K2, sync"},
            "gpu_launches": launches_total,
            "roofline": {"bound": "hbm", "kernel": "fma_k_page_copy_tma (K2 scatter, wake)" if args.kernel == "tma" else "fma_k_page_copy_ldg (K2)",
                         "achieved": round(achieved, 1) if achieved else None, "peak": peak, "unit": "GB/s",
                         "frac": round(achieved / peak, 4) if achieved else None, "traffic": traffic, "traffic_source": traffic_src,
                         "launches": k2_n, "bytes_per_launch": bytes_per_launch,
                         "avg_launch_us": round(k2_s / k2_n * 1e6, 2) if k2_n else None, "peak_source": peak_src,
                         "k1_gather_achieved": round(k1_b / k1_s / 1e9, 1) if k1_s > 0 else None, "k1_launches": k1_n},
            "pcie" if tier == L.FMA_TIER_HOST else "nvlink": {
                "bound": "pcie_gen5_x16" if tier == L.FMA_TIER_HOST else "nvlink5",
                "achieved_per_gpu": round(e2e_gbs / world, 3), "device_timed_per_gpu": round(W_total / wake_dev_med / 1e9 / world, 3),
                "peak": link_peak, "unit": "GB/s", "frac": round(e2e_gbs / world / link_peak, 4),
                "naive_pinned_h2d_per_gpu": round(ceiling, 3) if ceiling else None,
                "vs_naive_pinned_h2d": round(e2e_gbs / world / ceiling, 4) if ceiling else None,
                "naive_note": "min over ranks of a plain 8 GiB cudaMemcpyAsync from a torch pin_memory buffer, all ranks at once "
                              "(no NUMA placement, best of 3): the box's sustained copy-engine rate on the slowest rank's link"},
            "clocks": clocks,
        }
        if peer:
            out["peer_tier"] = peer
        if extras:
            out["extras"] = extras
        if roundrobin:
            out["roundrobin_config5"] = roundrobin
        if world == 1:
            eng.close()   # everything above is measured: give the HBM and the pinned store back before the baseline / extra processes run
        if world == 1 and "swap" in args.extras and tier == L.FMA_TIER_HOST:
            out["swap_config4"] = measure_swap(args, L, W)
        if world == 1 and "multipath" in args.extras and tier == L.FMA_TIER_HOST and torch.cuda.device_count() > 1:
            out["multipath_wake"] = measure_multipath(args, L, W, cfg, workload, torch.cuda.device_count())
        if world == 1 and "scaling_base" in args.extras and tier == L.FMA_TIER_HOST and workload != args.scaling_workload:
            out["n1_on_scaling_workload"] = measure_scaling_base(args, L, W, cfg)
        if world == 1 and not args.no_cpu_baseline:
            out["cpu_baseline"] = reference_sample(args, workload)
        if world == 1 and args.packed_extra and not args.pack and tier == L.FMA_TIER_HOST:
            out["packed_image"] = packed_image_extra(args, workload)
        print(json.dumps(out), flush=True)
    eng.close()
    group.close()


def dump_outputs(out_dir: str, eng, table, digests: list[int], suffix: str, block: int = 4096, blocks: int = 2048) -> None:
    """What the last timed wake handed back to its caller: the weight segments' contents.  weights_digest.npy holds the K3 digest
    of every weight segment as (high, low) 32-bit halves in float64; weights_sample.npy holds the bytes of `blocks` 4 KiB blocks
    drawn with a fixed seed from all weight segments, as float32 (32 MiB).  Both are the same from run to run unless a build
    computes different bytes."""
    import numpy as np

    os.makedirs(out_dir, exist_ok=True)
    idx = [i for i, s in enumerate(table) if s.tag == "weights"]
    d = np.array([digests[i] for i in idx], dtype=np.uint64)
    np.save(os.path.join(out_dir, f"weights_digest{suffix}.npy"), np.stack([d >> np.uint64(32), d & np.uint64(0xFFFFFFFF)], axis=1).astype(np.float64))
    starts = np.cumsum([0] + [table[i].bytes // block for i in idx])        # first block of each weight segment
    picks = np.sort(np.random.default_rng(0).choice(int(starts[-1]), size=min(blocks, int(starts[-1])), replace=False))
    sample = np.empty((len(picks), block), dtype=np.float32)
    for row, b in enumerate(picks):
        k = int(np.searchsorted(starts, b, side="right")) - 1
        sample[row] = np.frombuffer(eng.read(idx[k], block, offset=int(b - starts[k]) * block), dtype=np.uint8)
    np.save(os.path.join(out_dir, f"weights_sample{suffix}.npy"), sample)


def bench_config(args, workload: str, weight_bytes: int, n_segments: int, world: int, mode: str, packed: bool) -> dict:
    """The `config` object of BOTH arms' JSON lines (the reference arm runs on this arm's config: same table, same kv_cache
    region, same contents; the engine-only knobs describe what this arm would use)."""
    return {"workload": f"{workload} level-1 sleep->wake, {args.tier} tier, per-rank shard, no collective",
            "weights_gib_per_rank": round(weight_bytes / GiB, 3), "kv_cache_gib_per_rank": args.kv_gib,
            "segments_per_rank": n_segments, "mode": mode,
            "kernel": args.kernel, "chunk_mib": args.chunk_mib or "default", "copy_streams": args.copy_streams or "default",
            "contents": "splitmix64 bytes (incompressible)" if args.contents == "prng" else "bf16 U(-1e-3, 1e-3) (vLLM dummy weights)",
            "pack": packed, "incremental_sleep": bool(args.incremental),
            "phases": "executor semantics: every rank finishes sleeping before any rank wakes (host-side barrier between the phases)",
            "l2": "working set >> 126 MB L2 (no flush needed)", "parallelism": f"{world} independent ranks"}


def load_model(eng, W, model: str, kv_gib: float, seed: int):
    table = W.allocation_table(model, kv_cache_bytes=int(kv_gib * GiB))
    for s in table:
        eng.alloc(s.bytes, s.tag)
    first = 0
    for i, s in enumerate(table):
        if s.tag == "weights":
            eng.fill(i, seed, first)
            first += s.bytes // 8
    return table, W.weight_bytes(table)


def measure_swap(args, L, W, cycles: int = 10) -> dict:
    """BASELINE config 4: Llama-3-8B <-> Mistral-7B under one owner on one B200.  `fma_swap` = sleep(out) || wake(in): the D2H of
    the outgoing model and the H2D of the incoming one use the two PCIe directions at once.  Beside it, the serial form (sleep,
    then wake: what two independent reconciles of the reference controller produce, SURVEY.md section 3.4).  Medians over `cycles`."""
    import fma_b200

    try:
        A, B = fma_b200.Engine(0), fma_b200.Engine(0)
        ma, mb = args.swap_models.split(",")
        _, wa = load_model(A, W, ma, args.extras_kv_gib, 1)
        _, wb = load_model(B, W, mb, args.extras_kv_gib, 2)
        A.host_reserve(wa); B.host_reserve(wb)
        da, db = A.digest_all(["weights"]), B.digest_all(["weights"])
        B.sleep(["weights"])
        serial, swap, d2h, h2d = [], [], [], []
        for i in range(cycles + 2):
            t0 = time.perf_counter(); A.sleep(["weights"]); B.wake(None); t_ab = time.perf_counter() - t0
            t0 = time.perf_counter(); B.sleep(["weights"]); A.wake(None); t_ba = time.perf_counter() - t0
            t0 = time.perf_counter(); A.swap_out_for(B, ["weights"]); s_ab = time.perf_counter() - t0
            sa, sb = A.stats(), B.stats()
            t0 = time.perf_counter(); B.swap_out_for(A, ["weights"]); s_ba = time.perf_counter() - t0
            if i >= 2:
                serial += [t_ab, t_ba]; swap += [s_ab, s_ba]
                d2h.append(wa / sa["sleep_copy_seconds"] / 1e9); h2d.append(wb / sb["wake_copy_seconds"] / 1e9)
        ok = A.digest_all(["weights"]) == da
        A.swap_out_for(B, ["weights"]); ok = ok and B.digest_all(["weights"]) == db
        A.close(); B.close()
        med = statistics.median
        return {"models": f"{ma} ({wa / GiB:.2f} GiB) <-> {mb} ({wb / GiB:.2f} GiB), {args.extras_kv_gib:g} GiB kv_cache each, 1xB200, host tier",
                "swap_s_median": round(med(swap), 4), "swap_s_min_max": [round(min(swap), 4), round(max(swap), 4)],
                "serial_sleep_then_wake_s_median": round(med(serial), 4), "serial_s_min_max": [round(min(serial), 4), round(max(serial), 4)],
                "speedup_vs_serial": round(med(serial) / med(swap), 3),
                "d2h_gbs_during_swap_median": round(med(d2h), 2), "h2d_gbs_during_swap_median": round(med(h2d), 2),
                "both_directions_gbs": round(med(d2h) + med(h2d), 2), "cycles": len(swap), "bit_exact": bool(ok)}
    except Exception as e:
        return {"error": str(e)[:300]}


def measure_multipath(args, L, W, cfg, workload: str, n_visible: int, cycles: int = 6) -> dict:
    """MULTI-PATH wake (fma_paths_set) at N=1 with idle peers on the box: the same table, host tier; helpers = GPUs 1..k lend their
    PCIe links, K2 on GPU 0 gathers their staging slots over NVLink.  The single-link ceiling (55.6 GB/s measured) stops applying."""
    import fma_b200

    try:
        eng = fma_b200.Engine(0, cfg)
        _, wb = load_model(eng, W, workload, args.kv_gib, 1234)
        before = eng.digest_all(["weights"])
        rows = []
        ks = [k for k in (1, 3, 7) if k < n_visible]
        plans = [(k, 128, 3) for k in ks] + ([(ks[-1], 64, 4)] if ks else [])
        for k, slot_mib, slots in plans:
            eng.set_paths(list(range(1, k + 1)), slot_bytes=slot_mib << 20, slots=slots)
            wakes, devs, sleeps = [], [], []
            for i in range(cycles + 1):
                eng.sleep(["weights"]); ss = eng.stats(); eng.wake(None); st = eng.stats()
                if i:
                    wakes.append(st["wake_seconds"]); devs.append(st["wake_copy_seconds"]); sleeps.append(ss["sleep_seconds"])
            tl = eng.timeline()
            chunks = {r["idx"]: r["bytes"] for r in tl if r["kind"] == "path_chunks"}
            local = {r["idx"]: r["bytes"] for r in tl if r["kind"] == "path_local"}
            med = statistics.median
            rows.append({"helpers": k, "paths": k + 1, "slot_mib": slot_mib, "slots": slots, "wake_latency_s": round(med(wakes), 5),
                         "wake_latency_s_min_max": [round(min(wakes), 5), round(max(wakes), 5)], "e2e_gbs": round(wb / med(wakes) / 1e9, 1),
                         "device_gbs": round(wb / med(devs) / 1e9, 1), "x_single_link_64": round(wb / med(wakes) / 1e9 / PCIE_GEN5_X16_GBS, 2),
                         "sleep_latency_s": round(med(sleeps), 5), "sleep_e2e_gbs": round(wb / med(sleeps) / 1e9, 1),
                         "gib_per_path_device": {str(d): round(b / GiB, 2) for d, b in sorted(chunks.items())},
                         "gib_numa_local_per_path_device": {str(d): round(b / GiB, 2) for d, b in sorted(local.items())}})
        eng.set_paths([])
        ok = eng.digest_all(["weights"]) == before
        eng.close()
        best = min(rows, key=lambda r: r["wake_latency_s"]) if rows else None
        return {"workload": workload, "weights_gib": round(wb / GiB, 3), "visible_gpus": n_visible, "rows": rows,
                "best": {k: best[k] for k in ("helpers", "slot_mib", "wake_latency_s", "e2e_gbs")} if best else None, "bit_exact": bool(ok),
                "note": "helpers are idle GPUs of the same box (BASELINE config 5's parking GPUs, or any N=1 deployment on an 8-GPU node)"}
    except Exception as e:
        return {"error": str(e)[:300]}


def measure_scaling_base(args, L, W, cfg, cycles: int = 6) -> dict:
    """N=1 on the workload the N>1 lines use (one Llama-3-70B TP=8 shard), so the 1 -> 2 -> 4 -> 8 curve has a same-table base
    (the main N=1 line is BASELINE config[1], the 8B table, whose W differs by 10 %)."""
    import fma_b200

    try:
        eng = fma_b200.Engine(0, cfg)
        _, wb = load_model(eng, W, args.scaling_workload, args.kv_gib, 1234)
        eng.host_reserve(wb)
        before = eng.digest_all(["weights"])
        wakes, devs = [], []
        for i in range(cycles + 2):
            eng.sleep(["weights"]); eng.wake(None); st = eng.stats()
            if i >= 2:
                wakes.append(st["wake_seconds"]); devs.append(st["wake_copy_seconds"])
        ok = eng.digest_all(["weights"]) == before
        eng.close()
        med = statistics.median
        return {"workload": f"{args.scaling_workload} shard (the N>1 table) on 1 GPU", "weights_gib": round(wb / GiB, 3),
                "value": round(wb / med(devs) / 1e9, 3), "e2e": round(wb / med(wakes) / 1e9, 3), "unit": "GB/s",
                "wake_latency_s": round(med(wakes), 5), "wake_latency_s_min_max": [round(min(wakes), 5), round(max(wakes), 5)],
                "cycles": len(wakes), "bit_exact": bool(ok)}
    except Exception as e:
        return {"error": str(e)[:300]}


def measure_roundrobin(args, L, W, local_rank, rank, world, group, torch, rounds: int = 3) -> dict | None:
    """BASELINE config 5: N/2 sleeping Llama-3-8B models parked in the idle GPUs' HBM over NVSwitch (rank r < N/2 parks on GPU
    r + N/2), woken round-robin (one at a time, the other GPUs idle) and then all at once.  Ranks >= N/2 only lend their HBM."""
    import fma_b200

    half = world // 2
    out = None
    try:
        eng = None
        if rank < half:
            eng = fma_b200.Engine(local_rank)
            _, wb = load_model(eng, W, args.swap_models.split(",")[0], args.extras_kv_gib, 4321 + rank)
            before = eng.digest_all(["weights"])
            eng.peer_reserve(local_rank + half, wb)
            eng.sleep(["weights"], tier=L.FMA_TIER_PEER)
        single, single_dev, together = [], [], []
        for rnd in range(rounds + 1):
            for turn in range(half):
                group.phase_barrier()
                t = d = 0.0
                if rank == turn:
                    eng.wake(None); st = eng.stats(); t, d = st["wake_seconds"], st["wake_copy_seconds"]
                    eng.sleep(["weights"], tier=L.FMA_TIER_PEER)
                t, d = group.max(t), group.max(d)
                if rnd:
                    single.append(t); single_dev.append(d)
        for rnd in range(rounds + 1):
            group.phase_barrier()
            t = 0.0
            if rank < half:
                eng.wake(None); t = eng.stats()["wake_seconds"]
            t = group.max(t)
            group.phase_barrier()
            if rank < half:
                eng.sleep(["weights"], tier=L.FMA_TIER_PEER)
            if rnd:
                together.append(t)
        ok = True
        if rank < half:
            eng.wake(None)
            ok = eng.digest_all(["weights"]) == before
            wbytes = float(wb)
            eng.peer_release(); eng.close()
        else:
            wbytes = 0.0
        ok = group.all_true(ok)
        w8 = group.max(wbytes)
        med = statistics.median
        out = {"models": half, "model": f"{args.swap_models.split(',')[0]} ({w8 / GiB:.2f} GiB)", "placement": f"rank r < {half} parks on GPU r + {half}",
               "roundrobin_wake_s_median": round(med(single), 5), "roundrobin_wake_s_min_max": [round(min(single), 5), round(max(single), 5)],
               "roundrobin_gbs_e2e": round(w8 / med(single) / 1e9, 1), "roundrobin_gbs_device": round(w8 / med(single_dev) / 1e9, 1),
               "frac_of_nvlink_900": round(w8 / med(single) / 1e9 / NVLINK5_GBS, 4), "wakes": len(single),
               "all_at_once_wake_s_median": round(med(together), 5), "all_at_once_aggregate_gbs": round(half * w8 / med(together) / 1e9, 1),
               "bit_exact": bool(ok)}
    except Exception as e:
        out = {"error": str(e)[:300]}
    return out


def fill_weights(eng, table, seed: int, contents: str, torch) -> None:
    """Synthetic weights.  "prng": counter-based splitmix64 bytes (K0, on the device) — incompressible, the default.
    "bf16": bf16 values ~ U(-1e-3, 1e-3), what vLLM's --load-format dummy fills parameters with
    (vllm:model_executor/model_loader/weight_utils.py:1451-1471); one 1 GiB block generated on the GPU is written to
    every segment at a rotating offset (contents repeat across segments: irrelevant for bandwidth, digests still bite)."""
    first = 0
    if contents == "prng":
        for i, s in enumerate(table):
            if s.tag == "weights":
                eng.fill(i, seed, first)
                first += s.bytes // 8
        return
    n = min(512 << 20, max(1 << 20, max(s.bytes for s in table if s.tag == "weights") // 2))   # values in the block (<= 1 GiB)
    gen = torch.Generator(device="cuda"); gen.manual_seed(seed)
    src = torch.empty(n, dtype=torch.bfloat16, device="cuda").uniform_(-1e-3, 1e-3, generator=gen)
    host = torch.empty(n, dtype=torch.bfloat16, pin_memory=True).copy_(src)
    del src
    blk = n * 2
    for i, s in enumerate(table):
        if s.tag != "weights":
            continue
        o = 0
        while o < s.bytes:
            start = ((i * 7919 + o // (2 << 20)) * (2 << 20)) % blk
            m = min(s.bytes - o, blk - start)
            eng.write_ptr(i, host.data_ptr() + start, m, offset=o)
            o += m
    del host


def packed_image_extra(args, workload: str) -> dict:
    """Extra evidence at N=1 (like peer_tier at N>1; never fails the main line): the same table filled with bf16 dummy
    weights, slept and woken with the PACKED host image (config.pack: K4 encodes, K5 decodes, 0.758 of the bytes cross
    PCIe).  Runs in its OWN process with a timeout so that nothing it does can disturb the numbers above."""
    cmd = [sys.executable, os.path.abspath(__file__), "--packed-child", "--workload", workload, "--kv-gib", str(args.kv_gib),
           "--steps", "5", "--warmup", "3"]
    try:
        r = subprocess.run(cmd, capture_output=True, text=True, timeout=240, env=dict(os.environ, FMA_BENCH_NO_CLOCKS="1"))
        for line in reversed(r.stdout.strip().splitlines()):
            if line.startswith("{"):
                return json.loads(line)
        return {"error": f"no result (rc {r.returncode}): {(r.stderr or r.stdout)[-300:]}"}
    except subprocess.TimeoutExpired:
        return {"error": "timed out after 240 s"}
    except Exception as e:
        return {"error": str(e)[:200]}


def run_packed_child(args) -> None:
    import torch

    import fma_b200
    from fma_b200 import _lib as L
    from fma_b200 import workloads as W

    torch.cuda.set_device(0)
    eng = fma_b200.Engine(0, fma_b200.EngineConfig(pack=1))
    workload = workload_for(1, args.workload)
    table = W.allocation_table(workload, kv_cache_bytes=int(args.kv_gib * GiB))
    for s in table:
        eng.alloc(s.bytes, s.tag)
    Wb = W.weight_bytes(table)
    fill_weights(eng, table, 1234, "bf16", torch)
    before = eng.digest_all(["weights"])
    eng.host_reserve(Wb)
    rows = []
    for i in range(args.warmup + args.steps):
        eng.sleep(["weights"]); s1 = eng.stats()
        eng.wake(None); s2 = eng.stats()
        if i >= args.warmup:
            rows.append((s1, s2))
    ok = eng.digest_all(["weights"]) == before
    # INCREMENTAL sleep on the same engine: the first sleep with the option on seeds the digests, the following ones find the
    # image they need already in the host store and move nothing (K3 digest + unmap only)
    inc = {}
    try:
        eng.set_option("incremental", 1)
        irows = []
        for i in range(4):
            eng.sleep(["weights"]); s1 = eng.stats()
            eng.wake(None); s2 = eng.stats()
            irows.append((s1, s2))
        inc = {"sleep_latency_s": [round(r[0]["sleep_seconds"], 5) for r in irows], "sleep_bytes_copied": [r[0]["sleep_bytes_copied"] for r in irows],
               "wake_latency_s": [round(r[1]["wake_seconds"], 5) for r in irows], "bit_exact": bool(eng.digest_all(["weights"]) == before),
               "note": "cycle 0 seeds the digests (full sleep); later sleeps are clean: nothing crosses the link"}
        eng.set_option("incremental", 0)
    except Exception as e:
        inc = {"error": str(e)[:200]}
    mean = lambda xs: sum(xs) / len(xs)
    wake = mean([r[1]["wake_seconds"] for r in rows]); wake_dev = mean([r[1]["wake_copy_seconds"] for r in rows])
    sleep = mean([r[0]["sleep_seconds"] for r in rows])
    stored = rows[-1][0]["image_store_bytes"]
    k5_s = sum(r[1]["kernel_seconds"] for r in rows); k5_b = sum(r[1]["kernel_bytes"] for r in rows)
    k4_s = sum(r[0]["kernel_seconds"] for r in rows); k4_b = sum(r[0]["kernel_bytes"] for r in rows)
    peak, _ = hbm_peak()
    print(json.dumps({
        "contents": "bf16 U(-1e-3, 1e-3) (vLLM dummy weights)", "image_packed": bool(rows[-1][0]["image_packed"]),
        "bit_exact": bool(ok), "weights_gib": round(Wb / GiB, 3), "stored_gib": round(stored / GiB, 3), "stored_frac": round(stored / Wb, 4),
        "wake_latency_s": round(wake, 5), "wake_latency_s_median": round(statistics.median([r[1]["wake_seconds"] for r in rows]), 5),
        "sleep_latency_s": round(sleep, 5),
        "e2e_effective_gbs": round(Wb / wake / 1e9, 3), "e2e_link_gbs": round(stored / wake / 1e9, 3),
        "device_effective_gbs": round(Wb / wake_dev / 1e9, 3),
        "k5_unpack_gbs": round(k5_b / k5_s / 1e9, 1) if k5_s > 0 else None, "k5_frac_of_hbm_peak": round(k5_b / k5_s / 1e9 / peak, 4) if k5_s > 0 else None,
        "k4_pack_gbs": round(k4_b / k4_s / 1e9, 1) if k4_s > 0 else None,
        "steps": args.steps, "warmup": args.warmup, "incremental_sleep": inc,
        "note": "effective = weight bytes restored / time; link = bytes that crossed PCIe / time (bounded by the link)"}), flush=True)
    eng.close()


def pcie_ceiling_gbs(torch, nbytes: int = 8 << 30, reps: int = 2) -> float:
    """Plain H2D of one large pinned buffer on this rank's GPU, all ranks at the same time: 8 GiB per copy (about 0.15 s — long enough
    to be the link's SUSTAINED rate; round 1 used 2 GiB bursts, which flatter a link whose long-run rate is lower), best of `reps`."""
    try:
        h = torch.empty(nbytes, dtype=torch.uint8, pin_memory=True)
    except Exception:
        nbytes = 2 << 30
        h = torch.empty(nbytes, dtype=torch.uint8, pin_memory=True)
    d = torch.empty(nbytes, dtype=torch.uint8, device="cuda")
    best = 0.0
    for _ in range(reps + 1):
        e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
        e0.record(); d.copy_(h, non_blocking=True); e1.record(); torch.cuda.synchronize()
        best = max(best, nbytes / e0.elapsed_time(e1) / 1e6)
    del h, d
    return best


def measure_extras(args, eng, L, table, Wb, rank, world, barrier, max_over_ranks, sum_over_ranks, torch, group, steps=4):
    """--extras packed,incremental (opt-in; one torchrun then measures everything — an N=8 box is charged 8x): on the SAME
    engines, after the main measurement, every rank refills its shard with bf16 dummy weights and cycles with the PACKED image,
    then with INCREMENTAL sleep.  Aggregates like the main line: sum of bytes over ranks / max over ranks of the mean time."""
    out = {}
    try:
        from fma_b200 import ranks as R

        fill_weights(eng, table, R.shard_seed(rank), "bf16", torch)
        before = eng.digest_all(["weights"])
        mean = lambda xs: sum(xs) / len(xs)
        W_total = sum_over_ranks(float(Wb))
        if "packed" in args.extras:
            eng.set_option("pack", 1)
            rows = []
            for i in range(steps + 1):
                barrier(); eng.sleep(["weights"]); s1 = eng.stats()
                barrier(); eng.wake(None); s2 = eng.stats()
                if i:
                    rows.append((s1, s2))
            wake = max_over_ranks(mean([r[1]["wake_seconds"] for r in rows]))
            sleep = max_over_ranks(mean([r[0]["sleep_seconds"] for r in rows]))
            stored = sum_over_ranks(float(rows[-1][0]["image_store_bytes"]))
            out["packed"] = {"wake_latency_s": round(wake, 5), "sleep_latency_s": round(sleep, 5), "stored_frac": round(stored / W_total, 4),
                             "e2e_effective_gbs": round(W_total / wake / 1e9, 2), "e2e_link_gbs": round(stored / wake / 1e9, 2),
                             "image_packed": bool(rows[-1][0]["image_packed"]), "bit_exact": bool(group.all_true(eng.digest_all(["weights"]) == before))}
        if "incremental" in args.extras:
            eng.set_option("incremental", 1)
            rows = []
            for i in range(steps + 1):
                barrier(); eng.sleep(["weights"]); s1 = eng.stats()
                barrier(); eng.wake(None); s2 = eng.stats()
                if i:                                  # cycle 0 seeds the digests
                    rows.append((s1, s2))
            out["incremental"] = {"sleep_latency_s": round(max_over_ranks(mean([r[0]["sleep_seconds"] for r in rows])), 5),
                                  "sleep_bytes_copied": int(sum_over_ranks(float(rows[-1][0]["sleep_bytes_copied"]))),
                                  "wake_latency_s": round(max_over_ranks(mean([r[1]["wake_seconds"] for r in rows])), 5),
                                  "bit_exact": bool(group.all_true(eng.digest_all(["weights"]) == before))}
            eng.set_option("incremental", 0)
        eng.set_option("pack", args.pack)
    except Exception as e:       # extras never fail the main line
        out["error"] = str(e)[:200]
    return out


def measure_peer(eng, L, Wb, local_rank, world, barrier, max_over_ranks, before, steps=3):
    """Same shard parked in a peer GPU's HBM over NVLink (FMA_TIER_PEER): K1 gather -> peer, K2 scatter <- peer."""
    try:
        from fma_b200 import ranks

        peer_dev = ranks.parking_device(local_rank, world)
        eng.peer_reserve(peer_dev, Wb)
        rows = []
        for i in range(steps + 1):
            barrier()
            eng.sleep(["weights"], tier=L.FMA_TIER_PEER); s1 = eng.stats()
            barrier()
            eng.wake(None); s2 = eng.stats()
            if i:
                rows.append((s1, s2))
        ok = eng.digest_all(["weights"]) == before
        eng.peer_release()
        mean = lambda xs: sum(xs) / len(xs)
        wake_wall = max_over_ranks(mean([r[1]["wake_seconds"] for r in rows]))
        wake_dev = max_over_ranks(mean([r[1]["wake_copy_seconds"] for r in rows]))
        sleep_dev = max_over_ranks(mean([r[0]["sleep_copy_seconds"] for r in rows]))
        return {"wake_latency_s": round(wake_wall, 5), "wake_gbs_per_gpu_e2e": round(Wb / wake_wall / 1e9, 1),
                "wake_gbs_per_gpu_device": round(Wb / wake_dev / 1e9, 1), "sleep_gbs_per_gpu_device": round(Wb / sleep_dev / 1e9, 1),
                "frac_of_nvlink_900": round(Wb / wake_dev / 1e9 / NVLINK5_GBS, 4), "bit_exact": bool(ok),
                "placement": "rank r parks on GPU (r + N/2) % N"}
    except Exception as e:  # the peer tier is extra evidence; never fail the host-tier line because of it
        return {"error": str(e)[:200]}


# --------------------------------------------------------------------------------------------------
# reference arm: vLLM's own CuMemAllocator (vllm:device_allocator/cumem.py:177-249), unmodified
# --------------------------------------------------------------------------------------------------
def reference_cycle_worker(gpu: int, workload: str, kv_gib: float, steps: int, warmup: int, conn, start_barrier=None, contents: str = "prng"):
    """Runs in its own process: one GPU, the same allocation table, vLLM's allocator moving the bytes."""
    os.environ["CUDA_VISIBLE_DEVICES"] = str(gpu)
    try:
        import torch

        import fma_b200  # only for the table shapes (workloads.py holds no engine code)
        from fma_b200 import workloads as W
        from vllm.device_allocator.cumem import CuMemAllocator

        torch.cuda.set_device(0)
        table = W.allocation_table(workload, kv_cache_bytes=int(kv_gib * GiB))
        alloc = CuMemAllocator.get_instance()
        tensors = []
        gen = torch.Generator(device="cuda"); gen.manual_seed(1234 + gpu)
        with alloc.use_memory_pool(tag="weights"):
            for s in table:
                if s.tag == "weights":
                    tensors.append(torch.empty(s.bytes, dtype=torch.uint8, device="cuda"))
        with alloc.use_memory_pool(tag="kv_cache"):
            kv = [torch.empty(s.bytes, dtype=torch.uint8, device="cuda") for s in table if s.tag == "kv_cache"]
        for t in tensors:
            if contents == "bf16":     # what vLLM's dummy loader fills parameters with (weight_utils.py:1451-1471)
                t.view(torch.bfloat16).uniform_(-1e-3, 1e-3, generator=gen)
            else:
                t.view(torch.int64).random_(generator=gen)
        sums = [int(t.view(torch.int64).sum().item()) for t in tensors[:8]]
        Wb = sum(t.numel() for t in tensors)
        torch.cuda.synchronize()
        rows = []
        for i in range(warmup + steps):
            if start_barrier is not None:
                start_barrier.wait()
            torch.cuda.synchronize()
            a = time.perf_counter(); alloc.sleep(offload_tags=("weights",)); torch.cuda.synchronize(); b = time.perf_counter()
            if start_barrier is not None:
                start_barrier.wait()
            c = time.perf_counter(); alloc.wake_up(); torch.cuda.synchronize(); d = time.perf_counter()
            if i >= warmup:
                rows.append((b - a, d - c))
        ok = sums == [int(t.view(torch.int64).sum().item()) for t in tensors[:8]]
        conn.send({"ok": ok, "W": Wb, "rows": rows, "segments": len(alloc.pointer_to_data), "kv": len(kv)})
    except Exception as e:
        conn.send({"error": f"{type(e).__name__}: {e}"[:300]})


def run_reference_workers(n_gpus: int, workload: str, kv_gib: float, steps: int, warmup: int, contents: str = "prng"):
    import multiprocessing as mp

    ctx = mp.get_context("spawn")
    bar = ctx.Barrier(n_gpus) if n_gpus > 1 else None
    procs, conns = [], []
    for g in range(n_gpus):
        pc, cc = ctx.Pipe()
        p = ctx.Process(target=reference_cycle_worker, args=(g, workload, kv_gib, steps, warmup, cc, bar, contents))
        p.start()
        procs.append(p); conns.append(pc)
    results = [c.recv() for c in conns]
    for p in procs:
        p.join()
    return results


def summarise_reference(results, steps):
    """Same aggregation as this repo's arm: per-step job latency = slowest rank of that step; median (and mean) over the steps."""
    errs = [r["error"] for r in results if "error" in r]
    if errs:
        return None, errs[0]
    n = len(results)
    W_total = sum(r["W"] for r in results)
    k = min(len(r["rows"]) for r in results)
    wake_steps = [max(r["rows"][i][1] for r in results) for i in range(k)]
    sleep_steps = [max(r["rows"][i][0] for r in results) for i in range(k)]
    return {"W_total": W_total, "wake_s": statistics.median(wake_steps), "sleep_s": statistics.median(sleep_steps),
            "wake_s_mean": sum(wake_steps) / k, "sleep_s_mean": sum(sleep_steps) / k,
            "wake_steps": wake_steps, "ok": all(r["ok"] for r in results), "n": n,
            "segments": results[0]["segments"]}, None


def reference_sample(args, workload, cycles: int = 5) -> dict:
    """cpu_baseline: the reference data path timed on this box in the same run (bounded: 1 warm-up + 5 timed cycles; median)."""
    cores = os.cpu_count()
    try:
        res = run_reference_workers(1, workload, args.kv_gib, steps=cycles, warmup=1, contents=args.contents)
        summ, err = summarise_reference(res, cycles)
        if err:
            raise RuntimeError(err)
        ws = summ["wake_steps"]
        return {"value": round(summ["W_total"] / summ["wake_s"] / 1e9, 3), "unit": "GB/s", "cores": 1, "kind": "reference",
                "value_min_max": [round(summ["W_total"] / max(ws) / 1e9, 3), round(summ["W_total"] / min(ws) / 1e9, 3)],
                "wake_latency_s": round(summ["wake_s"], 4), "wake_latency_s_min_max": [round(min(ws), 4), round(max(ws), 4)],
                "sleep_latency_s": round(summ["sleep_s"], 4), "bit_exact": summ["ok"],
                "host_cores_available": cores,
                "sample": f"vLLM {vllm_version()} CuMemAllocator.sleep(('weights',)) -> wake_up() over the full {workload} table "
                          f"({summ['segments']} segments incl. kv_cache), 1 warm-up + {cycles} timed cycles (median; min-max beside it), "
                          f"one Python thread per rank"}
    except Exception as e:
        return port_sample(workload, note=f"vLLM allocator unavailable ({str(e)[:120]})")


def port_sample(workload, note="") -> dict:
    """Fallback baseline: the C restatement of the reference loops over host memory (oracle/fma_oracle.c)."""
    import ctypes as C

    import fma_b200  # noqa: F401
    from fma_b200 import workloads as W
    from oracle import oracle as O

    table = [s for s in W.allocation_table(workload) if s.tag == "weights"][:24]
    libc = C.CDLL(None); libc.malloc.restype = C.c_void_p; libc.malloc.argtypes = [C.c_size_t]
    segs = (O.seg_t * len(table))()
    for i, s in enumerate(table):
        p = libc.malloc(s.bytes); C.memset(p, i + 1, s.bytes)
        segs[i].dev, segs[i].bytes, segs[i].tag, segs[i].backup = p, s.bytes, 0, None
    Wb = sum(s.bytes for s in table)
    t0 = time.perf_counter(); O.lib().fma_oracle_sleep(segs, len(table), 1); t1 = time.perf_counter()
    O.lib().fma_oracle_wake(segs, len(table), 0, 0); t2 = time.perf_counter()
    return {"value": round(Wb / (t2 - t1) / 1e9, 3), "unit": "GB/s", "cores": 1, "kind": "port",
            "wake_latency_s": round(t2 - t1, 4), "sleep_latency_s": round(t1 - t0, 4),
            "sample": f"oracle/fma_oracle.c sleep->wake over the first {len(table)} weight segments of {workload} "
                      f"({Wb / GiB:.2f} GiB), host memcpy stand-in for device memory. {note}"}


def vllm_version() -> str:
    try:
        from importlib.metadata import version

        return version("vllm")
    except Exception:
        return "?"


def run_reference(args) -> None:
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return  # rank 0 alone runs the reference arm (it spawns one worker process per GPU itself)
    workload = workload_for(args.gpus, args.workload)
    t0 = time.perf_counter()
    try:
        res = run_reference_workers(args.gpus, workload, args.kv_gib, args.steps, args.warmup, contents=args.contents)
        summ, err = summarise_reference(res, args.steps)
        if err:
            raise RuntimeError(err)
        kind, cores = "reference", args.gpus
        value = summ["W_total"] / summ["wake_s"] / 1e9
        wake_s, sleep_s, ok = summ["wake_s"], summ["sleep_s"], summ["ok"]
        wake_mean, sleep_mean = summ["wake_s_mean"], summ["sleep_s_mean"]
        W_total = summ["W_total"]
        sample = (f"vLLM {vllm_version()} CuMemAllocator (unmodified, the data path POST /sleep and /wake_up reach through the "
                  f"reference launcher): sleep(('weights',)) -> wake_up() of the full {workload} table per GPU, "
                  f"{args.gpus} worker process(es), one Python thread each")
    except Exception as e:
        p = port_sample(workload, note=f"vLLM allocator unavailable ({str(e)[:120]})")
        kind, cores, value, wake_s, sleep_s, ok, sample = "port", 1, p["value"], p["wake_latency_s"], p["sleep_latency_s"], True, p["sample"]
        wake_mean, sleep_mean = wake_s, sleep_s
        W_total = 0
    total = time.perf_counter() - t0
    import fma_b200  # noqa: F401  (table shapes only: workloads.py holds no engine code)
    from fma_b200 import workloads as W

    table = W.allocation_table(workload, kv_cache_bytes=int(args.kv_gib * GiB))
    mode = args.mode if args.mode != "auto" else ("staged" if args.tier == "host" else "kernel")
    out = {"impl": "reference", "metric": "wake_h2d_gbs", "value": round(value, 3), "unit": "GB/s", "n_gpus": args.gpus,
           "steps": args.steps, "warmup": args.warmup, "ms_per_step": round((wake_mean + sleep_mean) * 1e3, 3),
           "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
           "config": bench_config(args, workload, W.weight_bytes(table), len(table), args.gpus, mode, False),
           "aggregation": "same as the repo's arm: whole-job bytes / MEDIAN over the K timed steps of the per-step job latency (max over ranks)",
           "value_mean": round(W_total / wake_mean / 1e9, 3) if W_total else None,
           "wake_latency_s": round(wake_s, 5), "wake_latency_s_mean": round(wake_mean, 5),
           "sleep_latency_s": round(sleep_s, 5), "bit_exact": bool(ok),
           "cpu_baseline": {"value": round(value, 3), "unit": "GB/s", "cores": cores, "kind": kind, "sample": sample},
           "e2e": {"value": round(value, 3), "unit": "GB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
           "gpu_launches": 0, "wall_s_total": round(total, 1)}
    print(json.dumps(out), flush=True)


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", choices=["ours", "reference"], default="ours")
    ap.add_argument("--workload", default=None, help="override: llama-3-8b | llama-3-70b-tp8 | mistral-7b | opt-125m")
    ap.add_argument("--kv-gib", type=float, default=32.0, help="kv_cache-tagged bytes per rank (discarded + remapped, never copied)")
    ap.add_argument("--tier", choices=["host", "peer", "local"], default="host")
    ap.add_argument("--mode", choices=["auto", "direct", "staged", "kernel"], default="auto")
    ap.add_argument("--kernel", choices=["tma", "ldg"], default="tma")
    ap.add_argument("--chunk-mib", type=int, default=0)
    ap.add_argument("--ring-slots", type=int, default=0)
    ap.add_argument("--copy-streams", type=int, default=0)
    ap.add_argument("--map-threads", type=int, default=0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--peer-extra", type=int, default=1, help="at N>1 also measure the NVLink peer-HBM tier (reported under peer_tier)")
    ap.add_argument("--contents", choices=["prng", "bf16"], default="prng", help="synthetic weights: incompressible bytes (default) or bf16 dummy weights")
    ap.add_argument("--pack", type=int, default=0, help="1 = PACKED host image (lossless bf16 page code; pays off with --contents bf16)")
    ap.add_argument("--incremental", type=int, default=0, help="1 = INCREMENTAL sleep: a sleep whose weights still match the image in the host store moves nothing")
    ap.add_argument("--packed-extra", type=int, default=1, help="at N=1 also measure the PACKED image on bf16 dummy weights in a child process (reported under packed_image)")
    ap.add_argument("--extras", default="swap,scaling_base,roundrobin,multipath",
                    help="comma list of extras measured after the main line: swap (N=1: BASELINE config 4, Llama-3-8B <-> Mistral-7B), scaling_base "
                         "(N=1: the N>1 table on one GPU), multipath (N=1 with more GPUs visible: MULTI-PATH wake over idle peers' links), roundrobin (N>=2: BASELINE config 5, N/2 parked 8B sleepers woken round-robin), "
                         "packed,incremental (any N, on the same engines; opt-in)")
    ap.add_argument("--swap-models", default="llama-3-8b,mistral-7b", help="the two models of the swap extra (the first is also the round-robin sleeper)")
    ap.add_argument("--scaling-workload", default="llama-3-70b-tp8", help="table of the scaling_base extra (= the N>1 workload)")
    ap.add_argument("--extras-kv-gib", type=float, default=16.0, help="kv_cache bytes per model in the swap / roundrobin extras")
    ap.add_argument("--timeline", default="", help="directory: every rank writes the per-phase timeline (fma_timeline) of its last timed sleep and wake there")
    ap.add_argument("--dump-outputs", default="", metavar="DIR",
                    help="after the timed steps, write the weights the last wake restored (digests and a fixed sample) to DIR/*.npy")
    ap.add_argument("--packed-child", action="store_true", help=argparse.SUPPRESS)
    args = ap.parse_args()
    if args.packed_child:
        run_packed_child(args)
        return
    if args.warmup < 3 and args.impl == "ours":
        args.warmup = 3  # timing rules: >= 3 warm-up steps
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()

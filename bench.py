#!/usr/bin/env python
"""bench.py — headline benchmark of the plugin hook-chain hot path on B200.

Metric (BASELINE.json): tool-call payloads/sec on 16 KiB JSON tool results.

  python bench.py --gpus N --steps K --warmup W              # our arm (one process per GPU under torchrun)
  python bench.py --impl reference ...                       # the reference chain's CPU path on the host cores
  python bench.py --workload scan ...                        # BASELINE configs[1] alone: the fused pattern scan (round-1 headline)

Default workload = the FULL CHAIN (BASELINE configs[3] semantics at 16 KiB): for every tool result the tool_post_invoke chain
harmful_content_detector (9 IGNORECASE regexes over every string) -> regex_filter (2 rules, rewrite on match) -> toon_encoder
(JSON -> TOON, kept when smaller) — one packed upload, one fused cf_run_batch per step (scan + rewrite of the flagged units +
TOON on the resident batch).  A "step" is one pass over one batch of `units` valid-JSON payloads of ~16 KiB per GPU (weak
scaling).  Rank 0 prints ONE JSON line; DESIGN.md §6 defines every field.
"""
from __future__ import annotations

import argparse
import asyncio
import ctypes
import json
import os
import re
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

PAYLOAD_BYTES = 16384
UNITS_CHAIN = 32768            # 32768 x 16 KiB = 512 MiB per step per GPU (4x the 126 MB L2)
UNITS_SCAN = 65536             # scan-only workload: 1 GiB per step per GPU
DISTINCT = 256                 # distinct seeded payloads, tiled to the batch
MIX = (("A", 0.5), ("B", 0.25), ("C", 0.25))
METRIC_CHAIN = "tool-call payloads/sec (16 KiB JSON), full tool_post_invoke chain: harmful scan + regex_filter + toon_encoder"
METRIC_SCAN = "tool-call payloads/sec (16 KiB JSON), fused regex/deny/harmful scan"

DENY = ["innovative", "groundbreaking", "revolutionary"]          # plugins/config.yaml:171-174
SUBS = [("crap", 0, "crud"), ("crud", 0, "yikes")]                # plugins/config.yaml:149-153

CHAIN_YAML = """
plugins:
  - name: "HarmfulContentDetector"
    kind: "mcp_context_forge_b200.plugins.harmful_content_detector.HarmfulContentDetectorPlugin"
    hooks: ["tool_post_invoke"]
    mode: "sequential"
    priority: 96
  - name: "ReplaceBadWordsPlugin"
    kind: "mcp_context_forge_b200.plugins.regex_filter.SearchReplacePlugin"
    hooks: ["tool_post_invoke"]
    mode: "sequential"
    priority: 150
    config:
      words:
        - {search: crap, replace: crud}
        - {search: crud, replace: yikes}
  - name: "ToonEncoder"
    kind: "mcp_context_forge_b200.plugins.toon_encoder.ToonEncoderPlugin"
    hooks: ["tool_post_invoke"]
    mode: "sequential"
    priority: 900
plugin_settings:
  plugin_timeout: 300
"""


def make_payloads(distinct: int = DISTINCT, valid_json: bool = True, hit_rate: float = 1e-4):
    """`distinct` seeded payloads of ~16 KiB in the MIX.  valid_json: every payload is a JSON document (prose is the body of a
    small JSON object; nested-config payloads are drawn until their size lands within 16 KiB +- 25 % — nothing is truncated)."""
    from mcp_context_forge_b200 import synth

    out = []
    for i in range(distinct):
        r = (i * 0.61803398875) % 1.0
        acc = 0.0
        shape = "A"
        for s, w in MIX:
            acc += w
            if r < acc:
                shape = s
                break
        if shape == "A":
            p = synth.payload("A", PAYLOAD_BYTES, seed=i, hit_rate=hit_rate)
        elif shape == "B":
            p, k = None, 0
            while p is None or not (0.75 * PAYLOAD_BYTES <= len(p) <= 1.25 * PAYLOAD_BYTES):
                p = synth.payload("B", int(PAYLOAD_BYTES * 0.6), seed=i * 131 + k, hit_rate=hit_rate)
                k += 1
                if k > 400:
                    break
        else:
            text = synth.payload("C", PAYLOAD_BYTES - 64, seed=i, hit_rate=hit_rate)
            p = json.dumps({"title": f"document {i}", "lang": "en", "body": text}, ensure_ascii=False, separators=(",", ":")) if valid_json else text
        out.append(p)
    return out


# ------------------------------------------------------------------------------------------------
# CPU arm: the oracle port of the reference chain (CPython `re`, toon.py restatement) on all host cores
# ------------------------------------------------------------------------------------------------
_W = {}


def _cpu_init():
    from oracle import hook_chain_ref as ref
    from oracle import toon_ref

    _W["cats"] = ref.harmful_compile(None)
    _W["rules"] = ref.regex_compile_rules([{"search": s, "replace": r} for s, _, r in SUBS])
    _W["ref"] = ref
    _W["toon"] = toon_ref


def _cpu_chain(payloads):
    """The reference tool_post_invoke chain for one tool result {"content": [{"type": "text", "text": payload}]}:
    harmful `_iter_strings` + 9 searches per string, regex_filter over the top-level str values, toon `_process_content_item`."""
    ref, toon = _W["ref"], _W["toon"]
    n = 0
    for p in payloads:
        result = {"content": [{"type": "text", "text": p}]}
        n += len(ref.harmful_tool_post(result, _W["cats"]))
        ref.regex_apply_dict(_W["rules"], result)
        t = toon.process_text(p)
        n += 0 if t is None else len(t)
    return n


def _cpu_scan(payloads):
    ref = _W["ref"]
    n = 0
    for p in payloads:
        n += len(ref.harmful_scan_text(p, _W["cats"]))
        n += 1 if any(w in p for w in DENY) else 0
        n += len(ref.regex_apply_str(_W["rules"], p))
    return n


def cpu_run(fn, payloads, total_units: int, cores: int) -> float:
    """payloads/s of the oracle chain over `total_units` payloads spread over `cores` processes."""
    import multiprocessing as mp

    per = max(1, total_units // cores)
    work = [[payloads[(c * per + i) % len(payloads)] for i in range(per)] for c in range(cores)]
    ctx = mp.get_context("fork")
    with ctx.Pool(cores, initializer=_cpu_init) as pool:
        pool.map(fn, [w[:2] for w in work])          # warm the workers
        t0 = time.perf_counter()
        pool.map(fn, work)
        dt = time.perf_counter() - t0
    return per * cores / dt


def host_cores() -> int:
    """Usable host threads: affinity mask, capped by the cgroup CPU quota when one is set."""
    try:
        n = len(os.sched_getaffinity(0))
    except Exception:
        n = os.cpu_count() or 1
    try:
        with open("/sys/fs/cgroup/cpu.max") as f:
            quota, period = f.read().split()
        if quota != "max":
            n = max(1, min(n, int(int(quota) / int(period))))
    except Exception:
        pass
    return n


# ------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = "index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, gpu_index: int):
        self.idx = gpu_index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100", "-i", str(self.idx)],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        for l in self.lines:
            f = [x.strip() for x in l.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons), "samples": len(sm)}


def read_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback 6.65 TB/s (B200_PROFILING.md)"


DUMP_SAMPLE_UNITS = 256        # units whose produced texts --dump-outputs writes (<= 256 x 20 KiB x 4 B: well under 64 MB)


def dump_outputs(directory: str, arrays: dict) -> None:
    """--dump-outputs: each array as DIR/<name>.npy.  Integer fields go out as float64 (exact below 2**53), bytes as float32."""
    import numpy as np

    os.makedirs(directory, exist_ok=True)
    for name, a in arrays.items():
        a = np.asarray(a)
        np.save(os.path.join(directory, name + ".npy"), a.astype(np.float32 if a.dtype == np.uint8 else np.float64))


def sampled_texts(out, oo, n: int):
    """The produced texts of a fixed, seeded sample of the units: (unit indices, their bytes concatenated, offsets into those bytes)."""
    import numpy as np

    idx = np.sort(np.random.default_rng(0).choice(n, size=min(n, DUMP_SAMPLE_UNITS), replace=False))
    parts = [out[int(oo[i]):int(oo[i + 1])] for i in idx]
    offs = np.zeros(len(parts) + 1, dtype=np.int64)
    np.cumsum([len(x) for x in parts], out=offs[1:])
    return idx, (np.concatenate(parts) if parts else np.zeros(0, dtype=np.uint8)), offs


def chain_config(world: int, units: int):
    return {"workload": "configs[3] semantics at 16 KiB: full tool_post_invoke chain — harmful_content_detector (9 IGNORECASE regexes) + regex_filter (2 rules, rewrite "
                        f"on match) + toon_encoder (JSON->TOON, kept when smaller); valid JSON payloads, {int(MIX[0][1]*100)}% tabular / {int(MIX[1][1]*100)}% nested config / "
                        f"{int(MIX[2][1]*100)}% prose-in-JSON, hit rate 1e-4 per word",
            "payload_bytes": PAYLOAD_BYTES, "units_per_gpu": units, "patterns": 11, "pattern_set": "reference defaults (plugins/config.yaml)",
            "l2_policy": "inputs_larger_than_l2 (512 MiB batch per GPU vs 126 MB L2)",
            "parallelism": (f"shard{world}: independent payload shards per GPU, one NCCL all_gather of 24-byte verdict records" if world > 1 else "single GPU")}


def scan_config(world: int, units: int):
    return {"workload": f"configs[1]: batched 16 KiB payloads ({int(MIX[0][1]*100)}% tabular JSON / {int(MIX[1][1]*100)}% nested JSON / {int(MIX[2][1]*100)}% prose, hit rate 1e-4), "
                        "fused harmful(9 IGNORECASE regex)+deny(3 literals)+regex_filter(2 rules) scan",
            "payload_bytes": PAYLOAD_BYTES, "units_per_gpu": units, "patterns": 14, "pattern_set": "reference defaults (plugins/config.yaml)",
            "l2_policy": "inputs_larger_than_l2 (1 GiB batch per GPU vs 126 MB L2)",
            "parallelism": f"shard{world}: independent payload shards per GPU, one NCCL all_gather of verdict bitmaps" if world > 1 else "single GPU"}


# ------------------------------------------------------------------------------------------------
def reference_arm(args, chain: bool):
    """The reference's CPU implementation of the path on all host cores (the reference is Python + one Rust crate: nothing
    compiles with gcc, so the oracle port — the reference's loops on CPython `re`, toon.py restated — is what is timed)."""
    payloads = make_payloads(64, valid_json=chain)
    cores = host_cores()
    fn = _cpu_chain if chain else _cpu_scan
    sample = max(cores * 4, min(args.units, (16 if chain else 64) * cores))
    vals = []
    for i in range(args.warmup + args.steps):
        v = cpu_run(fn, payloads, sample, cores)
        if i >= args.warmup:
            vals.append(v)
        if i == 0 and sample / v > 8.0:      # keep the whole run within a few minutes
            sample = max(cores * 2, int(sample * 4.0 / (sample / v)))
    val = sum(vals) / len(vals)
    config = chain_config(args.gpus, args.units) if chain else scan_config(args.gpus, args.units)
    what = ("oracle/hook_chain_ref.py + oracle/toon_ref.py = the reference plugins' loops on CPython re and toon.py restated"
            if chain else "oracle/hook_chain_ref.py = the reference plugins' loops on CPython re")
    line = {"impl": "reference", "metric": METRIC_CHAIN if chain else METRIC_SCAN, "value": val, "unit": "payloads/s", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * sample / val, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
            "config": config,
            "cpu_baseline": {"value": val, "unit": "payloads/s", "cores": cores, "kind": "port",
                             "sample": f"{sample} payloads of 16 KiB per step over {cores} processes; {what} (the reference is pure Python; cpex/orjson absent here)"},
            "e2e": {"value": val, "unit": "payloads/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))
    return 0


# ------------------------------------------------------------------------------------------------
def _api_worker(device: int, requests: int, waves: int, hit_rate: float, barrier, q):
    """One gateway worker process: its own event loop, its own BatchedPluginManager (and CUDA context) on GPU `device`."""
    from mcp_context_forge_b200 import framework as fw
    from mcp_context_forge_b200.cpex_compat.framework import HookPayloadPolicy
    from mcp_context_forge_b200.manager import BatchedPluginManager
    import logging

    logging.disable(logging.WARNING)       # the plugins log one warning per item TOON cannot encode, like the reference; not part of the measurement
    payloads = make_payloads(64, hit_rate=hit_rate)
    with tempfile.TemporaryDirectory() as td:
        cfg = os.path.join(td, "plugins.yaml")
        with open(cfg, "w") as f:
            f.write(CHAIN_YAML)
        m = BatchedPluginManager(cfg, timeout=300, hook_policies={"tool_post_invoke": HookPayloadPolicy(writable_fields=frozenset({"result"}))}, device=device)
        loop = asyncio.new_event_loop()
        loop.run_until_complete(m.initialize())
        gc = fw.GlobalContext(request_id="bench")
        posts = [fw.ToolPostInvokePayload(name="t", result={"content": [{"type": "text", "text": payloads[i % len(payloads)]}]}) for i in range(requests)]

        async def wave():
            return await asyncio.gather(*[m.invoke_hook("tool_post_invoke", p, gc) for p in posts])

        for _ in range(2):
            res = loop.run_until_complete(wave())
        a0, d0, r0 = m.assemble_s, m.device_s, m.replay_s
        barrier.wait()
        t0 = time.perf_counter()
        for _ in range(waves):
            res = loop.run_until_complete(wave())
        dt = time.perf_counter() - t0
        toon = [r.modified_payload.result["content"][0]["text"] for r, _ in res
                if r.modified_payload is not None and (r.modified_payload.result["content"][0].get("annotations") or {}).get("format") == "toon"]
        h2d = sum(len(p.result["content"][0]["text"].encode()) + 1 for p in posts) + 8 * (requests + 1) + requests
        d2h = 24 * requests + sum(len(t.encode()) for t in toon)
        q.put({"dt": dt, "requests": requests * waves, "h2d": h2d, "d2h": d2h, "converted": len(toon), "ms_assemble_python": (m.assemble_s - a0) / waves * 1e3,
               "ms_pack_h2d_kernels_d2h": (m.device_s - d0) / waves * 1e3, "ms_replay_python": (m.replay_s - r0) / waves * 1e3})
        loop.run_until_complete(m.shutdown())


def hook_api_e2e(requests: int, waves: int, device: int, workers: int, hit_rate: float):
    """payloads/s through the repo's own public API — `BatchedPluginManager.invoke_hook('tool_post_invoke', ...)` with host objects —
    as a gateway host runs it: `workers` worker processes (one event loop each, like gunicorn workers) sharing GPU `device`,
    `requests` concurrent calls per wave and worker.  Returns (payloads/s, h2d bytes, d2h bytes per step, stats)."""
    import multiprocessing as mp

    ctx = mp.get_context("spawn")
    barrier = ctx.Barrier(workers)
    q = ctx.Queue()
    procs = [ctx.Process(target=_api_worker, args=(device, requests, waves, hit_rate, barrier, q)) for _ in range(workers)]
    for p in procs:
        p.start()
    rs = [q.get(timeout=900) for _ in procs]
    for p in procs:
        p.join(120)
    dt = max(r["dt"] for r in rs)
    total = sum(r["requests"] for r in rs)
    stats = {"workers": workers, "requests_per_wave_per_worker": requests, "waves": waves, "ms_per_wave": dt / waves * 1e3,
             "ms_assemble_python": sum(r["ms_assemble_python"] for r in rs) / workers, "ms_pack_h2d_kernels_d2h": sum(r["ms_pack_h2d_kernels_d2h"] for r in rs) / workers,
             "ms_replay_python": sum(r["ms_replay_python"] for r in rs) / workers, "fused_launch_calls_per_wave_per_worker": 1,
             "toon_converted_per_wave": sum(r["converted"] for r in rs)}
    return total / dt, sum(r["h2d"] for r in rs), sum(r["d2h"] for r in rs), stats


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="chain", choices=["chain", "scan"])
    ap.add_argument("--units", type=int, default=0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--hit-rate", type=float, default=1e-4)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last timed step computed (rank 0's shard) as DIR/<name>.npy")
    args = ap.parse_args()
    args.warmup = max(args.warmup, 3)
    chain = args.workload == "chain"
    if not args.units:
        args.units = UNITS_CHAIN if chain else UNITS_SCAN

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))

    if args.impl == "reference":
        return 0 if rank != 0 else reference_arm(args, chain)
    if not chain:
        return scan_bench(args, rank, local_rank, world)

    # ------------------------------------------------------------------ our arm, full chain
    config = chain_config(world, args.units)
    payloads = make_payloads(hit_rate=args.hit_rate)
    cpu_base = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cores = host_cores()
        sample = 24 * cores                               # ~3-4 ms per payload per core: ~10-30 s of CPU work in total
        v = cpu_run(_cpu_chain, payloads, sample, cores)
        cpu_base = {"value": v, "unit": "payloads/s", "cores": cores, "kind": "port",
                    "sample": f"{sample} payloads of 16 KiB (same mix) over {cores} processes: oracle chain = harmful_tool_post + regex_apply_dict (CPython re) + toon_ref.process_text"}

    import numpy as np
    import torch

    from mcp_context_forge_b200 import engine
    from mcp_context_forge_b200._native import CF_STAGE_SCAN, CF_STAGE_SUB, CF_STAGE_TOON, CF_V_REWRITTEN, CF_V_TOON
    from mcp_context_forge_b200.plugins.harmful_content_detector import DEFAULT_LEXICONS   # product's copy of the reference defaults

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device — the B200 path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist

        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    ctx = engine.Context.get(local_rank)
    prog = engine.Program()
    for pats in DEFAULT_LEXICONS.values():
        for pat in pats:
            prog.add_search(pat, re.I)
    for s, f, r in SUBS:
        prog.add_sub(s, f, r)
    prog.compile(ctx)
    lib = ctx.lib
    STAGES = CF_STAGE_SCAN | CF_STAGE_SUB | CF_STAGE_TOON

    n = args.units
    units = [payloads[(i + rank * 7) % len(payloads)] for i in range(n)]
    stream, offs = engine.pack_units(units)
    nbytes = len(stream)
    h_stream = torch.empty(nbytes, dtype=torch.uint8, pin_memory=True)
    h_stream.numpy()[:] = np.frombuffer(stream, dtype=np.uint8)
    h_stream_np = h_stream.numpy()
    batch = engine.Batch(ctx, nbytes, n)
    batch.upload(h_stream_np, offs)
    torch.cuda.synchronize()
    # N > 1: the 24-byte verdict records of every shard are all-gathered every step (the path's only collective), on NCCL's
    # stream, overlapped with the next step's kernels
    words = engine.VERDICT_DTYPE.itemsize // 8
    d_local = [torch.zeros(n * words, dtype=torch.int64, device="cuda") for _ in range(2)] if world > 1 else None
    d_all = [torch.zeros(world * n * words, dtype=torch.int64, device="cuda") for _ in range(2)] if world > 1 else None
    pending = []
    step_no = [0]
    last = {}

    def step_resident():
        # stream=None: the batch is resident; outputs_resident: the produced texts are gathered in HBM and stay there (`value` has
        # no host<->device payload copies by definition; `e2e_cabi` below is the same call with host buffers on both sides)
        v, _out, oo, _ = engine.run_batch(prog, batch, None, offs, STAGES, outputs_resident=True)
        last["v"], last["oo"] = v, oo
        if world > 1:
            k = step_no[0] & 1
            step_no[0] += 1
            if len(pending) >= 2:
                pending.pop(0).wait()
            d_local[k].copy_(torch.from_numpy(v.view(np.int64)), non_blocking=True)
            pending.append(dist.all_gather_into_tensor(d_all[k], d_local[k], async_op=True))

    def step_cabi():
        v, out, oo, _ = engine.run_batch(prog, batch, h_stream_np, offs, STAGES)   # pinned host stream: H2D inside
        last["v"], last["out"], last["oo"] = v, out, oo

    def drain():
        while pending:
            pending.pop(0).wait()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        """cf_run_batch is synchronous (it returns the verdicts): wall clock around K calls, max over ranks."""
        barrier()
        t0 = time.perf_counter()
        for _ in range(steps):
            fn()
        if world > 1:
            drain()
        torch.cuda.synchronize()
        ms = (time.perf_counter() - t0) * 1e3
        if world > 1:
            t = torch.tensor([ms], dtype=torch.float64, device="cuda")
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        barrier()
        return ms

    for _ in range(args.warmup):
        step_resident()
    drain()
    torch.cuda.synchronize()

    sampler = ClockSampler(local_rank) if rank == 0 else None
    if sampler:
        sampler.start()
    l0 = ctx.kernel_launches
    ctx.check(lib.cf_profile_begin(ctx.h, 2 * args.steps), "profile_begin")
    ms_total = timed(step_resident, args.steps)
    each = (ctypes.c_double * (2 * args.steps + 2))()
    kn = ctypes.c_uint32()
    ctx.check(lib.cf_profile_collect_each(ctx.h, each, 2 * args.steps + 2, ctypes.byref(kn)), "profile_collect_each")
    ctx.check(lib.cf_profile_begin(ctx.h, 0), "profile_end")
    launches = ctx.kernel_launches - l0
    clocks = sampler.stop() if sampler else None
    scan_ms = [each[i] for i in range(0, kn.value, 2)]          # launch order inside cf_run_batch: scan, then the TOON stage
    toon_ms = [each[i] for i in range(1, kn.value, 2)]
    v_res = last["v"].copy()
    out_res, oo_res = engine.device_output(ctx), last["oo"].copy()       # un-timed copy of the resident outputs, for the parity checks below
    if args.dump_outputs and rank == 0:
        # the verdict record of every unit, and the texts produced (rewritten or TOON) for a fixed sample of the units
        idx, sample, sample_offs = sampled_texts(out_res, oo_res, n)
        dump_outputs(args.dump_outputs, {"verdict_match_bitmap": v_res["match_bitmap"], "verdict_flags": v_res["flags"], "verdict_out_len": v_res["out_len"],
                                         "verdict_aux": v_res["aux"], "text_sample_units": idx, "text_sample_bytes": sample, "text_sample_offsets": sample_offs})

    for _ in range(2):
        step_cabi()
    cabi_steps = max(3, min(args.steps, 5))
    ms_cabi = timed(step_cabi, cabi_steps)
    same = bool((last["v"] == v_res).all()) and bool((last["oo"] == oo_res).all()) and \
        bool((last["out"][: int(oo_res[-1])] == out_res[: int(oo_res[-1])]).all())     # resident outputs == host-buffer outputs, byte for byte

    # ---- parity of a sample of this run's outputs against the oracle (checker only)
    if rank == 0:
        from oracle import hook_chain_ref as ref
        from oracle import toon_ref

        for i in list(range(6)) + [n // 2, n - 1]:
            exp = toon_ref.process_text(units[i])
            got = out_res[int(oo_res[i]):int(oo_res[i + 1])].tobytes().decode() if v_res["flags"][i] & CF_V_TOON else None
            expb = ref.scan_bitmaps([units[i]], [(p, re.I) for pats in ref.DEFAULT_LEXICONS.values() for p in pats], [], [(s, f) for s, f, _ in SUBS])[0]
            dirty = (int(v_res["match_bitmap"][i]) >> 9) & 3
            if int(v_res["match_bitmap"][i]) != expb or (not dirty and got != exp) or not same:
                raise SystemExit(f"bench.py: parity check failed at unit {i} (resident==cabi: {same})")

    # ---- variants on a smaller batch (same call as `value`): hit rates 0 / 1e-2 and a large rule set (256 deny literals + 32 regexes)
    variants = None
    if rank == 0 and world == 1:
        variants = {}
        nv = min(n, 8192)

        def run_variant(vprog, vpayloads):
            vunits = [vpayloads[i % len(vpayloads)] for i in range(nv)]
            vs, vo = engine.pack_units(vunits)
            vb = engine.Batch(ctx, len(vs), nv)
            vb.upload(np.frombuffer(vs, dtype=np.uint8), vo)
            for _ in range(2):
                vv, _o, _oo, _f = engine.run_batch(vprog, vb, None, vo, STAGES, outputs_resident=True)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for _ in range(3):
                vv, _o, _oo, _f = engine.run_batch(vprog, vb, None, vo, STAGES, outputs_resident=True)
            dt = (time.perf_counter() - t0) / 3
            return {"payloads_per_s": nv / dt, "ms_per_step": dt * 1e3, "units": nv, "rewritten_units": int(((vv["flags"] & CF_V_REWRITTEN) != 0).sum()),
                    "flagged_units": int((vv["match_bitmap"] != 0).sum()), "toon_converted_units": int(((vv["flags"] & CF_V_TOON) != 0).sum())}

        variants["hit_rate_0"] = run_variant(prog, make_payloads(hit_rate=0.0))
        variants["hit_rate_1e-2"] = run_variant(prog, make_payloads(hit_rate=1e-2))
        sp = engine.Program()
        for pats in DEFAULT_LEXICONS.values():
            for pat in pats:
                sp.add_search(pat, re.I)
        import random as _random
        rr = _random.Random(5)
        syll = ["zor", "quix", "vald", "brem", "tosk", "jiv", "plun", "gax", "merv", "dwil", "skob", "frey", "hux", "nolt", "crim", "yast"]
        for k in range(256):
            sp.add_literal("".join(rr.choice(syll) for _ in range(3)) + str(k))
        for k in range(32 - 9):
            sp.add_search(r"\b" + rr.choice(syll) + r"[a-z]{2,5}" + rr.choice(syll) + r"\d+\b", re.I)
        for s_, f_, r_ in SUBS:
            sp.add_sub(s_, f_, r_)
        sp.compile(ctx)
        variants["stress_rule_set_256_literals_32_regexes"] = run_variant(sp, payloads)
        variants["stress_rule_set_256_literals_32_regexes"]["prefilter"] = "pair" if sp.compile_host().prefilter else "byte"

        # BASELINE configs[2]: the pattern scan + request_logging_masking on ONE upload (cf_run_batch, SCAN | MASK): the same JSON payloads as
        # request bodies; masked bodies come back to the host (they are what the middleware logs).  Last leg on this context, and it never
        # takes the line down: a failure is reported in place.
        def run_mask_variant():
            from mcp_context_forge_b200._native import CF_STAGE_MASK, CF_V_MASKED
            nm = min(n, 32768)                  # the headline's batch: one lane per body needs a full batch to fill the GPU at all
            munits = [payloads[i % len(payloads)] for i in range(nm)]
            ms_, mo = engine.pack_units(munits)
            mb = engine.Batch(ctx, len(ms_), nm)
            ms_np = np.frombuffer(ms_, dtype=np.uint8)
            for _ in range(2):
                mv, mout, moo, _f = engine.run_batch(prog, mb, ms_np, mo, CF_STAGE_SCAN | CF_STAGE_MASK)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for _ in range(3):
                mv, mout, moo, _f = engine.run_batch(prog, mb, ms_np, mo, CF_STAGE_SCAN | CF_STAGE_MASK)
            dt = (time.perf_counter() - t0) / 3
            from oracle import mask_ref
            ok = True
            for i in (0, 1, 2, nm // 2, nm - 1):
                got = mout[int(moo[i]):int(moo[i + 1])].tobytes() if mv["flags"][i] & CF_V_MASKED else None
                try:
                    exp = mask_ref.mask_json_bytes(munits[i] if isinstance(munits[i], bytes) else munits[i].encode(), 10)
                except ValueError:
                    exp = None
                ok = ok and got == exp
            n_out_m = int(moo[-1])
            return {"payloads_per_s": nm / dt, "ms_per_step": dt * 1e3, "units": nm, "in_bytes": len(ms_), "masked_out_bytes": n_out_m,
                    "masked_units": int(((mv["flags"] & CF_V_MASKED) != 0).sum()), "flagged_units": int((mv["match_bitmap"] != 0).sum()),
                    "gb_per_s_in_plus_out": (len(ms_) + n_out_m) / dt / 1e9, "oracle_sample_ok": bool(ok),
                    "what": "cf_run_batch(SCAN|MASK) with host buffers: H2D of the bodies, scan_kernel + mask_kernel (one lane per body, DESIGN 4.5) on the resident "
                            "batch, verdicts + masked bodies D2H; max_depth 10"}

        try:
            variants["configs2_scan_plus_masking"] = run_mask_variant()
        except Exception as exc:  # noqa: BLE001 - reported, never fatal for the headline line
            variants["configs2_scan_plus_masking"] = {"error": f"{type(exc).__name__}: {exc}"[:300]}

    # ---- end to end through the plugin API (host objects in, PluginResult out), one worker
    api = None
    if True:
        reqs = 2048
        # one gateway worker process per host core the rank may use (one core left to the launcher); at N > 1 at most 8 per rank
        workers = max(1, min(15 if world == 1 else 8, host_cores() // world - 1))
        api_val, api_h2d, api_d2h, api_stats = hook_api_e2e(reqs, 3, local_rank, workers, args.hit_rate)
        if world > 1:
            t = torch.tensor([api_val], dtype=torch.float64, device="cuda")
            dist.all_reduce(t, op=dist.ReduceOp.SUM)          # every GPU has its own gateway workers: the rates add up
            api_val = float(t.item())
        api = (api_val, api_h2d, api_d2h, api_stats)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return 0

    ms_step = ms_total / args.steps
    value = world * n / (ms_step / 1e3)
    cabi_val = world * n / (ms_cabi / cabi_steps / 1e3)
    peak, peak_src = read_peaks()
    n_out = int(v_res["out_len"][(v_res["flags"] & CF_V_TOON) != 0].sum())
    toon_k = sum(toon_ms) / max(1, len(toon_ms))
    scan_k = sum(scan_ms) / max(1, len(scan_ms))
    alg = nbytes + n_out + 24 * n                      # SURVEY §8(d): N_in + N_out + V (24-byte verdict record per payload)
    achieved = alg / (toon_k / 1e3) / 1e9 if toon_k > 0 else None
    traffic = None
    tp = os.path.join(ROOT, "profiles", "r02_toon_tp_traffic.json")
    if os.path.exists(tp):
        try:
            with open(tp) as f:
                tj = json.load(f)
            traffic = tj.get("dram_bytes_per_launch_scaled_to", {}).get(str(nbytes)) or (tj.get("dram_bytes_per_input_byte", 0) * nbytes or None)
        except Exception:
            pass
    line = {
        "metric": METRIC_CHAIN, "value": value, "unit": "payloads/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8",
        "data": f"synthetic: {DISTINCT} distinct seeded valid-JSON payloads tiled to {n} units per GPU", "config": config,
        "e2e": {"value": api[0], "unit": "payloads/s", "h2d_bytes_per_step": world * api[1], "d2h_bytes_per_step": world * api[2],
                "api": "BatchedPluginManager.invoke_hook('tool_post_invoke', ToolPostInvokePayload, GlobalContext) — host objects in, PluginResult out; "
                       "gateway worker processes (one event loop each) sharing the GPU, 2048 concurrent requests per wave and worker", **api[3]},
        "e2e_cabi": {"value": cabi_val, "unit": "payloads/s", "h2d_bytes_per_step": world * (nbytes + 8 * (n + 1)), "d2h_bytes_per_step": world * (24 * n + n_out),
                     "api": "cf_run_batch (C ABI, pinned host stream, synchronous): one H2D of the packed stream, scan + rewrite + TOON on the resident batch, verdicts + produced texts back",
                     "steps": cabi_steps},
        "gpu_launches": int(launches),
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": (achieved / peak) if achieved else None, "traffic": traffic,
                     "kernel": "toon_tp_kernel (+ the sequential hand-over launch)", "kernel_ms": toon_k, "algorithmic_bytes_per_launch": alg,
                     "algorithmic_bytes": {"n_in": nbytes, "n_out": n_out, "verdicts": 24 * n}, "read_frac": (nbytes / (toon_k / 1e3) / 1e9 / peak) if toon_k else None,
                     "peak_source": peak_src},
        "stages": {"scan_kernel": {"ms": scan_k, "gb_per_s": nbytes / scan_k / 1e6 if scan_k else None, "frac": (nbytes / scan_k / 1e6 / peak) if scan_k else None},
                   "toon_stage": {"ms": toon_k, "gb_per_s": nbytes / toon_k / 1e6 if toon_k else None, "frac": (nbytes / toon_k / 1e6 / peak) if toon_k else None},
                   "rewritten_units": int(((v_res["flags"] & CF_V_REWRITTEN) != 0).sum()), "toon_converted_units": int(((v_res["flags"] & CF_V_TOON) != 0).sum()),
                   "other_ms_per_step": ms_step - scan_k - toon_k,
                   "value_definition": "cf_run_batch(stream=NULL, CF_RUN_OUTPUTS_RESIDENT): batch resident in HBM, scan + TOON (+ hand-over) kernels, verdict D2H (24 B/unit), "
                                       "regex_filter rewriting of the matched units, gather of the produced texts into one device buffer; texts stay in HBM"},
        "variants": variants,
        "cpu_baseline": cpu_base,
        "clocks": clocks,
    }
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()
    return 0


# ------------------------------------------------------------------------------------------------
def scan_bench(args, rank, local_rank, world):
    """BASELINE configs[1]: the fused pattern scan alone (the round-1 headline), `--workload scan`."""
    config = scan_config(world, args.units)
    payloads = make_payloads(valid_json=False, hit_rate=args.hit_rate)
    cpu_base = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cores = host_cores()
        sample = 96 * cores
        v = cpu_run(_cpu_scan, payloads, sample, cores)
        cpu_base = {"value": v, "unit": "payloads/s", "cores": cores, "kind": "port",
                    "sample": f"{sample} payloads of 16 KiB (same mix) over {cores} processes, oracle/hook_chain_ref.py chain (CPython re)"}

    import numpy as np
    import torch

    from mcp_context_forge_b200 import engine
    from mcp_context_forge_b200.plugins.harmful_content_detector import DEFAULT_LEXICONS

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device — the B200 path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist

        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
        os.environ.setdefault("CF_SCAN_RESERVE_SMS", "4")     # leave NCCL's all-gather somewhere to run beside the persistent scan grid

    ctx = engine.Context.get(local_rank)
    prog = engine.Program()
    for pats in DEFAULT_LEXICONS.values():
        for pat in pats:
            prog.add_search(pat, re.I)
    for w in DENY:
        prog.add_literal(w)
    for s, f, r in SUBS:
        prog.add_sub(s, f, r)
    prog.compile(ctx)
    W = prog.words

    n = args.units
    units = [payloads[(i + rank * 7) % len(payloads)] for i in range(n)]
    stream, offs = engine.pack_units(units)
    nbytes = len(stream)
    h_stream = torch.empty(nbytes, dtype=torch.uint8, pin_memory=True)
    h_stream.numpy()[:] = np.frombuffer(stream, dtype=np.uint8)
    h_offs = torch.from_numpy(offs.astype(np.int64)).pin_memory()
    h_bm = torch.empty(n * W, dtype=torch.int64, pin_memory=True)
    d_bm = torch.zeros(n * W, dtype=torch.int64, device="cuda")
    d_bms = [d_bm, torch.zeros(n * W, dtype=torch.int64, device="cuda")] if world > 1 else [d_bm]
    # the gather carries 16 bits per unit (14 patterns), not the 64-bit word
    # (NCCL has no 16-bit integer type: the buffers are bytes, written through an int16 view)
    d_small = [torch.zeros(2 * n, dtype=torch.uint8, device="cuda") for _ in range(2)] if world > 1 else None
    d_alls = [torch.zeros(world * 2 * n, dtype=torch.uint8, device="cuda") for _ in range(2)] if world > 1 else None
    pending = []
    step_no = [0]
    batch = engine.Batch(ctx, nbytes, n)
    lib = ctx.lib
    cs = torch.cuda.current_stream().cuda_stream

    def upload():
        ctx.check(lib.cf_batch_upload(ctx.h, batch.h, h_stream.data_ptr(), nbytes, h_offs.data_ptr(), n, cs), "upload")

    def step_resident():
        k = step_no[0] & 1 if world > 1 else 0
        step_no[0] += 1
        if world > 1 and len(pending) >= 2:
            pending.pop(0).wait()
        ctx.check(lib.cf_scan(ctx.h, prog.h, batch.h, d_bms[k].data_ptr(), cs), "cf_scan")
        if world > 1:
            d_small[k].view(torch.int16).copy_(d_bms[k])    # W == 1: the low 16 bits hold all 14 pattern bits
            pending.append(dist.all_gather_into_tensor(d_alls[k], d_small[k], async_op=True))

    def drain():
        while pending:
            pending.pop(0).wait()

    def step_e2e():
        ctx.check(lib.cf_scan_host(ctx.h, prog.h, batch.h, h_stream.data_ptr(), nbytes, h_offs.data_ptr(), n, h_bm.data_ptr()), "cf_scan_host")

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps, use_events=True):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter()
        e0.record()
        for _ in range(steps):
            fn()
        if world > 1:
            drain()
        e1.record()
        torch.cuda.synchronize()
        wall = (time.perf_counter() - t0) * 1e3
        ms = e0.elapsed_time(e1) if use_events else wall
        if world > 1:
            t = torch.tensor([ms], dtype=torch.float64, device="cuda")
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        barrier()
        return ms

    upload()
    for _ in range(args.warmup):
        step_resident()
    if world > 1:
        drain()
    torch.cuda.synchronize()
    sampler = ClockSampler(local_rank) if rank == 0 else None
    if sampler:
        sampler.start()
    l0 = ctx.kernel_launches
    ctx.check(lib.cf_profile_begin(ctx.h, args.steps), "profile_begin")
    ms_total = timed(step_resident, args.steps)
    kms, kn = ctypes.c_double(), ctypes.c_uint32()
    ctx.check(lib.cf_profile_collect(ctx.h, ctypes.byref(kms), ctypes.byref(kn)), "profile_collect")
    ctx.check(lib.cf_profile_begin(ctx.h, 0), "profile_end")
    launches = ctx.kernel_launches - l0
    clocks = sampler.stop() if sampler else None
    cand, steps_dfa = ctx.scan_counters()
    if args.dump_outputs and rank == 0:
        # the match bitmaps of every unit (W words of 64 pattern bits each) the last timed scan wrote
        dump_outputs(args.dump_outputs, {"match_bitmap": d_bms[(step_no[0] - 1) & 1 if world > 1 else 0].cpu().numpy().view(np.uint64).reshape(n, W)})
    for _ in range(2):
        step_e2e()
    e2e_steps = max(3, min(args.steps, 10))
    ms_e2e = timed(step_e2e, e2e_steps, use_events=False)
    torch.cuda.synchronize()
    same = bool((h_bm.cuda() == d_bms[0]).all().item())
    if rank == 0:
        from oracle import hook_chain_ref as ref

        exp = ref.scan_bitmaps(units[:8], [(p, re.I) for pats in ref.DEFAULT_LEXICONS.values() for p in pats], DENY, [(s, f) for s, f, _ in SUBS])
        got = engine.bitmaps_to_ints(h_bm.numpy().view(np.uint64), 8, W)
        if got != exp or not same:
            raise SystemExit(f"bench.py: parity check failed (resident==e2e: {same})")
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return 0
    ms_step = ms_total / args.steps
    value = world * n / (ms_step / 1e3)
    e2e_val = world * n / (ms_e2e / e2e_steps / 1e3)
    peak, peak_src = read_peaks()
    k_ms = kms.value / max(1, kn.value)
    alg_bytes = nbytes + 8 * W * n
    achieved = alg_bytes / (k_ms / 1e3) / 1e9 if k_ms > 0 else None
    traffic = None
    tp = os.path.join(ROOT, "profiles", "scan_kernel_traffic.json")
    if os.path.exists(tp):
        try:
            with open(tp) as f:
                tj = json.load(f)
            if tj.get("stream_bytes") == nbytes:
                traffic = tj.get("dram_bytes_per_launch")
        except Exception:
            pass
    line = {"metric": METRIC_SCAN, "value": value, "unit": "payloads/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_step,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8",
            "data": f"synthetic: {DISTINCT} distinct seeded payloads tiled to {n} units per GPU", "config": config,
            "e2e": {"value": e2e_val, "unit": "payloads/s", "h2d_bytes_per_step": world * (nbytes + 8 * (n + 1)), "d2h_bytes_per_step": world * 8 * W * n,
                    "api": "cf_scan_host (C ABI, pinned host buffers, synchronous) — the scan stage only; the plugin-API number is the chain workload's e2e", "steps": e2e_steps},
            "gpu_launches": int(launches),
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": (achieved / peak) if achieved else None, "traffic": traffic,
                         "kernel": "scan_kernel", "kernel_ms": k_ms, "algorithmic_bytes_per_launch": alg_bytes, "peak_source": peak_src},
            "cpu_baseline": cpu_base, "clocks": clocks, "scan_counters": {"prefilter_candidates": cand, "dfa_steps": steps_dfa}}
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())

"""Container-only: live differential fuzz of the json_repair drop-in (on the engine's CPU simulator: JSON kernel source for "does it parse",
substitution routines for the trailing-comma rule) against the REFERENCE'S OWN plugins/json_repair/json_repair.py, imported unmodified from
/root/reference (orjson stood in for by the strict stdlib parser; texts that would expose an orjson / json delta are skipped).
usage: python tools/fuzz_json_repair_vs_reference.py [--record OUT] [seed] [cases]  |  --replay tests/golden/fuzz_json_repair.json.gz"""
import os
import random
import re
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, os.path.join(ROOT, "tools"))
import gen_golden  # noqa: E402
from fuzz_toon_tp import make_gen  # noqa: E402

_DELTA = re.compile(r"\d{18,}|[eE][+-]?\d{3,}|\\u[dD][89a-fA-F]|NaN|Infinity")


def texts(seed: int, n: int):
    rng = random.Random(seed)
    case = make_gen(rng)
    out = []
    while len(out) < n:
        t = case()
        k = rng.random()
        if k < 0.25:
            t = t.replace('"', "'")
        elif k < 0.5:
            t = re.sub(r"([}\]])", lambda m: rng.choice([",", ", ", ",\n", "", ""]) + m.group(1), t)
        elif k < 0.6 and t.startswith("{") and t.endswith("}"):
            t = t[1:-1]
        t = rng.choice(["", "", " ", "\n", " ", "\t"]) + t + rng.choice(["", "", " ", "\r\n", "　"])
        if _DELTA.search(t) or any(0xD800 <= ord(c) <= 0xDFFF for c in t) or t.count("[") + t.count("{") > 60:
            continue
        out.append(t)
    return out


def outcome(r):
    return {"continue_processing": r.continue_processing, "out_result": r.modified_payload.result if r.modified_payload is not None else None,
            "modified": r.modified_payload is not None, "metadata": r.metadata or {}}


def record(argv):
    seed = int(argv[0]) if len(argv) > 0 else 1
    n = int(argv[1]) if len(argv) > 1 else 3000
    gen_golden.install_shims()
    from cpex.framework import GlobalContext, PluginConfig, PluginContext, ToolPostInvokePayload
    from plugins.json_repair.json_repair import JSONRepairPlugin as RefPlugin

    ref = RefPlugin(PluginConfig(name="jr", kind="x", hooks=["tool_post_invoke"]))
    ctx = PluginContext(global_context=GlobalContext(request_id="fuzz"))
    ts = texts(seed, n)
    outputs = [gen_golden.digest(outcome(gen_golden.run(ref.tool_post_invoke(ToolPostInvokePayload(name="t", result=t), ctx)))) for t in ts]
    return {"seed": seed, "cases": n, "inputs": gen_golden.digest(ts), "outputs": outputs}


def compare(rec) -> int:
    import asyncio

    import pytest

    import hostsim_batcher
    from mcp_context_forge_b200 import framework as fw
    from mcp_context_forge_b200.plugins.json_repair import JSONRepairPlugin

    ts = texts(rec["seed"], rec["cases"])
    if gen_golden.digest(ts) != rec["inputs"]:
        print("the generator no longer yields the recorded texts: record the reference again (--record) bad=1")
        return 1
    hostsim_batcher.install(pytest.MonkeyPatch())
    t0 = time.time()
    plug = JSONRepairPlugin(fw.PluginConfig(name="jr", kind="x", hooks=["tool_post_invoke"]))
    ctx = fw.PluginContext(global_context=fw.GlobalContext(request_id="fuzz"))
    bad = repaired = 0
    for i in range(0, len(ts), 500):                            # all calls of a chunk concurrent: they share launches
        async def go():
            return await asyncio.gather(*[plug.tool_post_invoke(fw.ToolPostInvokePayload(name="t", result=t), ctx) for t in ts[i:i + 500]])

        for t, r, d in zip(ts[i:i + 500], gen_golden.run(go()), rec["outputs"][i:i + 500]):
            got = outcome(r)
            repaired += got["modified"]
            if gen_golden.digest(got) != d or (got["modified"] and r.modified_payload.name != "t"):
                bad += 1
                if bad <= 8:
                    print("BAD", repr(t)[:300], "\n   drop-in", repr(got)[:300])
    print(f"seed={rec['seed']} cases={len(ts)} repaired={repaired} bad={bad} time={time.time() - t0:.1f}s")
    return 1 if bad else 0


def main() -> int:
    return gen_golden.fuzz_main("fuzz_json_repair_vs_reference", sys.argv[1:], record, compare)


if __name__ == "__main__":
    sys.exit(main())

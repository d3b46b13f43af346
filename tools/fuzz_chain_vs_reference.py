"""Container-only: the whole product chain against the whole reference chain.  One YAML, two managers: the sequential `PluginManager` loading
the REFERENCE'S OWN plugin classes (kind: plugins.regex_filter.search_replace.SearchReplacePlugin, ... imported unmodified from /root/reference)
and `BatchedPluginManager` loading this repo's drop-ins (kind: mcp_context_forge_b200.plugins....) on the engine's CPU simulator — same priorities,
modes, conditions and hook policies, random waves of concurrent requests on the three hooks of the path, violations as results and as
exceptions.  Every request's (continue_processing, modified payload, violation, metadata) or raised error must be equal.
usage: python tools/fuzz_chain_vs_reference.py [--record OUT] [seed] [rounds] [requests per wave]  |  --replay tests/golden/fuzz_chain.json.gz"""
import asyncio
import json
import os
import random
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, os.path.join(ROOT, "tools"))
import gen_golden  # noqa: E402

OURS = {"harm": "mcp_context_forge_b200.plugins.harmful_content_detector.HarmfulContentDetectorPlugin", "deny": "mcp_context_forge_b200.plugins.deny_filter.DenyListPlugin",
        "regex": "mcp_context_forge_b200.plugins.regex_filter.SearchReplacePlugin", "sql": "mcp_context_forge_b200.plugins.sql_sanitizer.SQLSanitizerPlugin",
        "code": "mcp_context_forge_b200.plugins.code_safety_linter.CodeSafetyLinterPlugin", "repair": "mcp_context_forge_b200.plugins.json_repair.JSONRepairPlugin",
        "toon": "mcp_context_forge_b200.plugins.toon_encoder.ToonEncoderPlugin"}
REFS = {"harm": "plugins.harmful_content_detector.harmful_content_detector.HarmfulContentDetectorPlugin", "deny": "plugins.deny_filter.deny.DenyListPlugin",
        "regex": "plugins.regex_filter.search_replace.SearchReplacePlugin", "sql": "plugins.sql_sanitizer.sql_sanitizer.SQLSanitizerPlugin",
        "code": "plugins.code_safety_linter.code_safety_linter.CodeSafetyLinterPlugin", "repair": "plugins.json_repair.json_repair.JSONRepairPlugin",
        "toon": "plugins.toon_encoder.toon_encoder.ToonEncoderPlugin"}
WORDS = ["hello", "crap", "crud", "innovative", "kill him", "suicide", "normal text", "Kill her", "revolutionary idea", "I want to die", "racial slur", "fine", "DROP table t -- crap",
         "select 1 /* c */", "delete from t", "eval(x)", "rm -rf /", "é", "ſuicide", "日本語", "user@example.com", "12", "update t set a=1", "groundbreaking", "x", "", "bell\x07"]


def config(rng):
    """One random chain: which plugins, their modes / priorities / configs (the same dict rendered with either set of `kind`s)."""
    rules = [["crap", "crud"], ["crud", "yikes"], ["(?i)(kill) (him|her)", r"\2 <\1>"], [r"\d+", "#"], ["a*", "-"], [r"(\w+)@(\w+)\.com", r"\2 at \1"], [r"\s+", " "], ["é", "e"]]
    mode = lambda: rng.choice(["sequential", "sequential", "transform", "audit", "enforce", "enforce_ignore_error", "permissive", "fire_and_forget", "concurrent", "disabled"])   # noqa: E731
    plugs = [
        {"k": "harm", "hooks": ["prompt_pre_fetch", "tool_post_invoke"], "mode": mode(), "priority": rng.choice([96, 40, 500]),
         "config": rng.choice([{}, {"block_on": ["violence"]}, {"categories": {"spam": ["buy now", r"\bfine\b"]}, "block_on": ["spam", "self_harm"]}])},
        {"k": "deny", "hooks": ["prompt_pre_fetch"], "mode": mode(), "priority": 100, "config": {"words": rng.sample(["innovative", "groundbreaking", "revolutionary", "é", "x"], rng.randint(0, 3))}},
        {"k": "regex", "hooks": ["prompt_pre_fetch", "tool_pre_invoke", "tool_post_invoke"], "mode": mode(), "priority": rng.choice([150, 50, 97]),
         "config": {"words": [{"search": s, "replace": r} for s, r in rng.sample(rules, rng.randint(1, 4))]}},
        {"k": "sql", "hooks": ["prompt_pre_fetch", "tool_pre_invoke"], "mode": mode(), "priority": 45, "config": rng.choice([{"block_on_violation": False}, {}, {"strip_comments": False}])},
        {"k": "code", "hooks": ["tool_post_invoke"], "mode": mode(), "priority": rng.choice([120, 30]), "config": {}},
        {"k": "repair", "hooks": ["tool_post_invoke"], "mode": mode(), "priority": 145, "config": {}},
        {"k": "toon", "hooks": ["tool_post_invoke"], "mode": mode(), "priority": 900, "config": rng.choice([{"min_size_bytes": 10}, {}, {"min_size_bytes": 10, "add_format_marker": False}, {"min_size_bytes": 10, "skip_on_error": False}]),
         "conditions": rng.choice([None, [{"tools": ["t", "u"]}]])},
    ]
    conds = [None, None, None, [{"tools": ["t", "u"]}], [{"server_ids": ["s1"]}], [{"tenant_ids": ["acme"]}], [{"user_patterns": ["ali"]}], [{"prompts": ["p"]}, {"tools": ["other"]}],
             [{"server_ids": ["s2"], "tools": ["t"]}], [{"user_patterns": ["bob*", "zed"]}]]
    for p in plugs:
        p["on_error"] = rng.choice(["fail", "fail", "ignore", "disable"])
        if "conditions" not in p:
            p["conditions"] = rng.choice(conds)
    return [p for p in plugs if rng.random() < 0.8]


def render(plugs, kinds, fail_all=False):
    import yaml

    out = []
    for p in plugs:
        d = {"name": p["k"], "kind": kinds[p["k"]], "hooks": p["hooks"], "mode": p["mode"], "priority": p["priority"], "config": p["config"], "on_error": p["on_error"]}
        if p.get("conditions"):
            d["conditions"] = p["conditions"]
        out.append(d)
    return yaml.safe_dump({"plugins": out, "plugin_settings": {"plugin_timeout": 120, "fail_on_plugin_error": fail_all}})


HOOKS = ("prompt_pre_fetch", "tool_pre_invoke", "tool_post_invoke")


def rounds_of(seed: int, rounds: int, nreq: int):
    """The seeded inputs: per round the chain, its settings and `nreq` requests (prompt args, tool name + result, global context)."""
    from mcp_context_forge_b200 import synth

    rng = random.Random(seed)
    out = []
    for rd in range(rounds):
        r_ = {"plugs": config(rng), "fail_all": rng.random() < 0.2, "max_wave": rng.choice([8192, 8192, 7, 1, 33]), "window_us": rng.choice([0, 0, 50, 400]), "args": [], "post": []}
        for i in range(nreq):
            args = {f"k{j}": " ".join(rng.choice(WORDS) for _ in range(rng.randint(1, 6))) for j in range(rng.randint(0, 3))}
            if rng.random() < 0.15:
                args["n"] = rng.randint(0, 9)
            r_["args"].append(args)
            r = rng.random()
            if r < 0.45:
                text = synth.payload("A", rng.choice([300, 1500]), seed=i + rd * 1000) if rng.random() < 0.6 else json.dumps({"note": rng.choice(WORDS), "x": [1, 2, {"y": rng.choice(WORDS)}]})
                result = {"content": [{"type": "text", "text": text}, {"type": "text", "text": rng.choice(WORDS) * 3}], "summary": rng.choice(WORDS) + " crap"}
            elif r < 0.6:
                result = rng.choice(["{'a': 1, 'b': [1, 2,],}", '{"a": "crap", "b": [1, 2, 3]}', "[1, 2, 3,] crap", '"k": "kill him"', "{'x': 'eval(1)'}", "[1,2,3]", "not json " + rng.choice(WORDS)])
            elif r < 0.8:
                result = " ".join(rng.choice(WORDS) for _ in range(rng.randint(0, 8)))
            else:
                result = rng.choice([{"text": rng.choice(WORDS), "other": rng.choice(WORDS)}, None, 5, [rng.choice(WORDS)], {"a": {"b": rng.choice(WORDS)}, "c": [rng.choice(WORDS), 3]}])
            r_["post"].append([rng.choice(["t", "u", "other"]), result])
        r_["gcs"] = [[rng.choice([None, "s1", "s2"]), rng.choice([None, "acme", "other"]), rng.choice([None, "alice", "bob7", "zed"])] for i in range(nreq)]
        out.append(r_)
    return out


def waves(m, r_, loop):
    """Every request of the round through manager `m` on each hook, without and with violations_as_exceptions: normalised results."""
    import test_manager_gpu as tm
    from mcp_context_forge_b200 import framework as fw

    pre = [fw.PromptPrehookPayload(prompt_id="p", args=json.loads(json.dumps(a))) for a in r_["args"]]
    tpre = [fw.ToolPreInvokePayload(name="t", args=json.loads(json.dumps(a))) for a in r_["args"]]
    post = [fw.ToolPostInvokePayload(name=n, result=json.loads(json.dumps(res))) for n, res in r_["post"]]
    gcs = [fw.GlobalContext(request_id=f"r{i}", server_id=s, tenant_id=t, user=u) for i, (s, t, u) in enumerate(r_["gcs"])]
    out = []
    for hook, pls in zip(HOOKS, (pre, tpre, post)):
        for vae in (False, True):
            async def wave():
                return await asyncio.gather(*[m.invoke_hook(hook, p, g, None, vae) for p, g in zip(pls, gcs)], return_exceptions=True)
            out.append([tm.norm(u) for u in loop.run_until_complete(wave())])
    return out


def record(argv):
    seed = int(argv[0]) if len(argv) > 0 else 1
    rounds = int(argv[1]) if len(argv) > 1 else 20
    nreq = int(argv[2]) if len(argv) > 2 else 60
    gen_golden.install_shims()
    import logging

    import test_manager_gpu as tm
    from mcp_context_forge_b200 import framework as fw

    logging.disable(logging.ERROR)
    loop = asyncio.new_event_loop()
    rs = rounds_of(seed, rounds, nreq)
    outputs = []
    for r_ in rs:
        with tempfile.TemporaryDirectory() as td:
            a = os.path.join(td, "ref.yaml")
            with open(a, "w") as f:
                f.write(render(r_["plugs"], REFS, r_["fail_all"]))
            seq = fw.PluginManager(a, timeout=120, hook_policies=tm.POL)
            loop.run_until_complete(seq.initialize())
            outputs.append([[gen_golden.digest(x) for x in w] for w in waves(seq, r_, loop)])
    return {"seed": seed, "rounds": rounds, "requests": nreq, "inputs": gen_golden.digest(rs), "outputs": outputs}


def compare(rec) -> int:
    import logging

    import pytest

    import hostsim_batcher
    import test_manager_gpu as tm
    from mcp_context_forge_b200.manager import BatchedPluginManager
    from mcp_context_forge_b200.regex_frontend import UnsupportedPattern

    rs = rounds_of(rec["seed"], rec["rounds"], rec["requests"])
    if gen_golden.digest(rs) != rec["inputs"]:
        print("the generator no longer yields the recorded inputs: record the reference again (--record) bad=1")
        return 1
    logging.disable(logging.ERROR)
    hostsim_batcher.install(pytest.MonkeyPatch())
    loop = asyncio.new_event_loop()
    t0 = time.time()
    n = bad = rejected = slow = 0
    for r_, exp in zip(rs, rec["outputs"]):
        plugs = r_["plugs"]
        with tempfile.TemporaryDirectory() as td:
            b = os.path.join(td, "ours.yaml")
            with open(b, "w") as f:
                f.write(render(plugs, OURS, r_["fail_all"]))
            bat = BatchedPluginManager(b, timeout=120, hook_policies=tm.POL, max_wave=r_["max_wave"], window_us=r_["window_us"])
            try:
                loop.run_until_complete(bat.initialize())
            except (UnsupportedPattern, RuntimeError) as exc:
                if "Unsupported" not in repr(exc) and "unsupported" not in repr(exc):
                    raise
                rejected += 1
                continue
            for k, (got, want) in enumerate(zip(waves(bat, r_, loop), exp)):
                for i, (v, d) in enumerate(zip(got, want)):
                    n += 1
                    if gen_golden.digest(v) != d:
                        bad += 1
                        if bad <= 5:
                            print("BAD", HOOKS[k // 2], "vae", bool(k & 1), "\n  chain    ", [(p["k"], p["mode"], p["priority"]) for p in plugs], "\n  request  ",
                                  repr((r_["args"][i], r_["post"][i], r_["gcs"][i]))[:400], "\n  product  ", repr(v)[:600])
            slow += bat.slow_path_calls
    print(f"seed={rec['seed']} chains={rec['rounds']} rejected_loudly={rejected} requests={n} slow_path_calls={slow} bad={bad} time={time.time() - t0:.1f}s")
    return 1 if bad or not n else 0


def main() -> int:
    return gen_golden.fuzz_main("fuzz_chain_vs_reference", sys.argv[1:], record, compare)


if __name__ == "__main__":
    sys.exit(main())

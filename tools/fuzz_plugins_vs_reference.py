"""Container-only: live differential fuzz of the drop-in PLUGINS (their host logic — unit extraction, verdict -> result assembly, findings
order, payload rebuilding — on the engine's CPU simulator) against the REFERENCE'S OWN plugin classes, imported unmodified from /root/reference:
regex_filter, deny_filter, harmful_content_detector, sql_sanitizer, code_safety_linter, toon_encoder.  Random configurations (from pools that
include rules matching "", group-reference templates, invalid patterns, IGNORECASE Unicode traps) and random payload shapes (nested dicts /
lists / non-strings, every hook each plugin implements).  A configuration the engine rejects loudly (UnsupportedPattern) is skipped and counted.
usage: python tools/fuzz_plugins_vs_reference.py [--record OUT] [seed] [rounds]  |  --replay tests/golden/fuzz_plugins.json.gz"""
import asyncio
import json
import os
import random
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, os.path.join(ROOT, "tools"))
import gen_golden  # noqa: E402

WORDS = ["kill", "myself", "suicide", "self-harm", "want", "to", "die", "him", "her", "them", "someone", "shoot", "stab", "eradicate", "people", "racial", "slur", "hate", "speech", "crap",
         "crud", "innovative", "groundbreaking", "revolutionary", "the", "a", "of", "x", "Kill", "KILL", "ſuicide", "Kill", "é", "ß", "naïve", "日本語", "\U0001f600", "12", "_", "-", ".",
         ",", "\n", "DROP", "drop table t", "DELETE FROM t", "delete from t where x=1", "UPDATE t SET a=1", "update t set a=1 where b=2", "-- comment", "/* c */", "select * from t",
         "eval(", "exec (", "os.system('x')", "subprocess.run([", "rm -rf /", "'; --", "\"%s\" % x", "f\"{x}\"", "{} + {}", "buy now", "free", "xxy", "user@example.com", "555-1234", "a b",
         "zzz", "TRUNCATE", "alter", "GRANT all", "where", "#", "/*", "*/", "--", ";", "bell\x07", "\x01"]
SEPS = [" ", " ", " ", "", "  ", "\n", "-", "_", ".", "é", "1", "\t", ", "]
RULES = [("crap", "crud"), ("crud", "yikes"), (r"\bkill\b", "[k]"), ("(unclosed", "x"), (r"\d+", "#"), (r"cr[au]p+", "X"), (r"a|ab|abc", "<>"), ("a*", "-"), (r"(a)|b", r"[\1]"), (r"x*", "."),
         (r"(\w+)@(\w+)\.com", r"\2 at \1"), (r"\s+", " "), (r"(?i)kill", "K"), (r"é", "e"), (r"(?P<n>\d)(\d)", r"\g<n>-\2"), (r"^", ">"), (r"$", "<"), (r"\b", "|"), (r"[^\W\d_]+", "w"),
         (r"(a)\1", "bad"), (r"(?=x)", "la"), ("", "+"), (r"日本", "JP"), (r".", "d"), (r"\.", "dot")]
DENY = ["innovative", "groundbreaking", "revolutionary", "a b", "é", "x", "", "zzz", "kill", "Kill", "日本", "\n", "free", "--"]
HARM_CFG = [None, {"block_on": ["violence"]}, {"categories": {"spam": ["buy now", r"\bfree\b"], "x": ["x+y"]}, "block_on": ["spam"]}, {"block_on": []}, {"block_on": ["self_harm", "hate"]},
            {"categories": {"k": [r"k\w+l", "é+"], "w": [r"\bwhere\b"]}, "block_on": ["k", "w", "violence"]}]
import re as _re  # noqa: E402

HARM_CFG += [{"categories": {"c": [_re.compile("Kill"), _re.compile("him", _re.I), "Her"], "d": [_re.compile(r"k.ll\s+h", _re.S | _re.I), _re.compile(r"^die", _re.M)]}, "block_on": ["c", "d"]},
             {"categories": {"e": [_re.compile(r"\bé\w*", _re.I), _re.compile(r"ſ", _re.I), _re.compile(r"(?i)K")]}, "block_on": ["e"]}]
SQL_CFG = [None, {"block_on_violation": False}, {"block_on_violation": False, "require_parameterization": True, "fields": ["sql", "query"]}, {"strip_comments": False},
           {"fields": ["q"], "blocked_statements": [r"\bDROP\b", r"(?i)truncate\s+table"]}, {"require_parameterization": True}, {"block_delete_without_where": False, "block_update_without_where": False}]
CODE_CFG = [None, {"blocked_patterns": [r"curl\s+\S+\s*\|\s*sh", r"(?i)\bdrop\b", r"import\s+os"]}, {"blocked_patterns": []}, {"blocked_patterns": [r"rm\s+-rf", r"é+"]}]
TOON_CFG = [{"min_size_bytes": 10}, {"min_size_bytes": 10, "max_size_bytes": 300}, {"min_size_bytes": 10, "add_format_marker": False}, {"min_size_bytes": 40, "exclude_tools": ["other"]}, {"min_size_bytes": 10, "skip_on_error": False},
            {"min_size_bytes": 10, "skip_on_error": False, "add_format_marker": False}]


def text(rng, n=None):
    return "".join(rng.choice(WORDS) + rng.choice(SEPS) for _ in range(rng.randint(0, 7) if n is None else n))


def value(rng, depth):
    r = rng.random()
    if depth <= 0 or r < 0.45:
        return text(rng)
    if r < 0.55:
        return rng.choice([None, 5, 2.5, True, b"bytes".decode(), ""])
    if r < 0.75:
        return [value(rng, depth - 1) for _ in range(rng.randint(0, 3))]
    return {rng.choice(["sql", "query", "q", "text", "a", "b", "k1", "note", "content"]): value(rng, depth - 1) for _ in range(rng.randint(0, 4))}


def norm(r):
    v = r.violation.model_dump(include={"reason", "description", "code", "details"}) if r.violation is not None else None
    mp = r.modified_payload
    md = {k: x for k, x in (r.metadata or {}).items() if k != "conversion_time_ms"}
    res = getattr(mp, "result", None) if mp is not None else "-"
    if hasattr(res, "model_dump"):
        res = res.model_dump()
    return json.loads(json.dumps({"cont": r.continue_processing, "violation": v, "args": getattr(mp, "args", None) if mp is not None else "-", "result": res,
                                  "metadata": md}, default=str, sort_keys=True))


# plugin -> (the reference's class, this repository's drop-in)
CLASSES = {"regex_filter": ("plugins.regex_filter.search_replace.SearchReplacePlugin", "regex_filter.SearchReplacePlugin"),
           "deny_filter": ("plugins.deny_filter.deny.DenyListPlugin", "deny_filter.DenyListPlugin"),
           "harmful": ("plugins.harmful_content_detector.harmful_content_detector.HarmfulContentDetectorPlugin", "harmful_content_detector.HarmfulContentDetectorPlugin"),
           "sql_sanitizer": ("plugins.sql_sanitizer.sql_sanitizer.SQLSanitizerPlugin", "sql_sanitizer.SQLSanitizerPlugin"),
           "code_safety": ("plugins.code_safety_linter.code_safety_linter.CodeSafetyLinterPlugin", "code_safety_linter.CodeSafetyLinterPlugin"),
           "toon_encoder": ("plugins.toon_encoder.toon_encoder.ToonEncoderPlugin", "toon_encoder.ToonEncoderPlugin")}


def load_class(path):
    import importlib

    mod, _, cls = path.rpartition(".")
    return getattr(importlib.import_module(mod), cls)


def plans(seed: int, rounds: int):
    """The seeded inputs: per round and plugin (name, config, hooks, [(hook, args / result / rendered prompt)])."""
    rng = random.Random(seed)

    def payloads(kind):
        out = []
        for _ in range(24):
            if kind == "args":
                a = value(rng, 3)
                out.append(a if isinstance(a, dict) and rng.random() < 0.9 else {"k": text(rng), "sql": text(rng), "n": 7} if rng.random() < 0.8 else None)
            else:
                r = rng.random()
                out.append(text(rng) if r < 0.3 else value(rng, 3) if r < 0.7 else {"content": [{"type": "text", "text": json.dumps(value(rng, 3), ensure_ascii=False)}, {"type": "image", "data": "A"}], "isError": False})
        return out

    out = []
    for rd in range(rounds):
        plan = [
            ("regex_filter", {"words": [{"search": s, "replace": r} for s, r in rng.sample(RULES, rng.randint(0, 4))]}, ["prompt_pre_fetch", "tool_pre_invoke", "tool_post_invoke", "prompt_post_fetch"]),
            ("deny_filter", {"words": rng.sample(DENY, rng.randint(0, 4))}, ["prompt_pre_fetch"]),
            ("harmful", rng.choice(HARM_CFG), ["prompt_pre_fetch", "tool_post_invoke"]),
            ("sql_sanitizer", rng.choice(SQL_CFG), ["prompt_pre_fetch", "tool_pre_invoke"]),
            ("code_safety", rng.choice(CODE_CFG), ["tool_post_invoke"]),
            ("toon_encoder", rng.choice(TOON_CFG), ["tool_post_invoke"]),
        ]
        for name, cfg, hooks in plan:
            calls = []
            for hook in hooks:
                for p in payloads("args" if hook in ("prompt_pre_fetch", "tool_pre_invoke") else "result"):
                    if hook == "prompt_post_fetch":                                       # a rendered prompt: messages with text content
                        p = {"messages": [{"role": rng.choice(["user", "assistant"]), "content": {"type": "text", "text": text(rng)}} for _ in range(rng.randint(0, 4))]}
                    calls.append((hook, p))
            out.append((name, cfg, hooks, calls))
    return out


def make_payload(fw, hook, p):
    if hook == "prompt_post_fetch":
        return fw.PromptPosthookPayload(prompt_id="p", result=json.loads(json.dumps(p)))
    if hook == "prompt_pre_fetch":
        return fw.PromptPrehookPayload(prompt_id="p", args=p)
    if hook == "tool_pre_invoke":
        return fw.ToolPreInvokePayload(name="t", args=p)
    return fw.ToolPostInvokePayload(name="t", result=p)


def outcomes(fw, plug, calls, loop):
    """Per call the normalised result or the raised error (None: the payload model rejects the input), then the plugin's counters."""
    ctx = fw.PluginContext(global_context=fw.GlobalContext(request_id="fuzz"))
    out = []
    for hook, p in calls:
        try:
            pl = make_payload(fw, hook, p)
        except Exception:  # noqa: BLE001 - a payload shape the model rejects
            out.append(None)
            continue
        try:
            out.append(norm(loop.run_until_complete(getattr(plug, hook)(pl, ctx))))
        except Exception as exc:  # noqa: BLE001 - the reference raises: so must the drop-in
            out.append({"raises": type(exc).__name__, "message": str(exc)})
    return out, (plug.get_stats() if callable(getattr(plug, "get_stats", None)) else None)


def record(argv):
    seed = int(argv[0]) if len(argv) > 0 else 1
    rounds = int(argv[1]) if len(argv) > 1 else 40
    gen_golden.install_shims()
    import cpex.framework as fw

    loop = asyncio.new_event_loop()
    ps = plans(seed, rounds)
    outputs = []
    for name, cfg, hooks, calls in ps:
        res, stats = outcomes(fw, load_class(CLASSES[name][0])(fw.PluginConfig(name=name, kind="x", hooks=hooks, config=cfg)), calls, loop)
        outputs.append([[None if r is None else gen_golden.digest(r) for r in res], None if stats is None else gen_golden.digest(stats)])
    return {"seed": seed, "rounds": rounds, "inputs": gen_golden.digest(ps), "outputs": outputs}


def compare(rec) -> int:
    import pytest

    import hostsim_batcher
    from mcp_context_forge_b200 import framework as fw
    from mcp_context_forge_b200.regex_frontend import UnsupportedPattern

    ps = plans(rec["seed"], rec["rounds"])
    if gen_golden.digest(ps) != rec["inputs"]:
        print("the generator no longer yields the recorded inputs: record the reference again (--record) bad=1")
        return 1
    hostsim_batcher.install(pytest.MonkeyPatch())
    loop = asyncio.new_event_loop()
    t0 = time.time()
    n = bad = rejected = raised = 0
    for (name, cfg, hooks, calls), (exp, exp_stats) in zip(ps, rec["outputs"]):
        try:
            ours = load_class("mcp_context_forge_b200.plugins." + CLASSES[name][1])(fw.PluginConfig(name=name, kind="x", hooks=hooks, config=cfg))
        except UnsupportedPattern:
            rejected += 1
            continue
        got, stats = outcomes(fw, ours, calls, loop)
        for (hook, p), e, g in zip(calls, exp, got):
            if e is None and g is None:
                continue
            n += 1
            raised += isinstance(g, dict) and "raises" in g
            if g is None or gen_golden.digest(g) != e:
                bad += 1
                if bad <= 6:
                    print("BAD", name, hook, repr(cfg)[:300], "\n  payload  ", repr(p)[:400], "\n  drop-in  ", json.dumps(g, ensure_ascii=False)[:500])
        if exp_stats is not None:                              # toon_encoder's counters after the same calls
            n += 1
            if stats is None or gen_golden.digest(stats) != exp_stats:
                bad += 1
                if bad <= 6:
                    print("BAD stats", name, repr(cfg), stats)
    print(f"seed={rec['seed']} rounds={rec['rounds']} hook_calls={n} configs_rejected_loudly={rejected} drop_in_raised={raised} bad={bad} time={time.time() - t0:.1f}s")
    return 1 if bad or not n else 0


def main() -> int:
    return gen_golden.fuzz_main("fuzz_plugins_vs_reference", sys.argv[1:], record, compare)


if __name__ == "__main__":
    sys.exit(main())

#!/usr/bin/env python
"""Generate tests/golden/*.json by running the reference's OWN code (unmodified files under
/root/reference) in this container.  /root/reference does not exist on the GPU box, so the vectors
are committed; this script is the provenance.

How the reference code is made importable here (SURVEY.md §8c):
  * `cpex.framework`  -> mcp_context_forge_b200.cpex_compat (restated surface; cpex 0.1.0 is not installable)
  * `orjson`          -> tiny stand-in over stdlib json (loads/dumps/JSONDecodeError); inputs that would
                         expose orjson/json deltas (ints beyond u64, NaN literals) are not used in vectors
  * `mcpgateway.services.logging_service` -> stub LoggingService (deny.py:16 only needs a logger)
  * masking twin: the pure functions of mcpgateway/middleware/request_logging_middleware.py:83-291 are
    exec'd from the file's own source text (the module itself needs fastapi/sqlalchemy).

Run:  python tools/gen_golden.py        (writes tests/golden/*.json)
"""
from __future__ import annotations

import ast
import asyncio
import gzip
import hashlib
import json
import logging
import os
import random
import re
import sys
import types

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = "/root/reference"
sys.path.insert(0, ROOT)
OUT = os.path.join(ROOT, "tests", "golden")


def install_shims():
    from mcp_context_forge_b200.cpex_compat import install_as_cpex

    install_as_cpex(force=True)
    if "orjson" not in sys.modules:
        oj = types.ModuleType("orjson")

        class JSONDecodeError(ValueError):
            pass

        def loads(s):
            if isinstance(s, (bytes, bytearray, memoryview)):
                s = bytes(s).decode("utf-8")
            try:
                return json.loads(s, parse_constant=lambda c: (_ for _ in ()).throw(ValueError(c)))
            except ValueError as exc:
                raise JSONDecodeError(str(exc)) from exc

        def dumps(o):
            return json.dumps(o, separators=(",", ":"), ensure_ascii=False).encode("utf-8")

        oj.loads, oj.dumps, oj.JSONDecodeError = loads, dumps, JSONDecodeError
        sys.modules["orjson"] = oj
    for name in ("mcpgateway", "mcpgateway.services"):
        if name not in sys.modules:
            m = types.ModuleType(name)
            m.__path__ = []
            sys.modules[name] = m
    ls = types.ModuleType("mcpgateway.services.logging_service")

    class LoggingService:
        def get_logger(self, name):
            return logging.getLogger(name)

    ls.LoggingService = LoggingService
    sys.modules["mcpgateway.services.logging_service"] = ls
    if REF not in sys.path:
        sys.path.insert(0, REF)


def run(coro):
    return asyncio.new_event_loop().run_until_complete(coro)


def dump(name, obj):
    os.makedirs(OUT, exist_ok=True)
    path = os.path.join(OUT, name)
    with open(path, "w", encoding="utf-8") as f:
        json.dump(obj, f, ensure_ascii=True, indent=0, separators=(",", ":"))
        f.write("\n")
    print(f"wrote {path}: {os.path.getsize(path)} bytes")


def digest(obj) -> str:
    """32-bit digest of a value's canonical JSON (dict order ignored, as `==` does).  A fuzzer's recording keeps the reference's output
    for each case as this digest, and its inputs as the digest of the whole seeded sequence, which the fuzzer regenerates."""
    data = json.dumps(obj, ensure_ascii=True, sort_keys=True, separators=(",", ":"), default=repr).encode()
    return hashlib.sha256(data).hexdigest()[:8]


def save_recording(path, obj):
    """A differential fuzzer's recorded run as gzip-compressed JSON, byte-reproducible."""
    data = json.dumps(obj, ensure_ascii=True, separators=(",", ":")).encode()
    with open(path, "wb") as f:
        f.write(gzip.compress(data, compresslevel=9, mtime=0))
    print(f"wrote {path}: {os.path.getsize(path)} bytes")


def load_recording(path):
    with open(path, "rb") as f:
        return json.loads(gzip.decompress(f.read()))


def fuzz_main(name, argv, record, compare):
    """Command line of the differential fuzzers.  `[args]`: run the reference live and compare; `--record OUT [args]`: write the
    reference's side of the run to OUT; `--replay IN`: compare this repository against a recording (the reference is not needed)."""
    if argv[:1] == ["--replay"]:
        return compare(load_recording(argv[1]))
    out = None
    if argv[:1] == ["--record"]:
        out, argv = argv[1], argv[2:]
    if not os.path.isdir(REF):
        print(f"{name}: the reference checkout ({REF}) is not here; compare against a recording with --replay")
        return 0 if out is None else 1
    rec = record(argv)
    if out is not None:
        save_recording(out, rec)
        return 0
    return compare(rec)


# ------------------------------------------------------------------------------------------------
def rand_text(rng, n):
    words = ["kill", "myself", "suicide", "self-harm", "want", "to", "die", "him", "her", "them", "someone", "shoot", "stab", "eradicate", "people",
             "racial", "slur", "hate", "speech", "crap", "crud", "innovative", "groundbreaking", "revolutionary", "the", "a", "of", "x", "Kill", "KILL",
             "ſuicide", "Kill", "é", "ß", "naïve", "日本語", "\U0001f600", "12", "_", "-", ".", ",", "\n"]
    seps = [" ", " ", " ", "", "  ", "\n", "-", "_", ".", "é", "1"]
    return "".join(rng.choice(words) + rng.choice(seps) for _ in range(n))


def gen_pattern_plugins():
    from cpex.framework import GlobalContext, PluginConfig, PluginContext, PromptPrehookPayload, ToolPostInvokePayload, ToolPreInvokePayload
    from plugins.deny_filter.deny import DenyListPlugin
    from plugins.harmful_content_detector.harmful_content_detector import HarmfulContentDetectorPlugin
    from plugins.regex_filter.search_replace import SearchReplacePlugin

    ctx = PluginContext(global_context=GlobalContext(request_id="golden"))
    rng = random.Random(2024)
    out = {"regex_filter": [], "deny_filter": [], "harmful": []}

    # ---- regex_filter (plugins/regex_filter/search_replace.py)
    rule_sets = [
        [{"search": "crap", "replace": "crud"}, {"search": "crud", "replace": "yikes"}],          # plugins/config.yaml:149-153
        [{"search": r"\bkill\b", "replace": "[k]"}, {"search": "(unclosed", "replace": "x"}, {"search": r"\d+", "replace": "#"}],
        [{"search": r"cr[au]p+", "replace": "X"}, {"search": r"a|ab|abc", "replace": "<>"}],
        [{"search": r"\s{2,}", "replace": " "}, {"search": r"[^a-z\s]+", "replace": "·"}],
    ]
    for rules in rule_sets:
        plug = SearchReplacePlugin(PluginConfig(name="rf", kind="x", hooks=["tool_pre_invoke", "tool_post_invoke"], config={"words": rules}))
        cases = []
        for i in range(40):
            args = {f"k{j}": rand_text(rng, rng.randint(0, 12)) for j in range(rng.randint(0, 4))}
            if i % 5 == 0:
                args["n"] = 7
                args["nested"] = {"x": "crap"}
            r = run(plug.tool_pre_invoke(ToolPreInvokePayload(name="t", args=args), ctx))
            cases.append({"hook": "tool_pre_invoke", "args": args, "out_args": r.modified_payload.args})
        for i in range(20):
            res = rand_text(rng, rng.randint(0, 20)) if i % 2 else {"a": rand_text(rng, 8), "content": [{"type": "text", "text": "crap"}], "b": "crap crud"}
            r = run(plug.tool_post_invoke(ToolPostInvokePayload(name="t", result=res), ctx))
            cases.append({"hook": "tool_post_invoke", "result": res, "out_result": r.modified_payload.result})
        out["regex_filter"].append({"words": rules, "cases": cases})

    # ---- deny_filter (plugins/deny_filter/deny.py)
    for words in (["innovative", "groundbreaking", "revolutionary"], ["a b", "é", "x"], ["", "zzz"], []):
        plug = DenyListPlugin(PluginConfig(name="dl", kind="x", hooks=["prompt_pre_fetch"], config={"words": words}))
        cases = []
        for i in range(40):
            args = {f"k{j}": rand_text(rng, rng.randint(0, 10)) for j in range(rng.randint(0, 4))}
            r = run(plug.prompt_pre_fetch(PromptPrehookPayload(prompt_id="p", args=args), ctx))
            cases.append({"args": args, "blocked": not r.continue_processing,
                          "violation": r.violation.model_dump(exclude={"plugin_name", "http_status_code", "mcp_error_code", "http_headers"}) if r.violation else None})
        out["deny_filter"].append({"words": words, "cases": cases})

    # ---- harmful_content_detector (plugins/harmful_content_detector/harmful_content_detector.py)
    configs = [None, {"block_on": ["violence"]}, {"categories": {"spam": [r"buy now", r"\bfree\b"], "x": [r"x+y"]}, "block_on": ["spam"]}]
    for cfg in configs:
        plug = HarmfulContentDetectorPlugin(PluginConfig(name="hc", kind="x", hooks=["tool_post_invoke"], config=cfg))
        cases = []
        for i in range(80):
            kind = i % 4
            if kind == 0:
                result = rand_text(rng, rng.randint(0, 25))
            elif kind == 1:
                result = {"content": [{"type": "text", "text": rand_text(rng, rng.randint(0, 25))}, {"type": "text", "text": rand_text(rng, 5)}], "isError": False,
                          "meta": {"note": rand_text(rng, 6), "n": 3, "buy now": "free"}}
            elif kind == 2:
                result = [rand_text(rng, 6), {"a": [rand_text(rng, 6), 5, None]}, "buy now FREE xxy"]
            else:
                result = 12345
            r = run(plug.tool_post_invoke(ToolPostInvokePayload(name="t", result=result), ctx))
            cases.append({"result": result, "continue_processing": r.continue_processing, "metadata": r.metadata,
                          "violation": r.violation.model_dump(exclude={"plugin_name", "http_status_code", "mcp_error_code", "http_headers"}) if r.violation else None})
        out["harmful"].append({"config": cfg, "cases": cases})
    dump("pattern_plugins.json", out)


# ------------------------------------------------------------------------------------------------
def harvest_test_literals(path):
    """Every literal passed to encode()/assigned to `data` in the reference's own TOON tests."""
    tree = ast.parse(open(path, encoding="utf-8").read())
    found = []
    for node in ast.walk(tree):
        cands = []
        if isinstance(node, ast.Assign) and any(isinstance(t, ast.Name) and t.id in ("data", "original", "obj", "arr") for t in node.targets):
            cands.append(node.value)
        if isinstance(node, ast.Call) and getattr(node.func, "id", "") in ("encode", "toon_encode") and node.args:
            cands.append(node.args[0])
        for c in cands:
            try:
                found.append(ast.literal_eval(c))
            except Exception:
                pass
    return found


def jsonable(o):
    if isinstance(o, tuple):
        return [jsonable(x) for x in o]
    if isinstance(o, list):
        return [jsonable(x) for x in o]
    if isinstance(o, dict):
        return {str(k): jsonable(v) for k, v in o.items()}
    return o


def rand_json(rng, depth):
    r = rng.random()
    if depth <= 0 or r < 0.3:
        t = rng.random()
        if t < 0.25:
            return rng.choice(["", "a", "hello world", "has,comma", "x:y", "-5", "05", "1e5", "1E5", "+1", ".5", "0x1", "null", "true", "True", " lead", "trail ",
                               "q\"uote", "back\\slash", "tab\tx", "nl\nx", "cr\rx", "a-b", "-", "[x]", "{y}", "été", "日本", " nbsp", "1٢", "3.14",
                               "-0", "0", "00", "1.", "1.0", "ctrl\x01x", "user1@example.com", "2024-01-01", "n/a"])
        if t < 0.5:
            return rng.choice([0, 1, -1, 42, -17, 10**6, 2**31, 2**53 + 1, -(2**63), 2**64 - 1, 123456789012345678])
        if t < 0.8:
            return rng.choice([0.0, -0.0, 1.0, -2.5, 3.14, 1e-7, 1.5e-7, -1e-20, 1e-20, 1e15, 1e16, 1e21, 1.7976931348623157e308, 5e-324, 0.1 + 0.2, 1 / 3, 2 / 3,
                               99999999999999.98, 1234567890123456.5, 123456.789, round(rng.uniform(0, 100), 2), rng.uniform(-1e6, 1e6), rng.random() * 1e-5, 100.0, 1e100])
        return rng.choice([True, False, None])
    if r < 0.6:
        n = rng.randint(0, 5)
        style = rng.random()
        if style < 0.4:   # homogeneous rows (columnar candidates)
            keys = [rng.choice(["id", "name", "v", "has space", "k-2", "null", "a.b", "_x", "9z", ""]) for _ in range(rng.randint(1, 4))]
            rows = []
            for _ in range(n):
                ks = list(keys)
                if rng.random() < 0.2:
                    rng.shuffle(ks)
                row = {k: rand_json(rng, 0) for k in ks}
                if rng.random() < 0.1:
                    row["extra"] = 1
                if rng.random() < 0.1 and row:
                    row[next(iter(row))] = rand_json(rng, 1)
                rows.append(row)
            return rows
        return [rand_json(rng, depth - 1) for _ in range(n)]
    return {rng.choice(["a", "b", "key", "has space", "with:colon", "null", "true", "x.y", "_p", "1n", "", "k,c", "tab\tk", "é", "list", "obj", "id", "name"]): rand_json(rng, depth - 1)
            for _ in range(rng.randint(0, 5))}


def gen_toon():
    import importlib.util

    spec = importlib.util.spec_from_file_location("ref_toon", os.path.join(REF, "plugins/toon_encoder/toon.py"))
    toon = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(toon)
    from cpex.framework import GlobalContext, PluginConfig, PluginContext, ToolPostInvokePayload
    from plugins.toon_encoder.toon_encoder import ToonEncoderPlugin

    rng = random.Random(77)
    inputs = harvest_test_literals(os.path.join(REF, "tests/unit/plugins/toon_encoder/test_toon.py"))
    inputs += harvest_test_literals(os.path.join(REF, "tests/unit/plugins/toon_encoder/test_toon_encoder.py"))
    n_harvested = len(inputs)
    # SURVEY.md Appendix A-6 crash/quirk cases and layout quirks
    inputs += [
        {"meta": {"deep": {"arr": [{"x": 1, "y": [1, 2]}, {"x": 2, "y": []}]}}},
        [{"x": [1, 2]}, 5], [{"x": [{"p": 1}, 3]}, 5], [{"x": [{"p": 1}, {"p": 2}]}, 5], [{"x": [{"p": 1}, {"p": 2}], "y": [3, 4]}, 5],
        [{}, {"a": {}}, {"a": []}, []], {"e": {}, "l": [], "n": None}, [[]], [[], [1]], [[1, [2, [3, [4]]]]], {"a": [[1, 2], [3]]},
        [{"a": {"b": {"c": [{"d": 1}]}}}], {"has space": [{"a b": 1, "c": 2}, {"a b": 3, "c": 4}]}, [{"a": 1, "b": 2}, {"b": 3, "a": 4}], [{"a": 1}, {"b": 1}],
        [{"a": 1, "b": [1]}, {"a": 2, "b": [2]}], {"k": "ctrl\x01"}, ["ctrl\x02"], {"ctrl\x03k": 1}, [{"c": "ok"}, {"c": "bad\x04"}],
        [1.0, 2.5, -0.0, 1e21, 1e-7], {"f": 1.7976931348623157e308}, {"t": (1, 2)}, [True, 1, 1.0, "1"],
    ]
    # keys the reference emits unquoted with a RAW newline (its `$` admits a final "\n"; columnar header fields are never quoted): what follows
    # the newline is re-indented by every enclosing level that re-splits the nested text (ADVICE r1)
    newline_keys = [
        {"x": {"abc\n": 1}}, {"x": [[{"a\nb": 1}, {"a\nb": 2}]]}, {"x": {"y": [{"k\n": 1}, {"k\n": 2}]}}, {"a": {"b\nc": {"d\ne": 2}}}, [{"abc\n": 1, "z\n": {"q\n": 2}}],
        [{"k": [{"a\n b ": 1, "c": 2}, {"a\n b ": 3, "c": 4}], "m\n": [1, 2]}], {"p": [{"t\n": [{"u\nv": 1}, {"u\nv": 2}]}]}, {"o\n": {"i\n": {"j\n": [1, {"k\n": 2}]}}},
        [[{"h\n\nh": "v"}], {"w\n  y\t\n z ": 1}], {"L": [{"first": [{"\u00a0x\n\u2003y ": 1}], "second\n": 2}]},
    ]
    for _ in range(700):
        inputs.append(rand_json(rng, rng.randint(1, 5)))
    inputs += newline_keys          # appended: the vectors recorded in earlier rounds keep their positions
    enc_cases = []
    for obj in inputs:
        try:
            j = json.dumps(jsonable(obj), ensure_ascii=False)
        except (TypeError, ValueError):
            continue
        obj = json.loads(j)          # what a JSON parser hands to encode(): lists, never tuples
        try:
            res = {"toon": toon.encode(obj)}
        except Exception as exc:  # AttributeError crash path (A-6 iv) / ValueError control chars
            res = {"error": type(exc).__name__}
        enc_cases.append({"json": j, **res})
    helper = {
        "needs_quotes": [[s, toon._needs_quotes(s)] for s in ["", "null", "hello", "hello world", "has,comma", "123", "05", "-a", "-", " leading", "1E5", "+1", ".5", "0x1", "1٢",
                                                                "a-b", "x ", " x", "\x1cx", "x\x1f", "t\tx", "1.", "1.5e+3", "-0", "00", "0", "true", "True"]],
        "encode_key": [[s, toon._encode_key(s)] for s in ["simple", "has space", "with:colon", "_private", "camelCase", "with.dot", "name123", "123numeric", "key,comma", "null", "", "é", "a-b", "a\"b"]],
        "encode_float": [[repr(x), toon._encode_float(x)] for x in [0.0, -0.0, 1.0, 3.14, -2.5, 1e-20, -1e-20, 1.5e-7, 1 / 3, 99999999999999.98, 0.1 + 0.2, 1234567890123456.5, 1e15, 1e16,
                                                                   1e21, 1e22, 1.7976931348623157e308, 5e-324, 2.5e-5, 123456789.123456789, float("nan"), float("inf"), float("-inf"), 1e100, 4.35, 0.000123456789012345678]],
    }
    # plugin level (plugins/toon_encoder/toon_encoder.py:122-326)
    ctx = PluginContext(global_context=GlobalContext(request_id="golden"))
    plug_cases = []
    cfgs = [None, {"min_size_bytes": 10}, {"min_size_bytes": 10, "max_size_bytes": 300}, {"min_size_bytes": 10, "add_format_marker": False}, {"exclude_tools": ["t"]}, {"include_tools": ["other"]},
            {"min_size_bytes": 10, "skip_on_error": False}]
    texts = [c["json"] for c in enc_cases if len(c["json"]) > 10][:: max(1, len(enc_cases) // 120)]
    sys.path.insert(0, ROOT)
    from mcp_context_forge_b200 import synth

    texts += [synth.payload("A", 600, seed=1), synth.payload("B", 600, seed=2), "not json", "{\"a\": 1", "[1, 2, 3]", "\"just a string that is long enough to pass the size gate\"", "  {\"padded\": [1,2,3,4,5,6,7,8,9,10]}  "]
    for cfg in cfgs:
        plug = ToonEncoderPlugin(PluginConfig(name="toon", kind="x", hooks=["tool_post_invoke"], config=cfg))
        cases = []
        for i, t in enumerate(texts):
            item = {"type": "text", "text": t}
            if i % 3 == 1:
                item["annotations"] = {"audience": ["user"]}
            if i % 3 == 2:
                item["annotations"] = None
                item["_meta"] = {"x": 1}
            result = {"content": [item, {"type": "image", "data": "AAAA"}, {"type": "text", "text": 5}], "isError": False}
            try:
                r = run(plug.tool_post_invoke(ToolPostInvokePayload(name="t", result=result), ctx))
                md = dict(r.metadata or {})
                md.pop("conversion_time_ms", None)
                cases.append({"result": result, "modified": r.modified_payload.result if r.modified_payload else None, "metadata": md})
            except Exception as exc:
                cases.append({"result": result, "raises": type(exc).__name__, "message": str(exc)})
        non_dict = run(plug.tool_post_invoke(ToolPostInvokePayload(name="t", result="str result"), ctx))
        plug_cases.append({"config": cfg, "cases": cases, "stats": plug.get_stats(), "non_dict_modified": non_dict.modified_payload is not None})
    dump("toon.json", {"n_harvested_from_reference_tests": n_harvested, "encode": enc_cases, "helpers": helper, "plugin": plug_cases})


# ------------------------------------------------------------------------------------------------
def load_masking_twin():
    src = open(os.path.join(REF, "mcpgateway/middleware/request_logging_middleware.py"), encoding="utf-8").read().split("\n")
    start = next(i for i, l in enumerate(src) if l.startswith("SENSITIVE_KEYS = frozenset("))
    end = next(i for i, l in enumerate(src) if l.startswith("def _load_rust_request_logging_module"))
    code = "\n".join(src[start:end])
    ns = {"re": re, "orjson": sys.modules["orjson"], "settings": types.SimpleNamespace(experimental_rust_request_logging_masking_enabled=False),
          "logger": logging.getLogger("twin"), "SecurityValidator": None}
    exec(compile(code, "request_logging_middleware_twin", "exec"), ns)
    return ns


def gen_masking():
    ns = load_masking_twin()
    rng = random.Random(5)
    keys = ["password", "db_password", "clientSecret", "auth-token", "X-Api-Key", "X-Auth-Device", "X-Custom-JWT", "sessionToken", "authDevice", "privateKey", "APIKey", "Authorization",
            "__ClientSecret__", "auth-token---", "token", "passwordHash", "jwt", "o_auth", "ÉtokenÉ", "token_count", "tokenizer", "!!!", "X-Token-Count", "X-Auth-Count",
            "X-JWT_Status_Count", "auth_count", "api_key_id", "author", "secrets", "my_secret_name", "JWTToken", "a1B", "accessTokenTTL", "refresh_token_ttl", "tokens", "keyPrivate",
            "private_key_path", "jwt_id", "authz", "oauth", "", "_", "Cookie", "cookie", "X-Request-Id", "apiKey", "api-key", "API_KEY", "accessToken", "refreshToken", "client_secret",
            "jwtToken", "AUTH", "Auth0", "auth1Token", "secretKey", "topSecretValue", "passphrase", "pass_phrase", "user_password_length", "password_ms", "auth_url", "tokenURL",
            "HTTPAuth", "basicAUTH", "x", "ID", "key", "private", "privateKEY", "PrivateKeyPEM", "session", "sessionId", "name_secret", "type_token", "token_type"]
    classifier = [[k, ns["_normalize_key_for_masking"](k), ns["_is_sensitive_key"](k)] for k in keys]

    def rand_obj(depth):
        r = rng.random()
        if depth <= 0 or r < 0.3:
            return rng.choice(["v", 1, 2.5, True, None, "secret-value", -7, 1e16, 0.1, 10**15, "é", "q\"\\\n\t\x01/", 1.0, 100.0, 1e-7, 123456789012])
        if r < 0.55:
            return [rand_obj(depth - 1) for _ in range(rng.randint(0, 4))]
        return {rng.choice(keys): rand_obj(depth - 1) for _ in range(rng.randint(0, 5))}

    data_cases = []
    for i in range(150):
        obj = rand_obj(rng.randint(1, 6))
        for md in (10, 3, 1, 0):
            data_cases.append({"data": obj, "max_depth": md, "masked": ns["mask_sensitive_data"](obj, md)})
    # the reference's own parity vectors (tests/performance/test_request_logging_masking_native_extension_benchmark.py:174-190)
    for obj in [{"password": "secret", "nested": {"authToken": "abc", "count": 3}}, {"level": {"nested": {}}}, [{"apikey": "key1"}, {"data": "safe"}], "plain string",
                {"username": "john", "password": "secret123"}, {"user": {"name": "john", "token": "abc123"}}]:
        for md in (10, 1):
            data_cases.append({"data": obj, "max_depth": md, "masked": ns["mask_sensitive_data"](obj, md)})
    cookies = ["jwt_token=abc; theme=dark; session_id=xyz", "theme=dark", "", "a=b;c", " SESSION = 1 ;; x=y", "Auth=1;AUTHX=2;nope=3", "tokén=1; TOKEN=2", "noequals; jwt", "a=b=c; token=d=e",
               "\x1ctoken=1", "user=john; preference=light", "session_id=xyz; auth_token=secret", "jwt_token=abc123; theme=dark"]
    cookie_cases = [[c, ns["mask_jwt_in_cookies"](c)] for c in cookies]
    header_cases = []
    for i in range(40):
        h = {rng.choice(keys + ["Cookie", "cookie", "COOKIE", "Content-Type", "Accept"]): rng.choice(cookies + ["Bearer abc", "application/json"]) for _ in range(rng.randint(0, 6))}
        header_cases.append({"headers": h, "masked": ns["mask_sensitive_headers"](h)})
    dump("masking_twin.json", {"classifier": classifier, "mask_sensitive_data": data_cases, "cookies": cookie_cases, "headers": header_cases})


# ------------------------------------------------------------------------------------------------
def gen_sql_sanitizer():
    """plugins/sql_sanitizer/sql_sanitizer.py through its two hooks (SURVEY §8 row f-3)."""
    from cpex.framework import GlobalContext, PluginConfig, PluginContext, PromptPrehookPayload, ToolPreInvokePayload
    from plugins.sql_sanitizer.sql_sanitizer import SQLSanitizerPlugin

    ctx = PluginContext(global_context=GlobalContext(request_id="golden"))
    rng = random.Random(4242)
    frags = ["SELECT * FROM t", "select a, b from t where a = 1", "DROP TABLE users", "drop", "dropped", "Truncate x", "ALTER\ttable", "grant all", "REVOKE",
             "DELETE FROM t", "delete\n from t WHERE id=1", "DELETE  FROM", "deletefrom", "UPDATE t SET a=1", "update  é SET", "UPDATE ", "update t set a=1 where b=2",
             "nowhere", "WHERE", "-- comment", "--", "-", "a -- b\nc", "/* block */", "/* multi\nline */", "/*", "*/", "/*/", "/**/", "x /* DROP */ y",
             "-- DROP\n", "/* where */", "'a' + b", "%s", "%.2f", "{name}", "{", "}", "f\"{x}\"", ";", " ", "\n", "\r\n", "é", "ſelect", "İ", "K", "\u212a", "日本語", ""]

    def text():
        return rng.choice(["", " ", "\n", "; "]).join(rng.choice(frags) for _ in range(rng.randint(0, 5)))

    def value(d):
        r = rng.random()
        if d <= 0 or r < 0.5:
            return text()
        if r < 0.6:
            return rng.choice([7, None, True, 2.5])
        if r < 0.8:
            return {rng.choice(["sql", "query", "q", "note"]): value(d - 1) for _ in range(rng.randint(0, 3))}
        return [rng.choice([text(), {rng.choice(["sql", "q"]): value(d - 1)}, [text()], 5]) for _ in range(rng.randint(0, 3))]

    configs = [
        None,
        {"fields": None, "blocked_statements": _SQL_DEFAULT, "block_delete_without_where": True, "block_update_without_where": True, "strip_comments": True,
         "require_parameterization": False, "block_on_violation": True},                                    # tests/unit/plugins/test_sql_sanitizer.py:22-37
        {"block_on_violation": False},
        {"block_on_violation": False, "require_parameterization": True, "fields": ["sql", "query"]},
        {"strip_comments": False, "require_parameterization": True},
        {"strip_comments": False, "block_on_violation": False, "block_delete_without_where": False},
        {"blocked_statements": [r"\bEXEC(?:UTE)?\b", r"xp_\w+", r";\s*--"], "block_update_without_where": False, "block_on_violation": False},
        {"blocked_statements": [], "block_on_violation": False, "fields": []},
    ]
    out = []
    for cfg in configs:
        plug = SQLSanitizerPlugin(PluginConfig(name="sql", kind="x", hooks=["prompt_pre_fetch", "tool_pre_invoke"], config=cfg))
        cases = []
        fixed = [{"path": "sql.txt", "edits": [{"new": "DROP table tab1;", "old": "DROP table tab1;"}], "dry_run": False}, {"message": "DROP table asdf"},
                 {}, {"sql": "select 1 -- x", "nested": {"sql": "/* c */ select 2", "deep": {"query": "DELETE FROM t -- where"}}},
                 {"sql": ["DROP x", "ok -- c", {"sql": "update t set a=1 /* where */"}], "query": "a + b"}]
        for i in range(90):
            args = fixed[i] if i < len(fixed) else {rng.choice(["sql", "query", "q", "other"]): value(3) for _ in range(rng.randint(0, 4))}
            hook = "tool_pre_invoke" if i % 2 == 0 else "prompt_pre_fetch"
            if hook == "tool_pre_invoke":
                r = run(plug.tool_pre_invoke(ToolPreInvokePayload(name="t", args=args), ctx))
            else:
                r = run(plug.prompt_pre_fetch(PromptPrehookPayload(prompt_id="p", args=args), ctx))
            cases.append({"hook": hook, "args": args, "continue_processing": r.continue_processing, "metadata": r.metadata,
                          "out_args": r.modified_payload.args if r.modified_payload is not None else None,
                          "violation": r.violation.model_dump(exclude={"plugin_name", "http_status_code", "mcp_error_code", "http_headers"}) if r.violation else None})
        out.append({"config": cfg, "cases": cases})
    dump("sql_sanitizer.json", out)


_SQL_DEFAULT = [r"\bDROP\b", r"\bTRUNCATE\b", r"\bALTER\b", r"\bGRANT\b", r"\bREVOKE\b"]


# ------------------------------------------------------------------------------------------------
def gen_regex_filter_templates():
    """plugins/regex_filter/search_replace.py with rules whose patterns can match "" and whose replacements reference groups
    (SURVEY Appendix A-1): recorded from the reference's own plugin file."""
    from cpex.framework import GlobalContext, PluginConfig, PluginContext, ToolPostInvokePayload, ToolPreInvokePayload
    from plugins.regex_filter.search_replace import SearchReplacePlugin

    ctx = PluginContext(global_context=GlobalContext(request_id="golden"))
    rng = random.Random(777)
    rule_sets = [
        [{"search": r"(\w+)@(\w+)\.com", "replace": r"\2 at \1"}, {"search": r"\b(\d{3})-(\d{4})\b", "replace": r"***-\2"}],
        [{"search": r"(?P<word>crap|crud)", "replace": r"[\g<word>]"}, {"search": r"\[(\w+)\]", "replace": r"\1\1"}],
        [{"search": r"x*", "replace": "-"}, {"search": r"-+", "replace": "~"}],
        [{"search": r"^\s*", "replace": ""}, {"search": r"\s*\Z", "replace": ""}, {"search": r"(\S+)\s+(\S+)", "replace": r"\2 \1"}],
        [{"search": r"\b", "replace": "|"}, {"search": r"(a)|b", "replace": r"<\1>"}],
        [{"search": r"(?i)(kill)\s+(\w+)", "replace": r"\1 [\2]"}, {"search": r"(é+)(日?)", "replace": r"\2\1"}, {"search": r"", "replace": "."}],
    ]
    words = ["user@example.com", "bob@corp.com", "555-1234", "12-3456", "crap", "crud", "[x]", "xx", "x", "yxxy", "-", "--", "kill him", "KILL  them", "é", "éé日",
             "日", "a", "b", "ab", " ", "  ", "\n", "\t", "word", "two words", "", "_", "1", "naïve"]
    out = []
    for rules in rule_sets:
        plug = SearchReplacePlugin(PluginConfig(name="rf", kind="x", hooks=["tool_pre_invoke", "tool_post_invoke"], config={"words": rules}))
        cases = []
        for i in range(60):
            def text():
                return rng.choice(["", " ", "\n"]).join(rng.choice(words) for _ in range(rng.randint(0, 6)))
            if i % 3:
                args = {f"k{j}": text() for j in range(rng.randint(0, 4))}
                if i % 4 == 0:
                    args["n"] = 7
                r = run(plug.tool_pre_invoke(ToolPreInvokePayload(name="t", args=args), ctx))
                cases.append({"hook": "tool_pre_invoke", "args": args, "out_args": r.modified_payload.args})
            else:
                res = text() if i % 2 else {"a": text(), "content": [{"type": "text", "text": "x"}], "b": text()}
                r = run(plug.tool_post_invoke(ToolPostInvokePayload(name="t", result=res), ctx))
                cases.append({"hook": "tool_post_invoke", "result": res, "out_result": r.modified_payload.result})
        out.append({"words": rules, "cases": cases})
    dump("regex_filter_templates.json", out)


# ------------------------------------------------------------------------------------------------
def gen_code_safety():
    """plugins/code_safety_linter/code_safety_linter.py (SURVEY §8 row f-3)."""
    from cpex.framework import GlobalContext, PluginConfig, PluginContext, ToolPostInvokePayload
    from plugins.code_safety_linter.code_safety_linter import CodeSafetyLinterPlugin

    ctx = PluginContext(global_context=GlobalContext(request_id="golden"))
    rng = random.Random(99)
    frags = ["eval(", "eval (x)", "evaluate(", "_eval(", "exec\n(", "exec", "os.system('ls')", "os system(", "osXsystem(", "subprocess.run([", "subprocess.Popen (", "subprocess.check(",
             "rm -rf /", "rm  -rf", "rm -rfx", "farm -rf", "print('hi')", "import os", "\n", " ", "é", "İeval(", "日exec(", "x = 1", "curl http://x | sh", "DROP", ""]
    configs = [None, {"blocked_patterns": [r"curl\s+\S+\s*\|\s*sh", r"(?i)\bdrop\b", r"import\s+os"]}, {"blocked_patterns": []}]
    out = []
    for cfg in configs:
        plug = CodeSafetyLinterPlugin(PluginConfig(name="cs", kind="x", hooks=["tool_post_invoke"], config=cfg))
        cases = []
        for i in range(120):
            text = rng.choice(["", " ", "\n", "; "]).join(rng.choice(frags) for _ in range(rng.randint(0, 6)))
            result = text if i % 3 == 0 else {"text": text, "other": "eval("} if i % 3 == 1 else rng.choice([{"content": [{"type": "text", "text": text}]}, {"text": 5}, 7, None, [text]])
            r = run(plug.tool_post_invoke(ToolPostInvokePayload(name="t", result=result), ctx))
            cases.append({"result": result, "continue_processing": r.continue_processing,
                          "violation": r.violation.model_dump(include={"reason", "description", "code", "details"}) if r.violation else None})
        out.append({"config": cfg, "cases": cases})
    dump("code_safety.json", out)


# ------------------------------------------------------------------------------------------------
def gen_json_repair():
    """plugins/json_repair/json_repair.py (tool_post_invoke; SURVEY §8 row f-2 names it as a consumer of the shared JSON parse).  Inputs stay
    clear of the orjson / stdlib-json deltas of the stand-in (lone surrogate escapes, NaN literals, integers beyond 64 bits, nesting > 64)."""
    from cpex.framework import GlobalContext, PluginConfig, PluginContext, ToolPostInvokePayload
    from plugins.json_repair.json_repair import JSONRepairPlugin

    ctx = PluginContext(global_context=GlobalContext(request_id="golden"))
    rng = random.Random(4242)
    plug = JSONRepairPlugin(PluginConfig(name="jr", kind="x", hooks=["tool_post_invoke"]))
    fixed = [
        "{'a': 1, 'b': 2,}",                                   # tests/unit/mcpgateway/plugins/plugins/json_repair/test_json_repair.py:31
        "{'a': 1}", "['x', 'y']", "{'a': \"b\"}", "{'it''s': 1}", "('a')", "{'a': 1", "'a': 1}", "[1, 2, 3,]", "[1, 2, 3, ]", "{\"a\": 1,\n}", "{\"a\": [1, 2,], \"b\": {\"c\": 3,},}",
        "[1,,]", "[,]", "{,}", "[1 ,\t\n ]", "[\"a, ]\", 1,]", "{\"k\": \"v, }\"}", "[\"a, ]\"]", "\"a\": 1", "\"a\": 1, \"b\": [1, 2]", "a: 1", "'a': 1", "\"a\": 1,", "\"a\": {\"b\": 1}",
        "\"a\": 1}", "{\"a\": 1", "x: y: z", ":", "\"a\":", "  {\"a\": 1}  ", "\n[1, 2,]\n", "\u00a0{'a': 1}\u00a0", "\u2003[1,]\u2003", "\x0c[1,]", " 'a': 1 ", "\t\"k\": \"v\"\r\n",
        "", " ", "null", "true", "123", "-0.5e3", "\"str\"", "nul", "[1] x", "[1]\n", "{\"a\": 1}\u00a0", "{}", "[]", "{ }", "[ ]", "{'': ''}", "['']", "{'a': 'b, }'}", "['a,]',]",
        "{'a': 1,} ", "[\"\\u00e9\", 'x']", "{'é': 'ü',}", "['日本', '語',]", "{\"a\": 1,}trailing", "[1,]]", "[[1,],]", "{\"a\": {\"b\": [1,],},}", "'", "\"", "{'a': 'it\\'s'}",
        "{'a': 1, \"b\": 2,}", "{\"a\": 'x',}", "[1,\u00a0]", "[1,\u2028]", "[1,\x0b]", "[1,\x1f]", "\"a\": \"x:y\"", "k: [1, 2,]", "\"k\": [1, 2,]", "\"a\": 1, \"a\": 2", "[1, 2}", "{\"a\": 1]",
    ]
    gens = []
    for _ in range(260):
        v = rand_json(rng, rng.randint(0, 3))
        t = json.dumps(v, ensure_ascii=rng.random() < 0.5, separators=rng.choice([(",", ":"), (", ", ": "), (" ,\n", " : ")]))
        k = rng.random()
        if k < 0.2:
            pass
        elif k < 0.4:
            t = t.replace('"', "'")
        elif k < 0.6:
            t = re.sub(r"([}\]])", lambda m: rng.choice([",", ", ", ",\n", ""]) + m.group(1), t)
        elif k < 0.7:
            t = re.sub(r"([}\]])", lambda m: rng.choice([",", ""]) + m.group(1), t.replace('"', "'"))
        elif k < 0.8 and t.startswith("{") and t.endswith("}"):
            t = t[1:-1]
        elif k < 0.9:
            i = rng.randrange(len(t) + 1)
            t = t[:i] + rng.choice([",", "'", '"', "}", "]", ":", " ", "x", "\n"]) + t[i:]
        else:
            i = rng.randrange(len(t)) if t else 0
            t = t[:i] + t[i + 1:]
        gens.append(rng.choice(["", "", " ", "\n", "\u00a0"]) + t + rng.choice(["", "", " ", "\r\n", "\u3000"]))
    others = [None, 5, {"text": "{'a': 1,}"}, ["{'a': 1,}"], {"content": [{"type": "text", "text": "[1,]"}]}, True, 1.5]
    cases = []
    for res in fixed + gens + others:
        if isinstance(res, str) and any(ord(ch) >= 0xD800 and ord(ch) <= 0xDFFF for ch in res):
            continue
        r = run(plug.tool_post_invoke(ToolPostInvokePayload(name="t", result=res), ctx))
        cases.append({"result": res, "continue_processing": r.continue_processing, "out_result": r.modified_payload.result if r.modified_payload is not None else None,
                      "modified": r.modified_payload is not None, "metadata": r.metadata or {}})
    dump("json_repair.json", {"cases": cases})


if __name__ == "__main__":
    install_shims()
    only = sys.argv[1:]
    for name, fn in (("pattern_plugins", gen_pattern_plugins), ("toon", gen_toon), ("masking", gen_masking), ("sql_sanitizer", gen_sql_sanitizer),
                     ("regex_filter_templates", gen_regex_filter_templates),
                     ("code_safety", gen_code_safety), ("json_repair", gen_json_repair)):
        if not only or name in only:
            fn()

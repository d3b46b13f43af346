"""Container-only: live differential fuzz of the masker's source (csrc/json_mask.h on the host build: key classifier, depth rule, key order,
serialisation) against the REFERENCE'S OWN Python twin of the Rust crate (`mcpgateway/middleware/request_logging_middleware.py:83-291`, its pure
functions exec'd unmodified from /root/reference as tools/gen_golden.py does) — generated key names (token vocabulary x separators x casings),
random nested bodies, max_depth 0..12 — and against the oracle (oracle/mask_ref.py) byte for byte.
usage: python tools/fuzz_mask_vs_reference.py [--record OUT] [seed] [keys] [bodies]  |  --replay tests/golden/fuzz_mask.json.gz"""
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
import hostsim_util as hs  # noqa: E402
from oracle import mask_ref  # noqa: E402

VOCAB = ["auth", "token", "tokens", "tokenizer", "secret", "secrets", "key", "keys", "api", "jwt", "pass", "password", "passwd", "pwd", "word", "phrase", "session", "id", "count",
         "status", "private", "client", "access", "refresh", "cookie", "x", "url", "ttl", "hash", "name", "type", "o", "oauth", "credential", "cred", "bearer", "signature", "sig",
         "cert", "pin", "user", "authorization", "authz", "device", "custom", "ms", "length", "path", "value", "é", "ß", "1", "42", "a", "my", "top", "http", "basic", "pem"]
JOIN = ["", "_", "-", ".", " ", "__", "--", "_-", ":"]


def make_key(rng):
    n = rng.randint(1, 4)
    parts = []
    for _ in range(n):
        w = rng.choice(VOCAB)
        c = rng.random()
        parts.append(w if c < 0.4 else w.upper() if c < 0.55 else w.capitalize() if c < 0.9 else w[:1] + w[1:].upper())
    j = rng.choice(JOIN)
    k = j.join(parts) if rng.random() < 0.8 else "".join(p + rng.choice(JOIN) for p in parts)
    if rng.random() < 0.1:
        k = rng.choice(["X-", "x-", "_", "__", "-", " "]) + k
    if rng.random() < 0.05:
        k += rng.choice(["_", "-", "1", "S", "s", " "])
    return k


def cases(seed: int, nkeys: int, nbodies: int):
    """The seeded inputs: key names, JSON bodies for the kernel, (object, max_depth, headers) for the module, bodies of the non-JSON probe."""
    import math
    import struct

    rng = random.Random(seed)
    seen = {}
    for _ in range(nkeys):
        seen.setdefault(make_key(rng), None)
    keys = sorted(seen)

    def rand_prim():
        k = rng.random()
        if k < 0.35:                                            # any finite double: ryu's shortest digits and serde_json's layout (oracle: repr() digits)
            x = struct.unpack("<d", struct.pack("<Q", rng.getrandbits(64)))[0]
            return x if math.isfinite(x) else 0.5
        if k < 0.55:
            return rng.randint(-2 ** 63, 2 ** 64 - 1) >> rng.randint(0, 63)
        if k < 0.9:                                             # strings over controls, quotes, separators, BMP and astral code points: serde_json's escapes
            lo, hi = rng.choice([(0x00, 0x7F), (0x00, 0x1F), (0x7F, 0xFF), (0x2000, 0x2070), (0x3040, 0x30FF), (0x1F600, 0x1F64F), (0xFFF0, 0xFFFD)])
            return "".join(chr(rng.randint(lo, hi)) for _ in range(rng.choice([0, 1, 2, 5, 17, 40])))
        return round(rng.uniform(-1e9, 1e9), rng.randint(0, 12))

    def rand_obj(depth):
        r = rng.random()
        if depth <= 0 or r < 0.3:
            if rng.random() < 0.5:
                return rand_prim()
            return rng.choice(["v", 1, 2.5, True, None, "secret-value", -7, 1e16, 0.1, 10 ** 15, "é", "q\"\\\n\t\x01/", 1.0, 100.0, 1e-7, 123456789012, "", 0, -0.0, 5e-324, 1.7976931348623157e308])
        if r < 0.55:
            return [rand_obj(depth - 1) for _ in range(rng.randint(0, 4))]
        return {rng.choice(keys): rand_obj(depth - 1) for _ in range(rng.randint(0, 6))}

    bodies = []
    for _ in range(nbodies):
        obj = rand_obj(rng.randint(1, 7))
        md = rng.choice([10, 10, 3, 1, 0, 2, 12, 5])
        bodies.append((obj, md, json.dumps(obj, ensure_ascii=rng.random() < 0.5, separators=rng.choice([(",", ":"), (", ", ": ")])).encode()))
    # (no U+001C..U+001F around cookie names: Python's str.strip() of the twin strips them, Rust's trim() of the crate — which the drop-in
    # follows, lib.rs:199-231 — does not; tests/test_mask_gpu.py makes the same exclusion)
    cookies = ["jwt_token=abc; theme=dark; session_id=xyz", "theme=dark", "", "a=b;c", " SESSION = 1 ;; x=y", "Auth=1;AUTHX=2;nope=3", "tokén=1; TOKEN=2", "noequals; jwt", "a=b=c; token=d=e",
               "user=john; preference=light", "Bearer abc", "application/json", " \u00a0auth = 1\u3000; x = y ", "İauth=1; ſession=2; K=3"]
    module = []
    for _ in range(nbodies // 4):
        obj = rand_obj(rng.randint(1, 6))
        md = rng.choice([10, None, 3, 1, 0, 2])
        module.append((obj, md, {rng.choice(keys + ["Cookie", "cookie", "COOKIE", "CooKie", "Content-Type", "Accept"]): rng.choice(cookies) for _ in range(rng.randint(0, 6))}))
    words = ["password", "PassWord", "pass phrase", "secret", "SECRET", "toKen", "\u212aey", "api_\u212aey", "api-key", "APIKEY", "apikey", "access_token", "refresh-token", "client_secret",
             "Authorization", "auth_token", "jwt_token", "private_key", "private key", "İ", "ſecret", "hello", "x=1", "{", "\xff", "日本", " ", "&", "tok", "en"]
    fallback = [("".join(rng.choice(words) + rng.choice(["", " ", "=", "&", "\n"]) for _ in range(rng.randint(0, 6)))).encode("utf-8", "ignore") + rng.choice([b"", b"\xfe", b"\xc3"])
                for _ in range(nbodies // 4)]
    return keys, bodies, module, fallback


def record(argv):
    """The reference twin's side: one bit per key, the digest of each masked body / module call (data and headers) / fallback text."""
    seed = int(argv[0]) if len(argv) > 0 else 1
    nkeys = int(argv[1]) if len(argv) > 1 else 20000
    nbodies = int(argv[2]) if len(argv) > 2 else 2000
    gen_golden.install_shims()
    ns = gen_golden.load_masking_twin()
    keys, bodies, module, fallback = cases(seed, nkeys, nbodies)
    lows = tuple(ns["SENSITIVE_KEYS"])

    def fb(b_):
        s_ = b_.decode("utf-8", errors="ignore")                      # request_logging_middleware.py:661-667
        return "<contains sensitive data - masked>" if any(k in s_.lower() for k in lows) else s_

    return {"seed": seed, "keys": nkeys, "bodies": nbodies, "inputs": gen_golden.digest([keys, bodies, module, fallback]),
            "key_sensitive": "".join("1" if ns["_is_sensitive_key"](k) else "0" for k in keys),
            "masked": [gen_golden.digest(json.loads(json.dumps(ns["mask_sensitive_data"](obj, md)))) for obj, md, _ in bodies],
            "module": [gen_golden.digest([ns["mask_sensitive_data"](obj, 10 if md is None else md), ns["mask_sensitive_headers"](h)]) for obj, md, h in module],
            "fallback": [gen_golden.digest(fb(b_)) for b_ in fallback]}


def compare(rec) -> int:
    keys, bodies, module, fallback = cases(rec["seed"], rec["keys"], rec["bodies"])
    if gen_golden.digest([keys, bodies, module, fallback]) != rec["inputs"]:
        print("the generator no longer yields the recorded inputs: record the reference again (--record) bad=1")
        return 1
    t0 = time.time()
    bad = 0
    for k, exp in zip(keys, rec["key_sensitive"]):
        got = hs.key_sensitive_host(k)
        orc = mask_ref.is_sensitive_key(k)
        if not (exp == "01"[got] == "01"[orc]):
            bad += 1
            if bad <= 10:
                print("KEY", repr(k), "reference", exp == "1", "kernel", got, "oracle", orc)
    nb = 0
    for (obj, md, body), exp in zip(bodies, rec["masked"]):
        st, out = hs.mask_host(body, md)
        orc = mask_ref.mask_json_bytes(body, md)
        nb += 1
        if st != 0 or out != orc or gen_golden.digest(json.loads(out)) != exp:
            bad += 1
            if bad <= 10:
                print("BODY", body[:300], md, "\n  kernel   ", st, (out or b"")[:300], "\n  oracle   ", orc[:300])
    # ---- the module a gateway imports (request_logging_masking_native_extension -> mcp_context_forge_b200/masking.py): its host logic (key
    # collection, cookie splitting, header walk, fallback probes) with the launches on the CPU simulator, against the twin's functions
    import importlib

    import pytest

    import hostsim_batcher

    hostsim_batcher.install(pytest.MonkeyPatch())
    mod = importlib.import_module("request_logging_masking_native_extension")
    from mcp_context_forge_b200 import masking

    nm = 0
    for (obj, md, h), exp in zip(module, rec["module"]):
        got = mod.mask_sensitive_data(obj, md)
        hgot = mod.mask_sensitive_headers(h)
        nm += 2
        if gen_golden.digest([got, hgot]) != exp or masking.mask_sensitive_headers_batch([h, h])[1] != hgot:
            bad += 1
            if bad <= 10:
                print("MODULE", repr(obj)[:200], md, "\n  module   ", repr(got)[:200], "\n  headers", h, "\n  module   ", hgot)
    for b_, e_, g_ in zip(fallback, rec["fallback"], masking.non_json_fallback_batch(fallback)):
        nm += 1
        if gen_golden.digest(g_) != e_:
            bad += 1
            if bad <= 10:
                print("FALLBACK", b_, "module", repr(g_))
    print(f"seed={rec['seed']} keys={len(keys)} bodies={nb} module_calls={nm} bad={bad} time={time.time() - t0:.1f}s")
    return 1 if bad else 0


def main() -> int:
    return gen_golden.fuzz_main("fuzz_mask_vs_reference", sys.argv[1:], record, compare)


if __name__ == "__main__":
    sys.exit(main())

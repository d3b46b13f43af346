"""Container-only: live differential fuzz of the TOON kernels' source (sequential encoder csrc/json_toon.h on the host build; token-parallel kernel
body csrc/json_tp.h on the 32-fibre warp emulator) against the REFERENCE'S OWN `plugins/toon_encoder/toon.py`, imported unmodified from
/root/reference — no restatement in between (the oracle is compared too, so a gap in it shows).  Random JSON documents from the generator of
tools/fuzz_toon_tp.py (adversarial keys / strings / numbers, tables, byte-level mutations).  orjson is not installable here: the strict stdlib
parser stands in, and documents that would expose an orjson / json delta (integers beyond 64 bits, lone surrogates, non-finite floats) are skipped.
usage: python tools/fuzz_vs_reference.py [--record OUT] [seed] [cases] [gen1|gen2|synth]  |  --replay tests/golden/fuzz_toon.json.gz"""
import importlib.util
import json
import math
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
from fuzz_toon_tp import make_gen  # noqa: E402
from mcp_context_forge_b200.plugins.toon_encoder import _encode_error  # noqa: E402
from oracle import toon_ref  # noqa: E402


def load_reference_toon():
    spec = importlib.util.spec_from_file_location("ref_toon", os.path.join(gen_golden.REF, "plugins/toon_encoder/toon.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def delta_free(v) -> bool:
    """True when stdlib json and orjson agree on this parsed document."""
    if isinstance(v, bool) or v is None:
        return True
    if isinstance(v, int):
        return -(2 ** 63) <= v < 2 ** 64
    if isinstance(v, float):
        return math.isfinite(v)
    if isinstance(v, str):
        return not any(0xD800 <= ord(c) <= 0xDFFF for c in v)
    if isinstance(v, list):
        return all(delta_free(x) for x in v)
    return all(delta_free(k) and delta_free(x) for k, x in v.items())


def expected(toon, t: str):
    """(status, text) as include/cfgpu.h defines them for an unlimited output buffer: 0 = the reference's toon.encode(orjson.loads(t)),
    2 = not JSON, 3 / 4 = toon.encode raises ValueError / AttributeError."""
    try:
        t.encode("utf-8")
    except UnicodeEncodeError:
        return None
    try:
        doc = json.loads(t, parse_constant=lambda c: (_ for _ in ()).throw(ValueError(c)))
    except (ValueError, RecursionError):
        return (2, None)
    if not delta_free(doc):
        return None
    try:
        return (0, toon.encode(doc))
    except ValueError as exc:
        expected.message = str(exc)
        return (3, None)
    except AttributeError as exc:
        expected.message = str(exc)
        return (4, None)


def make_gen2(rng):
    """A second generator: strings over the whole BMP + astral planes (controls, quotes, separators, RTL, combining marks), numbers of every
    magnitude orjson and json agree on, deeper nesting, wide tables with missing / reordered / nested cells."""
    import struct

    pools = [(0x20, 0x7E), (0x00, 0x1F), (0x7F, 0xA0), (0xA0, 0x17F), (0x300, 0x36F), (0x590, 0x6FF), (0x2000, 0x206F), (0x3040, 0x30FF), (0xE000, 0xE010), (0xFFF0, 0xFFFD), (0x1F600, 0x1F64F)]

    def rstr():
        k = rng.random()
        if k < 0.3:
            return rng.choice(["", "null", "true", "false", "-", "- x", "1e5", "0x10", "007", "1.", ".5", "+3", "-0", "1_000", "NaN", "Infinity", " a", "a ", "a,b", "a:b", "a\"b", "[1]", "{}", "a\\b", "#", "x\ny", "\t"])
        n = rng.choice([1, 1, 2, 3, 5, 8, 20, 64])
        lo, hi = rng.choice(pools)
        return "".join(chr(rng.randint(*rng.choice([(lo, hi), (0x61, 0x7A)]))) for _ in range(n))

    def rnum():
        k = rng.random()
        if k < 0.3:
            return rng.randint(-2 ** 63, 2 ** 63 - 1) >> rng.randint(0, 62)
        if k < 0.4:
            return rng.choice([0, -0.0, 2 ** 53, 2 ** 53 + 1, -2 ** 63, 2 ** 64 - 1, 1e15, 1e16, 1e21, 1e22, 123456789012345.6, 0.1, 1 / 3, 5e-324, 1.7976931348623157e308, 2.2250738585072014e-308])
        if k < 0.7:
            x = struct.unpack("<d", struct.pack("<Q", rng.getrandbits(64)))[0]
            return x if math.isfinite(x) else 1.5
        return round(rng.uniform(-1e6, 1e6), rng.randint(0, 10))

    def rprim():
        k = rng.random()
        return rstr() if k < 0.45 else rnum() if k < 0.8 else rng.choice([None, True, False])

    def rkey():
        return rstr() if rng.random() < 0.5 else rng.choice(["id", "name", "a", "b", "value", "x.y", "_p", "k1", "A", "items", "é"])

    def rval(d):
        k = rng.random()
        if d <= 0 or k < 0.25:
            return rprim()
        if k < 0.4:
            return [rprim() for _ in range(rng.randint(0, 6))]
        if k < 0.6:
            keys = [rkey() for _ in range(rng.randint(1, 5))]
            rows = []
            for _ in range(rng.randint(1, 6)):
                ks = list(keys)
                q = rng.random()
                if q < 0.1:
                    rng.shuffle(ks)
                elif q < 0.15:
                    ks = ks[1:]
                rows.append({kk: (rprim() if rng.random() < 0.93 else rval(d - 1)) for kk in ks})
            if rng.random() < 0.1:
                rows.insert(rng.randint(0, len(rows)), rval(d - 1))
            return rows
        if k < 0.85:
            return {rkey(): rval(d - 1) for _ in range(rng.randint(0, 5))}
        return [rval(d - 1) for _ in range(rng.randint(0, 4))]

    def case():
        v = rval(rng.randint(0, 9))
        k = rng.random()
        if k < 0.5:
            return json.dumps(v, separators=(",", ":"), ensure_ascii=False)
        if k < 0.75:
            return json.dumps(v, ensure_ascii=True)
        return json.dumps(v, indent=rng.choice([None, 1, 3]), ensure_ascii=False)

    return case


def documents(seed: int, n: int, which: str):
    rng = random.Random(seed)
    if which == "synth":                                        # the bench's payload shapes (tabular / nested config / prose in JSON), 200 B .. 70 KB
        from mcp_context_forge_b200 import synth

        def case():
            shape = rng.choice("AABBC")
            p = synth.payload(shape, rng.choice([200, 600, 2000, 5000, 16384, 16384, 40000, 70000]), seed=rng.randrange(1 << 30), hit_rate=rng.choice([0, 1e-4, 1e-2]))
            return p if shape != "C" else json.dumps({"title": "d", "body": p}, ensure_ascii=rng.random() < 0.3)
    else:
        case = make_gen2(rng) if which == "gen2" else make_gen(rng)
    return [case() for _ in range(n)]


def record(argv):
    """The reference's side of a run: per document None (skipped) or the digest of (status, text, exception message)."""
    seed = int(argv[0]) if len(argv) > 0 else 1
    n = int(argv[1]) if len(argv) > 1 else 2000
    which = argv[2] if len(argv) > 2 else "gen1"
    toon = load_reference_toon()
    docs = documents(seed, n, which)
    outputs = []
    for t in docs:
        exp = expected(toon, t)
        if exp is None or (exp[0] == 2 and any(0xD800 <= ord(c) <= 0xDFFF for c in t)):
            outputs.append(None)
        else:
            outputs.append(gen_golden.digest([exp[0], exp[1], expected.message if exp[0] in (3, 4) else None]))
    return {"seed": seed, "cases": n, "generator": which, "inputs": gen_golden.digest(docs), "outputs": outputs}


def compare(rec) -> int:
    docs = documents(rec["seed"], rec["cases"], rec["generator"])
    if gen_golden.digest(docs) != rec["inputs"]:
        print("the generator no longer yields the recorded documents: record the reference again (--record) bad=1")
        return 1
    rng = random.Random(rec["seed"])                            # fibre orders of the token-parallel kernel
    t0 = time.time()
    done = skipped = handed = bad = worded = 0
    for it, (t, ref_digest) in enumerate(zip(docs, rec["outputs"])):
        if ref_digest is None:
            skipped += 1
            continue
        done += 1
        seq = hs.toon_host(t, unlimited=True)
        msg = str(_encode_error(seq[0], t)) if seq[0] in (3, 4) else None     # the wording the drop-in gives the exception (skip_on_error: false)
        worded += msg is not None
        if gen_golden.digest([seq[0], seq[1], msg]) != ref_digest:
            bad += 1
            if bad <= 8:
                print("BAD (differs from the reference)", repr(t)[:400], "\n   seq      ", repr(seq)[:300], "\n   message  ", msg)
        exp = seq                                               # == the reference's output unless reported above
        tp = hs.toon_tp(t, unlimited=True, report_errors=True, order=(it & 1) | (rng.randrange(16) << 4))
        if tp[0] == 7:
            handed += 1
            tp = exp
        try:
            orc = (0, toon_ref.encode(toon_ref.loads_strict(t)))
        except ValueError:
            orc = (2 if exp[0] == 2 else 3, None)
        except toon_ref.ToonCrash:
            orc = (4, None)
        # the product's rule on top (include/cfgpu.h): the text is kept only when strictly smaller than the JSON it came from
        small = exp if (exp[0] != 0 or len(exp[1].encode("utf-8")) < len(t.encode("utf-8"))) else (1, None)
        seq2, tp2 = hs.toon_host(t), hs.toon_tp(t, report_errors=True)
        if tp2[0] == 7:
            tp2 = small
        if not (seq2 == small and tp2 == small):
            bad += 1
            if bad <= 8:
                print("BAD (size rule)", repr(t)[:300], "\n   expected", repr(small)[:200], "\n   seq", repr(seq2)[:200], "\n   tp ", repr(tp2)[:200])
        if not (tp == exp and orc == exp):
            bad += 1
            if bad <= 8:
                print("BAD", repr(t)[:400], "\n   seq      ", repr(seq)[:300], "\n   tp       ", repr(tp)[:300], "\n   oracle   ", repr(orc)[:300])
    print(f"seed={rec['seed']} cases={rec['cases']} compared={done} skipped={skipped} handed_over={handed} error_messages_compared={worded} bad={bad} "
          f"time={time.time() - t0:.1f}s")
    return 1 if bad or not done else 0


def main() -> int:
    return gen_golden.fuzz_main("fuzz_vs_reference", sys.argv[1:], record, compare)


if __name__ == "__main__":
    sys.exit(main())

"""Regenerates tests/golden/golden_v1.json from the REFERENCE's own code (oracle/_ref/liblz4net_ref.so, i.e.
/root/reference/original/lz4.c + lz4hc.c compiled in place by oracle/Makefile).  Run only in the build container:

    python tests/golden/make_golden.py

The reference ships no golden vectors of its own (SURVEY.md 8c); these are outputs of the reference itself on
reproducible inputs (tests/cases.py), including the reference-defined AutoTest text (src/LZ4/LZ4Codec.cs:175-184).
It also writes tests/golden/reference_results.json: the reference's return values and output digests for the inputs
of tests/test_oracle.py's comparisons with the reference, computed by that module's own functions.
"""
import hashlib
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
import oracle  # noqa: E402
from tests import cases  # noqa: E402


def sha(b):
    return hashlib.sha256(b).hexdigest()


def main():
    out = []
    todo = [("autotest", "autotest", len(cases.AUTOTEST), 0)]
    for m in cases.MODELS:
        todo.append((f"{m}-64k", m, 65536, 1))
    for i, n in enumerate((0, 1, 12, 13, 20, 64, 300, 4096, 32768, 65535, 65546, 65547, 100000)):
        for m in ("mixed", "lowent", "ETEXT", "periodic"):
            todo.append((f"{m}-{n}", m, n if not (m == 'mixed' and n > 70000) else 70000, 50 + i))
    seen = set()
    for name, model, n, seed in todo:
        if name in seen:
            continue
        seen.add(name)
        data = cases.AUTOTEST if model == "autotest" else cases.content(model, n, seed).tobytes()
        c = {"name": name, "model": model, "n": len(data), "seed": seed, "input_sha256": sha(data)}
        for mode, fn in (("fast", oracle.encode), ("hc", oracle.encode_hc)):
            r, o = fn(data, impl="ref")
            r2, _ = fn(data, cap=len(data), impl="ref")
            c[mode] = {"len": r, "sha256": sha(o), "len_cap_n": r2}
            if r <= 512:
                c[mode]["hex"] = o.hex()
        out.append(c)
    path = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden_v1.json")
    json.dump({"source": "oracle/_ref (reference original/lz4.c + lz4hc.c, LZ4_ARCH64=1, LZ4_MK_OPT)", "cases": out},
              open(path, "w"), indent=1)
    print("wrote", path, len(out), "cases")
    reference_results()


def reference_results():
    from lz4net_b200 import synth
    from tests import test_oracle as t
    rl = {m: [[n, t.encode_results(d, "ref")[0]] for n, d in t.random_length_inputs(m)] for m in cases.MODELS}
    ar = [t.accept_reject_results(oracle.encode(d, impl="ref")[1], len(d), "ref") for _, d in t.accept_reject_inputs()]
    comps, streams = t.corrupt_streams("ref")
    cs = {"comp": t.digest(*comps), "verdicts": [t.unknown_result(c, n, "ref") for n, c in streams]}
    # tests/test_kernels_emu.py: a block on which r93's LZ4HC gives up at the bound
    d = synth.make_blocks("E0", 1, 65536, seed=3, first_block=1268)[0].tobytes()
    cap = oracle.bound(len(d))
    hc_bound = [oracle.encode_hc(d, cap=cap, impl="ref")[0], oracle.encode_hc(d, cap=cap + 4096, impl="ref")[0]]
    path = os.path.join(os.path.dirname(os.path.abspath(__file__)), "reference_results.json")
    doc = {"source": "oracle/_ref (reference original/lz4.c + lz4hc.c, LZ4_ARCH64=1, LZ4_MK_OPT)",
           "random_lengths": rl, "accept_reject": ar, "corrupt_streams": cs, "encode_hc_gives_up_at_the_bound": hc_bound}
    with open(path, "w") as f:                  # one entry of each list or object per line: diffs stay readable
        f.write("{\n" + ",\n".join(f"{json.dumps(k)}: {_one_entry_per_line(v)}" for k, v in doc.items()) + "\n}\n")
    print("wrote", path)


def _one_entry_per_line(v):
    if isinstance(v, dict):
        return "{\n" + ",\n".join(f" {json.dumps(k)}: {json.dumps(x)}" for k, x in v.items()) + "\n}"
    if isinstance(v, list) and v and isinstance(v[0], (list, dict)):
        return "[\n" + ",\n".join(" " + json.dumps(x) for x in v) + "\n]"
    return json.dumps(v)


if __name__ == "__main__":
    main()

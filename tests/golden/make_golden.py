"""Generates tests/golden/golden.json from the UNMODIFIED reference (oracle/_ref, built by
`make -C oracle ref` from the reference sources, see oracle/Makefile):

    python tests/golden/make_golden.py

Each case stores the input spec (tests/datasets.py), the input digest, and for both
compressors (-c hash table, -b BST) the stream length + sha256 (+ full hex when small).
"""
import hashlib
import json
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))

import datasets  # noqa: E402
import oracle_lib  # noqa: E402

SPECS = [
    "hex:616263",                      # "abc"      (SURVEY.md 8c)
    "rep:97:100",                      # 'a' x 100  (SURVEY.md 8c)
    "hex:00", "hex:0001", "rep:0:15", "rep:0:16", "rep:0:17", "rep:255:70",
    "rep:0:65536", "rep:0:65537", "rep:0:1048576",
    "corpus:random:2:0:1048576",
    "corpus:text:0:0:200000", "corpus:text:3:777:65536", "corpus:text:0:5:2049",
    "corpus:lowent:1:0:200000", "corpus:lowent:4:123:70001",
    "corpus:random:2:0:70000", "corpus:mixed:0:1000000:150000",
    "sym:5:1:100000", "sym:2:2:65537", "sym:3:3:4097",
    "period:7:1:70000", "period:300:2:131073", "period:4096:3:200000", "period:1:4:5000",
    "lz:1:100000", "lz:2:65536", "lz:3:300", "lz:4:131072",
] + [f"corpus:text:1:{s}:{s}" for s in (14, 15, 16, 17, 255, 256, 257, 2048, 4097, 65535)]


def main():
    oracle_lib.build(ref=True)
    ref = oracle_lib.Reference()
    cases = []
    for spec in SPECS:
        data = datasets.gen(spec)
        case = {"spec": spec, "size": int(data.size), "input_sha256": hashlib.sha256(data.tobytes()).hexdigest()}
        for name, mode in (("hash", 0), ("bst", 1)):
            s = ref.compress(data, mode)
            case[name] = {"len": int(s.size), "sha256": hashlib.sha256(s.tobytes()).hexdigest()}
            if s.size <= 64:
                case[name]["hex"] = s.tobytes().hex()
            # the reference decoder must invert its own stream (decoder refill bug aside, Q6)
            back = ref.decompress(s, data.size)
            case[name]["ref_roundtrip"] = bool(back.size == data.size and (back == data).all())
        cases.append(case)
    varints = [{"value": v, "hex": ref.varint_encode(v).hex()}
               for v in (0, 1, 127, 128, 227, 16384, 65536, 1 << 20, 1 << 30, (1 << 31) - 1, 1 << 32, (1 << 63) + 5)]
    with open(os.path.join(HERE, "golden.json"), "w") as f:
        json.dump({"source": "oracle/_ref built from the reference sources (gcc -O2)", "cases": cases,
                   "varints": varints}, f, indent=1)
    print(f"wrote {len(cases)} cases")


if __name__ == "__main__":
    main()

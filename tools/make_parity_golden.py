"""Generates tests/golden/reference_parity.json: the reference's answers on the seeded inputs of
tests/test_oracle_vs_reference.py, so that the port is compared with them where the reference is absent.

    python tools/make_parity_golden.py [--source reference|port]

--source reference (the default) drives the unmodified reference compiled into oracle/_ref (oracle/Makefile,
REF=<reference checkout>).  --source port records the oracle port instead; that is only a record of the
reference where the port has been shown to agree with it bit for bit on these same inputs.  The file says which
one it came from.  Large arrays are stored as SHA-256 digests of their fields, small ones as values.
"""
from __future__ import annotations

import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from oracle import oracle_lib as ol  # noqa: E402
from tools import corpus  # noqa: E402
from tools.make_golden import boundaries, packets_digest, sha  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden", "reference_parity.json")

# the inputs of tests/test_oracle_vs_reference.py
RAND_SEEDS, RAND_COUNT = (1, 42, 1673551), 2000
HEAP_SEED, HEAP_TRIALS = 7, 50
PARITY_CASES = [("text", 3000, 1), ("binary", 3000, 2), ("mixed", 6000, 3)]
ANNEAL_CASES = [("text", 1500, 0), ("binary", 1500, 0), ("mixed", 3000, 1), ("text", 3000, 2)]
ANNEAL_SEED, ANNEAL_EVALS = 11, 400
EDGE_INPUTS = (b"a", b"ab", b"aaaa", b"abcabcabcabc", bytes(300), bytes(range(256)))


def heap_inputs():
    """(keys, k) of every trial, in order."""
    rng = corpus.SplitMix64(HEAP_SEED)
    out = []
    for trial in range(HEAP_TRIALS):
        count = 1 + rng.below(300)
        k = 1 + rng.below(32)
        out.append(([int(rng.below(1 + trial % 9)) for _ in range(count)], k))
    return out


def topk_record(pops, counts) -> dict:
    return {"pops_digest": packets_digest(pops), "counts_sha256": sha(counts.astype("<i4").tobytes())}


def anneal(lib, data, slab, best, step):
    """(attempts, best_cost, cur_cost, trace): the reference's loop on its glibc rand() stream, seed of main.c:68."""
    if isinstance(lib, ol.Ref):
        return lib.anneal_epoch(data, slab, best, 0, 0, step=step, evals=ANNEAL_EVALS)
    attempts, bc, cc, _, trace = lib.anneal_epoch(data, slab, best, 0, 0, rng_mode=0, step=step, evals=ANNEAL_EVALS)
    return attempts, bc, cc, trace


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--source", choices=["reference", "port"], default="reference")
    args = ap.parse_args()
    port = ol.Port()
    lib = ol.Ref() if args.source == "reference" else port
    doc = {"generator": "tools/make_parity_golden.py", "source": args.source,
           "rand": {str(s): sha(lib.rand_stream(s, RAND_COUNT).astype("<i4").tobytes()) for s in RAND_SEEDS},
           "heap_pop_orders": [[int(x) for x in lib.heap_topk(keys, k)] for keys, k in heap_inputs()],
           "parity": [], "anneal": [], "edge": []}

    for kind, n, seed in PARITY_CASES:
        data = corpus.make(kind, n, seed)
        lit = ol.literal_slab(n)
        greedy = port.greedy_slab(data)  # the test builds its slab with the port too
        b = boundaries(greedy)
        case = {"kind": kind, "n": n, "seed": seed, "data_sha256": sha(data), "greedy_digest": packets_digest(greedy),
                "slabs": {}, "prefix": []}
        for name, slab in (("literal", lit), ("greedy", greedy)):
            enc = lib.encode_slab(data, slab)
            case["slabs"][name] = {"cost": lib.slab_cost(data, slab), "bytes_sha256": sha(enc), "bytes_len": len(enc)}
        for stop in (b[1], b[len(b) // 2], b[-1]):
            case["prefix"].append({"stop": int(stop), "cost": lib.prefix_cost(data, greedy, stop),
                                   "model_sha256": sha(lib.model_after_prefix(data, greedy, stop).tobytes())})
        case["topk_mode0"] = topk_record(*lib.topk_many(data, lit, 0, np.arange(n)))
        case["topk_mode1"] = topk_record(*lib.topk_many(data, greedy, 1, b))
        doc["parity"].append(case)

    for kind, n, step in ANNEAL_CASES:
        data = corpus.make(kind, n, ANNEAL_SEED)
        start = ol.literal_slab(n) if step == 0 else port.greedy_slab(data)
        slab, best = start.copy(), start.copy()
        attempts, bc, cc, trace = anneal(lib, data, slab, best, step)
        doc["anneal"].append({"kind": kind, "n": n, "step": step, "data_sha256": sha(data),
                              "start_digest": packets_digest(start), "attempts": attempts, "best_cost": bc,
                              "cur_cost": cc, "trace_len": int(trace.size), "trace_sha256": sha(trace.tobytes()),
                              "slab_digest": packets_digest(slab), "best_digest": packets_digest(best)})

    for data in EDGE_INPUTS:
        lit = ol.literal_slab(len(data))
        rec = {"input_hex": data.hex(), "cost": lib.slab_cost(data, lit), "bytes_hex": lib.encode_slab(data, lit).hex()}
        rec.update(topk_record(*lib.topk_many(data, lit, 0, np.arange(len(data)))))
        doc["edge"].append(rec)

    with open(OUT, "w") as f:
        json.dump(doc, f, indent=1)
        f.write("\n")
    print("wrote", OUT, os.path.getsize(OUT), "bytes")


if __name__ == "__main__":
    main()

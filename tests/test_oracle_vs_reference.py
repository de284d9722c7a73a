"""The oracle port against stored parity vectors on seeded inputs: tests/golden/reference_parity.json
(tools/make_parity_golden.py), plus the reference's struct sizes and price table in tests/golden/reference_vectors.json.

reference_parity.json says which implementation it was recorded from.  The committed file comes from the port
("source": "port"), not from the reference: it was recorded at commit 297a67c, whose oracle sources are those of
commit 1062593, where this module's 11 tests compared the port with the compiled reference on exactly these inputs
and passed.  So it pins the port to the answers it gave when it last agreed with the reference.  With a reference
checkout, `make -C oracle ref REF=<checkout>` and `python tools/make_parity_golden.py` record it from the reference."""
import json
import os

import numpy as np
import pytest

from oracle import oracle_lib as ol
from tools import corpus
from tools.make_golden import boundaries, packets_digest, sha
from tools.make_parity_golden import ANNEAL_EVALS, ANNEAL_SEED, EDGE_INPUTS, RAND_COUNT, RAND_SEEDS, heap_inputs

GOLDEN = os.path.join(os.path.dirname(__file__), "golden")


def load(name):
    with open(os.path.join(GOLDEN, name)) as f:
        return json.load(f)


@pytest.fixture(scope="module")
def gold():
    return load("reference_parity.json")


@pytest.fixture(scope="module")
def vectors():
    return load("reference_vectors.json")


def assert_topk(got, want):
    pops, counts = got
    assert sha(counts.astype("<i4").tobytes()) == want["counts_sha256"]
    assert packets_digest(pops) == want["pops_digest"]


def test_struct_sizes(vectors):
    # SURVEY.md Appendix B
    assert vectors["sizeof"]["LZMAPacket"] == 12 == ol.PACKET_DTYPE.itemsize
    # no port struct has the reference's LZMAState layout: this half only guards the stored record of it
    assert vectors["sizeof"]["LZMAState"] == 5280


def test_tables_and_rand(port, gold, vectors):
    assert sha(port.price_table().astype("<u8").tobytes()) == vectors["price_table_sha256"]
    for seed in RAND_SEEDS:
        assert sha(port.rand_stream(seed, RAND_COUNT).astype("<i4").tobytes()) == gold["rand"][str(seed)]


def test_heap_ties(port, gold):
    inputs = heap_inputs()
    assert len(inputs) == len(gold["heap_pop_orders"])
    for (keys, k), want in zip(inputs, gold["heap_pop_orders"]):
        assert port.heap_topk(keys, k).tolist() == want


def case_of(cases, **key):
    found = [c for c in cases if all(c[k] == v for k, v in key.items())]
    assert len(found) == 1, key
    return found[0]


@pytest.mark.parametrize("kind,n,seed", [("text", 3000, 1), ("binary", 3000, 2), ("mixed", 6000, 3)])
def test_three_parity_functions(port, gold, kind, n, seed):
    g = case_of(gold["parity"], kind=kind, n=n, seed=seed)
    data = corpus.make(kind, n, seed)
    assert sha(data) == g["data_sha256"], "synthetic corpus generator drifted"
    lit = ol.literal_slab(n)
    greedy = port.greedy_slab(data)
    assert packets_digest(greedy) == g["greedy_digest"]
    for name, slab in (("literal", lit), ("greedy", greedy)):
        want = g["slabs"][name]
        assert port.slab_cost(data, slab) == want["cost"]
        enc = port.encode_slab(data, slab)
        assert len(enc) == want["bytes_len"] and sha(enc) == want["bytes_sha256"]
    b = boundaries(greedy)
    assert [p["stop"] for p in g["prefix"]] == [b[1], b[len(b) // 2], b[-1]]
    for p in g["prefix"]:
        assert port.prefix_cost(data, greedy, p["stop"]) == p["cost"]
        assert sha(port.model_after_prefix(data, greedy, p["stop"]).tobytes()) == p["model_sha256"]
    assert_topk(port.topk_many(data, lit, 0, np.arange(n)), g["topk_mode0"])
    assert_topk(port.topk_many(data, greedy, 1, b), g["topk_mode1"])


@pytest.mark.parametrize("kind,n,step", [("text", 1500, 0), ("binary", 1500, 0), ("mixed", 3000, 1), ("text", 3000, 2)])
def test_anneal_epoch_trajectory(port, gold, kind, n, step):
    g = case_of(gold["anneal"], kind=kind, n=n, step=step)
    data = corpus.make(kind, n, ANNEAL_SEED)
    assert sha(data) == g["data_sha256"], "synthetic corpus generator drifted"
    start = ol.literal_slab(n) if step == 0 else port.greedy_slab(data)
    assert packets_digest(start) == g["start_digest"]
    s1, b1 = start.copy(), start.copy()
    attempts, bc, cc, _, trace = port.anneal_epoch(data, s1, b1, 0, 0, rng_mode=0, step=step, evals=ANNEAL_EVALS)
    assert (attempts, bc, cc) == (g["attempts"], g["best_cost"], g["cur_cost"])
    assert trace.size == g["trace_len"] and sha(trace.tobytes()) == g["trace_sha256"]
    assert packets_digest(s1) == g["slab_digest"] and packets_digest(b1) == g["best_digest"]


def test_edge_inputs(port, gold):
    assert [bytes.fromhex(e["input_hex"]) for e in gold["edge"]] == list(EDGE_INPUTS)
    for data, g in zip(EDGE_INPUTS, gold["edge"]):
        n = len(data)
        lit = ol.literal_slab(n)
        assert port.slab_cost(data, lit) == g["cost"]
        assert port.encode_slab(data, lit).hex() == g["bytes_hex"]
        assert_topk(port.topk_many(data, lit, 0, np.arange(n)), g)

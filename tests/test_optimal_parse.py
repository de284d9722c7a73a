"""Starting slabs from a shortest-path parse: mg_anneal_optimal_init / Annealer.optimal_init on the device, and
`megalania --optimal`.  The CPU tests pin a CPU parse built on the oracle port's pricing (tests/optimal_parse.c,
compiled into a temporary directory) and its match lists; the GPU tests hold the device parse to it packet for packet
(one region) and check the stitched slab of many regions."""
import ctypes
import lzma
import os
import subprocess

import numpy as np
import pytest

MIB = 1 << 20
LIST_CAP = 32


def live_chain(slab):
    out, p = [], 0
    while p < slab.size:
        out.append((p, int(slab[p]["type"]), int(slab[p]["dist"]), int(slab[p]["len"])))
        p += int(slab[p]["len"])
    return out


def brute_match_list(data, pos, max_occ, cap):
    """The match-list rule written from scratch: nearest occurrence of the bigram first, keep strictly longer ones."""
    n = len(data)
    if pos == 0 or pos + 1 >= n:
        return []
    max_occ = max_occ or 64
    limit = min(273, n - pos)
    occ = [o for o in range(pos - 1, -1, -1) if data[o:o + 2] == data[pos:pos + 2]][:max_occ]
    out, best = [], 0
    for o in occ:
        length = 2
        while length < limit and data[pos + length] == data[o + length]:
            length += 1
        if length <= best:
            continue
        if len(out) == cap:
            break
        out.append((length, pos - o - 1))
        best = length
        if length >= limit:
            break
    return out


class CpuParse:
    """ctypes binding of cpu_optimal_slab / cpu_match_list (tests/optimal_parse.c)."""

    def __init__(self, path: str):
        self.lib = ctypes.CDLL(path)
        vp, sz, u32 = ctypes.c_void_p, ctypes.c_size_t, ctypes.c_uint32
        self.lib.cpu_optimal_slab.restype = None
        self.lib.cpu_optimal_slab.argtypes = [vp, sz, u32, vp]
        self.lib.cpu_match_list.restype = sz
        self.lib.cpu_match_list.argtypes = [vp, sz, sz, u32, vp, sz]

    def optimal_slab(self, data, max_occ=0) -> np.ndarray:
        from oracle import oracle_lib
        d = np.ascontiguousarray(np.frombuffer(bytes(data), dtype=np.uint8))
        slab = oracle_lib.literal_slab(d.size)
        self.lib.cpu_optimal_slab(d.ctypes.data_as(ctypes.c_void_p), d.size, max_occ, slab.ctypes.data_as(ctypes.c_void_p))
        return slab

    def match_list(self, data, pos, max_occ=0, cap=LIST_CAP) -> np.ndarray:
        """(len, distance - 1) rows of the parse's match list at pos."""
        d = np.ascontiguousarray(np.frombuffer(bytes(data), dtype=np.uint8))
        out = np.zeros((max(cap, 1), 2), dtype=np.uint32)
        got = int(self.lib.cpu_match_list(d.ctypes.data_as(ctypes.c_void_p), d.size, pos, max_occ,
                                          out.ctypes.data_as(ctypes.c_void_p), cap))
        return out[:got]


@pytest.fixture(scope="module")
def parse(tmp_path_factory):
    """Compiled here, into a temporary directory: the tree may be read-only."""
    src = os.path.join(os.path.dirname(os.path.abspath(__file__)), "optimal_parse.c")
    lib = str(tmp_path_factory.mktemp("optimal_parse") / "liboptimal_parse.so")
    subprocess.run(["gcc", "-O2", "-std=gnu11", "-Wall", "-Wextra", "-fPIC", "-shared", "-o", lib, src, "-lm"], check=True)
    return CpuParse(lib)


def seeded_inputs():
    rng = np.random.default_rng(7)
    yield "alphabet4", bytes(rng.integers(0, 4, 3000, dtype=np.uint8))
    words = [b"abc", b"abcd", b"abcde", b"xyz", b"ab", b" "]
    yield "words", b"".join(words[i] for i in rng.integers(0, len(words), 900))
    yield "zeros", bytes(600) + bytes(rng.integers(0, 256, 200, dtype=np.uint8)) + bytes(600)


# ---- CPU: the CPU parse ------------------------------------------------------------------------------------
@pytest.mark.parametrize("max_occ,cap", [(0, LIST_CAP), (5, LIST_CAP), (64, 3), (1000, LIST_CAP)])
def test_match_list_is_the_rule(parse, max_occ, cap):
    for name, data in seeded_inputs():
        n = len(data)
        for pos in list(range(0, 40)) + list(range(40, n, 7)) + [n - 2, n - 1]:
            got = [tuple(int(v) for v in row) for row in parse.match_list(data, pos, max_occ, cap)]
            assert got == brute_match_list(data, pos, max_occ, cap), (name, pos)
            assert len(got) <= cap
            for k, (length, dist) in enumerate(got):
                # each entry reaches its length at its distance, and no nearer occurrence reaches it
                assert data[pos:pos + length] == data[pos - dist - 1:pos - dist - 1 + length]
                assert 2 <= length <= min(273, n - pos)
                if k:
                    assert length > got[k - 1][0] and dist > got[k - 1][1]
            if got and got[-1][0] == min(273, n - pos):
                assert got == brute_match_list(data, pos, 100000, 100000)[:len(got)]


def test_match_list_stops_at_273(parse):
    data = bytes(2000)
    assert [tuple(r) for r in parse.match_list(data, 500)] == [(273, 0)]
    assert [tuple(r) for r in parse.match_list(data, 1990)] == [(10, 0)]
    assert parse.match_list(data, 0).size == 0 and parse.match_list(data, 1999).size == 0


@pytest.mark.parametrize("kind", ["text", "binary", "mixed"])
@pytest.mark.parametrize("n", [4096, 65536])
def test_optimal_slab_is_valid_and_round_trips(port, parse, corpora, kind, n):
    data = corpora(kind, n)
    slab = parse.optimal_slab(data)
    assert port.slab_valid(data, slab)
    stream = port.encode_slab(data, slab)
    assert lzma.decompress(stream, format=lzma.FORMAT_ALONE) == data
    again = parse.optimal_slab(data)  # the parse draws nothing
    assert all((again[f] == slab[f]).all() for f in ("type", "dist", "len"))


def test_optimal_slab_beats_greedy_on_text(port, parse, corpora):
    data = corpora("text", 65536)
    assert port.slab_cost(data, parse.optimal_slab(data)) < port.slab_cost(data, port.greedy_slab(data))


def _cli():
    from megalania_b200 import build
    cli = build.build_cli() or build.CLI
    assert os.path.exists(cli)
    return cli


def test_cli_optimal_usage(tmp_path):
    cli = _cli()
    f = tmp_path / "in.bin"
    f.write_bytes(b"hello hello hello")
    for args in (["--optimal", "4", "--greedy", "4", "--time", "1"],
                 ["--optimal", "4", "--resume", str(f), "--time", "1"],
                 ["--optimal", "4"],
                 ["--optimal", "4", "--epochs", "1", "--steps", "1"],
                 ["--optimal"]):
        r = subprocess.run([cli] + args + [str(f)], capture_output=True)
        assert r.returncode == 255 and b"usage:" in r.stderr and r.stdout == b"", args


# ---- GPU: the device parse ---------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def mg():
    import megalania_b200 as m
    m.load_library()
    return m


@pytest.mark.gpu
@pytest.mark.parametrize("max_occ", [0, 8])
@pytest.mark.parametrize("kind,n", [("text", 4096), ("binary", 4096), ("text", 65536), ("mixed", 65536)])
def test_optimal_init_equals_the_cpu_parse(mg, port, parse, corpora, kind, n, max_occ):
    data = corpora(kind, n)
    want = parse.optimal_slab(data, max_occ)
    with mg.Context(data) as ctx:
        an = mg.Annealer(ctx, 2, seed=3)
        an.set_slab(None)
        cost = an.optimal_init(1, max_occ, 1)
        got = an.get_slab(1)
        assert live_chain(got) == live_chain(want)
        assert cost == port.slab_cost(data, want)
        st = ctx.optimal_stats()
        assert st["nodes"] == n and st["kernel_ms"] > 0
        an.close()


@pytest.mark.gpu
@pytest.mark.parametrize("kind,n,regions,below_greedy", [("text", 65536, 16, True), ("mixed", 65536, 16, True),
                                                          ("mixed", MIB, 1024, False)])
def test_optimal_init_regions(mg, port, corpora, kind, n, regions, below_greedy):
    """Many regions: the stitched slab is valid, priced exactly and round-trips.  With 4 KiB regions it is cheaper
    than the greedy parse of the same regions; with 1 KiB regions (1024 at 1 MiB) it is not (measured on a B200:
    6 958 805 274 against 6 822 651 662): every region is one block priced by a fresh model, whose flat prices the
    greedy parse leaves behind packet by packet."""
    data = corpora(kind, n)
    with mg.Context(data) as ctx:
        an = mg.Annealer(ctx, 2, seed=3)
        an.set_slab(None)
        cost = an.optimal_init(regions, 0, 0)
        slab = an.get_slab(0)
        assert port.slab_valid(data, slab)
        assert cost == ctx.score_slab(slab) == port.slab_cost(data, slab)
        assert lzma.decompress(ctx.encode_slab(slab), format=lzma.FORMAT_ALONE) == data
        assert ctx.optimal_stats()["nodes"] == n
        if below_greedy:
            greedy = an.greedy_init(regions, 1)
            assert cost < greedy, (cost, greedy)
        an.close()


@pytest.mark.gpu
def test_anneal_from_the_optimal_slab(mg, corpora):
    data = corpora("text", 65536)
    with mg.Context(data) as ctx:
        chains = 64
        an = mg.Annealer(ctx, chains, seed=5)
        an.set_slab(None)
        cost = an.optimal_init(16)
        an.broadcast_chain(0)
        cur, _ = an.costs()
        assert (cur == cost).all()
        an.run(50, schedule=mg.SCHEDULE_TEMPERATURE, temperatures=np.zeros(chains, dtype=np.float32))
        cur, best = an.costs()
        assert (cur <= cost).all()
        assert (best[best > 0] <= cost).all()
        an.close()


@pytest.mark.gpu
def test_cli_optimal(corpora, tmp_path):
    data = corpora("text", 65536)
    src = tmp_path / "in.bin"
    src.write_bytes(data)
    r = subprocess.run([_cli(), "--chains", "512", "--optimal", "16", "--time", "2", str(src)],
                       stdout=subprocess.PIPE, stderr=subprocess.PIPE)
    assert r.returncode == 0, r.stderr.decode(errors="replace")
    assert b"optimal parse" in r.stderr
    assert lzma.decompress(r.stdout, format=lzma.FORMAT_ALONE) == data

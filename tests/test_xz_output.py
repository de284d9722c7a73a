""".xz output: mg_encode_slab_xz / Context.encode_xz write a slab as one .xz stream whose LZMA2 chunks are range-coded
side by side on the device, and `megalania --format xz` writes its result that way.  The CPU tests pin a CPU writer
built on the oracle port (tests/xz_writer.c, compiled into a temporary directory): its streams decode with liblzma and
`xz -t`, and their chunk headers follow the plan rule of include/megalania_cuda.h.  The GPU tests hold the device
stream to it byte for byte."""
import ctypes
import lzma
import os
import shutil
import subprocess

import numpy as np
import pytest

MIB = 1 << 20
GRANULE = 4096
MAX_U, MAX_C = 1 << 21, 1 << 16
EINVAL = -1
INPUTS = [("binary", 4096), ("text", 65536), ("mixed", MIB)]
CHUNK_BYTES = (61440, 256)


class CpuXz:
    """ctypes binding of tests/xz_writer.c."""

    def __init__(self, path: str):
        self.lib = ctypes.CDLL(path)
        vp, sz, u32 = ctypes.c_void_p, ctypes.c_size_t, ctypes.c_uint32
        self.lib.cpu_encode_xz.restype = sz
        self.lib.cpu_encode_xz.argtypes = [vp, sz, vp, u32, vp, sz, vp, sz, ctypes.POINTER(sz)]
        self.lib.cpu_xz_candidates.restype = sz
        self.lib.cpu_xz_candidates.argtypes = [vp, sz, vp, vp, vp, sz]

    def encode(self, data, slab, chunk_bytes=0):
        """(stream, chunk bounds: starts and n)"""
        d = np.ascontiguousarray(np.frombuffer(bytes(data), dtype=np.uint8))
        cap = 2 * d.size + MAX_C
        out = np.zeros(cap, dtype=np.uint8)
        bounds = np.zeros(d.size // GRANULE + 2, dtype=np.uint32)
        chunks = ctypes.c_size_t(0)
        got = int(self.lib.cpu_encode_xz(d.ctypes.data, d.size, slab.ctypes.data, chunk_bytes, out.ctypes.data, cap,
                                         bounds.ctypes.data, bounds.size, ctypes.byref(chunks)))
        assert 0 < got <= cap
        return out[:got].tobytes(), bounds[:chunks.value + 1].astype(np.int64)

    def candidates(self, data, slab):
        """(positions, cost before each): 0, the first boundary at or after each multiple of 4096 below n, n"""
        d = np.ascontiguousarray(np.frombuffer(bytes(data), dtype=np.uint8))
        cap = d.size // GRANULE + 2
        pos = np.zeros(cap, dtype=np.uint32)
        cost = np.zeros(cap, dtype=np.uint64)
        got = int(self.lib.cpu_xz_candidates(d.ctypes.data, d.size, slab.ctypes.data, pos.ctypes.data, cost.ctypes.data, cap))
        assert got <= cap
        return pos[:got].astype(np.int64), cost[:got].astype(np.int64)


def _compile(tmp_path_factory, name):
    """Compiled here, into a temporary directory: the tree may be read-only."""
    src = os.path.join(os.path.dirname(os.path.abspath(__file__)), name + ".c")
    lib = str(tmp_path_factory.mktemp(name) / f"lib{name}.so")
    subprocess.run(["gcc", "-O2", "-std=gnu11", "-Wall", "-Wextra", "-fPIC", "-shared", "-o", lib, src, "-lm"], check=True)
    return lib


@pytest.fixture(scope="module")
def writer(tmp_path_factory):
    return CpuXz(_compile(tmp_path_factory, "xz_writer"))


@pytest.fixture(scope="module")
def decode_lzma(tmp_path_factory):
    """LZMA-alone stream -> slab, by the CPU decoder of tests/stream_decoder.c."""
    from oracle import oracle_lib
    lib = ctypes.CDLL(_compile(tmp_path_factory, "stream_decoder"))
    lib.cpu_decode_stream.restype = ctypes.c_int
    lib.cpu_decode_stream.argtypes = [ctypes.c_void_p, ctypes.c_size_t, ctypes.c_void_p, ctypes.c_size_t, ctypes.c_void_p]

    def decode(data, stream):
        d = np.frombuffer(bytes(data), dtype=np.uint8)
        s = np.frombuffer(bytes(stream), dtype=np.uint8)
        slab = oracle_lib.literal_slab(d.size)
        assert lib.cpu_decode_stream(d.ctypes.data, d.size, s.ctypes.data, s.size, slab.ctypes.data) == 0
        return slab
    return decode


def liblzma_lc0(data) -> bytes:
    return lzma.compress(data, format=lzma.FORMAT_ALONE,
                         filters=[{"id": lzma.FILTER_LZMA1, "preset": 6, "lc": 0, "lp": 0, "pb": 0}])


_SLABS = {}


def make_slab(port, corpora, decode_lzma, kind, n, which):
    """literal, greedy (the oracle's greedy parse: 4 KiB and 64 KiB only, it takes minutes at 1 MiB on the CPU) or
    liblzma (liblzma's lc = 0 stream decoded to a slab)."""
    key = (kind, n, which)
    if key not in _SLABS:
        from oracle import oracle_lib
        data = corpora(kind, n)
        if which == "literal":
            _SLABS[key] = oracle_lib.literal_slab(n)
        elif which == "greedy":
            _SLABS[key] = port.greedy_slab(data)
        else:
            _SLABS[key] = decode_lzma(data, liblzma_lc0(data))
    return _SLABS[key]


CASES = [(kind, n, which) for kind, n in INPUTS for which in ("literal", "greedy", "liblzma")
         if not (which == "greedy" and n == MIB)]


def parse_chunks(stream):
    """The LZMA2 chunks of a one-block .xz stream: (control, u, c, payload offset) each."""
    assert stream[:6] == b"\xfd7zXZ\x00" and stream[6:8] == b"\x00\x04" and stream[-2:] == b"YZ"
    at = 12 + (stream[12] + 1) * 4
    out = []
    while stream[at] != 0:
        ctl = stream[at]
        u = ((ctl & 0x1F) << 16 | stream[at + 1] << 8 | stream[at + 2]) + 1
        c = (stream[at + 3] << 8 | stream[at + 4]) + 1
        head = 6 if not out else 5
        if not out:
            assert stream[at + 5] == 0x00  # properties: lc = lp = pb = 0
        out.append((ctl, u, c, at + head))
        at += head + c
    return out


def check_stream(data, stream):
    assert lzma.decompress(stream, format=lzma.FORMAT_XZ) == data  # verifies the CRC64 too
    if shutil.which("xz"):
        subprocess.run(["xz", "-t", "-"], input=stream, check=True)
    chunks = parse_chunks(stream)
    assert 0xE0 <= chunks[0][0] <= 0xFF
    assert all(0x80 <= ctl <= 0x9F for ctl, _, _, _ in chunks[1:])
    for _, u, c, off in chunks:
        assert u <= MAX_U and c <= MAX_C
        assert stream[off] == 0  # every chunk's range coder restarts
    assert sum(u for _, u, _, _ in chunks) == len(data)
    return chunks


def plan(pos, cost, chunk_bytes):
    """The plan rule of include/megalania_cuda.h, restated."""
    budget = chunk_bytes * 8 * 2048
    bounds, s = [0], 0
    while s + 1 < len(pos):
        ok = [e for e in range(s + 1, len(pos)) if cost[e] - cost[s] <= budget and pos[e] - pos[s] <= MAX_U]
        s = ok[-1] if ok else s + 1
        bounds.append(int(pos[s]))
    return bounds


def live_positions(slab):
    out, p = [], 0
    while p < slab.size:
        out.append(p)
        p += int(slab[p]["len"])
    return out


# ---- CPU: the CPU writer -----------------------------------------------------------------------------------
@pytest.mark.parametrize("chunk_bytes", CHUNK_BYTES)
@pytest.mark.parametrize("kind,n,which", CASES)
def test_cpu_writer(port, corpora, decode_lzma, writer, kind, n, which, chunk_bytes):
    data = corpora(kind, n)
    slab = make_slab(port, corpora, decode_lzma, kind, n, which)
    stream, bounds = writer.encode(data, slab, chunk_bytes)
    chunks = check_stream(data, stream)
    assert len(chunks) == len(bounds) - 1
    assert [u for _, u, _, _ in chunks] == list(np.diff(bounds))
    # the cuts are the planned candidates, and the candidates are packet boundaries priced as the port prices them
    pos, cost = writer.candidates(data, slab)
    live = set(live_positions(slab)) | {n}
    assert set(pos.tolist()) <= live
    for k in range(1, len(pos) - 1):
        assert pos[k] >= k * GRANULE and pos[k] - k * GRANULE < 273
    for k in (len(pos) // 3, len(pos) - 1):
        assert cost[k] == port.prefix_cost(data, slab, int(pos[k]))
    assert list(bounds) == plan(pos, cost, chunk_bytes)
    # the same packets as the .lzma stream, plus the container and one header and flush per chunk
    lzma_len = len(port.encode_slab(data, slab))
    assert lzma_len - 13 < len(stream) <= lzma_len + 60 + 10 * len(chunks)


def test_cpu_writer_one_byte(port, writer):
    from oracle import oracle_lib
    stream, bounds = writer.encode(b"x", oracle_lib.literal_slab(1))
    assert list(bounds) == [0, 1]
    check_stream(b"x", stream)


def test_cpu_writer_match_across_a_granule(port, writer):
    """A 273-byte MATCH that straddles offset 4096: the cut moves to the packet's end."""
    from oracle import oracle_lib
    rng = np.random.default_rng(3)
    data = bytearray(rng.integers(0, 256, 8192, dtype=np.uint8).tobytes())
    data[4000:4273] = data[100:373]
    data = bytes(data)
    slab = oracle_lib.literal_slab(len(data))
    slab[4000] = (2, 4000 - 100 - 1, 273)
    assert port.slab_valid(data, slab)
    pos, _ = writer.candidates(data, slab)
    assert list(pos) == [0, 4273, 8192]
    stream, bounds = writer.encode(data, slab, 256)
    assert list(bounds) == [0, 4273, 8192]
    check_stream(data, stream)


def _cli():
    from megalania_b200 import build
    cli = build.build_cli() or build.CLI
    assert os.path.exists(cli)
    return cli


def test_cli_format_usage(tmp_path):
    f = tmp_path / "in.bin"
    f.write_bytes(b"hello hello hello")
    for args in (["--format", "foo"], ["--format"], ["--format", "XZ"]):
        r = subprocess.run([_cli()] + args + [str(f)], capture_output=True)
        assert r.returncode == 255 and b"usage:" in r.stderr and r.stdout == b"", args


# ---- GPU: the device stream against the CPU writer --------------------------------------------------------
@pytest.fixture(scope="module")
def mg():
    import megalania_b200 as m
    m.load_library()
    return m


@pytest.mark.gpu
def test_device_equals_cpu_writer(mg, port, corpora, decode_lzma, writer):
    for kind, n in INPUTS:
        data = corpora(kind, n)
        with mg.Context(data) as ctx:
            slabs = {which: make_slab(port, corpora, decode_lzma, kind, n, which) for k, m_, which in CASES if (k, m_) == (kind, n)}
            if n == MIB:
                # the device's greedy parse of one region is the oracle's greedy slab
                an = mg.Annealer(ctx, 1)
                an.set_slab(None)
                an.greedy_init(1)
                slabs["greedy"] = an.get_slab(0)
                an.close()
            for which, slab in slabs.items():
                for chunk_bytes in CHUNK_BYTES:
                    got = ctx.encode_xz(slab, chunk_bytes)
                    want, bounds = writer.encode(data, slab, chunk_bytes)
                    assert got == want, (kind, n, which, chunk_bytes)
                    st = ctx.encode_xz_stats()
                    chunks = parse_chunks(got)
                    assert st["chunks"] == len(chunks) == len(bounds) - 1
                    assert st["plan_ms"] > 0 and st["code_ms"] > 0
                    lzma_stream = ctx.encode_slab(slab)
                    assert st["events"] == ctx.encode_stats()["events"], (kind, n, which, chunk_bytes)
                    if len(chunks) == 1:
                        # one chunk: its payload is the LZMA-alone payload of the already-pinned coder
                        _, _, c, off = chunks[0]
                        assert got[off:off + c] == ctx.encode_slab_buffer(slab)[13:] == lzma_stream[13:]
            if n in (4096, 65536):
                assert ctx.encode_xz(slabs["literal"]) and ctx.encode_xz_stats()["chunks"] == 1
            if n == MIB:
                ctx.encode_xz(slabs["literal"], 256)
                assert ctx.encode_xz_stats()["chunks"] == MIB // GRANULE


@pytest.mark.gpu
def test_device_after_annealing_and_bad_arguments(mg, port, corpora, writer):
    data = corpora("text", 65536)
    with mg.Context(data) as ctx:
        an = mg.Annealer(ctx, 64, seed=9)
        an.set_slab(None)
        an.run(200)
        slab = an.get_slab(0)
        an.close()
        assert port.slab_valid(data, slab)
        for chunk_bytes in CHUNK_BYTES:
            assert ctx.encode_xz(slab, chunk_bytes) == writer.encode(data, slab, chunk_bytes)[0]
        for bad in (1, 255, 61441):
            with pytest.raises(mg.MegalaniaError) as err:
                ctx.encode_xz(slab, bad)
            assert err.value.code == EINVAL
        broken = slab.copy()
        broken[0] = (2, 5, 10)  # a match before any data
        with pytest.raises(mg.MegalaniaError) as err:
            ctx.encode_xz(broken)
        assert err.value.code == -4


@pytest.mark.gpu
def test_device_16mib_smoke(mg, corpora):
    data = corpora("corpus16", 16 * MIB)
    with mg.Context(data) as ctx:
        stream = ctx.encode_xz(mg.literal_slab(len(data)))
        st = ctx.encode_xz_stats()
    assert lzma.decompress(stream, format=lzma.FORMAT_XZ) == data
    assert st["chunks"] == len(parse_chunks(stream)) > 100


@pytest.mark.gpu
def test_cli_format_xz(port, corpora, tmp_path, writer, decode_lzma):
    """The epoch schedule computes the same slab on every run, so the .xz output is the CPU writer's stream of the
    slab the .lzma output holds; the rounds schedule (--greedy, clock-boxed) and --resume are checked for round trips."""
    cli = _cli()
    data = corpora("text", 65536)
    src = tmp_path / "in.bin"
    src.write_bytes(data)
    epochs = ["--chains", "256", "--iters", "200", "--epochs", "1", "--steps", "1"]

    def run(*args):
        r = subprocess.run([cli] + list(args) + [str(src)], stdout=subprocess.PIPE, stderr=subprocess.PIPE)
        assert r.returncode == 0, r.stderr.decode(errors="replace")
        return r.stdout

    as_lzma = run(*epochs)
    default = run(*epochs, "--format", "lzma")
    assert default == as_lzma
    as_xz = run(*epochs, "--format", "xz")
    chunks = check_stream(data, as_xz)
    slab = decode_lzma(data, as_lzma)
    assert as_xz == writer.encode(data, slab)[0]
    assert len(as_xz) <= len(as_lzma) + 60 + 10 * len(chunks)

    rounds = run("--chains", "512", "--rounds", "3", "--round-ms", "100", "--greedy", "16", "--format", "xz")
    check_stream(data, rounds)

    prev = tmp_path / "prev.lzma"
    prev.write_bytes(as_lzma)
    resumed_lzma = run(*epochs, "--resume", str(prev))
    resumed_xz = run(*epochs, "--resume", str(prev), "--format", "xz")
    check_stream(data, resumed_xz)
    assert resumed_xz == writer.encode(data, decode_lzma(data, resumed_lzma))[0]

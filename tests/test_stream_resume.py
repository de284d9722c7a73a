"""Resuming from an .lzma stream: mg_decode_stream / Context.decode_stream turn an LZMA-alone stream of the input
(lc = lp = pb = 0: an earlier megalania output, or liblzma's) back into a slab, and `megalania --resume` starts the
search from it.  The CPU tests pin a CPU decoder built on the oracle port's model (tests/stream_decoder.c, compiled
into a temporary directory); the GPU tests hold the device decoder to it, array for array."""
import ctypes
import lzma
import os
import subprocess

import numpy as np
import pytest

MIB = 1 << 20
EINVAL, ESLAB = -1, -4
INPUTS = [(kind, n) for kind in ("text", "binary", "mixed") for n in (4096, 65536)]
SLABS = ("literal", "greedy", "annealed")
PRESETS = {"preset0": 0, "preset6": 6, "preset9e": 9 | lzma.PRESET_EXTREME}


def lc0_filters(preset):
    return [{"id": lzma.FILTER_LZMA1, "preset": preset, "lc": 0, "lp": 0, "pb": 0}]


def xz_lc0(data, preset=9 | lzma.PRESET_EXTREME) -> bytes:
    """liblzma's LZMA-alone stream at lc = lp = pb = 0: size field all ones, ended by the end marker."""
    return lzma.compress(data, format=lzma.FORMAT_ALONE, filters=lc0_filters(preset))


def live_positions(slab):
    out, p = [], 0
    while p < slab.size:
        out.append(p)
        p += int(slab[p]["len"])
    return np.array(out, dtype=np.int64)


def canonical(slab):
    """What decoding the slab's stream gives: its live packets, LITERAL / 0 / 1 everywhere else."""
    from oracle import oracle_lib
    out = oracle_lib.literal_slab(slab.size)
    live = live_positions(slab)
    out[live] = slab[live]
    return out


def same(a, b):
    return all((a[f] == b[f]).all() for f in ("type", "dist", "len"))


class DecodeError(ValueError):
    def __init__(self, code: int):
        super().__init__(f"stream rejected with code {code}")
        self.code = code


class CpuDecoder:
    """ctypes binding of cpu_decode_stream (tests/stream_decoder.c)."""

    def __init__(self, path: str):
        self.lib = ctypes.CDLL(path)
        vp, sz = ctypes.c_void_p, ctypes.c_size_t
        self.lib.cpu_decode_stream.restype = ctypes.c_int
        self.lib.cpu_decode_stream.argtypes = [vp, sz, vp, sz, vp]

    def decode_stream(self, data, stream) -> np.ndarray:
        """LZMA-alone stream (lc = lp = pb = 0) of `data` -> slab; raises DecodeError(-1 header / -4 payload)."""
        from oracle import oracle_lib
        d = np.ascontiguousarray(np.frombuffer(bytes(data), dtype=np.uint8))
        s = np.ascontiguousarray(np.frombuffer(bytes(stream), dtype=np.uint8))
        slab = oracle_lib.literal_slab(d.size)
        rc = self.lib.cpu_decode_stream(d.ctypes.data_as(ctypes.c_void_p), d.size, s.ctypes.data_as(ctypes.c_void_p),
                                        s.size, slab.ctypes.data_as(ctypes.c_void_p))
        if rc != 0:
            raise DecodeError(rc)
        return slab


@pytest.fixture(scope="module")
def decoder(tmp_path_factory):
    """Compiled here, into a temporary directory: the tree may be read-only."""
    src = os.path.join(os.path.dirname(os.path.abspath(__file__)), "stream_decoder.c")
    lib = str(tmp_path_factory.mktemp("stream_decoder") / "libstream_decoder.so")
    subprocess.run(["gcc", "-O2", "-std=gnu11", "-Wall", "-Wextra", "-fPIC", "-shared", "-o", lib, src, "-lm"], check=True)
    return CpuDecoder(lib)


_SLAB_CACHE = {}


def make_slab(port, corpora, kind, n, which):
    key = (kind, n, which)
    if key not in _SLAB_CACHE:
        from oracle import oracle_lib
        data = corpora(kind, n)
        if which == "literal":
            slab = oracle_lib.literal_slab(n)
        elif which == "greedy":
            slab = port.greedy_slab(data)
        else:
            # a few hundred proposals of the oracle's annealer from the all-literal slab: matches, reps and the
            # hidden (non-live) slots they leave behind
            slab = oracle_lib.literal_slab(n)
            best = slab.copy()
            port.anneal_epoch(data, slab, best, 0, 0, rng_mode=1, rng_state=port.chain_seed(11, n), evals=300)
        _SLAB_CACHE[key] = slab
    return _SLAB_CACHE[key]


# ---- CPU: the CPU decoder ---------------------------------------------------------------------------------
@pytest.mark.parametrize("which", SLABS)
@pytest.mark.parametrize("kind,n", INPUTS)
def test_own_streams_round_trip(port, corpora, kind, n, which, decoder):
    data = corpora(kind, n)
    slab = make_slab(port, corpora, kind, n, which)
    stream = port.encode_slab(data, slab)
    decoded = decoder.decode_stream(data, stream)
    assert same(decoded, canonical(slab))
    assert port.encode_slab(data, decoded) == stream
    live = np.zeros(n, dtype=bool)
    live[live_positions(decoded)] = True
    hidden = decoded[~live]
    assert (hidden["type"] == 1).all() and (hidden["dist"] == 0).all() and (hidden["len"] == 1).all()


@pytest.mark.parametrize("preset", list(PRESETS))
@pytest.mark.parametrize("kind,n", INPUTS)
def test_liblzma_streams(port, corpora, kind, n, preset, decoder):
    data = corpora(kind, n)
    stream = xz_lc0(data, PRESETS[preset])
    assert stream[5:13] == b"\xff" * 8  # size unknown: the end marker closes the stream
    decoded = decoder.decode_stream(data, stream)
    assert port.slab_valid(data, decoded)
    again = port.encode_slab(data, decoded)
    assert lzma.decompress(again, format=lzma.FORMAT_ALONE) == data
    # the same packets without the end marker (> 30 bits) and with the size in the header
    assert len(again) < len(stream)


def rejections(port, corpora):
    """(name, stream, code) of the 64 KiB text's streams that must be refused, all deterministic."""
    data = corpora("text", 65536)
    own = port.encode_slab(data, make_slab(port, corpora, "text", 65536, "greedy"))
    other = corpora("binary", 65536)
    out = [("lc3", lzma.compress(data, format=lzma.FORMAT_ALONE), EINVAL),
           ("size", own[:5] + (65537).to_bytes(8, "little") + own[13:], EINVAL),
           ("too-short", own[:17], EINVAL),
           ("other-input", port.encode_slab(other, port.greedy_slab(other)), ESLAB),
           ("other-input-xz", xz_lc0(other), ESLAB),
           ("appended", own + b"\x00", ESLAB),
           ("first-byte", own[:13] + b"\x01" + own[14:], ESLAB)]
    for cut in (18, 100, len(own) // 2, len(own) - 1):
        out.append((f"cut{cut}", own[:cut], ESLAB))
    flip = bytearray(own)
    flip[len(own) // 3] ^= 0x10
    out.append(("flipped", bytes(flip), ESLAB))
    xz = xz_lc0(data)
    out.append(("xz-cut", xz[:-3], ESLAB))
    return data, out


def test_rejections(port, corpora, decoder):
    data, cases = rejections(port, corpora)
    for name, stream, code in cases:
        with pytest.raises(DecodeError) as err:
            decoder.decode_stream(data, stream)
        assert err.value.code == code, name


def _cli():
    from megalania_b200 import build
    cli = build.build_cli() or build.CLI
    assert os.path.exists(cli)
    return cli


def test_cli_resume_usage(tmp_path):
    cli = _cli()
    f = tmp_path / "in.bin"
    f.write_bytes(b"hello hello hello")
    r = subprocess.run([cli, "--resume"], capture_output=True)
    assert r.returncode == 255 and b"usage:" in r.stderr and r.stdout == b""
    r = subprocess.run([cli, "--resume", "x", "--greedy", "4", str(f)], capture_output=True)
    assert r.returncode == 255 and b"usage:" in r.stderr and r.stdout == b""
    r = subprocess.run([cli, "--resume", str(tmp_path / "missing.lzma"), str(f)], capture_output=True)
    assert r.returncode == 255 and r.stdout == b""


# ---- GPU: the device decoder against the oracle's --------------------------------------------------------
@pytest.fixture(scope="module")
def mg():
    import megalania_b200 as m
    m.load_library()
    return m


@pytest.mark.gpu
def test_device_decoder_matches_the_cpu_decoder(mg, port, corpora, decoder):
    for kind, n in INPUTS:
        data = corpora(kind, n)
        with mg.Context(data) as ctx:
            for which in SLABS:
                stream = port.encode_slab(data, make_slab(port, corpora, kind, n, which))
                got = ctx.decode_stream(stream)
                assert same(got, decoder.decode_stream(data, stream)), (kind, n, which)
                events = ctx.decode_stats()["events"]
                assert events > 0
                assert ctx.encode_slab(got) == stream, (kind, n, which)
                assert ctx.encode_stats()["events"] == events  # the same bits, coded and decoded
            for preset, p in PRESETS.items():
                stream = xz_lc0(data, p)
                got = ctx.decode_stream(stream)
                assert same(got, decoder.decode_stream(data, stream)), (kind, n, preset)
                assert ctx.decode_stats()["events"] > 0


@pytest.mark.gpu
def test_device_decoder_full_size(mg, port, corpora, decoder):
    """The 1 MiB mixed corpus: the stream of the device's greedy parse (one region = the oracle's greedy slab), and
    liblzma's -9e stream."""
    data = corpora("mixed", MIB)
    with mg.Context(data) as ctx:
        an = mg.Annealer(ctx, 1)
        an.set_slab(None)
        an.greedy_init(1)
        greedy = an.get_slab(0)
        an.close()
        for stream in (ctx.encode_slab(greedy), xz_lc0(data)):
            got = ctx.decode_stream(stream)
            st = ctx.decode_stats()
            assert st["events"] > 0 and st["kernel_ms"] > 0
            assert same(got, decoder.decode_stream(data, stream))
        assert same(ctx.decode_stream(ctx.encode_slab(greedy)), canonical(greedy))


@pytest.mark.gpu
def test_device_rejections(mg, port, corpora):
    data, cases = rejections(port, corpora)
    lit = mg.literal_slab(len(data))
    with mg.Context(data) as ctx:
        expect = ctx.score_slab(lit)
        for name, stream, code in cases:
            with pytest.raises(mg.MegalaniaError) as err:
                ctx.decode_stream(stream)
            assert err.value.code == code, (name, str(err.value))
            # no sticky CUDA error: the context still computes
            assert ctx.score_slab(lit) == expect, name
        assert "lc = 3" in str(pytest.raises(mg.MegalaniaError, ctx.decode_stream, cases[0][1]).value)


@pytest.mark.gpu
def test_annealer_from_a_decoded_slab(mg, port, corpora):
    data = corpora("text", 65536)
    with mg.Context(data) as ctx:
        decoded = ctx.decode_stream(xz_lc0(data))
        cost = port.slab_cost(data, decoded)
        assert ctx.score_slab(decoded) == cost
        chains = 64
        an = mg.Annealer(ctx, chains, seed=5)
        an.set_slab(decoded, adopt_cost=True)
        cur, _ = an.costs()
        assert (cur == cost).all()
        an.run(50, schedule=mg.SCHEDULE_TEMPERATURE, temperatures=np.zeros(chains, dtype=np.float32))
        cur, best = an.costs()
        assert (cur <= cost).all()
        assert (best[best > 0] <= cost).all()
        an.close()


def _decoded_cost(port, decoder, data, stream):
    return port.slab_cost(data, decoder.decode_stream(data, stream))


@pytest.mark.gpu
@pytest.mark.parametrize("schedule", [["--chains", "256", "--iters", "200", "--epochs", "1", "--steps", "1"],
                                      ["--chains", "512", "--rounds", "3", "--round-ms", "100"]],
                         ids=["epochs", "rounds"])
def test_cli_resume(port, corpora, tmp_path, schedule, decoder):
    cli = _cli()
    data = corpora("text", 65536)
    src = tmp_path / "in.bin"
    src.write_bytes(data)

    def run(*extra):
        return subprocess.run([cli] + schedule + list(extra) + [str(src)], stdout=subprocess.PIPE, stderr=subprocess.PIPE)

    first = run()
    assert first.returncode == 0, first.stderr.decode(errors="replace")
    prev = tmp_path / "first.lzma"
    prev.write_bytes(first.stdout)
    second = run("--resume", str(prev))
    assert second.returncode == 0, second.stderr.decode(errors="replace")
    assert b"resumed" in second.stderr
    assert lzma.decompress(second.stdout, format=lzma.FORMAT_ALONE) == data
    assert _decoded_cost(port, decoder, data, second.stdout) <= _decoded_cost(port, decoder, data, first.stdout)

    xz = xz_lc0(data)
    xzf = tmp_path / "xz.lzma"
    xzf.write_bytes(xz)
    third = run("--resume", str(xzf))
    assert third.returncode == 0, third.stderr.decode(errors="replace")
    assert lzma.decompress(third.stdout, format=lzma.FORMAT_ALONE) == data
    assert _decoded_cost(port, decoder, data, third.stdout) <= _decoded_cost(port, decoder, data, xz)
    assert len(third.stdout) <= len(xz)

    other = tmp_path / "other.lzma"
    other.write_bytes(xz_lc0(corpora("binary", 65536)))
    bad = run("--resume", str(other))
    assert bad.returncode == 255 and bad.stdout == b"" and b"mg_decode_stream" in bad.stderr

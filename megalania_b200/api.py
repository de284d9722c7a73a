"""ctypes binding of libmegalania_cuda.so — the Python mirror of the host interface.

The names follow the reference's vocabulary (slab, packet, top-k finder, perplexity = cost):
  Context(data)                 lzma_state_init + packet_enumerator_new + top_k_packet_finder_new
  Context.score_slabs(slabs)    perplexity_encoder total of a slab          (src/perplexity_encoder.c)
  Context.find_topk(...)        top_k_packet_finder_find + pop loop         (src/top_k_packet_finder.c)
  Context.encode_slab(slab)     header + range_encoder pass                 (src/main.c:110-119)
  Context.encode_xz(slab)       the same slab as an .xz stream, LZMA2 chunks coded side by side  (no reference counterpart)
  Context.decode_stream(stream) .lzma stream (lc = lp = pb = 0) -> slab, to resume a search (no reference counterpart)
  Annealer.optimal_init(...)    shortest-path parse as a starting slab                           (no reference counterpart)
  Annealer(ctx, chains, ...)    the loop of src/main.c:78-102 on many chains

There is no CPU path: importing works anywhere, but every compute call needs the CUDA library
(built in-tree by megalania_b200.build) and a GPU, and raises MegalaniaError otherwise.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

from . import build as _build

# LZMAPacket, reference src/lzma_packet.h:13-17
PACKET_DTYPE = np.dtype({"names": ["type", "dist", "len"], "formats": ["u1", "<u4", "<u2"],
                         "offsets": [0, 4, 8], "itemsize": 12})
TRACE_DTYPE = np.dtype([("cost", "<u8"), ("flags", "<u4"), ("undo_count", "<u4")])
MODEL_DTYPE = np.dtype({"names": ["probs", "ctx_state", "dists", "position", "cost"],
                        "formats": [("<u2", 2615), "u1", ("<u4", 4), "<u8", "<u8"],
                        "offsets": [0, 5230, 5232, 5248, 5256], "itemsize": 5264})
INVALID, LITERAL, MATCH, SHORT_REP, LONG_REP = 0, 1, 2, 3, 4
SCHEDULE_REFERENCE, SCHEDULE_TEMPERATURE = 0, 1
CONTINUE_EVALS = 0xFFFFFFFF
NO_OWNER = 0xFFFFFFFF  # merge_export: a region that lives on another process

ERRORS = {-1: "MG_EINVAL", -2: "MG_ECUDA", -3: "MG_ENOMEM", -4: "MG_ESLAB", -5: "MG_EOUTPUT", -6: "MG_ESTATE"}


class MegalaniaError(RuntimeError):
    def __init__(self, code: int, message: str):
        super().__init__(f"{ERRORS.get(code, code)}: {message}")
        self.code = code


class LZMAProperties(C.Structure):
    _fields_ = [("lc", C.c_uint8), ("lp", C.c_uint8), ("pb", C.c_uint8)]


class AnnealParams(C.Structure):
    _fields_ = [("chains", C.c_uint32), ("top_k", C.c_uint32), ("checkpoint_stride", C.c_uint32),
                ("edit_log_capacity", C.c_uint32), ("track_best", C.c_uint32), ("trace_capacity", C.c_uint32),
                ("seed", C.c_uint64)]


class AnnealRunParams(C.Structure):
    _fields_ = [("evals", C.c_uint32), ("max_attempts", C.c_uint32), ("schedule", C.c_uint32),
                ("step", C.c_uint32), ("num_iters", C.c_uint32), ("first_eval", C.c_uint32),
                ("temperatures", C.POINTER(C.c_float)), ("packet_budget", C.c_uint64), ("no_early_exit", C.c_uint32),
                ("suspend", C.c_uint32), ("cycle_budget", C.c_uint64), ("regions", C.POINTER(C.c_uint32))]


class AnnealStats(C.Structure):
    _fields_ = [(name, C.c_uint64) for name in (
        "evals", "attempts", "accepted", "new_best", "packets_scored", "bits_scored", "slab_bytes_read",
        "checkpoint_bytes", "finder_calls", "finder_candidates", "edits", "log_overflows", "rejoined", "finder_cycles", "chain_cycles",
        "finder_chunks", "max_chain_cycles", "finder_gave_up")] + [
        ("kernel_ms", C.c_double), ("launches", C.c_uint32)]

    def as_dict(self) -> dict:
        return {name: getattr(self, name) for name, _ in self._fields_}


WRITE_FN = C.CFUNCTYPE(C.c_bool, C.c_void_p, C.c_void_p, C.c_size_t)


class OutputInterface(C.Structure):
    """reference src/output_interface.h:8-13"""
    _fields_ = [("write", WRITE_FN), ("private_data", C.c_void_p)]


EXPORTS = [
    "mg_last_error", "mg_version", "mg_ctx_create", "mg_ctx_destroy", "mg_ctx_size", "mg_ctx_device",
    "mg_score_slabs", "mg_find_topk", "mg_encode_slab", "mg_encode_slab_buffer", "mg_anneal_create",
    "mg_anneal_destroy", "mg_anneal_chain_bytes", "mg_anneal_set_slab", "mg_anneal_run", "mg_anneal_costs",
    "mg_anneal_get_slab", "mg_anneal_get_trace", "mg_anneal_swap_chains", "mg_anneal_device_slab",
    "mg_anneal_refresh_chain", "mg_anneal_oneshot", "mg_debug_model_after_prefix", "mg_anneal_export_slab",
    "mg_anneal_import_slab", "mg_anneal_merge_regions", "mg_anneal_broadcast_chain", "mg_find_topk_stats",
    "mg_anneal_merge_export", "mg_anneal_merge_import", "mg_debug_index", "mg_encode_stats", "mg_ctx_full_wave", "mg_ctx_sm_clock_khz",
    "mg_comm_unique_id", "mg_comm_init", "mg_comm_destroy", "mg_comm_rank", "mg_comm_size", "mg_comm_exchange_best",
    "mg_comm_temper_exchange", "mg_temper_decide", "mg_comm_merge_regions", "mg_comm_stats", "mg_pool_trim",
    "mg_comm_broadcast_chain", "mg_comm_allgather_u64", "mg_ctx_set_finder_limits", "mg_anneal_greedy_init",
    "mg_decode_stream", "mg_decode_stats", "mg_anneal_optimal_init", "mg_optimal_stats", "mg_encode_slab_xz",
    "mg_encode_xz_stats",
]

_lib = None


def library_path() -> str:
    """The in-tree library; MEGALANIA_CUDA_LIB selects another build of the same sources (kernel experiments)."""
    return os.environ.get("MEGALANIA_CUDA_LIB") or _build.LIB


def load_library(build_if_missing: bool = True) -> C.CDLL:
    """Loads the CUDA library; raises if it is absent (there is nothing to fall back to)."""
    global _lib
    if _lib is not None:
        return _lib
    path = library_path()
    if not os.path.exists(path):
        if not build_if_missing:
            raise MegalaniaError(-2, f"{path} is missing: run `python -m megalania_b200.build`")
        _build.build_library()
    L = C.CDLL(path)
    vp, sz, u32, u64, i32 = C.c_void_p, C.c_size_t, C.c_uint32, C.c_uint64, C.c_int
    L.mg_last_error.restype = C.c_char_p
    L.mg_version.restype = u32
    L.mg_ctx_create.argtypes = [vp, sz, LZMAProperties, i32, C.POINTER(vp)]
    L.mg_ctx_destroy.argtypes = [vp]
    L.mg_ctx_destroy.restype = None
    L.mg_ctx_size.argtypes = [vp]
    L.mg_ctx_size.restype = sz
    L.mg_ctx_device.argtypes = [vp]
    L.mg_ctx_set_finder_limits.argtypes = [vp, sz, u32]
    L.mg_ctx_full_wave.argtypes = [vp]
    L.mg_ctx_full_wave.restype = u32
    L.mg_ctx_sm_clock_khz.argtypes = [vp]
    L.mg_ctx_sm_clock_khz.restype = u32
    L.mg_score_slabs.argtypes = [vp, vp, sz, vp]
    L.mg_find_topk.argtypes = [vp, vp, i32, vp, sz, i32, vp, vp, vp]
    L.mg_find_topk_stats.argtypes = [vp, C.POINTER(C.c_double), C.POINTER(u64)]
    L.mg_encode_slab.argtypes = [vp, vp, C.POINTER(OutputInterface)]
    L.mg_encode_slab_buffer.argtypes = [vp, vp, vp, sz, C.POINTER(sz)]
    L.mg_anneal_create.argtypes = [vp, C.POINTER(AnnealParams), C.POINTER(vp)]
    L.mg_anneal_destroy.argtypes = [vp]
    L.mg_anneal_destroy.restype = None
    L.mg_anneal_chain_bytes.argtypes = [vp, C.POINTER(AnnealParams)]
    L.mg_anneal_chain_bytes.restype = sz
    L.mg_anneal_set_slab.argtypes = [vp, u32, u32, vp, i32, i32]
    L.mg_anneal_run.argtypes = [vp, C.POINTER(AnnealRunParams), C.POINTER(AnnealStats)]
    L.mg_anneal_costs.argtypes = [vp, vp, vp]
    L.mg_anneal_get_slab.argtypes = [vp, u32, i32, vp]
    L.mg_anneal_get_trace.argtypes = [vp, u32, vp, sz, C.POINTER(sz)]
    L.mg_anneal_swap_chains.argtypes = [vp, u32, u32]
    L.mg_anneal_device_slab.argtypes = [vp, u32, i32, C.POINTER(vp), C.POINTER(sz)]
    L.mg_anneal_refresh_chain.argtypes = [vp, u32, i32]
    L.mg_anneal_merge_regions.argtypes = [vp, u32, vp, vp, u32, C.POINTER(u64)]
    L.mg_anneal_broadcast_chain.argtypes = [vp, u32]
    L.mg_anneal_greedy_init.argtypes = [vp, u32, u32, C.POINTER(u64)]
    L.mg_anneal_merge_export.argtypes = [vp, u32, vp, vp, vp, vp]
    L.mg_anneal_merge_import.argtypes = [vp, vp, vp, u32, C.POINTER(u64)]
    L.mg_anneal_export_slab.argtypes = [vp, u32, i32, vp]
    L.mg_anneal_import_slab.argtypes = [vp, u32, vp, i32]
    L.mg_anneal_oneshot.argtypes = [vp, C.POINTER(AnnealParams), C.POINTER(AnnealRunParams), vp, vp,
                                    C.POINTER(u64), C.POINTER(AnnealStats)]
    L.mg_debug_model_after_prefix.argtypes = [vp, vp, sz, vp]
    L.mg_debug_index.argtypes = [vp, vp, vp]
    L.mg_pool_trim.restype = None
    L.mg_comm_unique_id.argtypes = [vp]
    L.mg_comm_init.argtypes = [vp, i32, i32, vp]
    L.mg_comm_destroy.argtypes = [vp]
    L.mg_comm_destroy.restype = None
    L.mg_comm_rank.argtypes = [vp]
    L.mg_comm_size.argtypes = [vp]
    L.mg_comm_exchange_best.argtypes = [vp, C.POINTER(i32), C.POINTER(u64), C.POINTER(u32)]
    L.mg_comm_temper_exchange.argtypes = [vp, vp, u32, u64]
    L.mg_temper_decide.argtypes = [vp, vp, sz, u32, u64, vp]
    L.mg_comm_merge_regions.argtypes = [vp, u32, vp, vp, u32, C.POINTER(u64)]
    L.mg_comm_stats.argtypes = [vp, C.POINTER(u64), C.POINTER(u64), C.POINTER(u64)]
    L.mg_comm_broadcast_chain.argtypes = [vp, i32, u32, u32]
    L.mg_comm_allgather_u64.argtypes = [vp, u64, vp]
    L.mg_encode_stats.argtypes = [vp, C.POINTER(C.c_double), C.POINTER(u64)]
    L.mg_decode_stream.argtypes = [vp, vp, sz, vp]
    L.mg_decode_stats.argtypes = [vp, C.POINTER(C.c_double), C.POINTER(u64)]
    L.mg_anneal_optimal_init.argtypes = [vp, u32, u32, u32, C.POINTER(u64)]
    L.mg_optimal_stats.argtypes = [vp, C.POINTER(C.c_double), C.POINTER(u64)]
    L.mg_encode_slab_xz.argtypes = [vp, vp, u32, C.POINTER(OutputInterface)]
    L.mg_encode_xz_stats.argtypes = [vp, C.POINTER(C.c_double), C.POINTER(C.c_double), C.POINTER(u32), C.POINTER(u64)]
    _lib = L
    return L


def _check(rc: int) -> None:
    if rc != 0:
        raise MegalaniaError(rc, load_library().mg_last_error().decode(errors="replace"))


def literal_slab(n: int) -> np.ndarray:
    """packet_slab_new: every slot a LITERAL (src/packet_slab.c:30-32)."""
    slab = np.zeros(n, dtype=PACKET_DTYPE)
    slab["type"] = LITERAL
    slab["len"] = 1
    return slab


def as_slab(slab: np.ndarray) -> np.ndarray:
    """A contiguous array in the exact 12-byte LZMAPacket layout (numpy may repack struct dtypes)."""
    if slab.dtype == PACKET_DTYPE and slab.flags["C_CONTIGUOUS"]:
        return slab
    out = np.zeros(slab.shape, dtype=PACKET_DTYPE)
    for name in ("type", "dist", "len"):
        out[name] = slab[name]
    return out


def _slab_ptr(slab: np.ndarray, n: int, count: int = 1):
    if slab.dtype != PACKET_DTYPE or not slab.flags["C_CONTIGUOUS"] or slab.size != n * count:
        raise ValueError(f"slab must be a contiguous PACKET_DTYPE array of {n * count} packets")
    return slab.ctypes.data_as(C.c_void_p)


class Context:
    """One input resident on one GPU, with its bigram index and price tables."""

    def __init__(self, data: bytes, device: int = 0):
        self._lib = load_library()
        self._data = np.ascontiguousarray(np.frombuffer(bytes(data), dtype=np.uint8))
        self.n = int(self._data.size)
        self._h = C.c_void_p()
        self._children = []  # weak references to the Annealers living on this context
        _check(self._lib.mg_ctx_create(self._data.ctypes.data_as(C.c_void_p), self.n, LZMAProperties(0, 0, 0),
                                       device, C.byref(self._h)))

    def close(self) -> None:
        """Destroys the context; chain populations created on it are destroyed first (mg_ctx_destroy
        does the same on the C side), whatever order Python finalises the objects in."""
        if getattr(self, "_h", None):
            for ref in self._children:
                child = ref()
                if child is not None:
                    child.close()
            self._children = []
            self._lib.mg_ctx_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def score_slabs(self, slabs: np.ndarray) -> np.ndarray:
        slabs = as_slab(np.asarray(slabs))
        count = slabs.size // self.n
        out = np.zeros(count, dtype=np.uint64)
        _check(self._lib.mg_score_slabs(self._h, _slab_ptr(slabs.reshape(-1), self.n, count), count,
                                        out.ctypes.data_as(C.c_void_p)))
        return out

    def score_slab(self, slab: np.ndarray) -> int:
        return int(self.score_slabs(slab)[0])

    def find_topk(self, slab: np.ndarray, positions, state_mode: int = 0, k: int = 20):
        pos = np.ascontiguousarray(positions, dtype=np.uint64)
        slab = as_slab(slab)
        pops = np.zeros((pos.size, k), dtype=PACKET_DTYPE)
        prices = np.zeros((pos.size, k), dtype=np.uint32)
        counts = np.zeros(pos.size, dtype=np.int32)
        _check(self._lib.mg_find_topk(self._h, _slab_ptr(slab, self.n), state_mode, pos.ctypes.data_as(C.c_void_p),
                                      pos.size, k, pops.ctypes.data_as(C.c_void_p),
                                      prices.ctypes.data_as(C.c_void_p), counts.ctypes.data_as(C.c_void_p)))
        return pops, prices, counts

    def find_topk_stats(self) -> dict:
        ms, cand = C.c_double(0), C.c_uint64(0)
        _check(self._lib.mg_find_topk_stats(self._h, C.byref(ms), C.byref(cand)))
        return {"kernel_ms": ms.value, "candidates": int(cand.value)}

    def encode_slab(self, slab: np.ndarray) -> bytes:
        """Through the OutputInterface plug-in, exactly as a C host would receive it."""
        chunks: list[bytes] = []

        def _write(_iface, ptr, size):
            chunks.append(C.string_at(ptr, size))
            return True

        iface = OutputInterface(WRITE_FN(_write), None)
        _check(self._lib.mg_encode_slab(self._h, _slab_ptr(slab, self.n), C.byref(iface)))
        return b"".join(chunks)

    def encode_stats(self) -> dict:
        ms, ev = C.c_double(0), C.c_uint64(0)
        _check(self._lib.mg_encode_stats(self._h, C.byref(ms), C.byref(ev)))
        return {"kernel_ms": ms.value, "events": int(ev.value)}

    def encode_slab_buffer(self, slab: np.ndarray) -> bytes:
        cap = self.n * 2 + 8192
        out = np.zeros(cap, dtype=np.uint8)
        got = C.c_size_t(0)
        _check(self._lib.mg_encode_slab_buffer(self._h, _slab_ptr(slab, self.n), out.ctypes.data_as(C.c_void_p), cap,
                                               C.byref(got)))
        return out[:got.value].tobytes()

    def encode_xz(self, slab: np.ndarray, chunk_bytes: int = 0) -> bytes:
        """mg_encode_slab_xz: the slab as one .xz stream (one block, CRC64, LZMA2 chunks of at most chunk_bytes priced
        bytes, 0 = 61440, else 256..61440)."""
        chunks: list[bytes] = []

        def _write(_iface, ptr, size):
            chunks.append(C.string_at(ptr, size))
            return True

        iface = OutputInterface(WRITE_FN(_write), None)
        _check(self._lib.mg_encode_slab_xz(self._h, _slab_ptr(as_slab(slab), self.n), chunk_bytes, C.byref(iface)))
        return b"".join(chunks)

    def encode_xz_stats(self) -> dict:
        """Device time of the last encode_xz's plan walk and chunk kernel, its chunk count and coded events."""
        plan, code, chunks, ev = C.c_double(0), C.c_double(0), C.c_uint32(0), C.c_uint64(0)
        _check(self._lib.mg_encode_xz_stats(self._h, C.byref(plan), C.byref(code), C.byref(chunks), C.byref(ev)))
        return {"plan_ms": plan.value, "code_ms": code.value, "chunks": int(chunks.value), "events": int(ev.value)}

    def decode_stream(self, stream: bytes) -> np.ndarray:
        """An LZMA-alone stream of this input (lc = lp = pb = 0: an earlier output, or liblzma's) -> the slab that
        encodes to it, n packets; slots no packet starts at are LITERAL / 0 / 1.  Raises MegalaniaError with MG_EINVAL
        (header) or MG_ESLAB (a payload that is not this input's)."""
        buf = np.ascontiguousarray(np.frombuffer(bytes(stream), dtype=np.uint8))
        out = np.zeros(self.n, dtype=PACKET_DTYPE)
        _check(self._lib.mg_decode_stream(self._h, buf.ctypes.data_as(C.c_void_p), buf.size,
                                          out.ctypes.data_as(C.c_void_p)))
        return out

    def decode_stats(self) -> dict:
        ms, ev = C.c_double(0), C.c_uint64(0)
        _check(self._lib.mg_decode_stats(self._h, C.byref(ms), C.byref(ev)))
        return {"kernel_ms": ms.value, "events": int(ev.value)}

    def optimal_stats(self) -> dict:
        """Device time of the last Annealer.optimal_init's match-list and parse kernels, and the nodes it relaxed."""
        ms, nodes = C.c_double(0), C.c_uint64(0)
        _check(self._lib.mg_optimal_stats(self._h, C.byref(ms), C.byref(nodes)))
        return {"kernel_ms": ms.value, "nodes": int(nodes.value)}

    def model_after_prefix(self, slab: np.ndarray, stop: int):
        out = np.zeros(1, dtype=MODEL_DTYPE)
        _check(self._lib.mg_debug_model_after_prefix(self._h, _slab_ptr(slab, self.n), stop,
                                                     out.ctypes.data_as(C.c_void_p)))
        return out[0]

    # ---- several GPUs (NCCL behind the C ABI) ----
    @staticmethod
    def comm_unique_id() -> bytes:
        buf = C.create_string_buffer(128)
        _check(load_library().mg_comm_unique_id(buf))
        return buf.raw

    def comm_init(self, rank: int, nranks: int, unique_id: bytes) -> None:
        if len(unique_id) != 128:
            raise ValueError("an NCCL unique id is 128 bytes")
        _check(self._lib.mg_comm_init(self._h, rank, nranks, C.c_char_p(unique_id)))

    def comm_allgather(self, value: int) -> np.ndarray:
        size = int(self._lib.mg_comm_size(self._h))
        out = np.zeros(size, dtype=np.uint64)
        _check(self._lib.mg_comm_allgather_u64(self._h, int(value), out.ctypes.data_as(C.c_void_p)))
        return out

    def comm_stats(self) -> dict:
        a, b, c = C.c_uint64(0), C.c_uint64(0), C.c_uint64(0)
        _check(self._lib.mg_comm_stats(self._h, C.byref(a), C.byref(b), C.byref(c)))
        return {"exchanges": int(a.value), "installs_by_copy": int(b.value), "installs_by_rescore": int(c.value)}

    def set_finder_limits(self, window: int = 0, max_occurrences: int = 0) -> None:
        """0, 0 = the reference's unbounded enumeration (the default)."""
        _check(self._lib.mg_ctx_set_finder_limits(self._h, window, max_occurrences))

    def full_wave(self) -> int:
        """Chains that fill the device exactly once (SMs x chains per SM)."""
        return int(self._lib.mg_ctx_full_wave(self._h))

    def sm_clock_khz(self) -> int:
        """The device's SM clock in kHz (0 if unknown): step lengths in milliseconds x this = cycle_budget."""
        return int(self._lib.mg_ctx_sm_clock_khz(self._h))

    def bigram_index(self):
        """(occ_start[65537], occ[n-1]): the device-built index of src/substring_enumerator.c:26-47."""
        start = np.zeros(65537, dtype=np.uint32)
        occ = np.zeros(max(1, self.n - 1), dtype=np.uint32)
        _check(self._lib.mg_debug_index(self._h, start.ctypes.data_as(C.c_void_p), occ.ctypes.data_as(C.c_void_p)))
        return start, occ[:max(0, self.n - 1)]

    def chain_bytes(self, **params) -> int:
        p = AnnealParams(**params)
        return int(self._lib.mg_anneal_chain_bytes(self._h, C.byref(p)))


class Annealer:
    """A population of annealing chains (one warp each) over one Context."""

    def __init__(self, ctx: Context, chains: int, *, top_k: int = 20, checkpoint_stride: int = 0,
                 edit_log_capacity: int = 0, track_best: bool = True, trace_capacity: int = 0, seed: int = 1673551):
        self.ctx = ctx
        self._lib = ctx._lib
        self.chains = chains
        self.params = AnnealParams(chains, top_k, checkpoint_stride, edit_log_capacity, int(track_best),
                                   trace_capacity, seed)
        self._h = C.c_void_p()
        _check(self._lib.mg_anneal_create(ctx._h, C.byref(self.params), C.byref(self._h)))
        import weakref
        ctx._children.append(weakref.ref(self))

    def close(self) -> None:
        if getattr(self, "_h", None):
            self._lib.mg_anneal_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def set_slab(self, slab: np.ndarray | None = None, first: int = 0, count: int | None = None,
                 adopt_cost: bool | None = None, reset_best: bool = True) -> None:
        if count is None:
            count = self.chains - first
        if adopt_cost is None:
            adopt_cost = slab is not None
        ptr = _slab_ptr(slab, self.ctx.n) if slab is not None else None
        _check(self._lib.mg_anneal_set_slab(self._h, first, count, ptr, int(adopt_cost), int(reset_best)))

    def run(self, evals: int, *, schedule: int = SCHEDULE_REFERENCE, step: int = 0, num_iters: int = 0,
            first_eval: int = 0, max_attempts: int = 0, temperatures=None, packet_budget: int = 0,
            early_exit: bool = True, suspend: bool = False, cycle_budget: int = 0, regions=None) -> dict:
        temps = None
        tptr = None
        if temperatures is not None:
            temps = np.ascontiguousarray(temperatures, dtype=np.float32)
            if temps.size != self.chains:
                raise ValueError("one temperature per chain")
            tptr = temps.ctypes.data_as(C.POINTER(C.c_float))
        rptr = None
        if regions is not None:
            regs = np.ascontiguousarray(regions, dtype=np.uint32)
            if regs.shape != (self.chains, 2):
                raise ValueError("regions must be a [chains][2] array of byte ranges")
            rptr = regs.ctypes.data_as(C.POINTER(C.c_uint32))
        rp = AnnealRunParams(evals, max_attempts, schedule, step, num_iters, first_eval, tptr, packet_budget,
                             0 if early_exit else 1, int(suspend), cycle_budget, rptr)
        st = AnnealStats()
        _check(self._lib.mg_anneal_run(self._h, C.byref(rp), C.byref(st)))
        return st.as_dict()

    def costs(self):
        cur = np.zeros(self.chains, dtype=np.uint64)
        best = np.zeros(self.chains, dtype=np.uint64)
        _check(self._lib.mg_anneal_costs(self._h, cur.ctypes.data_as(C.c_void_p), best.ctypes.data_as(C.c_void_p)))
        return cur, best

    def get_slab(self, chain: int, best: bool = False) -> np.ndarray:
        out = np.zeros(self.ctx.n, dtype=PACKET_DTYPE)
        _check(self._lib.mg_anneal_get_slab(self._h, chain, int(best), out.ctypes.data_as(C.c_void_p)))
        return out

    def trace(self, chain: int) -> np.ndarray:
        cap = self.params.trace_capacity
        out = np.zeros(cap, dtype=TRACE_DTYPE)
        count = C.c_size_t(0)
        _check(self._lib.mg_anneal_get_trace(self._h, chain, out.ctypes.data_as(C.c_void_p), cap, C.byref(count)))
        return out[:min(cap, count.value)]

    def swap_chains(self, a: int, b: int) -> None:
        _check(self._lib.mg_anneal_swap_chains(self._h, a, b))

    def device_slab(self, chain: int, best: bool = False):
        ptr, size = C.c_void_p(), C.c_size_t()
        _check(self._lib.mg_anneal_device_slab(self._h, chain, int(best), C.byref(ptr), C.byref(size)))
        return ptr.value, size.value

    def export_slab(self, chain: int, best: bool, device_ptr: int) -> None:
        """Packed slab -> caller device buffer (n*8 bytes), e.g. a torch tensor's data_ptr()."""
        _check(self._lib.mg_anneal_export_slab(self._h, chain, int(best), C.c_void_p(device_ptr)))

    def import_slab(self, chain: int, device_ptr: int, adopt_cost: bool = True) -> None:
        _check(self._lib.mg_anneal_import_slab(self._h, chain, C.c_void_p(device_ptr), int(adopt_cost)))

    def merge_regions(self, bounds, owners, dst_chain: int = 0) -> int:
        """Region r = [bounds[r], bounds[r+1]) from chain owners[r] -> chain dst_chain, repaired and priced."""
        b = np.ascontiguousarray(bounds, dtype=np.uint32)
        o = np.ascontiguousarray(owners, dtype=np.uint32)
        if b.size != o.size + 1:
            raise ValueError("bounds must hold one more entry than owners")
        cost = C.c_uint64(0)
        _check(self._lib.mg_anneal_merge_regions(self._h, o.size, b.ctypes.data_as(C.c_void_p), o.ctypes.data_as(C.c_void_p),
                                                 dst_chain, C.byref(cost)))
        return int(cost.value)

    def merge_export(self, bounds, owners, dev_slab_ptr: int, dev_abs_ptr: int) -> None:
        """This process's part of a multi-GPU merge into two device buffers (n*8 and n*4 bytes); owners[r] = NO_OWNER
        for regions that live elsewhere."""
        b = np.ascontiguousarray(bounds, dtype=np.uint32)
        o = np.ascontiguousarray(owners, dtype=np.uint32)
        if b.size != o.size + 1:
            raise ValueError("bounds must hold one more entry than owners")
        _check(self._lib.mg_anneal_merge_export(self._h, o.size, b.ctypes.data_as(C.c_void_p), o.ctypes.data_as(C.c_void_p),
                                                C.c_void_p(dev_slab_ptr), C.c_void_p(dev_abs_ptr)))

    def merge_import(self, dev_slab_ptr: int, dev_abs_ptr: int, dst_chain: int = 0) -> int:
        cost = C.c_uint64(0)
        _check(self._lib.mg_anneal_merge_import(self._h, C.c_void_p(dev_slab_ptr), C.c_void_p(dev_abs_ptr), dst_chain,
                                                C.byref(cost)))
        return int(cost.value)

    def comm_exchange_best(self):
        """Collective: (winner rank or -1, global best cost, this rank's chain holding the slab); see mg_comm_exchange_best."""
        w, c, ch = C.c_int(-1), C.c_uint64(0), C.c_uint32(0)
        _check(self._lib.mg_comm_exchange_best(self._h, C.byref(w), C.byref(c), C.byref(ch)))
        return int(w.value), int(c.value), int(ch.value)

    def comm_broadcast_chain(self, root: int, src_chain: int, dst_chain: int) -> None:
        _check(self._lib.mg_comm_broadcast_chain(self._h, root, src_chain, dst_chain))

    def comm_temper_exchange(self, temps: np.ndarray, round_index: int, seed: int = 0) -> np.ndarray:
        """Collective: one replica-exchange round over the replicas of all ranks; returns this rank's new temperatures."""
        t = np.ascontiguousarray(temps, dtype=np.float32).copy()
        if t.size != self.chains:
            raise ValueError("one temperature per chain")
        _check(self._lib.mg_comm_temper_exchange(self._h, t.ctypes.data_as(C.c_void_p), round_index, seed))
        return t

    def comm_merge_regions(self, bounds, owners, dst_chain: int = 0) -> int:
        b = np.ascontiguousarray(bounds, dtype=np.uint32)
        o = np.ascontiguousarray(owners, dtype=np.uint32)
        cost = C.c_uint64(0)
        _check(self._lib.mg_comm_merge_regions(self._h, o.size, b.ctypes.data_as(C.c_void_p), o.ctypes.data_as(C.c_void_p),
                                               dst_chain, C.byref(cost)))
        return int(cost.value)

    def broadcast_chain(self, src_chain: int) -> None:
        _check(self._lib.mg_anneal_broadcast_chain(self._h, src_chain))

    def greedy_init(self, nregions: int = 1, dst_chain: int = 0) -> int:
        """mg_anneal_greedy_init: greedy parse of `nregions` byte regions side by side, stitched, repaired and priced
        into chain dst_chain; returns its cost.  One region, no finder limits = the oracle's greedy slab."""
        cost = C.c_uint64(0)
        _check(self._lib.mg_anneal_greedy_init(self._h, nregions, dst_chain, C.byref(cost)))
        return int(cost.value)

    def optimal_init(self, nregions: int = 1, max_occ: int = 0, dst_chain: int = 0) -> int:
        """mg_anneal_optimal_init: shortest-path parse of `nregions` byte regions side by side (match lists of at most
        max_occ occurrences, 0 = 64), stitched, repaired and priced into chain dst_chain; returns its cost.  One
        region = the CPU parse of the tests packet for packet."""
        cost = C.c_uint64(0)
        _check(self._lib.mg_anneal_optimal_init(self._h, nregions, max_occ, dst_chain, C.byref(cost)))
        return int(cost.value)

    def refresh_chain(self, chain: int, adopt_cost: bool = True) -> None:
        _check(self._lib.mg_anneal_refresh_chain(self._h, chain, int(adopt_cost)))


def temper_decide(costs, temps, round_index: int, seed: int = 0) -> np.ndarray:
    """mg_temper_decide: the replica-exchange swap rule (host only, runs without a GPU)."""
    c = np.ascontiguousarray(costs, dtype=np.uint64)
    t = np.ascontiguousarray(temps, dtype=np.float32)
    out = np.zeros_like(t)
    _check(load_library().mg_temper_decide(c.ctypes.data_as(C.c_void_p), t.ctypes.data_as(C.c_void_p), c.size, round_index, seed,
                                           out.ctypes.data_as(C.c_void_p)))
    return out


def anneal_oneshot(ctx: Context, *, chains: int, evals: int, init: np.ndarray | None = None, seed: int = 1673551,
                   top_k: int = 20, schedule: int = SCHEDULE_REFERENCE, step: int = 0, num_iters: int = 0,
                   packet_budget: int = 0, cycle_budget: int = 0, suspend: bool = False):
    """Host buffers in, host buffers out: the call the end-to-end benchmark times."""
    lib = ctx._lib
    p = AnnealParams(chains, top_k, 0, 0, 1, 0, seed)
    rp = AnnealRunParams(evals, 0, schedule, step, num_iters, 0, None, packet_budget, 0, int(suspend), cycle_budget, None)
    st = AnnealStats()
    best = np.zeros(ctx.n, dtype=PACKET_DTYPE)
    cost = C.c_uint64(0)
    iptr = _slab_ptr(init, ctx.n) if init is not None else None
    _check(lib.mg_anneal_oneshot(ctx._h, C.byref(p), C.byref(rp), iptr, best.ctypes.data_as(C.c_void_p),
                                 C.byref(cost), C.byref(st)))
    return best, int(cost.value), st.as_dict()

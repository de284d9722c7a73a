#!/usr/bin/env python
"""Benchmark of the annealing hot path (BASELINE.json: neighbour cost evals/sec).

    python bench.py [--gpus N] [--steps K] [--warmup W]            # the CUDA path
    python bench.py --impl reference [--gpus N] --steps K --warmup W  # the reference's CPU path
    python bench.py --steps K --warmup W --dump-outputs DIR          # also write the last step's results

A "step" = every chain runs successful neighbour proposals (mutate, repair, full cost, accept/undo)
until it has priced `--packet-budget` packets (a proposal cut by the budget is suspended at a checkpoint
and carried on by the next step), on the 1 MiB synthetic mixed text/binary input of BASELINE.json
configs[1], all chains starting from the all-literal slab like the reference does.  The budget is work,
not time, so the same arguments compute the same results on every run (see STEP_PACKETS for its cost).
`--packet-budget 0` ends steps on `--step-ms` of SM clocks instead, which keeps every warp busy to the
end of the step but makes how far the chains get depend on the clock.  `value` counts successful
evaluations of ALL chains on ALL GPUs per second of device time (CUDA events on the library's
launch stream, max over ranks).  `e2e` is the same metric through the one-shot host call with
host buffers in and out (input upload, index build, chain allocation, best slab read-back).

Under torchrun (N > 1) the timed arm is BASELINE.json configs[3]: the replicas of all ranks form one
temperature ladder (parallel tempering); every rank owns its own chains (weak scaling, no collective
inside a step); after EVERY step the ranks all-gather (cost, temperature) of every replica and swap
temperatures (mg_comm_temper_exchange), and every --exchange-every steps the cheapest best slab is
broadcast with its checkpoints and installed by copy (mg_comm_exchange_best).  The collectives are the
library's own NCCL calls behind the C ABI; torch.distributed only carries the rendezvous (NCCL id,
barriers, the final reductions of the timing numbers).

Rank 0 at N = 1 also reports, outside the timed region: `size` (the second half of the metric: .lzma bytes
after a fixed wall budget through the drop-in CLI, beside the reference harness on one core at the same
budget and xz -9e), `config3` (4 KiB exec-like input, thousands of chains) and `encode` (range-coder pass).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True  # the benchmark leaves the tree as it found it (it may be read-only)

from tools import corpus  # noqa: E402

METRIC = "neighbour_cost_evals_per_sec"
UNIT = "evals/s"
WORKLOAD = "1 MiB synthetic mixed text/binary (tools/corpus.py mixed, seed 7), all-literal start, reference schedule step 0"
ISSUE_CEILING_BITS_PER_S = 148 * 1.965e9 * 32 / 3  # SURVEY.md §8(d): shared-memory bank ceiling for the scorer
# packets each chain prices per step: the work a 1000 ms SM-clock step does from the all-literal start (5 timed steps
# after 3 warm-up ones: 828 323 evaluations against 823 389), so that the timed steps see slabs of the same age.
# Measured on a B200 at 1000 W and 1965 MHz: 1.26 s per step, 132 k evaluations/s against 164 k for --packet-budget 0,
# because chains given equal work finish unevenly (warp busy fraction 0.79 against 1.00)
STEP_PACKETS = 23_000_000


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            return json.load(f), "measured"
    return {"hbm_gbs": 6650.0, "sm_max_mhz": 1965.0}, "fallback"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled while the timed region runs."""

    QUERY = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
             "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, device: int):
        self.device = device
        self.proc = None
        self.lines: list[str] = []
        self.first = 0

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.device}", f"--query-gpu={self.QUERY}",
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except OSError:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def mark(self):
        """Samples read so far belong to the warm-up: the figures come from what follows."""
        self.first = len(self.lines)

    def stop(self) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, smax, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in self.lines[self.first:]:
            f = [x.strip() for x in line.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                smax.append(float(f[2]))
            except ValueError:
                continue
            for name, val in zip(names, f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(smax)), "reasons": sorted(reasons),
                "samples": len(sm)}


def dist_env():
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    return rank, world, local


# ------------------------------------------------------------------------------------------------
# CPU legs (the only places this file touches oracle/)
# ------------------------------------------------------------------------------------------------
_CORPUS_CACHE: dict = {}


def _corpus(kind: str, n: int) -> bytes:
    if (kind, n) not in _CORPUS_CACHE:
        _CORPUS_CACHE[(kind, n)] = corpus.make(kind, n)
    return _CORPUS_CACHE[(kind, n)]


def _cpu_worker(args):
    """One host core: the reference's own loop (src/main.c:78-102) for `evals` evaluations."""
    kind, n, evals, seed, which = args
    from oracle import oracle_lib as ol
    data = _corpus(kind, n)
    slab = ol.literal_slab(n)
    best = slab.copy()
    if which == "reference":
        lib = ol.Ref()
        t0 = time.perf_counter()
        lib.anneal_epoch(data, slab, best, 0, 0, seed=seed, evals=evals)
        dt = time.perf_counter() - t0
    else:
        lib = ol.Port()
        t0 = time.perf_counter()
        lib.anneal_epoch(data, slab, best, 0, 0, rng_mode=0, seed=seed, evals=evals)
        dt = time.perf_counter() - t0
    return evals, dt


def cpu_kind() -> str:
    from oracle import oracle_lib as ol
    ol.build()
    return "reference" if os.path.exists(ol.REF_SO) else "port"


def cpu_baseline(n: int, evals: int) -> dict:
    """Single-threaded reference on one host core, bounded sample (reported, not the target)."""
    kind = cpu_kind()
    done, dt = _cpu_worker(("mixed", n, evals, 1673551, kind))
    return {"value": done / dt, "unit": UNIT, "cores": 1, "kind": kind,
            "sample": f"first {done} successful evaluations from the all-literal slab, seed 1673551, {dt:.1f} s"}


def run_reference(args) -> None:
    """--impl reference: the reference's CPU implementation on all host cores it can use
    (it is single-threaded, so one independent annealing process per core, different seeds)."""
    rank, world, _ = dist_env()
    if rank != 0:
        return
    import multiprocessing as mp
    n = args.size
    kind = cpu_kind()
    cores = max(1, min(os.cpu_count() or 1, args.cpu_procs))
    evals = args.cpu_evals
    _corpus("mixed", n)  # generated once, inherited by the forked workers
    ctx = mp.get_context("fork")
    total_evals, total_time = 0, 0.0
    with ctx.Pool(cores) as pool:
        for step in range(args.warmup + args.steps):
            t0 = time.perf_counter()
            res = pool.map(_cpu_worker, [("mixed", n, evals, 1673551 + step * cores + w, kind) for w in range(cores)])
            dt = time.perf_counter() - t0
            if step >= args.warmup:
                total_evals += sum(r[0] for r in res)
                total_time += dt
    value = total_evals / total_time
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * total_time / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u16/u64 integer",
            "data": "synthetic",
            "config": {"workload": WORKLOAD, "input_bytes": n, "chains": cores, "evals_per_chain_per_step": evals},
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": kind,
                             "sample": f"{cores} independent single-threaded annealing processes x {evals} successful "
                                       f"evaluations per step from the all-literal slab"},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------
# the second half of the metric: .lzma bytes at equal wall time (rank 0, N = 1, outside the timed region)
# ------------------------------------------------------------------------------------------------
def _reference_size(kind: str, n: int, wall_s: float) -> dict:
    """The reference's own loop (src/main.c:78-102, step 0, from the all-literal slab) on ONE host core for
    `wall_s` seconds, then its range coder: bytes of the stream it would write."""
    from oracle import oracle_lib as ol
    which = cpu_kind()
    lib = ol.Ref() if which == "reference" else ol.Port()
    data = _corpus(kind, n)
    slab = ol.literal_slab(n)
    best = slab.copy()
    kw = {} if which == "reference" else {"rng_mode": 0}
    t0 = time.perf_counter()
    probe = 4
    _, bc, cc, *_ = lib.anneal_epoch(data, slab, best, 0, 0, seed=1673551, evals=probe, **kw)
    dt = max(1e-3, time.perf_counter() - t0)
    evals = probe
    rate = probe / dt
    remaining = wall_s - dt
    if remaining > 0:
        more = max(1, int(rate * remaining * 0.9))
        _, bc, cc, *_ = lib.anneal_epoch(data, slab, best, bc, cc, reseed=0, evals=more, **kw)
        evals += more
    used = time.perf_counter() - t0
    stream = lib.encode_slab(data, best if bc else slab)
    import lzma
    return {"bytes": len(stream), "evals": evals, "wall_s": used, "cores": 1, "kind": which,
            "round_trip": lzma.decompress(stream, format=lzma.FORMAT_ALONE) == data}


def size_leg(mg, wave: int, budget_s: float, device: int) -> list:
    import lzma
    import tempfile
    from megalania_b200 import build
    cli = build.CLI  # as build() left it: the benchmark compiles nothing into the tree
    out = []
    for name, kind, n, chains in (("config 1: 64 KiB synthetic English-like text", "text", 65536, wave),
                                  ("config 2: 1 MiB synthetic mixed text/binary", "mixed", 1 << 20, wave),
                                  ("config 3: 4 KiB synthetic executable-like binary", "binary", 4096, max(4096, wave))):
        data = _corpus(kind, n)
        with tempfile.NamedTemporaryFile(suffix=".bin") as f:
            f.write(data)
            f.flush()
            cmd = [cli, "--chains", str(chains), "--time", str(int(budget_s)), "--round-ms", "250", "--device", str(device)]
            if n >= (1 << 20):
                cmd += ["--greedy", "1024"]  # a greedy parse of 1024 regions as the starting slab (mg_anneal_greedy_init)
            cmd.append(f.name)
            t0 = time.perf_counter()
            r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.PIPE)
            wall = time.perf_counter() - t0
        rec = {"config": name, "input_bytes": n, "chains": chains, "wall_s": wall,
               "command": " ".join(["megalania"] + cmd[1:-1] + ["<file>"]) + "  (drop-in C CLI: cooperative regions, final "
                          "range-coder pass on the device)"}
        if r.returncode != 0:
            rec["error"] = r.stderr.decode(errors="replace")[-300:]
            out.append(rec)
            continue
        rec["bytes"] = len(r.stdout)
        try:
            rec["round_trip"] = lzma.decompress(r.stdout, format=lzma.FORMAT_ALONE) == data
        except lzma.LZMAError:
            rec["round_trip"] = False
        rec["xz_9e_bytes"] = len(lzma.compress(data, format=lzma.FORMAT_ALONE, preset=9 | lzma.PRESET_EXTREME))
        rec["reference_same_wall"] = _reference_size(kind, n, wall)
        rec["no_larger_than_reference"] = rec["bytes"] <= rec["reference_same_wall"]["bytes"]
        rec["smaller_than_xz_9e"] = rec["bytes"] < rec["xz_9e_bytes"]
        out.append(rec)
    return out


def config3_leg(mg, wave: int, seconds: float, sm_khz: int, device: int) -> dict:
    """BASELINE configs[2]: 4 KiB executable-like binary, thousands of chains, all-literal start."""
    n = 4096
    data = _corpus("binary", n)
    chains = max(4096, wave)
    chains = (chains + wave - 1) // wave * wave
    ctx = mg.Context(data, device=device)
    an = mg.Annealer(ctx, chains, seed=7)
    an.set_slab(None)
    budget = int(250 * sm_khz)
    for _ in range(2):
        an.run(1_000_000, first_eval=mg.CONTINUE_EVALS, cycle_budget=budget, suspend=True)
    evals, ms, steps = 0, 0.0, 0
    while ms < seconds * 1e3:
        st = an.run(1_000_000, first_eval=mg.CONTINUE_EVALS, cycle_budget=budget, suspend=True)
        evals += st["evals"]
        ms += st["kernel_ms"]
        steps += 1
    cur, best = an.costs()
    an.close()
    ctx.close()
    return {"workload": "4 KiB synthetic executable-like binary (tools/corpus.py binary, seed 7), all-literal start, reference schedule",
            "chains": chains, "evals_per_s": evals / (ms / 1e3), "evals_per_chain": evals / chains, "device_s": ms / 1e3,
            "steps": steps, "best_bytes_estimate": 18 + int(best[best > 0].min()) / 16384.0}


def encode_leg(mg, data: bytes, best_slab, device: int) -> dict:
    """The final range-coder pass (src/main.c:110-119) on the device beside the reference's CPU pass."""
    from oracle import oracle_lib as ol
    n = len(data)
    ctx = mg.Context(data, device=device)
    cpu = ol.Ref() if cpu_kind() == "reference" else ol.Port()
    out = {}
    for name, slab in (("all_literal", mg.literal_slab(n)), ("annealed_best", best_slab)):
        if slab is None:
            continue
        ctx.encode_slab_buffer(slab)
        stream = ctx.encode_slab_buffer(slab)
        st = ctx.encode_stats()
        t0 = time.perf_counter()
        want = cpu.encode_slab(data, slab)
        cpu_ms = 1e3 * (time.perf_counter() - t0)
        out[name] = {"bytes": len(stream), "events": st["events"], "device_ms": st["kernel_ms"], "cpu_ms": cpu_ms,
                     "identical_to_cpu": stream == want}
    ctx.close()
    return out


DUMP_SEED, DUMP_CHAINS, DUMP_POSITIONS = 2024, 8, 65536


def dump_outputs(an, out_dir: str, suffix: str = "") -> None:
    """What the timed path leaves its caller after the last timed step, as DIR/<name><suffix>.npy: every chain's
    current and best cost (float64, exact below 2^53) and, for a fixed seeded sample of chains and positions, the
    (type, dist, len) of those slots of their current and best slabs (float32, exact: dist < 2^24).  About 12 MB
    at the default size."""
    os.makedirs(out_dir, exist_ok=True)
    cur, best = an.costs()
    rng = np.random.default_rng(DUMP_SEED)
    chains = np.sort(rng.choice(an.chains, size=min(DUMP_CHAINS, an.chains), replace=False))
    pos = np.sort(rng.choice(an.ctx.n, size=min(DUMP_POSITIONS, an.ctx.n), replace=False))
    arrays = {"cur_cost": cur.astype(np.float64), "best_cost": best.astype(np.float64),
              "sample_chains": chains.astype(np.float64), "sample_positions": pos.astype(np.float64)}
    for name, is_best in (("cur_slab_sample", False), ("best_slab_sample", True)):
        slots = np.stack([an.get_slab(int(c), best=is_best)[pos] for c in chains])
        arrays[name] = np.stack([slots["type"], slots["dist"], slots["len"]], axis=-1).astype(np.float32)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, f"{name}{suffix}.npy"), a)


# ------------------------------------------------------------------------------------------------
# the CUDA arm
# ------------------------------------------------------------------------------------------------
def run_cuda(args) -> None:
    # stdout carries exactly one JSON line: anything libraries print on the way (NCCL's version
    # banner under NCCL_DEBUG) goes to stderr
    sys.stdout.flush()
    json_fd = os.dup(1)
    os.dup2(2, 1)
    import torch
    import megalania_b200 as mg

    rank, world, local = dist_env()
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the hot path has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    dist = None
    if world > 1:
        import torch.distributed as dist_mod
        dist = dist_mod
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    mg.load_library(build_if_missing=False)
    n = args.size
    data = _corpus("mixed", n)
    ctx = mg.Context(data, device=local)
    props = torch.cuda.get_device_properties(local)
    chains = args.chains or (props.multi_processor_count * args.warps_per_sm if args.warps_per_sm else ctx.full_wave())
    chain_bytes = ctx.chain_bytes(chains=chains, track_best=1)
    free, _ = torch.cuda.mem_get_info(local)
    wanted = chains
    while chains > 8 and chains * chain_bytes > 0.85 * free:
        chains //= 2
    if args.dump_outputs and chains != wanted:
        raise SystemExit(f"bench.py: only {chains} of {wanted} chains fit in free device memory; a dump of the smaller "
                         "population could not be compared with other runs")
    an = mg.Annealer(ctx, chains, seed=args.seed + 1000003 * rank)
    an.set_slab(None)

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    temps = None
    if dist is not None:
        # the library's own communicator (NCCL behind the C ABI); torch.distributed only carries the id
        box = [mg.Context.comm_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(box, src=0)
        ctx.comm_init(rank, world, box[0])
        from megalania_b200.tempering import temperature_ladder
        ladder = temperature_ladder(world * chains, args.t_min, args.t_max)
        temps = ladder[rank::world].copy()  # every rank holds rungs from the whole ladder

    step_no = [0]
    exchange_ms = [0.0]

    # SM clocks per millisecond: the library's own figure (cudaDevAttrClockRate), else torch's, else the measured peak file
    sm_khz = int(ctx.sm_clock_khz() or getattr(props, "clock_rate", 0) or peaks()[0].get("sm_max_mhz", 1965.0) * 1000)
    cycle_budget = 0 if args.packet_budget else int(args.step_ms * sm_khz)

    def step(first_eval):
        nonlocal temps
        if dist is None:
            st = an.run(args.evals, schedule=mg.SCHEDULE_REFERENCE, step=0, first_eval=mg.CONTINUE_EVALS,
                        packet_budget=args.packet_budget, cycle_budget=cycle_budget, suspend=True)
        else:
            st = an.run(args.evals, schedule=mg.SCHEDULE_TEMPERATURE, temperatures=temps, first_eval=mg.CONTINUE_EVALS,
                        packet_budget=args.packet_budget, cycle_budget=cycle_budget, suspend=True)
            t0 = time.perf_counter()
            temps = an.comm_temper_exchange(temps, step_no[0], seed=args.seed)       # every step
            if (step_no[0] + 1) % args.exchange_every == 0:
                an.comm_exchange_best()                                              # best-slab broadcast
            exchange_ms[0] += 1e3 * (time.perf_counter() - t0)
        step_no[0] += 1
        return st

    first_eval = 0
    sampler = ClockSampler(local)
    for w in range(args.warmup):
        if w == args.warmup - 1:
            # nvidia-smi holds the driver up for some tens of milliseconds while it starts (a 3-step run showed
            # 31 ms per step of wall clock the device never saw): it starts under the last warm-up step and only
            # the samples of the timed region count (mark())
            sampler.start()
        step(first_eval)
        first_eval += args.evals
    if args.warmup == 0:
        sampler.start()
    barrier()
    exchange_ms[0] = 0.0
    sampler.mark()
    t0 = time.perf_counter()
    agg = None
    per_launch_ms = []
    for _ in range(args.steps):
        st = step(first_eval)
        first_eval += args.evals
        per_launch_ms.append(st["kernel_ms"])
        if agg is None:
            agg = dict(st)
        else:
            for k, v in st.items():
                agg[k] += v
    barrier()
    wall = time.perf_counter() - t0
    clocks = sampler.stop()
    device_s = agg["kernel_ms"] / 1e3
    if args.dump_outputs:
        dump_outputs(an, args.dump_outputs, f"_rank{rank}" if world > 1 else "")

    # max over ranks (device time), sum over ranks (work)
    if dist is not None:
        t = torch.tensor([device_s, wall], dtype=torch.float64, device=f"cuda:{local}")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        device_s, wall = float(t[0]), float(t[1])
        w = torch.tensor([agg["evals"], agg["bits_scored"], agg["packets_scored"], agg["launches"]], dtype=torch.int64,
                         device=f"cuda:{local}")
        dist.all_reduce(w, op=dist.ReduceOp.SUM)
        total_evals, total_bits, total_packets, launches = (int(x) for x in w)
    else:
        total_evals, total_bits, total_packets, launches = agg["evals"], agg["bits_scored"], agg["packets_scored"], agg["launches"]
    # `value` uses the wall clock between the two barrier+synchronize brackets (launches, the
    # between-step exchange and all host work included); the CUDA-event time of the kernels alone
    # is reported beside it and feeds the roofline.
    value = total_evals / wall

    # ---- roofline of the dominant kernel (anneal_kernel), this rank ---------------------------
    pk, pk_src = peaks()
    # 9 B per byte walked (slab slot + data byte) + 3968 B per checkpoint moved + 16 B per edit, counted by the kernel.
    # The literal queues (32 B per literal priced from them) are read from L2, where the 48 B/byte table lives: they
    # show up in ncu's DRAM bytes only as far as they miss (traffic / algorithmic, below)
    alg_bytes = agg["slab_bytes_read"] + agg["checkpoint_bytes"] + 16 * agg["edits"]
    achieved = alg_bytes / (agg["kernel_ms"] / 1e3) / 1e9
    # DRAM traffic: ncu (dram__bytes_read + write of one captured launch of this kernel on this workload,
    # profiles/r02_final_traffic.json) as a ratio to the algorithmic bytes of that launch, SCALED to this run's
    # (not measured in this run: a number taken under a profiler is never a bench value)
    traffic, traffic_src = None, None
    tpath = os.path.join(ROOT, "profiles", "r02_final_traffic.json")
    if not os.path.exists(tpath):
        tpath = os.path.join(ROOT, "profiles", "r01_final_traffic.json")
    if os.path.exists(tpath):
        with open(tpath) as f:
            tj = json.load(f)
        traffic = tj["dram_over_algorithmic"] * alg_bytes / max(1, agg["launches"])
        traffic_src = f"ncu dram bytes / algorithmic bytes = {tj['dram_over_algorithmic']} on a {tj['launch_ms']} ms launch of the same workload, scaled to this launch"
    roofline = {"bound": "hbm", "achieved": achieved, "peak": pk["hbm_gbs"], "unit": "GB/s",
                "frac": achieved / pk["hbm_gbs"], "traffic": traffic, "traffic_source": traffic_src,
                "peak_source": pk_src, "kernel": "mg::anneal_kernel",
                "algorithmic_bytes_per_launch": alg_bytes / max(1, agg["launches"]),
                "avg_launch_ms": float(np.mean(per_launch_ms)),
                "note": "the scorer is issue/shared-memory bound, not HBM bound: see roofline_issue"}
    bits_per_s = agg["bits_scored"] / (agg["kernel_ms"] / 1e3)
    roofline_issue = {"bound": "shared-memory banks / issue slots", "achieved": bits_per_s,
                      "peak": ISSUE_CEILING_BITS_PER_S, "unit": "modelled bits/s", "frac": bits_per_s / ISSUE_CEILING_BITS_PER_S,
                      "bits_per_eval": agg["bits_scored"] / max(1, agg["attempts"]),
                      "note": "peak = 148 SMs x f_SM x 32 banks / 3 accesses per modelled bit (SURVEY 8d: every lane of every "
                              "shared-memory instruction useful); the per-lane literal queues issue ~2.1 shared-memory wavefronts per "
                              "9-bit literal (16 rounds x 3 accesses + conflicts per 32 literals: the hottest slots take one two-step "
                              "table lookup per two literals, the other lanes wait for them), LSU data pipe 86 % busy in the steady state (profiles/r02_parked_steady_anneal_kernel_ncu.txt, DESIGN.md 5); the match finder is 24 % of the warp time"}

    ctx_comm_stats = ctx.comm_stats() if dist is not None else None
    best_slab = None
    if rank == 0 and world == 1 and not args.no_size:
        _, bestc = an.costs()
        if (bestc > 0).any():
            best_slab = an.get_slab(int(np.where(bestc > 0, bestc, np.iinfo(np.uint64).max).argmin()), best=True)

    # ---- end to end through the one-shot host call (host buffers in and out) -------------------
    e2e = None
    if not args.no_e2e:
        an.close()
        ctx.close()
        e2e_chains = chains
        barrier()
        t0 = time.perf_counter()
        e2e_evals = 0
        for s in range(args.e2e_steps):
            c2 = mg.Context(data, device=local)                   # H2D of the input + index build
            best, cost, st2 = mg.anneal_oneshot(c2, chains=e2e_chains, evals=args.evals, seed=args.seed + s,
                                                packet_budget=args.packet_budget * args.e2e_step_factor,
                                                cycle_budget=cycle_budget * args.e2e_step_factor, suspend=True)
            e2e_evals += st2["evals"]                              # best slab + cost came back to the host
            c2.close()
        barrier()
        e2e_s = time.perf_counter() - t0
        if dist is not None:
            t = torch.tensor([e2e_s], dtype=torch.float64, device=f"cuda:{local}")
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            e2e_s = float(t[0])
            w = torch.tensor([e2e_evals], dtype=torch.int64, device=f"cuda:{local}")
            dist.all_reduce(w, op=dist.ReduceOp.SUM)
            e2e_evals = int(w[0])
        e2e = {"value": e2e_evals / e2e_s, "unit": UNIT, "h2d_bytes_per_step": n, "d2h_bytes_per_step": 12 * n + 8,
               "steps": args.e2e_steps, "step_ms": None if args.packet_budget else args.step_ms * args.e2e_step_factor,
               "step_packets": args.packet_budget * args.e2e_step_factor or None,
               "call": "mg_ctx_create + mg_anneal_oneshot (host data in, best slab + cost out); every step uploads the input, "
                       "builds the index, allocates and fills the chains, anneals, reads the best slab back and frees everything"}

    # ---- the match finder on its own (SURVEY 8d, K2): top-k at every position of the first 64 KiB plus
    # 4096 sampled ones, state-free pricing; reported beside the headline, not part of it
    finder = None
    if rank == 0 and world == 1 and not args.no_finder:
        fctx = mg.Context(data, device=local)
        fpos = np.concatenate([np.arange(min(n, 65536), dtype=np.uint64),
                               np.random.default_rng(7).integers(0, n, 4096).astype(np.uint64)])
        lit = mg.literal_slab(n)
        fctx.find_topk(lit, fpos[:256], state_mode=0)  # warm-up
        fctx.find_topk(lit, fpos, state_mode=0)
        fs = fctx.find_topk_stats()
        fctx.close()
        fsec = fs["kernel_ms"] / 1e3
        finder = {"kernel": "mg::topk_kernel", "positions": int(fpos.size), "kernel_ms": fs["kernel_ms"],
                  "positions_per_s": fpos.size / fsec, "candidates_per_s": fs["candidates"] / fsec,
                  "candidates_per_position": fs["candidates"] / fpos.size,
                  "hbm_algorithmic_GBps": 325.0 * fpos.size / fsec / 1e9,
                  "note": "325 B per query is the compulsory HBM traffic (SURVEY 8d); the kernel is bound by the serial "
                          "replay of the reference's heap and by L1/L2 reads of the window, not by HBM"}

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        cpu = cpu_baseline(n, args.cpu_evals)

    size = config3 = encode = None
    if rank == 0 and world == 1 and not args.no_size:
        wave = chains
        try:
            c0 = mg.Context(b"wave probe wave probe", device=local)
            wave = c0.full_wave()
            c0.close()
        except mg.MegalaniaError:
            pass
        encode = encode_leg(mg, data, best_slab, local)
        config3 = config3_leg(mg, wave, args.config3_seconds, sm_khz, local)
        size = size_leg(mg, wave, args.size_budget, local)

    if rank == 0:
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": 1e3 * wall / args.steps, "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": "u16 probabilities / u64 cost (integer)",
                "data": "synthetic",
                "config": {"workload": WORKLOAD, "input_bytes": n, "chains_per_gpu": chains,
                           "step": (f"each chain prices exactly {args.packet_budget} packets" if args.packet_budget else
                                    f"each chain anneals for {args.step_ms} ms of SM clocks ({cycle_budget} cycles)") +
                                   "; a proposal cut by the budget is suspended at a checkpoint and finished by the next step",
                           "top_k": 20, "l2": "inputs_exceed_l2",
                           "per_gpu_slab_bytes": chains * n * 8,
                           "multi_gpu": (None if world == 1 else
                                         f"BASELINE configs[3]: parallel tempering, one geometric ladder of {world * chains} temperatures "
                                         f"({args.t_min}..{args.t_max} in 1/2048 bit) over the replicas of all ranks; after every step an NCCL "
                                         f"all-gather of (cost, temperature) per replica and temperature swaps (mg_comm_temper_exchange); every "
                                         f"{args.exchange_every} steps the cheapest best slab is broadcast with its checkpoints and installed by copy "
                                         f"(mg_comm_exchange_best); collectives are the library's own NCCL calls behind the C ABI"),
                           "schedule": "reference rule src/main.c:86 (step 0)" if world == 1 else "Metropolis at the replica's ladder temperature"},
                "device_ms_per_step": 1e3 * device_s / args.steps,
                "timing": "value = evaluations / wall clock between barrier+cudaDeviceSynchronize brackets, max over ranks; "
                          "device_ms_per_step = CUDA events around the kernel on the library's launch stream",
                "clocks": clocks, "e2e": e2e, "gpu_launches": launches,
                "exchange_ms_per_step": exchange_ms[0] / args.steps if world > 1 else None,
                "comm": ctx_comm_stats,
                "roofline": roofline, "roofline_issue": roofline_issue, "finder": finder, "cpu_baseline": cpu,
                "size": size, "config3": config3, "encode": encode,
                "stats": {"evals": total_evals, "modelled_bits": total_bits, "packets": total_packets,
                          "attempts": agg["attempts"], "accepted": agg["accepted"],
                          "finder_candidates": agg["finder_candidates"], "log_overflows": agg["log_overflows"],
                          "finder_share_of_warp_time": agg["finder_cycles"] / max(1, agg["chain_cycles"]),
                          "warp_busy_fraction": agg["chain_cycles"] / max(1, chains * agg["max_chain_cycles"]) * 1.0 if args.steps == 1 else None,
                          "suspended_resumed": "proposals cut at the end of a step are finished by the next step"}}
        sys.stdout.flush()
        os.write(json_fd, (json.dumps(line) + "\n").encode())
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", choices=["cuda", "reference"], default="cuda")
    ap.add_argument("--size", type=int, default=1 << 20)
    ap.add_argument("--chains", type=int, default=0, help="chains per GPU (default: SMs x --warps-per-sm)")
    ap.add_argument("--warps-per-sm", type=int, default=0, help="0 = the library's own figure (chains per SM that fit shared memory)")
    ap.add_argument("--evals", type=int, default=1_000_000, help="cap on successful evaluations per chain per step")
    ap.add_argument("--packet-budget", type=int, default=STEP_PACKETS,
                    help="a chain ends its step when it has priced this many packets (reproducible); 0 = end steps on --step-ms")
    ap.add_argument("--step-ms", type=float, default=1000.0,
                    help="with --packet-budget 0: length of a step in milliseconds of SM clocks (results depend on the clock)")
    ap.add_argument("--seed", type=int, default=1673551)
    ap.add_argument("--exchange-every", type=int, default=4, help="multi-GPU: best-slab broadcast every this many steps")
    ap.add_argument("--t-min", type=float, default=16.0, help="multi-GPU: coldest ladder temperature, 1/2048 bit")
    ap.add_argument("--t-max", type=float, default=65536.0, help="multi-GPU: hottest ladder temperature, 1/2048 bit")
    ap.add_argument("--e2e-steps", type=int, default=2)
    ap.add_argument("--e2e-step-factor", type=int, default=3,
                    help="an end-to-end call anneals for this many bench steps (a one-shot call allocates ~90 GB of chains: "
                         "~0.3-0.7 s of fixed cost, which a one-second budget would not amortise)")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-finder", action="store_true")
    ap.add_argument("--no-size", action="store_true", help="skip the size / config 3 / encode legs")
    ap.add_argument("--size-budget", type=float, default=8.0, help="seconds of annealing per size-leg config (each side)")
    ap.add_argument("--config3-seconds", type=float, default=4.0)
    ap.add_argument("--cpu-evals", type=int, default=0, help="evaluations of the CPU sample (default: sized to ~15 s)")
    ap.add_argument("--cpu-procs", type=int, default=1 << 30)
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one left the chains with as DIR/<name>.npy "
                         "(per-chain costs, a seeded sample of slab slots; _rank<r> suffixes under torchrun)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.dump_outputs and args.impl != "cuda":
        ap.error("--dump-outputs writes the CUDA path's results")
    if args.cpu_evals == 0:
        # ~6.6 evals/s at 1 MiB on one core (BASELINE.md): ~15 s for the single-core sample,
        # ~2 s per step per core for the all-cores reference arm
        scale = max(1.0, (1 << 20) / args.size)
        args.cpu_evals = int((100 if args.impl == "cuda" else 12) * scale * scale)
    if args.impl == "reference":
        run_reference(args)
    else:
        run_cuda(args)


if __name__ == "__main__":
    main()

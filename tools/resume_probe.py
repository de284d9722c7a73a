"""How far `megalania --resume` gets from liblzma's lc = lp = pb = 0 parse, on the size leg's inputs and budget.

    python tools/resume_probe.py [--budget 8] [--device 0] [--out profiles/r03_resume_probe.json]

For each of bench.py's size-leg inputs (64 KiB text, 1 MiB mixed, 4 KiB binary, with the same chain counts): builds
liblzma's LZMA-alone -9e stream at lc = lp = pb = 0, decodes it on the device (mg_decode_stream: device time, events,
wall time of the call), runs the CLI with --resume at --time <budget> --round-ms 250, and records the output's bytes,
its round trip, xz -9e's bytes (lc = 3) and the resumed stream's own bytes - with the card's name and power limit,
read in the same run.  Uses the library and CLI as build() left them."""
from __future__ import annotations

import argparse
import json
import lzma
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import megalania_b200 as mg  # noqa: E402
from megalania_b200 import build  # noqa: E402
from tools import corpus  # noqa: E402


def card(device: int) -> dict:
    q = subprocess.run(["nvidia-smi", "-i", str(device), "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True)
    if q.returncode != 0:
        return {"error": q.stderr.strip()}
    name, power, clock = [x.strip() for x in q.stdout.strip().split("\n")[0].split(",")]
    return {"name": name, "power_limit": power, "max_sm_clock": clock}


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--budget", type=int, default=8, help="seconds of annealing (--time), the size leg's budget")
    ap.add_argument("--device", type=int, default=0)
    ap.add_argument("--repeats", type=int, default=3, help="decoder calls per input (the first loads the module)")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03_resume_probe.json"))
    args = ap.parse_args()
    with mg.Context(b"wave probe wave probe", device=args.device) as c0:
        wave = c0.full_wave()
    result = {"card": card(args.device), "budget_s": args.budget, "round_ms": 250, "configs": []}
    for name, kind, n, chains in (("config 1: 64 KiB synthetic English-like text", "text", 65536, wave),
                                  ("config 2: 1 MiB synthetic mixed text/binary", "mixed", 1 << 20, wave),
                                  ("config 3: 4 KiB synthetic executable-like binary", "binary", 4096, max(4096, wave))):
        data = corpus.make(kind, n)
        xz_lc0 = lzma.compress(data, format=lzma.FORMAT_ALONE,
                               filters=[{"id": lzma.FILTER_LZMA1, "preset": 9 | lzma.PRESET_EXTREME, "lc": 0, "lp": 0, "pb": 0}])
        rec = {"config": name, "input_bytes": n, "chains": chains, "resumed_stream_bytes": len(xz_lc0),
               "xz_9e_bytes": len(lzma.compress(data, format=lzma.FORMAT_ALONE, preset=9 | lzma.PRESET_EXTREME))}
        with mg.Context(data, device=args.device) as ctx:
            calls = []
            for _ in range(args.repeats):
                t0 = time.perf_counter()
                slab = ctx.decode_stream(xz_lc0)
                wall = time.perf_counter() - t0
                st = ctx.decode_stats()
                calls.append({"kernel_ms": st["kernel_ms"], "events": st["events"], "call_wall_ms": wall * 1e3})
            rec["decode"] = calls
            cost = ctx.score_slab(slab)
            rec["resumed_slab_bytes_estimate"] = 18 + cost / 16384.0
            rec["resumed_slab_reencoded_bytes"] = len(ctx.encode_slab(slab))
        with tempfile.TemporaryDirectory() as tmp:
            src = os.path.join(tmp, "in.bin")
            resume = os.path.join(tmp, "in.lzma")
            with open(src, "wb") as f:
                f.write(data)
            with open(resume, "wb") as f:
                f.write(xz_lc0)
            cmd = [build.CLI, "--chains", str(chains), "--time", str(args.budget), "--round-ms", "250", "--device",
                   str(args.device), "--resume", resume, src]
            t0 = time.perf_counter()
            r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.PIPE)
            rec["cli_wall_s"] = time.perf_counter() - t0
        rec["command"] = " ".join(["megalania"] + cmd[1:-3] + ["--resume", "<xz lc=0 -9e stream>", "<file>"])
        if r.returncode != 0:
            rec["error"] = r.stderr.decode(errors="replace")[-400:]
        else:
            rec["bytes"] = len(r.stdout)
            try:
                rec["round_trip"] = lzma.decompress(r.stdout, format=lzma.FORMAT_ALONE) == data
            except lzma.LZMAError:
                rec["round_trip"] = False
            rec["smaller_than_xz_9e"] = rec["bytes"] < rec["xz_9e_bytes"]
            rec["progress"] = r.stderr.decode(errors="replace").strip().split("\n")[-1]
        print(json.dumps(rec), flush=True)
        result["configs"].append(rec)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(result, f, indent=1)
    print(json.dumps({"card": result["card"]}))


if __name__ == "__main__":
    main()

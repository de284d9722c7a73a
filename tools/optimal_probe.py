"""Where the device's shortest-path parse (mg_anneal_optimal_init, `megalania --optimal`) starts and ends, against the
greedy parse, on the size leg's inputs and budget.

    python tools/optimal_probe.py [--budget 8] [--device 0] [--out profiles/r04_optimal_probe.json]

For each of bench.py's size-leg inputs (64 KiB text, 1 MiB mixed, 4 KiB binary, with the same chain counts):
optimal_init and greedy_init at the same region counts (1024 at 1 MiB, as the size leg's --greedy; 1 and 16 at the
small sizes; 1 and 64 at 1 MiB as well) - device time of the parse kernels, wall time of the call, exact cost as bytes - then the CLI with
--optimal R and with --greedy R (R = 1024 at 1 MiB, 16 otherwise) at --time <budget> --round-ms 250: the output's
bytes and round trip, and xz -9e's bytes (lc = 3), with the card's name and power limit read in the same run.  Uses
the library and CLI as build() left them."""
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
from tools.resume_probe import card  # noqa: E402


def as_bytes(cost: int) -> float:
    return 18 + cost / 16384.0  # header + 5 flush bytes, cost in 1/2048 bit


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--budget", type=int, default=8, help="seconds of annealing (--time), the size leg's budget")
    ap.add_argument("--device", type=int, default=0)
    ap.add_argument("--repeats", type=int, default=3, help="parse calls per setting (the first loads the module)")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r04_optimal_probe.json"))
    args = ap.parse_args()
    with mg.Context(b"wave probe wave probe", device=args.device) as c0:
        wave = c0.full_wave()
    result = {"card": card(args.device), "budget_s": args.budget, "round_ms": 250, "max_occ": 64, "configs": []}
    for name, kind, n, chains, inits, cli_regions in (
            ("config 1: 64 KiB synthetic English-like text", "text", 65536, wave, (1, 16), 16),
            ("config 2: 1 MiB synthetic mixed text/binary", "mixed", 1 << 20, wave, (1, 64, 1024), 1024),
            ("config 3: 4 KiB synthetic executable-like binary", "binary", 4096, max(4096, wave), (1, 16), 16)):
        data = corpus.make(kind, n)
        rec = {"config": name, "input_bytes": n, "chains": chains,
               "xz_9e_bytes": len(lzma.compress(data, format=lzma.FORMAT_ALONE, preset=9 | lzma.PRESET_EXTREME)),
               "init": []}
        with mg.Context(data, device=args.device) as ctx:
            an = mg.Annealer(ctx, 2)
            an.set_slab(None)
            for regions in inits:
                row = {"regions": regions, "optimal": [], "greedy": []}
                for _ in range(args.repeats):
                    t0 = time.perf_counter()
                    cost = an.optimal_init(regions, 0, 0)
                    wall = time.perf_counter() - t0
                    st = ctx.optimal_stats()
                    row["optimal"].append({"kernel_ms": st["kernel_ms"], "nodes": st["nodes"], "call_wall_ms": wall * 1e3,
                                           "cost": cost, "bytes_estimate": as_bytes(cost)})
                    t0 = time.perf_counter()
                    gcost = an.greedy_init(regions, 1)
                    row["greedy"].append({"call_wall_ms": (time.perf_counter() - t0) * 1e3, "cost": gcost,
                                          "bytes_estimate": as_bytes(gcost)})
                slab = an.get_slab(0)
                stream = ctx.encode_slab(slab)
                row["optimal_stream_bytes"] = len(stream)
                row["optimal_round_trip"] = lzma.decompress(stream, format=lzma.FORMAT_ALONE) == data
                row["optimal_below_greedy"] = row["optimal"][-1]["cost"] < row["greedy"][-1]["cost"]
                rec["init"].append(row)
            an.close()
        rec["cli"] = {}
        with tempfile.TemporaryDirectory() as tmp:
            src = os.path.join(tmp, "in.bin")
            with open(src, "wb") as f:
                f.write(data)
            for start in ("--optimal", "--greedy"):
                cmd = [build.CLI, "--chains", str(chains), "--time", str(args.budget), "--round-ms", "250", "--device",
                       str(args.device), start, str(cli_regions), src]
                t0 = time.perf_counter()
                r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.PIPE)
                leg = {"command": " ".join(["megalania"] + cmd[1:-1] + ["<file>"]), "cli_wall_s": time.perf_counter() - t0}
                if r.returncode != 0:
                    leg["error"] = r.stderr.decode(errors="replace")[-400:]
                else:
                    leg["bytes"] = len(r.stdout)
                    try:
                        leg["round_trip"] = lzma.decompress(r.stdout, format=lzma.FORMAT_ALONE) == data
                    except lzma.LZMAError:
                        leg["round_trip"] = False
                    leg["smaller_than_xz_9e"] = leg["bytes"] < rec["xz_9e_bytes"]
                    leg["progress"] = r.stderr.decode(errors="replace").strip().split("\n")[-1]
                rec["cli"][start.strip("-")] = leg
        o, g = rec["cli"]["optimal"].get("bytes"), rec["cli"]["greedy"].get("bytes")
        if o is not None and g is not None:
            rec["cli_optimal_below_greedy"] = o < g
        print(json.dumps(rec), flush=True)
        result["configs"].append(rec)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(result, f, indent=1)
    print(json.dumps({"card": result["card"]}))


if __name__ == "__main__":
    main()

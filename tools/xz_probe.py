"""What writing .xz costs against writing .lzma: device time of mg_encode_slab (one coder on one SM) against the plan
walk and chunk kernel of mg_encode_slab_xz (LZMA2 chunks coded side by side), and the bytes of both streams.

    python tools/xz_probe.py [--device 0] [--repeats 3] [--out profiles/r05_xz_probe.json]

Inputs: 4 KiB binary, 64 KiB text and 1 MiB mixed, each as the all-literal slab and as the device's greedy parse of
1024 regions (as --greedy 1024; fewer regions where the input has fewer than 64 bytes per region), and the 16 MiB corpus
of tools/big_probe.py as the all-literal slab.  Every output is checked with `xz -t`.  Times are the least of
--repeats calls (the first call of each kernel also loads the module).  The card's name and power limit are read in
the same run.  Uses the library as build() left it."""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import megalania_b200 as mg  # noqa: E402
from tools import corpus  # noqa: E402
from tools.resume_probe import card  # noqa: E402

INPUTS = [("binary", 4096), ("text", 65536), ("mixed", 1 << 20), ("corpus16", 16 << 20)]


def xz_test(stream: bytes, fmt: str) -> bool:
    return subprocess.run(["xz", "-t", f"--format={fmt}", "-"], input=stream, capture_output=True).returncode == 0


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--device", type=int, default=0)
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r05_xz_probe.json"))
    args = ap.parse_args()
    result = {"card": card(args.device), "rows": []}
    for kind, n in INPUTS:
        data = corpus.make(kind, n)
        with mg.Context(data, args.device) as ctx:
            slabs = {"literal": mg.literal_slab(n)}
            if n <= 1 << 20:
                regions = min(1024, n // 64)
                an = mg.Annealer(ctx, 1)
                an.set_slab(None)
                an.greedy_init(regions)
                slabs[f"greedy{regions}"] = an.get_slab(0)
                an.close()
            for name, slab in slabs.items():
                enc_ms, plan_ms, code_ms = [], [], []
                for _ in range(args.repeats):
                    lz = ctx.encode_slab(slab)
                    enc = ctx.encode_stats()
                    enc_ms.append(enc["kernel_ms"])
                    xz = ctx.encode_xz(slab)
                    st = ctx.encode_xz_stats()
                    plan_ms.append(st["plan_ms"])
                    code_ms.append(st["code_ms"])
                row = {"input": f"{kind}_{n}", "slab": name, "lzma_encode_ms": min(enc_ms),
                       "xz_plan_ms": min(plan_ms), "xz_code_ms": min(code_ms),
                       "xz_total_ms": min(p + c for p, c in zip(plan_ms, code_ms)), "chunks": st["chunks"],
                       "events": st["events"], "events_match": st["events"] == enc["events"],
                       "lzma_bytes": len(lz), "xz_bytes": len(xz), "lzma_xz_t": xz_test(lz, "lzma"),
                       "xz_xz_t": xz_test(xz, "xz")}
                print(json.dumps(row), flush=True)
                result["rows"].append(row)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(result, f, indent=1)


if __name__ == "__main__":
    main()

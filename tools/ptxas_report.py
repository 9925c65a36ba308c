#!/usr/bin/env python
"""Registers, spills and stack of every kernel of the last library build, from the `-Xptxas -v` log that
`poseestimationkf_b200/build.py` writes beside the library (build_ptxas.log), with demangled names.

  python tools/ptxas_report.py [--match replay_] [--gated | --general | --innov-steps | --general-innovation]
                               [--out profiles/r06_gating_registers.json]

--gated keeps the replay kernels instantiated with the innovation gate (the GATE template flag set), --general those
instantiated with general Q and R matrices (the GEN flag of the scalar kernels set), --innov-steps those with the
per-step innovation output (an InnovStepArgs in their parameter pack), --general-innovation those with general matrices
and the innovation terms (the GEN and INNOV flags both set).
"""
from __future__ import annotations

import argparse
import json
import os
import re
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def entries(log_text: str):
    out = []
    for chunk in re.split(r"ptxas info\s+: Compiling entry function '", log_text)[1:]:
        name = chunk.split("'")[0]
        regs = re.search(r"Used (\d+) registers", chunk)
        spill = re.search(r"(\d+) bytes spill stores, (\d+) bytes spill loads", chunk)
        stack = re.search(r"(\d+) bytes stack frame", chunk)
        out.append({"mangled": name, "registers": int(regs.group(1)) if regs else None,
                    "spill_store_bytes": int(spill.group(1)) if spill else None,
                    "spill_load_bytes": int(spill.group(2)) if spill else None,
                    "stack_bytes": int(stack.group(1)) if stack else None})
    names = subprocess.run(["c++filt"], input="\n".join(e["mangled"] for e in out), capture_output=True,
                           text=True).stdout.splitlines()
    for e, n in zip(out, names):
        e["kernel"] = n.split("(")[0]
    return out


def _flag(kernel: str, i: int) -> bool:
    m = re.search(r"replay_\w+_kernel<([^>]*)>", kernel)
    if not m:
        return False
    args = [a.strip() for a in m.group(1).split(",")]
    return len(args) > i and args[i] == "true"


def is_gated(kernel: str) -> bool:
    return _flag(kernel, 7)


def is_general(kernel: str) -> bool:
    return _flag(kernel, 8)


def is_general_innovation(kernel: str) -> bool:
    return _flag(kernel, 8) and _flag(kernel, 4)


def is_innov_steps(kernel: str) -> bool:
    return "InnovStepArgs" in kernel


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--log", default=os.path.join(ROOT, "poseestimationkf_b200", "build_ptxas.log"))
    ap.add_argument("--match", default="")
    ap.add_argument("--gated", action="store_true")
    ap.add_argument("--general", action="store_true")
    ap.add_argument("--innov-steps", action="store_true")
    ap.add_argument("--general-innovation", action="store_true")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    ents = [e for e in entries(open(a.log).read()) if a.match in e["kernel"] and (not a.gated or is_gated(e["kernel"]))
            and (not a.general or is_general(e["kernel"])) and (not a.innov_steps or is_innov_steps(e["kernel"]))
            and (not a.general_innovation or is_general_innovation(e["kernel"]))]
    for e in ents:
        del e["mangled"]
    res = {"source": "ptxas -v of the sm_100a build (nvcc flags of poseestimationkf_b200/build.py)",
           "kernels": len(ents), "spilling": sum(1 for e in ents if e["spill_store_bytes"] or e["spill_load_bytes"]),
           "max_registers": max((e["registers"] for e in ents), default=None), "entries": ents}
    text = json.dumps(res, indent=1)
    if a.out:
        with open(a.out, "w") as fh:
            fh.write(text + "\n")
    print(json.dumps({k: v for k, v in res.items() if k != "entries"}))
    return 0 if res["spilling"] == 0 else 1


if __name__ == "__main__":
    sys.exit(main())

#!/usr/bin/env python3
"""Fused passes over unaligned rows (``PlanOptions(unaligned=1)``) against what the same grid runs without the option
(one-operator kernels) and against the aligned sibling grid on its default plan, alternated in one process, three
rounds each.  Each sample is the device time of ``--reps`` back-to-back executions (CUDA events around all of them,
after warm-up) over ``--reps``.  Inputs are hash-filled on the device; the outputs of the two plans of one grid are
compared by their checksum bits.

Cases: Jacobi-3D 1024x1024x1022 x 8 (aligned sibling 1024^3), hdiff 1024x1024x78 (sibling 1024x1024x80), the
float64 2-D chain 32768x32767 x 16 (sibling 32768^2).  Prints the card's name and power limit, a table, and one
JSON line."""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))

from cluster_timing import card, per_execution_us  # noqa: E402

FILLS = {"a": (0.0, 1.0), "inp": (1.0, 2.0), "coeff": (0.0, 0.05)}


def load(path, opts):
    from stencilflow_b200.cuda_program import CudaProgram
    prog = CudaProgram(path, plan_options=opts, device=0)
    n = int(np.prod(prog.program.shape))
    for k, (name, f) in enumerate(sorted(prog.program.fields.items())):
        if f.kind == "input" and not f.is_scalar:
            lo, hi = FILLS.get(name, (0.0, 1.0))
            prog.rt.fill_hash(prog.buffers[name].dptr, n, f.data_type.type, seed=99 + k, lo=lo, hi=hi)
    return prog


def describe(prog):
    out = []
    for l in prog.lowered.launches:
        if l.family == "streamed":
            i = l.info
            out.append("streamed R{} w{} k{} tile {} sync {}{}".format(
                i["R"], i["warps"][0], i["threads_per_row"], i["tile"], i["sync"], " unaligned" if i.get("unaligned") else ""))
        else:
            out.append(l.family)
    return out


class ClockSampler:
    """SM clock and power draw (nvidia-smi, every 0.5 s) while a group of cases is timed: min / max of each."""

    def __init__(self):
        self.samples, self._stop = [], threading.Event()
        self._thread = threading.Thread(target=self._run, daemon=True)

    def _run(self):
        while not self._stop.is_set():
            try:
                out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=clocks.sm,power.draw",
                                      "--format=csv,noheader,nounits"], stdout=subprocess.PIPE, text=True,
                                     timeout=10).stdout.strip().split(",")
                self.samples.append((float(out[0]), float(out[1])))
            except (OSError, subprocess.SubprocessError, ValueError, IndexError):
                pass
            self._stop.wait(0.5)

    def __enter__(self):
        self._thread.start()
        return self

    def __exit__(self, *exc):
        self._stop.set()
        self._thread.join()

    def summary(self):
        if not self.samples:
            return {}
        mhz, watts = zip(*self.samples)
        return {"sm_mhz": [min(mhz), max(mhz)], "power_w": [min(watts), max(watts)], "samples": len(mhz)}


def compare(cases, reps, rounds):
    """cases: [(label, path, PlanOptions)]; the first two share a grid and must agree bit for bit."""
    progs = [(label, load(path, opts)) for label, path, opts in cases]
    rec = {label: {"plan": describe(p), "ms": []} for label, p in progs}
    for _, p in progs:
        per_execution_us(p, 3)
    with ClockSampler() as clocks:
        for _ in range(rounds):
            for label, p in progs:
                rec[label]["ms"].append(round(per_execution_us(p, reps) / 1e3, 3))
    rec["clocks_while_timed"] = clocks.summary()
    bits = []
    for label, p in progs[:2]:
        out = p.program.outputs[0]
        f = p.program.fields[out]
        bits.append(p.rt.checksum(p.buffers[out].dptr, int(np.prod(f.shape)), f.data_type.type)[1])
    for _, p in progs:
        p.close()
    rec["checksum_bits_equal"] = bits[0] == bits[1]
    return rec


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--reps", type=int, default=10, help="back-to-back executions per sample")
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--only", default="", help="comma-separated subset of jacobi3d,hdiff,jacobi2d")
    args = ap.parse_args()
    from stencilflow_b200 import build, programs
    from stencilflow_b200.planner import PlanOptions
    build.build_native()
    tmp = tempfile.mkdtemp(prefix="sfb200_unaligned_timing_")
    os.environ.setdefault("SFB200_CACHE", os.path.join(tmp, "cache"))      # cubins and programs stay out of the tree

    def write(prog, name):
        return programs.write_program(prog, name, tmp)

    groups = {
        "jacobi3d": [("1024x1024x1022 unaligned", write(programs.jacobi3d_chain([1024, 1024, 1022], 8), "j3_1022"),
                      PlanOptions(unaligned=1)),
                     ("1024x1024x1022 default", write(programs.jacobi3d_chain([1024, 1024, 1022], 8), "j3_1022"),
                      PlanOptions()),
                     ("1024^3 default", write(programs.jacobi3d_chain([1024, 1024, 1024], 8), "j3_1024"), PlanOptions())],
        "hdiff": [("1024x1024x78 unaligned", write(programs.hdiff([1024, 1024, 78]), "hd_78"), PlanOptions(unaligned=1)),
                  ("1024x1024x78 default", write(programs.hdiff([1024, 1024, 78]), "hd_78"), PlanOptions()),
                  ("1024x1024x80 default", write(programs.hdiff([1024, 1024, 80]), "hd_80"), PlanOptions())],
        "jacobi2d": [("32768x32767 unaligned", write(programs.jacobi2d_chain([32768, 32767], 16), "j2_32767"),
                      PlanOptions(unaligned=1)),
                     ("32768x32767 default", write(programs.jacobi2d_chain([32768, 32767], 16), "j2_32767"),
                      PlanOptions()),
                     ("32768^2 default", write(programs.jacobi2d_chain([32768, 32768], 16), "j2_32768"), PlanOptions())],
    }
    only = [g for g in args.only.split(",") if g] or list(groups)
    print("card: {}".format(card()), flush=True)
    result = {"card": card(), "reps": args.reps, "cases": {}}
    for g in only:
        rec = compare(groups[g], args.reps, args.rounds)
        result["cases"][g] = rec
        for label, _, _ in groups[g]:
            print("{:9s} {:28s} {} ms  {}".format(g, label, rec[label]["ms"], "; ".join(rec[label]["plan"])), flush=True)
        print("{:9s} checksum bits equal (unaligned vs default): {}; clocks while timed: {}".format(
            g, rec["checksum_bits_equal"], rec["clocks_while_timed"]), flush=True)
    print(json.dumps(result), flush=True)


if __name__ == "__main__":
    main()

#!/usr/bin/env python3
"""Freezes, per program of ``tests/programs`` and ``programs/``, a digest of the fused-pass (``sf_stream_*``)
kernel sources and of ``plan.describe()`` (without its options) for the default plan and for explicit fusion
depths 2 and 4.  ``tests/test_unaligned_plan.py`` checks that planning options which only concern other
programs leave these unchanged.  Run from the repository root:  python tests/golden/make_stream_digests.py
"""
import hashlib
import json
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)

DEPTHS = (None, 2, 4)
# the cost model's HBM rate is read from a per-machine file when it exists: digests are taken at the default
HBM_BYTES_PER_S = 6.1e12


def program_files():
    out = []
    for d in ("tests/programs", "programs"):
        for f in sorted(os.listdir(os.path.join(ROOT, d))):
            if f.endswith(".json"):
                out.append(os.path.join(d, f))
    return out


def digests(path, **extra):
    """{variant: [stream-source digest, describe digest]} of one program file."""
    from stencilflow_b200 import lower_stream
    from stencilflow_b200.kernel_chain_graph import KernelChainGraph
    from stencilflow_b200.planner import PlanOptions, plan_program
    from stencilflow_b200.stencil_op import make_program
    lower_stream.HBM_BYTES_PER_S = HBM_BYTES_PER_S
    program = make_program(KernelChainGraph(os.path.join(ROOT, path)))
    out = {}
    for depth in DEPTHS:
        opts = dict(extra)
        if depth:
            opts["max_depth"] = depth
        plan = plan_program(program, PlanOptions(**opts))
        text = "".join(k.source for name, k in sorted(plan.lowered.kernels.items()) if name.startswith("sf_stream_"))
        desc = {k: v for k, v in plan.describe().items() if k != "options"}
        out[str(depth or "default")] = [hashlib.sha1(text.encode()).hexdigest(),
                                        hashlib.sha1(json.dumps(desc, sort_keys=True, default=str).encode()).hexdigest()]
    return out


def main():
    for k in list(os.environ):
        if k.startswith("SFB200_"):
            del os.environ[k]
    table = {path: digests(path) for path in program_files()}
    with open(os.path.join(HERE, "sf_stream_digests.json"), "w") as f:
        json.dump(table, f, indent=1, sort_keys=True)
        f.write("\n")


if __name__ == "__main__":
    main()

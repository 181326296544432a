#!/usr/bin/env python3
"""Small grids: the default plan (one-operator kernels, replayed through a CUDA graph when there are three or
more) against the cluster family (``PlanOptions(cluster=1)``: the whole program in one launch of one
thread-block cluster), alternated in one process, three rounds each.  Each sample is the device time of
``--reps`` back-to-back executions (CUDA events around all of them, after warm-up) over ``--reps``; outputs
of the two plans are compared bit for bit.

Where the cluster kernel's time goes, from the same process:
* Jacobi-3D 32^3 with 1, 2, 4 and 8 operators on the cluster path: the slope is the cost of one operator
  (its compute and the cluster barrier before it), the intercept the launch, the input load, the final
  barrier and the exit;
* a kernel of 8 x 1024 threads that only runs cluster barriers (``barrier.cluster.arrive.release`` +
  ``wait.acquire``, as the generated code does): the cost of one barrier on its own.

Prints the card's name and power limit, a table, and one JSON line."""
import argparse
import json
import os
import subprocess
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

BARRIER_SOURCE = r"""
extern "C" __global__ void __cluster_dims__(8, 1, 1) __launch_bounds__(1024) sf_barrier_loop(int n, int* sink)
{
    for (int r = 0; r < n; ++r)
        asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
    if (threadIdx.x == 0 && n < 0) sink[blockIdx.x] = n;
}
"""


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             stdout=subprocess.PIPE, text=True, timeout=30).stdout.strip().splitlines()
        return out[0] if out else "unknown"
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def per_execution_us(prog, reps):
    rt = prog.rt
    e0, e1 = rt.event_create(), rt.event_create()
    rt.event_record(e0)
    for _ in range(reps):
        prog.execute()
    rt.event_record(e1)
    rt.event_synchronize(e1)
    ms = rt.elapsed_ms(e0, e1)
    rt.event_destroy(e0)
    rt.event_destroy(e1)
    return 1e3 * ms / reps


def load(path, opts, inputs):
    from stencilflow_b200.cuda_program import CudaProgram
    prog = CudaProgram(path, plan_options=opts, device=0)
    for name, value in inputs.items():
        prog.upload(name, value)
    return prog


def compare(path, reps, rounds):
    from stencilflow_b200 import synthetic
    from stencilflow_b200.planner import PlanOptions
    from stencilflow_b200.cuda_program import CudaProgram
    probe = CudaProgram(path, allocate=False)
    fields = probe.program.fields
    inputs = {n: synthetic.fill_hash(f.shape, f.data_type.type, 99) for n, f in fields.items()
              if f.kind == "input" and not f.is_scalar}
    out = probe.program.outputs[0]
    progs = {"default": load(path, PlanOptions(cluster=0), inputs), "cluster": load(path, PlanOptions(cluster=1), inputs)}
    rec = {label: {"launches": len(p.lowered.launches), "families": sorted({l.family for l in p.lowered.launches}),
                   "us": []} for label, p in progs.items()}
    rec["cluster"]["info"] = {k: progs["cluster"].lowered.launches[0].info[k]
                              for k in ("cluster", "threads", "barriers_before")}
    rec["cluster"]["smem"] = progs["cluster"].lowered.launches[0].smem
    for p in progs.values():
        per_execution_us(p, 20)                        # warm-up: module load, graph capture
    for _ in range(rounds):
        for label, p in progs.items():
            rec[label]["us"].append(round(per_execution_us(p, reps), 2))
    bits = [p.download(out).tobytes() for p in progs.values()]
    for p in progs.values():
        p.close()
    rec["bit_identical"] = bits[0] == bits[1]
    return rec


def barrier_cost(reps):
    from stencilflow_b200 import runtime as rt_mod
    from stencilflow_b200.cuda_program import compile_cached
    rt = rt_mod.Runtime.get(0)
    image, _, _ = compile_cached("sf_barrier_loop", BARRIER_SOURCE)
    module = rt.module_load(image)
    fn = rt.get_function(module, "sf_barrier_loop")
    sink = rt.malloc(64)
    import ctypes
    times = {}
    for n in (0, 1000):
        vals = [ctypes.c_int(n), ctypes.c_void_p(sink)]
        pack = rt_mod.pack_params(vals)
        for _ in range(5):
            rt.launch(fn, (8, 1, 1), (1024, 1, 1), 0, pack.array)
        e0, e1 = rt.event_create(), rt.event_create()
        rt.event_record(e0)
        for _ in range(reps):
            rt.launch(fn, (8, 1, 1), (1024, 1, 1), 0, pack.array)
        rt.event_record(e1)
        rt.event_synchronize(e1)
        times[n] = 1e3 * rt.elapsed_ms(e0, e1) / reps
        rt.event_destroy(e0)
        rt.event_destroy(e1)
    rt.free(sink)
    rt.module_unload(module)
    return {"empty_cluster_launch_us": round(times[0], 2),
            "ns_per_barrier": round(1e3 * (times[1000] - times[0]) / 1000, 1)}


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--reps", type=int, default=200, help="back-to-back executions per sample (>= 100)")
    ap.add_argument("--rounds", type=int, default=3)
    args = ap.parse_args()
    from stencilflow_b200 import build, programs
    build.build_native()
    tmp = tempfile.mkdtemp(prefix="sfb200_cluster_timing_")
    os.environ.setdefault("SFB200_CACHE", os.path.join(tmp, "cache"))      # generated programs and cubins stay out of the tree
    cases = []
    for n in (32, 48):
        cases.append(("jacobi3d_{0}x{0}x{0}_8itr".format(n),
                      programs.write_program(programs.jacobi3d_chain([n, n, n], 8), "jacobi3d_{}_8".format(n), tmp)))
    for name in ("ref_jacobi2d_128x128", "smooth1d_256"):
        cases.append((name, os.path.join(ROOT, "tests", "programs", name + ".json")))
    print("card: {}".format(card()))
    result = {"card": card(), "reps": args.reps, "cases": {}, "breakdown": {}}
    for name, path in cases:
        rec = compare(path, args.reps, args.rounds)
        result["cases"][name] = rec
        print("{:28s} default {:>2} launch(es) {} us | cluster C={} T={} smem={} B barriers={} {} us | bits equal: {}".format(
            name, rec["default"]["launches"], rec["default"]["us"], rec["cluster"]["info"]["cluster"],
            rec["cluster"]["info"]["threads"], rec["cluster"]["smem"], len(rec["cluster"]["info"]["barriers_before"]) + 1,
            rec["cluster"]["us"], rec["bit_identical"]), flush=True)
    from stencilflow_b200.planner import PlanOptions
    from stencilflow_b200 import synthetic
    for steps in (1, 2, 4, 8):
        path = programs.write_program(programs.jacobi3d_chain([32, 32, 32], steps), "jacobi3d_32_{}".format(steps), tmp)
        prog = load(path, PlanOptions(cluster=1), {"a": synthetic.fill_hash((32, 32, 32), np.float32, 99)})
        per_execution_us(prog, 20)
        us = [round(per_execution_us(prog, args.reps), 2) for _ in range(args.rounds)]
        prog.close()
        result["breakdown"]["jacobi3d_32_ops{}".format(steps)] = us
        print("cluster jacobi3d 32^3 x {}: {} us".format(steps, us), flush=True)
    xs = [1, 2, 4, 8]
    ys = [min(result["breakdown"]["jacobi3d_32_ops{}".format(s)]) for s in xs]
    slope, icpt = np.polyfit(xs, ys, 1)
    result["fit"] = {"us_per_operator": round(float(slope), 2), "us_fixed": round(float(icpt), 2)}
    result["barrier"] = barrier_cost(args.reps)
    print("per operator {:.2f} us (compute + one cluster barrier), fixed {:.2f} us (launch, load, exit)".format(
        slope, icpt))
    print("barrier-only kernel (8 x 1024 threads): {}".format(result["barrier"]))
    print(json.dumps(result), flush=True)


if __name__ == "__main__":
    main()

#!/usr/bin/env python3
"""Headline benchmark: stencil cell-updates/s and fraction of the HBM roofline (BASELINE.json).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--config C] [--impl ours|reference] [--dump-outputs DIR]

A *step* is one execution of the whole stencil program (all chained operators) over one synthetic
field.  Default workload = BASELINE.json configs[1]: Jacobi-3D, 8 chained operators, 1024^3 float32,
constant boundary.  For N > 1 (launched by torchrun, one rank per GPU) every rank owns a 1024^3 slab
of a (N*1024) x 1024 x 1024 domain and exchanges halos with its neighbours over NVLink once per
fused pass (weak scaling).  The same line also carries

* ``verify``: the timed result checked -- against the CPU oracle on a block of planes, against the
  one-operator kernels at full size, and (N > 1) bit for bit against one GPU running the whole domain;
* ``strong``: BASELINE.json configs[4] (Jacobi-3D 2048^3 x 64 operators) split over the same N GPUs,
  with the one-GPU time of the same box next to it.

One JSON line is printed by rank 0; see DESIGN.md section "Measurement" for the definition of every key.
Compiled kernels, generated programs and the CPU oracle's build go to a temporary directory (or to
``SFB200_CACHE`` if that is set), so the tree this runs from may be read-only.
"""
import argparse
import contextlib
import json
import os
import shutil
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "stencil_cell_updates_per_s"
UNIT = "cell-updates/s"


def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(path):
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region."""
    QUERY = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
             "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, device=0):
        self.device = device
        self.proc = None
        self.path = None

    def start(self):
        try:
            fd, self.path = tempfile.mkstemp(suffix=".csv")
            os.close(fd)
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.device), "--query-gpu=" + self.QUERY,
                 "--format=csv,noheader,nounits", "-lms", "20"],
                stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
        except OSError:
            self.proc = None

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, smax, power, reasons = [], [], [], set()
        with open(self.path) as f:
            for line in f:
                parts = [p.strip() for p in line.split(",")]
                if len(parts) < 9:
                    continue
                try:
                    sm.append(float(parts[1]))
                    smax.append(float(parts[2]))
                    power.append(float(parts[3]))
                except ValueError:
                    continue
                for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown",
                                      "sw_power_cap"), parts[5:9]):
                    if val.lower().startswith("active"):
                        reasons.add(name)
        os.unlink(self.path)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(smax)), "samples": len(sm),
                "power_w_max": float(max(power)), "reasons": sorted(reasons)}


VARIANT = None          # --variant: secondary form of a config (programs.VARIANTS)


def build_config(index, scale_i=1):
    from stencilflow_b200 import programs
    name, prog, halo = programs.baseline_config(index, VARIANT)
    if scale_i > 1:
        prog["dimensions"][0] *= scale_i
        name += "_x{}".format(scale_i)
    return name, prog, halo


INPUT_RANGES = {"inp": (1.0, 2.0), "coeff": (0.0, 0.05), "w": (0.9, 1.1)}   # hdiff; everything else U[0,1)
SEED = 1234


def fill_inputs(program, seed=SEED, index_offsets=None):
    rt = program.rt
    for k, (name, f) in enumerate(program.program.fields.items()):
        if f.kind != "input":
            continue
        if f.is_scalar:
            program.set_scalars({name: 0.5})
            continue
        lo, hi = INPUT_RANGES.get(name, (0.0, 1.0))
        n = int(np.prod(program.local_shape(name)))
        off = (index_offsets or {}).get(name, 0)
        rt.fill_hash(program.buffers[name].dptr, n, f.data_type.type, seed + k, lo, hi, off)
    rt.stream_synchronize()


def host_inputs(prog, dims, seed=SEED):
    """The synthetic input fields of ``prog`` restricted to the leading ``dims`` block, generated on
    the host (same counter hash as ``fill_inputs``: element values depend on the *global* flat index)."""
    from stencilflow_b200 import synthetic
    full = list(prog["dimensions"])
    iters = ["i", "j", "k"][3 - len(full):]
    out = {}
    for k, (name, cfg) in enumerate(prog["inputs"].items()):
        lo, hi = INPUT_RANGES.get(name, (0.0, 1.0))
        its = cfg.get("input_dims", iters)
        if not its:
            out[name] = np.dtype(cfg["data_type"]).type(0.5)
            continue
        fshape = tuple(n for it, n in zip(iters, full) if it in its)
        bshape = tuple(n for it, n in zip(iters, dims) if it in its)
        if fshape[1:] != bshape[1:]:
            raise ValueError("only the outermost dimension may be cut")
        # a leading block of a row-major field is a prefix of its flat index space
        out[name] = synthetic.fill_hash(bshape, np.dtype(cfg["data_type"]), seed + k, lo, hi)
    return out


@contextlib.contextmanager
def scratch_cache():
    """Points ``SFB200_CACHE`` (NVRTC cubins, generated programs, the oracle's build) at a fresh temporary
    directory for the duration of the run and removes it afterwards, unless the caller has set it."""
    if os.environ.get("SFB200_CACHE"):
        yield
        return
    path = tempfile.mkdtemp(prefix="sfb200_bench_")
    os.environ["SFB200_CACHE"] = path           # inherited by the ranks torchrun starts
    try:
        yield
    finally:
        shutil.rmtree(path, ignore_errors=True)


def oracle_build_dir():
    cache = os.environ.get("SFB200_CACHE")
    return os.path.join(cache, "oracle") if cache else None


DUMP_BYTES = 32 << 20       # all arrays of --dump-outputs together
DUMP_SEED = 4321


def dump_outputs(program, directory, halo):
    """``--dump-outputs``: every output field of ``program`` as it is on the device now, written as
    ``<directory>/<field>.npy`` in the field's data type.  The ``-halo`` border of shrink boundaries is cut
    off: its content is not defined.  A field larger than its share of DUMP_BYTES is written as its values
    at distinct flat indices drawn with DUMP_SEED, in ascending order (1-D), the same sample on every run."""
    os.makedirs(directory, exist_ok=True)
    outputs = program.program.outputs
    share = DUMP_BYTES // len(outputs)
    for name in outputs:
        arr = program.download(name)
        if halo:
            arr = arr[tuple(slice(halo, -halo) for _ in arr.shape)]
        if arr.nbytes > share:
            flat = np.unique(np.random.default_rng(DUMP_SEED).integers(0, arr.size, size=share // arr.itemsize))
            arr = arr[np.unravel_index(flat, arr.shape)]
        np.save(os.path.join(directory, name + ".npy"), np.ascontiguousarray(arr))


# ------------------------------------------------------------------------------------ CPU arm


class CpuSample:
    """The reference's CPU program (oracle/reference_cpp.py: OpenMP over the outermost loop, DaCe's flags
    -O3 -march=native -ffast-math, all transients live) built and allocated once for a bounded sample
    of a workload; ``run()`` times one execution."""

    def __init__(self, index, target_seconds=10.0, threads=None):
        from oracle import reference_cpp
        from stencilflow_b200 import programs, synthetic
        # all host threads, also under torchrun (which exports OMP_NUM_THREADS=1 to every rank);
        # SFB200_REF_THREADS overrides.  The count reported is the one the OpenMP runtime really uses.
        cores = threads or int(os.environ.get("SFB200_REF_THREADS", "0")) or os.cpu_count() or 1
        os.environ["OMP_NUM_THREADS"] = str(cores)
        self.name, prog, _ = programs.baseline_config(index, VARIANT)
        full = list(prog["dimensions"])
        self.nops = len(prog["program"])
        short = [d < 256 for d in full]                    # hdiff's vertical axis is kept as it is
        iters = ["i", "j", "k"][3 - len(full):]

        def sized(frac):
            return [d if sh else max(16, int(d * frac) // 8 * 8) for d, sh in zip(full, short)]

        def build(dims):
            p = json.loads(json.dumps(prog))
            p["dimensions"] = dims
            ref = reference_cpp.CompiledReference(p, build_dir=oracle_build_dir())
            inputs = {}
            for k, (iname, cfg) in enumerate(p["inputs"].items()):
                lo, hi = INPUT_RANGES.get(iname, (0.0, 1.0))
                shape = tuple(n for it, n in zip(iters, dims) if it in cfg.get("input_dims", iters))
                inputs[iname] = synthetic.fill_hash(shape, np.dtype(cfg["data_type"]), SEED + k, lo, hi)
            ref.allocate_transients()
            return ref, inputs

        # a small probe tells how large a sample fits the time budget (and the host's memory)
        probe_dims = sized(0.125 if full[0] >= 1024 else 1.0)
        ref, inputs = build(probe_dims)
        ref(**inputs)
        t0 = time.perf_counter()
        ref(**inputs)
        rate = self.nops * float(np.prod(probe_dims)) / (time.perf_counter() - t0)
        try:
            import psutil
            avail = psutil.virtual_memory().available
        except Exception:
            avail = 16 << 30
        itemsize = np.dtype(next(iter(prog["inputs"].values()))["data_type"]).itemsize
        mem_cells = 0.5 * avail / ((self.nops + 2) * itemsize)
        cells_full = float(np.prod(full))
        want_cells = min(cells_full, rate * target_seconds / self.nops, mem_cells)
        frac = (want_cells / cells_full) ** (1.0 / max(1, short.count(False)))
        dims = sized(min(1.0, frac))
        if np.prod(dims) > np.prod(probe_dims):
            del ref, inputs
            ref, inputs = build(dims)
            ref(**inputs)                                   # warm: page faults, OpenMP team
        else:
            dims = probe_dims
        self.ref, self.inputs, self.dims = ref, inputs, dims
        self.cores = ref.threads
        self.updates = self.nops * float(np.prod(dims))

    def run(self):
        t0 = time.perf_counter()
        self.ref(**self.inputs)
        return time.perf_counter() - t0

    def describe(self, timed):
        return "{} at {} ({} operators, all transients live), 1 warm + {} timed execution{}".format(
            self.name, "x".join(map(str, self.dims)), self.nops, timed, "" if timed == 1 else "s")


def cpu_reference_rate(index, target_seconds=10.0, threads=None):
    """(cell-updates/s, cores, sample description) of the CPU restatement on a bounded sample."""
    sample = CpuSample(index, target_seconds, threads)
    dt = sample.run()
    return sample.updates / dt, sample.cores, sample.describe(1)


def common_config(index, prog, world, scaling):
    dims = list(prog["dimensions"])
    fp64 = "float64" in json.dumps(prog["program"])
    per_gpu = [dims[0] // world] + dims[1:]
    return {"workload": workload_name(index, prog),
            "per_gpu": "x".join(map(str, per_gpu)),
            "l2": "no flush needed: every pass streams fields of {:.1f} GiB, far above the 126 MB L2".format(
                float(np.prod(per_gpu)) * (8 if fp64 else 4) / 2 ** 30),
            "input": "U[0,1) counter hash (seed {}), generated in HBM by the GPU arm".format(SEED)}


def run_reference_arm(args):
    """``--impl reference``: the reference's CPU path (the oracle's C++/OpenMP restatement -- the
    reference itself cannot be built here, DESIGN.md section 5) on all host cores: built and allocated once,
    warm executions, then exactly ``--steps`` timed executions of a bounded sample of the workload."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    world = args.gpus
    steps = max(1, args.steps)
    # the sample is sized so that warm-up + exactly ``steps`` timed executions take about two minutes
    sample = CpuSample(args.config, target_seconds=min(8.0, max(0.4, 110.0 / (steps + max(1, args.warmup)))))
    for _ in range(max(0, args.warmup - 1)):           # CpuSample already ran one warm execution
        sample.run()
    times = [sample.run() for _ in range(steps)]
    dt = float(np.mean(times))
    value = sample.updates / dt
    name, prog, _ = build_config(args.config, scale_i=world if args.scaling == "weak" else 1)
    config = common_config(args.config, prog, world, args.scaling)
    sample_text = sample.describe(len(times))
    if world > 1:
        config["reference_sample"] = sample_text        # the CPU arm times one bounded sample whatever N is
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world,
        "steps": len(times), "warmup": args.warmup, "ms_per_step": 1e3 * dt,
        "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None,
        "dtype": "f64" if "float64" in json.dumps(prog["program"]) else "f32", "data": "synthetic",
        "config": config,
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": sample.cores, "kind": "port", "sample": sample_text},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def workload_name(index, prog):
    dims = "x".join(map(str, prog["dimensions"]))
    nops = len(prog["program"])
    dt = next(iter(prog["program"].values()))["data_type"]
    kinds = {0: "Jacobi-3D chain", 1: "Jacobi-3D chain", 2: "COSMO hdiff", 3: "Jacobi-2D chain", 4: "Jacobi-3D chain"}
    tag = {"jki": ", layout J,K,I", "w1d": ", x 1-D weight w[k] per stage"}.get(VARIANT, "")
    return "{} {} {}, {} chained operators (BASELINE.json configs[{}]{})".format(kinds[index], dims, dt, nops, index, tag)


# ------------------------------------------------------------------------------------ GPU arm


def make_program(index, world, rank, local_rank, comm, scaling):
    from stencilflow_b200 import programs
    from stencilflow_b200.cuda_program import CudaProgram
    name, prog, halo = build_config(index, scale_i=world if scaling == "weak" else 1)
    path = programs.write_program(prog, name, programs.scratch_dir())
    if world > 1:
        from stencilflow_b200 import distributed
        program = distributed.SlabProgram(path, comm, device=local_rank)
    else:
        program = CudaProgram(path, device=local_rank)
    fill_inputs(program, index_offsets=getattr(program, "input_index_offsets", lambda: None)())
    return name, prog, path, program


def time_device(program, steps, warmup, comm, sampler=None):
    """``steps`` executions bracketed by a barrier + stream synchronisation on both sides, timed with
    CUDA events on the launch stream.  Returns (ms of this rank, max over ranks, launches)."""
    rtm = program.rt

    def barrier():
        rtm.stream_synchronize()
        if comm is not None:
            comm.barrier()

    for _ in range(warmup):
        program.execute()
    barrier()
    if sampler is not None:
        sampler.start()
    try:
        launches0 = program.launch_count
        e0, e1 = rtm.event_create(), rtm.event_create()
        barrier()
        rtm.event_record(e0)
        for _ in range(steps):
            program.execute()
        rtm.event_record(e1)
        rtm.event_synchronize(e1)
        barrier()
    except BaseException:
        if sampler is not None:
            sampler.stop()                  # no nvidia-smi left running behind a failed run
        raise
    ms_local = rtm.elapsed_ms(e0, e1)
    rtm.event_destroy(e0)
    rtm.event_destroy(e1)
    ms = comm.max_float(ms_local) if comm is not None else ms_local
    time_device.per_rank_ms = comm.allgather(ms_local) if comm is not None else [ms_local]
    return ms_local, ms, program.launch_count - launches0


def slab_checksums(program, field, bounds):
    """Bit checksums of ``field`` per plane range [b, e) of a single-GPU program."""
    f = program.program.fields[field]
    plane = int(np.prod(f.shape[1:]))
    out = []
    for (b, e) in bounds:
        out.append(program.rt.checksum(program.buffers[field].dptr + b * plane * f.data_type.bytes,
                                       (e - b) * plane, f.data_type.type)[1])
    return out


def verify_single(program, prog, path, index, local_rank, planes=128):
    """Checks the result the timed executions left in HBM (one GPU):
    ``oracle_block``: the first ``planes`` planes against the CPU oracle (the reference's program
    restated in C++), run on the leading block of the same synthetic input -- cells whose dependence cone
    stays inside the block; tolerance 1e-5 (float32) / 1e-12 (float64), BASELINE.json;
    ``fused_vs_general``: the whole result against the one-operator-per-launch kernels, compared on the
    device (``sfb_compare``)."""
    from oracle import reference_cpp, reference_numpy as rn
    from stencilflow_b200.cuda_program import CudaProgram
    from stencilflow_b200.planner import PlanOptions
    rtm = program.rt
    fields = program.program.fields
    out_name = program.program.outputs[0]
    f_out = fields[out_name]
    dims = list(prog["dimensions"])
    nops = len(prog["program"])
    result = {}
    # -- CPU oracle on a leading block
    t0 = time.perf_counter()
    reach = nops * 2                                  # generous bound on the accumulated extent along i
    block = min(dims[0], planes + reach)
    keep = planes if block < dims[0] else dims[0]
    sub = json.loads(json.dumps(prog))
    sub["dimensions"] = [block] + dims[1:]
    ref = reference_cpp.CompiledReference(sub, build_dir=oracle_build_dir())
    ins = host_inputs(prog, sub["dimensions"])
    expected = ref(**ins)[out_name]
    plane = int(np.prod(f_out.shape[1:]))
    got = np.empty((keep,) + tuple(f_out.shape[1:]), dtype=f_out.data_type.type)
    rtm.d2h(got, program.buffers[out_name].dptr, nbytes=keep * plane * f_out.data_type.bytes)
    rtm.stream_synchronize()
    halo = {2: 2, 3: 16}.get(index, 0)                # shrink boundaries: junk border excluded (-halo)
    a, b = expected[:keep], got
    if halo:
        # -halo trims every axis (stencilflow/run_program.py:202-209); the block's far side is cut off anyway
        sl = (slice(halo, None),) + tuple(slice(halo, -halo) for _ in range(a.ndim - 1))
        a, b = a[sl], b[sl]
    tol = 1e-12 if f_out.data_type.bytes == 8 else 1e-5
    err = float(rn.max_relative_error(a, b))
    result["oracle_block"] = {"planes": int(keep), "cells": int(a.size), "max_rel_err": err, "tolerance": tol,
                              "ok": bool(err <= tol), "seconds": round(time.perf_counter() - t0, 2)}
    del expected, got, ins
    # -- one-operator kernels, full size, compared on the device
    free_b, _ = rtm.mem_info()
    need = sum(f.nbytes for f in fields.values() if not f.is_scalar and f.kind != "intermediate") + 2 * f_out.nbytes
    if free_b > need + (2 << 30):
        general = CudaProgram(path, device=local_rank, plan_options=PlanOptions(fuse=False))
        for name, f in fields.items():
            if f.kind == "input" and not f.is_scalar:
                rtm.d2d(general.buffers[name].dptr, program.buffers[name].dptr, f.nbytes)
        general.scalar_values.update(program.scalar_values)
        general.execute()
        rtm.stream_synchronize()
        err, bad = rtm.compare(general.buffers[out_name].dptr, program.buffers[out_name].dptr,
                               f_out.size, f_out.data_type.type, tol)
        bits = (rtm.checksum(general.buffers[out_name].dptr, f_out.size, f_out.data_type.type)[1] ==
                rtm.checksum(program.buffers[out_name].dptr, f_out.size, f_out.data_type.type)[1])
        result["fused_vs_general"] = {"cells": int(f_out.size), "max_rel_err": float(err), "num_bad": int(bad),
                                      "bit_identical": bool(bits), "ok": bool(bad == 0)}
        general.close()
    else:
        result["fused_vs_general"] = {"skipped": "not enough free HBM for a second set of fields"}
    result["ok"] = all(v.get("ok", True) for v in result.values() if isinstance(v, dict))
    return result


def verify_multi(program, prog, path, comm, local_rank):
    """N > 1: the exchanged slab run against ONE GPU running the whole domain with the same plan
    (rank 0 does that), owned planes of every rank compared through bit checksums computed on the
    devices -- halo exchange, storage reuse and counters have to be exactly right for this to match."""
    from stencilflow_b200.cuda_program import CudaProgram
    rank = comm.rank
    out_name = program.program.outputs[0]
    mine = program.checksum_owned(out_name)[1]
    bounds = comm.allgather((program.slab.begin, program.slab.end))
    sums = comm.allgather(mine)
    result = None
    if rank == 0:
        fields = program.program.fields
        free_b, _ = program.rt.mem_info()
        need = 4 * max(f.nbytes for f in fields.values() if not f.is_scalar)
        if free_b > need + (2 << 30):
            single = CudaProgram(path, device=local_rank)
            fill_inputs(single)
            single.execute()
            single.rt.stream_synchronize()
            ref = slab_checksums(single, out_name, bounds)
            single.close()
            same = [int(a) == int(b) for a, b in zip(ref, sums)]
            result = {"single_gpu_whole_domain": "x".join(map(str, prog["dimensions"])),
                      "slabs_bit_identical": same, "ok": bool(all(same))}
        else:
            result = {"skipped": "whole domain does not fit one GPU next to the slab", "ok": True}
    comm.barrier()
    return result


def strong_block(args, world, rank, local_rank, comm, peak_gbs):
    """BASELINE.json configs[4] -- Jacobi-3D 2048^3 float32, 64 chained operators -- split into slabs
    over the N GPUs of this run, and on ONE GPU of the same box right after it (rank 0), so that the
    parallel efficiency t1 / (N * tN) comes from one lease.  The multi-GPU result is compared bit for
    bit with the one-GPU result (per-slab checksums)."""
    from stencilflow_b200.cuda_program import CudaProgram
    steps, warmup = 3, 3
    name, prog, path, program = make_program(4, world, rank, local_rank, comm, "strong")
    nops = len(prog["program"])
    updates = nops * float(np.prod(prog["dimensions"]))
    ms_local, ms, _ = time_device(program, steps, warmup, comm)
    out = {"workload": workload_name(4, prog), "n_gpus": world, "steps": steps, "warmup": warmup,
           "ms_per_step": ms / steps, "value": updates / (ms / steps * 1e-3), "unit": UNIT}
    alg = program.plan.algorithmic_bytes() / world
    out["roofline_frac"] = alg / (ms_local / steps * 1e-3) / 1e9 / peak_gbs
    out["launches_per_step"] = program.launches_per_execution
    if world > 1:
        out_name = program.program.outputs[0]
        # checksums of the state after exactly warmup + steps executions
        mine = program.checksum_owned(out_name)[1]
        bounds = comm.allgather((program.slab.begin, program.slab.end))
        sums = comm.allgather(mine)
        program.close()
        if rank == 0:
            single = CudaProgram(path, device=local_rank)
            fill_inputs(single)
            ms1_local, ms1, _ = time_device(single, steps, warmup, None)
            ref = slab_checksums(single, out_name, bounds)
            single.close()
            t1 = ms1 / steps
            out["one_gpu_ms_per_step"] = t1
            out["parallel_efficiency"] = t1 / (world * out["ms_per_step"])
            out["slabs_bit_identical_to_one_gpu"] = bool(all(int(a) == int(b) for a, b in zip(ref, sums)))
        comm.barrier()
    else:
        out["one_gpu_ms_per_step"] = out["ms_per_step"]
        out["parallel_efficiency"] = 1.0
        program.close()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100,
                    help="timed executions of the program, at least 1 (default 100: long enough for the clock "
                         "sampler to see the load and for the power cap to show)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--config", type=int, default=1, help="index into BASELINE.json configs")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--scaling", default=None, choices=["weak", "strong"],
                    help="N > 1: weak = every rank owns one copy of the config's domain (default for "
                         "configs 1-3); strong = the config's domain is split (default for config 4, "
                         "the 2048^3 x 64 slab-split case of BASELINE.json)")
    ap.add_argument("--variant", default=None, choices=["jki", "w1d"],
                    help="secondary form of a config (SURVEY 8d): jki = config 2 in the reference's COSMO "
                         "layout J,K,I (1024x80x1024); w1d = config 3 with a 1-D weight w[k] in every stage")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-verify", action="store_true")
    ap.add_argument("--no-strong", action="store_true",
                    help="skip the configs[4] strong-scaling block (default: measured when --config 1)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the program's output fields as DIR/<field>.npy "
                         "(fields above 32 MB as a fixed seeded sample; shrink borders cut off), so that "
                         "two builds can be compared output for output; --impl ours with one GPU only")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or args.gpus != 1):
        ap.error("--dump-outputs needs --impl ours and --gpus 1")
    global VARIANT
    VARIANT = args.variant
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    if args.scaling is None:
        args.scaling = "strong" if args.config == 4 else "weak"

    if args.impl == "reference":
        run_reference_arm(args)
        return

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            # convenience: re-launch ourselves under torchrun
            cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1",
                   "--nproc-per-node", str(args.gpus), "--master-addr", "127.0.0.1",
                   "--master-port", str(29500 + os.getpid() % 1000), os.path.abspath(__file__)] + sys.argv[1:]
            sys.exit(subprocess.call(cmd))
        raise SystemExit("WORLD_SIZE={} does not match --gpus {}".format(world, args.gpus))

    from stencilflow_b200 import build
    build.build_native()

    comm = None
    if world > 1:
        from stencilflow_b200 import distributed
        comm = distributed.make_comm()

    name, prog, path, program = make_program(args.config, world, rank, local_rank, comm, args.scaling)
    peak_gbs, peak_src = load_peaks()
    rtm = program.rt

    cells_total = int(np.prod(prog["dimensions"]))
    nops = len(prog["program"])
    updates_per_step = nops * cells_total                      # whole job, all ranks
    local_fraction = 1.0 / world

    sampler = ClockSampler(local_rank) if rank == 0 else None
    ms_local, ms, launches = time_device(program, args.steps, args.warmup, comm, sampler)
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs:
        dump_outputs(program, args.dump_outputs, build_config(args.config)[2])
    per_rank_ms = [t / args.steps for t in time_device.per_rank_ms]
    ms_per_step = ms / args.steps
    value = updates_per_step / (ms_per_step * 1e-3)

    # roofline of the dominant kernel: algorithmic bytes of one launch / its mean duration.
    # All launches of a step are stencil passes on one stream, so the mean launch duration is
    # (event-timed step) / (launches per step).
    alg_bytes_step = program.plan.algorithmic_bytes() * (1.0 if world == 1 else local_fraction)
    lps = program.launches_per_execution
    achieved = alg_bytes_step / (ms_local / args.steps * 1e-3) / 1e9
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.isfile(tpath):
        with open(tpath) as f:
            rec = json.load(f).get(str(args.config), {})
            # the ncu capture only describes the kernel it was taken from
            if rec.get("kernel") == program.lowered.launches[0].kernel and world == 1:
                traffic = rec.get("dram_bytes_per_launch")
    # fusion-independent companion figure (SURVEY 8d): the program's minimum off-chip volume
    # (every input read once, every output written once) over the same time
    fields = program.program.fields
    min_volume = sum(f.nbytes for f in fields.values() if f.kind in ("input", "output") and not f.is_scalar)
    min_volume *= (1.0 if world == 1 else local_fraction)
    l0 = program.lowered.launches[0]
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peak_gbs, "unit": "GB/s",
                "frac": achieved / peak_gbs, "traffic": traffic, "peak_source": peak_src,
                "algorithmic_bytes_per_launch": alg_bytes_step / lps, "launches_per_step": lps,
                "operators_per_launch": [len(l.ops) for l in program.lowered.launches],
                "min_volume_frac": min_volume / (ms_local / args.steps * 1e-3) / 1e9 / peak_gbs,
                "kernel": l0.kernel, "family": l0.family,
                "schedule": ("persistent CTAs, work list" if l0.info.get("persistent") else "one CTA per (tile, chunk)")
                if l0.family == "streamed" else "grid over cells"}

    # the result the timed executions left behind is checked before anything overwrites it
    verify = None
    if not args.no_verify:
        if world == 1:
            verify = verify_single(program, prog, path, args.config, local_rank)
        else:
            verify = verify_multi(program, prog, path, comm, local_rank)

    # end to end through the plugin call with host buffers, copies inside the timed region
    e2e = None
    if not args.no_e2e:
        e2e = measure_e2e(program, prog, args, updates_per_step, comm)

    plan_desc = [{"family": l.family, "ops": len(l.ops)} for l in program.lowered.launches]
    program.close()

    strong = None
    if args.config == 1 and not args.no_strong and VARIANT is None:
        strong = strong_block(args, world, rank, local_rank, comm, peak_gbs)

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        rate, cores, sample = cpu_reference_rate(args.config)
        cpu = {"value": rate, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample}

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_per_step, "ms_per_step_per_rank": per_rank_ms,
            "higher_is_better": True,
            "scaling": args.scaling, "vs_baseline": None,
            "dtype": "f64" if "float64" in json.dumps(prog["program"]) else "f32",
            "data": "synthetic",
            "config": common_config(args.config, prog, world, args.scaling),
            "plan": plan_desc,
            "roofline": roofline, "cpu_baseline": cpu, "clocks": clocks, "e2e": e2e,
            "verify": verify, "strong": strong,
            "gpu_launches": launches,
        }
        print(json.dumps(line), flush=True)
    if comm is not None:
        comm.close()


def pcie_duplex_rate(rtm, nbytes=1 << 30):
    """Measured ceiling of the end-to-end call: host->device and device->host copies of ``nbytes`` each
    running concurrently on two streams from pinned memory (GB/s per direction)."""
    a, pa = rtm.host_alloc((nbytes,), np.uint8)
    b, pb = rtm.host_alloc((nbytes,), np.uint8)
    d0, d1 = rtm.malloc(nbytes), rtm.malloc(nbytes)
    s0, s1 = rtm.stream_create(), rtm.stream_create()
    best = 0.0
    for it in range(3):
        rtm.stream_synchronize(s0)
        rtm.stream_synchronize(s1)
        t0 = time.perf_counter()
        rtm.h2d(d0, a, stream=s0)
        rtm.d2h(b, d1, stream=s1)
        rtm.stream_synchronize(s0)
        rtm.stream_synchronize(s1)
        dt = time.perf_counter() - t0
        if it:
            best = max(best, nbytes / dt / 1e9)
    rtm.free(d0)
    rtm.free(d1)
    rtm.host_free(pa)
    rtm.host_free(pb)
    return best


def measure_e2e(program, prog, args, updates_per_step, comm=None):
    """Same metric through the reference-facing call with HOST buffers: every step copies this rank's
    inputs host->device, runs the program and copies its outputs back (``CudaProgram.__call__`` on one
    GPU; the slab-wise equivalent on several).  Wall-clock, max over ranks.  The figure of record uses
    pinned host memory (``sfb_host_alloc``), as the bench contract specifies; ``numpy_arrays`` repeats it
    with plain numpy arrays, as the reference's driver allocates them (``run_program.py:145-159``) -- the
    call page-locks those on first use (``sfb_host_register``)."""
    rtm = program.rt
    fields = program.program.fields

    def allocate(pinned):
        host_in, host_out, free_host = {}, {}, []
        for name, f in fields.items():
            if f.is_scalar or f.kind == "intermediate":
                continue
            shape = program.local_shape(name)
            if pinned:
                arr, hptr = rtm.host_alloc(shape, f.data_type.type)
                free_host.append(hptr)
            else:
                arr = np.empty(shape, dtype=f.data_type.type)
            if f.kind == "input":
                rtm.d2h(arr, program.buffers[name].dptr)         # reuse the synthetic field as host data
                rtm.stream_synchronize()
                host_in[name] = arr
            else:
                host_out[name] = arr
        return host_in, host_out, free_host

    steps = max(2, min(args.steps, 5))

    def timed(host_in, host_out):
        kw = {k + "_host": v for k, v in host_in.items()}
        kw.update({k + "_host": v for k, v in host_out.items()})
        program(**kw)                                            # warm (page-locks numpy arrays once)
        if comm is not None:
            comm.barrier()
        t0 = time.perf_counter()
        for _ in range(steps):
            # the reference-facing call: CudaProgram.__call__ / SlabProgram.__call__ with host arrays
            program(**kw)
        rtm.stream_synchronize()
        dt = (time.perf_counter() - t0) / steps
        h2d = sum(a.nbytes for a in host_in.values())
        d2h = sum(a.nbytes for a in host_out.values())
        copied = getattr(program, "last_call_bytes", None)
        if copied:                                               # bytes the call actually moved per step
            h2d, d2h = int(copied[0]), int(copied[1])
        if comm is not None:
            dt = comm.max_float(dt)
            h2d = int(sum(comm.allgather(h2d)))
            d2h = int(sum(comm.allgather(d2h)))
        return dt, h2d, d2h

    host_in, host_out, _ = allocate(False)
    dt_numpy, _, _ = timed(host_in, host_out)
    del host_in, host_out
    host_in, host_out, free_host = allocate(True)
    dt, h2d, d2h = timed(host_in, host_out)
    for hptr in free_host:
        rtm.host_free(hptr)
    link = pcie_duplex_rate(rtm) if comm is None else None
    out = {"value": updates_per_step / dt, "unit": UNIT, "h2d_bytes_per_step": h2d,
           "d2h_bytes_per_step": d2h, "ms_per_step": dt * 1e3, "steps": steps,
           "host_memory": "pinned (sfb_host_alloc = cudaHostAlloc), as the bench contract asks",
           "numpy_arrays": {"value": updates_per_step / dt_numpy, "ms_per_step": dt_numpy * 1e3,
                            "host_memory": "plain numpy arrays as the reference's driver allocates them (run_program.py:"
                                           "145-159): pageable when handed over, page-locked by the call on first use"}}
    if link:
        # both directions run concurrently, so the call cannot be faster than its larger direction
        world = 1 if comm is None else comm.world
        floor = max(h2d, d2h) / world / (link * 1e9)
        out["roofline"] = {"bound": "pcie", "peak": link, "unit": "GB/s per direction, H2D and D2H concurrently",
                           "achieved": max(h2d, d2h) / world / dt / 1e9, "frac": floor / dt}
    return out


if __name__ == "__main__":
    with scratch_cache():
        main()

"""Parity tests proper: the CUDA path (through the C-ABI) against the oracle on the same seeded
inputs.  Tolerances are the north-star ones: max relative error 1e-5 for float32 results and 1e-12
for float64 results, the -halo border excluded for shrink boundaries."""
import json
import os

import numpy as np
import pytest

from conftest import GOLDEN, HALO, ROOT, all_programs, program_path, random_inputs

pytestmark = pytest.mark.gpu

TOL = {"float32": 1e-5, "float64": 1e-12}


@pytest.fixture(scope="module")
def gpu(native_lib):
    from stencilflow_b200 import runtime
    return runtime.Runtime.get()


def _run_cuda(name, inputs, plan_options=None):
    from stencilflow_b200.cuda_program import CudaProgram
    from oracle import reference_numpy as rn
    prog = CudaProgram(program_path(name), plan_options=plan_options)
    info = rn.ProgramInfo(rn.load_program(program_path(name)))
    outs = {o: np.zeros(info.shape, dtype=info.field_type(o)) for o in info.outputs}
    args = {}
    for k, v in inputs.items():
        args[k + "_host" if getattr(v, "ndim", 0) > 0 else k] = v
    for k, v in outs.items():
        args[k + "_host"] = v
    prog(**args)
    prog.close()
    return outs, prog


def _check(name, got, expected):
    from oracle import reference_numpy as rn
    h = HALO.get(name, 0)
    for field, ref in expected.items():
        err = rn.max_relative_error(rn.trim_halo(ref, h), rn.trim_halo(got[field], h))
        assert err <= TOL[ref.dtype.name], "{}:{} max rel err {}".format(name, field, err)


@pytest.mark.parametrize("name", all_programs())
def test_program_matches_oracle_general(gpu, name):
    """Every program, every operator as its own launch (fusion off)."""
    from oracle import reference_numpy as rn
    from stencilflow_b200.planner import PlanOptions
    inputs = random_inputs(name)
    expected = rn.run_reference(program_path(name), inputs)
    got, _ = _run_cuda(name, inputs, PlanOptions(fuse=False))
    _check(name, got, expected)


@pytest.mark.parametrize("name", all_programs())
def test_program_matches_oracle_planned(gpu, name):
    """Every program with the planner's default choice (fused passes where streamable)."""
    from oracle import reference_numpy as rn
    inputs = random_inputs(name, seed=11)
    expected = rn.run_reference(program_path(name), inputs)
    got, _ = _run_cuda(name, inputs)
    _check(name, got, expected)


@pytest.mark.parametrize("name", all_programs())
def test_program_matches_oracle_fused(gpu, name):
    """Every program with fusion requested (``max_depth=8``: the longest streamable runs of up to eight
    operators, whatever the cost model would say about grids this small)."""
    from oracle import reference_numpy as rn
    from stencilflow_b200.planner import PlanOptions
    inputs = random_inputs(name, seed=17)
    expected = rn.run_reference(program_path(name), inputs)
    got, _ = _run_cuda(name, inputs, PlanOptions(max_depth=8))
    _check(name, got, expected)


@pytest.mark.parametrize("name", [n for n in all_programs() if n.startswith("ref_")])
def test_reference_programs_match_known_answers(gpu, name):
    """The reference's own programs with their own inputs against the frozen known answers."""
    from oracle import reference_numpy as rn
    with open(os.path.join(GOLDEN, "known_answers.json")) as f:
        known = json.load(f)[name]
    inputs = rn.materialize_inputs(rn.load_program(program_path(name)))
    got, _ = _run_cuda(name, inputs)
    for field, rec in known.items():
        tol = TOL[rec["dtype"]]
        arr = got[field]
        assert abs(float(arr.sum(dtype=np.float64)) - rec["sum"]) <= 10 * tol * max(1.0, abs(rec["sum"]))
        if "values" in rec:
            assert rn.max_relative_error(np.array(rec["values"], dtype=arr.dtype), arr) <= tol
        for point, value in rec.get("points", []):
            assert abs(float(arr[tuple(point)]) - value) <= tol * max(1.0, abs(value))


with open(os.path.join(GOLDEN, "reference_sim.json")) as _f:
    REFERENCE_SIM = json.load(_f)


@pytest.mark.parametrize("fuse", [True, False], ids=["planned", "unfused"])
@pytest.mark.parametrize("case", sorted(REFERENCE_SIM))
def test_cuda_matches_reference_simulator(gpu, case, fuse):
    """The CUDA path against OUTPUTS OF THE REFERENCE ITSELF: its dataflow simulator run in the build
    container on the same program and inputs (tests/golden/reference_sim.npz, generator
    make_reference_sim_golden.py).  No oracle in between."""
    import sys
    if GOLDEN not in sys.path:
        sys.path.insert(0, GOLDEN)
    import make_reference_sim_golden as gen
    from oracle import reference_numpy as rn
    from stencilflow_b200.planner import PlanOptions
    rec = REFERENCE_SIM[case]
    inputs = gen.case_inputs(gen.case_program(rec["program"]), rec["seed"], rec.get("ranges"))
    got, _ = _run_cuda(rec["program"], inputs, None if fuse else PlanOptions(fuse=False))
    h = rec.get("halo", 0)          # shrink programs: the simulator ran them as constant -100000, interiors compared
    with np.load(os.path.join(GOLDEN, "reference_sim.npz")) as z:
        for field in rec["outputs"]:
            ref = z[case + "/" + field]
            assert got[field].dtype == ref.dtype
            err = rn.max_relative_error(rn.trim_halo(ref, h), rn.trim_halo(got[field], h))
            assert err <= TOL[ref.dtype.name], (case, field, err)


@pytest.mark.parametrize("name,halo", [(n, 0) for n in all_programs() if n.startswith("ref_")] +
                         [("hdiff_24x28x16", 2), ("jacobi2d_96x128_6itr_shrink_f64", 6),
                          ("upwind3d_fwd_24x16x32_4st", 0)])
def test_run_program_compare_to_reference(gpu, name, halo, tmp_path, monkeypatch):
    """`run_program.py prog.json cuda -compare-to-reference` end to end (drop-in driver), for every
    program of the reference's test/stencils (the north-star target: each of them verifies in cuda mode,
    as ``test/test_stencilflow.py:191-216`` requires of emulation mode) and two shrink programs with -halo."""
    from stencilflow_b200.run_program import run_program
    monkeypatch.chdir(tmp_path)
    ret = run_program(program_path(name), "cuda", compare_to_reference=True, halo=halo, log_level=0,
                      input_directory=os.path.dirname(program_path(name)))
    assert ret == 0
    base = os.path.splitext(os.path.basename(program_path(name)))[0].replace(".", "_")
    assert os.path.isdir(tmp_path / "results" / base / "reference")


@pytest.mark.parametrize("name,halo,compare", [("ref_simulator12", 0, False), ("ref_jacobi2d_128x128", 0, True),
                                               ("hdiff_16x20x8_f64", 2, True), ("ref_varying_dimensionality", 0, False)])
def test_run_program_with_simulation(gpu, name, halo, compare, tmp_path, monkeypatch, capsys):
    """`run_program.py prog.json cuda -run-simulation`: the dataflow simulator's result is compared with
    the device result (reference run_program.py:48-61,232-250)."""
    from stencilflow_b200.run_program import run_program
    monkeypatch.chdir(tmp_path)
    ret = run_program(program_path(name), "cuda", run_simulation=True, compare_to_reference=compare, halo=halo,
                      log_level=0, input_directory=os.path.dirname(program_path(name)))
    assert ret == 0
    out = capsys.readouterr().out
    assert "Comparing simulation results..." in out and "Results verified." in out


def test_mismatch_is_detected(gpu, tmp_path, monkeypatch):
    from stencilflow_b200 import run_program as rp
    monkeypatch.chdir(tmp_path)
    monkeypatch.setattr(rp, "tolerance_for", lambda dtype: -1.0)
    with pytest.raises(ValueError, match="Result mismatch"):
        rp.run_program(program_path("ref_simulator3"), "cuda", compare_to_reference=True, log_level=0)


def test_generate_input_and_repetitions(gpu, tmp_path, monkeypatch):
    from stencilflow_b200.run_program import run_program
    monkeypatch.chdir(tmp_path)
    assert run_program(program_path("ref_jacobi2d_128x128"), "cuda", compare_to_reference=True,
                       generate_input=True, repetitions=3, log_level=0) == 0
    assert run_program(program_path("ref_varying_dimensionality"), "cuda", compare_to_reference=True,
                       specialize_scalars=True, log_level=0) == 0
    assert run_program(program_path("ref_jacobi2d_128x128"), "cuda", compare_to_reference=True,
                       synthetic_reads=0.75, log_level=0) == 0


def test_device_utilities(gpu):
    """fill_hash is bit-identical to its host mirror; checksum/compare agree with numpy."""
    from stencilflow_b200 import synthetic
    n = 1 << 20
    for dt in (np.float32, np.float64):
        d = gpu.malloc(n * np.dtype(dt).itemsize)
        gpu.fill_hash(d, n, dt, seed=1234, lo=-1.0, hi=3.0, index_offset=5)
        host = np.empty(n, dtype=dt)
        gpu.d2h(host, d)
        gpu.stream_synchronize()
        mirror = synthetic.fill_hash((n,), dt, 1234, -1.0, 3.0, 5)
        assert np.array_equal(host, mirror)
        s, bits = gpu.checksum(d, n, dt)
        assert abs(s - float(host.sum(dtype=np.float64))) <= 1e-9 * n
        words = host.view(np.uint32 if dt == np.float32 else np.uint64).astype(np.uint64)
        assert bits == int(words.sum(dtype=np.uint64))
        d2 = gpu.malloc(n * np.dtype(dt).itemsize)
        other = host.copy()
        other[12345] *= dt(1.001)
        gpu.h2d(d2, other)
        m, bad = gpu.compare(d, d2, n, dt, 1e-5)
        assert bad == 1 and abs(m - 1e-3) < 2e-4
        gpu.free(d)
        gpu.free(d2)
    # indices beyond 2^32 use the high word
    a = synthetic.fill_hash((4,), np.float32, 1, index_offset=(1 << 33))
    b = synthetic.fill_hash((4,), np.float32, 1, index_offset=0)
    assert not np.array_equal(a, b)


def test_bench_dump_outputs_match_oracle(gpu, tmp_path):
    """``bench.py --dump-outputs`` writes what exactly ``--steps`` timed executions of BASELINE configs[0]
    computed; it equals the oracle on the same seeded inputs."""
    import subprocess
    import sys
    import bench
    from oracle import reference_numpy as rn
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--config", "0", "--steps", "2",
                          "--no-cpu-baseline", "--no-e2e", "--dump-outputs", str(tmp_path / "dump")],
                         stdout=subprocess.PIPE, text=True, timeout=600, check=True).stdout
    line = json.loads(out.strip().splitlines()[-1])
    assert line["steps"] == 2 and line["gpu_launches"] == 2 * line["roofline"]["launches_per_step"]
    assert line["verify"]["ok"]
    _, prog, _ = bench.build_config(0)
    expected = rn.run_reference(prog, bench.host_inputs(prog, prog["dimensions"]))
    for field, ref in expected.items():
        got = np.load(tmp_path / "dump" / (field + ".npy"))
        assert got.dtype == ref.dtype and got.shape == ref.shape
        assert rn.max_relative_error(ref, got) <= TOL[ref.dtype.name], field


def test_size_independent_properties_at_scale(gpu):
    """256^3 x 8 chained Jacobi on hash-generated input, checked by properties that do not need the
    oracle to hold nine 256^3 arrays: linearity and agreement of fused vs unfused execution."""
    from stencilflow_b200.cuda_program import CudaProgram
    from stencilflow_b200.planner import PlanOptions
    from stencilflow_b200 import programs, synthetic
    path = programs.write_program(programs.jacobi3d_chain([256, 256, 256], 8), "jacobi3d_256_8itr")
    n = 256 ** 3
    results = []
    for opts in (PlanOptions(fuse=False), None):
        p = CudaProgram(path, plan_options=opts)
        p.rt.fill_hash(p.buffers["a"].dptr, n, np.float32, seed=1234)
        p.execute()
        results.append(p.download("b7"))
        p.close()
    from oracle import reference_numpy as rn
    assert rn.max_relative_error(results[0], results[1]) <= 1e-5
    # oracle on a 64^3 corner problem with the same generator: exact same program at reduced size
    small = programs.write_program(programs.jacobi3d_chain([64, 64, 64], 8), "jacobi3d_64_8itr")
    a = synthetic.fill_hash((64, 64, 64), np.float32, 1234)
    expected = rn.run_reference(small, {"a": a})["b7"]
    p = CudaProgram(small)
    out = np.zeros((64, 64, 64), np.float32)
    p(a_host=a, b7_host=out)
    p.close()
    assert rn.max_relative_error(expected, out) <= 1e-5


PLAN_VARIANTS = [
    # (max_depth, rows_per_thread, warps, vector): every CTA shape / fusion depth the planner or the
    # tuner may pick, forced here on small programs so that each code shape is checked against the oracle
    (1, 4, 16, 0), (2, 4, 16, 0), (2, 3, 12, 0), (3, 4, 12, 0), (4, 4, 8, 0), (4, 2, 16, 0), (3, 1, 8, 0),
    (8, 2, 8, 0),
    # rows of 16 / 8 threads (two / four row groups per warp)
    (2, 4, 8, 0, 16), (4, 4, 8, 0, 16), (3, 2, 12, 0, 16), (2, 3, 8, 0, 8),
]


@pytest.mark.parametrize("variant", PLAN_VARIANTS, ids=lambda v: "d{}r{}w{}v{}".format(*v[:4]) + ("" if len(v) < 5 else "k{}".format(v[4])))
@pytest.mark.parametrize("name", ["ref_jacobi3d_32x32x32_8itr_8vec", "jacobi3d_16x24x32_5itr_const1",
                                  "jacobi3d_24x20x40_4itr_shrink_f64", "hdiff_24x28x16", "fork_join_20x16x24",
                                  "box3d_10x12x16"])
def test_plan_variants_3d(gpu, name, variant):
    from oracle import reference_numpy as rn
    from stencilflow_b200.planner import PlanOptions
    d, r, w, v = variant[:4]
    ks = variant[4] if len(variant) > 4 else 0
    inputs = random_inputs(name, seed=23)
    expected = rn.run_reference(program_path(name), inputs)
    got, prog = _run_cuda(name, inputs, PlanOptions(max_depth=d, rows_per_thread=r, warps=w, vector=v,
                                                    threads_per_row=ks))
    _check(name, got, expected)


@pytest.mark.parametrize("variant", [(1, 8, 0), (2, 8, 0), (4, 8, 0), (6, 16, 0), (4, 8, 4), (2, 16, 8), (3, 8, 8)],
                         ids=lambda v: "d{}w{}v{}".format(*v))
@pytest.mark.parametrize("name", ["jacobi2d_96x128_6itr_shrink_f64", "jacobi2d_64x64_4itr_const_f32",
                                  "ref_jacobi2d_128x128", "wide2d_8x2048_5itr_f64", "wide2d_6x4096_4itr_f32"])
def test_plan_variants_2d(gpu, name, variant, tmp_path):
    """2-D programs: fusion depths, CTA widths and cells per thread (the wide programs are there so
    that several CTAs and the longer per-thread runs actually occur)."""
    from oracle import reference_numpy as rn
    from stencilflow_b200 import programs
    from stencilflow_b200.cuda_program import CudaProgram
    from stencilflow_b200.planner import PlanOptions
    d, w, v = variant
    if name.startswith("wide2d"):
        dims = {"wide2d_8x2048_5itr_f64": ([8, 2048], 5, "float64"), "wide2d_6x4096_4itr_f32": ([6, 4096], 4, "float32")}[name]
        prog = programs.jacobi2d_chain(dims[0], dims[1], dtype=dims[2])
        path = str(tmp_path / (name + ".json"))
        with open(path, "w") as f:
            json.dump(prog, f)
        rng = np.random.default_rng(5)
        inputs = {"a": rng.random(dims[0]).astype(dims[2])}
        halo = dims[1]
    else:
        path = program_path(name)
        inputs = random_inputs(name, seed=29)
        halo = HALO.get(name, 0)
    expected = rn.run_reference(path, inputs)
    p = CudaProgram(path, plan_options=PlanOptions(max_depth=d, warps=w, vector=v))
    info = rn.ProgramInfo(rn.load_program(path))
    outs = {o: np.zeros(info.shape, dtype=info.field_type(o)) for o in info.outputs}
    args = {k + "_host": val for k, val in inputs.items()}
    args.update({k + "_host": val for k, val in outs.items()})
    p(**args)
    p.close()
    for field, ref in expected.items():
        err = rn.max_relative_error(rn.trim_halo(ref, halo), rn.trim_halo(outs[field], halo))
        assert err <= TOL[ref.dtype.name], "{}:{} max rel err {}".format(name, field, err)


@pytest.mark.parametrize("kind", ["jacobi3d", "hdiff", "jacobi2d", "jacobi2d_w1d"])
def test_pipelined_host_call(gpu, kind, monkeypatch):
    """The host-array call cut into pieces (copies overlapping the passes) gives bit-identical
    results to the plain upload / execute / download sequence, and matches the oracle."""
    from oracle import reference_numpy as rn
    from stencilflow_b200 import programs, synthetic
    from stencilflow_b200.cuda_program import CudaProgram
    if kind == "jacobi3d":
        prog, halo = programs.jacobi3d_chain([192, 160, 256], 8), 0
        inputs = {"a": synthetic.fill_hash((192, 160, 256), np.float32, 1234)}
    elif kind == "hdiff":
        prog, halo = programs.hdiff([384, 256, 80]), 2
        inputs = {"inp": synthetic.fill_hash((384, 256, 80), np.float32, 1, 1.0, 2.0),
                  "coeff": synthetic.fill_hash((384, 256, 80), np.float32, 2, 0.0, 0.05)}
    elif kind == "jacobi2d":
        prog, halo = programs.jacobi2d_chain([2048, 4096], 6), 6
        inputs = {"a": synthetic.fill_hash((2048, 4096), np.float64, 7)}
    else:
        # a 1-D coefficient array next to the streamed field: it goes up whole with the first piece
        prog, halo = programs.jacobi2d_chain([2048, 4096], 6), 6
        prog["inputs"]["w"] = {"data": "constant:0.9", "data_type": "float64", "input_dims": ["k"]}
        for op in prog["program"].values():
            op["computation_string"] = op["computation_string"].replace("0.25 *", "0.25 * w[k] *")
            op["boundary_conditions"]["w"] = {"type": "shrink"}
        inputs = {"a": synthetic.fill_hash((2048, 4096), np.float64, 7),
                  "w": synthetic.fill_hash((4096,), np.float64, 8, 0.5, 1.5)}
    path = programs.write_program(prog, "pipelined_" + kind)
    info = rn.ProgramInfo(rn.load_program(path))
    results = []
    for pieces in ("0", "8"):
        monkeypatch.setenv("SFB200_PIPELINE_PIECES", pieces)
        p = CudaProgram(path)
        monkeypatch.setattr(p, "PIPELINE_MIN_BYTES", 1 << 20)
        outs = {o: np.zeros(info.shape, dtype=info.field_type(o)) for o in info.outputs}
        args = {k + "_host": v for k, v in inputs.items()}
        args.update({k + "_host": v for k, v in outs.items()})
        # first call with other data: the second call must not see anything stale on the device
        other = {k + "_host": (v * v.dtype.type(0.5) + v.dtype.type(0.25)) for k, v in inputs.items()}
        other.update({k + "_host": v for k, v in outs.items()})
        p(**other)
        p(**args)                                   # a second call reuses the schedule
        if pieces != "0":
            assert getattr(p, "_pipe", None) is not None, "the pipelined path was not taken"
        p.close()
        results.append(outs)
    for o in info.outputs:
        assert np.array_equal(results[0][o], results[1][o])
    expected = rn.run_reference(path, inputs)
    for field, ref in expected.items():
        err = rn.max_relative_error(rn.trim_halo(ref, halo), rn.trim_halo(results[1][field], halo))
        assert err <= TOL[ref.dtype.name]


@pytest.mark.parametrize("kind", ["jacobi3d_64ops", "jacobi2d_16ops_f64"])
def test_long_chains_match_oracle(gpu, kind):
    """The shapes of BASELINE configs 4 and 3 at sizes the oracle finishes in seconds: a 64-operator
    Jacobi-3D chain (16 passes of 4 operators with the plan of the benchmark, intermediates sharing two
    ping-pong buffers; float32 drift over 64 stages stays inside the tolerance) and the 16-operator float64
    2-D ``shrink`` chain on its tuned plan (2-warp CTAs, 8 operators per pass)."""
    from oracle import reference_numpy as rn
    from stencilflow_b200 import programs, synthetic
    from stencilflow_b200.cuda_program import CudaProgram
    from stencilflow_b200.planner import PlanOptions
    if kind == "jacobi3d_64ops":
        shape, halo = (112, 96, 128), 0
        prog = programs.jacobi3d_chain(list(shape), 64)
        inputs = {"a": synthetic.fill_hash(shape, np.float32, 4321)}
        opts = PlanOptions(max_depth=4, rows_per_thread=3, warps=12, prefetch=5)
        out = "b63"
    else:
        shape, halo = (4096, 8192), 16
        prog = programs.jacobi2d_chain(list(shape), 16)
        inputs = {"a": synthetic.fill_hash(shape, np.float64, 77)}
        opts = PlanOptions(max_depth=8, vector=4, warps=2, prefetch=5)
        out = "b15"
    path = programs.write_program(prog, "longchain_" + kind)
    p = CudaProgram(path, plan_options=opts)
    streamed = [l for l in p.lowered.launches if l.family == "streamed"]
    assert len(streamed) == (16 if kind == "jacobi3d_64ops" else 2)
    if kind == "jacobi3d_64ops":
        assert len(set(p.plan.buffer_assignment().values())) <= 4          # input, output, two ping-pong buffers
    got = np.zeros(shape, dtype=inputs["a"].dtype)
    p(a_host=inputs["a"], **{out + "_host": got})
    p.close()
    expected = rn.run_reference(path, inputs)[out]
    err = rn.max_relative_error(rn.trim_halo(expected, halo), rn.trim_halo(got, halo))
    assert err <= TOL[expected.dtype.name], err


PAIR_VARIANTS_3D = [
    # (max_depth, rows_per_thread, warps, threads per row, prefetch): neighbour-only synchronisation with
    # per-warp TMA staging, and deeper TMA rings under both synchronisation schemes
    (4, 4, 8, 16, 2, "pair"), (4, 4, 8, 32, 5, "pair"), (2, 4, 16, 32, 3, "pair"), (3, 3, 12, 16, 5, "pair"),
    (4, 2, 16, 16, 2, "pair"), (1, 4, 8, 32, 2, "pair"), (4, 4, 8, 16, 5, "cta"), (3, 4, 12, 32, 3, "cta"),
    # per-field mbarriers instead of the CTA-wide barrier ("flags"; falls back to the barrier where a ring is
    # read after it was re-published, e.g. the fork/join program)
    (4, 3, 12, 16, 5, "flags"), (4, 4, 8, 16, 2, "flags"), (2, 4, 16, 32, 3, "flags"), (3, 2, 16, 16, 2, "flags"),
    (1, 4, 8, 32, 2, "flags"),
    # two half-CTAs sharing the tile: own barrier and TMA boxes per half, producer/consumer handshake at the seam
    (4, 3, 12, 16, 5, "halves"), (4, 4, 8, 16, 2, "halves"), (2, 4, 16, 32, 3, "halves"), (3, 2, 16, 16, 2, "halves"),
    (1, 4, 8, 32, 2, "halves"),
]


@pytest.mark.parametrize("variant", PAIR_VARIANTS_3D, ids=lambda v: "d{}r{}w{}k{}p{}{}".format(*v))
@pytest.mark.parametrize("name", ["ref_jacobi3d_32x32x32_8itr_8vec", "jacobi3d_16x24x32_5itr_const1",
                                  "jacobi3d_24x20x40_4itr_shrink_f64", "fork_join_20x16x24", "box3d_10x12x16"])
def test_pair_sync_and_prefetch_3d(gpu, name, variant):
    from oracle import reference_numpy as rn
    from stencilflow_b200.planner import PlanOptions
    d, r, w, ks, p, sync = variant
    inputs = random_inputs(name, seed=31)
    expected = rn.run_reference(program_path(name), inputs)
    got, prog = _run_cuda(name, inputs, PlanOptions(max_depth=d, rows_per_thread=r, warps=w, threads_per_row=ks,
                                                    prefetch=p, sync=sync))
    _check(name, got, expected)


DIRECT_VARIANTS_3D = [
    # (max_depth, rows_per_thread, warps, threads per row, prefetch): neighbour rows of the streamed
    # input read straight from the TMA ring (PlanOptions.direct); the ring depth prefetch + 2 must
    # divide the unroll factor
    (4, 3, 12, 16, 4), (4, 4, 8, 16, 4), (2, 4, 8, 32, 1), (3, 2, 8, 16, 1), (1, 4, 8, 32, 1), (4, 4, 8, 32, 4),
]


@pytest.mark.parametrize("variant", DIRECT_VARIANTS_3D, ids=lambda v: "d{}r{}w{}k{}p{}x".format(*v))
@pytest.mark.parametrize("name", ["ref_jacobi3d_32x32x32_8itr_8vec", "fork_join_20x16x24", "box3d_10x12x16",
                                  "jacobi3d_16x24x32_5itr_const1"])
def test_direct_input_rows_3d(gpu, name, variant):
    """(jacobi3d_16x24x32_5itr_const1 has a non-zero boundary value: its input needs the fix-up, so the
    option must leave it on the exchange ring and still be correct.)"""
    from oracle import reference_numpy as rn
    from stencilflow_b200.planner import PlanOptions
    d, r, w, ks, p = variant
    inputs = random_inputs(name, seed=37)
    expected = rn.run_reference(program_path(name), inputs)
    got, prog = _run_cuda(name, inputs, PlanOptions(max_depth=d, rows_per_thread=r, warps=w, threads_per_row=ks,
                                                    prefetch=p, direct=1))
    _check(name, got, expected)
    streamed = [l for l in prog.lowered.launches if l.family == "streamed"]
    if name == "ref_jacobi3d_32x32x32_8itr_8vec" and streamed:
        assert any(l.info.get("direct") for l in streamed)


def test_direct_input_rows_bit_identical_at_scale(gpu):
    """Many CTAs and waves: reading the input's neighbour rows from the TMA ring must reproduce the
    exchange-ring kernel bit for bit (a slot recycled too early would show as a difference)."""
    from stencilflow_b200 import programs
    from stencilflow_b200.cuda_program import CudaProgram
    from stencilflow_b200.planner import PlanOptions
    prog = programs.jacobi3d_chain([320, 448, 512], 8)
    path = programs.write_program(prog, "direct_jacobi3d")
    n = int(np.prod(prog["dimensions"]))
    sums = []
    for opts in (dict(max_depth=4, rows_per_thread=3, warps=12, prefetch=4),
                 dict(max_depth=4, rows_per_thread=3, warps=12, prefetch=4, direct=1),
                 dict(max_depth=4, rows_per_thread=4, warps=8, prefetch=4, direct=1),
                 dict(max_depth=2, rows_per_thread=4, warps=8, threads_per_row=32, prefetch=1, direct=1)):
        p = CudaProgram(path, plan_options=PlanOptions(**opts))
        p.rt.fill_hash(p.buffers["a"].dptr, n, np.float32, seed=99)
        for _ in range(3):
            p.execute()
        p.rt.stream_synchronize()
        sums.append(p.rt.checksum(p.buffers["b7"].dptr, n, np.float32))
        p.close()
    assert all(s[1] == sums[0][1] for s in sums[1:]), sums


def test_pair_sync_is_selected_when_asked(native_lib):
    """The knob reaches the generator: the streamed launches of a chain report pair synchronisation."""
    from stencilflow_b200.cuda_program import CudaProgram
    from stencilflow_b200.planner import PlanOptions
    p = CudaProgram(program_path("ref_jacobi3d_32x32x32_8itr_8vec"), allocate=False,
                    plan_options=PlanOptions(max_depth=4, rows_per_thread=4, warps=8, sync="pair"))
    assert all(l.info["sync"] == "pair" for l in p.lowered.launches if l.family == "streamed")
    p = CudaProgram(program_path("ref_jacobi3d_32x32x32_8itr_8vec"), allocate=False,
                    plan_options=PlanOptions(max_depth=4, rows_per_thread=3, warps=12, sync="flags"))
    assert all(l.info["sync"] == "flags" for l in p.lowered.launches if l.family == "streamed")
    p = CudaProgram(program_path("ref_jacobi3d_32x32x32_8itr_8vec"), allocate=False,
                    plan_options=PlanOptions(max_depth=4, rows_per_thread=3, warps=12, sync="halves"))
    assert all(l.info["sync"] == "halves" for l in p.lowered.launches if l.family == "streamed")
    # a field that is read through its ring by two operators keeps the CTA barrier
    p = CudaProgram(program_path("fork_join_20x16x24"), allocate=False,
                    plan_options=PlanOptions(max_depth=4, rows_per_thread=3, warps=12, sync="flags"))
    assert any(l.family == "streamed" for l in p.lowered.launches)


@pytest.mark.parametrize("kind", ["jacobi3d", "jacobi2d"])
def test_pair_sync_bit_identical_at_scale(gpu, kind):
    """Many CTAs, many waves: neighbour-only synchronisation with a deep TMA ring must reproduce the
    CTA-barrier kernel bit for bit (same per-cell arithmetic; any race would show as a difference)."""
    from stencilflow_b200 import programs
    from stencilflow_b200.cuda_program import CudaProgram
    from stencilflow_b200.planner import PlanOptions
    if kind == "jacobi3d":
        prog, out, dt = programs.jacobi3d_chain([320, 448, 512], 8), "b7", np.float32
        variants = [dict(max_depth=4, rows_per_thread=4, warps=8, sync="cta"),
                    dict(max_depth=4, rows_per_thread=4, warps=8, sync="pair", prefetch=5),
                    dict(max_depth=4, rows_per_thread=3, warps=12, sync="pair", prefetch=3),
                    dict(max_depth=4, rows_per_thread=3, warps=12, sync="flags", prefetch=5),
                    dict(max_depth=4, rows_per_thread=4, warps=8, sync="flags", prefetch=2),
                    dict(max_depth=4, rows_per_thread=3, warps=12, sync="halves", prefetch=5),
                    dict(max_depth=4, rows_per_thread=4, warps=8, sync="halves", prefetch=2)]
    else:
        prog, out, dt = programs.jacobi2d_chain([3000, 16384], 8), "b7", np.float64
        variants = [dict(max_depth=8, vector=4, warps=8, sync="cta"),
                    dict(max_depth=8, vector=4, warps=8, sync="pair", prefetch=5),
                    dict(max_depth=4, vector=2, warps=16, sync="pair", prefetch=3),
                    dict(max_depth=8, vector=4, warps=2, sync="flags", prefetch=5),
                    dict(max_depth=4, vector=4, warps=8, sync="flags", prefetch=5)]
    path = programs.write_program(prog, "pairsync_" + kind)
    n = int(np.prod(prog["dimensions"]))
    sums = []
    for opts in variants:
        p = CudaProgram(path, plan_options=PlanOptions(**opts))
        p.rt.fill_hash(p.buffers["a"].dptr, n, dt, seed=99)
        for _ in range(3):
            p.execute()
        p.rt.stream_synchronize()
        sums.append(p.rt.checksum(p.buffers[out].dptr, n, dt))
        p.close()
    assert all(s_[1] == sums[0][1] for s_ in sums[1:]), sums


GENERATOR_SWITCHES = [
    {"SFB200_SPLITBAR": "1"}, {"SFB200_HALO_SKIP": "1"}, {"SFB200_ST64": "5"}, {"SFB200_SPLITLOOP": "1"},
    {"SFB200_SPLITLOOP": "0"}, {"SFB200_BC_MODE": "thread"}, {"SFB200_BC_MODE": "cta", "SFB200_SCHED": "halving"},
    {"SFB200_UNROLL": "12", "SFB200_UNROLL_MULT": "2"}, {"SFB200_REASSOCIATE": "0"}, {"SFB200_L2HINT": "0"},
]


@pytest.mark.parametrize("switches", GENERATOR_SWITCHES, ids=lambda d: ",".join("{}={}".format(k[7:], v) for k, v in d.items()))
@pytest.mark.parametrize("name", ["ref_jacobi3d_32x32x32_8itr_8vec", "jacobi3d_16x24x32_5itr_const1",
                                  "jacobi2d_96x128_6itr_shrink_f64"])
def test_generator_switches_match_oracle(gpu, name, switches, monkeypatch):
    """The code-shape switches of DESIGN section 11 (measured alternatives the defaults were chosen against) stay
    correct: fused passes under each of them against the oracle."""
    from oracle import reference_numpy as rn
    from stencilflow_b200.planner import PlanOptions
    for k, v in switches.items():
        monkeypatch.setenv(k, v)
    inputs = random_inputs(name, seed=41)
    expected = rn.run_reference(program_path(name), inputs)
    opts = PlanOptions(max_depth=4, rows_per_thread=3, warps=12) if "3d" in name else PlanOptions(max_depth=6, vector=4, warps=2)
    got, prog = _run_cuda(name, inputs, opts)
    assert any(l.family == "streamed" for l in prog.lowered.launches)
    _check(name, got, expected)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["ref_jacobi3d_32x32x32_8itr_8vec", "hdiff_24x28x16", "fork_join_20x16x24",
                                  "jacobi2d_96x128_6itr_shrink_f64", "lowdim3d_20x24x48_3st_f32"])
def test_chunk_grid_still_matches_oracle(gpu, name, monkeypatch):
    """SFB200_PERSISTENT=0: the one-CTA-per-(tile, chunk) grid the persistent schedule replaced."""
    from oracle import reference_numpy as rn
    monkeypatch.setenv("SFB200_PERSISTENT", "0")
    inputs = random_inputs(name, seed=13)
    expected = rn.run_reference(program_path(name), inputs)
    got, prog = _run_cuda(name, inputs)
    assert not any(l.info.get("persistent") for l in prog.lowered.launches)
    _check(name, got, expected)


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["jacobi3d", "jacobi2d", "hdiff"])
def test_persistent_schedule_bit_identical_at_scale(gpu, kind, monkeypatch):
    """Persistent CTAs stream several (tile, plane-range) segments each, re-entering the pipeline at every
    segment; the result must equal the chunk grid's and the one-operator kernels' bit for bit, and the
    work table must have used every slot of the device."""
    from stencilflow_b200 import programs
    from stencilflow_b200.cuda_program import CudaProgram
    from stencilflow_b200.planner import PlanOptions
    if kind == "jacobi3d":
        prog, out, dt, fills = programs.jacobi3d_chain([320, 448, 512], 8), "b7", np.float32, {"a": (0.0, 1.0)}
    elif kind == "jacobi2d":
        prog, out, dt, fills = programs.jacobi2d_chain([3000, 16384], 8), "b7", np.float64, {"a": (0.0, 1.0)}
    else:
        prog, out, dt = programs.hdiff([192, 256, 80]), "out", np.float32
        fills = {"inp": (1.0, 2.0), "coeff": (0.0, 0.05)}
    path = programs.write_program(prog, "persist_" + kind)
    n = int(np.prod(prog["dimensions"]))
    sums = []
    for mode, opts in (("1", None), ("0", None), ("1", PlanOptions(fuse=False))):
        monkeypatch.setenv("SFB200_PERSISTENT", mode)
        p = CudaProgram(path, plan_options=opts)
        for k, (name, (lo, hi)) in enumerate(sorted(fills.items())):
            p.rt.fill_hash(p.buffers[name].dptr, n, dt, seed=99 + k, lo=lo, hi=hi)
        for _ in range(2):
            p.execute()
        p.rt.stream_synchronize()
        sums.append(p.rt.checksum(p.buffers[out].dptr, n, dt))
        if mode == "1" and opts is None:
            l, fn, grid, pack = p._packs[0]
            assert l.info["persistent"] and 0.9 * p._resident_ctas(l) <= grid[0] <= p._resident_ctas(l) and grid[1:] == (1, 1)
        p.close()
    assert sums[1][1] == sums[0][1] and sums[2][1] == sums[0][1], sums



def test_exported_program_conventions_end_to_end(gpu, tmp_path, monkeypatch):
    """A program as ``sdfg_to_stencilflow`` writes it (``stencilflow/sdfg_to_stencilflow.py:522-767``): J,K,I
    layout (``:46-68``), versioned field names (``out__1`` -> ``out``), ``constants`` with string values,
    ``btype`` boundary keys, newline-separated statements from astunparse, raw ``.dat`` inputs named
    ``<field>_<dims>_<dtype>.dat`` with ``input_dims`` -- through the drop-in driver with -compare-to-reference."""
    import json
    from stencilflow_b200 import helper
    from stencilflow_b200.run_program import run_program
    name = "sdfgexport_hdiff_jki_48x8x64_f64"
    with open(program_path(name)) as f:
        prog = json.load(f)
    inputs = random_inputs(name, seed=31)
    for field, cfg in prog["inputs"].items():
        helper.save_array(inputs[field], str(tmp_path / cfg["data"]))
    monkeypatch.chdir(tmp_path)
    assert run_program(program_path(name), "cuda", compare_to_reference=True, halo=2, log_level=0,
                       input_directory=str(tmp_path)) == 0
    # and directly against the oracle on the same arrays
    from oracle import reference_numpy as rn
    expected = rn.run_reference(program_path(name), inputs)
    got, prog_obj = _run_cuda(name, inputs)
    _check(name, got, expected)
    # ... and as one fused pass (asked for explicitly: on a grid this small the planner may prefer one-operator launches)
    from stencilflow_b200.planner import PlanOptions
    got, prog_obj = _run_cuda(name, inputs, PlanOptions(max_depth=8))
    _check(name, got, expected)
    assert [l.family for l in prog_obj.lowered.launches] == ["streamed"]


@pytest.mark.parametrize("name,opts", [("ref_jacobi3d_32x32x32_8itr_8vec", dict(max_depth=4)),
                                       ("ref_jacobi3d_32x32x32_8itr_8vec", dict(fuse=False)),
                                       ("hdiff_24x28x16", dict(max_depth=4)),
                                       ("jacobi2d_96x128_6itr_shrink_f64", dict(max_depth=3))])
def test_program_handle_round_trip(gpu, name, opts):
    """The per-program handle of the C ABI (``sfb_program_create / add_buffer / add_launch / bind / call /
    run / destroy``, the counterpart of DaCe's ``__dace_init / __program / __dace_exit``): host arrays are
    bound once, one library call copies in, runs every launch and copies out -- compared with the oracle;
    ``sfb_program_run`` then repeats the launches and reports the device time."""
    from oracle import reference_numpy as rn
    from stencilflow_b200.cuda_program import CudaProgram
    from stencilflow_b200.planner import PlanOptions
    inputs = random_inputs(name, seed=23)
    expected = rn.run_reference(program_path(name), inputs)
    prog = CudaProgram(program_path(name), plan_options=PlanOptions(**opts))
    assert prog.handle is not None
    prog.set_scalars({k: v for k, v in inputs.items() if getattr(v, "ndim", 0) == 0})
    prog._build_packs()
    rtm = prog.rt
    assert rtm.program_num_launches(prog.handle) == len(prog.lowered.launches)
    outs = {}
    for field, f in prog.program.fields.items():
        if f.is_scalar:
            continue
        if f.kind == "input":
            rtm.program_bind(prog.handle, field, np.ascontiguousarray(inputs[field]), 0)
        elif f.kind == "output":
            outs[field] = np.zeros(f.shape, dtype=f.data_type.type)
            rtm.program_bind(prog.handle, field, outs[field], 1)
    rtm.program_call(prog.handle)
    _check(name, outs, expected)
    ms = rtm.program_run(prog.handle, 3, timed=True)
    assert ms > 0.0
    # the fields the handle owns are the ones the Python object reports
    for field, buf in prog.buffers.items():
        assert rtm.program_buffer(prog.handle, field)[0] == buf.dptr
    prog.close()


@pytest.mark.parametrize("name,opts", [("ref_jacobi3d_32x32x32_8itr_8vec", dict(max_depth=4)),
                                       ("hdiff_24x28x16", dict(max_depth=4)),
                                       ("ref_varying_dimensionality", dict(fuse=False))])
def test_plain_c_host_runs_the_program_handle(gpu, name, opts, tmp_path):
    """No Python in the process that computes: ``examples/run_sfbplan.c`` (gcc, links libsfb200.so only)
    builds the per-program handle from an exported plan script, runs it and writes the outputs, which
    must match the oracle -- the C ABI is bindable from any language, as DaCe's init/program/exit trio is."""
    import subprocess
    from oracle import reference_numpy as rn
    from stencilflow_b200 import runtime
    from stencilflow_b200.cuda_program import CudaProgram
    from stencilflow_b200.planner import PlanOptions
    exe = str(tmp_path / "run_sfbplan")
    libdir = os.path.dirname(runtime.LIB_PATH)
    subprocess.run(["gcc", "-O2", "-I", os.path.join(ROOT, "include"), os.path.join(ROOT, "examples", "run_sfbplan.c"),
                    "-o", exe, "-L", libdir, "-lsfb200", "-Wl,-rpath," + libdir], check=True)
    inputs = random_inputs(name, seed=29)
    expected = rn.run_reference(program_path(name), inputs)
    prog = CudaProgram(program_path(name), plan_options=PlanOptions(**opts))
    script = prog.export_plan(str(tmp_path / "plan"), inputs)
    shapes = {o: (prog.program.fields[o].shape, prog.program.fields[o].data_type.type) for o in prog.program.outputs}
    prog.close()
    res = subprocess.run([exe, script, "0", "3"], stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=120)
    assert res.returncode == 0, res.stdout
    assert "launch(es), 3 repetitions" in res.stdout
    got = {o: np.fromfile(str(tmp_path / "plan" / (o + ".dat")), dtype=dt).reshape(shape)
           for o, (shape, dt) in shapes.items()}
    _check(name, got, expected)

"""Fused passes over unaligned rows (``PlanOptions(unaligned=1)``) on the GPU: every misaligned fixture and the
reference's misaligned programs against the oracle and, bit for bit, against the one-operator kernels; on the chunk
grid and on persistent CTAs, with parked window planes, through the pipelined host call, from the plain C host, and
at scale."""
import os
import subprocess

import numpy as np
import pytest

from conftest import program_path, random_inputs
from test_unaligned_plan import FIXTURES, fixture_path

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TOL = {"float32": 1e-5, "float64": 1e-12}
# the reference's programs whose innermost rows are not a multiple of 16 bytes, where a fused pass fits at their size
REFERENCE = ["ref_simulator", "ref_simulator2", "ref_simulator3", "ref_simulator4", "ref_simulator5",
             "ref_simulator6", "ref_simulator7", "ref_simulator8", "ref_simulator9", "ref_simulator10",
             "ref_simulator11", "ref_simulator12", "ref_simple_input_delay_buf"]


@pytest.fixture(scope="module")
def gpu(native_lib):
    from stencilflow_b200 import runtime
    return runtime.Runtime.get()


@pytest.fixture
def clean_env(monkeypatch):
    for k in list(os.environ):
        if k.startswith("SFB200_"):
            monkeypatch.delenv(k)
    return monkeypatch


def _inputs(path, seed):
    from oracle import reference_numpy as rn
    info = rn.ProgramInfo(rn.load_program(path))
    rng = np.random.default_rng(seed)
    out = {}
    for f in info.inputs:
        shape = info.field_shape(f)
        lo, hi = (1.0, 2.0) if f == "inp" else ((0.0, 0.05) if f == "coeff" else (0.0, 1.0))
        if len(shape) == 0:
            out[f] = info.field_type(f)(rng.uniform(0.5, 1.5))
        else:
            out[f] = rng.uniform(lo, hi, size=shape).astype(info.field_type(f))
    return out


def _run(path, inputs, opts):
    from oracle import reference_numpy as rn
    from stencilflow_b200.cuda_program import CudaProgram
    prog = CudaProgram(path, plan_options=opts)
    info = rn.ProgramInfo(rn.load_program(path))
    outs = {o: np.zeros(info.shape, dtype=info.field_type(o)) for o in info.outputs}
    args = {(k + "_host" if getattr(v, "ndim", 0) > 0 else k): v for k, v in inputs.items()}
    args.update({k + "_host": v for k, v in outs.items()})
    try:
        prog(**args)
    finally:
        prog.close()
    return outs, [l.info for l in prog.lowered.launches if l.family == "streamed"]


def _check_all(path, inputs, halo, runs):
    """Every run of ``runs`` [(label, PlanOptions, streamed?)] against the oracle; all of them bit-identical."""
    from oracle import reference_numpy as rn
    expected = rn.run_reference(path, inputs)
    results = {}
    for label, opts, fused in runs:
        got, streamed = _run(path, inputs, opts)
        if fused:
            assert streamed and all(i.get("unaligned") for i in streamed), label
        for field, ref in expected.items():
            err = rn.max_relative_error(rn.trim_halo(ref, halo), rn.trim_halo(got[field], halo))
            assert err <= TOL[ref.dtype.name], "{} {}: max rel err {}".format(label, field, err)
        results[label] = {f: np.ascontiguousarray(rn.trim_halo(a, halo)).tobytes() for f, a in got.items()}
    first = next(iter(results.values()))
    for label, res in results.items():
        assert res == first, label


@pytest.mark.parametrize("name", sorted(FIXTURES))
def test_fixture_matches_oracle_and_one_operator_kernels(gpu, clean_env, tmp_path, name):
    from stencilflow_b200.planner import PlanOptions
    path = fixture_path(name, tmp_path)
    _, opts, halo = FIXTURES[name]
    runs = [("unfused", PlanOptions(fuse=False), False), ("fused", PlanOptions(unaligned=1, **opts), True)]
    _check_all(path, _inputs(path, 11), halo, runs)
    clean_env.setenv("SFB200_PERSISTENT", "1")
    _check_all(path, _inputs(path, 11), halo, [runs[0], ("persistent", PlanOptions(unaligned=1, **opts), True)])


def test_jacobi3d_parked_planes(gpu, clean_env, tmp_path):
    from stencilflow_b200.planner import PlanOptions
    path = fixture_path("jacobi3d_f32_nk66", tmp_path)
    geo = dict(max_depth=4, rows_per_thread=3, warps=12, prefetch=5, sync="cta")
    runs = [("unfused", PlanOptions(fuse=False), False), ("parked", PlanOptions(unaligned=1, tmem=2, **geo), True),
            ("registers", PlanOptions(unaligned=1, tmem=0, **geo), True)]
    _check_all(path, _inputs(path, 12), 0, runs)
    _, streamed = _run(path, _inputs(path, 12), PlanOptions(unaligned=1, tmem=2, **geo))
    assert all(i["tmem"] for i in streamed)


@pytest.mark.parametrize("sync", ["pair", "halves", "flags"])
def test_other_synchronisation_schemes(gpu, clean_env, tmp_path, sync):
    from stencilflow_b200.planner import PlanOptions
    path = fixture_path("jacobi3d_f32_nk131", tmp_path)
    runs = [("unfused", PlanOptions(fuse=False), False),
            (sync, PlanOptions(unaligned=1, max_depth=3, rows_per_thread=4, warps=8, sync=sync), True)]
    _check_all(path, _inputs(path, 13), 0, runs)


@pytest.mark.parametrize("name", REFERENCE)
def test_reference_programs(gpu, clean_env, name):
    """At their own size (a 1x3x3 or 3^3 grid is one tile), every one of them with at least one fused pass."""
    from oracle import reference_numpy as rn
    from stencilflow_b200.planner import PlanOptions, plan_program
    from stencilflow_b200.kernel_chain_graph import KernelChainGraph
    from stencilflow_b200.stencil_op import make_program
    path = program_path(name)
    inputs = random_inputs(name, seed=5)
    opts = dict(unaligned=1, max_depth=8)
    plan = plan_program(make_program(KernelChainGraph(path)), PlanOptions(**opts))
    fused = any(l.family == "streamed" for l in plan.lowered.launches)
    runs = [("unfused", PlanOptions(fuse=False), False), ("option", PlanOptions(**opts), fused)]
    expected = rn.run_reference(path, inputs)
    results = []
    assert fused
    for label, o, f in runs:
        got, streamed = _run(path, inputs, o)
        if f:
            assert streamed and all(i.get("unaligned") for i in streamed), label
        for field, ref in expected.items():
            err = rn.max_relative_error(ref, got[field])
            assert err <= TOL[ref.dtype.name], "{} {}: max rel err {}".format(label, field, err)
        results.append({k: v.tobytes() for k, v in got.items()})
    assert results[0] == results[1]


def test_pipelined_host_call_matches_execute(gpu, clean_env, tmp_path):
    """A grid of more than 64 MiB per field and enough planes for 16 pieces of four times the passes' reach: the
    host-array call is cut into pieces; bit-identical to upload / execute / download."""
    from stencilflow_b200 import programs, synthetic
    from stencilflow_b200.cuda_program import CudaProgram
    from stencilflow_b200.planner import PlanOptions
    shape = [320, 256, 255]
    path = programs.write_program(programs.jacobi3d_chain(shape, 8), "unaligned_pipelined", str(tmp_path))
    a = synthetic.fill_hash(tuple(shape), np.float32, 1234)
    assert a.nbytes >= 64 << 20
    p = CudaProgram(path, plan_options=PlanOptions(unaligned=1, max_depth=4))
    try:
        assert all(l.info.get("unaligned") for l in p.lowered.launches)
        piped = np.zeros(shape, np.float32)
        p(a_host=a, b7_host=piped)
        assert getattr(p, "_pipe", None) is not None, "the pipelined path was not taken"
        p.upload("a", a)
        p.execute()
        plain = p.download("b7")
    finally:
        p.close()
    assert piped.tobytes() == np.asarray(plain).tobytes()


def test_plain_c_host_runs_the_exported_plan(gpu, clean_env, tmp_path):
    from oracle import reference_numpy as rn
    from stencilflow_b200 import runtime
    from stencilflow_b200.cuda_program import CudaProgram
    from stencilflow_b200.planner import PlanOptions
    exe = str(tmp_path / "run_sfbplan")
    libdir = os.path.dirname(runtime.LIB_PATH)
    subprocess.run(["gcc", "-O2", "-I", os.path.join(ROOT, "include"), os.path.join(ROOT, "examples", "run_sfbplan.c"),
                    "-o", exe, "-L", libdir, "-lsfb200", "-Wl,-rpath," + libdir], check=True)
    path = fixture_path("hdiff_f32_nk78", tmp_path)
    inputs = _inputs(path, 14)
    expected = rn.run_reference(path, inputs)
    prog = CudaProgram(path, plan_options=PlanOptions(unaligned=1, max_depth=4))
    script = prog.export_plan(str(tmp_path / "plan"), inputs)
    shapes = {o: (prog.program.fields[o].shape, prog.program.fields[o].data_type.type) for o in prog.program.outputs}
    prog.close()
    # the streamed launch passes its inputs as plain buffers
    assert not [line for line in open(script) if line.startswith("  tmap ")]
    res = subprocess.run([exe, script, "0", "3"], stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=120)
    assert res.returncode == 0, res.stdout
    got = {o: np.fromfile(str(tmp_path / "plan" / (o + ".dat")), dtype=dt).reshape(shape)
           for o, (shape, dt) in shapes.items()}
    for field, ref in expected.items():
        err = rn.max_relative_error(rn.trim_halo(ref, 2), rn.trim_halo(got[field], 2))
        assert err <= TOL["float32"], err


def _checksum_bits(path, opts, fills, out, dt, monkeypatch, env=None):
    from stencilflow_b200.cuda_program import CudaProgram
    for k, v in (env or {}).items():
        monkeypatch.setenv(k, v)
    p = CudaProgram(path, plan_options=opts)
    try:
        n = int(np.prod(p.program.shape))
        for k, (name, (lo, hi)) in enumerate(sorted(fills.items())):
            p.rt.fill_hash(p.buffers[name].dptr, n, dt, seed=99 + k, lo=lo, hi=hi)
        for _ in range(2):
            p.execute()
        p.rt.stream_synchronize()
        infos = [l.info for l in p.lowered.launches if l.family == "streamed"]
        return p.rt.checksum(p.buffers[out].dptr, n, dt)[1], infos
    finally:
        p.close()
        for k in (env or {}):
            monkeypatch.delenv(k)


def test_jacobi3d_1022_at_scale(gpu, clean_env, tmp_path):
    """1024x1024x1022 x 8 with the measured config-1 plan plus unaligned rows, on persistent CTAs and on the chunk
    grid: checksum bits equal to the one-operator kernels'."""
    from stencilflow_b200 import programs
    from stencilflow_b200.planner import PlanOptions
    path = programs.write_program(programs.jacobi3d_chain([1024, 1024, 1022], 8), "unaligned_j1022", str(tmp_path))
    fills = {"a": (0.0, 1.0)}
    ref, _ = _checksum_bits(path, PlanOptions(fuse=False), fills, "b7", np.float32, clean_env)
    clean_env.setenv("SFB200_UNALIGNED", "1")
    got, infos = _checksum_bits(path, PlanOptions(), fills, "b7", np.float32, clean_env)
    assert len(infos) == 2 and all(i["unaligned"] and i["persistent"] for i in infos)
    chunked, infos = _checksum_bits(path, PlanOptions(), fills, "b7", np.float32, clean_env, {"SFB200_PERSISTENT": "0"})
    assert not any(i["persistent"] for i in infos)
    assert ref == got == chunked


def test_jacobi2d_f64_32767_at_scale(gpu, clean_env, tmp_path):
    from stencilflow_b200 import programs
    from stencilflow_b200.planner import PlanOptions
    path = programs.write_program(programs.jacobi2d_chain([32768, 32767], 16), "unaligned_j2d", str(tmp_path))
    fills = {"a": (0.0, 1.0)}
    ref, _ = _checksum_bits(path, PlanOptions(fuse=False), fills, "b15", np.float64, clean_env)
    got, infos = _checksum_bits(path, PlanOptions(unaligned=1), fills, "b15", np.float64, clean_env)
    assert infos and all(i["unaligned"] for i in infos)
    assert ref == got

"""The cluster kernel family (``PlanOptions(cluster=1)``) on the GPU: a whole program in one launch of one
thread-block cluster, its fields in distributed shared memory.  The per-cell code is the one-operator kernel's,
so every program must be bit-identical to its ``fuse=False`` run, not only close to the oracle."""
import json
import os
import subprocess

import numpy as np
import pytest

from conftest import GOLDEN, HALO, ROOT, all_programs, program_path, random_inputs

pytestmark = pytest.mark.gpu

TOL = {"float32": 1e-5, "float64": 1e-12}
JACOBI_32 = "ref_jacobi3d_32x32x32_8itr_8vec"


def _takes_cluster(name):
    from stencilflow_b200.kernel_chain_graph import KernelChainGraph
    from stencilflow_b200.planner import PlanOptions, plan_program
    from stencilflow_b200.stencil_op import make_program
    plan = plan_program(make_program(KernelChainGraph(program_path(name))), PlanOptions(cluster=1))
    return [l.family for l in plan.lowered.launches] == ["cluster"]


CLUSTER_PROGRAMS = [n for n in all_programs() if _takes_cluster(n)]


@pytest.fixture(scope="module")
def gpu(native_lib):
    from stencilflow_b200 import runtime
    return runtime.Runtime.get()


def _run(name, inputs, **opts):
    """Outputs of one host-array call of ``name`` with the given plan options, and the launch families."""
    from stencilflow_b200.cuda_program import CudaProgram
    from stencilflow_b200.planner import PlanOptions
    prog = CudaProgram(program_path(name), plan_options=PlanOptions(**opts))
    outs = {o: np.zeros(prog.program.fields[o].shape, dtype=prog.program.fields[o].data_type.type)
            for o in prog.program.outputs}
    args = {(k + "_host" if getattr(v, "ndim", 0) > 0 else k): v for k, v in inputs.items()}
    args.update({o + "_host": v for o, v in outs.items()})
    prog(**args)
    families = [l.family for l in prog.lowered.launches]
    prog.close()
    return outs, families


def _check(name, got, expected, halo=None):
    from oracle import reference_numpy as rn
    h = HALO.get(name, 0) if halo is None else halo
    for field, ref in expected.items():
        assert got[field].dtype == ref.dtype
        err = rn.max_relative_error(rn.trim_halo(ref, h), rn.trim_halo(got[field], h))
        assert err <= TOL[ref.dtype.name], "{}:{} max rel err {}".format(name, field, err)


@pytest.mark.parametrize("name", CLUSTER_PROGRAMS)
def test_cluster_matches_oracle_and_is_bit_identical_to_one_operator_kernels(gpu, name):
    from oracle import reference_numpy as rn
    inputs = random_inputs(name, seed=31)
    expected = rn.run_reference(program_path(name), inputs)
    got, families = _run(name, inputs, cluster=1)
    assert families == ["cluster"]
    _check(name, got, expected)
    general, families = _run(name, inputs, fuse=False)
    assert set(families) == {"general"}
    for field in got:
        assert got[field].tobytes() == general[field].tobytes(), (name, field)


with open(os.path.join(GOLDEN, "reference_sim.json")) as _f:
    REFERENCE_SIM = json.load(_f)


@pytest.mark.parametrize("case", sorted(c for c in REFERENCE_SIM if REFERENCE_SIM[c]["program"] in CLUSTER_PROGRAMS))
def test_cluster_matches_reference_simulator(gpu, case):
    """Against outputs of the reference itself (its dataflow simulator, tests/golden/reference_sim.npz)."""
    import sys
    if GOLDEN not in sys.path:
        sys.path.insert(0, GOLDEN)
    import make_reference_sim_golden as gen
    rec = REFERENCE_SIM[case]
    inputs = gen.case_inputs(gen.case_program(rec["program"]), rec["seed"], rec.get("ranges"))
    got, families = _run(rec["program"], inputs, cluster=1)
    assert families == ["cluster"]
    with np.load(os.path.join(GOLDEN, "reference_sim.npz")) as z:
        _check(rec["program"], got, {f: z[case + "/" + f] for f in rec["outputs"]}, halo=rec.get("halo", 0))


@pytest.mark.parametrize("name", [n for n in CLUSTER_PROGRAMS if n.startswith("ref_")])
def test_run_program_compare_to_reference_with_cluster(gpu, name, tmp_path, monkeypatch):
    """The drop-in driver (`run_program.py prog.json cuda -compare-to-reference`) with SFB200_CLUSTER=1."""
    from stencilflow_b200.cuda_program import CudaProgram
    from stencilflow_b200.run_program import run_program
    monkeypatch.setenv("SFB200_CLUSTER", "1")
    monkeypatch.chdir(tmp_path)
    assert [l.family for l in CudaProgram(program_path(name), allocate=False).lowered.launches] == ["cluster"]
    ret = run_program(program_path(name), "cuda", compare_to_reference=True, halo=0, log_level=0,
                      input_directory=os.path.dirname(program_path(name)))
    assert ret == 0


def test_plain_c_host_runs_the_cluster_plan(gpu, tmp_path):
    """``examples/run_sfbplan.c`` runs the exported one-launch cluster plan unchanged."""
    from oracle import reference_numpy as rn
    from stencilflow_b200 import runtime
    from stencilflow_b200.cuda_program import CudaProgram
    from stencilflow_b200.planner import PlanOptions
    exe = str(tmp_path / "run_sfbplan")
    libdir = os.path.dirname(runtime.LIB_PATH)
    subprocess.run(["gcc", "-O2", "-I", os.path.join(ROOT, "include"), os.path.join(ROOT, "examples", "run_sfbplan.c"),
                    "-o", exe, "-L", libdir, "-lsfb200", "-Wl,-rpath," + libdir], check=True)
    inputs = random_inputs(JACOBI_32, seed=37)
    expected = rn.run_reference(program_path(JACOBI_32), inputs)
    prog = CudaProgram(program_path(JACOBI_32), plan_options=PlanOptions(cluster=1))
    assert [l.family for l in prog.lowered.launches] == ["cluster"]
    script = prog.export_plan(str(tmp_path / "plan"), inputs)
    prog.close()
    with open(script) as f:
        assert sum(1 for line in f if line.startswith("launch ")) == 1
    res = subprocess.run([exe, script, "0", "3"], stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=120)
    assert res.returncode == 0, res.stdout
    assert "launch(es), 3 repetitions" in res.stdout
    got = np.fromfile(str(tmp_path / "plan" / "b7.dat"), dtype=np.float32).reshape(32, 32, 32)
    _check(JACOBI_32, {"b7": got}, expected)


@pytest.mark.parametrize("name", [JACOBI_32, "smooth1d_256"])
def test_repeated_executions_are_one_launch_each_and_identical(gpu, name):
    from stencilflow_b200.cuda_program import CudaProgram
    from stencilflow_b200.planner import PlanOptions
    inputs = random_inputs(name, seed=41)
    prog = CudaProgram(program_path(name), plan_options=PlanOptions(cluster=1))
    for field, value in inputs.items():
        if getattr(value, "ndim", 0) > 0:
            prog.upload(field, value)
    prog.set_scalars({k: v for k, v in inputs.items() if getattr(v, "ndim", 0) == 0})
    out = prog.program.outputs[0]
    runs = []
    for n in range(3):
        before = prog.launch_count
        prog.execute()
        assert prog.launch_count == before + 1
        runs.append(prog.download(out).tobytes())
    assert prog._graph is None
    assert runs[0] == runs[1] == runs[2]
    prog.close()

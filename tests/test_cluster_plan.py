"""The cluster kernel family on the CPU: when ``PlanOptions(cluster=1)`` takes it, what its one launch
reads, writes and needs, that it leaves every other plan and the one-operator kernels' source alone, and that
the cubin holds the cluster barriers and the distributed-shared-memory reads."""
import hashlib
import json
import os
import re
import subprocess

import pytest

from conftest import GOLDEN, all_programs, program_path

# test programs whose fields do not fit one 8-CTA cluster (227 KB of shared memory a CTA): none yet
DOES_NOT_FIT = set()


def _program(path):
    from stencilflow_b200.kernel_chain_graph import KernelChainGraph
    from stencilflow_b200.stencil_op import make_program
    return make_program(KernelChainGraph(str(path)))


def _plan(path, **opts):
    from stencilflow_b200.planner import PlanOptions, plan_program
    return plan_program(_program(path), PlanOptions(**opts))


def _jacobi(tmp_path, n, steps=8):
    from stencilflow_b200 import programs
    path = tmp_path / "jacobi3d_{}_{}.json".format(n, steps)
    path.write_text(json.dumps(programs.jacobi3d_chain([n, n, n], steps)))
    return path


def _without_options(desc):
    return {k: v for k, v in desc.items() if k != "options"}


def test_jacobi3d_32_is_one_cluster_launch(tmp_path):
    plan = _plan(_jacobi(tmp_path, 32), cluster=1)
    (l,) = plan.lowered.launches
    assert l.family == "cluster" and l.kernel.startswith("sf_cluster_")
    C = l.info["cluster"]
    assert l.grid_fn(0, 32) == (C, 1, 1) and 1 <= C <= 8
    assert l.block[0] <= 1024 and l.block[1:] == (1, 1)
    assert 0 < l.smem <= 227 * 1024
    assert l.reads == ["a"] and l.writes == ["b7"]
    assert plan.algorithmic_bytes() == 2 * 32 ** 3 * 4
    desc = plan.describe()
    assert desc["passes"][0]["info"]["ranges"] == [[4 * c, 4 * c + 4] for c in range(8)]
    assert set(desc["passes"][0]["info"]["slots"]) == {"a", "b0", "b1", "b2", "b3", "b4", "b5", "b6"}
    # two slots of 4 planes of 32 x 32 floats: a field's slot is reused once it is dead
    assert l.smem == 2 * 4 * 32 * 32 * 4
    assert "__cluster_dims__(8, 1, 1)" in plan.lowered.source


def test_jacobi3d_64_does_not_fit_and_keeps_the_default_plan(tmp_path):
    path = _jacobi(tmp_path, 64)
    assert _without_options(_plan(path, cluster=1).describe()) == _without_options(_plan(path).describe())


def test_a_large_grid_that_keeps_nothing_in_shared_memory_does_not_fit(tmp_path):
    """Shared memory is not the only bound: the cells of a CTA must fit a few items per thread."""
    path = tmp_path / "wide.json"
    path.write_text(json.dumps({
        "inputs": {"w": {"data": "constant:1.0", "data_type": "float32", "input_dims": ["k"]}},
        "outputs": ["o"], "dimensions": [256, 256, 256],
        "program": {"o": {"computation_string": "o = w[k] + 1.0", "boundary_conditions": {}, "data_type": "float32"}}}))
    from stencilflow_b200 import lower_cluster
    layout = lower_cluster.ClusterLayout(_program(path))
    assert layout.smem_bytes == 0 and not layout.fits
    assert _without_options(_plan(path, cluster=1).describe()) == _without_options(_plan(path).describe())


def test_the_option_leaves_other_plans_alone(tmp_path, monkeypatch):
    plan = _plan(_jacobi(tmp_path, 32), cluster=1, fuse=False)
    assert [l.family for l in plan.lowered.launches] == ["general"] * 8
    from stencilflow_b200 import programs
    from stencilflow_b200.planner import PlanOptions, plan_program
    for index in (1, 2, 3):
        name, prog, _ = programs.baseline_config(index)
        path = programs.write_program(prog, name, str(tmp_path))
        program = _program(path)
        monkeypatch.delenv("SFB200_CLUSTER", raising=False)
        default = plan_program(program, PlanOptions())
        monkeypatch.setenv("SFB200_CLUSTER", "1")
        options = PlanOptions()
        assert options.is_default and options.cluster == 1
        clustered = plan_program(program, options)
        # the measured table still applies, and the kernels and tiles are those of the default plan
        assert clustered.tuned_from == default.tuned_from
        assert _without_options(clustered.describe()) == _without_options(default.describe()), index
        assert clustered.lowered.source == default.lowered.source


@pytest.fixture(scope="module")
def native(native_lib):
    return native_lib


def test_every_program_lowers_and_compiles_or_keeps_its_plan(native, tmp_path, monkeypatch):
    from stencilflow_b200.cuda_program import CudaProgram
    from stencilflow_b200.planner import PlanOptions
    monkeypatch.setenv("SFB200_CACHE", str(tmp_path / "cache"))
    clustered = []
    for name in all_programs():
        plan = _plan(program_path(name), cluster=1)
        families = [l.family for l in plan.lowered.launches]
        if families == ["cluster"]:
            clustered.append(name)
            prog = CudaProgram(program_path(name), plan_options=PlanOptions(cluster=1), allocate=False)
            assert len(prog.image) > 0
            assert [l.family for l in prog.lowered.launches] == ["cluster"]
        else:
            assert _without_options(plan.describe()) == _without_options(_plan(program_path(name)).describe())
    assert set(all_programs()) - set(clustered) == DOES_NOT_FIT
    for name in ("smooth1d_256",                         # 1-D: chunks of k
                 "ref_varying_dimensionality",           # float32 and float64, 0-D, 1-D and 2-D inputs
                 "ref_simple_input_delay_buf",           # 1 x 3 x 3: fewer planes than CTAs
                 "jacobi3d_12x12x16_3itr_copy",          # copy boundaries
                 "jacobi2d_96x128_6itr_shrink_f64"):     # shrink boundaries
        assert name in clustered, name
    info = _plan(program_path("ref_simple_input_delay_buf"), cluster=1).lowered.launches[0].info
    assert info["cluster"] == 1 and info["ranges"] == [[0, 1]]
    info = _plan(program_path("smooth1d_256"), cluster=1).lowered.launches[0].info
    assert info["outer"] == "k" and all((hi - lo) % 2 == 0 for lo, hi in info["ranges"])


def test_one_operator_kernels_are_unchanged():
    """The general kernels' source text (and so their names, which hash it) is what it was before the cluster
    family started to share their per-cell emitter."""
    from stencilflow_b200.planner import PlanOptions, plan_program
    with open(os.path.join(GOLDEN, "sf_general_digests.json")) as f:
        recorded = json.load(f)
    assert sorted(recorded) == all_programs()
    for name in all_programs():
        plan = plan_program(_program(program_path(name)), PlanOptions(fuse=False))
        text = "".join(k.source for k in plan.lowered.kernels.values())
        assert hashlib.sha1(text.encode()).hexdigest() == recorded[name], name


def test_cubin_holds_cluster_barriers_and_remote_reads(tmp_path):
    plan = _plan(_jacobi(tmp_path, 32), cluster=1)
    src = tmp_path / "cluster.cu"
    src.write_text(plan.lowered.source)
    cubin = tmp_path / "cluster.cubin"
    nvcc = os.environ.get("NVCC", "nvcc")
    # the flags programs are built with (cuda_program.compile_cached: -arch=sm_100a -std=c++17 -lineinfo)
    res = subprocess.run([nvcc, "-cubin", "-gencode", "arch=compute_100a,code=sm_100a", "-std=c++17", "-lineinfo",
                          "-Xptxas", "-v", "-o", str(cubin), str(src)],
                         stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, check=True)
    assert "0 bytes spill stores, 0 bytes spill loads" in res.stdout, res.stdout
    sass = subprocess.run(["cuobjdump", "-sass", str(cubin)], stdout=subprocess.PIPE, text=True, check=True).stdout
    ops = re.findall(r"\b(UCGABAR_ARV|UCGABAR_WAIT|LD\.E\.128|LDS\.128|STS\.128|STG\.E\.128|MEMBAR\.ALL\.GPU)\b", sass)
    count = {op: ops.count(op) for op in set(ops)}
    # one barrier after the input load and one before each later operator (all read the previous result), one at exit
    assert count["UCGABAR_ARV"] == count["UCGABAR_WAIT"] == 9
    # release at cluster scope: a memory barrier per arrive
    assert count["MEMBAR.ALL.GPU"] == 9
    # the i-1 and i+1 planes of every operator: mapa is address arithmetic, the load a generic 128-bit LD
    assert count["LD.E.128"] == 2 * 8
    assert count["LDS.128"] > 0 and count["STS.128"] > 0 and count["STG.E.128"] == 1

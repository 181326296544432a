"""Fused passes over unaligned rows (``PlanOptions(unaligned=1)``) on the CPU: the option leaves every program whose
rows are a multiple of 16 bytes alone, misaligned programs plan as streamed passes and compile, and the cubin
copies input cells with cp.async (LDGSTS) and stores results cell by cell."""
import json
import os
import re
import subprocess

import pytest

from conftest import GOLDEN

from stencilflow_b200 import programs

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

CONST0 = {"type": "constant", "value": 0.0}

# misaligned programs: name -> (program, plan options, halo of junk cells for ``shrink`` boundaries)
FIXTURES = {
    "jacobi3d_f32_nk15": (programs.jacobi3d_chain([20, 24, 15], 4), dict(max_depth=4), 0),
    "jacobi3d_f32_nk66": (programs.jacobi3d_chain([20, 24, 66], 4), dict(max_depth=4), 0),
    "jacobi3d_f32_nk131": (programs.jacobi3d_chain([12, 20, 131], 3), dict(max_depth=3), 0),
    # rows of 16 threads: 6 column tiles, so interior tiles between the two k-edge tiles, and 4 row tiles
    "jacobi3d_f32_nk301": (programs.jacobi3d_chain([24, 200, 301], 4), dict(max_depth=4, threads_per_row=16), 0),
    "jacobi3d_f64_nk33": (programs.jacobi3d_chain([16, 20, 33], 3, dtype="float64"), dict(max_depth=3), 0),
    "jacobi3d_f32_const1": (programs.jacobi3d_chain([16, 20, 30], 3, boundary={"type": "constant", "value": 1.0}),
                            dict(max_depth=3), 0),
    "jacobi3d_f32_shrink": (programs.jacobi3d_chain([16, 20, 30], 3, boundary={"type": "shrink"}),
                            dict(max_depth=3), 3),
    "jacobi3d_f32_copy": (programs.jacobi3d_chain([12, 12, 19], 3, boundary={"type": "copy"}), dict(max_depth=3), 0),
    "jacobi2d_f32_chain": (programs.jacobi2d_chain([64, 255], 4, dtype="float32", boundary=CONST0),
                           dict(max_depth=4), 0),
    "jacobi2d_f64_w1d": (programs.jacobi2d_weighted([64, 127], 4), dict(max_depth=4), 4),
    "hdiff_f32_nk78": (programs.hdiff([16, 20, 78]), dict(max_depth=4), 2),
}


def fixture_path(name, directory):
    return programs.write_program(FIXTURES[name][0], "unaligned_" + name, str(directory))


def _program(path):
    from stencilflow_b200.kernel_chain_graph import KernelChainGraph
    from stencilflow_b200.stencil_op import make_program
    return make_program(KernelChainGraph(str(path)))


def _plan(path, **opts):
    from stencilflow_b200.planner import PlanOptions, plan_program
    return plan_program(_program(path), PlanOptions(**opts))


@pytest.fixture
def clean_env(monkeypatch):
    for k in list(os.environ):
        if k.startswith("SFB200_"):
            monkeypatch.delenv(k)
    return monkeypatch


def _recorded():
    with open(os.path.join(GOLDEN, "sf_stream_digests.json")) as f:
        return json.load(f)


def _aligned(path):
    prog = _program(os.path.join(ROOT, path))
    return all((prog.shape[-1] * f.data_type.bytes) % 16 == 0 for f in prog.fields.values())


def test_without_the_option_no_plan_or_fused_kernel_changes(clean_env):
    """Digests of the ``sf_stream_*`` sources and of ``plan.describe()`` (without its options) recorded before the
    option existed: default and explicit-depth plans of every test program and every tracked program."""
    import sys
    sys.path.insert(0, GOLDEN)
    import make_stream_digests
    recorded = _recorded()
    assert sorted(recorded) == sorted(make_stream_digests.program_files())
    for path, want in recorded.items():
        assert make_stream_digests.digests(path) == want, path
        assert make_stream_digests.digests(path, unaligned=0) == want, path


def test_with_the_option_aligned_programs_are_unchanged(clean_env):
    import sys
    sys.path.insert(0, GOLDEN)
    import make_stream_digests
    aligned = 0
    for path, want in _recorded().items():
        if _aligned(path):
            aligned += 1
            assert make_stream_digests.digests(path, unaligned=1) == want, path
    assert aligned >= 40


def test_the_option_survives_the_measured_plan_table(clean_env, tmp_path):
    """A 1024x1024x1022 Jacobi-3D chain takes the measured config-1 plan plus unaligned rows."""
    path = programs.write_program(programs.jacobi3d_chain([1024, 1024, 1022], 8), "j1022", str(tmp_path))
    clean_env.setenv("SFB200_UNALIGNED", "1")
    from stencilflow_b200.planner import PlanOptions, plan_program
    options = PlanOptions()
    assert options.is_default and options.unaligned == 1
    plan = plan_program(_program(path), options)
    assert plan.tuned_from is not None
    infos = [l.info for l in plan.lowered.launches]
    assert [l.family for l in plan.lowered.launches] == ["streamed"] * 2
    assert all(i["unaligned"] and (i["R"], i["warps"][0], i["threads_per_row"]) == (3, 24, 16) for i in infos)
    assert all("unaligned" in p["info"] for p in plan.describe()["passes"])
    # without the option: one-operator kernels, as before
    clean_env.delenv("SFB200_UNALIGNED")
    assert [l.family for l in plan_program(_program(path), PlanOptions()).lowered.launches] == ["general"] * 8


def test_ignored_without_fusion_and_in_slab_mode(clean_env, tmp_path):
    path = fixture_path("jacobi3d_f32_nk66", tmp_path)
    assert {l.family for l in _plan(path, unaligned=1, fuse=False).lowered.launches} == {"general"}
    assert {l.family for l in _plan(path, unaligned=1, max_depth=4, peer_push=True).lowered.launches} == {"general"}


@pytest.mark.parametrize("name", sorted(FIXTURES))
def test_misaligned_fixtures_stream_and_compile(native_lib, clean_env, tmp_path, name):
    from stencilflow_b200.cuda_program import CudaProgram
    from stencilflow_b200.planner import PlanOptions
    clean_env.setenv("SFB200_CACHE", str(tmp_path / "cache"))
    path = fixture_path(name, tmp_path)
    opts = FIXTURES[name][1]
    assert {l.family for l in _plan(path, **opts).lowered.launches} == {"general"}
    plan = _plan(path, unaligned=1, **opts)
    streamed = [l for l in plan.lowered.launches if l.family == "streamed"]
    assert streamed and all(l.info["unaligned"] for l in streamed)
    for l in streamed:
        # the streamed inputs are plain buffers: no tensor map, so no 16-byte stride rule
        assert not any(a[0] == "tmap" for a in l.args)
    # input cells arrive by cp.async, results leave cell by cell
    for l in streamed:
        src = plan.lowered.kernels[l.kernel].source
        assert "sf_cp_async(" in src and "sf_stg1_if(" in src and "sf_tma_load" not in src and "sf_stg_if(" not in src
    prog = CudaProgram(path, plan_options=PlanOptions(unaligned=1, **opts), allocate=False)
    assert len(prog.image) > 0


def test_cubin_copies_cells_and_stores_cells(clean_env, tmp_path):
    """Config-1 geometry at 1024x1024x1022: input cells by LDGSTS completing on the ring's mbarrier, no TMA load, no
    128-bit result stores, no spills."""
    path = programs.write_program(programs.jacobi3d_chain([1024, 1024, 1022], 8), "j1022", str(tmp_path))
    plan = _plan(path, unaligned=1)
    src = tmp_path / "unaligned.cu"
    src.write_text(plan.lowered.source)
    cubin = tmp_path / "unaligned.cubin"
    nvcc = os.environ.get("NVCC", "nvcc")
    res = subprocess.run([nvcc, "-cubin", "-gencode", "arch=compute_100a,code=sm_100a", "-std=c++17", "-lineinfo",
                          "-Xptxas", "-v", "-o", str(cubin), str(src)],
                         stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, check=True)
    spills = re.findall(r"(\d+) bytes spill stores, (\d+) bytes spill loads", res.stdout)
    assert spills and all(st == "0" and ld == "0" for st, ld in spills), res.stdout
    sass = subprocess.run(["cuobjdump", "-sass", str(cubin)], stdout=subprocess.PIPE, text=True, check=True).stdout
    ops = re.findall(r"\b(UTMALDG\.\w+|LDGSTS\.E|ARRIVES\.LDGSTSBAR\.64\.ARVCNT|STG\.E\.128|STG\.E\.64|STG\.E)\b", sass)
    assert "LDGSTS.E" in ops and "ARRIVES.LDGSTSBAR.64.ARVCNT" in ops
    assert not any(o.startswith("UTMALDG") for o in ops)
    assert "STG.E.128" not in ops and "STG.E.64" not in ops and "STG.E" in ops

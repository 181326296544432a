"""Window planes parked in tensor memory (``PlanOptions.tmem``), on the GPU.  Every entry of the matrix runs one explicit
plan twice: with ``tmem=2`` (every slot that qualifies is parked, whatever the register estimate) and with ``tmem=0``.
Both runs must match the oracle, and they must be bit-identical, since parking a plane moves registers and changes no
arithmetic.  A wrong column parity, a missing ``tcgen05.wait::ld`` or swapped float64 words corrupt some planes
without a fault, so only a comparison of values catches them.  ``sync`` is always given, so that the switch to
per-field mbarriers that the cost model makes for parked passes does not change a second thing at once."""
import json

import numpy as np
import pytest

from conftest import HALO, program_path, random_inputs

pytestmark = pytest.mark.gpu

TOL = {"float32": 1e-5, "float64": 1e-12}

# d4 r3 w12 p5: the Jacobi-3D plan of BASELINE config 1.  Rows of 16 threads need an innermost extent of 32 V
# (or exactly 16 V), so most test programs take it with rows of 32 threads
GEO_A16 = dict(max_depth=4, rows_per_thread=3, warps=12, threads_per_row=16, prefetch=5)
GEO_A = dict(max_depth=4, rows_per_thread=3, warps=12, threads_per_row=32, prefetch=5)
GEO_B = dict(max_depth=4, rows_per_thread=4, warps=8, threads_per_row=32, prefetch=2)

# The reference's 3-D programs of 1x3x3 and 3^3 cells have no vector width that divides their innermost extent, so
# they never stream.  The same operators on this many cells do, with slot shapes no other program has: a slot of
# age 3 parked at the start of the step, and two pairs of fields parked after one operator each.
ENLARGED_SHAPE = [16, 12, 32]
ENLARGED_RANGES = {"ref_simple_input_delay_buf": {"wtgfac": (0.5, 1.5)},
                   # arrA changes sign, so that both arms of kernelB's select are taken; every sum stays positive
                   "ref_simulator12": {"arrA": (-0.5, 1.0), "arrB": (0.5, 1.5), "arrC": (0.5, 1.5)}}

JAC_1 = {"a": 2, "b0": 2, "b1": 2, "b2": 2}
JAC_2 = {"b3": 2, "b4": 2, "b5": 2, "b6": 2}
HDIFF = {"inp": 3, "flx": 2}

# (program, plan options, environment, the tensor-memory slots {field: age} of each streamed launch with tmem=2)
MATRIX = [
    ("ref_jacobi3d_32x32x32_8itr_8vec", dict(GEO_A, sync="cta"), {}, [JAC_1, JAC_2]),
    ("ref_jacobi3d_32x32x32_8itr_8vec", dict(GEO_B, sync="cta"), {}, [JAC_1, JAC_2]),
    ("jacobi3d_16x24x32_5itr_const1", dict(GEO_A, sync="cta"), {}, [JAC_1, {"b3": 2}]),
    ("jacobi3d_16x24x32_5itr_const1", dict(GEO_B, sync="cta"), {}, [JAC_1, {"b3": 2}]),
    ("jacobi3d_24x20x40_4itr_shrink_f64", dict(GEO_A, sync="cta"), {}, [JAC_1]),
    ("jacobi3d_24x20x40_4itr_shrink_f64", dict(GEO_B, sync="cta"), {}, [JAC_1]),
    ("upwind3d_bwd_20x12x32_5st_f64", dict(GEO_A16, sync="cta"), {}, [JAC_1, {"b3": 2}]),
    ("upwind3d_bwd_20x12x32_5st_f64", dict(GEO_B, sync="cta"), {}, [JAC_1, {"b3": 2}]),
    ("hdiff_24x28x16", dict(GEO_B, sync="cta"), {}, [HDIFF]),
    ("hdiff_16x20x8_f64", dict(GEO_B, sync="cta"), {}, [HDIFF]),
    ("fork_join_20x16x24", dict(GEO_A, sync="cta"), {}, [{"a": 2, "d": 2}]),
    ("fork_join_20x16x24", dict(GEO_B, sync="cta"), {}, [{"a": 2, "d": 2}]),
    ("diamond3d_12x10x16", dict(GEO_B, sync="cta"), {}, [{"a": 2, "r": 2}]),
    ("trig3d_8x10x12_f64", dict(GEO_B, sync="cta"), {}, [{"a": 2, "u": 3}]),
    ("ref_simple_input_delay_buf", dict(GEO_B, max_depth=6, sync="cta"), {}, [{"ppgk": 3}]),
    ("ref_simple_input_delay_buf", dict(GEO_B, max_depth=6, rows_per_thread=2, sync="cta"), {}, [{"ppgk": 3}]),
    ("ref_simulator12", dict(GEO_B, max_depth=6, sync="cta"), {},
     [{"arrA": 1, "arrB": 3, "kernelD": 1, "kernelE": 1}]),
    ("synth_fork_16x12x16_5st", dict(GEO_B, sync="cta"), {}, [{"a": 2, "b0": 2, "b1": 2, "a1": 2}, {}, {}]),
    ("lowdim3d_20x24x48_3st_f32", dict(GEO_A, sync="cta"), {}, [{"a": 2, "b0": 2}]),
    ("lowdim3d_20x24x48_3st_f32", dict(GEO_B, sync="cta"), {}, [{"a": 2, "b0": 2}]),
    # (at d4r4w8p2 this pass unrolls 3 steps, an odd number, and keeps its planes in registers)
    ("sdfgexport_hdiff_jki_48x8x64_f64", dict(GEO_A16, sync="cta"), {}, [{"inp": 2, "lap": 1, "flx": 1}, {}]),
    # the synchronisation schemes, direct input rows and the generator switches, on Jacobi and hdiff
    ("ref_jacobi3d_32x32x32_8itr_8vec", dict(GEO_B, sync="pair"), {}, [JAC_1, JAC_2]),
    ("hdiff_24x28x16", dict(GEO_B, sync="pair"), {}, [HDIFF]),
    ("ref_jacobi3d_32x32x32_8itr_8vec", dict(GEO_A, sync="flags"), {}, [JAC_1, JAC_2]),
    ("jacobi3d_16x24x32_5itr_const1", dict(GEO_B, sync="flags"), {}, [JAC_1, {"b3": 2}]),
    ("jacobi3d_16x24x32_5itr_const1", dict(GEO_A, sync="halves"), {}, [JAC_1, {"b3": 2}]),
    ("hdiff_16x20x8_f64", dict(GEO_B, sync="halves"), {}, [HDIFF]),
    ("ref_jacobi3d_32x32x32_8itr_8vec", dict(GEO_B, sync="cta", direct=1), {}, [JAC_1, JAC_2]),
    ("hdiff_24x28x16", dict(GEO_B, sync="cta", direct=1), {}, [HDIFF]),
    ("jacobi3d_16x24x32_5itr_const1", dict(GEO_A, sync="cta"), {"SFB200_PERSISTENT": "1"}, [JAC_1, {"b3": 2}]),
    ("hdiff_16x20x8_f64", dict(GEO_B, sync="cta"), {"SFB200_PERSISTENT": "1"}, [HDIFF]),
    ("ref_jacobi3d_32x32x32_8itr_8vec", dict(GEO_A, sync="cta"), {"SFB200_HALO_SKIP": "1"}, [JAC_1, JAC_2]),
    ("jacobi3d_16x24x32_5itr_const1", dict(GEO_B, sync="cta"), {"SFB200_HALO_SKIP": "1"}, [JAC_1, {"b3": 2}]),
    ("jacobi3d_16x24x32_5itr_const1", dict(GEO_A, sync="cta"), {"SFB200_SPLITLOOP": "1"}, [JAC_1, {"b3": 2}]),
    ("hdiff_16x20x8_f64", dict(GEO_B, sync="cta"), {"SFB200_SPLITLOOP": "1"}, [HDIFF]),
]


def matrix_id(entry):
    name, opts, env, _ = entry
    s = "{}-d{}r{}w{}k{}p{}-{}".format(name, opts["max_depth"], opts["rows_per_thread"], opts["warps"],
                                       opts["threads_per_row"], opts["prefetch"], opts["sync"])
    if opts.get("direct"):
        s += "-direct"
    return s + "".join("-{}={}".format(k[7:], v) for k, v in sorted(env.items()))


def case_path(name):
    """The program file of a matrix entry (the enlarged copy for the reference's tiny 3-D programs)."""
    if name not in ENLARGED_RANGES:
        return program_path(name)
    from stencilflow_b200 import programs
    with open(program_path(name)) as f:
        prog = json.load(f)
    prog["dimensions"] = list(ENLARGED_SHAPE)
    for cfg in prog["inputs"].values():
        cfg["data"] = "constant:1.0"
    return programs.write_program(prog, "{}_{}".format(name, "x".join(map(str, ENLARGED_SHAPE))))


def case_inputs(name, path, seed):
    if name not in ENLARGED_RANGES:
        return random_inputs(name, seed=seed)
    from oracle import reference_numpy as rn
    info = rn.ProgramInfo(rn.load_program(path))
    rng = np.random.default_rng(seed)
    return {f: rng.uniform(*ENLARGED_RANGES[name][f], size=info.field_shape(f)).astype(info.field_type(f))
            for f in info.inputs}


@pytest.fixture(scope="module")
def gpu(native_lib):
    from stencilflow_b200 import runtime
    return runtime.Runtime.get()


def _check_one_cta_per_sm(prog):
    """Every CTA of a parked pass allocates all 512 columns: the driver must place exactly one on each SM."""
    sms = int(prog.rt.props.sm_count)
    for l in prog.lowered.launches:
        if l.family == "streamed" and l.info["tmem"]:
            assert prog._resident_ctas(l) == sms, (l.kernel, prog._resident_ctas(l), sms)


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
        _check_one_cta_per_sm(prog)
    finally:
        prog.close()
    return outs, [l for l in prog.lowered.launches if l.family == "streamed"]


@pytest.mark.parametrize("entry", MATRIX, ids=matrix_id)
def test_parked_planes_match_oracle_and_registers(gpu, entry, monkeypatch):
    from oracle import reference_numpy as rn
    from stencilflow_b200.planner import PlanOptions
    name, opts, env, slots = entry
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    path = case_path(name)
    inputs = case_inputs(name, path, seed=43)
    expected = rn.run_reference(path, inputs)
    h = HALO.get(name, 0)
    results = []
    for tmem in (2, 0):
        got, streamed = _run(path, inputs, PlanOptions(tmem=tmem, **opts))
        assert [l.info["tmem"] for l in streamed] == (slots if tmem else [{}] * len(slots)), tmem
        assert all(l.info["sync"] == opts["sync"] for l in streamed if l.info["tmem"])
        if "SFB200_PERSISTENT" in env:
            assert all(l.info["persistent"] for l in streamed)
        for field, ref in expected.items():
            err = rn.max_relative_error(rn.trim_halo(ref, h), rn.trim_halo(got[field], h))
            assert err <= TOL[ref.dtype.name], "tmem={} {}: max rel err {}".format(tmem, field, err)
        results.append({f: np.ascontiguousarray(rn.trim_halo(a, h)) for f, a in got.items()})
    for field in expected:
        on, off = results[0][field], results[1][field]
        assert on.tobytes() == off.tobytes(), "{}: {} cells differ".format(field, int(np.sum(on != off)))


def _checksums(path, runs, fills, out, dt, monkeypatch):
    """{label: checksum bits of ``out``}, {label: infos of the streamed launches}, {label: plan options}, each run
    executed three times on the same hash-filled inputs: columns and work-table counters left behind by earlier work
    items and launches are in play."""
    from stencilflow_b200.cuda_program import CudaProgram
    from stencilflow_b200.planner import PlanOptions
    sums, streamed, plans = {}, {}, {}
    for label, opts, env in runs:
        monkeypatch.delenv("SFB200_PERSISTENT", raising=False)
        for k, v in env.items():
            monkeypatch.setenv(k, v)
        p = CudaProgram(path, plan_options=None if opts is None else PlanOptions(**opts))
        try:
            n = int(np.prod(p.program.shape))
            for k, (name, (lo, hi)) in enumerate(sorted(fills.items())):
                p.rt.fill_hash(p.buffers[name].dptr, n, dt, seed=99 + k, lo=lo, hi=hi)
            for _ in range(3):
                p.execute()
            p.rt.stream_synchronize()
            sums[label] = p.rt.checksum(p.buffers[out].dptr, n, dt)[1]
            _check_one_cta_per_sm(p)
            streamed[label] = [l.info for l in p.lowered.launches if l.family == "streamed"]
            plans[label] = p.plan.options.as_dict()
        finally:
            p.close()
    return sums, streamed, plans


@pytest.mark.parametrize("planes", [320, 317])
def test_jacobi3d_default_plan_bit_identical_at_scale(gpu, planes, monkeypatch):
    """The Jacobi-3D chain on its default plan parks its planes and synchronises by per-field mbarriers; the result
    equals, bit for bit, the same geometry with the planes in registers and the one-operator kernels -- on the chunk
    grid and on persistent CTAs.  317 planes are no multiple of the 6-step unroll: segments start at other steps."""
    from stencilflow_b200 import programs
    from stencilflow_b200.planner import PlanOptions
    for knob in PlanOptions.KNOBS + ("SFB200_TUNED",):
        monkeypatch.delenv(knob, raising=False)
    path = programs.write_program(programs.jacobi3d_chain([planes, 448, 512], 8), "tmem_jacobi3d_{}".format(planes))
    fills = {"a": (0.0, 1.0)}
    sums, streamed, plans = _checksums(path, [("default", None, {})], fills, "b7", np.float32, monkeypatch)
    plan = plans["default"]
    assert [i["tmem"] for i in streamed["default"]] == [JAC_1, JAC_2]
    assert all(i["sync"] == "flags" for i in streamed["default"])
    more, streamed2, _ = _checksums(path, [("registers", dict(plan, tmem=0), {}),
                                        ("persistent", plan, {"SFB200_PERSISTENT": "1"}),
                                        ("persistent registers", dict(plan, tmem=0), {"SFB200_PERSISTENT": "1"}),
                                        ("unfused", dict(fuse=False), {})], fills, "b7", np.float32, monkeypatch)
    sums.update(more)
    streamed.update(streamed2)
    geometry = ("V", "R", "warps", "threads_per_row", "prefetch", "sync", "unroll")
    for label in ("registers", "persistent", "persistent registers"):
        assert [[i[k] for k in geometry] for i in streamed[label]] == [[i[k] for k in geometry] for i in streamed["default"]]
    assert [i["tmem"] for i in streamed["persistent"]] == [JAC_1, JAC_2]
    assert all(i["persistent"] for i in streamed["persistent"]) and not any(i["persistent"] for i in streamed["default"])
    assert not any(i["tmem"] for i in streamed["registers"] + streamed["persistent registers"])
    assert len(set(sums.values())) == 1, sums


def test_hdiff_parked_planes_bit_identical_at_scale(gpu, monkeypatch):
    """hdiff parks an age-3 slot of its input and one of ``flx`` (rows of 20 threads, the plan of BASELINE config 2
    with tmem=2): bit-identical to the planes in registers and to the one-operator kernels."""
    from stencilflow_b200 import programs
    path = programs.write_program(programs.hdiff([192, 256, 80]), "tmem_hdiff")
    plan = dict(max_depth=4, rows_per_thread=2, prefetch=2, sync="cta")
    fills = {"inp": (1.0, 2.0), "coeff": (0.0, 0.05)}
    sums, streamed, _ = _checksums(path, [("parked", dict(plan, tmem=2), {}), ("registers", dict(plan, tmem=0), {}),
                                       ("persistent", dict(plan, tmem=2), {"SFB200_PERSISTENT": "1"}),
                                       ("unfused", dict(fuse=False), {})], fills, "out", np.float32, monkeypatch)
    assert [i["tmem"] for i in streamed["parked"]] == [HDIFF] == [i["tmem"] for i in streamed["persistent"]]
    assert streamed["persistent"][0]["persistent"] and [i["tmem"] for i in streamed["registers"]] == [{}]
    assert len(set(sums.values())) == 1, sums
